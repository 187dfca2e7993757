"""GPU parity of the string-graph container passes (SURVEY.md 8a rows a12-a18) against the
unmodified reference, function by function through the C ABI, on graphs the reference itself built."""
import ctypes as C

import numpy as np
import pytest

from miniasm_b200 import capi, synth
from miniasm_b200.capi import ARC_DT, DEL
from miniasm_b200.pipeline import Pipeline, canon_arcs
from tests import reference
from tests.tied_graph import FUZZ, tied_graph

pytestmark = pytest.mark.gpu

SETS = ["tiny_exact", "small_exact", "jitter30", "varlen300", "bubbles800", "chaos", "skew_small", "lowcov"]


@pytest.fixture(scope="module")
def graphs(ref, paf_dir):
    """name -> reference pipeline stopped right after ma_sg_gen (sorted + indexed raw graph)."""
    out = {}
    for name in SETS:
        paf = synth.generate(name, f"{paf_dir}/{name}.paf")
        out[name] = Pipeline(ref, paf).read().select().sg_gen()
    yield out
    for p in out.values():
        p.free()


def _clone_to(lib, src_lib, g):
    arcs, seq, idx, srt, symm = src_lib.read_graph(g)
    h = lib.make_graph(arcs, seq, srt, symm)
    if idx is not None:
        h.contents.idx = capi.c_malloc_copy(idx)
    return h


def _same_graph(prod, gp, ref, gr, exact_order=True):
    ap, sp, ip, srt_p, symm_p = prod.read_graph(gp)
    ar, sr, ir, srt_r, symm_r = ref.read_graph(gr)
    assert len(ap) == len(ar)
    assert np.array_equal(sp, sr)
    assert (srt_p, symm_p) == (srt_r, symm_r)
    if exact_order:
        assert np.array_equal(ap, ar)
    else:
        assert np.array_equal(ap["ul"], ar["ul"])          # same sort keys position by position
        assert np.array_equal(canon_arcs(ap), canon_arcs(ar))
    assert (ip is None) == (ir is None)
    if ip is not None:
        assert np.array_equal(ip, ir)


@pytest.mark.parametrize("name", SETS)
def test_del_trans(name, graphs, ref, prod):
    p = graphs[name]
    gr, gp = _clone_to(ref, ref, p.sg), _clone_to(prod, ref, p.sg)
    nr = ref.asg_arc_del_trans(gr, p.opt.gap_fuzz)
    n_p = prod.asg_arc_del_trans(gp, p.opt.gap_fuzz)
    assert n_p == nr
    _same_graph(prod, gp, ref, gr)
    ref.asg_destroy(gr), prod.asg_destroy(gp)


@pytest.mark.parametrize("fuzz", [0, 10, 100000])
def test_del_trans_fuzz(fuzz, graphs, ref, prod):
    p = graphs["chaos"]
    gr, gp = _clone_to(ref, ref, p.sg), _clone_to(prod, ref, p.sg)
    assert prod.asg_arc_del_trans(gp, fuzz) == ref.asg_arc_del_trans(gr, fuzz)
    _same_graph(prod, gp, ref, gr)
    ref.asg_destroy(gr), prod.asg_destroy(gp)


def test_del_trans_deleted_reads(graphs, ref, prod):
    """reads flagged del lose every arc (asg.c:158-161)."""
    p = graphs["jitter30"]
    arcs, seq, idx, _, _ = ref.read_graph(p.sg)
    seq = seq.copy()
    seq[::7] |= DEL
    gr, gp = ref.make_graph(arcs, seq, True), prod.make_graph(arcs, seq, True)
    gr.contents.idx, gp.contents.idx = capi.c_malloc_copy(idx), capi.c_malloc_copy(idx)
    assert prod.asg_arc_del_trans(gp, 1000) == ref.asg_arc_del_trans(gr, 1000)
    _same_graph(prod, gp, ref, gr)
    ref.asg_destroy(gr), prod.asg_destroy(gp)


@pytest.mark.parametrize("w2_first", [False, True])
def test_del_trans_tied_arcs(w2_first, ref, prod):
    """Two arcs tied on (source, length) whose targets overlap each other (tests/tied_graph.py): for either slab order the kernel
    reduces what the reference's sequential walk reduces -- the counter differs between the two orders, never between the two sides."""
    arcs, seq, idx = tied_graph(w2_first)
    gr, gp = ref.make_graph(arcs, seq, True), prod.make_graph(arcs, seq, True)
    gr.contents.idx, gp.contents.idx = capi.c_malloc_copy(idx), capi.c_malloc_copy(idx)
    nr = ref.asg_arc_del_trans(gr, FUZZ)
    assert prod.asg_arc_del_trans(gp, FUZZ) == nr
    assert nr == (4 if w2_first else 3)                        # v -> x is reduced by the pass itself only when w2 is walked first
    _same_graph(prod, gp, ref, gr)
    ref.asg_destroy(gr), prod.asg_destroy(gp)


@pytest.mark.parametrize("name", ["small_exact", "chaos", "skew_small"])
def test_cleanup_sorts_and_indexes(name, graphs, ref, prod):
    """asg_cleanup on a shuffled, partly deleted arc set: rm + sort + index (asg.c:57-80)."""
    p = graphs[name]
    arcs, seq, _, _, _ = ref.read_graph(p.sg)
    rng = np.random.default_rng(7)
    arcs = arcs[rng.permutation(len(arcs))].copy()
    arcs["ol_del"][rng.random(len(arcs)) < 0.1] |= DEL
    seq = seq.copy()
    seq[rng.random(len(seq)) < 0.02] |= DEL
    gr, gp = ref.make_graph(arcs, seq), prod.make_graph(arcs, seq)
    ref.asg_cleanup(gr), prod.asg_cleanup(gp)
    _same_graph(prod, gp, ref, gr, exact_order=False)   # the reference's radix sort is unstable: ties may permute
    a = prod.read_graph(gp)[0]
    assert np.all(a["ul"][1:] >= a["ul"][:-1])
    ref.asg_destroy(gr), prod.asg_destroy(gp)


@pytest.mark.parametrize("name", ["chaos", "bubbles800", "skew_small"])
def test_symm(name, graphs, ref, prod):
    """asg_symm = del_multi + del_asymm (asg.c:104-145) on a graph with planted duplicates / one-sided arcs."""
    p = graphs[name]
    arcs, seq, _, _, _ = ref.read_graph(p.sg)
    rng = np.random.default_rng(11)
    dup = arcs[rng.random(len(arcs)) < 0.01].copy()
    dup["ul"] += 3                                          # same source + target, longer: a multi-arc
    arcs = np.concatenate([arcs[rng.random(len(arcs)) > 0.01], dup])
    gr, gp = ref.make_graph(arcs, seq), prod.make_graph(arcs, seq)
    ref.asg_cleanup(gr), prod.asg_cleanup(gp)
    ref.asg_symm(gr), prod.asg_symm(gp)
    _same_graph(prod, gp, ref, gr, exact_order=False)
    ref.asg_destroy(gr), prod.asg_destroy(gp)


@pytest.mark.parametrize("ratio", [0.5, 0.6, 0.7, 0.8, 0.95])
def test_del_short(ratio, graphs, ref, prod):
    p = graphs["chaos"]
    gr = _clone_to(ref, ref, p.sg)
    ref.asg_arc_del_trans(gr, 1000)
    gp = _clone_to(prod, ref, gr)
    assert prod.asg_arc_del_short(gp, ratio) == ref.asg_arc_del_short(gr, ratio)
    _same_graph(prod, gp, ref, gr)
    ref.asg_destroy(gr), prod.asg_destroy(gp)


def test_big_slabs(ref, prod):
    """A hub vertex beyond the warp kernel (128 arcs) and beyond the CTA kernel (8192 arcs)."""
    rng = np.random.default_rng(5)
    n_seq = 12000
    seq = np.full(n_seq, 20000, dtype=np.uint32)
    rows = []
    def add(u, v, l):
        rows.append((u << 32 | l, v, 20000 - l))
        rows.append(((v ^ 1) << 32 | l, u ^ 1, 20000 - l))
    for hub, deg in ((0, 300), (2, 5000), (4, 9000)):
        tg = rng.choice(np.arange(6, 2 * n_seq), size=deg, replace=False)
        ls = np.sort(rng.integers(1, 18000, size=deg))
        for t, l in zip(tg, ls):
            add(hub, int(t), int(l))
        for k in range(0, deg - 1, 3):                      # chain some targets so that reductions happen
            add(int(tg[k]), int(tg[k + 1]), int(max(1, ls[k + 1] - ls[k])))
    arcs = np.array(rows, dtype=ARC_DT)
    gr = ref.make_graph(arcs, seq)
    ref.asg_cleanup(gr)
    gp = _clone_to(prod, ref, gr)      # same slab order on both sides: lengths tie heavily here (DESIGN.md "tie order")
    raw = reference.unpinned(ref)      # so the reduction follows the slab order: compared with the product only
    assert prod.asg_arc_del_trans(gp, 1000) == raw.asg_arc_del_trans(gr, 1000)
    _same_graph(prod, gp, raw, gr)
    ref.asg_destroy(gr), prod.asg_destroy(gp)


def test_empty_graph(ref, prod):
    seq = np.full(10, 5000, dtype=np.uint32)
    gp = prod.make_graph(np.zeros(0, dtype=ARC_DT), seq)
    prod.asg_cleanup(gp)
    assert prod.asg_arc_del_trans(gp, 1000) == 0
    arcs, s, idx, srt, _ = prod.read_graph(gp)
    assert len(arcs) == 0 and srt and idx is not None and not idx.any()
    prod.asg_destroy(gp)
