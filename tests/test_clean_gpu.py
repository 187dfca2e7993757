"""GPU parity of stage (iii) (SURVEY.md 8a rows a18-a25): the order-dependent cleaning passes, unitig
construction and the final GFA, against the unmodified reference on graphs with tips, bubbles, short
overlaps, internal sequences and bi-loops."""
import ctypes as C
import gzip
import os

import numpy as np
import pytest

from miniasm_b200 import capi, synth
from miniasm_b200.pipeline import Pipeline, gfa_canon
from tests import reference

pytestmark = pytest.mark.gpu

NOISY = ["bubbles800", "chaos", "chaos_small", "shuffled", "varlen300", "lowcov", "c1_ecoli_like", "jitter30"]
ALL = NOISY + ["tiny_exact", "small_exact", "skew_small"]


@pytest.fixture(scope="module")
def pafs(paf_dir):
    return {name: synth.generate(name, f"{paf_dir}/{name}.paf") for name in ALL}


def _clone_to(lib, src_lib, g):
    arcs, seq, idx, srt, symm = src_lib.read_graph(g)
    h = lib.make_graph(arcs, seq, srt, symm)
    if idx is not None:
        h.contents.idx = capi.c_malloc_copy(idx)
    return h


def _assert_same(prod, gp, ref, gr):
    ap, sp, ip, f1, f2 = prod.read_graph(gp)
    ar, sr, ir, g1, g2 = ref.read_graph(gr)
    assert np.array_equal(ap, ar) and np.array_equal(sp, sr) and (f1, f2) == (g1, g2)
    assert (ip is None) == (ir is None) and (ip is None or np.array_equal(ip, ir))


def _step(name, ref, prod, gr, *args):
    """Run one pass on the reference graph and, from the same pre-state, on the product; compare."""
    gp = _clone_to(prod, ref, gr)
    rr = getattr(ref, name)(gr, *args)
    rp = getattr(prod, name)(gp, *args)
    assert rp == rr, f"{name}: count {rp} != {rr}"
    _assert_same(prod, gp, ref, gr)
    prod.asg_destroy(gp)
    return rr


@pytest.mark.parametrize("name", NOISY)
def test_cleaning_passes_stepwise(name, pafs, ref, prod):
    r = Pipeline(ref, pafs[name]).read().select().sg_gen()
    o, g = r.opt, r.sg
    ref.asg_arc_del_trans(g, o.gap_fuzz)
    counts = {}
    counts["tip"] = _step("asg_cut_tip", ref, prod, g, o.max_ext)
    counts["bub"] = _step("asg_pop_bubble", ref, prod, g, o.bub_dist)
    for i in range(o.n_rounds + 1):
        ratio = float(np.float32(o.min_ovlp_drop_ratio) + (np.float32(o.max_ovlp_drop_ratio) - np.float32(o.min_ovlp_drop_ratio))
                      / np.float32(o.n_rounds) * np.float32(i))
        if _step("asg_arc_del_short", ref, prod, g, ratio):
            _step("asg_cut_tip", ref, prod, g, o.max_ext)
            _step("asg_pop_bubble", ref, prod, g, o.bub_dist)
    _step("asg_cut_internal", ref, prod, g, 1)
    _step("asg_cut_biloop", ref, prod, g, o.max_ext)
    _step("asg_cut_tip", ref, prod, g, o.max_ext)
    _step("asg_pop_bubble", ref, prod, g, o.bub_dist)
    if _step("asg_arc_del_short", ref, prod, g, o.final_ovlp_drop_ratio):
        _step("asg_cut_tip", ref, prod, g, o.max_ext)
        _step("asg_pop_bubble", ref, prod, g, o.bub_dist)
    # unitigs from the cleaned graph
    gp = _clone_to(prod, ref, g)
    ur, up = ref.ma_ug_gen(g), prod.ma_ug_gen(gp)
    tr = ref.print_to_string("ma_ug_print", ur, r.d, r.sub)
    tp = ref.print_to_string("ma_ug_print", up, r.d, r.sub)      # product structs through the reference's own writer
    tq = prod.print_to_string("ma_ug_print", up, r.d, r.sub)     # ... and through ours
    assert tp == tr and tq == tr
    ref.ma_ug_destroy(ur), prod.ma_ug_destroy(up), prod.asg_destroy(gp)
    r.free()


@pytest.mark.parametrize("ext,dist", [(1, 50000), (2, 5000), (8, 200000), (20, 1000)])
def test_cleaning_other_parameters(ext, dist, pafs, ref, prod):
    r = Pipeline(ref, pafs["chaos"]).read().select().sg_gen()
    g = r.sg
    ref.asg_arc_del_trans(g, 1000)
    _step("asg_cut_tip", ref, prod, g, ext)
    _step("asg_pop_bubble", ref, prod, g, dist)
    _step("asg_cut_internal", ref, prod, g, ext)
    _step("asg_cut_biloop", ref, prod, g, ext)
    r.free()


@pytest.mark.parametrize("name", ["chaos", "bubbles800", "tiny_exact"])
def test_ug_gen_on_raw_graph(name, pafs, ref, prod):
    """`-S5 -p ug`: unitigs straight from ma_sg_gen's graph (not symmetric: the literal replay path)."""
    r = Pipeline(ref, pafs[name]).read().select().sg_gen()
    gp = _clone_to(prod, ref, r.sg)
    ur, up = ref.ma_ug_gen(r.sg), prod.ma_ug_gen(gp)
    raw = reference.unpinned(ref)      # the raw graph's tied arcs order the unitig links: compared with the product only
    assert raw.print_to_string("ma_ug_print", up, r.d, r.sub) == raw.print_to_string("ma_ug_print", ur, r.d, r.sub)
    ref.ma_ug_destroy(ur), prod.ma_ug_destroy(up), prod.asg_destroy(gp)
    r.free()


@pytest.mark.parametrize("name", ALL)
def test_gfa_end_to_end(name, pafs, ref, prod):
    """The whole drop-in path, every call on the GPU: byte-identical GFA (and equal as sorted S/L/a/x multisets)."""
    tr = Pipeline(ref, pafs[name]).run_all()
    tp = Pipeline(prod, pafs[name]).run_all()
    assert gfa_canon(tp) == gfa_canon(tr)
    assert tp == tr


def _write_reads(paf, path, gz=False, fastq=False):
    lens = {}
    with open(paf) as f:
        for line in f:
            t = line.split("\t")
            lens[t[0]] = int(t[1]); lens[t[5]] = int(t[6])
    rng = np.random.default_rng(3)
    op = gzip.open if gz else open
    with op(path, "wt") as f:
        for k, (nm, ln) in enumerate(sorted(lens.items())):
            s = "".join(np.array(list("ACGTNacgtRY"))[rng.integers(0, 11, ln)])
            if fastq:
                f.write(f"@{nm} extra comment\n{s}\n+\n{'I' * ln}\n")
            else:
                f.write(f">{nm}\n" + "\n".join(s[i:i + 70] for i in range(0, ln, 70)) + "\n")
    return path


@pytest.mark.parametrize("fmt", ["fa", "fq.gz"])
def test_gfa_with_sequences(fmt, pafs, ref, prod, paf_dir):
    """-f reads: S lines carry the unitig sequence (ma_ug_seq, asm.c:236-290)."""
    paf = pafs["chaos_small"]
    reads = _write_reads(paf, os.path.join(paf_dir, f"reads.{fmt}"), gz=fmt.endswith("gz"), fastq=fmt.startswith("fq"))
    tr = Pipeline(ref, paf).run_all(reads)
    tp = Pipeline(prod, paf).run_all(reads)
    assert tp == tr and b"\tLN:i:" in tp and not tp.startswith(b"S\tutg000001l\t*")
