"""CPU tier: the oracle port step by step against the unmodified reference (oracle/_ref/libminiasm_ref.so) --
this is what pins the restatement, since the reference has no tests of its own."""
import ctypes as C
import os

import numpy as np
import pytest

from miniasm_b200 import capi, synth
from oracle import loaders
from miniasm_b200.pipeline import Pipeline, canon_arcs
from tests import reference

SETS = ["tiny_exact", "chaos_small", "chaos", "bubbles800", "shuffled", "lowcov", "varlen300", "skew_small", "c1_ecoli_like"]


@pytest.fixture(scope="module")
def port(built):
    return loaders.load_oracle_port()


def mask(h):
    h = h.copy()
    h["bl_del"] &= 0x7fffffff
    return h


@pytest.mark.parametrize("name", SETS)
def test_port_matches_reference_stepwise(name, ref, port, paf_dir):
    paf = synth.generate(name, f"{paf_dir}/{name}.paf")
    r, p = Pipeline(ref, paf).read(), Pipeline(port, paf).read()
    assert reference.pin(r.names()) == p.names()
    reference.pin(reference.hits(r.hits_np()))
    assert np.array_equal(np.sort(mask(r.hits_np()), order=list(capi.HIT_DT.names)), np.sort(mask(p.hits_np()), order=list(capi.HIT_DT.names)))
    p.free()
    p = Pipeline(port, paf, opt=r.opt).adopt(r)      # continue from the reference's own (tie-ordered) hit array
    for step in ("sub1", "cut", "flt", "sub2_cut_merge", "contained"):
        getattr(r, step)(), getattr(p, step)()
        assert r.n_hits == p.n_hits and np.array_equal(mask(r.hits_np()), mask(p.hits_np())), step
        assert np.array_equal(r.sub_np(), p.sub_np()), step
        reference.pin((reference.hits(r.hits_np()), r.sub_np(), r.cov.value))
    assert reference.pin(r.names()) == p.names()
    r.sg_gen(), p.sg_gen()
    (ar, sr, ir, _, _), (ap, sp, ip, _, _) = r.graph_np(), p.graph_np()
    assert np.array_equal(canon_arcs(ar), canon_arcs(ap)) and np.array_equal(sr, sp) and np.array_equal(ir, ip)
    o = r.opt
    for fn, args in [("asg_arc_del_trans", (o.gap_fuzz,)), ("asg_cut_tip", (o.max_ext,)), ("asg_pop_bubble", (o.bub_dist,)),
                     ("asg_arc_del_short", (0.5,)), ("asg_cut_tip", (o.max_ext,)), ("asg_pop_bubble", (o.bub_dist,)),
                     ("asg_arc_del_short", (0.7,)), ("asg_cut_internal", (1,)), ("asg_cut_biloop", (o.max_ext,)),
                     ("asg_cut_tip", (o.max_ext,)), ("asg_pop_bubble", (o.bub_dist,)), ("asg_arc_del_short", (0.8,))]:
        g2 = port.clone_graph(r.sg)                  # same pre-state for both
        a = getattr(ref, fn)(r.sg, *args)
        b = getattr(port, fn)(g2, *args)
        assert a == b, fn
        x, y = ref.read_graph(r.sg), port.read_graph(g2)
        assert np.array_equal(x[0], y[0]) and np.array_equal(x[1], y[1]) and x[3:] == y[3:], fn
        port.asg_destroy(g2)
    ur, up = ref.ma_ug_gen(r.sg), port.ma_ug_gen(r.sg)
    assert ref.print_to_string("ma_ug_print", ur, r.d, r.sub) == ref.print_to_string("ma_ug_print", up, r.d, r.sub)
    ref.ma_ug_destroy(ur), port.ma_ug_destroy(up)
    r.free(), p.free()


def test_tie_order_audit(ref, port, paf_dir):
    """SURVEY.md section 7.1: the reference's radix sort is unstable, ours (port and CUDA) are stable.  On data with
    thousands of tied sort keys the final GFA must not depend on it."""
    for name in ("jitter30", "chaos"):
        paf = synth.generate(name, f"{paf_dir}/{name}.paf")
        assert Pipeline(ref, paf).run_all() == Pipeline(port, paf).run_all()


def _reduce_tied(lib, w2_first):
    from tests.tied_graph import FUZZ, tied_graph
    arcs, seq, idx = tied_graph(w2_first)
    g = lib.make_graph(arcs, seq, is_srt=True)
    g.contents.idx = capi.c_malloc_copy(idx)
    n = lib.asg_arc_del_trans(g, FUZZ)
    out = lib.read_graph(g)
    lib.asg_destroy(g)
    return n, out


def test_tied_arcs_decide_the_counter_not_the_graph(ref, port):
    """ADVICE round 1: two arcs tied on (source, length) whose targets overlap each other.  Which one the reference explores first
    changes how many arcs asg_arc_del_trans itself reduces (asg.c:164-171); asg_symm inside the call (asg.c:188-191) takes the
    one-sided survivor, so the graph that comes out is the same.  The port follows the reference for either slab order."""
    res = {}
    for w2_first in (False, True):
        nr, gr = _reduce_tied(ref, w2_first)
        n_p, gp = _reduce_tied(port, w2_first)
        assert nr == n_p
        assert np.array_equal(gr[0], gp[0]) and np.array_equal(gr[1], gp[1]) and np.array_equal(gr[2], gp[2]) and gr[3:] == gp[3:]
        res[w2_first] = (nr, gr)
    assert res[True][0] == res[False][0] + 1                     # v -> x is reduced by the pass itself only when w2 comes first
    assert np.array_equal(canon_arcs(res[True][1][0]), canon_arcs(res[False][1][0]))
    assert len(res[True][1][0]) == 6                             # v -> w1 -> w2 -> x and the complement chain remain


@pytest.mark.parametrize("args", ["-n 4000 -l 2000 -L 30000 -c 30 -j 100 -s 41", "-n 6000 -l 1500 -L 40000 -c 40 -j 300 -s 42 -d 20000"])
@pytest.mark.parametrize("hang,frac", [(1000, 0.8), (200, 0.5), (4000, 0.95)])
def test_port_no_cont(args, hang, frac, ref, port, paf_dir):
    """-R (SURVEY.md 8f row 2): ma_hit_no_cont (hit.c:38-68) and ma_hit_read with its exclusion list (hit.c:86) -- read lengths
    spread over a factor of 20, so many reads lie clearly inside a read twice as long."""
    paf = synth.generate(args, f"{paf_dir}/nocont_{len(args)}.paf").encode()
    dr, dp = ref.ma_hit_no_cont(paf, 2000, 100, hang, frac), port.ma_hit_no_cont(paf, 2000, 100, hang, frac)
    names = lambda d: [(d.contents.seq[i].name, d.contents.seq[i].len) for i in range(d.contents.n_seq)]
    assert reference.pin(names(dr)) == names(dp) and (len(names(dr)) > 20 or hang == 4000)
    out = []
    for lib, excl in ((ref, dr), (port, dp)):
        d, n = lib.sd_init(), C.c_size_t(0)
        h = lib.ma_hit_read(paf, 2000, 100, d, C.byref(n), 1, excl)
        a = mask(capi.np_from_ptr(h, n.value, capi.HIT_DT))
        out.append((names(d), np.sort(a, order=list(capi.HIT_DT.names))))
        capi.c_free(h), lib.sd_destroy(d)
    assert out[0][0] == out[1][0] and np.array_equal(out[0][1], out[1][1])
    reference.pin(out[0])
    gone = {nm for nm, _ in names(dr)}
    assert gone and not gone & {nm for nm, _ in out[0][0]}
    ref.sd_destroy(dr), port.sd_destroy(dp)


@pytest.mark.parametrize("style,ext", [("fa_wrap", "fa"), ("fa_one_crlf", "fa"), ("fa_var_gaps_extra_dups_missing", "fa"), ("fa_wrap", "fa.gz"),
                                       ("fq", "fq"), ("fq_crlf_extra_dups", "fq"), ("fq_missing", "fq.gz"), ("fq_multi", "fq")])
def test_port_ug_seq(style, ext, ref, port, paf_dir):
    """-f reads (SURVEY.md 8f row 3): ma_ug_seq (asm.c:236-290 over kseq.h:163-211) -- FASTA / FASTQ, wrapped, CRLF, gzip, empty
    lines, multi-line FASTQ, records missing / foreign / repeated; the port fills the unitigs the reference built."""
    from tests.test_cli_gpu import _reads_file
    paf = synth.generate("chaos_small", f"{paf_dir}/chaos_small.paf")
    reads = _reads_file(paf, f"{paf_dir}/port_{style}.{ext}", style).encode()
    r = Pipeline(ref, paf).read().select().sg_gen().clean().ug_gen()
    want = r.gfa(reads.decode())                                  # reference fills r.ug and prints it
    ug2 = ref.ma_ug_gen(r.sg)                                    # a second, empty layout of the same graph for the port
    dp = port.sd_init()                                          # (a dictionary's index is private to the library that made it)
    for i in range(r.d.contents.n_seq):
        port.sd_put(dp, r.d.contents.seq[i].name, r.d.contents.seq[i].len)
    assert port.ma_ug_seq(ug2, dp, r.sub, reads) == 0
    got = ref.print_to_string("ma_ug_print", ug2, r.d, r.sub)
    ref.ma_ug_destroy(ug2)
    assert got == want and b"\t*\tLN" not in want and want.count(b"S\t") > 0
    assert port.ma_ug_seq(ref.ma_ug_gen(r.sg), dp, r.sub, b"/nonexistent/reads.fa") == -1      # asm.c:243
    port.sd_destroy(dp)
    r.free()
