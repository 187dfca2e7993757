"""CPU tier: the integer-conversion rules of ma_hit_cut (hit.c:162-193) and ma_hit2arc (miniasm.h:86-104) as the CUDA kernels
compile them (miniasm_b200/csrc/hit2arc.cuh, built for the host by tests/hostsim/hit_host.cpp), fuzzed against the unmodified
reference with hits no synthetic PAF produces: ends outside the kept intervals, wrapped spans (qe < qs), empty and deleted
intervals, self hits, palindromic self hits, every threshold from tiny to huge (SURVEY.md section 7 "hard part 2": which
comparisons are signed and which unsigned is part of the behaviour)."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from miniasm_b200 import capi
from miniasm_b200.capi import ARC_DT, DEL, HIT_DT, SUB_DT
from miniasm_b200.pipeline import canon_arcs
from tests import reference


ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SIM_SRC = os.path.join(ROOT, "tests", "hostsim", "hit_host.cpp")
SIM_SO = os.path.join(ROOT, "tests", "hostsim", "libhit_host.so")
HDRS = [os.path.join(ROOT, "miniasm_b200", "csrc", h) for h in ("hit2arc.cuh", "mab_common.cuh", "basecomp.cuh")]
CUDA_INC = "/usr/local/cuda/include"


@pytest.fixture(scope="module")
def sim(built):
    if not os.path.exists(SIM_SO) or os.path.getmtime(SIM_SO) < max(os.path.getmtime(p) for p in [SIM_SRC] + HDRS):
        # -ffp-contract=off: the one float product of ma_hit2arc is a plain IEEE multiply on both sides (the kernels use __fmul_rn)
        subprocess.run(["g++", "-O2", "-std=c++17", "-Wall", "-Wno-attributes", "-ffp-contract=off", "-shared", "-fPIC", "-I", CUDA_INC,
                        "-o", SIM_SO, SIM_SRC], check=True)
    dll = C.CDLL(SIM_SO)
    dll.hs_hit_cut.restype, dll.hs_hit_cut.argtypes = C.c_size_t, [C.c_void_p, C.c_int, C.c_size_t, C.c_void_p]
    dll.hs_hit_flt.restype, dll.hs_hit_flt.argtypes = C.c_size_t, [C.c_void_p, C.c_int, C.c_int, C.c_size_t, C.c_void_p, C.POINTER(C.c_ulonglong)]
    dll.hs_sg_arcs.restype = C.c_size_t
    dll.hs_sg_arcs.argtypes = [C.c_int, C.c_float, C.c_int, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p]
    dll.hs_comp.restype, dll.hs_comp.argtypes = C.c_ubyte, [C.c_ubyte]
    dll.hs_hit2arc.restype = C.c_int
    dll.hs_hit2arc.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_float, C.c_int, C.c_void_p]
    return dll


def layout_hits(rng, sub, n):
    """Hits between reads laid out on a line (random strands), alignment ends pulled in by U[0,1500] with probability 1/2 each:
    dovetails, containments and internal matches whose overhangs straddle the thresholds the tests sweep."""
    n_seq = len(sub)
    ln = (sub["e"] - (sub["s_del"] & np.uint32(0x7fffffff))).astype(np.int64)
    pos = rng.integers(0, 60000, n_seq)
    strand = rng.integers(0, 2, n_seq)
    q, t = rng.integers(0, n_seq, 4 * n), rng.integers(0, n_seq, 4 * n)
    a, b = np.maximum(pos[q], pos[t]), np.minimum(pos[q] + ln[q], pos[t] + ln[t])
    ok = (b - a > 200) & (q != t)
    q, t, a, b = q[ok][:n], t[ok][:n], a[ok][:n], b[ok][:n]
    m = len(q)
    b0 = b
    a = np.minimum(a + np.where(rng.random(m) < 0.5, rng.integers(0, 1500, m), 0), b0 - 1)
    b = np.maximum(b0 - np.where(rng.random(m) < 0.5, rng.integers(0, 1500, m), 0), a + 1)

    def on_read(r):
        lo, hi = a - pos[r], b - pos[r]
        return np.where(strand[r] == 1, ln[r] - hi, lo), np.where(strand[r] == 1, ln[r] - lo, hi)
    qs, qe = on_read(q)
    ts, te = on_read(t)
    h = np.zeros(m, dtype=HIT_DT)
    h["qns"] = (q.astype(np.uint64) << np.uint64(32)) | qs.astype(np.uint64)
    h["qe"], h["tn"], h["ts"], h["te"] = qe.astype(np.uint32), t.astype(np.uint32), ts.astype(np.uint32), te.astype(np.uint32)
    h["ml_rev"] = ((qe - qs) // 2).astype(np.uint32) | ((strand[q] != strand[t]).astype(np.uint32) << np.uint32(31))
    h["bl_del"] = (qe - qs).astype(np.uint32)
    return h[np.argsort(h["qns"], kind="stable")]


def fuzz(seed, n_seq=64, n=20000, wild=True):
    """Random interval table and hits.  wild=False keeps every hit inside the kept intervals (what the later stages see after
    ma_hit_cut); wild=True lets coordinates fall anywhere, spans wrap and intervals be empty or deleted; wild="layout": hits of a
    consistent layout (layout_hits), coordinates relative to the kept intervals."""
    rng = np.random.default_rng(seed)
    s = rng.integers(0, 4000, n_seq).astype(np.uint32)
    ln = rng.integers(0, 14000, n_seq).astype(np.uint32)
    ln[rng.random(n_seq) < 0.05] = 0                                    # empty kept interval
    sub = np.zeros(n_seq, dtype=SUB_DT)
    sub["s_del"], sub["e"] = s, s + ln
    if wild == "layout":
        return sub, layout_hits(rng, sub, n)
    if wild:
        sub["s_del"][rng.random(n_seq) < 0.08] |= DEL                   # reads ma_hit_sub dropped
    h = np.zeros(n, dtype=HIT_DT)
    q, t = rng.integers(0, n_seq, n), rng.integers(0, n_seq, n)
    same = rng.random(n) < 0.03
    t[same] = q[same]                                                   # self hits
    base_q = np.where(wild, 0, 0) + (sub["s_del"][q] & 0x7fffffff if wild else 0)
    lim_q = (sub["e"][q] if wild else ln[q]).astype(np.int64)
    lim_t = (sub["e"][t] if wild else ln[t]).astype(np.int64)
    base_t = (sub["s_del"][t] & 0x7fffffff) if wild else np.zeros(n, dtype=np.int64)

    def span(base, lim):
        a = base + rng.integers(-2500 if wild else 0, 6000, n)
        b = lim - rng.integers(-2500 if wild else 0, 6000, n)
        a = np.clip(a, 0, None)
        if not wild:
            a, b = np.clip(a, 0, lim), np.clip(b, 0, lim)
            a, b = np.minimum(a, b), np.maximum(a, b)
        return a.astype(np.int64), np.clip(b, 0, None).astype(np.int64)
    qs, qe = span(np.asarray(base_q, dtype=np.int64), lim_q)
    ts, te = span(np.asarray(base_t, dtype=np.int64), lim_t)
    pal = same & (rng.random(n) < 0.5)                                  # palindromic self hits (asm.c:27)
    ts[pal], te[pal] = qs[pal], qe[pal]
    rev = rng.random(n) < 0.5
    rev[pal] = True
    bl = np.maximum(np.abs(qe - qs), np.abs(te - ts)) + rng.integers(0, 50, n)
    ml = (bl * rng.random(n)).astype(np.int64)
    h["qns"] = (q.astype(np.uint64) << np.uint64(32)) | (qs.astype(np.uint64) & np.uint64(0xffffffff))
    h["qe"], h["tn"], h["ts"], h["te"] = qe.astype(np.uint32), t.astype(np.uint32), ts.astype(np.uint32), te.astype(np.uint32)
    h["ml_rev"] = (ml.astype(np.uint32) & np.uint32(0x7fffffff)) | (rev.astype(np.uint32) << np.uint32(31))
    h["bl_del"] = bl.astype(np.uint32) & np.uint32(0x7fffffff)
    order = np.argsort(h["qns"], kind="stable")                          # the arrays the reference passes around are sorted by qns
    return sub, h[order]


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


@pytest.mark.parametrize("seed", range(6))
@pytest.mark.parametrize("min_span", [1, 500, 2000, 9000])
def test_cut(seed, min_span, ref, sim):
    sub, h = fuzz(seed)
    a, b = h.copy(), h.copy()
    na = ref.ma_hit_cut(_ptr(sub), min_span, len(a), _ptr(a))
    nb = sim.hs_hit_cut(_ptr(sub), min_span, len(b), _ptr(b))
    assert na == nb and 0 < na < len(h)
    assert np.array_equal(reference.pin(a[:na]), b[:nb])


@pytest.mark.parametrize("seed", range(6))
@pytest.mark.parametrize("max_hang,min_ovlp", [(1500, 1000), (0, 0), (50, 5000), (100000, 1), (700, 20000)])
@pytest.mark.parametrize("wild", [False, True, "layout"])
def test_flt(seed, max_hang, min_ovlp, wild, ref, sim):
    sub, h = fuzz(100 + seed, wild=wild)
    a, b = h.copy(), h.copy()
    cov = C.c_float(0)
    na = ref.ma_hit_flt(_ptr(sub), max_hang, min_ovlp, len(a), _ptr(a), C.byref(cov))
    dp = C.c_ulonglong(0)
    nb = sim.hs_hit_flt(_ptr(sub), max_hang, min_ovlp, len(b), _ptr(b), C.byref(dp))
    assert na == nb
    assert np.array_equal(reference.pin(a[:na]), b[:nb])
    reference.pin(cov.value)
    if na:                                                               # the coverage the reference logs: tot_dp / tot_len (hit.c:208-212)
        k = a[:na]
        qid = (k["qns"] >> np.uint64(32)).astype(np.int64)
        last = np.r_[qid[1:] != qid[:-1], True]
        tot_len = int(((sub["e"][qid[last]] - (sub["s_del"][qid[last]] & 0x7fffffff)) & 0xffffffff).astype(np.uint64).sum())
        if tot_len:
            assert np.float32(dp.value / tot_len) == np.float32(cov.value)


@pytest.mark.parametrize("seed", range(6))
@pytest.mark.parametrize("max_hang,int_frac,min_ovlp", [(1000, 0.8, 2000), (0, 0.8, 2000), (1000, 0.0, 0), (1000, 1.0, 2000), (30000, 0.3, 1), (200, 0.95, 12000)])
@pytest.mark.parametrize("wild", [False, True, "layout"])
def test_sg_gen(seed, max_hang, int_frac, min_ovlp, wild, ref, sim):
    sub, h = fuzz(200 + seed, wild=wild)
    n_seq = len(sub)
    opt = ref.default_opt()
    opt.max_hang, opt.int_frac, opt.min_ovlp = max_hang, int_frac, min_ovlp
    d = ref.sd_init()
    for i in range(n_seq):
        ref.sd_put(d, f"r{i}".encode(), 20000)
    g = ref.ma_sg_gen(C.byref(opt), d, _ptr(sub), len(h), _ptr(h))
    arcs_r, seq_r, _, _, _ = ref.read_graph(g)
    ref.asg_destroy(g), ref.sd_destroy(d)

    seq = ((sub["e"] - (sub["s_del"] & np.uint32(0x7fffffff))) & np.uint32(0x7fffffff)) | (sub["s_del"] & DEL)   # asm.c:14-17
    seq = seq.astype(np.uint32)
    out = np.zeros(len(h), dtype=ARC_DT)
    m = sim.hs_sg_arcs(max_hang, int_frac, min_ovlp, len(h), _ptr(h), _ptr(seq), _ptr(out))
    arcs = out[:m]
    assert np.array_equal(seq, seq_r)
    dead = (seq & DEL) != 0                                              # asg_cleanup: asg_arc_rm + sort (asg.c:57-80)
    u, v = (arcs["ul"] >> np.uint64(33)).astype(np.int64), (arcs["v"] >> 1).astype(np.int64)
    arcs = arcs[~dead[u] & ~dead[v]]
    assert len(arcs) == len(arcs_r)
    assert np.array_equal(canon_arcs(arcs), canon_arcs(arcs_r))


def test_fuzz_reaches_every_class(sim):
    """What the inputs above exercise: every return class of ma_hit2arc, both strands, both arc directions."""
    seen = {}
    for wild in (False, True, "layout"):
        sub, h = fuzz(300, wild=wild)
        ln = (sub["e"] - (sub["s_del"] & np.uint32(0x7fffffff))).astype(np.int64)
        t = np.zeros(1, dtype=ARC_DT)
        for i in range(0, len(h), 7):
            r = sim.hs_hit2arc(_ptr(h[i:i + 1]), int(ln[int(h["qns"][i]) >> 32]) & 0x7fffffff, int(ln[h["tn"][i]]) & 0x7fffffff, 1000, 0.8, 2000, _ptr(t))
            key = ("arc", int(t["ul"][0] >> np.uint64(32)) & 1, int(h["ml_rev"][i] >> 31)) if r >= 0 else r
            seen[key] = seen.get(key, 0) + 1
    for cls in (-1, -2, -3, -4, ("arc", 0, 0), ("arc", 0, 1), ("arc", 1, 0), ("arc", 1, 1)):
        assert seen.get(cls, 0) > 0, (cls, seen)


def test_complement_of_every_byte(ref, sim, tmp_path):
    """The reverse-strand copy of ma_ug_seq (asm.c:277-282): complement through comp_tab (asm.c:224-233), bytes >= 128 become N.  The
    gather kernel of `-f reads` computes it arithmetically (basecomp.cuh); all byte values a FASTA line can carry are compared with
    what the reference's own ma_ug_seq writes for a one-read unitig on the reverse strand."""
    vals = [c for c in range(1, 256) if c not in (10, 13)]          # NUL, LF, CR cannot be sequence bytes of a FASTA line
    seq = bytes(vals) + b"ACGTacgtNn"
    fa = tmp_path / "all_bytes.fa"
    fa.write_bytes(b">r0\n" + seq + b"\n")
    d = ref.sd_init()
    ref.sd_put(d, b"r0", len(seq))
    item = np.array([(0 << 33) | (1 << 32) | len(seq)], dtype=np.uint64)       # read 0, reverse strand, whole length
    utg = (capi.MaUtg * 1)()
    utg[0].len_circ, utg[0].start, utg[0].end, utg[0].n, utg[0].m = len(seq), 1, 0, 1, 1
    utg[0].a, utg[0].s = item.ctypes.data_as(C.POINTER(C.c_uint64)), None
    ug = capi.MaUg()
    ug.n = ug.m = 1
    ug.a, ug.g = C.cast(utg, C.POINTER(capi.MaUtg)), None
    assert ref.ma_ug_seq(C.pointer(ug), d, None, str(fa).encode()) == 0
    got = C.string_at(C.cast(utg[0].s, C.c_void_p), len(seq))        # the unitig as the reference filled it
    want = bytes(sim.hs_comp(c) for c in reversed(seq))
    assert reference.pin(got) == want
    assert got != bytes(reversed(seq))                               # (it is not the identity)
    ref.sd_destroy(d)
    # the host reader of the drop-in level (host/gfa.c ma_ug_seq, also the fallback for multi-line FASTQ) on the same file
    prod = capi.load_product(strict=False)
    d2 = prod.sd_init()
    prod.sd_put(d2, b"r0", len(seq))
    utg2 = (capi.MaUtg * 1)()
    utg2[0].len_circ, utg2[0].start, utg2[0].end, utg2[0].n, utg2[0].m = len(seq), 1, 0, 1, 1
    utg2[0].a, utg2[0].s = item.ctypes.data_as(C.POINTER(C.c_uint64)), None
    ug2 = capi.MaUg()
    ug2.n = ug2.m = 1
    ug2.a, ug2.g = C.cast(utg2, C.POINTER(capi.MaUtg)), None
    assert prod.ma_ug_seq(C.pointer(ug2), d2, None, str(fa).encode()) == 0
    assert C.string_at(C.cast(utg2[0].s, C.c_void_p), len(seq)) == want
    prod.sd_destroy(d2)
