"""GPU parity of stage (i) (SURVEY.md 8a rows a4-a11): every drop-in entry point of hit.c / ma_sg_gen is run
on the state the unmodified reference produced for the previous step and compared bit for bit."""
import ctypes as C

import numpy as np
import pytest

from miniasm_b200 import capi, synth
from miniasm_b200.capi import HIT_DT, SUB_DT
from miniasm_b200.pipeline import Pipeline, canon_arcs
from tests import reference

pytestmark = pytest.mark.gpu

SETS = ["tiny_exact", "jitter30", "varlen300", "bubbles800", "chaos", "chaos_small", "shuffled", "skew_small", "lowcov", "c1_ecoli_like"]


def canon_mask(h):
    h = h.copy()
    h["bl_del"] &= 0x7fffffff
    return h


def canon_hits(h):
    h = h.copy()
    h["bl_del"] &= 0x7fffffff      # ma_hit_t::del is never written by the reference (uninitialised heap bit, hit.c:87-98)
    return np.sort(h, order=["qns", "tn", "qe", "ts", "te", "ml_rev", "bl_del"])


@pytest.fixture(scope="module")
def pafs(paf_dir):
    return {name: synth.generate(name, f"{paf_dir}/{name}.paf") for name in SETS}


@pytest.mark.parametrize("name", SETS)
def test_stage_i_stepwise(name, pafs, ref, prod):
    r = Pipeline(ref, pafs[name]).read()
    p = Pipeline(prod, pafs[name]).read()
    # ma_hit_read: same ids/names, same multiset of hits, same key order (ties may permute: unstable reference sort)
    assert reference.pin(r.names()) == p.names() and np.array_equal(reference.pin(r.seq_lens()), p.seq_lens())
    hr, hp = r.hits_np(), p.hits_np()
    reference.pin(reference.hits(hr))
    assert len(hr) == len(hp) and np.array_equal(hr["qns"], hp["qns"])
    assert np.array_equal(canon_hits(hr), canon_hits(hp))

    def fresh():
        return Pipeline(prod, pafs[name], opt=r.opt).adopt(r)

    def same_hits(x, y):
        reference.pin(reference.hits(x.hits_np()))
        return x.n_hits == y.n_hits and np.array_equal(canon_mask(x.hits_np()), canon_mask(y.hits_np()))

    # ma_hit_sub (round 1)
    q = fresh()
    r.sub1(), q.sub1()
    assert np.array_equal(reference.pin(r.sub_np()), q.sub_np())
    q.free()
    # ma_hit_cut
    q = fresh()
    r.cut(), q.cut()
    assert same_hits(r, q)
    q.free()
    # ma_hit_flt
    q = fresh()
    r.flt(), q.flt()
    assert same_hits(r, q)
    assert reference.pin(r.cov.value) == q.cov.value or (np.isnan(r.cov.value) and np.isnan(q.cov.value))
    q.free()
    # ma_hit_sub (round 2, end clip) + ma_hit_cut + ma_sub_merge
    q = fresh()
    r.sub2_cut_merge(), q.sub2_cut_merge()
    assert np.array_equal(reference.pin(r.sub_np()), q.sub_np())
    assert same_hits(r, q)
    q.free()
    # ma_hit_contained (+ dictionary squeeze)
    q = fresh()
    r.contained(), q.contained()
    assert reference.pin(r.names()) == q.names()
    assert np.array_equal(reference.pin(r.sub_np()), q.sub_np())
    assert same_hits(r, q)
    q.free()
    # ma_sg_gen
    q = fresh()
    r.sg_gen(), q.sg_gen()
    ar, sr, ir, _, _ = r.graph_np()
    aq, sq, iq, srt, _ = q.graph_np()
    assert srt and np.array_equal(sr, sq) and np.array_equal(ir, iq)
    assert np.array_equal(ar["ul"], aq["ul"]) and np.array_equal(canon_arcs(ar), canon_arcs(aq))
    q.free(), p.free(), r.free()


def test_sub_edge_cases(ref, prod):
    """Hand-made groups: depth exactly min_dp, ties between equally long stretches (first wins), end
    touching a start at the same coordinate, self hits and low-identity hits skipped, reads that never
    head a group (hit.c:109-160)."""
    rows = []
    def hit(q, qs, qe, t, ml=1000, bl=1000):
        rows.append((q << 32 | qs, qe, t, 0, qe - qs, ml, bl))
    for k in range(3):
        hit(0, 100, 5000, 1 + k)           # depth 3 on [100,5000)
    for k in range(3):
        hit(0, 6000, 10900, 4 + k)         # equally long stretch later: must lose to the first
    for k in range(2):
        hit(1, 0, 9000, 2 + k)             # depth 2 < min_dp: deleted
    for k in range(3):
        hit(2, 0, 3000, 5 + k)
    for k in range(3):
        hit(2, 3000, 8000, 8 + k)          # starts sort before ends at 3000: one stretch [0,8000)
    hit(3, 0, 9000, 3)                      # self hit ignored
    for k in range(3):
        hit(3, 10, 9000, 9 + k, ml=10, bl=1000)   # below min_iden: ignored -> deleted
    for k in range(4):
        hit(5, 500 + k, 7000 - k, 10 + k)   # nested: depth>=3 on [502,6998)
    a = np.array(rows, dtype=HIT_DT)
    a = a[np.argsort(a["qns"], kind="stable")]
    for clip in (0, 1000):
        pa = capi.c_malloc_copy(a)
        sr = ref.ma_hit_sub(3, 0.05, clip, len(a), pa, 16)
        sp = prod.ma_hit_sub(3, 0.05, clip, len(a), pa, 16)
        assert np.array_equal(reference.pin(capi.np_from_ptr(sr, 16, SUB_DT)), capi.np_from_ptr(sp, 16, SUB_DT))
        capi.c_free(sr), capi.c_free(sp), capi.c_free(pa)


def test_empty_inputs(prod):
    z = capi.c_malloc_copy(np.zeros(0, dtype=HIT_DT))
    s = prod.ma_hit_sub(3, 0.05, 0, 0, z, 4)
    assert not capi.np_from_ptr(s, 4, SUB_DT)["e"].any()
    assert prod.ma_hit_cut(s, 2000, 0, z) == 0
    capi.c_free(s), capi.c_free(z)


@pytest.mark.parametrize("span", [(30000, 20000), (9000, 11000), (200, 32000), (3, 40)], ids=["beyond32k", "reads10k", "edge32k", "tiny_coords"])
def test_sub_group_sizes(span, ref, prod):
    """Groups beyond the warp kernel (256 hits), beyond the CTA kernel (16384 hits) and tiny ones, in one array:
    the shared-memory paths and the device-wide-sort fallback of ma_hit_sub must agree with the reference.  `span` = (range of
    the interval starts, longest interval): below 32 768 the CTA kernel counts starts/ends per coordinate instead of sorting
    (many intervals share a coordinate in the small spans: the order of starts and ends at one coordinate matters)."""
    rng = np.random.default_rng(9)
    rows = []
    sizes = {0: 3, 1: 40, 2: 256, 3: 257, 4: 700, 5: 5000, 6: 16384, 7: 16385, 8: 20000, 9: 1, 10: 9000, 11: 12288}
    for q, n in sizes.items():
        qs = rng.integers(0, span[0], size=n)
        ln = rng.integers(min(500, span[1] // 2), span[1], size=n)
        for k in range(n):
            lowid = rng.random() < 0.05
            rows.append(((q << 32) | int(qs[k]), int(qs[k] + ln[k]), int(100 + rng.integers(0, 50)) if rng.random() > 0.02 else q,
                         0, int(ln[k]), 10 if lowid else 1000, 1000))
    a = np.array(rows, dtype=HIT_DT)
    a = a[np.argsort(a["qns"], kind="stable")]
    for dp, clip in ((3, 0), (3, 1000), (1, 0), (50, 300)):
        pa = capi.c_malloc_copy(a)
        sr = ref.ma_hit_sub(dp, 0.05, clip, len(a), pa, 200)
        sp = prod.ma_hit_sub(dp, 0.05, clip, len(a), pa, 200)
        assert np.array_equal(reference.pin(capi.np_from_ptr(sr, 200, SUB_DT)), capi.np_from_ptr(sp, 200, SUB_DT)), (dp, clip)
        capi.c_free(sr), capi.c_free(sp), capi.c_free(pa)


@pytest.mark.parametrize("name", ["tiny_exact", "chaos", "shuffled", "skew_small"])
def test_streamed_ingest_equals_two_calls(name, pafs, prod):
    """mab_load_ingest_text (chunks parsed while the next ones cross PCIe) must leave exactly the hits and the dictionary that
    mab_load_paf_text + mab_ingest leave; the weird-line file of test_cli_gpu exercises the short-line capacity fallback."""
    data = open(pafs[name], "rb").read()
    opt = prod.default_opt()
    res = []
    for stream in (False, True):
        ctx = prod.mab_create(0)
        if stream:
            assert prod.mab_load_ingest_text(ctx, data, len(data), opt.min_span, opt.min_match, 1) == 0
        else:
            assert prod.mab_load_paf_text(ctx, data, len(data)) == 0
            prod.mab_ingest(ctx, opt.min_span, opt.min_match, 1)
        n = C.c_size_t(0)
        hp = prod.mab_export_hits(ctx, C.byref(n))
        hits = capi.np_from_ptr(hp, n.value, HIT_DT)
        capi.c_free(hp)
        d = prod.mab_export_dict(ctx)
        names = [(d.contents.seq[i].name, d.contents.seq[i].len) for i in range(d.contents.n_seq)]
        prod.sd_destroy(d)
        prod.mab_destroy(ctx)
        res.append((canon_mask(hits), names))
    assert np.array_equal(res[0][0], res[1][0]) and res[0][1] == res[1][1]
    tiny = b"a\t1\t2\n\n\n\nq\t5000\t0\t4000\t+\tt\t5000\t1000\t5000\t800\t4000\t255\n" + b"\n" * 5000   # far more lines than len/24
    ctx = prod.mab_create(0)
    assert prod.mab_load_ingest_text(ctx, tiny, len(tiny), opt.min_span, opt.min_match, 1) == 0
    assert prod.mab_stats(ctx).contents.n_hits_stored == 2
    prod.mab_destroy(ctx)
