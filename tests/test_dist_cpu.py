"""CPU tier, world_size 2 (and 3) over gloo: the launcher-side logic of the sharded run (byte-range split at line ends,
ownership, hand-over of the communicator id), the rank aggregation bench.py uses, and a model of the sharding scheme itself
(global ids from per-rank dictionaries, hits to the owner of the query read, interval tables completed by all-reduce) with the
unmodified reference as every rank's compute, checked against a single-rank run."""
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from miniasm_b200 import sharded, synth


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, paf, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    data = open(paf, "rb").read()
    b, e = sharded.split_ranges(data, world)[rank]
    part = data[b:e]
    # every rank's piece ends at a line end; line counts add up
    n_lines = torch.tensor([part.count(b"\n")], dtype=torch.int64)
    dist.all_reduce(n_lines)
    ok = (e == len(data) or data[e - 1:e] == b"\n") and n_lines.item() == data.count(b"\n")
    # the id rank 0 makes reaches everybody unchanged
    box = [os.urandom(128) if rank == 0 else None]
    dist.broadcast_object_list(box, src=0)
    ids = [None] * world
    dist.all_gather_object(ids, box[0])
    ok = ok and all(i == ids[0] for i in ids) and len(ids[0]) == 128
    # bench aggregation: throughput = sum of work / max time
    t = torch.tensor([1.0 + rank, 100.0], dtype=torch.float64)
    mx, sm = t.clone(), t.clone()
    dist.all_reduce(mx, op=dist.ReduceOp.MAX)
    dist.all_reduce(sm, op=dist.ReduceOp.SUM)
    ok = ok and mx[0].item() == float(world) and sm[1].item() == 100.0 * world
    q.put((rank, ok, b, e))
    dist.barrier()
    dist.destroy_process_group()


def test_two_rank_launcher_logic(built, paf_dir):
    paf = synth.generate("-n 1500 -s 77 -j 100", f"{paf_dir}/dist.paf")
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    ps = [ctx.Process(target=_worker, args=(r, 2, port, paf, q)) for r in range(2)]
    for p in ps:
        p.start()
    res = sorted(q.get(timeout=120) for _ in ps)
    for p in ps:
        p.join(60)
    assert all(ok for _, ok, _, _ in res)
    assert res[0][2] == 0 and res[0][3] == res[1][2] and res[1][3] == os.path.getsize(paf)


@pytest.mark.parametrize("world", [1, 2, 3, 8])
def test_split_ranges_edge_cases(world):
    for data in (b"", b"a\n", b"a\nb", b"\n\n\n", b"x" * 50, b"l1\nl2\nl3\nl4\nl5\nl6\nl7\nl8\nl9\n"):
        rs = sharded.split_ranges(data, world)
        assert len(rs) == world and rs[0][0] == 0 and rs[-1][1] == len(data)
        assert all(rs[i][1] == rs[i + 1][0] for i in range(world - 1))
        assert all(e == len(data) or e == b or data[e - 1:e] == b"\n" for b, e in rs)
        assert b"".join(data[b:e] for b, e in rs) == data
    assert [sharded.owner(i, 4) for i in range(6)] == [0, 1, 2, 3, 0, 1]


# ---- the sharding scheme itself, modelled with the reference as every rank's compute -------------------------------------------------
def _model_body(rank, world, port, paf, q):
    """DESIGN.md section 8 steps 1-2 as a model: every rank parses its byte range with the UNMODIFIED reference (local ids), the ranks
    agree on global ids (first appearance in rank order = file order), hits travel to the owner of their query read (id mod world)
    keeping per-source order, the owner runs the reference's ma_hit_sub on what it received, the interval table is completed by an
    all-reduce(sum), ma_hit_cut + ma_hit_flt run owner-local against the full table.  Every rank checks its share against a
    single-rank run of the reference on the whole file."""
    import ctypes as C
    import tempfile

    import numpy as np

    from miniasm_b200 import capi
    from miniasm_b200.capi import HIT_DT, SUB_DT
    from miniasm_b200.pipeline import Pipeline
    from tests import reference
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    ref = reference.load()
    ref.set_verbose(0)
    data = open(paf, "rb").read()
    b, e = sharded.split_ranges(data, world)[rank]
    with tempfile.NamedTemporaryFile(suffix=".paf", delete=False) as tf:
        tf.write(data[b:e])
    mine = Pipeline(ref, tf.name).read()                     # local dictionary: ids = first appearance among MY stored lines
    os.unlink(tf.name)
    truth = Pipeline(ref, paf).read()                        # what one rank would have
    o = truth.opt

    # 1. global ids: walk the ranks in file order, a name keeps the id of its first appearance
    names = [None] * world
    dist.all_gather_object(names, mine.names())
    gid = {}
    for r in range(world):
        for nm in names[r]:
            gid.setdefault(nm, len(gid))
    ok = [nm for nm, _ in sorted(gid.items(), key=lambda kv: kv[1])] == truth.names()
    n_seq = len(gid)
    l2g = np.array([gid[nm] for nm in mine.names()], dtype=np.uint64)

    # 2. hits to the owner of the query read, per-source order kept; owner: concatenate in rank order, stable sort by (id, start)
    h = mine.hits_np()
    if len(h):
        h["qns"] = (l2g[(h["qns"] >> np.uint64(32)).astype(np.int64)] << np.uint64(32)) | (h["qns"] & np.uint64(0xffffffff))
        h["tn"] = l2g[h["tn"].astype(np.int64)].astype(np.uint32)
    dest = ((h["qns"] >> np.uint64(32)) % np.uint64(world)).astype(np.int64)
    box = [None] * world
    dist.all_gather_object(box, [h[dest == r].tobytes() for r in range(world)])
    got = np.concatenate([np.frombuffer(box[src][rank], dtype=HIT_DT) for src in range(world)])
    got = got[np.argsort(got["qns"], kind="stable")].copy()
    th = truth.hits_np()
    owned = ((th["qns"] >> np.uint64(32)) % np.uint64(world)).astype(np.int64) == rank
    key = ["qns", "qe", "tn", "ts", "te", "ml_rev"]        # (bl_del carries the del bit the reference never initialises)

    def same_hits(a, b):
        a, b = a.copy(), b.copy()
        a["bl_del"] &= 0x7fffffff
        b["bl_del"] &= 0x7fffffff
        return len(a) == len(b) and np.array_equal(np.sort(a, order=key + ["bl_del"]), np.sort(b, order=key + ["bl_del"]))
    ok = ok and same_hits(got, th[owned]) and np.array_equal(got["qns"], th[owned]["qns"])

    # 3. ma_hit_sub on the owner, all-reduce(sum) completes the table; cut + flt owner-local against the full table
    def sub_of(hits, clip):
        p = ref.ma_hit_sub(o.min_dp, o.min_iden, clip, len(hits), hits.ctypes.data_as(C.c_void_p), n_seq)
        t = capi.np_from_ptr(p, n_seq, SUB_DT)
        capi.c_free(p)
        rows = np.zeros(n_seq, dtype=bool)                     # rows of reads I do not own stay zero (calloc)
        rows[np.arange(n_seq) % world == rank] = True
        assert not t["s_del"][~rows].any() and not t["e"][~rows].any()
        w = torch.from_numpy(t.view(np.uint32).astype(np.int64))
        dist.all_reduce(w)
        return w.numpy().astype(np.uint32).view(SUB_DT).reshape(-1)
    sub = sub_of(got, 0)
    truth.sub1()
    ok = ok and np.array_equal(sub, truth.sub_np())
    n = ref.ma_hit_cut(sub.ctypes.data_as(C.c_void_p), o.min_span, len(got), got.ctypes.data_as(C.c_void_p))
    cov = C.c_float(0)
    n = ref.ma_hit_flt(sub.ctypes.data_as(C.c_void_p), int(o.max_hang * 1.5), int(o.min_ovlp * .5), n, got.ctypes.data_as(C.c_void_p), C.byref(cov))
    truth.cut().flt()
    th = truth.hits_np()
    owned = ((th["qns"] >> np.uint64(32)) % np.uint64(world)).astype(np.int64) == rank
    ok = ok and same_hits(got[:n], th[owned])
    tot = torch.tensor([n], dtype=torch.int64)
    dist.all_reduce(tot)
    ok = ok and tot.item() == truth.n_hits and n > 0
    # second round: same exchange with the clip of main.c:131
    sub2 = sub_of(got[:n].copy(), o.min_span // 2)
    p2 = ref.ma_hit_sub(o.min_dp, o.min_iden, o.min_span // 2, truth.n_hits, truth.hits, n_seq)
    ok = ok and np.array_equal(sub2, capi.np_from_ptr(p2, n_seq, SUB_DT))
    capi.c_free(p2)

    # 4. round-2 cut owner-local, merged table replicated (main.c:131-134)
    vp = lambda a: a.ctypes.data_as(C.c_void_p)
    n = ref.ma_hit_cut(vp(sub2), o.min_span, n, vp(got))
    merged = sub.copy()
    ref.ma_sub_merge(n_seq, vp(merged), vp(sub2))
    truth.cut(truth_sub2 := vp(sub2))
    ref.ma_sub_merge(n_seq, truth.sub, truth_sub2)
    th = truth.hits_np()
    owned = ((th["qns"] >> np.uint64(32)) % np.uint64(world)).astype(np.int64) == rank
    ok = ok and np.array_equal(merged, truth.sub_np()) and same_hits(got[:n], th[owned])

    # 5. ma_hit_contained (hit.c:225-256): containment flags of the owner's hits OR-ed over the ranks (all-reduce max), "used" marks
    #    likewise, renumbering replicated.  The local flags come from the reference itself: it runs on the owner's hits plus one
    #    inert self hit per read (classified "internal", so every read counts as used and only flagged reads leave the dictionary).
    gl_names = [nm for nm, _ in sorted(gid.items(), key=lambda kv: kv[1])]
    lens_box = [None] * world
    dist.all_gather_object(lens_box, dict(zip(mine.names(), mine.seq_lens().tolist())))
    gl_len = [next(lens_box[r][nm] for r in range(world) if nm in lens_box[r]) for nm in gl_names]   # sdict.c:36: first appearance
    ln = (merged["e"] - (merged["s_del"] & np.uint32(0x7fffffff))).astype(np.int64)
    inert = np.zeros(n_seq, dtype=HIT_DT)
    x = np.where(ln >= 2, 1, 0).astype(np.uint64)
    inert["qns"] = (np.arange(n_seq, dtype=np.uint64) << np.uint64(32)) | x
    inert["qe"] = inert["te"] = np.where(ln >= 2, 2, 0)
    inert["ts"], inert["tn"], inert["bl_del"] = x.astype(np.uint32), np.arange(n_seq, dtype=np.uint32), 1
    aug = np.concatenate([got[:n], inert])
    dloc = ref.sd_init()
    for nm, l in zip(gl_names, gl_len):
        ref.sd_put(dloc, nm, l)
    sub_copy = merged.copy()
    ref.ma_hit_contained(C.byref(o), dloc, vp(sub_copy), len(aug), vp(aug))
    left = {dloc.contents.seq[i].name for i in range(dloc.contents.n_seq)}
    ref.sd_destroy(dloc)
    flag = torch.tensor([nm not in left for nm in gl_names], dtype=torch.int32)
    used = torch.zeros(n_seq, dtype=torch.int32)
    used[torch.from_numpy((got[:n]["qns"] >> np.uint64(32)).astype(np.int64))] = 1
    used[torch.from_numpy(got[:n]["tn"].astype(np.int64))] = 1
    dist.all_reduce(flag, op=dist.ReduceOp.MAX)
    dist.all_reduce(used, op=dist.ReduceOp.MAX)
    flag, used = flag.numpy().astype(bool), used.numpy().astype(bool)
    ok = ok and not (used & (ln < 2)).any()                    # the inert hit of an empty interval may flag it: such reads are unused anyway
    dead = flag | ~used
    new_id = np.cumsum(~dead) - 1
    old_of_new = np.flatnonzero(~dead)
    loc = got[:n]
    lq, lt = (loc["qns"] >> np.uint64(32)).astype(np.int64), loc["tn"].astype(np.int64)
    loc = loc[~dead[lq] & ~dead[lt]].copy()
    loc["qns"] = (new_id[(loc["qns"] >> np.uint64(32)).astype(np.int64)].astype(np.uint64) << np.uint64(32)) | (loc["qns"] & np.uint64(0xffffffff))
    loc["tn"] = new_id[loc["tn"].astype(np.int64)].astype(np.uint32)
    sub_new = merged[~dead].copy()
    truth.contained()
    th = truth.hits_np()
    owned = old_of_new[(th["qns"] >> np.uint64(32)).astype(np.int64)] % world == rank     # ownership stays with the ORIGINAL id
    ok = ok and [gl_names[i] for i in old_of_new] == truth.names() and np.array_equal(sub_new, truth.sub_np()) and same_hits(loc, th[owned])

    # 6. ma_sg_gen (asm.c:9-39) on the owner; read flags OR-ed, arcs all-gathered and stably sorted by their key = the single-rank graph
    dnew = ref.sd_init()
    for i in old_of_new:
        ref.sd_put(dnew, gl_names[i], gl_len[i])
    g = ref.ma_sg_gen(C.byref(o), dnew, vp(sub_new), len(loc), vp(loc))
    arcs, seq, _, _, _ = ref.read_graph(g)
    ref.asg_destroy(g), ref.sd_destroy(dnew)
    sdel = torch.from_numpy((seq >> 31).astype(np.int32))
    dist.all_reduce(sdel, op=dist.ReduceOp.MAX)
    seq = (seq & np.uint32(0x7fffffff)) | (sdel.numpy().astype(np.uint32) << np.uint32(31))
    abox = [None] * world
    dist.all_gather_object(abox, arcs.tobytes())
    from miniasm_b200.capi import ARC_DT
    from miniasm_b200.pipeline import canon_arcs
    allarcs = np.concatenate([np.frombuffer(bts, dtype=ARC_DT) for bts in abox])
    gone = (seq >> 31).astype(bool)
    allarcs = allarcs[~gone[(allarcs["ul"] >> np.uint64(33)).astype(np.int64)] & ~gone[(allarcs["v"] >> 1).astype(np.int64)]]
    allarcs = allarcs[np.argsort(allarcs["ul"], kind="stable")]
    truth.sg_gen()
    tarcs, tseq, _, _, _ = truth.graph_np()
    ok = ok and np.array_equal(seq, tseq) and len(tarcs) > 0 and np.array_equal(allarcs["ul"], tarcs["ul"]) \
        and np.array_equal(canon_arcs(allarcs), canon_arcs(tarcs))
    q.put((rank, bool(ok), int(len(loc)), int(n_seq), int(flag.sum()), int(dead.sum()), int(len(tarcs))))
    dist.barrier()
    dist.destroy_process_group()


def _model_worker(rank, world, port, paf, q):
    try:
        _model_body(rank, world, port, paf, q)
    except BaseException as ex:  # noqa: BLE001 -- a rank that dies would leave the others waiting in a collective: report and let the parent stop them
        import traceback
        q.put((rank, False, traceback.format_exc()[-1500:] or repr(ex)))


@pytest.mark.parametrize("world", [2, 3])
def test_sharding_scheme_model(world, built, paf_dir):
    from tests import reference
    paf = synth.generate("-n 3000 -s 78 -j 300 -l 8000 -L 12000", f"{paf_dir}/dist_model.paf")
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    ps = [ctx.Process(target=_model_worker, args=(r, world, port, paf, q)) for r in range(world)]
    for p in ps:
        p.start()
    res = []
    try:
        for _ in ps:
            res.append(q.get(timeout=300))
            assert res[-1][1], res[-1]
    finally:
        if len(res) < world or not all(r[1] for r in res):
            for p in ps:
                p.terminate()
    for p in ps:
        p.join(60)
    res.sort()
    assert [r[0] for r in res] == list(range(world))
    assert all(r[1] for r in res), res
    # the model has teeth: hits on every rank, contained reads flagged, a non-trivial graph
    assert all(r[2] > 0 and r[4] > 100 and r[5] >= r[4] and r[6] > 100 for r in res), res
    reference.pin([r[2:] for r in res])                 # the counts the reference's compute gave every rank
    print(res)
