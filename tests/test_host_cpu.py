"""CPU tier: the host C side of the product (sdict.c, paf.c, gfa.c) -- no GPU involved."""
import ctypes as C
import gzip
import os

import pytest

from miniasm_b200 import capi, synth
from oracle import loaders
from miniasm_b200.pipeline import Pipeline
from tests import reference

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


class PafRec(C.Structure):                                   # paf_rec_t, paf.h:20-24
    _fields_ = [("qn", C.c_char_p), ("tn", C.c_char_p), ("ql", C.c_uint32), ("qs", C.c_uint32), ("qe", C.c_uint32),
                ("tl", C.c_uint32), ("ts", C.c_uint32), ("te", C.c_uint32), ("ml_rev", C.c_uint32), ("bl", C.c_uint32)]


def paf_records(lib, path):
    lib.dll.paf_open.restype = C.c_void_p
    lib.dll.paf_open.argtypes = [C.c_char_p]
    lib.dll.paf_read.argtypes = [C.c_void_p, C.POINTER(PafRec)]
    lib.dll.paf_close.argtypes = [C.c_void_p]
    fp = lib.dll.paf_open(path.encode())
    assert fp
    r, out = PafRec(), []
    while lib.dll.paf_read(fp, C.byref(r)) >= 0:
        out.append((r.qn, r.ql, r.qs, r.qe, r.ml_rev >> 31, r.tn, r.tl, r.ts, r.te, r.ml_rev & 0x7fffffff, r.bl))
    lib.dll.paf_close(fp)
    return out


WEIRD = (b"q1\t1000\t10\t900\t+\tt1\t2000\t5\t800\t700\t890\t255\n"
         b"q2\t1000\t+10\t 900\t-\tt1\t2000\t5\t800\t700abc\t890\t255\ttp:A:S\r\n"
         b"\n"
         b"short\tline\n"
         b"q3\t1000\t0\t1000\t-\tt2\t3000\t0\t1000\t999\n"                 # 10 fields: bl stays 890
         b"q4\t99999999999999999999\t-5\t77\t*\tt3\t1\t2\t3\t4\t5\t6\t7\t8\n"
         b"q5\t1\t2\t3\t-\tt5\t6\t7\t8\t9\t10")                            # no trailing newline


def test_paf_reader_corner_cases(built, tmp_path):
    prod = capi.load_product()
    p = tmp_path / "weird.paf"
    p.write_bytes(WEIRD)
    got = paf_records(prod, str(p))
    assert got == [
        (b"q1", 1000, 10, 900, 0, b"t1", 2000, 5, 800, 700, 890),
        (b"q2", 1000, 10, 900, 1, b"t1", 2000, 5, 800, 700, 890),
        (b"q3", 1000, 0, 1000, 1, b"t2", 3000, 0, 1000, 999, 890),
        (b"q4", 0xffffffff, 0xfffffffb, 77, 0, b"t3", 1, 2, 3, 4, 5),
        (b"q5", 1, 2, 3, 1, b"t5", 6, 7, 8, 9, 10),
    ]
    if os.path.exists(loaders.REFERENCE_SO):
        assert paf_records(loaders.load_reference(), str(p)) == got
    gz = tmp_path / "weird.paf.gz"
    with gzip.open(gz, "wb") as f:
        f.write(WEIRD)
    assert paf_records(prod, str(gz)) == got


def test_sdict(built):
    prod = capi.load_product()
    d = prod.sd_init()
    names = [f"read/{i}".encode() for i in range(5000)]
    for i, n in enumerate(names):
        assert prod.sd_put(d, n, 100 + i) == i
    assert prod.sd_put(d, names[17], 1) == 17 and d.contents.seq[17].len == 117      # first length wins
    assert prod.sd_get(d, b"nope") == -1 and prod.sd_get(d, names[4999]) == 4999
    for i in range(0, 5000, 3):
        d.contents.seq[i].aux_del |= 0x80000000
    m = capi.np_from_ptr(prod.sd_squeeze(d), 5000, "<i4")
    assert d.contents.n_seq == 5000 - len(range(0, 5000, 3))
    assert m[0] == -1 and m[1] == 0 and m[2] == 1 and m[4] == 2
    assert prod.sd_get(d, names[3]) == -1 and prod.sd_get(d, names[4]) == 2
    prod.sd_destroy(d)


def test_writers_and_ug_seq_against_reference(built, ref, paf_dir):
    from tests.test_clean_gpu import _write_reads
    prod = capi.load_product()
    paf = synth.generate("chaos_small", f"{paf_dir}/hc.paf")
    for fmt in ("fa", "fq.gz"):
        reads = _write_reads(paf, os.path.join(paf_dir, f"hc_reads.{fmt}"), gz=fmt.endswith("gz"), fastq=fmt.startswith("fq"))
        a = Pipeline(ref, paf).read().select().sg_gen().clean().ug_gen()
        want = a.gfa(reads)
        b = Pipeline(ref, paf).read().select().sg_gen().clean().ug_gen()
        d2 = prod.sd_init()                                                           # sdict_t::h is private to each library: rebuild the dictionary on our side
        for i, nm in enumerate(b.names()):
            assert prod.sd_put(d2, nm, b.d.contents.seq[i].len) == i
        prod.ma_ug_seq(b.ug, d2, b.sub, reads.encode())                               # our ma_ug_seq fills the reference's unitig structs
        assert prod.print_to_string("ma_ug_print", b.ug, d2, b.sub) == want
        prod.sd_destroy(d2)
        assert prod.print_to_string("ma_sg_print", b.sg, b.d, b.sub) == a.sg_text()
        assert prod.print_to_string("ma_sg_print", b.sg, b.d, None) == ref.print_to_string("ma_sg_print", a.sg, a.d, None)
        a.free(), b.free()


def test_ug_seq_refuses_a_short_record(built, paf_dir):
    """asm.c:263 asserts that a record covers the interval the layout keeps; ours must not read past a shorter record either
    (a reads file that does not belong to the PAF): message + abort, in a child process."""
    import subprocess
    import sys
    code = f"""
import sys, os
sys.path.insert(0, {ROOT!r})
from miniasm_b200 import capi, synth
from miniasm_b200.pipeline import Pipeline
from tests import reference
ref = reference.load(); ref.set_verbose(0)
prod = capi.load_product(); prod.set_verbose(0)
paf = synth.generate("tiny_exact", {paf_dir!r} + "/short.paf")
b = Pipeline(ref, paf).read().select().sg_gen().clean().ug_gen()
names = b.names()
with open({paf_dir!r} + "/short.fa", "w") as f:
    for nm in names:
        f.write(">" + nm.decode() + "\\nACGTACGTAC\\n")          # 10 bases where the layout needs thousands
d2 = prod.sd_init()
for i, nm in enumerate(names):
    prod.sd_put(d2, nm, b.d.contents.seq[i].len)
prod.ma_ug_seq(b.ug, d2, b.sub, ({paf_dir!r} + "/short.fa").encode())
print("survived")
"""
    r = subprocess.run([sys.executable, "-c", code], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
    assert r.returncode != 0 and "survived" not in r.stdout
    assert "[E::ma_ug_seq]" in r.stderr and "wrong reads file" in r.stderr


def test_no_cont_prefilter_against_reference(built, ref, paf_dir):
    prod = capi.load_product()
    paf = synth.generate("-n 4000 -l 2000 -L 30000 -c 30 -j 100 -s 41", f"{paf_dir}/nocont.paf")
    a = ref.ma_hit_no_cont(paf.encode(), 2000, 100, 1000, 0.8)
    b = prod.ma_hit_no_cont(paf.encode(), 2000, 100, 1000, 0.8)
    na = [a.contents.seq[i].name for i in range(a.contents.n_seq)]
    nb = [b.contents.seq[i].name for i in range(b.contents.n_seq)]
    assert reference.pin(na) == nb and len(na) > 10


def test_device_parser_matches_host_reader(built, paf_dir):
    """The GPU line parser (ingest_dev.cu parse_line, compiled for the host through mab_test_parse_line) against the host
    reader on ~140 K lines with CRLF, 9/10-field lines, tags, signs, junk, blanks, empty lines."""
    from tests.test_cli_gpu import test_weird_lines  # noqa: F401  (same recipe, rebuilt here without the GPU)
    prod = capi.load_product()
    f = prod.dll.mab_test_parse_line
    f.argtypes = [C.c_char_p, C.c_size_t, C.POINTER(C.c_uint32)]
    base = synth.generate("-n 3000 -s 31 -j 200 -C 200000", os.path.join(paf_dir, "pw_base.paf"))
    out = []
    for i, ln in enumerate(open(base, "rb").read().split(b"\n")):
        if not ln:
            continue
        fl = ln.rstrip(b"\r").split(b"\t")
        if i % 11 == 0 and i > 0:
            out.append(b"\t".join(fl[:10]))
        elif i % 13 == 0:
            out.append(b"\t".join(fl[:9]))
        elif i % 17 == 0:
            out.append(ln + b"\ttp:A:S\tcm:i:12")
        elif i % 19 == 0:
            out += [b"", ln]
        elif i % 23 == 0:
            fl[2] = b"+" + fl[2]; fl[9] = fl[9] + b"xyz"; fl[7] = b"-" + fl[7]; out.append(b"\t".join(fl))
        elif i % 29 == 0:
            fl[1] = b" " + fl[1]; fl[6] = b"000000000000000000000" + fl[6]; out.append(b"\t".join(fl) + b"\r")
        elif i % 31 == 0:
            fl[3] = b"99999999999999999999999"; fl[8] = b"-99999999999999999999999"; out.append(b"\t".join(fl))
        else:
            out.append(ln)
    path = os.path.join(paf_dir, "pw.paf")
    with open(path, "wb") as fo:
        fo.write(b"\n".join(out))
    want = paf_records(prod, path)
    got, stale = [], 0
    for ln in out:
        o = (C.c_uint32 * 13)()
        f(ln, len(ln), o)
        o = list(o)
        if o[0] >= 11:
            stale = o[9]
        if o[0] >= 10:
            l2 = ln[:-1] if len(ln) > 1 and ln.endswith(b"\r") else ln
            got.append((l2[:o[10]], o[1], o[2], o[3], o[4], l2[o[12]:o[12] + o[11]], o[5], o[6], o[7], o[8], o[9] if o[0] >= 11 else stale))
    assert len(got) == len(want) > 100000 and got == want


def _synthetic_layout(lib, n_utg, seed):
    """A ma_ug_t built by hand (miniasm.h:42-55): unitigs of 1..3000 reads, some circular, plus a few links."""
    import numpy as np
    rng = np.random.default_rng(seed)
    n_reads = 40000
    d = lib.sd_init()
    for i in range(n_reads):
        lib.sd_put(d, b"r%d_%s" % (i * 7919 % 100003, b"x" * (i % 23)), 5000 + i % 9000)
    sub = np.zeros(n_reads, dtype=capi.SUB_DT)
    sub["s_del"] = rng.integers(0, 500, n_reads)
    sub["e"] = 5000 + rng.integers(0, 3000, n_reads)
    keep = []                                                              # numpy buffers the C structs point into
    utg = (capi.MaUtg * n_utg)()
    for i in range(n_utg):
        n = int(rng.choice([1, 2, 3, 50, 700, 3000, 4095, 4096, 4097]))
        a = (rng.integers(0, n_reads, n).astype(np.uint64) << np.uint64(33)) | (rng.integers(0, 2, n).astype(np.uint64) << np.uint64(32)) \
            | rng.integers(1, 20000, n).astype(np.uint64)
        keep.append(a)
        circ = i % 5 == 3
        utg[i].len_circ = int(a.astype(np.uint32).sum() & 0x7fffffff) | (int(circ) << 31)
        utg[i].start = 0xffffffff if circ else int(a[0] >> np.uint64(32))
        utg[i].end = 0xffffffff if circ else int(a[-1] >> np.uint64(32)) ^ 1
        utg[i].n = utg[i].m = n
        utg[i].a = a.ctypes.data_as(C.POINTER(C.c_uint64))
        utg[i].s = None
    arcs = np.zeros(7, dtype=capi.ARC_DT)
    arcs["ul"] = (rng.integers(0, 2 * n_utg, 7).astype(np.uint64) << np.uint64(32)) | rng.integers(1, 9999, 7).astype(np.uint64)
    arcs["v"] = rng.integers(0, 2 * n_utg, 7)
    arcs["ol_del"] = rng.integers(1, 5000, 7)
    idx = rng.integers(0, 3, 2 * n_utg).astype(np.uint64)
    g = capi.AsgT()
    g.m_arc, g.n_arc_srt, g.arc = 7, 7, arcs.ctypes.data
    g.m_seq, g.n_seq_symm, g.seq, g.idx = n_utg, n_utg, None, idx.ctypes.data
    ug = capi.MaUg()
    ug.n = ug.m = n_utg
    ug.a = C.cast(utg, C.POINTER(capi.MaUtg))
    ug.g = C.pointer(g)
    keep += [utg, arcs, idx, g]
    return ug, d, sub, keep


def test_ug_writer_threads_keep_the_byte_stream(built, monkeypatch):
    """ma_ug_print formats large layouts with worker threads (gfa.c); the bytes must not depend on the thread count."""
    prod = capi.load_product(strict=False)
    ug, d, sub, keep = _synthetic_layout(prod, 60, 5)
    subp = C.c_void_p(sub.ctypes.data)
    outs = {}
    for t in ("0", "1", "3", "7", "16"):
        monkeypatch.setenv("MAB_WRITER_THREADS", t)
        outs[t] = prod.print_to_string("ma_ug_print", C.pointer(ug), d, subp)
    assert len(outs["0"]) > 1_000_000 and outs["0"].count(b"\na\t") > 50_000
    for t in outs:
        assert outs[t] == outs["0"], t
    plain = {}
    for t in ("0", "5"):                                                  # sub == NULL: names without the :s-e suffix
        monkeypatch.setenv("MAB_WRITER_THREADS", t)
        plain[t] = prod.print_to_string("ma_ug_print", C.pointer(ug), d, None)
    assert plain["0"] == plain["5"] and len(plain["0"]) < len(outs["0"])
    if os.path.exists(loaders.REFERENCE_SO):                                # and they are the reference's bytes (asm.c:64-116)
        ref = loaders.load_reference()
        d2 = ref.sd_init()
        for i in range(d.contents.n_seq):
            ref.sd_put(d2, d.contents.seq[i].name, d.contents.seq[i].len)
        assert ref.print_to_string("ma_ug_print", C.pointer(ug), d2, subp) == outs["0"]


def test_device_gfa_formatter_matches_host_writer(built):
    """gfa_dev.cu's record emitter (what mab_write_gfa runs one thread per line of) compiled for the CPU through
    mab_test_gfa_host, against ma_ug_print on the same hand-built layout: S/L/a/x lines, circular unitigs, links."""
    prod = capi.load_product(strict=False)
    f = prod.dll.mab_test_gfa_host
    f.restype = C.c_size_t
    f.argtypes = [C.POINTER(capi.MaUg), C.POINTER(capi.Sdict), C.c_void_p, C.c_void_p, C.c_size_t]
    for seed, with_sub in ((5, True), (6, False), (7, True)):
        ug, d, sub, keep = _synthetic_layout(prod, 40, seed)
        subp = C.c_void_p(sub.ctypes.data) if with_sub else None
        want = prod.print_to_string("ma_ug_print", C.pointer(ug), d, subp)
        n = f(C.pointer(ug), d, subp, None, 0)
        assert n == len(want)
        buf = C.create_string_buffer(n)
        assert f(C.pointer(ug), d, subp, buf, n) == n
        assert buf.raw == want
