"""The drop-in command line: `miniasm-b200 [options] in.paf` against the unmodified reference binary on the
same input, option by option (main.c:44-74 flag surface, -S stage dumps of SURVEY.md section 4)."""
import gzip
import os
import shutil
import subprocess

import pytest

from miniasm_b200 import synth
from tests import reference

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLI = os.path.join(ROOT, "miniasm_b200", "miniasm-b200")


def run(binary, args, stdin=None):
    r = subprocess.run([binary] + args, stdout=subprocess.PIPE, stderr=subprocess.PIPE, stdin=stdin)
    return r.returncode, r.stdout, r.stderr


@pytest.fixture(scope="module")
def pafs(built, paf_dir):
    return {name: synth.generate(name, f"{paf_dir}/{name}.paf") for name in ["chaos_small", "chaos", "bubbles800", "tiny_exact", "shuffled"]}


def same(args, exact=True):
    rc_c, out_c, err_c = run(CLI, args)
    if exact:
        reference.match((rc_c, out_c, err_c), args, lambda r: (r[0], r[1]))
    else:  # outputs whose line order depends on ties of the reference's unstable radix sort
        reference.match((rc_c, out_c, err_c), args, lambda r: (r[0], sorted(r[1].splitlines())))
    return out_c


@pytest.mark.parametrize("name", ["chaos_small", "chaos", "bubbles800", "tiny_exact", "shuffled"])
def test_default_gfa(name, pafs):
    out = same([pafs[name]])
    assert out.startswith(b"S\tutg000001")


@pytest.mark.parametrize("opts", [
    ["-c", "2"], ["-c", "5"], ["-e", "2"], ["-e", "10"], ["-n", "1"], ["-n", "5"], ["-r", "0.8,0.4"], ["-F", "0.9"],
    ["-h", "500"], ["-h", "3000"], ["-I", "0.6"], ["-o", "3000"], ["-m", "2500"], ["-i", "0.3"], ["-s", "1500"], ["-s", "4000"],
    ["-g", "10"], ["-g", "100000"], ["-d", "2000"], ["-d", "500000"], ["-1"], ["-2"], ["-1", "-2"], ["-b"], ["-B"], ["-R"], ["-R", "-b"],
])
def test_options(opts, pafs):
    same(opts + [pafs["chaos_small"]])


@pytest.mark.parametrize("stage", [2, 3, 4, 5])
def test_stage_dumps_paf(stage, pafs):
    same(["-S", str(stage), "-p", "paf", pafs["chaos_small"]], exact=False)


@pytest.mark.parametrize("stage", [2, 3, 4, 5, 100])
def test_bed(stage, pafs):
    same(["-S", str(stage), "-p", "bed", pafs["chaos_small"]])


@pytest.mark.parametrize("stage", [1, 5, 6, 7, 9, 10, 11])
def test_stage_dumps_sg_ug(stage, pafs):
    same(["-S", str(stage), "-p", "sg", pafs["chaos"]], exact=False)
    # before transitive reduction the raw graph has equal-key arcs; their order (unstable sort in the reference)
    # decides the order of tied unitig links, so the early dumps are compared as multisets
    same(["-S", str(stage), "-p", "ug", pafs["chaos"]], exact=stage >= 6)


def test_gzip_and_stdin(pafs, paf_dir):
    gz = os.path.join(paf_dir, "in.paf.gz")
    with open(pafs["chaos_small"], "rb") as f, gzip.open(gz, "wb") as g:
        shutil.copyfileobj(f, g)
    plain = same([pafs["chaos_small"]])
    assert same([gz]) == plain
    with open(pafs["chaos_small"], "rb") as f:
        rc, out, _ = run(CLI, ["-"], stdin=f)
    assert rc == 0 and out == plain


def _counters(err):
    """The reference's [M::...] progress lines with the timestamps masked (sys_timestamp: "::<real>*<cpu ratio>")."""
    import re
    out = []
    for ln in err.decode().splitlines():
        if not ln.startswith("[M::") or ln.startswith(("[M::main] Version", "[M::main] CMD", "[M::main] Real time")):
            continue
        out.append(re.sub(r"::\d+\.\d+\*\d+\.\d+\]", "]", ln))
    return out


@pytest.mark.parametrize("name", ["chaos_small", "chaos", "bubbles800", "tiny_exact"])
@pytest.mark.parametrize("opts", [[], ["-c", "2", "-e", "2"], ["-R"]], ids=["default", "c2e2", "R"])
def test_stderr_counters(name, opts, pafs):
    """SURVEY.md section 5: the [M::...] lines carry the counts of every step (hits stored, reads kept, arcs reduced, tips cut,
    bubbles popped ...) and are reproduced verbatim."""
    reference.match(run(CLI, opts + [pafs[name]]), opts + [pafs[name]], lambda r: _counters(r[2]))


def test_bubble_dense_300k(paf_dir):
    """300 K reads with jittered ends: 3 713 bubbles popped along genome-ordered ids (the set on which one-commit-per-round
    schemes crawl); output bytes and every stderr counter against the reference."""
    paf = synth.generate("-n 300000 -l 9000 -L 11000 -j 800 -c 30 -s 15", os.path.join(paf_dir, "bub300k.paf"))
    rc_c, out_c, err_c = run(CLI, [paf])
    assert rc_c == 0, err_c.decode()[-2000:]
    reference.match((rc_c, out_c, err_c), [paf], lambda r: (r[0], r[1]))
    # Equal-length arcs out of one vertex are common with 800 bp of jitter at 300 K reads; which of two tied neighbours is explored
    # first follows the order the reference's unstable in-place radix sort left them in (ksort.h:134-183; ours are stable), and on
    # this set that moves 5 of 1 875 013 transitive reductions into the asymmetric-arc removal that follows -- the graph after
    # asg_symm, every later counter and the GFA are identical (DESIGN.md "Tie order").  The two lines are compared as a sum.
    def norm(lines):
        i = next(k for k, x in enumerate(lines) if "transitively reduced" in x)
        j = next(k for k, x in enumerate(lines) if k > i and "asymmetric arcs" in x)
        num = lambda x: int([t for t in x.split() if t.isdigit()][0])
        return [x for k, x in enumerate(lines) if k not in (i, j)], num(lines[i]) + num(lines[j])
    reference.match((rc_c, out_c, err_c), [paf], lambda r: norm(_counters(r[2])))
    assert any("popped 3713 bubbles" in x for x in _counters(err_c))


@pytest.mark.parametrize("args", ["-n 4000 -l 2000 -L 30000 -c 30 -j 100 -s 41", "-n 20000 -l 1500 -L 40000 -c 40 -j 300 -s 42 -d 20000"])
def test_R_prefilter_on_the_gpu(args, paf_dir):
    """-R (ma_hit_no_cont, hit.c:38-68): read lengths spread over a factor of 20, so hundreds of reads are clearly contained in a
    read twice as long; ids are first appearances among the lines that survive the exclusion.  Output and counters vs the reference."""
    paf = synth.generate(args, os.path.join(paf_dir, "nocont_cli.paf"))
    for extra in ([], ["-b"], ["-c", "2"]):
        rc_c, out_c, err_c = run(CLI, ["-R"] + extra + [paf])
        assert rc_c == 0, err_c.decode()[-2000:]
        reference.match((rc_c, out_c, err_c), ["-R"] + extra + [paf], lambda r: (r[0], r[1], _counters(r[2])))
        dropped = [x for x in _counters(err_c) if "dropped" in x]
        assert dropped and int(dropped[0].split("dropped")[1].split()[0]) > 50
    same(["-R", "-S", "2", "-p", "paf", paf], exact=False)
    same(["-R", "-p", "bed", paf])


def test_version_usage_and_missing_file(pafs):
    reference.match(run(CLI, ["-V"]), ["-V"], lambda r: r[:2])
    rc, out, err = run(CLI, [])
    assert rc == 1 and out == b"" and b"Usage:" in err
    rc_c, out, err = run(CLI, ["/nonexistent.paf"])
    assert rc_c == 1 and b"could not open PAF file" in err
    reference.match((rc_c, out, err), ["/nonexistent.paf"], lambda r: r[0])


def test_with_reads(pafs, paf_dir):
    from tests.test_clean_gpu import _write_reads
    reads = _write_reads(pafs["chaos_small"], os.path.join(paf_dir, "cli_reads.fa"))
    out = same(["-f", reads, pafs["chaos_small"]])
    assert b"\t*\tLN" not in out


def _read_lengths(paf):
    lens = {}
    with open(paf) as f:
        for line in f:
            t = line.split("\t")
            lens[t[0]] = int(t[1]); lens[t[5]] = int(t[6])
    return lens


def _reads_file(paf, path, style, seed=7):
    """A reads file for `paf` in one of the layouts ma_ug_seq (asm.c:236-290, kseq.h:163-211) must cope with."""
    import numpy as np
    rng = np.random.default_rng(seed)
    lens = _read_lengths(paf)
    alphabet = np.frombuffer(b"ACGTNacgtnRYKMBDHVUuWSrykm", dtype=np.uint8)
    names = sorted(lens)
    rng.shuffle(names)
    op = gzip.open if path.endswith(".gz") else open
    eol = b"\r\n" if "crlf" in style else b"\n"
    with op(path, "wb") as f:
        def record(nm, seq):
            if style.startswith("fq"):
                qual = bytes(rng.integers(33, 74, len(seq), dtype=np.uint8))       # includes '@' (64) and '>' (62) and '+' (43) as first bytes now and then
                if "multi" in style:                                               # multi-line FASTQ: only a sequential reader can cut it
                    h = len(seq) // 2
                    f.write(b"@" + nm + b" c" + eol + seq[:h] + eol + seq[h:] + eol + b"+" + eol + qual[:h] + eol + qual[h:] + eol)
                else:
                    f.write(b"@" + nm + b"\tx=1" + eol + seq + eol + b"+" + nm + eol + qual + eol)
            else:
                w = 70 if "wrap" in style else (len(seq) if "one" in style else int(rng.integers(40, 200)))
                f.write(b">" + nm + (b" some comment" if rng.random() < .5 else b"") + eol)
                for i in range(0, len(seq), w):
                    f.write(seq[i:i + w] + eol)
                    if "gaps" in style and rng.random() < .05:
                        f.write(eol)                                               # empty lines are skipped (kseq.h:181)
        for k, nm in enumerate(names):
            if "missing" in style and k % 9 == 0:
                continue                                                           # reads that are not in the file stay N's
            seq = bytes(alphabet[rng.integers(0, len(alphabet), lens[nm])])
            record(nm.encode(), seq)
            if "dups" in style and k % 7 == 0:                                     # same name again with other bases: the later record wins
                record(nm.encode(), bytes(alphabet[rng.integers(0, len(alphabet), lens[nm])]))
            if "extra" in style and k % 5 == 0:
                record(b"not_in_the_layout_%d" % k, b"ACGT" * 50)
    return path


@pytest.mark.parametrize("style,ext", [("fa_wrap", "fa"), ("fa_one_crlf", "fa"), ("fa_var_gaps_extra_dups_missing", "fa"), ("fa_wrap", "fa.gz"),
                                       ("fq", "fq"), ("fq_crlf_extra_dups", "fq"), ("fq_missing", "fq.gz"), ("fq_multi", "fq")])
@pytest.mark.parametrize("name", ["chaos_small", "bubbles800"])
def test_reads_on_the_gpu(style, ext, name, pafs, paf_dir):
    """-f reads: the record index, name table and base gather of ma_ug_seq on the GPU (or, for multi-line FASTQ, the host reader it
    falls back to) against the reference, for FASTA/FASTQ layouts, line ends, compression, missing / foreign / repeated records."""
    reads = _reads_file(pafs[name], os.path.join(paf_dir, f"r_{name}_{style}.{ext}"), style)
    out = same(["-f", reads, pafs[name]])
    assert b"\t*\tLN" not in out
    same(["-f", reads, "-c", "2", "-e", "2", pafs[name]])


def test_reads_wrong_file_is_refused(pafs, paf_dir):
    """asm.c:263 asserts that a record covers the kept interval: a reads file with shorter records aborts with a message."""
    lens = _read_lengths(pafs["chaos_small"])
    path = os.path.join(paf_dir, "short_reads.fa")
    with open(path, "w") as f:
        for nm in lens:
            f.write(f">{nm}\nACGTACGT\n")
    rc, out, err = run(CLI, ["-f", path, pafs["chaos_small"]])
    assert rc != 0 and b"[E::ma_ug_seq]" in err
    rc, out, err = run(CLI, ["-f", "/nonexistent.fa", pafs["chaos_small"]])       # unreadable file: GFA without sequences, like the reference
    assert rc == 0 and b"\t*\tLN" in out
    reference.match((rc, out, err), ["-f", "/nonexistent.fa", pafs["chaos_small"]], lambda r: (r[0], r[1]))


def test_reads_c2_size(paf_dir):
    """BASELINE config 2 (100 K reads / 5 M overlaps) with its 1 GB reads file: -f parity at size, and the wall clocks."""
    import time
    import numpy as np
    paf = synth.generate("c2_100k", os.path.join(paf_dir, "c2.paf"))
    lens = _read_lengths(paf)
    reads = os.path.join(paf_dir, "c2_reads.fa")
    rng = np.random.default_rng(11)
    acgt = np.frombuffer(b"ACGT", dtype=np.uint8)
    with open(reads, "wb") as f:
        for nm, ln in lens.items():
            seq = acgt[rng.integers(0, 4, ln)]
            lines = np.full((ln + 69) // 70 * 71, 10, dtype=np.uint8)
            body = lines.reshape(-1, 71)
            flat = np.concatenate([seq, np.zeros(body.shape[0] * 70 - ln, dtype=np.uint8)]).reshape(-1, 70)
            body[:, :70] = flat
            txt = body.tobytes().replace(b"\x00", b"")
            f.write(b">" + nm.encode() + b"\n" + txt)
    t0 = time.time(); reference.cli(["-f", reads, paf]); t_ref = time.time() - t0
    t0 = time.time(); rc_c, out_c, err_c = run(CLI, ["-f", reads, paf]); t_cli = time.time() - t0
    assert rc_c == 0, err_c.decode()[-2000:]
    reference.match((rc_c, out_c, err_c), ["-f", reads, paf], lambda r: (r[0], r[1]))
    t_ref = f"{t_ref:.2f} s" if reference.LIVE else "not run"
    print(f"c2 with -f: reference {t_ref}, miniasm-b200 {t_cli:.2f} s ({os.path.getsize(reads) / 1e9:.2f} GB of reads)")
    os.unlink(reads)


def test_weird_lines(paf_dir):
    """Parser corners (paf.c:34-67): CRLF, short lines, 10-field lines (stale bl), extra tags, empty lines,
    signs and junk in numeric fields, no trailing newline."""
    base = synth.generate("-n 3000 -s 31 -j 200 -C 200000", os.path.join(paf_dir, "weird_base.paf"))
    lines = open(base, "rb").read().split(b"\n")
    out = []
    for i, ln in enumerate(lines):
        if not ln:
            continue
        f = ln.rstrip(b"\r").split(b"\t")
        if i % 11 == 0 and i > 0:                             # (not the first line: there the reference's bl is uninitialised stack memory)
            out.append(b"\t".join(f[:10]))                    # 10 fields: bl stays stale
        elif i % 13 == 0:
            out.append(b"\t".join(f[:9]))                     # too short: skipped
        elif i % 17 == 0:
            out.append(ln + b"\ttp:A:S\tcm:i:12")             # optional tags
        elif i % 19 == 0:
            out.append(b"")                                   # empty line
            out.append(ln)
        elif i % 23 == 0:
            f[2] = b"+" + f[2]; f[9] = f[9] + b"xyz"
            out.append(b"\t".join(f))                         # strtol corner cases
        elif i % 29 == 0:
            f[1] = b" " + f[1]
            out.append(b"\t".join(f) + b"\r")
        else:
            out.append(ln)
    path = os.path.join(paf_dir, "weird.paf")
    with open(path, "wb") as fo:
        fo.write(b"\n".join(out))                             # no newline at the end
    same([path])
    same(["-S", "2", "-p", "paf", path], exact=False)


SEAM = os.path.join(ROOT, "oracle", "_ref", "miniasm_seam")


@pytest.mark.skipif(not os.path.exists(SEAM), reason="oracle/_ref/miniasm_seam not built")
@pytest.mark.parametrize("opts", [[], ["-p", "sg"], ["-R"], ["-c", "2", "-e", "2"]])
def test_link_seam(opts, pafs):
    """The reference's own main.o (compiled from its main.c, untouched) linked against libminiasm_b200.so:
    every library call of main.c:108-199 lands in the CUDA path, the GFA must be the reference's."""
    rc_r, out_r, _ = run(reference.REF_CLI, opts + [pafs["chaos_small"]])
    rc_s, out_s, err = run(SEAM, opts + [pafs["chaos_small"]])
    assert rc_s == rc_r == 0, err.decode()[-2000:]
    if "sg" in opts:
        assert sorted(out_s.splitlines()) == sorted(out_r.splitlines())
    else:
        assert out_s == out_r


@pytest.mark.parametrize("content", [b"", b"\n", b"\n\n\n", b"not a paf line\n", b"a\t1\t2\n",
                                     b"q\t5000\t0\t4000\t+\tt\t5000\t1000\t5000\t800\t4000\t255\n",            # one overlap: too shallow for min_dp
                                     b"q\t5000\t0\t100\t+\tt\t5000\t0\t100\t80\t100\t255\n",                   # below min_span: nothing stored
                                     b"q\t5000\t0\t4000\t+\tq\t5000\t1000\t5000\t800\t4000\t255\n"])           # self hit only
def test_degenerate_inputs(content, paf_dir):
    """Empty / all-filtered / single-line inputs: same (possibly empty) output and exit status as the reference."""
    path = os.path.join(paf_dir, "degenerate.paf")
    with open(path, "wb") as f:
        f.write(content)
    same([path])
    same(["-S", "2", "-p", "paf", path], exact=False)
    same(["-p", "sg", path], exact=False)


def test_long_read_names(built, paf_dir, tmp_path):
    """Read names beyond 65535 bytes (ADVICE round 1: the round-1 parser kept 16-bit name lengths and gave up; the reference takes
    any length, paf.c / kseq getuntil).  Two of the names differ only in their last byte, which the dictionary's witness comparison
    has to reach."""
    src = synth.generate("tiny_exact", f"{paf_dir}/tiny_exact.paf")
    long_a, long_b = "L" * 70000 + "a", "L" * 70000 + "b"
    ren = {"r206": long_a, "r27": long_b, "r172": "M" * 66000}
    dst = str(tmp_path / "long.paf")
    with open(src) as f, open(dst, "w") as g:
        for line in f:
            c = line.split("\t")
            c[0], c[5] = ren.get(c[0], c[0]), ren.get(c[5], c[5])
            g.write("\t".join(c))
    same([dst])
    bed = same(["-S", "2", "-p", "bed", dst])
    assert long_a.encode() + b"\t" in bed and long_b.encode() + b"\t" in bed and b"M" * 66000 + b"\t" in bed
    same(["-R", dst])
