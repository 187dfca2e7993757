#!/usr/bin/env python
"""bench.py -- PAF overlaps/s, ingest -> GFA, on synthetic PAF of the shapes BASELINE.json names.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload NAME] [--impl b200|reference] [--quick] [--dump-outputs DIR]

One "step" = one pass of the whole hot path over one PAF: parse -> read selection -> string graph ->
transitive reduction -> cleaning -> unitigs (main.c:108-199 of the reference).

Workload: N=1 BASELINE config 3 (1 M reads / 50 M overlaps); N=2 the same law at 2 M reads; N=4 config 4 (4 M / 200 M);
N=8 config 5 (8 M reads / 400 M overlaps, two hot loci of 10 000 reads).  At N>1 the job is ONE PAF cut into N parts in
file order (rank r generates and holds part r), read ids are hash-sharded (owner = id mod N).

* value  : whole-job PAF records/s with the PAF bytes already resident in HBM (timed on the device, CUDA
           events on the library's stream, max over ranks).
* e2e    : the same through the C ABI with HOST buffers: pinned PAF text -> H2D (in chunks; at N=1 the chunks that have arrived
           are parsed while the next ones cross PCIe, mab_load_ingest_text) -> all steps -> GFA text (formatted on the GPU, one
           D2H, written to /dev/null by rank 0); wall clock bracketed by device synchronisation.
* roofline : asg_arc_del_trans kernel, algorithmic bytes / CUDA-event time vs the measured HBM copy peak;
  roofline_phases: the other phases against SURVEY.md 8(d)'s byte counts.
* check  : sha256 of the GFA text of the last step (compared with tests/golden/configs.json when the workload has a
           digest of the reference's GFA there), arcs reduced, unitigs.
* cpu_baseline : the unmodified reference (oracle/_ref, single-threaded as it is) on a bounded sample of the same law;
  cpu_full_size: ONE run of it on the full workload (N=1 only; cached in /dev/shm between the two arms of a bench run).
* cli    : the drop-in command line, cold process, PAF in /dev/shm, GFA to /dev/null (cli_wall_s).
* noisy  : a 600 K-read set with jittered ends (tips, thousands of bubbles) through the same legs, next to the
           reference's time on the same file.
* host_affinity : every rank runs on the host cores NVML names for its GPU (bound before the pinned buffers are allocated).
--impl reference prints the same line for the reference's own CPU implementation (rank 0 only).
--dump-outputs DIR writes the unitig graph the last timed step left (what mab_export_ug / _dict / _sub hand a caller) as
float64 .npy files, so that two builds can be compared output for output on the same seeded input.
"""
import argparse
import ctypes as C
import hashlib
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from miniasm_b200 import synth  # noqa: E402

# workload -> pafgen options (SURVEY.md section 8d: fixed 10 kb reads, 62.5x, >= 2 kb overlaps, ~50 lines/read)
WORKLOADS = {
    "c2_100k": dict(args=synth.CONFIGS["c2_100k"], label="Synthetic PAF: 100K reads / 5M overlaps"),
    "c3_1m": dict(args=synth.CONFIGS["c3_1m"], label="Synthetic PAF: 1M reads / 50M overlaps (C. elegans-scale)"),
    "c3_2m": dict(args=synth.CONFIGS["c3_2m"], label="Synthetic PAF: 2M reads / 100M overlaps (config 3's law)"),
    "c4_4m": dict(args=synth.CONFIGS["c4_4m"], label="Synthetic PAF: 4M reads / 200M overlaps"),
    "c5_8m_skew": dict(args=synth.CONFIGS["c5_8m_skew"], label="Synthetic PAF: 8M reads / 400M overlaps, skewed degree (hot loci of 10 000 reads)"),
    "noisy_600k": dict(args="-n 600000 -l 9000 -L 11000 -j 800 -c 30 -s 15", label="Synthetic PAF: 600K reads U[9k,11k] / 30x / ends jittered by U[0,800] (tips and bubbles)"),
    "skew_1m": dict(args="-n 1000000 -s 5 -H 1 -R 10000 -W 8000", label="Synthetic PAF: 1M reads / 50M overlaps + one hot locus of 10 000 reads (50M more overlaps, ~10 000 hits per hot read)"),
    "tiny": dict(args="-n 20000 -s 12", label="Synthetic PAF: 20K reads / 1M overlaps (smoke)"),
}
BY_GPUS = {1: "c3_1m", 2: "c3_2m", 4: "c4_4m", 8: "c5_8m_skew"}
CPU_SAMPLE = "-n 100000 -s 2"  # reference arm / cpu_baseline sample: config 3's law at 100K reads ~ 5M PAF lines (~5-8 s of CPU)
METRIC = "paf_overlaps_per_sec_ingest_to_gfa"
DTYPE = "int64/uint32 (+3 float32 predicates)"


class PafgenOpt(C.Structure):
    _fields_ = [("n_reads", C.c_uint32), ("len_min", C.c_uint32), ("len_max", C.c_uint32), ("coverage", C.c_double),
                ("min_olap", C.c_uint32), ("jitter", C.c_uint32), ("seed", C.c_uint64),
                ("n_hot", C.c_uint32), ("hot_reads", C.c_uint32), ("hot_span", C.c_uint32),
                ("dup_ppm", C.c_uint32), ("self_ppm", C.c_uint32), ("internal_ppm", C.c_uint32), ("lowid_ppm", C.c_uint32),
                ("shuffle", C.c_uint32), ("flip_ppm", C.c_uint32), ("name_base", C.c_uint32), ("part", C.c_uint32), ("n_parts", C.c_uint32)]


class PafgenStat(C.Structure):
    _fields_ = [("n_lines", C.c_uint64), ("n_bytes", C.c_uint64), ("genome_len", C.c_uint64), ("n_reads_total", C.c_uint32)]


_OPT_FIELDS = {"-n": ("n_reads", int), "-l": ("len_min", int), "-L": ("len_max", int), "-c": ("coverage", float), "-m": ("min_olap", int),
               "-j": ("jitter", int), "-s": ("seed", int), "-H": ("n_hot", int), "-R": ("hot_reads", int), "-W": ("hot_span", int),
               "-d": ("dup_ppm", int), "-S": ("self_ppm", int), "-I": ("internal_ppm", int), "-D": ("lowid_ppm", int), "-C": ("flip_ppm", int)}


def generate_args(args, part=0, n_parts=1):
    """PAF text for a pafgen command line, in C heap memory: (pointer, n_bytes, n_lines, free_fn).  n_parts > 1: only part `part`."""
    synth.build()
    lib = C.CDLL(synth.LIB)
    lib.pafgen_defaults.argtypes = [C.POINTER(PafgenOpt)]
    lib.pafgen_generate.restype = C.c_size_t
    lib.pafgen_generate.argtypes = [C.POINTER(PafgenOpt), C.POINTER(C.c_void_p), C.POINTER(PafgenStat)]
    lib.pafgen_free.argtypes = [C.c_void_p]
    o, st, buf = PafgenOpt(), PafgenStat(), C.c_void_p()
    lib.pafgen_defaults(C.byref(o))
    tok = args.split()
    i = 0
    while i < len(tok):
        if tok[i] == "-x":
            o.shuffle = 1
            i += 1
            continue
        name, conv = _OPT_FIELDS[tok[i]]
        setattr(o, name, conv(tok[i + 1]))
        i += 2
    if o.len_max < o.len_min:
        o.len_max = o.len_min
    o.part, o.n_parts = part, n_parts
    n = lib.pafgen_generate(C.byref(o), C.byref(buf), C.byref(st))
    return buf, n, st.n_lines, lambda: lib.pafgen_free(buf)


def generate(n_reads, seed, name_base=0):
    """Config-3 law at n_reads reads (kept for the tests that name a BASELINE config by (n_reads, seed))."""
    return generate_args(f"-n {n_reads} -s {seed}")


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu):
        super().__init__(daemon=True)
        self.gpu, self.rows, self.stop_flag, self.proc = gpu, [], False, None

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                self.rows.append([x.strip() for x in line.split(",")])
                if self.stop_flag:
                    break
        except Exception:
            pass

    def finish(self):
        self.stop_flag = True
        if self.proc:
            self.proc.terminate()
        sm = sorted(int(r[0]) for r in self.rows if r and r[0].isdigit())
        busy = [x for x in sm if x > 0]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            for k, nm in enumerate(names):
                if len(r) > 3 + k and r[3 + k].lower().startswith("active"):
                    reasons.add(nm)
        mx = max((int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()), default=None)
        return {"sm_mhz": busy[len(busy) // 2] if busy else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(self.rows)}


REF_TIMED = os.path.join(ROOT, "oracle", "_ref", "miniasm_ref_timed")


def write_paf(args, path):
    """PAF of a pafgen command line as a file (+ .n with its line count); reused if it is already there."""
    if not (os.path.exists(path) and os.path.exists(path + ".n")):
        buf, n, n_lines, free = generate_args(args)
        with open(path, "wb") as f:
            f.write((C.c_char * n).from_address(buf.value))
        free()
        with open(path + ".n", "w") as f:
            f.write(str(n_lines))
    return int(open(path + ".n").read())


def run_reference(paf, n_lines):
    """One run of the unmodified reference (oracle/_ref/miniasm_ref_timed) on a PAF file; returns its timing dict."""
    if not os.path.exists(REF_TIMED):
        raise FileNotFoundError("oracle/_ref/miniasm_ref_timed missing (run __graft_entry__.build() where /root/reference is mounted)")
    t0 = time.perf_counter()
    r = subprocess.run([REF_TIMED, paf], stdout=subprocess.DEVNULL, stderr=subprocess.PIPE, text=True)
    wall = time.perf_counter() - t0
    tj = [ln for ln in r.stderr.splitlines() if ln.startswith("[T] ")]
    t = json.loads(tj[-1][4:]) if tj else {}
    t["wall"], t["n_lines"] = wall, n_lines
    return t


def reference_full_size(name, shm, model, cores):
    """cpu_full_size: ONE run of the reference on the whole workload; the result is kept in /dev/shm so that the two arms of
    one bench run (reference arm first, then ours) pay for it once."""
    cache = os.path.join(shm, f"mab_ref_full_{name}.json")
    if os.path.exists(cache):
        try:
            d = json.load(open(cache))
            d["cached"] = True
            return d
        except (OSError, ValueError):
            pass
    paf = os.path.join(shm, f"mab_{name}.paf")
    n_lines = write_paf(WORKLOADS[name]["args"], paf)
    t = run_reference(paf, n_lines)
    d = {"value": n_lines / t["wall"], "unit": "PAF records/s", "seconds": t["wall"], "n_lines": n_lines, "cores": 1, "kind": "reference",
         "workload": name, "host": f"{model} ({cores} logical cores; the reference is single-threaded)",
         "del_trans_arcs_per_sec": t["n_arc_del_trans_in"] / t["asg_arc_del_trans"] if t.get("asg_arc_del_trans") else None,
         "seconds_by_function": {k: round(v, 4) for k, v in t.items() if isinstance(v, float) and k not in ("total", "wall")}, "cached": False}
    try:
        json.dump(d, open(cache, "w"))
    except OSError:
        pass
    return d


def bind_near_gpu(torch, ordinal):
    """Run this process on the host cores next to its GPU (NVML's CPU affinity of the device), before any pinned buffer exists: the
    buffers then live on that NUMA node and the H2D copies of several ranks do not cross the socket link.  Best effort: any
    failure leaves the affinity as it was.  Returns what was done, for the JSON line."""
    try:
        import pynvml
        pynvml.nvmlInit()
        try:
            pr = torch.cuda.get_device_properties(ordinal)
            h = pynvml.nvmlDeviceGetHandleByPciBusId(f"{pr.pci_domain_id:08X}:{pr.pci_bus_id:02X}:{pr.pci_device_id:02X}.0")
        except Exception:  # noqa: BLE001 -- older torch without the PCI fields: NVML order = CUDA order unless CUDA_VISIBLE_DEVICES reorders
            h = pynvml.nvmlDeviceGetHandleByIndex(ordinal)
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        cpus = {64 * w + b for w, word in enumerate(words) for b in range(64) if word >> b & 1} & os.sched_getaffinity(0)
        if not cpus:
            return {"bound": False, "why": "NVML affinity mask does not meet the allowed CPUs"}
        os.sched_setaffinity(0, cpus)
        return {"bound": True, "cpus": len(cpus), "source": "NVML CPU affinity of the GPU"}
    except Exception as ex:  # noqa: BLE001
        return {"bound": False, "why": f"{type(ex).__name__}: {ex}"[:120]}


def host_cpu():
    model = "unknown"
    try:
        for ln in open("/proc/cpuinfo"):
            if ln.startswith("model name"):
                model = ln.split(":", 1)[1].strip()
                break
    except OSError:
        pass
    return model, os.cpu_count()


def config_of(name, world):
    """The `config` object: identical in both arms (the reference arm describes its bounded sample in cpu_baseline.sample)."""
    return {"workload": WORKLOADS[name]["label"], "name": name, "pafgen": WORKLOADS[name]["args"],
            "l2": "inputs larger than L2 (PAF text and hit arrays are GBs; no flush needed)",
            "parallelism": (f"one PAF cut into {world} parts in file order; read ids hash-sharded over {world} GPUs (owner = id mod {world}); NCCL "
                            f"all-to-all of hits, all-reduce of interval/flag tables, all-gather of names and surviving arcs, neighbour slabs read from peers over NVLink")
            if world > 1 else "1 GPU"}


DUMP_MAX_BYTES = 60 << 20   # whole dump; rows beyond an even share per array are a seeded sample (the limit is 64 MB)


def dump_outputs(lib, ctx, out_dir):
    """The layout the pipeline hands a caller, as float64 arrays (every value below 2^53, so exact).  Each array's column 0 is
    the row index, so that a sampled array (a fixed, seeded sample of the rows beyond its share of DUMP_MAX_BYTES) can still be
    compared row by row.  Tables without rows are not written."""
    import numpy as np
    from miniasm_b200 import capi
    d, sub, ug = lib.mab_export_dict(ctx), lib.mab_export_sub(ctx), lib.mab_export_ug(ctx)
    u, n_seq = ug.contents, d.contents.n_seq
    utgs = [u.a[i] for i in range(u.n)]
    reads = capi.np_from_ptr(sub, n_seq, capi.SUB_DT) if sub else np.zeros(n_seq, dtype=capi.SUB_DT)
    seq_len = np.array([d.contents.seq[i].len for i in range(n_seq)], dtype=np.float64)
    members = np.concatenate([capi.np_from_ptr(x.a, x.n, np.uint64) for x in utgs]) if utgs else np.zeros(0, np.uint64)
    arcs = lib.read_graph(u.g)[0]
    tables = {
        "unitigs": np.array([[x.len_circ & 0x7fffffff, x.len_circ >> 31, x.start, x.end, x.n] for x in utgs]).reshape(-1, 5),  # length, circular, ends, reads
        "unitig_reads": np.stack([np.repeat(np.arange(len(utgs)), [x.n for x in utgs]), members >> 32, members & 0xffffffff], 1),
        "unitig_arcs": np.stack([arcs["ul"] >> 32, arcs["ul"] & 0xffffffff, arcs["v"], arcs["ol_del"] & 0x7fffffff, arcs["ol_del"] >> 31], 1),
        "reads": np.stack([seq_len, reads["s_del"] & 0x7fffffff, reads["s_del"] >> 31, reads["e"]], 1),            # length, kept interval
    }
    tables = {k: t for k, t in tables.items() if len(t)}       # e.g. no links between unitigs: an empty array compares nothing
    max_rows = DUMP_MAX_BYTES // (8 * sum(t.shape[1] + 1 for t in tables.values()))
    os.makedirs(out_dir, exist_ok=True)
    total = 0
    for name, t in tables.items():
        t = t.astype(np.float64)
        rows = np.arange(len(t))
        if len(t) > max_rows:
            rows = np.sort(np.random.default_rng(0).choice(len(t), max_rows, replace=False))
        t = np.concatenate([rows[:, None].astype(np.float64), t[rows]], 1)
        np.save(os.path.join(out_dir, f"{name}.npy"), t)
        total += t.nbytes
    lib.ma_ug_destroy(ug), capi.c_free(sub), lib.sd_destroy(d)
    assert total <= 64 << 20, total


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default=None, choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--quick", action="store_true", help="skip the extra legs: full-size reference run, cold CLI wall clock, noisy workload")
    ap.add_argument("--host-gfa", action="store_true", help="e2e leg: host structs + ma_ug_print instead of the GFA text formatted on the GPU (mab_write_gfa)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the unitig graph of the last timed step to DIR/<name>.npy (float64)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    name = a.workload or BY_GPUS.get(world) or "c3_1m"
    wl = WORKLOADS[name]
    model, cores = host_cpu()
    shm = "/dev/shm" if os.path.isdir("/dev/shm") else tempfile.gettempdir()
    extras = world == 1 and not a.quick and not a.no_cpu_baseline and name == "c3_1m"

    # ------------------------------------------------------------------ reference arm
    if a.impl == "reference":
        if rank != 0:
            return
        paf = os.path.join(shm, "mab_cpu_sample.paf")
        n_lines = write_paf(CPU_SAMPLE, paf)
        secs, t = [], {}
        for i in range(a.warmup + a.steps):
            t = run_reference(paf, n_lines)
            if i >= a.warmup:
                secs.append(t["wall"])
        mean = sum(secs) / len(secs)
        v = n_lines / mean
        sample = f"pafgen {CPU_SAMPLE}: 100 000 reads / {n_lines} PAF lines of config 3's law (fixed 10 kb reads, 62.5x); one full run of the reference per step"
        line = {
            "impl": "reference", "metric": METRIC, "value": v, "unit": "PAF records/s", "n_gpus": a.gpus,
            "steps": a.steps, "warmup": a.warmup, "ms_per_step": mean * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": DTYPE, "data": "synthetic", "config": config_of(name, world),
            "cpu_baseline": {"value": v, "unit": "PAF records/s", "cores": 1, "kind": "reference", "sample": sample,
                             "host": f"{model} ({cores} logical cores; the reference is single-threaded)",
                             "del_trans_arcs_per_sec": t.get("n_arc_del_trans_in", 0) / t["asg_arc_del_trans"] if t.get("asg_arc_del_trans") else None},
            "e2e": {"value": v, "unit": "PAF records/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        }
        if world == 1 and not a.quick and name == "c3_1m":
            try:
                line["cpu_full_size"] = reference_full_size(name, shm, model, cores)
            except Exception as ex:  # noqa: BLE001
                line["cpu_full_size"] = {"value": None, "error": str(ex)}
        print(json.dumps(line))
        return

    # ------------------------------------------------------------------ B200 arm
    os.environ.setdefault("NCCL_DEBUG", "WARN")
    saved_stdout = os.dup(1)                  # libraries (NCCL banner ...) must not add lines to stdout: the JSON line is the only one
    os.dup2(2, 1)
    import torch
    import torch.distributed as dist
    from miniasm_b200 import capi
    if not torch.cuda.is_available():
        sys.exit("bench.py: no CUDA device; the product has no CPU path")
    torch.cuda.set_device(local_rank)
    affinity = bind_near_gpu(torch, local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    lib = capi.load_product()
    lib.set_verbose(0)
    ctx = lib.mab_create(local_rank)
    opt = lib.default_opt()
    if world > 1:
        from miniasm_b200 import sharded
        sharded.init(lib, ctx, rank, world)        # NCCL communicator inside the library (id handed over through torch.distributed)
    devnull = capi._libc.fopen(b"/dev/null", b"w")

    def device_steps():
        if world > 1:
            lib.mab_ingest_sharded(ctx, opt.min_span, opt.min_match, 1)
            lib.mab_select_sharded(ctx, C.byref(opt))
            lib.mab_layout_sharded(ctx, C.byref(opt))
        else:
            lib.mab_ingest(ctx, opt.min_span, opt.min_match, 1)
            lib.mab_select(ctx, C.byref(opt), 0, 0, 100)
            lib.mab_layout(ctx, C.byref(opt), 100)
        lib.mab_unitigs(ctx)

    def barrier():
        lib.mab_sync(ctx)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    def measure(args_str, steps, warmup, with_roofline, dump_dir=None):
        """value + e2e legs over one PAF (this rank's part of it)."""
        buf, n_bytes, n_lines, free = generate_args(args_str, rank, world)
        pinned = torch.empty(max(n_bytes, 1), dtype=torch.uint8, pin_memory=True)
        C.memmove(pinned.data_ptr(), buf, n_bytes)
        free()

        def e2e_step():
            if world > 1:                                                      # H2D in chunks, parsed while the next ones arrive
                lib.mab_load_ingest_text_sharded(ctx, pinned.data_ptr(), n_bytes, opt.min_span, opt.min_match, 1)
                lib.mab_select_sharded(ctx, C.byref(opt))
                lib.mab_layout_sharded(ctx, C.byref(opt))
                lib.mab_unitigs(ctx)
            else:
                lib.mab_load_ingest_text(ctx, pinned.data_ptr(), n_bytes, opt.min_span, opt.min_match, 1)
                lib.mab_select(ctx, C.byref(opt), 0, 0, 100)
                lib.mab_layout(ctx, C.byref(opt), 100)
                lib.mab_unitigs(ctx)
            if rank != 0:                                                      # the result is replicated; rank 0 writes it
                return 0
            if not a.host_gfa:                                                 # GFA text formatted on the GPU, one D2H of the text
                return lib.mab_write_gfa(ctx, devnull)
            d, sub, ug = lib.mab_export_dict(ctx), lib.mab_export_sub(ctx), lib.mab_export_ug(ctx)   # D2H
            lib.ma_ug_print(ug, d, sub, devnull)                               # GFA text (host C writer)
            g = ug.contents.g.contents
            nb = (g.n_arc_srt & 0x7fffffff) * 16 + (g.n_seq_symm & 0x7fffffff) * 20
            nb += sum(ug.contents.a[i].n for i in range(min(ug.contents.n, 100000))) * 8 + ug.contents.n * 24
            nb += d.contents.n_seq * (8 + 12)
            lib.ma_ug_destroy(ug), capi.c_free(sub), lib.sd_destroy(d)
            return nb

        # ---- value: inputs resident in HBM, device-timed
        lib.mab_load_paf_text(ctx, pinned.data_ptr(), n_bytes)
        inner = 0
        if with_roofline:
            lib.mab_count_del_trans_inner(1)      # one untimed pass with the instrumented kernel: inner-loop iterations I
            device_steps()
            inner = lib.mab_stats(ctx).contents.trans_inner   # (N > 1: this rank's share of the vertices)
            lib.mab_count_del_trans_inner(0)
        for _ in range(warmup):
            device_steps()
        st = lib.mab_stats(ctx).contents
        launches0, libcalls0 = st.n_kernel_launches, st.n_lib_calls
        e0, e1 = lib.mab_event_create(), lib.mab_event_create()
        barrier()
        dt_ms, t_wall0 = [], time.perf_counter()
        for _ in range(steps):
            lib.mab_event_record(ctx, e0)
            device_steps()
            lib.mab_event_record(ctx, e1)
            ms = lib.mab_event_elapsed_ms(e0, e1)
            lib.mab_sync(ctx)
            dt_ms.append((ms, lib.mab_stats(ctx).contents.ms_del_trans_kernel))
        barrier()
        wall_dev = time.perf_counter() - t_wall0
        if dump_dir and rank == 0:                  # untimed; the graph is replicated on every rank
            dump_outputs(lib, ctx, dump_dir)
        st = lib.mab_stats(ctx).contents
        cl = [C.c_uint32() for _ in range(4)]
        lib.mab_clean_totals(*[C.byref(x) for x in cl])
        res = {"n_lines": n_lines, "n_bytes": n_bytes, "inner": inner, "dev_ms": sum(x[0] for x in dt_ms), "kernel_ms": sum(x[1] for x in dt_ms) / len(dt_ms),
               "launches": st.n_kernel_launches - launches0, "libcalls": st.n_lib_calls - libcalls0, "wall_dev": wall_dev,
               "n_arc_in": st.n_arc_trans_in, "n_vtx": 2 * st.n_seq_final // world, "n_reduced": st.n_reduced, "n_utg": st.n_utg, "n_arc_sg": st.n_arc_sg,
               "n_hits": st.n_hits_stored, "n_hits_final": st.n_hits_final, "n_seq": st.n_seq_in,
               "phases": {"ingest": st.ms_ingest, "select": st.ms_select, "layout": st.ms_layout, "unitigs": st.ms_unitigs},
               "cleaning": {"passes": cl[0].value, "max_sweeps_of_a_pass": cl[1].value, "sweeps": cl[2].value, "actions": cl[3].value}}
        lib.mab_event_destroy(e0), lib.mab_event_destroy(e1)
        # ---- e2e: host buffers in, GFA text out
        for _ in range(min(warmup, 2)):
            e2e_step()
        barrier()
        t0 = time.perf_counter()
        d2h = 0
        for _ in range(steps):
            d2h = e2e_step()
        barrier()
        res["e2e_s"], res["d2h"] = time.perf_counter() - t0, d2h
        # ---- check: digest of the GFA text of the state the last step left (untimed)
        if rank == 0:
            with tempfile.NamedTemporaryFile(dir=shm, delete=False) as tf:
                path = tf.name
            fp = capi._libc.fopen(path.encode(), b"w")
            lib.mab_write_gfa(ctx, fp)
            capi._libc.fclose(fp)
            h = hashlib.sha256()
            with open(path, "rb") as f:
                for blk in iter(lambda: f.read(1 << 24), b""):
                    h.update(blk)
            res["gfa_sha256"], res["gfa_bytes"] = h.hexdigest(), os.path.getsize(path)
            os.unlink(path)
        del pinned
        return res

    def reduce_ranks(res):
        tot = torch.tensor([res["dev_ms"], res["e2e_s"], float(res["n_lines"]), float(res["n_bytes"])], dtype=torch.float64, device="cuda")
        if world > 1:
            mx, sm = tot.clone(), tot.clone()
            dist.all_reduce(mx, op=dist.ReduceOp.MAX)
            dist.all_reduce(sm, op=dist.ReduceOp.SUM)
            return mx[0].item(), mx[1].item(), sm[2].item(), sm[3].item()
        return res["dev_ms"], res["e2e_s"], float(res["n_lines"]), float(res["n_bytes"])

    sampler = ClockSampler(local_rank)
    sampler.start()
    res = measure(wl["args"], a.steps, a.warmup, True, a.dump_outputs)
    clocks = sampler.finish()
    dev_ms, e2e_s, lines_all, bytes_all = reduce_ranks(res)

    noisy = None
    if extras:  # the bubble/tip-dense set through the same legs (1 GPU only)
        nres = measure(WORKLOADS["noisy_600k"]["args"], 3, 1, False)
        noisy = {"workload": WORKLOADS["noisy_600k"]["label"], "pafgen": WORKLOADS["noisy_600k"]["args"], "paf_lines": nres["n_lines"],
                 "value": nres["n_lines"] * 3 / (nres["dev_ms"] * 1e-3), "ms_per_step": nres["dev_ms"] / 3,
                 "e2e": {"value": nres["n_lines"] * 3 / nres["e2e_s"], "ms_per_step": nres["e2e_s"] / 3 * 1e3},
                 "phase_ms_last_step": nres["phases"], "n_reduced": nres["n_reduced"], "n_utg": nres["n_utg"], "gfa_sha256": nres["gfa_sha256"],
                 "cleaning_passes": nres["cleaning"]}

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except OSError:
            pass
        peak, peak_src = (peaks["hbm_gbs"], "measured (MEASURED_PEAKS.json, burst copy)") if "hbm_gbs" in peaks else (6650.0, "fallback (B200_PROFILING.md)")
        n_arc_in, n_vtx, inner, kms = res["n_arc_in"], res["n_vtx"], res["inner"], res["kernel_ms"]
        alg_bytes = 16 * n_arc_in + 16 * inner + 1 * n_arc_in + 12 * n_vtx     # DESIGN.md "roofline": own slab + explored neighbour prefixes + flag byte + idx/seq
        achieved = alg_bytes / (kms * 1e-3) / 1e9 if kms else 0.0
        traffic = None                             # measured DRAM bytes of one launch: from the committed ncu capture of THIS kernel on THIS workload, 1 GPU only
        prof = os.path.join(ROOT, "profiles", "del_trans_r02.json")
        if world == 1 and os.path.exists(prof):
            try:
                pj = json.load(open(prof))
                if pj.get("workload") == name:
                    traffic = pj.get("dram_bytes_per_launch")
            except (OSError, ValueError):
                pass
        # the other phases against SURVEY.md 8(d): algorithmic bytes / CUDA-event time of the phase (rank 0's share at N > 1)
        n_hits, n_arc_sg, ph = res["n_hits"] // world, res["n_arc_sg"] // world, res["phases"]
        hit_bits = 32 + max(1, (max(res["n_seq"], 2) - 1).bit_length())
        hit_passes = (hit_bits + 7) // 8
        ingest_b = 61 * res["n_lines"] + 2 * 32 * res["n_lines"] + 32 * n_hits * (2 * hit_passes + 1)
        select_b = 208 * n_hits
        sg_b = 32 * (res["n_hits_final"] // world) + 16 * n_arc_sg + 16 * n_arc_sg * 3   # read the hits, write the arcs, order them (one more read + write) and index them
        phases = {}
        for k, b, ms, what in (("ingest", ingest_b, ph["ingest"], "61 B text + 2x32 B hits per line + 32 B x n_hits x (2P+1) for the P-pass hit sort"),
                               ("select", select_b, ph["select"], "208 B per stored hit (fused floor of the six passes)"),
                               ("layout", sg_b + alg_bytes, ph["layout"], "ma_sg_gen (32 B hit in, 16 B arc out, ordering) + asg_arc_del_trans bytes; the rest of the phase works on the 2 % graph")):
            gbs = b / (ms * 1e-3) / 1e9 if ms else 0.0
            phases[k] = {"ms": ms, "algorithmic_bytes": b, "achieved": gbs, "frac": gbs / peak if peak else None, "bytes": what}
        gold = None
        try:
            gj = json.load(open(os.path.join(ROOT, "tests", "golden", "configs.json")))
            if name in gj:
                gold = gj[name]["gfa_sha256"]
        except (OSError, ValueError):
            pass
        cpu = full = cli = None
        if not a.no_cpu_baseline and world == 1:
            try:
                paf = os.path.join(shm, "mab_cpu_sample.paf")
                n_s = write_paf(CPU_SAMPLE, paf)
                t = run_reference(paf, n_s)
                cpu = {"value": n_s / t["total"], "unit": "PAF records/s", "cores": 1, "kind": "reference",
                       "sample": f"pafgen {CPU_SAMPLE}: 100 000 reads / {n_s} PAF lines of config 3's law, one run of oracle/_ref/miniasm_ref_timed ({t['total']:.2f} s)",
                       "host": f"{model} ({cores} logical cores; the reference is single-threaded)",
                       "del_trans_arcs_per_sec": t["n_arc_del_trans_in"] / t["asg_arc_del_trans"],
                       "seconds_by_function": {k: round(v, 4) for k, v in t.items() if isinstance(v, float) and k not in ("total", "wall")}}
            except Exception as ex:  # noqa: BLE001
                cpu = {"value": None, "error": str(ex)}
        if extras:
            try:
                full = reference_full_size(name, shm, model, cores)
            except Exception as ex:  # noqa: BLE001
                full = {"value": None, "error": str(ex)}
            exe = os.path.join(ROOT, "miniasm_b200", "miniasm-b200")
            env = {**os.environ, "MINIASM_B200_DEVICE": str(local_rank)}
            try:   # the drop-in command line, cold: new process, CUDA context, arena, file read from /dev/shm, GFA to /dev/null
                paf = os.path.join(shm, f"mab_{name}.paf")
                n_l = write_paf(wl["args"], paf)
                t0 = time.perf_counter()
                r = subprocess.run([exe, paf], stdout=subprocess.DEVNULL, stderr=subprocess.PIPE, text=True, env=env)
                w = time.perf_counter() - t0
                foot = [ln for ln in r.stderr.splitlines() if "Real time" in ln]
                cli = {"cli_wall_s": w, "rc": r.returncode, "records_per_s": n_l / w, "footer": foot[-1] if foot else None,
                       "cmd": "miniasm-b200 /dev/shm/<c3>.paf > /dev/null (cold process; the bench process keeps its own context alive meanwhile)"}
            except Exception as ex:  # noqa: BLE001
                cli = {"cli_wall_s": None, "error": str(ex)}
            if noisy is not None:
                try:
                    paf = os.path.join(shm, "mab_noisy_600k.paf")
                    n_l = write_paf(WORKLOADS["noisy_600k"]["args"], paf)
                    t = run_reference(paf, n_l)
                    noisy["reference"] = {"seconds": t["wall"], "value": n_l / t["wall"],
                                          "cleaning_seconds": sum(t.get(k, 0.0) for k in ("asg_cut_tip", "asg_pop_bubble", "asg_cut_internal", "asg_cut_biloop", "asg_arc_del_short"))}
                    t0 = time.perf_counter()
                    subprocess.run([exe, paf], stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL, env=env)
                    noisy["cli_wall_s"] = time.perf_counter() - t0
                except Exception as ex:  # noqa: BLE001
                    noisy["reference"] = {"error": str(ex)}
        sys.stdout.flush()
        os.dup2(saved_stdout, 1)
        line = {
            "metric": METRIC, "value": lines_all * a.steps / (dev_ms * 1e-3), "unit": "PAF records/s",
            "n_gpus": world, "steps": a.steps, "warmup": a.warmup, "ms_per_step": dev_ms / a.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": DTYPE, "data": "synthetic", "config": config_of(name, world),
            "input": {"paf_lines": int(lines_all), "paf_bytes": int(bytes_all), "paf_lines_rank0": res["n_lines"], "paf_bytes_rank0": res["n_bytes"]},
            "e2e": {"value": lines_all * a.steps / e2e_s, "unit": "PAF records/s", "ms_per_step": e2e_s / a.steps * 1e3,
                    "h2d_bytes_per_step": int(bytes_all), "d2h_bytes_per_step": res["d2h"],
                    "writer": "mab_export_* + ma_ug_print (host)" if a.host_gfa else "mab_write_gfa (text formatted on the GPU)"},
            "check": {"gfa_sha256": res["gfa_sha256"], "gfa_bytes": res["gfa_bytes"], "n_reduced": res["n_reduced"], "n_utg": res["n_utg"],
                      "reference_gfa_sha256": gold, "matches_reference": (res["gfa_sha256"] == gold) if gold else None},
            "gpu_launches": res["launches"], "lib_calls": res["libcalls"],
            "arcs_per_sec_del_trans": n_arc_in / (kms * 1e-3) if kms else None,
            "del_trans": {"n_arc_in": n_arc_in, "inner_iters": inner, "n_vtx": n_vtx, "kernel_ms": kms},
            "phase_ms_last_step": res["phases"], "cleaning_passes": res["cleaning"],
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak if peak else None,
                         "frac_kind": "algorithmic bytes / kernel time / measured copy peak", "traffic": traffic,
                         "dram_gbs": traffic / (kms * 1e-3) / 1e9 if traffic and kms else None,
                         "peak_source": peak_src, "kernel": "k_del_trans_warp", "algorithmic_bytes": alg_bytes, "formula": "16*n_arc + 16*inner_iters + 1*n_arc + 12*n_vtx"},
            "roofline_phases": phases,
            "cpu_baseline": cpu, "cpu_full_size": full, "cli": cli, "noisy": noisy,
            "clocks": clocks, "host_affinity": affinity, "wall_s_timed_region": res["wall_dev"], "wall_ms_per_step": res["wall_dev"] / a.steps * 1e3,
        }
        print(json.dumps(line), flush=True)
        os.dup2(2, 1)
    lib.mab_destroy(ctx)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
