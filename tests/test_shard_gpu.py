"""Multi-GPU parity (SURVEY.md 8e): the hash-sharded pipeline on 2 (or more) GPUs must print the GFA the reference
prints for the whole PAF -- byte for byte.  Needs >= 2 visible GPUs (gpurun --gpus 2); skipped otherwise."""
import os
import subprocess
import sys

import pytest

from miniasm_b200 import synth
from tests import reference

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.path.join(ROOT, "oracle", "_ref", "miniasm_ref")


def n_gpus():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


WORLDS = [w for w in (2, 3, 4, 8) if w <= n_gpus()]


@pytest.mark.skipif(n_gpus() < 2, reason="needs at least 2 GPUs")
@pytest.mark.parametrize("name", ["chaos_small", "chaos", "bubbles800", "tiny_exact", "shuffled", "lowcov"])
@pytest.mark.parametrize("world", WORLDS or [2])
def test_sharded_gfa_equals_reference(name, world, built, paf_dir):
    paf = synth.generate(name, f"{paf_dir}/sh_{name}.paf")
    out = f"{paf_dir}/sh_{name}_{world}.gfa"
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr", "127.0.0.1",
           "--master-port", "29533", os.path.join(ROOT, "tests", "shard_worker.py"), paf, out]
    # half of the sets load and ingest in two calls, the other half overlapped (MAB_SHARD_STREAM, tests/shard_worker.py)
    env = {**os.environ, "MAB_SHARD_STREAM": "0" if name in ("chaos_small", "bubbles800", "shuffled") else "1"}
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600, env=env)
    assert r.returncode == 0, r.stdout[-3000:]
    want = subprocess.run([REF, paf], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL).stdout
    assert open(out, "rb").read() == want


FULL = [("c3_1m", 2), ("c3_1m", 8), ("c4_4m", 2), ("c4_4m", 4), ("c5_8m_skew", 8)]


@pytest.mark.skipif(n_gpus() < 2 or os.environ.get("MAB_TEST_FULL") != "1", reason="needs >= 2 GPUs and MAB_TEST_FULL=1 (minutes)")
@pytest.mark.parametrize("name,world", [c for c in FULL if c[1] <= max(n_gpus(), 2)])
def test_sharded_full_config_digest(name, world, built, paf_dir):
    """BASELINE configs 3 / 4 / 5 (1 M / 4 M / 8 M reads, the last one skewed) as ONE PAF cut into `world` parts, hash-sharded
    over `world` GPUs: the GFA must have the sha256 of the reference's GFA for the same PAF (tests/golden/configs.json)."""
    import hashlib
    import json
    gold = json.load(open(os.path.join(ROOT, "tests", "golden", "configs.json")))
    if name not in gold:
        pytest.skip(f"no golden digest for {name}")
    out = f"{paf_dir}/shfull_{name}_{world}.gfa"
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr", "127.0.0.1",
           "--master-port", "29534", os.path.join(ROOT, "tests", "shard_worker.py"), f"gen:{name}", out]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=1800)
    assert r.returncode == 0, r.stdout[-3000:]
    h = hashlib.sha256()
    with open(out, "rb") as f:
        for blk in iter(lambda: f.read(1 << 24), b""):
            h.update(blk)
    size = os.path.getsize(out)
    os.unlink(out)
    assert size == gold[name]["gfa_bytes"] and h.hexdigest() == gold[name]["gfa_sha256"]


CLI = os.path.join(ROOT, "miniasm_b200", "miniasm-b200")


@pytest.mark.skipif(n_gpus() < 2, reason="needs at least 2 GPUs")
@pytest.mark.parametrize("name", ["chaos_small", "chaos", "bubbles800", "tiny_exact"])
@pytest.mark.parametrize("world", WORLDS or [2])
@pytest.mark.parametrize("extra", [[], ["-p", "sg"]], ids=["ug", "sg"])
def test_cli_multi_gpu(name, world, extra, built, paf_dir):
    """The drop-in command line with MINIASM_B200_GPUS=N (threads of one process, NCCL + peer access inside the library):
    same bytes on stdout as the reference, same counts on stderr."""
    import re
    paf = synth.generate(name, f"{paf_dir}/sh_{name}.paf")
    want = subprocess.run([REF] + extra + [paf], stdout=subprocess.PIPE, stderr=subprocess.PIPE)
    for p2p in ("1", "0"):
        got = subprocess.run([CLI] + extra + [paf], stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=600,
                             env={**os.environ, "MINIASM_B200_GPUS": str(world), "MAB_SHARD_P2P": p2p})
        assert got.returncode == 0, got.stderr.decode()[-3000:]
        if extra:   # raw-graph dumps: arcs of equal (vertex, length) print in the order the reference's unstable sort left them
            assert sorted(got.stdout.splitlines()) == sorted(want.stdout.splitlines())
        else:
            assert got.stdout == want.stdout
        cnt = lambda err: [re.sub(r"::\d+\.\d+\*\d+\.\d+\]", "]", x) for x in err.decode().splitlines()
                           if x.startswith("[M::") and "::main]" not in x and any(k in x for k in ("ma_hit_read", "ma_hit_contained", "ma_sg_gen", "asg_")) and "===>" not in x]
        assert cnt(got.stderr) == cnt(want.stderr)


@pytest.mark.parametrize("name,stream", [("chaos", "1"), ("bubbles800", "0"), ("lowcov", "0"), ("c2_100k", "1")])
def test_sharded_pipeline_world1(name, stream, built, paf_dir):
    """The sharded code path with ONE rank on one GPU: every kernel of it runs (count / scan / staged emit into the receive buffer, the
    global name table, the replicated tail), only the collectives degenerate -- keeps the multi-GPU path under test on 1-GPU boxes."""
    paf = synth.generate(name, f"{paf_dir}/sh1_{name}.paf")
    out = f"{paf_dir}/sh1_{name}_{stream}.gfa"
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=1", "--master-addr", "127.0.0.1",
           "--master-port", "29535", os.path.join(ROOT, "tests", "shard_worker.py"), paf, out]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600, env={**os.environ, "MAB_SHARD_STREAM": stream})
    assert r.returncode == 0, r.stdout[-3000:]
    reference.match((0, open(out, "rb").read(), b""), [paf], lambda x: x[1])
