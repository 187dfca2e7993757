"""Runtime switches of the CUDA library (DESIGN.md "Runtime switches"): every alternative code path must give the
reference's GFA.  The switches are read once per process, so each case runs the command-line tool in a fresh
process with the variable set and compares its output with the unmodified reference binary's.

Sets: tips/bubbles/multi-arcs/hot spots/deep groups, i.e. every kernel variant (warp / CTA / device-wide) is reached."""
import os
import subprocess

import pytest

from miniasm_b200 import synth
from tests import reference
from tests.gfa_compare import assert_same_gfa

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLI = os.path.join(ROOT, "miniasm_b200", "miniasm-b200")

SETS = {
    "chaos": "chaos",
    "bubbles800": "bubbles800",
    "shuffled": "shuffled",
    "deep": "-n 1500 -l 3000 -L 12000 -c 400 -j 30 -s 77",      # several hundred hits per read: the CTA-per-read kernels
    "multi": "-n 5000 -s 5 -d 200000 -j 30",                          # 20 % duplicated overlaps -> multi-arcs (shared marks in the transitive reduction)
    "skew": "skew_small",                                             # hot spots: slabs beyond the warp kernels' limits
    "bubbly": "-n 60000 -l 9000 -L 11000 -j 800 -c 30 -s 21",     # thousands of bubbles/tips along sorted ids
}
# "multi": jitter 30 on 10 kb reads makes equal-length arcs out of one unitig end common; the order of the L lines of such
# ties is the order the reference's unstable in-place radix sort happens to leave (DESIGN.md "Tie order")
TIES = {"multi"}
SWITCHES = [{}, {"MAB_CUB_SELECT": "1"}, {"MAB_SUB_SMEM_SORT": "1"}, {"MAB_GPU_GFA": "0", "MAB_WRITER_THREADS": "3"}, {"MAB_GPU_GFA": "0"},
            {"MAB_SG_SEGSORT": "0"}, {"MAB_CUB_SELECT": "1", "MAB_SUB_SMEM_SORT": "1", "MAB_GPU_GFA": "0", "MAB_SG_SEGSORT": "0"}]


@pytest.fixture(scope="module")
def pafs(built, paf_dir):
    return {k: synth.generate(v, f"{paf_dir}/sw_{k}.paf") for k, v in SETS.items()}


@pytest.mark.parametrize("name", list(SETS))
@pytest.mark.parametrize("env", SWITCHES, ids=lambda e: "+".join(f"{k}={v}" for k, v in e.items()) or "default")
def test_switch(env, name, pafs):
    r = subprocess.run([CLI, pafs[name]], stdout=subprocess.PIPE, stderr=subprocess.PIPE, env={**os.environ, **env})
    assert r.returncode == 0, r.stderr.decode()[-2000:]
    want = reference.cli([pafs[name]])
    if want is not None:
        assert want[0] == 0
        assert_same_gfa(r.stdout, want[1], tie_order_free=name in TIES)
    # the digest carries the comparison where the reference is not built; for tied sets only as the sorted line multiset
    reference.match((r.returncode, r.stdout, r.stderr), [pafs[name]],
                    lambda x: (x[0], sorted(x[1].split(b"\n")) if name in TIES else x[1]))
