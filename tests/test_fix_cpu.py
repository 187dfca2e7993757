"""CPU tier: the timestamp fixed point that the CUDA cleaning passes run (miniasm_b200/csrc/clean_fix.cuh, compiled for
the host by tests/hostsim/) against the unmodified reference, pass by pass from identical pre-states
(asg.c:238-306 tips / internal / bi-loops, asg.c:312-433 bubbles)."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from miniasm_b200 import capi, synth
from miniasm_b200.pipeline import Pipeline

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SIM_SRC = os.path.join(ROOT, "tests", "hostsim", "fix_host.cpp")
SIM_SO = os.path.join(ROOT, "tests", "hostsim", "libfix_host.so")
HDR = os.path.join(ROOT, "miniasm_b200", "csrc", "clean_fix.cuh")

NOISY = ["bubbles800", "chaos", "chaos_small", "shuffled", "varlen300", "lowcov", "c1_ecoli_like", "jitter30"]
EXTRA = {"bubbly": "-n 60000 -l 9000 -L 11000 -j 800 -c 30 -s 21", "multi": "-n 5000 -s 5 -d 200000 -j 30"}


@pytest.fixture(scope="module")
def sim(built):
    if not os.path.exists(SIM_SO) or os.path.getmtime(SIM_SO) < max(os.path.getmtime(SIM_SRC), os.path.getmtime(HDR)):
        subprocess.run(["g++", "-O2", "-std=c++14", "-Wall", "-shared", "-fPIC", "-o", SIM_SO, SIM_SRC], check=True)
    dll = C.CDLL(SIM_SO)
    for n in ("asg_cut_tip", "asg_cut_internal", "asg_cut_biloop"):
        getattr(dll, n).restype, getattr(dll, n).argtypes = C.c_int, [C.POINTER(capi.AsgT), C.c_int]
    dll.fx_pop_bubble.restype, dll.fx_pop_bubble.argtypes = C.c_uint64, [C.POINTER(capi.AsgT), C.c_int]
    return dll


class Stepper:
    def __init__(self, ref, sim):
        self.ref, self.sim, self.sweeps, self.acted = ref, sim, {}, {}

    def step(self, name, g, *args):
        ref, sim = self.ref, self.sim
        h = ref.clone_graph(g)
        want = getattr(ref, name)(g, *args)
        if name == "asg_pop_bubble":
            if not h.contents.n_seq_symm >> 31:
                ref.asg_symm(h)
            got = sim.fx_pop_bubble(h, *args)
            assert C.c_int.in_dll(sim, "fx_last_nonmono").value == 0
            got = C.c_int(got & 0xffffffff).value      # the reference returns the 64-bit count through an int
        else:
            got = getattr(sim, name)(h, *args)
        if got:
            ref.asg_cleanup(h)
        assert got == want, f"{name}: {got} != {want}"
        # read back unpinned: on jittered sets the arcs a pass leaves marked can follow the order of tied arcs, which the reference's
        # unstable sort and the port's stable one settle differently (DESIGN.md "Tie order"); the counts are pinned
        a, s, i, f1, f2 = capi.Lib.read_graph(h)
        b, t, j, g1, g2 = capi.Lib.read_graph(g)
        assert np.array_equal(a, b) and np.array_equal(s, t) and (f1, f2) == (g1, g2), name
        assert (i is None) == (j is None) and (i is None or np.array_equal(i, j))
        ref.asg_destroy(h)
        k = C.c_int.in_dll(sim, "fx_last_sweeps").value
        self.sweeps[name] = max(self.sweeps.get(name, 0), k)
        self.acted[name] = self.acted.get(name, 0) + (want & 0xffffffff)
        return want


def _all_passes(st, ref, paf):
    r = Pipeline(ref, paf).read().select().sg_gen()
    o, g = r.opt, r.sg
    ref.asg_arc_del_trans(g, o.gap_fuzz)
    st.step("asg_cut_tip", g, o.max_ext)
    st.step("asg_pop_bubble", g, o.bub_dist)
    for i in range(o.n_rounds + 1):
        ratio = float(np.float32(o.min_ovlp_drop_ratio) + (np.float32(o.max_ovlp_drop_ratio) - np.float32(o.min_ovlp_drop_ratio))
                      / np.float32(o.n_rounds) * np.float32(i))
        if ref.asg_arc_del_short(g, ratio):
            st.step("asg_cut_tip", g, o.max_ext)
            st.step("asg_pop_bubble", g, o.bub_dist)
    st.step("asg_cut_internal", g, 1)
    st.step("asg_cut_biloop", g, o.max_ext)
    st.step("asg_cut_tip", g, o.max_ext)
    st.step("asg_pop_bubble", g, o.bub_dist)
    if ref.asg_arc_del_short(g, o.final_ovlp_drop_ratio):
        st.step("asg_cut_tip", g, o.max_ext)
        st.step("asg_pop_bubble", g, o.bub_dist)
    r.free()


@pytest.mark.parametrize("name", NOISY + list(EXTRA))
def test_fixpoint_passes_stepwise(name, ref, sim, paf_dir):
    paf = synth.generate(EXTRA.get(name, name), f"{paf_dir}/fx_{name}.paf")
    st = Stepper(ref, sim)
    _all_passes(st, ref, paf)
    print(name, "max sweeps per pass:", st.sweeps, "actions:", st.acted)
    assert max(st.sweeps.values()) <= 64      # dependency chains are short; one round per bubble would be in the thousands


@pytest.mark.parametrize("ext,dist", [(1, 50000), (2, 5000), (8, 200000), (20, 1000), (100, 50000)])
def test_fixpoint_other_parameters(ext, dist, ref, sim, paf_dir):
    paf = synth.generate("chaos", f"{paf_dir}/fx_chaos.paf")
    r = Pipeline(ref, paf).read().select().sg_gen()
    g = r.sg
    ref.asg_arc_del_trans(g, 1000)
    st = Stepper(ref, sim)
    st.step("asg_cut_tip", g, ext)
    st.step("asg_pop_bubble", g, dist)
    st.step("asg_cut_internal", g, ext)
    st.step("asg_cut_biloop", g, ext)
    r.free()
