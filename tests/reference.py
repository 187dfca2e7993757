"""What the parity tests compare against: the unmodified reference, live or as stored digests.

Where oracle/_ref/ is built (oracle/Makefile compiles the reference when its sources are at hand), the tests run it and
compare with it directly.  Every reference-side result a test compares is also folded, in order, into one sha256 per test;
with MAB_RECORD_REFERENCE=<file> those digests are written to <file> (to be merged into tests/golden/reference_digests.json).

Without oracle/_ref/ the library-level tests drive the oracle port (oracle/ma_oracle.c, our CPU restatement of the
reference) in the reference's place, and the command-line tests have no reference binary to run.  The same results are then
folded into the test's digest -- the port's for library calls, ours where the reference's output would have been -- and the
digest must equal the one recorded from the reference: every comparison with the reference still holds, through its digest.
"""
import ctypes as C
import hashlib
import json
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_SO = os.path.join(ROOT, "oracle", "_ref", "libminiasm_ref.so")
REF_CLI = os.path.join(ROOT, "oracle", "_ref", "miniasm_ref")
DIGESTS = os.path.join(ROOT, "tests", "golden", "reference_digests.json")
LIVE = os.path.exists(REF_SO) and os.path.exists(REF_CLI)


def _canon(v):
    """Bytes of a compared value; arc arrays in canonical order (ties of the reference's unstable sort may permute)."""
    if isinstance(v, np.ndarray):
        if v.dtype.names and "ul" in v.dtype.names:
            from miniasm_b200.pipeline import canon_arcs
            v = canon_arcs(v)
        return v.dtype.str.encode() + np.ascontiguousarray(v).tobytes()
    if isinstance(v, (bytes, bytearray)):
        return bytes(v)
    if isinstance(v, (tuple, list)):
        return b"(" + b",".join(_canon(x) for x in v) + b")"
    return repr(v).encode()


class Pins:
    """The reference-side results of one test, folded in order into a sha256."""

    def __init__(self):
        self.h, self.n, self.used = hashlib.sha256(), 0, False

    def add(self, v):
        self.h.update(_canon(v))
        self.h.update(b"|")
        self.n += 1
        return v

    def hexdigest(self):
        return self.h.hexdigest()[:32]


CURRENT = [Pins()]          # the running test's pins (tests/conftest.py starts a new one per test)


def pin(v):
    return CURRENT[0].add(v)


def hits(h):
    """A hit array as the reference's can be pinned: ma_hit_t::del masked (the reference never writes it, hit.c:87-98) and rows
    sorted (equal keys leave its unstable sort in no fixed order)."""
    h = h.copy()
    h["bl_del"] &= 0x7fffffff
    return np.sort(h, order=list(h.dtype.names))


_INT_TYPES = (C.c_int, C.c_uint, C.c_long, C.c_ulong, C.c_longlong, C.c_ulonglong, C.c_int32, C.c_uint32, C.c_int64, C.c_uint64, C.c_float)


class PinnedLib:
    """A miniasm-ABI library whose compared results (counts returned by entry points, graphs read back, text written) are pinned."""

    def __init__(self, lib):
        self._lib = lib

    def __getattr__(self, name):
        CURRENT[0].used = True
        v = getattr(self._lib, name)
        if name in ("read_graph", "print_to_string"):
            return lambda *a: pin(v(*a))
        if getattr(v, "restype", None) in _INT_TYPES:
            return lambda *a: pin(v(*a))
        return v


def unpinned(lib):
    """The library behind a PinnedLib: for results that follow the order of tied arcs, which the reference's unstable sort and
    the port's stable one settle differently (DESIGN.md "Tie order"), so that no digest of the reference's can stand for them."""
    return getattr(lib, "_lib", lib)


def load():
    """The reference when built, else the oracle port; either way with its compared results pinned."""
    from oracle import loaders
    return PinnedLib(loaders.load_reference() if LIVE else loaders.load_oracle_port())


_runs = {}


def cli(args):
    """(rc, stdout, stderr) of the reference command line, or None when it is not built (then compare with `match`)."""
    if not LIVE:
        return None
    key = tuple((a, os.stat(a).st_mtime_ns, os.stat(a).st_size) if os.path.isfile(a) else a for a in args)   # files get rewritten
    if key not in _runs:
        r = subprocess.run([REF_CLI] + list(args), stdout=subprocess.PIPE, stderr=subprocess.PIPE)
        _runs[key] = (r.returncode, r.stdout, r.stderr)
    return _runs[key]


def match(ours, args, form=lambda r: r):
    """form(ours) must equal form(the reference's (rc, stdout, stderr) for `args`): compared directly where the reference is
    built, through the test's digest where it is not."""
    CURRENT[0].used = True
    want = cli(args)
    got = form(ours)
    if want is None:
        pin(got)
        return got
    assert got == pin(form(want))
    return got


def stored():
    try:
        with open(DIGESTS) as f:
            return json.load(f)
    except FileNotFoundError:
        return {}
