"""Host build of the constant-time window-table selection (csrc/dkg_ct_select.cuh) that the direct
and grouped kernels run in constant-time mode: for every table size 2^w - 1 (w = 1..6) and every
digit, including the digit-0 / Montgomery-one markers, the selected value is the wanted entry and
the sequence of addresses read is the same."""
from __future__ import annotations

import ctypes
import os
import random
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "protocols", "distributed_keygen_b200", "csrc")
VW = 4


@pytest.fixture(scope="module")
def lib(tmp_path_factory):
    out = tmp_path_factory.mktemp("ct_select_host") / "libct_select_host.so"
    subprocess.run(
        ["g++", "-O1", "-w", "-shared", "-fPIC", "-I", CSRC, "-o", str(out),
         os.path.join(ROOT, "tests", "host", "ct_select_host.cpp")],
        check=True,
    )
    lib = ctypes.CDLL(str(out))
    vp = ctypes.c_void_p
    lib.host_ct_select.argtypes = [vp, vp, ctypes.c_int, ctypes.c_int, ctypes.c_uint32, vp, vp, ctypes.c_int]
    lib.host_ct_select.restype = ctypes.c_int
    return lib


@pytest.mark.parametrize("w", [1, 2, 3, 4, 5, 6])
@pytest.mark.parametrize("nvec", [1, 3])
def test_ct_select_value_and_address_trace(lib, w, nvec):
    n = (1 << w) - 1
    rng = np.random.default_rng(100 * w + nvec)
    table = rng.integers(0, 1 << 32, size=(n, nvec * VW), dtype=np.uint64).astype(np.uint32)
    one = rng.integers(0, 1 << 32, size=nvec * VW, dtype=np.uint64).astype(np.uint32)
    cap = (n + 1) * nvec * VW
    traces = {}
    # table indices, the direct kernel's digit-0 marker 0xfe and the grouped kernels' digit - 1
    # for digit 0 (wrapped around)
    for idx in [*range(n), 0xFE, 0xFFFFFFFF]:
        out = np.zeros(nvec * VW, dtype=np.uint32)
        trace = (ctypes.c_void_p * cap)()
        length = lib.host_ct_select(table.ctypes.data, one.ctypes.data, n, nvec, idx, out.ctypes.data, trace, cap)
        assert length == cap, (w, idx, length)
        want = table[idx] if idx < n else one
        assert np.array_equal(out, want), (w, nvec, idx)
        # addresses as offsets into the two arrays read: the same sequence for every digit
        base_t, base_o = table.ctypes.data, one.ctypes.data
        traces[idx] = tuple(("one", a - base_o) if base_o <= a < base_o + one.nbytes else ("tab", a - base_t)
                            for a in trace)
    first = next(iter(traces.values()))
    assert all(t == first for t in traces.values()), (w, nvec)
    # every word of every entry and of the one is read exactly once
    assert sorted(first) == sorted([("one", 4 * i) for i in range(nvec * VW)] + [("tab", 4 * i) for i in range(n * nvec * VW)])


def test_ct_select_random_digits_match_direct_indexing(lib):
    """Digits drawn as the kernels see them (a digit d of a w-bit window, index d - 1) for random tables."""
    rng = random.Random(5)
    for w in range(1, 7):
        n = (1 << w) - 1
        table = np.array([[rng.getrandbits(32) for _ in range(2 * VW)] for _ in range(n)], dtype=np.uint32)
        one = np.array([rng.getrandbits(32) for _ in range(2 * VW)], dtype=np.uint32)
        for _ in range(20):
            d = rng.randrange(1 << w)
            out = np.zeros(2 * VW, dtype=np.uint32)
            trace = (ctypes.c_void_p * ((n + 1) * 2 * VW))()
            lib.host_ct_select(table.ctypes.data, one.ctypes.data, n, 2, (d - 1) & 0xFFFFFFFF, out.ctypes.data,
                               trace, (n + 1) * 2 * VW)
            assert np.array_equal(out, table[d - 1] if d else one), (w, d)
