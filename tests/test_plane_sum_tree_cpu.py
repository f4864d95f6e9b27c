"""The shape of NumPy's float32 pairwise-sum tree as the plane-mean kernels derive it on the device (prepost.cuh:
plane_sum_tree, sum_node, leaf_part), run through the host emulation (tests/host_emu) and compared with NumPy's own
split rule (loops_utils.h.src, pairwise_sum): runs of more than 128 elements split at n2 = n/2 - (n/2) % 8, shorter
runs are leaves.  Every leaf must be found with its depth, index within the depth, first element and length.  The
kernels rely on NumPy's leaves sitting on two adjacent depths: leaf_sum_kernel sums each node of level L as a leaf or as
two leaves."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT

EMU_DIR = os.path.join(ROOT, "tests", "host_emu")


@pytest.fixture(scope="module")
def emu():
    so = os.path.join(EMU_DIR, "libpysp_emu.so")
    srcs = [os.path.join(EMU_DIR, "emu.cpp")] + [os.path.join(ROOT, "pysp_b200", "csrc", f)
                                                 for f in os.listdir(os.path.join(ROOT, "pysp_b200", "csrc"))]
    if not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in srcs):
        if not os.path.exists("/usr/bin/g++"):
            pytest.skip("g++ not available")
        subprocess.check_call([os.path.join(EMU_DIR, "build.sh")])
    lib = C.CDLL(so)
    lib.emu_plane_sum_leaves.argtypes = [C.c_longlong, C.POINTER(C.c_int), C.c_void_p, C.c_int]
    return lib


def numpy_leaves(ns):
    """NumPy's recursion for every n of `ns` at once, one depth at a time: rows (n index, depth, index, first, count) of
    the leaves, ordered by n and then from left to right"""
    ns = np.asarray(ns, dtype=np.int64)
    node = np.stack([np.arange(len(ns)), np.zeros_like(ns), np.zeros_like(ns), np.zeros_like(ns), ns], axis=1)
    leaves = []
    while len(node):
        leaf = node[:, 4] <= 128
        leaves.append(node[leaf])
        k, d, i, first, n = node[~leaf].T
        n2 = n // 2
        n2 -= n2 % 8
        node = np.concatenate([np.stack([k, d + 1, 2 * i, first, n2], axis=1),
                               np.stack([k, d + 1, 2 * i + 1, first + n2, n - n2], axis=1)])
    rows = np.concatenate(leaves)
    return rows[np.lexsort((rows[:, 3], rows[:, 0]))]


def emu_leaves(lib, ns):
    """the same rows as leaf_sum_kernel finds them, and L per n"""
    cap = int(max(ns)) // 64 + 2                    # every leaf but a lone root holds at least 64 elements
    buf = np.empty((sum(int(n) // 64 + 2 for n in ns), 4), dtype=np.int64)
    L = np.empty(len(ns), dtype=np.int64)
    ids, at, lv = [], 0, C.c_int()
    for k, n in enumerate(ns):
        got = lib.emu_plane_sum_leaves(int(n), C.byref(lv), buf[at:].ctypes.data, cap)
        assert got > 0, "n = %d: emu_plane_sum_leaves returned %d" % (n, got)
        ids.append(np.full(got, k))
        L[k] = lv.value
        at += got
    return np.concatenate([np.concatenate(ids)[:, None], buf[:at]], axis=1), L


def check(lib, ns):
    got, L = emu_leaves(lib, ns)
    want = numpy_leaves(ns)
    assert got.shape == want.shape, "n in [%d, %d]: %d leaves, NumPy's recursion has %d" % (ns[0], ns[-1], len(got), len(want))
    bad = np.flatnonzero((got != want).any(axis=1))
    assert not len(bad), "n = %d: leaf (depth, index, first, count) %s, NumPy's %s" % (
        ns[got[bad[0], 0]], got[bad[0], 1:].tolist(), want[bad[0], 1:].tolist())
    depth, first_of_n = want[:, 1], np.flatnonzero(np.diff(want[:, 0], prepend=-1))
    assert (np.maximum.reduceat(depth, first_of_n) - np.minimum.reduceat(depth, first_of_n) <= 1).all(), "leaves on three depths"
    assert ((depth == L[want[:, 0]]) | (depth == L[want[:, 0]] + 1)).all(), "leaves off the levels L and L + 1"


def test_every_n_up_to_65536(emu):
    for lo in range(1, 65537, 2048):
        check(emu, np.arange(lo, min(lo + 2048, 65537)))


@pytest.mark.parametrize("n", [6_000_000, 16_785_409, 25_011_525])
def test_large_planes(emu, n):
    """a 24 MP frame's plane (6000 x 4000 / 4), 8194 x 8194 (leaves on two depths) and 8662 x 11550 (above 2^24 sites)"""
    check(emu, np.array([n]))
