"""Sharded ragged batches in the host (g++) build of the kernel sources: the multi-destination (NDST = 2) forms of the
ragged pair and default-mode kernels, with one constants bag and with per-satellite constants, run as two shards of a
mixed constellation (shard_ranges_by_work), each storing into both gathered buffers at its global columns
s (K_cap - 1) + k.  Both buffers must come out bit for bit as the single-destination ragged launch of the whole batch on
the live columns; padding columns stay NaN, and after the first shard so do the second shard's columns.  A second build
under AddressSanitizer + UBSan runs the same launches with exactly sized buffers."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

import hostk
import test_ragged_kernel_source_on_host as R
import test_units_kernel_source_on_host as U
from conftest import ROOT
from mpconstellation_b200.distributed import shard_ranges_by_work

HERE = os.path.join(ROOT, "tests", "hostk")
D = ctypes.c_double
K_SAT = np.array([7, 2, 12, 5, 12, 3], np.int32)
K_CAP = 14                      # a capacity above the largest count, as RaggedGather keeps it


def _build(sanitize=False):
    """libmpc_hostk_shard[_asan].so: tests/hostk/shard_main.cpp over the sources hostk.build() prepared"""
    hostk.build(sanitize=sanitize)
    so = os.path.join(hostk.BUILD, "libmpc_hostk_shard_asan.so" if sanitize else "libmpc_hostk_shard.so")
    src = os.path.join(HERE, "shard_main.cpp")
    deps = [src, os.path.join(HERE, "hostk_main.cpp"), os.path.join(hostk.BUILD, "libmpc_hostk_asan.so" if sanitize else "libmpc_hostk.so")]
    if not (os.path.exists(so) and all(os.path.getmtime(so) >= os.path.getmtime(d) for d in deps)):
        opt = (["-O1", "-g", "-fsanitize=address,undefined", "-fno-sanitize-recover=undefined", "-fno-omit-frame-pointer"]
               if sanitize else ["-O2"])
        tmp = f"{so}.{os.getpid()}.tmp"
        cmd = ["g++"] + opt + ["-std=c++17", "-pthread", "-shared", "-fPIC", "-mfma", "-ffp-contract=fast", "-fno-math-errno",
                               "-w", "-I", os.path.join(HERE, "include"), "-I", hostk.BUILD, "-o", tmp, src]
        res = subprocess.run(cmd, capture_output=True, text=True)
        assert res.returncode == 0, res.stdout + res.stderr
        os.replace(tmp, so)
    return so


def _lib(sanitize=False):
    return ctypes.CDLL(_build(sanitize))


def batch(K_sat=K_SAT, K_cap=K_CAP):
    """the mixed constellation of the units tests on its own grids, padded to K_cap (NaN)"""
    y0, consts = U.mixed_constellation(len(K_sat))
    x, u = U._trajectories(y0, consts, K_sat)
    N, _, Kmax = x.shape
    xp, up = np.full((N, 7, K_cap), np.nan), np.full((N, 3, K_cap), np.nan)
    xp[:, :, :Kmax], up[:, :, :Kmax] = x, u
    return xp, up, consts


def shard(L, x, u, tf, consts, K_sat, s0, s1, psc, adaptive, out0, out1, include_J2=False, n_sub=100, skip_const=0):
    """satellites [s0, s1) of the batch through one NDST = 2 launch into out0, out1 [105, N (K_cap - 1)]"""
    K_cap = x.shape[2]
    xs, us = np.ascontiguousarray(x[s0:s1]), np.ascontiguousarray(u[s0:s1])
    n = s1 - s0
    first = np.concatenate([[0], np.cumsum(K_sat[s0:s1].astype(np.int64) - 1)]).astype(np.int64)
    c8 = U._c8(consts[s0:s1] if psc else consts[:1])
    status = np.full(n * (K_cap - 1), -1, np.int32)
    nodes = np.full(n * (K_cap - 1), -1, np.int32)
    L.hostk_discretize_shard(hostk._p(xs), hostk._p(us), hostk._p(np.full(n, float(tf))), hostk._p(c8), int(psc),
                             int(include_J2), n, K_cap, hostk._p(first), int(adaptive), int(n_sub), D(1e-3), D(1e-6), D(1e-2),
                             hostk._p(out0), hostk._p(out1), ctypes.c_longlong(out0.shape[1]),
                             ctypes.c_longlong(s0 * (K_cap - 1)), int(skip_const), hostk._p(status), hostk._p(nodes), 1)
    return status.reshape(n, K_cap - 1), nodes.reshape(n, K_cap - 1)


def live(K_sat, K_cap, sats):
    """global columns of the live intervals of satellites `sats`"""
    return np.concatenate([s * (K_cap - 1) + np.arange(K_sat[s] - 1) for s in sats] or [np.zeros(0, int)])


@pytest.mark.parametrize("psc", [False, True])
@pytest.mark.parametrize("adaptive", [False, True])
@pytest.mark.parametrize("j2", [False, True])
def test_two_shards_store_bit_identical_results_into_both_buffers(psc, adaptive, j2):
    L = _lib()
    x, u, consts = batch()
    N = len(K_SAT)
    if psc:
        ref, rst, rnodes = U.discretize_units(U._lib(), x, u, 0.3, consts, K_SAT, adaptive, include_J2=j2)
    else:
        ref, rst, rnodes = R.discretize_ragged(R._lib(), x, u, 0.3, consts[0], K_SAT, adaptive, include_J2=j2)
    ranges = shard_ranges_by_work(K_SAT, 2)
    assert all(b > a for a, b in ranges)
    bufs = [np.full((105, N * (K_CAP - 1)), np.nan) for _ in range(2)]
    all_cols = np.arange(N * (K_CAP - 1))
    for r, (s0, s1) in enumerate(ranges):
        st, nodes = shard(L, x, u, 0.3, consts, K_SAT, s0, s1, psc, adaptive, bufs[r], bufs[1 - r], include_J2=j2)
        mine = live(K_SAT, K_CAP, range(s0, s1))
        loc = mine - s0 * (K_CAP - 1)
        assert np.array_equal(st.reshape(-1)[loc], rst.reshape(-1)[mine])
        if adaptive:
            assert np.array_equal(nodes.reshape(-1)[loc], rnodes.reshape(-1)[mine])
        pad = np.setdiff1d(np.arange(st.size), loc)
        assert (st.reshape(-1)[pad] == -1).all()
        if r == 0:      # the other shard's columns and all padding: untouched in both buffers
            rest = np.setdiff1d(all_cols, mine)
            assert all(np.isnan(b[:, rest]).all() for b in bufs)
    cols = live(K_SAT, K_CAP, range(N))
    pad = np.setdiff1d(all_cols, cols)
    for b in bufs:
        assert np.array_equal(b[:, cols], ref[:, cols])
        assert np.isnan(b[:, pad]).all()


def test_skip_const_leaves_the_constant_rows_to_the_fill():
    """skip_const 1: rows 42..48 (0 .. 0 1) go to the own buffer only, 2: to neither; every other row to both"""
    L = _lib()
    x, u, consts = batch()
    N = len(K_SAT)
    s0, s1 = shard_ranges_by_work(K_SAT, 2)[1]
    cols = live(K_SAT, K_CAP, range(s0, s1))
    rows = np.r_[0:42, 49:105]
    for skip in (1, 2):
        b0, b1 = (np.full((105, N * (K_CAP - 1)), np.nan) for _ in range(2))
        shard(L, x, u, 0.3, consts, K_SAT, s0, s1, True, True, b0, b1, skip_const=skip)
        assert np.array_equal(b0[rows][:, cols], b1[rows][:, cols]) and np.isfinite(b0[rows][:, cols]).all()
        assert np.isnan(b1[42:49][:, cols]).all()
        if skip == 1:
            assert (b0[42:48][:, cols] == 0).all() and (b0[48][cols] == 1).all()
        else:
            assert np.isnan(b0[42:49][:, cols]).all()


def test_shard_kernels_under_address_sanitizer():
    asan = subprocess.run(["gcc", "-print-file-name=libasan.so"], capture_output=True, text=True).stdout.strip()
    if not os.path.isabs(asan) or not os.path.exists(asan):
        pytest.skip("no AddressSanitizer runtime next to this gcc")
    _build(sanitize=True)
    code = (
        "import sys, numpy as np\n"
        f"sys.path.insert(0, {os.path.join(ROOT, 'tests')!r}); sys.path.insert(0, {ROOT!r})\n"
        "import test_shard_kernel_source_on_host as T\n"
        "from mpconstellation_b200.distributed import shard_ranges_by_work\n"
        "L = T._lib(sanitize=True)\n"
        "for K_sat, K_cap, world in (([2], 2, 2), ([9, 2, 9], 9, 2), ([2, 5, 3, 9], 11, 3)):\n"
        "    K_sat = np.array(K_sat, np.int32)\n"
        "    x, u, consts = T.batch(K_sat, K_cap)\n"
        "    N = len(K_sat)\n"
        "    for psc in (0, 1):\n"
        "        for ad in (0, 1):\n"
        "            for j2 in (0, 1):\n"
        "                b0, b1 = np.full((105, N * (K_cap - 1)), np.nan), np.full((105, N * (K_cap - 1)), np.nan)\n"
        "                for s0, s1 in shard_ranges_by_work(K_sat, world):\n"
        "                    if s1 > s0:\n"
        "                        T.shard(L, x, u, 0.3, consts, K_sat, s0, s1, psc, ad, b0, b1, include_J2=j2,\n"
        "                                n_sub=100 if ad else 6, skip_const=psc)\n"
        "print('shard launches clean')\n")
    env = dict(os.environ, HOSTK_SANITIZE="1", LD_PRELOAD=asan, ASAN_OPTIONS="detect_leaks=0:halt_on_error=1")
    res = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, timeout=900)
    assert res.returncode == 0 and "shard launches clean" in res.stdout, res.stdout[-2000:] + res.stderr[-4000:]
    assert "AddressSanitizer" not in res.stderr and "runtime error" not in res.stderr
