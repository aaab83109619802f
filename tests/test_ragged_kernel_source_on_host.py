"""Ragged batches in the host (g++) build of the kernel sources: satellite s on its own K_s nodes through ONE launch of
the pair (fixed-step) and default-mode kernels, and per-lane sample counts / table lengths in the RK45 propagator.  Every
satellite must come out bit for bit as the rectangular host launch of that satellite at K_s, and the padding columns
must stay untouched (NaN, status -1).  A second build under AddressSanitizer + UBSan memchecks the indexing on ragged
shapes with K_s = 2 and K_s = Kmax, exactly sized buffers."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

import hostk
from conftest import GOLDEN, ROOT, synth_batch

HERE = os.path.join(ROOT, "tests", "hostk")


def _lib(sanitize=False):
    """libmpc_hostk_ragged[_asan].so, loaded (the _asan build only in a process that runs under the ASan runtime)"""
    return ctypes.CDLL(_build(sanitize))


def _build(sanitize=False):
    """libmpc_hostk_ragged[_asan].so: tests/hostk/ragged_main.cpp over the sources hostk.build() prepared"""
    hostk.build(sanitize=sanitize)
    so = os.path.join(hostk.BUILD, "libmpc_hostk_ragged_asan.so" if sanitize else "libmpc_hostk_ragged.so")
    src = os.path.join(HERE, "ragged_main.cpp")
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


def discretize_ragged(L, x, u, tf, const, K_sat, adaptive, include_J2=False, n_sub=100, em=1):
    """one ragged launch over x [N,7,Kmax], u [N,3,Kmax] -> SoA [105, N (Kmax-1)] (NaN padding), status, n_nodes; em as
    DstTab::em (1: what hostk.discretize sets)"""
    x = np.ascontiguousarray(x, dtype=np.float64)
    u = np.ascontiguousarray(u, dtype=np.float64)
    N, _, Kmax = x.shape
    tfv = np.ascontiguousarray(np.broadcast_to(np.asarray(tf, dtype=np.float64), (N,)))
    first = np.concatenate([[0], np.cumsum(np.asarray(K_sat, dtype=np.int64) - 1)]).astype(np.int64)
    pitch = N * (Kmax - 1)
    out = np.full((105, pitch), np.nan)
    status = np.full(pitch, -1, dtype=np.int32)
    nodes = np.full(pitch, -1, dtype=np.int32)
    D = ctypes.c_double
    L.hostk_discretize_ragged(hostk._p(x), hostk._p(u), hostk._p(tfv), hostk._p(hostk._const8(const)), int(include_J2), N, Kmax,
                              hostk._p(first), int(adaptive), int(n_sub), D(1e-3), D(1e-6), D(1e-2), hostk._p(out),
                              ctypes.c_longlong(pitch), hostk._p(status), hostk._p(nodes), int(em))
    return out, status.reshape(N, Kmax - 1), nodes.reshape(N, Kmax - 1)


def _batch(const, K_sat, tf=0.3, seed=20240531):
    """x, u [N,.,Kmax]: satellite s sampled on its own K_s nodes (oracle propagation), padding poisoned with NaN"""
    N, Kmax = len(K_sat), int(max(K_sat))
    y0, _, _ = synth_batch(N, 2, tf, const, seed=seed)
    x = np.full((N, 7, Kmax), np.nan)
    u = np.full((N, 3, Kmax), np.nan)
    for s, k in enumerate(K_sat):
        _, xs, us = synth_batch(N, int(k), tf, const, seed=seed)
        x[s, :, :k], u[s, :, :k] = xs[s], us[s]
    return y0, x, u


@pytest.mark.parametrize("adaptive", [False, True])
@pytest.mark.parametrize("j2", [False, True])
def test_ragged_launch_is_bit_identical_to_per_satellite_rectangular_launches(const, adaptive, j2):
    K_sat = np.array([7, 2, 12, 5, 12, 3], np.int32)
    Kmax = int(K_sat.max())
    _, x, u = _batch(const, K_sat)
    out, st, nodes = discretize_ragged(_lib(), x, u, 0.3, const, K_sat, adaptive, include_J2=j2)
    for s, k in enumerate(K_sat):
        n = k - 1
        cols = slice(s * (Kmax - 1), s * (Kmax - 1) + n)
        xs, us = x[s:s + 1, :, :k], u[s:s + 1, :, :k]
        if adaptive:
            ref, rst, rnodes = hostk.discretize_adaptive(xs, us, 0.3, const, include_J2=j2)
            assert np.array_equal(nodes[s, :n], rnodes)
        else:
            ref, rst = hostk.discretize(xs, us, 0.3, const, include_J2=j2)
        assert np.array_equal(out[:, cols], ref) and np.array_equal(st[s, :n], rst)
        assert np.isnan(out[:, s * (Kmax - 1) + n:(s + 1) * (Kmax - 1)]).all() and (st[s, n:] == -1).all()


def test_ragged_rk45_lanes_match_rectangular_runs(const):
    L = _lib()
    y0, _, _ = synth_batch(5, 2, 1.0, const)
    N, T_max, Ku = 5, 40, 12
    T_sat = np.array([40, 2, 17, 33, 9], np.int32)
    ku = np.array([12, 2, 7, 12, 4], np.int32)
    tab = 0.2 * np.random.default_rng(3).standard_normal((N, 3, Ku))
    for kind in (2, 3):
        y = np.full((N, 7, T_max), np.nan)
        uo = np.full((N, 3, T_max), np.nan)
        st = np.full(N, -1, np.int32)
        steps = np.zeros(N, np.int32)
        L.hostk_propagate_rk45_ragged(hostk._p(y0), hostk._p(np.full(N, 1.0)), hostk._p(hostk._const8(const)), kind,
                                      ctypes.c_double(0.5), hostk._p(tab), Ku, hostk._p(ku), N, T_max, hostk._p(T_sat),
                                      hostk._p(y), hostk._p(uo), hostk._p(st), hostk._p(steps))
        for s in range(N):
            t = int(T_sat[s])
            table = np.ascontiguousarray(tab[s:s + 1, :, :ku[s]]) if kind == 3 else None
            yr, ur, sr, nr, _ = hostk.propagate_rk45(y0[s:s + 1], 1.0, const, kind=kind, thrust=(0.5, 0, 0), table=table, T=t)
            assert np.array_equal(y[s, :, :t], yr[0]) and np.array_equal(uo[s, :, :t], ur[0])
            assert st[s] == sr[0] == 0 and steps[s] == nr[0]
            assert np.isnan(y[s, :, t:]).all() and np.isnan(uo[s, :, t:]).all()


def test_ragged_kernels_under_address_sanitizer(const):
    asan = subprocess.run(["gcc", "-print-file-name=libasan.so"], capture_output=True, text=True).stdout.strip()
    if not os.path.isabs(asan) or not os.path.exists(asan):
        pytest.skip("no AddressSanitizer runtime next to this gcc")
    _build(sanitize=True)
    code = (
        "import sys, ctypes, numpy as np\n"
        f"sys.path.insert(0, {os.path.join(ROOT, 'tests')!r}); sys.path.insert(0, {ROOT!r})\n"
        "import test_ragged_kernel_source_on_host as T\n"
        "from oracle.mpc_oracle import OracleConstants\n"
        f"const = OracleConstants(*np.load({os.path.join(GOLDEN, 'discretize.npz')!r})['const'])\n"
        "L = T._lib(sanitize=True)\n"
        "for K_sat in ([2, 9, 3], [9], [2, 2], [4, 9, 2, 9, 6]):\n"
        "    K_sat = np.array(K_sat, np.int32)\n"
        "    _, x, u = T._batch(const, K_sat)\n"
        "    for ad in (0, 1):\n"
        "        for j2 in (0, 1):\n"
        "            T.discretize_ragged(L, x, u, 0.3, const, K_sat, ad, include_J2=j2, n_sub=100 if ad else 6)\n"
        "print('ragged launches clean')\n")
    env = dict(os.environ, HOSTK_SANITIZE="1", LD_PRELOAD=asan, ASAN_OPTIONS="detect_leaks=0:halt_on_error=1")
    res = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, timeout=900)
    assert res.returncode == 0 and "ragged launches clean" in res.stdout, res.stdout[-2000:] + res.stderr[-4000:]
    assert "AddressSanitizer" not in res.stderr and "runtime error" not in res.stderr
