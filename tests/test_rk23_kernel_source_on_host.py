"""The default quadrature mode with scipy's RK23 (discretize_rk23_kernel) in the host (g++) build of the kernel sources:
against the reference's own call, interval_matrices(ivp_solver="RK23") -- the same accepted steps (n_nodes ==
len(sol.t) for every interval) and the matrices to 1e-10 norm-relative -- on the Hubble family, eccentric, polar and
retrograde orbits, a coast-to-thrust switch with exactly-zero inputs, J2 on and off, a short horizon on which max_step
binds and a loose max_step on which scipy rejects steps; the controller's x^(-1/3) against pow; ragged and
per-satellite-constants launches bit-identical to single-satellite ones; status words; an ASan + UBSan run."""
import ctypes
import dataclasses
import os
import shutil
import subprocess
import sys

import numpy as np
import pytest

import hostk
import orbit_sweep as O
from conftest import NAMES, ROOT, rel_err, synth_batch
from oracle import mpc_oracle as M

HERE = os.path.join(ROOT, "tests", "hostk")
D = ctypes.c_double
TOL = 1e-10


def _build(sanitize=False):
    """libmpc_hostk_rk23[_asan].so: tests/hostk/rk23_main.cpp over the sources hostk.build() prepared, plus
    discretize_rk23_kernel.cuh copied next to them"""
    hostk.build(sanitize=sanitize)
    hdr = os.path.join(hostk.CSRC, "discretize_rk23_kernel.cuh")
    text = open(hdr).read()
    assert "asm(" not in text, "inline PTX the host build does not know"
    dst = os.path.join(hostk.BUILD, "discretize_rk23_kernel.cuh")
    if not os.path.exists(dst) or open(dst).read() != text:
        tmp = f"{dst}.{os.getpid()}.tmp"
        shutil.copyfile(hdr, tmp)
        os.replace(tmp, dst)
    so = os.path.join(hostk.BUILD, "libmpc_hostk_rk23_asan.so" if sanitize else "libmpc_hostk_rk23.so")
    src = os.path.join(HERE, "rk23_main.cpp")
    deps = [src, dst, os.path.join(HERE, "hostk_main.cpp"),
            os.path.join(hostk.BUILD, "libmpc_hostk_asan.so" if sanitize else "libmpc_hostk.so")]
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


_LIBS = {}


def _lib(sanitize=False):
    if sanitize not in _LIBS:
        _LIBS[sanitize] = ctypes.CDLL(_build(sanitize))
    return _LIBS[sanitize]


def run(x, u, tf, const, j2=False, K_sat=None, rtol=1e-3, atol=1e-6, max_step=1e-2, L=None):
    """the host kernel: const one Constants bag or a list of N (per-satellite constants); K_sat None (rectangular) or
    int [N] (ragged, x / u padded) -> SoA [105, N (K-1)], status [N (K-1)], n_nodes [N (K-1)]"""
    L = L or _lib()
    x = np.ascontiguousarray(x, dtype=np.float64)
    u = np.ascontiguousarray(u, dtype=np.float64)
    N, _, K = x.shape
    tfv = np.ascontiguousarray(np.broadcast_to(np.asarray(tf, dtype=np.float64), (N,)))
    psc = isinstance(const, (list, tuple))
    c8 = np.ascontiguousarray(np.concatenate([hostk._const8(c) for c in const]) if psc else hostk._const8(const))
    first = None
    if K_sat is not None:
        first = np.zeros(N + 1, dtype=np.int64)
        first[1:] = np.cumsum(np.asarray(K_sat) - 1)
    n_int = N * (K - 1)
    out = np.full((105, n_int), np.nan)
    st = np.full(n_int, -1, dtype=np.int32)
    nodes = np.zeros(n_int, dtype=np.int32)
    p = hostk._p
    L.hostk_discretize_rk23(p(x), p(u), p(tfv), p(c8), int(psc), int(j2), N, K, p(first), D(rtol), D(atol), D(max_step),
                            p(out), ctypes.c_longlong(n_int), p(st), p(nodes))
    return out, st, nodes


def reference(k, x, u, tf, const, j2, max_step=1e-2):
    """the reference's RK23 call for interval k -> (matrices, scipy's solution object)"""
    rec = []
    orig = M.integrate.solve_ivp

    def spy(*a, **kw):
        rec.append(orig(*a, **kw))
        return rec[-1]
    M.integrate.solve_ivp = spy
    try:
        mats = M.interval_matrices(k, x, u, tf, const, include_J2=j2, ivp_solver="RK23", ivp_max_step=max_step)
    finally:
        M.integrate.solve_ivp = orig
    assert rec[0].status == 0
    return mats, rec[0]


def check(x, u, tf, const, j2, pairs, max_step=1e-2):
    """host kernel against the reference on the (s, k) pairs -> list of (n_nodes, nfev) of scipy's solutions"""
    out, st, nodes = run(x, u, tf, const, j2=j2, max_step=max_step)
    assert st.max() == 0 and st.min() == 0
    N, _, K = x.shape
    got = hostk.stacked(out, N, K)
    tfv = np.broadcast_to(np.asarray(tf, dtype=np.float64), (N,))
    seen = []
    for s, k in pairs:
        ref, sol = reference(k, x[s], u[s], float(tfv[s]), const, j2, max_step)
        assert nodes[s * (K - 1) + k] == len(sol.t), (s, k)
        for i, n in enumerate(NAMES):
            g = got[i][s, k] if i < 3 else got[i][s, :, k]
            assert rel_err(g, ref[i]) <= TOL, (s, k, n, rel_err(g, ref[i]))
        seen.append((len(sol.t), sol.nfev))
    return seen


def _rejects(n, nfev):
    # a run without rejections costs 2 evaluations (f0, select_initial_step) plus 3 per accepted step
    return nfev > 2 + 3 * (n - 1)


@pytest.mark.parametrize("j2", [False, True])
def test_hubble_tangential(const, j2):
    """the Hubble family (conftest.synth_batch), tangential thrust 0.5, K = 200, tf = 2: one or two steps per interval"""
    _, x, u = synth_batch(2, 200, 2.0, const)
    check(x, u, 2.0, const, j2, [(s, k) for s in range(2) for k in (0, 1, 50, 123, 197, 198)])


@pytest.mark.parametrize("j2", [False, True])
def test_eccentric_polar_retrograde_orbits(const, j2):
    """orbit_sweep's elements: e = 0.6 / 0.8, inclinations 0, 90 and 160 degrees, starting at and after perigee"""
    el = O.sweep_elements()
    pick = np.flatnonzero((el["e"] >= 0.6) & (el["nu0"] >= 0))[::2]
    Y0 = O.kepler_states(const, **{k: v[pick] for k, v in el.items()})
    K = 4
    r = np.linalg.norm(Y0[:, 0:3], axis=1)
    tf = 0.05 * 2 * np.pi * np.sqrt(r ** 3 / const.MU) * (K - 1)
    _, x, u = O.kepler_batch(const, K, tf, "tangential", Y0=Y0)
    assert {0.0, 90.0, 160.0} <= set(np.round(np.degrees(el["inc"][pick])))
    seen = check(x, u, tf, const, j2, [(s, k) for s in range(len(pick)) for k in range(K - 1)])
    assert max(n for n, _ in seen) > 30         # max_step = 1e-2 of an interval of 1/3


def test_coast_to_thrust_switch_with_zero_inputs(const):
    """u exactly zero on the first nodes, thrust after: the guarded 1/|u| of the node term and the hold across the switch"""
    _, x, u = synth_batch(2, 12, 0.5, const)
    u = u.copy()
    u[:, :, :6] = 0.0
    for j2 in (False, True):
        check(x, u, 0.5, const, j2, [(s, k) for s in range(2) for k in range(11)])


def test_short_horizon_max_step_binds(const):
    """K = 5: intervals of 1/4 in tau, so max_step = 1e-2 caps every step (26 nodes or more per interval)"""
    _, x, u = synth_batch(2, 5, 0.3, const)
    for j2 in (False, True):
        seen = check(x, u, 0.3, const, j2, [(s, k) for s in range(2) for k in range(4)])
        assert min(n for n, _ in seen) >= 26


def test_rejected_steps(const):
    """eccentric orbits with a loose max_step (1.0): the error controller decides the steps and scipy rejects some
    (nfev > 2 + 3 (len(sol.t) - 1)); the kernel takes the same decisions"""
    el = O.sweep_elements()
    pick = np.flatnonzero((el["e"] >= 0.6) & (el["nu0"] >= 0))[::2]
    Y0 = O.kepler_states(const, **{k: v[pick] for k, v in el.items()})
    K = 4
    r = np.linalg.norm(Y0[:, 0:3], axis=1)
    tf = 0.2 * 2 * np.pi * np.sqrt(r ** 3 / const.MU) * (K - 1)
    _, x, u = O.kepler_batch(const, K, tf, "tangential", Y0=Y0)
    seen = check(x, u, tf, const, False, [(s, k) for s in range(len(pick)) for k in range(K - 1)], max_step=1.0)
    assert any(_rejects(n, f) for n, f in seen)


def test_inv_cube_root_against_pow():
    """x^(-1/3) of the controller and the initial step: to rounding over the double range (float seed + Newton on the
    reduced argument), and the clamped factors of scipy's controller exactly where pow gives them, at the clamp edges"""
    L = _lib()
    L.hostk_inv_cube_root.restype = None
    edges = [0.09 ** 3, 4.5 ** 3, 1.0]            # 0.9 x^(-1/3) = 10 (MAX_FACTOR), = 0.2 (MIN_FACTOR); accept / reject
    xs = [np.nextafter(e, d) for e in edges for d in (0.0, np.inf)] + edges
    xs += list(np.logspace(-300, 300, 241)) + [5e-324, 2.2250738585072014e-308, 1e-45, 1e-39, 3.4e38, 1e39, 1.7976931348623157e308]
    xs += list(np.random.default_rng(7).uniform(0.0, 100.0, 2000))
    x = np.ascontiguousarray(xs, dtype=np.float64)
    y = np.empty_like(x)
    L.hostk_inv_cube_root(hostk._p(x), len(x), hostk._p(y))
    assert np.max(np.abs(y * np.cbrt(x) - 1.0)) <= 4e-16
    # scipy's err ** (-1/3) rounds the exponent: |ln x| 2e-17 apart from the exact root, <= 4e-16 where the controller
    # and the initial step evaluate it
    ref = x ** (-1.0 / 3.0)
    sel = (x >= 1e-8) & (x <= 1e4)
    assert np.max(np.abs(y[sel] / ref[sel] - 1.0)) <= 6e-16
    acc = np.minimum(10.0, 0.9 * y)
    rej = np.maximum(0.2, 0.9 * y)
    assert np.array_equal(acc <= 10.0, np.minimum(10.0, 0.9 * ref) <= 10.0)
    for e, f in ((edges[0], 10.0), (edges[1], 0.2)):
        i = list(x).index(e)
        assert abs((acc if f == 10.0 else rej)[i] - f) <= 4e-15
    # x = 0 (err == 0: the caller takes MAX_FACTOR) and x = inf (a rejection: MIN_FACTOR) come out as NaN, which the
    # clamps turn into what pow's 0 / inf give
    sp = np.array([0.0, np.inf, np.nan])
    z = np.empty_like(sp)
    L.hostk_inv_cube_root(hostk._p(sp), 3, hostk._p(z))
    assert np.isnan(z).all()
    assert np.fmax(0.2, 0.9 * z[1]) == max(0.2, 0.9 * np.inf ** (-1 / 3))


def test_ragged_and_units_bit_identical_to_single_launches(const):
    """a ragged batch (K_s from 3 to 9 nodes) and a constellation in per-satellite constants: every satellite's columns,
    status and node counts bit for bit those of a rectangular single-constant launch on it alone"""
    N, Kmax = 4, 9
    _, x, u = synth_batch(N, Kmax, 0.4, const)
    K_sat = np.array([9, 3, 6, 2], dtype=np.int32)
    xp, up = x.copy(), u.copy()
    for s, k in enumerate(K_sat):
        xp[s, :, k:] = np.nan
        up[s, :, k:] = np.nan
    tfs = np.array([0.4, 0.3, 0.45, 0.2])
    consts = [dataclasses.replace(const, MU=const.MU * (1.0 + 0.01 * s), ISP=const.ISP * (1.0 - 0.02 * s)) for s in range(N)]
    for j2 in (False, True):
        for cc in (const, consts):
            out, st, nodes = run(xp, up, tfs, cc, j2=j2, K_sat=K_sat)
            for s, k in enumerate(K_sat):
                one = consts[s] if isinstance(cc, list) else const
                o1, s1, n1 = run(np.ascontiguousarray(x[s:s + 1, :, :k]), np.ascontiguousarray(u[s:s + 1, :, :k]), tfs[s], one, j2=j2)
                cols = slice(s * (Kmax - 1), s * (Kmax - 1) + k - 1)
                assert np.array_equal(out[:, cols], o1, equal_nan=True), (j2, s)
                assert np.array_equal(st[cols], s1) and np.array_equal(nodes[cols], n1)
                assert np.isnan(out[:, s * (Kmax - 1) + k - 1:(s + 1) * (Kmax - 1)]).all()   # padding not written
            rect, _, _ = run(x, u, tfs, cc, j2=j2)
            assert np.array_equal(rect[:, 0:Kmax - 1], out[:, 0:Kmax - 1])


def test_status_words(const):
    """zero mass: ST_MASS (the reference raises); NaN input: ST_NONFINITE"""
    _, x, u = synth_batch(2, 4, 0.3, const)
    xm = x.copy()
    xm[0, 6, :] = 0.0
    _, st, _ = run(xm, u, 0.3, const)
    assert (st[:3] == 1).all() and (st[3:] == 0).all()
    xn = x.copy()
    xn[1, 0, 1] = np.nan
    _, st, _ = run(xn, u, 0.3, const)
    assert st[4] == 2 and (np.delete(st, 4) == 0).all()      # interval k starts from x[:, k] only


def test_rk23_kernel_under_address_sanitizer():
    """edge shapes (K = 2, batches that do not fill or straddle a warp, ragged counts of 2, per-satellite constants) under
    AddressSanitizer + UBSan, as tests/hostk/sanitize_driver.py runs the other kernel sources"""
    asan = subprocess.run(["gcc", "-print-file-name=libasan.so"], capture_output=True, text=True).stdout.strip()
    if not os.path.isabs(asan) or not os.path.exists(asan):
        pytest.skip("no AddressSanitizer runtime next to this gcc")
    _build(sanitize=True)
    code = (
        "import sys, numpy as np\n"
        f"sys.path.insert(0, {os.path.join(ROOT, 'tests')!r}); sys.path.insert(0, {ROOT!r})\n"
        "import test_rk23_kernel_source_on_host as T\n"
        "from conftest import synth_batch\n"
        "from oracle.mpc_oracle import OracleConstants\n"
        f"const = OracleConstants(*np.load({os.path.join(ROOT, 'tests', 'golden', 'discretize.npz')!r})['const'])\n"
        "L = T._lib(sanitize=True)\n"
        "n = 0\n"
        "for N, K in ((1, 2), (3, 5), (33, 4), (7, 13)):\n"
        "    _, x, u = synth_batch(N, K, 0.3, const)\n"
        "    ks = np.array([2 + (s * 5) % (K - 1) for s in range(N)], np.int32)\n"
        "    for j2 in (False, True):\n"
        "        for cc in (const, [const] * N):\n"
        "            for K_sat in (None, ks):\n"
        "                for ms in (1e-2, 1.0):\n"
        "                    T.run(x, u, 0.3, cc, j2=j2, K_sat=K_sat, max_step=ms, L=L)\n"
        "                    n += 1\n"
        "print(f'rk23 launches clean: {n}')\n")
    env = dict(os.environ, HOSTK_SANITIZE="1", LD_PRELOAD=asan, ASAN_OPTIONS="detect_leaks=0:halt_on_error=1")
    res = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, timeout=900)
    assert res.returncode == 0 and "rk23 launches clean" in res.stdout, res.stdout[-2000:] + res.stderr[-4000:]
    assert "AddressSanitizer" not in res.stderr and "runtime error" not in res.stderr
