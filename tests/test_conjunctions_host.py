"""Conjunction screening without a GPU: the kernel sources (conjunction_kernel.cuh) in the host build against the numpy
oracle (conj_oracle.py) -- the per-interval functions on 1e5 random pair-intervals, the bounding spheres, the pre-pass
under ASan + UBSan, an analytic two-body encounter, a constellation in one constants bag and in per-satellite units -- and
what screen_conjunctions and the C-ABI reject before any device work."""
import ctypes
import os
import shutil
import subprocess
import sys

import numpy as np
import pytest

import conj_oracle as O
import hostk
import mpconstellation_b200 as M
from conftest import ROOT
from mpconstellation_b200 import _lib, batch, conjunctions

HERE = os.path.join(ROOT, "tests", "hostk")
D_ = ctypes.c_double
MAXEV = 6


def _build(sanitize=False):
    """libmpc_hostk_conj[_asan].so: tests/hostk/conj_main.cpp over hostk's sources plus conjunction_kernel.cuh"""
    hostk.build(sanitize=sanitize)
    hdr = os.path.join(hostk.CSRC, "conjunction_kernel.cuh")
    text = open(hdr).read()
    assert "asm(" not in text, "inline PTX the host build does not know"
    dst = os.path.join(hostk.BUILD, "conjunction_kernel.cuh")
    if not os.path.exists(dst) or open(dst).read() != text:
        tmp = f"{dst}.{os.getpid()}.tmp"
        shutil.copyfile(hdr, tmp)
        os.replace(tmp, dst)
    so = os.path.join(hostk.BUILD, "libmpc_hostk_conj_asan.so" if sanitize else "libmpc_hostk_conj.so")
    src = os.path.join(HERE, "conj_main.cpp")
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


def _hl(sanitize=False):
    if sanitize not in _LIBS:
        _LIBS[sanitize] = ctypes.CDLL(_build(sanitize))
    return _LIBS[sanitize]


p = hostk._p


def prepass(y, scale, D, L=None):
    L = L or _hl()
    y = np.ascontiguousarray(y, dtype=np.float64)
    N, _, T = y.shape
    X, S = np.full((T, 6, N), -7.0), np.full((T - 1, 4, N), -7.0)
    sk = np.full(N, -1, dtype=np.int32)
    L.hostk_conj_prepass(p(y), p(np.ascontiguousarray(scale)), N, T, D_(D / (T - 1)), p(X), p(S), p(sk))
    return X, S, sk


def host_screen(y, tf, const, thr, capacity=1 << 16, L=None):
    """the host build of the whole screen -> (events as (i, j, k, t_ca, d_min, v_rel) sorted, flags, skipped, passed)"""
    L = L or _hl()
    y = np.ascontiguousarray(y, dtype=np.float64)
    scale, D = conjunctions.screen_scales(y.shape, tf, const, thr)
    N, _, T = y.shape
    X, S = np.empty((T, 6, N)), np.empty((T - 1, 4, N))
    sk = np.empty(N, dtype=np.int32)
    ev = np.zeros(capacity, dtype=_lib.CONJUNCTION_DTYPE)
    cnt = np.zeros(3, dtype=np.int64)
    L.hostk_conj_screen(p(y), p(scale), N, T, D_(D / (T - 1)), D_(thr), p(X), p(S), p(sk), p(ev), ctypes.c_longlong(capacity),
                        p(cnt))
    ev = ev[:cnt[0]]
    ev = ev[np.lexsort((ev["t_ca"], ev["j"], ev["i"]))]
    return ([(int(e["i"]), int(e["j"]), int(e["k"]), float(e["t_ca"]), float(e["d_min"]), float(e["v_rel"])) for e in ev],
            ev["flags"], sk, int(cnt[2]))


def random_pair_intervals(m, h=30.0, spread=4.0e4, seed=0):
    """m pair-intervals of two satellites a few tens of km apart, moving at up to ~2 km/s relative to each other, on
    smooth (Kepler-like) segments: q [m, 4, 6] (qi0, qi1, qj0, qj1)"""
    rng = np.random.default_rng(seed)
    r = rng.standard_normal((m, 3))
    r *= (6.9e6 + 5e5 * rng.random((m, 1))) / np.linalg.norm(r, axis=1, keepdims=True)
    t = np.cross(r, rng.standard_normal((m, 3)))
    v = 7.5e3 * t / np.linalg.norm(t, axis=1, keepdims=True)

    def step(r, v):    # two-body Taylor step over h: the next sample
        a = -O.MU_EARTH * r / np.linalg.norm(r, axis=1, keepdims=True) ** 3
        return r + h * v + 0.5 * h * h * a, v + h * a
    ri1, vi1 = step(r, v)
    dr = spread * rng.standard_normal((m, 3))
    dv = 1.0e3 * rng.standard_normal((m, 3))
    dr -= h * rng.random((m, 1)) * dv            # aim the relative track through the neighbourhood of 0
    rj, vj = r + dr, v + dv
    rj1, vj1 = step(rj, vj)
    q = np.stack([np.concatenate([r, v], 1), np.concatenate([ri1, vi1], 1), np.concatenate([rj, vj], 1),
                  np.concatenate([rj1, vj1], 1)], axis=1)
    return np.ascontiguousarray(q)


def host_intervals(q, fl, h, thr):
    ev = np.zeros((len(q), MAXEV, 4))
    n = np.zeros(len(q), dtype=np.int32)
    L = _hl()
    assert L.hostk_conj_interval(p(q), p(np.ascontiguousarray(fl, dtype=np.int32)), len(q), D_(h), D_(thr), p(ev), p(n)) == MAXEV
    return ev, n


def test_interval_functions_against_oracle():
    """1e5 random pair-intervals (first / last flags at random): the same events as the oracle's real roots of the
    quintic, d_min to 1e-9 relative (or 1e-6 m), t_ca to 1e-6 h; pair-intervals with a minimum within 1e-6 relative of
    the threshold are left out (either answer is right there)"""
    m, h, thr = 100000, 30.0, 2.0e4
    q = random_pair_intervals(m, h)
    rng = np.random.default_rng(1)
    fl = rng.integers(0, 4, m)
    ev, n = host_intervals(q, fl, h, thr)
    assert (ev[:, :, 3] == 0).all()
    first, last = (fl & 1).astype(bool), (fl & 2).astype(bool)
    ref_lo = O.interval_events(q[:, 0], q[:, 1], q[:, 2], q[:, 3], h, thr * (1 - 1e-6), first, last)
    ref_hi = O.interval_events(q[:, 0], q[:, 1], q[:, 2], q[:, 3], h, thr * (1 + 1e-6), first, last)
    compared = n_ev = 0
    for e in range(m):
        if len(ref_lo[e]) != len(ref_hi[e]):
            continue
        ref = ref_lo[e]
        assert n[e] == len(ref), (e, n[e], ref)
        for a, (s, d, v) in enumerate(ref):
            assert abs(ev[e, a, 0] - s) <= 1e-6, (e, ev[e, a], s)
            assert abs(ev[e, a, 1] - d) <= max(1e-9 * d, 1e-6), (e, ev[e, a], d)
            assert abs(ev[e, a, 2] - v) <= max(1e-7 * v, 1e-6), (e, ev[e, a], v)
        compared += 1
        n_ev += len(ref)
    assert compared >= m - 10 and n_ev > 5000, (compared, n_ev)
    # the oracle itself against dense sampling: every discrete local minimum of d below the threshold on 1001 points has
    # an event within 1e-3 of it, no farther than the grid allows
    s = np.linspace(0.0, 1.0, 1001)
    A = O.cubic(q[:2000, 0], q[:2000, 1], q[:2000, 2], q[:2000, 3], h)
    P = A[0][:, None] + s[None, :, None] * (A[1][:, None] + s[None, :, None] * (A[2][:, None] + s[None, :, None] * A[3][:, None]))
    d = np.linalg.norm(P, axis=-1)
    for e in range(2000):
        loc = np.flatnonzero((d[e, 1:-1] < d[e, :-2]) & (d[e, 1:-1] < d[e, 2:]) & (d[e, 1:-1] < 0.999 * thr)) + 1
        for li in loc:
            near = [x for x in ref_lo[e] if abs(x[0] - s[li]) <= 1e-3]
            assert near and min(x[1] for x in near) <= d[e, li] + 1e-9, (e, s[li], ref_lo[e])


def test_bounding_spheres_contain_segments():
    """every Hermite segment sampled at 1001 points lies in its sphere, for satellites in LEO to GEO and h up to an
    eighth of an orbit; a non-finite sample gives a NaN sphere"""
    rng = np.random.default_rng(3)
    m = 4000
    q = random_pair_intervals(m, 30.0, seed=5)
    h = np.exp(rng.uniform(np.log(1.0), np.log(900.0), m))
    s = np.linspace(0.0, 1.0, 1001)[:, None]
    for e in range(m):
        q0, q1 = q[e, 0], q[e, 1]
        out = np.zeros(4)
        _hl().hostk_conj_sphere(p(q0), p(q1), 1, D_(h[e]), p(out))
        h00, h10, h01, h11 = 2 * s ** 3 - 3 * s ** 2 + 1, s ** 3 - 2 * s ** 2 + s, -2 * s ** 3 + 3 * s ** 2, s ** 3 - s ** 2
        pts = h00 * q0[:3] + h10 * h[e] * q0[3:] + h01 * q1[:3] + h11 * h[e] * q1[3:]
        assert np.linalg.norm(pts - out[:3], axis=1).max() <= out[3], e
    bad = q[0, 1].copy()
    bad[4] = np.nan
    out = np.zeros(4)
    _hl().hostk_conj_sphere(p(q[0, 0]), p(bad), 1, D_(30.0), p(out))
    assert np.isnan(out).all()


def test_prepass_layout_and_skipped():
    """X [T][6][N] in SI, S [T-1][4][N], skipped counts the intervals with a non-finite end sample"""
    y, tf, const = O.fly(O.shell(5, seed=2), 600.0, 7)
    y[3, 4, 2] = np.nan
    y[1, 6, :] = np.nan                      # the mass row is not read
    scale, D = conjunctions.screen_scales(y.shape, tf, const, 1.0)
    X, S, sk = prepass(y, scale, D)
    ref = O.si_states(y, const)
    assert np.allclose(np.transpose(X, (2, 1, 0)), ref, rtol=1e-15, atol=0, equal_nan=True)
    assert list(sk) == [0, 0, 0, 2, 0]
    assert np.isnan(S[1:3, :, 3]).all() and np.isfinite(np.delete(S, 3, axis=2)).all()


def test_prepass_under_address_sanitizer():
    """the pre-pass on edge shapes (T = 2, N not a multiple of 32, one satellite over a warp) and the whole host screen
    under AddressSanitizer + UBSan: every buffer exactly of its documented size"""
    asan = subprocess.run(["gcc", "-print-file-name=libasan.so"], capture_output=True, text=True).stdout.strip()
    if not os.path.isabs(asan) or not os.path.exists(asan):
        pytest.skip("no AddressSanitizer runtime next to this gcc")
    _build(sanitize=True)
    code = (
        "import sys, numpy as np\n"
        f"sys.path.insert(0, {os.path.join(ROOT, 'tests')!r}); sys.path.insert(0, {ROOT!r})\n"
        "import test_conjunctions_host as T, conj_oracle as O\n"
        "L = T._hl(sanitize=True)\n"
        "n = 0\n"
        "for N, Tn in ((2, 2), (3, 5), (33, 4), (7, 13)):\n"
        "    y, tf, c = O.fly(O.shell(N, seed=N), 300.0, Tn)\n"
        "    y[N - 1, 0, Tn - 1] = np.nan\n"
        "    sc = np.ascontiguousarray(np.tile([c.R0, c.R0 * 1e-3], (N, 1)))\n"
        "    X, S, sk = T.prepass(y, sc, 300.0, L=L)\n"
        "    assert sk[N - 1] == 1\n"
        "    T.host_screen(y, tf, c, 1e6, capacity=3, L=L)\n"
        "    n += 2\n"
        "print(f'conj launches clean: {n}')\n")
    env = dict(os.environ, HOSTK_SANITIZE="1", LD_PRELOAD=asan, ASAN_OPTIONS="detect_leaks=0:halt_on_error=1")
    res = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, timeout=900)
    assert res.returncode == 0 and "conj launches clean" in res.stdout, res.stdout[-2000:] + res.stderr[-4000:]
    assert "AddressSanitizer" not in res.stderr and "runtime error" not in res.stderr


def two_body_case(T=361, a=7.0e6, alpha=np.radians(30.0), dtheta=0.01, u_mid=0.8):
    """two circular orbits of radius a, planes alpha apart about the x axis (the line of nodes), the satellites dtheta
    apart in phase: closest approach when they stand symmetric about the line of nodes (mean argument of latitude 0 or
    pi), d_min = 2 a sin(dtheta / 2) cos(alpha / 2).  One orbit period, starting at mean argument of latitude -u_mid."""
    n = np.sqrt(O.MU_EARTH / a ** 3)
    D = 2 * np.pi / n
    st = np.array([O.circular_state(a, 0.0, 0.0, -u_mid - dtheta / 2), O.circular_state(a, alpha, 0.0, -u_mid + dtheta / 2)])
    t_exact = np.array([u_mid, u_mid + np.pi]) / n
    d_exact = 2 * a * np.sin(dtheta / 2) * np.cos(alpha / 2)
    return st, D, n, t_exact, d_exact


def test_two_body_analytic_encounter():
    """two_body_case on 361 samples of one period, in the host build and in the oracle.  The bound of the check: the cubic
    Hermite interpolant of a smooth curve errs by at most h^4 max|p''''| / 384 in position and h^3 max|p''''| sqrt(3) /
    216 in velocity, and on a circular orbit |p''''| = a n^4.  The samples themselves (the RK45 restatement) err by e_r,
    e_v against the exact orbit, which the interpolant carries with weights <= 1 (positions) and <= 4 h / 27
    (velocities).  For the pair: eps_p = 2 (Hermite + e_r + 4 h e_v / 27), eps_v = 2 (Hermite' + 2 e_r / h + e_v).  Then
    |d_min error| <= eps_p, and the instant of the minimum, a root of dp . dv whose slope is >= |dv|^2 - d |da| with
    |da| <= 2 a n^2, moves by at most (eps_p |dv| + d eps_v) / (|dv|^2 - 2 d a n^2)."""
    st, D, n, t_exact, d_exact = two_body_case()
    T = 361
    y, tf, const = O.fly(st, D, T)
    X = O.si_states(y, const)
    h = D / (T - 1)
    a = 7.0e6
    # sample errors of the flight against the exact circular orbits
    t = np.linspace(0.0, D, T)
    e_r = e_v = 0.0
    for s, (inc, u0) in enumerate(((0.0, -0.8 - 0.005), (np.radians(30.0), -0.8 + 0.005))):
        ex = np.array([O.circular_state(a, inc, 0.0, u0 + n * tt)[:6] for tt in t]).T
        e_r = max(e_r, np.abs(np.linalg.norm(X[s, :3] - ex[:3], axis=0)).max())
        e_v = max(e_v, np.abs(np.linalg.norm(X[s, 3:] - ex[3:], axis=0)).max())
    herm_p = h ** 4 * a * n ** 4 / 384
    herm_v = h ** 3 * a * n ** 4 * np.sqrt(3) / 216
    eps_p = 2 * (herm_p + e_r + 4 * h * e_v / 27)
    eps_v = 2 * (herm_v + 2 * e_r / h + e_v)
    dv = np.linalg.norm(O.circular_state(a, 0.0, 0.0, -0.005)[3:6] - O.circular_state(a, np.radians(30.0), 0.0, 0.005)[3:6])
    dt_bound = (eps_p * dv + d_exact * eps_v) / (dv ** 2 - 2 * d_exact * a * n ** 2)
    ev, flags, sk, _ = host_screen(y, tf, const, 1.0e5)
    assert len(ev) == 2 and (flags == 0).all() and (sk == 0).all()
    for e, te in zip(ev, t_exact):
        assert abs(e[4] - d_exact) <= eps_p, (e, d_exact, eps_p)
        assert abs(e[3] - te) <= dt_bound, (e, te, dt_bound)
        assert abs(e[5] - dv) <= eps_v + 1e-6 * dv
    assert eps_p < 1.0 and dt_bound < 1e-2                 # the bound is tight enough to mean something
    # and the oracle on the same samples
    ref, _ = O.screen(X, D, 1.0e5)
    O.match(ev, ref, h)


def test_one_bag_and_per_satellite_units_agree():
    """the same SI trajectories expressed in one constants bag and in every satellite's own units (tf_s = D / s0_s):
    the same events, values to 1e-9; both equal to the oracle"""
    states = O.shell(48, n_planes=6, seed=11)
    D, T = 1500.0, 51
    y, tf, const = O.fly(states, D, T)
    X = O.si_states(y, const)
    yu, inv_s0, consts = O.renormalize(X, states)
    thr = O.pick_threshold(X, D, 3.0e5)
    ev1, _, _, passed = host_screen(y, tf, const, thr)
    ev2, _, _, _ = host_screen(yu, D * inv_s0, consts, thr)
    assert len(ev1) >= 5, len(ev1)
    O.match(ev1, ev2, D / (T - 1), rel=1e-9, t_tol=1e-9)
    ref, _ = O.screen(X, D, thr)
    O.match(ev1, ref, D / (T - 1))
    assert passed < 48 * 47 // 2 * (T - 1) // 4      # the sphere filter passes over most pair-intervals


def test_screen_scales_and_value_errors():
    states = O.shell(4, seed=1)
    y, tf, const = O.fly(states, 300.0, 5)
    scale, D = conjunctions.screen_scales(y.shape, tf, const, 10.0)
    s0 = 2 * np.pi * np.sqrt(const.R0 ** 3 / O.MU_EARTH)
    assert np.allclose(scale, [[const.R0, const.R0 / s0]] * 4, rtol=1e-15) and abs(D - 300.0) <= 1e-9
    yu, inv_s0, consts = O.renormalize(O.si_states(y, const), states)
    tfs = 300.0 * inv_s0
    conjunctions.screen_scales(yu.shape, tfs, consts, 10.0)
    tfs[2] *= 1 + 1e-10
    with pytest.raises(ValueError, match="satellite 2"):
        conjunctions.screen_scales(yu.shape, tfs, consts, 10.0)
    with pytest.raises(ValueError, match="satellite 1"):
        conjunctions.screen_scales(y.shape, tf, const, 10.0, T_sat=[5, 4, 5, 5])
    for thr in (0.0, -1.0, np.inf, np.nan):
        with pytest.raises(ValueError, match="threshold"):
            conjunctions.screen_scales(y.shape, tf, const, thr)
    with pytest.raises(ValueError, match="N = 1"):
        conjunctions.screen_scales((1, 7, 5), tf, const, 1.0)
    with pytest.raises(ValueError, match="T = 1"):
        conjunctions.screen_scales((3, 7, 1), tf, const, 1.0)
    with pytest.raises(ValueError, match=r"\[N, 7, T\]"):
        conjunctions.screen_scales((3, 6, 5), tf, const, 1.0)
    with pytest.raises(ValueError, match="expected 4"):
        conjunctions.screen_scales(y.shape, tf, consts[:3], 1.0)
    with pytest.raises(ValueError, match="satellite 0"):
        conjunctions.screen_scales(y.shape, 0.0, const, 1.0)


def test_rejections_before_device_work(monkeypatch):
    """(the context is never created: _ctx raising would show a device call)"""
    def no_device(*a, **k):
        raise AssertionError("device work before the argument checks")
    monkeypatch.setattr(batch, "_ctx", no_device)
    y, tf, const = O.fly(O.shell(3, seed=4), 300.0, 4)
    with pytest.raises(ValueError, match="satellite 1"):
        M.screen_conjunctions(y, [tf, 2 * tf, tf], const, 1e4)
    with pytest.raises(ValueError, match="threshold"):
        M.screen_conjunctions(y, tf, const, 0.0)
    with pytest.raises(ValueError, match="ragged"):
        M.screen_conjunctions(y, tf, const, 1e4, T_sat=[4, 4, 3])
    with pytest.raises(ValueError, match="CUDA tensor"):
        M.screen_conjunctions_device(y, tf, const, 1e4)


def test_c_abi_rejects_before_touching_the_device():
    L = _lib.lib()
    N, T = 3, 4
    y = np.zeros((N, 7, T))
    scale = np.ones((N, 2))
    cnt, fl = ctypes.c_int64(-1), ctypes.c_int64(-1)
    sk = np.zeros(N, np.int32)
    ev = np.zeros(4, dtype=_lib.CONJUNCTION_DTYPE)
    assert ev.itemsize == 40

    def host(ctx=1, y=y, n=N, T=T, sc=scale, D=10.0, thr=1.0, ev=ev, cap=4):
        return L.mpc_screen_conjunctions_host(ctx, _lib.addr(y), n, T, _lib.addr(sc), D, thr, _lib.addr(ev), cap,
                                              ctypes.byref(cnt), ctypes.byref(fl), _lib.addr(sk))

    def dev(y=y, n=N, T=T, sc=scale, D=10.0, thr=1.0, scratch=1, ev=1, cap=4, counters=1, skipped=1):
        return L.mpc_screen_conjunctions(_lib.addr(y), n, T, _lib.addr(sc), D, thr, scratch, ev, cap, counters, skipped, None)
    # (a bogus non-null ctx / device pointers: the checks come first and none of them is dereferenced)
    for f in (host, dev):
        assert f(y=None) == _lib.E_INVALID
        assert f(sc=None) == _lib.E_INVALID
        assert f(n=1) == _lib.E_INVALID and b"n_sats >= 2" in L.mpc_last_error()
        assert f(T=1) == _lib.E_INVALID
        for thr in (0.0, -1.0, np.inf, np.nan):
            assert f(thr=thr) == _lib.E_INVALID and b"threshold" in L.mpc_last_error()
        for D in (0.0, np.nan):
            assert f(D=D) == _lib.E_INVALID and b"duration" in L.mpc_last_error()
        for v in (0.0, -2.0, np.inf, np.nan):
            bad = scale.copy()
            bad[2, 1] = v
            assert f(sc=bad) == _lib.E_INVALID and b"scale[2][1]" in L.mpc_last_error()
    assert host(ctx=None) == _lib.E_INVALID
    assert host(ev=None) == _lib.E_INVALID and host(cap=-1) == _lib.E_INVALID
    assert dev(scratch=None) == _lib.E_INVALID and dev(counters=None) == _lib.E_INVALID
    assert dev(skipped=None) == _lib.E_INVALID and dev(ev=None) == _lib.E_INVALID
    assert L.mpc_conjunction_scratch_doubles(4096, 200) == 4096 * (6 * 200 + 4 * 199 + 2)
