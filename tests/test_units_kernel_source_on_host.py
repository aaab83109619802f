"""Per-satellite designer units in the host (g++) build of the kernel sources: a constellation that mixes altitudes,
masses, eccentricities and inclinations, every satellite normalized by its own SatelliteScale, through ONE launch of the
PSC instantiations (pair and default-mode discretization, RK45 propagation, constraint terms; rectangular and ragged).
Every satellite must come out bit for bit as the rectangular host launch of that satellite under its own constants
alone, with the same status / node / step counts, and the padding must stay untouched.  A second build under
AddressSanitizer + UBSan runs the same kernels at edge shapes with exactly sized buffers."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

import hostk
from conftest import ROOT

HERE = os.path.join(ROOT, "tests", "hostk")
D = ctypes.c_double


def _build(sanitize=False):
    """libmpc_hostk_units[_asan].so: tests/hostk/units_main.cpp over the sources hostk.build() prepared"""
    hostk.build(sanitize=sanitize)
    so = os.path.join(hostk.BUILD, "libmpc_hostk_units_asan.so" if sanitize else "libmpc_hostk_units.so")
    src = os.path.join(HERE, "units_main.cpp")
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


def mixed_constellation(n=6):
    """Satellites from dimensional states: perigee altitudes 400 km ... 20,000 km, masses 300 ... 12,200 kg,
    eccentricities 0 ... 0.3, inclinations 0 ... 98 deg.  -> (y0 [n,7], [n] Constants), each in its own units."""
    from mpconstellation_b200.model import MU_EARTH, R_EARTH, Satellite, sat_units
    alt = np.array([400e3, 20000e3, 1200e3, 7000e3, 550e3, 3500e3])
    mass = np.array([12200.0, 300.0, 2500.0, 800.0, 5000.0, 1500.0])
    ecc = np.array([0.0, 0.05, 0.3, 0.0, 0.1, 0.2])
    inc = np.radians([28.5, 0.0, 63.4, 98.0, 51.6, 10.0])
    sats = []
    for i in range(n):
        j = i % 6
        rp = R_EARTH + alt[j] * (1 + 0.01 * (i // 6))
        vp = np.sqrt(MU_EARTH * (1 + ecc[j]) / rp)
        ci, si = np.cos(inc[j]), np.sin(inc[j])
        sats.append(Satellite(np.array([rp, 0.0, 0.0]), np.array([0.0, vp * ci, vp * si]), mass[j]))
    return sat_units(sats)


def _c8(consts):
    return np.ascontiguousarray([hostk._const8(c) for c in consts], dtype=np.float64)


def _trajectories(y0, consts, K_sat, tf=0.3):
    """x, u [N,.,Kmax]: satellite s propagated in its own units (host RK45 replay, tangential thrust), NaN padding"""
    N, Kmax = len(K_sat), int(max(K_sat))
    x, u = np.full((N, 7, Kmax), np.nan), np.full((N, 3, Kmax), np.nan)
    for s, k in enumerate(K_sat):
        y, uo, st, _, _ = hostk.propagate_rk45(y0[s:s + 1], tf, consts[s], kind=2, thrust=(0.05, 0, 0), T=int(k))
        assert st[0] == 0
        x[s, :, :k], u[s, :, :k] = y[0], uo[0]
    return x, u


def discretize_units(L, x, u, tf, consts, K_sat, adaptive, include_J2=False, n_sub=100, em=1):
    x = np.ascontiguousarray(x)
    u = np.ascontiguousarray(u)
    N, _, K = x.shape
    tfv = np.full(N, float(tf))
    first = None if K_sat is None else np.concatenate([[0], np.cumsum(np.asarray(K_sat, np.int64) - 1)]).astype(np.int64)
    pitch = N * (K - 1)
    out = np.full((105, pitch), np.nan)
    status = np.full(pitch, -1, np.int32)
    nodes = np.full(pitch, -1, np.int32)
    L.hostk_discretize_units(hostk._p(x), hostk._p(u), hostk._p(tfv), hostk._p(_c8(consts)), int(include_J2), N, K,
                             hostk._p(first), int(adaptive), int(n_sub), D(1e-3), D(1e-6), D(1e-2), hostk._p(out),
                             ctypes.c_longlong(pitch), hostk._p(status), hostk._p(nodes), int(em))
    return out, status.reshape(N, K - 1), nodes.reshape(N, K - 1)


@pytest.mark.parametrize("ragged", [False, True])
@pytest.mark.parametrize("adaptive", [False, True])
@pytest.mark.parametrize("j2", [False, True])
def test_units_discretize_is_bit_identical_to_per_satellite_launches(ragged, adaptive, j2):
    y0, consts = mixed_constellation()
    K_sat = np.array([7, 2, 12, 5, 12, 3] if ragged else [9] * 6, np.int32)
    Kmax = int(K_sat.max())
    x, u = _trajectories(y0, consts, K_sat)
    out, st, nodes = discretize_units(_lib(), x, u, 0.3, consts, K_sat if ragged else None, adaptive, include_J2=j2)
    for s, k in enumerate(K_sat):
        n = k - 1
        cols = slice(s * (Kmax - 1), s * (Kmax - 1) + n)
        xs, us = x[s:s + 1, :, :k], u[s:s + 1, :, :k]
        if adaptive:
            ref, rst, rnodes = hostk.discretize_adaptive(xs, us, 0.3, consts[s], include_J2=j2)
            assert np.array_equal(nodes[s, :n], rnodes)
        else:
            ref, rst = hostk.discretize(xs, us, 0.3, consts[s], include_J2=j2)
        assert np.array_equal(out[:, cols], ref) and np.array_equal(st[s, :n], rst), s
        assert np.isnan(out[:, s * (Kmax - 1) + n:(s + 1) * (Kmax - 1)]).all() and (st[s, n:] == -1).all()


def test_units_differ_from_a_common_scale():
    """the table is read per satellite: the same inputs under satellite 0's constants give other matrices"""
    y0, consts = mixed_constellation()
    K_sat = np.array([9] * 6, np.int32)
    x, u = _trajectories(y0, consts, K_sat)
    out, _, _ = discretize_units(_lib(), x, u, 0.3, consts, None, False)
    one, _, _ = discretize_units(_lib(), x, u, 0.3, [consts[0]] * 6, None, False)
    n = 8
    assert np.array_equal(out[:, :n], one[:, :n])
    assert all(not np.array_equal(out[:, s * n:(s + 1) * n], one[:, s * n:(s + 1) * n]) for s in range(1, 6))


@pytest.mark.parametrize("ragged", [False, True])
@pytest.mark.parametrize("j2", [False, True])
def test_units_rk45_lanes_match_per_satellite_runs(ragged, j2):
    L = _lib()
    y0, consts = mixed_constellation()
    N, T_max, Ku = 6, 40, 12
    T_sat = np.array([40, 2, 17, 33, 9, 40], np.int32) if ragged else None
    ku = np.array([12, 2, 7, 12, 4, 9], np.int32) if ragged else None
    tab = 0.05 * np.random.default_rng(3).standard_normal((N, 3, Ku))
    for kind in (2, 3):
        y = np.full((N, 7, T_max), np.nan)
        uo = np.full((N, 3, T_max), np.nan)
        st = np.full(N, -1, np.int32)
        steps = np.zeros(N, np.int32)
        L.hostk_propagate_rk45_units(hostk._p(y0), hostk._p(np.full(N, 0.5)), hostk._p(_c8(consts)), int(j2), kind, D(0.05),
                                     hostk._p(tab), Ku, hostk._p(ku), N, T_max, hostk._p(T_sat), hostk._p(y), hostk._p(uo),
                                     hostk._p(st), hostk._p(steps))
        for s in range(N):
            t = int(T_sat[s]) if ragged else T_max
            k = int(ku[s]) if ragged else Ku
            table = np.ascontiguousarray(tab[s:s + 1, :, :k]) if kind == 3 else None
            yr, ur, sr, nr, _ = hostk.propagate_rk45(y0[s:s + 1], 0.5, consts[s], kind=kind, thrust=(0.05, 0, 0), table=table,
                                                     T=t, include_J2=j2)
            assert np.array_equal(y[s, :, :t], yr[0]) and np.array_equal(uo[s, :, :t], ur[0]), (kind, s)
            assert st[s] == sr[0] == 0 and steps[s] == nr[0]
            assert np.isnan(y[s, :, t:]).all() and np.isnan(uo[s, :, t:]).all()


@pytest.mark.parametrize("ragged", [False, True])
def test_units_constraint_terms_match_per_satellite_launches(ragged):
    L = _lib()
    y0, consts = mixed_constellation()
    K_sat = np.array([7, 2, 12, 5, 12, 3] if ragged else [9] * 6, np.int32)
    N, Kmax = 6, int(K_sat.max())
    x, u = _trajectories(y0, consts, K_sat)
    first = np.concatenate([[0], np.cumsum(K_sat.astype(np.int64) - 1)]).astype(np.int64) if ragged else None
    rbar, ubar, fin = np.full((N, 3, Kmax - 1), np.nan), np.full((N, 3, Kmax), np.nan), np.full((N, 32), np.nan)
    mu = np.array([c.MU for c in consts])
    L.hostk_constraint_terms_units(hostk._p(x), hostk._p(u), N, Kmax, hostk._p(first), hostk._p(mu), hostk._p(rbar),
                                   hostk._p(ubar), hostk._p(fin))
    for s, k in enumerate(K_sat):
        r, ub, f = hostk.constraint_terms(x[s:s + 1, :, :k], u[s:s + 1, :, :k], consts[s].MU)
        assert np.array_equal(rbar[s, :, :k - 1], r[0]) and np.array_equal(ubar[s, :, :k], ub[0]) and np.array_equal(fin[s], f[0])
        assert np.isnan(rbar[s, :, k - 1:]).all() and np.isnan(ubar[s, :, k:]).all()


def test_units_kernels_under_address_sanitizer():
    asan = subprocess.run(["gcc", "-print-file-name=libasan.so"], capture_output=True, text=True).stdout.strip()
    if not os.path.isabs(asan) or not os.path.exists(asan):
        pytest.skip("no AddressSanitizer runtime next to this gcc")
    _build(sanitize=True)
    code = (
        "import sys, ctypes, numpy as np\n"
        f"sys.path.insert(0, {os.path.join(ROOT, 'tests')!r}); sys.path.insert(0, {ROOT!r})\n"
        "import hostk, test_units_kernel_source_on_host as T\n"
        "L = T._lib(sanitize=True)\n"
        "for N, K_sat in ((1, [2]), (1, [9]), (3, [2, 9, 2]), (2, [9, 9])):\n"
        "    y0, consts = T.mixed_constellation(N)\n"
        "    K_sat = np.array(K_sat, np.int32)\n"
        "    x, u = T._trajectories(y0, consts, K_sat)\n"
        "    for ragged in (False, True):\n"
        "        if not ragged and len(set(K_sat.tolist())) > 1: continue\n"
        "        for ad in (0, 1):\n"
        "            for j2 in (0, 1):\n"
        "                T.discretize_units(L, x, u, 0.3, consts, K_sat if ragged else None, ad, include_J2=j2, n_sub=100 if ad else 6)\n"
        "        first = np.concatenate([[0], np.cumsum(K_sat.astype(np.int64) - 1)]) if ragged else None\n"
        "        Kmax = int(K_sat.max())\n"
        "        r, ub, f = np.empty((N, 3, Kmax - 1)), np.empty((N, 3, Kmax)), np.empty((N, 32))\n"
        "        L.hostk_constraint_terms_units(hostk._p(x), hostk._p(u), N, Kmax, hostk._p(first),\n"
        "                                       hostk._p(np.array([c.MU for c in consts])), hostk._p(r), hostk._p(ub), hostk._p(f))\n"
        "        for kind in (2, 3):\n"
        "            Ku = Kmax\n"
        "            tab = 0.05 * np.ones((N, 3, Ku))\n"
        "            T_sat = K_sat if ragged else None\n"
        "            ku = K_sat if ragged else None\n"
        "            y, uo = np.empty((N, 7, Kmax)), np.empty((N, 3, Kmax))\n"
        "            st, steps = np.empty(N, np.int32), np.empty(N, np.int32)\n"
        "            L.hostk_propagate_rk45_units(hostk._p(y0), hostk._p(np.full(N, 0.3)), hostk._p(T._c8(consts)), 1, kind,\n"
        "                                         T.D(0.05), hostk._p(tab), Ku, hostk._p(ku), N, Kmax, hostk._p(T_sat), hostk._p(y),\n"
        "                                         hostk._p(uo), hostk._p(st), hostk._p(steps))\n"
        "print('units launches clean')\n")
    env = dict(os.environ, HOSTK_SANITIZE="1", LD_PRELOAD=asan, ASAN_OPTIONS="detect_leaks=0:halt_on_error=1")
    res = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, timeout=900)
    assert res.returncode == 0 and "units launches clean" in res.stdout, res.stdout[-2000:] + res.stderr[-4000:]
    assert "AddressSanitizer" not in res.stderr and "runtime error" not in res.stderr


NAMES = ("A_k", "B_kp", "B_kn", "Sigma_k", "xi_k")
# fixed-step forms against the literal 101-node sums (README): A_k on the 51-node form (the loosest), the quadrature rows
# with all 101 nodes (the loosest)
FIXED_BOUND = {"A_k": 5e-11, "B_kp": 1.6e-11, "B_kn": 1.6e-11, "Sigma_k": 1.6e-11, "xi_k": 1.6e-11}


@pytest.mark.parametrize("j2", [False, True])
def test_units_batch_against_the_c_oracle_per_satellite(j2):
    """every satellite of the mixed batch, through one PSC launch, against the plain-C oracle run on that satellite alone
    with its own constants: default mode with the same node counts and matrices to 1.3e-11, the fixed-step form within
    the README's per-form bounds, the RK45 propagation with the same attempted steps and states to 5e-12"""
    from conftest import rel_err
    from oracle import c_oracle as C
    L = _lib()
    y0, consts = mixed_constellation()
    N, K, tf = 6, 9, 0.3
    x, u = _trajectories(y0, consts, [K] * N, tf)
    soa_f, st_f, _ = discretize_units(L, x, u, tf, consts, None, False, include_J2=j2)
    soa_a, st_a, nodes = discretize_units(L, x, u, tf, consts, None, True, include_J2=j2)
    assert st_f.max() == 0 and st_a.max() == 0
    got_f, got_a = hostk.stacked(soa_f, N, K), hostk.stacked(soa_a, N, K)
    for s in range(N):
        xs, us = x[s:s + 1], u[s:s + 1]
        ref_f = C.discretize_batch(xs, us, tf, consts[s], include_J2=j2)
        ref_a = C.discretize_batch_adaptive(xs, us, tf, consts[s], include_J2=j2)
        assert ref_f[5].max() == 0 and ref_a[5].max() == 0
        assert np.array_equal(nodes[s], ref_a[6][0]), s
        for i, name in enumerate(NAMES):
            assert rel_err(got_f[i][s], ref_f[i][0]) <= FIXED_BOUND[name], (s, name, rel_err(got_f[i][s], ref_f[i][0]))
            assert rel_err(got_a[i][s], ref_a[i][0]) <= 1.3e-11, (s, name, rel_err(got_a[i][s], ref_a[i][0]))
    # propagation: tangential thrust so that 1 / (G0 ISP) matters, steps long enough for rejections on the e = 0.3 orbit
    T, thrust = 40, 0.05
    y = np.full((N, 7, T), np.nan)
    uo = np.full((N, 3, T), np.nan)
    st = np.full(N, -1, np.int32)
    steps = np.zeros(N, np.int32)
    L.hostk_propagate_rk45_units(hostk._p(y0), hostk._p(np.full(N, 0.5)), hostk._p(_c8(consts)), int(j2), 2, D(thrust),
                                 None, 0, None, N, T, None, hostk._p(y), hostk._p(uo), hostk._p(st), hostk._p(steps))
    assert st.max() == 0
    for s in range(N):
        yc, _, stc, acc_c, rej_c = C.propagate_batch_rk45(y0[s:s + 1], 0.5, consts[s], C.CTRL_TANGENTIAL, (thrust, 0, 0),
                                                          include_drag=False, include_J2=j2, T=T)
        assert stc[0] == 0 and steps[s] == acc_c[0] + rej_c[0], s
        assert rel_err(y[s], yc[0]) <= 5e-12, (s, rel_err(y[s], yc[0]))
