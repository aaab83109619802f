"""The RK45 replay under an altitude-dependent atmosphere (propagate_rk45_atmo_kernel) in the host (g++) build of the
kernel sources: against the plain-C oracle with the same series (attempted steps and states), against scipy's solve_ivp
on the Python callable, against the constant-density kernel for a constant model, bit-identity of ragged and
per-satellite-constants batches to single-satellite launches, the out-of-range status, and an ASan + UBSan run."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

import hostk
from conftest import ROOT, rel_err

HERE = os.path.join(ROOT, "tests", "hostk")
D = ctypes.c_double
S_SCALE = 1e4            # S scaled as in the drag fixtures, so that drag shows within a few orbits
RHO_CONST = 9.983e-13


def _build(sanitize=False):
    """libmpc_hostk_atmo[_asan].so: tests/hostk/atmo_main.cpp over the sources hostk.build() prepared"""
    hostk.build(sanitize=sanitize)
    so = os.path.join(hostk.BUILD, "libmpc_hostk_atmo_asan.so" if sanitize else "libmpc_hostk_atmo.so")
    src = os.path.join(HERE, "atmo_main.cpp")
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


def power_law(h):
    return 8e26 * h ** -6.828          # the reference authors' model (simulator.py:110)


def exponential(h):
    return 1e-12 * np.exp(-(h - 500e3) / 60e3)


def fitted(rho, lo, hi):
    from mpconstellation_b200 import fit_atmosphere
    return fit_atmosphere(rho, lo, hi)


def leo(alts=(400e3,), mass=122000.0, inc=51.6, s_scale=S_SCALE):
    """circular orbits at the given altitudes, normalized by the first one's scale -> (y0 [n,7], Constants with S scaled);
    the mass keeps a 400 km orbit above 300 km for three orbits at the scaled S"""
    from mpconstellation_b200.model import MU_EARTH, R_EARTH, Satellite, SatelliteScale
    ci, si = np.cos(np.radians(inc)), np.sin(np.radians(inc))
    sats = []
    for h in alts:
        r = R_EARTH + h
        v = np.sqrt(MU_EARTH / r)
        sats.append(Satellite(np.array([r, 0.0, 0.0]), np.array([0.0, v * ci, v * si]), mass))
    sc = SatelliteScale(sat=sats[0])
    const = sc.get_normalized_constants()
    const.S *= s_scale
    return np.array([sc.normalize_state(s.get_state_vector()) for s in sats]), const


def _atmo_vec(a):
    from mpconstellation_b200.model import R_EARTH
    return np.concatenate([[a.h_min, a.h_max, R_EARTH, len(a.coef)], a.coef]).astype(np.float64)


def run(L, y0, tf, consts, atmo, kind=2, thrust=(0.02, 0.0, 0.0), j2=True, T=50, table=None, ku=None, T_sat=None,
        end_tau=1.0, lpw=32):
    """the host kernel: consts one Constants (psc = 0) or a list of N (psc = 1) -> y, u, status, steps"""
    y0 = np.ascontiguousarray(y0, dtype=np.float64)
    N = y0.shape[0]
    psc = isinstance(consts, (list, tuple))
    c8 = np.ascontiguousarray([hostk._const8(c) for c in consts] if psc else hostk._const8(consts), dtype=np.float64)
    y, uo = np.full((N, 7, T), np.nan), np.full((N, 3, T), np.nan)
    st, steps = np.full(N, -1, np.int32), np.zeros(N, np.int32)
    th = np.ascontiguousarray(thrust, dtype=np.float64)
    tab = None if table is None else np.ascontiguousarray(table, dtype=np.float64)
    tfv = np.ascontiguousarray(np.broadcast_to(np.asarray(tf, dtype=np.float64), (N,)))
    L.hostk_propagate_rk45_atmo(hostk._p(y0), hostk._p(tfv), hostk._p(c8), int(psc), int(j2), D(2.5), int(kind),
                                hostk._p(th), hostk._p(tab), 0 if tab is None else tab.shape[-1], hostk._p(ku), D(end_tau), N,
                                int(T), hostk._p(T_sat), hostk._p(_atmo_vec(atmo)), int(lpw), hostk._p(y), hostk._p(uo),
                                hostk._p(st), hostk._p(steps))
    return y, uo, st, steps


LAWS = [(0, (0.0, 0.0, 0.0)), (1, (0.01, -0.02, 0.005)), (2, (0.02, 0.0, 0.0)), (3, None)]


@pytest.mark.parametrize("j2", [False, True])
@pytest.mark.parametrize("law", range(4))
def test_atmo_kernel_matches_the_c_oracle(law, j2):
    """every controller law, J2 on and off: the same attempted steps as the C oracle flying the same series, states
    within 5e-12"""
    import atmo_oracle as A
    L = _lib()
    atmo = fitted(power_law, 150e3, 1000e3)
    y0, const = leo((400e3, 450e3, 520e3))
    kind, thrust = LAWS[law]
    tab = 0.02 * np.random.default_rng(7).standard_normal((3, 3, 9)) if kind == 3 else None
    T, tf = 60, 1.5
    y, uo, st, steps = run(L, y0, tf, const, atmo, kind=kind, thrust=thrust or (0, 0, 0), j2=j2, T=T, table=tab,
                           end_tau=0.8)
    yc, uc, stc, acc, rej = A.propagate_batch_rk45(y0, tf, const, kind, thrust or (0, 0, 0), table=tab, end_tau=0.8,
                                                   include_J2=j2, T=T, atmosphere=atmo)
    assert st.max() == 0 and stc.max() == 0
    assert np.array_equal(steps, acc + rej), (steps, acc + rej)
    assert rel_err(y, yc) <= 5e-12, rel_err(y, yc)
    assert rel_err(uo, uc) <= 5e-12


def test_atmo_kernel_against_scipy_and_the_constant_density():
    """a 400 km orbit over three orbits under the power law: scipy's solve_ivp RK45 (max_step 0.001) on the numpy
    oracle's dynamics with the Python callable agrees to 1e-9; the constant-density flight is far from both"""
    import atmo_oracle as A
    from oracle import mpc_oracle as O
    L = _lib()
    atmo = fitted(power_law, 150e3, 1000e3)
    y0, const = leo((400e3,))
    T, tf = 61, 3.0
    y, _, st, _ = run(L, y0, tf, const, atmo, kind=0, j2=True, T=T)
    assert st[0] == 0
    ys, _ = A.propagate_scipy(y0[0], tf, O.ctrl_zero(), const, power_law, include_J2=True, eval_points=T)
    assert rel_err(y[0], ys) <= 1e-9, rel_err(y[0], ys)
    yk, _, _, _, _ = hostk.propagate_rk45(y0, tf, const, kind=0, include_drag=True, include_J2=True, T=T)
    assert rel_err(yk[0], ys) > 1e-5, rel_err(yk[0], ys)
    # the altitude decays faster under the denser 400 km air of the power law than under the 500 km constant
    assert np.linalg.norm(y[0, 0:3, -1]) < np.linalg.norm(yk[0, 0:3, -1])


@pytest.mark.parametrize("kind", [0, 2])
def test_constant_model_matches_the_constant_density_kernel(kind):
    """rho = 9.983e-13 everywhere through the series: the same attempted steps as the existing kernel, states to 1e-13"""
    L = _lib()
    atmo = fitted(lambda h: RHO_CONST, 100e3, 2000e3)
    y0, const = leo((400e3, 700e3))
    y, _, st, steps = run(L, y0, 1.0, const, atmo, kind=kind, j2=True, T=40)
    yk, _, stk, stepsk, _ = hostk.propagate_rk45(y0, 1.0, const, kind=kind, thrust=(0.02, 0, 0), include_drag=True,
                                                 include_J2=True, T=40)
    assert st.max() == 0 and stk.max() == 0
    assert np.array_equal(steps, stepsk)
    assert rel_err(y, yk) <= 1e-13, rel_err(y, yk)


def _exp_constellation(n=6):
    from test_units_kernel_source_on_host import mixed_constellation
    y0, consts = mixed_constellation(n)
    for c in consts:
        c.S *= S_SCALE
    return y0, consts


@pytest.mark.parametrize("ragged", [False, True])
@pytest.mark.parametrize("psc", [False, True])
def test_atmo_batches_are_bit_identical_to_single_satellite_launches(ragged, psc):
    """rectangular / ragged, one bag / per-satellite constants (400 ... 20,000 km, each in its own units, under the
    exponential model): every satellite bit for bit as a launch of it alone, padding untouched"""
    L = _lib()
    atmo = fitted(exponential, 200e3, 40000e3)
    y0, consts = _exp_constellation()
    if not psc:                            # one bag: the first satellite's units for all
        consts = consts[0]
        y0 = np.array([y0[0] * (1 + 0.05 * i) for i in range(6)])
    N, T_max, Ku = 6, 30, 10
    T_sat = np.array([30, 2, 17, 23, 9, 30], np.int32) if ragged else None
    ku = np.array([10, 2, 7, 10, 4, 9], np.int32) if ragged else None
    tab = 0.02 * np.random.default_rng(3).standard_normal((N, 3, Ku))
    for kind in (2, 3):
        y, uo, st, steps = run(L, y0, 0.4, consts, atmo, kind=kind, T=T_max, table=tab, ku=ku, T_sat=T_sat, lpw=4)
        assert st.max() == 0
        for s in range(N):
            t = int(T_sat[s]) if ragged else T_max
            k = int(ku[s]) if ragged else Ku
            one = consts[s] if psc else consts
            yr, ur, sr, nr = run(L, y0[s:s + 1], 0.4, one, atmo, kind=kind, T=t,
                                 table=np.ascontiguousarray(tab[s:s + 1, :, :k]))
            assert np.array_equal(y[s, :, :t], yr[0]) and np.array_equal(uo[s, :, :t], ur[0]), (kind, s)
            assert st[s] == sr[0] == 0 and steps[s] == nr[0]
            assert np.isnan(y[s, :, t:]).all() and np.isnan(uo[s, :, t:]).all()


def test_units_constellation_against_the_c_oracle_per_satellite():
    """each satellite of the mixed constellation in its own constants against the C oracle on that satellite alone"""
    import atmo_oracle as A
    L = _lib()
    atmo = fitted(exponential, 200e3, 40000e3)
    y0, consts = _exp_constellation()
    y, _, st, steps = run(L, y0, 0.5, consts, atmo, kind=2, T=40)
    assert st.max() == 0
    for s in range(6):
        yc, _, stc, acc, rej = A.propagate_batch_rk45(y0[s:s + 1], 0.5, consts[s], A.C.CTRL_TANGENTIAL, (0.02, 0, 0),
                                                      include_J2=True, T=40, atmosphere=atmo)
        assert stc[0] == 0 and steps[s] == acc[0] + rej[0], s
        assert rel_err(y[s], yc[0]) <= 5e-12, (s, rel_err(y[s], yc[0]))


def test_out_of_range_sets_the_atmosphere_status_for_that_satellite_only():
    import atmo_oracle as A
    L = _lib()
    atmo = fitted(power_law, 300e3, 1000e3)
    y0, const = leo((400e3, 250e3, 600e3))
    y, uo, st, _ = run(L, y0, 0.5, const, atmo, kind=0, T=20)
    assert st.tolist() == [0, 4, 0]
    assert np.isnan(y[1]).all() and np.isfinite(y[[0, 2]]).all()
    _, _, stc, _, _ = A.propagate_batch_rk45(y0, 0.5, const, include_J2=True, T=20, atmosphere=atmo)
    assert stc.tolist() == [0, 2, 0]
    # a satellite that decays out of the range mid-flight stops there: its samples before the exit are kept
    atmo_n = fitted(power_law, 390e3, 1000e3)
    y, _, st, _ = run(L, y0[:1], 1.0, const, atmo_n, kind=0, T=20)
    assert st[0] == 4 and np.isfinite(y[0, :, 0]).all() and np.isnan(y[0, :, -1]).all()


def test_atmo_kernels_under_address_sanitizer():
    asan = subprocess.run(["gcc", "-print-file-name=libasan.so"], capture_output=True, text=True).stdout.strip()
    if not os.path.isabs(asan) or not os.path.exists(asan):
        pytest.skip("no AddressSanitizer runtime next to this gcc")
    _build(sanitize=True)
    code = (
        "import sys, numpy as np\n"
        f"sys.path.insert(0, {os.path.join(ROOT, 'tests')!r}); sys.path.insert(0, {ROOT!r})\n"
        "import test_atmosphere_kernel_source_on_host as T\n"
        "L = T._lib(sanitize=True)\n"
        "atmo = T.fitted(T.exponential, 200e3, 40000e3)\n"
        "for N, T_sat in ((1, [2]), (1, [7]), (3, [2, 7, 2]), (33, None)):\n"
        "    y0, consts = T._exp_constellation(N)\n"
        "    T_max = 7 if T_sat is None else max(T_sat)\n"
        "    ts = None if T_sat is None else np.array(T_sat, np.int32)\n"
        "    tab = 0.02 * np.ones((N, 3, 5))\n"
        "    ku = None if T_sat is None else np.full(N, 3, np.int32)\n"
        "    for psc in (False, True):\n"
        "        for kind in (0, 1, 2, 3):\n"
        "            for lpw in (1, 32):\n"
        "                T.run(L, y0, 0.2, consts if psc else consts[0], atmo, kind=kind, T=T_max, table=tab, ku=ku,\n"
        "                      T_sat=ts, lpw=lpw)\n"
        "    T.run(L, y0[:1] * 0.9, 0.2, consts[0], T.fitted(T.power_law, 300e3, 1000e3), kind=0, T=T_max)\n"
        "print('atmo launches clean')\n")
    env = dict(os.environ, HOSTK_SANITIZE="1", LD_PRELOAD=asan, ASAN_OPTIONS="detect_leaks=0:halt_on_error=1")
    res = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, timeout=900)
    assert res.returncode == 0 and "atmo launches clean" in res.stdout, res.stdout[-2000:] + res.stderr[-4000:]
    assert "AddressSanitizer" not in res.stderr and "runtime error" not in res.stderr
