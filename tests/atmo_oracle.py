"""TEST INFRASTRUCTURE ONLY -- oracles of the drag under an altitude-dependent atmosphere:

  propagate_batch_rk45   tests/atmo_oracle.c: the plain-C restatement of the reference's RK45 call (oracle/mpc_oracle.c,
                         included unchanged) with the density from the Atmosphere's series at h = |r| R0 - R_EARTH;
  propagate_scipy        scipy's solve_ivp (RK45, max_step) on the numpy oracle's dynamics without drag plus the drag of
                         simulator.py:150-153 with a Python callable rho(h) -- the altitude-dependent models of
                         simulator.py:110-111 as the reference's authors would have flown them.

Nothing in mpconstellation_b200/ imports this.
"""
import ctypes
import os
import subprocess

import numpy as np
from scipy import integrate

from oracle import c_oracle as C
from oracle import mpc_oracle as O

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "atmo_oracle.c")
BUILD = os.path.join(HERE, "hostk", "_build")
SO = os.path.join(BUILD, "libatmo_oracle.so")
R_EARTH = 6.371e6   # m (constants.py)


class OrcAtmo(ctypes.Structure):
    """orc_atmo (the layout of mpc_atmosphere)"""
    _fields_ = [("h_min", ctypes.c_double), ("h_max", ctypes.c_double), ("r_earth", ctypes.c_double),
                ("n", ctypes.c_int), ("reserved", ctypes.c_int), ("coef", ctypes.c_double * 32)]


_lib = None


def lib():
    global _lib
    if _lib is None:
        deps = [SRC, os.path.join(os.path.dirname(HERE), "oracle", "mpc_oracle.c")]
        if not (os.path.exists(SO) and all(os.path.getmtime(SO) >= os.path.getmtime(d) for d in deps)):
            os.makedirs(BUILD, exist_ok=True)
            tmp = f"{SO}.{os.getpid()}.tmp"
            # the flags of oracle/Makefile (the system gcc: the one with libgomp)
            subprocess.check_call(["/usr/bin/gcc", "-O2", "-fPIC", "-fopenmp", "-ffp-contract=off", "-shared", "-o", tmp, SRC,
                                   "-lm"])
            os.replace(tmp, SO)
        _lib = ctypes.CDLL(SO)
        dp, ip = ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_int)
        _lib.orc_propagate_rk45_atmo.argtypes = [dp, dp, ctypes.POINTER(C.OrcParams), ctypes.c_int, dp, dp, ctypes.c_int,
                                                 ctypes.c_int, ctypes.c_double, dp, ctypes.c_int, ctypes.c_int,
                                                 ctypes.c_double, ctypes.c_double, ctypes.c_double, dp, dp, ip, ip, ip,
                                                 ctypes.c_int, ctypes.POINTER(OrcAtmo)]
        _lib.orc_propagate_rk45_atmo.restype = ctypes.c_int
    return _lib


def _atmo(a):
    """an Atmosphere (mpconstellation_b200.fit_atmosphere: h_min, h_max, coef) -> OrcAtmo"""
    o = OrcAtmo(float(a.h_min), float(a.h_max), R_EARTH, len(a.coef), 0)
    for k, c in enumerate(a.coef):
        o.coef[k] = float(c)
    return o


def propagate_batch_rk45(y0, tf, const, kind=C.CTRL_ZERO, cparams=(0.0, 0.0, 0.0), table=None, end_tau=1.0,
                         include_J2=True, T=100, rtol=1e-3, atol=1e-6, max_step=1e-3, atmosphere=None):
    """oracle.c_oracle.propagate_batch_rk45 with drag under `atmosphere` -> (y[N,7,T], u[N,3,T], status[N] (2: an
    altitude outside the model's range), n_steps[N], n_rejected[N])"""
    y0 = np.ascontiguousarray(y0, dtype=np.float64)
    N = y0.shape[0]
    tf = np.ascontiguousarray(np.broadcast_to(np.asarray(tf, dtype=np.float64), (N,)))
    cp = np.ascontiguousarray(np.resize(np.asarray(cparams, dtype=np.float64), 3))
    Ku, per_sat = 0, 0
    if table is not None:
        table = np.ascontiguousarray(table, dtype=np.float64)
        Ku = table.shape[-1]
        per_sat = int(table.ndim == 3)
    y = np.zeros((N, 7, T))
    uo = np.zeros((N, 3, T))
    status = np.zeros(N, dtype=np.int32)
    steps = np.zeros(N, dtype=np.int32)
    rej = np.zeros(N, dtype=np.int32)
    p = C.make_params(const, include_J2, True)
    ip = ctypes.POINTER(ctypes.c_int)
    dp = C._dp
    lib().orc_propagate_rk45_atmo(dp(y0), dp(tf), ctypes.byref(p), kind, dp(cp), dp(table), Ku, per_sat, float(end_tau),
                                  None, N, T, rtol, atol, max_step, dp(y), dp(uo), status.ctypes.data_as(ip),
                                  steps.ctypes.data_as(ip), rej.ctypes.data_as(ip), 0, ctypes.byref(_atmo(atmosphere)))
    return y, uo, status, steps, rej


def propagate_scipy(y0, tf, u_func, const, density, include_J2=True, eval_points=100, max_step=0.001):
    """solve_ivp(RK45, max_step) of the reference's dynamics with rho(h) in the drag -> (y[7,T], t[T])"""
    ts = np.linspace(0, 1, eval_points)

    def rhs(t, y):
        dy = O.dynamics(y, u_func(y, t), tf, const, include_drag=False, include_J2=include_J2)
        r, v, m = y[0:3], y[3:6], y[6]
        rho = float(density(np.linalg.norm(r) * const.R0 - R_EARTH))
        dy[3:6] += tf * (-0.5 * O.C_D * const.S * (1 / m) * (rho / const.RHO) * np.linalg.norm(v) * v)
        return dy

    sol = integrate.solve_ivp(rhs, [0, 1], np.asarray(y0, dtype=float), t_eval=ts, max_step=max_step)
    return sol.y, sol.t
