"""Discretizer.ivp_solver = 'RK23', host logic (no GPU): what raises NotImplementedError before any device work, and what
the C-ABI entries mpc_discretize_batch_rk23[_host] reject before they touch the device."""
import ctypes

import numpy as np
import pytest

import mpconstellation_b200 as M
from mpconstellation_b200 import _lib, batch
from mpconstellation_b200.batch import _units_of
from mpconstellation_b200.model import Satellite, sat_units


def satellite_dynamics(*a, **k):      # the name the Discretizer accepts (Simulator.satellite_dynamics)
    raise AssertionError("never called")


def _consts(n):
    sats = [Satellite(np.array([7.0e6 + 1.0e6 * i, 0.0, 0.0]), np.array([0.0, 7.5e3 - 300.0 * i, 0.0]), 500.0 + 1000.0 * i)
            for i in range(n)]
    return sat_units(sats)


def _xu(N=2, K=5, Ku=None):
    x = np.ones((N, 7, K))
    u = np.zeros((N, 3, Ku or K))
    return x, u


def test_discretizer_rejections():
    _, consts = _consts(1)
    c = consts[0]
    x, u = _xu(1)
    d = M.Discretizer(c)
    d.ivp_solver = "RK23"
    d.use_uniform_steps = True
    with pytest.raises(NotImplementedError, match="dense output"):
        d.discretize(satellite_dynamics, x[0], u[0], 1.0)
    c.CD = 2.2
    d = M.Discretizer(c, rho_func=lambda r: 1.0, drho_func=lambda r: 0.0, include_drag=True)
    d.ivp_solver = "RK23"
    with pytest.raises(NotImplementedError, match="include_drag"):
        d.discretize(satellite_dynamics, x[0], u[0], 1.0)
    d = M.Discretizer(consts[0])
    for name in ("DOP853", "Radau", "BDF", "LSODA", "rk23"):
        d.ivp_solver = name
        with pytest.raises(NotImplementedError, match="RK45 and RK23 only"):
            d.discretize(satellite_dynamics, x[0], u[0], 1.0)


def test_batch_rejections_before_device_work(monkeypatch):
    """(the context is never created: _ctx raising would show a device call)"""
    def no_device(*a, **k):
        raise AssertionError("device work before the argument checks")
    monkeypatch.setattr(batch, "_ctx", no_device)
    monkeypatch.setattr(batch, "_torch", no_device)
    _, consts = _consts(1)
    x, u = _xu()
    with pytest.raises(NotImplementedError, match="own grid"):
        batch.discretize_batch(x, _xu(Ku=9)[1], 1.0, consts[0], adaptive=dict(method="RK23"))
    with pytest.raises(NotImplementedError, match="include_drag"):
        batch.discretize_batch(x, u, 1.0, consts[0], include_drag=True, disc_drag=(2.2, 1.0), adaptive=dict(method="RK23"))
    for m in ("DOP853", "Radau"):
        with pytest.raises(NotImplementedError, match="RK45 and RK23 only"):
            batch.discretize_batch(x, u, 1.0, consts[0], adaptive=dict(method=m))
        with pytest.raises(NotImplementedError, match="RK45 and RK23 only"):
            batch.discretize_batch_device(x, u, np.ones(2), consts[0], adaptive=dict(method=m))
    with pytest.raises(NotImplementedError, match="one destination"):
        batch.discretize_batch_device(x, u, np.ones(2), consts[0], adaptive=dict(method="RK23"), extra_dst=[0])
    assert batch._rk23(None) is False and batch._rk23({}) is False and batch._rk23(dict(method="RK45")) is False
    assert batch._rk23(dict(method="RK23", rtol=1e-3)) is True


def test_c_abi_rejects_before_touching_the_device():
    L = _lib.lib()
    _, consts = _consts(2)
    psc, _ = _units_of(consts, 2)
    N, K = 2, 5
    x, u, tf = np.zeros((N, 7, K)), np.zeros((N, 3, K)), np.ones(N)
    out, status = np.zeros((105, N * (K - 1))), np.zeros(N * (K - 1), np.int32)
    scratch = np.zeros(N * _lib.SAT_SCRATCH_DOUBLES)
    first = np.zeros(N + 1, np.int64)
    p = _lib.make_params(consts[0])

    def disc(p=p, cs=None, K_sat=None, rtol=1e-3, K=K, xp=x, o=out):
        return L.mpc_discretize_batch_rk23(_lib.addr(xp), _lib.addr(u), _lib.addr(tf), ctypes.byref(p), cs, N, K,
                                           _lib.addr(K_sat), _lib.addr(first), _lib.addr(scratch), rtol, 1e-6, 1e-2,
                                           _lib.addr(o), N * (K - 1), 0, _lib.addr(status), None, None)
    p_drag = _lib.make_params(consts[0], include_drag=True, disc_drag=(2.2, 1.0))
    assert disc(p_drag) == _lib.E_UNSUPPORTED and b"drag" in L.mpc_last_error()
    assert disc(p_drag, psc) == _lib.E_UNSUPPORTED
    bad = (_lib.MpcSatConsts * 2)(psc[0], psc[1])
    bad[1].mu = 0.0
    assert disc(cs=bad) == _lib.E_INVALID and b"consts[1]" in L.mpc_last_error()
    bad[1].mu, bad[1].isp = psc[1].mu, float("inf")
    assert disc(cs=bad) == _lib.E_INVALID and b"consts[1]" in L.mpc_last_error()
    assert disc(K_sat=np.array([5, 1], np.int32)) == _lib.E_INVALID and b"K_sat[1]" in L.mpc_last_error()
    assert disc(K_sat=np.array([6, 3], np.int32)) == _lib.E_INVALID
    assert disc(rtol=0.0) == _lib.E_INVALID and b"rtol" in L.mpc_last_error()
    assert disc(K=1) == _lib.E_INVALID
    assert disc(xp=None) == _lib.E_INVALID
    assert disc(o=None) == _lib.E_INVALID
    rc = L.mpc_discretize_batch_rk23(_lib.addr(x), _lib.addr(u), _lib.addr(tf), ctypes.byref(p), None, N, K,
                                     _lib.addr(np.array([5, 3], np.int32)), None, None, 1e-3, 1e-6, 1e-2, _lib.addr(out),
                                     N * (K - 1), 0, _lib.addr(status), None, None)
    assert rc == _lib.E_INVALID and b"first" in L.mpc_last_error()
    rc = L.mpc_discretize_batch_rk23(_lib.addr(x), _lib.addr(u), _lib.addr(tf), ctypes.byref(p), None, N, K, None, None,
                                     None, 1e-3, 1e-6, 1e-2, _lib.addr(out), N * (K - 1) - 1, 0, _lib.addr(status), None, None)
    assert rc == _lib.E_INVALID and b"out_pitch" in L.mpc_last_error()
    # an empty batch is a no-op
    assert L.mpc_discretize_batch_rk23(_lib.addr(x), _lib.addr(u), _lib.addr(tf), ctypes.byref(p), None, 0, K, None, None,
                                       None, 1e-3, 1e-6, 1e-2, _lib.addr(out), 0, 0, None, None, None) == 0
    assert L.mpc_discretize_batch_rk23_host(None, _lib.addr(x), _lib.addr(u), _lib.addr(tf), ctypes.byref(p), None, N, K,
                                            None, 1e-3, 1e-6, 1e-2, _lib.addr(out), _lib.addr(status), None) == _lib.E_INVALID
