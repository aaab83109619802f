"""Per-satellite constants, host logic (no GPU): which calls take the single-constant launches, which raise, and what
the C-ABI rejects before it touches the device."""
import ctypes

import numpy as np
import pytest

from mpconstellation_b200 import _lib
from mpconstellation_b200.batch import _units_of
from mpconstellation_b200.model import Constants, Satellite, SatelliteScale, sat_units
from mpconstellation_b200.scp import BatchedSCP


def _consts(n):
    sats = [Satellite(np.array([7.0e6 + 1.0e6 * i, 0.0, 0.0]), np.array([0.0, 7.5e3 - 300.0 * i, 0.0]), 500.0 + 1000.0 * i)
            for i in range(n)]
    return sat_units(sats)


def test_sat_units_normalizes_each_satellite_by_its_own_scale():
    sats = [Satellite(np.array([7.0e6, 0.0, 0.0]), np.array([0.0, 7.5e3, 0.0]), 12200.0),
            Satellite(np.array([0.0, 2.6e7, 0.0]), np.array([-3.9e3, 0.0, 0.0]), 300.0)]
    y0, consts = sat_units(sats)
    for s, sat in enumerate(sats):
        sc = SatelliteScale(sat=sat)
        assert np.array_equal(y0[s], sc.normalize_state(sat.get_state_vector()))
        assert vars(consts[s]) == vars(sc.get_normalized_constants())
    assert consts[0].R_E != consts[1].R_E and consts[0].RHO != consts[1].RHO


def test_equal_constants_take_the_single_constant_path():
    _, consts = _consts(1)
    same = [Constants(**vars(consts[0])) for _ in range(4)]
    psc, one = _units_of(same, 4)
    assert psc is None and one is same[0]
    psc, one = _units_of(consts[0], 4)
    assert psc is None and one is consts[0]


def test_differing_constants_pack_the_seven_fields():
    _, consts = _consts(3)
    psc, one = _units_of(consts, 3)
    assert one is consts[0] and len(psc) == 3
    for s, c in enumerate(consts):
        assert (psc[s].mu, psc[s].r_e, psc[s].j2, psc[s].g0, psc[s].isp, psc[s].s_area, psc[s].rho) == \
            (c.MU, c.R_E, c.J2, c.G0, c.ISP, c.S, c.RHO)


def test_length_and_attribute_errors():
    _, consts = _consts(3)
    with pytest.raises(ValueError, match="expected 4"):
        _units_of(consts, 4)

    class NoRho:
        MU, R_E, J2, G0, ISP, S = 1.0, 1.0, 1.0, 1.0, 1.0, 1.0
    with pytest.raises(ValueError, match="RHO"):
        _units_of([consts[0], NoRho()], 2)


def test_rejected_combinations_raise():
    y0, consts = _consts(3)
    with pytest.raises(ValueError, match="drag"):
        _units_of(consts, 3, drag=True)
    with pytest.raises(ValueError, match="own grid"):
        _units_of(consts, 3, ugrid=True)
    with pytest.raises(NotImplementedError, match="per-satellite constants"):
        BatchedSCP(consts).run_segments(y0, 1)


def _c_consts(consts):
    psc, _ = _units_of(consts, len(consts))
    return psc


def test_c_abi_rejects_before_touching_the_device():
    """argument checks of the *_units entry points (no device call is made before them)"""
    L = _lib.lib()
    y0, consts = _consts(2)
    psc = _c_consts(consts)
    N, K = 2, 5
    x, u, tf = np.zeros((N, 7, K)), np.zeros((N, 3, K)), np.ones(N)
    out, status = np.zeros((105, N * (K - 1))), np.zeros(N * (K - 1), np.int32)
    scratch = np.zeros(N * _lib.SAT_SCRATCH_DOUBLES)

    def disc(p, cs, adaptive=0):
        return L.mpc_discretize_batch_units(_lib.addr(x), _lib.addr(u), _lib.addr(tf), ctypes.byref(p), cs, N, K, None, None,
                                            _lib.addr(scratch), adaptive, 100, 1e-3, 1e-6, 1e-2, _lib.addr(out), N * (K - 1), 0,
                                            _lib.addr(status), None, None)
    p_drag = _lib.make_params(consts[0], include_drag=True, disc_drag=(2.2, 1.0))
    assert disc(p_drag, psc) == _lib.E_UNSUPPORTED and b"drag" in L.mpc_last_error()
    bad = (_lib.MpcSatConsts * 2)(psc[0], psc[1])
    bad[1].g0 = 0.0
    assert disc(_lib.make_params(consts[0]), bad) == _lib.E_INVALID and b"consts[1]" in L.mpc_last_error()
    bad[1].g0, bad[1].rho = psc[1].g0, float("nan")
    assert disc(_lib.make_params(consts[0]), bad) == _lib.E_INVALID and b"consts[1]" in L.mpc_last_error()
    assert L.mpc_set_tuning(9) == 0
    try:
        assert disc(_lib.make_params(consts[0]), psc, adaptive=1) == _lib.E_UNSUPPORTED and b"round-1" in L.mpc_last_error()
    finally:
        assert L.mpc_set_tuning(10) == 0
    # the propagation names the satellite whose constants are invalid
    c = _lib.MpcController()
    c.kind = _lib.CTRL_ZERO
    y = np.zeros((N, 7, K))
    rc = L.mpc_propagate_batch_rk45_units(_lib.addr(y0), _lib.addr(tf), ctypes.byref(_lib.make_params(consts[0])), bad,
                                          ctypes.byref(c), N, K, None, None, _lib.addr(scratch), 1e-3, 1e-6, 1e-3, _lib.addr(y),
                                          None, None, None, None)
    assert rc == _lib.E_INVALID and b"consts[1]" in L.mpc_last_error()


def test_any_sequence_of_bags_and_nothing_else():
    _, consts = _consts(3)
    arr = np.empty(3, dtype=object)
    arr[:] = consts
    psc, one = _units_of(arr, 3)
    assert one is consts[0] and len(psc) == 3
    with pytest.raises(ValueError, match="sequence of 3"):
        _units_of(1.0, 3)


def test_rk4_propagator_rejects_per_satellite_constants():
    import mpconstellation_b200 as M
    y0, consts = _consts(3)
    ctrl = M.ConstantTangentialThrustController(tangential_thrust=0.1)
    with pytest.raises(ValueError, match="RK4"):
        M.propagate_batch(y0, 0.3, ctrl, consts, T=10, n_sub=10)
    torch = pytest.importorskip("torch")
    with pytest.raises(ValueError, match="RK4"):
        M.propagate_batch_device(torch.as_tensor(y0), torch.ones(3, dtype=torch.float64), ctrl, consts, T=10, n_sub=10)


@pytest.mark.parametrize("uniform", [False, True])
def test_batched_scp_routes_per_satellite_constants_past_the_fused_pass(monkeypatch, uniform):
    """per-satellite constants: one propagation and one discretization call per pass, with the constants list and the
    per-satellite counts, never the fused overlapped pass; one bag in uniform mode keeps the fused pass"""
    from mpconstellation_b200 import batch, scp
    y0, consts = _consts(3)
    calls = []

    def prop(y0_, tf, ctrl, const, **kw):
        calls.append(("propagate", const, kw.get("T")))
        T = int(np.max(kw["T"]))
        return np.zeros((3, 7, T)), np.zeros((3, 3, T)), None, None

    def disc(x, u, tf, const, **kw):
        calls.append(("discretize", const, kw.get("K")))
        return None

    def fused(*a, **kw):
        calls.append(("fused",))
        K = kw["T"]
        return None, np.zeros((3, 7, K)), np.zeros((3, 3, K))
    monkeypatch.setattr(batch, "propagate_batch", prop)
    monkeypatch.setattr(batch, "discretize_batch", disc)
    monkeypatch.setattr(batch, "propagate_discretize", fused)
    ctrl = scp.ConstantTangentialThrustController(tangential_thrust=0.1)
    lin = BatchedSCP(consts, base_res=30, use_uniform_steps=uniform).linearize(y0, 2.0, ctrl)
    assert [c[0] for c in calls] == ["propagate", "discretize"]
    assert calls[0][1] is consts and calls[1][1] is consts and lin.const is consts
    assert np.array_equal(calls[0][2], [60] * 3) and np.array_equal(calls[1][2], [60] * 3)
    if uniform:
        calls.clear()
        BatchedSCP(consts[0], base_res=30, use_uniform_steps=True).linearize(y0, 2.0, ctrl)
        assert [c[0] for c in calls] == ["fused"]
