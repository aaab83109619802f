"""The altitude-dependent atmosphere on the B200: propagate_rk45_atmo_kernel through the public interface against the C
oracle and scipy, the host build, the kernel names, Simulator, BatchedSCP.run_segments at config 5's shape and a
per-satellite-units constellation from 400 to 20,000 km."""
import numpy as np
import pytest

from conftest import rel_err, synth_batch
from test_atmosphere_kernel_source_on_host import (LAWS, _exp_constellation, _lib as host_lib, exponential,
                                                   fitted, leo, power_law, run as host_run)

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def M():
    import mpconstellation_b200 as M
    M._lib.require_gpu()
    return M


def _spec(M, kind, thrust, tab=None, end_tau=1.0):
    return M.ControllerSpec(kind, tuple(thrust), tab, end_tau)


@pytest.mark.parametrize("j2", [False, True])
@pytest.mark.parametrize("law", range(4))
def test_device_against_the_oracle_and_the_host_build(M, law, j2):
    import atmo_oracle as A
    atmo = fitted(power_law, 150e3, 1000e3)
    y0, const = leo((400e3, 450e3, 520e3))
    kind, thrust = LAWS[law]
    thrust = thrust or (0.0, 0.0, 0.0)
    tab = 0.02 * np.random.default_rng(7).standard_normal((3, 3, 9)) if kind == 3 else None
    T, tf = 60, 1.5
    steps = np.zeros(3, np.int32)
    y, u, _, st = M.propagate_batch(y0, tf, _spec(M, kind, thrust, tab, 0.8), const, include_J2=j2, T=T, n_steps=steps,
                                    atmosphere=atmo)
    yc, uc, stc, acc, rej = A.propagate_batch_rk45(y0, tf, const, kind, thrust, table=tab, end_tau=0.8,
                                                   include_J2=j2, T=T, atmosphere=atmo)
    assert st.max() == 0 and stc.max() == 0
    assert np.array_equal(steps, acc + rej)
    assert rel_err(y, yc) <= 5e-12 and rel_err(u, uc) <= 5e-12, (rel_err(y, yc), rel_err(u, uc))
    # the host build of the same kernel: the same steps; log / exp of the two math libraries may differ in the last bit
    yh, uh, sth, nh = host_run(host_lib(), y0, tf, const, atmo, kind=kind, thrust=thrust, j2=j2, T=T, table=tab,
                               end_tau=0.8)
    assert np.array_equal(steps, nh) and sth.max() == 0
    assert rel_err(y, yh) <= 1e-13 and rel_err(u, uh) <= 1e-13, (rel_err(y, yh), rel_err(u, uh))


def test_one_launch_of_the_new_kernels_and_none_without_an_atmosphere(M):
    import torch
    from torch.profiler import ProfilerActivity, profile
    atmo = fitted(power_law, 150e3, 1000e3)
    y0, const = leo((400e3, 450e3, 520e3))
    y0d = torch.as_tensor(y0, device="cuda")
    tfd = torch.full((3,), 0.5, dtype=torch.float64, device="cuda")
    ctrl = M.ConstantTangentialThrustController(tangential_thrust=0.02)
    names, ys = {}, {}
    for key, a in (("atmo", atmo), ("const", None)):
        M.propagate_batch_device(y0d, tfd, ctrl, const, T=20, atmosphere=a)   # warm-up
        torch.cuda.synchronize()
        before = M.launch_count()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            y, u, st = M.propagate_batch_device(y0d, tfd, ctrl, const, T=20, atmosphere=a)
            torch.cuda.synchronize()
        assert M.launch_count() - before == 1 and int(st.max()) == 0
        ys[key] = y.cpu().numpy()
        names[key] = [e.name for e in prof.events() if "propagate" in e.name and e.device_type.name == "CUDA"]
    assert len(names["atmo"]) == 1 and "propagate_rk45_atmo_kernel" in names["atmo"][0], names
    assert len(names["const"]) == 1 and "propagate_rk45_kernel" in names["const"][0], names
    # device form = host form, per-satellite constants included
    y_h, u_h, _, _ = M.propagate_batch(y0, 0.5, ctrl, const, T=20, atmosphere=atmo)
    assert np.array_equal(ys["atmo"], y_h) and not np.array_equal(ys["const"], y_h)
    y0u, consts = _exp_constellation()
    atmo_e = fitted(exponential, 200e3, 40000e3)
    yd, _, std = M.propagate_batch_device(torch.as_tensor(y0u, device="cuda"), torch.full((6,), 0.4, dtype=torch.float64,
                                          device="cuda"), ctrl, consts, T=20, atmosphere=atmo_e)
    yh2, _, _, _ = M.propagate_batch(y0u, 0.4, ctrl, consts, T=20, atmosphere=atmo_e)
    assert int(std.max()) == 0 and np.array_equal(yd.cpu().numpy(), yh2)


def test_simulator_run_with_the_model_against_scipy(M):
    import atmo_oracle as A
    from oracle import mpc_oracle as O
    from mpconstellation_b200.model import MU_EARTH, R_EARTH
    atmo = fitted(power_law, 150e3, 1000e3)
    r = R_EARTH + 400e3
    v = np.sqrt(MU_EARTH / r)
    sat = M.Satellite(np.array([r, 0.0, 0.0]), np.array([0.0, v * 0.6, v * 0.8]), 1000.0)
    scale = M.SatelliteScale(sat=sat)
    sim = M.Simulator(sats=[sat], scale=scale, base_res=30)
    sim.atmosphere = atmo
    data, _ = sim.run(tf=2)
    ys, _ = A.propagate_scipy(scale.normalize_state(sat.get_state_vector()), 2, O.ctrl_zero(),
                              scale.get_normalized_constants(), power_law, include_J2=True, eval_points=60)
    assert rel_err(data[sat.id], ys) <= 1e-9, rel_err(data[sat.id], ys)


def test_config5_run_segments_with_the_model(M, const):
    """256 satellites, base_res=30, tf_horizon=2, two segments of one orbit; the first flight segment per satellite
    against the C oracle flying the same series (the exponential model: the synthetic constellation's eccentric orbits
    leave the power law's 300 ... 1,000 km)"""
    from mpconstellation_b200.scp import BatchedSCP
    import atmo_oracle as A
    atmo = fitted(exponential, 200e3, 40000e3)
    y0, _, _ = synth_batch(256, 2, 1.0, const)
    scp = BatchedSCP(const, base_res=30, tf_horizon=2.0, tf_interval=1.0, n_iterations=2)
    before = M.launch_count()
    traj, plans = scp.run_segments(y0, n_segments=2, atmosphere=atmo)
    assert M.launch_count() - before == 2 * (2 * 2 + 1)
    assert traj.shape == (256, 7, 200) and np.all(np.isfinite(traj))
    u_tab = plans[0][1].u_bar
    for s in (0, 100, 255):
        yr, _, st, _, _ = A.propagate_batch_rk45(y0[s:s + 1], 1.0, const, A.C.CTRL_SEQUENCE, table=u_tab[s], end_tau=2.0,
                                                 include_J2=True, T=100, atmosphere=atmo)
        assert st[0] == 0 and rel_err(traj[s, :, :100], yr[0]) < 2e-12, rel_err(traj[s, :, :100], yr[0])


def test_units_constellation_from_400_to_20000_km(M):
    """each satellite in its own constants under the exponential model: the C oracle on that satellite alone, and the
    drag's effect follows its own altitude (large at 400 km, nil at 20,000 km)"""
    import atmo_oracle as A
    atmo = fitted(exponential, 200e3, 40000e3)
    y0, consts = _exp_constellation()
    ctrl = M.ConstantTangentialThrustController(tangential_thrust=0.02)
    steps = np.zeros(6, np.int32)
    y, _, _, st = M.propagate_batch(y0, 0.5, ctrl, consts, T=40, n_steps=steps, atmosphere=atmo)
    y_nd, _, _, _ = M.propagate_batch(y0, 0.5, ctrl, consts, T=40, include_drag=False)
    assert st.max() == 0
    for s in range(6):
        yc, _, stc, acc, rej = A.propagate_batch_rk45(y0[s:s + 1], 0.5, consts[s], A.C.CTRL_TANGENTIAL, (0.02, 0, 0),
                                                      include_J2=True, T=40, atmosphere=atmo)
        assert stc[0] == 0 and steps[s] == acc[0] + rej[0] and rel_err(y[s], yc[0]) <= 5e-12, s
    effect = [rel_err(y[s], y_nd[s]) for s in range(6)]
    assert effect[0] > 1e-7 and effect[1] < 1e-15, effect       # 400 km / 20,000 km perigee


def test_out_of_range_flight_raises(M):
    atmo = fitted(power_law, 300e3, 1000e3)
    y0, const = leo((400e3, 250e3, 600e3))
    with pytest.raises(ValueError, match=r"satellite 1: .*\[300000, 1e\+06\] m"):
        M.propagate_batch(y0, 0.5, M.Controller(), const, T=20, atmosphere=atmo)
    _, _, _, st = M.propagate_batch(y0, 0.5, M.Controller(), const, T=20, atmosphere=atmo, check=False)
    assert st.tolist() == [0, M._lib.ST_ATMO, 0]
