"""Per-satellite designer units on the B200: a constellation that mixes altitudes and masses, each satellite in the
units of its own SatelliteScale, through one launch per leg.  Satellite s must come out bit for bit as a launch of the
same kernel under its own constants alone (the whole batch under consts[s], block s kept).  Batch sizes come from the
launch thresholds of mpc_b200.cu so that every launch branch runs once."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

# mpc_b200.cu: pair kernel in 128-thread CTAs for 148*32 < n <= 148*128 intervals, one-warp CTAs below 148*9*32*2,
# 128-thread CTAs above; the default-mode kernel in one-warp CTAs below 148*256 intervals
PAIR_BAND, PAIR_BIG, DEFAULT_BIG = 148 * 32, 148 * 9 * 32 * 2, 148 * 256


def _mixed(n):
    """n satellites over the six scales of mixed_constellation: satellite s has the constants of scale s % 6 (its speed
    varied slightly), so that one launch of the batch under consts[c] is the reference of every satellite s % 6 == c"""
    from test_units_kernel_source_on_host import mixed_constellation
    y6, c6 = mixed_constellation(6)
    y0 = y6[np.arange(n) % 6].copy()
    y0[:, 3:6] *= (1 + 1e-3 * np.arange(n) / max(n, 1))[:, None]
    return y0, [c6[s % 6] for s in range(n)]


@pytest.fixture(scope="module")
def M():
    import mpconstellation_b200 as M
    from mpconstellation_b200 import _lib
    _lib.require_gpu()
    return M


def _traj(M, y0, consts, K, tf=0.3):
    x, u, _, st = M.propagate_batch(y0, tf, M.ConstantTangentialThrustController(tangential_thrust=0.05), consts,
                                    include_drag=False, include_J2=False, T=K)
    assert (st == 0).all()
    return np.ascontiguousarray(x), np.ascontiguousarray(u)


def _no_group(M):
    from mpconstellation_b200 import _lib
    assert _lib.lib().mpc_set_tuning(23) == 0      # the rectangular reference takes the pair kernel, as _units does


def _group_back(M):
    from mpconstellation_b200 import _lib
    assert _lib.lib().mpc_set_tuning(24) == 0


def _kernels(fn):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return " ".join(e.key for e in prof.key_averages())


@pytest.mark.parametrize("n_int, adaptive, kernel", [
    (600, False, "discretize_pair_kernel<false, 32, 255, 1, true, true>"),
    (PAIR_BAND + 1000, False, "discretize_pair_kernel<false, 128, 255, 1, true, true>"),
    (PAIR_BIG + 1000, False, "discretize_pair_kernel<false, 128, 255, 1, true, true>"),
    (600, True, "discretize_default_units_kernel<false, 32, false>"),
    (DEFAULT_BIG + 1000, True, "discretize_default_units_kernel<false, 256, false>"),
])
def test_units_discretize_rectangular(M, n_int, adaptive, kernel):
    K = 60
    N = -(-n_int // (K - 1))
    y0, consts = _mixed(N)
    x, u = _traj(M, y0, consts, K)
    ad = dict(rtol=1e-3, atol=1e-6, max_step=1e-2) if adaptive else None
    xd, ud, tfd = (torch.as_tensor(a).cuda() for a in (x, u, np.full(N, 0.3)))
    names = _kernels(lambda: M.discretize_batch_device(xd, ud, tfd, consts, adaptive=ad))
    assert kernel in names
    before = M.launch_count()
    out, st = M.discretize_batch_device(xd, ud, tfd, consts, adaptive=ad)
    torch.cuda.synchronize()
    assert M.launch_count() - before == 1
    host = M.discretize_batch(x, u, 0.3, consts, adaptive=ad)
    assert np.array_equal(out.cpu().numpy(), host.soa) and np.array_equal(st.cpu().numpy().reshape(N, K - 1), host.status)
    got = out.cpu().numpy().reshape(105, N, K - 1)
    _no_group(M)
    try:
        for c in range(6):
            ref, rst = M.discretize_batch_device(xd, ud, tfd, consts[c], adaptive=ad)
            ref = ref.cpu().numpy().reshape(105, N, K - 1)
            idx = np.arange(c, N, 6)
            assert np.array_equal(got[:, idx], ref[:, idx]), c
    finally:
        _group_back(M)


@pytest.mark.parametrize("adaptive", [False, True])
def test_units_discretize_ragged(M, adaptive):
    N, Kmax = 300, 60
    y0, consts = _mixed(N)
    K_sat = np.array([2 + (7 * s) % (Kmax - 1) for s in range(N)], np.int32)
    K_sat[0] = Kmax
    x, u = _traj(M, y0, consts, Kmax)
    ad = dict(rtol=1e-3, atol=1e-6, max_step=1e-2) if adaptive else None
    res = M.discretize_batch(x, u, 0.3, consts, adaptive=ad, K=K_sat)
    for c in range(6):
        ref = M.discretize_batch(x, u, 0.3, consts[c], adaptive=ad, K=K_sat)
        for s in range(c, N, 6):
            assert all(np.array_equal(a, b) for a, b in zip(res.sat(s), ref.sat(s))), s


@pytest.mark.parametrize("ragged", [False, True])
def test_units_rk45(M, ragged):
    N, T = 600, 60
    y0, consts = _mixed(N)
    T_arg = np.array([2 + (5 * s) % (T - 1) for s in range(N)], np.int32) if ragged else T
    ctrl = M.ConstantTangentialThrustController(tangential_thrust=0.05)
    y0d, tfd = torch.as_tensor(y0).cuda(), torch.full((N,), 0.5, dtype=torch.float64, device="cuda")
    names = _kernels(lambda: M.propagate_batch_device(y0d, tfd, ctrl, consts, include_drag=True, include_J2=True, T=T_arg))
    assert "propagate_rk45_kernel<32, 2, true, true, true, true, true>" in names
    steps = np.zeros(N, np.int32)
    before = M.launch_count()
    y, u, _, st = M.propagate_batch(y0, 0.5, ctrl, consts, T=T_arg, n_steps=steps)
    assert M.launch_count() - before == 1 and (st == 0).all()
    yd, ud, _ = M.propagate_batch_device(y0d, tfd, ctrl, consts, T=T_arg)
    if not ragged:       # (the device form leaves the padding of a ragged batch unwritten)
        assert np.array_equal(yd.cpu().numpy(), y) and np.array_equal(ud.cpu().numpy(), u)
    for c in range(6):
        rs = np.zeros(N, np.int32)
        yr, ur, _, _ = M.propagate_batch(y0, 0.5, ctrl, consts[c], T=T_arg, n_steps=rs)
        idx = np.arange(c, N, 6)
        assert np.array_equal(y[idx], yr[idx], equal_nan=True) and np.array_equal(u[idx], ur[idx], equal_nan=True), c
        assert np.array_equal(steps[idx], rs[idx])


@pytest.mark.parametrize("ragged", [False, True])
def test_units_constraint_terms(M, ragged):
    N, K = 300, 30
    y0, consts = _mixed(N)
    x, u = _traj(M, y0, consts, K)
    K_sat = np.array([2 + (3 * s) % (K - 1) for s in range(N)], np.int32) if ragged else None
    before = M.launch_count()
    got = M.constraint_terms_batch(x, u, consts, K=K_sat)
    assert M.launch_count() - before == 1
    r, ub, f = M.constraint_terms_device(torch.as_tensor(x).cuda(), torch.as_tensor(u).cuda(), consts, K=K_sat)
    if not ragged:
        assert np.array_equal(r.cpu().numpy(), got["rbar_hat"]) and np.array_equal(ub.cpu().numpy(), got["ubar_hat"])
    for c in range(6):
        ref = M.constraint_terms_batch(x, u, consts[c], K=K_sat)   # (one launch of the batch under scale c)
        idx = np.arange(c, N, 6)
        for key in got:
            assert np.array_equal(got[key][idx], ref[key][idx], equal_nan=True), (c, key)


@pytest.mark.parametrize("tf", ["equal", "differing"])
def test_units_batched_scp_plan_matches_single_satellite_plans(M, tf):
    from mpconstellation_b200.scp import BatchedSCP, hold_reference_solver
    N = 6
    y0, consts = _mixed(N)
    horizons = np.full(N, 0.6) if tf == "equal" else np.array([0.6, 0.5, 0.7, 0.4, 0.6, 0.55])
    plans = []

    def solver(lin):
        u, _ = hold_reference_solver(lin)
        return u, horizons.copy()
    scp = BatchedSCP(consts, base_res=40, tf_horizon=0.6, n_iterations=2)
    before = M.launch_count()
    tab, tf_u, hist = scp.plan(y0, solver)
    assert M.launch_count() - before == 2 * 2          # one propagation and one discretization launch per pass
    for s in range(N):
        one = BatchedSCP(consts[s], base_res=40, tf_horizon=0.6, n_iterations=2)
        t1, tf1, h1 = one.plan(y0[s:s + 1], lambda lin, s=s: (hold_reference_solver(lin)[0], horizons[s:s + 1].copy()))
        k = t1.shape[2]
        assert np.array_equal(tab[s, :, :k], t1[0]) and tf_u[s] == tf1[0]
        for a, b in zip(hist, h1):
            assert all(np.array_equal(p, q) for p, q in zip(a.sat(s), b.sat(0)))
        plans.append(t1)
    lin = hist[-1]
    terms = M.constraint_terms_batch(lin.x_bar, lin.u_bar, lin.const, K=lin.K)
    for s in range(N):
        k = int(lin.K[s])
        one = M.constraint_terms_batch(lin.x_bar[s:s + 1, :, :k], lin.u_bar[s:s + 1, :, :k], consts[s])
        assert all(np.array_equal(np.asarray(terms[key])[s][..., :np.shape(one[key])[-1]] if np.ndim(one[key]) > 1 else terms[key][s],
                                  one[key][0]) for key in one)
