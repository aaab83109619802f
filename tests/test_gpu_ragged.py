"""GPU: ragged batches -- every satellite on its own node / sample count (K_s = int(base_res * tf_s)) through one
propagate and one discretize launch, against the rectangular entry points, per-satellite launches and the C oracle."""
import numpy as np
import pytest

from conftest import rel_err, synth_batch

pytestmark = pytest.mark.gpu

ADAPTIVE = dict(rtol=1e-3, atol=1e-6, max_step=1e-2)
GROUPS = ((0, 49), (49, 70), (70, 91), (91, 98), (98, 105))


@pytest.fixture(scope="module")
def M():
    import mpconstellation_b200 as m
    m._lib.require_gpu()
    return m


def _ragged_inputs(M, const, K_sat, tf, seed=3):
    """x, u [N,.,Kmax]: satellite s propagated on its own K_s samples (NaN past them), tangential seed law"""
    N = len(K_sat)
    y0, _, _ = synth_batch(N, 2, 1.0, const, seed=seed)
    ctrl = M.ConstantTangentialThrustController(tangential_thrust=0.5)
    x, u, t, st = M.propagate_batch(y0, tf, ctrl, const, include_drag=False, include_J2=False, T=K_sat)
    return y0, ctrl, np.array(x), np.array(u), t


def test_equal_counts_are_bit_identical_to_the_rectangular_entry_points(M, const):
    N, K = 64, 60                                   # 3776 intervals: the rectangular launch takes the pair kernel as well
    y0, _, _ = synth_batch(N, 2, 1.0, const)
    ctrl = M.ConstantTangentialThrustController(tangential_thrust=0.5)
    steps_r, steps_g = np.zeros(N, np.int32), np.zeros(N, np.int32)
    x, u, t, st = M.propagate_batch(y0, 1.4, ctrl, const, include_drag=False, include_J2=True, T=K, n_steps=steps_r)
    xg, ug, tg, stg = M.propagate_batch(y0, 1.4, ctrl, const, include_drag=False, include_J2=True, T=np.full(N, K),
                                        n_steps=steps_g)
    assert np.array_equal(x, xg) and np.array_equal(u, ug) and np.array_equal(steps_r, steps_g)
    assert tg.shape == (N, K) and np.array_equal(tg[7], t)
    for j2 in (False, True):
        for ad in (None, ADAPTIVE):
            r = M.discretize_batch(x, u, 1.4, const, include_J2=j2, adaptive=ad)
            g = M.discretize_batch(x, u, 1.4, const, include_J2=j2, adaptive=ad, K=np.full(N, K))
            assert np.array_equal(r.soa, g.soa) and np.array_equal(r.status, g.status)
            if ad is not None:
                assert np.array_equal(r.n_nodes, g.n_nodes)


@pytest.mark.parametrize("j2", [False, True])
def test_seeded_ragged_batch_matches_per_satellite_launches_and_the_oracle(M, const, j2):
    from oracle import c_oracle as C
    rng = np.random.default_rng(7 + j2)
    N = 64
    K_sat = rng.integers(20, 101, N).astype(np.int32)
    K_sat[0], K_sat[1] = 2, 100                     # the smallest grid and Kmax itself
    tf = 1.0 + rng.random(N)
    y0, ctrl, x, u, t = _ragged_inputs(M, const, K_sat, tf)
    Kmax = int(K_sat.max())
    for s in range(N):
        assert np.isnan(x[s, :, K_sat[s]:]).all() and np.isfinite(x[s, :, :K_sat[s]]).all()
        assert np.isnan(t[s, K_sat[s]:]).all() and t[s, K_sat[s] - 1] == 1.0
    # propagation: per-satellite rectangular launches, same steps
    steps = np.zeros(N, np.int32)
    M.propagate_batch(y0, tf, ctrl, const, include_drag=False, include_J2=False, T=K_sat, n_steps=steps)
    for s in (0, 1, 17, 40):
        st1 = np.zeros(1, np.int32)
        x1, u1, _, _ = M.propagate_batch(y0[s:s + 1], tf[s], ctrl, const, include_drag=False, include_J2=False,
                                         T=int(K_sat[s]), n_steps=st1)
        assert np.array_equal(x1[0], x[s, :, :K_sat[s]]) and np.array_equal(u1[0], u[s, :, :K_sat[s]])
        assert st1[0] == steps[s]
        yr, _, sr, _, _ = C.propagate_batch_rk45(y0[s:s + 1], tf[s], const, C.CTRL_TANGENTIAL, (0.5, 0, 0),
                                                 include_drag=False, include_J2=False, T=int(K_sat[s]))
        assert sr[0] == 0 and rel_err(x[s, :, :K_sat[s]], yr[0]) < 2e-12
    for ad in (ADAPTIVE, None):
        g = M.discretize_batch(x, u, tf, const, include_J2=j2, adaptive=ad, K=K_sat)
        assert g.soa.shape == (105, N * (Kmax - 1))
        for s in range(N):
            n = K_sat[s] - 1
            pad = g.soa[:, s * (Kmax - 1) + n:(s + 1) * (Kmax - 1)]
            assert np.isnan(pad).all() and (g.status[s, n:] == 0).all() and (g.status[s, :n] == 0).all()
        for s in (0, 1, 5, 33, 63):
            n = int(K_sat[s]) - 1
            xs, us = x[s:s + 1, :, :n + 1], u[s:s + 1, :, :n + 1]
            r = M.discretize_batch(xs, us, tf[s], const, include_J2=j2, adaptive=ad)
            got = g.soa[:, s * (Kmax - 1):s * (Kmax - 1) + n]
            # default mode: the same kernel build either way (one-warp CTAs): bit-identical.  Fixed-step mode: the one-
            # satellite launch takes the thread-group kernel, the ragged one the pair kernel: equal to rounding.
            if ad is not None:
                assert np.array_equal(got, r.soa) and np.array_equal(g.n_nodes[s, :n], r.n_nodes[0])
            else:
                for a, b in GROUPS:
                    assert rel_err(got[a:b], r.soa[a:b]) <= 1e-12
            mine = g.sat(s)
            assert [m.shape for m in mine] == [(n, 7, 7), (n, 7, 3), (n, 7, 3), (7, n), (7, n)]
            if n == 1:
                continue        # (one interval over the whole horizon: compared with the rectangular launch above only)
            # the C oracle, with the tolerances of the rectangular tests (test_gpu_discretize.py)
            if ad is not None:
                o = C.discretize_batch_adaptive(xs, us, tf[s], const, include_J2=j2)
                assert np.array_equal(g.n_nodes[s, :n], o[6][0])
            else:
                o = C.discretize_batch(xs, us, tf[s], const, include_J2=j2)
            for name_i in range(5):
                assert rel_err(mine[name_i], o[name_i][0]) < (1e-8 if ad is not None else 1e-10)


def test_ragged_device_entry_leaves_poisoned_padding_alone(M, const):
    import ctypes
    import torch
    K_sat = np.array([5, 12, 2, 9], np.int32)
    y0, ctrl, x, u, t = _ragged_inputs(M, const, K_sat, 1.3)
    N, Kmax = len(K_sat), int(K_sat.max())
    dev = torch.device("cuda")
    xd = torch.as_tensor(np.nan_to_num(x)).to(dev).contiguous()
    ud = torch.as_tensor(np.nan_to_num(u)).to(dev).contiguous()
    tfd = torch.full((N,), 1.3, dtype=torch.float64, device=dev)
    out = torch.full((105, N * (Kmax - 1)), float("nan"), dtype=torch.float64, device=dev)
    status = torch.full((N * (Kmax - 1),), 0, dtype=torch.int32, device=dev)
    first = torch.empty(N + 1, dtype=torch.int64, device=dev)
    p = M._lib.make_params(const, False, False)
    stream = torch.cuda.current_stream().cuda_stream
    M._lib.check(M._lib.lib().mpc_discretize_batch_ragged(
        xd.data_ptr(), ud.data_ptr(), tfd.data_ptr(), ctypes.byref(p), N, Kmax, K_sat.ctypes.data, first.data_ptr(), 0, 100,
        0.0, 0.0, 0.0, out.data_ptr(), N * (Kmax - 1), 0, status.data_ptr(), None, stream))
    torch.cuda.synchronize()
    o = out.cpu().numpy()
    ref = M.discretize_batch(x, u, 1.3, const, K=K_sat)
    assert np.array_equal(np.isnan(o), np.isnan(ref.soa))
    assert np.array_equal(o[~np.isnan(o)], ref.soa[~np.isnan(ref.soa)])
    assert np.array_equal(first.cpu().numpy(), np.concatenate([[0], np.cumsum(K_sat - 1)]))
    # invalid counts and the drag branch are rejected
    bad = np.array([5, 13, 2, 9], np.int32)
    rc = M._lib.lib().mpc_discretize_batch_ragged(
        xd.data_ptr(), ud.data_ptr(), tfd.data_ptr(), ctypes.byref(p), N, Kmax, bad.ctypes.data, first.data_ptr(), 0, 100,
        0.0, 0.0, 0.0, out.data_ptr(), N * (Kmax - 1), 0, status.data_ptr(), None, stream)
    assert rc == M._lib.E_INVALID
    pd = M._lib.make_params(const, False, True, disc_drag=(2.2, 4.0e4))
    rc = M._lib.lib().mpc_discretize_batch_ragged(
        xd.data_ptr(), ud.data_ptr(), tfd.data_ptr(), ctypes.byref(pd), N, Kmax, K_sat.ctypes.data, first.data_ptr(), 0, 100,
        0.0, 0.0, 0.0, out.data_ptr(), N * (Kmax - 1), 0, status.data_ptr(), None, stream)
    assert rc == M._lib.E_UNSUPPORTED


def test_per_satellite_table_lengths_match_the_oracle(M, const):
    from oracle import c_oracle as C
    y0, _, _ = synth_batch(5, 2, 1.0, const)
    rng = np.random.default_rng(5)
    lens = np.array([12, 4, 9, 2, 12], np.int32)
    tabs = np.zeros((5, 3, 12))
    for s in range(5):
        tabs[s, :, :lens[s]] = 0.2 * rng.standard_normal((3, lens[s]))
    spec = M.ControllerSpec(M._lib.CTRL_SEQUENCE, (0.0, 0.0, 0.0), tabs, 1.0, lens)
    T_sat = np.array([30, 41, 2, 17, 41], np.int32)
    y, u, t, st = M.propagate_batch(y0, 1.3, spec, const, include_drag=True, include_J2=True, T=T_sat)
    for s in range(5):
        yr, ur, sr, _, _ = C.propagate_batch_rk45(y0[s:s + 1], 1.3, const, C.CTRL_SEQUENCE, table=tabs[s, :, :lens[s]],
                                                  end_tau=1.0, include_drag=True, include_J2=True, T=int(T_sat[s]))
        assert sr[0] == 0 and rel_err(y[s, :, :T_sat[s]], yr[0]) < 2e-12 and rel_err(u[s, :, :T_sat[s]], ur[0]) < 1e-10
        assert np.isnan(y[s, :, T_sat[s]:]).all()
    # a rectangular T with per-satellite lengths runs the same kernel (all counts equal)
    y2, _, _, _ = M.propagate_batch(y0, 1.3, spec, const, include_drag=True, include_J2=True, T=41)
    assert np.array_equal(y2[[1, 4]], y[[1, 4]])
    with pytest.raises(ValueError):                # the fixed-step RK4 propagator takes no per-satellite lengths
        M.propagate_batch(y0, 1.3, spec, const, T=20, n_sub=4)


def test_batched_scp_with_differing_horizons_keeps_one_launch_per_leg(M, const):
    from mpconstellation_b200.scp import BatchedSCP
    N = 12
    y0, _, _ = synth_batch(N, 2, 1.0, const)
    tf_new = np.linspace(1.0, 2.0, N)

    def shrink(lin):                               # stand-in solver: the reference input, per-satellite horizons
        return np.array(lin.u_bar), tf_new.copy()

    def launches(solver, uniform):
        scp = BatchedSCP(const, base_res=30, tf_horizon=2.0, n_iterations=2, use_uniform_steps=uniform)
        before = M.launch_count()
        _, tf_u, hist = scp.plan(y0, solver)
        return M.launch_count() - before, hist

    n_equal, _ = launches(lambda lin: (np.array(lin.u_bar), np.full(N, 1.4)), False)
    n_ragged, hist = launches(shrink, False)
    assert n_ragged == n_equal == 4                 # 2 iterations x (propagate + discretize)
    # uniform mode: the first (rectangular) pass is the fused windowed one, the ragged pass two launches
    _, hist_u = launches(shrink, True)
    assert np.array_equal(hist_u[1].K, [int(30 * t) for t in tf_new]) and hist_u[1].matrices.status.max() == 0
    # the second linearization flies each satellite's own horizon on int(base_res * tf_s) nodes
    lin = hist[1]
    K_ref = np.array([int(30 * t) for t in tf_new])
    assert np.array_equal(lin.K, K_ref)
    for s in (0, 4, N - 1):
        A_k, B_kp, B_kn, Sigma_k, xi_k = lin.sat(s)
        assert A_k.shape == (K_ref[s] - 1, 7, 7) and Sigma_k.shape == (7, K_ref[s] - 1)
        alone = BatchedSCP(const, base_res=30, tf_horizon=2.0, n_iterations=2)
        ctrl = M.ControllerSpec(M._lib.CTRL_SEQUENCE, (0.0, 0.0, 0.0), hist[0].u_bar[s:s + 1, :, :hist[0].K[s]], 1.0)
        one = alone.linearize(y0[s:s + 1], tf_new[s:s + 1], ctrl)
        for a, b in zip(lin.sat(s), one.sat(0)):
            assert a.shape == b.shape and rel_err(a, b) <= 1e-12
        res = lin.dynamics_residual(s, lin.x_bar[s], lin.u_bar[s], tf_new[s])
        assert res.shape == (7, K_ref[s] - 1) and np.isfinite(res).all()
