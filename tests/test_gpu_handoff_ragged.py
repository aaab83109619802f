"""GPU: the hand-off of a ragged batch (every satellite on its own K_s = int(base_res * tf_s) nodes) to the convex
subproblem -- constraint terms and the per-satellite sparse dynamics constraint, one launch each -- against the host build
of the same kernel sources, the rectangular library calls per satellite, and through the device-tensor chain
propagate -> discretize -> constraint terms -> Jacobian."""
import numpy as np
import pytest

import test_handoff_ragged_on_host as H

pytestmark = pytest.mark.gpu

ADAPTIVE = dict(rtol=1e-3, atol=1e-6, max_step=1e-2)
TOL = 5e-13                  # terminal terms vs the host build: a few 3x3 products, contracted by each compiler its own way


@pytest.fixture(scope="module")
def M():
    import mpconstellation_b200 as m
    m._lib.require_gpu()
    return m


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.int64)


def _fin(out):
    """the terminal block [N,32] back from the dict of constraint_terms_batch"""
    from mpconstellation_b200 import _lib
    N = out["Vc"].shape[0]
    fin = np.empty((N, 32))
    for key, (off, ln) in _lib.FINAL_TERM_LAYOUT.items():
        fin[:, off:off + max(ln, 1)] = out[key].reshape(N, -1)
    return fin


def _live_equal(a, b, K_sat, width):
    """bit-identity of the live columns k < K_s + width of two [N, rows, Kmax(-1)] arrays"""
    return all(np.array_equal(_bits(a[s, :, :k + width]), _bits(b[s, :, :k + width])) for s, k in enumerate(K_sat.tolist()))


def test_library_host_and_device_forms_are_the_host_build(M, const):
    import torch
    from mpconstellation_b200.batch import DiscretizedBatch
    from mpconstellation_b200.constraints import constraint_terms_batch, constraint_terms_device, dynamics_jacobian, \
        dynamics_jacobian_device
    K_sat = H._counts()
    N, Kmax = len(K_sat), int(K_sat.max())
    tf = np.linspace(1.0, 2.0, N)
    x, u = H._batch(const, K_sat, 1.3)
    hr, hu, hf = H.constraint_terms_ragged(H._lib(), x, u, K_sat, const.MU)
    out = constraint_terms_batch(x, u, const, K=K_sat)
    np.testing.assert_array_equal(out["rbar_hat"], hr)              # NaN in the same places: padding and 0/0
    np.testing.assert_array_equal(out["ubar_hat"], hu)
    assert _live_equal(out["rbar_hat"], hr, K_sat, -1) and _live_equal(out["ubar_hat"], hu, K_sat, 0)
    fin = _fin(out)
    assert np.isfinite(fin).all() and np.max(np.abs(fin - hf) / np.maximum(np.abs(hf), 1.0)) <= TOL
    xd, ud = torch.from_numpy(x).cuda(), torch.from_numpy(u).cuda()        # NaN in the padding: never read
    rb, ub, fd = constraint_terms_device(xd, ud, const, K=K_sat)
    assert _live_equal(rb.cpu().numpy(), hr, K_sat, -1) and _live_equal(ub.cpu().numpy(), hu, K_sat, 0)
    assert np.array_equal(_bits(fd.cpu().numpy()), _bits(fin))
    # the Jacobian has no arithmetic but signs: every bit and index of the host build, host and device forms
    soa = H._soa(const, x, u, K_sat, tf)
    hv, hc, hrhs = H.dynamics_jacobian_ragged(H._lib(), soa, N, Kmax, K_sat)
    jac = dynamics_jacobian(DiscretizedBatch(soa, np.zeros((N, Kmax - 1), np.int32), N, Kmax, K_sat=K_sat))
    assert np.array_equal(_bits(jac.values), _bits(hv.ravel())) and np.array_equal(jac.indices, hc.ravel())
    assert np.array_equal(_bits(jac.rhs), _bits(hrhs))
    v, c, r = dynamics_jacobian_device(torch.from_numpy(soa).cuda(), N, Kmax, K_sat=K_sat, with_indices=False)
    assert c is None and np.array_equal(_bits(v.cpu().numpy()), _bits(hv.ravel()))
    # invalid counts and a pitch that does not hold the batch are rejected
    bad = K_sat.copy()
    bad[3] = Kmax + 1
    with pytest.raises(M._lib.MpcError):
        M._lib.check(M._lib.lib().mpc_constraint_terms_ragged_host(M.batch._ctx(0), x.ctypes.data, u.ctypes.data, N, Kmax,
                                                                    bad.ctypes.data, const.MU, hr.ctypes.data,
                                                                    hu.ctypes.data, hf.ctypes.data))
    first = torch.empty(N + 1, dtype=torch.int64, device="cuda")
    sd = torch.from_numpy(soa).cuda()
    rc = M._lib.lib().mpc_dynamics_jacobian_ragged(sd.data_ptr(), N * (Kmax - 1) - 1, 0, N, Kmax, K_sat.ctypes.data,
                                                   first.data_ptr(), v.data_ptr(), None, r.data_ptr(), None)
    assert rc == M._lib.E_INVALID


def test_batched_scp_pass_at_config5_shape_hands_off_in_one_launch_each(M, const):
    from conftest import synth_batch
    from mpconstellation_b200.batch import DiscretizedBatch
    from mpconstellation_b200.constraints import constraint_terms_batch, dynamics_jacobian, get_constraint_terms
    from mpconstellation_b200.scp import BatchedSCP
    N = 256
    y0, _, _ = synth_batch(N, 2, 1.0, const)
    tf_new = np.linspace(1.0, 2.0, N)
    scp = BatchedSCP(const, base_res=30, tf_horizon=2.0, n_iterations=2)
    _, _, hist = scp.plan(y0, lambda lin: (np.array(lin.u_bar), tf_new.copy()))
    lin = hist[1]
    K_sat = lin.K
    Kmax = int(K_sat.max())
    assert lin.matrices.K_sat is not None and len(np.unique(K_sat)) > 1
    n0 = M.launch_count()
    ct = constraint_terms_batch(lin.x_bar, lin.u_bar, const, K=lin.K)
    n1 = M.launch_count()
    jac = dynamics_jacobian(lin.matrices, K=lin.K)
    n2 = M.launch_count()
    assert n1 - n0 == 1 and n2 - n1 == 1
    assert np.isfinite(_fin(ct)).all() and np.isfinite(jac.values).all() and np.isfinite(jac.rhs).all()
    for s, k in enumerate(K_sat.tolist()):
        assert np.isfinite(ct["rbar_hat"][s, :, :k - 1]).all() and np.isfinite(ct["ubar_hat"][s, :, :k]).all()
    fin = _fin(ct)
    for s in (0, 1, 77, 128, 200, N - 1):
        k = int(K_sat[s])
        one = constraint_terms_batch(lin.x_bar[s:s + 1, :, :k], lin.u_bar[s:s + 1, :, :k], const)
        assert np.array_equal(_bits(ct["rbar_hat"][s, :, :k - 1]), _bits(one["rbar_hat"][0]))
        assert np.array_equal(_bits(ct["ubar_hat"][s, :, :k]), _bits(one["ubar_hat"][0]))
        assert np.array_equal(_bits(fin[s]), _bits(_fin(one)[0]))
        n = k - 1
        soa_s = np.ascontiguousarray(lin.matrices.soa[:, s * (Kmax - 1):s * (Kmax - 1) + n])
        rect = dynamics_jacobian(DiscretizedBatch(soa_s, np.zeros((1, n), np.int32), 1, k))
        rows, cols = jac.block(s)
        assert np.array_equal(_bits(jac.values.reshape(-1, 16)[rows]), _bits(rect.values.reshape(-1, 16)))
        assert np.array_equal(jac.indices.reshape(-1, 16)[rows], rect.indices.reshape(-1, 16) + cols.start)
        assert np.array_equal(_bits(jac.rhs[rows]), _bits(rect.rhs))
    # the optimizer's list form: one ragged launch, per-satellite widths
    n0 = M.launch_count()
    lists = get_constraint_terms([lin.x_bar[s, :, :k] for s, k in enumerate(K_sat.tolist())],
                                 [lin.u_bar[s, :, :k] for s, k in enumerate(K_sat.tolist())], const)
    assert M.launch_count() - n0 == 1
    assert lists["rbar_hat"][9].shape == (3, K_sat[9] - 1) and lists["ubar_hat"][9].shape == (3, K_sat[9])
    assert np.array_equal(lists["DrVn_DvVn"][9], ct["DrVn_DvVn"][9]) and lists["Vc"][9] == ct["Vc"][9]
    # the first (rectangular) pass with its counts: the per-satellite form of the same numbers
    lin0 = hist[0]
    j0 = dynamics_jacobian(lin0.matrices, K=lin0.K)
    jr = dynamics_jacobian(lin0.matrices)
    assert j0.K_sat is not None and j0.rows == jr.rows and j0.cols == jr.cols + N - 1
    assert np.array_equal(_bits(j0.values), _bits(jr.values)) and np.array_equal(_bits(j0.rhs), _bits(jr.rhs))


def test_device_chain_stays_in_hbm_and_gives_the_host_forms_bits(M, const):
    import torch
    from conftest import synth_batch
    from mpconstellation_b200.constraints import constraint_terms_batch, constraint_terms_device, dynamics_jacobian, \
        dynamics_jacobian_device
    N = 96
    tf = np.linspace(1.0, 2.0, N)
    K_sat = np.array([int(30 * t) for t in tf], np.int32)
    Kmax = int(K_sat.max())
    y0, _, _ = synth_batch(N, 2, 1.0, const)
    ctrl = M.ConstantTangentialThrustController(tangential_thrust=0.5)
    x, u, _, _ = M.propagate_batch(y0, tf, ctrl, const, include_drag=False, include_J2=False, T=K_sat)
    x, u = np.array(x), np.array(u)
    mats = M.discretize_batch(x, u, tf, const, adaptive=ADAPTIVE, K=K_sat)
    ct = constraint_terms_batch(x, u, const, K=K_sat)
    jac = dynamics_jacobian(mats)
    dev = torch.device("cuda")
    y0d, tfd = torch.from_numpy(y0).to(dev), torch.from_numpy(tf).to(dev)
    n0 = M.launch_count()
    xd, ud, sp = M.propagate_batch_device(y0d, tfd, ctrl, const, include_drag=False, include_J2=False, T=K_sat)
    nodes = torch.zeros(N * (Kmax - 1), dtype=torch.int32, device=dev)
    out, sd = M.discretize_batch_device(xd, ud, tfd, const, adaptive=ADAPTIVE, n_nodes=nodes, K=K_sat)
    rb, ub, fd = constraint_terms_device(xd, ud, const, K=K_sat)
    v, c, r = dynamics_jacobian_device(out, N, Kmax, K_sat=K_sat)
    torch.cuda.synchronize()
    assert M.launch_count() - n0 == 4
    assert sp.max().item() == 0 and sd.max().item() == 0
    assert _live_equal(xd.cpu().numpy(), x, K_sat, 0) and _live_equal(ud.cpu().numpy(), u, K_sat, 0)
    o = out.cpu().numpy()
    for s, k in enumerate(K_sat.tolist()):
        cols = slice(s * (Kmax - 1), s * (Kmax - 1) + k - 1)
        assert np.array_equal(_bits(o[:, cols]), _bits(mats.soa[:, cols]))
    assert np.array_equal(nodes.cpu().numpy().reshape(N, Kmax - 1), mats.n_nodes)
    assert _live_equal(rb.cpu().numpy(), ct["rbar_hat"], K_sat, -1) and _live_equal(ub.cpu().numpy(), ct["ubar_hat"], K_sat, 0)
    assert np.array_equal(_bits(fd.cpu().numpy()), _bits(_fin(ct)))
    assert np.array_equal(_bits(v.cpu().numpy()), _bits(jac.values)) and np.array_equal(c.cpu().numpy(), jac.indices)
    assert np.array_equal(_bits(r.cpu().numpy()), _bits(jac.rhs))


def test_profiler_names_the_ragged_kernels(M, const):
    import torch
    from torch.profiler import ProfilerActivity, profile
    from mpconstellation_b200.constraints import constraint_terms_device, dynamics_jacobian_device
    K_sat = np.array([5, 12, 2, 9], np.int32)
    N, Kmax = len(K_sat), int(K_sat.max())
    x = torch.rand((N, 7, Kmax), dtype=torch.float64, device="cuda") + 1.0
    u = torch.rand((N, 3, Kmax), dtype=torch.float64, device="cuda")
    soa = torch.rand((105, N * (Kmax - 1)), dtype=torch.float64, device="cuda")
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        constraint_terms_device(x, u, const, K=K_sat)
        dynamics_jacobian_device(soa, N, Kmax, K_sat=K_sat)
        torch.cuda.synchronize()
    names = " ".join(e.name for e in prof.events())
    assert "constraint_terms_kernel<true>" in names and "dynamics_jacobian_kernel<true>" in names, names[:2000]
