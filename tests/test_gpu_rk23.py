"""Discretizer.ivp_solver = 'RK23' on the B200: the library's RK23 replay of the default quadrature mode against the
reference's own call, interval_matrices(ivp_solver="RK23") -- identical node counts (len(sol.t)) and the matrices to
1e-10 norm-relative -- on the cases of tests/test_rk23_kernel_source_on_host.py; ragged batches and a mixed
constellation in its own units bit for bit as single-satellite rectangular launches, in one-warp and full CTAs; the
status words; the device entry point against the host one; the RK45 dispatch unchanged."""
import numpy as np
import pytest

import orbit_sweep as O
from conftest import NAMES, rel_err, synth_batch
from test_rk23_kernel_source_on_host import TOL, _rejects, reference

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

DEFAULT_BIG = 148 * 256      # mpc_b200.cu: one-warp CTAs below this many intervals, 256-thread CTAs above


@pytest.fixture(scope="module")
def M():
    import mpconstellation_b200 as M
    from mpconstellation_b200 import _lib
    _lib.require_gpu()
    return M


def rk23(**kw):
    return dict(method="RK23", **kw)


def check(M, x, u, tf, const, j2, pairs, max_step=1e-2):
    res = M.discretize_batch(x, u, tf, const, include_J2=j2, adaptive=rk23(max_step=max_step))
    assert (res.status == 0).all()
    got = res.stacked()
    tfv = np.broadcast_to(np.asarray(tf, dtype=np.float64), (x.shape[0],))
    seen = []
    for s, k in pairs:
        ref, sol = reference(k, x[s], u[s], float(tfv[s]), const, j2, max_step)
        assert res.n_nodes[s, k] == len(sol.t), (s, k)
        for i, n in enumerate(NAMES):
            g = got[i][s, k] if i < 3 else got[i][s, :, k]
            assert rel_err(g, ref[i]) <= TOL, (s, k, n, rel_err(g, ref[i]))
        seen.append((len(sol.t), sol.nfev))
    return seen


def _eccentric(const, fac):
    el = O.sweep_elements()
    pick = np.flatnonzero((el["e"] >= 0.6) & (el["nu0"] >= 0))[::2]
    Y0 = O.kepler_states(const, **{k: v[pick] for k, v in el.items()})
    r = np.linalg.norm(Y0[:, 0:3], axis=1)
    tf = fac * 2 * np.pi * np.sqrt(r ** 3 / const.MU) * 3
    _, x, u = O.kepler_batch(const, 4, tf, "tangential", Y0=Y0)
    return x, u, tf


@pytest.mark.parametrize("j2", [False, True])
def test_against_the_reference(M, const, j2):
    _, x, u = synth_batch(2, 200, 2.0, const)
    check(M, x, u, 2.0, const, j2, [(s, k) for s in range(2) for k in (0, 1, 50, 123, 197, 198)])
    x, u, tf = _eccentric(const, 0.05)
    check(M, x, u, tf, const, j2, [(s, k) for s in range(x.shape[0]) for k in range(3)])
    _, x, u = synth_batch(2, 12, 0.5, const)
    u = u.copy()
    u[:, :, :6] = 0.0                                   # coast, then thrust: exactly-zero inputs
    check(M, x, u, 0.5, const, j2, [(s, k) for s in range(2) for k in range(11)])
    _, x, u = synth_batch(2, 5, 0.3, const)             # max_step binds
    seen = check(M, x, u, 0.3, const, j2, [(s, k) for s in range(2) for k in range(4)])
    assert min(n for n, _ in seen) >= 26


def test_rejected_steps(M, const):
    x, u, tf = _eccentric(const, 0.2)
    seen = check(M, x, u, tf, const, False, [(s, k) for s in range(x.shape[0]) for k in range(3)], max_step=1.0)
    assert any(_rejects(n, f) for n, f in seen)


def test_discretizer_honours_ivp_solver(M, const):
    """Discretizer.discretize / discretize_batch (ndarray and list inputs) with ivp_solver = 'RK23'"""
    _, x, u = synth_batch(3, 9, 0.4, const)

    def satellite_dynamics():
        pass
    d = M.Discretizer(const)
    d.ivp_solver = "RK23"
    one = d.discretize(satellite_dynamics, x[1], u[1], 0.4)
    for k in (0, 4, 7):
        ref, _ = reference(k, x[1], u[1], 0.4, const, False)
        for i in range(5):
            g = one[i][k] if i < 3 else one[i][:, k]
            assert rel_err(g, ref[i]) <= TOL
    K_s = [9, 4, 6]
    rag = d.discretize_batch(satellite_dynamics, [x[s, :, :k] for s, k in enumerate(K_s)],
                             [u[s, :, :k] for s, k in enumerate(K_s)], 0.4)
    for s, k in enumerate(K_s):
        alone = d.discretize(satellite_dynamics, x[s, :, :k], u[s, :, :k], 0.4)
        for a, b in zip(rag.sat(s), alone):
            assert np.array_equal(a, b)
    d.ivp_solver = "RK45"                               # the RK45 replay is still what the default gives
    r45 = d.discretize(satellite_dynamics, x[1], u[1], 0.4)
    ref45 = M.discretize_batch(x[1:2], u[1:2], 0.4, const, adaptive=dict(rtol=1e-3, atol=1e-6, max_step=1e-2)).sat(0)
    for a, b in zip(r45, ref45):
        assert np.array_equal(a, b)
    assert max(rel_err(a, b) for a, b in zip(one, r45)) > 1e-7      # RK23 is not RK45


def _single(M, x, u, tf, c, j2):
    return M.discretize_batch(np.ascontiguousarray(x[None]), np.ascontiguousarray(u[None]), tf, c, include_J2=j2,
                              adaptive=rk23(), check=False)


@pytest.mark.parametrize("big", [False, True])
def test_ragged_and_units_bit_identical_to_single_launches(M, const, big):
    """K_s from node_counts over tf_s in [1, 2]; a mixed constellation in its own units (model.sat_units): every
    satellite bit for bit a rectangular single-constant RK23 launch on it alone.  big: above the 256-thread CTA threshold."""
    from mpconstellation_b200.scp import node_counts
    from test_units_kernel_source_on_host import mixed_constellation
    rng = np.random.default_rng(3)
    N = 700 if big else 9
    base_res = 40
    tfs = rng.uniform(1.0, 2.0, N)
    K_sat = node_counts(base_res, tfs)
    Kmax = int(K_sat.max())
    y6, c6 = mixed_constellation(6)
    consts = [c6[s % 6] for s in range(N)]
    y0 = y6[np.arange(N) % 6]
    x, u, _, st = M.propagate_batch(y0, tfs, M.ConstantTangentialThrustController(tangential_thrust=0.05), consts,
                                    include_drag=False, include_J2=False, T=Kmax)
    assert (st == 0).all()
    x, u = np.ascontiguousarray(x), np.ascontiguousarray(u)
    assert big == (int((K_sat - 1).sum()) >= DEFAULT_BIG)
    picks = range(N) if not big else list(range(0, N, 97)) + [N - 1]
    for j2 in (False, True):
        for cc in (consts[0], consts):
            res = M.discretize_batch(x, u, tfs, cc, include_J2=j2, adaptive=rk23(), K=K_sat, check=False)
            rect = M.discretize_batch(x, u, tfs, cc, include_J2=j2, adaptive=rk23(), check=False)
            for s in picks:
                k = int(K_sat[s])
                c = consts[s] if isinstance(cc, list) else cc
                one = _single(M, x[s, :, :k], u[s, :, :k], tfs[s], c, j2)
                cols = slice(s * (Kmax - 1), s * (Kmax - 1) + k - 1)
                assert np.array_equal(res.soa[:, cols], one.soa), (j2, s)
                assert np.array_equal(res.status.reshape(-1)[cols], one.status.reshape(-1))
                assert np.array_equal(res.n_nodes.reshape(-1)[cols], one.n_nodes.reshape(-1))
                full = _single(M, x[s], u[s], tfs[s], c, j2)
                assert np.array_equal(rect.soa[:, s * (Kmax - 1):(s + 1) * (Kmax - 1)], full.soa)
            # the device entry point: the same bits
            xd, ud = torch.as_tensor(x, device="cuda"), torch.as_tensor(u, device="cuda")
            tfd = torch.as_tensor(tfs, device="cuda")
            nn = torch.zeros(N * (Kmax - 1), dtype=torch.int32, device="cuda")
            out = torch.full((105, N * (Kmax - 1)), float("nan"), dtype=torch.float64, device="cuda")
            _, std = M.discretize_batch_device(xd, ud, tfd, cc, include_J2=j2, adaptive=rk23(), K=K_sat, out=out, n_nodes=nn)
            torch.cuda.synchronize()
            live = np.concatenate([np.arange(s * (Kmax - 1), s * (Kmax - 1) + int(K_sat[s]) - 1) for s in range(N)])
            o = out.cpu().numpy()
            assert np.array_equal(o[0:42][:, live], res.soa[0:42][:, live])     # (rows 42..48: filled by the host entry)
            assert np.array_equal(o[49:][:, live], res.soa[49:][:, live])
            assert np.array_equal(nn.cpu().numpy()[live], res.n_nodes.reshape(-1)[live])
            assert np.array_equal(std.cpu().numpy()[live], res.status.reshape(-1)[live])


def test_status_words(M, const):
    _, x, u = synth_batch(2, 4, 0.3, const)
    xm = x.copy()
    xm[0, 6, :] = 0.0
    with pytest.raises(Exception, match="INVALID SATELLITE MASS"):
        M.discretize_batch(xm, u, 0.3, const, adaptive=rk23())
    xn = x.copy()
    xn[1, 0, 1] = np.nan
    res = M.discretize_batch(xn, u, 0.3, const, adaptive=rk23(), check=False)
    st = res.status.reshape(-1)
    assert st[4] == 2 and (np.delete(st, 4) == 0).all()
    with pytest.raises(FloatingPointError):
        res.raise_on_error()


def test_rk45_dispatch_unchanged(M, const):
    """adaptive without a method and with method="RK45" take the unchanged RK45 launches, bit for bit"""
    _, x, u = synth_batch(40, 30, 0.5, const)
    a = M.discretize_batch(x, u, 0.5, const, adaptive=dict(rtol=1e-3, atol=1e-6, max_step=1e-2))
    b = M.discretize_batch(x, u, 0.5, const, adaptive=dict(rtol=1e-3, atol=1e-6, max_step=1e-2, method="RK45"))
    c = M.discretize_batch(x, u, 0.5, const, adaptive=dict(rtol=1e-3, atol=1e-6, max_step=1e-2, method="RK23"))
    assert np.array_equal(a.soa, b.soa) and np.array_equal(a.n_nodes, b.n_nodes)
    assert not np.array_equal(a.soa, c.soa)
