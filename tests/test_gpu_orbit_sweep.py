"""GPU: the eccentric / polar / retrograde sweep of orbit_sweep.py through the library, with batch sizes chosen so that
every launch branch of the fixed-step, default-mode and ragged discretizations runs once, against the extended-precision
101-node sums (fixed step) and the host build of the same kernel source (default mode).  The sample of intervals compared
includes the last interval of the batch and the intervals on both sides of CTA boundaries."""
import re

import numpy as np
import pytest

import hostk
import orbit_sweep as O
from conftest import rel_err
from test_orbit_sweep_on_host import TOL

pytestmark = pytest.mark.gpu

# launch branches of csrc/mpc_b200.cu for a 148-SM B200: launch_disc_n (fixed step, one destination), launch_adaptive_k
# (default mode) and launch_ragged
SMS = 148
GROUP_MAX = 2560                      # kGroupMaxIntervals: the 8-lanes-per-interval kernel up to here
BAND = (SMS * 32, SMS * 128)          # (4736, 18944]: the pair kernel in 128-thread CTAs, one per SM
WIDE = SMS * 9 * 32 * 2               # 85248: from here the production 128-thread pair kernel; below it one-warp CTAs
DEFAULT_WIDE = SMS * 256              # 37888: the default-mode kernels take 256-thread CTAs from here
HOST_CHUNK = SMS * 9 * 32             # chunk_sats: intervals per chunk of the host entry points (one launch each)
ADAPTIVE = dict(rtol=1e-3, atol=1e-6, max_step=1e-2)


@pytest.fixture(scope="module")
def M():
    import mpconstellation_b200 as m
    m._lib.require_gpu()
    return m


def _base(const, K):
    """the sweep under tangential and constant inertial thrust, intervals of 0.009 and 0.03 of the circular orbit at
    perigee (the 11- and the 51-node forms) and on both sides of the 51-node bound: 180 satellites"""
    Y0 = O.kepler_states(const, **O.sweep_elements())
    per = 2 * np.pi * np.sqrt(np.linalg.norm(Y0[:, 0:3], axis=1) ** 3 / const.MU)
    xs, us, tfs = [], [], []
    for law in ("tangential", "inertial"):
        for frac in (0.009, 0.03):
            tf = frac * per * (K - 1)
            _, x, u = O.kepler_batch(const, K, tf, law, Y0=Y0)
            xs.append(x), us.append(u), tfs.append(tf)
    _, x, u, tf = O.intervals_at_gate(const, K, "inertial")[("51", "out")]
    xs.append(x), us.append(u), tfs.append(tf)
    return np.concatenate(xs), np.concatenate(us), np.concatenate(tfs)


def _tiled(const, K, N):
    x, u, tf = _base(const, K)
    idx = np.arange(N) % x.shape[0]
    return np.ascontiguousarray(x[idx]), np.ascontiguousarray(u[idx]), np.ascontiguousarray(tf[idx])


def _sample(n_int, block, seed=0, n_rand=24):
    """seeded intervals, the last one and both sides of the first, a middle and the last CTA boundary"""
    rng = np.random.default_rng(seed)
    b = [block, (n_int // block // 2) * block, (n_int - 1) // block * block]
    cols = set(rng.integers(0, n_int, n_rand).tolist()) | {0, n_int - 1}
    for c in b:
        if 0 < c < n_int:
            cols |= {c - 1, c}
    return np.array(sorted(cols))


def _kernels(fn):
    """(kernel name, block) of the library's kernels launched by fn(), when torch.profiler reports them by name"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    names = [e.name for e in prof.events()]
    return out, {(m.group(1), int(m.group(2))) for n in names
                 for m in [re.search(r"(discretize_\w+?_kernel)<(?:true|false), (\d+)", n)] if m}


def _tuned(M, variants, fn):
    L = M._lib.lib()
    try:
        for v in variants:
            assert L.mpc_set_tuning(v) == 0
        return fn()
    finally:
        assert L.mpc_set_tuning(38) == 0 and L.mpc_set_tuning(40) == 0


def _check_fixed(M, const, x, u, tf, soa_of, block, expect_kernel, j2, K_sat=None):
    """soa_of(): SoA [105, pitch] of the batch, columns s (Kmax-1) + k.  Three settings: tiers on, 11-node form off
    (mpc_set_tuning(39)), every node evaluated (37); the sample against sums101_longdouble within its tier's tolerance"""
    N, _, K = x.shape
    Ks = np.full(N, K) if K_sat is None else K_sat
    live = np.concatenate([s * (K - 1) + np.arange(Ks[s] - 1) for s in range(N)])      # live index -> column
    cols = live[_sample(live.size, block)]
    s_idx, k_idx = cols // (K - 1), cols % (K - 1)
    ref = np.full((105, cols.size), np.nan)
    tier = np.zeros(cols.size, int)
    tier1 = np.zeros(cols.size, int)
    for Kg in np.unique(Ks[s_idx]):
        sel = Ks[s_idx] == Kg
        sats, inv = np.unique(s_idx[sel], return_inverse=True)
        xs, us = x[sats, :, :Kg], u[sats, :, :Kg]
        loc = inv * (Kg - 1) + k_idx[sel]
        ref[:, sel] = O.to_soa(O.sums101_longdouble(xs, us, tf[sats], const, j2, cols=loc))
        tier[sel] = O.tiers(xs, us, tf[sats], const).ravel()[loc]
        tier1[sel] = O.tiers(xs, us, tf[sats], const, em11=False).ravel()[loc]
    worst = {}
    for name, variants, t_of in (("on", (), tier), ("11 off", (39,), tier1), ("all nodes", (37,), np.zeros_like(tier))):
        (out, kern) = _tuned(M, variants, lambda: _kernels(soa_of))
        if kern:
            assert expect_kernel in kern, (expect_kernel, kern)
        got = out[:, cols]
        for t in np.unique(t_of):
            sel = t_of == t
            for grp, e in O.group_errors(got[:, sel], ref[:, sel]).items():
                assert e <= TOL[t][grp], (name, O.TIER_NAMES[t], grp, e)
                worst[(name, O.TIER_NAMES[t], grp)] = max(worst.get((name, O.TIER_NAMES[t], grp), 0.0), e)
    print(expect_kernel, kern, "J2" if j2 else "", " ".join(f"{k}={v:.1e}" for k, v in sorted(worst.items())))
    return worst


def _host_call(M, const, j2, K_sat=None):
    def run(x, u, tf):
        return lambda: M.discretize_batch(x, u, tf, const, include_J2=j2, K=K_sat).soa
    return run


@pytest.mark.parametrize("j2", [False, True])
@pytest.mark.parametrize("n_int,block,kernel", [
    (GROUP_MAX - 40, 32, ("discretize_group_kernel", 32)),
    (BAND[0] - 136, 32, ("discretize_pair_kernel", 32)),
    (BAND[1] - 144, 128, ("discretize_pair_kernel", 128)),
])
def test_fixed_step_launch_branches_through_the_host_entry(M, const, j2, n_int, block, kernel):
    K = 9
    x, u, tf = _tiled(const, K, n_int // (K - 1))
    assert (n_int <= GROUP_MAX) == (kernel[0] == "discretize_group_kernel") and (n_int > BAND[0]) == (block == 128)
    _check_fixed(M, const, x, u, tf, _host_call(M, const, j2)(x, u, tf), block, kernel, j2)


def test_fixed_step_wide_launch_through_the_device_entry(M, const):
    """one launch of >= 85,248 intervals (the host entry points cut batches into chunks of 42,624): the production
    128-thread pair kernel"""
    import torch
    K = 9
    N = (WIDE + 8 * 128) // (K - 1)
    x, u, tf = _tiled(const, K, N)
    assert N * (K - 1) >= WIDE
    dx, du, dtf = (torch.from_numpy(a).cuda() for a in (x, u, tf))

    def run():
        out, st = M.discretize_batch_device(dx, du, dtf, const, include_J2=True)
        assert int(st.max()) == 0
        return out.cpu().numpy()
    _check_fixed(M, const, x, u, tf, run, 128, ("discretize_pair_kernel", 128), True)


@pytest.mark.parametrize("j2", [False, True])
def test_ragged_pair_kernel_in_the_128_thread_band(M, const, j2):
    K = 41
    N = 360
    x, u, tf = _tiled(const, K, N)
    K_sat = np.random.default_rng(5).integers(20, K + 1, N).astype(np.int32)
    K_sat[-1] = K
    tf = tf * (K_sat - 1) / (K - 1)                  # every satellite keeps the interval length of its tier
    live = int((K_sat - 1).sum())
    assert BAND[0] < live <= BAND[1]
    _check_fixed(M, const, x, u, tf, _host_call(M, const, j2, K_sat)(x, u, tf), 128, ("discretize_pair_kernel", 128), j2,
                 K_sat=K_sat)


def _check_default(M, const, run, x, u, tf, block, kernel, K_sat=None, j2=False):
    N, _, K = x.shape
    (res, kern) = _kernels(run)
    if kern:
        assert kernel in kern, (kernel, kern)
    soa, nodes = res
    Ks = np.full(N, K) if K_sat is None else K_sat
    live = np.concatenate([s * (K - 1) + np.arange(Ks[s] - 1) for s in range(N)])
    cols = live[_sample(live.size, block, n_rand=16)]
    sats = np.unique(cols // (K - 1))
    for s in sats:
        Kg = int(Ks[s])
        out, st, nn = hostk.discretize_adaptive(x[s:s + 1, :, :Kg], u[s:s + 1, :, :Kg], tf[s], const, include_J2=j2, **ADAPTIVE)
        assert st.max() == 0
        c = s * (K - 1) + np.arange(Kg - 1)
        assert np.array_equal(nodes[c], nn)
        assert rel_err(soa[:, c], out) <= 1e-12, s


@pytest.mark.parametrize("n_int,block,kernel", [(DEFAULT_WIDE - 888, 32, ("discretize_default_kernel", 32)),
                                                (DEFAULT_WIDE + 1112, 256, ("discretize_default_kernel", 256))])
def test_default_mode_launch_branches(M, const, n_int, block, kernel):
    import torch
    K = 9
    x, u, tf = _tiled(const, K, n_int // (K - 1))
    dx, du, dtf = (torch.from_numpy(a).cuda() for a in (x, u, tf))

    def run():
        nn = torch.zeros(dx.shape[0] * (K - 1), dtype=torch.int32, device="cuda")
        out, st = M.discretize_batch_device(dx, du, dtf, const, include_J2=True, adaptive=ADAPTIVE, n_nodes=nn)
        assert int(st.max()) == 0
        return out.cpu().numpy(), nn.cpu().numpy()
    _check_default(M, const, run, x, u, tf, block, kernel, j2=True)


def test_ragged_default_mode_in_256_thread_ctas(M, const):
    """a ragged batch with >= 37,888 live intervals in one chunk of the host entry point"""
    K = 49
    N = HOST_CHUNK // (K - 1)
    x, u, tf = _tiled(const, K, N)
    K_sat = np.full(N, K, dtype=np.int32)
    K_sat[::10] = 25
    tf = tf * (K_sat - 1) / (K - 1)
    live = int((K_sat - 1).sum())
    assert live >= DEFAULT_WIDE and N * (K - 1) <= HOST_CHUNK

    def run():
        r = M.discretize_batch(x, u, tf, const, adaptive=ADAPTIVE, K=K_sat)
        return r.soa, r.n_nodes.ravel()
    _check_default(M, const, run, x, u, tf, 256, ("discretize_default_ragged_kernel", 256), K_sat=K_sat)


def test_rk45_propagation_of_the_sweep(M, const):
    """the RK45 replay on the sweep's eccentric orbits with steps long enough to be rejected: the attempted steps of the
    C oracle's replica and its states to 5e-12, rectangular and ragged (measured on a B200: 2.8e-12 -- the device
    contracts to FMA where the C replica does not, and 0.2-long steps carry that further than the reference's 1e-3; the
    host build, contracted like the device, agrees with scipy itself to 1e-12, test_orbit_sweep_on_host.py)"""
    from oracle import c_oracle as C
    Y0 = O.kepler_states(const, **O.sweep_elements())
    tf, T = 3.0, 40
    o = dict(rtol=1e-3, atol=1e-6, max_step=0.2)
    ctrl = M.ConstantTangentialThrustController(tangential_thrust=0.02)
    steps = np.zeros(len(Y0), np.int32)
    y, _, _, st = M.propagate_batch(Y0, tf, ctrl, const, include_drag=False, include_J2=True, T=T, rk45=o, n_steps=steps)
    yc, _, stc, acc, rej = C.propagate_batch_rk45(Y0, tf, const, C.CTRL_TANGENTIAL, (0.02, 0, 0), include_drag=False,
                                                   include_J2=True, T=T, max_step=0.2)
    assert st.max() == 0 and stc.max() == 0 and rej.max() > 0
    assert np.array_equal(steps, acc + rej)
    assert rel_err(y, yc) <= 5e-12
    T_sat = np.random.default_rng(1).integers(2, T + 1, len(Y0)).astype(np.int32)
    steps_r = np.zeros(len(Y0), np.int32)
    yr, _, _, _ = M.propagate_batch(Y0, tf, ctrl, const, include_drag=False, include_J2=True, T=T_sat, rk45=o,
                                    n_steps=steps_r)
    assert np.array_equal(steps_r, steps)
    for s in range(len(Y0)):
        ys, _, _, _, _ = C.propagate_batch_rk45(Y0[s:s + 1], tf, const, C.CTRL_TANGENTIAL, (0.02, 0, 0), include_drag=False,
                                                include_J2=True, T=int(T_sat[s]), max_step=0.2)
        assert rel_err(yr[s, :, :T_sat[s]], ys[0]) <= 5e-12, s
