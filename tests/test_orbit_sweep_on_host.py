"""The host build of the fixed-step, default-mode and RK45 kernels on eccentric (e up to 0.8, perigee 2-5 % of R_E above
the surface), equatorial, polar and retrograde orbits, against an extended-precision reference of the same operation
(orbit_sweep.sums101_longdouble) and the reference's own scipy calls.  Every interval is checked against the tolerance of
the form of the sums it takes (11-, 21-, 51- or all 101 nodes), with the form taken read off the gate quantities and
confirmed by bit-identity with the launches that switch the shorter forms off."""
import numpy as np
import pytest

import hostk
import orbit_sweep as O
from conftest import NAMES, rel_err, synth_batch
from oracle import c_oracle as C
from test_11_node_rule import discretize as disc_em, discretize_group as group_em

# Norm-relative error per row group against the 101-node sums of the exact flow, by the form of the sums an interval
# takes, for e <= 0.8 with and without J2 (measured maxima at the gate edges on the host build: 11-node 3.4e-13 /
# 4.4e-14 / 2.7e-14 / 5.4e-14, 21-node 1.7e-11 / 6.7e-13 / 4.5e-13 / 9.2e-13, 51-node 5.0e-11 / 4.2e-12 / 3.4e-12 /
# 6.8e-12, all 101 nodes with the Hermite midpoint 1.3e-11 / 2.2e-12 / 1.6e-11 / 4.0e-12).  The gate bounds the
# circular rate at the start node; at perigee the angular rate is sqrt(1 + e) times that, so eccentric orbits sit
# closer to each tier's limit than the Hubble family does (include/mpc_b200.h, mpc_discretize_batch).
TOL = {O.TIER_11: {"A_k": 1e-12, "B_pm": 1e-13, "Sigma": 1e-13, "xi": 1.5e-13},
       O.TIER_21: {"A_k": 4e-11, "B_pm": 1.5e-12, "Sigma": 1e-12, "xi": 2e-12},
       O.TIER_51: {"A_k": 1e-10, "B_pm": 1e-11, "Sigma": 8e-12, "xi": 1.5e-11},
       O.TIER_ALL: {"A_k": 3e-11, "B_pm": 5e-12, "Sigma": 4e-11, "xi": 1e-11}}


def _perigee_period(const, Y0):
    r = np.linalg.norm(Y0[:, 0:3], axis=1)
    return 2 * np.pi * np.sqrt(r ** 3 / const.MU)


def check_tiers_and_errors(x, u, tf, const, j2, ref=None):
    """pair kernel with the 11-node form on (em11), off (21/51-node forms only) and every node evaluated, group kernel
    with the 11-node form: the form per interval from the gate quantities, confirmed bit for bit, and every launch within
    its tier's tolerance of sums101_longdouble.  Returns (tier [n], {tier: {group: max error}})."""
    a2, s2 = disc_em(x, u, tf, const, include_J2=j2, em11=True)
    a1, s1 = disc_em(x, u, tf, const, include_J2=j2)
    a0, s0 = disc_em(x, u, tf, const, include_J2=j2, em=False)
    g2, sg = group_em(x, u, tf, const, include_J2=j2, em11=True)
    assert s2.max() == 0 and s1.max() == 0 and s0.max() == 0 and sg.max() == 0
    tier = O.tiers(x, u, tf, const).ravel()
    tier1 = O.tiers(x, u, tf, const, em11=False).ravel()
    same20, same21, same10 = np.all(a2 == a0, axis=0), np.all(a2 == a1, axis=0), np.all(a1 == a0, axis=0)
    assert np.array_equal(same20, tier == O.TIER_ALL)
    assert np.array_equal(same21, tier != O.TIER_11)
    assert np.array_equal(same10, tier1 == O.TIER_ALL)
    if ref is None:
        ref = O.to_soa(O.sums101_longdouble(x, u, tf, const, j2))
    worst = {}
    for out, t_of in ((a2, tier), (g2, tier), (a1, tier1), (a0, np.full_like(tier, O.TIER_ALL))):
        for t in np.unique(t_of):
            sel = t_of == t
            for grp, e in O.group_errors(out[:, sel], ref[:, sel]).items():
                assert e <= TOL[t][grp], (O.TIER_NAMES[t], grp, e)
                w = worst.setdefault(t, {})
                w[grp] = max(w.get(grp, 0.0), e)
    return tier, worst


def test_reference_converges_and_agrees_with_the_c_oracle_on_the_hubble_family(const):
    """sums101_longdouble with m and 2m RK4 steps per panel agree to 1e-15 on the hardest intervals of the sweep (the
    outer edge of the 51-node gate at e = 0.8, J2 on); on the Hubble family the C oracle's fixed-step sums agree with it
    to 1e-12"""
    _, x, u, tf = O.intervals_at_gate(const, 3, "tangential")[("51", "out")]
    sel = np.arange(0, x.shape[0] * 2, 5)
    a = O.sums101_longdouble(x, u, tf, const, True, cols=sel, m=8)
    b = O.sums101_longdouble(x, u, tf, const, True, cols=sel, m=16)
    for p, q in zip(a, b):
        assert rel_err(p, q) <= 1e-15
    for j2 in (False, True):
        _, xh, uh = synth_batch(3, 5, 0.05, const)
        ref = O.sums101_longdouble(xh, uh, 0.05, const, j2)
        orc = C.discretize_batch(xh, uh, 0.05, const, include_J2=j2)
        assert orc[5].max() == 0
        for i, n in enumerate(NAMES):
            r = ref[i] if i < 3 else ref[i].T
            o = orc[i].reshape((-1,) + orc[i].shape[2:]) if i < 3 else orc[i].transpose(1, 0, 2).reshape(7, -1)
            assert rel_err(o, r) <= 1e-12, n


@pytest.mark.parametrize("law", O.LAWS)
@pytest.mark.parametrize("frac", [0.009, 0.03])
def test_fixed_step_kernels_on_the_sweep(const, law, frac):
    """the sweep's 36 satellites, 2 intervals each of `frac` of the circular orbit at perigee (the 11- and the 51-node
    forms on the near-circular orbits), with and without J2"""
    K = 3
    Y0 = O.kepler_states(const, **O.sweep_elements())
    tf = frac * _perigee_period(const, Y0) * (K - 1)
    _, x, u = O.kepler_batch(const, K, tf, law, Y0=Y0)
    if law in ("tangential", "radial"):                                 # in-plane: equatorial orbits keep z = 0
        assert np.all(x[O.sweep_elements()["inc"] == 0, 2] == 0.0)
    for j2 in (False, True):
        tier, _ = check_tiers_and_errors(x, u, tf, const, j2)
        assert np.mean(tier == (O.TIER_11 if frac < 0.011 else O.TIER_51)) > 0.5


@pytest.mark.parametrize("law", ["inertial", "tangential"])
def test_both_sides_of_every_orbital_threshold(const, law):
    """tf puts the start node of the first interval 1e-9 inside / outside each threshold: the expected form is taken on
    each side (constant inertial thrust is smooth everywhere; the tangential law turns with the orbit) and each side is
    within its form's tolerance, the interval that starts just after perigee included"""
    K = 3
    el = O.sweep_elements()
    expect = {("11/21", "in"): O.TIER_11, ("11/21", "out"): O.TIER_51, ("51", "in"): O.TIER_51,
              ("51", "out"): O.TIER_ALL, ("hermite", "in"): O.TIER_51, ("hermite", "out"): O.TIER_51}
    for (name, side), (Y0, x, u, tf) in O.intervals_at_gate(const, K, law).items():
        w = O.w2H2(x, tf, K, const)[:, 0]
        thr = {"11/21": O.ORBIT_11 / O.ORBIT_SCALE_11, "51": O.ORBIT_51, "hermite": O.ORBIT_HERMITE}[name]
        assert np.all(w <= thr) if side == "in" else np.all(w > thr)
        for j2 in (False, True):
            tier, _ = check_tiers_and_errors(x, u, tf, const, j2)
            first = tier.reshape(-1, K - 1)[:, 0]
            if law == "inertial":
                assert np.all(first == expect[(name, side)]), (name, side)
            else:
                assert np.all((first == expect[(name, side)]) | (first == O.TIER_ALL)), (name, side)
                assert np.any(first == expect[(name, side)])
            assert np.any((el["nu0"] > 0) & (first == expect[(name, side)]))
        if name == "hermite":
            # every node evaluated: two nodes per step inside the bound, one step per node outside it (the launch
            # without the two-node steps, discretize_kernel)
            a0, _ = disc_em(x, u, tf, const, em=False)
            p1, _ = hostk.discretize(x, u, tf, const, pair=False, em=False)
            f0 = np.all(a0 == p1, axis=0).reshape(-1, K - 1)[:, 0]
            assert np.all(~f0) if side == "in" else np.all(f0)


@pytest.mark.parametrize("bound", [O.SMOOTH_11, O.SMOOTH_21])
def test_both_sides_of_every_smoothness_threshold(const, bound):
    """input tables whose first interval changes by sqrt(bound) of the input's size, one ulp inside and one ulp outside:
    the 11-node form / the 21-node form / all 101 nodes as the gate says, each within its tolerance"""
    K, n = 6, 4
    Y0 = O.kepler_states(const, **O.sweep_elements())[::4][:2 * n]
    tf = 0.008 * _perigee_period(const, Y0) * (K - 1)
    _, x, _ = O.kepler_batch(const, K, tf, "inertial", Y0=Y0)
    u = O.smoothness_tables(K, bound, n)
    d2, m2 = O.smoothness(u)
    assert np.all(d2[:n, 0] <= bound * m2[:n, 0]) and np.all(d2[n:, 0] > bound * m2[n:, 0])
    for j2 in (False, True):
        tier, _ = check_tiers_and_errors(x, u, tf, const, j2)
        first = tier.reshape(-1, K - 1)[:, 0]
        inside, outside = (O.TIER_11, O.TIER_21) if bound == O.SMOOTH_11 else (O.TIER_21, O.TIER_ALL)
        assert np.all(first[:n] == inside) and np.all(first[n:] == outside)


def test_default_mode_on_eccentric_orbits(const):
    """the default-mode kernel (the reference's RK45 controller replayed per interval) against the reference's own call,
    interval_matrices(use_uniform_steps=False): the same accepted steps (node counts) and the matrices to 1.3e-11"""
    from oracle.mpc_oracle import interval_matrices
    el = O.sweep_elements()
    pick = np.flatnonzero((el["e"] >= 0.6) & (el["nu0"] >= 0))[::2]
    Y0 = O.kepler_states(const, **{k: v[pick] for k, v in el.items()})
    K = 4
    tf = 0.05 * _perigee_period(const, Y0) * (K - 1)
    _, x, u = O.kepler_batch(const, K, tf, "tangential", Y0=Y0)
    for j2 in (False, True):
        out, st, nodes = hostk.discretize_adaptive(x, u, tf, const, include_J2=j2)
        assert st.max() == 0
        got = hostk.stacked(out, len(pick), K)
        for s in range(len(pick)):
            for k in range(K - 1):
                ref = interval_matrices(k, x[s], u[s], tf[s], const, include_J2=j2)
                for i, n in enumerate(NAMES):
                    g = got[i][s, k] if i < 3 else got[i][s, :, k]
                    assert rel_err(g, ref[i]) <= 1.3e-11, (s, k, n)
        assert nodes.max() > 3


def test_rk45_propagation_on_eccentric_orbits(const):
    """the RK45 propagator against the reference's solve_ivp on eccentric orbits whose perigee passes make the step-size
    controller reject steps: the same attempted steps as the C oracle's replica, 6 function evaluations per attempted
    step plus 2 (the first-step heuristic) in scipy, states to 1e-12"""
    from oracle import mpc_oracle as MO
    el = O.sweep_elements()
    pick = np.flatnonzero(el["nu0"] == 0.0)[::3]
    Y0 = O.kepler_states(const, **{k: v[pick] for k, v in el.items()})
    tf, T, max_step, thrust = 3.0, 40, 0.2, 0.02      # steps long enough for the error estimate to reject some
    for j2 in (False, True):
        y, uo, st, steps, _ = hostk.propagate_rk45(Y0, tf, const, kind=C.CTRL_TANGENTIAL, thrust=(thrust, 0, 0),
                                                   include_J2=j2, T=T, max_step=max_step)
        yc, _, stc, acc_c, rej_c = C.propagate_batch_rk45(Y0, tf, const, C.CTRL_TANGENTIAL, (thrust, 0, 0),
                                                          include_drag=False, include_J2=j2, T=T, max_step=max_step)
        assert st.max() == 0 and stc.max() == 0
        assert np.array_equal(steps, acc_c + rej_c)                     # attempted = accepted + rejected
        assert np.any(rej_c[el["e"][pick] > 0] > 0)
        for s in range(len(pick)):
            law = MO.ctrl_tangential(thrust)
            calls = [0]

            def counted(xx, tau):
                calls[0] += 1
                return law(xx, tau)
            ys, _ = MO.propagate(Y0[s], tf, counted, const, include_drag=False, include_J2=j2, eval_points=T,
                                 max_step=max_step)
            assert calls[0] == 2 + 6 * steps[s], (s, calls[0], steps[s])
            assert rel_err(y[s], ys) <= 1e-12, s
