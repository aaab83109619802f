"""The 11-node form of the reference's 101-node trapezoid sums on ten fifth-order Nystrom steps (kEmW3, column_step5 /
state_step5 in csrc/discretize_kernel.cuh): the rule, the tableau, the host build of the fixed-step kernels with the form
switched on (em11=True below, what the launcher does by default) and off, and the gate on the benchmark's own constellation."""
import ctypes
import os
import re
from fractions import Fraction as F

import numpy as np
import pytest

import hostk
from conftest import GOLDEN, NAMES, ROOT, rel_err, synth_batch
from oracle import c_oracle as C

SRC = os.path.join(ROOT, "mpconstellation_b200", "csrc", "discretize_kernel.cuh")
W_COMB = [F(11189689, 8000000), F(-13088691, 32000000), F(2089791, 200000000), F(-110789, 800000000)]
GROUPS = ((0, 49), (49, 70), (70, 91), (91, 98), (98, 105))


def _em_level(em, em11):
    """DstTab::em: 0 every node evaluated, 1 the 21- / 51-node forms, 2 also the 11-node form (the launcher's default,
    mpc_set_tuning(40))"""
    return (2 if em11 else 1) if em else 0


def discretize(x, u, tf, const, include_J2=False, n_sub=100, em=True, em11=False):
    """hostk.discretize (the fixed-step kernels, one thread per interval, whole batch) with the 11-node form selectable:
    em11=True takes it where the gate admits it"""
    x = np.ascontiguousarray(x, dtype=np.float64)
    u = np.ascontiguousarray(u, dtype=np.float64)
    N, _, K = x.shape
    tfv = np.ascontiguousarray(np.broadcast_to(np.asarray(tf, dtype=np.float64), (N,)))
    n_int = N * (K - 1)
    out = np.full((105, n_int), np.nan)
    status = np.full(n_int, -1, dtype=np.int32)
    hostk.lib().hostk_discretize(hostk._p(x), hostk._p(u), hostk._p(tfv), hostk._p(hostk._const8(const)), int(include_J2), N, K,
                                 int(n_sub), 1, 0, -1, hostk._p(out), ctypes.c_longlong(n_int), ctypes.c_longlong(0),
                                 hostk._p(status), ctypes.c_longlong(0), ctypes.c_longlong(0), _em_level(em, em11))
    return out, status


def discretize_group(x, u, tf, const, include_J2=False, n_sub=100, em=True, em11=False):
    """hostk.discretize_group (8 lanes per interval) with the 11-node form selectable, as discretize above"""
    x = np.ascontiguousarray(x, dtype=np.float64)
    u = np.ascontiguousarray(u, dtype=np.float64)
    N, _, K = x.shape
    tfv = np.ascontiguousarray(np.broadcast_to(np.asarray(tf, dtype=np.float64), (N,)))
    n_int = N * (K - 1)
    out = np.full((105, n_int), np.nan)
    status = np.full(n_int, -1, dtype=np.int32)
    hostk.lib().hostk_discretize_group(hostk._p(x), hostk._p(u), hostk._p(tfv), hostk._p(hostk._const8(const)), int(include_J2),
                                       N, K, int(n_sub), hostk._p(out), ctypes.c_longlong(n_int), ctypes.c_longlong(0),
                                       hostk._p(status), 0, _em_level(em, em11))
    return out, status


def _rule():
    """the trapezoid sums over every n-th node, n = 10, 20, 50, 100, combined with W_COMB, collected node by node on the
    nodes j = 0, 10, ..., 100 (weights in units of 10 h)"""
    W = [F(0)] * 11
    for wn, n in zip(W_COMB, (1, 2, 5, 10)):
        p = 10 // n
        for j in range(p + 1):
            W[j * n] += wn * n * (F(1, 2) if j in (0, p) else 1)
    return W


def test_the_11_node_rule_literals_are_the_exact_combination_of_four_trapezoid_sums():
    for r in range(4):                                   # sum w n^2r = 1: the h^2, h^4, h^6 terms cancel
        assert sum(w * F(10 * n) ** (2 * r) for w, n in zip(W_COMB, (1, 2, 5, 10))) == 1
    W = _rule()
    body = re.search(r"kEmW3\[11\] = \{(.*?)\};", open(SRC).read(), re.S).group(1)
    lits = [F(int(float(a)), int(b)) for a, b in re.findall(r"([0-9.]+) / ([0-9]+)", body)]
    assert lits == W and sum(W) == 10 and all(q > 0 for q in W) and W == W[::-1]
    # exact against the 101-node trapezoid sum (not the integral) for every polynomial through degree 7
    for p in range(8):
        full = sum(F(j, 100) ** p * (F(1, 2) if j in (0, 100) else 1) for j in range(101)) / 100
        assert sum(W[i] * F(i, 10) ** p for i in range(11)) / 10 == full, p


@pytest.mark.parametrize("theta,bound", [(0.066, 1e-15), (0.25, 1e-14), (0.5, 1e-12), (1.0, 2e-10)])
def test_the_11_node_rule_remainder_grows_with_the_turn_of_the_integrand(theta, bound):
    """remainder against the literal 101-node sum of cos(theta tau + 0.4): rounding at the benchmark's 0.066 rad per
    interval, 2.5e-13 at 0.5 rad, 5e-11 at 1 rad (the 21-node rule: 3e-14 at 1 rad)"""
    W = [float(q) for q in _rule()]
    t = np.linspace(0.0, 1.0, 101)
    g = np.cos(theta * t + 0.4)
    full = 0.01 * (g[0] / 2 + g[-1] / 2 + g[1:-1].sum())
    em = 0.1 * sum(W[i] * g[10 * i] for i in range(11))
    assert abs(em - full) <= bound
    if theta >= 0.5:
        assert abs(em - full) > bound / 100                # it is a remainder of the rule, not rounding


def test_the_fifth_order_nystrom_tableau_satisfies_the_order_conditions():
    """Nystrom (1925), 4 stages: the conditions of a Runge-Kutta-Nystrom method for y'' = f(t, y) through order 5,
    in exact fractions, with the coefficients as written in column_step5"""
    c = [F(0), F(1, 5), F(2, 3), F(1)]
    a = {(1, 0): F(1, 50), (2, 0): F(-1, 27), (2, 1): F(7, 27), (3, 0): F(3, 10), (3, 1): F(-2, 35), (3, 2): F(9, 35)}
    bbar = [F(14, 336), F(100, 336), F(54, 336), F(0)]
    b = [F(14, 336), F(125, 336), F(162, 336), F(35, 336)]
    A = [[a.get((i, j), F(0)) for j in range(4)] for i in range(4)]
    for i in range(4):
        assert sum(A[i]) == c[i] ** 2 / 2
    for q in range(5):                                   # b c^q = 1/(q+1), q <= 4
        assert sum(b[i] * c[i] ** q for i in range(4)) == F(1, q + 1)
    for q in range(4):                                   # bbar c^q = 1/((q+1)(q+2)), q <= 3
        assert sum(bbar[i] * c[i] ** q for i in range(4)) == F(1, (q + 1) * (q + 2))
    # the remaining trees: sum b_i g(c_i) stands for int_0^1 g, sum_j a_ij g(c_j) for int_0^c_i (c_i - s) g(s) ds,
    # sum bbar_i g(c_i) for int_0^1 (1 - t) g(t) dt
    Ac = [sum(A[i][j] * c[j] for j in range(4)) for i in range(4)]
    Ac2 = [sum(A[i][j] * c[j] ** 2 for j in range(4)) for i in range(4)]
    AAc = [sum(A[i][j] * sum(A[j]) for j in range(4)) for i in range(4)]
    assert sum(b[i] * Ac[i] for i in range(4)) == F(1, 24)                  # order 4
    assert sum(b[i] * c[i] * Ac[i] for i in range(4)) == F(1, 30)           # order 5
    assert sum(b[i] * Ac2[i] for i in range(4)) == F(1, 60)
    assert sum(b[i] * AAc[i] for i in range(4)) == F(1, 120)
    assert sum(bbar[i] * Ac[i] for i in range(4)) == F(1, 120)              # positions, order 5
    assert sum(bbar[i] * c[i] * sum(A[i]) for i in range(4)) == F(1, 40)
    # the coefficients are the ones the kernel source uses (p+ = b + k1/24 + 25/84 k2 + 9/56 k3, p'+ = ... 5/48 k4)
    assert [F(1, 24), F(25, 84), F(9, 56)] == bbar[:3] and [F(1, 24), F(125, 336), F(27, 56), F(5, 48)] == b
    src = open(SRC).read()
    body = src[src.index("void column_step5"):src.index("void stage_accel")]
    for lit in ("1.0 / 50", "0.2", "7.0 / 27", "-1.0 / 27", "2.0 / 3", "9.0 / 35", "-2.0 / 35", "0.3", "9.0 / 56",
                "25.0 / 84", "1.0 / 24", "5.0 / 48", "27.0 / 56", "125.0 / 336"):
        assert lit in body, lit


def test_the_mass_quadrature_weights_integrate_the_cubic_exactly():
    """state_step5: m at c_s is m + the integral to c_s of the cubic through mdot at c = (0, 1/5, 2/3, 1)"""
    c = [F(0), F(1, 5), F(2, 3), F(1)]
    src = open(SRC).read()
    body = src[src.index("void state_step5"):]
    rows = {1: (F(253, 3000), F(209, 1680), F(-81, 7000), F(17, 6000)), 2: (F(1, 81), F(250, 567), F(5, 21), F(-2, 81)),
            3: (F(1, 24), F(125, 336), F(27, 56), F(5, 48))}
    for s, w in rows.items():
        for p in range(4):
            assert sum(w[j] * c[j] ** p for j in range(4)) == c[s] ** (p + 1) / (p + 1)
        for q in w:
            assert f"{q.numerator}.0 / {q.denominator}" in body or f"{-q.numerator}.0 / {q.denominator}" in body


@pytest.mark.parametrize("j2", [False, True])
def test_11_node_form_agrees_with_the_21_node_form_and_the_101_nodes(const, j2):
    """pair and group kernel with the 11-node form against the 21-node form (quadrature rows to 1e-12, A_k to 2e-11: the
    21-node form's own integrator error), against every node evaluated (A_k to 1e-12 -- closer than the 21-node form --,
    quadrature to 1e-12) and against the plain-C oracle's literal sums; pair vs group to 1e-14 in A_k"""
    for n_sats, K, tf in ((5, 23, 0.23), (3, 50, 0.5)):
        _, x, u = synth_batch(n_sats, K, tf, const)
        a, sa = discretize(x, u, tf, const, include_J2=j2, em11=True)
        o, so = discretize(x, u, tf, const, include_J2=j2)
        b, sb = discretize(x, u, tf, const, include_J2=j2, em=False)
        g, sg = discretize_group(x, u, tf, const, include_J2=j2, em11=True)
        assert sa.max() == 0 and so.max() == 0 and sb.max() == 0 and sg.max() == 0
        assert not np.any(np.all(a == o, axis=0))                          # every interval takes the new form
        assert rel_err(a[0:49], o[0:49]) < 2e-11
        for r0, r1 in GROUPS[1:]:
            assert rel_err(a[r0:r1], o[r0:r1]) < 1e-12, (r0, K)
            assert rel_err(a[r0:r1], b[r0:r1]) < 1e-12, (r0, K)
        assert rel_err(a[0:49], b[0:49]) < 1e-12 < rel_err(o[0:49], b[0:49])
        assert rel_err(a[0:49], g[0:49]) < 1e-14 and rel_err(a, g) < 1e-13
        ref = C.discretize_batch(x, u, tf, const, include_J2=j2)
        for n, v in zip(NAMES, hostk.stacked(a, n_sats, K)):
            assert rel_err(v, ref[NAMES.index(n)]) < 2e-11, n


def test_11_node_form_is_fifth_order(const):
    """A_k against a fine-step launch (1000 nodes, 500 steps; A_k does not depend on the quadrature) on 0.01- and
    0.005-orbit intervals, with J2 made 1000x larger so that the integrator's error stands above rounding inside the
    gate: halving the interval cuts the error by about 2^5 (the 21-node form's fourth-order steps: 2^4)"""
    import dataclasses
    stiff = dataclasses.replace(const, J2=const.J2 * 1000.0) if dataclasses.is_dataclass(const) else \
        const._replace(J2=const.J2 * 1000.0)
    err, err4 = [], []
    for K in (21, 41):
        _, x, u = synth_batch(3, K, 0.2, const)
        a, sa = discretize(x, u, 0.2, stiff, include_J2=True, em11=True)
        o, _ = discretize(x, u, 0.2, stiff, include_J2=True)
        r, _ = discretize(x, u, 0.2, stiff, include_J2=True, em=False, n_sub=1000)
        assert sa.max() == 0 and not np.any(np.all(a == o, axis=0))
        err.append(rel_err(a[0:49], r[0:49]))
        err4.append(rel_err(o[0:49], r[0:49]))
    assert 2 ** 4.5 < err[0] / err[1] < 2 ** 6.5, err
    assert err[0] < err4[0] / 50
    assert 2 ** 3.5 < err4[0] / err4[1] < 2 ** 4.5, err4


def _tiers(u):
    """per interval, from the gate's smoothness measure |u_k+1 - u_k|^2 / max(|u_k|^2, |u_k+1|^2): 3 = the 11-node form
    (<= 1/64), 1 = the 21-node form (<= 1/16), 0 = all 101 nodes (on intervals the orbital bound admits)"""
    u0, u1 = u[:, :, :-1], u[:, :, 1:]
    d2, m2 = np.sum((u1 - u0) ** 2, axis=1), np.maximum(np.sum(u0 ** 2, axis=1), np.sum(u1 ** 2, axis=1))
    q2 = np.divide(d2, m2, out=np.zeros_like(d2), where=m2 > 0)     # a coast arc (u = 0 at both nodes) counts as smooth
    return np.where(q2 <= 1 / 64, 3, np.where(q2 <= 1 / 16, 1, 0)).ravel()


def test_11_node_form_is_taken_where_the_input_changes_by_at_most_an_eighth(const):
    """same per-interval gate as the 21-node form with the smoothness bound halved: thrust jumps, sign flips and
    coast-to-thrust switches take all 101 nodes (bit-identical to the launch without the rules), inputs that change by
    1/8 ... 1/4 of their size the 21-node form (bit-identical to the launch without the 11-node form), long intervals the
    51-node rule, other node counts are untouched"""
    n_sats, K, tf = 4, 23, 0.23
    _, x, u = synth_batch(n_sats, K, tf, const)
    u = u.copy()
    u[0, :, 8:] *= 1.5
    u[1, :, 5:9] = 0.0
    u[2, :, 12:] *= -1.0
    u[3, :, 10] *= 1.2                    # a 1/6 change on both sides of node 10: the 21-node form
    a, sa = discretize(x, u, tf, const, em11=True)
    o, _ = discretize(x, u, tf, const)
    b, _ = discretize(x, u, tf, const, em=False)
    g, _ = discretize_group(x, u, tf, const, em11=True)
    assert sa.max() == 0
    expect_all = np.zeros((n_sats, K - 1), dtype=bool)
    expect_all[0, 7] = expect_all[1, 4] = expect_all[1, 8] = expect_all[2, 11] = True
    expect_21 = np.zeros((n_sats, K - 1), dtype=bool)
    expect_21[3, 9] = expect_21[3, 10] = True
    assert np.array_equal(np.all(a == b, axis=0).reshape(n_sats, K - 1), expect_all)
    assert np.array_equal(np.all(a == o, axis=0).reshape(n_sats, K - 1), expect_all | expect_21)
    assert np.array_equal(_tiers(u).reshape(n_sats, K - 1), np.where(expect_all, 0, np.where(expect_21, 1, 3)))
    assert rel_err(a, g) < 1e-13
    new = ~(expect_all | expect_21).ravel()
    assert rel_err(a[0:49, new], b[0:49, new]) < 1e-12
    for r0, r1 in GROUPS[1:]:
        assert rel_err(a[r0:r1, new], b[r0:r1, new]) < 1e-12
    _, x2, u2 = synth_batch(2, 16, 0.5, const)                          # 0.033-orbit intervals: the 51-node rule
    assert np.array_equal(discretize(x2, u2, 0.5, const, em11=True)[0], discretize(x2, u2, 0.5, const)[0])
    assert np.array_equal(discretize(x, u, tf, const, n_sub=50, em11=True)[0],
                          discretize(x, u, tf, const, n_sub=50, em=False)[0])


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_11_node_form_on_random_thrust_tables(const, seed):
    """inputs whose direction and size change from node to node by 0 ... 40 % of their size, so that every tier is
    taken: the 11-node intervals within 1e-12 of every node evaluated (A_k and quadrature), the others bit-identical to
    the launch without the 11-node form"""
    rng = np.random.default_rng(seed)
    n_sats, K = 6, int(rng.integers(12, 40))
    tf = 0.0101 * (K - 1) * float(rng.uniform(0.5, 1.05))
    _, x, u = synth_batch(n_sats, K, tf, const)
    u = u.copy()
    for s in range(n_sats):
        for k in range(1, K):
            d = rng.normal(size=3)
            d *= rng.uniform(0.0, 0.4) * np.linalg.norm(u[s, :, k - 1]) / np.linalg.norm(d)
            u[s, :, k] = u[s, :, k - 1] + d
    j2 = bool(seed % 2)
    a, sa = discretize(x, u, tf, const, include_J2=j2, em11=True)
    o, so = discretize(x, u, tf, const, include_J2=j2)
    b, sb = discretize(x, u, tf, const, include_J2=j2, em=False)
    assert sa.max() == 0 and so.max() == 0 and sb.max() == 0
    tier = _tiers(u)
    assert all(0.1 < (tier == t).mean() < 0.8 for t in (0, 1, 3))
    assert np.array_equal(np.all(a == o, axis=0), tier != 3)
    new = tier == 3
    for r0, r1 in GROUPS:
        assert rel_err(a[r0:r1, new], b[r0:r1, new]) < 1e-12, (r0, seed)
        assert rel_err(a[r0:r1], b[r0:r1]) < (2e-11 if r0 == 0 else 2e-12), (r0, seed)


def test_with_the_11_node_form_off_the_kernels_compute_what_they_did_before_it():
    """em11=False (mpc_set_tuning(39) on the device): bit-identical to the outputs of the kernels before the 11-node form
    was added (tests/golden/discretize_em21.npz: the host build of those sources, J2 on, a thrust jump in satellite 0)"""
    from oracle.mpc_oracle import OracleConstants
    const = OracleConstants(*np.load(os.path.join(GOLDEN, "discretize.npz"))["const"])
    g = np.load(os.path.join(GOLDEN, "discretize_em21.npz"))
    x, u, tf = g["x"], g["u"], float(g["tf"])
    a, _ = hostk.discretize(x, u, tf, const, include_J2=True)
    b, _ = hostk.discretize_group(x, u, tf, const, include_J2=True)
    assert np.array_equal(a, g["pair"]) and np.array_equal(b, g["group"])
    assert not np.array_equal(discretize(x, u, tf, const, include_J2=True, em11=True)[0], g["pair"])


def test_every_interval_of_the_benchmark_constellation_takes_the_11_node_form():
    """bench.py's workload (4096 satellites of make_constellation, K = 200, tf = 2, tangential thrust 0.5), propagated by
    the C oracle's restatement of the reference's RK45, with the gate quantities evaluated as discretize_pair_kernel does:
    every interval passes -- the benchmark measures the 11-node form, not a silent fallback"""
    import bench
    Y, const = bench.make_constellation(4096)
    K, tf = 200, 2.0
    x, u, st, _, _ = C.propagate_batch_rk45(Y, tf, const, C.CTRL_TANGENTIAL, (0.5, 0.0, 0.0), include_drag=False,
                                            include_J2=False, T=K)
    assert st.max() == 0
    u0, u1 = u[:, :, :-1], u[:, :, 1:]
    d2 = np.sum((u1 - u0) ** 2, axis=1)
    smooth = d2 / np.maximum(np.sum(u0 ** 2, axis=1), np.sum(u1 ** 2, axis=1))
    r2 = np.sum(x[:, 0:3, :-1] ** 2, axis=1)
    H = 2.0 * tf * (1.0 / 100) / (K - 1)
    orbit = const.MU * H * H / (r2 * np.sqrt(r2)) * 6.25
    assert smooth.max() <= 0.015625 / 2, smooth.max()          # with margin: the input changes by < 1/11 of its size
    assert orbit.max() <= 1.2e-5 * 0.99, orbit.max()
