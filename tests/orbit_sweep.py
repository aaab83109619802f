"""TEST INFRASTRUCTURE ONLY -- orbits away from the Hubble family, intervals placed on the tier gates of the fixed-step
discretization, and an extended-precision reference of the reference's 101-node trapezoid sums.

Every other fixture of the suite starts from the one near-circular, 28.5-degree Hubble state under a slowly turning
tangential thrust.  kepler_batch builds constellations from orbital elements instead (eccentric, equatorial, polar and
retrograde, start nodes around perigee, four thrust laws, masses down to 0.3); intervals_at_gate sizes the intervals so
that their start node lands just inside and just outside each threshold of the per-interval tier gate; sums101_longdouble
integrates every interval with np.longdouble and forms the 101-node sums of oracle/mpc_oracle.py: interval_matrices
(use_uniform_steps=True) from the exact flow, so that the kernels are checked against something other than a restatement
of their own algorithm.
"""
import numpy as np

from oracle import c_oracle as C

# The per-interval tier gate of discretize_pair_kernel (csrc/discretize_pair_kernel.cuh, the block that picks the form of
# the sums) and discretize_group_kernel (csrc/discretize_group_kernel.cuh, the same conditions), with n_sub = 100:
#   w2H2 = MU H^2 / |r_k|^3, H = 2 tf / (n_sub (K - 1)): the circular orbital rate at the start node times two panels
#   smooth: |u_k+1 - u_k|^2 <= SMOOTH_21 max(|u_k|^2, |u_k+1|^2)
#   smooth and ORBIT_SCALE_11 w2H2 <= ORBIT_11: 10 fifth-order steps + the 11-node rule if also |du|^2 <= SMOOTH_11 max|u|^2
#                                              (and the 11-node form is on), else 20 steps + the 21-node rule
#   smooth and ORBIT_11 < 6.25 w2H2, w2H2 <= ORBIT_51: 50 steps + the 51-node rule
#   otherwise all 101 nodes: two nodes per step with the Hermite midpoint where w2H2 <= ORBIT_HERMITE, else one per node
SMOOTH_11 = 0.015625          # 1/64: the input changes by at most an eighth of its size
SMOOTH_21 = 0.0625            # 1/16: ... a quarter
ORBIT_SCALE_11 = 6.25         # (5 h / 2 h)^2: the gate of the 11/21-node forms is on the rate times five panels
ORBIT_11 = 1.2e-5
ORBIT_51 = 1.94e-5
ORBIT_HERMITE = 1.0e-5

TIER_ALL, TIER_21, TIER_51, TIER_11 = 0, 1, 2, 3
TIER_NAMES = {TIER_ALL: "101 nodes", TIER_21: "21-node", TIER_51: "51-node", TIER_11: "11-node"}
GROUPS = {"A_k": (0, 49), "B_pm": (49, 91), "Sigma": (91, 98), "xi": (98, 105)}
LAWS = ("tangential", "inertial", "radial", "normal")


def w2H2(x, tf, K, const, n_sub=100):
    """the gate's orbital quantity at the start node of every interval, [N, K-1], as the kernels form it"""
    tf = np.broadcast_to(np.asarray(tf, dtype=np.float64), (x.shape[0],))[:, None]
    H = 2.0 * (tf * ((1.0 / n_sub) / (K - 1)))
    r2 = np.sum(x[:, 0:3, :-1] ** 2, axis=1)
    return const.MU * (H * H) / (r2 * np.sqrt(r2))


def smoothness(u):
    """(d2, max(a2, b2)) of the gate, [N, K-1], with the kernels' operations (exact for inputs along one axis)"""
    u0 = u[:, :, :-1]
    du = u[:, :, 1:] - u0
    e0 = u0 + du
    return np.sum(du * du, axis=1), np.maximum(np.sum(u0 * u0, axis=1), np.sum(e0 * e0, axis=1))


def tiers(x, u, tf, const, em11=True, n_sub=100):
    """the form of the sums every interval takes, [N, K-1] (TIER_*), from the gate quantities"""
    w = w2H2(x, tf, x.shape[2], const, n_sub)
    d2, m2 = smoothness(u)
    smooth = d2 <= SMOOTH_21 * m2
    t = np.full(w.shape, TIER_ALL)
    if n_sub != 100:
        return t
    short = w * ORBIT_SCALE_11 <= ORBIT_11
    t[smooth & ~short & (w <= ORBIT_51)] = TIER_51
    t[smooth & short] = TIER_21
    if em11:
        t[smooth & short & (d2 <= SMOOTH_11 * m2)] = TIER_11
    return t


# ---------------------------------------------------------------------------------------------------- constellations

def kepler_states(const, e, inc, nu0, alt=0.04, mass=1.0, raan=0.0, argp=0.0):
    """normalized states [N,7] from elements: perigee radius R_E (1 + alt), eccentricity e, inclination inc, true anomaly
    nu0 at the start (all radians, broadcast).  inc = 0 gives z = vz = 0 exactly."""
    e, inc, nu0, alt, mass, raan, argp = np.broadcast_arrays(*[np.asarray(v, dtype=np.float64) for v in
                                                              (e, inc, nu0, alt, mass, raan, argp)])
    rp = const.R_E * (1.0 + alt)
    p = rp * (1.0 + e)
    r = p / (1.0 + e * np.cos(nu0))
    vs = np.sqrt(const.MU / p)
    P = np.stack([r * np.cos(nu0), r * np.sin(nu0), np.zeros_like(r)])            # perifocal frame
    V = np.stack([-vs * np.sin(nu0), vs * (e + np.cos(nu0)), np.zeros_like(r)])
    cO, sO, ci, si, cw, sw = np.cos(raan), np.sin(raan), np.cos(inc), np.sin(inc), np.cos(argp), np.sin(argp)
    R = np.array([[cO * cw - sO * sw * ci, -cO * sw - sO * cw * ci, sO * si],
                  [sO * cw + cO * sw * ci, -sO * sw + cO * cw * ci, -cO * si],
                  [sw * si, cw * si, ci]])
    R[2, 0:2] = np.where(si == 0.0, 0.0, R[2, 0:2])
    Y = np.zeros(e.shape + (7,))
    Y[..., 0:3] = np.einsum("ij...,j...->...i", R, P)
    Y[..., 3:6] = np.einsum("ij...,j...->...i", R, V)
    Y[..., 6] = mass
    return Y


def sweep_elements(seed=20261020, n_nu=3):
    """the element grid of the sweep: e in (0, 0.3, 0.6, 0.8) x inclination (0, 90, 160 degrees) x start node (just
    before, at and just after perigee); perigee altitudes in [0.02, 0.05] R_E, node / argument of perigee and the mass in
    [0.3, 1] seeded.  Returns dict of [N] arrays."""
    rng = np.random.default_rng(seed)
    E, I, NU = np.meshgrid([0.0, 0.3, 0.6, 0.8], np.radians([0.0, 90.0, 160.0]), [-0.02, 0.0, 0.02][:n_nu], indexing="ij")
    n = E.size
    return dict(e=E.ravel(), inc=I.ravel(), nu0=NU.ravel(), alt=rng.uniform(0.02, 0.05, n), mass=rng.uniform(0.3, 1.0, n),
                raan=rng.uniform(0, 2 * np.pi, n), argp=rng.uniform(0, 2 * np.pi, n))


INERTIAL_DIR = (0.6, 0.0, 0.8)


def law_inputs(x, law, thrust=0.5):
    """node inputs [N,3,K] of a thrust law evaluated on the states x [N,7,K]"""
    r, v = x[:, 0:3], x[:, 3:6]
    rh = r / np.linalg.norm(r, axis=1, keepdims=True)
    h = np.cross(r, v, axis=1)
    hh = h / np.linalg.norm(h, axis=1, keepdims=True)
    if law == "radial":
        return thrust * rh
    if law == "normal":
        return thrust * hh
    if law == "tangential":
        return thrust * np.cross(hh, rh, axis=1)
    if law == "inertial":
        return np.broadcast_to(thrust * np.asarray(INERTIAL_DIR)[None, :, None], x[:, 0:3].shape).copy()
    raise ValueError(law)


def kepler_batch(const, K, tf, law="tangential", Y0=None, seed=20261020, thrust=0.5, n_nu=3):
    """a constellation of sweep_elements (or the states Y0), propagated by the C oracle as conftest.synth_batch does
    (fixed-step RK4 at <= 1e-3 of the horizon per step, no J2): tangential and constant inertial thrust fly under their
    own law, radial and normal thrust are evaluated on a coast arc.  tf scalar or [N].  Returns Y0, x [N,7,K], u [N,3,K]."""
    if Y0 is None:
        Y0 = kepler_states(const, **sweep_elements(seed, n_nu))
    n_sub = max(1, int(np.ceil(1000 / max(K - 1, 1))))
    kind, cp = {"tangential": (C.CTRL_TANGENTIAL, (thrust, 0.0, 0.0)),
                "inertial": (C.CTRL_CONSTANT, tuple(thrust * np.asarray(INERTIAL_DIR)))}.get(
                    law, (C.CTRL_ZERO, (0.0, 0.0, 0.0)))
    x, u, st = C.propagate_batch(Y0, tf, const, kind, cp, include_drag=False, include_J2=False, T=K, n_sub=n_sub)
    assert st.max() == 0
    if law in ("radial", "normal"):
        u = law_inputs(x, law, thrust)
    return Y0, x, u


def tf_for_w2H2(const, Y0, K, value, n_sub=100):
    """tf [N] that puts the start node of the first interval at w2H2 = value"""
    r = np.linalg.norm(Y0[:, 0:3], axis=1)
    return 0.5 * n_sub * (K - 1) * np.sqrt(np.asarray(value) * r ** 3 / const.MU)


def intervals_at_gate(const, K=4, law="tangential", rel=1e-9, seed=20261020):
    """the orbital thresholds: for every threshold (ORBIT_11 through ORBIT_SCALE_11, ORBIT_51, ORBIT_HERMITE) the sweep's
    satellites with tf set so that the first interval's w2H2 lies `rel` inside and `rel` outside it.
    Returns {(name, side): (Y0, x, u, tf)}, side "in" / "out"."""
    Y0 = kepler_states(const, **sweep_elements(seed))
    out = {}
    for name, thr in (("11/21", ORBIT_11 / ORBIT_SCALE_11), ("51", ORBIT_51), ("hermite", ORBIT_HERMITE)):
        for side, f in (("in", 1.0 - rel), ("out", 1.0 + rel)):
            tf = tf_for_w2H2(const, Y0, K, thr * f)
            _, x, u = kepler_batch(const, K, tf, law, Y0=Y0)
            out[(name, side)] = (Y0, x, u, tf)
    return out


def smoothness_tables(K, bound, n_sats=2):
    """input tables [2 n_sats, 3, K] along one axis whose FIRST interval has |du|^2 / max|u|^2 one ulp of the input
    inside (satellites 0..n_sats-1) and outside (n_sats..) `bound` (SMOOTH_11 or SMOOTH_21), as the kernels evaluate it;
    the later intervals shrink by the same ratio as the first one (inside the bound up to rounding, continuous at the
    nodes).  The magnitudes are 0.5 ... 0.75."""
    q = np.sqrt(bound)                                   # 1/8 or 1/4
    c = 0.75
    target = c * (1.0 - q)

    def inside(u1):
        d = u1 - c
        e = c + d
        return d * d <= bound * max(c * c, e * e)
    lo = hi = target                                     # walk to the last inside / first outside value of u1
    while inside(lo):
        lo = np.nextafter(lo, 0.0)
    while not inside(lo):
        lo = np.nextafter(lo, 1.0)
    hi = np.nextafter(lo, 0.0)
    assert inside(lo) and not inside(hi)
    tabs = []
    for u1 in [lo] * n_sats + [hi] * n_sats:
        t = np.zeros((3, K))
        t[0, 0] = c
        t[0, 1:] = u1 * (u1 / c) ** np.arange(K - 1)
        tabs.append(t)
    return np.stack(tabs)


# ---------------------------------------------------------------------------------------------------- the reference

def _rhs(y, P, u, tf, const, j2):
    """d/ds of (r, v, m, Phi rows 0..5) over one interval in the local s in [0, 1] (tau = tau_k + s / (K-1)), longdouble.
    y: state [M,7], P: Phi rows 0..5 [M,6,7] (row 6 of Phi stays e7: the last row of A is zero)."""
    r, v, m = y[:, 0:3], y[:, 3:6], y[:, 6]
    r2 = np.sum(r * r, axis=1)
    rn = np.sqrt(r2)
    ir3 = 1 / (r2 * rn)
    G = const["MU"] * (3 * (r[:, :, None] * r[:, None, :]) / r2[:, None, None] - np.eye(3, dtype=np.longdouble)) * \
        ir3[:, None, None]
    acc = -const["MU"] * ir3[:, None] * r + u / m[:, None]
    if j2:
        kJ2 = 1.5 * const["J2"] * const["MU"] * const["R_E"] ** 2
        q = 5 * r[:, 2] ** 2 / r2
        shape = np.stack([q - 1, q - 1, q - 3], axis=1)
        k5 = kJ2 / (r2 * r2 * rn)
        acc = acc + k5[:, None] * shape * r
        # the reference's Jacobian of the J2 term (linearize_discretize.py:150-158), which is its exact derivative
        ddr = -2 * q[:, None] * r / r2[:, None]
        ddr[:, 2] += 10 * r[:, 2] / r2
        G = G + k5[:, None, None] * ((-5 * (shape * r)[:, :, None] * r[:, None, :]) / r2[:, None, None]
                                     + r[:, :, None] * ddr[:, None, :] + shape[:, :, None] * np.eye(3, dtype=np.longdouble))
    un = np.sqrt(np.sum(u * u, axis=1))
    a6 = -u / (m * m)[:, None]
    dy = np.empty_like(y)
    dy[:, 0:3] = v
    dy[:, 3:6] = acc
    dy[:, 6] = -un / (const["G0"] * const["ISP"])
    dP = np.empty_like(P)
    dP[:, 0:3] = P[:, 3:6]
    dP[:, 3:6] = np.einsum("mij,mjc->mic", G, P[:, 0:3])
    dP[:, 3:6, 6] += a6
    f = tf[:, None]
    return dy * f, dP * f[:, :, None], G, a6, acc, un


def _node_terms(y, P, u, tf, const, j2):
    """the reference's integrands at one node (interval_matrices: Bs, Ss, Xs) and Phi [M,7,7]"""
    M = y.shape[0]
    _, _, G, a6, acc, un = _rhs(y, P, u, tf, const, j2)
    Phi = np.zeros((M, 7, 7), dtype=np.longdouble)
    Phi[:, 0:6] = P
    Phi[:, 6, 6] = 1
    A = np.zeros((M, 7, 7), dtype=np.longdouble)
    A[:, 0:3, 3:6] = np.eye(3, dtype=np.longdouble)
    A[:, 3:6, 0:3] = G
    A[:, 3:6, 6] = a6
    A *= tf[:, None, None]
    B = np.zeros((M, 7, 3), dtype=np.longdouble)
    B[:, 3:6, :] = np.eye(3, dtype=np.longdouble) / y[:, 6, None, None]
    big = un > np.finfo(np.float64).eps
    B[big, 6, :] = -u[big] / (const["G0"] * const["ISP"] * un[big, None])
    B *= tf[:, None, None]
    S = np.empty((M, 7), dtype=np.longdouble)
    S[:, 0:3] = y[:, 3:6]
    S[:, 3:6] = acc
    S[:, 6] = -un / (const["G0"] * const["ISP"])
    X = -(np.einsum("mij,mj->mi", A, y) + np.einsum("mij,mj->mi", B, u))
    return Phi, B, S, X


def _inv(Phi):
    """Phi^-1 to longdouble precision: the float64 inverse refined by two Newton steps"""
    X = np.linalg.inv(Phi.astype(np.float64)).astype(np.longdouble)
    I2 = 2 * np.eye(7, dtype=np.longdouble)
    for _ in range(2):
        X = X @ (I2 - Phi @ X)
    return X


def sums101_longdouble(x, u, tf, const, j2=False, cols=None, m=8, n_nodes=101):
    """The reference's fixed-step discretization (interval_matrices with use_uniform_steps=True, integrator_steps=101) of
    the intervals `cols` (global index s (K-1) + k, default all), with the flow integrated exactly instead of by RK45:
    state + Phi stepped in np.longdouble by classical RK4, m steps per trapezoid panel, sampled on the 101 uniform nodes;
    the input held linearly between u_k and u_k+1; the reference's integrands at the nodes and its trapezoid sums formed
    in longdouble.  Returns float64 (A [n,7,7], B_kp [n,7,3], B_kn [n,7,3], Sigma [n,7], xi [n,7])."""
    N, _, K = x.shape
    cols = np.arange(N * (K - 1)) if cols is None else np.asarray(cols)
    s_idx, k_idx = cols // (K - 1), cols % (K - 1)
    L = np.longdouble
    cst = {k: L(getattr(const, k)) for k in ("MU", "R_E", "J2", "G0", "ISP")}
    tfv = np.broadcast_to(np.asarray(tf, dtype=np.float64), (N,))[s_idx].astype(L)
    dtau = L(1) / (K - 1)
    tfs = tfv * dtau                                     # d/ds = tf / (K-1) d/dt
    y = x[s_idx, :, k_idx].astype(L)
    u0 = u[s_idx, :, k_idx].astype(L)
    du = u[s_idx, :, k_idx + 1].astype(L) - u0
    M = cols.size
    P = np.zeros((M, 6, 7), dtype=L)
    P[:, np.arange(6), np.arange(6)] = 1
    n_pan = n_nodes - 1
    h = L(1) / (n_pan * m)
    sumB = np.zeros((M, 2, 7, 3), dtype=L)               # sum w Phi^-1 B lam_p, lam_n
    sumS = np.zeros((M, 7), dtype=L)
    sumX = np.zeros((M, 7), dtype=L)

    def f(s, y, P):
        dy, dP, *_ = _rhs(y, P, u0 + s * du, tfs, cst, j2)
        return dy, dP

    for j in range(n_nodes):
        s = L(j) / n_pan
        w = L(0.5) if j in (0, n_pan) else L(1)
        Phi, B, S, X = _node_terms(y, P, u0 + s * du, tfv, cst, j2)
        Pi = _inv(Phi)
        PB = Pi @ B
        sumB[:, 0] += (w * s) * PB
        sumB[:, 1] += (w * (1 - s)) * PB
        sumS += w * np.einsum("mij,mj->mi", Pi, S)
        sumX += w * np.einsum("mij,mj->mi", Pi, X)
        if j == n_pan:
            break
        for i in range(m):
            t = s + i * h
            k1y, k1P = f(t, y, P)
            k2y, k2P = f(t + h / 2, y + (h / 2) * k1y, P + (h / 2) * k1P)
            k3y, k3P = f(t + h / 2, y + (h / 2) * k2y, P + (h / 2) * k2P)
            k4y, k4P = f(t + h, y + h * k3y, P + h * k3P)
            y = y + (h / 6) * (k1y + 2 * k2y + 2 * k3y + k4y)
            P = P + (h / 6) * (k1P + 2 * k2P + 2 * k3P + k4P)
    wq = dtau / n_pan
    Bp = Phi @ sumB[:, 0] * wq
    Bn = Phi @ sumB[:, 1] * wq
    Sg = np.einsum("mij,mj->mi", Phi, sumS) * wq
    Xi = np.einsum("mij,mj->mi", Phi, sumX) * wq
    return tuple(a.astype(np.float64) for a in (Phi, Bp, Bn, Sg, Xi))


def to_soa(ref):
    """(A, B_kp, B_kn, Sigma, xi) with a leading interval axis -> SoA [105, n] (the kernels' row order)"""
    A, Bp, Bn, S, X = ref
    n = A.shape[0]
    return np.concatenate([A.reshape(n, 49), Bp.reshape(n, 21), Bn.reshape(n, 21), S, X], axis=1).T


def group_errors(out, ref_soa):
    """{row group: norm-relative error max|a-b| / max|b|} of SoA columns against the reference"""
    res = {}
    for g, (r0, r1) in GROUPS.items():
        a, b = out[r0:r1], ref_soa[r0:r1]
        res[g] = float(np.max(np.abs(a - b)) / np.max(np.abs(b)))
    return res
