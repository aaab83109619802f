"""TEST INFRASTRUCTURE ONLY -- numpy oracle of the conjunction screening (mpconstellation_b200.screen_conjunctions).

The same trajectory model as conjunction_kernel.cuh (each satellite on the cubic Hermite curve through its samples), the
same event rule (local minima of the pair distance below the threshold, t = 0 / t = D by the sign of d' there, a minimum
at a sample belongs to the interval that starts there), but its own arithmetic: every pair-interval of the brute force,
a lower bound of |dp|^2 from the Bernstein coefficients of the sextic (not the kernel's spheres) to pass over the far
ones, and the real roots of the quintic g = dp . dp' from the eigenvalues of its companion matrix, polished by Newton.
"""
import numpy as np

MU_EARTH = 3.986004418e14


def si_states(y, const):
    """y [N,7,T] normalized, const one bag or N -> X [N,6,T] (m, m/s)"""
    N = y.shape[0]
    bags = [const] * N if hasattr(const, "MU") else list(const)
    X = np.empty((N, 6, y.shape[2]))
    for s, c in enumerate(bags):
        s0 = np.sqrt(c.MU * c.R0 ** 3 / MU_EARTH)
        X[s, 0:3] = y[s, 0:3] * c.R0
        X[s, 3:6] = y[s, 3:6] * (c.R0 / s0)
    return X


def cubic(qi0, qi1, qj0, qj1, h):
    """[..., 6] end states of the two satellites -> A [4, ..., 3], the relative cubic's power coefficients"""
    P0, P1 = qi0[..., 0:3] - qj0[..., 0:3], qi1[..., 0:3] - qj1[..., 0:3]
    M0, M1 = h * (qi0[..., 3:6] - qj0[..., 3:6]), h * (qi1[..., 3:6] - qj1[..., 3:6])
    return np.stack([P0, M0, 3.0 * (P1 - P0) - 2.0 * M0 - M1, 2.0 * (P0 - P1) + M0 + M1])


def quintic(A):
    """A [4, ..., 3] -> c [..., 6]: g(s) = dp . dp' = sum c_n s^n"""
    d = lambda a, b: np.sum(A[a] * A[b], axis=-1)
    return np.stack([d(0, 1), 2 * d(0, 2) + d(1, 1), 3 * (d(0, 3) + d(1, 2)), 4 * d(1, 3) + 2 * d(2, 2), 5 * d(2, 3),
                     3 * d(3, 3)], axis=-1)


def f_lower_bound(A):
    """min over the Bernstein coefficients of |dp(s)|^2 (degree 6): <= |dp(s)|^2 on [0, 1]"""
    d = lambda a, b: np.sum(A[a] * A[b], axis=-1)
    e = [d(0, 0), 2 * d(0, 1), 2 * d(0, 2) + d(1, 1), 2 * (d(0, 3) + d(1, 2)), 2 * d(1, 3) + d(2, 2), 2 * d(2, 3), d(3, 3)]
    from math import comb
    b = [sum(comb(k, i) / comb(6, i) * e[i] for i in range(k + 1)) for k in range(7)]
    return np.min(np.stack(b), axis=0)


def _polyval(c, s):
    g = np.zeros_like(s) + c[..., 5]
    dg = np.zeros_like(s)
    for n in range(4, -1, -1):
        dg = dg * s + g
        g = g * s + c[..., n]
    return g, dg


def rising_roots(c):
    """c [m, 6] -> list of arrays: the roots of g in [0, 1] where g changes sign from - to +"""
    out = [np.empty(0) for _ in range(len(c))]
    ok = np.abs(c[:, 5]) > 0
    comp = np.zeros((len(c), 5, 5))
    comp[:, 1:, :-1] = np.eye(4)
    comp[:, :, -1] = -c[:, :5] / np.where(ok, c[:, 5], 1.0)[:, None]
    lam = np.linalg.eigvals(comp)
    for e in np.flatnonzero(ok):
        r = lam[e]
        r = np.real(r[(np.abs(np.imag(r)) < 1e-5) & (np.real(r) > -1e-6) & (np.real(r) < 1 + 1e-6)])
        for _ in range(4):                              # Newton polish on the power form
            g, dg = _polyval(c[e], r)
            r = r - np.where(dg != 0, g / np.where(dg != 0, dg, 1.0), 0.0)
        g, dg = _polyval(c[e], r)
        r = np.sort(r[(dg > 0) & (r >= 0.0) & (r <= 1.0)])
        out[e] = r[np.concatenate([[True], np.diff(r) > 1e-12])] if r.size else r
    for e in np.flatnonzero(~ok):                       # degenerate (dp' constant along a line): np.roots
        r = np.roots(c[e][::-1])
        r = np.real(r[np.abs(np.imag(r)) < 1e-9])
        g, dg = _polyval(c[e], r)
        out[e] = np.sort(r[(dg > 0) & (r >= 0.0) & (r <= 1.0)])
    return out


def interval_events(qi0, qi1, qj0, qj1, h, thr, first, last):
    """m pair-intervals ([m, 6] each; first / last bool [m]) -> list of m lists of (s, d, v).  thr = inf: every minimum."""
    A = cubic(qi0, qi1, qj0, qj1, h)
    c = quintic(A)
    roots = rising_roots(c)
    g0, g1 = c[:, 0], c.sum(axis=1)
    res = []
    for e in range(len(c)):
        ss = list(roots[e][roots[e] < 1.0]) if not last[e] else list(roots[e])
        if first[e] and g0[e] > 0:
            ss = [0.0] + ss
        if last[e] and not g1[e] > 0:
            ss = ss + [1.0]
        ev = []
        for s in ss:
            p = ((A[3, e] * s + A[2, e]) * s + A[1, e]) * s + A[0, e]
            v = (3 * A[3, e] * s + 2 * A[2, e]) * s + A[1, e]
            d = float(np.linalg.norm(p))
            if d < thr:
                ev.append((float(s), d, float(np.linalg.norm(v)) / h))
        res.append(ev)
    return res


def screen(X, D, thr):
    """Brute force over every pair i < j and interval: X [N,6,T] SI -> structured events sorted by (i, j, t_ca) as a
    list of (i, j, k, t_ca, d_min, v_rel), and skipped [N]"""
    N, _, T = X.shape
    h = D / (T - 1)
    fin = np.isfinite(X).all(axis=1)
    okint = fin[:, :-1] & fin[:, 1:]
    skipped = (~okint).sum(axis=1).astype(np.int32)
    events = []
    for i in range(N - 1):
        j = np.arange(i + 1, N)
        qi0 = np.broadcast_to(X[i, :, :-1].T, (len(j), T - 1, 6))
        qi1 = np.broadcast_to(X[i, :, 1:].T, (len(j), T - 1, 6))
        qj0 = np.transpose(X[j, :, :-1], (0, 2, 1))
        qj1 = np.transpose(X[j, :, 1:], (0, 2, 1))
        with np.errstate(invalid="ignore", over="ignore"):
            A = cubic(qi0, qi1, qj0, qj1, h)
            lb = f_lower_bound(A)
        cand = np.argwhere((lb <= thr * thr * (1 + 1e-6)) & okint[i][None, :] & okint[j])
        if not len(cand):
            continue
        jj, kk = cand[:, 0], cand[:, 1]
        evs = interval_events(qi0[jj, kk], qi1[jj, kk], qj0[jj, kk], qj1[jj, kk], h, thr, kk == 0, kk == T - 2)
        for e, ev in enumerate(evs):
            for s, d, v in ev:
                events.append((i, int(j[jj[e]]), int(kk[e]), kk[e] * h + s * h, d, v))
    events.sort(key=lambda r: (r[0], r[1], r[3]))
    return events, skipped


def pick_threshold(X, D, want, rel=1e-6):
    """a threshold near `want` at least `rel` relative away from every d_min of the brute force"""
    ev, _ = screen(X, D, want * 1.01)
    dmins = np.array([r[4] for r in ev])
    thr = float(want)
    for _ in range(1000):
        if dmins.size == 0 or np.min(np.abs(dmins - thr)) > rel * thr:
            return thr
        thr *= 1.0 + 7.3e-6
    raise AssertionError("no threshold clear of the minima")


def circular_state(a, inc, raan, u):
    """SI state on a circular orbit of radius a: inclination inc, node raan, argument of latitude u"""
    n_vec = np.array([np.cos(raan), np.sin(raan), 0.0])
    w = np.array([-np.sin(raan) * np.cos(inc), np.cos(raan) * np.cos(inc), np.sin(inc)])
    v = np.sqrt(MU_EARTH / a)
    return np.concatenate([a * (np.cos(u) * n_vec + np.sin(u) * w), v * (-np.sin(u) * n_vec + np.cos(u) * w), [500.0]])


def shell(N, n_planes=16, inc=np.radians(53.0), a=6.921e6, seed=0):
    """N satellites in n_planes planes of one shell, random phases -> SI states [N, 7]"""
    rng = np.random.default_rng(seed)
    return np.array([circular_state(a * (1 + 1e-4 * rng.standard_normal()), inc, 2 * np.pi * (s % n_planes) / n_planes,
                                    rng.uniform(0, 2 * np.pi)) for s in range(N)])


def fly(states, D, T, units=False):
    """SI initial states [N, 7] flown for D seconds (two-body, the reference's RK45 restated in C), T samples ->
    (y [N,7,T] normalized, tf, const): one SatelliteScale of satellite 0 (tf scalar), or with units=True every satellite
    in its own (tf_s = D / s0_s)."""
    from mpconstellation_b200.model import SatelliteScale
    from oracle import c_oracle as C
    if not units:
        sc = SatelliteScale(x=states[0])
        const = sc.get_normalized_constants()
        y0 = np.array([sc.normalize_state(x) for x in states])
        tf = D / sc._s0
        y, _, st, _, _ = C.propagate_batch_rk45(y0, tf, const, include_drag=False, include_J2=False, T=T)
        assert st.max() == 0
        return y, tf, const
    y = np.empty((len(states), 7, T))
    consts, tfs = [], []
    for s, x in enumerate(states):
        sc = SatelliteScale(x=x)
        c = sc.get_normalized_constants()
        ys, _, st, _, _ = C.propagate_batch_rk45(sc.normalize_state(x)[None], D / sc._s0, c, include_drag=False,
                                                  include_J2=False, T=T)
        assert st.max() == 0
        y[s] = ys[0]
        consts.append(c)
        tfs.append(D / sc._s0)
    return y, np.array(tfs), consts


def renormalize(X, states):
    """SI trajectories X [N,6,T] -> the same trajectories in each satellite's own units: (y [N,7,T], tf [N], consts) for a
    duration D to be passed as tf_s = D / s0_s by the caller (tf returned as 1 / s0_s)"""
    from mpconstellation_b200.model import SatelliteScale
    N, _, T = X.shape
    y = np.empty((N, 7, T))
    consts, inv_s0 = [], []
    for s in range(N):
        sc = SatelliteScale(x=states[s])
        y[s, 0:3] = X[s, 0:3] / sc._r0
        y[s, 3:6] = X[s, 3:6] / sc._v0
        y[s, 6] = 1.0
        consts.append(sc.get_normalized_constants())
        inv_s0.append(1.0 / sc._s0)
    return y, np.array(inv_s0), consts


def match(got, ref, h, rel=1e-9, t_tol=1e-6):
    """got / ref: lists of (i, j, k, t_ca, d_min, v_rel) sorted -> raises unless the sets agree"""
    assert len(got) == len(ref), (len(got), len(ref))
    for g, r in zip(got, ref):
        assert g[0:3] == r[0:3], (g, r)
        assert abs(g[3] - r[3]) <= t_tol * h, (g, r)
        assert abs(g[4] - r[4]) <= max(rel * r[4], 1e-6), (g, r)
        assert abs(g[5] - r[5]) <= max(1e-7 * r[5], 1e-6), (g, r)
