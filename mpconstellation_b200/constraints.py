"""Optimizer.get_constraint_terms (optimizer.py:80-170) for a batch of satellites, on the GPU.

This is the step that follows the discretization inside Optimizer.solve_OPT (optimizer.py:243-262): unit vectors
of the reference positions / thrusts and the linearised circular-orbit terminal conditions.  The reference's
formulas are mirrored literally, including its inverted `ubar_hat` mask (optimizer.py:137-138) and the operator
precedence of `Dv_h_hat` (optimizer.py:121) -- they define what the optimizer is handed.
"""
import ctypes

import numpy as np

from . import _lib
from .batch import _counts, _ctx, _f64, _lock

KEYS = ['rbar_hat', 'ubar_hat', 'rf_hat', 'Vc', 'DrVc', 'DrVc_rbar', 'Vt', 'DrVt_DvVt', 'DrVt_DvVt_bar',
        'Vr', 'DrVr_DvVr', 'DrVr_DvVr_bar', 'Vn', 'DrVn_DvVn', 'DrVn_DvVn_bar']    # optimizer.py:101-104


def _split_final(fin):
    """[N,32] terminal block -> {key: [N] or [N,len]} views (layout: include/mpc_b200.h MPC_FT_*)."""
    out = {}
    for key, (off, ln) in _lib.FINAL_TERM_LAYOUT.items():
        out[key] = fin[:, off] if ln == 0 else fin[:, off:off + ln]
    return out


def constraint_terms_batch(x, u, const, device=0, K=None):
    """x [N,7,K], u [N,3,Ku] (host arrays) -> dict of stacked arrays: rbar_hat [N,3,K-1], ubar_hat [N,3,Ku],
    rf_hat [N,3], Vc [N], DrVc [N,3], ... with the reference's keys.

    K = int array [N]: a ragged batch (Linearization.K) -- satellite s on its own K_s <= x.shape[2] nodes (the first K_s
    columns of x[s], u[s]; u must be on the nodes of x), one launch for all.  rbar_hat / ubar_hat keep the padded shapes
    with NaN past K_s - 1 / K_s, and the terminal terms come from node K_s - 1.

    const: one Constants bag, or a sequence of N (satellite s in the units of its own scale; the terminal terms read its
    MU).  N bags that agree bit for bit take the single-constant launch; otherwise u must be on the nodes of x."""
    ctx = _ctx(device)
    x = _f64(x)
    u = _f64(u)
    if x.ndim != 3 or x.shape[1] != 7 or x.shape[2] < 2:
        raise ValueError(f"x must be [N,7,K] with K >= 2, got {x.shape}")
    N, _, Kx = x.shape
    if u.ndim != 3 or u.shape[:2] != (N, 3) or u.shape[2] < 1:
        raise ValueError(f"u must be [N,3,Ku], got {u.shape}")
    Ku = u.shape[2]
    K_sat = None
    if K is not None:
        K_sat = _counts(K, N, Kx, "K")
        if Ku != Kx:
            raise ValueError("a ragged batch needs u on the nodes of x ([N,3,Kmax])")
    psc, const = _lib.sat_consts(const, N)
    if psc is not None and Ku != Kx:
        raise ValueError("per-satellite constants need u on the nodes of x ([N,3,K])")
    rbar = np.empty((N, 3, Kx - 1))
    ubar = np.empty((N, 3, Ku))
    fin = np.empty((N, _lib.FINAL_TERMS))
    with _lock(device):
        if psc is not None:
            _lib.check(_lib.lib().mpc_constraint_terms_units_host(ctx, _lib.addr(x), _lib.addr(u), N, Kx, _lib.addr(K_sat), psc,
                                                                  _lib.addr(rbar), _lib.addr(ubar), _lib.addr(fin)))
        elif K_sat is not None:
            _lib.check(_lib.lib().mpc_constraint_terms_ragged_host(ctx, _lib.addr(x), _lib.addr(u), N, Kx, _lib.addr(K_sat),
                                                                   float(const.MU), _lib.addr(rbar), _lib.addr(ubar),
                                                                   _lib.addr(fin)))
        else:
            _lib.check(_lib.lib().mpc_constraint_terms_host(ctx, _lib.addr(x), _lib.addr(u), N, Kx, Ku, float(const.MU),
                                                            _lib.addr(rbar), _lib.addr(ubar), _lib.addr(fin)))
    out = {"rbar_hat": rbar, "ubar_hat": ubar}
    out.update(_split_final(fin))
    return out


def constraint_terms_device(x, u, const, rbar_hat=None, ubar_hat=None, final_terms=None, K=None, first=None):
    """Device form: x [N,7,K], u [N,3,Ku] float64 CUDA tensors; enqueued on torch's current stream.
    Returns (rbar_hat [N,3,K-1], ubar_hat [N,3,Ku], final_terms [N,32]).
    K = int array [N] (host): a ragged batch as in constraint_terms_batch; `first` is an int64 CUDA tensor [N+1] the call
    fills with the prefix sums of K_s - 1 (allocated when None).  The padding columns of the outputs are not written.
    const: one Constants bag or a sequence of N, as in constraint_terms_batch."""
    import torch
    N, _, Kx = x.shape
    Ku = u.shape[2]
    assert x.is_cuda and x.dtype == torch.float64 and x.is_contiguous() and u.is_contiguous() and u.shape[:2] == (N, 3)
    K_sat = None
    if K is not None:
        K_sat = _counts(K, N, Kx, "K")
        if Ku != Kx:
            raise ValueError("a ragged batch needs u on the nodes of x ([N,3,Kmax])")
    psc, const = _lib.sat_consts(const, N)
    if psc is not None and Ku != Kx:
        raise ValueError("per-satellite constants need u on the nodes of x ([N,3,K])")
    if K_sat is not None and first is None:
        first = torch.empty(N + 1, dtype=torch.int64, device=x.device)
    if rbar_hat is None:
        rbar_hat = torch.empty((N, 3, Kx - 1), dtype=torch.float64, device=x.device)
    if ubar_hat is None:
        ubar_hat = torch.empty((N, 3, Ku), dtype=torch.float64, device=x.device)
    if final_terms is None:
        final_terms = torch.empty((N, _lib.FINAL_TERMS), dtype=torch.float64, device=x.device)
    stream = torch.cuda.current_stream(x.device).cuda_stream
    if psc is not None:
        scratch = torch.empty(N * _lib.SAT_SCRATCH_DOUBLES, dtype=torch.float64, device=x.device)
        _lib.check(_lib.lib().mpc_constraint_terms_units(x.data_ptr(), u.data_ptr(), N, Kx, _lib.addr(K_sat),
                                                         first.data_ptr() if first is not None else None, psc,
                                                         scratch.data_ptr(), rbar_hat.data_ptr(), ubar_hat.data_ptr(),
                                                         final_terms.data_ptr(), stream))
        scratch.record_stream(torch.cuda.current_stream(x.device))
    elif K_sat is not None:
        _lib.check(_lib.lib().mpc_constraint_terms_ragged(x.data_ptr(), u.data_ptr(), N, Kx, _lib.addr(K_sat),
                                                          first.data_ptr(), float(const.MU), rbar_hat.data_ptr(),
                                                          ubar_hat.data_ptr(), final_terms.data_ptr(), stream))
    else:
        _lib.check(_lib.lib().mpc_constraint_terms(x.data_ptr(), u.data_ptr(), N, Kx, Ku, float(const.MU),
                                                   rbar_hat.data_ptr(), ubar_hat.data_ptr(), final_terms.data_ptr(),
                                                   stream))
    return rbar_hat, ubar_hat, final_terms


def get_constraint_terms(x_bar, u_bar, const, device=0):
    """Drop-in for Optimizer.get_constraint_terms: x_bar / u_bar are the optimizer's N-element lists of (7,K) /
    (3,K) arrays; returns the same dict of N-element lists (optimizer.py:84-100).  Lists whose widths differ (every
    satellite on its own K_s nodes) take one ragged launch and return arrays of each satellite's own widths; then every
    u_bar[s] must have the width of x_bar[s]."""
    if len(x_bar) == 0:
        return {k: [] for k in KEYS}
    xs = [np.asarray(a, dtype=np.float64) for a in x_bar]
    us = [np.asarray(a, dtype=np.float64) for a in u_bar]
    n = len(xs)
    widths = np.array([a.shape[-1] for a in xs])
    if (widths == widths[0]).all():
        stacked = constraint_terms_batch(np.stack(xs), np.stack(us), const, device=device)
        return {k: [stacked[k][i] if stacked[k].ndim > 1 else float(stacked[k][i]) for i in range(n)] for k in KEYS}
    if len(us) != n or any(a.ndim != 2 or b.ndim != 2 or b.shape[1] != a.shape[1] for a, b in zip(xs, us)):
        raise ValueError("a ragged batch needs every u_bar[s] on the nodes of x_bar[s] ((3,K_s) with (7,K_s))")
    Kmax = int(widths.max())
    x = np.zeros((n, 7, Kmax))
    u = np.zeros((n, 3, Kmax))
    for s in range(n):
        x[s, :, :widths[s]], u[s, :, :widths[s]] = xs[s], us[s]
    stacked = constraint_terms_batch(x, u, const, device=device, K=widths)
    out = {"rbar_hat": [stacked["rbar_hat"][s, :, :widths[s] - 1] for s in range(n)],
           "ubar_hat": [stacked["ubar_hat"][s, :, :widths[s]] for s in range(n)]}
    for k in KEYS[2:]:
        out[k] = [stacked[k][s] if stacked[k].ndim > 1 else float(stacked[k][s]) for s in range(n)]
    return out


# ------------------------------------------------------------------ sparse dynamics constraint (optimizer.py:327-339)

NNZ_PER_ROW = 16


class DynamicsJacobian:
    """CSR form  J z = rhs  of the reference's dynamics constraint (dynamics_const_rule, optimizer.py:327-339) for N
    satellites: rows in pyomo's generation order (s, i, k), row = (s*7+i)*(K-1)+k; 16 non-zeros per row; variables
    z = [x (N,7,K) | u (N,3,K) | nu (N,7,K) | tf] flattened C-order (include/mpc_b200.h, mpc_dynamics_jacobian).

    Per-satellite form (K_sat [N], a ragged batch or counts passed to dynamics_jacobian): N independent single-satellite
    systems, each with its own final time tf_s, as every satellite's own Optimizer builds them.  Block s is the numbering
    above with N = 1, K = K_s, its rows starting at 7 first[s] and its variables z_s = [x_s (7,K_s) | u_s (3,K_s) |
    nu_s (7,K_s) | tf_s] at V_s = 17 (first[s] + s) + s, first[s] = sum_{r<s} (K_r - 1) (mpc_dynamics_jacobian_ragged)."""

    def __init__(self, values, indices, rhs, n_sats, K, K_sat=None):
        self.values, self.indices, self.rhs, self.n_sats, self.K = values, indices, rhs, n_sats, K
        self.K_sat = None if K_sat is None else np.asarray(K_sat, dtype=np.int64)
        if self.K_sat is None:
            self.rows = n_sats * 7 * (K - 1)
            self.cols = 17 * n_sats * K + 1
        else:
            self.first = np.concatenate([[0], np.cumsum(self.K_sat - 1)])
            self.rows = int(7 * self.first[-1])
            self.cols = int(17 * (self.first[-1] + n_sats) + n_sats)

    @property
    def indptr(self):
        return np.arange(self.rows + 1, dtype=np.int64) * NNZ_PER_ROW

    def block(self, s):
        """(rows, cols) slices of satellite s's diagonal block (per-satellite form)"""
        f, Ks = int(self.first[s]), int(self.K_sat[s])
        V = 17 * (f + s) + s
        return slice(7 * f, 7 * (f + Ks - 1)), slice(V, V + 17 * Ks + 1)

    def pack(self, x, u, nu, tf):
        """decision vector z from x [N,7,K], u [N,3,K], nu [N,7,K] (last column unused by the constraint), tf scalar.
        Per-satellite form: x, u, nu are N-element sequences of (7,K_s), (3,K_s), (7,K_s) arrays (or padded arrays:
        the first K_s columns are taken), tf one final time per satellite."""
        if self.K_sat is None:
            return np.concatenate([np.ravel(x), np.ravel(u), np.ravel(nu), [float(tf)]])
        tf = np.broadcast_to(np.asarray(tf, dtype=np.float64), (self.n_sats,))
        parts = []
        for s, Ks in enumerate(self.K_sat):
            for a, m in ((x[s], 7), (u[s], 3), (nu[s], 7)):
                a = np.asarray(a, dtype=np.float64)[:, :Ks]
                if a.shape != (m, Ks):
                    raise ValueError(f"satellite {s}: expected ({m},{Ks}) columns, got {a.shape}")
                parts.append(a.ravel())
            parts.append([tf[s]])
        return np.concatenate(parts)

    def residual(self, z):
        """J z - rhs, reshaped [N,7,K-1] (per-satellite form: a list of [7,K_s-1]): zero where the reference's
        constraint holds"""
        v = np.asarray(self.values).reshape(self.rows, NNZ_PER_ROW)
        c = np.asarray(self.indices).reshape(self.rows, NNZ_PER_ROW)
        r = (v * np.asarray(z)[c]).sum(axis=1) - np.asarray(self.rhs)
        if self.K_sat is None:
            return r.reshape(self.n_sats, 7, self.K - 1)
        return [r[self.block(s)[0]].reshape(7, int(self.K_sat[s]) - 1) for s in range(self.n_sats)]

    def to_scipy(self):
        from scipy.sparse import csr_matrix
        return csr_matrix((np.asarray(self.values), np.asarray(self.indices), self.indptr), shape=(self.rows, self.cols))


def dynamics_jacobian_device(soa, n_sats, K, pitch=None, offset=0, values=None, indices=None, rhs=None,
                             with_indices=True, K_sat=None, first=None):
    """Device form: soa is the [105, pitch] float64 CUDA tensor a discretization wrote (columns offset.. hold the
    batch).  Returns (values [rows*16] f64, indices [rows*16] i64 or None, rhs [rows] f64) CUDA tensors; enqueued on
    torch's current stream.  Between SCP iterations only the values change: pass with_indices=False.
    K_sat = int array [N] (host): the per-satellite form (DynamicsJacobian) of a ragged result of K = Kmax (or of a
    rectangular one, all counts K); `first` is an int64 CUDA tensor [N+1] the call fills (allocated when None)."""
    import torch
    pitch = soa.shape[1] if pitch is None else int(pitch)
    assert soa.is_cuda and soa.dtype == torch.float64 and soa.is_contiguous()
    if K_sat is not None:
        K_sat = _counts(K_sat, n_sats, K, "K_sat")
        rows = 7 * int((K_sat.astype(np.int64) - 1).sum())
        if first is None:
            first = torch.empty(n_sats + 1, dtype=torch.int64, device=soa.device)
    else:
        rows = n_sats * 7 * (K - 1)
    if values is None:
        values = torch.empty(rows * NNZ_PER_ROW, dtype=torch.float64, device=soa.device)
    if indices is None and with_indices:
        indices = torch.empty(rows * NNZ_PER_ROW, dtype=torch.int64, device=soa.device)
    if rhs is None:
        rhs = torch.empty(rows, dtype=torch.float64, device=soa.device)
    stream = torch.cuda.current_stream(soa.device).cuda_stream
    idx = indices.data_ptr() if indices is not None else None
    if K_sat is not None:
        _lib.check(_lib.lib().mpc_dynamics_jacobian_ragged(soa.data_ptr(), pitch, int(offset), int(n_sats), int(K),
                                                           _lib.addr(K_sat), first.data_ptr(), values.data_ptr(), idx,
                                                           rhs.data_ptr(), stream))
    else:
        _lib.check(_lib.lib().mpc_dynamics_jacobian(soa.data_ptr(), pitch, int(offset), int(n_sats), int(K),
                                                    values.data_ptr(), idx, rhs.data_ptr(), stream))
    return values, indices, rhs


def dynamics_jacobian(matrices, K=None):
    """Host form: `matrices` is a DiscretizedBatch (e.g. Linearization.matrices); the assembly runs on the GPU.
    Returns a DynamicsJacobian with numpy arrays.  With K (int array [N], e.g. Linearization.K) or a ragged `matrices`
    (K_sat set) the result is the per-satellite form: one system and one final time per satellite.  Without, it is the
    reference's multi-satellite Optimizer: one shared tf."""
    import torch
    _lib.require_gpu()
    counts = matrices.K_sat if K is None else K
    if K is not None and matrices.K_sat is not None and not np.array_equal(np.asarray(K), matrices.K_sat):
        raise ValueError("K differs from the node counts the matrices were discretized on (matrices.K_sat)")
    host = matrices.soa
    if getattr(matrices, "layout", "satmajor") == "kmajor":        # the assembly kernel reads per-satellite column blocks
        N, n = matrices.n_sats, matrices.K - 1
        host = host.reshape(_lib.MPC_OUT_ROWS, n, N).transpose(0, 2, 1).reshape(_lib.MPC_OUT_ROWS, N * n)
    soa = torch.from_numpy(np.ascontiguousarray(host)).cuda()
    K_sat = None if counts is None else _counts(counts, matrices.n_sats, matrices.K, "K")
    v, c, r = dynamics_jacobian_device(soa, matrices.n_sats, matrices.K, K_sat=K_sat)
    return DynamicsJacobian(v.cpu().numpy(), c.cpu().numpy(), r.cpu().numpy(), matrices.n_sats, matrices.K, K_sat=K_sat)
