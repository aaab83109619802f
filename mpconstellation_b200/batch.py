"""Batched entry points over the C-ABI: every (satellite, interval) / satellite is one GPU work unit.

Host arrays (numpy) go through the library's host API (chunked copy/compute pipeline); torch CUDA
tensors go through the device API on torch's current stream.  Shapes follow the reference with a
leading batch axis: x [N,7,K], u [N,3,K], tf [N] -> SoA [105, N*(K-1)].
"""
import ctypes
import math
import threading

import numpy as np

from . import _lib
from .control import ControllerSpec, spec_from

_ctx_lock = threading.Lock()
_ctxs = {}
_call_locks = {}


def _lock(device=0):
    """One lock per device context: an mpc_ctx owns ONE workspace (device buffers, events, pinned staging), and ctypes
    releases the GIL during a call, so two Python threads must not be inside host-API calls of the same ctx at once."""
    with _ctx_lock:
        return _call_locks.setdefault(device, threading.RLock())


def _ctx(device=0):
    with _ctx_lock:
        if device not in _ctxs:
            _lib.require_gpu()
            h = ctypes.c_void_p()
            _lib.check(_lib.lib().mpc_ctx_create(int(device), ctypes.byref(h)))
            _ctxs[device] = h
        return _ctxs[device]


def _f64(a, shape=None):
    a = np.ascontiguousarray(a, dtype=np.float64)
    if shape is not None and a.shape != tuple(shape):
        raise ValueError(f"expected shape {tuple(shape)}, got {a.shape}")
    return a


def _tf_vec(tf, n):
    return np.ascontiguousarray(np.broadcast_to(np.asarray(tf, dtype=np.float64), (n,)))


class DiscretizedBatch:
    """SoA result of a batched discretization plus reference-shaped views.

    soa: [105, N*(K-1)] float64 (rows: A 49 | B_kp 21 | B_kn 21 | Sigma 7 | xi 7), status: [N, K-1] int32.
    layout "satmajor": column = s (K-1) + k (per-satellite blocks); "kmajor": column = k N + s (what the streamed host
    pass propagate_discretize(layout="kmajor") writes).  sat(s) returns (A_k, B_kp, B_kn, Sigma_k, xi_k) with the shapes
    and order of Discretizer.discretize (linearize_discretize.py:390); they are views in either layout, no copy is made.
    Ragged batches (K_sat [N]: satellite s on its own K_s nodes) keep the layout of K = max K_s: satellite s owns the
    columns s (K-1) + k, k < K_s - 1, and sat(s) returns its K_s - 1 intervals; the padding columns hold NaN (status 0).
    """

    def __init__(self, soa, status, n_sats, K, layout="satmajor", K_sat=None):
        self.soa, self.status, self.n_sats, self.K, self.layout = soa, status, n_sats, K, layout
        self.K_sat = None if K_sat is None else np.asarray(K_sat, dtype=np.int32)

    def _n(self, s):
        return (self.K if self.K_sat is None else int(self.K_sat[s])) - 1

    def _rows(self, r0, nrows, s):
        n = self.K - 1
        if self.layout == "kmajor":
            return self.soa[r0:r0 + nrows, s::self.n_sats]
        return self.soa[r0:r0 + nrows, s * n:s * n + self._n(s)]

    def sat(self, s):
        n = self._n(s)
        A = self._rows(_lib.ROW_A, 49, s).T.reshape(n, 7, 7)
        Bp = self._rows(_lib.ROW_BP, 21, s).T.reshape(n, 7, 3)
        Bn = self._rows(_lib.ROW_BN, 21, s).T.reshape(n, 7, 3)
        return A, Bp, Bn, self._rows(_lib.ROW_SIGMA, 7, s), self._rows(_lib.ROW_XI, 7, s)

    def stacked(self):
        """(A[N,K-1,7,7], B_kp[N,K-1,7,3], B_kn[N,K-1,7,3], Sigma[N,7,K-1], xi[N,7,K-1]) as views (ragged: padded, NaN
        past K_s - 1)."""
        N, n = self.n_sats, self.K - 1
        if self.layout == "kmajor":
            v = self.soa.reshape(_lib.MPC_OUT_ROWS, n, N).transpose(0, 2, 1)      # [105, N, n], strided
        else:
            v = self.soa.reshape(_lib.MPC_OUT_ROWS, N, n)
        A = v[0:49].transpose(1, 2, 0).reshape(N, n, 7, 7)
        Bp = v[49:70].transpose(1, 2, 0).reshape(N, n, 7, 3)
        Bn = v[70:91].transpose(1, 2, 0).reshape(N, n, 7, 3)
        return A, Bp, Bn, v[91:98].transpose(1, 0, 2), v[98:105].transpose(1, 0, 2)

    def raise_on_error(self):
        raise_on_status(self.status)


def raise_on_status(status, atmosphere=None):
    st = np.asarray(status)
    if st.size and st.max() != 0:
        idx = np.argwhere(st != 0)[0]
        code = int(st[tuple(idx)])
        if code == _lib.ST_ATMO:
            rng = "" if atmosphere is None else f" [{atmosphere.h_min:.6g}, {atmosphere.h_max:.6g}] m"
            raise ValueError(f"satellite {int(idx[0])}: the altitude left the range of the fitted atmosphere{rng}; "
                             "the density is not extrapolated")
        if code == _lib.ST_MASS:
            # same exception type / text as simulator.py:135-136
            raise Exception(f"ERROR: INVALID SATELLITE MASS: non-positive mass at unit {tuple(int(i) for i in idx)}")
        if code == _lib.ST_STEP:
            raise RuntimeError(f"adaptive integration failed (step size underflow) at unit {tuple(int(i) for i in idx)}")
        raise FloatingPointError(f"non-finite result at unit {tuple(int(i) for i in idx)}")


def _counts(c, n, cmax, what):
    """per-satellite node / sample counts as int32 [n], each 2 <= c <= cmax"""
    c = np.ascontiguousarray(c, dtype=np.int32)
    if c.shape != (n,):
        raise ValueError(f"{what} must have shape [{n}], got {c.shape}")
    if n and (c.min() < 2 or c.max() > cmax):
        raise ValueError(f"every {what} must be >= 2 and <= {cmax}")
    return c


def _rk23(adaptive, include_drag=False, ugrid=False):
    """True when adaptive asks for scipy's RK23 (adaptive["method"]; missing or "RK45": the RK45 replay).  Raises
    NotImplementedError, before any device work, for another method and for what RK23 has no device form of."""
    method = (adaptive or {}).get("method", "RK45")
    if method == "RK45":
        return False
    if method != "RK23":
        raise NotImplementedError(f"adaptive method {method!r}: the device replays scipy's RK45 and RK23 only; "
                                  "DOP853 and the implicit methods have no device form and there is no CPU fallback")
    if include_drag:
        raise NotImplementedError("RK23 with include_drag: the drag linearisation is replayed with RK45 only")
    if ugrid:
        raise NotImplementedError("RK23 with u on its own grid: the RK23 replay needs u on the nodes of x")
    return True


def discretize_batch(x, u, tf, const, include_J2=False, include_drag=False, n_sub=100, out=None, status=None,
                     device=0, check=True, adaptive=None, disc_drag=None, K=None):
    """Discretize every interval of every satellite in one launch sequence (host arrays).

    x [N,7,K], u [N,3,K], tf scalar or [N]; `out` may be a preallocated (ideally pinned) [105, N*(K-1)]
    array.  Returns a DiscretizedBatch.  ref: linearize_discretize.py:334-390 / :8-82.

    adaptive=None: fixed-step fourth-order Runge-Kutta-Nystrom, trapezoid on n_sub+1 nodes (the reference's
    use_uniform_steps=True node set).  adaptive=dict(rtol=1e-3, atol=1e-6, max_step=1e-2): the reference's
    default mode, quadrature on the steps scipy's RK45 controller accepts; the result carries `.n_nodes`.

    include_drag=True needs disc_drag=(CD, rho): const.CD and the (constant) value of rho_func the reference's drag
    branch reads (linearize_discretize.py:162-168); without them the call is rejected like the reference's.

    adaptive=dict(method="RK23", ...): the same with scipy's RK23 controller (Discretizer.ivp_solver = 'RK23'); u on the
    nodes of x, no drag.  A missing method or "RK45" is the RK45 replay; any other method raises NotImplementedError.

    K=None: every satellite on the K = x.shape[2] nodes.  K = int array [N]: a ragged batch -- satellite s on its own
    K_s <= x.shape[2] nodes (the first K_s columns of x[s], u[s]), one launch for all; the result keeps the layout of
    Kmax = x.shape[2] with NaN in the padding columns (DiscretizedBatch.sat(s) returns K_s - 1 intervals).  u must be on
    the nodes of x, and the drag linearisation is not available for ragged batches.

    const: one Constants bag, or a sequence of N -- satellite s linearized in the units of its own scale (model.
    sat_units), one launch for the batch, as N single-satellite calls would give it.  N bags that agree bit for bit in
    the seven per-scale fields take the single-constant launches.  Per-satellite constants need u on the nodes of x and
    are not available with include_drag.
    """
    rk23 = adaptive is not None and _rk23(adaptive, include_drag, np.ndim(u) == 3 and np.ndim(x) == 3 and
                                          np.shape(u)[2] != np.shape(x)[2])
    ctx = _ctx(device)
    counts, K = K, None
    x = _f64(x)
    if x.ndim != 3 or x.shape[1] != 7:
        raise ValueError(f"x must be [N,7,K], got {x.shape}")
    N, _, K = x.shape
    u = _f64(u)
    if u.ndim != 3 or u.shape[:2] != (N, 3) or u.shape[2] < 2:
        raise ValueError(f"u must be [N,3,Ku] with Ku >= 2, got {u.shape}")
    Ku = u.shape[2]                      # Ku != K: u lives on its own grid (linearize_discretize.py:308-315)
    tfv = _tf_vec(tf, N)
    n_int = N * (K - 1)
    if out is None:
        out = _lib.pinned_empty((_lib.MPC_OUT_ROWS, n_int))
    elif out.shape != (_lib.MPC_OUT_ROWS, n_int) or out.dtype != np.float64 or not out.flags["C_CONTIGUOUS"]:
        raise ValueError("out must be C-contiguous float64 [105, N*(K-1)]")
    if status is None:
        status = np.zeros(n_int, dtype=np.int32)
    psc, const = _units_of(const, N, Ku != K, include_drag)
    p = _lib.make_params(const, include_J2, include_drag, disc_drag=disc_drag)
    n_nodes = None
    K_sat = None
    if counts is not None:
        K_sat = _counts(counts, N, K, "K")
        if Ku != K:
            raise ValueError("a ragged batch needs u on the nodes of x ([N,3,Kmax])")
    with _lock(device):
        if rk23:
            n_nodes = np.zeros(n_int, dtype=np.int32)
            _lib.check(_lib.lib().mpc_discretize_batch_rk23_host(
                ctx, _lib.addr(x), _lib.addr(u), _lib.addr(tfv), ctypes.byref(p), psc, N, K, _lib.addr(K_sat),
                float(adaptive.get("rtol", 1e-3)), float(adaptive.get("atol", 1e-6)), float(adaptive.get("max_step", 1e-2)),
                _lib.addr(out), _lib.addr(status), _lib.addr(n_nodes)))
        elif psc is not None:
            ad = adaptive or {}
            n_nodes = np.zeros(n_int, dtype=np.int32) if adaptive is not None else None
            _lib.check(_lib.lib().mpc_discretize_batch_units_host(
                ctx, _lib.addr(x), _lib.addr(u), _lib.addr(tfv), ctypes.byref(p), psc, N, K, _lib.addr(K_sat),
                int(adaptive is not None), int(n_sub), float(ad.get("rtol", 1e-3)), float(ad.get("atol", 1e-6)),
                float(ad.get("max_step", 1e-2)), _lib.addr(out), _lib.addr(status), _lib.addr(n_nodes)))
        elif K_sat is not None:
            ad = adaptive or {}
            n_nodes = np.zeros(n_int, dtype=np.int32) if adaptive is not None else None
            _lib.check(_lib.lib().mpc_discretize_batch_ragged_host(
                ctx, _lib.addr(x), _lib.addr(u), _lib.addr(tfv), ctypes.byref(p), N, K, _lib.addr(K_sat),
                int(adaptive is not None), int(n_sub), float(ad.get("rtol", 1e-3)), float(ad.get("atol", 1e-6)),
                float(ad.get("max_step", 1e-2)), _lib.addr(out), _lib.addr(status), _lib.addr(n_nodes)))
        elif Ku != K:
            ad = adaptive or {}
            n_nodes = np.zeros(n_int, dtype=np.int32) if adaptive is not None else None
            _lib.check(_lib.lib().mpc_discretize_batch_ugrid_host(
                ctx, _lib.addr(x), _lib.addr(u), Ku, _lib.addr(tfv), ctypes.byref(p), N, K, int(adaptive is not None),
                int(n_sub), float(ad.get("rtol", 1e-3)), float(ad.get("atol", 1e-6)), float(ad.get("max_step", 1e-2)),
                _lib.addr(out), _lib.addr(status), _lib.addr(n_nodes)))
        elif adaptive is None:
            _lib.check(_lib.lib().mpc_discretize_batch_host(ctx, _lib.addr(x), _lib.addr(u), _lib.addr(tfv),
                                                            ctypes.byref(p), N, K, int(n_sub), _lib.addr(out),
                                                            _lib.addr(status)))
        else:
            n_nodes = np.zeros(n_int, dtype=np.int32)
            _lib.check(_lib.lib().mpc_discretize_batch_adaptive_host(
                ctx, _lib.addr(x), _lib.addr(u), _lib.addr(tfv), ctypes.byref(p), N, K, float(adaptive.get("rtol", 1e-3)),
                float(adaptive.get("atol", 1e-6)), float(adaptive.get("max_step", 1e-2)), _lib.addr(out), _lib.addr(status),
                _lib.addr(n_nodes)))
    res = DiscretizedBatch(out, status.reshape(N, K - 1), N, K, K_sat=K_sat)
    res.n_nodes = None if n_nodes is None else n_nodes.reshape(N, K - 1)
    if check:
        res.raise_on_error()
    return res


def _units_of(const, n, ugrid=False, drag=False):
    """(mpc_sat_consts [n] or None, the bag for mpc_params): see _lib.sat_consts; rejects what has no per-satellite form"""
    psc, one = _lib.sat_consts(const, n)
    if psc is None:
        return None, one
    if ugrid:
        raise ValueError("per-satellite constants need u on the nodes of x (no u on its own grid)")
    if drag:
        raise ValueError("the drag linearisation (include_drag=True) is not available with per-satellite constants")
    return psc, list(const)[0]


def _rk4_units(const, n, n_sub):
    """per-satellite constants need the reference integrator: raise before any device work when n_sub asks for RK4"""
    if n_sub not in (None, 0) and _lib.sat_consts(const, n)[0] is not None:
        raise ValueError("per-satellite constants need the reference integrator (n_sub=None); the fixed-step RK4 "
                         "propagator has no per-satellite form")


def _atmosphere(atmosphere, include_drag, n_sub):
    """the mpc_atmosphere of an Atmosphere (None: the constant density), after the checks that raise before any device
    work: the model is the density of the drag, flown by the reference integrator"""
    if atmosphere is None:
        return None
    from .atmosphere import Atmosphere
    if not isinstance(atmosphere, Atmosphere):
        raise ValueError(f"atmosphere must be an Atmosphere (fit_atmosphere), got {type(atmosphere).__name__}")
    if not include_drag:
        raise ValueError("an atmosphere is the density of the drag: it needs include_drag=True")
    if n_sub not in (None, 0):
        raise ValueError("an atmosphere needs the reference integrator (n_sub=None); the fixed-step RK4 propagator "
                         "flies the constant density only")
    return atmosphere.struct()


def _no_atmosphere(atmosphere, what):
    if atmosphere is not None:
        raise ValueError(f"{what} flies the constant density only: propagate with propagate_batch[_device]"
                         "(atmosphere=...) instead")


def _ctrl_struct(spec, n_sats, table_addr=None, end_tau_addr=None):
    c = _lib.MpcController()
    c.kind = spec.kind
    c.thrust[0], c.thrust[1], c.thrust[2] = [float(t) for t in spec.thrust]
    keep = None
    if np.ndim(spec.end_tau) == 0:
        c.end_tau = float(spec.end_tau)
    else:
        et = np.ascontiguousarray(spec.end_tau, dtype=np.float64)
        if et.shape != (n_sats,):
            raise ValueError("per-satellite end_tau must have shape [N]")
        c.end_tau = float(et[0])
        c.end_tau_per_sat = end_tau_addr if end_tau_addr is not None else et.ctypes.data
        keep = [et]
    if spec.kind == _lib.CTRL_SEQUENCE:
        tab = spec.table
        if tab.ndim == 3 and tab.shape[0] != n_sats:
            raise ValueError("per-satellite sequence table must be [N,3,Ku]")
        c.table_len = tab.shape[-1]
        c.table_per_sat = int(tab.ndim == 3)
        keep = [keep, tab]
        c.table = table_addr if table_addr is not None else tab.ctypes.data
    return c, keep


def _rectangular_law(spec):
    if spec.kind == _lib.CTRL_SEQUENCE and spec.table_len is not None:
        raise ValueError("per-satellite table lengths (ControllerSpec.table_len) are taken by propagate_batch only")


def default_n_sub(T, max_step=0.001):
    """RK4 steps between samples so that the step in tau is <= max_step (simulator.py:186)."""
    if T < 2:
        return 1
    return max(1, int(math.ceil(1.0 / (max_step * (T - 1)) - 1e-9)))


def propagate_batch(y0, tf, controller, const, include_drag=True, include_J2=True, T=100, n_sub=None,
                    want_u=True, device=0, check=True, y_out=None, u_out=None, rk45=None, n_steps=None, atmosphere=None):
    """Propagate N satellites over tau in [0,1] and sample at linspace(0,1,T) (host arrays).

    y0 [N,7] normalized states; returns (y [N,7,T], u [N,3,T] or None, t [T], status [N]).
    ref: simulator.py:164-189 (+ extract_uk, linearize_discretize.py:393-411).

    T = int array [N]: satellite s sampled at linspace(0, 1, T_s) (the reference's int(base_res * tf_s) of every
    satellite's own horizon), one launch for all; y / u are [N,7,Tmax] / [N,3,Tmax] and t is [N,Tmax], NaN past T_s.
    The steps do not depend on the samples (n_steps as for a rectangular run).  Reference integrator only (n_sub=None),
    as is a sequence law with per-satellite table lengths (ControllerSpec.table_len).

    n_sub=None (default): the reference's own integrator, replayed on the device -- scipy's RK45 with its step-size
    controller exactly as simulator.py:185-187 calls it (max_step=0.001, rtol 1e-3, atol 1e-6, dense-output samples);
    `rk45=dict(rtol=, atol=, max_step=)` overrides those numbers, `n_steps` (int32 [N]) receives the steps attempted.
    n_sub >= 1: fixed-step RK4 with n_sub steps between samples (default_n_sub(T) mirrors max_step=0.001).

    const: one Constants bag, or a sequence of N (satellite s integrated in the units of its own scale, one launch; N bags
    that agree bit for bit take the single-constant launch).  Per-satellite constants need the reference integrator.

    atmosphere: an Atmosphere (fit_atmosphere) -- the drag's density rho(h) at every stage instead of the constant of
    Simulator.get_atmo_density, satellite s at the altitude |r| r0 - R_EARTH of its own scale.  Needs include_drag and
    the reference integrator (ValueError otherwise); a satellite that leaves the fitted range raises ValueError.
    """
    y0 = _f64(y0)
    if y0.ndim != 2 or y0.shape[1] != 7:
        raise ValueError(f"y0 must be [N,7], got {y0.shape}")
    N = y0.shape[0]
    _rk4_units(const, N, n_sub)
    atmo = _atmosphere(atmosphere, include_drag, n_sub)
    ctx = _ctx(device)
    spec = spec_from(controller)
    T_sat = tab_len = None
    if spec.kind == _lib.CTRL_SEQUENCE and spec.table_len is not None:
        tab_len = _counts(spec.table_len, N, np.shape(spec.table)[-1], "table_len")
    if np.ndim(T) != 0:
        T_sat = _counts(T, N, int(np.max(T)) if N else 2, "T")
        T = int(T_sat.max()) if N else 2
    T = int(T)
    if (T_sat is not None or tab_len is not None) and n_sub not in (None, 0):
        raise ValueError("per-satellite sample counts / table lengths need the reference integrator (n_sub=None)")
    tfv = _tf_vec(tf, N)
    if n_sub is None:
        n_sub = 0
    if n_sub != 0 and rk45 is not None:
        raise ValueError("rk45 options only apply to the reference integrator (n_sub=None)")
    y = y_out if y_out is not None else _lib.pinned_empty((N, 7, T))
    uo = (u_out if u_out is not None else _lib.pinned_empty((N, 3, T))) if want_u else None
    status = np.zeros(N, dtype=np.int32)
    if T_sat is None:
        t = np.linspace(0, 1, T)
    else:
        t = np.full((N, T), np.nan)
        for s_, ts in enumerate(T_sat):
            t[s_, :ts] = np.linspace(0, 1, ts)
    if N == 0 or T == 0:
        return y, uo, t, status
    psc, const = _units_of(const, N)
    p = _lib.make_params(const, include_J2, include_drag)
    c, _keep = _ctrl_struct(spec, N)
    if n_sub == 0:
        o = rk45 or {}
        if n_steps is not None and (n_steps.shape != (N,) or n_steps.dtype != np.int32):
            raise ValueError("n_steps must be int32 [N]")
        with _lock(device):
            if atmo is not None:
                _lib.check(_lib.lib().mpc_propagate_batch_rk45_atmo_host(
                    ctx, _lib.addr(y0), _lib.addr(tfv), ctypes.byref(p), psc, ctypes.byref(c), N, T, _lib.addr(T_sat),
                    _lib.addr(tab_len), float(o.get("rtol", 1e-3)), float(o.get("atol", 1e-6)), float(o.get("max_step", 1e-3)),
                    _lib.addr(y), _lib.addr(uo), _lib.addr(status), _lib.addr(n_steps), ctypes.byref(atmo)))
            elif psc is not None:
                _lib.check(_lib.lib().mpc_propagate_batch_rk45_units_host(
                    ctx, _lib.addr(y0), _lib.addr(tfv), ctypes.byref(p), psc, ctypes.byref(c), N, T, _lib.addr(T_sat),
                    _lib.addr(tab_len), float(o.get("rtol", 1e-3)), float(o.get("atol", 1e-6)), float(o.get("max_step", 1e-3)),
                    _lib.addr(y), _lib.addr(uo), _lib.addr(status), _lib.addr(n_steps)))
            elif T_sat is not None or tab_len is not None:
                counts = T_sat if T_sat is not None else np.full(N, T, dtype=np.int32)
                _lib.check(_lib.lib().mpc_propagate_batch_rk45_ragged_host(
                    ctx, _lib.addr(y0), _lib.addr(tfv), ctypes.byref(p), ctypes.byref(c), N, T, _lib.addr(counts),
                    _lib.addr(tab_len), float(o.get("rtol", 1e-3)), float(o.get("atol", 1e-6)), float(o.get("max_step", 1e-3)), _lib.addr(y),
                    _lib.addr(uo), _lib.addr(status), _lib.addr(n_steps)))
            else:
                _lib.check(_lib.lib().mpc_propagate_batch_rk45_host(
                    ctx, _lib.addr(y0), _lib.addr(tfv), ctypes.byref(p), ctypes.byref(c), N, T, float(o.get("rtol", 1e-3)),
                    float(o.get("atol", 1e-6)), float(o.get("max_step", 1e-3)), _lib.addr(y), _lib.addr(uo),
                    _lib.addr(status), _lib.addr(n_steps)))
    else:
        with _lock(device):
            _lib.check(_lib.lib().mpc_propagate_batch_host(ctx, _lib.addr(y0), _lib.addr(tfv), ctypes.byref(p),
                                                           ctypes.byref(c), N, T, int(n_sub), _lib.addr(y),
                                                           _lib.addr(uo), _lib.addr(status)))
    if check:
        raise_on_status(status, atmosphere)
    return y, uo, t, status


def propagate_discretize(y0, tf, controller, const, T, prop_drag=False, prop_J2=False, disc_J2=False,
                         n_sub_prop=None, n_sub_disc=100, out=None, y_out=None, u_out=None, device=0, check=True,
                         status=None, layout="satmajor", atmosphere=None):
    """One SCP linearization pass on the device: propagate -> extract_uk -> discretize, the reference
    trajectory staying in HBM between the kernels (control.py:180-188 pattern).  K = T.
    layout="kmajor": the matrices come back in the k-major layout (DiscretizedBatch views hide it) through the streamed
    pass -- windows along k gated on the propagation's progress, every window read back while the next one runs.
    Returns (DiscretizedBatch, y [N,7,T], u [N,3,T]).  An atmosphere raises ValueError: the fused pass flies the constant
    density only."""
    _no_atmosphere(atmosphere, "propagate_discretize")
    ctx = _ctx(device)
    y0 = _f64(y0)
    N = y0.shape[0]
    T = int(T)
    spec = spec_from(controller)
    _rectangular_law(spec)
    tfv = _tf_vec(tf, N)
    n_int = N * (T - 1)
    if n_sub_prop is None:
        n_sub_prop = 0                    # the reference's RK45, replayed (see propagate_batch)
    if out is None:
        out = _lib.pinned_empty((_lib.MPC_OUT_ROWS, n_int))
    y = y_out if y_out is not None else _lib.pinned_empty((N, 7, T))
    uo = u_out if u_out is not None else _lib.pinned_empty((N, 3, T))
    if status is None:
        status = np.zeros(n_int, dtype=np.int32)
    elif status.shape != (n_int,) or status.dtype != np.int32 or not status.flags["C_CONTIGUOUS"]:
        raise ValueError("status must be C-contiguous int32 [N*(T-1)] (pinned: pinned_empty(n, np.int32))")
    pp = _lib.make_params(const, prop_J2, prop_drag)
    pd = _lib.make_params(const, disc_J2, False)
    c, _keep = _ctrl_struct(spec, N)
    if layout not in ("satmajor", "kmajor"):
        raise ValueError(f"unknown layout {layout!r}")
    with _lock(device):
        _lib.check(_lib.lib().mpc_propagate_discretize_host_layout(
            ctx, _lib.addr(y0), _lib.addr(tfv), ctypes.byref(pp), ctypes.byref(pd), ctypes.byref(c), N, T, int(n_sub_prop),
            int(n_sub_disc), _lib.addr(y), _lib.addr(uo), _lib.addr(out), _lib.addr(status),
            _lib.LAYOUT_K_MAJOR if layout == "kmajor" else _lib.LAYOUT_SAT_MAJOR))
    res = DiscretizedBatch(out, status.reshape(N, T - 1), N, T, layout)
    if check:
        res.raise_on_error()
    return res, y, uo


# ------------------------------------------------------------------ device-tensor API (torch CUDA tensors)

def _torch():
    import torch
    return torch


def discretize_batch_device(x, u, tf, const, include_J2=False, n_sub=100, out=None, out_pitch=None, out_offset=0,
                            status=None, extra_dst=None, adaptive=None, n_nodes=None, K=None, first=None):
    """Device form: x [N,7,K], u [N,3,K], tf [N] are float64 CUDA tensors; work is enqueued on torch's
    current stream, nothing synchronises.  `out` is [105, pitch]; `extra_dst` is an optional list of
    further [105, pitch] buffers (e.g. peer-mapped) every result is also stored to (total 1,2,4 or 8).
    K = int array [N] (host): a ragged batch as in discretize_batch (x, u [N,.,Kmax]); `first` is an int64 CUDA tensor
    [N+1] the call fills with the prefix sums of K_s - 1 (allocated when None).  The padding columns of `out` are not
    written; status (zeroed when allocated here) and n_nodes keep the [N*(Kmax-1)] layout.
    const: one Constants bag or a sequence of N, as in discretize_batch (no extra_dst with per-satellite constants).
    adaptive=dict(method="RK23", ...): scipy's RK23 controller, as in discretize_batch (one destination)."""
    rk23 = adaptive is not None and _rk23(adaptive)
    if rk23 and extra_dst:
        raise NotImplementedError("RK23 stores into one destination (no extra_dst)")
    torch = _torch()
    N, _, K_ = x.shape
    n_int = N * (K_ - 1)
    assert x.is_cuda and x.dtype == torch.float64 and x.is_contiguous()
    assert u.shape == (N, 3, K_) and u.is_contiguous() and tf.shape == (N,)
    K_sat = None
    if K is not None:
        K_sat = _counts(K, N, K_, "K")
        if extra_dst:
            raise ValueError("a ragged batch has one destination")
        if first is None:
            first = torch.empty(N + 1, dtype=torch.int64, device=x.device)
    if out is None:
        out = torch.empty((_lib.MPC_OUT_ROWS, n_int), dtype=torch.float64, device=x.device)
    pitch = out.shape[1] if out_pitch is None else int(out_pitch)
    if status is None:
        status = (torch.zeros if K_sat is not None else torch.empty)(n_int, dtype=torch.int32, device=x.device)
    psc, const = _units_of(const, N)
    if psc is not None and extra_dst:
        raise ValueError("per-satellite constants have one destination")
    p = _lib.make_params(const, include_J2, False)
    stream = torch.cuda.current_stream(x.device).cuda_stream
    L = _lib.lib()
    if rk23:
        scratch = None if psc is None else torch.empty(N * _lib.SAT_SCRATCH_DOUBLES, dtype=torch.float64, device=x.device)
        _lib.check(L.mpc_discretize_batch_rk23(
            x.data_ptr(), u.data_ptr(), tf.data_ptr(), ctypes.byref(p), psc, N, K_, _lib.addr(K_sat),
            first.data_ptr() if first is not None else None, scratch.data_ptr() if scratch is not None else None,
            float(adaptive.get("rtol", 1e-3)), float(adaptive.get("atol", 1e-6)), float(adaptive.get("max_step", 1e-2)),
            out.data_ptr(), pitch, int(out_offset), status.data_ptr(), n_nodes.data_ptr() if n_nodes is not None else None,
            stream))
        if scratch is not None:
            scratch.record_stream(torch.cuda.current_stream(x.device))
    elif psc is not None:
        ad = adaptive or {}
        scratch = torch.empty(N * _lib.SAT_SCRATCH_DOUBLES, dtype=torch.float64, device=x.device)
        _lib.check(L.mpc_discretize_batch_units(
            x.data_ptr(), u.data_ptr(), tf.data_ptr(), ctypes.byref(p), psc, N, K_, _lib.addr(K_sat),
            first.data_ptr() if first is not None else None, scratch.data_ptr(), int(adaptive is not None), int(n_sub),
            float(ad.get("rtol", 1e-3)), float(ad.get("atol", 1e-6)), float(ad.get("max_step", 1e-2)), out.data_ptr(), pitch,
            int(out_offset), status.data_ptr(), n_nodes.data_ptr() if n_nodes is not None else None, stream))
        scratch.record_stream(torch.cuda.current_stream(x.device))
    elif K_sat is not None:
        ad = adaptive or {}
        _lib.check(L.mpc_discretize_batch_ragged(
            x.data_ptr(), u.data_ptr(), tf.data_ptr(), ctypes.byref(p), N, K_, _lib.addr(K_sat), first.data_ptr(),
            int(adaptive is not None), int(n_sub), float(ad.get("rtol", 1e-3)), float(ad.get("atol", 1e-6)),
            float(ad.get("max_step", 1e-2)), out.data_ptr(), pitch, int(out_offset), status.data_ptr(),
            n_nodes.data_ptr() if n_nodes is not None else None, stream))
    elif adaptive is not None:
        _lib.check(L.mpc_discretize_batch_adaptive(
            x.data_ptr(), u.data_ptr(), tf.data_ptr(), ctypes.byref(p), N, K_, float(adaptive.get("rtol", 1e-3)),
            float(adaptive.get("atol", 1e-6)), float(adaptive.get("max_step", 1e-2)), out.data_ptr(), pitch,
            int(out_offset), status.data_ptr(), n_nodes.data_ptr() if n_nodes is not None else None, stream))
    elif extra_dst:
        ptrs = [out.data_ptr()] + [int(d if isinstance(d, int) else d.data_ptr()) for d in extra_dst]
        arr = (ctypes.c_void_p * len(ptrs))(*ptrs)
        _lib.check(L.mpc_discretize_batch_multi(x.data_ptr(), u.data_ptr(), tf.data_ptr(), ctypes.byref(p), N, K_,
                                                int(n_sub), arr, len(ptrs), pitch, int(out_offset),
                                                status.data_ptr(), stream))
    else:
        _lib.check(L.mpc_discretize_batch(x.data_ptr(), u.data_ptr(), tf.data_ptr(), ctypes.byref(p), N, K_,
                                          int(n_sub), out.data_ptr(), pitch, int(out_offset), status.data_ptr(),
                                          stream))
    return out, status


def propagate_batch_device(y0, tf, controller, const, include_drag=True, include_J2=True, T=100, n_sub=None,
                           y=None, u_out=None, status=None, T_max=None, atmosphere=None):
    """Device form of propagate_batch: y0 [N,7], tf [N] float64 CUDA tensors -> y [N,7,T], u [N,3,T], status [N].
    T = int array [N] (host): satellite s sampled at linspace(0, 1, T_s) into the first T_s columns of y / u [.,.,Tmax]
    (the padding columns are not written), the reference integrator only, as propagate_batch; so is a sequence law
    with per-satellite table lengths (ControllerSpec.table_len).  T_max: the column stride of y / u of such a batch
    (default max T_s; a fixed capacity keeps the layout of a buffer whose counts change from call to call).
    const: one Constants bag or a sequence of N, as in propagate_batch; atmosphere as in propagate_batch (the status
    words report a satellite that left the fitted range as ST_ATMO; raise_on_status(status, atmosphere) raises for it)."""
    atmo = _atmosphere(atmosphere, include_drag, n_sub)
    torch = _torch()
    N = y0.shape[0]
    _rk4_units(const, N, n_sub)
    spec = spec_from(controller)
    T_sat = tab_len = None
    if spec.kind == _lib.CTRL_SEQUENCE and spec.table_len is not None:
        tab_len = _counts(spec.table_len, N, np.shape(spec.table)[-1], "table_len")
    if np.ndim(T) != 0:
        T_sat = _counts(T, N, int(np.max(T)) if N else 2, "T")
        T = int(T_sat.max()) if N else 2
        if T_max is not None:
            if int(T_max) < T:
                raise ValueError(f"T_max = {T_max} is below the largest count {T}")
            T = int(T_max)
    T = int(T)
    if (T_sat is not None or tab_len is not None) and n_sub not in (None, 0):
        raise ValueError("per-satellite sample counts / table lengths need the reference integrator (n_sub=None)")
    if n_sub is None:
        n_sub = 0                         # the reference's RK45, replayed (see propagate_batch)
    if y is None:
        y = torch.empty((N, 7, T), dtype=torch.float64, device=y0.device)
    if u_out is None:
        u_out = torch.empty((N, 3, T), dtype=torch.float64, device=y0.device)
    if status is None:
        status = torch.empty(N, dtype=torch.int32, device=y0.device)
    tab_dev = et_dev = cnt_dev = len_dev = None
    if spec.kind == _lib.CTRL_SEQUENCE:
        tab_dev = torch.as_tensor(spec.table, dtype=torch.float64).to(y0.device).contiguous()
        if np.ndim(spec.end_tau) != 0:
            et_dev = torch.as_tensor(np.asarray(spec.end_tau, dtype=np.float64)).to(y0.device).contiguous()
    c, _keep = _ctrl_struct(spec, N, table_addr=tab_dev.data_ptr() if tab_dev is not None else None,
                            end_tau_addr=et_dev.data_ptr() if et_dev is not None else None)
    psc, const = _units_of(const, N)
    p = _lib.make_params(const, include_J2, include_drag)
    stream = torch.cuda.current_stream(y0.device).cuda_stream
    if atmo is not None:
        cnt_dev = torch.as_tensor(T_sat).to(y0.device) if T_sat is not None else None
        len_dev = torch.as_tensor(tab_len).to(y0.device) if tab_len is not None else None
        scratch = torch.empty(N * _lib.SAT_SCRATCH_DOUBLES, dtype=torch.float64, device=y0.device) if psc is not None else None
        _lib.check(_lib.lib().mpc_propagate_batch_rk45_atmo(
            y0.data_ptr(), tf.data_ptr(), ctypes.byref(p), psc, ctypes.byref(c), N, T,
            cnt_dev.data_ptr() if cnt_dev is not None else None, len_dev.data_ptr() if len_dev is not None else None,
            scratch.data_ptr() if scratch is not None else None, 1e-3, 1e-6, 1e-3, y.data_ptr(), u_out.data_ptr(),
            status.data_ptr(), None, ctypes.byref(atmo), stream))
        if scratch is not None:
            scratch.record_stream(torch.cuda.current_stream(y0.device))
    elif psc is not None:
        cnt_dev = torch.as_tensor(T_sat).to(y0.device) if T_sat is not None else None
        len_dev = torch.as_tensor(tab_len).to(y0.device) if tab_len is not None else None
        scratch = torch.empty(N * _lib.SAT_SCRATCH_DOUBLES, dtype=torch.float64, device=y0.device)
        _lib.check(_lib.lib().mpc_propagate_batch_rk45_units(
            y0.data_ptr(), tf.data_ptr(), ctypes.byref(p), psc, ctypes.byref(c), N, T,
            cnt_dev.data_ptr() if cnt_dev is not None else None, len_dev.data_ptr() if len_dev is not None else None,
            scratch.data_ptr(), 1e-3, 1e-6, 1e-3, y.data_ptr(), u_out.data_ptr(), status.data_ptr(), None, stream))
        scratch.record_stream(torch.cuda.current_stream(y0.device))
    elif T_sat is not None or tab_len is not None:
        # the ragged entry point reads the counts on the device
        cnt_dev = torch.as_tensor(T_sat if T_sat is not None else np.full(N, T, dtype=np.int32)).to(y0.device)
        len_dev = torch.as_tensor(tab_len).to(y0.device) if tab_len is not None else None
        _lib.check(_lib.lib().mpc_propagate_batch_rk45_ragged(
            y0.data_ptr(), tf.data_ptr(), ctypes.byref(p), ctypes.byref(c), N, T, cnt_dev.data_ptr(),
            len_dev.data_ptr() if len_dev is not None else None, 1e-3, 1e-6, 1e-3, y.data_ptr(), u_out.data_ptr(),
            status.data_ptr(), None, stream))
    else:
        _lib.check(_lib.lib().mpc_propagate_batch(y0.data_ptr(), tf.data_ptr(), ctypes.byref(p), ctypes.byref(c), N,
                                                  int(T), int(n_sub), y.data_ptr(), u_out.data_ptr(),
                                                  status.data_ptr(), stream))
    for t_ in (tab_dev, et_dev, cnt_dev, len_dev):
        if t_ is not None:
            t_.record_stream(torch.cuda.current_stream(y0.device))
    return y, u_out, status


def propagate_discretize_device(y0, tf, controller, const, T, prop_drag=False, prop_J2=False, disc_J2=False,
                                n_sub_prop=None, n_sub_disc=100, y=None, u_out=None, out=None, out_pitch=None,
                                out_offset=0, status_prop=None, status_disc=None, n_windows=0, extra_dst=None,
                                out_ptr=None, gather=None, atmosphere=None):
    """Device form of propagate_discretize: one SCP linearization pass (control.py:180-188) on CUDA tensors, enqueued on
    torch's current stream, with the propagation overlapped with the discretization (mpc_propagate_discretize: the
    intervals are discretized window by window along k as the propagation publishes its progress).  Bit-identical to
    propagate_batch_device followed by discretize_batch_device.  y0 [N,7], tf [N] float64 CUDA tensors; K = T.
    `extra_dst`: further [105, pitch] buffers (tensors or raw peer-mapped addresses) every result is also stored to
    (total 1, 2, 4 or 8: the fused all-gather); `out_ptr`: raw address used instead of out.data_ptr() (a multicast
    mapping of `out`); `gather`: an _lib.MpcGatherOpts -- layout (satellite- or k-major), n_sats_total, sat_offset and the
    gather options for this call (then out_pitch / out_offset are implied).
    Returns (out [105, pitch], y [N,7,T], u [N,3,T], status_prop [N], status_disc [N*(T-1)]).  An atmosphere raises
    ValueError: the overlapped, streamed and gathered passes fly the constant density only."""
    _no_atmosphere(atmosphere, "propagate_discretize_device")
    torch = _torch()
    N = y0.shape[0]
    T = int(T)
    dev = y0.device
    assert y0.is_cuda and y0.dtype == torch.float64 and y0.is_contiguous() and y0.shape == (N, 7) and tf.shape == (N,)
    n_int = N * (T - 1)
    spec = spec_from(controller)
    _rectangular_law(spec)
    if n_sub_prop is None:
        n_sub_prop = 0                    # the reference's RK45, replayed (see propagate_batch)
    if y is None:
        y = torch.empty((N, 7, T), dtype=torch.float64, device=dev)
    if u_out is None:
        u_out = torch.empty((N, 3, T), dtype=torch.float64, device=dev)
    if out is None:
        out = torch.empty((_lib.MPC_OUT_ROWS, n_int), dtype=torch.float64, device=dev)
    pitch = out.shape[1] if out_pitch is None else int(out_pitch)
    if status_prop is None:
        status_prop = torch.empty(N, dtype=torch.int32, device=dev)
    if status_disc is None:
        status_disc = torch.empty(n_int, dtype=torch.int32, device=dev)
    assert y.shape == (N, 7, T) and u_out.shape == (N, 3, T) and y.is_contiguous() and u_out.is_contiguous()
    tab_dev = et_dev = None
    if spec.kind == _lib.CTRL_SEQUENCE:
        tab_dev = torch.as_tensor(spec.table, dtype=torch.float64).to(dev).contiguous()
        if np.ndim(spec.end_tau) != 0:
            et_dev = torch.as_tensor(np.asarray(spec.end_tau, dtype=np.float64)).to(dev).contiguous()
    c, _keep = _ctrl_struct(spec, N, table_addr=tab_dev.data_ptr() if tab_dev is not None else None,
                            end_tau_addr=et_dev.data_ptr() if et_dev is not None else None)
    pp = _lib.make_params(const, prop_J2, prop_drag)
    pd = _lib.make_params(const, disc_J2, False)
    cur = torch.cuda.current_stream(dev)
    ptrs = [int(out_ptr) if out_ptr is not None else out.data_ptr()]
    ptrs += [int(d_ if isinstance(d_, int) else d_.data_ptr()) for d_ in (extra_dst or [])]
    arr = (ctypes.c_void_p * len(ptrs))(*ptrs)
    dev_i = dev.index if dev.index is not None else torch.cuda.current_device()
    with _lock(dev_i):   # the ctx owns the internal streams / progress words of the overlapped pass
        if gather is not None:      # fused all-gather with per-call options / layout (mpc_propagate_discretize_gather)
            _lib.check(_lib.lib().mpc_propagate_discretize_gather(
                _ctx(dev_i), y0.data_ptr(), tf.data_ptr(),
                ctypes.byref(pp), ctypes.byref(pd), ctypes.byref(c), N, T, int(n_sub_prop), int(n_sub_disc), y.data_ptr(),
                u_out.data_ptr(), arr, len(ptrs), ctypes.byref(gather), status_prop.data_ptr(), status_disc.data_ptr(),
                int(n_windows), cur.cuda_stream))
        else:
            _lib.check(_lib.lib().mpc_propagate_discretize_multi(
                _ctx(dev_i), y0.data_ptr(), tf.data_ptr(),
                ctypes.byref(pp), ctypes.byref(pd), ctypes.byref(c), N, T, int(n_sub_prop), int(n_sub_disc), y.data_ptr(),
                u_out.data_ptr(), arr, len(ptrs), pitch, int(out_offset), status_prop.data_ptr(), status_disc.data_ptr(),
                int(n_windows), cur.cuda_stream))
    for t_ in (tab_dev, et_dev):
        if t_ is not None:
            t_.record_stream(cur)
    return out, y, u_out, status_prop, status_disc


def fp64_peak_tflops(device=0, repeats=5):
    _lib.require_gpu()
    tf_, ms = ctypes.c_double(), ctypes.c_double()
    _lib.check(_lib.lib().mpc_fp64_peak_probe(int(device), int(repeats), ctypes.byref(tf_), ctypes.byref(ms)))
    return tf_.value, ms.value


def launch_count():
    return int(_lib.lib().mpc_launch_count())
