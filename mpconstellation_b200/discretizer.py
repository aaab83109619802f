"""Discretizer: the reference's class (linearize_discretize.py:85-411) with the per-interval work on the GPU.

Constructor, attributes, `discretize(f, x, u, tf)` signature, return order (A_k, B_kp, B_kn, Sigma_k, xi_k)
and shapes are the reference's, so `optimizer.py:243-249` can hold one of these as `self.d` unchanged.
"""
import numpy as np

from . import batch
from .control import spec_from


RHO_CHEB = 32          # coefficients per series (include/mpc_b200.h MPC_RHO_CHEB)


def _cheb_fit(f, lo, hi, n=RHO_CHEB):
    """Coefficients c_k of sum_k c_k T_k(t), t = (r - mid) / half, interpolating f at the n Chebyshev points of [lo, hi]."""
    j = np.arange(n)
    t = np.cos(np.pi * (j + 0.5) / n)
    mid, half = 0.5 * (lo + hi), 0.5 * (hi - lo)
    fv = np.array([float(f(mid + half * tj)) for tj in t])
    c = np.array([2.0 / n * np.sum(fv * np.cos(np.pi * k * (j + 0.5) / n)) for k in range(n)])
    c[0] *= 0.5
    return c


def _scalar(v):
    """drho_func returns d rho / d|r| (the factor of r^T/|r| in linearize_discretize.py:166): one number"""
    v = np.asarray(v, dtype=np.float64)
    if v.size != 1:
        raise NotImplementedError("drho_func must return the scalar d rho / d|r| (linearize_discretize.py:166)")
    return float(v.reshape(-1)[0])


def _cheb_val(c, t):
    return np.polynomial.chebyshev.chebval(t, c)


def fit_density(rho_func, drho_func, pos, tol=1e-9):
    """What the device needs of rho_func / drho_func (linearize_discretize.py:164-165) for a batch whose normalized
    positions are pos [M,3]: the float rho when the density is constant along the batch and its gradient zero, else
    {"r_mid", "r_ihalf", "rho_c", "drho_c"}: Chebyshev series in t = (|r| - r_mid) r_ihalf over the radii of the batch
    (padded by 2 %: the integrator's stages leave the sampled radii by O(h^2)), each fitted along one direction and then
    CHECKED against the callables at the batch's own positions (all directions): agreement to tol of the largest value,
    or NotImplementedError -- the density depends on more than |r|, or is not smooth enough for 32 terms."""
    pos = np.asarray(pos, dtype=np.float64).reshape(-1, 3)
    if pos.shape[0] == 0:
        return 0.0
    if pos.shape[0] > 256:
        pos = pos[np.linspace(0, pos.shape[0] - 1, 256).astype(int)]
    rho = np.array([float(rho_func(r)) for r in pos])
    drho = np.array([_scalar(drho_func(r)) for r in pos])
    if np.ptp(rho) == 0.0 and not np.any(drho != 0.0):
        return float(rho[0])
    if not (np.all(np.isfinite(rho)) and np.all(np.isfinite(drho))):
        raise NotImplementedError("rho_func / drho_func return non-finite values on this batch")
    rad = np.linalg.norm(pos, axis=1)
    lo, hi = float(rad.min()), float(rad.max())
    pad = 0.02 * (hi - lo) + 1e-9 * hi
    lo, hi = lo - pad, hi + pad
    e = pos[0] / rad[0]
    rho_c = _cheb_fit(lambda r: rho_func(r * e), lo, hi)
    drho_c = _cheb_fit(lambda r: _scalar(drho_func(r * e)), lo, hi) if np.any(drho != 0.0) else np.zeros(0)
    mid, ihalf = 0.5 * (lo + hi), 2.0 / (hi - lo)
    t = (rad - mid) * ihalf
    err_r = np.max(np.abs(_cheb_val(rho_c, t) - rho)) / max(np.max(np.abs(rho)), 1e-300)
    err_d = 0.0 if drho_c.size == 0 else np.max(np.abs(_cheb_val(drho_c, t) - drho)) / max(np.max(np.abs(drho)), 1e-300)
    if not (err_r <= tol and err_d <= tol):
        raise NotImplementedError(
            "the GPU discretizer linearizes drag for a density that is a smooth function of |r| over the batch "
            f"(rho_func / drho_func differ from their radial Chebyshev fit by {err_r:.1e} / {err_d:.1e}); "
            "there is no CPU fallback")
    return {"r_mid": mid, "r_ihalf": ihalf, "rho_c": rho_c, "drho_c": drho_c}


class Discretizer:
    def __init__(self, const, rho_func=None, drho_func=None, include_drag=False, include_J2=False,
                 use_scipy_ZOH=False):
        self.const = const
        self.include_drag = include_drag
        self.include_J2 = include_J2
        # the reference's two input holds (u_FOH / scipy interp1d 'linear') are the same function of tau
        # (linearize_discretize.py:327-331); the kernel evaluates that first-order hold directly
        self.use_scipy_ZOH = use_scipy_ZOH
        self.rho_func = rho_func
        self.drho_func = drho_func
        # ODE solver parameters (linearize_discretize.py:104-105)
        self.ivp_max_step = 1e-2
        self.ivp_solver = 'RK45'
        # numerical integration parameters (linearize_discretize.py:108-109)
        self.integrator_steps = 101
        self.use_uniform_steps = False
        # scipy.integrate.solve_ivp defaults (the reference passes neither, linearize_discretize.py:37-41)
        self.ivp_rtol = 1e-3
        self.ivp_atol = 1e-6
        self.device = 0

    # -- option handling ---------------------------------------------------------------------------
    def _check_options(self, f):
        name = getattr(f, "__name__", None)
        if name != "satellite_dynamics":
            raise NotImplementedError(
                "the GPU discretizer integrates the reference's Simulator.satellite_dynamics on the device; "
                f"an arbitrary Python f ({f!r}) cannot be linearized there and there is no CPU fallback")
        if self.include_drag:
            # the reference cannot run this branch either: rho_func defaults to None and Constants has no
            # CD attribute (linearize_discretize.py:162-169, constants.py:11-20)
            if self.rho_func is None:
                raise TypeError("'NoneType' object is not callable")
            if not hasattr(self.const, "CD"):
                raise AttributeError("'Constants' object has no attribute 'CD'")
            if self.drho_func is None:
                raise TypeError("'NoneType' object is not callable")
        if self.ivp_solver not in ('RK45', 'RK23'):
            raise NotImplementedError(f"ivp_solver={self.ivp_solver!r}: the device replays scipy's RK45 and RK23 only; "
                                      "DOP853 and the implicit methods have no device form and there is no CPU fallback")
        if self.ivp_solver == 'RK23' and self.use_uniform_steps:
            raise NotImplementedError(
                "ivp_solver='RK23' with use_uniform_steps=True: the reference then integrates on RK23's dense output at "
                "the integrator_steps nodes, which is 1.9e-6 from the converged flow, so the fixed-step device integrator "
                "is no stand-in; only the default quadrature mode (use_uniform_steps=False) replays RK23")
        if self.ivp_solver == 'RK23' and self.include_drag:
            raise NotImplementedError("ivp_solver='RK23' with include_drag: the drag linearisation is replayed with RK45 only")
        if self.use_uniform_steps and int(self.integrator_steps) < 2:
            raise ValueError("integrator_steps must be >= 2")

    def _disc_drag(self, x):
        """(CD, rho) for the device, or None.  The drag branch (linearize_discretize.py:160-169) calls rho_func(r) and
        drho_func(r) at every state.  The kernels take the density as a function of |r|: a constant (what
        Simulator.get_atmo_density returns, simulator.py:112) or a smooth radial model such as the fits of
        simulator.py:110-111, handed over as Chebyshev series (fit_density).  Anything else -- a density that depends on the
        direction of r, or one the series cannot follow -- is rejected loudly: there is no CPU fallback."""
        if not self.include_drag:
            return None
        pos = np.moveaxis(x[:, 0:3, :], 1, 2).reshape(-1, 3)
        return float(self.const.CD), fit_density(self.rho_func, self.drho_func, pos)

    # -- the reference entry point -------------------------------------------------------------------
    def discretize(self, f, x, u, tf):
        """x (7,K), u (3,K), tf scalar -> A_k (K-1,7,7), B_kp (K-1,7,3), B_kn (K-1,7,3), Sigma_k (7,K-1),
        xi_k (7,K-1).  ref: linearize_discretize.py:334-390."""
        x = np.asarray(x, dtype=np.float64)
        u = np.asarray(u, dtype=np.float64)
        if x.ndim != 2 or x.shape[0] != 7:
            raise ValueError(f"x must be (7, K), got {x.shape}")
        res = self.discretize_batch(f, x[None], u[None] if u.ndim == 2 else u, tf)
        return res.sat(0)

    # -- batched form ------------------------------------------------------------------------------
    def discretize_batch(self, f, x, u, tf, out=None, check=True):
        """x [N,7,K], u [N,3,K], tf scalar or [N] -> batch.DiscretizedBatch (SoA + reference-shaped views).
        x, u may also be lists of the per-satellite (7,K_s) / (3,K_s) arrays Optimizer.solve_OPT holds (optimizer.py:
        243-249): they are packed into one ragged batch (padded to max K_s) and discretized in one launch."""
        self._check_options(f)
        K_sat = None
        if isinstance(x, (list, tuple)):
            x, u, K_sat = pack_ragged(x, u)
        x = np.asarray(x, dtype=np.float64)
        u = np.asarray(u, dtype=np.float64)
        K = x.shape[2]
        if K < 2:
            raise ValueError("need at least K = 2 temporal nodes")
        # u may have its own column count: the reference's hold takes its grid from u (linearize_discretize.py:308-315)
        # use_uniform_steps=False (the reference default): quadrature on the steps scipy's RK45 controller accepts
        # (replayed on the device, scipy's default rtol/atol as the reference passes none);
        # use_uniform_steps=True: fixed-step fourth-order Runge-Kutta(-Nystrom) on the uniform integrator_steps grid.
        # ivp_solver = 'RK23' (default mode only, _check_options): scipy's RK23 controller replayed the same way.
        adaptive = None if self.use_uniform_steps else dict(rtol=self.ivp_rtol, atol=self.ivp_atol,
                                                            max_step=float(self.ivp_max_step), method=self.ivp_solver)
        return batch.discretize_batch(x, u, tf, self.const, include_J2=self.include_J2,
                                      include_drag=bool(self.include_drag), disc_drag=self._disc_drag(x),
                                      n_sub=max(1, int(self.integrator_steps) - 1), out=out, device=self.device,
                                      check=check, adaptive=adaptive, K=K_sat)

    @staticmethod
    def extract_uk(x_k, tau_k, controller):
        """3 x K controller outputs at the sampled states.  ref: linearize_discretize.py:393-411.
        (Simulator.run on the GPU already returns these next to the trajectory: sim.sim_u.)"""
        u_func = spec_from(controller).host_u_func() if not callable(controller) or hasattr(controller, "device_spec") \
            else controller
        return np.column_stack([u_func(x_k[:, i], tau_k[i]) for i in range(x_k.shape[1])])


def pack_ragged(xs, us):
    """Per-satellite arrays (7,K_s) / (3,K_s) -> x [N,7,Kmax], u [N,3,Kmax] (NaN past K_s), K_sat int32 [N]."""
    if len(xs) != len(us) or not xs:
        raise ValueError("need one (7,K_s) and one (3,K_s) array per satellite")
    K_sat = np.array([np.shape(a)[1] for a in xs], dtype=np.int32)
    if any(np.shape(a) != (7, k) for a, k in zip(xs, K_sat)) or any(np.shape(b) != (3, k) for b, k in zip(us, K_sat)):
        raise ValueError("satellite s needs x (7,K_s) and u (3,K_s) on the same K_s nodes")
    Kmax = int(K_sat.max())
    x = np.full((len(xs), 7, Kmax), np.nan)
    u = np.full((len(us), 3, Kmax), np.nan)
    for s, (a, b) in enumerate(zip(xs, us)):
        x[s, :, :K_sat[s]] = a
        u[s, :, :K_sat[s]] = b
    return x, u, K_sat
