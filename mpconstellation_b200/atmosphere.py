"""An altitude-dependent atmosphere for the propagator's drag: the user's rho(h) fitted once on the host, flown on the device.

Every flight with drag otherwise uses the one density of Simulator.get_atmo_density (simulator.py:112, 500 km).  The
reference's authors wrote the power law 8E26 * h**-6.828 for 400-600 km (simulator.py:110) and dropped it because a
Python call per right-hand side slowed the solver down; on the device a Chebyshev series of log rho in log h costs a
log, an exp and a few dozen FMAs per stage evaluation.
"""
import numpy as np

from . import _lib
from .discretizer import RHO_CHEB, _cheb_fit
from .model import R_EARTH

CHECK_POINTS = 2001     # the fit is checked against rho at this many points of [h_min, h_max], both ends included
TOL = 1e-9              # largest relative error in rho the check accepts


class Atmosphere:
    """An immutable fitted density model (fit_atmosphere): log rho as sum_k coef[k] T_k(t) in
    t = (log h - (log h_min + log h_max) / 2) / ((log h_max - log h_min) / 2), h = |r| r0 - R_EARTH in metres, valid on
    [h_min, h_max].  max_rel_err is the largest relative error in rho the check found."""
    __slots__ = ("h_min", "h_max", "coef", "max_rel_err")

    def __init__(self, h_min, h_max, coef, max_rel_err):
        coef = np.array(coef, dtype=np.float64)
        coef.flags.writeable = False
        for k, v in (("h_min", float(h_min)), ("h_max", float(h_max)), ("coef", coef), ("max_rel_err", float(max_rel_err))):
            object.__setattr__(self, k, v)

    def __setattr__(self, name, value):
        raise AttributeError("Atmosphere is immutable: fit a new one")

    def __delattr__(self, name):
        raise AttributeError("Atmosphere is immutable: fit a new one")

    def __repr__(self):
        return (f"Atmosphere(h_min={self.h_min:.6g} m, h_max={self.h_max:.6g} m, {len(self.coef)} terms, "
                f"max_rel_err={self.max_rel_err:.1e})")

    def log_density(self, h):
        """log rho at altitudes h (m), from the series"""
        lo, hi = np.log(self.h_min), np.log(self.h_max)
        t = (np.log(np.asarray(h, dtype=np.float64)) - 0.5 * (lo + hi)) / (0.5 * (hi - lo))
        return np.polynomial.chebyshev.chebval(t, self.coef)

    def density(self, h):
        """rho (kg/m^3) at altitudes h (m), from the series"""
        return np.exp(self.log_density(h))

    def struct(self):
        """the mpc_atmosphere of the C-ABI"""
        a = _lib.MpcAtmosphere()
        a.h_min, a.h_max, a.r_earth, a.n = self.h_min, self.h_max, R_EARTH, len(self.coef)
        for k, c in enumerate(self.coef):
            a.coef[k] = float(c)
        return a


def _rho(rho, h):
    v = float(rho(float(h)))
    if not np.isfinite(v):
        raise ValueError(f"rho({h:.6g} m) = {v}: the density must be finite")
    if not v > 0.0:
        raise ValueError(f"rho({h:.6g} m) = {v}: the density must be positive")
    return v


def fit_atmosphere(rho, h_min, h_max):
    """Fit the density model rho(h) (h the altitude in metres, h = |r| r0 - R_EARTH; returns kg/m^3) over
    [h_min, h_max] for the propagator: log rho as a Chebyshev series of at most 32 terms (MPC_RHO_CHEB) in log h, where
    a power law is exactly linear and an exponential atmosphere stays smooth from 200 to 20,000 km.  The series is
    checked against rho at 2,001 points of the range, the ends included: a relative error in rho above 1e-9 raises
    NotImplementedError (a model with kinks, such as the larger of two exponentials, cannot be followed: there is no CPU
    fallback).  ValueError: not 0 < h_min < h_max, or rho not finite and positive there.  Returns an immutable
    Atmosphere, fitted once and reused for every flight segment."""
    h_min, h_max = float(h_min), float(h_max)
    if not (np.isfinite(h_min) and np.isfinite(h_max) and 0.0 < h_min < h_max):
        raise ValueError(f"need 0 < h_min < h_max (got {h_min!r}, {h_max!r})")
    lo, hi = np.log(h_min), np.log(h_max)
    coef = _cheb_fit(lambda s: np.log(_rho(rho, np.exp(s))), lo, hi, RHO_CHEB)
    h = np.exp(np.linspace(lo, hi, CHECK_POINTS))
    h[0], h[-1] = h_min, h_max
    want = np.array([_rho(rho, x) for x in h])
    # the shortest leading part of the series that checks no worse than all of it: the trailing terms of a power law
    # (exactly linear in log h) or of a constant are rounding noise of the fit, and each term costs an FMA per stage
    errs = [np.max(np.abs(Atmosphere(h_min, h_max, coef[:n], 0.0).density(h) / want - 1.0)) for n in range(1, len(coef) + 1)]
    errs = np.nan_to_num(np.array(errs), nan=np.inf)
    n = next(n for n in range(1, len(coef) + 1) if errs[n - 1] <= errs[-1])
    err = errs[n - 1]
    if not err <= TOL:
        raise NotImplementedError(
            f"the device propagates drag under a density that is a smooth function of the altitude over [{h_min:.6g}, "
            f"{h_max:.6g}] m (rho differs from its {RHO_CHEB}-term Chebyshev fit in log h by {err:.1e}, more than "
            f"{TOL:.0e}); there is no CPU fallback")
    return Atmosphere(h_min, h_max, coef[:n], err)
