"""Host-side state containers mirroring the reference's data model (Python, as in the reference).

    Satellite        ref: satellite.py:4-46
    SatelliteScale   ref: satellite_scale.py:4-100
    Constants        ref: constants.py:11-20
"""
import uuid

import numpy as np

# ref: constants.py:1-8
MU_EARTH = 3.986004418e14   # m^3 / s^2
R_EARTH = 6.371e6           # m, mean radius
J2 = 1.08262668e-3
G0 = 9.80665                # m / s^2
ISP = 500                   # s
C_D = 2.5
S = 55.44                   # m^2
RHO_ATMO = 9.983e-13        # kg / m^3, the constant the reference's density model returns (simulator.py:112)


class Constants:
    """Bag of (normalized) constants handed to the dynamics (constants.py:11-20).  A plain class like the reference's:
    callers may add attributes -- Discretizer(include_drag=True) reads `const.CD` (linearize_discretize.py:165-168),
    which the reference's own Constants never sets."""

    def __init__(self, MU, R_E, J2, G0, ISP, S, R0, RHO):
        self.MU, self.R_E, self.J2, self.G0 = MU, R_E, J2, G0
        self.ISP, self.S, self.R0, self.RHO = ISP, S, R0, RHO


class Satellite:
    """Position (3), velocity (3), mass and a 128-bit id."""

    def __init__(self, position=None, velocity=None, mass=0.):
        self.position = np.zeros(3) if position is None else position
        self.velocity = np.zeros(3) if velocity is None else velocity
        self.mass = mass
        self.id = uuid.uuid4().int

    def get_state_vector(self):
        return np.concatenate([self.position, self.velocity, np.array([self.mass])])

    def update_state_vector(self, state):
        self.position, self.velocity, self.mass = state[0:3], state[3:6], state[6]

    def __str__(self):
        return (f"Satellite {hex(self.id)} with mass {self.mass}:\n"
                f"position: {self.position}\nvelocity: {self.velocity}")


class SatelliteScale:
    """Designer-unit scaling derived from one reference state."""

    def __init__(self, x=None, sat=None):
        if sat is not None:
            x = sat.get_state_vector()
        elif x is None:
            x = np.array([1, 0, 0, 0, 0, 0, 1])
        self._r0 = np.linalg.norm(x[0:3])
        self._s0 = 2 * np.pi * np.sqrt(self._r0 ** 3 / MU_EARTH)
        self._v0 = self._r0 / self._s0
        self._a0 = self._r0 / self._s0 ** 2
        self._m0 = x[6]
        self._T0 = self._m0 * self._r0 / self._s0 ** 2
        self._mu0 = self._r0 ** 3 / self._s0 ** 2

    def get_normalized_constants(self):
        return Constants(MU=MU_EARTH / self._mu0, R_E=R_EARTH / self._r0, J2=J2, G0=G0 / self._a0,
                         ISP=ISP / self._s0, S=S / self._r0 ** 2, R0=self._r0, RHO=self._m0 / self._r0 ** 3)

    def _apply(self, x, fr, fv, fm):
        x = np.asarray(x)
        if x.ndim == 1:
            return np.concatenate([x[0:3] * fr, x[3:6] * fv, [x[6] * fm]])
        assert x.shape[0] == 7, "If x is 2D, must be shaped as 7 x N"
        return np.vstack([x[0:3, :] * fr, x[3:6, :] * fv, x[6, :] * fm])

    def redim_state(self, x):
        return self._apply(x, self._r0, self._v0, self._m0)

    def normalize_state(self, x):
        x = np.asarray(x)
        if x.ndim == 1:
            return np.concatenate([x[0:3] / self._r0, x[3:6] / self._v0, np.array([x[6] / self._m0])])
        assert x.shape[0] == 7, "If x is 2D, must be shaped as 7 x N"
        return np.vstack([x[0:3, :] / self._r0, x[3:6, :] / self._v0, x[6, :] / self._m0])

    def redim_thrust(self, u):
        return u * self._T0

    def normalize_thrust(self, u):
        return u / self._T0


def sat_units(sats):
    """Each satellite normalized by its own SatelliteScale, as N OptimalControllers of the reference compute it
    (control.py:164): -> (y0 [N,7] normalized states, [N] Constants).  The constants list goes to propagate_batch,
    discretize_batch, constraint_terms_batch and BatchedSCP as `const`."""
    scales = [SatelliteScale(sat=s) for s in sats]
    y0 = np.array([sc.normalize_state(s.get_state_vector()) for sc, s in zip(scales, sats)], dtype=np.float64).reshape(-1, 7)
    return y0, [sc.get_normalized_constants() for sc in scales]
