"""Controller laws (host mirror of the reference's control.py) and their device encoding.

Every controller here yields two things:
  * get_u_func() -> u(x, tau): a host callable with the reference's signature (control.py:20,47,82,127),
    tagged with `.mpc_spec` so the GPU propagator can recognise it;
  * device_spec() -> ControllerSpec: the enum + parameters the propagate kernel evaluates on the device.

`spec_from(obj)` also recognises the REFERENCE's own controller objects and the closures their
get_u_func() returns (by class name / closure contents), so a Simulator from this package can be
driven by the reference's controllers unchanged.  The SCP/MPC loop itself (OptimalController.update,
control.py:170-235) is a caller of this path and stays in the reference.
"""
from dataclasses import dataclass, field

import numpy as np

from . import _lib


@dataclass
class ControllerSpec:
    kind: int = _lib.CTRL_ZERO
    thrust: tuple = (0.0, 0.0, 0.0)
    table: np.ndarray = field(default=None, repr=False)   # (3,Ku) or (N,3,Ku)
    end_tau: object = 1.0                                  # scalar, or [N] array (one end_tau per satellite)
    table_len: object = None                               # None, or int [N]: satellite s uses the first table_len[s]
                                                           # columns of its (N,3,Ku) table (per-satellite horizons)

    def host_u_func(self):
        """u(x, tau) on the host, same arithmetic as the device law (used by extract_uk on the host
        and handed to code that wants a callable)."""
        kind, th, tab, end_tau = self.kind, np.asarray(self.thrust, dtype=float), self.table, self.end_tau
        if kind == _lib.CTRL_ZERO:
            fn = lambda x, tau: np.zeros(3)
        elif kind == _lib.CTRL_CONSTANT:
            fn = lambda x, tau: th
        elif kind == _lib.CTRL_TANGENTIAL:
            def fn(x, tau):
                r, v = np.asarray(x[0:3], dtype=float), np.asarray(x[3:6], dtype=float)
                n = r / np.linalg.norm(r)
                h = np.cross(r, v)
                return th[0] * np.cross(h / np.linalg.norm(h), n)
        else:
            def fn(x, tau):
                if tau > end_tau:
                    return np.zeros(3)
                t = tau / end_tau       # (host law: scalar end_tau only)
                Ku = tab.shape[-1]
                if t == 1:
                    return tab[..., -1]
                k = min(max(int(np.floor(t * (Ku - 1))), 0), Ku - 2)
                lo, hi = k / (Ku - 1), (k + 1) / (Ku - 1)
                return (hi - t) / (hi - lo) * tab[..., k] + (t - lo) / (hi - lo) * tab[..., k + 1]
        fn.mpc_spec = self
        return fn


class Controller:
    """Zero thrust.  ref: control.py:8-35."""

    def __init__(self, sats=None):
        self.sats = [] if sats is None else sats
        self.sat_ids = set(s.id for s in self.sats)

    def device_spec(self):
        return ControllerSpec()

    def get_u_func(self, sat_id=None):
        return self.device_spec().host_u_func()

    def update(self):
        pass


class ConstantThrustController(Controller):
    """ref: control.py:37-53."""

    def __init__(self, sats=None, thrust=np.array([1., 1., 1.])):
        super().__init__(sats)
        self.thrust = thrust

    def device_spec(self):
        return ControllerSpec(_lib.CTRL_CONSTANT, tuple(float(t) for t in np.asarray(self.thrust).ravel()[:3]))


class ConstantTangentialThrustController(Controller):
    """Constant magnitude along t_hat = h_hat x r_hat.  ref: control.py:55-84."""

    def __init__(self, sats=None, tangential_thrust=1):
        super().__init__(sats)
        self.tangential_thrust = tangential_thrust

    def device_spec(self):
        return ControllerSpec(_lib.CTRL_TANGENTIAL, (float(self.tangential_thrust), 0.0, 0.0))


class SequenceController(Controller):
    """First-order hold of a (3,Ku) table over tau/end_tau, zero after end_tau.  ref: control.py:86-143."""

    def __init__(self, sats=None, u=np.array([]), tf_u=1, tf_sim=1):
        super().__init__(sats)
        self.end_tau = tf_u / tf_sim
        self.u = u

    def device_spec(self):
        tab = np.ascontiguousarray(self.u, dtype=np.float64)
        if tab.ndim not in (2, 3) or tab.shape[-2] != 3 or tab.shape[-1] < 2:
            raise ValueError("SequenceController needs u of shape (3, Ku) with Ku >= 2")
        return ControllerSpec(_lib.CTRL_SEQUENCE, (0.0, 0.0, 0.0), tab, float(self.end_tau))


_BY_NAME = {
    "Controller": lambda c: ControllerSpec(),
    "ConstantThrustController": lambda c: ControllerSpec(_lib.CTRL_CONSTANT, tuple(float(t) for t in np.asarray(c.thrust).ravel()[:3])),
    "ConstantTangentialThrustController": lambda c: ControllerSpec(_lib.CTRL_TANGENTIAL, (float(c.tangential_thrust), 0.0, 0.0)),
    "SequenceController": lambda c: ControllerSpec(_lib.CTRL_SEQUENCE, (0.0, 0.0, 0.0), np.ascontiguousarray(c.u, dtype=np.float64), float(c.end_tau)),
}


def _known_law(obj):
    """ControllerSpec of a controller OBJECT whose control law is one the device evaluates, else None.  Only exact
    classes qualify: a subclass may override get_u_func (a feedback law on top of ConstantThrustController, say) and
    would silently fly its parent's law, so it is refused unless its get_u_func is still the known implementation."""
    klass = type(obj)
    if isinstance(obj, Controller):                      # this package's controllers
        if klass.get_u_func is Controller.get_u_func and klass.device_spec in _OWN_SPECS:
            return obj.device_spec()
        return None
    if klass.__name__ in _BY_NAME:                       # the reference's own classes, by exact name
        return _BY_NAME[klass.__name__](obj)
    return None


def stateless(controller):
    """True when controller.update() cannot change the law between satellites (what lets run_segment propagate every
    satellite in one launch): this package's controllers with the inherited no-op update, or reference controllers
    whose update is the base class's `pass` (control.py:31-35)."""
    klass = type(controller)
    if isinstance(controller, Controller):
        return klass.update is Controller.update
    base = [k for k in klass.__mro__ if k.__name__ == "Controller"]
    return bool(base) and getattr(klass, "update", None) is getattr(base[0], "update", None)


def spec_from(obj):
    """ControllerSpec from: a ControllerSpec, one of this package's controllers, a reference controller object (exact
    class, matched by name), an OptimalController after update() (its sequence_controller), or a u_func closure produced
    by any of those.  Anything else -- subclasses with their own law included -- cannot run on the device:
    NotImplementedError (the package never falls back to calling Python per stage)."""
    if isinstance(obj, ControllerSpec):
        return obj
    if hasattr(obj, "mpc_spec"):
        return obj.mpc_spec
    if hasattr(obj, "sequence_controller"):              # reference OptimalController after update() (control.py:217,245)
        return spec_from(obj.sequence_controller)
    if type(obj).__name__ == "OptimalController":
        # before the first update() the reference's get_u_func (control.py:244-245) raises exactly this
        raise AttributeError("'OptimalController' object has no attribute 'sequence_controller'")
    if not callable(obj) or isinstance(obj, Controller):
        spec = _known_law(obj)
        if spec is not None:
            return spec
    elif callable(obj):
        qual = getattr(obj, "__qualname__", "")
        cells = [c.cell_contents for c in (getattr(obj, "__closure__", None) or ())]
        for c in cells:                            # reference lambdas close over `self`
            if type(c).__name__ != "Controller":
                spec = None if isinstance(c, (int, float, str, np.ndarray)) else _known_law(c)
                if spec is not None:
                    return spec
        if qual.startswith("Controller.get_u_func"):
            return ControllerSpec()
    raise NotImplementedError(
        f"controller / u_func {obj!r} has no device encoding: the GPU propagator evaluates the reference's "
        "controller laws (zero, constant, tangential, sequence) on the device and cannot call back into Python")


_OWN_SPECS = (Controller.device_spec, ConstantThrustController.device_spec,
              ConstantTangentialThrustController.device_spec, SequenceController.device_spec)
