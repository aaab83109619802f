"""Batched SCP linearization pass and closed-loop driver: the callers either side of the hot path.

The reference's OptimalController.update (control.py:170-235) does, for ONE satellite and serially:
    reference trajectory (run_nonlinear, :180)  ->  extract_uk (:188)  ->  Optimizer(...).solve_OPT (:198-199, which calls
    Discretizer.discretize, optimizer.py:243-249)  ->  new SequenceController  ->  run_nonlinear again (:227)
and Simulator.run_segments (simulator.py:79-94) advances the satellites segment by segment.

`BatchedSCP` keeps that control flow but evaluates both hot-path legs for ALL satellites at once on the GPU.  The
convex subproblem itself (pyomo + ipopt, optimizer.py:251-613) is out of scope and is injected as a callable:
    solver(hand_off) -> (u_new [N,3,Kmax] padded, or a list of (3,K_s) arrays; tf_new [N])
where `hand_off.sat(s)` yields exactly the five arrays optimizer.py:327-339 indexes.  Every satellite is linearized on
its own K_s = int(base_res * tf_s) nodes, as the reference's per-satellite controllers do (control.py:221,227,
simulator.py:38); batches whose K_s differ run as one ragged launch per leg.  `const` may be one Constants bag or one per
satellite (model.sat_units: each satellite in the designer units of its own SatelliteScale, as N OptimalControllers of
the reference plan it); per-satellite constants also run one launch per leg.  With pyomo/ipopt installed one
wraps the reference's Optimizer in such a callable; `hold_reference_solver` is a deterministic stand-in (it returns the
reference input unchanged) for boxes without a solver, clearly NOT an optimizer.
"""
from dataclasses import dataclass

import numpy as np

from . import batch
from .control import ConstantTangentialThrustController, ControllerSpec, spec_from
from . import _lib


@dataclass
class Linearization:
    """Result of one batched linearization pass (the hand-off to the subproblem)."""
    x_bar: np.ndarray        # [N,7,Kmax] reference trajectories (NaN past K_s)
    u_bar: np.ndarray        # [N,3,Kmax] reference inputs (extract_uk)
    tf: np.ndarray           # [N]
    matrices: "batch.DiscretizedBatch"
    K: np.ndarray = None     # [N] nodes of every satellite, int(base_res * tf_s)
    const: object = None     # the Constants of the pass: one bag or one per satellite (constraint_terms_batch hand-off)

    def sat(self, s):
        """(A_k, B_kp, B_kn, Sigma_k, xi_k) of satellite s -- what Optimizer.solve_OPT appends at optimizer.py:243-249."""
        return self.matrices.sat(s)

    def dynamics_residual(self, s, x, u, tf, nu=None):
        """Residual of the reference's dynamics constraint (optimizer.py:327-339) for a candidate (x [7,K], u [3,K], tf),
        indexed exactly as the pyomo rule does: one value per (i, k)."""
        A_k, B_kp, B_kn, Sigma_k, xi_k = self.sat(s)
        K = int(self.K[s]) if self.K is not None else x.shape[1]
        res = np.zeros((7, K - 1))
        for k in range(K - 1):
            for i in range(7):
                rhs = (sum(A_k[k, i, j] * x[j, k] for j in range(7))
                       + sum(B_kn[k, i, j] * u[j, k] for j in range(3))
                       + sum(B_kp[k, i, j] * u[j, k + 1] for j in range(3))
                       + Sigma_k[i, k] * tf + xi_k[i, k] + (nu[i, k] if nu is not None else 0.0))
                res[i, k] = x[i, k + 1] - rhs
        return res


def hold_reference_solver(lin):
    """Stand-in for the pyomo/ipopt subproblem: keeps the reference input and final time (NOT an optimizer)."""
    return np.array(lin.u_bar), np.array(lin.tf)


def node_counts(base_res, tf):
    """K_s = int(base_res * tf_s) per satellite, the reference's own expression (simulator.py:38); K_s < 2 raises."""
    K = np.array([int(base_res * float(t)) for t in np.atleast_1d(tf)], dtype=np.int32)
    if K.size and K.min() < 2:
        raise ValueError(f"int(base_res * tf) < 2 nodes for satellite {int(np.argmin(K))} (tf = "
                         f"{float(np.atleast_1d(tf)[np.argmin(K)])}, base_res = {base_res})")
    return K


def sequence_table(u_new, K):
    """The solver's inputs as a sequence table: (table [N,3,Ku], per-satellite lengths or None when all are equal).
    u_new: [N,3,Kmax] padded (satellite s has K[s] columns) or a list of (3,K_s) arrays."""
    if isinstance(u_new, (list, tuple)):
        lens = np.array([np.shape(a)[1] for a in u_new], dtype=np.int32)
        tab = np.zeros((len(u_new), 3, int(lens.max())))
        for s, a in enumerate(u_new):
            tab[s, :, :lens[s]] = a
    else:
        tab = np.ascontiguousarray(u_new, dtype=np.float64)
        lens = np.minimum(np.asarray(K, dtype=np.int32), tab.shape[2])
    if (lens == lens[0]).all():
        return np.ascontiguousarray(tab[:, :, :lens[0]]), None
    tab = np.ascontiguousarray(np.nan_to_num(tab, nan=0.0))   # (padding is never read; keep it finite)
    return tab, lens


class BatchedSCP:
    def __init__(self, const, base_res=30, tf_horizon=2.0, tf_interval=1.0, n_iterations=2, seed_thrust=0.5,
                 include_J2=False, use_uniform_steps=False, integrator_steps=101, device=0):
        self.const = const
        self.base_res = base_res                  # OptimalController.base_res        (control.py:161)
        self.horizon = float(tf_horizon)          # OptimalController.horizon         (control.py:159)
        self.interval = float(tf_interval)        # OptimalController.interval        (control.py:160)
        self.n_iterations = n_iterations          # SCPn_iterations                   (control.py:166)
        self.seed_thrust = seed_thrust            # T_tan_mag of the seed trajectory  (control.py:178)
        self.include_J2 = include_J2
        self.use_uniform_steps = use_uniform_steps
        self.integrator_steps = integrator_steps
        self.device = device

    def linearize(self, y0, tf, controller):
        """run_nonlinear + extract_uk + discretize for every satellite (control.py:180-188 without the solve).
        The reference trajectory is propagated without drag / J2, as OptimalController.run_nonlinear does (:238-239)."""
        y0 = np.ascontiguousarray(y0, dtype=np.float64)
        N = y0.shape[0]
        tfv = np.ascontiguousarray(np.broadcast_to(np.asarray(tf, dtype=np.float64), (N,)))
        K_sat = node_counts(self.base_res, tfv)
        ragged_law = getattr(spec_from(controller), "table_len", None) is not None
        units = _lib.sat_consts(self.const, N)[0] is not None
        if (K_sat != K_sat[0]).any() or ragged_law or units:
            # one ragged launch per leg: every satellite on its own grid and / or in its own units (the fused pass is
            # rectangular and single-constant only)
            x, u, _, _ = batch.propagate_batch(y0, tfv, controller, self.const, include_drag=False, include_J2=False,
                                               T=K_sat, device=self.device)
            if self.use_uniform_steps:
                res = batch.discretize_batch(x, u, tfv, self.const, include_J2=self.include_J2, device=self.device,
                                             n_sub=self.integrator_steps - 1, K=K_sat)
            else:
                res = batch.discretize_batch(x, u, tfv, self.const, include_J2=self.include_J2, device=self.device,
                                             adaptive=dict(rtol=1e-3, atol=1e-6, max_step=1e-2), K=K_sat)
            return Linearization(np.asarray(x), np.asarray(u), tfv, res, K_sat, self.const)
        K = int(K_sat[0])
        if self.use_uniform_steps:
            # (k-major layout: the streamed host pass; the per-satellite views of the result hide it)
            res, x, u = batch.propagate_discretize(y0, tfv, controller, self.const, T=K, disc_J2=self.include_J2,
                                                   n_sub_disc=self.integrator_steps - 1, device=self.device,
                                                   layout="kmajor")
        else:
            x, u, _, _ = batch.propagate_batch(y0, tfv, controller, self.const, include_drag=False, include_J2=False,
                                               T=K, device=self.device)
            res = batch.discretize_batch(x, u, tfv, self.const, include_J2=self.include_J2, device=self.device,
                                         adaptive=dict(rtol=1e-3, atol=1e-6, max_step=1e-2))
        return Linearization(np.asarray(x), np.asarray(u), tfv, res, K_sat, self.const)

    def plan(self, y0, solver=hold_reference_solver):
        """OptimalController.update for N satellites: seed trajectory, then n_iterations of (linearize, solve,
        re-propagate with the solved inputs).  Returns the per-satellite input tables [N,3,Ku] (satellite s: the K_s
        columns of its last solve, zero-padded) and their tf_u."""
        tab, _, tf_u, history = self._plan(y0, solver)
        return tab, tf_u, history

    def _plan(self, y0, solver):
        N = y0.shape[0]
        ctrl = ConstantTangentialThrustController(tangential_thrust=self.seed_thrust)
        tf_u = np.full(N, self.horizon)
        history = []
        for _ in range(self.n_iterations):
            lin = self.linearize(y0, tf_u, ctrl)
            u_new, tf_u = solver(lin)
            tab, lens = sequence_table(u_new, lin.K)
            history.append(lin)
            # SequenceController(u=u_opt, tf_u=tf_u, tf_sim=tf_u) -> end_tau = 1 (control.py:221); satellite s's table
            # has the K_s columns of its own solve
            ctrl = ControllerSpec(_lib.CTRL_SEQUENCE, (0.0, 0.0, 0.0), tab, 1.0, lens)
        return tab, lens, tf_u, history

    def run_segments(self, y0, n_segments, solver=hold_reference_solver, include_drag=True, include_J2=True,
                     sim_base_res=100, atmosphere=None):
        """Simulator.run_segments with an OptimalController (test_simulator.py:79-95) for N satellites: before every
        segment the controller re-plans (plan), then the satellites fly `interval` with the planned inputs
        (SequenceController(u, tf_u, tf_sim=interval), control.py:217) under the full dynamics.  atmosphere: an
        Atmosphere (fit_atmosphere), the density of the flight's drag; the plans stay drag-free (control.py:238-239)."""
        y = np.ascontiguousarray(y0, dtype=np.float64)
        N = y.shape[0]
        batch._atmosphere(atmosphere, include_drag, None)     # (raises before any device work)
        if _lib.sat_consts(self.const, N)[0] is not None:
            raise NotImplementedError("run_segments with per-satellite constants: the flight runs in the Simulator's one "
                                      "scale, and carrying each controller's plan across that unit boundary is not "
                                      "implemented")
        traj, plans = [], []
        for _ in range(n_segments):
            u_tab, lens, tf_u, hist = self._plan(y, solver)
            plans.append(hist)
            end_tau = np.asarray(tf_u, dtype=np.float64) / self.interval     # one end_tau per satellite
            ctrl = ControllerSpec(_lib.CTRL_SEQUENCE, (0.0, 0.0, 0.0), u_tab, end_tau, lens)
            T = int(sim_base_res * self.interval)
            ys, _, _, _ = batch.propagate_batch(y, self.interval, ctrl, self.const, include_drag=include_drag,
                                                include_J2=include_J2, T=T, device=self.device, atmosphere=atmosphere)
            traj.append(np.array(ys))
            y = np.ascontiguousarray(ys[:, :, -1])
            if self.horizon - self.interval > 0.1:          # control.py:234-235
                self.horizon -= self.interval
        return np.concatenate(traj, axis=2), plans
