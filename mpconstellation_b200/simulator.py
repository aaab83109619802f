"""Simulator: the reference's class (simulator.py:9-201) with the trajectory integration on the GPU.

All satellites of a run are propagated in ONE batched kernel launch instead of the reference's serial
loop over solve_ivp calls (simulator.py:41-45,58-62); signatures, return structures, segment
bookkeeping and the mass-error behaviour follow the reference.
"""
import os
from datetime import datetime
from types import SimpleNamespace

import numpy as np

from . import batch
from .control import Controller, spec_from, stateless
from .model import C_D, RHO_ATMO, R_EARTH, SatelliteScale


class Simulator:
    def __init__(self, sats=None, controller=None, scale=None, base_res=100, include_drag=True,
                 include_J2=True, verbose=False):
        self.sim_data = {}
        self.sim_time = {}
        self.sim_u = {}            # controller output at every sample (what extract_uk would recompute)
        self.sats = [] if sats is None else sats
        self.base_res = base_res
        self.eval_points = self.base_res
        self.controller = Controller() if controller is None else controller
        self.include_drag = include_drag
        self.include_J2 = include_J2
        self.scale = SatelliteScale() if scale is None else scale
        self.verbose = verbose
        self.max_time_step = 0.001   # simulator.py:186: solve_ivp's max_step
        # "rk45": the reference's integrator (scipy RK45 + step-size controller + dense-output samples, simulator.py:185-187)
        # replayed step for step on the device; "rk4": fixed-step RK4, ceil(1/(max_time_step (T-1))) steps per sample
        self.integrator = "rk45"
        self.last_n_steps = None
        self.device = 0
        # an Atmosphere (fit_atmosphere): the density of the drag as a function of the altitude instead of the constant of
        # get_atmo_density; used when include_drag is set (the reference integrator only)
        self.atmosphere = None

    # -- batched core --------------------------------------------------------------------------------
    def _propagate(self, sats, tf, controller):
        const = self.scale.get_normalized_constants()
        y0 = np.stack([self.scale.normalize_state(s.get_state_vector()) for s in sats]) if sats else np.zeros((0, 7))
        T = int(self.eval_points)
        if self.integrator == "rk45":
            mode = dict(n_sub=None, rk45=dict(max_step=self.max_time_step))
        elif self.integrator == "rk4":
            mode = dict(n_sub=batch.default_n_sub(T, self.max_time_step))
        else:
            raise ValueError(f"unknown integrator {self.integrator!r} (rk45 | rk4)")
        if self.integrator == "rk45":
            mode["n_steps"] = np.zeros(len(sats), dtype=np.int32)
        atmosphere = self.atmosphere if self.include_drag else None
        y, u, t, _ = batch.propagate_batch(y0, tf, controller, const, include_drag=self.include_drag,
                                           include_J2=self.include_J2, T=T, device=self.device, atmosphere=atmosphere,
                                           **mode)
        # steps attempted per satellite by the replayed integrator (scipy's sol.nfev = 2 + 6 steps)
        self.last_n_steps = mode.get("n_steps")
        return y, u, t

    def run(self, tf=10):
        """ref: simulator.py:29-48.  Returns ({sat.id: (7,T)}, {sat.id: (T,)})."""
        self.eval_points = int(self.base_res * tf)
        y, u, t = self._propagate(self.sats, tf, self.controller)
        self.sim_data = {s.id: y[i] for i, s in enumerate(self.sats)}
        self.sim_time = {s.id: t.copy() for s in self.sats}
        self.sim_u = {s.id: u[i] for i, s in enumerate(self.sats)}
        return self.sim_data, self.sim_time

    def run_segment(self, tf=1):
        """ref: simulator.py:50-77.  The reference goes satellite by satellite: controller.update(), propagate, write the
        final state back to the satellite.  With a controller whose update() is the base class's no-op that order cannot
        matter and all satellites are propagated in ONE launch; a controller that re-plans in update() (the reference's
        OptimalController reads the satellite state and shortens its horizon there, control.py:170-235) is served in the
        reference's order, one satellite per launch, so that every satellite flies the plan made for it."""
        self.eval_points = int(self.base_res * tf)
        if stateless(self.controller):
            for _ in self.sats:
                self.controller.update()
            y, u, t = self._propagate(self.sats, tf, self.controller)
            for i, sat in enumerate(self.sats):
                self._append_segment(sat, y[i], u[i], t, tf)
            return
        for sat in self.sats:
            self.controller.update()
            y, u, t = self._propagate([sat], tf, spec_from(self.controller))
            self._append_segment(sat, y[0], u[0], t, tf)

    def _append_segment(self, sat, y, u, t, tf):
        sat.update_state_vector(self.scale.redim_state(y[:, -1]))
        if sat.id in self.sim_data and sat.id in self.sim_time:
            time = t + self.sim_time.get(sat.id, [0])[-1] * tf + 0.0000001      # simulator.py:70
            self.sim_data[sat.id] = np.concatenate([self.sim_data[sat.id], y], axis=1)
            self.sim_time[sat.id] = np.concatenate([self.sim_time[sat.id], time])
            self.sim_u[sat.id] = np.concatenate([self.sim_u[sat.id], u], axis=1)
        else:
            self.sim_data[sat.id] = np.array(y)
            self.sim_time[sat.id] = t.copy()
            self.sim_u[sat.id] = np.array(u)

    def run_segments(self, tf=1, num_segments=1):
        """ref: simulator.py:79-94."""
        tf_step = tf / float(num_segments)
        for n in range(num_segments):
            if self.verbose:
                print(f"\nRunning segment {n+1} of {num_segments}; tf {tf_step*(n+1)} of {tf}")
            self.run_segment(tf=tf_step)

    def get_trajectory_ODE(self, sat, tf, u_func):
        """ref: simulator.py:164-189.  Returns an object with .y (7,T) and .t (T,) like solve_ivp's."""
        y, u, t = self._propagate([sat], tf, spec_from(u_func))
        nfev = None if self.last_n_steps is None else 2 + 6 * int(self.last_n_steps[0])     # as solve_ivp counts them
        return SimpleNamespace(y=y[0], t=t, u=u[0], success=True, status=0, nfev=nfev,
                               message=f"{self.integrator} on sm_100a")

    def save_to_csv(self, suffix="", redimensionalize=True, directory="."):
        """ref: simulator.py:192-201 -- one `trajectory_<date>_<sat.id><suffix>.csv` per satellite, rows = samples,
        7 comma-separated columns (np.savetxt default '%.18e'), read by the reference's visualizer.m.
        `directory` is an addition (the reference writes into the working directory); returns the paths."""
        date = datetime.today().strftime('%Y-%m-%d-%H-%M-%S')
        paths = []
        for sat in self.sats:
            data = self.sim_data[sat.id]
            if redimensionalize:
                data = self.scale.redim_state(data)
            path = os.path.join(directory, f"trajectory_{date}_{sat.id}{suffix}.csv")
            np.savetxt(path, np.asarray(data).T, delimiter=",")
            paths.append(path)
        return paths

    # -- reference statics kept as host callables ------------------------------------------------------
    @staticmethod
    def get_atmo_density(r, r0):
        """ref: simulator.py:96-112 (constant 500 km density)."""
        return RHO_ATMO

    @staticmethod
    def satellite_dynamics(tau, y, u_func, tf, const, include_drag=True, include_J2=True):
        """Host evaluation of the dynamics, reference signature (simulator.py:115-161).  This is the callable
        users pass as `f` to Discretizer.discretize; the GPU kernels implement the same equations."""
        y = np.asarray(y, dtype=float)
        r, v, m = y[0:3], y[3:6], y[6]
        if m <= 0.1:
            print(f"WARNING: low mass {m}")
        if m <= 0:
            raise Exception(f"ERROR: INVALID SATELLITE MASS: {m}")
        rn = np.linalg.norm(r)
        u = np.asarray(u_func(y, tau), dtype=float)
        acc = -const.MU / rn ** 3 * r + u / m
        if include_drag:
            acc = acc - 0.5 * C_D * const.S / m * (Simulator.get_atmo_density(r, const.R0) / const.RHO) * np.linalg.norm(v) * v
        if include_J2:
            q = 5 * (r[2] / rn) ** 2
            acc = acc + 1.5 * const.J2 * const.MU * const.R_E ** 2 / rn ** 5 * np.array([q - 1, q - 1, q - 3]) * r
        return tf * np.concatenate([v, acc, [-np.linalg.norm(u) / (const.G0 * const.ISP)]])
