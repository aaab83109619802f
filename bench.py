#!/usr/bin/env python
"""bench.py -- discretized intervals/sec of the batched SCvx linearize-and-discretize hot path.

Workload (BASELINE.json configs[2], the largest single-GPU configuration): 4096 satellites x K=200
nodes (815,104 intervals), tangential thrust 0.5, tf=2.  One STEP = one SCP linearization pass over the
batch: propagate every satellite (reference trajectory + extract_uk) and discretize every interval
(integrator_steps=101: 100 fixed fourth-order Runge-Kutta(-Nystrom) steps + 101-node trapezoid per interval).
The propagation runs beside the discretization (windows of k gated on its progress, mpc_propagate_discretize;
bit-identical to the two kernels back to back, which --no-overlap times instead).

    python bench.py [--gpus N] [--steps K] [--warmup W]            # this repo's CUDA path
    python bench.py --impl reference [...]                          # the reference algorithm on the host cores
    python bench.py --dump-outputs DIR [...]                        # also save a sample of the last timed step's results

`--dump-outputs` writes what the last timed step returned to its caller as DIR/<name>.npy (float64, a fixed seeded sample
of the satellites, under 64 MB in all), so that two builds run with the same arguments can be compared output for output.

Under torchrun (N>1) every rank processes its own 4096-satellite shard (weak scaling) and the discretized
matrices are all-gathered over NVLink inside the timed step, as north_star asks (fused into the kernel: peer stores;
--gather nccl for the NCCL baseline).  `--total-sats 5025` is BASELINE configs[3]: ONE 1 M-interval sweep sharded over
the ranks (strong scaling).  At N=1 the line also carries `configs`: BASELINE configs 1, 2 and 5 timed on the GPU, the
plain-C port and (config 5) the reference path on the same shapes.

Prints ONE JSON line (rank 0).  Timing: CUDA events on the launching stream, >= 3 warm-up steps, L2 flushed
between timed steps (256 MiB write), max over ranks, clocks sampled during the timed region.
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

HUBBLE = np.array([5371.4806e3, -4133.1393e3, 1399.9594e3, 4.6921e3, 4.9848e3, -3.2752e3, 12200.0])
FP64_NOMINAL_TFLOPS = 148 * 64 * 2 * 1.965e9 / 1e12      # 148 SM x 64 DFMA/clk x 2 flop x 1.965 GHz = 37.2


def flops_per_interval(n_sub, include_j2=False, em=True):
    """ALGORITHMIC FP64 work of one interval: the arithmetic of the algorithm DESIGN.md section 4 states (42 live Phi
    entries, symmetric G, Nystrom's 3-stage fourth-order Runge-Kutta method in step-normalised variables with steps that
    span two quadrature nodes and a cubic-Hermite midpoint, symplectic inverse, 56 accumulators), FMA = 2 flop,
    mul/add = 1, MUFU seeds not counted.  One thread does one interval with no recomputation, so this equals the
    executed DFMA/DMUL/DADD count: per integrator step (= two quadrature nodes) 754 FMA + 242 mul + 99 add (J2: 798 /
    298 / 116), plus the last node and the Phi_end * [integrals] epilogue (1249 flop; J2 1310).  An odd n_sub runs one
    step per node (532 / 182 / 55; J2 571 / 230 / 69).  Counted from the SASS of the shipped kernel
    (scripts/sass_reuse.py) and cross-checked against ncu smsp__sass_thread_inst_executed_op_{dfma,dmul,dadd}_pred_on.
    em (what the library launches for n_sub = 100 unless mpc_set_tuning(37)): see below; em=False prices the same
    throughput at the work of evaluating all 101 nodes (`all_nodes_alg` in the bench line)."""
    tail = 1310 if include_j2 else 1249
    if em and n_sub == 100:
        # the reference's integrator_steps = 101 as shipped: the 101-node trapezoid sums through their Euler-Maclaurin
        # expansion (kEmW, csrc/discretize_kernel.cuh) -- 20 one-node steps whose ends are the 21 nodes of the rule
        return EM_STEPS * ((2 * 571 + 230 + 69) if include_j2 else (2 * 532 + 182 + 55)) + tail
    if n_sub % 2 == 0:
        return (n_sub // 2) * ((2 * 798 + 298 + 116) if include_j2 else (2 * 754 + 242 + 99)) + tail
    return n_sub * ((2 * 571 + 230 + 69) if include_j2 else (2 * 532 + 182 + 55)) + tail


EM_STEPS = 20


def fp64_instr_per_interval(n_sub, include_j2=False, em=True):
    """FP64-pipe instructions (DFMA+DMUL+DADD) per interval: the pipe-occupancy view of the same work."""
    tail = 785 if include_j2 else 742
    if em and n_sub == 100:
        return EM_STEPS * ((571 + 230 + 69) if include_j2 else (532 + 182 + 55)) + tail
    if n_sub % 2 == 0:
        return (n_sub // 2) * ((798 + 298 + 116) if include_j2 else (754 + 242 + 99)) + tail
    return n_sub * ((571 + 230 + 69) if include_j2 else (532 + 182 + 55)) + tail


def kernel_counters():
    """Per-launch hardware counters of the shipped kernels, measured with ncu on this workload and committed under
    profiles/ (each entry names the summary it was read from): dram traffic, executed flop of the default-mode kernel.
    bench.py never hard-codes them; a kernel change means a new capture and a new entry."""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "kernel_counters.json")))
    except Exception:
        return {}


def bytes_per_interval():
    return 13 * 8 + 105 * 8       # read x_k, u_k, u_k+1; write 105 doubles (SURVEY 8d)


# ------------------------------------------------------------------------------------------ inputs

def make_constellation(n_sats, seed=20240531):
    """SURVEY 8(d): Hubble state rotated about z by 2*pi*i/N, speed scaled by 1+0.1*U[0,1), one scale from sat 0."""
    import mpconstellation_b200 as M
    scale = M.SatelliteScale(x=HUBBLE)
    const = scale.get_normalized_constants()
    y = scale.normalize_state(HUBBLE)
    rng = np.random.default_rng(seed)
    ang = 2 * np.pi * np.arange(n_sats) / max(n_sats, 1)
    ca, sa = np.cos(ang), np.sin(ang)
    f = 1 + 0.1 * rng.random(n_sats)
    Y = np.tile(y, (n_sats, 1))
    Y[:, 0], Y[:, 1] = ca * y[0] - sa * y[1], sa * y[0] + ca * y[1]
    Y[:, 3], Y[:, 4] = (ca * y[3] - sa * y[4]) * f, (sa * y[3] + ca * y[4]) * f
    Y[:, 5] = y[5] * f
    return Y, const


DUMP_BYTES = 48 << 20


def dump_outputs(path, out, x, u, status_prop, status_disc):
    """--dump-outputs: the arrays the step hands its caller (the [105, N*(K-1)] matrices, the propagated states [N,7,K] and
    inputs [N,3,K], both status arrays), restricted to a seeded sample of satellites that depends on N and K only, with
    every interval of a sampled satellite kept; at most DUMP_BYTES of float64 (status codes as numbers)."""
    import torch
    N, _, K = x.shape
    per_sat = 8 * (105 * (K - 1) + 10 * K + 1 + (K - 1))
    n = min(N, max(1, DUMP_BYTES // per_sat))
    sats = np.sort(np.random.default_rng(0).choice(N, size=n, replace=False))
    cols = (sats[:, None] * (K - 1) + np.arange(K - 1)).ravel()
    si, ci = torch.from_numpy(sats).to(x.device), torch.from_numpy(cols).to(x.device)
    os.makedirs(path, exist_ok=True)
    for name, a in (("out", out[:, ci]), ("x", x[si]), ("u", u[si]), ("status_prop", status_prop[si]),
                    ("status_disc", status_disc[ci])):
        np.save(os.path.join(path, name + ".npy"), a.cpu().numpy().astype(np.float64))


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons through NVML while the timed region runs."""

    def __init__(self, index=0, period=0.004):
        super().__init__(daemon=True)
        self.period, self.samples, self.reasons, self.max_mhz = period, [], set(), None
        self._halt = threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
                 nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap",
                 nv.nvmlClocksThrottleReasonHwPowerBrakeSlowdown: "hw_power_brake"}
        while not self._halt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, nm in names.items():
                    if r & bit:
                        self.reasons.add(nm)
            except Exception:
                pass
            time.sleep(self.period)

    def stop(self):
        self._halt.set()
        self.join(timeout=2)
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


# ------------------------------------------------------------------------------------------ CPU arms

def cpu_port_baseline(n_sats, K, tf, n_sub, budget_s=12.0):
    """oracle/mpc_oracle.c (plain-C port of the same RK4/trapezoid algorithm, OpenMP over intervals) on a
    bounded sample of the workload: the first S satellites."""
    from oracle import c_oracle as C
    from oracle.mpc_oracle import OracleConstants
    Y, const_m = make_constellation(n_sats)
    const = OracleConstants(const_m.MU, const_m.R_E, const_m.J2, const_m.G0, const_m.ISP, const_m.S, const_m.R0, const_m.RHO)
    cores = C.max_threads()
    n_prop = max(1, int(np.ceil(1000 / (K - 1))))

    def run(S):
        t0 = time.perf_counter()
        x, u, st = C.propagate_batch(Y[:S], tf, const, C.CTRL_TANGENTIAL, (0.5, 0, 0), include_drag=False,
                                     include_J2=False, T=K, n_sub=n_prop)
        out = C.discretize_batch(x, u, tf, const, n_sub=n_sub)
        assert out[5].max() == 0
        return time.perf_counter() - t0
    S = min(n_sats, 2 * cores)
    t = run(S)                                   # calibration (also warms the OpenMP pool)
    S = int(min(n_sats, max(S, S * budget_s / max(t, 1e-3))))
    t = run(S)
    return {"value": S * (K - 1) / t, "unit": "intervals/s", "cores": cores, "kind": "port",
            "sample": f"first {S} of {n_sats} satellites x {K-1} intervals (propagate + discretize, n_sub={n_sub}), "
                      f"{t:.1f} s of oracle/mpc_oracle.c with OpenMP"}


def reference_arm(args):
    """--impl reference: the UNMODIFIED reference on the box's host cores.  Its hot-path modules are compiled to Python
    bytecode under oracle/_ref/ by build() where /root/reference is mounted (oracle/refshim.py; no source is copied),
    and run here through the reference's own public API, per satellite as its callers do (simulator.py:41-45,
    control.py:180-188, optimizer.py:243-249): Simulator.run (scipy RK45, max_step 0.001) -> Discretizer.extract_uk ->
    Discretizer.discretize (one mp.Pool over the intervals per call).  A bounded sample of the workload per step.
    Falls back to the numpy restatement (oracle/mpc_oracle.py, kind "port") only when the bytecode is absent."""
    import warnings
    warnings.filterwarnings("ignore")
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import refshim
    n_sats, K, tf = args.sats, args.nodes, args.tf
    cores = os.cpu_count() or 1
    S = args.ref_sats
    Yn, _ = make_constellation(n_sats)
    root, kind = refshim.reference_location()
    if root is not None:
        import contextlib
        import io
        R = refshim.load_reference()
        hub = R.Satellite(HUBBLE[0:3].copy(), HUBBLE[3:6].copy(), float(HUBBLE[6]))
        scale = R.SatelliteScale(sat=hub)
        const = scale.get_normalized_constants()
        ctrl = R.ConstantTangentialThrustController(tangential_thrust=0.5)
        F = R.Simulator.satellite_dynamics

        def one_pass(s, uniform):
            yd = scale.redim_state(Yn[s])
            sat = R.Satellite(yd[0:3], yd[3:6], float(yd[6]))
            sim = R.Simulator(sats=[sat], controller=ctrl, scale=scale, base_res=int(round(K / tf)), include_drag=False,
                              include_J2=False)
            sim.run(tf=tf)
            x, t = sim.sim_data[sat.id], sim.sim_time[sat.id]
            d = R.Discretizer(const)
            d.use_uniform_steps = uniform
            d.integrator_steps = args.n_sub + 1
            with contextlib.redirect_stdout(io.StringIO()):
                return d.discretize(F, x, R.Discretizer.extract_uk(x, t, ctrl), tf)
        impl_kind = "reference"
        what = f"the unmodified reference ({kind} under {os.path.relpath(root, ROOT) if root.startswith(ROOT) else root})"
    else:
        from oracle import mpc_oracle as O
        const = O.normalized_constants(O.scale_factors(HUBBLE))
        ctrl = O.ctrl_tangential(0.5)

        def one_pass(s, uniform):
            x, t = O.propagate(Yn[s], tf, ctrl, const, False, False, K)
            return O.discretize(x, O.extract_uk(x, t, ctrl), tf, const, use_uniform_steps=uniform,
                                integrator_steps=args.n_sub + 1, processes=cores)
        impl_kind = "port"
        what = "oracle/mpc_oracle.py (numpy/scipy restatement; oracle/_ref bytecode not built)"

    def step():
        for s in range(S):
            one_pass(s, True)
    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = (time.perf_counter() - t0) / args.steps
    val = S * (K - 1) / dt
    # the reference's shipped default (use_uniform_steps=False: quadrature on the 4-8 accepted RK45 steps), once, for the record
    t1 = time.perf_counter()
    for s in range(min(S, 4)):
        one_pass(s, False)
    default_mode = min(S, 4) * (K - 1) / (time.perf_counter() - t1)
    sample = (f"{S} of {n_sats} satellites x {K-1} intervals per step; per satellite Simulator.run + extract_uk + "
              f"Discretizer.discretize (use_uniform_steps=True, integrator_steps={args.n_sub + 1}), mp.Pool({cores}) per "
              f"discretize call as the reference does; {what}")
    cfg = workload_config(args)
    cfg["integrator"] = ("scipy solve_ivp RK45 (rtol 1e-3, atol 1e-6): propagation with max_step 0.001 and dense-output samples; "
                         f"discretization per interval, Phi and x read off the dense output at {args.n_sub + 1} uniform nodes "
                         "(use_uniform_steps=True), np.linalg.inv per node, trapezoid rule")
    cfg["parallelism"] = f"mp.Pool({cores}) over the intervals of one satellite; satellites serial"
    print(json.dumps({
        "impl": "reference", "metric": "discretized intervals/sec", "value": val, "unit": "intervals/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": cfg,
        "cpu_baseline": {"value": val, "unit": "intervals/s", "cores": cores, "kind": impl_kind, "sample": sample},
        "e2e": {"value": val, "unit": "intervals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "default_mode_intervals_per_s": default_mode,
        "gpu_launches": 0,
    }))


def workload_config(args):
    if getattr(args, "total_sats", 0):
        wl = (f"{args.total_sats} satellites x K={args.nodes} nodes ({args.total_sats * (args.nodes - 1)} intervals) IN TOTAL, sharded "
              f"over {args.gpus} GPU(s): propagate (tangential thrust 0.5, no drag/J2) + discretize, BASELINE configs[3]")
    else:
        wl = (f"{args.sats} satellites x K={args.nodes} nodes ({args.sats * (args.nodes - 1)} intervals) per GPU: "
              "propagate (tangential thrust 0.5, no drag/J2) + discretize, BASELINE configs[2]")
    return {"workload": wl,
            "sats_per_gpu": args.sats, "K": args.nodes, "tf": args.tf, "integrator_steps": args.n_sub + 1,
            "integrator": "fixed-step fourth-order Runge-Kutta-Nystrom (3 stages); the trapezoid sums over the reference's 101 nodes evaluated through their Euler-Maclaurin expansion (21 of the nodes = the ends of 20 integrator steps; agrees with the literal 101-node sums to 1e-13, per-interval fallback to all 101 nodes where the held input is not smooth)", "l2": "flushed between timed steps (256 MiB write)",
            "parallelism": f"satellites sharded over {args.gpus} GPU(s)" + (f", all-gather of the SoA matrices inside the step ({args.gather})" if args.gpus > 1 else "")}


# ------------------------------------------------------------------------------------------ BASELINE configs 1, 2, 5

def small_configs_record(M, dev, const, with_cpu=True):
    """BASELINE configs[0], [1], [4] on the same GPU (rank 0, N=1): kernel times on device buffers (CUDA events, mean of 5
    after 2 warm-ups, the reference's integrator replayed for the propagation), and for config 5 the per-SCP-pass and
    per-MPC-step wall time through the host API (BatchedSCP: control.py:170-235 for all satellites at once), next to the
    plain-C port on the same shapes and -- config 5 -- the reference path itself on a 2-satellite sample."""
    import torch
    from mpconstellation_b200.scp import BatchedSCP
    ctrl = M.ConstantTangentialThrustController(tangential_thrust=0.5)
    ad = dict(rtol=1e-3, atol=1e-6, max_step=1e-2)

    def ev_ms(fn, n=5):
        ts = []
        for i in range(n + 2):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize(dev)
            a.record()
            fn()
            b.record()
            torch.cuda.synchronize(dev)
            if i >= 2:
                ts.append(a.elapsed_time(b))
        return float(np.mean(ts))

    def wall_ms(fn, n=3):
        fn()
        t0 = time.perf_counter()
        for _ in range(n):
            fn()
        return (time.perf_counter() - t0) / n * 1e3

    rec = {}
    shapes = (("config1", 1, 50, 0.5, "single satellite, K=50 (test_discretizer.py default scenario)"),
              ("config2", 64, 100, 1.0, "64 satellites x K=100, one SCP linearization pass"),
              ("config5", 256, 60, 2.0, "256-satellite closed loop: base_res 30, horizon 2 -> K=60, 2 SCP passes per segment"))
    for name, Ns, Ks, tfs, what in shapes:
        Ys, _ = make_constellation(Ns)
        y0 = torch.from_numpy(Ys).to(dev)
        tfd = torch.full((Ns,), tfs, dtype=torch.float64, device=dev)
        x, u, _ = M.propagate_batch_device(y0, tfd, ctrl, const, include_drag=False, include_J2=False, T=Ks)
        r = {"what": what, "satellites": Ns, "K": Ks, "intervals": Ns * (Ks - 1),
             "propagate_ms": ev_ms(lambda: M.propagate_batch_device(y0, tfd, ctrl, const, include_drag=False, include_J2=False, T=Ks)),
             "discretize_uniform_ms": ev_ms(lambda: M.discretize_batch_device(x, u, tfd, const, n_sub=100)),
             "discretize_default_ms": ev_ms(lambda: M.discretize_batch_device(x, u, tfd, const, adaptive=ad)),
             "pass_uniform_ms": ev_ms(lambda: M.propagate_discretize_device(y0, tfd, ctrl, const, Ks, n_sub_disc=100))}
        if with_cpu:
            from oracle import c_oracle as C
            from oracle.mpc_oracle import OracleConstants
            oc = OracleConstants(const.MU, const.R_E, const.J2, const.G0, const.ISP, const.S, const.R0, const.RHO)
            t0 = time.perf_counter()
            xr, ur, _, _, _ = C.propagate_batch_rk45(Ys, tfs, oc, C.CTRL_TANGENTIAL, (0.5, 0, 0), include_drag=False,
                                                     include_J2=False, T=Ks)
            t1 = time.perf_counter()
            C.discretize_batch(xr, ur, tfs, oc)
            t2 = time.perf_counter()
            C.discretize_batch_adaptive(xr, ur, tfs, oc)
            t3 = time.perf_counter()
            r["cpu_port_ms"] = {"propagate": (t1 - t0) * 1e3, "discretize_uniform": (t2 - t1) * 1e3,
                                "discretize_default": (t3 - t2) * 1e3, "cores": C.max_threads()}
        rec[name] = r
    # config 5 through the host API, as the closed loop runs it: linearize = propagate + extract_uk + discretize (default
    # quadrature mode, control.py:187) for all 256 satellites; one MPC step = plan (2 passes) + flight (drag + J2)
    Ys, _ = make_constellation(256)
    scp = BatchedSCP(const, base_res=30, tf_horizon=2.0, tf_interval=1.0, n_iterations=2)
    c5 = rec["config5"]
    c5["scp_pass_host_ms"] = wall_ms(lambda: scp.linearize(Ys, 2.0, ctrl))
    scp_u = BatchedSCP(const, base_res=30, tf_horizon=2.0, tf_interval=1.0, n_iterations=2, use_uniform_steps=True)
    c5["scp_pass_host_uniform_ms"] = wall_ms(lambda: scp_u.linearize(Ys, 2.0, ctrl))

    def mpc_step():
        s_ = BatchedSCP(const, base_res=30, tf_horizon=2.0, tf_interval=1.0, n_iterations=2)
        s_.run_segments(Ys, n_segments=1)
    c5["mpc_step_host_ms"] = wall_ms(mpc_step)
    c5["mpc_step_note"] = ("one segment of BatchedSCP.run_segments: 2 x (propagate + extract_uk + default-mode discretize) + the "
                           "flight of the interval with drag + J2, host arrays in and out; the pyomo/ipopt subproblem is not "
                           "part of this path and is stood in for by hold_reference_solver (no solve time on either side)")
    if with_cpu:
        # the reference path on the same shape (control.py:180-188,227 per satellite, serial over satellites), 2-satellite sample
        try:
            import contextlib
            import io
            import warnings
            warnings.filterwarnings("ignore")
            from oracle import refshim
            R = refshim.load_reference()
            hub = R.Satellite(HUBBLE[0:3].copy(), HUBBLE[3:6].copy(), float(HUBBLE[6]))
            scale = R.SatelliteScale(sat=hub)
            rconst = scale.get_normalized_constants()
            rc = R.ConstantTangentialThrustController(tangential_thrust=0.5)
            t0 = time.perf_counter()
            for s in range(2):
                yd = scale.redim_state(Ys[s])
                for _ in range(2):                                   # SCPn_iterations (control.py:166)
                    sat = R.Satellite(yd[0:3], yd[3:6], float(yd[6]))
                    sim = R.Simulator(sats=[sat], controller=rc, scale=scale, base_res=30, include_drag=False, include_J2=False)
                    sim.run(tf=2.0)
                    xx, tt = sim.sim_data[sat.id], sim.sim_time[sat.id]
                    with contextlib.redirect_stdout(io.StringIO()):
                        R.Discretizer(rconst).discretize(R.Simulator.satellite_dynamics, xx, R.Discretizer.extract_uk(xx, tt, rc), 2.0)
                sat = R.Satellite(yd[0:3], yd[3:6], float(yd[6]))
                R.Simulator(sats=[sat], controller=rc, scale=scale, base_res=100).run(tf=1.0)   # the flight, drag + J2
            per_sat = (time.perf_counter() - t0) / 2
            c5["reference_path"] = {"ms_per_satellite_per_mpc_step": per_sat * 1e3, "ms_per_mpc_step_256_satellites": per_sat * 256e3,
                                    "sample": "2 satellites, unmodified reference (oracle/_ref bytecode), serial over satellites as "
                                              "Simulator.run_segment / OptimalController.update are, mp.Pool per discretize call; "
                                              "subproblem solve excluded on both sides", "cores": os.cpu_count()}
            c5["mpc_step_vs_reference_path"] = per_sat * 256e3 / c5["mpc_step_host_ms"]
        except Exception as exc:        # bytecode not built on this box
            c5["reference_path"] = {"unavailable": str(exc)}
    return rec


# ------------------------------------------------------------------------------------------ GPU arm

def gpu_arm(args):
    import torch
    import mpconstellation_b200 as M
    from mpconstellation_b200 import _lib
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    _lib.require_gpu()
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    try:
        local_phys = int(vis.split(",")[local]) if vis else local      # NVML index of this rank's GPU
    except (ValueError, IndexError):
        local_phys = local
    dist = None
    if world > 1:
        import torch.distributed as dist
        # stdout carries exactly one JSON line: keep NCCL's version banner off it (NCCL_DEBUG=INFO etc. is respected)
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"
        dist.init_process_group("nccl", device_id=dev)
    from mpconstellation_b200 import distributed as D
    K, tf, n_sub = args.nodes, args.tf, args.n_sub
    # weak scaling: args.sats satellites per rank; strong scaling (--total-sats): one batch sharded over the ranks
    N_total = args.total_sats if args.total_sats else args.sats * world
    s0, s1 = D.shard_range(N_total, rank, world)
    N = s1 - s0
    n_int = N * (K - 1)
    n_int_total = N_total * (K - 1)
    Y, const = make_constellation(N_total)
    Y = np.ascontiguousarray(Y[s0:s1])
    ctrl = M.ConstantTangentialThrustController(tangential_thrust=0.5)

    # ---- device-resident step --------------------------------------------------------------------
    y0 = torch.from_numpy(Y).to(dev)
    tfd = torch.full((N,), tf, dtype=torch.float64, device=dev)
    x = torch.empty((N, 7, K), dtype=torch.float64, device=dev)
    u = torch.empty((N, 3, K), dtype=torch.float64, device=dev)
    stp = torch.empty(N, dtype=torch.int32, device=dev)
    std = torch.empty(n_int, dtype=torch.int32, device=dev)
    out = torch.empty((105, n_int), dtype=torch.float64, device=dev) if world == 1 else None
    flush = torch.empty(256 * 1024 * 1024 // 8, dtype=torch.float64, device=dev)
    n_prop = M.batch.default_n_sub(K) if args.prop == "rk4" else 0   # 0: the reference's RK45, replayed (default)
    fused = None
    gather_mode = "none"
    if world > 1:
        gather_mode = args.gather
        if gather_mode == "nccl" and N_total % world:
            raise SystemExit("--gather nccl needs equal shards (total satellites divisible by the number of ranks)")
        if gather_mode == "fused":
            try:
                fused = D.FusedGather(N_total, K, device=dev, mode=args.fused_mode, chunk_waves=args.chunk_waves,
                                      layout=args.layout)
            except Exception as exc:            # no peer mapping on this box: fall back to the NCCL baseline
                if rank == 0:
                    print(f"[bench] symmetric memory unavailable ({exc}); using the NCCL all-gather", file=sys.stderr)
                gather_mode = "nccl"
        if gather_mode == "nccl":
            local_out = torch.empty((105, n_int), dtype=torch.float64, device=dev)
            comm_stream = torch.cuda.Stream(dev)
            col_chunk = ((N + args.chunks - 1) // args.chunks) * (K - 1)

    # One linearization pass.  Default: the propagation is hidden behind the discretization (the intervals are
    # discretized window by window along k as the propagation publishes its progress, mpc_propagate_discretize);
    # --no-overlap runs the two kernels back to back (what the ncu launch list under profiles/ serialises anyway).
    overlap = not args.no_overlap and (world == 1 or (fused is not None and fused.overlap_ok and
                                                      args.fused_mode in ("unicast", "multicast")))
    if N == 0:
        raise SystemExit("a rank without satellites: use fewer GPUs for this --total-sats")

    def step():
        if overlap and world == 1:
            M.propagate_discretize_device(y0, tfd, ctrl, const, K, n_sub_prop=n_prop, n_sub_disc=n_sub, y=x, u_out=u,
                                          out=out, status_prop=stp, status_disc=std, n_windows=args.windows)
            return
        if overlap:
            # ... and every result is stored into all ranks' gathered buffers (peer stores over NVLink)
            fused.propagate_discretize(y0, tfd, ctrl, const, n_sub_prop=n_prop, n_sub=n_sub, y=x, u_out=u, status_prop=stp,
                                       barrier=True, n_windows=args.windows)
            return
        M.propagate_batch_device(y0, tfd, ctrl, const, include_drag=False, include_J2=False, T=K, n_sub=n_prop,
                                 y=x, u_out=u, status=stp)
        if world == 1:
            M.discretize_batch_device(x, u, tfd, const, n_sub=n_sub, out=out, status=std)
        elif fused is not None:
            # the kernel stores every result into all ranks' gathered buffers (peer stores over NVLink)
            fused.discretize(x, u, tfd, const, n_sub=n_sub, barrier=True)
        else:
            def produce(c0, c1):
                s0, s1 = c0 // (K - 1), c1 // (K - 1)
                M.discretize_batch_device(x[s0:s1], u[s0:s1], tfd[s0:s1], const, n_sub=n_sub, out=local_out,
                                          out_offset=c0, status=std[c0:c1])
            step.gathered = D.nccl_gather_chunks(local_out, args.chunks, side_stream=comm_stream, produce=produce,
                                                 chunk_cols=col_chunk)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize(dev)

    for _ in range(max(args.warmup, 3)):
        step()
    barrier()
    assert int(stp.max()) == 0 and int((fused.status if fused is not None else std).max()) == 0, "device status flags set"
    peak_tflops, _ = M.fp64_peak_tflops(local, repeats=5)
    sampler = ClockSampler(local)
    sampler.start()
    launches0 = M.launch_count()
    step_ms, disc_ms, prop_ms = [], [], []
    for _ in range(args.steps):
        flush.fill_(1.0)
        barrier()
        e0, e3 = (torch.cuda.Event(enable_timing=True) for _ in range(2))
        e0.record()
        step()
        e3.record()
        torch.cuda.synchronize(dev)
        step_ms.append(e0.elapsed_time(e3))
    launches = M.launch_count() - launches0
    if args.dump_outputs:
        # before the stand-alone kernel timings below overwrite the buffers
        dump_outputs(args.dump_outputs, out, x, u, stp, std)
    # The two kernels on their own (same inputs, same L2 flush, same clock sampling window): the discretization
    # kernel's launch duration is what `roofline` is computed from.  Inside the overlapped step the same kernel runs
    # as windows beside the propagation, so it cannot be bracketed by events there.
    scratch = out if world == 1 else torch.empty((105, n_int), dtype=torch.float64, device=dev)
    # (one untimed call first: the stand-alone launch of the propagator is a different kernel instantiation than the one
    #  the overlapped step uses, and the driver loads a kernel's code at its first launch -- ~8 ms, once)
    M.propagate_batch_device(y0, tfd, ctrl, const, include_drag=False, include_J2=False, T=K, n_sub=n_prop,
                             y=x, u_out=u, status=stp)
    M.discretize_batch_device(x, u, tfd, const, n_sub=n_sub, out=scratch, status=std)
    for _ in range(args.steps):
        flush.fill_(1.0)
        torch.cuda.synchronize(dev)
        e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        e0.record()
        M.propagate_batch_device(y0, tfd, ctrl, const, include_drag=False, include_J2=False, T=K, n_sub=n_prop,
                                 y=x, u_out=u, status=stp)
        e1.record()
        M.discretize_batch_device(x, u, tfd, const, n_sub=n_sub, out=scratch, status=std)
        e2.record()
        torch.cuda.synchronize(dev)
        prop_ms.append(e0.elapsed_time(e1))
        disc_ms.append(e1.elapsed_time(e2))
    clocks = sampler.stop()
    if world > 1:
        del scratch
    # the reference's shipped default quadrature mode (adaptive RK45 nodes, replayed on the device): reported
    # next to the headline, which is the fixed-step RK4 / 101-node mode north_star names
    adaptive_ms = None
    if world == 1:
        nn = torch.empty(n_int, dtype=torch.int32, device=dev)
        ts = []
        for _ in range(4):
            ea, eb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ea.record()
            M.discretize_batch_device(x, u, tfd, const, out=out, status=std, adaptive=dict(rtol=1e-3, atol=1e-6, max_step=1e-2),
                                      n_nodes=nn)
            eb.record()
            torch.cuda.synchronize(dev)
            ts.append(ea.elapsed_time(eb))
        adaptive_ms = float(min(ts[1:]))
        adaptive_nodes = (int(nn.min()), int(nn.max()))
        M.discretize_batch_device(x, u, tfd, const, n_sub=n_sub, out=out, status=std)   # restore the headline result
        torch.cuda.synchronize(dev)
    total_ms = float(np.sum(step_ms))
    if dist is not None:
        t = torch.tensor([total_ms, float(np.sum(disc_ms)), float(np.sum(prop_ms))], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms, disc_total, prop_total = float(t[0]), float(t[1]), float(t[2])
        lt = torch.tensor([launches], dtype=torch.int64, device=dev)
        dist.all_reduce(lt)
        launches = int(lt[0])
    else:
        disc_total, prop_total = float(np.sum(disc_ms)), float(np.sum(prop_ms))
    prop_ms_avg = prop_total / args.steps
    ms_per_step = total_ms / args.steps
    value = n_int_total / (ms_per_step * 1e-3)
    disc_ms_avg = disc_total / args.steps

    # ---- end to end through the public host API (pinned host buffers, H2D + D2H inside the timed region) --
    # every rank keeps its host thread and its pinned buffers on the NUMA node of its own GPU (first touch)
    cpus0 = os.sched_getaffinity(0)
    cpus = M.bind_host_to_gpu(local_phys)
    y0_h = M.pinned_empty((N, 7))
    y0_h[:] = Y
    out_h = M.pinned_empty((105, n_int))
    y_h = M.pinned_empty((N, 7, K))
    u_h = M.pinned_empty((N, 3, K))
    st_h = M.pinned_empty(n_int, np.int32)
    e2e_t = []
    for i in range(2 + max(3, args.steps // 2)):
        barrier()
        t0 = time.perf_counter()
        res, _, _ = M.propagate_discretize(y0_h, tf, ctrl, const, T=K, n_sub_prop=n_prop, n_sub_disc=n_sub, out=out_h,
                                           y_out=y_h, u_out=u_h, status=st_h, device=local, layout=args.e2e_layout)
        dt = time.perf_counter() - t0
        if i >= 2:
            e2e_t.append(dt)
    e2e_s = float(np.mean(e2e_t))
    os.sched_setaffinity(0, cpus0)          # the CPU baseline below uses every host core again
    if dist is not None:
        t = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t[0])
    # parity spot check inside the bench: device-resident result == host-API result
    if world == 1:
        dev_cols = out[:, :K - 1]
    elif fused is not None:
        # the K-1 intervals of this rank's first satellite, wherever the gathered layout puts them
        dev_cols = (fused.buf[:, s0:s0 + (K - 1) * N_total:N_total] if fused.layout == "kmajor"
                    else fused.buf[:, s0 * (K - 1):(s0 + 1) * (K - 1)])
    else:
        dev_cols = local_out[:, :K - 1]
    # (the K-1 intervals of the first satellite of this rank, wherever the host layout puts them)
    host_cols = out_h[:, 0:(K - 1) * N:N] if args.e2e_layout == "kmajor" else out_h[:, :K - 1]
    same = bool(np.array_equal(host_cols, dev_cols.cpu().numpy()))
    gathered_ok = None
    if fused is not None:
        # every rank must hold every other rank's block: compare a column of each peer block with its owner
        # (interval k = 7 of the first satellite of every rank)
        first = [D.shard_range(N_total, r, world)[0] for r in range(world)]
        colof = (lambda sg: 7 * N_total + sg) if fused.layout == "kmajor" else (lambda sg: sg * (K - 1) + 7)
        probe = torch.stack([fused.buf[:, colof(first[r])] for r in range(world)])
        mine = fused.buf[:, colof(s0)].clone()
        allm = [torch.empty_like(mine) for _ in range(world)]
        dist.all_gather(allm, mine)
        gathered_ok = bool(all(torch.equal(probe[r], allm[r]) for r in range(world)))

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak, hbm_src = (peaks["hbm_gbs"], "MEASURED_PEAKS.json") if "hbm_gbs" in peaks else (6650.0, "fallback (B200_PROFILING.md)")
    counters = kernel_counters()
    is_cfg3 = (N, K, n_sub, world) == (4096, 200, 100, 1)
    pair_ctr = counters.get("discretize_pair_kernel", {}) if is_cfg3 else {}
    # executed FP64 work per interval: the ncu count of this very workload where one is committed (profiles/
    # kernel_counters.json), the count from the SASS of the loop bodies otherwise (within 2 % of each other)
    fl = pair_ctr.get("flop_per_interval") or flops_per_interval(n_sub)
    fp64_ipi = pair_ctr.get("fp64_instr_per_interval") or fp64_instr_per_interval(n_sub)
    achieved_tflops = fl * n_int / (disc_ms_avg * 1e-3) / 1e12
    dflt_ctr = counters.get("discretize_default_kernel", {}) if is_cfg3 else {}
    # the CPU baseline is a rank-0, N=1 measurement (under torchrun OMP_NUM_THREADS=1 would make it a one-core number)
    cpu = cpu_port_baseline(N, K, tf, n_sub) if (world == 1 and not args.no_cpu_baseline) else None
    line = {
        "metric": "discretized intervals/sec", "value": value, "unit": "intervals/s", "n_gpus": world,
        "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True,
        "scaling": "strong" if args.total_sats else "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args),
        "e2e": {"value": n_int_total / e2e_s, "unit": "intervals/s", "ms_per_step": e2e_s * 1e3,
                "h2d_bytes_per_step": int(y0_h.nbytes + N * 8),
                # (the 7 structural-constant rows of A_k are written by the host, not copied: 98 of the 105 rows cross PCIe)
                "d2h_bytes_per_step": int(out_h.nbytes // 105 * 98 + y_h.nbytes + u_h.nbytes + n_int * 4),
                "api": ("mpconstellation_b200.propagate_discretize(layout='kmajor') (C-ABI mpc_propagate_discretize_host_layout: k-windows "
                        "gated on the propagation's progress, every window read back while the next one runs), pinned host buffers"
                        if args.e2e_layout == "kmajor" else
                        "mpconstellation_b200.propagate_discretize (C-ABI mpc_propagate_discretize_host), pinned host buffers"),
                "host_cpus_rank0": len(cpus),
                "matches_device_path": same},
        "gather": {"mode": gather_mode + (":" + args.fused_mode if fused is not None else ""), "verified": gathered_ok,
                   "layout": fused.layout if fused is not None else "rank blocks",
                   "bytes_received_per_rank_per_step": int((n_int_total - n_int) * 8 * (98 if fused is not None and fused.skip_const else 105)),
                   "note": "rows 42..48 of the SoA result (last row of A_k, constants) are written once by the owner and never sent"
                           if fused is not None and fused.skip_const else None} if world > 1 else None,
        "gpu_launches": int(launches),
        "kernel": {"discretize_ms": disc_ms_avg, "propagate_ms": prop_ms_avg,
                   "timing": "each kernel launched on its own right after the timed steps (CUDA events, L2 flushed); "
                             "back_to_back_ms is their sum, ms_per_step the step as shipped",
                   "back_to_back_ms": disc_ms_avg + prop_ms_avg,
                   "overlap": ("propagation hidden behind the discretization: windows along k gated by stream memory operations "
                               "(mpc_propagate_discretize), bit-identical results") if overlap else "none (kernels back to back)",
                   # SURVEY 8(d): propagation is sequential in tau (latency-bound), reported as satellite-steps/s
                   "propagator": "scipy RK45 replayed (max_step 0.001: 1000 steps x 6 stages per satellite), dense-output samples"
                                 if n_prop == 0 else f"fixed-step RK4, {(K - 1) * n_prop} steps x 4 stages per satellite",
                   "propagate_sat_steps_per_s": N * (1000 if n_prop == 0 else (K - 1) * n_prop) / (prop_ms_avg * 1e-3),
                   "discretize_intervals_per_s_per_gpu": n_int / (disc_ms_avg * 1e-3),
                   "default_mode_adaptive_rk45": None if adaptive_ms is None else {
                       "discretize_ms": adaptive_ms, "intervals_per_s": n_int / (adaptive_ms * 1e-3),
                       "nodes_per_interval": list(adaptive_nodes),
                       "note": "use_uniform_steps=False (reference default): quadrature on scipy-RK45 accepted steps"}},
        "roofline": {"bound": "fp64", "achieved": achieved_tflops, "peak": peak_tflops, "unit": "TFLOP/s",
                     "frac": achieved_tflops / peak_tflops,
                     # the conservative reading: the same flops over the WHOLE step (propagation, window gating and
                     # -- at N > 1 -- the exchange included)
                     "in_step": {"achieved": fl * n_int / (ms_per_step * 1e-3) / 1e12,
                                 "frac": fl * n_int / (ms_per_step * 1e-3) / 1e12 / peak_tflops},
                     # dram__bytes_read.sum + dram__bytes_write.sum of one full-batch launch, ncu --set full capture of
                     # this command (profiles/r01_n_discretize_pair_windows.txt, third kernel: 65.80 + 628.39 MB);
                     # algorithmic = 944 B x 815,104 = 769.5 MB (the 13 input doubles are shared by neighbours in L2)
                     # committed in profiles/kernel_counters.json together with the name of the summary it was read from
                     "traffic": pair_ctr.get("dram_bytes"), "traffic_source": pair_ctr.get("source"),
                     "peak_source": "DFMA-chain microbenchmark (mpc_fp64_peak_probe) in this run; MEASURED_PEAKS.json has no FP64 entry",
                     "peak_nominal": FP64_NOMINAL_TFLOPS, "flop_per_interval": fl,
                     # SURVEY.md 8(d) counts the reference formulation (plain RK4 on 42+7 unknowns, dense Phi^-1
                     # products): 2084 n_sub + 1386 flop per interval.  The kernel executes fewer (Nystrom form,
                     # symplectic inverse, Euler identity), so `achieved`/`frac` above use the EXECUTED count (the
                     # conservative reading); this is the same throughput priced at the survey's count.
                     # the same throughput priced at the work of evaluating all 101 nodes (the kernel of
                     # mpc_set_tuning(37): two-node steps with a Hermite midpoint), for comparison with round 1
                     "all_nodes_alg": {"flop_per_interval": flops_per_interval(n_sub, em=False),
                                       "achieved": flops_per_interval(n_sub, em=False) * n_int / (disc_ms_avg * 1e-3) / 1e12,
                                       "frac": flops_per_interval(n_sub, em=False) * n_int / (disc_ms_avg * 1e-3) / 1e12 / peak_tflops},
                     "survey_alg": {"flop_per_interval": 2084 * n_sub + 1386,
                                    "achieved": (2084 * n_sub + 1386) * n_int / (disc_ms_avg * 1e-3) / 1e12,
                                    "frac": (2084 * n_sub + 1386) * n_int / (disc_ms_avg * 1e-3) / 1e12 / peak_tflops},
                     "fp64_pipe_frac": fp64_ipi * n_int / (disc_ms_avg * 1e-3) / (peak_tflops * 1e12 / 2),
                     "flop_source": pair_ctr.get("source") or "bench.py: flops_per_interval (SASS count of the loop bodies)",
                     "fp64_pipe_note": "FP64 instructions issued / (measured DFMA issue rate): DMUL/DADD occupy a DFMA slot but count 1 flop",
                     "kernel": "mpc::discretize_pair_kernel",
                     "hbm": {"achieved": bytes_per_interval() * n_int / (disc_ms_avg * 1e-3) / 1e9, "peak": hbm_peak,
                             "unit": "GB/s", "peak_source": hbm_src, "bytes_per_interval": bytes_per_interval()}},
        "clocks": clocks,
    }
    if adaptive_ms is not None:
        # the reference's DEFAULT quadrature mode (what control.py:187 runs): its own roofline block.  The executed flop
        # count depends on the data (3-4 accepted RK45 steps per interval here) and is the ncu count of this workload
        fpi, ipi = dflt_ctr.get("flop_per_interval"), dflt_ctr.get("fp64_instr_per_interval")
        line["roofline_default_mode"] = {
            "kernel": "mpc::discretize_default_kernel", "bound": "fp64", "discretize_ms": adaptive_ms,
            "intervals_per_s": n_int / (adaptive_ms * 1e-3), "nodes_per_interval": list(adaptive_nodes),
            "flop_per_interval": fpi, "flop_source": dflt_ctr.get("source"),
            "achieved": None if fpi is None else fpi * n_int / (adaptive_ms * 1e-3) / 1e12, "peak": peak_tflops, "unit": "TFLOP/s",
            "frac": None if fpi is None else fpi * n_int / (adaptive_ms * 1e-3) / 1e12 / peak_tflops,
            "fp64_pipe_frac": None if ipi is None else ipi * n_int / (adaptive_ms * 1e-3) / (peak_tflops * 1e12 / 2),
            "traffic": dflt_ctr.get("dram_bytes"),
            "note": "use_uniform_steps=False: scipy's RK45 controller replayed per interval, trapezoid on the accepted steps"}
    if cpu is not None:
        line["cpu_baseline"] = cpu
        line["vs_cpu_port"] = {"device": value / cpu["value"], "e2e": line["e2e"]["value"] / cpu["value"],
                               "note": "this line's value and e2e over cpu_baseline.value (oracle/mpc_oracle.c, OpenMP, all host cores)"}
    if world == 1 and not args.no_configs:
        line["configs"] = small_configs_record(M, dev, const, not args.no_cpu_baseline)
    print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--sats", type=int, default=4096, help="satellites per GPU")
    ap.add_argument("--nodes", type=int, default=200, help="K temporal nodes")
    ap.add_argument("--tf", type=float, default=2.0)
    ap.add_argument("--n-sub", dest="n_sub", type=int, default=100, help="RK4 steps per interval (integrator_steps-1)")
    ap.add_argument("--chunks", type=int, default=8, help="compute/all-gather overlap chunks (N>1, --gather nccl)")
    ap.add_argument("--fused-mode", dest="fused_mode", default="unicast", choices=["unicast", "multicast", "push", "pushk"])
    ap.add_argument("--chunk-waves", dest="chunk_waves", type=int, default=1, help="--fused-mode push: kernel waves per pushed chunk")
    ap.add_argument("--gather", default="fused", choices=["fused", "nccl"],
                    help="N>1: all-gather by peer stores from inside the kernel (fused) or chunked NCCL all-gather")
    ap.add_argument("--ref-sats", dest="ref_sats", type=int, default=8, help="satellites per step of the reference arm")
    ap.add_argument("--total-sats", dest="total_sats", type=int, default=0,
                    help="strong scaling: this many satellites in total, sharded over the ranks (5025 = BASELINE configs[3])")
    ap.add_argument("--no-configs", dest="no_configs", action="store_true", help="skip the configs 1/2/5 record (N=1)")
    ap.add_argument("--e2e-layout", dest="e2e_layout", default="kmajor", choices=["satmajor", "kmajor"],
                    help="layout of the matrices the end-to-end leg hands back (kmajor: the streamed pass)")
    ap.add_argument("--layout", default=None, choices=["satmajor", "kmajor"], help="gathered layout of the fused all-gather")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-overlap", dest="no_overlap", action="store_true",
                    help="run propagate and discretize back to back instead of overlapped")
    ap.add_argument("--prop", default="rk45", choices=["rk45", "rk4"],
                    help="propagator: the reference's RK45 replayed step for step (default) or fixed-step RK4")
    ap.add_argument("--windows", type=int, default=0, help="windows along k of the overlapped pass (0 = library default)")
    ap.add_argument("--dump-outputs", dest="dump_outputs", metavar="DIR", default=None,
                    help="write a seeded sample of the last timed step's results to DIR/<name>.npy (one GPU)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.gpus != 1 or int(os.environ.get("WORLD_SIZE", "1")) != 1):
        ap.error("--dump-outputs needs the CUDA path on one GPU")
    if args.impl == "reference":
        reference_arm(args)
    else:
        gpu_arm(args)


if __name__ == "__main__":
    main()
