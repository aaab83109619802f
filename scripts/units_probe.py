"""Per-satellite designer units on one GPU: what the one-launch-per-leg form costs.

  config 5's shape (256 satellites, K = 60, every satellite in its own units): one *_units launch per leg (RK45
           propagation, default-mode and fixed-step discretization, constraint terms) against 256 per-satellite launches
           of the same leg, and against one single-constant launch of the batch (wrong units: a cost reference only);
  config 3 (4096 x 200, all constants equal): the fixed-step (without and with J2) and default-mode discretization forced
           through the *_units entry point against the rectangular entry point, alternated in the same process -- the
           cost of the table (and, fixed-step, of taking the ragged kernel with equal counts).

CUDA events around each variant over `--reps` repetitions, the L2 flushed (256 MB written) before every one; medians
with min / max.  Writes profiles/units_probe.json with the card name and power limit read in the same run.

    python scripts/units_probe.py [--reps 15] [--out profiles/units_probe.json]
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def mixed_constellation(n):
    """n satellites from dimensional states: perigee altitudes 400 km ... 20,000 km, masses 300 ... 12,200 kg,
    eccentricities 0 ... 0.3, inclinations 0 ... 98 deg, each normalized by its own SatelliteScale (the constellation of
    the tests of the per-satellite kernels)"""
    from mpconstellation_b200.model import MU_EARTH, R_EARTH, Satellite, sat_units
    alt = np.array([400e3, 20000e3, 1200e3, 7000e3, 550e3, 3500e3])
    mass = np.array([12200.0, 300.0, 2500.0, 800.0, 5000.0, 1500.0])
    ecc = np.array([0.0, 0.05, 0.3, 0.0, 0.1, 0.2])
    inc = np.radians([28.5, 0.0, 63.4, 98.0, 51.6, 10.0])
    sats = []
    for i in range(n):
        j = i % 6
        rp = R_EARTH + alt[j] * (1 + 0.01 * (i // 6))
        vp = np.sqrt(MU_EARTH * (1 + ecc[j]) / rp)
        ci, si = np.cos(inc[j]), np.sin(inc[j])
        sats.append(Satellite(np.array([rp, 0.0, 0.0]), np.array([0.0, vp * ci, vp * si]), mass[j]))
    return sat_units(sats)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=15)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "units_probe.json"))
    a = ap.parse_args()
    import torch
    import mpconstellation_b200 as M
    from mpconstellation_b200 import _lib
    _lib.require_gpu()
    L = _lib.lib()
    dev = torch.device("cuda")
    stream = torch.cuda.current_stream().cuda_stream
    flush = torch.empty(256 * 1024 * 1024 // 8, dtype=torch.float64, device=dev)

    def timed(fn):
        fn()
        torch.cuda.synchronize()
        ts = []
        for _ in range(a.reps):
            flush.fill_(1.0)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1))
        return {"median_ms": float(np.median(ts)), "min_ms": float(np.min(ts)), "max_ms": float(np.max(ts))}

    res = {}
    # ---- config 5's shape, heterogeneous constants ------------------------------------------------------------------
    N, K, tf = 256, 60, 0.3
    y0, consts = mixed_constellation(N)
    ctrl = M.ConstantTangentialThrustController(tangential_thrust=0.05)
    y0d, tfd = torch.as_tensor(y0).to(dev), torch.full((N,), tf, dtype=torch.float64, device=dev)
    y = torch.empty((N, 7, K), dtype=torch.float64, device=dev)
    u = torch.empty((N, 3, K), dtype=torch.float64, device=dev)
    st = torch.empty(N, dtype=torch.int32, device=dev)
    M.propagate_batch_device(y0d, tfd, ctrl, consts, include_drag=False, include_J2=False, T=K, y=y, u_out=u, status=st)
    torch.cuda.synchronize()
    assert int(st.max()) == 0
    out = torch.empty((105, N * (K - 1)), dtype=torch.float64, device=dev)
    ds = torch.empty(N * (K - 1), dtype=torch.int32, device=dev)
    AD = dict(rtol=1e-3, atol=1e-6, max_step=1e-2)
    legs = {
        "rk45": lambda c, sl: M.propagate_batch_device(y0d[sl], tfd[sl], ctrl, c, include_drag=False, include_J2=False, T=K,
                                                      y=y[sl], u_out=u[sl], status=st[sl]),
        "default_mode": lambda c, sl: M.discretize_batch_device(y[sl], u[sl], tfd[sl], c, adaptive=AD),
        "fixed_step": lambda c, sl: M.discretize_batch_device(y[sl], u[sl], tfd[sl], c, n_sub=100),
        "constraint_terms": lambda c, sl: M.constraint_terms_device(y[sl], u[sl], c),
    }
    c5 = {}
    for name, leg in legs.items():
        all_ = slice(0, N)

        def per_sat(leg=leg):
            for s in range(N):
                leg(consts[s], slice(s, s + 1))
        c5[name] = {"units_one_launch": timed(lambda leg=leg: leg(consts, all_)),
                    "per_satellite_launches": timed(per_sat),
                    "single_constant_launch_wrong_units": timed(lambda leg=leg: leg(consts[0], all_))}
    res["config5_256x60_mixed_units"] = c5

    # ---- config 3, all constants equal: the cost of reading the table -----------------------------------------------
    N3, K3 = 4096, 200
    y03, c3 = mixed_constellation(1)
    y03 = np.repeat(y03, N3, axis=0)
    y03[:, 3:6] *= (1 + 1e-3 * np.arange(N3) / N3)[:, None]
    y3d, tf3 = torch.as_tensor(y03).to(dev), torch.full((N3,), tf, dtype=torch.float64, device=dev)
    x3, u3, st3 = M.propagate_batch_device(y3d, tf3, ctrl, c3[0], include_drag=False, include_J2=False, T=K3)
    torch.cuda.synchronize()
    out3 = torch.empty((105, N3 * (K3 - 1)), dtype=torch.float64, device=dev)
    s3 = torch.empty(N3 * (K3 - 1), dtype=torch.int32, device=dev)
    nn3 = torch.empty(N3 * (K3 - 1), dtype=torch.int32, device=dev)
    scratch = torch.empty(N3 * _lib.SAT_SCRATCH_DOUBLES, dtype=torch.float64, device=dev)
    arr = (_lib.MpcSatConsts * N3)()
    c = c3[0]
    for s in range(N3):
        arr[s] = _lib.MpcSatConsts(c.MU, c.R_E, c.J2, c.G0, c.ISP, c.S, c.RHO)

    def units(adaptive, j2=False):
        p = _lib.make_params(c, include_J2=j2)
        _lib.check(L.mpc_discretize_batch_units(x3.data_ptr(), u3.data_ptr(), tf3.data_ptr(), ctypes.byref(p), arr, N3, K3,
                                                None, None, scratch.data_ptr(), int(adaptive), 100, 1e-3, 1e-6, 1e-2,
                                                out3.data_ptr(), N3 * (K3 - 1), 0, s3.data_ptr(), nn3.data_ptr(), stream))

    def rect(adaptive, j2=False):
        M.discretize_batch_device(x3, u3, tf3, c, include_J2=j2, adaptive=AD if adaptive else None, out=out3, status=s3,
                                  n_nodes=nn3 if adaptive else None)
    c3r = {}
    for name, adaptive, j2 in (("fixed_step", False, False), ("fixed_step_j2", False, True), ("default_mode", True, False)):
        rect(adaptive, j2)
        torch.cuda.synchronize()
        ref = out3.clone()
        units(adaptive, j2)
        torch.cuda.synchronize()
        same = bool(torch.equal(ref, out3))
        r_runs, u_runs = [], []
        for _ in range(2):                        # alternated: r, u, r, u
            r_runs.append(timed(lambda: rect(adaptive, j2)))
            u_runs.append(timed(lambda: units(adaptive, j2)))
        rm = float(np.median([r["median_ms"] for r in r_runs]))
        um = float(np.median([r["median_ms"] for r in u_runs]))
        c3r[name] = {"rectangular": r_runs, "units_all_equal": u_runs, "units_over_rectangular": um / rm,
                     "bit_identical": same}
    res["config3_4096x200_equal_constants"] = c3r
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip()
    res["gpu"] = q
    res["reps"] = a.reps
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
