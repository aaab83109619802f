"""Discretizer.ivp_solver = 'RK23' on one GPU: the RK23 replay of the default quadrature mode against the RK45 one.

  config 3 (4096 x 200, tf = 2, tangential thrust 0.5 on the Hubble family; 0.05 on the mixed constellation): rectangular with one constants bag;
           ragged (K_s = node_counts(100, tf_s), tf_s in [1, 2]: K_s in [100, 200]); every satellite in its own units (mixed constellation);
  config 5's shape (256 satellites, K = 60, mixed constellation in its own units): rectangular and ragged
           (K_s = node_counts(30, tf_s), tf_s in [1, 2]).

Each case runs the RK45 and the RK23 launch of the same batch through discretize_batch_device, alternated in one process
(RK45, RK23, RK45, RK23, ...): CUDA events around each launch, the L2 flushed (256 MB written) before every one, medians
with min / max over `--reps` pairs, and the mean quadrature nodes per interval of each method.  Writes the JSON with the
card name and power limit read in the same run.

    python scripts/rk23_probe.py [--reps 15] [--out profiles/rk23_probe.json]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=15)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "rk23_probe.json"))
    a = ap.parse_args()
    import torch
    import mpconstellation_b200 as M
    from mpconstellation_b200 import _lib
    from mpconstellation_b200.scp import node_counts
    from units_probe import mixed_constellation
    _lib.require_gpu()
    dev = torch.device("cuda")
    flush = torch.empty(256 * 1024 * 1024 // 8, dtype=torch.float64, device=dev)
    AD = dict(rtol=1e-3, atol=1e-6, max_step=1e-2)

    def traj(y0, tf, const, T, thrust=0.05):
        ctrl = M.ConstantTangentialThrustController(tangential_thrust=thrust)
        N = y0.shape[0]
        tfd = torch.as_tensor(np.broadcast_to(np.asarray(tf, dtype=np.float64), (N,)).copy()).to(dev)
        x, u, st = M.propagate_batch_device(torch.as_tensor(y0).to(dev), tfd, ctrl, const, include_drag=False,
                                            include_J2=False, T=T)
        torch.cuda.synchronize()
        assert int(st.max()) == 0
        return x, u, tfd

    def case(x, u, tfd, const, K_sat=None):
        N, _, K = x.shape
        out = torch.empty((105, N * (K - 1)), dtype=torch.float64, device=dev)
        st = torch.zeros(N * (K - 1), dtype=torch.int32, device=dev)
        nn = {m: torch.zeros(N * (K - 1), dtype=torch.int32, device=dev) for m in ("RK45", "RK23")}

        def run(m):
            M.discretize_batch_device(x, u, tfd, const, adaptive=dict(AD, method=m), out=out, status=st, n_nodes=nn[m],
                                      K=K_sat)
        times = {"RK45": [], "RK23": []}
        for m in times:                            # warm-up, every shape and both kernels
            run(m)
        torch.cuda.synchronize()
        assert int(st.max()) == 0
        for _ in range(a.reps):
            for m in ("RK45", "RK23"):
                flush.fill_(1.0)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                run(m)
                e1.record()
                torch.cuda.synchronize()
                times[m].append(e0.elapsed_time(e1))
        live = (nn["RK45"] > 0)
        r = {"n_sats": N, "K_max": K, "intervals": int(live.sum())}
        for m, ts in times.items():
            r[m] = {"median_ms": float(np.median(ts)), "min_ms": float(np.min(ts)), "max_ms": float(np.max(ts)),
                    "mean_nodes_per_interval": float(nn[m][live].double().mean())}
        r["rk23_over_rk45"] = r["RK23"]["median_ms"] / r["RK45"]["median_ms"]
        print(json.dumps(r), flush=True)
        return r

    res = {}
    rng = np.random.default_rng(20261021)
    # ---- config 3: 4096 x 200 --------------------------------------------------------------------------------------
    N3, K3 = 4096, 200
    hubble = np.array([5371.4806e3, -4133.1393e3, 1399.9594e3, 4.6921e3, 4.9848e3, -3.2752e3, 12200.0])
    scale = M.SatelliteScale(x=hubble)
    c1 = scale.get_normalized_constants()
    y0 = np.tile(scale.normalize_state(hubble), (N3, 1))
    y0[:, 3:6] *= (1 + 0.1 * rng.random(N3))[:, None]
    x, u, tfd = traj(y0, 2.0, c1, K3, 0.5)
    res["config3_4096x200_rectangular"] = case(x, u, tfd, c1)
    tfs = rng.uniform(1.0, 2.0, N3)
    K_sat = node_counts(100, tfs)
    x, u, tfd = traj(y0, tfs, c1, K3, 0.5)
    res["config3_4096x200_ragged"] = case(x, u, tfd, c1, K_sat)
    yu, cu = mixed_constellation(N3)
    x, u, tfd = traj(yu, 0.3, cu, K3)
    res["config3_4096x200_units"] = case(x, u, tfd, cu)
    # ---- config 5's shape: 256 x 60, every satellite in its own units -----------------------------------------------
    N5, K5 = 256, 60
    y5, c5 = mixed_constellation(N5)
    x, u, tfd = traj(y5, 0.3, c5, K5)
    res["config5_256x60_units"] = case(x, u, tfd, c5)
    tf5 = rng.uniform(1.0, 2.0, N5)
    K5s = node_counts(30, tf5)
    x, u, tfd = traj(y5, 0.3 * tf5, c5, K5)
    res["config5_256x60_units_ragged"] = case(x, u, tfd, c5, K5s)
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip()
    res["gpu"] = q
    res["reps"] = a.reps
    res["timing"] = "CUDA events per launch, L2 flushed before each, RK45 / RK23 alternated; medians over reps"
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
