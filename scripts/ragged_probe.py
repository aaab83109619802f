"""Ragged batches on one GPU: what one launch per leg costs against the launches that reproduce the reference's
per-satellite grids today.

Config 5's shape (256 satellites, base_res 30, tf_s spread over [1, 2], so K_s = int(30 tf_s) in 30..60), both modes of
the discretization plus the RK45 propagation, each timed with CUDA events over `--reps` repetitions, the L2 flushed before
every one:
  (a) ragged  -- one ragged launch for the whole batch (device entry points, per-satellite counts)
  (b) per_K   -- one rectangular launch per distinct K_s (what a user has to do today to get the reference's grids)
  (c) padded  -- one rectangular launch at Kmax for every satellite (the wrong grid; the cost floor)
and config 3 (4096 x 200) with all counts equal through the ragged entry against the rectangular one (the index search).
Writes profiles/ragged_probe.json with the card name and power limit.

    python scripts/ragged_probe.py [--reps 20] [--out profiles/ragged_probe.json]
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
sys.path.insert(0, os.path.join(ROOT, "tests"))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "ragged_probe.json"))
    a = ap.parse_args()
    import torch
    import mpconstellation_b200 as M
    from conftest import synth_batch
    from oracle.mpc_oracle import OracleConstants
    M._lib.require_gpu()
    L = M._lib.lib()
    const = OracleConstants(*np.load(os.path.join(ROOT, "tests", "golden", "discretize.npz"))["const"])
    dev = torch.device("cuda")
    stream = torch.cuda.current_stream().cuda_stream
    flush = torch.empty(256 * 1024 * 1024 // 8, dtype=torch.float64, device=dev)   # 256 MB > 126 MB of L2

    def timed(fn):
        fn()                                             # warm-up: module load, smem carve-out
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

    p_disc = M._lib.make_params(const, False, False)
    p_prop = M._lib.make_params(const, False, False)
    ctrl = M._lib.MpcController()
    ctrl.kind = M._lib.CTRL_TANGENTIAL
    ctrl.thrust[0] = 0.5

    def disc_rect(xd, ud, tfd, N, K, adaptive, out, status, nodes):
        if adaptive:
            M._lib.check(L.mpc_discretize_batch_adaptive(xd.data_ptr(), ud.data_ptr(), tfd.data_ptr(), ctypes.byref(p_disc), N, K,
                                                         1e-3, 1e-6, 1e-2, out.data_ptr(), out.shape[1], 0, status.data_ptr(),
                                                         nodes.data_ptr(), stream))
        else:
            M._lib.check(L.mpc_discretize_batch(xd.data_ptr(), ud.data_ptr(), tfd.data_ptr(), ctypes.byref(p_disc), N, K, 100,
                                                out.data_ptr(), out.shape[1], 0, status.data_ptr(), stream))

    def disc_ragged(xd, ud, tfd, K_sat, first, adaptive, out, status, nodes):
        N, Kmax = xd.shape[0], xd.shape[2]
        M._lib.check(L.mpc_discretize_batch_ragged(xd.data_ptr(), ud.data_ptr(), tfd.data_ptr(), ctypes.byref(p_disc), N, Kmax,
                                                   K_sat.ctypes.data, first.data_ptr(), int(adaptive), 100, 1e-3, 1e-6, 1e-2,
                                                   out.data_ptr(), out.shape[1], 0, status.data_ptr(),
                                                   nodes.data_ptr() if adaptive else None, stream))

    res = {"gpu": torch.cuda.get_device_name(0)}
    try:
        res["power_limit"] = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                                            capture_output=True, text=True).stdout.strip()
    except OSError:
        res["power_limit"] = "unknown"

    # ---- config 5: 256 satellites, tf_s over [1, 2] -----------------------------------------------------------------
    N = 256
    tf = np.linspace(1.0, 2.0, N)
    K_sat = np.array([int(30 * t) for t in tf], dtype=np.int32)
    Kmax = int(K_sat.max())
    y0, _, _ = synth_batch(N, 2, 1.0, const)
    ctl = M.ConstantTangentialThrustController(tangential_thrust=0.5)
    x, u, _, _ = M.propagate_batch(y0, tf, ctl, const, include_drag=False, include_J2=False, T=K_sat)
    xd = torch.as_tensor(np.nan_to_num(np.array(x))).to(dev).contiguous()
    ud = torch.as_tensor(np.nan_to_num(np.array(u))).to(dev).contiguous()
    tfd = torch.as_tensor(tf).to(dev).contiguous()
    y0d = torch.as_tensor(y0).to(dev).contiguous()
    # (c): what BatchedSCP did before per-satellite grids -- every satellite propagated and discretized on Kmax nodes
    xp, up, _, _ = M.propagate_batch(y0, tf, ctl, const, include_drag=False, include_J2=False, T=Kmax)
    xpd = torch.as_tensor(np.array(xp)).to(dev).contiguous()
    upd = torch.as_tensor(np.array(up)).to(dev).contiguous()
    out = torch.empty((105, N * (Kmax - 1)), dtype=torch.float64, device=dev)
    status = torch.zeros(N * (Kmax - 1), dtype=torch.int32, device=dev)
    nodes = torch.zeros(N * (Kmax - 1), dtype=torch.int32, device=dev)
    first = torch.empty(N + 1, dtype=torch.int64, device=dev)
    groups = {}
    for k in np.unique(K_sat):                          # (b): contiguous copies per distinct K, made outside the timing
        idx = np.nonzero(K_sat == k)[0]
        it = torch.as_tensor(idx, device=dev)
        groups[int(k)] = (xd[it, :, :k].contiguous(), ud[it, :, :k].contiguous(), tfd[it].contiguous(), y0d[it].contiguous(),
                          torch.empty((105, len(idx) * (k - 1)), dtype=torch.float64, device=dev),
                          torch.zeros(len(idx) * (k - 1), dtype=torch.int32, device=dev),
                          torch.zeros(len(idx) * (k - 1), dtype=torch.int32, device=dev), len(idx))
    c5 = {"n_sats": N, "distinct_K": len(groups), "K_range": [int(K_sat.min()), Kmax],
          "live_intervals": int((K_sat - 1).sum()), "padded_intervals": N * (Kmax - 1)}
    for mode, adaptive in (("default", True), ("fixed_step", False)):
        c5[mode] = {
            "a_ragged": timed(lambda: disc_ragged(xd, ud, tfd, K_sat, first, adaptive, out, status, nodes)),
            "b_per_K": timed(lambda: [disc_rect(g[0], g[1], g[2], g[7], k, adaptive, g[4], g[5], g[6]) for k, g in groups.items()]),
            "c_padded": timed(lambda: disc_rect(xpd, upd, tfd, N, Kmax, adaptive, out, status, nodes)),
        }
    # propagation leg (RK45, the reference's integrator)
    T_dev = torch.as_tensor(K_sat).to(dev)
    yb = torch.empty((N, 7, Kmax), dtype=torch.float64, device=dev)
    ub = torch.empty((N, 3, Kmax), dtype=torch.float64, device=dev)
    sp = torch.zeros(N, dtype=torch.int32, device=dev)

    def prop_ragged():
        M._lib.check(L.mpc_propagate_batch_rk45_ragged(y0d.data_ptr(), tfd.data_ptr(), ctypes.byref(p_prop), ctypes.byref(ctrl),
                                                       N, Kmax, T_dev.data_ptr(), None, 1e-3, 1e-6, 1e-3, yb.data_ptr(), ub.data_ptr(),
                                                       sp.data_ptr(), None, stream))

    def prop_rect(y0_, tf_, n, T):
        M._lib.check(L.mpc_propagate_batch_rk45(y0_.data_ptr(), tf_.data_ptr(), ctypes.byref(p_prop), ctypes.byref(ctrl), n, T,
                                                1e-3, 1e-6, 1e-3, yb.data_ptr(), ub.data_ptr(), sp.data_ptr(), None, stream))

    c5["propagate_rk45"] = {
        "a_ragged": timed(prop_ragged),
        "b_per_K": timed(lambda: [prop_rect(g[3], g[2], g[7], k) for k, g in groups.items()]),
        "c_padded": timed(lambda: prop_rect(y0d, tfd, N, Kmax)),
    }
    res["config5"] = c5

    # ---- config 3: 4096 x 200, all counts equal: the ragged entry against the rectangular one ---------------------------
    N3, K3 = 4096, 200
    y3, x3, u3 = synth_batch(N3, K3, 1.0, const)
    x3d, u3d = torch.as_tensor(x3).to(dev).contiguous(), torch.as_tensor(u3).to(dev).contiguous()
    tf3 = torch.ones(N3, dtype=torch.float64, device=dev)
    out3 = torch.empty((105, N3 * (K3 - 1)), dtype=torch.float64, device=dev)
    st3 = torch.zeros(N3 * (K3 - 1), dtype=torch.int32, device=dev)
    nn3 = torch.zeros(N3 * (K3 - 1), dtype=torch.int32, device=dev)
    f3 = torch.empty(N3 + 1, dtype=torch.int64, device=dev)
    Ks3 = np.full(N3, K3, dtype=np.int32)
    c3 = {"n_sats": N3, "K": K3}
    for mode, adaptive in (("default", True), ("fixed_step", False)):
        # alternate the two so that drift of the shared machine hits both alike
        r1 = timed(lambda: disc_rect(x3d, u3d, tf3, N3, K3, adaptive, out3, st3, nn3))
        g1 = timed(lambda: disc_ragged(x3d, u3d, tf3, Ks3, f3, adaptive, out3, st3, nn3))
        r2 = timed(lambda: disc_rect(x3d, u3d, tf3, N3, K3, adaptive, out3, st3, nn3))
        g2 = timed(lambda: disc_ragged(x3d, u3d, tf3, Ks3, f3, adaptive, out3, st3, nn3))
        c3[mode] = {"rectangular": [r1, r2], "ragged_equal_counts": [g1, g2]}
    res["config3"] = c3
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
