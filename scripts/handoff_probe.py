"""The ragged hand-off kernels (constraint terms, sparse dynamics Jacobian) against their rectangular forms on one GPU.

  config 3 (4096 x 200, all counts equal, 815,104 intervals): rectangular vs ragged launch of each kernel, alternated
           in the same process (r, g, r, g) so that drift of the shared machine hits both alike;
  config 5 (256 satellites, base_res 30, tf_s over [1, 2], K_s = int(30 tf_s)): one ragged launch vs the 256
           per-satellite rectangular launches that give the same per-satellite numbering today.

Each variant is timed with CUDA events over `--reps` repetitions, the L2 flushed (256 MB written) before every one;
medians with min / max.  GB/s are against the bytes the kernel has to move (below), not a measured DRAM count.  Writes
profiles/handoff_probe.json with the card name and power limit read in the same run.

    python scripts/handoff_probe.py [--reps 30] [--out profiles/handoff_probe.json]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

JAC_READ, JAC_WRITE_IDX, JAC_WRITE = 840, 1848, 952      # bytes per interval: 105 SoA values; 7 rows x (16 values +
#                                                          16 indices + rhs) with indices, 7 x (16 + 1) doubles without
CT_COL, CT_SAT = 96, 6 * 8 + 32 * 8                     # bytes per node: x, u rows read, rbar / ubar written; per
#                                                          satellite: the terminal node read, 32 terms written


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "handoff_probe.json"))
    a = ap.parse_args()
    import torch
    import mpconstellation_b200 as M
    from conftest import synth_batch
    from oracle.mpc_oracle import OracleConstants
    M._lib.require_gpu()
    L = M._lib.lib()
    const = OracleConstants(*np.load(os.path.join(ROOT, "tests", "golden", "discretize.npz"))["const"])
    mu = float(const.MU)
    dev = torch.device("cuda")
    stream = torch.cuda.current_stream().cuda_stream
    flush = torch.empty(256 * 1024 * 1024 // 8, dtype=torch.float64, device=dev)   # 256 MB > 126 MB of L2

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

    def gbps(t, nbytes):
        return round(nbytes / (t["median_ms"] * 1e-3) / 1e9, 1)

    res = {"gpu": torch.cuda.get_device_name(0)}
    try:
        res["power_limit"] = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                                            capture_output=True, text=True).stdout.strip()
    except OSError:
        res["power_limit"] = "unknown"

    def ct_rect(xd, ud, N, K, rb, ub, fin):
        M._lib.check(L.mpc_constraint_terms(xd.data_ptr(), ud.data_ptr(), N, K, K, mu, rb.data_ptr(), ub.data_ptr(),
                                            fin.data_ptr(), stream))

    def ct_rag(xd, ud, K_sat, first, rb, ub, fin):
        N, Kmax = xd.shape[0], xd.shape[2]
        M._lib.check(L.mpc_constraint_terms_ragged(xd.data_ptr(), ud.data_ptr(), N, Kmax, K_sat.ctypes.data, first.data_ptr(),
                                                   mu, rb.data_ptr(), ub.data_ptr(), fin.data_ptr(), stream))

    def jac_rect(soa, pitch, off, N, K, v, c, r):
        M._lib.check(L.mpc_dynamics_jacobian(soa.data_ptr(), pitch, off, N, K, v, c, r, stream))

    def jac_rag(soa, N, Kmax, K_sat, first, v, c, r):
        M._lib.check(L.mpc_dynamics_jacobian_ragged(soa.data_ptr(), soa.shape[1], 0, N, Kmax, K_sat.ctypes.data,
                                                    first.data_ptr(), v, c, r, stream))

    # ---- config 3: 4096 x 200, all counts equal ----------------------------------------------------------------------
    N3, K3 = 4096, 200
    n3 = N3 * (K3 - 1)
    _, x3, u3 = synth_batch(N3, K3, 1.0, const)
    x3d, u3d = torch.as_tensor(x3).to(dev).contiguous(), torch.as_tensor(u3).to(dev).contiguous()
    Ks3 = np.full(N3, K3, np.int32)
    f3 = torch.empty(N3 + 1, dtype=torch.int64, device=dev)
    rb3 = torch.empty((N3, 3, K3 - 1), dtype=torch.float64, device=dev)
    ub3 = torch.empty((N3, 3, K3), dtype=torch.float64, device=dev)
    fn3 = torch.empty((N3, 32), dtype=torch.float64, device=dev)
    out3, st3 = M.discretize_batch_device(x3d, u3d, torch.ones(N3, dtype=torch.float64, device=dev), const)
    vals = torch.empty(7 * n3 * 16, dtype=torch.float64, device=dev)
    idx = torch.empty(7 * n3 * 16, dtype=torch.int64, device=dev)
    rhs = torch.empty(7 * n3, dtype=torch.float64, device=dev)
    c3 = {"n_sats": N3, "K": K3, "intervals": n3}
    ct_bytes = N3 * K3 * CT_COL + N3 * CT_SAT
    r = [timed(lambda: ct_rect(x3d, u3d, N3, K3, rb3, ub3, fn3)), timed(lambda: ct_rag(x3d, u3d, Ks3, f3, rb3, ub3, fn3)),
         timed(lambda: ct_rect(x3d, u3d, N3, K3, rb3, ub3, fn3)), timed(lambda: ct_rag(x3d, u3d, Ks3, f3, rb3, ub3, fn3))]
    c3["constraint_terms"] = {"bytes": ct_bytes, "rectangular": [r[0], r[2]], "ragged": [r[1], r[3]],
                              "GBps_rectangular": [gbps(r[0], ct_bytes), gbps(r[2], ct_bytes)],
                              "GBps_ragged": [gbps(r[1], ct_bytes), gbps(r[3], ct_bytes)]}
    for tag, ci, wb in (("jacobian_with_indices", idx.data_ptr(), JAC_WRITE_IDX), ("jacobian_values_only", None, JAC_WRITE)):
        nbytes = n3 * (JAC_READ + wb)
        rr = [timed(lambda: jac_rect(out3, n3, 0, N3, K3, vals.data_ptr(), ci, rhs.data_ptr())),
              timed(lambda: jac_rag(out3, N3, K3, Ks3, f3, vals.data_ptr(), ci, rhs.data_ptr())),
              timed(lambda: jac_rect(out3, n3, 0, N3, K3, vals.data_ptr(), ci, rhs.data_ptr())),
              timed(lambda: jac_rag(out3, N3, K3, Ks3, f3, vals.data_ptr(), ci, rhs.data_ptr()))]
        c3[tag] = {"bytes": nbytes, "floor_ms_at_7.7TBps": round(nbytes / 7.7e12 * 1e3, 4),
                   "rectangular": [rr[0], rr[2]], "ragged": [rr[1], rr[3]],
                   "GBps_rectangular": [gbps(rr[0], nbytes), gbps(rr[2], nbytes)],
                   "GBps_ragged": [gbps(rr[1], nbytes), gbps(rr[3], nbytes)]}
    res["config3_equal_counts"] = c3
    del out3, vals, idx, rhs

    # ---- config 5: 256 satellites, K_s = int(30 tf_s), tf_s over [1, 2] ---------------------------------------------
    N = 256
    tf = np.linspace(1.0, 2.0, N)
    K_sat = np.array([int(30 * t) for t in tf], dtype=np.int32)
    Kmax = int(K_sat.max())
    first_h = np.concatenate([[0], np.cumsum(K_sat.astype(np.int64) - 1)])
    n_live = int(first_h[-1])
    y0, _, _ = synth_batch(N, 2, 1.0, const)
    ctl = M.ConstantTangentialThrustController(tangential_thrust=0.5)
    x, u, _, _ = M.propagate_batch(y0, tf, ctl, const, include_drag=False, include_J2=False, T=K_sat)
    xd = torch.as_tensor(np.nan_to_num(np.array(x))).to(dev).contiguous()
    ud = torch.as_tensor(np.nan_to_num(np.array(u))).to(dev).contiguous()
    tfd = torch.as_tensor(tf).to(dev).contiguous()
    soa, _ = M.discretize_batch_device(xd, ud, tfd, const, adaptive=dict(rtol=1e-3, atol=1e-6, max_step=1e-2), K=K_sat)
    first = torch.empty(N + 1, dtype=torch.int64, device=dev)
    rb = torch.empty((N, 3, Kmax - 1), dtype=torch.float64, device=dev)
    ub = torch.empty((N, 3, Kmax), dtype=torch.float64, device=dev)
    fin = torch.empty((N, 32), dtype=torch.float64, device=dev)
    per_sat = [(xd[s:s + 1, :, :k].contiguous(), ud[s:s + 1, :, :k].contiguous(), int(k)) for s, k in enumerate(K_sat)]
    vals = torch.empty(7 * n_live * 16, dtype=torch.float64, device=dev)
    idx = torch.empty(7 * n_live * 16, dtype=torch.int64, device=dev)
    rhs = torch.empty(7 * n_live, dtype=torch.float64, device=dev)
    V, I, R = vals.data_ptr(), idx.data_ptr(), rhs.data_ptr()

    def ct_each():
        for s, (xs, us, k) in enumerate(per_sat):
            ct_rect(xs, us, 1, k, rb[s], ub[s], fin[s])

    def jac_each(ci):
        for s, k in enumerate(K_sat.tolist()):
            r0 = 7 * int(first_h[s])
            jac_rect(soa, soa.shape[1], s * (Kmax - 1), 1, k, V + r0 * 16 * 8, ci + r0 * 16 * 8 if ci else None, R + r0 * 8)

    c5 = {"n_sats": N, "K_range": [int(K_sat.min()), Kmax], "live_intervals": n_live}
    ct5 = int(K_sat.sum()) * CT_COL + N * CT_SAT
    r = [timed(lambda: ct_rag(xd, ud, K_sat, first, rb, ub, fin)), timed(ct_each),
         timed(lambda: ct_rag(xd, ud, K_sat, first, rb, ub, fin)), timed(ct_each)]
    c5["constraint_terms"] = {"bytes": ct5, "ragged_one_launch": [r[0], r[2]], "per_satellite_256_launches": [r[1], r[3]]}
    nb = n_live * (JAC_READ + JAC_WRITE_IDX)
    r = [timed(lambda: jac_rag(soa, N, Kmax, K_sat, first, V, I, R)), timed(lambda: jac_each(I)),
         timed(lambda: jac_rag(soa, N, Kmax, K_sat, first, V, I, R)), timed(lambda: jac_each(I))]
    c5["jacobian_with_indices"] = {"bytes": nb, "ragged_one_launch": [r[0], r[2]], "per_satellite_256_launches": [r[1], r[3]]}
    res["config5_ragged"] = c5
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
