"""What the altitude-dependent atmosphere costs on one GPU: the RK45 replay with drag under the constant density
(propagate_rk45_kernel / the per-satellite-units kernels) against the same flight under a fitted model
(propagate_rk45_atmo_kernel), alternated in one process.

  config 3   4096 satellites, T = 200, tangential law, drag + J2, one constants bag;
  config 5   the table-law flight of BatchedSCP.run_segments: 256 satellites, per-satellite tables [256,3,60], end_tau 2,
             T = 100, drag + J2;
  units      256 satellites of the mixed 400 ... 20,000 km constellation, each in its own constants, tangential law.

The model is the exponential atmosphere rho0 exp(-(h - h0) / H) fitted over 200 ... 40,000 km (22 terms), and for
config 3 also the power law of simulator.py:110 over 300 ... 1,000 km (2 terms) on near-circular orbits.  CUDA events
around one propagate_batch_device call, warm-up first, medians (min / max) over --reps runs per variant.  The working
set is a few MB and the kernels are latency-bound chains of dependent stages, so the L2 is not flushed.  Writes
profiles/atmo_probe.json with the card name and power limit read in the same run.

    python scripts/atmo_probe.py [--reps 25] [--out profiles/atmo_probe.json]
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
    ap.add_argument("--reps", type=int, default=25)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "atmo_probe.json"))
    a = ap.parse_args()
    import torch
    import mpconstellation_b200 as M
    from mpconstellation_b200 import _lib
    from units_probe import mixed_constellation
    _lib.require_gpu()
    dev = torch.device("cuda")
    expo = M.fit_atmosphere(lambda h: 3.7e-12 * np.exp(-(h - 400e3) / 58e3), 200e3, 40000e3)
    plaw = M.fit_atmosphere(lambda h: 8e26 * h ** -6.828, 300e3, 1000e3)

    def timed(fn):
        fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1)

    def compare(name, variants, check):
        t = {k: [] for k in variants}
        for k, fn in variants.items():     # warm-up of every shape
            fn()
        for _ in range(a.reps):
            for k, fn in variants.items():
                t[k].append(timed(fn))
        out = {k: {"median_ms": float(np.median(v)), "min_ms": float(np.min(v)), "max_ms": float(np.max(v))} for k, v in t.items()}
        base = out["constant"]["median_ms"]
        for k in out:
            out[k]["vs_constant"] = out[k]["median_ms"] / base
        out["status_max"] = check()
        print(name, json.dumps(out))
        return out

    res = {"reps": a.reps, "models": {"exponential": {"range_m": [200e3, 40000e3], "terms": len(expo.coef)},
                                      "power_law": {"range_m": [300e3, 1000e3], "terms": len(plaw.coef)}}}
    # config 3: Hubble's state rotated about z, speed scaled by 1 + 0.1 U[0,1) (SURVEY.md section 8(d)); the power law
    # on the same satellites with speeds within 0.5 % of circular, so that they stay inside its 300 ... 1,000 km
    hubble = np.array([5371.4806e3, -4133.1393e3, 1399.9594e3, 4.6921e3, 4.9848e3, -3.2752e3, 12200.0])
    scale = M.SatelliteScale(x=hubble)
    const = scale.get_normalized_constants()
    N3, T3 = 4096, 200

    def constellation(spread):
        y0 = np.tile(scale.normalize_state(hubble), (N3, 1))
        ang = 2 * np.pi * np.arange(N3) / N3
        ca, sa = np.cos(ang), np.sin(ang)
        for i in (0, 3):
            x, y = y0[:, i].copy(), y0[:, i + 1].copy()
            y0[:, i], y0[:, i + 1] = ca * x - sa * y, sa * x + ca * y
        y0[:, 3:6] *= (1 + spread * np.random.default_rng(1).random(N3))[:, None]
        return torch.as_tensor(y0, device=dev)
    y3, y3c = constellation(0.1), constellation(0.005)
    tf3 = torch.full((N3,), 1.0, dtype=torch.float64, device=dev)
    ctrl = M.ConstantTangentialThrustController(tangential_thrust=0.05)
    buf = [torch.empty((N3, 7, T3), dtype=torch.float64, device=dev), torch.empty((N3, 3, T3), dtype=torch.float64, device=dev),
           torch.empty(N3, dtype=torch.int32, device=dev)]

    def prop3(y0, atmo):
        return lambda: M.propagate_batch_device(y0, tf3, ctrl, const, T=T3, y=buf[0], u_out=buf[1], status=buf[2], atmosphere=atmo)

    def st3():
        return int(buf[2].max())
    res["config3"] = compare("config3", {"constant": prop3(y3, None), "exponential": prop3(y3, expo)}, st3)
    res["config3_circular"] = compare("config3_circular", {"constant": prop3(y3c, None), "power_law": prop3(y3c, plaw),
                                                           "exponential": prop3(y3c, expo)}, st3)
    # config 5's table-law flight
    N5, T5 = 256, 100
    y5 = y3[:: N3 // N5].contiguous()
    tf5 = torch.full((N5,), 1.0, dtype=torch.float64, device=dev)
    spec5 = M.ControllerSpec(_lib.CTRL_SEQUENCE, (0.0, 0.0, 0.0), 0.05 * np.random.default_rng(5).standard_normal((N5, 3, 60)),
                             2.0)
    st5 = torch.empty(N5, dtype=torch.int32, device=dev)

    def prop5(atmo):
        return lambda: M.propagate_batch_device(y5, tf5, spec5, const, T=T5, status=st5, atmosphere=atmo)
    res["config5_flight"] = compare("config5_flight", {"constant": prop5(None), "exponential": prop5(expo)},
                                    lambda: int(st5.max()))
    # the mixed-units constellation
    yu, consts = mixed_constellation(256)
    yud = torch.as_tensor(yu, device=dev)
    tfu = torch.full((256,), 0.5, dtype=torch.float64, device=dev)
    stu = torch.empty(256, dtype=torch.int32, device=dev)

    def propu(atmo):
        return lambda: M.propagate_batch_device(yud, tfu, ctrl, consts, T=60, status=stu, atmosphere=atmo)
    res["units_256"] = compare("units_256", {"constant": propu(None), "exponential": propu(expo)}, lambda: int(stu.max()))
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    res["gpu"] = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name()
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
