"""Cost of the conjunction screening on one GPU (screen_conjunctions_device / mpc_screen_conjunctions).

  config 3's shape: 4096 satellites x 200 samples; config 5's shape: 256 x 60.  Each is a shell at ~550 km (16 planes at
  53 degrees, random phases, the radius spread by 0.1 %), flown for one orbit with J2 by propagate_batch_device, and
  screened at thresholds of 1, 10 and 100 km.

Per case: the kernels alone (mpc_screen_conjunctions, CUDA events around the two launches) and the whole device call
(screen_conjunctions_device: the launches, the count read back and the sort), warmed, medians with min / max over
`--reps`; pair-intervals per second of the kernels; the fraction of pair-intervals that pass the sphere prefilter
(counted afterwards from the spheres the pre-pass left in the scratch); the event count.  Writes the JSON with the card
name and power limit read in the same run.

    python scripts/conjunction_probe.py [--reps 20] [--out profiles/conjunction_probe.json]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def shell_states(N, seed, a=6.921e6, inc=np.radians(53.0), planes=16):
    from mpconstellation_b200.model import MU_EARTH
    rng = np.random.default_rng(seed)
    out = np.empty((N, 7))
    for s in range(N):
        r = a * (1 + 1e-3 * rng.standard_normal())
        raan, u = 2 * np.pi * (s % planes) / planes, rng.uniform(0, 2 * np.pi)
        nv = np.array([np.cos(raan), np.sin(raan), 0.0])
        wv = np.array([-np.sin(raan) * np.cos(inc), np.cos(raan) * np.cos(inc), np.sin(inc)])
        v = np.sqrt(MU_EARTH / r)
        out[s] = np.concatenate([r * (np.cos(u) * nv + np.sin(u) * wv), v * (-np.sin(u) * nv + np.cos(u) * wv), [500.0]])
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "conjunction_probe.json"))
    a = ap.parse_args()
    import torch
    import mpconstellation_b200 as M
    from mpconstellation_b200 import _lib
    _lib.require_gpu()
    dev = torch.device("cuda")
    L = _lib.lib()

    def case(N, T, seed):
        st = shell_states(N, seed)
        sc = M.SatelliteScale(x=st[0])
        const = sc.get_normalized_constants()
        y0 = torch.as_tensor(np.array([sc.normalize_state(x) for x in st])).to(dev)
        tf = torch.full((N,), 1.0, dtype=torch.float64, device=dev)             # one period of the scale orbit
        ctrl = M.ConstantTangentialThrustController(tangential_thrust=0.0)
        y, _, status = M.propagate_batch_device(y0, tf, ctrl, const, include_drag=False, include_J2=True, T=T)
        torch.cuda.synchronize()
        assert int(status.max()) == 0
        scale, D = M.conjunctions.screen_scales(tuple(y.shape), 1.0, const, 1.0)
        out = {}
        for thr_km in (1, 10, 100):
            thr = thr_km * 1e3
            res = M.screen_conjunctions_device(y, 1.0, const, thr)
            cap = max(len(res), 1)
            scratch = torch.empty(int(L.mpc_conjunction_scratch_doubles(N, T)), dtype=torch.float64, device=dev)
            ev = torch.empty((cap, 5), dtype=torch.float64, device=dev)
            cnt = torch.zeros(2, dtype=torch.int64, device=dev)
            sk = torch.empty(N, dtype=torch.int32, device=dev)
            stream = torch.cuda.current_stream(dev).cuda_stream

            def kernels():
                _lib.check(L.mpc_screen_conjunctions(y.data_ptr(), N, T, _lib.addr(scale), D, thr, scratch.data_ptr(),
                                                     ev.data_ptr(), cap, cnt.data_ptr(), sk.data_ptr(), stream))

            def call():
                M.screen_conjunctions_device(y, 1.0, const, thr, capacity=cap)
            r = {}
            for name, fn in (("kernels", kernels), ("device_call", call)):
                for _ in range(3):
                    fn()
                torch.cuda.synchronize()
                ts = []
                for _ in range(a.reps):
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    fn()
                    e1.record()
                    torch.cuda.synchronize()
                    ts.append(e0.elapsed_time(e1))
                r[name] = {"median_ms": float(np.median(ts)), "min_ms": float(np.min(ts)), "max_ms": float(np.max(ts))}
            assert int(cnt[0]) == len(res)
            # the prefilter's pass count, from the spheres S [T-1][4][N] in the scratch
            S = scratch[N * 6 * T: N * 6 * T + N * 4 * (T - 1)].view(T - 1, 4, N)
            passed = 0
            iu = torch.triu_indices(N, N, 1, device=dev)
            for k in range(T - 1):
                c = S[k, 0:3].T
                rho = S[k, 3]
                dist = torch.cdist(c, c)
                ok = dist <= rho[:, None] + rho[None, :] + thr
                passed += int(ok[iu[0], iu[1]].sum())
            n_pi = N * (N - 1) // 2 * (T - 1)
            r.update({"pair_intervals": n_pi, "pair_intervals_per_s": n_pi / (r["kernels"]["median_ms"] * 1e-3),
                      "prefilter_pass_fraction": passed / n_pi, "events": len(res), "flagged": res.n_flagged})
            out[f"{thr_km}km"] = r
            print(N, T, thr_km, json.dumps(r), flush=True)
        return out

    result = {"config3_4096x200": case(4096, 200, 3), "config5_256x60": case(256, 60, 5)}
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True).stdout.strip()
    result["gpu"] = q
    result["reps"] = a.reps
    result["timing"] = ("CUDA events, warmed (3 calls), medians over reps; kernels = mpc_screen_conjunctions (pre-pass + "
                        "pair kernel); device_call = screen_conjunctions_device (launches, count read-back, sort)")
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result, indent=1))


if __name__ == "__main__":
    main()
