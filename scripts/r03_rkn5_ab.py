"""Same-process A/B of the 11-node form of the 101-node sums on fifth-order steps (kEmW3, mpc_set_tuning(40)) against the
21-node form it replaces on the benchmark's intervals (mpc_set_tuning(39)), at bench.py's default workload: 4096 satellites
x K = 200, tf = 2, n_sub = 100, the RK45 propagator.

Times, alternating the two settings, each repetition after a 256 MiB L2 flush (CUDA events):
  * discretize_batch_device alone, on the propagated x, u
  * propagate_discretize_device (the overlapped pass bench.py times), library default windows
and then, with the tier on, the overlapped pass for several window counts.  Prints the median and the spread (min..max)
of each, the card's name and power limit, and compares the outputs of the two settings in the layout of
bench.py --dump-outputs (written under DIR/on and DIR/off): x, u and both status arrays bit-identical, A_k rows to 2e-11,
the other row groups to 1e-12, norm-relative.

usage: python scripts/r03_rkn5_ab.py [--reps 15] [--out DIR]   (default DIR: r03_rkn5_ab in the temporary directory)"""
import argparse
import json
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import torch

import mpconstellation_b200 as M
from bench import dump_outputs, make_constellation


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as exc:       # no nvidia-smi: the name from the runtime only
        q = f"{name}, power limit unknown ({exc})"
    return q


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=15)
    ap.add_argument("--out", default=os.path.join(tempfile.gettempdir(), "r03_rkn5_ab"))
    ap.add_argument("--windows", default="4,8,12,16,24,32", help="window counts of the sweep (tier on)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    N, K, tf, n_sub = 4096, 200, 2.0, 100
    dev = torch.device("cuda:0")
    L = M._lib.lib()
    Y, const = make_constellation(N)
    ctrl = M.ConstantTangentialThrustController(tangential_thrust=0.5)
    y0 = torch.from_numpy(Y).to(dev)
    tfd = torch.full((N,), tf, dtype=torch.float64, device=dev)
    x = torch.empty((N, 7, K), dtype=torch.float64, device=dev)
    u = torch.empty((N, 3, K), dtype=torch.float64, device=dev)
    out = torch.empty((105, N * (K - 1)), dtype=torch.float64, device=dev)
    sp = torch.empty(N, dtype=torch.int32, device=dev)
    sd = torch.empty(N * (K - 1), dtype=torch.int32, device=dev)
    flush = torch.empty(256 * 1024 * 1024 // 8, dtype=torch.float64, device=dev)

    def disc():
        M.discretize_batch_device(x, u, tfd, const, n_sub=n_sub, out=out, status=sd)

    def pass_(nw=0):
        M.propagate_discretize_device(y0, tfd, ctrl, const, K, n_sub_prop=0, n_sub_disc=n_sub, y=x, u_out=u, out=out,
                                      status_prop=sp, status_disc=sd, n_windows=nw)

    def once(fn):
        flush.fill_(1.0)
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b)

    def tier(on):
        assert L.mpc_set_tuning(40 if on else 39) == 0

    res = {"card": card(), "workload": dict(n_sats=N, K=K, tf=tf, n_sub=n_sub, propagator="rk45"), "reps": args.reps}
    # outputs of the two settings, dumped as bench.py --dump-outputs does
    for on in (False, True):
        tier(on)
        for _ in range(3):
            pass_()
        torch.cuda.synchronize()
        assert int(sp.max()) == 0 and int(sd.max()) == 0
        dump_outputs(os.path.join(args.out, "on" if on else "off"), out, x, u, sp, sd)
    d = {t: {n: np.load(os.path.join(args.out, t, n + ".npy")) for n in ("out", "x", "u", "status_prop", "status_disc")}
         for t in ("on", "off")}

    def rel(a, b):
        return float(np.max(np.abs(a - b)) / np.max(np.abs(b)))
    cmp = {n: bool(np.array_equal(d["on"][n], d["off"][n])) for n in ("x", "u", "status_prop", "status_disc")}
    groups = {"A_k": (0, 49), "B_kp": (49, 70), "B_kn": (70, 91), "Sigma_k": (91, 98), "xi_k": (98, 105)}
    cmp.update({g: rel(d["on"]["out"][r0:r1], d["off"]["out"][r0:r1]) for g, (r0, r1) in groups.items()})
    ok = all(cmp[n] for n in ("x", "u", "status_prop", "status_disc")) and cmp["A_k"] <= 2e-11 and \
        all(cmp[g] <= 1e-12 for g in groups if g != "A_k")
    res["outputs_on_vs_off"] = cmp
    res["outputs_ok"] = ok

    # alternating timings
    t = {("disc", True): [], ("disc", False): [], ("pass", True): [], ("pass", False): []}
    for on in (True, False):
        tier(on)
        for _ in range(3):
            once(disc)
            once(pass_)
    for _ in range(args.reps):
        for on in (True, False):
            tier(on)
            t[("disc", on)].append(once(disc))
            t[("pass", on)].append(once(pass_))

    def stat(v):
        v = np.asarray(v)
        return {"median_ms": round(float(np.median(v)), 4), "min_ms": round(float(v.min()), 4),
                "max_ms": round(float(v.max()), 4)}
    res["timing"] = {f"{k}_{'on' if on else 'off'}": stat(v) for (k, on), v in t.items()}
    for k in ("disc", "pass"):
        on, off = np.median(t[(k, True)]), np.median(t[(k, False)])
        res["timing"][f"{k}_gain_pct"] = round(100.0 * (off - on) / off, 2)

    # the overlapped pass with the tier on, for several window counts (0 = library default)
    tier(True)
    once(disc)                       # the reference: the back-to-back sequence with the tier on
    ref = out.clone()
    sweep = {}
    for nw in [0] + [int(a) for a in args.windows.split(",") if a]:
        for _ in range(2):
            once(lambda: pass_(nw))
        v = [once(lambda: pass_(nw)) for _ in range(args.reps)]
        sweep[str(nw)] = dict(stat(v), identical=bool(torch.equal(out, ref)))
    res["windows_sweep_tier_on"] = sweep
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "result.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))
    if not ok:
        raise SystemExit("outputs of the two settings differ beyond the bounds")


if __name__ == "__main__":
    main()
