"""Sharded linearization of ragged / per-satellite-units batches (RaggedGather) over the GPUs of one box.

    torchrun --nproc_per_node W scripts/shard_probe.py [--reps 10] [--out profiles/shard_probe.json]

Batches (every satellite in the designer units of its own SatelliteScale, model.sat_units):
  mixed4096  4096 satellites, tf_s spread over [1, 2] (seeded), base_res = 100: K_s = int(100 tf_s) in [100, 200], K_cap 200
  config5    config 5's shape: 256 satellites, tf = 2, base_res = 30: K = 60 everywhere
Both quadrature modes (default: the reference's RK45 node set; fixed: use_uniform_steps, 101 integrator steps).  Per
batch and mode:
  step_ms      RaggedGather.linearize (propagate shard, fused-store discretization, x_bar / u_bar copies, barriers, status
               combine), CUDA events on every rank, the L2 flushed (256 MB written) before each repetition; the median
               of rank 0 and the slowest rank's median
  disc_ms      the discretization kernel of every rank alone (events around its launch inside the same steps): the load
               imbalance of shard_ranges_by_work
  single_ms    the single-GPU ragged / units calls on the whole batch (propagate_batch_device + discretize_batch_device),
               same timing, on rank 0 while the others wait
  check        every rank's gathered matrices, x_bar and u_bar bit-identical on the live columns to the single-GPU result
With all counts and constants equal (fixed step; mixed4096 -> 4096 x 200, config5 -> 256 x 60, constants of satellite 0):
  rect_ragged_ms  RaggedGather.linearize;  rect_fused_ms  the rectangular FusedGather (satellite-major, unicast), shard
                  propagated then discretized back to back (propagate_batch_device + FusedGather.discretize).
Rank 0 writes the JSON with the card name and power limit read in the same run.
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


def batches():
    from units_probe import mixed_constellation
    rng = np.random.default_rng(7)
    y4, c4 = mixed_constellation(4096)
    tf4 = rng.uniform(1.0, 2.0, 4096)
    y5, c5 = mixed_constellation(256)
    return {"mixed4096": (y4, c4, tf4, 100, 200), "config5": (y5, c5, np.full(256, 2.0), 30, 60)}


def single_gpu(y0, tf, ctrl, const, K_sat, uniform, include_J2=False):
    """the single-GPU ragged / units calls of BatchedSCP.linearize, device-resident: (soa, x, u)"""
    import torch
    from mpconstellation_b200 import batch
    dev = torch.device("cuda")
    y0t = torch.as_tensor(y0, dtype=torch.float64, device=dev)
    tft = torch.as_tensor(tf, dtype=torch.float64, device=dev)
    x, u, _ = batch.propagate_batch_device(y0t, tft, ctrl, const, include_drag=False, include_J2=False, T=K_sat)
    out, _ = batch.discretize_batch_device(x, u, tft, const, include_J2=include_J2, n_sub=100, K=K_sat,
                                           adaptive=None if uniform else dict(rtol=1e-3, atol=1e-6, max_step=1e-2))
    return out, x, u


def live_columns(K_sat, K):
    import torch
    k = torch.as_tensor(K_sat, dtype=torch.int64)
    s = torch.repeat_interleave(torch.arange(len(K_sat)), k - 1)
    off = torch.repeat_interleave(torch.cumsum(k - 1, 0) - (k - 1), k - 1)
    return s * (K - 1) + torch.arange(int((k - 1).sum())) - off


def same_as_single(res, ref, K_sat):
    """bit-identical live columns of the matrices and live samples of x_bar / u_bar"""
    import torch
    soa, x, u = ref
    dev = soa.device
    Kc, Km = res.x_bar.shape[2], x.shape[2]
    ok = torch.equal(res.soa[:, live_columns(K_sat, Kc).to(dev)], soa[:, live_columns(K_sat, Km).to(dev)])
    mask = torch.arange(Km, device=dev)[None, :] < torch.as_tensor(K_sat, device=dev)[:, None]
    for a, b in ((res.x_bar, x), (res.u_bar, u)):
        ok &= torch.equal(a[:, :, :Km].transpose(1, 2)[mask], b.transpose(1, 2)[mask])
    return bool(ok)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "shard_probe.json"))
    a = ap.parse_args()
    import torch
    import torch.distributed as dist
    from mpconstellation_b200 import ConstantTangentialThrustController, _lib, batch
    from mpconstellation_b200.distributed import FusedGather, RaggedGather
    from mpconstellation_b200.scp import node_counts
    _lib.require_gpu()
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", 0)))
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", torch.cuda.current_device()))
    dev = torch.device("cuda", torch.cuda.current_device())
    flush = torch.empty(256 * 1024 * 1024 // 8, dtype=torch.float64, device=dev)
    ctrl = ConstantTangentialThrustController(tangential_thrust=0.5)
    L = _lib.lib()
    launch = L.mpc_discretize_batch_ragged_gather
    disc_events = []

    def timed_launch(*args):          # events around this rank's discretization kernel
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        rc = launch(*args)
        e1.record()
        disc_events.append((e0, e1))
        return rc
    L.mpc_discretize_batch_ragged_gather = timed_launch

    def timed(fn, reps=a.reps):
        fn()
        torch.cuda.synchronize()
        dist.barrier()
        ts = []
        disc_events.clear()
        for _ in range(reps):
            flush.fill_(1.0)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1))
        disc = [b.elapsed_time(c) for b, c in disc_events]
        return float(np.median(ts)), (float(np.median(disc)) if disc else 0.0)

    def over_ranks(v):
        t = torch.tensor([float(v)], dtype=torch.float64, device=dev)
        out = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(out, t)
        return [float(o.item()) for o in out]

    res = {"world": world, "reps": a.reps, "batches": {}}
    for name, (y0, consts, tf, base_res, K_cap) in batches().items():
        K_sat = node_counts(base_res, tf)
        N = len(K_sat)
        g = RaggedGather(N, K_cap)
        entry = {"n_sats": N, "K_cap": K_cap, "live_intervals": int((K_sat - 1).sum())}
        for mode, uniform in (("default", False), ("fixed", True)):
            step, disc = timed(lambda: g.linearize(y0, tf, ctrl, consts, K_sat, use_uniform_steps=uniform))
            out = g.linearize(y0, tf, ctrl, consts, K_sat, use_uniform_steps=uniform)
            ref = single_gpu(y0, tf, ctrl, consts, K_sat, uniform)
            torch.cuda.synchronize()
            ok = all(over_ranks(same_as_single(out, ref, K_sat)))
            del ref
            single = None
            dist.barrier()
            if rank == 0:
                ts = []
                single_gpu(y0, tf, ctrl, consts, K_sat, uniform)
                torch.cuda.synchronize()
                for _ in range(a.reps):
                    flush.fill_(1.0)
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    single_gpu(y0, tf, ctrl, consts, K_sat, uniform)
                    e1.record()
                    torch.cuda.synchronize()
                    ts.append(e0.elapsed_time(e1))
                single = float(np.median(ts))
            dist.barrier()
            steps = over_ranks(step)
            entry[mode] = {"step_ms_rank0": steps[0], "step_ms_slowest_rank": max(steps), "disc_ms_per_rank": over_ranks(disc),
                           "live_intervals_per_rank": [int((K_sat[s0:s1] - 1).sum()) for s0, s1 in out.ranges],
                           "single_gpu_ms": single, "check_bit_identical": ok}
        # all counts and constants equal, fixed step: RaggedGather against the rectangular FusedGather, back to back
        Ke = np.full(N, K_cap, np.int32)
        tfe = np.full(N, K_cap / base_res)
        one = consts[0]
        fg = FusedGather(N, K_cap, layout="satmajor")
        yt = torch.as_tensor(y0, dtype=torch.float64, device=dev)
        tft = torch.as_tensor(tfe, dtype=torch.float64, device=dev)

        def fused():
            y, u, st = batch.propagate_batch_device(yt[fg.s0:fg.s1], tft[fg.s0:fg.s1], ctrl, one, include_drag=False,
                                                    include_J2=False, T=K_cap)
            fg.discretize(y, u, tft[fg.s0:fg.s1], one)
        rect_ragged, _ = timed(lambda: g.linearize(y0, tfe, ctrl, one, Ke, use_uniform_steps=True))
        rect_fused, _ = timed(fused)
        entry["equal_counts_and_constants_fixed"] = {"ragged_gather_step_ms_slowest_rank": max(over_ranks(rect_ragged)),
                                                     "fused_gather_step_ms_slowest_rank": max(over_ranks(rect_fused))}
        res["batches"][name] = entry
        del g, fg
        torch.cuda.empty_cache()
    if rank == 0:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True).stdout.strip().splitlines()
        res["gpus"] = q[:world]
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        json.dump(res, open(a.out, "w"), indent=1)
        print(json.dumps(res))
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
