"""GPU, 2 ranks (NCCL): RaggedGather on a mixed constellation -- 4096 satellites in their own units with horizons spread
over [1, 2] (K_s = int(100 tf_s)), and config 5's shape (256 x 60, own units) -- in both quadrature modes.  Every rank's
gathered matrices and reference trajectories must be bit-identical on the live columns to the single-GPU ragged / units
calls on the whole batch, the subproblem hand-off run on rank 0 over the gathered buffers bit-identical to the
single-GPU hand-off, and a zero-mass satellite on rank 1 must raise the reference's Exception on both ranks."""
import os
import socket
import sys

import numpy as np
import pytest

from conftest import ROOT

pytestmark = pytest.mark.gpu
sys.path.insert(0, os.path.join(ROOT, "scripts"))


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, tmp):
    import torch
    import torch.distributed as dist
    import shard_probe as P
    from mpconstellation_b200 import ConstantTangentialThrustController
    from mpconstellation_b200.constraints import constraint_terms_device, dynamics_jacobian_device
    from mpconstellation_b200.distributed import RaggedGather
    from mpconstellation_b200.scp import node_counts
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    out = {}
    try:
        ctrl = ConstantTangentialThrustController(tangential_thrust=0.5)
        for name, (y0, consts, tf, base_res, K_cap) in P.batches().items():
            K_sat = node_counts(base_res, tf)
            g = RaggedGather(len(K_sat), K_cap)
            for uniform in (False, True):
                res = g.linearize(y0, tf, ctrl, consts, K_sat, use_uniform_steps=uniform)
                ref = P.single_gpu(y0, tf, ctrl, consts, K_sat, uniform)
                key = f"{name}_{'fixed' if uniform else 'default'}"
                out[key] = P.same_as_single(res, ref, K_sat)
                if rank == 0:
                    N, Km = len(K_sat), ref[1].shape[2]
                    a = constraint_terms_device(res.x_bar, res.u_bar, consts, K=K_sat)
                    b = constraint_terms_device(ref[1], ref[2], consts, K=K_sat)
                    mask = torch.arange(Km, device=ref[1].device)[None, :] < torch.as_tensor(K_sat, device=ref[1].device)[:, None]
                    ok = torch.equal(a[0][:, :, :Km - 1].transpose(1, 2)[mask[:, 1:]], b[0].transpose(1, 2)[mask[:, 1:]])
                    ok &= torch.equal(a[1][:, :, :Km].transpose(1, 2)[mask], b[1].transpose(1, 2)[mask])
                    ok &= torch.equal(a[2], b[2])
                    ja = dynamics_jacobian_device(res.soa, N, K_cap, K_sat=K_sat)
                    jb = dynamics_jacobian_device(ref[0], N, Km, K_sat=K_sat)
                    ok &= all(torch.equal(p, q) for p, q in zip(ja, jb))
                    out[key + "_handoff"] = bool(ok)
                torch.cuda.synchronize()
            # a zero-mass satellite of rank 1's range
            s_bad = g.linearize(y0, tf, ctrl, consts, K_sat).ranges[1][0]
            y_bad = np.array(y0)
            y_bad[s_bad, 6] = 0.0
            try:
                g.linearize(y_bad, tf, ctrl, consts, K_sat)
                out[name + "_zero_mass"] = "no exception"
            except Exception as e:     # noqa: BLE001 -- the reference raises a plain Exception
                out[name + "_zero_mass"] = f"{type(e).__name__}: {e}"
            del g
        np.save(os.path.join(tmp, f"rank{rank}.npy"), out, allow_pickle=True)
    finally:
        dist.barrier()
        dist.destroy_process_group()


def test_ragged_gather_two_ranks_match_single_gpu(tmp_path):
    import torch
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    ctx = mp.start_processes(_worker, args=(2, _free_port(), str(tmp_path)), nprocs=2, join=False, start_method="spawn")
    try:
        for _ in range(600):               # 10 minutes at most
            if ctx.join(timeout=1):
                break
        else:
            pytest.fail("the ranks did not finish within 10 minutes")
    finally:
        for p in ctx.processes:
            if p.is_alive():
                p.kill()
                p.join()
    for rank in (0, 1):
        got = np.load(tmp_path / f"rank{rank}.npy", allow_pickle=True).item()
        for key, v in got.items():
            if key.endswith("_zero_mass"):
                assert v.startswith("Exception: ERROR: INVALID SATELLITE MASS"), (rank, key, v)
            else:
                assert v is True, (rank, key)
        assert sum(k.endswith("_handoff") for k in got) == (4 if rank == 0 else 0)


def _shard_launch(x, u, tf, consts, K_sat, s0, s1, dst, pitch, adaptive, skip_const):
    """one rank's launch of mpc_discretize_batch_ragged_gather: satellites [s0, s1) of x / u [N, ., K_cap] into dst"""
    import ctypes
    import torch
    from mpconstellation_b200 import _lib, batch
    n, K_cap = s1 - s0, x.shape[2]
    psc, one = batch._units_of(consts[s0:s1], n)
    p = _lib.make_params(one, False, False)
    status = torch.zeros(n * (K_cap - 1), dtype=torch.int32, device=x.device)
    first = torch.empty(n + 1, dtype=torch.int64, device=x.device)
    scratch = torch.empty(n * _lib.SAT_SCRATCH_DOUBLES, dtype=torch.float64, device=x.device)
    arr = (ctypes.c_void_p * len(dst))(*[d.data_ptr() for d in dst])
    _lib.check(_lib.lib().mpc_discretize_batch_ragged_gather(
        x[s0:s1].data_ptr(), u[s0:s1].data_ptr(), tf[s0:s1].data_ptr(), ctypes.byref(p), psc, n, K_cap,
        _lib.addr(np.ascontiguousarray(K_sat[s0:s1])), first.data_ptr(), scratch.data_ptr() if psc is not None else None,
        int(adaptive), 100, 1e-3, 1e-6, 1e-2, arr, len(dst), pitch, s0 * (K_cap - 1), skip_const, status.data_ptr(), None,
        torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    return status


@pytest.mark.parametrize("n_dst", [2, 4, 8])
@pytest.mark.parametrize("adaptive", [False, True])
def test_multi_destination_shards_on_one_gpu(n_dst, adaptive):
    """the NDST = 2 / 4 / 8 kernels on one B200, local buffers standing in for the peers: n_dst shards of the mixed
    constellation (per-satellite constants) each store into all n_dst buffers; every buffer must equal the single-GPU
    units call on the live columns, rows 42..48 left to the fill (skip_const 1) in all but the own buffer"""
    import torch
    import shard_probe as P
    from mpconstellation_b200 import ConstantTangentialThrustController, _lib, batch
    from mpconstellation_b200.distributed import shard_ranges_by_work
    from mpconstellation_b200.scp import node_counts
    y0, consts, tf, base_res, K_cap = P.batches()["mixed4096"]
    N = 1024                                   # the first 1024 satellites: every altitude / mass of the mix
    y0, consts, tf = y0[:N], consts[:N], tf[:N]
    K_sat = node_counts(base_res, tf)
    ctrl = ConstantTangentialThrustController(tangential_thrust=0.5)
    ref, x, u = P.single_gpu(y0, tf, ctrl, consts, K_sat, not adaptive)
    dev = x.device
    xc = torch.full((N, 7, K_cap), float("nan"), dtype=torch.float64, device=dev)
    uc = torch.full((N, 3, K_cap), float("nan"), dtype=torch.float64, device=dev)
    xc[:, :, :x.shape[2]], uc[:, :, :u.shape[2]] = x, u
    tft = torch.as_tensor(tf, dtype=torch.float64, device=dev)
    pitch = N * (K_cap - 1)
    bufs = [torch.full((105, pitch), float("nan"), dtype=torch.float64, device=dev) for _ in range(n_dst)]
    for b in bufs:
        _lib.check(_lib.lib().mpc_fill_const_rows(b.data_ptr(), pitch, torch.cuda.current_stream().cuda_stream))
    ranges = shard_ranges_by_work(K_sat, n_dst)
    for r, (s0, s1) in enumerate(ranges):
        if s1 > s0:
            st = _shard_launch(xc, uc, tft, consts, K_sat, s0, s1, [bufs[(r + i) % n_dst] for i in range(n_dst)], pitch,
                               adaptive, 1)
            assert int(st.max()) == 0
    cols_g = P.live_columns(K_sat, K_cap).to(dev)
    cols_r = P.live_columns(K_sat, x.shape[2]).to(dev)
    pad = torch.ones(pitch, dtype=torch.bool, device=dev)
    pad[cols_g] = False
    for b in bufs:
        assert torch.equal(b[:, cols_g], ref[:, cols_r])
        assert torch.isnan(b[:42][:, pad]).all() and torch.isnan(b[49:][:, pad]).all()
    # one bag for all: the single-constant multi-destination kernels
    one = [consts[0]] * N
    ref1, _ = batch.discretize_batch_device(xc, uc, tft, consts[0], n_sub=100, K=K_sat,
                                            adaptive=dict(rtol=1e-3, atol=1e-6, max_step=1e-2) if adaptive else None)
    bufs = [torch.full((105, pitch), float("nan"), dtype=torch.float64, device=dev) for _ in range(n_dst)]
    for r, (s0, s1) in enumerate(ranges):
        if s1 > s0:
            _shard_launch(xc, uc, tft, one, K_sat, s0, s1, [bufs[(r + i) % n_dst] for i in range(n_dst)], pitch, adaptive, 0)
    for b in bufs:
        assert torch.equal(b[:, cols_g], ref1[:, cols_g])


def _worker_world1(rank, port, tmp):
    import torch
    import torch.distributed as dist
    import shard_probe as P
    from mpconstellation_b200 import ConstantTangentialThrustController
    from mpconstellation_b200.distributed import RaggedGather
    from mpconstellation_b200.scp import node_counts
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(0)
    dist.init_process_group("nccl", rank=0, world_size=1, device_id=torch.device("cuda", 0))
    try:
        y0, consts, tf, base_res, K_cap = P.batches()["config5"]
        K_sat = node_counts(base_res, tf)
        ctrl = ConstantTangentialThrustController(tangential_thrust=0.5)
        g = RaggedGather(len(K_sat), K_cap)
        out = {}
        for uniform in (False, True):
            res = g.linearize(y0, tf, ctrl, consts, K_sat, use_uniform_steps=uniform)
            out[uniform] = P.same_as_single(res, P.single_gpu(y0, tf, ctrl, consts, K_sat, uniform), K_sat)
        y_bad = np.array(y0)
        y_bad[3, 6] = 0.0
        try:
            g.linearize(y_bad, tf, ctrl, consts, K_sat)
            out["zero_mass"] = "no exception"
        except Exception as e:     # noqa: BLE001
            out["zero_mass"] = f"{type(e).__name__}: {e}"
        np.save(os.path.join(tmp, "world1.npy"), out, allow_pickle=True)
    finally:
        dist.destroy_process_group()


def test_ragged_gather_world1_runs_the_single_gpu_calls(tmp_path):
    import torch.multiprocessing as mp
    ctx = mp.start_processes(_worker_world1, args=(_free_port(), str(tmp_path)), nprocs=1, join=False, start_method="spawn")
    try:
        for _ in range(300):
            if ctx.join(timeout=1):
                break
        else:
            pytest.fail("the rank did not finish within 5 minutes")
    finally:
        for p in ctx.processes:
            if p.is_alive():
                p.kill()
                p.join()
    got = np.load(tmp_path / "world1.npy", allow_pickle=True).item()
    assert got[False] is True and got[True] is True
    assert got["zero_mass"].startswith("Exception: ERROR: INVALID SATELLITE MASS"), got["zero_mass"]
