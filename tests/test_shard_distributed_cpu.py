"""CPU: the sharded linearization of ragged / per-satellite-units batches (RaggedGather) -- work-balanced satellite
ranges, the exchange of the reference trajectories and matrices, the status words combined over the ranks and the
gathered per-satellite views -- under gloo, world size 2.  The per-rank computation is stood in for by the host build of
the kernel sources (single-destination launches on the shard, tests/hostk); the slicing, exchange, status and view code
is the product's (mpconstellation_b200/distributed.py)."""
import os
import socket

import numpy as np
import pytest

from mpconstellation_b200 import distributed as D


def _bound(K_sat, world):
    w = np.asarray(K_sat, np.int64) - 1
    return -(-int(w.sum()) // world) + int(w.max())


@pytest.mark.parametrize("K_sat, world", [
    ([7, 2, 12, 5, 12, 3], 2), ([7, 2, 12, 5, 12, 3], 4), ([100] * 5 + [2] * 300, 8), ([2, 2, 2], 8), ([50], 3),
    ([400, 2, 2, 2, 2, 2, 2, 2, 2], 2), (list(np.random.default_rng(5).integers(2, 300, 4096)), 8), ([], 2)])
def test_shard_ranges_by_work_cover_are_contiguous_and_balanced(K_sat, world):
    ranges = D.shard_ranges_by_work(K_sat, world)
    assert len(ranges) == world
    assert ranges[0][0] == 0 and ranges[-1][1] == len(K_sat)
    w = np.asarray(K_sat, np.int64) - 1
    for r, (s0, s1) in enumerate(ranges):
        assert 0 <= s0 <= s1 <= len(K_sat)
        if r:
            assert s0 == ranges[r - 1][1]
        if len(K_sat):
            assert int(w[s0:s1].sum()) <= _bound(K_sat, world)


def test_shard_ranges_by_work_balance_live_intervals_not_satellites():
    K_sat = [101] * 10 + [3] * 90          # 1000 + 180 live intervals
    (a0, a1), (b0, b1) = D.shard_ranges_by_work(K_sat, 2)
    assert a1 - a0 < 10 and b1 - b0 > 90   # the long horizons are split, not the first half of the satellites
    with pytest.raises(ValueError):
        D.shard_ranges_by_work([5, 1], 2)
    with pytest.raises(ValueError):
        D.shard_ranges_by_work([5], 0)


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


K_SAT = np.array([7, 2, 12, 5, 12, 3], np.int32)
K_CAP, TF = 14, 0.3


class _HostShard(D.RaggedGather):
    """RaggedGather with the per-rank computation of the host build: the shard's trajectories (RK45 replay, tangential
    thrust) and its matrices (ragged per-satellite-constants launch) written where the CUDA path writes them"""
    bad_rank = None

    def _compute(self, y0, tf, spec, const, K_sat, s0, include_J2, adaptive, n_sub, n_nodes):
        import torch
        import test_units_kernel_source_on_host as U
        n = y0.shape[0]
        words = torch.zeros(2, dtype=torch.int32)
        if n:
            x, u = U._trajectories(y0.numpy(), const, K_sat, TF)
            self.x_bar[s0:s0 + n, :, :x.shape[2]] = torch.from_numpy(x)
            self.u_bar[s0:s0 + n, :, :u.shape[2]] = torch.from_numpy(u)
            out, st, _ = U.discretize_units(U._lib(), self.x_bar[s0:s0 + n].numpy(), self.u_bar[s0:s0 + n].numpy(), TF, const,
                                            K_sat, adaptive is not None, include_J2=include_J2)
            live = ~np.isnan(out[0])
            cols = np.arange(out.shape[1])[live] + s0 * (self.K_cap - 1)
            self.buf[:, cols] = torch.from_numpy(np.ascontiguousarray(out[:, live]))
            words[1] = int(st.max())
        if self.rank == self.bad_rank:
            words[0] = 1                   # a non-positive mass in this rank's propagation
        return words


def _worker(rank, world, port, tmp, bad_rank):
    import torch.distributed as dist
    import test_units_kernel_source_on_host as U
    from mpconstellation_b200 import ConstantTangentialThrustController
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        y0, consts = U.mixed_constellation(len(K_SAT))
        g = _HostShard(len(K_SAT), K_CAP)
        g.bad_rank = bad_rank
        try:
            res = g.linearize(y0, TF, ConstantTangentialThrustController(tangential_thrust=0.05), consts, K_SAT)
        except Exception as e:            # noqa: BLE001 -- the reference raises a plain Exception
            open(os.path.join(tmp, f"raised{rank}.txt"), "w").write(f"{type(e).__name__}: {e}")
            return
        np.savez(os.path.join(tmp, f"rank{rank}.npz"), soa=res.soa.numpy(), x=res.x_bar.numpy(), u=res.u_bar.numpy(),
                 ranges=np.array(res.ranges), A3=res.sat(3)[0].numpy(), xi2=res.sat(2)[4].numpy())
    finally:
        dist.barrier()
        dist.destroy_process_group()


def _run(tmp_path, bad_rank=None):
    import torch.multiprocessing as mp
    mp.spawn(_worker, args=(2, _free_port(), str(tmp_path), bad_rank), nprocs=2, join=True)


def test_ragged_units_gather_world2_matches_single_process(tmp_path):
    import test_units_kernel_source_on_host as U
    _run(tmp_path)
    y0, consts = U.mixed_constellation(len(K_SAT))
    x, u = U._trajectories(y0, consts, K_SAT, TF)
    ref, _, _ = U.discretize_units(U._lib(), x, u, TF, consts, K_SAT, True)
    Kmax = int(K_SAT.max())
    for rank in (0, 1):
        got = np.load(tmp_path / f"rank{rank}.npz")
        assert [tuple(r) for r in got["ranges"]] == D.shard_ranges_by_work(K_SAT, 2)
        for s, k in enumerate(K_SAT):
            n = k - 1
            assert np.array_equal(got["soa"][:, s * (K_CAP - 1):s * (K_CAP - 1) + n], ref[:, s * (Kmax - 1):s * (Kmax - 1) + n])
            assert np.array_equal(got["x"][s, :, :k], x[s, :, :k]) and np.array_equal(got["u"][s, :, :k], u[s, :, :k])
        A = ref[0:49, 3 * (Kmax - 1):3 * (Kmax - 1) + K_SAT[3] - 1].T.reshape(-1, 7, 7)
        assert np.array_equal(got["A3"], A)
        assert np.array_equal(got["xi2"], ref[98:105, 2 * (Kmax - 1):2 * (Kmax - 1) + K_SAT[2] - 1])


def test_non_positive_mass_on_one_rank_raises_on_both(tmp_path):
    _run(tmp_path, bad_rank=1)
    for rank in (0, 1):
        text = (tmp_path / f"raised{rank}.txt").read_text()
        assert text.startswith("Exception: ERROR: INVALID SATELLITE MASS"), text
