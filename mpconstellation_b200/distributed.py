"""Multi-GPU: satellites sharded over ranks, the all-gather of the discretized matrices fused into the kernel.

Every (satellite, interval) is independent given the reference trajectory (linearize_discretize.py:31-34),
so the path shards by satellite with no exchange until the end; the one exchange north_star names is the
all-gather of the SoA matrices to the rank(s) driving the optimizer.  One process per GPU (torchrun);
`torch.distributed` does the plumbing.

Two implementations of the exchange:

* `FusedGather` (the product path on NVLink/NVSwitch boxes): every rank owns a symmetric-memory buffer in
  the FINAL gathered layout  G[row][global column],  global column = global_satellite * (K-1) + k.
  The discretization kernel of rank r stores each result directly into column range r of EVERY rank's
  buffer (`mpc_discretize_batch_multi`, peer-mapped pointers): the transfer is spread over the whole
  compute-bound kernel instead of following it, no staging copy, no separate collective launch.
  A symmetric-memory barrier closes the step.
* `nccl_gather_chunks` (baseline / fallback when peer mapping is unavailable): chunked
  `all_gather_into_tensor` on a side stream, overlapping the gather of chunk c with the compute of chunk c+1.

`GatheredView` hands out the reference-shaped per-satellite views of either result, so optimizer-side code
indexes exactly as before (optimizer.py:327-339).

`RaggedGather` is the sharded linearization of the batches `BatchedSCP` produces after the first solve: every satellite on
its own grid K_s and / or in its own designer units.  Satellites are split by live intervals (`shard_ranges_by_work`),
the ragged discretization kernels store into every rank's buffer (`mpc_discretize_batch_ragged_gather`) and the
reference trajectories follow by one copy per peer.
"""
from dataclasses import dataclass

import numpy as np

from . import _lib


def shard_sizes(n_sats, world):
    """Contiguous blocks of ceil(N/G) satellites; trailing ranks may be short or empty."""
    per = (n_sats + world - 1) // world if world > 0 else 0
    return [max(0, min(per, n_sats - r * per)) for r in range(world)]


def shard_range(n_sats, rank, world):
    per = (n_sats + world - 1) // world
    s0 = min(n_sats, rank * per)
    return s0, min(n_sats, s0 + per)


def shard_ranges_by_work(K_sat, world):
    """Contiguous satellite ranges [(s0, s1)] * world balanced by live intervals sum(K_s - 1), not by satellite count
    (the discretization sets the balance: the propagation costs about the same per satellite up to far larger batches).
    Rank r takes the satellites up to the first prefix sum >= r ceil(total / world), so each rank's live count is at
    most ceil(total / world) + max(K_s - 1) - 1.  Ranges may be empty (world > N included)."""
    w = np.asarray(K_sat, dtype=np.int64).reshape(-1) - 1
    if world < 1:
        raise ValueError(f"world must be >= 1, got {world}")
    if w.size and w.min() < 1:
        raise ValueError("every K_s must be >= 2")
    prefix = np.concatenate([[0], np.cumsum(w)])
    target = -(-int(prefix[-1]) // world)
    edges = [0] + [int(np.searchsorted(prefix, r * target, side="left")) for r in range(1, world)] + [int(w.size)]
    edges = [min(e, int(w.size)) for e in edges]
    return [(edges[r], max(edges[r], edges[r + 1])) for r in range(world)]


def _np(a):
    return a if isinstance(a, np.ndarray) else a.detach().cpu().numpy()


class GatheredView:
    """Per-satellite access to a gathered SoA buffer.

    layout "global":  buf[105, n_sats*(K-1)], column = s (K-1) + k     (FusedGather, satellite-major)
    layout "kmajor":  buf[105, n_sats*(K-1)], column = k n_sats + s     (FusedGather, k-major: a strided view per satellite)
    layout "rank":    buf[world, 105, per*(K-1)]                        (NCCL all-gather of equal rank blocks)
    """

    def __init__(self, buf, n_sats, K, world, layout="global"):
        self.buf, self.n_sats, self.K, self.world, self.layout = buf, n_sats, K, world, layout
        self.per = (n_sats + world - 1) // world

    def block(self, s):
        if not 0 <= s < self.n_sats:
            raise IndexError(s)
        n = self.K - 1
        if self.layout == "global":
            return _np(self.buf[:, s * n:(s + 1) * n])
        if self.layout == "kmajor":
            return _np(self.buf[:, s:s + n * self.n_sats:self.n_sats])
        r, ls = s // self.per, s % self.per
        return _np(self.buf[r][:, ls * n:(ls + 1) * n])

    def sat(self, s):
        """(A_k, B_kp, B_kn, Sigma_k, xi_k) of GLOBAL satellite s; shapes/order of linearize_discretize.py:390."""
        n = self.K - 1
        blk = self.block(s)
        A = blk[_lib.ROW_A:_lib.ROW_A + 49].T.reshape(n, 7, 7)
        Bp = blk[_lib.ROW_BP:_lib.ROW_BP + 21].T.reshape(n, 7, 3)
        Bn = blk[_lib.ROW_BN:_lib.ROW_BN + 21].T.reshape(n, 7, 3)
        return A, Bp, Bn, blk[_lib.ROW_SIGMA:_lib.ROW_SIGMA + 7], blk[_lib.ROW_XI:_lib.ROW_XI + 7]


def _dst_count(world):
    for n in (1, 2, 4, 8):
        if world <= n:
            return n
    raise ValueError("FusedGather supports up to 8 ranks (one NVSwitch box)")


class FusedGather:
    """All-gather of the discretized matrices by peer stores from inside the discretization kernel."""

    def __init__(self, n_sats_total, K, group=None, device=None, mode="unicast", chunk_waves=1, skip_const=True,
                 stagger=None, layout=None):
        """mode "unicast": one peer-mapped store per destination rank (works on any P2P-capable box);
        mode "multicast": one store to the NVSwitch multicast address of the symmetric buffer, replicated by the
        switch to every rank (NVLS) -- 1/world of the SM store instructions and of the egress traffic;
        mode "push": the kernel stores locally, chunk by chunk, and the copy engines push every finished chunk to
        the peers' buffers over NVLink while the next chunk is computed (`mpc_discretize_batch_push`): no SM time
        and no store-queue stalls go into the exchange, and the structurally constant rows are not sent;
        mode "pushk": the same pipeline with a small highest-priority copy kernel per chunk instead of the copy engines.
        skip_const: rows 42..48 (the last row of A_k, constants 0..0 1) are written once into every buffer here and
        never sent again (6.7 % less NVLink traffic).  stagger: see mpc_set_gather_tuning.
        layout: "satmajor" (column = s (K-1) + k, per-satellite blocks) or "kmajor" (column = k N + s): in the k-major
        layout a k-window of the overlapped pass stores whole runs of consecutive columns, so the propagation can hide
        behind the discretization at any world size (satellite-major: world <= 2 only).  Default: kmajor (push modes:
        satmajor)."""
        import torch
        import torch.distributed as dist
        import torch.distributed._symmetric_memory as symm_mem
        self.group = dist.group.WORLD if group is None else group
        self.world = dist.get_world_size(self.group)
        self.rank = dist.get_rank(self.group)
        self.n_sats, self.K = n_sats_total, K
        self.pitch = n_sats_total * (K - 1)
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else device
        self.buf = symm_mem.empty((_lib.MPC_OUT_ROWS, self.pitch), dtype=torch.float64, device=self.device)
        self.handle = symm_mem.rendezvous(self.buf, self.group)
        ptrs = [int(p) for p in self.handle.buffer_ptrs]
        # own buffer first (it is also the kernel's "local" destination), then the peers, rotated so that the
        # ranks do not all hammer the same peer at the same time; padded to 1/2/4/8 with the own pointer
        order = [(self.rank + i) % self.world for i in range(self.world)]
        self.dst = [ptrs[r] for r in order]
        while len(self.dst) < _dst_count(self.world):
            self.dst.append(ptrs[self.rank])
        self.mode = mode
        self.mc_ptr = int(getattr(self.handle, "multicast_ptr", 0) or 0)
        if mode == "multicast" and not self.mc_ptr:
            raise RuntimeError("this box / torch build exposes no multicast (NVLS) mapping for symmetric memory")
        self.chunk_waves = int(chunk_waves)
        self.skip_const = bool(skip_const) or mode in ("push", "pushk")
        # measured on 8xB200 (profiles/r01_e_multi_gpu.txt): 4 phases help once the step is NVLink-ingress bound
        self.stagger = int(stagger) if stagger is not None else (4 if self.world >= 8 and mode == "unicast" else 0)
        if self.skip_const:
            # rows 42..48 of every buffer are constants that are never sent: written once, here, by the owner
            _lib.check(_lib.lib().mpc_fill_const_rows(self.buf.data_ptr(), self.pitch,
                                                      torch.cuda.current_stream(self.device).cuda_stream))
            torch.cuda.synchronize(self.device)
            self.handle.barrier()
        if mode in ("push", "pushk"):
            self.peers = [ptrs[self.rank]] + [ptrs[r] for r in order[1:]]
        # (measured, profiles/r02_*_multi_gpu_w*: k-major is the faster layout of the overlapped pass at 2, 4 and 8 GPUs;
        # the push modes copy per-satellite column blocks and keep the satellite-major one)
        self.layout = layout if layout is not None else ("satmajor" if mode in ("push", "pushk") else "kmajor")
        if self.layout not in ("satmajor", "kmajor"):
            raise ValueError(f"unknown layout {self.layout!r}")
        if self.layout == "kmajor" and mode in ("push", "pushk"):
            raise ValueError("the push modes copy per-satellite column blocks: satellite-major layout only")
        self.overlap_ok = self.world <= 2 or self.layout == "kmajor"     # see propagate_discretize
        self.s0, self.s1 = shard_range(n_sats_total, self.rank, self.world)
        self.status = torch.zeros(max(1, (self.s1 - self.s0) * (K - 1)), dtype=torch.int32, device=self.device)

    def _pre_barrier(self, pre_barrier):
        """The kernel of this rank stores into EVERY rank's buffer.  The barrier after the kernel only says "all results
        of this step have landed"; nothing there stops a fast rank from starting the next step and overwriting its column
        range in a peer's buffer while that peer is still reading the previous result.  So every step opens with a
        barrier as well, enqueued on the current stream behind whatever the caller enqueued there to consume the
        previous result: "every rank is done with step n" before any store of step n+1 (a few microseconds).  A caller
        that synchronises all ranks itself between consuming and the next step may pass pre_barrier=False."""
        if pre_barrier and self.world > 1:
            self.handle.barrier(channel=1)

    def discretize(self, x, u, tf, const, include_J2=False, n_sub=100, barrier=True, pre_barrier=True):
        """x [n_local,7,K], u [n_local,3,K], tf [n_local] (this rank's shard_range block, CUDA float64).  Enqueues
        the kernel on the current stream; with barrier=True also the cross-rank barrier after which every
        rank's `self.buf` holds all N satellites (pre_barrier: see _pre_barrier)."""
        from . import batch
        assert x.shape[0] == self.s1 - self.s0 and x.shape[2] == self.K
        self._pre_barrier(pre_barrier)
        self._launch(x, u, tf, const, include_J2, n_sub)
        if barrier:
            self.handle.barrier()
        return self.buf

    def propagate_discretize(self, y0, tf, controller, const, include_J2=False, n_sub_prop=None, n_sub=100, y=None,
                             u_out=None, status_prop=None, barrier=True, n_windows=0, pre_barrier=True):
        """One SCP linearization pass of this rank's shard with the all-gather fused in AND the propagation hidden
        behind the discretization (`mpc_propagate_discretize_gather`): y0 [n_local,7], tf [n_local] CUDA float64.
        Modes "unicast" and "multicast".  In the satellite-major layout a k-window stores runs of ~13 columns per row and
        satellite -- fine for HBM and for one peer, but with 7 peers the step is NVLink-ingress bound and the fragmented
        peer stores cost more than the hidden propagation buys (8 x B200: 7.77 ms back to back, 13.8 ms windowed;
        profiles/r01_n_overlap.txt) -- so there the overlapped pass is used at world <= 2 only.  In the k-major layout
        (the default) a window stores whole runs of consecutive columns and the overlapped pass is used at any
        world size.  The push modes keep the two-kernel sequence.
        Returns (buf, y, u, status_prop); results are bit-identical to propagate_batch_device + discretize()."""
        from . import batch
        assert y0.shape[0] == self.s1 - self.s0
        if self.mode in ("push", "pushk") or y0.shape[0] == 0 or not self.overlap_ok:
            y, u_out, status_prop = batch.propagate_batch_device(y0, tf, controller, const, include_drag=False,
                                                                 include_J2=include_J2, T=self.K, n_sub=n_sub_prop,
                                                                 y=y, u_out=u_out, status=status_prop)
            self.discretize(y, u_out, tf, const, include_J2=include_J2, n_sub=n_sub, barrier=barrier,
                            pre_barrier=pre_barrier)
            return self.buf, y, u_out, status_prop
        self._pre_barrier(pre_barrier)
        mc = self.mode == "multicast"
        _, y, u_out, status_prop, _ = batch.propagate_discretize_device(
            y0, tf, controller, const, self.K, prop_J2=include_J2, disc_J2=include_J2, n_sub_prop=n_sub_prop,
            n_sub_disc=n_sub, y=y, u_out=u_out, out=self.buf, status_prop=status_prop, status_disc=self.status,
            n_windows=n_windows, extra_dst=None if mc else self.dst[1:], out_ptr=self.mc_ptr if mc else None,
            gather=self._opts())
        if barrier:
            self.handle.barrier()
        return self.buf, y, u_out, status_prop

    def _opts(self):
        """Options of one fused-gather launch (passed per call: nothing process-wide is touched)."""
        return _lib.MpcGatherOpts(_lib.LAYOUT_K_MAJOR if self.layout == "kmajor" else _lib.LAYOUT_SAT_MAJOR,
                                  (2 if self.mode == "multicast" else 1) if self.skip_const else 0,
                                  self.stagger if self.stagger > 1 else 0, 0, self.n_sats, self.s0)

    def _launch(self, x, u, tf, const, include_J2, n_sub):
        from . import batch
        if x.shape[0] > 0 and self.mode in ("unicast", "multicast"):
            import ctypes
            import torch
            p = _lib.make_params(const, include_J2, False)
            stream = torch.cuda.current_stream(x.device).cuda_stream
            ptrs = [self.mc_ptr] if self.mode == "multicast" else self.dst
            arr = (ctypes.c_void_p * len(ptrs))(*ptrs)
            g = self._opts()
            _lib.check(_lib.lib().mpc_discretize_batch_gather(x.data_ptr(), u.data_ptr(), tf.data_ptr(), ctypes.byref(p),
                                                              x.shape[0], self.K, int(n_sub), arr, len(ptrs),
                                                              ctypes.byref(g), self.status.data_ptr(), stream))
        elif x.shape[0] > 0 and self.mode in ("push", "pushk"):
            import ctypes
            import torch
            p = _lib.make_params(const, include_J2, False)
            stream = torch.cuda.current_stream(x.device).cuda_stream
            arr = (ctypes.c_void_p * len(self.peers))(*self.peers)
            _lib.check(_lib.lib().mpc_discretize_batch_push(
                batch._ctx(self.device.index or 0), x.data_ptr(), u.data_ptr(), tf.data_ptr(), ctypes.byref(p), x.shape[0],
                self.K, int(n_sub), arr, len(self.peers), self.pitch, self.s0 * (self.K - 1), self.status.data_ptr(),
                self.chunk_waves, int(self.mode == "pushk"), stream))

    def view(self):
        return GatheredView(self.buf, self.n_sats, self.K, self.world, layout="kmajor" if self.layout == "kmajor" else "global")


def nccl_gather_chunks(local, n_chunks, group=None, side_stream=None, produce=None, chunk_cols=None):
    """Baseline exchange: `local` is this rank's [105, cols] block (equal cols on every rank).  It is gathered
    in `n_chunks` column chunks (or chunks of exactly `chunk_cols` columns); if `produce(c0, c1)` is given it is called right before chunk [c0,c1) is
    gathered (that is where the caller launches the kernel for those columns), so gather(c) overlaps
    produce(c+1).  Returns the list of gathered chunk tensors [world, 105, chunk_cols] and the chunk bounds.
    Works on CPU tensors with gloo (used by the CPU tests) and CUDA tensors with NCCL."""
    import torch
    import torch.distributed as dist
    world = dist.get_world_size(group)
    cols = local.shape[1]
    csz = int(chunk_cols) if chunk_cols else max(1, (cols + n_chunks - 1) // n_chunks)
    cuda = local.is_cuda
    if cuda and side_stream is None:
        side_stream = torch.cuda.Stream(local.device)
    out, bounds = [], []
    for c0 in range(0, cols, csz):
        c1 = min(cols, c0 + csz)
        if produce is not None:
            produce(c0, c1)
        piece = local[:, c0:c1].contiguous()
        recv = torch.empty((world,) + tuple(piece.shape), dtype=local.dtype, device=local.device)
        if cuda:
            ev = torch.cuda.Event()
            ev.record(torch.cuda.current_stream(local.device))
            side_stream.wait_event(ev)
            with torch.cuda.stream(side_stream):
                dist.all_gather_into_tensor(recv.view(-1, piece.shape[1]), piece, group=group)
            piece.record_stream(side_stream)
        else:
            dist.all_gather_into_tensor(recv.view(-1, piece.shape[1]), piece, group=group)
        out.append(recv)
        bounds.append((c0, c1))
    if cuda:
        torch.cuda.current_stream(local.device).wait_stream(side_stream)
    return out, bounds


def assemble_rank_major(chunks, bounds, world):
    """[world, 105, cols] from the chunk list of nccl_gather_chunks (a copy; for consumers that want one buffer)."""
    import torch
    cols = bounds[-1][1]
    full = torch.empty((world, chunks[0].shape[1], cols), dtype=chunks[0].dtype, device=chunks[0].device)
    for t, (c0, c1) in zip(chunks, bounds):
        full[:, :, c0:c1] = t
    return full


@dataclass
class ShardedLinearization:
    """Result of RaggedGather.linearize on every rank, device-resident and in the single-GPU ragged layout at the
    capacity K_cap (views of the gatherer's buffers: the next linearize overwrites them; padding columns are not written).
      soa     [105, N (K_cap - 1)]: satellite s on columns s (K_cap - 1) + k, k < K_s - 1
      x_bar   [N, 7, K_cap], u_bar [N, 3, K_cap]: the reference trajectories (first K_s columns of satellite s)
      tf [N], K_sat [N] (host int32), const: what the pass ran with
      n_nodes [s1 - s0, K_cap - 1] (default mode): node counts of THIS rank's satellites ranges[rank] only
    Feeds the hand-off as the single-GPU result does: constraint_terms_device(x_bar, u_bar, const, K=K_sat),
    dynamics_jacobian_device(soa, N, K_cap, K_sat=K_sat)."""
    soa: object
    x_bar: object
    u_bar: object
    tf: object
    K_sat: np.ndarray
    const: object
    ranges: list
    n_nodes: object = None

    def sat(self, s):
        """(A_k, B_kp, B_kn, Sigma_k, xi_k) of GLOBAL satellite s on its K_s - 1 intervals; shapes of
        linearize_discretize.py:390 (device tensors)."""
        from .batch import DiscretizedBatch
        return DiscretizedBatch(self.soa, None, len(self.K_sat), self.x_bar.shape[2], K_sat=self.K_sat).sat(s)


def _shard_spec(spec, s0, s1):
    """the controller law of satellites [s0, s1): the per-satellite tables / end_tau / table lengths sliced"""
    from .control import ControllerSpec
    tab = spec.table
    if tab is not None and np.ndim(tab) == 3:
        tab = np.ascontiguousarray(np.asarray(tab)[s0:s1])
    end_tau = spec.end_tau if np.ndim(spec.end_tau) == 0 else np.asarray(spec.end_tau)[s0:s1]
    lens = None if spec.table_len is None else np.asarray(spec.table_len)[s0:s1]
    return ControllerSpec(spec.kind, spec.thrust, tab, end_tau, lens)


def _raise_status(code, what):
    """the exceptions of batch.raise_on_status for a status code combined over the ranks"""
    if code == _lib.ST_MASS:
        # same exception type / text as simulator.py:135-136
        raise Exception(f"ERROR: INVALID SATELLITE MASS: non-positive mass in the sharded {what}")
    if code == _lib.ST_STEP:
        raise RuntimeError(f"adaptive integration failed (step size underflow) in the sharded {what}")
    raise FloatingPointError(f"non-finite result in the sharded {what}")


class RaggedGather:
    """Sharded SCP linearization of a ragged and / or per-satellite-units constellation over the ranks of one box.

    The buffers -- matrices [105, N (K_cap - 1)], x_bar [N, 7, K_cap], u_bar [N, 3, K_cap] -- are ONE symmetric-memory
    allocation made here, once: the node counts change from one SCP iteration to the next, the layout (capacity K_cap)
    does not, so no allocation or rendezvous happens per call.  Each rank takes the contiguous satellite range
    shard_ranges_by_work gives it for the call's counts.  On a gloo group (CPU tensors) the buffers are plain tensors and
    the exchange is a broadcast of every rank's blocks; the computation itself needs CUDA (_compute)."""

    def __init__(self, n_sats, K_cap, group=None, device=None, skip_const=True):
        import torch
        import torch.distributed as dist
        if n_sats < 0 or K_cap < 2:
            raise ValueError(f"need n_sats >= 0 and K_cap >= 2 (got {n_sats}, {K_cap})")
        self.group = dist.group.WORLD if group is None else group
        self.world = dist.get_world_size(self.group)
        self.rank = dist.get_rank(self.group)
        self.n_sats, self.K_cap = int(n_sats), int(K_cap)
        self.pitch = self.n_sats * (self.K_cap - 1)
        self.cuda = dist.get_backend(self.group) != "gloo"
        if device is None:
            device = torch.device("cuda", torch.cuda.current_device()) if self.cuda else torch.device("cpu")
        self.device = torch.device(device)
        n_buf, n_x = _lib.MPC_OUT_ROWS * self.pitch, self.n_sats * 7 * self.K_cap
        n_all = n_buf + n_x + self.n_sats * 3 * self.K_cap
        self._off = (0, n_buf, n_buf + n_x)             # element offsets of buf, x_bar, u_bar
        if self.cuda:
            import torch.distributed._symmetric_memory as symm_mem
            self.flat = symm_mem.empty((max(1, n_all),), dtype=torch.float64, device=self.device)
            self.handle = symm_mem.rendezvous(self.flat, self.group)
        else:
            self.flat, self.handle = torch.empty((max(1, n_all),), dtype=torch.float64), None
        self.flat.fill_(float("nan"))
        self.buf = self.flat[:n_buf].view(_lib.MPC_OUT_ROWS, self.pitch)
        self.x_bar = self.flat[n_buf:n_buf + n_x].view(self.n_sats, 7, self.K_cap)
        self.u_bar = self.flat[n_buf + n_x:n_all].view(self.n_sats, 3, self.K_cap)
        self.skip_const = bool(skip_const) and self.world > 1
        if self.cuda:
            ptrs = [int(p) for p in self.handle.buffer_ptrs]
            self._base = (self.flat.data_ptr() - ptrs[self.rank]) // 8     # the tensor's place in its allocation
            # own buffer first (the kernel's local destination), then the peers rotated as in FusedGather, padded to
            # 1/2/4/8 with the own one
            order = [(self.rank + i) % self.world for i in range(self.world)]
            self.peers = order[1:]
            self.dst = [ptrs[r] + 8 * self._base for r in order]
            while len(self.dst) < _dst_count(self.world):
                self.dst.append(self.dst[0])
        if self.skip_const and self.pitch:
            # rows 42..48 (the last row of A_k: constants 0..0 1) are written once into every buffer here, never sent
            if self.cuda:
                _lib.check(_lib.lib().mpc_fill_const_rows(self.buf.data_ptr(), self.pitch,
                                                          torch.cuda.current_stream(self.device).cuda_stream))
                torch.cuda.synchronize(self.device)
            else:
                self.buf[42:49] = 0.0
                self.buf[48] = 1.0
        self._barrier()

    def _barrier(self, channel=0):
        import torch.distributed as dist
        if self.world == 1:
            return
        if self.cuda:
            self.handle.barrier(channel=channel)
        else:
            dist.barrier(self.group)

    def linearize(self, y0, tf, controller, const, K_sat, include_J2=False, use_uniform_steps=False, integrator_steps=101,
                  check=True, pre_barrier=True):
        """One SCP linearization pass of the whole constellation, sharded: run_nonlinear + extract_uk + discretize of
        every satellite on its own K_s nodes (and, with N Constants, in its own units), as BatchedSCP.linearize computes
        it on one GPU.  Every rank passes the FULL inputs: y0 [N,7], tf [N] (numpy or tensors), controller (a sequence law
        may carry per-satellite tables / table lengths), const (one bag or N), K_sat [N] (2 <= K_s <= K_cap).
        Each rank propagates its shard (RK45 replay, no drag / J2, as OptimalController.run_nonlinear), discretizes it
        into every rank's buffer, copies its x_bar / u_bar block to every peer and meets the others at a barrier; then
        the status words are combined over the ranks (max), and with check=True a non-positive mass raises the
        reference's Exception on every rank (non-finite results / step underflow raise as in raise_on_status).
        pre_barrier: see FusedGather._pre_barrier.  Returns a ShardedLinearization."""
        import torch
        import torch.distributed as dist
        from .control import spec_from
        N, Kc = self.n_sats, self.K_cap
        K_sat = np.ascontiguousarray(K_sat, dtype=np.int32)
        if K_sat.shape != (N,) or (N and (K_sat.min() < 2 or K_sat.max() > Kc)):
            raise ValueError(f"K_sat must be [{N}] with every count in [2, {Kc}]")
        y0 = torch.as_tensor(y0, dtype=torch.float64).to(self.device).contiguous()
        tfv = torch.as_tensor(tf, dtype=torch.float64, device=self.device).reshape(-1).expand(N).contiguous()
        if y0.shape != (N, 7):
            raise ValueError(f"y0 must be [{N}, 7], got {tuple(y0.shape)}")
        one_bag = hasattr(const, "MU")
        if not one_bag and len(const) != N:          # (the bags themselves are checked where they are packed)
            raise ValueError(f"per-satellite constants: expected {N} Constants, got {len(const)}")
        ranges = shard_ranges_by_work(K_sat, self.world)
        s0, s1 = ranges[self.rank]
        shard_const = const if one_bag else list(const)[s0:s1]
        spec = _shard_spec(spec_from(controller), s0, s1)
        adaptive = None if use_uniform_steps else dict(rtol=1e-3, atol=1e-6, max_step=1e-2)
        n_nodes = None if use_uniform_steps else torch.zeros(((s1 - s0), Kc - 1), dtype=torch.int32, device=self.device)
        if self.world == 1:
            # the single-GPU calls, into the same buffers
            if N:
                from . import batch
                _, _, st_prop = batch.propagate_batch_device(y0, tfv, spec, const, include_drag=False, include_J2=False,
                                                             T=K_sat, T_max=Kc, y=self.x_bar, u_out=self.u_bar)
                _, st_disc = batch.discretize_batch_device(self.x_bar, self.u_bar, tfv, const, include_J2=include_J2,
                                                           n_sub=integrator_steps - 1, out=self.buf, adaptive=adaptive,
                                                           n_nodes=n_nodes, K=K_sat)
                words = torch.stack([st_prop.max(), st_disc.max()])
            else:
                words = torch.zeros(2, dtype=torch.int32, device=self.device)
        else:
            if pre_barrier:
                self._barrier(channel=1)
            words = self._compute(y0[s0:s1], tfv[s0:s1], spec, shard_const, K_sat[s0:s1], s0, include_J2, adaptive,
                                  integrator_steps - 1, n_nodes)
            self._publish(ranges)
            self._barrier()
            dist.all_reduce(words, op=dist.ReduceOp.MAX, group=self.group)
        if check:
            codes = words.tolist()
            if codes[0]:
                _raise_status(codes[0], "propagation")
            if codes[1]:
                _raise_status(codes[1], "discretization")
        res = ShardedLinearization(self.buf, self.x_bar, self.u_bar, tfv, K_sat, const, ranges, n_nodes)
        res.status = words
        return res

    def _compute(self, y0, tf, spec, const, K_sat, s0, include_J2, adaptive, n_sub, n_nodes):
        """this rank's shard: propagate into the own x_bar / u_bar rows, discretize into every rank's buffer; returns the
        device int32 [2] (max propagation status, max discretization status) of the shard"""
        import ctypes
        import torch
        from . import batch
        n, Kc = y0.shape[0], self.K_cap
        if n == 0:
            return torch.zeros(2, dtype=torch.int32, device=self.device)
        x, u = self.x_bar[s0:s0 + n], self.u_bar[s0:s0 + n]
        _, _, st_prop = batch.propagate_batch_device(y0, tf, spec, const, include_drag=False, include_J2=False, T=K_sat,
                                                     T_max=Kc, y=x, u_out=u)
        psc, one = batch._units_of(const, n)
        p = _lib.make_params(one, include_J2, False)
        cur = torch.cuda.current_stream(self.device)
        status = torch.zeros(n * (Kc - 1), dtype=torch.int32, device=self.device)
        first = torch.empty(n + 1, dtype=torch.int64, device=self.device)
        scratch = torch.empty(n * _lib.SAT_SCRATCH_DOUBLES, dtype=torch.float64, device=self.device) if psc is not None else None
        arr = (ctypes.c_void_p * len(self.dst))(*self.dst)
        ad = adaptive or {}
        _lib.check(_lib.lib().mpc_discretize_batch_ragged_gather(
            x.data_ptr(), u.data_ptr(), tf.data_ptr(), ctypes.byref(p), psc, n, Kc, _lib.addr(K_sat), first.data_ptr(),
            scratch.data_ptr() if scratch is not None else None, int(adaptive is not None), int(n_sub),
            float(ad.get("rtol", 1e-3)), float(ad.get("atol", 1e-6)), float(ad.get("max_step", 1e-2)), arr, len(self.dst),
            self.pitch, s0 * (Kc - 1), 1 if self.skip_const else 0, status.data_ptr(),
            n_nodes.data_ptr() if n_nodes is not None else None, cur.cuda_stream))
        for t_ in (first, scratch):
            if t_ is not None:
                t_.record_stream(cur)
        return torch.stack([st_prop.max(), status.max()])

    def _publish(self, ranges):
        """x_bar / u_bar rows of this rank's satellites into every peer's buffers: one copy per peer and array (the
        matrices are already there: the kernel stored them).  gloo: every rank's blocks broadcast from their owner."""
        import torch.distributed as dist
        Kc = self.K_cap
        if self.cuda:
            s0, s1 = ranges[self.rank]
            if s1 == s0:
                return
            for off, rows, arr in ((self._off[1], 7, self.x_bar), (self._off[2], 3, self.u_bar)):
                n_el = (s1 - s0) * rows * Kc
                src = arr[s0:s1].reshape(-1)
                for r in self.peers:
                    self.handle.get_buffer(r, (n_el,), src.dtype, self._base + off + s0 * rows * Kc).copy_(src)
            return
        for r, (a, b) in enumerate(ranges):
            if b == a:
                continue
            for arr in (self.x_bar, self.u_bar):
                dist.broadcast(arr[a:b], src=r, group=self.group)
            blk = self.buf[:, a * (Kc - 1):b * (Kc - 1)].contiguous()
            dist.broadcast(blk, src=r, group=self.group)
            self.buf[:, a * (Kc - 1):b * (Kc - 1)] = blk
