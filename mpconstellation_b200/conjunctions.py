"""Close-approach screening of a constellation's trajectories: every satellite pair of one propagate_batch[_device] run
in one device pass (include/mpc_b200.h, mpc_screen_conjunctions).

Satellite s is taken to SI in its own units: r = y[0:3] R0_s, v = y[3:6] R0_s / s0_s with s0_s = sqrt(MU_s R0_s^3 /
MU_EARTH) (a SatelliteScale's 2 pi sqrt(R0^3 / MU_EARTH)); its run lasts D_s = tf_s s0_s seconds.  Every D_s must be the
same D (to 1e-12 relative), so that sample j is the instant j D / (T - 1) for every satellite: a mixed constellation
flies with tf_s = D / s0_s.  Between two samples each satellite follows the cubic Hermite curve through its positions and
velocities there; an event is a local minimum of a pair's distance below the threshold (see conjunction_kernel.cuh).
"""
import ctypes
from dataclasses import dataclass

import numpy as np

from . import _lib
from .model import MU_EARTH

DEFAULT_CAPACITY = 1 << 16
_FIELDS = ("i", "j", "k", "flags", "t_ca", "d_min", "v_rel")


@dataclass
class Conjunctions:
    """Events sorted by (i, j, t_ca): i < j the satellites, k the sample interval, t_ca (s from the start of the run),
    d_min (m), v_rel (m/s at t_ca), flags (MPC_CONJ_FLAG_DEPTH: the root isolation hit its depth cap, t_ca known to
    2^-20 of an interval).  numpy arrays from screen_conjunctions, CUDA tensors from screen_conjunctions_device.
    skipped [N]: intervals of satellite s with a non-finite end sample (left out for every pair with s); n_flagged: events
    with a flag; duration: D (s)."""
    i: object
    j: object
    k: object
    flags: object
    t_ca: object
    d_min: object
    v_rel: object
    skipped: object
    n_flagged: int
    duration: float

    def __len__(self):
        return int(self.i.shape[0])


def _bags(const, n):
    if hasattr(const, "MU"):
        return [const] * n
    try:
        const = list(const)
    except TypeError:
        raise ValueError(f"const must be a Constants bag or a sequence of {n} of them, got {type(const).__name__}") from None
    if len(const) != n:
        raise ValueError(f"per-satellite constants: expected {n} Constants, got {len(const)}")
    return const


def screen_scales(shape, tf, const, threshold_m, T_sat=None):
    """The checks and the scale table of a screening call, before any device work -> (scale [N, 2] = (R0_s, R0_s / s0_s),
    D).  Raises ValueError for a bad shape or threshold, a ragged T_sat, non-finite or non-positive constants or tf, or
    durations D_s that differ from satellite 0's by more than 1e-12 relative (naming the satellite)."""
    if len(shape) != 3 or shape[1] != 7:
        raise ValueError(f"y must be [N, 7, T], got shape {tuple(shape)}")
    N, _, T = (int(v) for v in shape)
    if N < 2 or T < 2:
        raise ValueError(f"need at least 2 satellites and 2 samples (got N = {N}, T = {T})")
    thr = float(threshold_m)
    if not (np.isfinite(thr) and thr > 0.0):
        raise ValueError(f"threshold_m must be finite and > 0 (got {threshold_m})")
    if T_sat is not None:
        ts = np.broadcast_to(np.asarray(T_sat), (N,))
        bad = np.flatnonzero(ts != T)
        if bad.size:
            raise ValueError(f"satellite {bad[0]} has T_sat = {ts[bad[0]]}: screening needs every satellite on the same "
                             f"{T} samples (ragged batches are not supported)")
    try:
        tfv = np.broadcast_to(np.asarray(tf, dtype=np.float64), (N,))
    except ValueError:
        raise ValueError(f"tf must be a scalar or [N = {N}], got shape {np.shape(tf)}") from None
    bags = _bags(const, N)
    scale = np.empty((N, 2))
    dur = np.empty(N)
    for s, c in enumerate(bags):
        r0, mu = float(c.R0), float(c.MU)
        if not (np.isfinite(r0) and r0 > 0.0 and np.isfinite(mu) and mu > 0.0):
            raise ValueError(f"satellite {s}: need finite R0 > 0 and MU > 0 (got {r0}, {mu})")
        s0 = np.sqrt(mu * r0 ** 3 / MU_EARTH)
        scale[s] = (r0, r0 / s0)
        dur[s] = float(tfv[s]) * s0
        if not (np.isfinite(dur[s]) and dur[s] > 0.0):
            raise ValueError(f"satellite {s}: need a finite tf > 0 (got {tfv[s]})")
    D = float(dur[0])
    off = np.flatnonzero(np.abs(dur - D) > 1e-12 * D)
    if off.size:
        s = int(off[0])
        raise ValueError(f"satellite {s} flies {dur[s]!r} s, satellite 0 {D!r} s: every run must last the same time "
                         f"(tf_s = D / s0_s)")
    return np.ascontiguousarray(scale), D


def _sorted_host(ev, skipped, n_flagged, D):
    order = np.lexsort((ev["t_ca"], ev["j"], ev["i"]))
    ev = ev[order]
    return Conjunctions(*(np.ascontiguousarray(ev[f]) for f in _FIELDS), skipped=skipped, n_flagged=int(n_flagged),
                        duration=D)


def screen_conjunctions(y, tf, const, threshold_m, capacity=DEFAULT_CAPACITY, T_sat=None, device=0):
    """Every close approach below threshold_m (m) between two satellites of one propagation: y [N, 7, T] host array as
    propagate_batch returns it (normalized), tf a scalar or [N], const one Constants bag or N of them (as for every other
    entry point) -> Conjunctions (numpy).  When the device finds more than `capacity` events it runs once more with room
    for all of them."""
    from .batch import _ctx, _lock
    y = np.ascontiguousarray(y, dtype=np.float64)
    scale, D = screen_scales(y.shape, tf, const, threshold_m, T_sat)
    N, _, T = y.shape
    L = _lib.lib()
    cap = max(int(capacity), 1)
    count, flagged = ctypes.c_int64(), ctypes.c_int64()
    skipped = np.zeros(N, dtype=np.int32)
    with _lock(device):
        h = _ctx(device)
        for _ in range(2):
            ev = np.zeros(cap, dtype=_lib.CONJUNCTION_DTYPE)
            _lib.check(L.mpc_screen_conjunctions_host(h, _lib.addr(y), N, T, _lib.addr(scale), D, float(threshold_m),
                                                      _lib.addr(ev), cap, ctypes.byref(count), ctypes.byref(flagged),
                                                      _lib.addr(skipped)))
            if count.value <= cap:
                break
            cap = int(count.value)
    return _sorted_host(ev[:count.value], skipped, flagged.value, D)


def screen_conjunctions_device(y, tf, const, threshold_m, capacity=DEFAULT_CAPACITY, T_sat=None):
    """Device form: y [N, 7, T] float64 CUDA tensor (propagate_batch_device), tf a number, a host array or a tensor of N
    (read on the host for the duration check) -> Conjunctions of CUDA tensors, sorted on the device.  Runs on the current
    stream of y's device; reading the event count synchronizes with it."""
    import torch
    if not (isinstance(y, torch.Tensor) and y.is_cuda and y.dtype == torch.float64):
        raise ValueError("y must be a float64 CUDA tensor")
    if isinstance(tf, torch.Tensor):
        tf = tf.detach().cpu().numpy()
    scale, D = screen_scales(tuple(y.shape), tf, const, threshold_m, T_sat)
    N, _, T = y.shape
    y = y.contiguous()
    dev = y.device
    L = _lib.lib()
    stream = torch.cuda.current_stream(dev).cuda_stream
    rec = _lib.CONJUNCTION_DTYPE.itemsize // 8
    scratch = torch.empty(int(L.mpc_conjunction_scratch_doubles(N, T)), dtype=torch.float64, device=dev)
    counters = torch.zeros(2, dtype=torch.int64, device=dev)
    skipped = torch.empty(N, dtype=torch.int32, device=dev)
    cap = max(int(capacity), 1)
    for _ in range(2):
        ev = torch.empty((cap, rec), dtype=torch.float64, device=dev)
        _lib.check(L.mpc_screen_conjunctions(y.data_ptr(), N, T, _lib.addr(scale), D, float(threshold_m), scratch.data_ptr(),
                                             ev.data_ptr(), cap, counters.data_ptr(), skipped.data_ptr(), stream))
        count, flagged = (int(v) for v in counters.cpu())
        if count <= cap:
            break
        cap = count
    ev = ev[:count]
    ints = ev[:, 0:2].contiguous().view(torch.int32)          # i, j, k, flags
    t_ca, d_min, v_rel = ev[:, 2], ev[:, 3], ev[:, 4]
    order = torch.argsort(t_ca, stable=True)
    order = order[torch.argsort(ints[order, 1], stable=True)]
    order = order[torch.argsort(ints[order, 0], stable=True)]
    ints = ints[order]
    return Conjunctions(ints[:, 0].contiguous(), ints[:, 1].contiguous(), ints[:, 2].contiguous(), ints[:, 3].contiguous(),
                        t_ca[order].contiguous(), d_min[order].contiguous(), v_rel[order].contiguous(), skipped,
                        flagged, D)
