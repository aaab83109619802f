"""Conjunction screening on the device (mpc_screen_conjunctions: the pre-pass and the tiled pair kernel) against the
brute-force numpy oracle (conj_oracle.py): the analytic two-body encounter, a constellation in one constants bag and in
per-satellite units, a 512-satellite shell; bit-identical repeats, capacity overflow and its relaunch, non-finite samples,
and the device form against the host form."""
import numpy as np
import pytest

import conj_oracle as O
import mpconstellation_b200 as M

pytestmark = pytest.mark.gpu


def _rows(r):
    return [(int(r.i[e]), int(r.j[e]), int(r.k[e]), float(r.t_ca[e]), float(r.d_min[e]), float(r.v_rel[e])) for e in range(len(r))]


def _dev_rows(r):
    return [(int(a), int(b), int(c), float(t), float(d), float(v)) for a, b, c, t, d, v in
            zip(*(x.cpu().numpy() for x in (r.i, r.j, r.k, r.t_ca, r.d_min, r.v_rel)))]


@pytest.fixture(scope="module")
def shell512():
    states = O.shell(512, n_planes=16, seed=21)
    D, T = 1800.0, 61
    y, tf, const = O.fly(states, D, T)
    X = O.si_states(y, const)
    thr = O.pick_threshold(X, D, 5.0e4)
    ref, _ = O.screen(X, D, thr)
    return y, tf, const, D, T, thr, ref


def test_two_body_analytic_encounter():
    from test_conjunctions_host import two_body_case
    st, D, n, t_exact, d_exact = two_body_case()
    T = 361
    y, tf, const = O.fly(st, D, T)
    X = O.si_states(y, const)
    ref, _ = O.screen(X, D, 1.0e5)
    r = M.screen_conjunctions(y, tf, const, 1.0e5)
    assert len(r) == 2 and r.n_flagged == 0
    O.match(_rows(r), ref, D / (T - 1))
    assert np.abs(r.d_min - d_exact).max() < 1.0 and np.abs(r.t_ca - t_exact).max() < 1e-2


def test_one_bag_and_per_satellite_units():
    states = O.shell(96, n_planes=8, seed=11)
    D, T = 1500.0, 51
    y, tf, const = O.fly(states, D, T)
    X = O.si_states(y, const)
    yu, inv_s0, consts = O.renormalize(X, states)
    thr = O.pick_threshold(X, D, 3.0e5)
    ref, _ = O.screen(X, D, thr)
    r1 = M.screen_conjunctions(y, tf, const, thr)
    r2 = M.screen_conjunctions(yu, D * inv_s0, consts, thr)
    assert len(ref) >= 5
    O.match(_rows(r1), ref, D / (T - 1))
    O.match(_rows(r1), _rows(r2), D / (T - 1), rel=1e-9, t_tol=1e-9)


def test_shell_512_against_brute_force(shell512):
    y, tf, const, D, T, thr, ref = shell512
    r = M.screen_conjunctions(y, tf, const, thr)
    assert len(ref) >= 10, len(ref)
    O.match(_rows(r), ref, D / (T - 1))
    assert (r.skipped == 0).all() and r.n_flagged == 0


def test_repeat_calls_bit_identical(shell512):
    import torch
    y, tf, const, D, T, thr, ref = shell512
    a = M.screen_conjunctions(y, tf, const, thr)
    b = M.screen_conjunctions(y, tf, const, thr)
    for f in ("i", "j", "k", "flags", "t_ca", "d_min", "v_rel"):
        assert getattr(a, f).tobytes() == getattr(b, f).tobytes(), f
    yd = torch.as_tensor(y).cuda()
    c = M.screen_conjunctions_device(yd, tf, const, thr)
    d = M.screen_conjunctions_device(yd, tf, const, thr)
    for f in ("i", "j", "k", "flags", "t_ca", "d_min", "v_rel"):
        assert torch.equal(getattr(c, f), getattr(d, f)), f


def test_capacity_overflow_relaunch(shell512):
    import torch
    from mpconstellation_b200 import _lib
    y, tf, const, D, T, thr, ref = shell512
    full = M.screen_conjunctions(y, tf, const, thr)
    small = M.screen_conjunctions(y, tf, const, thr, capacity=3)
    assert len(small) == len(full) == len(ref)
    assert _rows(small) == _rows(full)
    # the C-ABI reports the full count with a buffer too small
    import ctypes
    scale, D2 = M.conjunctions.screen_scales(y.shape, tf, const, thr)
    N = y.shape[0]
    yd = torch.as_tensor(y).cuda()
    scratch = torch.empty(int(_lib.lib().mpc_conjunction_scratch_doubles(N, T)), dtype=torch.float64, device="cuda")
    ev = torch.zeros((2, 5), dtype=torch.float64, device="cuda")
    cnt = torch.zeros(2, dtype=torch.int64, device="cuda")
    sk = torch.zeros(N, dtype=torch.int32, device="cuda")
    _lib.check(_lib.lib().mpc_screen_conjunctions(yd.data_ptr(), N, T, _lib.addr(scale), D2, thr, scratch.data_ptr(),
                                                  ev.data_ptr(), 2, cnt.data_ptr(), sk.data_ptr(),
                                                  torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    assert int(cnt[0]) == len(ref) and int(cnt[1]) == 0


def test_nonfinite_samples_skipped(shell512):
    y, tf, const, D, T, thr, ref = shell512
    y = y.copy()
    y[5, 1, 10] = np.nan          # intervals 9 and 10 of satellite 5
    y[300, 3, T - 1] = np.inf     # the last interval of satellite 300
    y[7, 6, :] = np.nan           # the mass row is not read
    r = M.screen_conjunctions(y, tf, const, thr)
    want = np.zeros(512, np.int32)
    want[5], want[300] = 2, 1
    assert np.array_equal(r.skipped, want)
    keep = [e for e in ref if not ((5 in e[:2] and e[2] in (9, 10)) or (300 in e[:2] and e[2] == T - 2))]
    O.match(_rows(r), keep, D / (T - 1))


def test_device_form_matches_host_form(shell512):
    import torch
    y, tf, const, D, T, thr, ref = shell512
    h = M.screen_conjunctions(y, tf, const, thr)
    d = M.screen_conjunctions_device(torch.as_tensor(y).cuda(), torch.as_tensor(np.full(512, tf)).cuda(), const, thr,
                                     capacity=4)
    assert _dev_rows(d) == _rows(h)
    assert np.array_equal(d.skipped.cpu().numpy(), h.skipped) and d.n_flagged == h.n_flagged == 0
