"""Host logic of ragged batches (no GPU): per-satellite views of a padded result, packing of per-satellite arrays, the
node counts BatchedSCP derives from every satellite's horizon, and the sequence table it hands on."""
import numpy as np
import pytest

from mpconstellation_b200 import batch
from mpconstellation_b200.discretizer import pack_ragged
from mpconstellation_b200.scp import node_counts, sequence_table


def test_sat_views_of_a_ragged_result():
    K_sat = np.array([4, 2, 6], np.int32)
    N, Kmax = 3, 6
    soa = np.full((105, N * (Kmax - 1)), np.nan)
    for s in range(N):
        for k in range(K_sat[s] - 1):
            soa[:, s * (Kmax - 1) + k] = 1000 * s + k + np.arange(105) / 1000
    res = batch.DiscretizedBatch(soa, np.zeros((N, Kmax - 1), np.int32), N, Kmax, K_sat=K_sat)
    for s in range(N):
        A, Bp, Bn, Sig, xi = res.sat(s)
        n = K_sat[s] - 1
        assert A.shape == (n, 7, 7) and Bp.shape == (n, 7, 3) and Bn.shape == (n, 7, 3)
        assert Sig.shape == (7, n) and xi.shape == (7, n)
        assert np.isfinite(A).all() and np.shares_memory(Sig, soa)
        if n:
            assert A[n - 1, 0, 0] == 1000 * s + n - 1 and xi[6, 0] == 1000 * s + 104 / 1000
    A, Bp, Bn, Sig, xi = res.stacked()
    assert A.shape == (N, Kmax - 1, 7, 7) and np.isnan(A[1, 1:]).all() and np.isfinite(A[2]).all()


def test_pack_ragged_pads_with_nan_and_checks_shapes():
    rng = np.random.default_rng(0)
    xs = [rng.random((7, k)) for k in (5, 3, 8)]
    us = [rng.random((3, k)) for k in (5, 3, 8)]
    x, u, K = pack_ragged(xs, us)
    assert x.shape == (3, 7, 8) and u.shape == (3, 3, 8) and K.tolist() == [5, 3, 8] and K.dtype == np.int32
    assert np.array_equal(x[1, :, :3], xs[1]) and np.isnan(x[1, :, 3:]).all() and np.isnan(u[0, :, 5:]).all()
    with pytest.raises(ValueError):
        pack_ragged(xs, [us[0], us[2], us[1]])


def test_node_counts_use_the_reference_expression_and_reject_short_grids():
    assert node_counts(30, [1.4])[0] == int(30 * 1.4) == 42
    assert node_counts(30, [2.0, 1.0, 1.999]).tolist() == [60, 30, 59]
    with pytest.raises(ValueError):
        node_counts(30, [1.0, 0.05])
    with pytest.raises(ValueError):
        node_counts(1, [1.9])


def test_sequence_table_lengths():
    u = np.arange(2 * 3 * 5, dtype=float).reshape(2, 3, 5)
    tab, lens = sequence_table(u, np.array([5, 5]))
    assert lens is None and np.array_equal(tab, u)
    u2 = u.copy()
    u2[1, :, 3:] = np.nan
    tab, lens = sequence_table(u2, np.array([5, 3]))
    assert lens.tolist() == [5, 3] and np.isfinite(tab).all() and np.array_equal(tab[1, :, :3], u[1, :, :3])
    tab, lens = sequence_table([u[0, :, :4], u[1, :, :2]], None)
    assert lens.tolist() == [4, 2] and tab.shape == (2, 3, 4)


def test_counts_are_validated():
    with pytest.raises(ValueError):
        batch._counts([2, 1], 2, 5, "K")
    with pytest.raises(ValueError):
        batch._counts([2, 6], 2, 5, "K")
    with pytest.raises(ValueError):
        batch._counts([2, 3, 4], 2, 5, "K")
    assert batch._counts([2, 5], 2, 5, "K").dtype == np.int32
