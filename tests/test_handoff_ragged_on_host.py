"""The hand-off of a ragged batch to the convex subproblem in the host (g++) build of the kernel sources: constraint terms
and the sparse dynamics constraint with satellite s on its own K_s nodes, through ONE launch each.

Every satellite must come out bit for bit as the rectangular host launch of that satellite alone at K_s (the Jacobian's
column indices shifted by the start V_s of its variable block), the padding never written and never read, and the
per-satellite system must be the reference's dynamics_const_rule (optimizer.py:327-339) with satellite s's own tf_s.  A
second build under AddressSanitizer + UBSan memchecks the indexing on exactly sized buffers."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

import hostk
from conftest import GOLDEN, ROOT, synth_batch

HERE = os.path.join(ROOT, "tests", "hostk")
KEYS = {"rf_hat": (0, 3), "Vc": (3, 0), "DrVc": (4, 3), "DrVc_rbar": (7, 0), "Vt": (8, 0), "DrVt_DvVt": (9, 6),
        "DrVt_DvVt_bar": (15, 0), "Vr": (16, 0), "DrVr_DvVr": (17, 6), "DrVr_DvVr_bar": (23, 0), "Vn": (24, 0),
        "DrVn_DvVn": (25, 6), "DrVn_DvVn_bar": (31, 0)}


def _lib(sanitize=False):
    """libmpc_hostk_handoff[_asan].so, loaded (the _asan build only in a process that runs under the ASan runtime)"""
    return ctypes.CDLL(_build(sanitize))


def _build(sanitize=False):
    """libmpc_hostk_handoff[_asan].so: tests/hostk/handoff_main.cpp over the sources hostk.build() prepared"""
    hostk.build(sanitize=sanitize)
    so = os.path.join(hostk.BUILD, "libmpc_hostk_handoff_asan.so" if sanitize else "libmpc_hostk_handoff.so")
    src = os.path.join(HERE, "handoff_main.cpp")
    deps = [src, os.path.join(HERE, "hostk_main.cpp"), os.path.join(hostk.BUILD, "libmpc_hostk_asan.so" if sanitize else "libmpc_hostk.so")]
    if not (os.path.exists(so) and all(os.path.getmtime(so) >= os.path.getmtime(d) for d in deps)):
        opt = (["-O1", "-g", "-fsanitize=address,undefined", "-fno-sanitize-recover=undefined", "-fno-omit-frame-pointer"]
               if sanitize else ["-O2"])
        tmp = f"{so}.{os.getpid()}.tmp"
        cmd = ["g++"] + opt + ["-std=c++17", "-pthread", "-shared", "-fPIC", "-mfma", "-ffp-contract=fast", "-fno-math-errno",
                               "-w", "-I", os.path.join(HERE, "include"), "-I", hostk.BUILD, "-o", tmp, src]
        res = subprocess.run(cmd, capture_output=True, text=True)
        assert res.returncode == 0, res.stdout + res.stderr
        os.replace(tmp, so)
    return so


def _first(K_sat):
    return np.concatenate([[0], np.cumsum(np.asarray(K_sat, dtype=np.int64) - 1)]).astype(np.int64)


def constraint_terms_ragged(L, x, u, K_sat, mu):
    """one ragged launch over x [N,7,Kmax], u [N,3,Kmax] -> rbar_hat [N,3,Kmax-1], ubar_hat [N,3,Kmax], fin [N,32], all
    pre-filled with NaN"""
    x = np.ascontiguousarray(x, dtype=np.float64)
    u = np.ascontiguousarray(u, dtype=np.float64)
    N, _, Kmax = x.shape
    first = _first(K_sat)
    rbar, ubar, fin = np.full((N, 3, Kmax - 1), np.nan), np.full((N, 3, Kmax), np.nan), np.full((N, 32), np.nan)
    L.hostk_constraint_terms_ragged(hostk._p(x), hostk._p(u), N, Kmax, hostk._p(first), ctypes.c_double(mu), hostk._p(rbar),
                                    hostk._p(ubar), hostk._p(fin))
    return rbar, ubar, fin


def dynamics_jacobian_ragged(L, soa, N, Kmax, K_sat):
    """one ragged launch over the SoA [105, N (Kmax-1)] -> values [rows,16], indices [rows,16], rhs [rows]"""
    soa = np.ascontiguousarray(soa, dtype=np.float64)
    first = _first(K_sat)
    rows = 7 * int(first[-1])
    values, indices, rhs = np.full((rows, 16), np.nan), np.full((rows, 16), -1, dtype=np.int64), np.full(rows, np.nan)
    L.hostk_dynamics_jacobian_ragged(hostk._p(soa), ctypes.c_longlong(soa.shape[1]), ctypes.c_longlong(0), N, Kmax,
                                     hostk._p(first), hostk._p(values), hostk._p(indices), hostk._p(rhs))
    return values, indices, rhs


def _counts(N=24, Kmax=17, seed=11):
    K_sat = np.random.default_rng(seed).integers(2, Kmax + 1, N).astype(np.int32)
    K_sat[0], K_sat[5], K_sat[N - 1] = 2, Kmax, Kmax          # the smallest grid and Kmax itself, also last
    return K_sat


def _batch(const, K_sat, tf, seed=20240531):
    """x, u [N,.,Kmax]: satellite s sampled on its own K_s nodes (oracle propagation), padding poisoned with NaN; some input
    columns exactly zero, some tiny on both sides of the eps mask of ubar_hat"""
    N, Kmax = len(K_sat), int(max(K_sat))
    x = np.full((N, 7, Kmax), np.nan)
    u = np.full((N, 3, Kmax), np.nan)
    for k in np.unique(K_sat):
        _, xs, us = synth_batch(N, int(k), tf, const, seed=seed)
        idx = K_sat == k
        x[idx, :, :k], u[idx, :, :k] = xs[idx], us[idx]
    rng = np.random.default_rng(seed)
    for s, k in enumerate(K_sat):
        u[s, :, rng.integers(0, k)] = 0.0
        u[s, :, k - 1] = (1e-17 if s % 2 else 1e-15) * rng.standard_normal(3)      # the last column, both sides of eps
    return x, u


def _soa(const, x, u, K_sat, tf):
    """the ragged discretization result: every satellite's own rectangular host launch at K_s in its column block, NaN in
    the padding (mpc_discretize_batch_ragged gives these bits, tests/test_ragged_kernel_source_on_host.py)"""
    N, _, Kmax = x.shape
    soa = np.full((105, N * (Kmax - 1)), np.nan)
    for s, k in enumerate(K_sat.tolist()):
        soa[:, s * (Kmax - 1):s * (Kmax - 1) + k - 1] = hostk.discretize(x[s:s + 1, :, :k], u[s:s + 1, :, :k], tf[s], const,
                                                                         n_sub=10)[0]
    return soa


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.int64)


def test_ragged_constraint_terms_are_the_per_satellite_launches_bit_for_bit(const):
    from oracle import mpc_oracle as O
    K_sat = _counts()
    x, u = _batch(const, K_sat, 1.3)
    rbar, ubar, fin = constraint_terms_ragged(_lib(), x, u, K_sat, const.MU)
    assert np.isnan(ubar).any() and (ubar == 0).any()         # the inverted mask: 0/0 where |u| <= eps, 0 elsewhere
    for s, k in enumerate(K_sat.tolist()):
        rr, ur, fr = hostk.constraint_terms(x[s:s + 1, :, :k], u[s:s + 1, :, :k], const.MU)
        assert np.array_equal(_bits(rbar[s, :, :k - 1]), _bits(rr[0])) and np.array_equal(_bits(ubar[s, :, :k]), _bits(ur[0]))
        assert np.array_equal(_bits(fin[s]), _bits(fr[0])), s
        assert np.isnan(rbar[s, :, k - 1:]).all() and np.isnan(ubar[s, :, k:]).all()
        ref = O.constraint_terms(x[s, :, :k], u[s, :, :k], const.MU)
        np.testing.assert_array_equal(rbar[s, :, :k - 1], ref["rbar_hat"])
        np.testing.assert_array_equal(ubar[s, :, :k], ref["ubar_hat"])
        for key, (off, ln) in KEYS.items():
            got = fin[s, off:off + ln] if ln else fin[s, off]
            want = np.asarray(ref[key])
            assert np.max(np.abs(got - want)) <= 5e-13 * max(np.max(np.abs(want)), 1.0), (s, key)
    assert np.isfinite(fin).all()


def test_ragged_jacobian_is_block_diagonal_with_one_final_time_per_satellite(const):
    from mpconstellation_b200.batch import DiscretizedBatch
    from mpconstellation_b200.constraints import DynamicsJacobian
    from mpconstellation_b200.scp import Linearization
    K_sat = _counts()
    N, Kmax = len(K_sat), int(K_sat.max())
    tf = np.linspace(1.0, 2.0, N)
    x, u = _batch(const, K_sat, 1.3)
    soa = _soa(const, x, u, K_sat, tf)
    values, indices, rhs = dynamics_jacobian_ragged(_lib(), soa, N, Kmax, K_sat)
    jac = DynamicsJacobian(values.ravel(), indices.ravel(), rhs, N, Kmax, K_sat=K_sat)
    first = _first(K_sat)
    assert jac.rows == 7 * first[-1] == values.shape[0] and jac.cols == 17 * (first[-1] + N) + N
    # every value finite although the SoA's padding columns are NaN: the padding is never read
    assert np.isfinite(values).all() and np.isfinite(rhs).all()
    assert np.all(np.diff(indices, axis=1) > 0) and indices.min() == 0 and indices.max() == jac.cols - 1
    for s, k in enumerate(K_sat):
        rv, ri, rr = hostk.dynamics_jacobian(soa[:, s * (Kmax - 1):s * (Kmax - 1) + k - 1], 1, int(k))
        rows, cols = jac.block(s)
        V = 17 * (first[s] + s) + s
        assert rows == slice(7 * first[s], 7 * first[s + 1]) and cols == slice(V, V + 17 * k + 1)
        assert np.array_equal(_bits(values[rows]), _bits(rv)) and np.array_equal(_bits(rhs[rows]), _bits(rr))
        assert np.array_equal(indices[rows], ri + V)
    # J z - rhs against the pyomo rule, written out per satellite, with every satellite's own tf_s
    lin = Linearization(x, u, tf, DiscretizedBatch(soa, np.zeros((N, Kmax - 1), np.int32), N, Kmax, K_sat=K_sat), K_sat)
    rng = np.random.default_rng(3)
    xz = [rng.standard_normal((7, k)) for k in K_sat]
    uz = [rng.standard_normal((3, k)) for k in K_sat]
    nz = [rng.standard_normal((7, k)) for k in K_sat]
    tz = 1.0 + rng.random(N)
    z = jac.pack(xz, uz, nz, tz)
    assert z.shape == (jac.cols,)
    res = jac.residual(z)
    for s in range(N):
        want = lin.dynamics_residual(s, xz[s], uz[s], tz[s], nu=nz[s])
        assert res[s].shape == (7, K_sat[s] - 1)
        assert np.max(np.abs(res[s] - want)) < 1e-12 * max(1.0, np.max(np.abs(want))), s
    J = jac.to_scipy()
    assert J.shape == (jac.rows, jac.cols) and J.nnz == 16 * jac.rows
    assert np.allclose(J @ z - rhs, np.concatenate([r.ravel() for r in res]), rtol=0, atol=1e-12)
    for s in (0, 5, N - 1):                                   # no coupling between satellites: J is block-diagonal
        rows, cols = jac.block(s)
        assert J[rows][:, :cols.start].nnz == 0 and J[rows][:, cols.stop:].nnz == 0
    # on the reference point with nu = the first-order-hold defect the constraint holds; the padded arrays pack alike
    nu0 = np.zeros((N, 7, Kmax))
    for s, k in enumerate(K_sat):
        nu0[s, :, :k - 1] = lin.dynamics_residual(s, x[s, :, :k], u[s, :, :k], tf[s])
    assert max(np.max(np.abs(r)) for r in jac.residual(jac.pack(x, u, nu0, tf))) < 1e-13


def test_equal_counts_are_the_rectangular_numbering_per_satellite(const):
    """all K_s = K: the per-satellite system is the rectangular one with one tf column inserted after every satellite"""
    N, K = 4, 6
    K_sat = np.full(N, K, np.int32)
    x, u = _batch(const, K_sat, 0.9)
    soa = _soa(const, x, u, K_sat, np.full(N, 0.9))
    v, c, r = dynamics_jacobian_ragged(_lib(), soa, N, K, K_sat)
    rv, rc, rr = hostk.dynamics_jacobian(soa, N, K)
    assert np.array_equal(_bits(v), _bits(rv)) and np.array_equal(_bits(r), _bits(rr))
    s = np.arange(7 * N * (K - 1)) // (7 * (K - 1))
    assert not np.array_equal(c, rc)
    for sv in range(N):          # rectangular x | u | nu blocks of all satellites -> satellite sv's own [x u nu tf] block
        own = c[s == sv] - (17 * K + 1) * sv
        glob = rc[s == sv]
        x_part, u_part, nu_part = glob < 7 * N * K, (glob >= 7 * N * K) & (glob < 10 * N * K), glob >= 10 * N * K
        assert np.array_equal(own[x_part], glob[x_part] - 7 * K * sv)
        assert np.array_equal(own[u_part], glob[u_part] - 7 * N * K - 3 * K * sv + 7 * K)
        assert np.array_equal(own[nu_part & (glob < 17 * N * K)], glob[nu_part & (glob < 17 * N * K)] - 10 * N * K - 7 * K * sv + 10 * K)
        assert (own[glob == 17 * N * K] == 17 * K).all()


def test_ragged_lists_are_checked_before_any_launch(const):
    from mpconstellation_b200.constraints import get_constraint_terms
    x = [np.zeros((7, 5)), np.zeros((7, 8))]
    with pytest.raises(ValueError):
        get_constraint_terms(x, [np.zeros((3, 5)), np.zeros((3, 7))], const)


def test_ragged_handoff_kernels_under_address_sanitizer(const):
    asan = subprocess.run(["gcc", "-print-file-name=libasan.so"], capture_output=True, text=True).stdout.strip()
    if not os.path.isabs(asan) or not os.path.exists(asan):
        pytest.skip("no AddressSanitizer runtime next to this gcc")
    _build(sanitize=True)
    code = (
        "import sys, numpy as np\n"
        f"sys.path.insert(0, {os.path.join(ROOT, 'tests')!r}); sys.path.insert(0, {ROOT!r})\n"
        "import test_handoff_ragged_on_host as T\n"
        "from oracle.mpc_oracle import OracleConstants\n"
        f"const = OracleConstants(*np.load({os.path.join(GOLDEN, 'discretize.npz')!r})['const'])\n"
        "L = T._lib(sanitize=True)\n"
        "for K_sat in ([2, 9, 3], [9], [2, 2], [4, 9, 2, 9, 6], [2] * 33):\n"
        "    K_sat = np.array(K_sat, np.int32)\n"
        "    N, Kmax = len(K_sat), int(K_sat.max())\n"
        "    x, u = T._batch(const, K_sat, 0.7)\n"
        "    T.constraint_terms_ragged(L, x, u, K_sat, const.MU)\n"
        "    soa = np.full((105, N * (Kmax - 1)), 0.5)\n"
        "    v, c, r = T.dynamics_jacobian_ragged(L, soa, N, Kmax, K_sat)\n"
        "    assert np.isfinite(v).all() and c.min() >= 0\n"
        "print('ragged hand-off launches clean')\n")
    env = dict(os.environ, HOSTK_SANITIZE="1", LD_PRELOAD=asan, ASAN_OPTIONS="detect_leaks=0:halt_on_error=1")
    res = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, timeout=900)
    assert res.returncode == 0 and "ragged hand-off launches clean" in res.stdout, res.stdout[-2000:] + res.stderr[-4000:]
    assert "AddressSanitizer" not in res.stderr and "runtime error" not in res.stderr
