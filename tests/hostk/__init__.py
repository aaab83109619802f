"""TEST INFRASTRUCTURE ONLY -- the CUDA kernel sources (mpconstellation_b200/csrc/*.cuh) compiled for the HOST with g++.

Purpose: `pytest -m "not gpu"` runs in a container without a GPU; this lets it exercise the arithmetic, the thread ->
(satellite, interval) indexing, the windowed launches and the status logic of the very source that nvcc compiles for
sm_100a, against the oracles and the reference fixtures.  The sources are copied into tests/hostk/_build/ with exactly
two lines replaced (the inline-PTX MUFU seeds of fast_rcp / fast_rsqrt -> a float-precision host seed; the Newton
refinement that follows is the kernel's own), CUDA keywords are defined away by include/hostk_shim.h, and the threads
of a launch run one after the other (every kernel is one independent thread per work unit).

This is a checker, like oracle/: nothing in mpconstellation_b200/ may import it, it is never what is measured or
shipped, and it says nothing about performance.
"""
import ctypes
import fcntl
import os
import re
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(os.path.dirname(os.path.dirname(HERE)), "mpconstellation_b200", "csrc")
BUILD = os.path.join(HERE, "_build")
SO = os.path.join(BUILD, "libmpc_hostk.so")
SOURCES = ["discretize_kernel.cuh", "discretize_adaptive_kernel.cuh", "discretize_default_kernel.cuh", "discretize_pair_kernel.cuh",
           "discretize_group_kernel.cuh",
           "discretize_drag_kernel.cuh", "propagate_kernel.cuh", "propagate_rk45_kernel.cuh", "constraint_terms_kernel.cuh"]
_SEEDS = [(r'asm\("rcp\.approx\.ftz\.f64 %0, %1;" : "=d"\(y\) : "d"\(a\)\);', "y = hostk_rcp_seed(a);"),
          (r'asm\("rsqrt\.approx\.ftz\.f64 %0, %1;" : "=d"\(y\) : "d"\(a\)\);', "y = hostk_rsqrt_seed(a);")]


def build(force=False, sanitize=False):
    """g++ build of the kernel sources.  sanitize=True: a second library with AddressSanitizer + UBSan instrumentation
    (tests/hostk/sanitize_driver.py runs it in a subprocess with the ASan runtime preloaded)."""
    if sanitize:
        return _build(os.path.join(BUILD, "libmpc_hostk_asan.so"), force,
                      ["-O1", "-g", "-fsanitize=address,undefined", "-fno-sanitize-recover=undefined", "-fno-omit-frame-pointer"])
    return _build(SO, force, ["-O2"])


def _build(SO, force, opt):
    srcs = [os.path.join(CSRC, s) for s in SOURCES] + [os.path.join(HERE, "hostk_main.cpp"),
                                                       os.path.join(HERE, "include", "hostk_shim.h"), __file__]

    def fresh():
        return os.path.exists(SO) and all(os.path.getmtime(SO) >= os.path.getmtime(s) for s in srcs)
    if not force and fresh():
        return SO
    os.makedirs(BUILD, exist_ok=True)
    # Several processes can ask for the library at once (the spawned ranks of tests/test_distributed_cpu.py on a fresh
    # checkout): one builds while the others wait, and the library is renamed into place, so that no process loads a
    # partly written file.
    with open(os.path.join(BUILD, ".lock"), "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        if not force and fresh():
            return SO
        n_sub = 0
        for s in SOURCES:
            text = open(os.path.join(CSRC, s)).read()
            for pat, rep in _SEEDS:
                text, n = re.subn(pat, rep, text)
                n_sub += n
            assert "asm(" not in text, f"{s}: inline PTX the host build does not know"
            open(os.path.join(BUILD, s), "w").write(text)
        assert n_sub == 3, "expected exactly the three MUFU seeds (fast_rcp, fast_rcp1, fast_rsqrt) to be replaced"
        tmp = f"{SO}.{os.getpid()}.tmp"
        cmd = ["g++"] + opt + ["-std=c++17", "-pthread", "-shared", "-fPIC", "-mfma", "-ffp-contract=fast", "-fno-math-errno",
               "-w", "-I", os.path.join(HERE, "include"), "-I", BUILD, "-o", tmp, os.path.join(HERE, "hostk_main.cpp")]
        res = subprocess.run(cmd, capture_output=True, text=True)
        if res.returncode != 0:
            raise RuntimeError("g++ failed:\n" + res.stdout + res.stderr)
        os.replace(tmp, SO)
    return SO


_lib = None


def lib():
    global _lib
    if _lib is None:
        _lib = ctypes.CDLL(build(sanitize=bool(os.environ.get("HOSTK_SANITIZE"))))
    return _lib


def _p(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


def _const8(const):
    return np.array([const.MU, const.R_E, const.J2, const.G0, const.ISP, const.S, const.R0, const.RHO], dtype=np.float64)


def discretize(x, u, tf, const, include_J2=False, n_sub=100, pair=True, k0=0, kc=-1, out=None, pitch=None, offset=0,
               status=None, km_ntot=0, km_soff=0, em=True):
    """The fixed-step kernels (discretize_pair_kernel / discretize_kernel) on host arrays x [N,7,K], u [N,3,K] -> SoA
    [105, pitch] + status, with the launch window (k0, kc) of the overlapped pass.  em: what the launcher sets by default
    (the pair kernel may take the 21-node form of the 101-node sums); em=False: every node evaluated."""
    x = np.ascontiguousarray(x, dtype=np.float64)
    u = np.ascontiguousarray(u, dtype=np.float64)
    N, _, K = x.shape
    tfv = np.ascontiguousarray(np.broadcast_to(np.asarray(tf, dtype=np.float64), (N,)))
    n_int = N * (K - 1)
    pitch = n_int if pitch is None else int(pitch)
    if out is None:
        out = np.full((105, pitch), np.nan)
    if status is None:
        status = np.full(n_int, -1, dtype=np.int32)
    c8 = _const8(const)
    lib().hostk_discretize(_p(x), _p(u), _p(tfv), _p(c8), int(include_J2), N, K, int(n_sub), int(pair), int(k0), int(kc),
                           _p(out), ctypes.c_longlong(pitch), ctypes.c_longlong(offset), _p(status),
                           ctypes.c_longlong(km_ntot), ctypes.c_longlong(km_soff), int(bool(em)))
    return out, status


def discretize_group(x, u, tf, const, include_J2=False, n_sub=100, extra_groups=0, em=True):
    """discretize_group_kernel (8 lanes per interval, the small-batch mapping) on host arrays -> SoA [105, N*(K-1)], status"""
    x = np.ascontiguousarray(x, dtype=np.float64)
    u = np.ascontiguousarray(u, dtype=np.float64)
    N, _, K = x.shape
    tfv = np.ascontiguousarray(np.broadcast_to(np.asarray(tf, dtype=np.float64), (N,)))
    n_int = N * (K - 1)
    out = np.full((105, n_int), np.nan)
    status = np.full(n_int, -1, dtype=np.int32)
    c8 = _const8(const)
    lib().hostk_discretize_group(_p(x), _p(u), _p(tfv), _p(c8), int(include_J2), N, K, int(n_sub), _p(out),
                                 ctypes.c_longlong(n_int), ctypes.c_longlong(0), _p(status), int(extra_groups), int(bool(em)))
    return out, status


def discretize_adaptive(x, u, tf, const, include_J2=False, rtol=1e-3, atol=1e-6, max_step=1e-2, v1=False):
    """the default-mode kernel (discretize_default_kernel); v1=True: the round-1 build (discretize_adaptive_kernel)"""
    x = np.ascontiguousarray(x, dtype=np.float64)
    u = np.ascontiguousarray(u, dtype=np.float64)
    N, _, K = x.shape
    tfv = np.ascontiguousarray(np.broadcast_to(np.asarray(tf, dtype=np.float64), (N,)))
    n_int = N * (K - 1)
    out = np.full((105, n_int), np.nan)
    status = np.full(n_int, -1, dtype=np.int32)
    nodes = np.zeros(n_int, dtype=np.int32)
    c8 = _const8(const)
    lib().hostk_discretize_adaptive(_p(x), _p(u), _p(tfv), _p(c8), int(include_J2), N, K, ctypes.c_double(rtol),
                                    ctypes.c_double(atol), ctypes.c_double(max_step), _p(out), ctypes.c_longlong(n_int),
                                    ctypes.c_longlong(0), _p(status), _p(nodes), int(v1))
    return out, status, nodes


def propagate(y0, tf, const, kind=0, thrust=(0.0, 0.0, 0.0), table=None, end_tau=1.0, include_drag=False, include_J2=False,
              T=100, n_sub=1, c_d=2.5, rho_atm=9.983e-13, seg_len=0):
    """propagate_kernel on host arrays y0 [N,7] -> y [N,7,T], u [N,3,T], status [N], progress words (seg_len > 0)."""
    y0 = np.ascontiguousarray(y0, dtype=np.float64)
    N = y0.shape[0]
    tfv = np.ascontiguousarray(np.broadcast_to(np.asarray(tf, dtype=np.float64), (N,)))
    y = np.full((N, 7, T), np.nan)
    uo = np.full((N, 3, T), np.nan)
    status = np.full(N, -1, dtype=np.int32)
    progress = np.zeros(64, dtype=np.uint32) if seg_len > 0 else None
    th = np.ascontiguousarray(np.asarray(thrust, dtype=np.float64))
    tab = None if table is None else np.ascontiguousarray(table, dtype=np.float64)
    c8 = _const8(const)
    lib().hostk_propagate(_p(y0), _p(tfv), _p(c8), int(include_J2), int(include_drag), ctypes.c_double(c_d),
                          ctypes.c_double(rho_atm), int(kind), _p(th), _p(tab), 0 if tab is None else tab.shape[-1],
                          int(tab is not None and tab.ndim == 3), ctypes.c_double(end_tau), N, int(T), int(n_sub), _p(y), _p(uo), _p(status), _p(progress),
                          int(seg_len))
    return y, uo, status, progress


def propagate_rk45(y0, tf, const, kind=0, thrust=(0.0, 0.0, 0.0), table=None, end_tau=1.0, include_drag=False,
                   include_J2=False, T=100, rtol=1e-3, atol=1e-6, max_step=1e-3, spec=True, lpw=32, c_d=2.5,
                   rho_atm=9.983e-13, seg_len=0):
    """propagate_rk45_kernel (the reference's solve_ivp call, replayed) on host arrays y0 [N,7] -> y [N,7,T], u [N,3,T],
    status [N], n_steps [N] (attempted steps), progress words (seg_len > 0).  end_tau: scalar or [N]."""
    y0 = np.ascontiguousarray(y0, dtype=np.float64)
    N = y0.shape[0]
    tfv = np.ascontiguousarray(np.broadcast_to(np.asarray(tf, dtype=np.float64), (N,)))
    y = np.full((N, 7, T), np.nan)
    uo = np.full((N, 3, T), np.nan)
    status = np.full(N, -1, dtype=np.int32)
    steps = np.zeros(N, dtype=np.int32)
    progress = np.zeros(64, dtype=np.uint32) if seg_len > 0 else None
    th = np.ascontiguousarray(np.asarray(thrust, dtype=np.float64))
    tab = None if table is None else np.ascontiguousarray(table, dtype=np.float64)
    et_arr = None
    if np.ndim(end_tau) != 0:
        et_arr = np.ascontiguousarray(end_tau, dtype=np.float64)
        end_tau = float(et_arr[0])
    c8 = _const8(const)
    D = ctypes.c_double
    lib().hostk_propagate_rk45(_p(y0), _p(tfv), _p(c8), int(include_J2), int(include_drag), D(c_d), D(rho_atm), int(kind),
                               _p(th), _p(tab), 0 if tab is None else tab.shape[-1], int(tab is not None and tab.ndim == 3),
                               D(end_tau), _p(et_arr), N, int(T), D(rtol), D(atol), D(max_step), int(spec), int(lpw),
                               _p(y), _p(uo), _p(status), _p(steps), _p(progress), int(seg_len))
    return y, uo, status, steps, progress


def discretize_drag(x, u, tf, const, drag, include_J2=False, n_sub=100, adaptive=None, c_d=2.5, rho_atm=9.983e-13, em=True):
    """The drag kernels (discretize_drag_kernel / the DRAG variant of the adaptive kernel); drag = (const.CD, rho_func
    value) or (const.CD, density model: the dict Discretizer fits for a radial rho_func / drho_func), as
    mpconstellation_b200.discretize_batch(disc_drag=...)."""
    x = np.ascontiguousarray(x, dtype=np.float64)
    u = np.ascontiguousarray(u, dtype=np.float64)
    N, _, K = x.shape
    tfv = np.ascontiguousarray(np.broadcast_to(np.asarray(tf, dtype=np.float64), (N,)))
    n_int = N * (K - 1)
    out = np.full((105, n_int), np.nan)
    status = np.full(n_int, -1, dtype=np.int32)
    nodes = np.zeros(n_int, dtype=np.int32)
    c8 = _const8(const)
    kf = 0.5 * c_d * const.S * (rho_atm / const.RHO)
    model = None
    if isinstance(drag[1], dict):
        m = drag[1]
        ka = 0.5 * drag[0] * const.S
        model = np.zeros(4 + 64)
        model[0:4] = m["r_mid"], m["r_ihalf"], len(m["rho_c"]), len(m["drho_c"])
        model[4:4 + len(m["rho_c"])] = m["rho_c"]
        model[36:36 + len(m["drho_c"])] = m["drho_c"]
    else:
        ka = 0.5 * drag[0] * const.S * drag[1]
    ad = adaptive if adaptive is not None else {}
    D = ctypes.c_double
    lib().hostk_discretize_drag(_p(x), _p(u), _p(tfv), _p(c8), int(include_J2), D(kf), D(ka), N, K, int(n_sub),
                                int(adaptive is not None), D(ad.get("rtol", 1e-3)), D(ad.get("atol", 1e-6)),
                                D(ad.get("max_step", 1e-2)), _p(out), ctypes.c_longlong(n_int), _p(status), _p(nodes),
                                int(bool(em)), _p(model) if model is not None else None)
    return out, status, nodes


def discretize_ugrid(x, u, tf, const, include_J2=False, n_sub=100, adaptive=None):
    """u [N,3,Ku] on its own grid (Ku != K): the GENU builds of discretize_kernel / discretize_adaptive_kernel."""
    x = np.ascontiguousarray(x, dtype=np.float64)
    u = np.ascontiguousarray(u, dtype=np.float64)
    N, _, K = x.shape
    tfv = np.ascontiguousarray(np.broadcast_to(np.asarray(tf, dtype=np.float64), (N,)))
    n_int = N * (K - 1)
    out = np.full((105, n_int), np.nan)
    status = np.full(n_int, -1, dtype=np.int32)
    nodes = np.zeros(n_int, dtype=np.int32)
    ad = adaptive if adaptive is not None else {}
    D = ctypes.c_double
    c8 = _const8(const)
    lib().hostk_discretize_ugrid(_p(x), _p(u), int(u.shape[2]), _p(tfv), _p(c8), int(include_J2), N, K,
                                 int(adaptive is not None), int(n_sub), D(ad.get("rtol", 1e-3)), D(ad.get("atol", 1e-6)),
                                 D(ad.get("max_step", 1e-2)), _p(out), ctypes.c_longlong(n_int), _p(status), _p(nodes))
    return out, status, nodes


def ref_node_input(us, f=1.0):
    """ref_node_input of the kernels at every node of the grid of us [3, Ku] -> [Ku, 3]"""
    us = np.ascontiguousarray(us, dtype=np.float64)
    Ku = us.shape[1]
    out = np.full((Ku, 3), np.nan)
    lib().hostk_ref_node_input(_p(us), Ku, ctypes.c_double(f), _p(out))
    return out


def constraint_terms(x, u, mu):
    """constraint_terms_kernel on host arrays x [N,7,K], u [N,3,Ku] -> rbar_hat [N,3,K-1], ubar_hat [N,3,Ku], fin [N,32]"""
    x = np.ascontiguousarray(x, dtype=np.float64)
    u = np.ascontiguousarray(u, dtype=np.float64)
    N, _, K = x.shape
    Ku = u.shape[2]
    rbar, ubar, fin = np.full((N, 3, K - 1), np.nan), np.full((N, 3, Ku), np.nan), np.full((N, 32), np.nan)
    lib().hostk_constraint_terms(_p(x), _p(u), N, K, Ku, ctypes.c_double(mu), _p(rbar), _p(ubar), _p(fin))
    return rbar, ubar, fin


def dynamics_jacobian(soa, n_sats, K):
    """dynamics_jacobian_kernel: CSR values [rows,16], indices [rows,16], rhs [rows] of the dynamics constraint"""
    soa = np.ascontiguousarray(soa, dtype=np.float64)
    rows = n_sats * 7 * (K - 1)
    values = np.full((rows, 16), np.nan)
    indices = np.full((rows, 16), -1, dtype=np.int64)
    rhs = np.full(rows, np.nan)
    lib().hostk_dynamics_jacobian(_p(soa), ctypes.c_longlong(soa.shape[1]), ctypes.c_longlong(0), n_sats, K, _p(values),
                                  _p(indices), _p(rhs))
    return values, indices, rhs


def stacked(soa, N, K):
    """SoA [105, N*(K-1)] -> (A, B_kp, B_kn, Sigma, xi) in the reference's shapes with a leading satellite axis."""
    n = K - 1
    v = soa.reshape(105, N, n)
    A = v[0:49].transpose(1, 2, 0).reshape(N, n, 7, 7)
    Bp = v[49:70].transpose(1, 2, 0).reshape(N, n, 7, 3)
    Bn = v[70:91].transpose(1, 2, 0).reshape(N, n, 7, 3)
    return A, Bp, Bn, v[91:98].transpose(1, 0, 2), v[98:105].transpose(1, 0, 2)
