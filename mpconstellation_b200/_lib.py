"""ctypes binding of csrc/libmpc_b200.so (C-ABI: include/mpc_b200.h).

There is no CPU fallback: if the shared library is missing or no CUDA device is usable, the
functions here raise.  `build()` compiles the library in-tree with nvcc for sm_100a.
"""
import ctypes
import os
import subprocess
import sys
import weakref

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
SO_PATH = os.path.join(CSRC, "libmpc_b200.so")
# the drag-branch kernels, the per-satellite-constants kernels, the multi-destination ragged kernels, the RK45 replay
# under an altitude-dependent atmosphere, the default quadrature mode with RK23 and the conjunction screening have a
# translation unit each
SOURCES = ["mpc_b200.cu", "mpc_b200_drag.cu", "mpc_b200_units.cu", "mpc_b200_shard.cu", "mpc_b200_atmo.cu", "mpc_b200_rk23.cu",
           "mpc_b200_conj.cu"]
HEADERS = ["discretize_kernel.cuh", "discretize_adaptive_kernel.cuh", "discretize_default_kernel.cuh", "propagate_kernel.cuh", "propagate_rk45_kernel.cuh", "discretize_group_kernel.cuh", "constraint_terms_kernel.cuh", "discretize_drag_kernel.cuh", "discretize_pair_kernel.cuh", "mpc_b200_drag.h", "mpc_b200_units.h", "mpc_b200_shard.h", "mpc_b200_atmo.h", "discretize_rk23_kernel.cuh", "mpc_b200_rk23.h", "conjunction_kernel.cuh", "mpc_b200_conj.h", os.path.join("..", "..", "include", "mpc_b200.h")]
# No -split-compile: with it nvcc partitions the module for parallel compilation and the register allocation of the
# 250-register kernels comes out differently from build to build (the same source gave discretize_default_kernel 253
# registers / 296 B of stack in one build and 255 / 536 B in the next: 1.366 vs 1.390 ms on BASELINE configs[2];
# profiles/r02_zz_ab_default_*.log).  Unsplit, every kernel compiles as it does on its own: 1.327 ms.  The two
# translation units are compiled side by side instead (build()).
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC"]

MPC_OUT_ROWS = 105
ROW_A, ROW_BP, ROW_BN, ROW_SIGMA, ROW_XI = 0, 49, 70, 91, 98
CTRL_ZERO, CTRL_CONSTANT, CTRL_TANGENTIAL, CTRL_SEQUENCE = 0, 1, 2, 3
ST_OK, ST_MASS, ST_NONFINITE, ST_STEP, ST_ATMO = 0, 1, 2, 3, 4
FINAL_TERMS = 32
# key -> (offset, length) inside the per-satellite terminal block (include/mpc_b200.h MPC_FT_*); length 0 = scalar
FINAL_TERM_LAYOUT = {"rf_hat": (0, 3), "Vc": (3, 0), "DrVc": (4, 3), "DrVc_rbar": (7, 0), "Vt": (8, 0),
                     "DrVt_DvVt": (9, 6), "DrVt_DvVt_bar": (15, 0), "Vr": (16, 0), "DrVr_DvVr": (17, 6),
                     "DrVr_DvVr_bar": (23, 0), "Vn": (24, 0), "DrVn_DvVn": (25, 6), "DrVn_DvVn_bar": (31, 0)}
E_INVALID, E_CUDA, E_UNSUPPORTED, E_NOMEM = -1, -2, -3, -4


class MpcParams(ctypes.Structure):
    _fields_ = [(n, ctypes.c_double) for n in
                ("mu", "r_e", "j2", "g0", "isp", "s_area", "r0", "rho", "c_d", "rho_atm", "disc_cd", "disc_rho")] + \
               [("include_j2", ctypes.c_int32), ("include_drag", ctypes.c_int32),
                ("disc_n_rho", ctypes.c_int32), ("disc_n_drho", ctypes.c_int32),
                ("disc_r_mid", ctypes.c_double), ("disc_r_ihalf", ctypes.c_double),
                ("disc_rho_cheb", ctypes.c_double * 32), ("disc_drho_cheb", ctypes.c_double * 32)]


RHO_CHEB = 32


class MpcSatConsts(ctypes.Structure):
    """mpc_sat_consts: the per-scale fields of one satellite's normalized Constants"""
    _fields_ = [(n, ctypes.c_double) for n in ("mu", "r_e", "j2", "g0", "isp", "s_area", "rho")]


SAT_SCRATCH_DOUBLES = 8    # MPC_SAT_SCRATCH_DOUBLES


class MpcAtmosphere(ctypes.Structure):
    """mpc_atmosphere: log rho as a Chebyshev series in log h over [h_min, h_max] (atmosphere.fit_atmosphere)"""
    _fields_ = [("h_min", ctypes.c_double), ("h_max", ctypes.c_double), ("r_earth", ctypes.c_double),
                ("n", ctypes.c_int32), ("reserved", ctypes.c_int32), ("coef", ctypes.c_double * 32)]


class MpcController(ctypes.Structure):
    _fields_ = [("kind", ctypes.c_int32), ("table_len", ctypes.c_int32), ("table_per_sat", ctypes.c_int32),
                ("reserved", ctypes.c_int32), ("thrust", ctypes.c_double * 3), ("end_tau", ctypes.c_double),
                ("table", ctypes.c_void_p), ("end_tau_per_sat", ctypes.c_void_p)]


class MpcGatherOpts(ctypes.Structure):
    _fields_ = [("layout", ctypes.c_int32), ("skip_const", ctypes.c_int32), ("stagger_phases", ctypes.c_int32),
                ("reserved", ctypes.c_int32), ("n_sats_total", ctypes.c_int64), ("sat_offset", ctypes.c_int64)]


LAYOUT_SAT_MAJOR, LAYOUT_K_MAJOR = 0, 1

# mpc_conjunction, one close approach (include/mpc_b200.h)
CONJUNCTION_DTYPE = np.dtype([("i", "<i4"), ("j", "<i4"), ("k", "<i4"), ("flags", "<i4"), ("t_ca", "<f8"), ("d_min", "<f8"),
                              ("v_rel", "<f8")])
CONJ_FLAG_DEPTH = 1     # MPC_CONJ_FLAG_DEPTH


class MpcError(RuntimeError):
    def __init__(self, code, text):
        super().__init__(f"libmpc_b200 error {code}: {text}")
        self.code = code


def needs_build():
    if not os.path.exists(SO_PATH):
        return True
    t = os.path.getmtime(SO_PATH)
    deps = [os.path.join(CSRC, s) for s in SOURCES + HEADERS]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    """Compile csrc/*.cu into csrc/libmpc_b200.so for sm_100a (nvcc cross-compiles without a GPU)."""
    if not force and not needs_build():
        return SO_PATH
    import concurrent.futures
    objs = [os.path.join(CSRC, os.path.splitext(src)[0] + ".o") for src in SOURCES]

    def compile_one(src, obj):
        cmd = ["nvcc"] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", "-o", obj, os.path.join(CSRC, src)]
        return subprocess.run(cmd, capture_output=True, text=True)

    with concurrent.futures.ThreadPoolExecutor(len(SOURCES)) as ex:
        results = list(ex.map(compile_one, SOURCES, objs))
    for res in results:
        if res.returncode != 0:
            raise RuntimeError("nvcc failed:\n" + res.stdout + res.stderr)
        if verbose:
            sys.stderr.write(res.stderr)
    res = subprocess.run(["nvcc", "-shared", "-o", SO_PATH] + objs, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("nvcc (link) failed:\n" + res.stdout + res.stderr)
    for obj in objs:
        os.remove(obj)
    return SO_PATH


_lib = None

_DP = ctypes.c_void_p  # all array pointers are passed as raw addresses


def lib():
    """Loads the shared library (once).  Raises ImportError when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(SO_PATH):
        raise ImportError(f"{SO_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                          "(there is no CPU fallback)")
    L = ctypes.CDLL(SO_PATH)
    i, i64, vp = ctypes.c_int, ctypes.c_int64, ctypes.c_void_p
    pp, pc = ctypes.POINTER(MpcParams), ctypes.POINTER(MpcController)
    L.mpc_version.restype = i
    L.mpc_last_error.restype = ctypes.c_char_p
    L.mpc_device_count.restype = i
    L.mpc_device_info.argtypes = [i, ctypes.c_char_p, i, ctypes.POINTER(i), ctypes.POINTER(i), ctypes.POINTER(i)]
    L.mpc_launch_count.restype = i64
    L.mpc_discretize_batch.argtypes = [_DP, _DP, _DP, pp, i, i, i, _DP, i64, i64, _DP, vp]
    L.mpc_discretize_batch_multi.argtypes = [_DP, _DP, _DP, pp, i, i, i, ctypes.POINTER(ctypes.c_void_p), i, i64, i64, _DP, vp]
    d = ctypes.c_double
    L.mpc_discretize_batch_adaptive.argtypes = [_DP, _DP, _DP, pp, i, i, d, d, d, _DP, i64, i64, _DP, _DP, vp]
    L.mpc_discretize_batch_adaptive_host.argtypes = [vp, _DP, _DP, _DP, pp, i, i, d, d, d, _DP, _DP, _DP]
    L.mpc_discretize_batch_ugrid.argtypes = [_DP, _DP, i, _DP, pp, i, i, i, i, d, d, d, _DP, i64, i64, _DP, _DP, vp]
    L.mpc_discretize_batch_ugrid_host.argtypes = [vp, _DP, _DP, i, _DP, pp, i, i, i, i, d, d, d, _DP, _DP, _DP]
    L.mpc_propagate_batch.argtypes = [_DP, _DP, pp, pc, i, i, i, _DP, _DP, _DP, vp]
    L.mpc_propagate_batch_rk45.argtypes = [_DP, _DP, pp, pc, i, i, d, d, d, _DP, _DP, _DP, _DP, vp]
    L.mpc_propagate_batch_rk45_host.argtypes = [vp, _DP, _DP, pp, pc, i, i, d, d, d, _DP, _DP, _DP, _DP]
    L.mpc_discretize_batch_ragged.argtypes = [_DP, _DP, _DP, pp, i, i, _DP, _DP, i, i, d, d, d, _DP, i64, i64, _DP, _DP, vp]
    L.mpc_discretize_batch_ragged_host.argtypes = [vp, _DP, _DP, _DP, pp, i, i, _DP, i, i, d, d, d, _DP, _DP, _DP]
    L.mpc_propagate_batch_rk45_ragged.argtypes = [_DP, _DP, pp, pc, i, i, _DP, _DP, d, d, d, _DP, _DP, _DP, _DP, vp]
    L.mpc_propagate_batch_rk45_ragged_host.argtypes = [vp, _DP, _DP, pp, pc, i, i, _DP, _DP, d, d, d, _DP, _DP, _DP, _DP]
    L.mpc_ctx_create.argtypes = [i, ctypes.POINTER(vp)]
    L.mpc_ctx_destroy.argtypes = [vp]
    L.mpc_host_alloc.argtypes = [ctypes.c_size_t]
    L.mpc_host_alloc.restype = vp
    L.mpc_host_free.argtypes = [vp]
    L.mpc_host_free.restype = None
    L.mpc_discretize_batch_host.argtypes = [vp, _DP, _DP, _DP, pp, i, i, i, _DP, _DP]
    L.mpc_propagate_batch_host.argtypes = [vp, _DP, _DP, pp, pc, i, i, i, _DP, _DP, _DP]
    L.mpc_propagate_discretize_host.argtypes = [vp, _DP, _DP, pp, pp, pc, i, i, i, i, _DP, _DP, _DP, _DP]
    L.mpc_propagate_discretize_host_layout.argtypes = [vp, _DP, _DP, pp, pp, pc, i, i, i, i, _DP, _DP, _DP, _DP, i]
    L.mpc_propagate_discretize.argtypes = [vp, _DP, _DP, pp, pp, pc, i, i, i, i, _DP, _DP, _DP, i64, i64, _DP, _DP, i, vp]
    L.mpc_propagate_discretize_multi.argtypes = [vp, _DP, _DP, pp, pp, pc, i, i, i, i, _DP, _DP, ctypes.POINTER(ctypes.c_void_p), i, i64, i64, _DP, _DP, i, vp]
    pg = ctypes.POINTER(MpcGatherOpts)
    L.mpc_discretize_batch_gather.argtypes = [_DP, _DP, _DP, pp, i, i, i, ctypes.POINTER(ctypes.c_void_p), i, pg, _DP, vp]
    L.mpc_propagate_discretize_gather.argtypes = [vp, _DP, _DP, pp, pp, pc, i, i, i, i, _DP, _DP, ctypes.POINTER(ctypes.c_void_p), i, pg, _DP, _DP, i, vp]
    L.mpc_discretize_batch_push.argtypes = [vp, _DP, _DP, _DP, pp, i, i, i, ctypes.POINTER(ctypes.c_void_p), i, i64, i64, _DP, i, i, vp]
    L.mpc_fill_const_rows.argtypes = [_DP, i64, vp]
    L.mpc_dynamics_jacobian.argtypes = [_DP, i64, i64, i, i, _DP, _DP, _DP, vp]
    L.mpc_constraint_terms.argtypes = [_DP, _DP, i, i, i, d, _DP, _DP, _DP, vp]
    L.mpc_constraint_terms_host.argtypes = [vp, _DP, _DP, i, i, i, d, _DP, _DP, _DP]
    L.mpc_constraint_terms_ragged.argtypes = [_DP, _DP, i, i, _DP, _DP, d, _DP, _DP, _DP, vp]
    L.mpc_constraint_terms_ragged_host.argtypes = [vp, _DP, _DP, i, i, _DP, d, _DP, _DP, _DP]
    L.mpc_dynamics_jacobian_ragged.argtypes = [_DP, i64, i64, i, i, _DP, _DP, _DP, _DP, _DP, vp]
    L.mpc_discretize_batch_units.argtypes = [_DP, _DP, _DP, pp, _DP, i, i, _DP, _DP, _DP, i, i, d, d, d, _DP, i64, i64, _DP, _DP, vp]
    L.mpc_discretize_batch_units_host.argtypes = [vp, _DP, _DP, _DP, pp, _DP, i, i, _DP, i, i, d, d, d, _DP, _DP, _DP]
    L.mpc_discretize_batch_ragged_gather.argtypes = [_DP, _DP, _DP, pp, _DP, i, i, _DP, _DP, _DP, i, i, d, d, d,
                                                     ctypes.POINTER(ctypes.c_void_p), i, i64, i64, i, _DP, _DP, vp]
    L.mpc_propagate_batch_rk45_units.argtypes = [_DP, _DP, pp, _DP, pc, i, i, _DP, _DP, _DP, d, d, d, _DP, _DP, _DP, _DP, vp]
    L.mpc_propagate_batch_rk45_units_host.argtypes = [vp, _DP, _DP, pp, _DP, pc, i, i, _DP, _DP, d, d, d, _DP, _DP, _DP, _DP]
    L.mpc_discretize_batch_rk23.argtypes = [_DP, _DP, _DP, pp, _DP, i, i, _DP, _DP, _DP, d, d, d, _DP, i64, i64, _DP, _DP, vp]
    L.mpc_discretize_batch_rk23_host.argtypes = [vp, _DP, _DP, _DP, pp, _DP, i, i, _DP, d, d, d, _DP, _DP, _DP]
    pa = ctypes.POINTER(MpcAtmosphere)
    L.mpc_propagate_batch_rk45_atmo.argtypes = [_DP, _DP, pp, _DP, pc, i, i, _DP, _DP, _DP, d, d, d, _DP, _DP, _DP, _DP, pa, vp]
    L.mpc_propagate_batch_rk45_atmo_host.argtypes = [vp, _DP, _DP, pp, _DP, pc, i, i, _DP, _DP, d, d, d, _DP, _DP, _DP, _DP, pa]
    L.mpc_constraint_terms_units.argtypes = [_DP, _DP, i, i, _DP, _DP, _DP, _DP, _DP, _DP, _DP, vp]
    L.mpc_constraint_terms_units_host.argtypes = [vp, _DP, _DP, i, i, _DP, _DP, _DP, _DP, _DP]
    L.mpc_conjunction_scratch_doubles.argtypes = [i, i]
    L.mpc_conjunction_scratch_doubles.restype = i64
    L.mpc_screen_conjunctions.argtypes = [_DP, i, i, _DP, d, d, _DP, _DP, i64, _DP, _DP, vp]
    L.mpc_screen_conjunctions_host.argtypes = [vp, _DP, i, i, _DP, d, d, _DP, i64, ctypes.POINTER(i64), ctypes.POINTER(i64), _DP]
    L.mpc_fp64_peak_probe.argtypes = [i, i, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_double)]
    L.mpc_set_gather_tuning.argtypes = [i, i]
    L.mpc_set_gather_tuning.restype = i
    L.mpc_set_tuning.argtypes = [i]
    L.mpc_set_tuning.restype = i
    for name in ("mpc_propagate_batch_rk45_atmo", "mpc_propagate_batch_rk45_atmo_host", "mpc_propagate_discretize_host_layout", "mpc_discretize_batch_gather", "mpc_propagate_discretize_gather", "mpc_propagate_batch_rk45", "mpc_propagate_batch_rk45_host", "mpc_device_info", "mpc_discretize_batch", "mpc_discretize_batch_multi", "mpc_propagate_batch",
                 "mpc_discretize_batch_adaptive", "mpc_discretize_batch_adaptive_host",
                 "mpc_discretize_batch_ugrid", "mpc_discretize_batch_ugrid_host",
                 "mpc_ctx_create", "mpc_ctx_destroy", "mpc_discretize_batch_host", "mpc_propagate_batch_host",
                 "mpc_propagate_discretize_host", "mpc_propagate_discretize", "mpc_propagate_discretize_multi", "mpc_fp64_peak_probe", "mpc_constraint_terms",
                 "mpc_constraint_terms_host", "mpc_discretize_batch_push", "mpc_fill_const_rows", "mpc_dynamics_jacobian",
                 "mpc_constraint_terms_ragged", "mpc_constraint_terms_ragged_host", "mpc_dynamics_jacobian_ragged",
                 "mpc_discretize_batch_units", "mpc_discretize_batch_units_host", "mpc_propagate_batch_rk45_units",
                 "mpc_propagate_batch_rk45_units_host", "mpc_discretize_batch_ragged_gather", "mpc_constraint_terms_units", "mpc_constraint_terms_units_host",
                 "mpc_discretize_batch_rk23", "mpc_discretize_batch_rk23_host", "mpc_screen_conjunctions",
                 "mpc_screen_conjunctions_host"):
        getattr(L, name).restype = i
    _lib = L
    return L


EXPORTED_SYMBOLS = [
    "mpc_version", "mpc_last_error", "mpc_device_count", "mpc_device_info", "mpc_launch_count",
    "mpc_discretize_batch", "mpc_discretize_batch_multi", "mpc_discretize_batch_adaptive", "mpc_discretize_batch_ugrid", "mpc_propagate_batch",
    "mpc_propagate_batch_rk45", "mpc_propagate_batch_rk45_host", "mpc_discretize_batch_gather", "mpc_propagate_discretize_gather",
    "mpc_propagate_discretize_host_layout",
    "mpc_discretize_batch_ragged", "mpc_discretize_batch_ragged_host", "mpc_propagate_batch_rk45_ragged",
    "mpc_propagate_batch_rk45_ragged_host",
    "mpc_ctx_create", "mpc_ctx_destroy", "mpc_host_alloc", "mpc_host_free",
    "mpc_discretize_batch_host", "mpc_discretize_batch_adaptive_host", "mpc_discretize_batch_ugrid_host", "mpc_propagate_batch_host", "mpc_propagate_discretize_host", "mpc_propagate_discretize", "mpc_propagate_discretize_multi",
    "mpc_constraint_terms", "mpc_constraint_terms_host", "mpc_discretize_batch_push", "mpc_fill_const_rows",
    "mpc_dynamics_jacobian",
    "mpc_constraint_terms_ragged", "mpc_constraint_terms_ragged_host", "mpc_dynamics_jacobian_ragged",
    "mpc_discretize_batch_units", "mpc_discretize_batch_units_host", "mpc_propagate_batch_rk45_units",
    "mpc_propagate_batch_rk45_units_host", "mpc_constraint_terms_units", "mpc_constraint_terms_units_host",
    "mpc_discretize_batch_ragged_gather", "mpc_fp64_peak_probe", "mpc_set_tuning", "mpc_set_gather_tuning",
    "mpc_propagate_batch_rk45_atmo", "mpc_propagate_batch_rk45_atmo_host",
    "mpc_discretize_batch_rk23", "mpc_discretize_batch_rk23_host",
    "mpc_conjunction_scratch_doubles", "mpc_screen_conjunctions", "mpc_screen_conjunctions_host",
]


SAT_CONST_FIELDS = ("MU", "R_E", "J2", "G0", "ISP", "S", "RHO")   # what mpc_sat_consts carries, in its order


def sat_consts(const, n):
    """const: one Constants bag or a sequence of n of them -> (None, one bag) when every satellite has the same seven
    per-scale values bit for bit (the single-constant launches apply), else (mpc_sat_consts [n], None).  A length other
    than n, or a bag without one of the seven attributes, raises ValueError."""
    if hasattr(const, "MU"):             # one bag
        return None, const
    try:
        const = list(const)              # any sequence of bags: list, tuple, numpy object array, ...
    except TypeError:
        raise ValueError(f"const must be a Constants bag or a sequence of {n} of them, got {type(const).__name__}") from None
    if len(const) != n:
        raise ValueError(f"per-satellite constants: expected {n} Constants, got {len(const)}")
    rows = []
    for s, c in enumerate(const):
        try:
            rows.append([float(getattr(c, f)) for f in SAT_CONST_FIELDS])
        except AttributeError as e:
            raise ValueError(f"per-satellite constants: const[{s}] has no attribute {e.name!r}") from None
    vals = np.array(rows, dtype=np.float64).reshape(n, 7)
    if n == 0 or (vals.view(np.uint64) == vals[0].view(np.uint64)).all():
        return None, (const[0] if n else None)
    return (MpcSatConsts * n).from_buffer_copy(np.ascontiguousarray(vals)), None


def check(rc):
    if rc != 0:
        raise MpcError(rc, lib().mpc_last_error().decode("utf-8", "replace"))


def require_gpu():
    if lib().mpc_device_count() < 1:
        raise RuntimeError("mpconstellation_b200 needs a CUDA device (sm_100a); none is visible and there is no CPU fallback")


def make_params(const, include_J2=False, include_drag=False, c_d=2.5, rho_atm=9.983e-13, disc_drag=None):
    """Pack a reference-style Constants bag (constants.py:11-20) into the C struct.  disc_drag = (CD, rho): what the
    discretizer's drag branch reads (const.CD, rho_func(r); linearize_discretize.py:162-168); rho is a number (constant
    density) or the dict discretizer.fit_density returns for a density that depends on |r|."""
    g = lambda n, d=0.0: float(getattr(const, n, d))
    model = None
    if disc_drag is not None and isinstance(disc_drag[1], dict):     # a fitted radial density (discretizer.fit_density)
        model = disc_drag[1]
        disc_drag = (disc_drag[0], float(model["rho_c"][0]))
    cd_a, rho_a = (0.0, 0.0) if disc_drag is None else (float(disc_drag[0]), float(disc_drag[1]))
    p = MpcParams(g("MU"), g("R_E"), g("J2"), g("G0"), g("ISP"), g("S"), g("R0", 1.0), g("RHO", 1.0),
                  float(c_d), float(rho_atm), cd_a, rho_a, int(bool(include_J2)), int(bool(include_drag)))
    if model is not None:
        rc, dc = list(model["rho_c"]), list(model["drho_c"])
        if not (1 <= len(rc) <= RHO_CHEB and len(dc) <= RHO_CHEB):
            raise ValueError(f"density model: 1..{RHO_CHEB} Chebyshev coefficients")
        p.disc_n_rho, p.disc_n_drho = len(rc), len(dc)
        p.disc_r_mid, p.disc_r_ihalf = float(model["r_mid"]), float(model["r_ihalf"])
        for i, v in enumerate(rc):
            p.disc_rho_cheb[i] = float(v)
        for i, v in enumerate(dc):
            p.disc_drho_cheb[i] = float(v)
    return p


# Page-locked buffers are expensive to create (cudaHostAlloc: ~0.1-1 ms plus ~0.2 ms per MiB) and the host API hands out
# three of them per call (trajectory, inputs, matrices).  Buffers whose numpy array has been garbage-collected go back
# to a small size-bucketed pool instead of being freed, so a loop of calls (the SCP iterations: control.py:183-227)
# pays for them once.
_POOL = {}                 # bucket size in bytes -> [addresses]
_POOL_BYTES = 0
_POOL_CAP = 2 << 30        # at most 2 GiB parked


def _bucket(nbytes):
    b = 4096
    while b < nbytes:
        b <<= 1
    return b


def _release(ptr, bucket):
    global _POOL_BYTES
    if _POOL_BYTES + bucket <= _POOL_CAP:
        _POOL.setdefault(bucket, []).append(ptr)
        _POOL_BYTES += bucket
    else:
        lib().mpc_host_free(ptr)


def pinned_empty(shape, dtype=np.float64):
    """numpy array over page-locked host memory (cudaHostAlloc through the C-ABI), pooled (see above)."""
    global _POOL_BYTES
    dtype = np.dtype(dtype)
    shape = tuple(int(s) for s in (shape if isinstance(shape, (tuple, list)) else (shape,)))
    nbytes = int(np.prod(shape, dtype=np.int64)) * dtype.itemsize
    bucket = _bucket(max(nbytes, 1))
    L = lib()
    free = _POOL.get(bucket)
    if free:
        ptr = free.pop()
        _POOL_BYTES -= bucket
    else:
        ptr = L.mpc_host_alloc(bucket)
        if not ptr:
            raise MemoryError(L.mpc_last_error().decode())
    buf = (ctypes.c_char * bucket).from_address(ptr)
    arr = np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape, dtype=np.int64))).reshape(shape)
    weakref.finalize(buf, _release, ptr, bucket)
    return arr


def addr(a):
    """Raw address of a C-contiguous numpy array (None -> NULL)."""
    if a is None:
        return None
    assert a.flags["C_CONTIGUOUS"]
    return a.ctypes.data
