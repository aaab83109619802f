/*
 * mpc_b200.h -- C-ABI of libmpc_b200.so: the B200 (sm_100a) implementation of mpconstellation's
 * batched SCvx linearize-and-discretize step and nonlinear orbit propagation.
 *
 * The reference (rgovindjee/mpconstellation) is pure Python and has no FFI layer; the boundary
 * it offers is two call signatures, Discretizer.discretize (linearize_discretize.py:334-390)
 * and Simulator.get_trajectory_ODE / run (simulator.py:29-48,164-189).  Each entry point below
 * names the reference interface it replaces.  INTEGRATION.md shows the ctypes binding a
 * maintainer of the reference would add.
 *
 * Conventions
 *   - every function returns 0 on success or a negative MPC_E_* code; mpc_last_error() gives text
 *   - all arrays are float64, C-contiguous, in the reference's own per-satellite shapes with a
 *     leading batch axis:  x [N][7][K], u [N][3][K], y [N][7][T]
 *   - "device API": pointers are device pointers owned by the caller, work is enqueued on the
 *     caller's stream (a cudaStream_t passed as void*), nothing is allocated, nothing synchronises
 *   - "host API": pointers are host pointers (pinned memory recommended: mpc_host_alloc);
 *     an mpc_ctx owns the device workspace, streams and the chunked copy/compute pipeline
 *   - there is NO CPU fallback anywhere in this library
 */
#ifndef MPC_B200_H
#define MPC_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MPC_B200_VERSION 100 /* major*10000 + minor*100 + patch */

/* rows of the structure-of-arrays discretization output, out[row][interval] */
#define MPC_OUT_ROWS 105
#define MPC_ROW_A 0      /* 49 rows: A_k  = Phi(tau_{k+1}), row-major 7x7   linearize_discretize.py:43-44 */
#define MPC_ROW_BP 49    /* 21 rows: B_kp (B+), row-major 7x3               linearize_discretize.py:72,77 */
#define MPC_ROW_BN 70    /* 21 rows: B_kn (B-), row-major 7x3               linearize_discretize.py:71,78 */
#define MPC_ROW_SIGMA 91 /*  7 rows: Sigma_k                                linearize_discretize.py:74,79 */
#define MPC_ROW_XI 98    /*  7 rows: xi_k                                   linearize_discretize.py:75,80 */

/* layouts of a [105][n_sats (K-1)] result: column = s (K-1) + k (per-satellite blocks) or k n_sats + s (interval k of all
 * satellites adjacent; see mpc_discretize_batch_gather / mpc_propagate_discretize_host_layout) */
#define MPC_LAYOUT_SAT_MAJOR 0
#define MPC_LAYOUT_K_MAJOR 1

/* return codes */
#define MPC_SUCCESS 0
#define MPC_E_INVALID (-1)     /* bad argument */
#define MPC_E_CUDA (-2)        /* CUDA runtime error (text in mpc_last_error) */
#define MPC_E_UNSUPPORTED (-3) /* option the reference cannot run either (e.g. drag in the discretizer) */
#define MPC_E_NOMEM (-4)

/* per-unit status written by the kernels (one int32 per interval / per satellite) */
#define MPC_ST_OK 0
#define MPC_ST_MASS 1      /* mass <= 0 met while integrating: simulator.py:135-136 raises here */
#define MPC_ST_NONFINITE 2 /* a non-finite result */
#define MPC_ST_STEP 3      /* adaptive mode: step size underflow / too many steps (solve_ivp would fail) */
#define MPC_ST_ATMO 4      /* mpc_propagate_batch_rk45_atmo: an altitude outside the fitted atmosphere's range */

/* Normalized constants: the reference's Constants bag (constants.py:11-20) as produced by
 * SatelliteScale.get_normalized_constants (satellite_scale.py:36-44), plus the two module-level
 * values the dynamics read directly (C_D constants.py:7; density simulator.py:112). */
typedef struct mpc_params {
    double mu, r_e, j2, g0, isp;
    double s_area, r0, rho;
    double c_d, rho_atm;  /* drag of the DYNAMICS: module-level C_D and density        simulator.py:150-153 */
    double disc_cd;       /* drag of the LINEARISATION: const.CD ...                  linearize_discretize.py:165-168 */
    double disc_rho;      /* ... and rho_func(r) when the density is constant (drho_func = 0); 0, 0 = not supplied */
    int32_t include_j2;   /* Discretizer(include_J2=...) / Simulator(include_J2=...) */
    int32_t include_drag; /* Simulator(include_drag=...); Discretizer(include_drag=...): needs disc_cd / disc_rho --
                             without them the reference raises (rho_func is None, Constants has no CD) and so do we */
    /* Altitude-dependent density in the drag LINEARISATION (rho_func(r), drho_func(r) of linearize_discretize.py:164-166,
     * e.g. the power law of simulator.py:110): Chebyshev series in t = (|r| - disc_r_mid) * disc_r_ihalf over the radii of
     * the batch, sum_k c_k T_k(t).  disc_n_rho = 0: the constant disc_rho above (and no gradient).  disc_n_drho = 0:
     * drho_func = 0.  Fitted and verified by the host (mpconstellation_b200/discretizer.py: fit_density). */
    int32_t disc_n_rho, disc_n_drho; /* 0 .. MPC_RHO_CHEB */
    double disc_r_mid, disc_r_ihalf;
    double disc_rho_cheb[32], disc_drho_cheb[32];
} mpc_params;
#define MPC_RHO_CHEB 32

/* Controller laws the propagator can evaluate on the device (control.py). */
#define MPC_CTRL_ZERO 0       /* Controller.get_u_func                      control.py:20-29   */
#define MPC_CTRL_CONSTANT 1   /* ConstantThrustController                   control.py:47-53   */
#define MPC_CTRL_TANGENTIAL 2 /* ConstantTangentialThrustController         control.py:66-84   */
#define MPC_CTRL_SEQUENCE 3   /* SequenceController (FOH table, end_tau)    control.py:104-143 */

typedef struct mpc_controller {
    int32_t kind;          /* MPC_CTRL_* */
    int32_t table_len;     /* Ku: columns of the sequence table (>= 2 for MPC_CTRL_SEQUENCE) */
    int32_t table_per_sat; /* 1: table is [N][3][Ku]; 0: one [3][Ku] table shared by all satellites */
    int32_t reserved;
    double thrust[3];      /* CONSTANT: the vector; TANGENTIAL: thrust[0] = magnitude */
    double end_tau;        /* SEQUENCE: tf_u / tf_sim (control.py:101) */
    const double *table;   /* SEQUENCE: device pointer (device API) or host pointer (host API) */
    const double *end_tau_per_sat; /* SEQUENCE, optional [N]: per-satellite end_tau (overrides end_tau); same
                                      pointer kind as `table`; NULL = use the scalar */
} mpc_controller;

/* ---------------------------------------------------------------- library */
int mpc_version(void);
const char *mpc_last_error(void);
int mpc_device_count(void);
/* name / SM count / clock of a device; returns MPC_E_CUDA when there is no usable GPU */
int mpc_device_info(int device, char *name, int name_len, int *sm_count, int *cc_major, int *cc_minor);

/* ---------------------------------------------------------------- device API */

/*
 * Replaces Discretizer.discretize (linearize_discretize.py:334-390) + get_matrices (:8-82) for a
 * whole batch: every (satellite, interval) pair is one independent unit.
 *
 *   x   [n_sats][7][K]   reference trajectories (scaled states)            discretize() arg `x`
 *   u   [n_sats][3][K]   reference inputs on the same K nodes              discretize() arg `u`
 *   tf  [n_sats]         reference final time per satellite                discretize() arg `tf`
 *   n_sub                trapezoid panels per interval = integrator_steps - 1 (quadrature nodes = n_sub + 1).  The
 *                        integrator (fixed-step fourth-order Runge-Kutta-Nystrom) takes one step per panel, or one
 *                        step per TWO panels with the node in between read off the step's cubic Hermite interpolant
 *                        where that is accurate to ~1e-12 (even n_sub, step short against the orbital rate; decided
 *                        per interval on the device; mpc_set_tuning(7) forces one step per panel everywhere).
 *                        n_sub = 100 (the reference's integrator_steps = 101): the 101-node trapezoid sums are evaluated
 *                        through their Euler-Maclaurin expansion -- T(h) = sum_n w_n T(n h), n = 5, 10, 20, 25: one rule on
 *                        the 21 nodes 0, 5, ..., 100, which are the ends of 20 integrator steps -- wherever the held
 *                        input changes by at most a quarter of its size across the interval and the interval is at
 *                        most ~0.011 orbit (up to ~0.035 orbit: n = 2, 4, 10, 20, the 51 even nodes, 50 steps); all
 *                        101 nodes otherwise, decided per interval on the device.  The gate bounds the circular
 *                        orbital rate at the interval's start node; on an eccentric orbit the angular rate at perigee
 *                        is sqrt(1+e) times that, so the error is bounded per form, not by one number.  Against the
 *                        101-node sums of the exact flow, norm-relative, for e <= 0.8 and perigees down to 2 % of R_E
 *                        above the surface, at the edges of the gate: the 11-node form (the default where the input
 *                        changes by at most an eighth) A_k 3.4e-13, B/Sigma/xi 5.4e-14; the 21-node form 1.7e-11 /
 *                        9.2e-13; the 51-node form 5e-11 / 6.8e-12; all 101 nodes 1.3e-11 / 1.6e-11
 *                        (tests/test_orbit_sweep_on_host.py).  All far below the reference's own RK45 error
 *                        (~1e-9).  mpc_set_tuning(37) evaluates all 101 nodes everywhere
 *   out                  SoA, out[row * out_pitch + out_offset + s*(K-1) + k], row in [0,105)
 *   status [n_sats*(K-1)] MPC_ST_* per interval (may be NULL)
 *
 * out_pitch >= out_offset + n_sats*(K-1).  Passing a pitch/offset larger than the local batch lets
 * several ranks write disjoint column ranges of one gathered buffer.
 */
int mpc_discretize_batch(const double *x, const double *u, const double *tf, const mpc_params *p, int n_sats,
                         int K, int n_sub, double *out, int64_t out_pitch, int64_t out_offset, int32_t *status,
                         void *stream);

/*
 * Same computation; every result is stored to n_dst destination buffers (for example the local
 * buffer plus NVLink peer-mapped buffers of the other ranks: the all-gather of the discretized
 * matrices fused into the producing kernel).  dst is a HOST array of n_dst device pointers
 * (n_dst <= MPC_MAX_DST).
 */
#define MPC_MAX_DST 8
int mpc_discretize_batch_multi(const double *x, const double *u, const double *tf, const mpc_params *p,
                               int n_sats, int K, int n_sub, double *const *dst, int n_dst, int64_t out_pitch,
                               int64_t out_offset, int32_t *status, void *stream);

/*
 * The reference's DEFAULT quadrature mode (Discretizer.use_uniform_steps = False, linearize_discretize.py:
 * 29-30,49-50,109): the nodes of every interval are the steps scipy's solve_ivp(RK45) accepts.  The kernel
 * replays scipy's step-size controller per interval (Dormand-Prince 5(4), rtol/atol error norm, first-step
 * heuristic, max_step = Discretizer.ivp_max_step) and applies the non-uniform trapezoid rule on those nodes,
 * so the matrices match what the unmodified reference hands to the optimizer.  scipy defaults: rtol 1e-3,
 * atol 1e-6.  n_nodes [n_sats*(K-1)] (may be NULL) receives the node count of every interval (len(sol.t)).
 * Other arguments as mpc_discretize_batch.
 */
int mpc_discretize_batch_adaptive(const double *x, const double *u, const double *tf, const mpc_params *p,
                                  int n_sats, int K, double rtol, double atol, double max_step, double *out,
                                  int64_t out_pitch, int64_t out_offset, int32_t *status, int32_t *n_nodes,
                                  void *stream);

/*
 * u on its own grid: u is [n_sats][3][u_cols] with u_cols != K.  The reference accepts this (u_FOH takes its grid
 * from u itself, linearize_discretize.py:308-315; its own test_linearize_many passes a (3,3K) array,
 * test_discretizer.py:103): the hold is evaluated on u's global grid inside every interval.  adaptive = 0: fixed-step
 * mode (n_sub used), adaptive = 1: default mode (rtol, atol, max_step, n_nodes used).
 */
int mpc_discretize_batch_ugrid(const double *x, const double *u, int u_cols, const double *tf, const mpc_params *p,
                               int n_sats, int K, int adaptive, int n_sub, double rtol, double atol, double max_step,
                               double *out, int64_t out_pitch, int64_t out_offset, int32_t *status, int32_t *n_nodes,
                               void *stream);

/*
 * Replaces Simulator.get_trajectory_ODE (simulator.py:164-189) for a batch of satellites, and
 * Discretizer.extract_uk (linearize_discretize.py:393-411) on the sampled trajectory.
 *
 *   y0  [n_sats][7]      normalized initial states (scale.normalize_state(sat.get_state_vector()))
 *   tf  [n_sats]
 *   T                    eval_points = int(base_res * tf)    (simulator.py:38,185)
 *   n_sub                0: THE REFERENCE'S INTEGRATOR, replayed step for step -- scipy's RK45 (Dormand-Prince 5(4))
 *                        with its step-size controller, max_step = 0.001 and default tolerances exactly as
 *                        simulator.py:185-187 calls solve_ivp, samples read off the 4th-order dense output of the step
 *                        that covers them (propagate_rk45_kernel; agrees with the reference to ~1e-13, also where the
 *                        thrust jumps inside a run: control.py:127-141).
 *                        >= 1: fixed-step classical RK4 with n_sub steps between consecutive samples (the reference's
 *                        max_step corresponds to n_sub = ceil(1000/(T-1))); agrees with the reference to ~1e-8 on
 *                        smooth inputs only
 *   y   [n_sats][7][T]   sol.y per satellite; sample times are linspace(0,1,T)
 *   u_out [n_sats][3][T] controller output at every sample (may be NULL)
 *   status [n_sats]      MPC_ST_* (may be NULL)
 */
int mpc_propagate_batch(const double *y0, const double *tf, const mpc_params *p, const mpc_controller *ctrl,
                        int n_sats, int T, int n_sub, double *y, double *u_out, int32_t *status, void *stream);

/*
 * mpc_propagate_batch(n_sub = 0) with the three numbers solve_ivp would take (simulator.py:185-187 hard-codes
 * max_step = 0.001 and leaves rtol = 1e-3, atol = 1e-6 at scipy's defaults).  n_steps [n_sats] (may be NULL) receives
 * the number of steps attempted per satellite (accepted + rejected; scipy's nfev = 2 + 6 n_steps).
 */
int mpc_propagate_batch_rk45(const double *y0, const double *tf, const mpc_params *p, const mpc_controller *ctrl,
                             int n_sats, int T, double rtol, double atol, double max_step, double *y, double *u_out,
                             int32_t *status, int32_t *n_steps, void *stream);

/*
 * Ragged batches: satellite s has its own node count K_s = K_sat[s] (2 <= K_s <= K_max), the reference's
 * int(base_res * tf_s) of every satellite's own horizon.  x [n_sats][7][K_max] and u [n_sats][3][K_max] are padded: only
 * the first K_s columns of satellite s are read.  The result keeps the rectangular layout of K_max:
 * out[row][out_offset + s (K_max-1) + k] for k < K_s - 1, status / n_nodes [n_sats][K_max-1]; the padding columns are
 * never written.  One launch for the whole batch, the threads mapped to live intervals only.  adaptive = 0: fixed-step
 * mode (n_sub), 1: default mode (rtol, atol, max_step, n_nodes), as mpc_discretize_batch_ugrid.
 *   K_sat      HOST array [n_sats] (validated; it also sizes the launch)
 *   first      DEVICE scratch of n_sats + 1 int64, filled by the call (prefix sums of K_s - 1) and read by the kernel
 * MPC_E_UNSUPPORTED: include_drag.
 */
int mpc_discretize_batch_ragged(const double *x, const double *u, const double *tf, const mpc_params *p, int n_sats,
                                int K_max, const int32_t *K_sat, int64_t *first, int adaptive, int n_sub, double rtol,
                                double atol, double max_step, double *out, int64_t out_pitch, int64_t out_offset,
                                int32_t *status, int32_t *n_nodes, void *stream);

/*
 * mpc_propagate_batch_rk45 with a sample count per satellite: satellite s is sampled at linspace(0, 1, T_sat[s]) into the
 * first T_sat[s] columns of y [n_sats][7][T_max] (and u_out [n_sats][3][T_max]); the padding columns are never written.
 * The steps do not depend on the samples: n_steps equals a rectangular run of the same satellite.
 *   T_sat          DEVICE array [n_sats] (not read by the host; the kernel keeps every count inside [0, T_max])
 *   table_len_sat  MPC_CTRL_SEQUENCE with a per-satellite table [n_sats][3][table_len]: satellite s uses its first
 *                  table_len_sat[s] columns (2 .. table_len; table_len stays the stride).  DEVICE array [n_sats] or NULL
 *                  (every satellite: table_len)
 */
int mpc_propagate_batch_rk45_ragged(const double *y0, const double *tf, const mpc_params *p, const mpc_controller *ctrl,
                                    int n_sats, int T_max, const int32_t *T_sat, const int32_t *table_len_sat, double rtol,
                                    double atol, double max_step, double *y, double *u_out, int32_t *status,
                                    int32_t *n_steps, void *stream);

/* ---------------------------------------------------------------- host API */
typedef struct mpc_ctx mpc_ctx;

int mpc_ctx_create(int device, mpc_ctx **ctx);
int mpc_ctx_destroy(mpc_ctx *ctx);

/* page-locked host memory (cudaHostAlloc); NULL on failure */
void *mpc_host_alloc(size_t bytes);
void mpc_host_free(void *p);

/*
 * Host-buffer form of mpc_discretize_batch: copies x/u/tf to the device, runs the kernel and
 * copies the SoA result back, pipelined in satellite chunks over two streams.
 * out_host is [105][n_sats*(K-1)] (pitch = n_sats*(K-1)); status_host [n_sats*(K-1)] or NULL.
 * Rows 42..48 (the last row of A_k, structurally 0 0 0 0 0 0 1 because the last row of the Jacobian is zero,
 * linearize_discretize.py:177-179) are not moved over PCIe: the library writes them into out_host itself.
 */
int mpc_discretize_batch_host(mpc_ctx *ctx, const double *x, const double *u, const double *tf,
                              const mpc_params *p, int n_sats, int K, int n_sub, double *out_host,
                              int32_t *status_host);

/* Host-buffer form of mpc_discretize_batch_adaptive. */
int mpc_discretize_batch_adaptive_host(mpc_ctx *ctx, const double *x, const double *u, const double *tf,
                                       const mpc_params *p, int n_sats, int K, double rtol, double atol,
                                       double max_step, double *out_host, int32_t *status_host,
                                       int32_t *n_nodes_host);

/* Host-buffer form of mpc_discretize_batch_ugrid. */
int mpc_discretize_batch_ugrid_host(mpc_ctx *ctx, const double *x, const double *u, int u_cols, const double *tf,
                                    const mpc_params *p, int n_sats, int K, int adaptive, int n_sub, double rtol,
                                    double atol, double max_step, double *out_host, int32_t *status_host,
                                    int32_t *n_nodes_host);

/* Host-buffer form of mpc_propagate_batch (ctrl->table is a host pointer here). */
int mpc_propagate_batch_host(mpc_ctx *ctx, const double *y0, const double *tf, const mpc_params *p,
                             const mpc_controller *ctrl, int n_sats, int T, int n_sub, double *y_host,
                             double *u_host, int32_t *status_host);

/* Host-buffer form of mpc_propagate_batch_rk45. */
int mpc_propagate_batch_rk45_host(mpc_ctx *ctx, const double *y0, const double *tf, const mpc_params *p,
                                  const mpc_controller *ctrl, int n_sats, int T, double rtol, double atol,
                                  double max_step, double *y_host, double *u_host, int32_t *status_host,
                                  int32_t *n_steps_host);

/* Host-buffer form of mpc_discretize_batch_ragged: K_sat is a host array (validated: 2 <= K_s <= K_max), out_host is
 * [105][n_sats (K_max-1)] with NaN in the padding columns, status_host / n_nodes_host [n_sats][K_max-1] with 0 there. */
int mpc_discretize_batch_ragged_host(mpc_ctx *ctx, const double *x, const double *u, const double *tf, const mpc_params *p,
                                     int n_sats, int K_max, const int32_t *K_sat, int adaptive, int n_sub, double rtol,
                                     double atol, double max_step, double *out_host, int32_t *status_host,
                                     int32_t *n_nodes_host);

/* Host-buffer form of mpc_propagate_batch_rk45_ragged: T_sat and table_len_sat are host arrays (validated:
 * 2 <= T_s <= T_max, 2 <= table length <= table_len); y_host / u_host padding columns are NaN. */
int mpc_propagate_batch_rk45_ragged_host(mpc_ctx *ctx, const double *y0, const double *tf, const mpc_params *p,
                                         const mpc_controller *ctrl, int n_sats, int T_max, const int32_t *T_sat,
                                         const int32_t *table_len_sat, double rtol, double atol, double max_step,
                                         double *y_host, double *u_host, int32_t *status_host, int32_t *n_steps_host);

/*
 * SCP inner step on host buffers, fused on the device (control.py:180-188 pattern): propagate the
 * batch, evaluate the controller on the samples (extract_uk), discretize about the result.  The
 * reference trajectory never leaves HBM between the two kernels.  K = T.
 * Any of y_host / u_host may be NULL when the caller only wants the matrices.  n_sub_prop as n_sub of
 * mpc_propagate_batch (0 = the reference's RK45, replayed), here and in the two entry points below.
 */
int mpc_propagate_discretize_host(mpc_ctx *ctx, const double *y0, const double *tf, const mpc_params *p_prop,
                                  const mpc_params *p_disc, const mpc_controller *ctrl, int n_sats, int T,
                                  int n_sub_prop, int n_sub_disc, double *y_host, double *u_host,
                                  double *out_host, int32_t *status_host);

/*
 * mpc_propagate_discretize_host with the result in the K-MAJOR layout (out_host[row][k n_sats + s], see
 * MPC_LAYOUT_K_MAJOR) and the propagation hidden behind the discretization AND the read-back: the intervals are
 * discretized window by window along k as the propagation publishes its progress (mpc_propagate_discretize), and the
 * columns of a finished window -- one contiguous range per row in this layout -- go back over PCIe while the next window
 * runs.  The first byte leaves the device ~0.3 ms after the call starts instead of after the whole propagation (1.1 ms).
 * status_host stays [n_sats][T-1].  layout = MPC_LAYOUT_SAT_MAJOR is mpc_propagate_discretize_host.
 */
int mpc_propagate_discretize_host_layout(mpc_ctx *ctx, const double *y0, const double *tf, const mpc_params *p_prop,
                                         const mpc_params *p_disc, const mpc_controller *ctrl, int n_sats, int T,
                                         int n_sub_prop, int n_sub_disc, double *y_host, double *u_host, double *out_host,
                                         int32_t *status_host, int layout);

/*
 * The same SCP inner step on DEVICE buffers, enqueued on `stream`, with the propagation overlapped with the
 * discretization (control.py:180-188: run_nonlinear -> extract_uk -> Discretizer.discretize, for every satellite).
 * The propagation is sequential in tau and latency-bound; interval k only needs the samples k and k+1.  The intervals
 * are cut into `n_windows` windows along k (0 = default, 16); the propagation kernel publishes a progress word per
 * window and the discretization of window b is gated on it by a stream memory operation (cuStreamWaitValue32) on an
 * internal stream -- no kernel spins.  Results (x [N][7][T], u [N][3][T], the SoA matrices, both status arrays) are
 * bit-identical to mpc_propagate_batch followed by mpc_discretize_batch.  Batches too small for windows to fill the
 * machine, and the drag branch, run the two kernels back to back on `stream`.  ctrl->table / end_tau_per_sat are
 * device pointers (as in mpc_propagate_batch).  One call per ctx may be in flight at a time; `stream` continues only
 * when everything has finished.
 */
int mpc_propagate_discretize(mpc_ctx *ctx, const double *y0, const double *tf, const mpc_params *p_prop,
                             const mpc_params *p_disc, const mpc_controller *ctrl, int n_sats, int T, int n_sub_prop,
                             int n_sub_disc, double *x, double *u, double *out, int64_t out_pitch, int64_t out_offset,
                             int32_t *status_prop, int32_t *status_disc, int n_windows, void *stream);

/* mpc_propagate_discretize with the multi-destination store of mpc_discretize_batch_multi (fused all-gather: dst[0] is
 * the local buffer, dst[1..] peer-mapped buffers of the same layout; n_dst = 1, 2, 4 or 8; honours
 * mpc_set_gather_tuning, the staggered start applying to the first window only). */
int mpc_propagate_discretize_multi(mpc_ctx *ctx, const double *y0, const double *tf, const mpc_params *p_prop,
                                   const mpc_params *p_disc, const mpc_controller *ctrl, int n_sats, int T,
                                   int n_sub_prop, int n_sub_disc, double *x, double *u, double *const *dst, int n_dst,
                                   int64_t out_pitch, int64_t out_offset, int32_t *status_prop, int32_t *status_disc,
                                   int n_windows, void *stream);

/*
 * The fused all-gather with its options passed per call (the two entry points above read the process-wide knobs of
 * mpc_set_gather_tuning), and with a choice of the gathered layout.  Every destination buffer is [105][n_sats_total (K-1)]:
 *   MPC_LAYOUT_SAT_MAJOR  column = (sat_offset + s) (K-1) + k      (what mpc_discretize_batch writes; per-satellite blocks)
 *   MPC_LAYOUT_K_MAJOR    column = k n_sats_total + sat_offset + s  (interval k of ALL satellites adjacent)
 * n_sats_total: satellites of all ranks, sat_offset: first satellite of this rank (s = 0..n_sats-1 are this call's).
 * In the k-major layout a window of k of the overlapped pass stores whole runs of n_sats consecutive columns per row --
 * full 256-byte lines per warp, also to the peers -- where the satellite-major layout gives 13-column fragments; that is
 * what lets the propagation hide behind the discretization at 4 and 8 GPUs as well.  The consumer indexes elements
 * (optimizer.py:327-339), so the layout is a stride, not a copy (GatheredView in the Python package).
 * skip_const / stagger_phases: as mpc_set_gather_tuning.  Fixed-step (two-node-step) kernel only.
 */
typedef struct mpc_gather_opts {
    int32_t layout;         /* MPC_LAYOUT_* */
    int32_t skip_const;     /* 0, 1, 2: see mpc_set_gather_tuning */
    int32_t stagger_phases; /* 0 = off */
    int32_t reserved;
    int64_t n_sats_total;
    int64_t sat_offset;
} mpc_gather_opts;
int mpc_discretize_batch_gather(const double *x, const double *u, const double *tf, const mpc_params *p, int n_sats,
                                int K, int n_sub, double *const *dst, int n_dst, const mpc_gather_opts *g,
                                int32_t *status, void *stream);
int mpc_propagate_discretize_gather(mpc_ctx *ctx, const double *y0, const double *tf, const mpc_params *p_prop,
                                    const mpc_params *p_disc, const mpc_controller *ctrl, int n_sats, int T,
                                    int n_sub_prop, int n_sub_disc, double *x, double *u, double *const *dst, int n_dst,
                                    const mpc_gather_opts *g, int32_t *status_prop, int32_t *status_disc, int n_windows,
                                    void *stream);

/*
 * All-gather of the discretized matrices by the COPY ENGINES, overlapped with the kernel: the batch is discretized
 * in chunks of `chunk_waves` full waves of the kernel into dst[0] (local); as soon as a chunk is done its columns
 * are pushed to dst[1..n_dst-1] (peer-mapped buffers of the other ranks, same layout) by cudaMemcpy2DAsync on one
 * stream per peer -- NVLink carries chunk c while the SMs compute chunk c+1, no SM time and no store-queue stalls
 * are spent on the exchange.  When the call returns, everything is enqueued and `stream` waits for the pushes.
 * Rows 42..48 (structural constants, see mpc_discretize_batch_host) are NOT pushed: every destination buffer must
 * have been initialised once with mpc_fill_const_rows.  x, u, tf, dst[] device pointers; ctx owns the push streams.
 * use_copy_kernel = 1: the pushes are done by a small copy kernel on a highest-priority stream instead of the copy
 * engines (one launch per chunk writing to all peers).
 */
int mpc_discretize_batch_push(mpc_ctx *ctx, const double *x, const double *u, const double *tf, const mpc_params *p,
                              int n_sats, int K, int n_sub, double *const *dst, int n_dst, int64_t out_pitch,
                              int64_t out_offset, int32_t *status, int chunk_waves, int use_copy_kernel, void *stream);
/* Writes the structural constants (rows 42..47 = 0, row 48 = 1) into all out_pitch columns of a SoA buffer. */
int mpc_fill_const_rows(double *out, int64_t out_pitch, void *stream);

/* ---------------------------------------------------------------- constraint terms (next step of the path) */

/*
 * Replaces Optimizer.get_constraint_terms (optimizer.py:80-170) for a batch of satellites: the step that follows
 * the discretization inside Optimizer.solve_OPT (optimizer.py:243-262).
 *
 *   x  [n_sats][7][K], u [n_sats][3][u_cols]   the reference trajectories / inputs (x_bar, u_bar)
 *   mu                                         const.MU
 *   rbar_hat [n_sats][3][K-1]                  r_bar/|r_bar| on nodes 0..K-2            optimizer.py:128-129
 *   ubar_hat [n_sats][3][u_cols]               as the reference computes it (filled only where |u| <= eps,
 *                                              i.e. 0/0 = NaN for zero thrust, 0 elsewhere) optimizer.py:132-139
 *   final_terms [n_sats][MPC_FINAL_TERMS]      terminal-node terms, offsets MPC_FT_*    optimizer.py:108-168
 */
#define MPC_FINAL_TERMS 32
#define MPC_FT_RF_HAT 0         /* 3 */
#define MPC_FT_VC 3             /* 1 */
#define MPC_FT_DRVC 4           /* 3 */
#define MPC_FT_DRVC_RBAR 7      /* 1 */
#define MPC_FT_VT 8             /* 1 */
#define MPC_FT_DRVT_DVVT 9      /* 6 */
#define MPC_FT_DRVT_DVVT_BAR 15 /* 1 */
#define MPC_FT_VR 16            /* 1 */
#define MPC_FT_DRVR_DVVR 17     /* 6 */
#define MPC_FT_DRVR_DVVR_BAR 23 /* 1 */
#define MPC_FT_VN 24            /* 1 */
#define MPC_FT_DRVN_DVVN 25     /* 6 */
#define MPC_FT_DRVN_DVVN_BAR 31 /* 1 */
int mpc_constraint_terms(const double *x, const double *u, int n_sats, int K, int u_cols, double mu, double *rbar_hat,
                         double *ubar_hat, double *final_terms, void *stream);
/* Host-buffer form. */
int mpc_constraint_terms_host(mpc_ctx *ctx, const double *x, const double *u, int n_sats, int K, int u_cols, double mu,
                              double *rbar_hat, double *ubar_hat, double *final_terms);

/*
 * Sparse (CSR) assembly of the dynamics constraint optimizer.py:327-339 from a SoA discretization result on the
 * device:  J z = rhs,  one row per (s, i, k) in pyomo's generation order, row = (s*7 + i)*(K-1) + k, exactly
 * MPC_JAC_NNZ_PER_ROW = 16 non-zeros per row in ascending column order (indptr[r] = 16 r), variables numbered
 *   x[s,i,k] -> (s*7+i)*K + k | u[s,j,k] -> 7NK + (s*3+j)*K + k | nu[s,i,k] -> 10NK + (s*7+i)*K + k | tf -> 17NK.
 * values [rows*16], indices [rows*16] (int64; may be NULL when only the values change between SCP iterations),
 * rhs [rows] = xi_k.  soa / pitch / offset as written by mpc_discretize_batch.  Device pointers, caller's stream.
 */
#define MPC_JAC_NNZ_PER_ROW 16
int mpc_dynamics_jacobian(const double *soa, int64_t pitch, int64_t offset, int n_sats, int K, double *values,
                          int64_t *indices, double *rhs, void *stream);

/*
 * Ragged batches (satellite s on its own K_s = K_sat[s] nodes, 2 <= K_s <= K_max; the hand-off of
 * mpc_discretize_batch_ragged).  Buffers stay padded to K_max and the padding is never written; one launch for the
 * batch, the threads mapped to the live intervals only.
 *   K_sat   HOST array [n_sats] (validated; it also sizes the launch)
 *   first   DEVICE scratch of n_sats + 1 int64, filled by the call (prefix sums first[s] = sum_{r<s} (K_r - 1))
 *
 * mpc_constraint_terms_ragged: x [n_sats][7][K_max], u [n_sats][3][K_max] on the nodes of x.  Satellite s gets
 * rbar_hat [n_sats][3][K_max-1] columns k < K_s - 1, ubar_hat [n_sats][3][K_max] columns k < K_s and final_terms
 * [n_sats][MPC_FINAL_TERMS] from node K_s - 1: bit for bit what mpc_constraint_terms gives for that satellite alone at
 * K = u_cols = K_s.
 */
int mpc_constraint_terms_ragged(const double *x, const double *u, int n_sats, int K_max, const int32_t *K_sat, int64_t *first,
                                double mu, double *rbar_hat, double *ubar_hat, double *final_terms, void *stream);
/* Host-buffer form: x, u, K_sat and the outputs are host arrays; the padding columns of rbar_hat / ubar_hat are NaN. */
int mpc_constraint_terms_ragged_host(mpc_ctx *ctx, const double *x, const double *u, int n_sats, int K_max,
                                     const int32_t *K_sat, double mu, double *rbar_hat, double *ubar_hat, double *final_terms);

/*
 * mpc_dynamics_jacobian_ragged: the dynamics constraint of a ragged batch as a block-diagonal CSR of n_sats independent
 * single-satellite systems, each with its own final time tf_s (every satellite's Optimizer has its own tf variable,
 * optimizer.py:281).  Block s is the numbering of mpc_dynamics_jacobian with n_sats = 1, K = K_s, shifted:
 *   rows       R_s = 7 first[s];   row = R_s + i (K_s-1) + k                       (7 first[n_sats] rows)
 *   variables  V_s = sum_{r<s} (17 K_r + 1) = 17 (first[s] + s) + s                (17 (first[n_sats] + n_sats) + n_sats)
 *              x[i,k] -> V_s + i K_s + k          u[j,k] -> V_s + 7 K_s + j K_s + k
 *              nu[i,k] -> V_s + 10 K_s + i K_s + k   tf_s -> V_s + 17 K_s
 * Still MPC_JAC_NNZ_PER_ROW non-zeros per row in ascending column order (indptr[r] = 16 r).  soa holds the ragged
 * result of mpc_discretize_batch_ragged: satellite s, interval k at column offset + s (K_max-1) + k, pitch >= offset +
 * n_sats (K_max-1).  indices may be NULL (only the values change between SCP iterations).  Device pointers except K_sat.
 */
int mpc_dynamics_jacobian_ragged(const double *soa, int64_t pitch, int64_t offset, int n_sats, int K_max,
                                 const int32_t *K_sat, int64_t *first, double *values, int64_t *indices, double *rhs,
                                 void *stream);

/* ---------------------------------------------------------------- per-satellite designer units */

/*
 * The per-scale fields of one satellite's normalized Constants (SatelliteScale.get_normalized_constants of THAT
 * satellite, satellite_scale.py:36-44): what the kernels read.  A constellation that mixes altitudes and masses is
 * linearized satellite by satellite in these units, as N separate controllers of the reference do (control.py:164,187).
 * Everything else stays launch-wide in mpc_params: include_j2, include_drag, c_d, rho_atm (its mu .. rho are not read).
 */
typedef struct mpc_sat_consts {
    double mu, r_e, j2, g0, isp, s_area, rho;
} mpc_sat_consts;

/* doubles of device scratch per satellite the *_units device entry points fill with the derived kernel constants */
#define MPC_SAT_SCRATCH_DOUBLES 8

/*
 * *_units: the computation of the single-constant entry point for every satellite s in the units of consts[s], one
 * launch for the batch; satellite s comes out bit for bit as a launch of the same kernel under consts[s] alone.
 *   consts          HOST array [n_sats], validated (every value finite, mu > 0, g0 * isp > 0; otherwise MPC_E_INVALID
 *                   naming the satellite).  The kernel constants are derived on the host with the expressions of the
 *                   single-constant path and copied (cudaMemcpyAsync on `stream`) into
 *   consts_scratch  DEVICE scratch of n_sats * MPC_SAT_SCRATCH_DOUBLES doubles, which the call fills.
 * Not available (MPC_E_UNSUPPORTED): the drag linearisation (include_drag in the discretization), the fixed-step RK4
 * propagator, u on its own grid, the round-1 default-mode kernel (mpc_set_tuning(9)), the fused overlapped pass and the
 * rectangular multi-GPU gather entry points (mpc_discretize_batch_ragged_gather takes per-satellite constants).
 *
 * mpc_discretize_batch_units: mpc_discretize_batch_ragged with per-satellite constants; K_sat == NULL means a rectangular
 * batch (K = K_max nodes for every satellite; `first` is then not used and may be NULL).  The fixed-step form always
 * takes the two-node-step kernel (small batches in one-warp CTAs, no thread-group kernel), in its ragged form: a
 * rectangular batch runs as one with K_max nodes everywhere, its prefix sums written into consts_scratch.
 */
int mpc_discretize_batch_units(const double *x, const double *u, const double *tf, const mpc_params *p,
                               const mpc_sat_consts *consts, int n_sats, int K_max, const int32_t *K_sat, int64_t *first,
                               double *consts_scratch, int adaptive, int n_sub, double rtol, double atol, double max_step,
                               double *out, int64_t out_pitch, int64_t out_offset, int32_t *status, int32_t *n_nodes,
                               void *stream);
/* Host-buffer form (context-owned scratch): as mpc_discretize_batch_ragged_host, K_sat == NULL: rectangular. */
int mpc_discretize_batch_units_host(mpc_ctx *ctx, const double *x, const double *u, const double *tf, const mpc_params *p,
                                    const mpc_sat_consts *consts, int n_sats, int K_max, const int32_t *K_sat, int adaptive,
                                    int n_sub, double rtol, double atol, double max_step, double *out_host,
                                    int32_t *status_host, int32_t *n_nodes_host);

/*
 * mpc_discretize_batch_rk23: the default quadrature mode (as mpc_discretize_batch_adaptive) with scipy's RK23 in place of
 * RK45 -- the reference's Discretizer.ivp_solver = 'RK23' (solve_ivp(method='RK23')): Bogacki-Shampine 3(2), its own
 * initial step and step-size controller, replayed per interval; the quadrature on the steps it accepts.  The arguments
 * are those of mpc_discretize_batch_units without adaptive and n_sub:
 *   consts    NULL: one constants bag (p; consts_scratch is then not used and may be NULL); else per-satellite
 *             constants [n_sats], validated as in mpc_discretize_batch_units, with their DEVICE consts_scratch.
 *   K_sat     NULL: a rectangular batch (K_max nodes everywhere; first may be NULL); else a ragged batch as in
 *             mpc_discretize_batch_ragged (host counts, `first` their device prefix sums).
 * n_nodes [n_sats (K_max - 1)] (may be NULL) receives len(sol.t) of every interval.  Not available: include_drag
 * (MPC_E_UNSUPPORTED); u is on the nodes of x.
 */
int mpc_discretize_batch_rk23(const double *x, const double *u, const double *tf, const mpc_params *p,
                              const mpc_sat_consts *consts, int n_sats, int K_max, const int32_t *K_sat, int64_t *first,
                              double *consts_scratch, double rtol, double atol, double max_step, double *out, int64_t out_pitch,
                              int64_t out_offset, int32_t *status, int32_t *n_nodes, void *stream);
/* Host-buffer form (context-owned scratch); consts and K_sat as above. */
int mpc_discretize_batch_rk23_host(mpc_ctx *ctx, const double *x, const double *u, const double *tf, const mpc_params *p,
                                   const mpc_sat_consts *consts, int n_sats, int K_max, const int32_t *K_sat, double rtol,
                                   double atol, double max_step, double *out_host, int32_t *status_host,
                                   int32_t *n_nodes_host);

/*
 * mpc_discretize_batch_ragged_gather: one rank's shard of a ragged batch (multi-GPU, satellites sharded over ranks), every
 * result stored into every rank's gathered buffer.  The gathered layout is the single-GPU ragged layout at a fixed
 * capacity K_cap: global satellite g on columns g (K_cap - 1) + k, k < K_g - 1.  A rank holding satellites [s0, s1)
 * passes x [n_sats][7][K_cap], u [n_sats][3][K_cap], tf [n_sats] of those satellites, its own counts K_sat (HOST, each
 * 2 <= K_s <= K_cap; `first` is their DEVICE scratch of n_sats + 1 prefix sums) and out_offset = s0 (K_cap - 1).
 *   consts      NULL: one constants bag (p), as mpc_discretize_batch_ragged; else per-satellite constants [n_sats] with
 *               their consts_scratch, as mpc_discretize_batch_units.
 *   adaptive    0: fixed step (n_sub), 1: the default quadrature mode (rtol, atol, max_step; n_nodes may be NULL).
 *   dst         n_dst (1, 2, 4 or 8) buffers [105][out_pitch] (the own one first: it also holds the default mode's scratch
 *               rows while the kernel runs; the others typically peer-mapped).  Padding columns are never written.
 *   skip_const  0: rows 42..48 stored everywhere; 1: to dst[0] only; 2: nowhere (buffers filled once by
 *               mpc_fill_const_rows).
 *   status, n_nodes  [n_sats (K_cap - 1)] of this rank (not gathered), padding not written.
 * Satellite s comes out bit for bit as in mpc_discretize_batch_ragged / _units.  Not available: include_drag.
 */
int mpc_discretize_batch_ragged_gather(const double *x, const double *u, const double *tf, const mpc_params *p,
                                       const mpc_sat_consts *consts, int n_sats, int K_cap, const int32_t *K_sat, int64_t *first,
                                       double *consts_scratch, int adaptive, int n_sub, double rtol, double atol,
                                       double max_step, double *const *dst, int n_dst, int64_t out_pitch, int64_t out_offset,
                                       int skip_const, int32_t *status, int32_t *n_nodes, void *stream);

/*
 * mpc_propagate_batch_rk45_units: mpc_propagate_batch_rk45_ragged with per-satellite constants (mu, kj2, 1/(g0 isp) and,
 * with include_drag, the drag coefficient 0.5 c_d s_area rho_atm / rho of each satellite).  T_sat == NULL (and
 * table_len_sat == NULL): every satellite on T_max samples, the rectangular run.  T_sat / table_len_sat are DEVICE
 * arrays as in the ragged entry point.
 */
int mpc_propagate_batch_rk45_units(const double *y0, const double *tf, const mpc_params *p, const mpc_sat_consts *consts,
                                   const mpc_controller *ctrl, int n_sats, int T_max, const int32_t *T_sat,
                                   const int32_t *table_len_sat, double *consts_scratch, double rtol, double atol,
                                   double max_step, double *y, double *u_out, int32_t *status, int32_t *n_steps,
                                   void *stream);
/* Host-buffer form: T_sat / table_len_sat are host arrays or NULL, as in mpc_propagate_batch_rk45_ragged_host. */
int mpc_propagate_batch_rk45_units_host(mpc_ctx *ctx, const double *y0, const double *tf, const mpc_params *p,
                                        const mpc_sat_consts *consts, const mpc_controller *ctrl, int n_sats, int T_max,
                                        const int32_t *T_sat, const int32_t *table_len_sat, double rtol, double atol,
                                        double max_step, double *y_host, double *u_host, int32_t *status_host,
                                        int32_t *n_steps_host);

/* ---------------------------------------------------------------- altitude-dependent atmosphere */

/*
 * A density model of the propagator's drag: log rho (kg/m^3) as a Chebyshev series sum_k coef[k] T_k(t) in
 * t = (log h - (log h_min + log h_max) / 2) * 2 / (log h_max - log h_min), h the altitude in metres, valid on
 * [h_min, h_max].  Fitted and checked against the user's rho(h) by mpconstellation_b200.fit_atmosphere.
 * Satellite s flies at the altitude h = |r| L - r_earth, L = r_earth / r_e the metres per unit length of its constants
 * (SatelliteScale: r_e = R_EARTH / r0, so L is its r0), and its drag acceleration is
 *     -(0.5 c_d s_area / rho) rho(h) / m |v| v
 * in those units: the dynamics of simulator.py:150-153 with rho(h) in place of Simulator.get_atmo_density.
 */
typedef struct mpc_atmosphere {
    double h_min, h_max;  /* m, 0 < h_min < h_max */
    double r_earth;       /* m */
    int32_t n;            /* terms, 1 .. MPC_RHO_CHEB */
    int32_t reserved;
    double coef[32];
} mpc_atmosphere;

/*
 * mpc_propagate_batch_rk45_atmo: the RK45 replay with drag under the atmosphere *atmo (passed by value to the kernel).
 * The arguments of mpc_propagate_batch_rk45_units plus atmo; consts == NULL: one constants bag (p; consts_scratch is
 * then not used and may be NULL), otherwise satellite s in the units of consts[s] (its own L and rho).  T_sat == NULL:
 * a rectangular batch.  p->include_drag must be set (rho_atm is not read).  The first stage evaluation at an altitude
 * outside [h_min, h_max] ends that satellite's run with status MPC_ST_ATMO (no extrapolation), as a non-positive mass
 * ends it with MPC_ST_MASS.  MPC_E_INVALID: a bad atmosphere (n, range, non-finite coefficients), r_e <= 0, or drag off.
 */
int mpc_propagate_batch_rk45_atmo(const double *y0, const double *tf, const mpc_params *p, const mpc_sat_consts *consts,
                                  const mpc_controller *ctrl, int n_sats, int T_max, const int32_t *T_sat,
                                  const int32_t *table_len_sat, double *consts_scratch, double rtol, double atol,
                                  double max_step, double *y, double *u_out, int32_t *status, int32_t *n_steps,
                                  const mpc_atmosphere *atmo, void *stream);
/* Host-buffer form: T_sat / table_len_sat are host arrays or NULL, as in mpc_propagate_batch_rk45_units_host. */
int mpc_propagate_batch_rk45_atmo_host(mpc_ctx *ctx, const double *y0, const double *tf, const mpc_params *p,
                                       const mpc_sat_consts *consts, const mpc_controller *ctrl, int n_sats, int T_max,
                                       const int32_t *T_sat, const int32_t *table_len_sat, double rtol, double atol,
                                       double max_step, double *y_host, double *u_host, int32_t *status_host,
                                       int32_t *n_steps_host, const mpc_atmosphere *atmo);

/*
 * mpc_constraint_terms_units: the terminal terms of satellite s with consts[s].mu (the only constant the constraint terms
 * read).  K_sat == NULL: rectangular, u on the nodes of x (u_cols = K_max; `first` may be NULL); otherwise as
 * mpc_constraint_terms_ragged (K_sat a host array, `first` its device scratch).
 */
int mpc_constraint_terms_units(const double *x, const double *u, int n_sats, int K_max, const int32_t *K_sat, int64_t *first,
                               const mpc_sat_consts *consts, double *consts_scratch, double *rbar_hat, double *ubar_hat,
                               double *final_terms, void *stream);
/* Host-buffer form; the padding columns of a ragged batch come back NaN. */
int mpc_constraint_terms_units_host(mpc_ctx *ctx, const double *x, const double *u, int n_sats, int K_max,
                                    const int32_t *K_sat, const mpc_sat_consts *consts, double *rbar_hat, double *ubar_hat,
                                    double *final_terms);

/* ---------------------------------------------------------------- conjunction screening */

/*
 * Close approaches between every pair of satellites of one propagation (mpc_propagate_batch*: y [n_sats][7][T],
 * normalized, sampled at T common instants).  Satellite s is taken to SI with scale[s] = (R0_s, R0_s / s0_s): position
 * y[0:3] R0_s (m), velocity y[3:6] R0_s / s0_s (m/s); the run lasts `duration` seconds for every satellite (sample k at
 * t_k = k h, h = duration / (T - 1)); the mass row is not read.  Between two samples each satellite follows the cubic
 * Hermite curve through its positions and velocities there.  An event is a local minimum of a pair's distance d(t) on
 * [0, duration] with d < threshold: t = 0 counts when d increases there, t = duration when d does not increase there,
 * and a minimum belongs to the interval whose half-open [t_k, t_k+1) holds it (the last interval is closed).
 * An interval with a non-finite end sample of satellite s is skipped for every pair with s, and counted in skipped[s].
 */
typedef struct mpc_conjunction {
    int32_t i, j;      /* satellites, i < j */
    int32_t k;         /* interval [t_k, t_k+1] */
    int32_t flags;     /* MPC_CONJ_FLAG_* */
    double t_ca;       /* s from the start of the run */
    double d_min;      /* m */
    double v_rel;      /* m/s at t_ca */
} mpc_conjunction;
/* the root isolation reached its depth cap (pieces of 2^-20 of an interval) before isolating this minimum: t_ca is
 * then known to that width only */
#define MPC_CONJ_FLAG_DEPTH 1

/* doubles of device scratch mpc_screen_conjunctions needs: n_sats (6 T + 4 (T - 1) + 2) */
int64_t mpc_conjunction_scratch_doubles(int n_sats, int T);

/*
 * mpc_screen_conjunctions: y [n_sats][7][T] DEVICE; scale [n_sats][2] HOST (every value finite and > 0); duration > 0
 * (s) and threshold > 0 (m) finite; scratch DEVICE of mpc_conjunction_scratch_doubles(n_sats, T); events DEVICE
 * [capacity] (capacity >= 0; may be NULL when 0) in no particular order; counters DEVICE [2] receives the number of
 * events found (which may exceed capacity: only the first `capacity` are stored) and the number with
 * MPC_CONJ_FLAG_DEPTH; skipped DEVICE [n_sats].  Two kernel launches on `stream`; nothing is synchronized.
 * MPC_E_INVALID before any device call: a null pointer, n_sats < 2, T < 2, a bad duration, threshold or scale.
 */
int mpc_screen_conjunctions(const double *y, int n_sats, int T, const double *scale, double duration, double threshold,
                            double *scratch, mpc_conjunction *events, int64_t capacity, uint64_t *counters,
                            int32_t *skipped, void *stream);
/* Host-buffer form (context-owned device buffers; returns when the results are in the host buffers): *count and
 * *n_flagged as counters above; min(*count, capacity) events in events_host, in no particular order. */
int mpc_screen_conjunctions_host(mpc_ctx *ctx, const double *y, int n_sats, int T, const double *scale, double duration,
                                 double threshold, mpc_conjunction *events_host, int64_t capacity, int64_t *count,
                                 int64_t *n_flagged, int32_t *skipped_host);

/* ---------------------------------------------------------------- measurement helpers */

/* FP64 FMA-chain microbenchmark: measured DFMA peak of `device` in TFLOP/s (2 flop per FMA). */
int mpc_fp64_peak_probe(int device, int repeats, double *tflops, double *ms);

/* Number of kernels this library has launched since load (bench.py's gpu_launches evidence). */
int64_t mpc_launch_count(void);

/* Experiment knob: 1..6 select an alternative block-size / register-cap build of the one-step-per-node discretization
 * kernel (0 = production; results identical, only occupancy differs; DESIGN.md, tuning table).  7 / 8 switch the
 * two-node integrator steps of the production kernel off / on (results differ by ~1e-12).  9 / 10 switch to the
 * round-1 build of the default-mode (adaptive) kernel and back (same results to rounding; A/B measurements).  11 / 12: RK45 propagator without / with the speculative first stage
 * of the next step (same results).  13: satellites per warp of the RK45 propagator chosen automatically, 14..19: forced
 * to 32, 16, 8, 4, 2, 1 (same results).  20 / 21 / 22: CTA size of the default-mode kernel 32 / 128 / 256 threads (same
 * results).  23 / 24 / 25: the thread-group kernel for small batches (8 lanes per interval) off / on / at any batch size
 * (results equal to rounding).  26..29: k-windows of the streamed host pass (mpc_propagate_discretize_host_layout) 16 / 32 /
 * 48 / 64 (same results).  37 / 38: the 21-node Euler-Maclaurin form of the 101-node trapezoid sums (n_sub = 100) off / on
 * (quadrature equal to 1e-13, A_k to 1e-11).  39 / 40: where the 21-node form applies, its 11-node form on ten
 * fifth-order Nystrom steps off / on (quadrature equal to 1e-12, A_k to 1e-11). */
int mpc_set_tuning(int variant);

/* Options of the fused (in-kernel store) all-gather, applied by mpc_discretize_batch / _multi:
 *   skip_const 1: rows 42..48 (structural constants) are stored to dst[0] only, 2: to no destination -- the other
 *                 buffers must have been initialised with mpc_fill_const_rows (6.7 % less NVLink traffic);
 *   stagger_phases > 1: the CTAs of the first wave start with a delay of (blockIdx % phases)/phases of one interval's
 *                 run time, which spreads the store phases of the CTAs over time (NVLink egress stays busy instead
 *                 of alternating between bursts and silence).  Results are unchanged.  0, 0 = off (default). */
int mpc_set_gather_tuning(int skip_const, int stagger_phases);

#ifdef __cplusplus
}
#endif
#endif /* MPC_B200_H */
