// propagate_rk45_kernel.cuh -- the reference's own trajectory integrator, replayed on the device.
//
// Simulator.get_trajectory_ODE (simulator.py:164-189) calls
//     solve_ivp(satellite_dynamics, [0, 1], y0, t_eval=linspace(0, 1, T), max_step=0.001)     (RK45, rtol 1e-3, atol 1e-6)
// so what the reference hands on is not "the solution of the ODE" but the output of scipy's Dormand-Prince 5(4) with its
// step-size controller, sampled through the 4th-order dense output of the step that covers each sample.  Wherever the
// thrust jumps inside a run (SequenceController with end_tau < 1, control.py:127-141, reachable from control.py:217) that
// output carries an O(h) error of its own which no other method reproduces; the reference's answer is the specification,
// so this kernel steps exactly as scipy does (scipy 1.18.1: integrate/_ivp/rk.py RungeKutta._step_impl, rk_step,
// RK45 tableau A/B/C/E/P, RkDenseOutput._call_impl; common.py select_initial_step, norm; ivp.py t_eval handling:
// samples with t_old < t_eval <= t, searchsorted side='right'):
//   * first step from select_initial_step (order 4), clamped to max_step; min_step = 10 ulp(t)
//   * a step is accepted when the RMS of err / (atol + rtol max(|y|, |y_new|)) is < 1; the next step is h * min(10,
//     0.9 err^-1/5) (at most h after a rejection), a rejected one shrinks by max(0.2, 0.9 err^-1/5)
//   * the last step is clipped to t = 1; FSAL: f(t + h, y_new) is both the 7th error stage and the next step's first
//   * samples: y_old + h Q [x, x^2, x^3, x^4], Q = K^T P, x = (t_eval - t_old) / h
// scipy is a third-party dependency the reference neither vendors nor pins; the tests pin this kernel to trajectories
// produced by the unmodified reference (tests/golden/propagate.npz, p0..p6: <= 4e-13).
//
// One thread per satellite; the 7 stage derivatives live in registers.  The chain of dependent stages (6 per step,
// ~1000 steps) bounds the run time, so (a) the tableau is pre-multiplied by the step (one FMA from the newest stage
// derivative to the next stage state) and (b) SPEC: the first stage of the NEXT step is evaluated with the predicted
// step size (the controller almost always returns max_step again) while the error norm of the current one is still
// being formed; a wrong prediction just recomputes that stage.  `lpw` lanes of every warp carry satellites (the rest
// exit at once): fewer satellites per warp spread a small batch over more SM sub-partitions.
#ifndef MPC_RK45_BODY
#ifndef MPC_PROPAGATE_RK45_KERNEL_CUH
#define MPC_PROPAGATE_RK45_KERNEL_CUH
#include "propagate_kernel.cuh"

namespace mpc {

struct Rk45Opts {
    double rtol, atol, max_step;
};

__device__ __forceinline__ double rk45_min_step(double t)
{
    // 10 * |nextafter(t, inf) - t|, t >= 0 (rk.py:119)
    const double up = (t == 0.0) ? 4.9406564584124654e-324 : __longlong_as_double(__double_as_longlong(t) + 1LL);
    return 10.0 * (up - t);
}

// 0.9 * err^-0.2 (rk.py SAFETY * error_norm ** error_exponent) from err^2
__device__ __forceinline__ double rk45_factor(double err2) { return 0.9 * pow(err2, -0.1); }

// RAG: a ragged batch (launched without progress words): T is the padded stride Tmax of y_out / u_out, lane s samples
// linspace(0, 1, T_sat[s]) and stores those T_sat[s] samples only (T_sat == nullptr: all T); its sequence table (stride
// C.table_len) has Ku_sat[s] columns (Ku_sat == nullptr: all C.table_len).  The steps do not depend on the samples.  The
// counts are clamped into the buffers (T_sat to [0, T], Ku_sat to [2, C.table_len]); the entry points validate them.
// PSC: per-satellite constants (mpc_propagate_batch_rk45_units) -- lane s integrates with its own PropParams, from the
// device table [n_sats] passed in place of the progress words (such a launch has none).  The table travels in an
// existing parameter because ptxas's register allocation of these ~250-register kernels follows the entry's parameter
// list: one more parameter changed the SASS of every single-constant instantiation.
// ATMO (propagate_rk45_atmo_kernel): drag under the altitude-dependent atmosphere A, in a kernel of its own for that
// reason; with PSC its per-satellite table is `asat` (AtmoSat: the constants and the satellite's length unit).
template <int BLOCK, int KIND, bool DRAG, bool J2, bool SPEC, bool RAG = false, bool PSC = false>
__global__ void __launch_bounds__(BLOCK)
propagate_rk45_kernel(const double *__restrict__ y0, const double *__restrict__ tf_arr, PropParams P, CtrlParams C,
                      Rk45Opts O, int n_sats, int T, int lpw, double *__restrict__ y_out, double *__restrict__ u_out,
                      int32_t *__restrict__ status, int32_t *__restrict__ n_steps, unsigned int *progress, int seg_len,
                      const int32_t *__restrict__ T_sat = nullptr, const int32_t *__restrict__ Ku_sat = nullptr)
{
#define MPC_RK45_ATMO 0
#define MPC_RK45_BODY
#include "propagate_rk45_kernel.cuh"
#undef MPC_RK45_BODY
#undef MPC_RK45_ATMO
}

// The RK45 replay with drag under the altitude-dependent atmosphere A (mpc_propagate_batch_rk45_atmo): always the ragged
// form (T_sat / Ku_sat == nullptr: the rectangular run), one-warp CTAs.  PSC: satellite s takes its constants and its
// length unit from asat[s] (P is then not read).  No progress words: never beside the discretization.  The speculative
// first stage (which changes the schedule, not the result) is on except for the table law: its knot-interval cache
// already holds that kernel at 254-255 registers, and log, exp and the series on top of the speculative stage's state
// spilled.
template <int KIND, bool J2, bool PSC>
__global__ void __launch_bounds__(32)
propagate_rk45_atmo_kernel(const double *__restrict__ y0, const double *__restrict__ tf_arr, PropParams P, CtrlParams C,
                           Rk45Opts O, int n_sats, int T, int lpw, double *__restrict__ y_out, double *__restrict__ u_out,
                           int32_t *__restrict__ status, int32_t *__restrict__ n_steps, const int32_t *__restrict__ T_sat,
                           const int32_t *__restrict__ Ku_sat, const __grid_constant__ AtmoParams Aparam,
                           const AtmoSat *__restrict__ asat)
{
    constexpr int BLOCK = 32;
    constexpr bool DRAG = true, SPEC = (KIND != 3), RAG = true;
    const AtmoParams *const A = &Aparam;
    unsigned int *progress = nullptr;
    const int seg_len = 0;
#define MPC_RK45_ATMO 1
#define MPC_RK45_BODY
#include "propagate_rk45_kernel.cuh"
#undef MPC_RK45_BODY
#undef MPC_RK45_ATMO
}

}  // namespace mpc

#endif  // MPC_PROPAGATE_RK45_KERNEL_CUH
#else   // MPC_RK45_BODY
// The body of the RK45 replay, included by this file into its two kernels above (and nowhere else).  It is one body for
// both; it is included rather than called because ptxas's code generation of these ~250-register kernels follows their
// structure: the same body behind an inlined call changed the SASS of every existing instantiation, and so does any
// difference in its text.  MPC_RK45_ATMO (0 / 1, set by the including kernel) switches the atmosphere's lines in by the
// preprocessor, so that the other kernels compile the text they always had.  In scope: the template flags BLOCK, KIND,
// DRAG, J2, SPEC, RAG, PSC, the kernel parameters and, with MPC_RK45_ATMO, A (the atmosphere) and asat (its
// per-satellite table, PSC).
#if MPC_RK45_ATMO
#define MPC_RK45_ATMO_ARGS , A, alen
#else
#define MPC_RK45_ATMO_ARGS
#endif
    // progress != nullptr (the overlapped pass, see propagate_kernel): window b of the discretization needs the samples
    // up to e_b = min((b+1) seg_len, T-1).  Lanes may take different numbers of steps here, so every LANE that has stored
    // sample e_b counts itself into progress[b] (fence first; lanes of a warp that arrive together are aggregated into
    // one atomic); the stream memory operation waits for progress[b] == n_sats.
    const int lane = threadIdx.x & 31;
    const int warp = (int)((blockIdx.x * (unsigned)BLOCK + threadIdx.x) >> 5);
    const int s = warp * lpw + lane;
    if (lane >= lpw || s >= n_sats) return;
    // PSC: `progress` is the table of per-satellite constants (see above), read here and then cleared, so that every use
    // of the progress words below sees none.  Nothing may read `progress` before this point.
    static_assert(alignof(PropParams) == alignof(double) && sizeof(PropParams) % alignof(double) == 0,
                  "the per-satellite table is an array of PropParams at a double-aligned address");
#if MPC_RK45_ATMO
    double alen;                  // metres per unit length of this satellite's constants
    if constexpr (PSC) {
        P = asat[s].P;
        alen = asat[s].len;
    } else {
        alen = A->len;
    }
#else
    if constexpr (PSC) {
        P = reinterpret_cast<const PropParams *>(progress)[s];
        progress = nullptr;
    }
#endif
    const double *tab = C.table ? C.table + (C.table_per_sat ? (long long)s * 3 * C.table_len : 0) : nullptr;
    // samples of this lane (T: the stride) and columns of its table (0: C.table_len), held inside the buffers
    const int Tn = (RAG && T_sat) ? min(max(T_sat[s], 0), T) : T;
    const int ku = (RAG && Ku_sat) ? min(max(Ku_sat[s], 2), C.table_len) : 0;
    const double end_tau = C.end_tau_arr ? C.end_tau_arr[s] : C.end_tau;
    const double tf = tf_arr[s];
    const double rtol = O.rtol, atol = O.atol, max_step = O.max_step;
    // Zero, constant and tangential thrust burn mass at a constant rate: every stage derivative of the mass is the same
    // number cm, the stage masses are m + h c_s cm (sum_l a_sl = c_s), its error estimate is zero (sum E = 0) and its dense
    // output is the straight line -- none of the 7-term sums is formed for that component (NC = 6).
    constexpr bool CM = (KIND != 3);
    constexpr int NC = CM ? 6 : 7;
    // err^2 <= sum (e_i h)^2 / (7 atol^2) because every scale is >= atol: when even that bound is below 0.09^10 the
    // controller's decision (accept, factor 10) is known without forming the 7 scales and their reciprocals
    const double tiny_thr = 3.486784401e-11 * 7.0 * atol * atol;
    double y[7], K[7][7];
#pragma unroll
    for (int c = 0; c < 7; ++c) y[c] = y0[(long long)s * 7 + c];
    double *yo = y_out + (long long)s * 7 * T;
    double *uo = u_out ? u_out + (long long)s * 3 * T : nullptr;
    // t_eval = np.linspace(0, 1, T): arange(T) * step, the last point exactly 1
    const double lstep = (Tn > 1) ? 1.0 / (double)(Tn - 1) : 0.0;
    int ti = 0;                   // next sample to write
    double te = 0.0;              // its time
    int bad = 0, fail = 0, steps = 0;
    double t = 0.0;

    FohCache foh;                 // KIND 3: knot interval of the table law shared by consecutive stage evaluations
    foh_cache_init(foh, RAG && ku > 0 ? ku : C.table_len, end_tau);
    FohCache *const fc = (KIND == 3) ? &foh : nullptr;
    bad |= prop_rhs<KIND, DRAG, J2, MPC_RK45_ATMO>(P, C, tab, end_tau, y, 0.0, K[0], nullptr, ku MPC_RK45_ATMO_ARGS);
    // ---- select_initial_step (common.py), f = tf * k ------------------------------------------------------------
    double h_abs;
    {
        double d0sq = 0.0, d1sq = 0.0, d2sq = 0.0, y1[7], k1[7];
#pragma unroll
        for (int i = 0; i < 7; ++i) {
            const double isc = 1.0 / (atol + fabs(y[i]) * rtol);
            d0sq = fma(y[i] * isc, y[i] * isc, d0sq);
            d1sq = fma(tf * K[0][i] * isc, tf * K[0][i] * isc, d1sq);
        }
        const double d0 = sqrt(d0sq * (1.0 / 7.0)), d1 = sqrt(d1sq * (1.0 / 7.0));
        double h0 = (d0 < 1e-5 || d1 < 1e-5) ? 1e-6 : 0.01 * d0 / d1;
        h0 = fmin(h0, 1.0);
#pragma unroll
        for (int i = 0; i < 7; ++i) y1[i] = fma(h0 * tf, K[0][i], y[i]);
        bad |= prop_rhs<KIND, DRAG, J2, MPC_RK45_ATMO>(P, C, tab, end_tau, y1, h0, k1, nullptr, ku MPC_RK45_ATMO_ARGS);
#pragma unroll
        for (int i = 0; i < 7; ++i) {
            const double q = tf * (k1[i] - K[0][i]) / (atol + fabs(y[i]) * rtol);
            d2sq = fma(q, q, d2sq);
        }
        const double d2 = sqrt(d2sq * (1.0 / 7.0)) / h0;
        const double h1 = (d1 <= 1e-15 && d2 <= 1e-15) ? fmax(1e-6, h0 * 1e-3) : pow(0.01 / fmax(d1, d2), 0.2);
        h_abs = fmin(fmin(100.0 * h0, h1), fmin(1.0, max_step));
    }

    bool have_k1 = false;         // SPEC: K[1] already holds the stage-1 derivative for the step size h_k1
    double h_k1 = 0.0;
    int bad_k1 = 0;
    while (t < 1.0 && !bad && !fail) {
        const double min_step = rk45_min_step(t);
        if (h_abs > max_step) h_abs = max_step;
        else if (h_abs < min_step) h_abs = min_step;
        bool accepted = false, rejected = false;
        double t_new = t, h = 0.0, yn[7];
        while (!accepted) {
            if (h_abs < min_step) {
                fail = 1;
                break;
            }
            t_new = t + h_abs;
            if (t_new - 1.0 > 0.0) t_new = 1.0;
            h = t_new - t;
            h_abs = fabs(h);
            const double hs = h * tf;
            // -- rk_step: stage states with the tableau pre-multiplied by the step ------------------------------------
            if (SPEC && have_k1 && h_k1 == h) {
                bad |= bad_k1;
            } else {
                double ys[7];
                const double a10 = hs * (1.0 / 5);
#pragma unroll
                for (int i = 0; i < NC; ++i) ys[i] = fma(K[0][i], a10, y[i]);
                if (CM) ys[6] = fma(K[0][6], hs * (1.0 / 5), y[6]);
                bad |= prop_rhs<KIND, DRAG, J2, MPC_RK45_ATMO>(P, C, tab, end_tau, ys, t + (1.0 / 5) * h, K[1], fc, ku MPC_RK45_ATMO_ARGS);
            }
            have_k1 = false;
            {
                double ys[7];
                const double a0 = hs * (3.0 / 40), a1 = hs * (9.0 / 40);
#pragma unroll
                for (int i = 0; i < NC; ++i) ys[i] = fma(K[1][i], a1, fma(K[0][i], a0, y[i]));
                if (CM) ys[6] = fma(K[0][6], hs * (3.0 / 10), y[6]);
                bad |= prop_rhs<KIND, DRAG, J2, MPC_RK45_ATMO>(P, C, tab, end_tau, ys, t + (3.0 / 10) * h, K[2], fc, ku MPC_RK45_ATMO_ARGS);
            }
            {
                double ys[7];
                const double a0 = hs * (44.0 / 45), a1 = hs * (-56.0 / 15), a2 = hs * (32.0 / 9);
#pragma unroll
                for (int i = 0; i < NC; ++i) ys[i] = fma(K[2][i], a2, fma(K[1][i], a1, fma(K[0][i], a0, y[i])));
                if (CM) ys[6] = fma(K[0][6], hs * (4.0 / 5), y[6]);
                bad |= prop_rhs<KIND, DRAG, J2, MPC_RK45_ATMO>(P, C, tab, end_tau, ys, t + (4.0 / 5) * h, K[3], fc, ku MPC_RK45_ATMO_ARGS);
            }
            {
                double ys[7];
                const double a0 = hs * (19372.0 / 6561), a1 = hs * (-25360.0 / 2187), a2 = hs * (64448.0 / 6561),
                             a3 = hs * (-212.0 / 729);
#pragma unroll
                for (int i = 0; i < NC; ++i)
                    ys[i] = fma(K[3][i], a3, fma(K[2][i], a2, fma(K[1][i], a1, fma(K[0][i], a0, y[i]))));
                if (CM) ys[6] = fma(K[0][6], hs * (8.0 / 9), y[6]);
                bad |= prop_rhs<KIND, DRAG, J2, MPC_RK45_ATMO>(P, C, tab, end_tau, ys, t + (8.0 / 9) * h, K[4], fc, ku MPC_RK45_ATMO_ARGS);
            }
            {
                double ys[7];
                const double a0 = hs * (9017.0 / 3168), a1 = hs * (-355.0 / 33), a2 = hs * (46732.0 / 5247),
                             a3 = hs * (49.0 / 176), a4 = hs * (-5103.0 / 18656);
#pragma unroll
                for (int i = 0; i < NC; ++i)
                    ys[i] = fma(K[4][i], a4, fma(K[3][i], a3, fma(K[2][i], a2, fma(K[1][i], a1, fma(K[0][i], a0, y[i])))));
                if (CM) ys[6] = fma(K[0][6], hs, y[6]);
                bad |= prop_rhs<KIND, DRAG, J2, MPC_RK45_ATMO>(P, C, tab, end_tau, ys, t + h, K[5], fc, ku MPC_RK45_ATMO_ARGS);
            }
            {
                const double b0 = hs * (35.0 / 384), b2 = hs * (500.0 / 1113), b3 = hs * (125.0 / 192),
                             b4 = hs * (-2187.0 / 6784), b5 = hs * (11.0 / 84);
#pragma unroll
                for (int i = 0; i < NC; ++i)
                    yn[i] = fma(K[5][i], b5, fma(K[4][i], b4, fma(K[3][i], b3, fma(K[2][i], b2, fma(K[0][i], b0, y[i])))));
                if (CM) yn[6] = fma(K[0][6], hs, y[6]);
                bad |= prop_rhs<KIND, DRAG, J2, MPC_RK45_ATMO>(P, C, tab, end_tau, yn, t + h, K[6], fc, ku MPC_RK45_ATMO_ARGS);
            }
            double k1n[7];
            int bad_n = 0;
            double h_pred = 0.0;
            if (SPEC) {
                // first stage of the next step, assuming the controller hands back max_step (it does unless the error norm
                // exceeds 0.59 or a step was rejected): independent of the error norm below, so the two chains overlap
                double ys[7], tp = t_new + fmin(h_abs * 10.0, max_step);
                if (tp - 1.0 > 0.0) tp = 1.0;
                h_pred = tp - t_new;
                const double a10 = (h_pred * tf) * (1.0 / 5);
#pragma unroll
                for (int i = 0; i < NC; ++i) ys[i] = fma(K[6][i], a10, yn[i]);
                if (CM) ys[6] = fma(K[0][6], a10, yn[6]);
                bad_n = prop_rhs<KIND, DRAG, J2, MPC_RK45_ATMO>(P, C, tab, end_tau, ys, t_new + (1.0 / 5) * h_pred, k1n, fc, ku MPC_RK45_ATMO_ARGS);
            }
            // -- error norm (rk.py _estimate_error_norm) ---------------------------------------------------------------
            double eh[NC], esum0 = 0.0;
#pragma unroll
            for (int i = 0; i < NC; ++i) {
                double e = K[6][i] * (1.0 / 40);
                e = fma(K[5][i], -22.0 / 525, e);
                e = fma(K[4][i], 17253.0 / 339200, e);
                e = fma(K[3][i], -71.0 / 1920, e);
                e = fma(K[2][i], 71.0 / 16695, e);
                e = fma(K[0][i], -71.0 / 57600, e);
                eh[i] = e * hs;
                esum0 = fma(eh[i], eh[i], esum0);
            }
            double err2 = 0.0;                         // error_norm^2 (the decisions below need no square root)
            if (!(esum0 <= tiny_thr)) {                // (also taken by a NaN)
                double esum = 0.0;
#pragma unroll
                for (int i = 0; i < NC; ++i) {
                    const double q = eh[i] * fast_rcp(atol + fmax(fabs(y[i]), fabs(yn[i])) * rtol);
                    esum = fma(q, q, esum);
                }
                err2 = esum * (1.0 / 7.0);
            }
            if (bad) break;
            if (err2 < 1.0) {
                // min(10, 0.9 err^-0.2) = 10  <=>  err <= 0.09^5: the common case needs no pow
                double factor = (err2 <= 3.486784401e-11) ? 10.0 : fmin(10.0, rk45_factor(err2));
                if (rejected) factor = fmin(1.0, factor);
                h_abs *= factor;
                accepted = true;
                if (SPEC) {
                    have_k1 = true;
                    h_k1 = h_pred;
                    bad_k1 = bad_n;
                }
            } else {
                // (a NaN error norm lands here: the step shrinks by 0.2 until it underflows min_step, as in scipy)
                const double f = rk45_factor(err2);
                h_abs *= (f > 0.2) ? f : 0.2;
                rejected = true;
            }
            if (++steps > (1 << 22)) fail = 1;
            if (fail) break;
            if (accepted && SPEC) {
                // K[1] of the next step (K[0] = K[6] is assigned below)
#pragma unroll
                for (int i = 0; i < 7; ++i) K[1][i] = k1n[i];
            }
        }
        if (bad || fail) break;
        // ---- samples with t_eval <= t_new off the dense output of this step (ivp.py:712-728, rk.py:723-737) ----------
        if (ti < Tn && te <= t_new) {
            // Q = K^T P; column 0 of P is e_1 and its row 1 is zero
            double Q[7][4];
            const double hs = h * tf;
#pragma unroll
            for (int i = 0; i < NC; ++i) {
                Q[i][0] = K[0][i];
                Q[i][1] = K[0][i] * (-8048581381.0 / 2820520608.0);
                Q[i][2] = K[0][i] * (8663915743.0 / 2820520608.0);
                Q[i][3] = K[0][i] * (-12715105075.0 / 11282082432.0);
            }
            // rows 2..6 of P; in SPEC mode K[1] already belongs to the next step (P's row 1 is zero: not needed)
#define MPC_QROW(l, p1, p2, p3)                     \
    _Pragma("unroll") for (int i = 0; i < NC; ++i) \
    {                                               \
        Q[i][1] = fma(K[l][i], p1, Q[i][1]);        \
        Q[i][2] = fma(K[l][i], p2, Q[i][2]);        \
        Q[i][3] = fma(K[l][i], p3, Q[i][3]);        \
    }
            MPC_QROW(2, 131558114200.0 / 32700410799.0, -68118460800.0 / 10900136933.0, 87487479700.0 / 32700410799.0)
            MPC_QROW(3, -1754552775.0 / 470086768.0, 14199869525.0 / 1410260304.0, -10690763975.0 / 1880347072.0)
            MPC_QROW(4, 127303824393.0 / 49829197408.0, -318862633887.0 / 49829197408.0, 701980252875.0 / 199316789632.0)
            MPC_QROW(5, -282668133.0 / 205662961.0, 2019193451.0 / 616988883.0, -1453857185.0 / 822651844.0)
            MPC_QROW(6, 40617522.0 / 29380423.0, -110615467.0 / 29380423.0, 69997945.0 / 29380423.0)
#undef MPC_QROW
            while (ti < Tn && te <= t_new) {
                const double xx = (te - t) / h;
                const double x2 = xx * xx, x3 = x2 * xx, x4 = x3 * xx;
                double ys[7];
#pragma unroll
                for (int i = 0; i < NC; ++i) {
                    const double q = fma(Q[i][3], x4, fma(Q[i][2], x3, fma(Q[i][1], x2, Q[i][0] * xx)));
                    ys[i] = fma(hs, q, y[i]);
                    yo[(long long)i * T + ti] = ys[i];
                }
                if (CM) {
                    ys[6] = fma(hs * xx, K[0][6], y[6]);
                    yo[(long long)6 * T + ti] = ys[6];
                }
                if (uo) {   // Discretizer.extract_uk (linearize_discretize.py:393-411) on the sample
                    double ux, uy, uz;
                    const double irs = fast_rsqrt(fma(ys[0], ys[0], fma(ys[1], ys[1], ys[2] * ys[2])));
                    ctrl_eval<KIND>(C, tab, end_tau, ys, irs, te, ux, uy, uz, ku);
                    uo[ti] = ux;
                    uo[T + ti] = uy;
                    uo[2 * (long long)T + ti] = uz;
                }
                // a window is released one sample after its last interval ends (its end node's input lookup may reach one
                // node further, see propagate_kernel), the last window at T-1
                // (a PSC launch passed its constants table in `progress` and cleared it at thread start: no progress words)
                if (progress && ti > 1 && (ti - 1) % seg_len == 0 && (ti - 1) < T - 1) {
                    const int b = (ti - 1) / seg_len - 1;
                    __threadfence();
                    const unsigned peers = __match_any_sync(__activemask(), b);
                    if (lane == __ffs(peers) - 1) atomicAdd(progress + b, (unsigned)__popc(peers));
                }
                if (progress && ti == T - 1 && ti > 0) {
                    const int b = (T - 2) / seg_len;
                    __threadfence();
                    const unsigned peers = __match_any_sync(__activemask(), b);
                    if (lane == __ffs(peers) - 1) atomicAdd(progress + b, (unsigned)__popc(peers));
                }
                ++ti;
                te = (ti == Tn - 1) ? 1.0 : (double)ti * lstep;
            }
        }
#pragma unroll
        for (int i = 0; i < 7; ++i) {
            y[i] = yn[i];
            K[0][i] = K[6][i];
        }
        t = t_new;
    }
    if (bad || fail) {
        // the reference raises here (simulator.py:135-136) or solve_ivp reports failure: nothing is handed on.  The
        // samples not yet written become NaN, and the windows waiting on them are released.
        const double qnan = __longlong_as_double(0x7ff8000000000000LL);
        for (; ti < Tn; ++ti) {
#pragma unroll
            for (int c = 0; c < 7; ++c) yo[(long long)c * T + ti] = qnan;
            if (uo) {
                uo[ti] = qnan;
                uo[T + ti] = qnan;
                uo[2 * (long long)T + ti] = qnan;
            }
            if (progress && ti > 1 && (ti - 1) % seg_len == 0 && (ti - 1) < T - 1) {   // (nullptr in a PSC launch)
                __threadfence();
                atomicAdd(progress + ((ti - 1) / seg_len - 1), 1u);
            }
            if (progress && ti == T - 1 && ti > 0) {
                __threadfence();
                atomicAdd(progress + (T - 2) / seg_len, 1u);
            }
        }
    }
#if MPC_RK45_ATMO
    // prop_rhs reports the atmosphere's range as 4 (MPC_ST_ATMO); a non-positive mass takes precedence
    if (status) status[s] = bad ? ((bad & 1) ? 1 : 4) : (fail ? 3 : 0);
#else
    if (status) status[s] = bad ? 1 : (fail ? 3 : 0);
#endif
    if (n_steps) n_steps[s] = steps;
#undef MPC_RK45_ATMO_ARGS
#endif  // MPC_RK45_BODY
