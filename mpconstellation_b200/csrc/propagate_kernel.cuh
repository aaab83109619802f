// propagate_kernel.cuh -- batched nonlinear orbit propagation, one thread per satellite.
//
// Replaces Simulator.get_trajectory_ODE (simulator.py:164-189): integrate
//   y' = tf * f(y, u(y,tau))   over tau in [0,1]          (simulator.py:115-161)
// and sample at linspace(0,1,T).  The reference's solve_ivp(RK45, max_step=0.001) becomes
// fixed-step classical RK4 with n_sub steps between consecutive samples.  The controller law
// u(y,tau) (control.py) is evaluated on the device at every stage, and once more at every
// sample to produce Discretizer.extract_uk's output (linearize_discretize.py:393-411).
//
// Propagation is sequential in tau, so this kernel is latency-bound by construction: one warp per
// CTA spreads the satellites over as many SMs as possible.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "discretize_kernel.cuh"

namespace mpc {

struct PropParams {
    double mu, kj2, inv_ve;
    double drag_k;  // 0.5 * C_D * S * (rho_atm / RHO)   (simulator.py:152)
    int include_j2, include_drag;
};

struct CtrlParams {
    int kind, table_len, table_per_sat, pad;
    double t0, t1, t2;  // constant thrust vector, or t0 = tangential magnitude
    double end_tau;
    const double *table;
    const double *end_tau_arr;  // optional per-satellite end_tau
};

// Controller law, compile-time kind (straight-line code per law); `ir` = 1/|r| of y, already needed by gravity.
// ku > 0: the table law of a ragged batch -- this satellite's table has ku columns, stored with the stride C.table_len
template <int KIND>
__device__ __forceinline__ void ctrl_eval(const CtrlParams &C, const double *__restrict__ tab, double end_tau,
                                          const double (&y)[7], double ir, double tau, double &ux, double &uy,
                                          double &uz, int ku = 0)
{
    ux = uy = uz = 0.0;
    if (KIND == 1) {  // control.py:47-53
        ux = C.t0;
        uy = C.t1;
        uz = C.t2;
    } else if (KIND == 2) {  // control.py:66-84: thrust along t_hat = h_hat x r_hat
        const double hx = fma(y[1], y[5], -y[2] * y[4]);
        const double hy = fma(y[2], y[3], -y[0] * y[5]);
        const double hz = fma(y[0], y[4], -y[1] * y[3]);
        const double sc = C.t0 * ir * fast_rsqrt(fma(hx, hx, fma(hy, hy, hz * hz)));   // mag / (|h| |r|)
        ux = sc * fma(hy, y[2], -hz * y[1]);
        uy = sc * fma(hz, y[0], -hx * y[2]);
        uz = sc * fma(hx, y[1], -hy * y[0]);
    } else if (KIND == 3) {  // control.py:104-143: FOH table on tau/end_tau, zero after end_tau
        if (tau <= end_tau) {
            const int ld = C.table_len, Ku = (ku > 0) ? ku : ld;
            const double t = tau / end_tau;
            if (t == 1.0) {
                ux = tab[Ku - 1];
                uy = tab[ld + Ku - 1];
                uz = tab[2 * ld + Ku - 1];
            } else {
                const double km1 = (double)(Ku - 1);
                int k = (int)floor(t * km1);
                k = min(max(k, 0), Ku - 2);
                const double lo = (double)k / km1, hi = (double)(k + 1) / km1;
                const double iw = 1.0 / (hi - lo);
                const double ln = (hi - t) * iw, lp = (t - lo) * iw;
                ux = fma(ln, tab[k], lp * tab[k + 1]);
                uy = fma(ln, tab[ld + k], lp * tab[ld + k + 1]);
                uz = fma(ln, tab[2 * ld + k], lp * tab[2 * ld + k + 1]);
            }
        }
    }
}

// The FOH table law (KIND 3) evaluated through a one-entry cache of its knot interval.  The integrator's steps (0.001) are
// short against the knot spacing (end_tau / (Ku - 1)), so consecutive stage times almost always fall between the same
// two knots: the three divisions that place the interval (k / (Ku-1), (k+1) / (Ku-1), 1 / (hi - lo)) and the six table
// loads are then the previous evaluation's (same values as ctrl_eval<3>; see ctrl_eval_foh_cached for the two places where
// the arithmetic differs from it by a rounding).
struct FohCache {
    int k;
    double lo, hi, iw, a[3], b[3];
    double km1, inv_et;          // Ku - 1 and 1 / end_tau (set once, foh_cache_init)
};

__device__ __forceinline__ void foh_cache_init(FohCache &fc, int Ku, double end_tau)
{
    fc.k = -1;
    fc.km1 = (double)(Ku - 1);
    fc.inv_et = 1.0 / end_tau;
}

// The refill is a real call (the result comes back by value, so the cache itself stays in registers): inlined into the
// seven stage evaluations of a step it made the hot loop 28 KB of code, most of it never executed.
__device__ __noinline__ FohCache foh_cache_fill(const double *__restrict__ tab, int Ku, int k, double km1, double inv_et)
{
    FohCache fc;
    fc.k = k;
    fc.km1 = km1;
    fc.inv_et = inv_et;
    fc.lo = (double)k / km1;
    fc.hi = (double)(k + 1) / km1;
    fc.iw = 1.0 / (fc.hi - fc.lo);
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        fc.a[i] = tab[i * Ku + k];
        fc.b[i] = tab[i * Ku + k + 1];
    }
    return fc;
}

// Straight-line on the common path (the only branch is the refill): the quotient tau / end_tau from the stored reciprocal
// and one correction step (q = tau y; q += (tau - q end_tau) y: the correctly rounded quotient but for rare last-bit
// cases), the end point t = 1 through the last interval (lambda- = 0 there) and the cut-off after end_tau by a select --
// the branches and slow-path guards of the literal form kept ptxas from scheduling across the seven stage evaluations.
__device__ __forceinline__ void ctrl_eval_foh_cached(const CtrlParams &C, const double *__restrict__ tab, double end_tau,
                                                     double tau, FohCache &fc, double &ux, double &uy, double &uz, int ku = 0)
{
    const int Ku = (ku > 0) ? ku : C.table_len;
    double t = tau * fc.inv_et;
    t = fma(fma(-t, end_tau, tau), fc.inv_et, t);
    int k = (int)(t * fc.km1);
    k = min(max(k, 0), Ku - 2);
    if (k != fc.k) fc = foh_cache_fill(tab, C.table_len, k, fc.km1, fc.inv_et);
    const double ln = (fc.hi - t) * fc.iw, lp = (t - fc.lo) * fc.iw;
    const bool on = tau <= end_tau;
    const double vx = fma(ln, fc.a[0], lp * fc.b[0]), vy = fma(ln, fc.a[1], lp * fc.b[1]), vz = fma(ln, fc.a[2], lp * fc.b[2]);
    ux = on ? vx : 0.0;
    uy = on ? vy : 0.0;
    uz = on ? vz : 0.0;
}

// An altitude-dependent atmosphere (mpc_atmosphere, fitted and checked on the host: atmosphere.fit_atmosphere): log rho
// as a Chebyshev series in t = (log h - s_mid) s_ihalf, h = |r| len - r_earth the altitude in metres, valid on
// [h_min, h_max].  With it the drag coefficient drag_k of PropParams is 0.5 C_D S / RHO and the density rho(h) multiplies
// it at every stage evaluation.
constexpr int kAtmoCheb = 32;
struct AtmoParams {
    double coef[kAtmoCheb];
    double s_mid, s_ihalf, h_min, h_max, r_earth;
    double len;                 // metres per unit length of the launch-wide constants (per-satellite: AtmoSat::len)
    int n, pad;
};
// one satellite's entry of the per-satellite constants table of the atmosphere kernels
struct AtmoSat {
    PropParams P;
    double len;
};

__device__ __forceinline__ double atmo_density(const AtmoParams &A, double h)
{
    const double t = (log(h) - A.s_mid) * A.s_ihalf;
    // Clenshaw: sum_k c_k T_k(t)
    double b1 = 0.0, b2 = 0.0;
    const double t2 = 2.0 * t;
    for (int k = A.n - 1; k >= 1; --k) {
        const double b = fma(t2, b1, A.coef[k]) - b2;
        b2 = b1;
        b1 = b;
    }
    return exp(fma(t, b1, A.coef[0]) - b2);
}

// f(y,u) without the tf factor (simulator.py:130-160); returns nonzero on non-positive mass (1) and, with ATMO, an
// altitude outside the fitted atmosphere (4, MPC_ST_ATMO).  fc: the knot-interval cache of the table law (KIND 3 only;
// nullptr = evaluate the law from scratch); ku: see ctrl_eval; A / len: the atmosphere and the satellite's length unit
template <int KIND, bool DRAG, bool J2, bool ATMO = false>
__device__ __forceinline__ int prop_rhs(const PropParams &P, const CtrlParams &C, const double *__restrict__ tab,
                                        double end_tau, const double (&y)[7], double tau, double (&dy)[7],
                                        FohCache *fc = nullptr, int ku = 0, const AtmoParams *A = nullptr, double len = 0.0)
{
    int out = 0;
    const double m = y[6];
    const double r2 = fma(y[0], y[0], fma(y[1], y[1], y[2] * y[2]));
    const double ir = fast_rsqrt(r2);
    const double ir2 = ir * ir;
    const double mu3 = P.mu * ir * ir2;
    const double im = fast_rcp(m);
    double ux = 0.0, uy = 0.0, uz = 0.0, ax, ay, az;
    if (KIND == 2) {
        // the tangential law (ctrl_eval<2>) with 1/m folded into its scale: u/m = (mag / (|h| |r| m)) (h x r) -- two
        // multiplications per evaluation fewer than forming u first (|u| is the constant mag, below)
        const double hx = fma(y[1], y[5], -y[2] * y[4]);
        const double hy = fma(y[2], y[3], -y[0] * y[5]);
        const double hz = fma(y[0], y[4], -y[1] * y[3]);
        const double scm = C.t0 * ir * fast_rsqrt(fma(hx, hx, fma(hy, hy, hz * hz))) * im;
        ax = fma(scm, fma(hy, y[2], -hz * y[1]), -mu3 * y[0]);
        ay = fma(scm, fma(hz, y[0], -hx * y[2]), -mu3 * y[1]);
        az = fma(scm, fma(hx, y[1], -hy * y[0]), -mu3 * y[2]);
    } else {
        if (KIND == 3 && fc) ctrl_eval_foh_cached(C, tab, end_tau, tau, *fc, ux, uy, uz, ku);
        else ctrl_eval<KIND>(C, tab, end_tau, y, ir, tau, ux, uy, uz, ku);
        ax = fma(-mu3, y[0], ux * im);
        ay = fma(-mu3, y[1], uy * im);
        az = fma(-mu3, y[2], uz * im);
    }
    if (DRAG) {
        const double v2 = fma(y[3], y[3], fma(y[4], y[4], y[5] * y[5]));
        const double vn = (v2 > 0.0) ? v2 * fast_rsqrt(v2) : 0.0;
        double kd = P.drag_k;
        if constexpr (ATMO) {
            const double h = fma(r2 * ir, len, -A->r_earth);
            if (h < A->h_min || h > A->h_max) out = 4;
            kd *= atmo_density(*A, h);
        }
        const double c = -kd * im * vn;
        ax = fma(c, y[3], ax);
        ay = fma(c, y[4], ay);
        az = fma(c, y[5], az);
    }
    if (J2) {
        const double nz = y[2] * ir;
        const double q5 = 5.0 * nz * nz;
        const double k5 = P.kj2 * ir2 * ir2 * ir;
        const double c1 = k5 * (q5 - 1.0);
        ax = fma(c1, y[0], ax);
        ay = fma(c1, y[1], ay);
        az = fma(k5 * (q5 - 3.0), y[2], az);
    }
    double un;
    if (KIND == 0) un = 0.0;
    else if (KIND == 2) un = fabs(C.t0);          // |t_hat| = 1: the tangential law has constant magnitude
    else {
        const double uu = fma(ux, ux, fma(uy, uy, uz * uz));
        un = (uu > 0.0) ? uu * fast_rsqrt(uu) : 0.0;
    }
    dy[0] = y[3];
    dy[1] = y[4];
    dy[2] = y[5];
    dy[3] = ax;
    dy[4] = ay;
    dy[5] = az;
    dy[6] = -un * P.inv_ve;
    if constexpr (ATMO) return (int)!(m > 0.0) | out;
    else return !(m > 0.0);
}

template <int BLOCK, int KIND, bool DRAG, bool J2>
__global__ void __launch_bounds__(BLOCK)
propagate_kernel(const double *__restrict__ y0, const double *__restrict__ tf_arr, PropParams P, CtrlParams C,
                 int n_sats, int T, int n_sub, double *__restrict__ y_out, double *__restrict__ u_out,
                 int32_t *__restrict__ status, unsigned int *progress = nullptr, int seg_len = 0)
{
    // progress != nullptr: the kernel publishes how far it has come.  Window b of the discretization covers the intervals
    // [b seg_len, min((b+1) seg_len, T-1)) and needs the samples up to min(e_b + 1, T-1), e_b = min((b+1) seg_len, T-1)
    // (one past its last interval: see below): once every lane of a warp has stored that sample, the warp adds 1 to
    // progress[b] (stores fenced first).  A stream memory operation on the
    // discretization's stream waits for progress[b] == number of warps (mpc_propagate_discretize): no kernel ever spins.
    const int s = blockIdx.x * BLOCK + threadIdx.x;
    if (s >= n_sats) return;
    const double *tab = C.table ? C.table + (C.table_per_sat ? (long long)s * 3 * C.table_len : 0) : nullptr;
    const double end_tau = C.end_tau_arr ? C.end_tau_arr[s] : C.end_tau;
    const double tf = tf_arr[s];
    double y[7], k1[7], k2[7], k3[7], k4[7], yt[7];
#pragma unroll
    for (int c = 0; c < 7; ++c) y[c] = y0[(long long)s * 7 + c];
    const double Tm1 = (T > 1) ? (double)(T - 1) : 1.0;
    const double h = 1.0 / (Tm1 * (double)n_sub);
    const double hs = tf * h, hh = 0.5 * hs, hs_6 = hs * (1.0 / 6.0);
    double *yo = y_out + (long long)s * 7 * T;
    double *uo = u_out ? u_out + (long long)s * 3 * T : nullptr;
    int bad = 0;
    for (int j = 0; j < T; ++j) {
        const double tau_j = (T > 1) ? (double)j / Tm1 : 0.0;
        if (bad) {
            const double qnan = __longlong_as_double(0x7ff8000000000000LL);
#pragma unroll
            for (int c = 0; c < 7; ++c) yo[(long long)c * T + j] = qnan;
            if (uo) {
                uo[j] = qnan;
                uo[T + j] = qnan;
                uo[2 * (long long)T + j] = qnan;
            }
        } else {
#pragma unroll
            for (int c = 0; c < 7; ++c) yo[(long long)c * T + j] = y[c];
            if (uo) {
                double ux, uy, uz;
                const double irs = fast_rsqrt(fma(y[0], y[0], fma(y[1], y[1], y[2] * y[2])));
                ctrl_eval<KIND>(C, tab, end_tau, y, irs, tau_j, ux, uy, uz);
                uo[j] = ux;
                uo[T + j] = uy;
                uo[2 * (long long)T + j] = uz;
            }
        }
        // Window b needs the samples up to e_b + 1 (e_b = min((b+1) seg_len, T-1)): its last interval reads the inputs of
        // node e_b, and the reference's global-grid lookup of that end node may interpolate towards node e_b + 1
        // (ref_node_input).  So a window is released one sample later than its last interval ends, the last one at T-1.
        if (progress && j > 1 && (j - 1) % seg_len == 0 && (j - 1) < T - 1) {
            __threadfence();
            __syncwarp();
            if ((threadIdx.x & 31) == 0) atomicAdd(progress + ((j - 1) / seg_len - 1), 1u);
        }
        if (progress && j == T - 1 && j > 0) {
            __threadfence();
            __syncwarp();
            if ((threadIdx.x & 31) == 0) atomicAdd(progress + (T - 2) / seg_len, 1u);
        }
        if (bad) continue;
        if (j == T - 1) break;
        const double tau_n = (double)(j + 1) / Tm1;
        for (int n = 0; n < n_sub; ++n) {
            // step end points from integers: the last one is exactly tau_{j+1} (1.0 at the end of the run)
            const double t0 = (n == 0) ? tau_j : fma((double)n, h, tau_j);
            const double t1 = (n == n_sub - 1) ? tau_n : fma((double)(n + 1), h, tau_j);
            const double tm = 0.5 * (t0 + t1);
            bad |= prop_rhs<KIND, DRAG, J2>(P, C, tab, end_tau, y, t0, k1);
#pragma unroll
            for (int c = 0; c < 7; ++c) yt[c] = fma(hh, k1[c], y[c]);
            bad |= prop_rhs<KIND, DRAG, J2>(P, C, tab, end_tau, yt, tm, k2);
#pragma unroll
            for (int c = 0; c < 7; ++c) yt[c] = fma(hh, k2[c], y[c]);
            bad |= prop_rhs<KIND, DRAG, J2>(P, C, tab, end_tau, yt, tm, k3);
#pragma unroll
            for (int c = 0; c < 7; ++c) yt[c] = fma(hs, k3[c], y[c]);
            bad |= prop_rhs<KIND, DRAG, J2>(P, C, tab, end_tau, yt, t1, k4);
            if (bad) break;
#pragma unroll
            for (int c = 0; c < 7; ++c) y[c] = fma(hs_6, (k1[c] + k4[c]) + 2.0 * (k2[c] + k3[c]), y[c]);
        }
    }
    if (status) status[s] = bad ? 1 : 0;
}

// FP64 FMA throughput probe: 8 independent chains per thread, `iters` rounds.
__global__ void __launch_bounds__(256) fp64_probe_kernel(double *out, int iters, double seed)
{
    double a0 = seed + threadIdx.x, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6,
           a7 = a0 + 7;
    const double b = 0.999999, c = 1e-9;
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int r = 0; r < 8; ++r) {
            a0 = fma(a0, b, c);
            a1 = fma(a1, b, c);
            a2 = fma(a2, b, c);
            a3 = fma(a3, b, c);
            a4 = fma(a4, b, c);
            a5 = fma(a5, b, c);
            a6 = fma(a6, b, c);
            a7 = fma(a7, b, c);
        }
    }
    out[(long long)blockIdx.x * blockDim.x + threadIdx.x] = ((a0 + a1) + (a2 + a3)) + ((a4 + a5) + (a6 + a7));
}

__global__ void fill_kernel(double *__restrict__ p, long long n, double v)
{
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) p[i] = v;
}

// Push the columns [off, off+nc) of a SoA result (all rows but the structurally constant 42..48) from the local buffer
// to n_peers peer-mapped buffers of the same layout: the SM-driven alternative to the copy engines for the all-gather
// (a store to a peer sustains the full NVLink rate from a handful of CTAs; scripts/micro/nvl_store.cu).
struct PeerTab {
    double *p[8];
};

__global__ void __launch_bounds__(256)
push_chunk_kernel(const double *__restrict__ src, PeerTab peers, int n_peers, long long pitch, long long off, long long nc)
{
    const long long n_el = 98 * nc;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n_el; i += (long long)gridDim.x * blockDim.x) {
        const int r98 = (int)(i / nc);
        const long long c = i - (long long)r98 * nc;
        const int row = r98 < 42 ? r98 : r98 + 7;
        const long long a = (long long)row * pitch + off + c;
        const double v = src[a];
        for (int d = 0; d < n_peers; ++d) peers.p[d][a] = v;
    }
}

}  // namespace mpc
