// conjunction_kernel.cuh -- close-approach screening of a constellation's trajectories (mpc_screen_conjunctions).
//
// Input: the SI states of N satellites at T common instants t_k = k h, h = D / (T - 1).  Between samples k and k + 1
// every satellite follows the cubic Hermite curve through its positions and velocities at the two samples,
//     p(s) = B0 b0(s) + B1 b1(s) + B2 b2(s) + B3 b3(s),  s = (t - t_k) / h in [0, 1],
//     B0 = r_k,  B1 = r_k + h v_k / 3,  B2 = r_{k+1} - h v_{k+1} / 3,  B3 = r_{k+1}
// (b_i the cubic Bernstein polynomials), so a pair's distance d(t) is C^1 over the whole run.  An event is a local
// minimum of d with d < threshold; a minimum belongs to the interval whose half-open [t_k, t_{k+1}) holds it (the last
// interval is closed), t = 0 counts when d increases there and t = D when d does not increase there.
//
// Two kernels:
//   conj_prepass_kernel  one thread per (satellite, sample): the SI states in the k-major layout X [T][6][N] and, per
//                        interval, a sphere (centre, radius) S [T-1][4][N] that contains the satellite's Hermite segment
//                        (conj_sphere); a non-finite end sample gives a NaN sphere and counts in skipped[s].
//   conj_pair_kernel     one CTA per (i-block, j-block) tile of the upper triangle (32 x 32 satellites); both blocks'
//                        states and spheres for kConjKc intervals at a time in shared memory; one thread per pair and
//                        interval.  A pair-interval whose spheres are farther apart than rho_i + rho_j + threshold
//                        cannot come closer than the threshold and is skipped; the others go to conj_interval.  Events
//                        are appended through a warp-aggregated atomic counter to a buffer of fixed capacity; the
//                        counter ends at the full count even when it exceeds the capacity.
//
// The per-interval functions (conj_sphere, conj_interval) and the pre-pass compile for the host as well (the tests build
// them with g++); the pair kernel, which needs the warp collectives and a CTA barrier, is device-only.
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

namespace mpc {

constexpr int kConjTile = 32;        // satellites per side of a pair tile
constexpr int kConjThreads = 256;    // threads of a pair CTA: 8 warps, 4 pairs per thread per interval
constexpr int kConjKc = 8;           // intervals staged in shared memory per round
constexpr int kConjDepth = 20;       // depth cap of the Bernstein subdivision: pieces of 2^-20 of an interval
constexpr int kConjMaxEv = 6;        // events one pair-interval can report (at most 4 local minima of a sextic on [0, 1])
constexpr int kConjFlagDepth = 1;    // flag bit: the subdivision reached kConjDepth before isolating this minimum

// one event as the C-ABI returns it (mpc_conjunction)
struct ConjRecord {
    int32_t i, j, k, flags;
    double t_ca, d_min, v_rel;
};

// one event of a pair-interval: s in [0, 1], distance (m), relative speed (m/s)
struct ConjEvent {
    double s, d, v;
    int flags;
};

__device__ __forceinline__ bool conj_finite6(const double *q)
{
    bool ok = true;
    for (int c = 0; c < 6; ++c) ok = ok && isfinite(q[c]);
    return ok;
}

// Bounding sphere of one satellite's Hermite segment on an interval: q0, q1 = (r, v) at its two samples (SI), h its
// length in seconds -> out = (centre x, y, z, radius).
//
// The bound: p(s) = sum_i B_i b_i(s) with b_i >= 0 and sum_i b_i = 1 on [0, 1], so p(s) lies in the convex hull of the
// control points B0..B3 and, for any centre c, |p(s) - c| <= max_i |B_i - c| =: r.  c is the mean of the B_i.  The
// radius returned is rho = r + 1e-12 (|c| + r): the relative margin covers the rounding of c, of the B_i here and of
// the pair's relative cubic in conj_interval (all a few ulp of |c| + r, 1e-16 relative), so the filter
//     |c_i - c_j| <= rho_i + rho_j + threshold
// never discards a pair-interval on which the Hermite model comes closer than the threshold.
// A non-finite sample gives a NaN centre and radius: every comparison with it is false.
__device__ __forceinline__ void conj_sphere(const double *q0, const double *q1, double h, double *out)
{
    double B[4][3], c[3];
    for (int x = 0; x < 3; ++x) {
        B[0][x] = q0[x];
        B[1][x] = q0[x] + h * q0[3 + x] * (1.0 / 3.0);
        B[2][x] = q1[x] - h * q1[3 + x] * (1.0 / 3.0);
        B[3][x] = q1[x];
        c[x] = 0.25 * ((B[0][x] + B[1][x]) + (B[2][x] + B[3][x]));
    }
    double r2 = 0.0;
    for (int i = 0; i < 4; ++i) {
        const double dx = B[i][0] - c[0], dy = B[i][1] - c[1], dz = B[i][2] - c[2];
        r2 = fmax(r2, dx * dx + dy * dy + dz * dz);
    }
    const double r = sqrt(r2);
    const double rho = r + 1e-12 * (sqrt(c[0] * c[0] + c[1] * c[1] + c[2] * c[2]) + r);
    const bool ok = conj_finite6(q0) && conj_finite6(q1);
    const double nan = __longlong_as_double(0x7ff8000000000000LL);
    out[0] = ok ? c[0] : nan;
    out[1] = ok ? c[1] : nan;
    out[2] = ok ? c[2] : nan;
    out[3] = ok ? rho : nan;
}

// g(s) = (1/2) d/ds |dp(s)|^2 (a quintic, power basis c[0..5]) and g'(s) at s
__device__ __forceinline__ void conj_g(const double *c, double s, double &g, double &dg)
{
    g = c[5];
    dg = 0.0;
    for (int n = 4; n >= 0; --n) {
        dg = fma(dg, s, g);
        g = fma(g, s, c[n]);
    }
}

// the rising root of g in [a, b] (g(a) <= 0 < g(b)) by safeguarded Newton-bisection: a Newton step from the current
// iterate when it stays inside the bracket, the midpoint otherwise; the bracket shrinks at every step
__device__ __forceinline__ double conj_refine(const double *c, double a, double b)
{
    double x = 0.5 * (a + b);
    for (int it = 0; it < 100; ++it) {
        double g, dg;
        conj_g(c, x, g, dg);
        if (g <= 0.0) a = x;
        else b = x;
        double xn = x - g / dg;
        if (!(dg > 0.0) || !(xn > a && xn < b)) xn = 0.5 * (a + b);
        const bool done = fabs(xn - x) <= 2e-16 || b - a <= 4e-16;
        x = xn;
        if (done) break;
    }
    return x;
}

// Bernstein coefficients (degree 5) of g(lo + w t), t in [0, 1]: Taylor shift of the power form to lo, scaled by w
__device__ __forceinline__ void conj_piece(const double *c, double lo, double w, double *b)
{
    double d[6];
    for (int n = 0; n < 6; ++n) d[n] = c[n];
    for (int m = 0; m < 5; ++m)                 // synthetic division: d[n] <- g^(n)(lo) / n!
        for (int n = 4; n >= m; --n) d[n] = fma(d[n + 1], lo, d[n]);
    double wn = w;
    for (int n = 1; n < 6; ++n) {
        d[n] *= wn;
        wn *= w;
    }
    // b_k = sum_{i <= k} C(k, i) / C(5, i) d_i
    b[0] = d[0];
    b[1] = d[0] + 0.2 * d[1];
    b[2] = d[0] + 0.4 * d[1] + 0.1 * d[2];
    b[3] = d[0] + 0.6 * d[1] + 0.3 * d[2] + 0.1 * d[3];
    b[4] = d[0] + 0.8 * d[1] + 0.6 * d[2] + 0.4 * d[3] + 0.2 * d[4];
    b[5] = d[0] + d[1] + d[2] + d[3] + d[4] + d[5];
}

// The events of one pair-interval.  qi0 / qi1, qj0 / qj1: (r, v) of satellites i and j at the interval's two samples
// (SI), h its length (s), thr the threshold (m); first / last: the interval starts / ends the run.  -> number of events
// written to ev (s ascending).
//
// The relative position dp(s) = ri(s) - rj(s) is the cubic Hermite curve of P0 = ri0 - rj0, M0 = h (vi0 - vj0),
// P1, M1: dp(s) = A0 + A1 s + A2 s^2 + A3 s^3 with A0 = P0, A1 = M0, A2 = 3 (P1 - P0) - 2 M0 - M1,
// A3 = 2 (P0 - P1) + M0 + M1.  The minima of d = |dp| are those of f = |dp|^2, i.e. the roots of the quintic
// g = dp . dp' at which g changes sign from <= 0 to > 0.  They are isolated in Bernstein form: a dyadic piece of [0, 1]
// whose coefficients show no sign change holds no such root; one change (first coefficient <= 0 < last) holds exactly
// one, which conj_refine polishes; more changes split the piece, down to kConjDepth.  A piece that still shows several
// changes at that depth is reported at its rising root (or, when g has the same sign at both ends, at its midpoint)
// with kConjFlagDepth set.  The pieces are visited depth first, left to right, without a stack: the next piece after a
// leaf (idx, depth) is the right sibling of the nearest ancestor that is a left child.
__device__ __forceinline__ int conj_interval(const double *qi0, const double *qi1, const double *qj0, const double *qj1,
                                             double h, double thr, bool first, bool last, ConjEvent *ev)
{
    double A0[3], A1[3], A2[3], A3[3];
    for (int x = 0; x < 3; ++x) {
        const double P0 = qi0[x] - qj0[x], P1 = qi1[x] - qj1[x];
        const double M0 = h * (qi0[3 + x] - qj0[3 + x]), M1 = h * (qi1[3 + x] - qj1[3 + x]);
        A0[x] = P0;
        A1[x] = M0;
        A2[x] = 3.0 * (P1 - P0) - 2.0 * M0 - M1;
        A3[x] = 2.0 * (P0 - P1) + M0 + M1;
    }
    auto dot = [](const double *a, const double *b) { return a[0] * b[0] + a[1] * b[1] + a[2] * b[2]; };
    // f = |dp|^2 in power form e[0..6]; its Bernstein coefficients bound f from below on [0, 1]: no minimum below the
    // threshold when the smallest is above thr^2 (with a margin for the rounding of the coefficients)
    const double a00 = dot(A0, A0), a01 = dot(A0, A1), a02 = dot(A0, A2), a03 = dot(A0, A3);
    const double a11 = dot(A1, A1), a12 = dot(A1, A2), a13 = dot(A1, A3), a22 = dot(A2, A2), a23 = dot(A2, A3);
    const double a33 = dot(A3, A3);
    {
        const double e0 = a00, e1 = 2.0 * a01, e2 = 2.0 * a02 + a11, e3 = 2.0 * (a03 + a12), e4 = 2.0 * a13 + a22;
        const double e5 = 2.0 * a23, e6 = a33;
        // b_k = sum_{i <= k} C(k, i) / C(6, i) e_i
        double lb = e0;
        lb = fmin(lb, e0 + e1 * (1.0 / 6.0));
        lb = fmin(lb, e0 + e1 * (2.0 / 6.0) + e2 * (1.0 / 15.0));
        lb = fmin(lb, e0 + e1 * (3.0 / 6.0) + e2 * (3.0 / 15.0) + e3 * (1.0 / 20.0));
        lb = fmin(lb, e0 + e1 * (4.0 / 6.0) + e2 * (6.0 / 15.0) + e3 * (4.0 / 20.0) + e4 * (1.0 / 15.0));
        lb = fmin(lb, e0 + e1 * (5.0 / 6.0) + e2 * (10.0 / 15.0) + e3 * (10.0 / 20.0) + e4 * (5.0 / 15.0) + e5 * (1.0 / 6.0));
        lb = fmin(lb, e0 + e1 + e2 + e3 + e4 + e5 + e6);
        const double scale = a00 + a11 + a22 + a33;
        if (!(lb <= thr * thr * (1.0 + 1e-9) + 1e-12 * scale)) return 0;
    }
    // g = dp . dp' = sum_n c_n s^n
    double c[6];
    c[0] = a01;
    c[1] = 2.0 * a02 + a11;
    c[2] = 3.0 * (a03 + a12);
    c[3] = 4.0 * a13 + 2.0 * a22;
    c[4] = 5.0 * a23;
    c[5] = 3.0 * a33;

    int n = 0;
    auto emit = [&](double s, int flags) {
        double p[3], v[3];
        for (int x = 0; x < 3; ++x) {
            p[x] = fma(fma(fma(A3[x], s, A2[x]), s, A1[x]), s, A0[x]);
            v[x] = fma(fma(3.0 * A3[x], s, 2.0 * A2[x]), s, A1[x]);
        }
        const double d = sqrt(dot(p, p));
        if (d < thr && n < kConjMaxEv) ev[n++] = ConjEvent{s, d, sqrt(dot(v, v)) / h, flags};
    };
    if (first && c[0] > 0.0) emit(0.0, 0);                   // d increasing at t = 0
    unsigned idx = 0;
    int depth = 0;
    for (;;) {
        const double w = ldexp(1.0, -depth), lo = idx * w;
        double b[6];
        conj_piece(c, lo, w, b);
        int changes = 0;
        for (int i = 0; i < 5; ++i) changes += (b[i] > 0.0) != (b[i + 1] > 0.0);
        const bool rising = !(b[0] > 0.0) && b[5] > 0.0;
        if (changes >= 2 && depth < kConjDepth) {            // split: go to the left child
            idx <<= 1;
            ++depth;
            continue;
        }
        if (changes == 1) {
            if (rising) emit(conj_refine(c, lo, lo + w), 0);
        } else if (changes >= 2) {                           // at the depth cap
            emit(rising ? conj_refine(c, lo, lo + w) : lo + 0.5 * w, kConjFlagDepth);
        }
        while (idx & 1u) {                                   // up past the right children
            idx >>= 1;
            --depth;
        }
        if (depth == 0) break;
        idx += 1;                                            // the right sibling
    }
    if (last && !(c[0] + c[1] + c[2] + c[3] + c[4] + c[5] > 0.0)) emit(1.0, 0);   // d not increasing at t = D
    return n;
}

// Pre-pass: thread (k, s) -> X [T][6][N] (r in m, v in m/s) and, for k < T - 1, S [T-1][4][N] (conj_sphere) and the
// skipped count of satellite s.  y [N][7][T] normalized (propagate_batch), scale [N][2] = (R0_s, R0_s / s0_s).
template <int BLOCK>
__global__ void __launch_bounds__(BLOCK) conj_prepass_kernel(const double *__restrict__ y, const double *__restrict__ scale,
                                                             int n_sats, int T, double h, double *__restrict__ X,
                                                             double *__restrict__ S, int32_t *__restrict__ skipped)
{
    const long long t = (long long)blockIdx.x * BLOCK + threadIdx.x;
    if (t >= (long long)n_sats * T) return;
    const int k = (int)(t / n_sats), s = (int)(t - (long long)k * n_sats);
    const double R = scale[2 * s], V = scale[2 * s + 1];
    const double *ys = y + (size_t)s * 7 * T;
    double q0[6], q1[6];
    for (int c = 0; c < 6; ++c) {
        q0[c] = ys[(size_t)c * T + k] * (c < 3 ? R : V);
        X[((size_t)k * 6 + c) * n_sats + s] = q0[c];
    }
    if (k == T - 1) return;
    for (int c = 0; c < 6; ++c) q1[c] = ys[(size_t)c * T + k + 1] * (c < 3 ? R : V);
    double sp[4];
    conj_sphere(q0, q1, h, sp);
    for (int c = 0; c < 4; ++c) S[((size_t)k * 4 + c) * n_sats + s] = sp[c];
    if (!(conj_finite6(q0) && conj_finite6(q1))) atomicAdd((unsigned *)&skipped[s], 1u);
}

#ifdef __CUDACC__
// The pair-interval events of a warp go out through one atomicAdd: an inclusive scan of the per-lane counts, lane 31
// reserves the warp's range, and every lane writes its events at base + (exclusive prefix).  Called by all 32 lanes.
__device__ __forceinline__ void conj_warp_append(const ConjEvent *ev, int n, int i, int j, int k, double h, ConjRecord *out,
                                                 long long capacity, unsigned long long *counters)
{
    const unsigned full = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    int incl = n;
    for (int off = 1; off < 32; off <<= 1) {
        const int v = __shfl_up_sync(full, incl, off);
        if (lane >= off) incl += v;
    }
    const int total = __shfl_sync(full, incl, 31);
    if (total == 0) return;
    unsigned long long base = 0;
    if (lane == 31) base = atomicAdd(&counters[0], (unsigned long long)total);
    base = __shfl_sync(full, base, 31) + (unsigned long long)(incl - n);
    for (int e = 0; e < n; ++e) {
        if (ev[e].flags) atomicAdd(&counters[1], 1ull);
        if (base + e < (unsigned long long)capacity)
            out[base + e] = ConjRecord{i, j, k, ev[e].flags, fma((double)k, h, ev[e].s * h), ev[e].d, ev[e].v};
    }
}

// grid (n_blocks, n_blocks): blockIdx.x = j-block, blockIdx.y = i-block; the tiles below the diagonal exit at once.
// Thread t of a tile takes satellite i = lane of the i-block against j = t / 32 + 8 q (q = 0..3) of the j-block.
__global__ void __launch_bounds__(kConjThreads) conj_pair_kernel(const double *__restrict__ X, const double *__restrict__ S,
                                                                 int n_sats, int T, double h, double thr, ConjRecord *out,
                                                                 long long capacity, unsigned long long *counters)
{
    const int ib = blockIdx.y, jb = blockIdx.x;
    if (jb < ib) return;
    __shared__ double sx[kConjKc + 1][6][2 * kConjTile];   // states of the i-block (0..31) and the j-block (32..63)
    __shared__ double ss[kConjKc][4][2 * kConjTile];       // spheres
    const int lane = threadIdx.x & 31, wj = threadIdx.x >> 5;
    const int i = ib * kConjTile + lane;
    const int n_int = T - 1;
    for (int k0 = 0; k0 < n_int; k0 += kConjKc) {
        const int nk = min(kConjKc, n_int - k0);
        __syncthreads();
        for (int e = threadIdx.x; e < (nk + 1) * 6 * 2 * kConjTile; e += kConjThreads) {
            const int l = e & (2 * kConjTile - 1), row = e / (2 * kConjTile);
            const int s = l < kConjTile ? ib * kConjTile + l : jb * kConjTile + l - kConjTile;
            (&sx[0][0][0])[e] = s < n_sats ? X[((size_t)k0 * 6 + row) * n_sats + s] : 0.0;
        }
        for (int e = threadIdx.x; e < nk * 4 * 2 * kConjTile; e += kConjThreads) {
            const int l = e & (2 * kConjTile - 1), row = e / (2 * kConjTile);
            const int s = l < kConjTile ? ib * kConjTile + l : jb * kConjTile + l - kConjTile;
            (&ss[0][0][0])[e] = s < n_sats ? S[((size_t)k0 * 4 + row) * n_sats + s] : __longlong_as_double(0x7ff8000000000000LL);
        }
        __syncthreads();
        for (int kk = 0; kk < nk; ++kk) {
            const int k = k0 + kk;
            const double cix = ss[kk][0][lane], ciy = ss[kk][1][lane], ciz = ss[kk][2][lane], ri = ss[kk][3][lane];
#pragma unroll 1
            for (int q = 0; q < 4; ++q) {
                const int jl = wj + 8 * q, j = jb * kConjTile + jl;
                const bool valid = i < n_sats && j < n_sats && (ib != jb || lane < jl);
                const double dx = cix - ss[kk][0][kConjTile + jl], dy = ciy - ss[kk][1][kConjTile + jl];
                const double dz = ciz - ss[kk][2][kConjTile + jl], R = ri + ss[kk][3][kConjTile + jl] + thr;
                const bool pass = valid && dx * dx + dy * dy + dz * dz <= R * R;
                if (__ballot_sync(0xffffffffu, pass) == 0u) continue;
                ConjEvent ev[kConjMaxEv];
                int n = 0;
                if (pass) {
                    double qi0[6], qi1[6], qj0[6], qj1[6];
                    for (int c = 0; c < 6; ++c) {
                        qi0[c] = sx[kk][c][lane];
                        qi1[c] = sx[kk + 1][c][lane];
                        qj0[c] = sx[kk][c][kConjTile + jl];
                        qj1[c] = sx[kk + 1][c][kConjTile + jl];
                    }
                    n = conj_interval(qi0, qi1, qj0, qj1, h, thr, k == 0, k == n_int - 1, ev);
                }
                conj_warp_append(ev, n, i, j, k, h, out, capacity, counters);
            }
        }
    }
}
#endif

}  // namespace mpc
