// constraint_terms_kernel.cuh -- Optimizer.get_constraint_terms (optimizer.py:80-170) for a batch of satellites.
//
// The step immediately after the discretization on the reference's path: unit vectors of the reference
// positions / thrusts along the horizon (trust-region and thrust-cone constraint terms) and the linearised
// circular-orbit terminal conditions at the final node (orbital speed V_c, tangential / radial / normal
// velocity and their gradients with respect to r and v).  HBM-bound, trivial arithmetic: one thread per
// (satellite, node); the thread of the last node also evaluates the 32 terminal terms.
//
// The reference's formulas are followed literally, including two that are probably not what its authors meant
// (they define what the optimizer receives, so they are mirrored, not fixed):
//   * optimizer.py:121  Dv_h_hat = I/|h| - (h h^T/|h|^3) @ skew(r)   ('@' binds tighter than '-')
//   * optimizer.py:137-138  ubar_hat is populated only where |u| <= eps (mask inverted): 0/0 = NaN there, 0 elsewhere
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "discretize_kernel.cuh"   // ragged_locate

namespace mpc {

constexpr int kFinalTerms = 32;
// offsets into the per-satellite terminal block
constexpr int kOffRf = 0;     // rf_hat (3)
constexpr int kOffVc = 3;     // Vc
constexpr int kOffDrVc = 4;   // DrVc (3)
constexpr int kOffDrVcR = 7;  // DrVc_rbar
constexpr int kOffVt = 8;     // Vt
constexpr int kOffDVt = 9;    // DrVt_DvVt (6)
constexpr int kOffDVtB = 15;  // DrVt_DvVt_bar
constexpr int kOffVr = 16;    // Vr
constexpr int kOffDVr = 17;   // DrVr_DvVr (6)
constexpr int kOffDVrB = 23;  // DrVr_DvVr_bar
constexpr int kOffVn = 24;    // Vn
constexpr int kOffDVn = 25;   // DrVn_DvVn (6)
constexpr int kOffDVnB = 31;  // DrVn_DvVn_bar

struct M3 {
    double a[3][3];
};

__device__ __forceinline__ M3 m3_skew(const double (&x)[3])   // optimizer.py:41-45
{
    M3 s;
    s.a[0][0] = 0.0;   s.a[0][1] = -x[2]; s.a[0][2] = x[1];
    s.a[1][0] = x[2];  s.a[1][1] = 0.0;   s.a[1][2] = -x[0];
    s.a[2][0] = -x[1]; s.a[2][1] = x[0];  s.a[2][2] = 0.0;
    return s;
}

__device__ __forceinline__ M3 m3_mul(const M3 &p, const M3 &q)
{
    M3 r;
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) r.a[i][j] = p.a[i][0] * q.a[0][j] + p.a[i][1] * q.a[1][j] + p.a[i][2] * q.a[2][j];
    return r;
}

// s1 * I - s3 * x x^T
__device__ __forceinline__ M3 m3_projector(const double (&x)[3], double s1, double s3)
{
    M3 r;
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) r.a[i][j] = (i == j ? s1 : 0.0) - s3 * x[i] * x[j];
    return r;
}

__device__ __forceinline__ double dot3(const double (&p)[3], const double (&q)[3])
{
    return p[0] * q[0] + p[1] * q[1] + p[2] * q[2];
}

// row vector times matrix: out_j = sum_i v_i M_ij   (np.dot(v, M))
__device__ __forceinline__ void vecmat(const double (&v)[3], const M3 &m, double (&out)[3])
{
#pragma unroll
    for (int j = 0; j < 3; ++j) out[j] = v[0] * m.a[0][j] + v[1] * m.a[1][j] + v[2] * m.a[2][j];
}

// optimizer.py:108-168 for one satellite: r, v = final node of the reference trajectory
__device__ inline void terminal_terms(const double (&r)[3], const double (&v)[3], double mu, double *__restrict__ o)
{
    const double nr = sqrt(dot3(r, r));
    double h[3] = {r[1] * v[2] - r[2] * v[1], r[2] * v[0] - r[0] * v[2], r[0] * v[1] - r[1] * v[0]};
    const double nh = sqrt(dot3(h, h));
    double rh[3], hh[3];
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        rh[i] = r[i] / nr;
        hh[i] = h[i] / nh;
    }
    double th[3] = {hh[1] * rh[2] - hh[2] * rh[1], hh[2] * rh[0] - hh[0] * rh[2], hh[0] * rh[1] - hh[1] * rh[0]};
    const double inh = 1.0 / nh, inh3 = 1.0 / (nh * nh * nh), inr = 1.0 / nr, inr3 = 1.0 / (nr * nr * nr);
    const M3 sk_v = m3_skew(v), sk_r = m3_skew(r), sk_rh = m3_skew(rh), sk_hh = m3_skew(hh);
    // :120  Dr_h_hat = (I/|h| - h h^T/|h|^3) @ (-skew(v))
    M3 neg_sk_v = sk_v;
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) neg_sk_v.a[i][j] = -sk_v.a[i][j];
    const M3 Dr_h = m3_mul(m3_projector(h, inh, inh3), neg_sk_v);
    // :121  Dv_h_hat = I/|h| - (h h^T/|h|^3) @ skew(r)        (literal operator precedence)
    M3 hhT;
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) hhT.a[i][j] = inh3 * h[i] * h[j];
    M3 Dv_h = m3_mul(hhT, sk_r);
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) Dv_h.a[i][j] = (i == j ? inh : 0.0) - Dv_h.a[i][j];
    const M3 Dr_r = m3_projector(r, inr, inr3);   // :122
    // :123  Dr_t_hat = -skew(r_hat) @ Dr_h_hat + skew(h_hat) @ Dr_r_hat ;  :124  Dv_t_hat = -skew(r_hat) @ Dv_h_hat
    const M3 t1 = m3_mul(sk_rh, Dr_h), t2 = m3_mul(sk_hh, Dr_r), t3 = m3_mul(sk_rh, Dv_h);
    M3 Dr_t, Dv_t;
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            Dr_t.a[i][j] = -t1.a[i][j] + t2.a[i][j];
            Dv_t.a[i][j] = -t3.a[i][j];
        }
    double tmp[3];
#pragma unroll
    for (int i = 0; i < 3; ++i) o[kOffRf + i] = rh[i];                       // :143
    o[kOffVc] = sqrt(mu / nr);                                                // :145
    const double cvc = -0.5 * sqrt(mu) / (nr * nr * sqrt(nr));                // :146  -1/2 sqrt(MU) |r|^(-5/2)
    double drvc[3] = {cvc * r[0], cvc * r[1], cvc * r[2]};
#pragma unroll
    for (int i = 0; i < 3; ++i) o[kOffDrVc + i] = drvc[i];
    o[kOffDrVcR] = dot3(drvc, r);                                             // :148
    // tangential :149-154
    o[kOffVt] = dot3(v, th);
    double g[6];
    vecmat(v, Dr_t, tmp);
    g[0] = tmp[0]; g[1] = tmp[1]; g[2] = tmp[2];
    vecmat(v, Dv_t, tmp);
    g[3] = th[0] + tmp[0]; g[4] = th[1] + tmp[1]; g[5] = th[2] + tmp[2];
#pragma unroll
    for (int i = 0; i < 6; ++i) o[kOffDVt + i] = g[i];
    o[kOffDVtB] = g[0] * r[0] + g[1] * r[1] + g[2] * r[2] + g[3] * v[0] + g[4] * v[1] + g[5] * v[2];
    // radial :156-161
    o[kOffVr] = dot3(v, rh);
    vecmat(v, Dr_r, tmp);
    g[0] = tmp[0]; g[1] = tmp[1]; g[2] = tmp[2];
    g[3] = rh[0]; g[4] = rh[1]; g[5] = rh[2];
#pragma unroll
    for (int i = 0; i < 6; ++i) o[kOffDVr + i] = g[i];
    o[kOffDVrB] = g[0] * r[0] + g[1] * r[1] + g[2] * r[2] + g[3] * v[0] + g[4] * v[1] + g[5] * v[2];
    // normal :163-168
    o[kOffVn] = dot3(v, hh);
    vecmat(v, Dr_h, tmp);
    g[0] = tmp[0]; g[1] = tmp[1]; g[2] = tmp[2];
    vecmat(v, Dv_h, tmp);
    g[3] = hh[0] + tmp[0]; g[4] = hh[1] + tmp[1]; g[5] = hh[2] + tmp[2];
#pragma unroll
    for (int i = 0; i < 6; ++i) o[kOffDVn + i] = g[i];
    o[kOffDVnB] = g[0] * r[0] + g[1] * r[1] + g[2] * r[2] + g[3] * v[0] + g[4] * v[1] + g[5] * v[2];
}

// The per-column pieces of optimizer.py:128-168, shared by the rectangular and the ragged launch.  Satellite s's blocks:
// x [7][ld], rbar_hat [3][ld-1], u and ubar_hat [3][ldu].
__device__ __forceinline__ void rbar_column(const double *__restrict__ xs, int ld, int c, double *__restrict__ rbar_hat, int s)
{   // :128-129  r_bar / ||r_bar||  (columns 0..K-2); no contraction, bit-identical to numpy
    const double r0 = xs[c], r1 = xs[ld + c], r2 = xs[2 * ld + c];
    const double n = __dsqrt_rn(__dadd_rn(__dadd_rn(__dmul_rn(r0, r0), __dmul_rn(r1, r1)), __dmul_rn(r2, r2)));
    double *o = rbar_hat + (size_t)s * 3 * (ld - 1);
    o[c] = __ddiv_rn(r0, n);
    o[(ld - 1) + c] = __ddiv_rn(r1, n);
    o[2 * (ld - 1) + c] = __ddiv_rn(r2, n);
}

__device__ __forceinline__ void ubar_column(const double *__restrict__ u, int ldu, int c, double eps, double *__restrict__ ubar_hat,
                                            int s)
{   // :132-139  (mask as written: filled where the norm is <= eps, zero elsewhere)
    const double *us = u + (size_t)s * 3 * ldu;
    const double u0 = us[c], u1 = us[ldu + c], u2 = us[2 * ldu + c];
    const double n = __dsqrt_rn(__dadd_rn(__dadd_rn(__dmul_rn(u0, u0), __dmul_rn(u1, u1)), __dmul_rn(u2, u2)));
    const bool fill = n <= eps;
    double *o = ubar_hat + (size_t)s * 3 * ldu;
    o[c] = fill ? __ddiv_rn(u0, n) : 0.0;
    o[ldu + c] = fill ? __ddiv_rn(u1, n) : 0.0;
    o[2 * ldu + c] = fill ? __ddiv_rn(u2, n) : 0.0;
}

// x [N][7][K], u [N][3][Ku] -> rbar_hat [N][3][K-1], ubar_hat [N][3][Ku], fin [N][32].
// Thread i covers column c = i % C of satellite s = i / C, C = max(K, Ku): consecutive threads touch
// consecutive addresses of every row.
//
// RAG: a ragged batch.  K = Ku = Kmax is the padded stride and first[] the prefix sums of K_s - 1 (ragged_locate); the
// launch covers the live intervals of every satellite.  The thread of interval k writes column k of rbar_hat and
// ubar_hat; the thread of the last interval (k = K_s - 2) also writes ubar_hat column K_s - 1 and the terminal terms of
// node K_s - 1.  Satellite s gets exactly the bits of a rectangular launch of that satellite at K = Ku = K_s; the padding
// columns are never written.
template <bool RAG = false>
__global__ void __launch_bounds__(256)
constraint_terms_kernel(const double *__restrict__ x, const double *__restrict__ u, int n_sats, int K, int Ku,
                        double mu, double eps, double *__restrict__ rbar_hat, double *__restrict__ ubar_hat,
                        double *__restrict__ fin, const long long *__restrict__ first = nullptr)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (RAG) {
        if (i >= first[n_sats] - first[0]) return;
        int s, k, Ks;
        ragged_locate(first, n_sats, i, s, k, Ks);
        const double *xs = x + (size_t)s * 7 * K;
        rbar_column(xs, K, k, rbar_hat, s);
        ubar_column(u, K, k, eps, ubar_hat, s);
        if (k == Ks - 2) {
            ubar_column(u, K, Ks - 1, eps, ubar_hat, s);
            const double r[3] = {xs[Ks - 1], xs[K + Ks - 1], xs[2 * K + Ks - 1]};
            const double v[3] = {xs[3 * K + Ks - 1], xs[4 * K + Ks - 1], xs[5 * K + Ks - 1]};
            double o[kFinalTerms];
            terminal_terms(r, v, mu, o);
            double *dst = fin + (size_t)s * kFinalTerms;
#pragma unroll
            for (int j = 0; j < kFinalTerms; ++j) dst[j] = o[j];
        }
        return;
    }
    const int C = K > Ku ? K : Ku;
    if (i >= (long long)n_sats * C) return;
    const int s = (int)(i / C), c = (int)(i % C);
    const double *xs = x + (size_t)s * 7 * K;
    if (c < K - 1) rbar_column(xs, K, c, rbar_hat, s);
    if (c < Ku) ubar_column(u, Ku, c, eps, ubar_hat, s);
    if (c == K - 1) {
        const double r[3] = {xs[K - 1], xs[2 * K - 1], xs[3 * K - 1]};
        const double v[3] = {xs[4 * K - 1], xs[5 * K - 1], xs[6 * K - 1]};
        double o[kFinalTerms];
        terminal_terms(r, v, mu, o);
        double *dst = fin + (size_t)s * kFinalTerms;
#pragma unroll
        for (int j = 0; j < kFinalTerms; ++j) dst[j] = o[j];
    }
}

// Per-satellite constants (mpc_constraint_terms_units): constraint_terms_kernel with satellite s's MU read from mu_sat[s],
// rectangular (first == nullptr, u on the nodes of x: Ku = K) or ragged.  A kernel of its own rather than a template flag
// on the one above, whose instantiations keep their names and code.
template <bool RAG>
__global__ void __launch_bounds__(256)
constraint_terms_units_kernel(const double *__restrict__ x, const double *__restrict__ u, int n_sats, int K,
                              const double *__restrict__ mu_sat, double eps, double *__restrict__ rbar_hat,
                              double *__restrict__ ubar_hat, double *__restrict__ fin, const long long *__restrict__ first)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    int s, c, Ks = K;             // c: interval (ragged) or column (rectangular)
    if (RAG) {
        if (i >= first[n_sats] - first[0]) return;
        ragged_locate(first, n_sats, i, s, c, Ks);
    } else {
        if (i >= (long long)n_sats * K) return;
        s = (int)(i / K);
        c = (int)(i % K);
    }
    const double *xs = x + (size_t)s * 7 * K;
    if (c < Ks - 1) rbar_column(xs, K, c, rbar_hat, s);
    ubar_column(u, K, c, eps, ubar_hat, s);
    if (c == Ks - 1 || (RAG && c == Ks - 2)) {
        if (RAG) ubar_column(u, K, Ks - 1, eps, ubar_hat, s);
        const double r[3] = {xs[Ks - 1], xs[K + Ks - 1], xs[2 * K + Ks - 1]};
        const double v[3] = {xs[3 * K + Ks - 1], xs[4 * K + Ks - 1], xs[5 * K + Ks - 1]};
        double o[kFinalTerms];
        terminal_terms(r, v, mu_sat[s], o);
        double *dst = fin + (size_t)s * kFinalTerms;
#pragma unroll
        for (int j = 0; j < kFinalTerms; ++j) dst[j] = o[j];
    }
}

// ---------------------------------------------------------------------------------------------------------------
// Sparse assembly of the dynamics constraint (optimizer.py:327-339) from the SoA discretization result.
//
//   x[s,i,k+1] - ( sum_j A_k[s][k,i,j] x[s,j,k] + sum_j B_kn[s][k,i,j] u[s,j,k] + sum_j B_kp[s][k,i,j] u[s,j,k+1]
//                  + Sigma_k[s][i,k] tf + xi_k[s][i,k] + nu[s,i,k] ) == 0
//
// is one row of   J z = rhs   with rhs = xi_k[s][i,k].  Rows follow the order pyomo generates them in
// (Constraint(sIDX, xIDX, kIDX), k = K-1 skipped):  row = (s*7 + i)*(K-1) + k.  Variables are numbered
//   x[s,i,k]  -> (s*7 + i)*K + k                    u[s,j,k] -> 7NK + (s*3 + j)*K + k
//   nu[s,i,k] -> 10NK + (s*7 + i)*K + k             tf       -> 17NK           (one shared final time, optimizer.py:281)
// Every row has exactly 16 structural non-zeros, stored in ascending column order:
//   [ -A[i,0..6] with +1 at x[s,i,k+1] merged in order ] ... see the column list in the kernel.
// CSR: indptr[r] = 16 r (implicit), indices [rows*16], values [rows*16], rhs [rows].
// One thread per row; consecutive threads = consecutive k, so the SoA reads are coalesced.
//
// RAG: a ragged batch, assembled as N independent single-satellite systems (block-diagonal J), each with its own final
// time tf_s.  K is the padded stride Kmax of the SoA result (column offset + s (Kmax-1) + k), first[] the prefix sums of
// K_s - 1 (ragged_locate).  Satellite s's rows start at R_s = 7 first[s], row = R_s + i (K_s-1) + k; its variables at
// V_s = sum_{r<s} (17 K_r + 1) = 17 (first[s] + s) + s:
//   x[i,k] -> V_s + i K_s + k | u[j,k] -> V_s + 7K_s + j K_s + k | nu[i,k] -> V_s + 10K_s + i K_s + k | tf_s -> V_s + 17K_s
// i.e. the rectangular numbering of n_sats = 1, K = K_s shifted by V_s.  One thread per live interval writes its 7 rows
// (one index search per interval instead of one per row); consecutive threads still walk k, so every SoA read and every
// row store of a warp covers consecutive columns / rows as in the rectangular kernel.
constexpr int kJacNnzPerRow = 16;

// Row r of the system: state row i of interval k, read from SoA column col; x0 / u0 / nu0 / tfc: the columns of x[s,0,0],
// u[s,0,0], nu[s,i,0] and tf; Kc: nodes of the satellite's grid.
__device__ __forceinline__ void jacobian_row(const double *__restrict__ soa, long long pitch, long long col, int i, int k,
                                             int Kc, long long r, long long x0, long long u0, long long nu0, long long tfc,
                                             double *__restrict__ values, int64_t *__restrict__ indices,
                                             double *__restrict__ rhs)
{
    double *vo = values + r * kJacNnzPerRow;
    int64_t *co = indices ? indices + r * kJacNnzPerRow : nullptr;
    auto put = [&](int pos, double val, long long column) {
        vo[pos] = val;
        if (co) co[pos] = column;
    };
    // ascending column order: x[s,0..i,k] | x[s,i,k+1] | x[s,i+1..6,k] | u[s,j,k], u[s,j,k+1] per j | nu | tf
#pragma unroll
    for (int j = 0; j < 7; ++j)                                                          // -A_k[k,i,j] * x[s,j,k]
        put(j + (j > i ? 1 : 0), -soa[(long long)(i * 7 + j) * pitch + col], x0 + (long long)j * Kc + k);
    put(i + 1, 1.0, x0 + (long long)i * Kc + k + 1);                                     // +x[s,i,k+1]
#pragma unroll
    for (int j = 0; j < 3; ++j) {
        put(8 + 2 * j, -soa[(long long)(70 + i * 3 + j) * pitch + col], u0 + (long long)j * Kc + k);       // -B_kn u[s,j,k]
        put(9 + 2 * j, -soa[(long long)(49 + i * 3 + j) * pitch + col], u0 + (long long)j * Kc + k + 1);   // -B_kp u[s,j,k+1]
    }
    put(14, -1.0, nu0 + k);                                                               // -nu[s,i,k]
    put(15, -soa[(long long)(91 + i) * pitch + col], tfc);                                // -Sigma_k[i,k] * tf
    rhs[r] = soa[(long long)(98 + i) * pitch + col];                     // xi_k[i,k]
}

template <bool RAG = false>
__global__ void __launch_bounds__(256)
dynamics_jacobian_kernel(const double *__restrict__ soa, long long pitch, long long offset, int n_sats, int K,
                         double *__restrict__ values, int64_t *__restrict__ indices, double *__restrict__ rhs,
                         const long long *__restrict__ first = nullptr)
{
    if (RAG) {
        const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
        if (t >= first[n_sats] - first[0]) return;
        int s, k, Ks;
        ragged_locate(first, n_sats, t, s, k, Ks);
        const long long f = first[s] - first[0];
        const long long V = 17 * (f + s) + s;
        const long long col = offset + (long long)s * (K - 1) + k;
#pragma unroll
        for (int i = 0; i < 7; ++i)
            jacobian_row(soa, pitch, col, i, k, Ks, 7 * f + (long long)i * (Ks - 1) + k, V, V + 7LL * Ks,
                         V + 10LL * Ks + (long long)i * Ks, V + 17LL * Ks, values, indices, rhs);
        return;
    }
    const long long rows = (long long)n_sats * 7 * (K - 1);
    const long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= rows) return;
    const int k = (int)(r % (K - 1));
    const long long si = r / (K - 1);
    const int i = (int)(si % 7);
    const long long s = si / 7;
    const long long col = offset + s * (K - 1) + k;   // column of this interval in the SoA result
    const long long NK = (long long)n_sats * K;
    jacobian_row(soa, pitch, col, i, k, K, r, s * 7 * K, 7 * NK + s * 3 * K, 10 * NK + (s * 7 + i) * (long long)K, 17 * NK,
                 values, indices, rhs);
}

}  // namespace mpc
