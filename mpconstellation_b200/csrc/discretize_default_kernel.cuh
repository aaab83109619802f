// discretize_default_kernel.cuh -- the reference's DEFAULT quadrature mode, second build (round 2).
//
// Same mathematics as discretize_adaptive_kernel (see its header: scipy's RK45 controller replayed per interval,
// non-uniform trapezoid rule on the accepted steps, linearize_discretize.py:29-30,49-50,77-80,109), restructured for
// what limited that kernel (profiles/r01_g: one warp per scheduler because of 52 KiB of shared memory per warp, and a
// 41 KB hot loop that does not fit the 32 KB instruction cache):
//
//   * Phi does not live in shared memory.  The two copies a step needs (the accepted Phi and the candidate of the step
//     being tried -- a rejected step must not destroy the former) ping-pong between two row blocks of the OUTPUT buffer
//     itself: rows 0..41 (where A_k ends up anyway) and rows 49..90 (B_kp / B_kn, written only by the epilogue).  The
//     layout is the SoA one, [row][interval]: every access of a warp is one coalesced 256-byte line, it stays in L2
//     for the life of the warp, and each entry is read / written once per step.  Shared memory per thread drops from
//     203 to 111 slots (48 accumulators + 7 stage linearisations of 9; the 8 accumulators of row 6, plain sums that
//     need no Phi, are kept in rows 91..98 of the output buffer as well), i.e. 8 instead of 4 warps per SM.
//   * every quadrature node is evaluated ONCE, with its full trapezoid weight (t_{j+1} - t_{j-1})/2, when the step that
//     leaves it has been accepted (the old build evaluated both ends of every panel: 2 (n-1) instead of n node terms,
//     each with a 6x6 solve), and the step loop is arranged so that the node term has a single call site;
//   * launched as ONE 8-warp CTA per SM: the hot loop (36 KB of SASS) is larger than the SM's instruction cache, and
//     one-warp CTAs walk it out of phase, each paying its own instruction misses (measured: 3.75 warps stalled on
//     instruction fetch per issue, the GPC-level instruction cache 98 % busy, 2.64 ms).  The warps of one CTA start
//     together and take the same 4-5 steps, stay within a few cache lines of each other and share every fetched line
//     (instruction-cache hit rate 68 % -> 93 %, 1.97 ms; profiles/r02_b, r02_c).
// Results agree with the first build to rounding (the panel sums are associated differently) and with the unmodified
// reference's default-mode fixtures to <= 1e-10; node counts are identical.
#pragma once
#include "discretize_adaptive_kernel.cuh"

namespace mpc {

constexpr int kDfAcc = 48;                        // accumulators in shared memory: slots 0..47 of the kAccSlots layout; the 8
                                                  // of row 6 (slots 48..55) live in the output buffer (rows kDfRow6..)
constexpr int kDfSlots = kDfAcc + 7 * 9;          // + G_s (6), d_s (3) of the 7 stages: 111 slots, 8 warps per SM
constexpr int kDfSlotsDrag = kDfAcc + 7 * 18;     // drag branch of the linearisation: G_s + W_s (9, not symmetric), d_s (3), V_s (6)
constexpr int kDfPhiA = 0, kDfPhiB = 49;          // the two Phi row blocks inside the output buffer
constexpr int kDfRow6 = 91;                       // rows 91..98: the row-6 accumulators until the epilogue
constexpr int kDfEndU = 99;                       // rows 99..101: input of the far end node (ref_node_input), parked

#define SM(e) sm[(e) * BLOCK]

// x^(-1/5) of the step-size controller (scipy: 0.9 * err^(-0.2)): single-precision seed, two Newton steps
// y <- y (6 - x y^5) / 5 (relative error 3 e^2 per step: 1e-7 -> 3e-14 -> rounding).  A tenth of the instructions of
// pow(double, double), on the FP32 pipe for the seed.  x = 0, inf, NaN, or outside the float range give 0 / inf / NaN,
// which the clamps of the caller (fmin / fmax return their finite argument) turn into the same factors pow would.
__device__ __forceinline__ double inv_fifth_root(double x)
{
    double y = (double)powf((float)x, -0.2f);
#pragma unroll
    for (int i = 0; i < 2; ++i) {
        const double y2 = y * y, y5 = y2 * y2 * y;
        y *= fma(-0.2 * x, y5, 1.2);
    }
    return y;
}

// The stage linearisations are stored in the units of the step: hs^2 G_s, hs^2 d_s (and hs V_s), see the column loop.
template <int BLOCK, bool DRAG>
__device__ __forceinline__ void df_store_stage(volatile double *sm, int s, const typename AdStageSel<DRAG>::type &st, double hs, double hs2)
{
    const int b = kDfAcc + s * (DRAG ? 18 : 9);
    if constexpr (DRAG) {
        // hs^2 (G + W), W = gw r_hat^T (the density gradient's term, discretize_drag_kernel.cuh), row-major; d; hs V
        SM(b + 0) = hs2 * fma(st.gw[0], st.rh[0], st.g.xx);
        SM(b + 1) = hs2 * fma(st.gw[0], st.rh[1], st.g.xy);
        SM(b + 2) = hs2 * fma(st.gw[0], st.rh[2], st.g.xz);
        SM(b + 3) = hs2 * fma(st.gw[1], st.rh[0], st.g.xy);
        SM(b + 4) = hs2 * fma(st.gw[1], st.rh[1], st.g.yy);
        SM(b + 5) = hs2 * fma(st.gw[1], st.rh[2], st.g.yz);
        SM(b + 6) = hs2 * fma(st.gw[2], st.rh[0], st.g.xz);
        SM(b + 7) = hs2 * fma(st.gw[2], st.rh[1], st.g.yz);
        SM(b + 8) = hs2 * fma(st.gw[2], st.rh[2], st.g.zz);
        SM(b + 9) = hs2 * st.d[0];
        SM(b + 10) = hs2 * st.d[1];
        SM(b + 11) = hs2 * st.d[2];
        SM(b + 12) = hs * st.v.xx;
        SM(b + 13) = hs * st.v.xy;
        SM(b + 14) = hs * st.v.xz;
        SM(b + 15) = hs * st.v.yy;
        SM(b + 16) = hs * st.v.yz;
        SM(b + 17) = hs * st.v.zz;
    } else {
        SM(b + 0) = hs2 * st.g.xx;
        SM(b + 1) = hs2 * st.g.xy;
        SM(b + 2) = hs2 * st.g.xz;
        SM(b + 3) = hs2 * st.g.yy;
        SM(b + 4) = hs2 * st.g.yz;
        SM(b + 5) = hs2 * st.g.zz;
        SM(b + 6) = hs2 * st.d[0];
        SM(b + 7) = hs2 * st.d[1];
        SM(b + 8) = hs2 * st.d[2];
    }
}

// RAG: a ragged batch (discretize_default_ragged_kernel): K is the padded stride Kmax, first[] the prefix sums of K_s - 1
// (ragged_locate); threads map to live intervals only, gid below is the interval's output column s (Kmax-1) + k.
// PSC: per-satellite constants (discretize_default_units_kernel): the thread of satellite `sat` reads psc[sat] where the
// others read P.  The table is read where the constants are used, inside the step loop (it is not __restrict__: the
// stores to the output buffer keep the loads where they are), so that this 254-register body keeps no more values live.
// NDST: the results are stored into dst.p[0 .. NDST-1] (the fused all-gather of a sharded batch); the Phi scratch rows
// stay in dst.p[0], the local buffer.
template <bool J2, int BLOCK, bool GENU, bool DRAG, bool RAG = false, bool PSC = false, int NDST = 1>
__device__ __forceinline__ void
discretize_default_body(const double *__restrict__ x_in, const double *__restrict__ u_in,
                        const double *__restrict__ tf_arr, const DiscParams &P0, int n_sats, int K, int Ku, double rtol, double atol,
                        double max_step, const DstTab &dst, long long pitch, long long offset, int32_t *__restrict__ status,
                        int32_t *__restrict__ n_nodes, double kf, const DragLin *L, const long long *__restrict__ first = nullptr,
                        const DiscParams *psc = nullptr)
{
    constexpr int kStage = DRAG ? 18 : 9;
    extern __shared__ double acc_smem[];
    long long gid;
    int sat, k, Kg = K;           // Kg: nodes of this satellite's grid
    if constexpr (RAG) {
        const long long tid = (long long)blockIdx.x * BLOCK + threadIdx.x;
        if (tid >= first[n_sats] - first[0]) return;
        ragged_locate(first, n_sats, tid, sat, k, Kg);
        gid = (long long)sat * (K - 1) + k;
    } else {
        const long long n_int = (long long)n_sats * (K - 1);
        gid = (long long)blockIdx.x * BLOCK + threadIdx.x;
        if (gid >= n_int) return;
        sat = (int)(gid / (K - 1));
        k = (int)(gid - (long long)sat * (K - 1));
    }
    const DiscParams &P = PSC ? psc[sat] : P0;
    volatile double *sm = acc_smem + threadIdx.x;
    const double tf = tf_arr[sat];
    const double *xs = x_in + ((long long)sat * 7) * K + k;
    double x[7];
#pragma unroll
    for (int c = 0; c < 7; ++c) x[c] = xs[(long long)c * K];
    UHold<GENU> hold;
    hold.init(u_in, sat, k, K, Ku);
    // tau = np.linspace(0, 1, K) (:356): start + i*step, last point exactly 1
    const double step = 1.0 / (double)(Kg - 1);
    const double t0 = (double)k * step, t1 = (k + 1 == Kg - 1) ? 1.0 : (double)(k + 1) * step;
    const double ilen = 1.0 / (t1 - t0);
    // this thread's column of the output buffer: Phi scratch blocks at rows kDfPhiA.. and kDfPhiB..
    double *const col = dst.p[0] + offset + gid;
    double *cur = col + (long long)kDfPhiA * pitch, *nxt = col + (long long)kDfPhiB * pitch;

#pragma unroll 1
    for (int e = 0; e < kDfAcc; ++e) SM(e) = 0.0;
    double *const row6 = col + (long long)kDfRow6 * pitch;
#pragma unroll
    for (int q = 0; q < 8; ++q) row6[(long long)q * pitch] = 0.0;
    if (!GENU) {       // input of the far end node as the reference looks it up: computed once, parked in the buffer
        double e[3];
        if (RAG) ref_node_input_ld(u_in + (long long)sat * 3 * K, K, Kg, k + 1, 1.0, e[0], e[1], e[2]);
        else ref_node_input(u_in + (long long)sat * 3 * K, K, k + 1, 1.0, e[0], e[1], e[2]);
#pragma unroll
        for (int q = 0; q < 3; ++q) col[(long long)(kDfEndU + q) * pitch] = e[q];
    }
    int bad = 0, fail = 0, nodes = 1;
    double t = t0;
    // Phi(tau_k) = I (:34)
#pragma unroll
    for (int e = 0; e < 42; ++e) cur[(long long)e * pitch] = (e % 7 == 0 && e < 36) ? 1.0 : 0.0;

    typename AdStageSel<DRAG>::type st0;
    bad |= ad_eval<J2, GENU, DRAG>(P, kf, L, x, 0.0, t0, hold, st0);
    // ---- select_initial_step (common.py); f = tf * k, y0 = [I, x] ----------------------------------------------
    double h_abs;
    {
        const double interval_length = fabs(t1 - t0);
        // (the error scales take three kinds of values -- atol, atol + rtol, atol + |x_i| rtol --: nine reciprocals,
        //  with tf folded in, instead of a division per term)
        const double s1 = atol + rtol, s0 = atol;
        const double is1 = tf / s1, is0 = tf / s0;
        double d0sq = 7.0 / (s1 * s1), d1sq = 0.0, isc[7];
#pragma unroll
        for (int i = 0; i < 7; ++i) {
            const double sc = atol + fabs(x[i]) * rtol, r_ = 1.0 / sc;
            isc[i] = tf * r_;
            d0sq += (x[i] * r_) * (x[i] * r_);
            d1sq += (st0.k[i] * isc[i]) * (st0.k[i] * isc[i]);
        }
        // G (+ W = gw r_hat^T with drag: the density gradient's term, not symmetric)
        const double g[9] = {MPC_G9(DRAG, st0)};
        double v0[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0}, vA[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
        if (DRAG) {
            const double t_[9] = {st0.v.xx, st0.v.xy, st0.v.xz, st0.v.xy, st0.v.yy, st0.v.yz, st0.v.xz, st0.v.yz, st0.v.zz};
#pragma unroll
            for (int i = 0; i < 9; ++i) {
                v0[i] = t_[i];
                const double isc_ = (i % 4 == 0) ? is1 : is0;
                d1sq += (t_[i] * isc_) * (t_[i] * isc_);
            }
        }
        d1sq += 3.0 * is0 * is0;
#pragma unroll
        for (int i = 0; i < 9; ++i) d1sq += (g[i] * is0) * (g[i] * is0);
#pragma unroll
        for (int i = 0; i < 3; ++i) d1sq += (st0.d[i] * is0) * (st0.d[i] * is0);
        const double d0 = sqrt(d0sq / 56.0), d1 = sqrt(d1sq / 56.0);
        double h0 = (d0 < 1e-5 || d1 < 1e-5) ? 1e-6 : 0.01 * d0 / d1;
        h0 = fmin(h0, interval_length);
        const double hs0 = h0 * tf;
        double x1[7];
#pragma unroll
        for (int i = 0; i < 7; ++i) x1[i] = fma(hs0, st0.k[i], x[i]);
        typename AdStageSel<DRAG>::type stA;
        bad |= ad_eval<J2, GENU, DRAG>(P, kf, L, x1, h0 * ilen, t0 + h0, hold, stA);
        double d2sq = 0.0;
#pragma unroll
        for (int i = 0; i < 7; ++i) {
            const double df = (stA.k[i] - st0.k[i]) * isc[i];
            d2sq += df * df;
        }
        const double g1[9] = {MPC_G9(DRAG, stA)};
        if (DRAG) {
            const double t_[9] = {stA.v.xx, stA.v.xy, stA.v.xz, stA.v.xy, stA.v.yy, stA.v.yz, stA.v.xz, stA.v.yz, stA.v.zz};
#pragma unroll
            for (int i = 0; i < 9; ++i) vA[i] = t_[i];
        }
#pragma unroll
        for (int c = 0; c < 7; ++c) {
            double p1r[3], p1v[3], f0r[3], f0v[3];
#pragma unroll
            for (int a = 0; a < 3; ++a) {
                f0r[a] = (c == a + 3) ? 1.0 : 0.0;
                f0v[a] = (c < 3) ? g[a * 3 + c] : ((c == 6) ? st0.d[a] : v0[a * 3 + (c - 3)]);
                p1r[a] = ((c == a) ? 1.0 : 0.0) + hs0 * f0r[a];
                p1v[a] = ((c == a + 3) ? 1.0 : 0.0) + hs0 * f0v[a];
            }
#pragma unroll
            for (int a = 0; a < 3; ++a) {
                const double f1r = p1v[a];
                double f1v = g1[a * 3 + 0] * p1r[0] + g1[a * 3 + 1] * p1r[1] + g1[a * 3 + 2] * p1r[2];
                if (DRAG) f1v += vA[a * 3 + 0] * p1v[0] + vA[a * 3 + 1] * p1v[1] + vA[a * 3 + 2] * p1v[2];
                if (c == 6) f1v += stA.d[a];
                const double e1 = (f1r - f0r[a]) * ((c == a) ? is1 : is0), e2 = (f1v - f0v[a]) * ((c == a + 3) ? is1 : is0);
                d2sq += e1 * e1 + e2 * e2;
            }
        }
        const double d2 = sqrt(d2sq / 56.0) / h0;
        const double h1 = (d1 <= 1e-15 && d2 <= 1e-15) ? fmax(1e-6, h0 * 1e-3) : inv_fifth_root(100.0 * fmax(d1, d2));
        h_abs = fmin(fmin(100.0 * h0, h1), fmin(interval_length, max_step));
    }

    // ---- solve_ivp main loop.  One trip per quadrature node: try steps from node j until one is accepted (none when
    // t has reached the end), then add node j with its full trapezoid weight, then move on. ---------------------------
    // the node term of tau_k reads the reference's lookup of u there
    if (RAG) ad_end_node_input_ld(st0, u_in, sat, K, Kg, k);
    else ad_end_node_input<GENU>(st0, u_in, sat, K, k);
    double half_prev = 0.0;       // (t_j - t_{j-1}) / 2
#pragma unroll 1
    for (;;) {
        const bool last = !(t < t1);
        double half_next = 0.0, t_new = t;
        double xn[7];
        typename AdStageSel<DRAG>::type st6;
        if (!last) {
            const double min_step = 10.0 * fabs(nextafter(t, CUDART_INF) - t);
            if (h_abs > max_step) h_abs = max_step;
            else if (h_abs < min_step) h_abs = min_step;
            bool accepted = false, rejected = false;
            while (!accepted) {
                if (h_abs < min_step) {
                    fail = 1;
                    break;
                }
                t_new = t + h_abs;
                if (t_new - t1 > 0.0) t_new = t1;
                const double h = t_new - t;
                h_abs = fabs(h);
                const double hs = h * tf, hs2 = hs * hs, ihs = 1.0 / hs;
                // -- state stages (registers) ------------------------------------------------------------------------
                double kx[6][7];
#pragma unroll
                for (int i = 0; i < 7; ++i) kx[0][i] = st0.k[i];
                df_store_stage<BLOCK, DRAG>(sm, 0, st0, hs, hs2);
                const double cs[6] = {0.0, 1.0 / 5, 3.0 / 10, 4.0 / 5, 8.0 / 9, 1.0};
#pragma unroll
                for (int s = 1; s < 6; ++s) {
                    double xs_[7];
#pragma unroll
                    for (int i = 0; i < 7; ++i) {
                        double dy = 0.0;
#pragma unroll
                        for (int l = 0; l < s; ++l) dy = fma(kx[l][i], kDpA[s][l], dy);
                        xs_[i] = fma(dy, hs, x[i]);
                    }
                    typename AdStageSel<DRAG>::type sg;
                    bad |= ad_eval<J2, GENU, DRAG>(P, kf, L, xs_, (t + cs[s] * h - t0) * ilen, t + cs[s] * h, hold, sg);
#pragma unroll
                    for (int i = 0; i < 7; ++i) kx[s][i] = sg.k[i];
                    df_store_stage<BLOCK, DRAG>(sm, s, sg, hs, hs2);
                }
                const double bw[6] = {35.0 / 384, 0.0, 500.0 / 1113, 125.0 / 192, -2187.0 / 6784, 11.0 / 84};
                const double ew[7] = {-71.0 / 57600, 0.0, 71.0 / 16695, -71.0 / 1920, 17253.0 / 339200, -22.0 / 525, 1.0 / 40};
#pragma unroll
                for (int i = 0; i < 7; ++i) {
                    double dy = 0.0;
#pragma unroll
                    for (int l = 0; l < 6; ++l) dy = fma(kx[l][i], bw[l], dy);
                    xn[i] = fma(hs, dy, x[i]);
                }
                bad |= ad_eval<J2, GENU, DRAG>(P, kf, L, xn, (t + h - t0) * ilen, t + h, hold, st6);
                df_store_stage<BLOCK, DRAG>(sm, 6, st6, hs, hs2);
                double esum = 0.0;
#pragma unroll
                for (int i = 0; i < 7; ++i) {
                    double e = st6.k[i] * ew[6];
#pragma unroll
                    for (int l = 0; l < 6; ++l) e = fma(kx[l][i], ew[l], e);
                    const double q = e * hs * fast_rcp1(atol + fmax(fabs(x[i]), fabs(xn[i])) * rtol);
                    esum = fma(q, q, esum);
                }
                // -- Phi columns: global (L2) -> registers -> global, stage matrices from shared memory ----------------
                // Each column (p_r, p_v) obeys p_r' = p_v, p_v' = G p_r (+ V p_v) (+ d): stepped in the units of the
                // step, P = hs p_v, K_s = hs^2 p_v'(stage s), the Dormand-Prince stages read
                //     q_r(s) = p_r + c_s P + sum_m (A A)_sm K_m,      hs q_v(s) = P + sum_m A_sm K_m,
                // the position rows through the squared tableau (the stage derivative of a position row is the stage's
                // velocity row, itself a combination of the K_m).  Same stages, same result to rounding; every
                // coefficient is a literal, no product with hs inside the stages and nothing but K to keep per stage.
                // Error estimate h K^T E of the position rows likewise: sum_m (E A)_m K_m (sum(E) = 0 exactly).
                // (the next column is requested from L2 while this one is stepped)
                const double a2[7][5] = {{0, 0, 0, 0, 0},
                                         {0, 0, 0, 0, 0},
                                         {9.0 / 200, 0, 0, 0, 0},
                                         {-12.0 / 25, 4.0 / 5, 0, 0, 0},
                                         {-12248.0 / 6561, 7208.0 / 2187, -6784.0 / 6561, 0, 0},
                                         {-533.0 / 264, 91.0 / 22, -56.0 / 33, 7.0 / 88, 0},
                                         {35.0 / 384, 0.0, 50.0 / 159, 25.0 / 192, -243.0 / 6784}};
                const double ea[6] = {-611.0 / 230400, 0.0, 514.0 / 83475, -391.0 / 38400, 4617.0 / 1356800, 11.0 / 3360};
                double pn[6];
#pragma unroll
                for (int i = 0; i < 6; ++i) pn[i] = cur[(long long)i * pitch];
#pragma unroll 1
                for (int c = 0; c < 7; ++c) {
                    double pr_[3], pv_[3], Pv[3], kk[7][3];
#pragma unroll
                    for (int i = 0; i < 3; ++i) {
                        pr_[i] = pn[i];
                        pv_[i] = pn[3 + i];
                        Pv[i] = hs * pn[3 + i];
                    }
                    if (c < 6) {
#pragma unroll
                        for (int i = 0; i < 6; ++i) pn[i] = cur[(long long)((c + 1) * 6 + i) * pitch];
                    }
#pragma unroll
                    for (int s = 0; s < 7; ++s) {
                        double qr[3], qv[3];       // q_r(s), hs q_v(s)
#pragma unroll
                        for (int i = 0; i < 3; ++i) {
                            if (s == 0) {
                                qr[i] = pr_[i];
                                qv[i] = Pv[i];
                            } else {
                                double r_ = fma(cs[s == 6 ? 5 : s], Pv[i], pr_[i]), v_ = Pv[i];
#pragma unroll
                                for (int m = 0; m + 1 < s && m < 5; ++m) r_ = fma(kk[m][i], a2[s][m], r_);
#pragma unroll
                                for (int m = 0; m < s && m < 6; ++m) v_ = fma(kk[m][i], (s == 6) ? bw[m] : kDpA[s < 6 ? s : 5][m < 5 ? m : 4], v_);
                                qr[i] = r_;
                                qv[i] = v_;
                            }
                        }
                        const int b = kDfAcc + s * kStage;
                        if (DRAG) {
                            // general (G + W): 9 entries, then d (mass column), then (hs V) (hs q_v)
                            double dx = 0.0, dy_ = 0.0, dz = 0.0;
                            if (c == 6) {
                                dx = SM(b + 9);
                                dy_ = SM(b + 10);
                                dz = SM(b + 11);
                            }
                            const double vxx = SM(b + 12), vxy = SM(b + 13), vxz = SM(b + 14), vyy = SM(b + 15), vyz = SM(b + 16), vzz = SM(b + 17);
                            dx = fma(vxz, qv[2], fma(vxy, qv[1], fma(vxx, qv[0], dx)));
                            dy_ = fma(vyz, qv[2], fma(vyy, qv[1], fma(vxy, qv[0], dy_)));
                            dz = fma(vzz, qv[2], fma(vyz, qv[1], fma(vxz, qv[0], dz)));
                            kk[s][0] = fma(SM(b + 2), qr[2], fma(SM(b + 1), qr[1], fma(SM(b + 0), qr[0], dx)));
                            kk[s][1] = fma(SM(b + 5), qr[2], fma(SM(b + 4), qr[1], fma(SM(b + 3), qr[0], dy_)));
                            kk[s][2] = fma(SM(b + 8), qr[2], fma(SM(b + 7), qr[1], fma(SM(b + 6), qr[0], dz)));
                        } else {
                            const double gxx = SM(b), gxy = SM(b + 1), gxz = SM(b + 2), gyy = SM(b + 3), gyz = SM(b + 4), gzz = SM(b + 5);
                            // (d = -u/m^2 forces the mass column only: loaded for c == 6, a warp-uniform condition)
                            double dx = 0.0, dy_ = 0.0, dz = 0.0;
                            if (c == 6) {
                                dx = SM(b + 6);
                                dy_ = SM(b + 7);
                                dz = SM(b + 8);
                            }
                            kk[s][0] = fma(gxz, qr[2], fma(gxy, qr[1], fma(gxx, qr[0], dx)));
                            kk[s][1] = fma(gyz, qr[2], fma(gyy, qr[1], fma(gxy, qr[0], dy_)));
                            kk[s][2] = fma(gzz, qr[2], fma(gyz, qr[1], fma(gxz, qr[0], dz)));
                        }
                        if (s == 6) {      // (qr, qv / hs) is the new column: store, error estimate
#pragma unroll
                            for (int i = 0; i < 3; ++i) {
                                const double yv = qv[i] * ihs;
                                nxt[(long long)(c * 6 + i) * pitch] = qr[i];
                                nxt[(long long)(c * 6 + 3 + i) * pitch] = yv;
                                double er = 0.0, ev = 0.0;
#pragma unroll
                                for (int m = 0; m < 6; ++m) er = fma(kk[m][i], ea[m], er);
#pragma unroll
                                for (int l = 0; l < 7; ++l) ev = fma(kk[l][i], ew[l], ev);
                                const double q1 = er * fast_rcp1(atol + fmax(fabs(pr_[i]), fabs(qr[i])) * rtol);
                                const double q2 = ev * ihs * fast_rcp1(atol + fmax(fabs(pv_[i]), fabs(yv)) * rtol);
                                esum = fma(q1, q1, esum);
                                esum = fma(q2, q2, esum);
                            }
                        }
                    }
                }
                const double err = sqrt(esum * (1.0 / 56.0));
                const double ef = 0.9 * inv_fifth_root(err);
                if (!(err >= 1.0)) {   // also accepts a NaN error so that a poisoned unit terminates (status flags it)
                    double factor = (err == 0.0) ? 10.0 : fmin(10.0, ef);
                    if (rejected) factor = fmin(1.0, factor);
                    if (!(factor == factor)) factor = 1.0;
                    h_abs *= factor;
                    accepted = true;
                } else {
                    h_abs *= fmax(0.2, ef);
                    rejected = true;
                }
            }
            half_next = 0.5 * (t_new - t);
        }
        // ---- node j: w_j = (t_j - t_{j-1})/2 + (t_{j+1} - t_j)/2, np.trapz with x = sol.t (:77-80) ---------------------
        // (after a step-size underflow nothing is accumulated any more: the unit is flagged)
        if (!fail) {
            double pr[7][3], pv[7][3];
#pragma unroll
            for (int c = 0; c < 7; ++c)
#pragma unroll
                for (int a = 0; a < 3; ++a) {
                    pr[c][a] = cur[(long long)(c * 6 + a) * pitch];
                    pv[c][a] = cur[(long long)(c * 6 + 3 + a) * pitch];
                }
            if (!GENU && last) {       // far end node: the node term reads u, 1/|u| (guarded), |u| of the reference's lookup
                const double *e = col + (long long)kDfEndU * pitch;
                st0.ux = e[0];
                st0.uy = e[pitch];
                st0.uz = e[2 * pitch];
                const double uu = fma(st0.ux, st0.ux, fma(st0.uy, st0.uy, st0.uz * st0.uz));
                st0.iun = (uu > 4.930380657631324e-32) ? fast_rsqrt(uu) : 0.0;
                st0.un = uu * st0.iun;
            }
            const double w = half_prev + half_next;
            // The reference inverts the NUMERICAL Phi (np.linalg.inv, :69): general 6x6 solve, see discretize_adaptive_kernel
            node_accumulate_general<BLOCK>(sm, pr, pv, P, st0, x, w, w * ((t - t0) * ilen), row6, pitch);
        }
        if (last || fail) break;
        double *const tmp = cur;
        cur = nxt;
        nxt = tmp;
#pragma unroll
        for (int i = 0; i < 7; ++i) x[i] = xn[i];
        st0 = st6;
        half_prev = half_next;
        t = t_new;
        if (++nodes > 4096) {
            fail = 1;
            break;
        }
    }

    double pr[7][3], pv[7][3];
#pragma unroll
    for (int c = 0; c < 7; ++c)
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            pr[c][a] = cur[(long long)(c * 6 + a) * pitch];
            pv[c][a] = cur[(long long)(c * 6 + 3 + a) * pitch];
        }
#pragma unroll
    for (int q = 0; q < 8; ++q) SM(48 + q) = row6[(long long)q * pitch];   // (the stage slots are dead by now)
    const int nonfinite = epilogue_store<BLOCK, NDST>(sm, pr, pv, tf, 1.0, tf, dst, pitch, offset + gid);
    if (status) status[gid] = bad ? 1 : (nonfinite ? 2 : (fail ? 3 : 0));
    if (n_nodes) n_nodes[gid] = nodes;
}
#undef SM

// (the body takes the parameter structs by reference: ptxas then reads them from the constant bank where they are used
//  instead of copying them into registers at entry; 1.47 -> 1.44 ms on config 3, same box)
// (DRAG is always false here and the two trailing parameters are unused: the drag branch has its own entry below.  They are
//  kept because ptxas's register allocation of this 254-register kernel turned out to depend on the entry's signature --
//  the same PTX body with two parameters fewer came out at 255 registers and 240 B more stack, 3-5 % slower on config 3.)
template <bool J2, int BLOCK, bool GENU, bool DRAG>
__global__ void __launch_bounds__(BLOCK)
discretize_default_kernel(const double *__restrict__ x_in, const double *__restrict__ u_in,
                          const double *__restrict__ tf_arr, DiscParams P, int n_sats, int K, int Ku, double rtol, double atol,
                          double max_step, DstTab dst, long long pitch, long long offset, int32_t *__restrict__ status,
                          int32_t *__restrict__ n_nodes, double kf = 0.0, double ka = 0.0)
{
    static_assert(!DRAG, "the drag branch is discretize_default_drag_kernel");
    discretize_default_body<J2, BLOCK, GENU, false>(x_in, u_in, tf_arr, P, n_sats, K, Ku, rtol, atol, max_step, dst, pitch, offset,
                                                    status, n_nodes, kf, nullptr);
}

// the drag branch of the linearisation (linearize_discretize.py:160-169): kf for the dynamics, L for the Jacobian
template <bool J2, int BLOCK>
__global__ void __launch_bounds__(BLOCK)
discretize_default_drag_kernel(const double *__restrict__ x_in, const double *__restrict__ u_in,
                               const double *__restrict__ tf_arr, DiscParams P, int n_sats, int K, double rtol, double atol,
                               double max_step, DstTab dst, long long pitch, long long offset, int32_t *__restrict__ status,
                               int32_t *__restrict__ n_nodes, double kf, const __grid_constant__ DragLin L)
{
    discretize_default_body<J2, BLOCK, false, true>(x_in, u_in, tf_arr, P, n_sats, K, 0, rtol, atol, max_step, dst, pitch, offset,
                                                    status, n_nodes, kf, &L);
}

// ragged batch: satellite s on K_s = first[s+1] - first[s] + 1 nodes, x / u padded to K = Kmax columns, results, status and
// node counts in columns offset + s (Kmax-1) + k (k < K_s - 1); the padding columns are never written
template <bool J2, int BLOCK>
__global__ void __launch_bounds__(BLOCK)
discretize_default_ragged_kernel(const double *__restrict__ x_in, const double *__restrict__ u_in,
                                 const double *__restrict__ tf_arr, DiscParams P, int n_sats, int K, double rtol, double atol,
                                 double max_step, DstTab dst, long long pitch, long long offset, int32_t *__restrict__ status,
                                 int32_t *__restrict__ n_nodes, const long long *__restrict__ first)
{
    discretize_default_body<J2, BLOCK, false, false, true>(x_in, u_in, tf_arr, P, n_sats, K, K, rtol, atol, max_step, dst, pitch,
                                                           offset, status, n_nodes, 0.0, nullptr, first);
}

// per-satellite constants (mpc_discretize_batch_units): satellite s runs with psc[s] in place of the launch-wide
// DiscParams; RAG as discretize_default_ragged_kernel (first == nullptr otherwise)
template <bool J2, int BLOCK, bool RAG>
__global__ void __launch_bounds__(BLOCK)
discretize_default_units_kernel(const double *__restrict__ x_in, const double *__restrict__ u_in,
                                const double *__restrict__ tf_arr, const DiscParams *psc, int n_sats, int K, double rtol,
                                double atol, double max_step, DstTab dst, long long pitch, long long offset,
                                int32_t *__restrict__ status, int32_t *__restrict__ n_nodes, const long long *__restrict__ first)
{
    discretize_default_body<J2, BLOCK, false, false, RAG, true>(x_in, u_in, tf_arr, psc[0], n_sats, K, K, rtol, atol, max_step,
                                                                dst, pitch, offset, status, n_nodes, 0.0, nullptr, first, psc);
}

// ragged batch (with or without per-satellite constants) stored into NDST > 1 buffers: one rank's shard of the fused
// all-gather (mpc_discretize_batch_ragged_gather).  The signatures are those of the single-destination forms above.
template <bool J2, int BLOCK, int NDST>
__global__ void __launch_bounds__(BLOCK)
discretize_default_ragged_multi_kernel(const double *__restrict__ x_in, const double *__restrict__ u_in,
                                       const double *__restrict__ tf_arr, DiscParams P, int n_sats, int K, double rtol,
                                       double atol, double max_step, DstTab dst, long long pitch, long long offset,
                                       int32_t *__restrict__ status, int32_t *__restrict__ n_nodes,
                                       const long long *__restrict__ first)
{
    discretize_default_body<J2, BLOCK, false, false, true, false, NDST>(x_in, u_in, tf_arr, P, n_sats, K, K, rtol, atol, max_step,
                                                                        dst, pitch, offset, status, n_nodes, 0.0, nullptr, first);
}

template <bool J2, int BLOCK, int NDST>
__global__ void __launch_bounds__(BLOCK)
discretize_default_units_multi_kernel(const double *__restrict__ x_in, const double *__restrict__ u_in,
                                      const double *__restrict__ tf_arr, const DiscParams *psc, int n_sats, int K, double rtol,
                                      double atol, double max_step, DstTab dst, long long pitch, long long offset,
                                      int32_t *__restrict__ status, int32_t *__restrict__ n_nodes,
                                      const long long *__restrict__ first)
{
    discretize_default_body<J2, BLOCK, false, false, true, true, NDST>(x_in, u_in, tf_arr, psc[0], n_sats, K, K, rtol, atol,
                                                                       max_step, dst, pitch, offset, status, n_nodes, 0.0, nullptr,
                                                                       first, psc);
}

}  // namespace mpc
