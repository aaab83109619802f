// discretize_rk23_kernel.cuh -- the reference's DEFAULT quadrature mode with Discretizer.ivp_solver = 'RK23'.
//
// The reference hands ivp_solver to solve_ivp(method=...) (linearize_discretize.py:37-41), and its quadrature rides on
// the steps the solver accepts, so the solver decides the result at the 1e-3 level: this is scipy's RK23
// (scipy/integrate/_ivp/rk.py) replayed per interval [t_k, t_{k+1}] on the augmented state [Phi (49), x (7)], as
// discretize_default_body replays RK45:
//
//   * Bogacki-Shampine 3(2): C = [0, 1/2, 3/4], A = [[0,0,0], [1/2,0,0], [0,3/4,0]], B = [2/9, 1/3, 4/9],
//     E = [5/72, -1/12, -1/9, 1/8]; 3 stages plus the FSAL evaluation at the new point;
//   * error_estimator_order = 2: the controller's exponent is -1/3 (SAFETY 0.9, MIN_FACTOR 0.2, MAX_FACTOR 10, as RK45),
//     and select_initial_step takes order 2, i.e. h1 = (0.01 / max(d1, d2))^(1/3);
//   * every step decision (accept / reject, the next h) is scipy's, so the node count of an interval is len(sol.t).
//
// Everything else is the RK45 body's: the Phi ping-pong in the output rows 0..41 / 49..90, the row-6 accumulators in
// rows 91..98, the far end node's input parked in rows 99..101, each quadrature node evaluated once with its full
// trapezoid weight (node_accumulate_general), the same epilogue (epilogue_store), thread mapping (ragged_locate) and
// status words.  Only the stepper differs, and with it the stage slots: 4 x 9 stage linearisations instead of 7 x 9.
// The body is a sibling of discretize_default_body rather than a template flag of it, so that the RK45 kernels keep
// their code generation; its kernels are instantiated in mpc_b200_rk23.cu only.
#pragma once
#include "discretize_default_kernel.cuh"

namespace mpc {

constexpr int kRkSlots = kDfAcc + 4 * 9;          // 48 accumulators + G_s (6), d_s (3) of the 4 stages: 84 slots

// x^(-1/3) of the RK23 controller (scipy: 0.9 * err^(-1/3)) and of its initial step (0.01 / max(d1, d2))^(1/3).
// x = m 2^(3q) with m in [1/2, 4) (exact), a single-precision seed of m^(-1/3), two Newton steps
// y <- y (4 - m y^3) / 3 (relative error 2 e^2 per step: 1e-7 -> 2e-14 -> rounding), then the exact scaling by 2^-q:
// over the whole double range, not only the float one.  x = 0, inf or NaN give NaN, which the clamps of the caller
// (fmin / fmax return their other argument) turn into the factors pow would give: x = 0 only reaches the controller
// together with err == 0 (factor MAX_FACTOR), x = inf is a rejection (factor MIN_FACTOR).
__device__ __forceinline__ double inv_cube_root(double x)
{
    int e;
    const double m = frexp(x, &e);                      // x = m 2^e, m in [1/2, 1)
    const int q = (e >= 0) ? e / 3 : -((2 - e) / 3);    // floor(e / 3)
    const double mr = ldexp(m, e - 3 * q);              // in [1/2, 4)
    double y = (double)powf((float)mr, -1.0f / 3.0f);
#pragma unroll
    for (int i = 0; i < 2; ++i) {
        const double y3 = y * y * y;
        y *= fma(mr * (-1.0 / 3.0), y3, 4.0 / 3.0);
    }
    return ldexp(y, -q);
}

#define SM(e) sm[(e) * BLOCK]

// RAG, PSC: as discretize_default_body (ragged batch with first[] the prefix sums of K_s - 1; per-satellite constants
// psc[sat] in place of P0).  u on the nodes of x, no drag branch, one destination.
template <bool J2, int BLOCK, bool RAG, bool PSC>
__device__ __forceinline__ void
discretize_rk23_body(const double *__restrict__ x_in, const double *__restrict__ u_in, const double *__restrict__ tf_arr,
                     const DiscParams &P0, int n_sats, int K, double rtol, double atol, double max_step, double *out,
                     long long pitch, long long offset, int32_t *__restrict__ status, int32_t *__restrict__ n_nodes,
                     const long long *__restrict__ first, const DiscParams *psc)
{
    constexpr bool GENU = false, DRAG = false;
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
    hold.init(u_in, sat, k, K, K);
    // tau = np.linspace(0, 1, K) (:356): start + i*step, last point exactly 1
    const double step = 1.0 / (double)(Kg - 1);
    const double t0 = (double)k * step, t1 = (k + 1 == Kg - 1) ? 1.0 : (double)(k + 1) * step;
    const double ilen = 1.0 / (t1 - t0);
    double *const col = out + offset + gid;
    double *cur = col + (long long)kDfPhiA * pitch, *nxt = col + (long long)kDfPhiB * pitch;

#pragma unroll 1
    for (int e = 0; e < kDfAcc; ++e) SM(e) = 0.0;
    double *const row6 = col + (long long)kDfRow6 * pitch;
#pragma unroll
    for (int q = 0; q < 8; ++q) row6[(long long)q * pitch] = 0.0;
    {       // input of the far end node as the reference looks it up: computed once, parked in the buffer
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

    AdStage st0;
    bad |= ad_eval<J2, GENU, DRAG>(P, 0.0, nullptr, x, 0.0, t0, hold, st0);
    // ---- select_initial_step (common.py) with order = 2; f = tf * k, y0 = [I, x] ---------------------------------
    double h_abs;
    {
        const double interval_length = fabs(t1 - t0);
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
        const double g[9] = {MPC_G9(DRAG, st0)};
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
        AdStage stA;
        bad |= ad_eval<J2, GENU, DRAG>(P, 0.0, nullptr, x1, h0 * ilen, t0 + h0, hold, stA);
        double d2sq = 0.0;
#pragma unroll
        for (int i = 0; i < 7; ++i) {
            const double df = (stA.k[i] - st0.k[i]) * isc[i];
            d2sq += df * df;
        }
        const double g1[9] = {MPC_G9(DRAG, stA)};
#pragma unroll
        for (int c = 0; c < 7; ++c) {
            double p1r[3], p1v[3], f0r[3], f0v[3];
#pragma unroll
            for (int a = 0; a < 3; ++a) {
                f0r[a] = (c == a + 3) ? 1.0 : 0.0;
                f0v[a] = (c < 3) ? g[a * 3 + c] : ((c == 6) ? st0.d[a] : 0.0);
                p1r[a] = ((c == a) ? 1.0 : 0.0) + hs0 * f0r[a];
                p1v[a] = ((c == a + 3) ? 1.0 : 0.0) + hs0 * f0v[a];
            }
#pragma unroll
            for (int a = 0; a < 3; ++a) {
                const double f1r = p1v[a];
                double f1v = g1[a * 3 + 0] * p1r[0] + g1[a * 3 + 1] * p1r[1] + g1[a * 3 + 2] * p1r[2];
                if (c == 6) f1v += stA.d[a];
                const double e1 = (f1r - f0r[a]) * ((c == a) ? is1 : is0), e2 = (f1v - f0v[a]) * ((c == a + 3) ? is1 : is0);
                d2sq += e1 * e1 + e2 * e2;
            }
        }
        const double d2 = sqrt(d2sq / 56.0) / h0;
        const double h1 = (d1 <= 1e-15 && d2 <= 1e-15) ? fmax(1e-6, h0 * 1e-3) : inv_cube_root(100.0 * fmax(d1, d2));
        h_abs = fmin(fmin(100.0 * h0, h1), fmin(interval_length, max_step));
    }

    // ---- solve_ivp main loop, one trip per quadrature node (see discretize_default_body) ---------------------------
    if (RAG) ad_end_node_input_ld(st0, u_in, sat, K, Kg, k);
    else ad_end_node_input<GENU>(st0, u_in, sat, K, k);
    // Bogacki-Shampine: stage s of the state is x + hs sum_l A_sl k_l; the FSAL stage 3 is the new point (row B)
    const double cs[4] = {0.0, 1.0 / 2, 3.0 / 4, 1.0};
    const double bw[3] = {2.0 / 9, 1.0 / 3, 4.0 / 9};
    const double ew[4] = {5.0 / 72, -1.0 / 12, -1.0 / 9, 1.0 / 8};
    double half_prev = 0.0;       // (t_j - t_{j-1}) / 2
#pragma unroll 1
    for (;;) {
        const bool last = !(t < t1);
        double half_next = 0.0, t_new = t;
        double xn[7];
        AdStage st3;
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
                double kx[3][7];
#pragma unroll
                for (int i = 0; i < 7; ++i) kx[0][i] = st0.k[i];
                df_store_stage<BLOCK, DRAG>(sm, 0, st0, hs, hs2);
#pragma unroll
                for (int s = 1; s < 3; ++s) {
                    double xs_[7];
#pragma unroll
                    for (int i = 0; i < 7; ++i) xs_[i] = fma(kx[s - 1][i] * cs[s], hs, x[i]);   // A = diag(1/2, 3/4) below
                    AdStage sg;
                    bad |= ad_eval<J2, GENU, DRAG>(P, 0.0, nullptr, xs_, (t + cs[s] * h - t0) * ilen, t + cs[s] * h, hold, sg);
#pragma unroll
                    for (int i = 0; i < 7; ++i) kx[s][i] = sg.k[i];
                    df_store_stage<BLOCK, DRAG>(sm, s, sg, hs, hs2);
                }
#pragma unroll
                for (int i = 0; i < 7; ++i) {
                    double dy = 0.0;
#pragma unroll
                    for (int l = 0; l < 3; ++l) dy = fma(kx[l][i], bw[l], dy);
                    xn[i] = fma(hs, dy, x[i]);
                }
                bad |= ad_eval<J2, GENU, DRAG>(P, 0.0, nullptr, xn, (t + h - t0) * ilen, t + h, hold, st3);
                df_store_stage<BLOCK, DRAG>(sm, 3, st3, hs, hs2);
                double esum = 0.0;
#pragma unroll
                for (int i = 0; i < 7; ++i) {
                    double e = st3.k[i] * ew[3];
#pragma unroll
                    for (int l = 0; l < 3; ++l) e = fma(kx[l][i], ew[l], e);
                    const double q = e * hs * fast_rcp1(atol + fmax(fabs(x[i]), fabs(xn[i])) * rtol);
                    esum = fma(q, q, esum);
                }
                // -- Phi columns: global (L2) -> registers -> global, stage matrices from shared memory ----------------
                // As in discretize_default_body: P = hs p_v, K_s = hs^2 p_v'(stage s),
                //     q_r(s) = p_r + c_s P + sum_m (A A)_sm K_m,      hs q_v(s) = P + sum_m A_sm K_m,
                // with A extended by its FSAL row B (stage 3 is the new column).  A A: row 2 = [3/8], row 3 = [1/6, 1/3].
                // Position rows' error estimate: sum_m (E A)_m K_m, E A = [-1/72, -1/24, 1/18] (sum(E) = 0 exactly).
                const double a2[4][2] = {{0, 0}, {0, 0}, {3.0 / 8, 0}, {1.0 / 6, 1.0 / 3}};
                const double av[4][3] = {{0, 0, 0}, {1.0 / 2, 0, 0}, {0, 3.0 / 4, 0}, {2.0 / 9, 1.0 / 3, 4.0 / 9}};
                const double ea[3] = {-1.0 / 72, -1.0 / 24, 1.0 / 18};
                double pn[6];
#pragma unroll
                for (int i = 0; i < 6; ++i) pn[i] = cur[(long long)i * pitch];
#pragma unroll 1
                for (int c = 0; c < 7; ++c) {
                    double pr_[3], pv_[3], Pv[3], kk[4][3];
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
                    for (int s = 0; s < 4; ++s) {
                        double qr[3], qv[3];       // q_r(s), hs q_v(s)
#pragma unroll
                        for (int i = 0; i < 3; ++i) {
                            if (s == 0) {
                                qr[i] = pr_[i];
                                qv[i] = Pv[i];
                            } else {
                                double r_ = fma(cs[s], Pv[i], pr_[i]), v_ = Pv[i];
#pragma unroll
                                for (int m = 0; m + 1 < s; ++m) r_ = fma(kk[m][i], a2[s][m], r_);
#pragma unroll
                                for (int m = 0; m < s; ++m)
                                    if (av[s][m] != 0.0) v_ = fma(kk[m][i], av[s][m], v_);
                                qr[i] = r_;
                                qv[i] = v_;
                            }
                        }
                        const int b = kDfAcc + s * 9;
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
                        if (s == 3) {      // (qr, qv / hs) is the new column: store, error estimate
#pragma unroll
                            for (int i = 0; i < 3; ++i) {
                                const double yv = qv[i] * ihs;
                                nxt[(long long)(c * 6 + i) * pitch] = qr[i];
                                nxt[(long long)(c * 6 + 3 + i) * pitch] = yv;
                                double er = 0.0, ev = 0.0;
#pragma unroll
                                for (int m = 0; m < 3; ++m) er = fma(kk[m][i], ea[m], er);
#pragma unroll
                                for (int l = 0; l < 4; ++l) ev = fma(kk[l][i], ew[l], ev);
                                const double q1 = er * fast_rcp1(atol + fmax(fabs(pr_[i]), fabs(qr[i])) * rtol);
                                const double q2 = ev * ihs * fast_rcp1(atol + fmax(fabs(pv_[i]), fabs(yv)) * rtol);
                                esum = fma(q1, q1, esum);
                                esum = fma(q2, q2, esum);
                            }
                        }
                    }
                }
                const double err = sqrt(esum * (1.0 / 56.0));
                const double ef = 0.9 * inv_cube_root(err);
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
        if (!fail) {
            double pr[7][3], pv[7][3];
#pragma unroll
            for (int c = 0; c < 7; ++c)
#pragma unroll
                for (int a = 0; a < 3; ++a) {
                    pr[c][a] = cur[(long long)(c * 6 + a) * pitch];
                    pv[c][a] = cur[(long long)(c * 6 + 3 + a) * pitch];
                }
            if (last) {       // far end node: the node term reads u, 1/|u| (guarded), |u| of the reference's lookup
                const double *e = col + (long long)kDfEndU * pitch;
                st0.ux = e[0];
                st0.uy = e[pitch];
                st0.uz = e[2 * pitch];
                const double uu = fma(st0.ux, st0.ux, fma(st0.uy, st0.uy, st0.uz * st0.uz));
                st0.iun = (uu > 4.930380657631324e-32) ? fast_rsqrt(uu) : 0.0;
                st0.un = uu * st0.iun;
            }
            const double w = half_prev + half_next;
            node_accumulate_general<BLOCK>(sm, pr, pv, P, st0, x, w, w * ((t - t0) * ilen), row6, pitch);
        }
        if (last || fail) break;
        double *const tmp = cur;
        cur = nxt;
        nxt = tmp;
#pragma unroll
        for (int i = 0; i < 7; ++i) x[i] = xn[i];
        st0 = st3;
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
    DstTab dst{};
    dst.p[0] = out;
    const int nonfinite = epilogue_store<BLOCK, 1>(sm, pr, pv, tf, 1.0, tf, dst, pitch, offset + gid);
    if (status) status[gid] = bad ? 1 : (nonfinite ? 2 : (fail ? 3 : 0));
    if (n_nodes) n_nodes[gid] = nodes;
}
#undef SM

// One entry for the four batch kinds: RAG (first[] the prefix sums of K_s - 1, x / u padded to K = Kmax columns; results,
// status and node counts in columns offset + s (Kmax-1) + k, padding never written) and PSC (satellite s runs with
// psc[s]; P is not read).
template <bool J2, int BLOCK, bool RAG, bool PSC>
__global__ void __launch_bounds__(BLOCK)
discretize_rk23_kernel(const double *__restrict__ x_in, const double *__restrict__ u_in, const double *__restrict__ tf_arr,
                       DiscParams P, const DiscParams *psc, int n_sats, int K, double rtol, double atol, double max_step,
                       double *out, long long pitch, long long offset, int32_t *__restrict__ status,
                       int32_t *__restrict__ n_nodes, const long long *__restrict__ first)
{
    discretize_rk23_body<J2, BLOCK, RAG, PSC>(x_in, u_in, tf_arr, P, n_sats, K, rtol, atol, max_step, out, pitch, offset,
                                              status, n_nodes, first, psc);
}

}  // namespace mpc
