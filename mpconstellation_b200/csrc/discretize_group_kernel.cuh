// discretize_group_kernel.cuh -- the fixed-step discretization for SMALL batches: a thread-group of 8 lanes per interval.
//
// north_star: "each independent interval maps to a warp or thread-group".  One thread per interval (discretize_pair_kernel)
// is the right mapping when there are enough intervals to fill the machine -- every lane does identical work, nothing is
// exchanged.  Below one wave it is latency-bound by construction: 50 two-node steps of ~1100 dependent-ish FP64
// instructions in ONE instruction stream (0.113 ms for 49 intervals or for 6,336: BASELINE configs 1-2, and every
// per-satellite Discretizer.discretize call the reference makes, optimizer.py:243-249).  This kernel cuts the stream:
//
//   lane c = 0..6 of a group owns COLUMN c of Phi (6 doubles, registers) and the 8 quadrature accumulators of the
//   Phi^-1-row that column produces (column 3+a gives row a, column a gives row 3+a, node_accumulate; lane 6: row 6);
//   lane 7 idles (it stores the structural-constant rows).  The 7-dimensional state is integrated REDUNDANTLY by all
//   lanes (no exchange, no divergence: 3 gravity evaluations per step), each lane steps its own column with the shared
//   stage matrices and adds its own row of the node terms.  The only traffic between lanes is the mass column (lane 6)
//   at every node -- 6 doubles by shuffle -- and the epilogue's Phi_end * [integrals] reduction.
//
// Per step a lane issues ~330 FP64 instructions instead of ~1100, so a small batch finishes in about a third of the time;
// the whole warp-instruction count per interval is ~2.4x that of the one-thread kernel, which is why the launcher uses this
// mapping only below one wave.  Same scheme (Nystrom 3-stage steps over two nodes with the Hermite midpoint where the step
// is short against the orbital rate, one step per node otherwise -- decided per interval, like discretize_pair_kernel),
// same node formulas, no shared memory; results agree with the one-thread kernels to rounding (the epilogue sums across
// lanes in a different order).  linearize_discretize.py:8-82.
#pragma once
#include "discretize_pair_kernel.cuh"

namespace mpc {

// The groups of a warp may take different paths (step counts differ when their intervals choose different step modes), so
// every shuffle names only the 8 lanes of its own group.
__device__ __forceinline__ unsigned grp_mask() { return 0xFFu << (threadIdx.x & 24); }

__device__ __forceinline__ double grp_bcast(double v, int src)   // value of lane `src` of this 8-lane group
{
    return __shfl_sync(grp_mask(), v, src, 8);
}

__device__ __forceinline__ double grp_sum(double v)              // sum over the 8 lanes of the group, on every lane
{
    const unsigned m = grp_mask();
    v += __shfl_xor_sync(m, v, 1, 8);
    v += __shfl_xor_sync(m, v, 2, 8);
    v += __shfl_xor_sync(m, v, 4, 8);
    return v;
}

// One lane's share of a node term: column (pr, pv) of Phi at the node gives one row of Phi^-1 [Duf, Sigma, xi'].
//   sgn = +1: column 3+a -> row a (TOP), sgn = -1: column a -> row 3+a; row6: this lane holds row 6 (= e7^T) instead.
struct GrpAcc {
    double A0[3], A1[3], AS, AX;
};

__device__ __forceinline__ void grp_node(GrpAcc &A, const double (&pr)[3], const double (&pv)[3], const double (&cr)[3],
                                         const double (&cv)[3], const double (&vv)[3], const double (&aa)[3],
                                         const double (&gg)[3], const double (&b)[3], double im, double md, double mdb,
                                         double w, double ws, double sgn, bool row6)
{
    double e = pr[0] * cv[0], dv = pv[0] * vv[0], pa = pr[0] * aa[0], pg = pr[0] * gg[0];
#pragma unroll
    for (int i = 1; i < 3; ++i) {
        e = fma(pr[i], cv[i], e);
        dv = fma(pv[i], vv[i], dv);
        pa = fma(pr[i], aa[i], pa);
        pg = fma(pr[i], gg[i], pg);
    }
#pragma unroll
    for (int i = 0; i < 3; ++i) e = fma(-pv[i], cr[i], e);
    e *= sgn;
    const double sdv = sgn * dv;
    double S = fma(e, md, sdv) - sgn * pa;          // e md + s dv - s pr.a
    double X = sgn * pg - fma(e, mdb, sdv);         // s pr.(G r) - e mdb - s dv
    const double sim = -sgn * im;
    if (row6) {                                     // Phi^-1 row 6 = e7^T: last rows of Duf, Sigma, xi'
        S = md;
        X = -mdb;
    }
#pragma unroll
    for (int j = 0; j < 3; ++j) {
        const double q = row6 ? b[j] : fma(b[j], e, sim * pr[j]);
        A.A0[j] = fma(w, q, A.A0[j]);
        A.A1[j] = fma(ws, q, A.A1[j]);
    }
    A.AS = fma(w, S, A.AS);
    A.AX = fma(w, X, A.AX);
}

template <bool J2, int BLOCK>
__global__ void __launch_bounds__(BLOCK)
discretize_group_kernel(const double *__restrict__ x, const double *__restrict__ u, const double *__restrict__ tf_arr,
                        DiscParams P, int n_sats, int K, int n_sub, DstTab dst, long long pitch, long long offset,
                        int32_t *__restrict__ status)
{
    const long long n_int = (long long)n_sats * (K - 1);
    const int lane = threadIdx.x & 7;
    long long gid = ((long long)blockIdx.x * BLOCK + threadIdx.x) >> 3;
    const bool live = gid < n_int;
    if (!live) gid = n_int - 1;              // whole groups only diverge at the end of the grid; keep the warp converged
    const int s = (int)(gid / (K - 1));
    const int k = (int)(gid - (long long)s * (K - 1));
    const double tf = tf_arr[s];
    const double *xs = x + ((long long)s * 7) * K + k;
    double rx = xs[0], ry = xs[K], rz = xs[2 * (long long)K];
    double vx = xs[3 * (long long)K], vy = xs[4 * (long long)K], vz = xs[5 * (long long)K];
    double m = xs[6 * (long long)K];
    UHold<false> hold;
    hold.init(u, s, k, K, K);

    const double inv_n = 1.0 / (double)n_sub;
    const double h = inv_n / (double)(K - 1);  // node spacing in tau
    const double hn = tf * h;                  // node spacing of the unscaled system
    // two-node steps where discretize_pair_kernel takes them (even number of panels, step short against the orbital rate)
    // ... and the 21-node form of the 101-node sums (kEmW, discretize_kernel.cuh) where discretize_pair_kernel takes it:
    // 20 steps of five nodes, the step ends are the nodes of the rule; or its 11-node form kEmW3 on 10 fifth-order steps
    // (state_step5 / column_step5, the code of discretize_thread) under the same per-interval conditions
    bool pairmode;
    int em = 0;                     // 1: 20 steps + kEmW, 2: 50 steps + kEmW2, 3: 10 fifth-order steps + kEmW3
    {
        const double r2 = fma(rx, rx, fma(ry, ry, rz * rz));
        const double w2H2 = P.mu * (4.0 * hn * hn) / (r2 * sqrt(r2));
        pairmode = !(n_sub & 1) && (w2H2 <= 1.0e-5);
        if (dst.em && n_sub == 100) {
            const double d2 = fma(hold.dux, hold.dux, fma(hold.duy, hold.duy, hold.duz * hold.duz));
            const double e0x = hold.u0x + hold.dux, e0y = hold.u0y + hold.duy, e0z = hold.u0z + hold.duz;
            const double a2 = fma(hold.u0x, hold.u0x, fma(hold.u0y, hold.u0y, hold.u0z * hold.u0z));
            const double b2 = fma(e0x, e0x, fma(e0y, e0y, e0z * e0z));
            if (d2 <= 0.0625 * fmax(a2, b2))
                em = (w2H2 * 6.25 <= 1.2e-5) ? ((dst.em >= 2 && d2 <= 0.015625 * fmax(a2, b2)) ? 3 : 1)
                                              : ((w2H2 <= 1.94e-5) ? 2 : 0);
        }
        if (em) pairmode = false;
    }
    const int nodes_per_step = (em == 3) ? 10 : (em == 1) ? 5 : ((em == 2 || pairmode) ? 2 : 1);
    const int n_steps = n_sub / nodes_per_step;
    const double H = hn * (double)nodes_per_step;      // integrator step
    // step-normalised variables as in discretize_kernel, with the step H
    const double H2 = H * H;
    DiscParams Ph;
    Ph.mu = P.mu * H2;
    Ph.kj2 = P.kj2 * H2;
    Ph.inv_ve = P.inv_ve / H;
    hold.scale(H2);
    const double eps2 = 4.930380657631324e-32 * (H2 * H2);
    vx *= H;
    vy *= H;
    vz *= H;
    constexpr double c6 = 1.0 / 6.0, c12 = 1.0 / 12.0, c24 = 1.0 / 24.0, c48 = 1.0 / 48.0;

    // this lane's column of Phi(tau_k) = I  (:34) and its role
    double pr[3], pv[3];
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        pr[a] = (lane == a) ? 1.0 : 0.0;
        pv[a] = (lane == a + 3) ? 1.0 : 0.0;
    }
    const double dflag = (lane == 6) ? 1.0 : 0.0;      // the mass column is forced by d = -u/m^2
    const double sgn = (lane < 3) ? -1.0 : 1.0;
    const bool row6 = lane == 6;
    GrpAcc A;
#pragma unroll
    for (int j = 0; j < 3; ++j) A.A0[j] = A.A1[j] = 0.0;
    A.AS = A.AX = 0.0;

    int bad = 0;
    double ux, uy, uz, e1x, e1y, e1z;
    // the two end nodes: as the reference looks them up (ref_node_input)
    ref_node_input(u + (long long)s * 3 * K, K, k + 1, H2, e1x, e1y, e1z);
    ref_node_input(u + (long long)s * 3 * K, K, k, H2, ux, uy, uz);
    double uu = fma(ux, ux, fma(uy, uy, uz * uz));
    double iun = inv_norm_guarded(uu, eps2);
    double un = uu * iun;
    double jn = 0.0;                                   // node index of the step's first node, as a double

    for (int j = 0; j <= n_steps; ++j) {
        if (j == n_steps) {                                                         // the other end node
            ux = e1x;
            uy = e1y;
            uz = e1z;
            uu = fma(ux, ux, fma(uy, uy, uz * uz));
            iun = inv_norm_guarded(uu, eps2);
            un = uu * iun;
        }
        // ---- stage 1 == quadrature node at the start of the step ---------------------------------------------------
        StageLin s1;
        double a1x, a1y, a1z;
        double gr[3];
        gravity<J2>(Ph, rx, ry, rz, a1x, a1y, a1z, s1.g, gr);
        bad |= !(m > 0.0);
        const double im = fast_rcp(m);
        const double tx = ux * im, ty = uy * im, tz = uz * im;
        a1x += tx;
        a1y += ty;
        a1z += tz;
        s1.dx = -tx * im * dflag;
        s1.dy = -ty * im * dflag;
        s1.dz = -tz * im * dflag;
        const double md1 = -un * Ph.inv_ve;
        {
            const double w = (em == 3) ? 10.0 * kEmW3[j] : (em == 1) ? 5.0 * kEmW[j] :
                             ((em == 2) ? 2.0 * kEmW2[j] : ((j == 0 || j == n_steps) ? 0.5 : 1.0));
            const double bs = -P.inv_ve * iun;
            const double b[3] = {bs * ux, bs * uy, bs * uz};
            const double cr[3] = {grp_bcast(pr[0], 6), grp_bcast(pr[1], 6), grp_bcast(pr[2], 6)};
            const double cv[3] = {grp_bcast(pv[0], 6), grp_bcast(pv[1], 6), grp_bcast(pv[2], 6)};
            const double vv[3] = {vx, vy, vz}, aa[3] = {a1x, a1y, a1z};
            grp_node(A, pr, pv, cr, cv, vv, aa, gr, b, im * H, md1, (iun != 0.0) ? md1 : 0.0, w, w * (jn * inv_n), sgn, row6);
        }
        if (j == n_steps) break;

        if (em == 3) {   // ---- the fifth-order step: state (every lane) and this lane's column ------------------------
            StageLin s2, s3, s4;
            double ue[3], uue, iune;
            state_step5<J2>(Ph, hold, jn * inv_n, 10.0 * inv_n, eps2, rx, ry, rz, vx, vy, vz, m, a1x, a1y, a1z, md1, s2, s3, s4,
                            ue, uue, iune, bad);
            s2.dx *= dflag; s2.dy *= dflag; s2.dz *= dflag;
            s3.dx *= dflag; s3.dy *= dflag; s3.dz *= dflag;
            s4.dx *= dflag; s4.dy *= dflag; s4.dz *= dflag;
            column_step5<true>(pr, pv, s1, s2, s3, s4);
            ux = ue[0];
            uy = ue[1];
            uz = ue[2];
            iun = iune;
            un = uue * iune;
            jn += 10.0;
            continue;
        }

        // ---- inputs and masses at the middle and the end of the step --------------------------------------------------
        const double sm = (jn + 0.5 * (double)nodes_per_step) * inv_n, se = (jn + (double)nodes_per_step) * inv_n;
        double umx, umy, umz, uex, uey, uez;
        hold.at(sm, 0.0, umx, umy, umz);
        hold.at(se, 0.0, uex, uey, uez);
        const double uum = fma(umx, umx, fma(umy, umy, umz * umz));
        const double uue = fma(uex, uex, fma(uey, uey, uez * uez));
        const double iunm = inv_norm_guarded(uum, eps2);
        const double iune = inv_norm_guarded(uue, eps2);
        const double mdm = -(uum * iunm) * Ph.inv_ve;
        const double mde = -(uue * iune) * Ph.inv_ve;
        const double m2 = fma(c24, fma(8.0, mdm, 5.0 * md1) - mde, m);
        const double m3 = fma(c6, fma(4.0, mdm, md1) + mde, m);
        bad |= !(m3 > 0.0);

        // ---- stages 2, 3 of the state (every lane) ----------------------------------------------------------------------
        StageLin s2, s3;
        double a2x, a2y, a2z, a3x, a3y, a3z;
        const double hx = fma(0.5, vx, rx), hy = fma(0.5, vy, ry), hz = fma(0.5, vz, rz);
        const double r2x = fma(0.125, a1x, hx), r2y = fma(0.125, a1y, hy), r2z = fma(0.125, a1z, hz);
        gravity<J2>(Ph, r2x, r2y, r2z, a2x, a2y, a2z, s2.g);
        const double i2 = fast_rcp(m2);
        {
            const double qx = umx * i2, qy = umy * i2, qz = umz * i2;
            a2x += qx;
            a2y += qy;
            a2z += qz;
            s2.dx = -qx * i2 * dflag;
            s2.dy = -qy * i2 * dflag;
            s2.dz = -qz * i2 * dflag;
        }
        const double bx = vx + rx, by = vy + ry, bz = vz + rz;
        const double r3x = fma(0.5, a2x, bx), r3y = fma(0.5, a2y, by), r3z = fma(0.5, a2z, bz);
        gravity<J2>(Ph, r3x, r3y, r3z, a3x, a3y, a3z, s3.g);
        {
            const double i3 = fast_rcp(m3);
            const double qx = uex * i3, qy = uey * i3, qz = uez * i3;
            a3x += qx;
            a3y += qy;
            a3z += qz;
            s3.dx = -qx * i3 * dflag;
            s3.dy = -qy * i3 * dflag;
            s3.dz = -qz * i3 * dflag;
        }
        // ---- state: end of the step and Hermite midpoint ------------------------------------------------------------------
        double vmid[3], amid[3], gmid[3];
        {
            const double Ax = fma(2.0, a2x, a1x), Ay = fma(2.0, a2y, a1y), Az = fma(2.0, a2z, a1z);
            const double Tx = fma(4.0, a2x, a1x) + a3x, Ty = fma(4.0, a2y, a1y) + a3y, Tz = fma(4.0, a2z, a1z) + a3z;
            const double rmx = fma(-c48, Tx, fma(c12, Ax, hx)), rmy = fma(-c48, Ty, fma(c12, Ay, hy)),
                         rmz = fma(-c48, Tz, fma(c12, Az, hz));
            vmid[0] = fma(-c24, Tx, fma(0.25, Ax, vx));
            vmid[1] = fma(-c24, Ty, fma(0.25, Ay, vy));
            vmid[2] = fma(-c24, Tz, fma(0.25, Az, vz));
            rx = fma(c6, Ax, bx);
            ry = fma(c6, Ay, by);
            rz = fma(c6, Az, bz);
            vx = fma(c6, Tx, vx);
            vy = fma(c6, Ty, vy);
            vz = fma(c6, Tz, vz);
            m = m3;
            if (pairmode) {      // node in the middle: acceleration and G r at the interpolated position
                Sym3 gdead;
                double amx, amy, amz;
                gravity<J2>(Ph, rmx, rmy, rmz, amx, amy, amz, gdead, gmid);
                amid[0] = fma(umx, i2, amx);
                amid[1] = fma(umy, i2, amy);
                amid[2] = fma(umz, i2, amz);
            }
        }
        // ---- this lane's column: step (the d of the stages is zero except on lane 6) and the middle node's row ------------
        double mr[3], mv[3];
        column_step_mid<true>(pr, pv, s1, s2, s3, mr, mv);
        if (pairmode) {
            const double bs = -P.inv_ve * iunm;
            const double b[3] = {bs * umx, bs * umy, bs * umz};
            const double cr[3] = {grp_bcast(mr[0], 6), grp_bcast(mr[1], 6), grp_bcast(mr[2], 6)};
            const double cv[3] = {grp_bcast(mv[0], 6), grp_bcast(mv[1], 6), grp_bcast(mv[2], 6)};
            grp_node(A, mr, mv, cr, cv, vmid, amid, gmid, b, i2 * H, mdm, (iunm != 0.0) ? mdm : 0.0, 1.0, sm, sgn, row6);
        }
        ux = uex;
        uy = uey;
        uz = uez;
        iun = iune;
        un = uue * iune;
        jn += (double)nodes_per_step;
    }

    // ---- epilogue: A_k = Phi_end, [B_kp B_kn Sigma_k xi_k] = Phi_end * integrals (:43-44,77-80) --------------------------
    // scalings as epilogue_store(acc, pr, pv, sB = hn, sS = h/H, sX = hn/H, ..., cs = H, vs = 1/H)
    const double iH = 1.0 / H;
    const double sB = hn, sS = h * iH, sX = hn * iH, cs = H, vs = iH;
    const long long col = out_col(dst, offset, s, k, K);
    double *const o = dst.p[0] + col;
    int nonfinite = 0;
    auto store = [&](int row, double v) {
        nonfinite |= !(fabs(v) <= 1.79769313486231570e308);
        if (live) o[(long long)row * pitch] = v;
    };
    if (lane < 7) {
        const bool vcol = lane >= 3 && lane < 6;
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            store(a * 7 + lane, vcol ? pr[a] * cs : pr[a]);
            store((a + 3) * 7 + lane, vcol ? pv[a] : pv[a] * vs);
        }
    } else {
#pragma unroll
        for (int c = 0; c < 7; ++c) store(42 + c, (c == 6) ? 1.0 : 0.0);
    }
    // The accumulators of Phi^-1-row r sit on the lane that owns column (r < 3 ? r + 3 : r < 6 ? r - 3 : 6); the product
    // needs row r next to COLUMN r of Phi_end: swap them between the partner lanes, multiply, sum over the group.
    const int partner = (lane < 3) ? lane + 3 : (lane < 6) ? lane - 3 : lane;
    double I[8];      // integrals of row `lane`, as the 8 result vectors: Bp[0..2], Bn[0..2], Sigma, xi
#pragma unroll
    for (int j = 0; j < 3; ++j) {
        const double i0 = grp_bcast(A.A0[j], partner), i1 = grp_bcast(A.A1[j], partner);
        I[j] = sB * i1;
        I[3 + j] = sB * (i0 - i1);
    }
    I[6] = sS * grp_bcast(A.AS, partner);
    I[7] = sX * grp_bcast(A.AX, partner);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        double mine = 0.0;      // the value this lane stores: row `lane` of result vector j
#pragma unroll
        for (int a = 0; a < 7; ++a) {
            // Phi_end[a][lane] * I[lane][j];  row 6 of Phi_end is e7^T; lane 7 owns no column
            double t;
            if (a < 3) t = pr[a] * I[j];
            else if (a < 6) t = pv[a - 3] * I[j];
            else t = (lane == 6) ? I[j] : 0.0;
            if (lane == 7) t = 0.0;
            double v = grp_sum(t);
            if (a >= 3 && a < 6) v *= vs;
            if (lane == a) mine = v;
        }
        if (lane < 7) {
            const int row = (j < 3) ? (49 + lane * 3 + j) : (j < 6) ? (70 + lane * 3 + (j - 3)) : (j == 6) ? (91 + lane) : (98 + lane);
            store(row, mine);
        }
    }
    // status: one word per interval, any lane's finding counts
    int flag = bad ? 1 : (nonfinite ? 2 : 0);
#pragma unroll
    for (int d = 1; d < 8; d <<= 1) {
        const int other = __shfl_xor_sync(grp_mask(), flag, d, 8);
        flag = (flag == 1 || other == 1) ? 1 : max(flag, other);
    }
    if (status && live && lane == 0) status[gid] = flag;
}

}  // namespace mpc
