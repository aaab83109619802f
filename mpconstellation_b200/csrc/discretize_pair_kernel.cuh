// discretize_pair_kernel.cuh -- the fixed-step discretization with integrator steps that span TWO quadrature nodes.
//
// Same mathematics and the same 101 (integrator_steps) trapezoid nodes as discretize_kernel.  The difference is where
// the node values come from.  The reference takes them from the DENSE OUTPUT of its integrator (solve_ivp with t_eval:
// 1-4 RK45 steps per interval, 101 nodes read off the interpolant, linearize_discretize.py:37-48).  discretize_kernel
// takes one Runge-Kutta-Nystrom step per node; this kernel takes one step per two nodes and reads the node in the
// middle off the step's cubic Hermite interpolant (positions and velocities at both ends: for a midpoint that is
// O(h^4) accurate in the value AND in the derivative).  With the step-normalised variables the interpolation is four
// FMAs per position/velocity pair, because the sums the step already formed (K12 = k1 + 2 k2, K = k1 + 4 k2 + k3) are
// all it needs:
//     p_mid  = (p + 1/2 p') + 1/12 K12 - 1/48 K          p'_mid = p' + 1/4 K12 - 1/24 K
// On the reference's grids (0.005-0.03 orbit per interval) the result differs from one-step-per-node by 1e-13 ... 7e-12
// (the CPU restatement used by the tests implements both; DESIGN.md section 4), two to four orders below the
// reference's own integration error, for 29 % fewer FP64 instructions.
//
// The middle node's quadrature terms are accumulated COLUMN BY COLUMN while the columns are being stepped (column c of
// Phi gives row c-3 / c+3 of every Phi^-1 product, see node_accumulate), so the interpolated Phi never has to exist as
// a whole: no second copy of the 42 entries in registers.
//
// Per thread, the two-node steps are used for an even number of panels and steps short against the orbital rate
// (omega H <= 3.2e-3 rad); otherwise the thread runs discretize_thread (one step per node).
#pragma once
#include "discretize_kernel.cuh"

namespace mpc {

// One column through one RKN4 step (see column_step) that also returns the Hermite midpoint of the step.
template <bool MASSCOL>
__device__ __forceinline__ void column_step_mid(double (&pr)[3], double (&pv)[3], const StageLin &s1, const StageLin &s2,
                                                const StageLin &s3, double (&mr)[3], double (&mv)[3])
{
    constexpr double c6 = 1.0 / 6.0, c12 = 1.0 / 12.0, c24 = 1.0 / 24.0, c48 = 1.0 / 48.0;
    double k1x, k1y, k1z, k2x, k2y, k2z, k3x, k3y, k3z;
    if (MASSCOL) sym_mul_add(s1.g, pr[0], pr[1], pr[2], s1.dx, s1.dy, s1.dz, k1x, k1y, k1z);
    else sym_mul(s1.g, pr[0], pr[1], pr[2], k1x, k1y, k1z);
    const double hx = fma(0.5, pv[0], pr[0]), hy = fma(0.5, pv[1], pr[1]), hz = fma(0.5, pv[2], pr[2]);   // p + 1/2 p'
    const double q2x = fma(0.125, k1x, hx), q2y = fma(0.125, k1y, hy), q2z = fma(0.125, k1z, hz);
    if (MASSCOL) sym_mul_add(s2.g, q2x, q2y, q2z, s2.dx, s2.dy, s2.dz, k2x, k2y, k2z);
    else sym_mul(s2.g, q2x, q2y, q2z, k2x, k2y, k2z);
    const double bx = pv[0] + pr[0], by = pv[1] + pr[1], bz = pv[2] + pr[2];
    const double q3x = fma(0.5, k2x, bx), q3y = fma(0.5, k2y, by), q3z = fma(0.5, k2z, bz);
    if (MASSCOL) sym_mul_add(s3.g, q3x, q3y, q3z, s3.dx, s3.dy, s3.dz, k3x, k3y, k3z);
    else sym_mul(s3.g, q3x, q3y, q3z, k3x, k3y, k3z);
    const double ax = fma(2.0, k2x, k1x), ay = fma(2.0, k2y, k1y), az = fma(2.0, k2z, k1z);               // K12
    const double tx = fma(4.0, k2x, k1x) + k3x, ty = fma(4.0, k2y, k1y) + k3y, tz = fma(4.0, k2z, k1z) + k3z;   // K
    mr[0] = fma(-c48, tx, fma(c12, ax, hx));
    mr[1] = fma(-c48, ty, fma(c12, ay, hy));
    mr[2] = fma(-c48, tz, fma(c12, az, hz));
    mv[0] = fma(-c24, tx, fma(0.25, ax, pv[0]));
    mv[1] = fma(-c24, ty, fma(0.25, ay, pv[1]));
    mv[2] = fma(-c24, tz, fma(0.25, az, pv[2]));
    pr[0] = fma(c6, ax, bx);
    pr[1] = fma(c6, ay, by);
    pr[2] = fma(c6, az, bz);
    pv[0] = fma(c6, tx, pv[0]);
    pv[1] = fma(c6, ty, pv[1]);
    pv[2] = fma(c6, tz, pv[2]);
}

// What node_accumulate needs from the node itself (not from Phi), for the column-by-column form.
struct NodeVec {
    double cr[3], cv[3];            // mass column of Phi at the node
    double vv[3], aa[3], gg[3];     // v, a = f[3:6], G r   (scaled as discretize_kernel scales them)
    double b[3];                    // last row of Duf
    double im, md, mdb, w, ws;
};

// Contribution of ONE column of Phi (values pr, pv at the node) to the quadrature accumulators: column 3+a gives row a
// of every Phi^-1 product (TOP), column a gives row 3+a (see node_accumulate for the algebra; s = +1 / -1).
#define ACC(e) acc[(e) * BLOCK]
// Split in two so that the caller can issue the eight shared-memory loads BEFORE it steps the column: their latency
// then hides behind the column's arithmetic instead of stalling the accumulation (the accesses are volatile, they stay
// where the source puts them).
struct ColAcc {
    double A0[3], A1[3], AS, AX;
};

template <int BLOCK, bool TOP>
__device__ __forceinline__ void column_acc_load(volatile double *acc, int a, ColAcc &c)
{
    const int i0 = (TOP ? 0 : 9) + a * 3, i1 = (TOP ? 18 : 27) + a * 3, is = (TOP ? 36 : 39) + a, ix = (TOP ? 42 : 45) + a;
#pragma unroll
    for (int j = 0; j < 3; ++j) {
        c.A0[j] = ACC(i0 + j);
        c.A1[j] = ACC(i1 + j);
    }
    c.AS = ACC(is);
    c.AX = ACC(ix);
}

template <int BLOCK, bool TOP>
__device__ __forceinline__ void node_accumulate_column(volatile double *acc, int a, const double (&pr)[3], const double (&pv)[3],
                                                       const NodeVec &n, const ColAcc &c)
{
    const int i0 = (TOP ? 0 : 9) + a * 3, i1 = (TOP ? 18 : 27) + a * 3, is = (TOP ? 36 : 39) + a, ix = (TOP ? 42 : 45) + a;
    // e = s (pr.cv - pv.cr),  dv = pv.v,  pa = pr.a,  pg = pr.(G r)
    double e = pr[0] * n.cv[0], dv = pv[0] * n.vv[0], pa = pr[0] * n.aa[0], pg = pr[0] * n.gg[0];
#pragma unroll
    for (int i = 1; i < 3; ++i) {
        e = fma(pr[i], n.cv[i], e);
        dv = fma(pv[i], n.vv[i], dv);
        pa = fma(pr[i], n.aa[i], pa);
        pg = fma(pr[i], n.gg[i], pg);
    }
#pragma unroll
    for (int i = 0; i < 3; ++i) e = fma(-pv[i], n.cr[i], e);
    if (!TOP) e = -e;
    const double sdv = TOP ? dv : -dv;
    const double S = fma(e, n.md, sdv) - (TOP ? pa : -pa);          // e md + s dv - s pr.a
    const double X = (TOP ? pg : -pg) - fma(e, n.mdb, sdv);         // -e mdb - s dv + s pr.(G r)
    const double sim = TOP ? -n.im : n.im;
#pragma unroll
    for (int j = 0; j < 3; ++j) {
        const double q = fma(n.b[j], e, sim * pr[j]);               // b_j e - s im pr_j
        ACC(i0 + j) = fma(n.w, q, c.A0[j]);
        ACC(i1 + j) = fma(n.ws, q, c.A1[j]);
    }
    ACC(is) = fma(n.w, S, c.AS);
    ACC(ix) = fma(n.w, X, c.AX);
}

template <bool J2, int BLOCK, int MAXREG, int NDST>
__global__ void __launch_bounds__(BLOCK) __maxnreg__(MAXREG)
discretize_pair_kernel(const double *__restrict__ x, const double *__restrict__ u, const double *__restrict__ tf_arr,
                       DiscParams P, int n_sats, int K, int n_sub, DstTab dst, long long pitch, long long offset,
                       int32_t *__restrict__ status, int k0, int kc)
{
    // The launch covers the intervals k in [k0, k0 + kc) of every satellite (the whole batch: k0 = 0, kc = K - 1).  A
    // window of k is what the overlapped propagate -> discretize pass launches as soon as the propagation has produced
    // the samples up to k0 + kc (mpc_propagate_discretize).  gid is the interval's global index s (K-1) + k either way.
    extern __shared__ double acc_smem[];
    const long long tid = (long long)blockIdx.x * BLOCK + threadIdx.x;
    if (tid >= (long long)n_sats * kc) return;
    if (dst.stagger_phases > 1 && (int)blockIdx.x < dst.first_wave_ctas) {
        const long long wait = dst.stagger_cycles * (long long)(blockIdx.x % dst.stagger_phases) / dst.stagger_phases;
        const long long t0 = clock64();
        while (clock64() - t0 < wait) __nanosleep(2000);
    }
    volatile double *acc = acc_smem + threadIdx.x;

    // thread -> (satellite, interval): consecutive threads walk the direction in which the output columns are adjacent
    // (k for the satellite-major layout, the satellite for the k-major one), so that every store of a warp is one line
    int s, k;
    if (dst.km_ntot) {
        const int kk = (int)(tid / n_sats);
        s = (int)(tid - (long long)kk * n_sats);
        k = k0 + kk;
    } else {
        s = (int)(tid / kc);
        k = k0 + (int)(tid - (long long)s * kc);
    }
    const long long gid = (long long)s * (K - 1) + k;
    const double tf = tf_arr[s];
    const double *xs = x + ((long long)s * 7) * K + k;
    double rx = xs[0], ry = xs[K], rz = xs[2 * (long long)K];
    double vx = xs[3 * (long long)K], vy = xs[4 * (long long)K], vz = xs[5 * (long long)K];
    double m = xs[6 * (long long)K];
    UHold<false> hold;
    hold.init(u, s, k, K, K);

    const int n_pairs = n_sub >> 1;
    const double inv_n = 1.0 / (double)n_sub;
    const double h = inv_n / (double)(K - 1);  // node spacing in tau
    const double hn = tf * h;                  // node spacing of the unscaled system
    const double H = 2.0 * hn;                 // integrator step = two nodes
    {
        // The midpoint interpolation is O((omega H)^4): it is used only where the step is short against the local orbital
        // rate omega = sqrt(MU/|r|^3) -- omega H <= 3.2e-3 rad (5e-4 orbit), where it agrees with one step per node to
        // < 1e-11 -- and for an even number of panels.  Everything else (coarse user-chosen integrator_steps, very long
        // intervals, non-finite inputs) takes one step per node, like discretize_kernel.
        const double r2 = fma(rx, rx, fma(ry, ry, rz * rz));
        const double w2H2 = P.mu * H * H / (r2 * sqrt(r2));
        // The reference's setting, integrator_steps = 101: 20 steps and the 21-node rule kEmW (discretize_kernel.cuh) where
        // the integrands are smooth across the interval -- the held input changes by at most a quarter of its size between
        // the two nodes (|u_k+1 - u_k| <= 0.25 max|u|; both zero, a coast arc, counts), so |u(tau)| stays away from the kink
        // at zero -- and the step 5 h is short against the orbital rate (omega 5h <= 3.5e-3 rad: 0.011-orbit intervals).
        if (dst.em && n_sub == 100) {
            const double d2 = fma(hold.dux, hold.dux, fma(hold.duy, hold.duy, hold.duz * hold.duz));
            const double e0x = hold.u0x + hold.dux, e0y = hold.u0y + hold.duy, e0z = hold.u0z + hold.duz;
            const double a2 = fma(hold.u0x, hold.u0x, fma(hold.u0y, hold.u0y, hold.u0z * hold.u0z));
            const double b2 = fma(e0x, e0x, fma(e0y, e0y, e0z * e0z));
            if (d2 <= 0.0625 * fmax(a2, b2)) {
                if (w2H2 * 6.25 <= 1.2e-5) {
                    // the same orbital bound (omega 10h <= 7e-3 rad) and a held input that changes by at most an eighth
                    // of its size: 10 fifth-order steps and the 11-node rule kEmW3 (its remainder grows like the eighth
                    // power of that change: 2.5e-13 of the 101-node sums at 1/8, 4e-11 at 1/4)
                    if (dst.em >= 2 && d2 <= 0.015625 * fmax(a2, b2)) {
                        discretize_thread<J2, BLOCK, NDST, false, 3>(x, u, tf_arr, P, K, K, kEmSteps3, dst, pitch, offset, status, gid, acc);
                        return;
                    }
                    discretize_thread<J2, BLOCK, NDST, false, 1>(x, u, tf_arr, P, K, K, kEmSteps, dst, pitch, offset, status, gid, acc);
                    return;
                }
                // longer intervals (omega 2h <= 4.4e-3 rad: 0.035-orbit intervals): 50 steps and the 51-node rule kEmW2
                if (w2H2 <= 1.94e-5) {
                    discretize_thread<J2, BLOCK, NDST, false, 2>(x, u, tf_arr, P, K, K, kEmSteps2, dst, pitch, offset, status, gid, acc);
                    return;
                }
            }
        }
        if ((n_sub & 1) || !(w2H2 <= 1.0e-5)) {
            discretize_thread<J2, BLOCK, NDST, false>(x, u, tf_arr, P, K, K, n_sub, dst, pitch, offset, status, gid, acc);
            return;
        }
    }
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

    double pr[7][3], pv[7][3];
#pragma unroll
    for (int c = 0; c < 7; ++c)
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            pr[c][a] = (c == a) ? 1.0 : 0.0;
            pv[c][a] = (c == a + 3) ? 1.0 : 0.0;
        }
#pragma unroll
    for (int e = 0; e < kAccSlots; ++e) ACC(e) = 0.0;

    int bad = 0;
    double ux, uy, uz;
    // the two end nodes: as the reference looks them up (ref_node_input); the far one waits in shared memory
    ref_node_input(u + (long long)s * 3 * K, K, k + 1, H2, ux, uy, uz);
    ACC(kEndU) = ux;
    ACC(kEndU + 1) = uy;
    ACC(kEndU + 2) = uz;
    ref_node_input(u + (long long)s * 3 * K, K, k, H2, ux, uy, uz);
    double uu = fma(ux, ux, fma(uy, uy, uz * uz));
    double iun = inv_norm_guarded(uu, eps2);
    double un = uu * iun;

    for (int j = 0; j <= n_pairs; ++j) {
        if (j == n_pairs) {                                                         // the other end node
            ux = ACC(kEndU);
            uy = ACC(kEndU + 1);
            uz = ACC(kEndU + 2);
            uu = fma(ux, ux, fma(uy, uy, uz * uz));
            iun = inv_norm_guarded(uu, eps2);
            un = uu * iun;
        }
        // ---- stage 1 == even quadrature node 2j -----------------------------------------------------------------
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
        s1.dx = -tx * im;
        s1.dy = -ty * im;
        s1.dz = -tz * im;
        const double md1 = -un * Ph.inv_ve;
        {
            const double sfrac = (double)(2 * j) * inv_n;
            const double w = (j == 0 || j == n_pairs) ? 0.5 : 1.0;
            node_accumulate<BLOCK>(acc, pr, pv, P, im * H, ux, uy, uz, iun, md1, vx, vy, vz, a1x, a1y, a1z, gr[0], gr[1], gr[2],
                                   w, w * sfrac);
        }
        if (j == n_pairs) break;

        // ---- inputs and masses at the middle (node 2j+1) and the end (node 2j+2) of the step ---------------------
        const double sm = (double)(2 * j + 1) * inv_n, se = (double)(2 * j + 2) * inv_n;
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

        // ---- stages 2, 3 of the state --------------------------------------------------------------------------
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
            s2.dx = -qx * i2;
            s2.dy = -qy * i2;
            s2.dz = -qz * i2;
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
            s3.dx = -qx * i3;
            s3.dy = -qy * i3;
            s3.dz = -qz * i3;
        }
        // row-6 accumulators of the middle node: loaded here, used after the state update (latency hidden)
        double r6a[3], r6b[3];
#pragma unroll
        for (int jj = 0; jj < 3; ++jj) {
            r6a[jj] = ACC(48 + jj);
            r6b[jj] = ACC(51 + jj);
        }
        const double r6s = ACC(54), r6x = ACC(55);
        // ---- state: end of the step and Hermite midpoint ----------------------------------------------------------
        NodeVec nv;
        {
            const double Ax = fma(2.0, a2x, a1x), Ay = fma(2.0, a2y, a1y), Az = fma(2.0, a2z, a1z);
            const double Tx = fma(4.0, a2x, a1x) + a3x, Ty = fma(4.0, a2y, a1y) + a3y, Tz = fma(4.0, a2z, a1z) + a3z;
            const double rmx = fma(-c48, Tx, fma(c12, Ax, hx)), rmy = fma(-c48, Ty, fma(c12, Ay, hy)),
                         rmz = fma(-c48, Tz, fma(c12, Az, hz));
            nv.vv[0] = fma(-c24, Tx, fma(0.25, Ax, vx));
            nv.vv[1] = fma(-c24, Ty, fma(0.25, Ay, vy));
            nv.vv[2] = fma(-c24, Tz, fma(0.25, Az, vz));
            rx = fma(c6, Ax, bx);
            ry = fma(c6, Ay, by);
            rz = fma(c6, Az, bz);
            vx = fma(c6, Tx, vx);
            vy = fma(c6, Ty, vy);
            vz = fma(c6, Tz, vz);
            m = m3;
            // node 2j+1: acceleration and G r at the interpolated position (G itself is not needed at a node)
            Sym3 gdead;
            double amx, amy, amz;
            gravity<J2>(Ph, rmx, rmy, rmz, amx, amy, amz, gdead, nv.gg);
            nv.aa[0] = fma(umx, i2, amx);
            nv.aa[1] = fma(umy, i2, amy);
            nv.aa[2] = fma(umz, i2, amz);
        }
        {
            const double bs = -P.inv_ve * iunm;
            nv.b[0] = bs * umx;
            nv.b[1] = bs * umy;
            nv.b[2] = bs * umz;
            nv.im = i2 * H;
            nv.md = mdm;
            nv.mdb = (iunm != 0.0) ? mdm : 0.0;
            nv.w = 1.0;                                    // an odd node is never an end point of the trapezoid rule
            nv.ws = sm;
            // row 6 of the middle node: Phi^-1 row 6 = e7^T
#pragma unroll
            for (int jj = 0; jj < 3; ++jj) {
                ACC(48 + jj) = r6a[jj] + nv.b[jj];
                ACC(51 + jj) = fma(nv.ws, nv.b[jj], r6b[jj]);
            }
            ACC(54) = r6s + nv.md;
            ACC(55) = r6x - nv.mdb;
        }
        // ---- variational columns: step, and the middle node's terms column by column -------------------------------
        column_step_mid<true>(pr[6], pv[6], s1, s2, s3, nv.cr, nv.cv);
#pragma unroll
        for (int c = 0; c < 6; ++c) {
            double mr[3], mv[3];
            ColAcc ca;
            if (c < 3) column_acc_load<BLOCK, false>(acc, c, ca);
            else column_acc_load<BLOCK, true>(acc, c - 3, ca);
            column_step_mid<false>(pr[c], pv[c], s1, s2, s3, mr, mv);
            if (c < 3) node_accumulate_column<BLOCK, false>(acc, c, mr, mv, nv, ca);
            else node_accumulate_column<BLOCK, true>(acc, c - 3, mr, mv, nv, ca);
        }
        ux = uex;
        uy = uey;
        uz = uez;
        iun = iune;
        un = uue * iune;
    }

    // B and xi carry tf (tf h = hn per panel), Sigma does not (h); the accumulated Sigma / xi vectors carry the factor H,
    // the accumulated Duf vectors do not; cs / vs undo D = diag(I, H I, 1)
    const double iH = 1.0 / H;
    const int nonfinite = epilogue_store<BLOCK, NDST>(acc, pr, pv, hn, h * iH, hn * iH, dst, pitch, out_col(dst, offset, s, k, K), H, iH);
    if (status) status[gid] = bad ? 1 : (nonfinite ? 2 : 0);
}
#undef ACC

}  // namespace mpc
