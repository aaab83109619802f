// discretize_kernel.cuh -- batched SCvx linearize-and-discretize, one thread per (satellite, interval).
//
// What one thread computes (reference: linearize_discretize.py:8-82, get_matrices):
//   integrate  Phi' = A(x,u) Phi,  x' = f(x,u)  over [tau_k, tau_{k+1}]  (:262-290)
//   with u(tau) the first-order hold between u_k and u_{k+1}             (:294-315)
//   and at every node  accumulate  Phi^-1 [B lam-, B lam+, Sigma, xi]    (:63-75)
//   then  A_k = Phi_end,  [B_kn B_kp Sigma_k xi_k] = Phi_end * trapz(..) (:43-44, :77-80)
//
// Structure this kernel exploits (none of it changes the mathematics):
//   * every term of the RHS carries the factor tf (simulator.py:161, linearize_discretize.py:182,214),
//     so the kernel integrates the unscaled system with step hs = tf*h
//   * A = [[0 I 0],[G 0 d],[0 0 0]] with G symmetric (gravity gradient, + J2 gradient) and
//     d = -u/m^2 (linearize_discretize.py:146-179): the last row of Phi stays e7^T, each of the
//     7 columns of Phi is an independent second-order system  p_r'' = G(tau) p_r (+ d)
//   * a second-order system whose force does not depend on the velocity can be integrated with Nystrom's 3-stage
//     fourth-order Runge-Kutta method (three force evaluations per step instead of the classical scheme's four,
//     same order); the 3 stage matrices G1..G3 come from the state trajectory alone, so they are computed once
//     per step and shared by the 7 columns
//   * the 6x6 block of Phi is symplectic (G symmetric, no drag in the discretizer), so
//     Phi6^-1 = [[Pvv^T, -Prv^T],[-Pvr^T, Prr^T]]  and  Phi^-1 = [[Phi6^-1, -Phi6^-1 c],[0 1]]:
//     the per-node inverse (:69) costs no factorisation
//   * mass flow depends on tau only (|u(tau)|), so the mass stages are explicit
//
// Per-thread storage: Phi (42 doubles) and the state live in registers; the 56 quadrature
// accumulators live in shared memory, laid out [entry][thread] (conflict-free, 2 wavefronts per access).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace mpc {

struct DiscParams {
    double mu;       // MU
    double kj2;      // 1.5 * J2 * MU * R_E^2       (linearize_discretize.py:150, simulator.py:157)
    double inv_ve;   // 1 / (G0 * ISP)              (simulator.py:160)
};

struct Sym3 {  // symmetric 3x3
    double xx, xy, xz, yy, yz, zz;
};

struct StageLin {  // what the variational equation needs from one RK stage
    Sym3 g;        // d a / d r
    double dx, dy, dz;  // d a / d m = -u/m^2
};

__device__ __forceinline__ double fast_rcp(double a)
{
    // reciprocal: MUFU.RCP64H seed (relative error < 2^-20) and ONE third-order step, y (1 + e + e^2) with e = 1 - a y:
    // error e^3 < 1e-18, i.e. rounding-limited, in three dependent operations instead of the four of two Newton steps
    // (a > 0, normal range)
    double y;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(a));
    const double e = fma(-a, y, 1.0);
    return fma(y, fma(e, e, e), y);
}

// reciprocal to ~1e-12 (MUFU seed + ONE Newton step): for the scales of the RK45 error norm, where the controller turns
// a relative error of 1e-12 into a step-size change of 2e-13
__device__ __forceinline__ double fast_rcp1(double a)
{
    double y;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(a));
    const double e = fma(-a, y, 1.0);
    return fma(y, e, y);
}

__device__ __forceinline__ double fast_rsqrt(double a)
{
    // reciprocal square root: MUFU.RSQ64H seed (relative error d < 2^-20) and ONE third-order step,
    // y (1 + e/2 + 3 e^2/8) with e = 1 - a y^2 = 2 d: the next term, 5 e^3/16 < 3e-18, is below rounding.  Five operations,
    // four of them dependent, instead of the seven / six of two Newton steps (a > 0, normal range)
    double y;
    asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(a));
    const double e = fma(-(a * y), y, 1.0);
    return fma(y * e, fma(e, 0.375, 0.5), y);
}

// 1/sqrt(uu) if uu > thr, else 0 (the reference's |u| <= eps guard, linearize_discretize.py:208), without a branch:
// the Newton sequence always runs (on a harmless argument when the guard trips) and a select picks the result, so
// a warp with mixed thrust / no-thrust intervals does not diverge and no BSSY/BSYNC pair sits in the step loop.
__device__ __forceinline__ double inv_norm_guarded(double uu, double thr)
{
    const bool on = uu > thr;
    const double r = fast_rsqrt(on ? uu : 1.0);
    return on ? r : 0.0;
}

// acceleration (without the thrust/mass part) and its gradient at position r.
// G r comes for free from Euler's theorem on homogeneous functions: a_g is homogeneous of degree -2 in r and a_J2 of
// degree -4, so (d a_g/d r) r = -2 a_g and (d a_J2/d r) r = -4 a_J2  =>  G r = -2 a - 2 a_J2  (a = a_g + a_J2).
template <bool J2>
__device__ __forceinline__ void gravity(const DiscParams &P, double rx, double ry, double rz, double &ax,
                                        double &ay, double &az, Sym3 &g, double *gr = nullptr)
{
    const double r2 = fma(rx, rx, fma(ry, ry, rz * rz));
    const double ir = fast_rsqrt(r2);
    const double ir2 = ir * ir;
    const double mu3 = P.mu * ir * ir2;  // MU / |r|^3
    const double nx = rx * ir, ny = ry * ir, nz = rz * ir;
    const double t3 = 3.0 * mu3;
    const double tx = t3 * nx, ty = t3 * ny, tz = t3 * nz;
    // G = -MU/|r|^3 I + 3 MU/|r|^5 r r^T            (linearize_discretize.py:146-147)
    g.xx = fma(tx, nx, -mu3);
    g.yy = fma(ty, ny, -mu3);
    g.zz = fma(tz, nz, -mu3);
    g.xy = tx * ny;
    g.xz = tx * nz;
    g.yz = ty * nz;
    // a_g = -MU r / |r|^3                            (simulator.py:145)
    ax = -mu3 * rx;
    ay = -mu3 * ry;
    az = -mu3 * rz;
    if (gr) {
        gr[0] = -2.0 * ax;
        gr[1] = -2.0 * ay;
        gr[2] = -2.0 * az;
    }
    if (J2) {
        // a_J2 = kJ2/|r|^5 diag(5q-1, 5q-1, 5q-3) r,  q = (z/|r|)^2      (simulator.py:156-157)
        // its gradient (the symmetric Hessian of the J2 potential; equals the reference's
        // Dr_aJ2, linearize_discretize.py:150-158) written in the unit vector n = r/|r|:
        //   J = kJ2/|r|^5 [ diag(c1,c1,c3) - (35q-5) n n^T + 10 q-terms ]  (see DESIGN.md)
        const double q = nz * nz;
        const double k5 = P.kj2 * ir2 * ir2 * ir;
        const double c1 = fma(5.0, q, -1.0);
        const double c3 = fma(5.0, q, -3.0);
        const double k5c1 = k5 * c1;
        const double jx = k5c1 * rx, jy = k5c1 * ry, jz = (k5 * c3) * rz;
        ax += jx;
        ay += jy;
        az += jz;
        if (gr) {
            gr[0] = fma(-4.0, jx, gr[0]);
            gr[1] = fma(-4.0, jy, gr[1]);
            gr[2] = fma(-4.0, jz, gr[2]);
        }
        const double e = k5 * fma(35.0, q, -5.0);   // k5 (35q - 5)
        const double f = k5 * fma(-35.0, q, 15.0);  // k5 (15 - 35q)
        const double ex = e * nx, ey = e * ny;
        g.xx += fma(-ex, nx, k5c1);
        g.yy += fma(-ey, ny, k5c1);
        g.xy = fma(-ex, ny, g.xy);
        g.xz = fma(f * nx, nz, g.xz);
        g.yz = fma(f * ny, nz, g.yz);
        g.zz = fma(k5, fma(q, fma(-35.0, q, 30.0), -3.0), g.zz);
    }
}

__device__ __forceinline__ void sym_mul(const Sym3 &g, double px, double py, double pz, double &ox, double &oy,
                                        double &oz)
{
    ox = fma(g.xz, pz, fma(g.xy, py, g.xx * px));
    oy = fma(g.yz, pz, fma(g.yy, py, g.xy * px));
    oz = fma(g.zz, pz, fma(g.yz, py, g.xz * px));
}

__device__ __forceinline__ void sym_mul_add(const Sym3 &g, double px, double py, double pz, double cx, double cy,
                                            double cz, double &ox, double &oy, double &oz)
{
    ox = fma(g.xz, pz, fma(g.xy, py, fma(g.xx, px, cx)));
    oy = fma(g.yz, pz, fma(g.yy, py, fma(g.xy, px, cy)));
    oz = fma(g.zz, pz, fma(g.yz, py, fma(g.xz, px, cz)));
}

// One column of Phi through one step of Nystrom's 3-stage fourth-order method for p'' = G(t) p (+ d):
//     k1 = G1 p,  k2 = G2 (p + 1/2 p' + 1/8 k1),  k3 = G3 (p + p' + 1/2 k2),
//     p+ = p + p' + 1/6 (k1 + 2 k2),   p'+ = p' + 1/6 (k1 + 4 k2 + k3)
// in the STEP-NORMALISED variables of discretize_kernel: velocities scaled by the step hs, G and d scaled by hs^2, so
// the step is 1 and every coefficient is a literal (an immediate / constant-bank operand instead of a third register
// operand: a DFMA with three distinct register sources issues every 3 cycles on sm_100a, with two every 2).
// G1..G3 are the stage matrices of the SAME scheme applied to the state, so Phi is the exact derivative of the
// numerical flow.  MASSCOL: column 6, whose forcing is d_j = -u/m^2 at each stage (Phi[6][6] == 1).
template <bool MASSCOL>
__device__ __forceinline__ void column_step(double (&pr)[3], double (&pv)[3], const StageLin &s1,
                                            const StageLin &s2, const StageLin &s3)
{
    constexpr double c6 = 1.0 / 6.0;
    double k1x, k1y, k1z, k2x, k2y, k2z, k3x, k3y, k3z;
    if (MASSCOL) sym_mul_add(s1.g, pr[0], pr[1], pr[2], s1.dx, s1.dy, s1.dz, k1x, k1y, k1z);
    else sym_mul(s1.g, pr[0], pr[1], pr[2], k1x, k1y, k1z);
    // stage 2 position: p + 1/2 p_v + 1/8 k1
    const double q2x = fma(0.125, k1x, fma(0.5, pv[0], pr[0])), q2y = fma(0.125, k1y, fma(0.5, pv[1], pr[1])),
                 q2z = fma(0.125, k1z, fma(0.5, pv[2], pr[2]));
    if (MASSCOL) sym_mul_add(s2.g, q2x, q2y, q2z, s2.dx, s2.dy, s2.dz, k2x, k2y, k2z);
    else sym_mul(s2.g, q2x, q2y, q2z, k2x, k2y, k2z);
    // stage 3 position: p + p_v + 1/2 k2
    const double bx = pv[0] + pr[0], by = pv[1] + pr[1], bz = pv[2] + pr[2];
    const double q3x = fma(0.5, k2x, bx), q3y = fma(0.5, k2y, by), q3z = fma(0.5, k2z, bz);
    if (MASSCOL) sym_mul_add(s3.g, q3x, q3y, q3z, s3.dx, s3.dy, s3.dz, k3x, k3y, k3z);
    else sym_mul(s3.g, q3x, q3y, q3z, k3x, k3y, k3z);
    pr[0] = fma(c6, fma(2.0, k2x, k1x), bx);
    pr[1] = fma(c6, fma(2.0, k2y, k1y), by);
    pr[2] = fma(c6, fma(2.0, k2z, k1z), bz);
    pv[0] = fma(c6, fma(4.0, k2x, k1x) + k3x, pv[0]);
    pv[1] = fma(c6, fma(4.0, k2y, k1y) + k3y, pv[1]);
    pv[2] = fma(c6, fma(4.0, k2z, k1z) + k3z, pv[2]);
}

// Python's float floor division v // w for v >= 0, w > 0 (CPython float_divmod): NOT floor(v / w) -- 0.5 // 0.1 is 4.
__device__ __forceinline__ double py_floordiv(double v, double w)
{
    const double mod = fmod(v, w);
    const double div = (v - mod) / w;
    if (div == 0.0) return 0.0;
    double fl = floor(div);
    if (div - fl > 0.5) fl += 1.0;
    return fl;
}

// The input the REFERENCE sees at node i of tau = np.linspace(0, 1, Ku): Discretizer.u_FOH (linearize_discretize.py:
// 294-315) looks the node up on the global grid, k = int(tau // dtau), and interpolates there.  Rounding decides whether
// tau_i lands in the interval left or right of it (tau_6 = 0.6000000000000001 of an 11-node grid lands in [6, 7], tau_5 =
// 0.5 in [4, 5]), so the value is u_i only up to ~1e-16 (u_{i+-1} - u_i).  That is immaterial everywhere except in the
// |u| <= eps guard of B_func (:208): where u_i is exactly 0 next to a thrusting node the reference gets |u| ~ 1e-15 > eps
// and a unit thrust direction (taken from the NEIGHBOUR) in the mass row of B, where a straight hold gets 0.  The kernels
// therefore take the inputs of the two END nodes of every interval from here (interior nodes are always looked up in
// their own interval).  us: u of this satellite, [3][Ku]; f: the kernel's scaling of u.  Called twice per interval.
__device__ __noinline__ void ref_node_input(const double *__restrict__ us, int Ku, int i, double f, double &ux, double &uy,
                                            double &uz)
{
    if (i >= Ku - 1) {                       // tau == 1: the last column (:305-306)
        ux = f * us[Ku - 1];
        uy = f * us[2 * Ku - 1];
        uz = f * us[3 * (long long)Ku - 1];
        return;
    }
    const double km1 = (double)(Ku - 1);
    const double dtau = 1.0 / km1;
    const double tau = (double)i * dtau;     // np.linspace: arange(Ku) * step
    // int(tau // dtau) with Python's float floor division (py_floordiv).  For tau = fl(i * dtau) the quotient is i when the
    // product was rounded up or is exact and i - 1 when it was rounded down (fmod then returns dtau - |rounding error|),
    // and the sign of the rounding error is one FMA: checked against CPython for every node of every grid up to 1200
    // nodes (741 k cases, 351 k of them i - 1).  fmod and the division of py_floordiv cost ~700 instructions a call.
    int kq = i - (fma((double)i, dtau, -tau) > 0.0 ? 1 : 0);
    kq = min(max(kq, 0), Ku - 2);
    const double tk = (double)kq / km1, tk1 = (double)(kq + 1) / km1;
    // (one division for the two weights: whether a weight is exactly 0 -- the only thing that matters, see above -- is
    //  decided by its numerator)
    const double iw = 1.0 / (tk1 - tk);
    const double ln = (tk1 - tau) * iw, lp = (tau - tk) * iw;
    ux = f * __dadd_rn(__dmul_rn(ln, us[kq]), __dmul_rn(lp, us[kq + 1]));
    uy = f * __dadd_rn(__dmul_rn(ln, us[Ku + kq]), __dmul_rn(lp, us[Ku + kq + 1]));
    uz = f * __dadd_rn(__dmul_rn(ln, us[2 * (long long)Ku + kq]), __dmul_rn(lp, us[2 * (long long)Ku + kq + 1]));
}

// Input hold u(tau).  GENU = false: u is given on the K nodes of x, so inside one interval the reference's
// first-order hold (linearize_discretize.py:294-315) is the straight line between u_k and u_{k+1}.
// GENU = true: u has its own column count Ku (the reference accepts that: u_FOH takes its grid from u itself,
// :308-315; its own test_linearize_many does it, test_discretizer.py:103) -- the hold is evaluated on u's global
// grid with the reference's index arithmetic (tau == 1 -> last column, k = floor(tau / dtau)).
template <bool GENU>
struct UHold;

template <>
struct UHold<false> {
    double u0x, u0y, u0z, dux, duy, duz;
    __device__ __forceinline__ void init(const double *u, int sat, int k, int K, int)
    {
        const double *us = u + ((long long)sat * 3) * K + k;
        u0x = us[0];
        u0y = us[K];
        u0z = us[2 * (long long)K];
        dux = us[1] - u0x;
        duy = us[K + 1] - u0y;
        duz = us[2 * (long long)K + 1] - u0z;
    }
    __device__ __forceinline__ void scale(double f)   // hold f*u(tau) from now on
    {
        u0x *= f; u0y *= f; u0z *= f;
        dux *= f; duy *= f; duz *= f;
    }
    // s: position inside the interval in [0,1];  tau: the same point on the global grid (unused here)
    __device__ __forceinline__ void at(double s, double, double &ux, double &uy, double &uz) const
    {
        ux = fma(s, dux, u0x);
        uy = fma(s, duy, u0y);
        uz = fma(s, duz, u0z);
    }
};

template <>
struct UHold<true> {
    const double *base;
    int Ku;
    double f;
    __device__ __forceinline__ void init(const double *u, int sat, int, int, int Ku_)
    {
        Ku = Ku_;
        f = 1.0;
        base = u + ((long long)sat * 3) * Ku_;
    }
    __device__ __forceinline__ void scale(double f_) { f = f_; }
    __device__ __forceinline__ void at(double, double tau, double &ux, double &uy, double &uz) const
    {
        if (tau == 1.0 || Ku < 2) {
            ux = f * base[Ku - 1];
            uy = f * base[2 * Ku - 1];
            uz = f * base[3 * (long long)Ku - 1];
            return;
        }
        const double km1 = (double)(Ku - 1);
        const double dtau = 1.0 / km1;
        int k = (int)py_floordiv(tau, dtau);
        k = min(max(k, 0), Ku - 2);
        const double lo = (double)k / km1, hi = (double)(k + 1) / km1;
        const double ln = (hi - tau) / (hi - lo), lp = (tau - lo) / (hi - lo);
        ux = f * fma(ln, base[k], lp * base[k + 1]);
        uy = f * fma(ln, base[Ku + k], lp * base[Ku + k + 1]);
        uz = f * fma(ln, base[2 * (long long)Ku + k], lp * base[2 * (long long)Ku + k + 1]);
    }
};

// Shared-memory accumulator slots (per thread), entry e at smem[e * BLOCK + tid]:
//   0..17  I0[a][j]   sum w   Phi^-1 Duf   rows a = 0..5 (row 6 handled below), j = 0..2
//  18..35  I1[a][j]   sum w s Phi^-1 Duf
//  36..41  IS[a]      sum w   Phi^-1 f(tf=1)
//  42..47  IX[a]      sum w   Phi^-1 xi'
//  48..50  I0m[j], 51..53 I1m[j], 54 ISm, 55 IXm   (row 6: Phi^-1 row 6 = e7^T)
constexpr int kAccSlots = 56;
constexpr int kEndU = kAccSlots;          // 3 more slots: the input of the interval's END node (ref_node_input), parked
constexpr int kDiscSlots = kAccSlots + 3; //   there from the start of the kernel so that no call sits in the step loop
constexpr int kMaxDst = 8;

struct DstTab {  // destination buffers of the (optionally multi-destination) SoA store
    double *p[kMaxDst];
    // fused all-gather options (all zero for a plain launch):
    int skip_const;            // 1: rows 42..48 (structural constants) go to p[0] only; 2: to no destination
    int stagger_phases;        // > 1: CTAs of the first wave start with a delay of (blockIdx % phases)/phases of one
    int first_wave_ctas;       //      interval's run time, so that the store phases of the CTAs sharing the NVLink
    long long stagger_cycles;  //      egress do not coincide; stagger_cycles = run time of one interval in SM clocks
    // k-major gathered layout (0 = the default, satellite-major: column = offset + s (K-1) + k).  km_ntot > 0: column =
    // k * km_ntot + km_soff + s, with km_ntot the satellites of ALL ranks and km_soff the first satellite of this one:
    // the intervals k of all satellites are adjacent, so a window of k (the overlapped pass) writes whole rows of
    // consecutive columns -- whole 256-byte lines per warp, also to the peers -- instead of 13-column fragments.
    long long km_ntot, km_soff;
    // != 0: the launch may evaluate the 101-node trapezoid sums of an interval through their Euler-Maclaurin expansion
    // (kEmW, kEmW2 below; discretize_pair_kernel decides per interval); >= 2: also through the 11-node form kEmW3 on
    // fifth-order steps.  Set by the launcher, mpc_set_tuning(37/38) and (39/40).
    int em;
};

// column of interval (s, k) in the SoA output
__device__ __forceinline__ long long out_col(const DstTab &d, long long offset, int s, int k, int K)
{
    return d.km_ntot ? (long long)k * d.km_ntot + d.km_soff + s : offset + (long long)s * (K - 1) + k;
}

// Quadrature-node accumulation shared by the fixed-step and the adaptive kernel:
//   acc += w * Phi^-1 [Duf, Sigma, xi']   and   acc1 += w*lambda+ * Phi^-1 Duf      (ws = w * lambda+)
// with Phi given by its columns (pr, pv), Phi^-1 from the symplectic structure, and the slots laid out as
// documented at kAccSlots.  linearize_discretize.py:63-75.
#define ACC(e) acc[(e) * BLOCK]
template <int BLOCK>
__device__ __forceinline__ void node_accumulate(volatile double *acc, const double (&pr)[7][3], const double (&pv)[7][3],
                                                const DiscParams &P, double im, double ux, double uy, double uz,
                                                double iun, double md1, double vx, double vy, double vz, double a1x,
                                                double a1y, double a1z, double grx, double gry, double grz, double w,
                                                double ws)
{
    // Duf = [0; I/m; b^T],  b = -u / (G0 ISP |u|)  (0 when |u| <= eps)      (:200-212)
    const double bs = -P.inv_ve * iun;
    const double b[3] = {bs * ux, bs * uy, bs * uz};
    // Sigma = f(tf=1) = [v; a; mdot] (:252-253);  xi' = -[v; G r; mdot_B] with mdot_B the
    // (Duf u) last row, which is 0 under the eps guard
    const double mdb = (iun != 0.0) ? md1 : 0.0;
    // Row pairs: column 3+a of Phi gives row a of every Phi^-1 product, column a gives row 3+a
    //   e = -Phi6^-1 c (c = column 6):  et[a] = pr[3+a].cv - pv[3+a].cr ,  eb[a] = pv[a].cr - pr[a].cv
    //   Q = Phi^-1 Duf:   row a: -pr[3+a][j]/m + b_j et[a] ;  row 3+a: pr[a][j]/m + b_j eb[a]
    //   Phi^-1 w = [Phi6^-1 w6 + e wm ; wm] :  row a: pv[3+a].wr - pr[3+a].wv ;  row 3+a: pr[a].wv - pv[a].wr
    // Loops run with the vector COMPONENT outermost so that consecutive FMAs share one source (cv[i], cr[i],
    // v[i], a[i], (G r)[i]): a DFMA with three distinct register sources issues every 3 cycles on sm_100a,
    // one whose source sits in the operand-reuse cache every 2 (profiles/r01_micro_fp64_pipe.txt).
    const double vv[3] = {vx, vy, vz}, aa[3] = {a1x, a1y, a1z}, gg[3] = {grx, gry, grz};
    double et[3], eb[3], dvt[3], dvb[3], st[3], sb[3], xt[3], xb[3];
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        et[a] = pr[3 + a][0] * pv[6][0];
        eb[a] = -pr[a][0] * pv[6][0];
    }
#pragma unroll
    for (int i = 1; i < 3; ++i)
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            et[a] = fma(pr[3 + a][i], pv[6][i], et[a]);
            eb[a] = fma(-pr[a][i], pv[6][i], eb[a]);
        }
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            et[a] = fma(-pv[3 + a][i], pr[6][i], et[a]);
            eb[a] = fma(pv[a][i], pr[6][i], eb[a]);
        }
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        dvt[a] = pv[3 + a][0] * vv[0];
        dvb[a] = pv[a][0] * vv[0];
    }
#pragma unroll
    for (int i = 1; i < 3; ++i)
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            dvt[a] = fma(pv[3 + a][i], vv[i], dvt[a]);
            dvb[a] = fma(pv[a][i], vv[i], dvb[a]);
        }
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        st[a] = fma(et[a], md1, dvt[a]);
        sb[a] = fma(eb[a], md1, -dvb[a]);
        xt[a] = -fma(et[a], mdb, dvt[a]);
        xb[a] = fma(-eb[a], mdb, dvb[a]);
    }
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            st[a] = fma(-pr[3 + a][i], aa[i], st[a]);
            sb[a] = fma(pr[a][i], aa[i], sb[a]);
        }
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            xt[a] = fma(pr[3 + a][i], gg[i], xt[a]);
            xb[a] = fma(-pr[a][i], gg[i], xb[a]);
        }
    // The 16 accumulators of a row pair are loaded together, updated, stored together (the volatile
    // accesses keep program order, so grouping them exposes one shared-memory latency per group).
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        double A0t[3], A1t[3], A0b[3], A1b[3];
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            A0t[j] = ACC(a * 3 + j);
            A1t[j] = ACC(18 + a * 3 + j);
            A0b[j] = ACC(9 + a * 3 + j);
            A1b[j] = ACC(27 + a * 3 + j);
        }
        double ASt = ACC(36 + a), ASb = ACC(39 + a), AXt = ACC(42 + a), AXb = ACC(45 + a);
        double qt[3], qb[3];
#pragma unroll
        for (int j = 0; j < 3; ++j) qt[j] = fma(b[j], et[a], -im * pr[3 + a][j]);
#pragma unroll
        for (int j = 0; j < 3; ++j) qb[j] = fma(b[j], eb[a], im * pr[a][j]);
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            A0t[j] = fma(w, qt[j], A0t[j]);
            A0b[j] = fma(w, qb[j], A0b[j]);
        }
        ASt = fma(w, st[a], ASt);
        ASb = fma(w, sb[a], ASb);
        AXt = fma(w, xt[a], AXt);
        AXb = fma(w, xb[a], AXb);
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            A1t[j] = fma(ws, qt[j], A1t[j]);
            A1b[j] = fma(ws, qb[j], A1b[j]);
        }
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            ACC(a * 3 + j) = A0t[j];
            ACC(18 + a * 3 + j) = A1t[j];
            ACC(9 + a * 3 + j) = A0b[j];
            ACC(27 + a * 3 + j) = A1b[j];
        }
        ACC(36 + a) = ASt;
        ACC(39 + a) = ASb;
        ACC(42 + a) = AXt;
        ACC(45 + a) = AXb;
    }
    {   // row 6: Phi^-1 row 6 = e7^T, so the integrands are the last rows of Duf, Sigma, xi'
        double m0[3], m1[3];
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            m0[j] = ACC(48 + j);
            m1[j] = ACC(51 + j);
        }
        double mS = ACC(54), mX = ACC(55);
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            ACC(48 + j) = fma(w, b[j], m0[j]);
            ACC(51 + j) = fma(ws, b[j], m1[j]);
        }
        ACC(54) = fma(w, md1, mS);
        ACC(55) = fma(-w, mdb, mX);
    }
}

// Epilogue shared by both kernels: A_k = Phi_end; [B_kp B_kn Sigma_k xi_k] = Phi_end * integrals, with the
// integrals scaled by sB (B carries tf, :182,214) / sS (Sigma does not, :252) / sX (xi; = sB unless the caller's
// accumulated xi vectors carry a factor of their own); SoA store to NDST buffers.
// linearize_discretize.py:43-44,77-80.  Returns nonzero when a stored value is not finite.
// cs / vs undo a similarity scaling of the velocity block: the caller's Phi is D Phi D^-1 and its integrals are
// D * (integrals) with D = diag(I3, cs I3, 1), vs = 1/cs (discretize_kernel: cs = step; adaptive kernel: cs = vs = 1,
// and the multiplications by 1.0 leave every bit unchanged).
template <int BLOCK, int NDST>
__device__ __forceinline__ int epilogue_store(volatile double *acc, const double (&pr)[7][3], const double (&pv)[7][3],
                                              double sB, double sS, double sX, const DstTab &dst, long long pitch,
                                              long long col, double cs = 1.0, double vs = 1.0)
{
    double *dsts[NDST];
#pragma unroll
    for (int d = 0; d < NDST; ++d) dsts[d] = dst.p[d];
    int nonfinite = 0;
    auto store = [&](int row, double v) {
        nonfinite |= !(fabs(v) <= 1.79769313486231570e308);
#pragma unroll
        for (int d = 0; d < NDST; ++d) dsts[d][(long long)row * pitch + col] = v;
    };
    // A_k = Phi_end (row-major 7x7)
#pragma unroll
    for (int a = 0; a < 3; ++a)
#pragma unroll
        for (int c = 0; c < 7; ++c) {
            const bool vcol = (c >= 3 && c < 6);
            store(a * 7 + c, vcol ? pr[c][a] * cs : pr[c][a]);
            store((a + 3) * 7 + c, vcol ? pv[c][a] : pv[c][a] * vs);
        }
    if (dst.skip_const == 0) {
#pragma unroll
        for (int c = 0; c < 7; ++c) store(42 + c, (c == 6) ? 1.0 : 0.0);
    } else if (dst.skip_const == 1) {   // remote buffers were initialised once with the constants
#pragma unroll
        for (int c = 0; c < 7; ++c) dsts[0][(long long)(42 + c) * pitch + col] = (c == 6) ? 1.0 : 0.0;
    }
    // Bp = sB*I1, Bn = sB*(I0 - I1), Sigma = sS*IS, xi = sB*IX
    // result row a: sum_c Phi[a][c] I[c][.],  Phi[a][c] = pr[c][a] (a<3) / pv[c][a-3] (a<6); row 6 = I[6][.]
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        double I[7];
        if (j < 3) {
#pragma unroll
            for (int c = 0; c < 6; ++c) I[c] = sB * ACC(18 + c * 3 + j);
            I[6] = sB * ACC(51 + j);
        } else if (j < 6) {
#pragma unroll
            for (int c = 0; c < 6; ++c) I[c] = sB * (ACC(c * 3 + (j - 3)) - ACC(18 + c * 3 + (j - 3)));
            I[6] = sB * (ACC(48 + (j - 3)) - ACC(51 + (j - 3)));
        } else if (j == 6) {
#pragma unroll
            for (int c = 0; c < 6; ++c) I[c] = sS * ACC(36 + c);
            I[6] = sS * ACC(54);
        } else {
#pragma unroll
            for (int c = 0; c < 6; ++c) I[c] = sX * ACC(42 + c);
            I[6] = sX * ACC(55);
        }
#pragma unroll
        for (int a = 0; a < 7; ++a) {
            double v;
            if (a < 3) {
                v = pr[0][a] * I[0];
#pragma unroll
                for (int c = 1; c < 7; ++c) v = fma(pr[c][a], I[c], v);
            } else if (a < 6) {
                v = pv[0][a - 3] * I[0];
#pragma unroll
                for (int c = 1; c < 7; ++c) v = fma(pv[c][a - 3], I[c], v);
                v *= vs;
            } else {
                v = I[6];
            }
            const int row = (j < 3) ? (49 + a * 3 + j) : (j < 6) ? (70 + a * 3 + (j - 3)) : (j == 6) ? (91 + a) : (98 + a);
            store(row, v);
        }
    }
    return nonfinite;
}
#undef ACC

// One interval, one integrator step per quadrature node: the whole per-thread computation (the kernel below is a thin
// wrapper; discretize_pair_kernel falls back to it for intervals whose steps are too long for its midpoint interpolation).
// The composite trapezoid sum over the reference's 101 uniform nodes (linearize_discretize.py:27-28, 77-80), from 21 of
// them.  For a smooth integrand g the trapezoid sum with spacing h is, by the Euler-Maclaurin formula,
//     T(h) = I + c2 h^2 + c4 h^4 + c6 h^6 + O(h^8),
// with I the integral and c2, c4, c6 fixed by derivatives of g at the two ends of the interval -- the same numbers for every
// h.  The sums over every 5th, 10th, 20th and 25th node, T(5h), T(10h), T(20h), T(25h), therefore determine T(h): with the
// weights w solving sum w = 1, sum w n^2 = 1, sum w n^4 = 1, sum w n^6 = 1 for n = (5, 10, 20, 25),
//     T(h) = sum_n w_n T(n h) + O((25 h)^8 g^(8)) .
// w = (114114/78125, -7904/15625, 4576/78125, -209/15625); collecting the four sums node by node gives ONE rule on the 21
// nodes j = 0, 5, ..., 100 with the positive weights below (in units of 5 h; they add up to 20).  On the reference's
// scenarios the rule reproduces the 101-node sum to 1e-15 (the remainder is 1e-20); what it needs is that the integrand
// Phi^-1 [B lambda, Sigma, xi'] is smooth across the interval, i.e. that the held input does not come near zero inside it
// -- discretize_pair_kernel checks that per interval and takes the 101 nodes otherwise.  Nothing is interpolated: the 21
// nodes are the ends of 20 Nystrom steps, whose own error at this step (5 h) is 6e-12 on 0.01-orbit intervals.
__device__ __constant__ double kEmW[21] = {
    48153.0 / 156250, 114114.0 / 78125, 35074.0 / 78125, 114114.0 / 78125, 53378.0 / 78125, 108889.0 / 78125, 35074.0 / 78125,
    114114.0 / 78125, 53378.0 / 78125,  114114.0 / 78125, 29849.0 / 78125, 114114.0 / 78125, 53378.0 / 78125, 114114.0 / 78125,
    35074.0 / 78125,  108889.0 / 78125, 53378.0 / 78125,  114114.0 / 78125, 35074.0 / 78125, 114114.0 / 78125, 48153.0 / 156250};
constexpr int kEmSteps = 20;      // integrator steps of the rule above (n_sub = 100 only)
// The same construction for intervals too long for the step 5 h (up to ~0.035 orbit: BASELINE config 5): the sums over
// every 2nd, 4th, 10th and 20th node, w = (665/512, -627/2048, 19/2560, -1/10240), one rule on the 51 even nodes = the ends
// of 50 steps (weights in units of 2 h; they add up to 50).  Half the node terms of the all-nodes path and no midpoint.
__device__ __constant__ double kEmW2[51] = {
    185.0 / 512, 665.0 / 512, 703.0 / 1024, 665.0 / 512, 703.0 / 1024, 171.0 / 128, 703.0 / 1024, 665.0 / 512, 703.0 /
    1024, 665.0 / 512, 185.0 / 256, 665.0 / 512, 703.0 / 1024, 665.0 / 512, 703.0 / 1024, 171.0 / 128, 703.0 / 1024,
    665.0 / 512, 703.0 / 1024, 665.0 / 512, 185.0 / 256, 665.0 / 512, 703.0 / 1024, 665.0 / 512, 703.0 / 1024, 171.0 /
    128, 703.0 / 1024, 665.0 / 512, 703.0 / 1024, 665.0 / 512, 185.0 / 256, 665.0 / 512, 703.0 / 1024, 665.0 / 512,
    703.0 / 1024, 171.0 / 128, 703.0 / 1024, 665.0 / 512, 703.0 / 1024, 665.0 / 512, 185.0 / 256, 665.0 / 512, 703.0 /
    1024, 665.0 / 512, 703.0 / 1024, 171.0 / 128, 703.0 / 1024, 665.0 / 512, 703.0 / 1024, 665.0 / 512, 185.0 / 512};
constexpr int kEmSteps2 = 50;
// The same construction on every 10th node, for the intervals of kEmW whose integrands are smoothest: the sums over every
// 10th, 20th, 50th and 100th node, w = (11189689/8000000, -13088691/32000000, 2089791/200000000, -110789/800000000)
// (sum w n^2r = 1, r = 0..3), one rule on the 11 nodes j = 0, 10, ..., 100 (weights in units of 10 h; they add up to 10).
// Its remainder is 1e-16 of the 101-node sum where the integrand turns by 0.07 rad across the interval (the orbital motion
// of a 0.01-orbit interval), 1e-15 at 0.25 rad and 2.5e-13 at 0.5 rad, so it is used for a smooth held input only.  The
// 11 nodes are the ends of 10 steps of Nystrom's 4-stage fifth-order method (column_step5), whose own error at the step
// 10 h is at rounding on 0.01-orbit intervals.
__device__ __constant__ double kEmW3[11] = {
    12630557.0 / 40000000, 11189689.0 / 8000000, 9290687.0 / 16000000, 11189689.0 / 8000000, 9290687.0 / 16000000,
    14509559.0 / 10000000, 9290687.0 / 16000000, 11189689.0 / 8000000, 9290687.0 / 16000000, 11189689.0 / 8000000,
    12630557.0 / 40000000};
constexpr int kEmSteps3 = 10;

// Nystrom's 4-stage fifth-order method (1925) for p'' = F(t, p), in units of the step:
//     c = (0, 1/5, 2/3, 1),  P_s = p + c_s p' + sum_j abar_sj k_j,  k_s = F(c_s, P_s),
//     abar_21 = 1/50,  abar_3 = (-1/27, 7/27),  abar_4 = (3/10, -2/35, 9/35),
//     p+ = p + p' + (14 k1 + 100 k2 + 54 k3) / 336,   p'+ = p' + (14 k1 + 125 k2 + 162 k3 + 35 k4) / 336
// One column of Phi through one step, with the stage matrices G_s (and d_s, MASSCOL) of the same scheme applied to the
// state, so that Phi stays the exact derivative of the numerical flow (as column_step).
template <bool MASSCOL>
__device__ __forceinline__ void column_step5(double (&pr)[3], double (&pv)[3], const StageLin &s1, const StageLin &s2,
                                             const StageLin &s3, const StageLin &s4)
{
    double k1[3], k2[3], k3[3], k4[3], q[3], b[3];
    if (MASSCOL) sym_mul_add(s1.g, pr[0], pr[1], pr[2], s1.dx, s1.dy, s1.dz, k1[0], k1[1], k1[2]);
    else sym_mul(s1.g, pr[0], pr[1], pr[2], k1[0], k1[1], k1[2]);
#pragma unroll
    for (int i = 0; i < 3; ++i) q[i] = fma(1.0 / 50, k1[i], fma(0.2, pv[i], pr[i]));
    if (MASSCOL) sym_mul_add(s2.g, q[0], q[1], q[2], s2.dx, s2.dy, s2.dz, k2[0], k2[1], k2[2]);
    else sym_mul(s2.g, q[0], q[1], q[2], k2[0], k2[1], k2[2]);
#pragma unroll
    for (int i = 0; i < 3; ++i) q[i] = fma(7.0 / 27, k2[i], fma(-1.0 / 27, k1[i], fma(2.0 / 3, pv[i], pr[i])));
    if (MASSCOL) sym_mul_add(s3.g, q[0], q[1], q[2], s3.dx, s3.dy, s3.dz, k3[0], k3[1], k3[2]);
    else sym_mul(s3.g, q[0], q[1], q[2], k3[0], k3[1], k3[2]);
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        b[i] = pv[i] + pr[i];
        q[i] = fma(9.0 / 35, k3[i], fma(-2.0 / 35, k2[i], fma(0.3, k1[i], b[i])));
    }
    if (MASSCOL) sym_mul_add(s4.g, q[0], q[1], q[2], s4.dx, s4.dy, s4.dz, k4[0], k4[1], k4[2]);
    else sym_mul(s4.g, q[0], q[1], q[2], k4[0], k4[1], k4[2]);
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        pr[i] = fma(9.0 / 56, k3[i], fma(25.0 / 84, k2[i], fma(1.0 / 24, k1[i], b[i])));
        pv[i] = fma(5.0 / 48, k4[i], fma(27.0 / 56, k3[i], fma(125.0 / 336, k2[i], fma(1.0 / 24, k1[i], pv[i]))));
    }
}

// Acceleration of the state at one stage: gravity at (rx, ry, rz) plus the held input over the stage's mass, and the
// stage's StageLin (d = -u/m^2).
template <bool J2>
__device__ __forceinline__ void stage_accel(const DiscParams &Ph, double rx, double ry, double rz, double ux, double uy,
                                            double uz, double mass, double &ax, double &ay, double &az, StageLin &s)
{
    gravity<J2>(Ph, rx, ry, rz, ax, ay, az, s.g);
    const double im = fast_rcp(mass);
    const double qx = ux * im, qy = uy * im, qz = uz * im;
    ax += qx;
    ay += qy;
    az += qz;
    s.dx = -qx * im;
    s.dy = -qy * im;
    s.dz = -qz * im;
}

// The state through one step of the fifth-order method above, from stage 1 (a1 = the acceleration at the step's start,
// md1 = its mass flow) -- shared by discretize_thread and discretize_group_kernel.  The held input is evaluated at the
// stage abscissae s0 + c_s ds (u at the end is returned in ue, with its guarded inverse norm); the mass is a quadrature
// of mdot(tau): the cubic through mdot at the four abscissae, integrated exactly to each c_s (to c = 1 that is the
// velocity weights b).  Returns the stage matrices of stages 2..4 for the variational columns.
template <bool J2>
__device__ __forceinline__ void state_step5(const DiscParams &Ph, const UHold<false> &hold, double s0, double ds, double eps2,
                                            double &rx, double &ry, double &rz, double &vx, double &vy, double &vz, double &m,
                                            double a1x, double a1y, double a1z, double md1, StageLin &s2, StageLin &s3,
                                            StageLin &s4, double (&ue)[3], double &uue, double &iune, int &bad)
{
    double u2[3], u3[3];
    hold.at(fma(0.2, ds, s0), 0.0, u2[0], u2[1], u2[2]);
    hold.at(fma(2.0 / 3, ds, s0), 0.0, u3[0], u3[1], u3[2]);
    hold.at(s0 + ds, 0.0, ue[0], ue[1], ue[2]);
    const double uu2 = fma(u2[0], u2[0], fma(u2[1], u2[1], u2[2] * u2[2]));
    const double uu3 = fma(u3[0], u3[0], fma(u3[1], u3[1], u3[2] * u3[2]));
    uue = fma(ue[0], ue[0], fma(ue[1], ue[1], ue[2] * ue[2]));
    iune = inv_norm_guarded(uue, eps2);
    const double md2 = -(uu2 * inv_norm_guarded(uu2, eps2)) * Ph.inv_ve;
    const double md3 = -(uu3 * inv_norm_guarded(uu3, eps2)) * Ph.inv_ve;
    const double md4 = -(uue * iune) * Ph.inv_ve;
    const double m2 = fma(17.0 / 6000, md4, fma(-81.0 / 7000, md3, fma(209.0 / 1680, md2, fma(253.0 / 3000, md1, m))));
    const double m3 = fma(-2.0 / 81, md4, fma(5.0 / 21, md3, fma(250.0 / 567, md2, fma(1.0 / 81, md1, m))));
    const double m4 = fma(5.0 / 48, md4, fma(27.0 / 56, md3, fma(125.0 / 336, md2, fma(1.0 / 24, md1, m))));
    bad |= !(m4 > 0.0);

    double a2x, a2y, a2z, a3x, a3y, a3z, a4x, a4y, a4z;
    stage_accel<J2>(Ph, fma(1.0 / 50, a1x, fma(0.2, vx, rx)), fma(1.0 / 50, a1y, fma(0.2, vy, ry)),
                    fma(1.0 / 50, a1z, fma(0.2, vz, rz)), u2[0], u2[1], u2[2], m2, a2x, a2y, a2z, s2);
    stage_accel<J2>(Ph, fma(7.0 / 27, a2x, fma(-1.0 / 27, a1x, fma(2.0 / 3, vx, rx))),
                    fma(7.0 / 27, a2y, fma(-1.0 / 27, a1y, fma(2.0 / 3, vy, ry))),
                    fma(7.0 / 27, a2z, fma(-1.0 / 27, a1z, fma(2.0 / 3, vz, rz))), u3[0], u3[1], u3[2], m3, a3x, a3y, a3z, s3);
    const double bx = vx + rx, by = vy + ry, bz = vz + rz;
    stage_accel<J2>(Ph, fma(9.0 / 35, a3x, fma(-2.0 / 35, a2x, fma(0.3, a1x, bx))),
                    fma(9.0 / 35, a3y, fma(-2.0 / 35, a2y, fma(0.3, a1y, by))),
                    fma(9.0 / 35, a3z, fma(-2.0 / 35, a2z, fma(0.3, a1z, bz))), ue[0], ue[1], ue[2], m4, a4x, a4y, a4z, s4);
    rx = fma(9.0 / 56, a3x, fma(25.0 / 84, a2x, fma(1.0 / 24, a1x, bx)));
    ry = fma(9.0 / 56, a3y, fma(25.0 / 84, a2y, fma(1.0 / 24, a1y, by)));
    rz = fma(9.0 / 56, a3z, fma(25.0 / 84, a2z, fma(1.0 / 24, a1z, bz)));
    vx = fma(5.0 / 48, a4x, fma(27.0 / 56, a3x, fma(125.0 / 336, a2x, fma(1.0 / 24, a1x, vx))));
    vy = fma(5.0 / 48, a4y, fma(27.0 / 56, a3y, fma(125.0 / 336, a2y, fma(1.0 / 24, a1y, vy))));
    vz = fma(5.0 / 48, a4z, fma(27.0 / 56, a3z, fma(125.0 / 336, a2z, fma(1.0 / 24, a1z, vz))));
    m = m4;
}

#define ACC(e) acc[(e) * BLOCK]
// EM = 1 / 2 / 3: n_sub is kEmSteps / kEmSteps2 / kEmSteps3 and node n carries the weight kEmW[n] / kEmW2[n] / kEmW3[n]
// instead of the trapezoid's 1/2, 1, ..., 1, 1/2.  EM = 3 takes the fifth-order steps (state_step5, column_step5).
template <bool J2, int BLOCK, int NDST, bool GENU, int EM = 0>
__device__ __forceinline__ void discretize_thread(const double *__restrict__ x, const double *__restrict__ u,
                                                  const double *__restrict__ tf_arr, const DiscParams &P, int K, int Ku,
                                                  int n_sub, const DstTab &dst, long long pitch, long long offset,
                                                  int32_t *__restrict__ status, long long gid, volatile double *acc)
{

    const int s = (int)(gid / (K - 1));
    const int k = (int)(gid - (long long)s * (K - 1));
    const double tf = tf_arr[s];
    const double *xs = x + ((long long)s * 7) * K + k;
    double rx = xs[0], ry = xs[K], rz = xs[2 * (long long)K];
    double vx = xs[3 * (long long)K], vy = xs[4 * (long long)K], vz = xs[5 * (long long)K];
    double m = xs[6 * (long long)K];
    UHold<GENU> hold;
    hold.init(u, s, k, K, Ku);
    const double tau0 = (double)k / (double)(K - 1), dtau_k = 1.0 / (double)(K - 1);  // interval [tau_k, tau_k+1]

    const double inv_n = 1.0 / (double)n_sub;
    const double h = inv_n / (double)(K - 1);  // step in tau
    const double hs = tf * h;                  // step of the unscaled system
    // ---- step-normalised variables ------------------------------------------------------------------
    // With D = diag(I3, hs I3, 1) the kernel carries D x (velocity times the step) and D Phi D^-1, and integrates in
    // units of the step: r' = v~, v~' = hs^2 a, m' = hs mdot.  hs^2 is folded into MU, kJ2 and the held input
    // (u~ = hs^2 u), hs into 1/(G0 ISP), so it costs nothing per step, and every Runge-Kutta coefficient becomes a
    // literal.  D Phi D^-1 is symplectic too (D^T J D = hs J), so the inverse formula is unchanged.  The
    // quadrature accumulates Phi~^-1 (D g) -- for Sigma and xi' with the common factor 1/hs taken out -- and the
    // epilogue undoes D.  Same arithmetic as before up to rounding.
    const double hs2 = hs * hs;
    DiscParams Ph;
    Ph.mu = P.mu * hs2;
    Ph.kj2 = P.kj2 * hs2;
    Ph.inv_ve = P.inv_ve / hs;                 // mdot~ = hs mdot = -|u~| / (hs G0 ISP)
    hold.scale(hs2);
    const double eps2 = 4.930380657631324e-32 * (hs2 * hs2);   // |u| <= eps  <=>  |u~|^2 <= eps^2 hs^4   (:208)
    vx *= hs;
    vy *= hs;
    vz *= hs;
    constexpr double c6 = 1.0 / 6.0;

    // Phi columns: pr[c] = rows 0..2 of column c, pv[c] = rows 3..5.  Phi(tau_k) = I   (:34)
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
    // thrust at the current node and its norm
    double ux, uy, uz;
    if (GENU) hold.at(0.0, tau0, ux, uy, uz);
    else {       // the two end nodes: as the reference looks them up; the far one waits in shared memory
        ref_node_input(u + (long long)s * 3 * K, K, k + 1, hs2, ux, uy, uz);
        ACC(kEndU) = ux;
        ACC(kEndU + 1) = uy;
        ACC(kEndU + 2) = uz;
        ref_node_input(u + (long long)s * 3 * K, K, k, hs2, ux, uy, uz);
    }
    double uu = fma(ux, ux, fma(uy, uy, uz * uz));
    double iun = inv_norm_guarded(uu, eps2);
    double un = uu * iun;

    for (int n = 0; n <= n_sub; ++n) {
        if (!GENU && n == n_sub) {                                                  // the other end node
            ux = ACC(kEndU);
            uy = ACC(kEndU + 1);
            uz = ACC(kEndU + 2);
            uu = fma(ux, ux, fma(uy, uy, uz * uz));
            iun = inv_norm_guarded(uu, eps2);
            un = uu * iun;
        }
        // ---- stage 1 == quadrature node n ------------------------------------------------------
        StageLin s1;
        double a1x, a1y, a1z;
        double gr[3];   // G r of xi' = -(Dxf x + Duf u) = -[v; G r; mdot]  (the -u/m and +u/m terms cancel, :232-235)
        gravity<J2>(Ph, rx, ry, rz, a1x, a1y, a1z, s1.g, gr);
        bad |= !(m > 0.0);
        const double im = fast_rcp(m);
        const double tx = ux * im, ty = uy * im, tz = uz * im;  // u~/m
        const double grx = gr[0], gry = gr[1], grz = gr[2];
        a1x += tx;
        a1y += ty;
        a1z += tz;
        s1.dx = -tx * im;
        s1.dy = -ty * im;
        s1.dz = -tz * im;
        const double md1 = -un * Ph.inv_ve;  // hs * mass flow (simulator.py:160)
        {
            const double sfrac = (double)n * inv_n;                     // lambda+   (:61)
            const double w = (EM == 1) ? kEmW[n] : ((EM == 2) ? kEmW2[n] : ((EM == 3) ? kEmW3[n] :
                             ((n == 0 || n == n_sub) ? 0.5 : 1.0)));   // trapezoid end weights (:77-80)
            const double ws = w * sfrac;
            // D Duf = [0; hs I/m; b^T];  hs D Sigma = [v~; a~; mdot~];  hs D xi' = -[v~; G~ r; mdot~_B]
            node_accumulate<BLOCK>(acc, pr, pv, P, im * hs, ux, uy, uz, iun, md1, vx, vy, vz, a1x, a1y, a1z, grx, gry, grz, w, ws);
        }
        if (n == n_sub) break;

        if constexpr (EM == 3 && !GENU) {
            // ---- stages 2..4 of the state and the columns: Nystrom's 4-stage fifth-order method ----------------------
            StageLin s2, s3, s4;
            double ue[3], uue, iune;
            state_step5<J2>(Ph, hold, (double)n * inv_n, inv_n, eps2, rx, ry, rz, vx, vy, vz, m, a1x, a1y, a1z, md1, s2, s3,
                            s4, ue, uue, iune, bad);
            column_step5<true>(pr[6], pv[6], s1, s2, s3, s4);
#pragma unroll
            for (int c = 0; c < 6; ++c) column_step5<false>(pr[c], pv[c], s1, s2, s3, s4);
            ux = ue[0];
            uy = ue[1];
            uz = ue[2];
            iun = iune;
            un = uue * iune;
            continue;
        }

        // ---- stages 2, 3 of the state: Nystrom's 3-stage fourth-order method for r'' = a(tau, r) ----------------
        // (the mass is a quadrature of mdot(tau): m at the half step from the quadratic through the three mdot
        //  values, m at the end by Simpson -- which is also the mass update)
        const double sm = ((double)n + 0.5) * inv_n, se = (double)(n + 1) * inv_n;
        double umx, umy, umz, uex, uey, uez;
        hold.at(sm, fma(sm, dtau_k, tau0), umx, umy, umz);
        hold.at(se, (n + 1 == n_sub && k + 2 == K) ? 1.0 : fma(se, dtau_k, tau0), uex, uey, uez);
        const double uum = fma(umx, umx, fma(umy, umy, umz * umz));
        const double uue = fma(uex, uex, fma(uey, uey, uez * uez));
        const double iunm = inv_norm_guarded(uum, eps2);
        const double iune = inv_norm_guarded(uue, eps2);
        const double mdm = -(uum * iunm) * Ph.inv_ve;
        const double mde = -(uue * iune) * Ph.inv_ve;
        const double m2 = fma(1.0 / 24.0, fma(8.0, mdm, 5.0 * md1) - mde, m);
        const double m3 = fma(c6, fma(4.0, mdm, md1) + mde, m);
        bad |= !(m3 > 0.0);

        StageLin s2, s3;
        double a2x, a2y, a2z, a3x, a3y, a3z;
        const double r2x = fma(0.125, a1x, fma(0.5, vx, rx)), r2y = fma(0.125, a1y, fma(0.5, vy, ry)),
                     r2z = fma(0.125, a1z, fma(0.5, vz, rz));
        gravity<J2>(Ph, r2x, r2y, r2z, a2x, a2y, a2z, s2.g);
        {
            const double i2 = fast_rcp(m2);
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
        // ---- state update -------------------------------------------------------------------------
        rx = fma(c6, fma(2.0, a2x, a1x), bx);
        ry = fma(c6, fma(2.0, a2y, a1y), by);
        rz = fma(c6, fma(2.0, a2z, a1z), bz);
        vx = fma(c6, fma(4.0, a2x, a1x) + a3x, vx);
        vy = fma(c6, fma(4.0, a2y, a1y) + a3y, vy);
        vz = fma(c6, fma(4.0, a2z, a1z) + a3z, vz);
        m = m3;
        // ---- variational columns ----------------------------------------------------------------
        // the mass column first: its forcing terms d1..d3 are dead for the remaining six columns
        column_step<true>(pr[6], pv[6], s1, s2, s3);
#pragma unroll
        for (int c = 0; c < 6; ++c) column_step<false>(pr[c], pv[c], s1, s2, s3);
        ux = uex;
        uy = uey;
        uz = uez;
        iun = iune;
        un = uue * iune;
    }

    // ---- epilogue: left-multiply by Phi_end, undo D, scale by the step, store SoA -----------------
    // B and xi carry tf (scale tf h = hs), Sigma does not (h); the accumulated Sigma and xi vectors carry the factor hs
    const double ihs = 1.0 / hs;
    const int nonfinite = epilogue_store<BLOCK, NDST>(acc, pr, pv, hs, h * ihs, 1.0, dst, pitch, out_col(dst, offset, s, k, K), hs, ihs);
    if (status) status[gid] = bad ? 1 : (nonfinite ? 2 : 0);
}
#undef ACC

template <bool J2, int BLOCK, int MAXREG, int NDST, bool GENU>
__global__ void __launch_bounds__(BLOCK) __maxnreg__(MAXREG)
discretize_kernel(const double *__restrict__ x, const double *__restrict__ u, const double *__restrict__ tf_arr,
                  DiscParams P, int n_sats, int K, int Ku, int n_sub, DstTab dst, long long pitch, long long offset,
                  int32_t *__restrict__ status)
{
    extern __shared__ double acc_smem[];
    const long long n_int = (long long)n_sats * (K - 1);
    const long long gid = (long long)blockIdx.x * BLOCK + threadIdx.x;
    if (gid >= n_int) return;
    if (dst.stagger_phases > 1 && (int)blockIdx.x < dst.first_wave_ctas) {
        const long long wait = dst.stagger_cycles * (long long)(blockIdx.x % dst.stagger_phases) / dst.stagger_phases;
        const long long t0 = clock64();
        while (clock64() - t0 < wait) __nanosleep(2000);
    }
    // volatile: keep the accumulators IN shared memory (the compiler would otherwise promote these
    // thread-private slots to registers and spill them to local memory, which is write-through to L2)
    discretize_thread<J2, BLOCK, NDST, GENU>(x, u, tf_arr, P, K, Ku, n_sub, dst, pitch, offset, status, gid,
                                             acc_smem + threadIdx.x);
}

}  // namespace mpc
