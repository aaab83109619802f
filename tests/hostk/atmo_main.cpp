// TEST INFRASTRUCTURE ONLY -- the RK45 replay under an altitude-dependent atmosphere (propagate_rk45_atmo_kernel, one
// constants bag or per-satellite constants, rectangular or ragged) of the host build, on top of the wrappers of
// hostk_main.cpp.  Built by tests/test_atmosphere_kernel_source_on_host.py next to libmpc_hostk.so; the threads of a
// launch run one after the other.  The kernel constants are derived as mpc_b200.cu derives them (atmo_prop_params,
// atmo_sat, atmo_params).
#include <cmath>
#include <vector>

#include "hostk_main.cpp"

namespace {

// const8: MU, R_E, J2, G0, ISP, S, R0, RHO (tests/hostk/__init__.py _const8)
mpc::PropParams atmo_prop(const double *c, int include_j2, double c_d)
{
    mpc::PropParams P;
    P.mu = c[0];
    P.kj2 = 1.5 * c[2] * c[0] * c[1] * c[1];
    P.inv_ve = 1.0 / (c[3] * c[4]);
    P.drag_k = 0.5 * c_d * c[5] / c[7];
    P.include_j2 = include_j2;
    P.include_drag = 1;
    return P;
}

}  // namespace

// atmo: h_min, h_max, r_earth, n, coef[n] (doubles).  psc = 0: one bag const8 [8]; 1: const8 [n_sats][8].
// table [n_sats][3][table_len] (kind 3) with ku [n_sats] columns each (may be NULL); T_sat NULL: every lane on T_max samples.
extern "C" int hostk_propagate_rk45_atmo(const double *y0, const double *tf, const double *const8, int psc, int include_j2,
                                         double c_d, int kind, const double *thrust, const double *table, int table_len,
                                         const int32_t *ku, double end_tau, int n_sats, int T_max, const int32_t *T_sat,
                                         const double *atmo, int lpw, double *y, double *u_out, int32_t *status,
                                         int32_t *n_steps)
{
    mpc::AtmoParams A{};
    A.h_min = atmo[0];
    A.h_max = atmo[1];
    A.r_earth = atmo[2];
    A.n = (int)atmo[3];
    for (int k = 0; k < A.n; ++k) A.coef[k] = atmo[4 + k];
    const double lo = std::log(A.h_min), hi = std::log(A.h_max);
    A.s_mid = 0.5 * (lo + hi);
    A.s_ihalf = 2.0 / (hi - lo);
    A.len = A.r_earth / const8[1];
    const mpc::PropParams P = atmo_prop(const8, include_j2, c_d);
    std::vector<mpc::AtmoSat> sat(psc ? (size_t)n_sats : 0);
    for (size_t s = 0; s < sat.size(); ++s) {
        sat[s].P = atmo_prop(const8 + 8 * s, include_j2, c_d);
        sat[s].len = A.r_earth / const8[8 * s + 1];
    }
    mpc::CtrlParams C{};
    C.kind = kind;
    C.t0 = thrust[0];
    C.t1 = thrust[1];
    C.t2 = thrust[2];
    C.end_tau = end_tau;
    C.table_len = table_len;
    C.table_per_sat = 1;
    C.table = kind == 3 ? table : nullptr;
    const mpc::Rk45Opts O{1e-3, 1e-6, 1e-3};
    const long long n_threads = (long long)((n_sats + lpw - 1) / lpw) * 32;
#define HK_A45(KIND, J2, PSC)                                                                                                \
    run_grid(n_threads, [&] {                                                                                                \
        mpc::propagate_rk45_atmo_kernel<KIND, J2, PSC>(y0, tf, P, C, O, n_sats, T_max, lpw, y, u_out, status, n_steps, T_sat, \
                                                       kind == 3 ? ku : nullptr, A, sat.data());                              \
    })
#define HK_A45_K(KIND)                                          \
    do {                                                        \
        if (psc) {                                              \
            if (include_j2) HK_A45(KIND, true, true);           \
            else HK_A45(KIND, false, true);                     \
        } else {                                                \
            if (include_j2) HK_A45(KIND, true, false);          \
            else HK_A45(KIND, false, false);                    \
        }                                                       \
    } while (0)
    switch (kind) {
        case 0: HK_A45_K(0); break;
        case 1: HK_A45_K(1); break;
        case 2: HK_A45_K(2); break;
        default: HK_A45_K(3); break;
    }
#undef HK_A45_K
#undef HK_A45
    return 0;
}
