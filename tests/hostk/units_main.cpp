// TEST INFRASTRUCTURE ONLY -- the per-satellite-constants kernels (discretize_pair_kernel / propagate_rk45_kernel with
// PSC = true, discretize_default_units_kernel, constraint_terms_units_kernel; rectangular and ragged) of the host
// build, on top of the wrappers of hostk_main.cpp.  Built by tests/test_units_kernel_source_on_host.py next to
// libmpc_hostk.so; the threads of a launch run one after the other.
#include <vector>

#include "hostk_main.cpp"

// const8_sat [n_sats][8]: satellite s's constants in the order of const8.  first [n_sats+1] (prefix sums of K_s - 1) or
// NULL: a rectangular batch.  adaptive = 0: the fixed-step pair kernel (em as hostk_discretize), 1: the default-mode kernel.
extern "C" int hostk_discretize_units(const double *x, const double *u, const double *tf, const double *const8_sat,
                                      int include_j2, int n_sats, int K, const long long *first, int adaptive, int n_sub,
                                      double rtol, double atol, double max_step, double *out, long long pitch,
                                      int32_t *status, int32_t *n_nodes, int em)
{
    std::vector<mpc::DiscParams> psc((size_t)n_sats);
    for (int s = 0; s < n_sats; ++s) psc[s] = disc_params(const8_sat + 8 * s, include_j2);
    mpc::DstTab dst{};
    dst.p[0] = out;
    dst.em = em;
    const long long n = first ? first[n_sats] - first[0] : (long long)n_sats * (K - 1);
    const mpc::DiscParams *t = psc.data();
    std::vector<long long> eq((size_t)n_sats + 1);
    for (int s = 0; s <= n_sats; ++s) eq[s] = (long long)s * (K - 1);
    run_grid(n, [&] {
        if (adaptive) {
            if (first) {
                if (include_j2) mpc::discretize_default_units_kernel<true, kBlock, true>(x, u, tf, t, n_sats, K, rtol, atol, max_step, dst, pitch, 0, status, n_nodes, first);
                else mpc::discretize_default_units_kernel<false, kBlock, true>(x, u, tf, t, n_sats, K, rtol, atol, max_step, dst, pitch, 0, status, n_nodes, first);
            } else {
                if (include_j2) mpc::discretize_default_units_kernel<true, kBlock, false>(x, u, tf, t, n_sats, K, rtol, atol, max_step, dst, pitch, 0, status, n_nodes, nullptr);
                else mpc::discretize_default_units_kernel<false, kBlock, false>(x, u, tf, t, n_sats, K, rtol, atol, max_step, dst, pitch, 0, status, n_nodes, nullptr);
            }
        } else {
            // (ragged only, as in the library: a rectangular batch runs with equal counts)
            const mpc::DiscParams none{};
            const long long *f = first ? first : eq.data();
            if (include_j2) mpc::discretize_pair_kernel<true, kBlock, 255, 1, true, true>(x, u, tf, none, n_sats, K, n_sub, dst, pitch, 0, status, 0, K - 1, f, t);
            else mpc::discretize_pair_kernel<false, kBlock, 255, 1, true, true>(x, u, tf, none, n_sats, K, n_sub, dst, pitch, 0, status, 0, K - 1, f, t);
        }
    });
    return 0;
}

// the RK45 replay with per-lane constants: tangential law (kind 2) or a per-satellite sequence table [n_sats][3][table_len]
// with ku [n_sats] columns each (kind 3, ku may be NULL); T_sat NULL: every lane on T_max samples (the rectangular run)
extern "C" int hostk_propagate_rk45_units(const double *y0, const double *tf, const double *const8_sat, int include_j2, int kind,
                                          double thrust, const double *table, int table_len, const int32_t *ku, int n_sats,
                                          int T_max, const int32_t *T_sat, double *y, double *u_out, int32_t *status,
                                          int32_t *n_steps)
{
    std::vector<mpc::PropParams> psc((size_t)n_sats);
    for (int s = 0; s < n_sats; ++s) {
        const double *c = const8_sat + 8 * s;
        psc[s].mu = c[0];
        psc[s].kj2 = 1.5 * c[2] * c[0] * c[1] * c[1];
        psc[s].inv_ve = 1.0 / (c[3] * c[4]);
        psc[s].drag_k = 0.0;
        psc[s].include_j2 = include_j2;
        psc[s].include_drag = 0;
    }
    mpc::CtrlParams C{};
    C.kind = kind;
    C.t0 = thrust;
    C.end_tau = 1.0;
    C.table_len = table_len;
    C.table_per_sat = 1;
    C.table = kind == 3 ? table : nullptr;
    const mpc::Rk45Opts O{1e-3, 1e-6, 1e-3};
    run_grid(n_sats, [&] {
#define HK_U45(KIND, J2) \
    mpc::propagate_rk45_kernel<kBlock, KIND, false, J2, true, true, true>(y0, tf, mpc::PropParams{}, C, O, n_sats, T_max, 32, y, u_out, status, n_steps, (unsigned int *)psc.data(), 0, T_sat, ku)
        if (kind == 3) {
            if (include_j2) HK_U45(3, true);
            else HK_U45(3, false);
        } else {
            if (include_j2) HK_U45(2, true);
            else HK_U45(2, false);
        }
#undef HK_U45
    });
    return 0;
}

// first == NULL: rectangular (u on the nodes of x); mu_sat [n_sats]
extern "C" int hostk_constraint_terms_units(const double *x, const double *u, int n_sats, int K, const long long *first,
                                            const double *mu_sat, double *rbar_hat, double *ubar_hat, double *fin)
{
    const long long n = first ? first[n_sats] - first[0] : (long long)n_sats * K;
    run_grid(n, [&] {
        if (first) mpc::constraint_terms_units_kernel<true>(x, u, n_sats, K, mu_sat, 2.220446049250313e-16, rbar_hat, ubar_hat, fin, first);
        else mpc::constraint_terms_units_kernel<false>(x, u, n_sats, K, mu_sat, 2.220446049250313e-16, rbar_hat, ubar_hat, fin, nullptr);
    });
    return 0;
}
