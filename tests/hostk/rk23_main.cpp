// TEST INFRASTRUCTURE ONLY -- the default quadrature mode with scipy's RK23 (discretize_rk23_kernel: one constants bag or
// per-satellite constants, rectangular or ragged) of the host build, on top of the wrappers of hostk_main.cpp.  Built by
// tests/test_rk23_kernel_source_on_host.py next to libmpc_hostk.so; the threads of a launch run one after the other.
#include <vector>

#include "hostk_main.cpp"
#include "discretize_rk23_kernel.cuh"

// psc = 0: const8 [8], one bag; 1: const8 [n_sats][8].  first [n_sats+1] (prefix sums of K_s - 1) or NULL: rectangular.
extern "C" int hostk_discretize_rk23(const double *x, const double *u, const double *tf, const double *const8, int psc,
                                     int include_j2, int n_sats, int K, const long long *first, double rtol, double atol,
                                     double max_step, double *out, long long pitch, int32_t *status, int32_t *n_nodes)
{
    std::vector<mpc::DiscParams> tab(psc ? (size_t)n_sats : 0);
    for (size_t s = 0; s < tab.size(); ++s) tab[s] = disc_params(const8 + 8 * s, include_j2);
    const mpc::DiscParams P = psc ? mpc::DiscParams{} : disc_params(const8, include_j2);
    const mpc::DiscParams *t = psc ? tab.data() : nullptr;
    const long long n = first ? first[n_sats] - first[0] : (long long)n_sats * (K - 1);
#define HK_R23(J2, RAG, PSC) \
    mpc::discretize_rk23_kernel<J2, kBlock, RAG, PSC>(x, u, tf, P, t, n_sats, K, rtol, atol, max_step, out, pitch, 0, status, n_nodes, first)
#define HK_R23_J(RAG, PSC)              \
    do {                                \
        if (include_j2) HK_R23(true, RAG, PSC); \
        else HK_R23(false, RAG, PSC);   \
    } while (0)
    run_grid(n, [&] {
        if (first) {
            if (psc) HK_R23_J(true, true);
            else HK_R23_J(true, false);
        } else {
            if (psc) HK_R23_J(false, true);
            else HK_R23_J(false, false);
        }
    });
#undef HK_R23_J
#undef HK_R23
    return 0;
}

// the controller's x^(-1/3) (inv_cube_root) at n points
extern "C" void hostk_inv_cube_root(const double *x, int n, double *y)
{
    for (int i = 0; i < n; ++i) y[i] = mpc::inv_cube_root(x[i]);
}
