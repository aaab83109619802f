// TEST INFRASTRUCTURE ONLY -- the multi-destination ragged kernels (discretize_pair_kernel with NDST = 2, RAG = true,
// PSC = false / true; discretize_default_ragged_multi_kernel / discretize_default_units_multi_kernel with NDST = 2) of
// the host build, on top of the wrappers of hostk_main.cpp: one rank's shard of a sharded batch stored into two gathered
// buffers.  Built by tests/test_shard_kernel_source_on_host.py next to libmpc_hostk.so; the threads of a launch run one
// after the other.
#include <vector>

#include "hostk_main.cpp"

// const8_sat [n_sats][8]: satellite s's constants in the order of const8; psc = 0: every satellite runs with row 0 as the
// launch-wide constants.  first [n_sats+1]: the shard's own prefix sums of K_s - 1.  Results go to columns
// offset + s (K - 1) + k of out0 AND out1 (skip_const as DstTab::skip_const).  adaptive = 0: the fixed-step pair kernel
// (em as hostk_discretize), 1: the default-mode kernel.
extern "C" int hostk_discretize_shard(const double *x, const double *u, const double *tf, const double *const8_sat, int psc,
                                      int include_j2, int n_sats, int K, const long long *first, int adaptive, int n_sub,
                                      double rtol, double atol, double max_step, double *out0, double *out1, long long pitch,
                                      long long offset, int skip_const, int32_t *status, int32_t *n_nodes, int em)
{
    std::vector<mpc::DiscParams> tab((size_t)n_sats);
    for (int s = 0; s < n_sats; ++s) tab[s] = disc_params(const8_sat + (psc ? 8 * s : 0), include_j2);
    const mpc::DiscParams P = tab.empty() ? mpc::DiscParams{} : tab[0];
    mpc::DstTab dst{};
    dst.p[0] = out0;
    dst.p[1] = out1;
    dst.skip_const = skip_const;
    dst.em = em;
    const mpc::DiscParams *t = tab.data();
    run_grid(first[n_sats] - first[0], [&] {
#define HK_SHARD(J2)                                                                                                                  \
    if (adaptive && psc)                                                                                                              \
        mpc::discretize_default_units_multi_kernel<J2, kBlock, 2>(x, u, tf, t, n_sats, K, rtol, atol, max_step, dst, pitch, offset,   \
                                                                  status, n_nodes, first);                                            \
    else if (adaptive)                                                                                                                \
        mpc::discretize_default_ragged_multi_kernel<J2, kBlock, 2>(x, u, tf, P, n_sats, K, rtol, atol, max_step, dst, pitch, offset,  \
                                                                   status, n_nodes, first);                                           \
    else if (psc)                                                                                                                     \
        mpc::discretize_pair_kernel<J2, kBlock, 255, 2, true, true>(x, u, tf, mpc::DiscParams{}, n_sats, K, n_sub, dst, pitch,        \
                                                                    offset, status, 0, K - 1, first, t);                              \
    else                                                                                                                              \
        mpc::discretize_pair_kernel<J2, kBlock, 255, 2, true, false>(x, u, tf, P, n_sats, K, n_sub, dst, pitch, offset, status, 0,   \
                                                                     K - 1, first, nullptr)
        if (include_j2) HK_SHARD(true);
        else HK_SHARD(false);
#undef HK_SHARD
    });
    return 0;
}
