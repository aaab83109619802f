// TEST INFRASTRUCTURE ONLY -- the ragged-batch kernels (discretize_pair_kernel / propagate_rk45_kernel with RAG = true,
// discretize_default_ragged_kernel) of the host build, on top of the wrappers of hostk_main.cpp.  Built by
// tests/test_ragged_kernel_source_on_host.py next to libmpc_hostk.so; the threads of a launch run one after the other.
#include "hostk_main.cpp"

// first [n_sats+1]: prefix sums of K_s - 1; the launch covers first[n_sats] - first[0] live intervals.  adaptive = 0: the
// fixed-step pair kernel (em as hostk_discretize), 1: the default-mode kernel.
extern "C" int hostk_discretize_ragged(const double *x, const double *u, const double *tf, const double *const8, int include_j2,
                                       int n_sats, int K_max, const long long *first, int adaptive, int n_sub, double rtol,
                                       double atol, double max_step, double *out, long long pitch, int32_t *status,
                                       int32_t *n_nodes, int em)
{
    const mpc::DiscParams P = disc_params(const8, include_j2);
    mpc::DstTab dst{};
    dst.p[0] = out;
    dst.em = em;
    const long long n_live = first[n_sats] - first[0];
    run_grid(n_live, [&] {
        if (adaptive) {
            if (include_j2)
                mpc::discretize_default_ragged_kernel<true, kBlock>(x, u, tf, P, n_sats, K_max, rtol, atol, max_step, dst, pitch, 0, status, n_nodes, first);
            else
                mpc::discretize_default_ragged_kernel<false, kBlock>(x, u, tf, P, n_sats, K_max, rtol, atol, max_step, dst, pitch, 0, status, n_nodes, first);
        } else {
            if (include_j2) mpc::discretize_pair_kernel<true, kBlock, 255, 1, true>(x, u, tf, P, n_sats, K_max, n_sub, dst, pitch, 0, status, 0, K_max - 1, first);
            else mpc::discretize_pair_kernel<false, kBlock, 255, 1, true>(x, u, tf, P, n_sats, K_max, n_sub, dst, pitch, 0, status, 0, K_max - 1, first);
        }
    });
    return 0;
}

// tangential law (kind 2) or a per-satellite sequence table [n_sats][3][table_len] with ku [n_sats] columns each (kind 3)
extern "C" int hostk_propagate_rk45_ragged(const double *y0, const double *tf, const double *const8, int kind, double thrust,
                                           const double *table, int table_len, const int32_t *ku, int n_sats, int T_max,
                                           const int32_t *T_sat, double *y, double *u_out, int32_t *status, int32_t *n_steps)
{
    mpc::PropParams PP;
    PP.mu = const8[0];
    PP.kj2 = 1.5 * const8[2] * const8[0] * const8[1] * const8[1];
    PP.inv_ve = 1.0 / (const8[3] * const8[4]);
    PP.drag_k = 0.0;
    PP.include_j2 = 0;
    PP.include_drag = 0;
    mpc::CtrlParams C{};
    C.kind = kind;
    C.t0 = thrust;
    C.end_tau = 1.0;
    C.table_len = table_len;
    C.table_per_sat = 1;
    C.table = kind == 3 ? table : nullptr;
    const mpc::Rk45Opts O{1e-3, 1e-6, 1e-3};
    run_grid(n_sats, [&] {
        if (kind == 3)
            mpc::propagate_rk45_kernel<kBlock, 3, false, false, true, true>(y0, tf, PP, C, O, n_sats, T_max, 32, y, u_out, status, n_steps, nullptr, 0, T_sat, ku);
        else
            mpc::propagate_rk45_kernel<kBlock, 2, false, false, true, true>(y0, tf, PP, C, O, n_sats, T_max, 32, y, u_out, status, n_steps, nullptr, 0, T_sat, nullptr);
    });
    return 0;
}
