// TEST INFRASTRUCTURE ONLY -- the ragged forms (RAG = true) of constraint_terms_kernel and dynamics_jacobian_kernel in
// the host build, on top of the wrappers of hostk_main.cpp.  Built by tests/test_handoff_ragged_on_host.py next to
// libmpc_hostk.so; the threads of a launch run one after the other.
#include "hostk_main.cpp"

// first [n_sats+1]: prefix sums of K_s - 1; x [n_sats][7][K_max], u [n_sats][3][K_max]
extern "C" int hostk_constraint_terms_ragged(const double *x, const double *u, int n_sats, int K_max, const long long *first,
                                             double mu, double *rbar_hat, double *ubar_hat, double *fin)
{
    run_grid(first[n_sats] - first[0], [&] {
        mpc::constraint_terms_kernel<true>(x, u, n_sats, K_max, K_max, mu, 2.220446049250313e-16, rbar_hat, ubar_hat, fin, first);
    });
    return 0;
}

// soa: the ragged discretization result, satellite s at columns offset + s (K_max-1) + k
extern "C" int hostk_dynamics_jacobian_ragged(const double *soa, long long pitch, long long offset, int n_sats, int K_max,
                                              const long long *first, double *values, int64_t *indices, double *rhs)
{
    run_grid(first[n_sats] - first[0],
             [&] { mpc::dynamics_jacobian_kernel<true>(soa, pitch, offset, n_sats, K_max, values, indices, rhs, first); });
    return 0;
}
