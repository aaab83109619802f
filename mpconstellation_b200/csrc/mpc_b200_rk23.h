// mpc_b200_rk23.h -- interface between mpc_b200.cu and mpc_b200_rk23.cu (the translation unit of the default quadrature
// mode with scipy's RK23, discretize_rk23_kernel.cuh).  The launch policy (validation, block size, the constants tables)
// stays in mpc_b200.cu.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

struct MpcRk23Disc {
    const double *x, *u, *tf;
    const void *P;             // host mpc::DiscParams of a launch without per-satellite constants (passed by value)
    const void *psc;           // device mpc::DiscParams [n_sats], or NULL: one constants bag (P)
    const long long *first;    // ragged batch: device prefix sums of K_s - 1; NULL: rectangular
    long long n_units;         // threads: live intervals (ragged) or n_sats (K-1)
    int include_j2, n_sats, K;
    int block;                 // 32 or 256 threads per CTA
    double rtol, atol, max_step;
    double *out;
    long long pitch, offset;
    int32_t *status, *n_nodes;
    cudaStream_t stream;
};

size_t mpc_rk23_sizeof();      // sizeof(mpc::DiscParams)
cudaError_t mpc_rk23_launch_disc(const MpcRk23Disc *a);
