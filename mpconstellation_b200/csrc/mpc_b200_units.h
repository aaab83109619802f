// mpc_b200_units.h -- interface between mpc_b200.cu and mpc_b200_units.cu (the translation unit of the per-satellite-
// constants kernels, PSC = true).  The launch policy (block size, validation, the constants tables) stays in mpc_b200.cu.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

struct MpcUnitsDisc {
    const double *x, *u, *tf;
    const void *psc;           // device mpc::DiscParams [n_sats]
    const void *dst_tab;       // mpc::DstTab (em set by the caller)
    const long long *first;    // ragged batch: device prefix sums of K_s - 1; NULL: rectangular
    long long n_units;         // threads: live intervals (ragged) or n_sats (K-1)
    int include_j2, n_sats, K, n_sub;
    int adaptive, block;       // adaptive: the default-mode kernel (CTA 32 / 128 / 256), else the pair kernel (32 / 128)
    double rtol, atol, max_step;
    long long pitch, offset;
    int32_t *status, *n_nodes;
    cudaStream_t stream;
};

struct MpcUnitsProp {
    const double *y0, *tf;
    const void *psc;           // device mpc::PropParams [n_sats]
    const void *ctrl;          // mpc::CtrlParams
    const void *opts;          // mpc::Rk45Opts
    int kind, include_drag, include_j2;
    int n_sats, T, lpw;
    unsigned n_warps;
    double *y, *u_out;
    int32_t *status, *n_steps;
    const int32_t *T_sat, *ku;  // device, may be NULL (all T / all table_len)
    cudaStream_t stream;
    const void *prop;          // mpc::PropParams of a launch without per-satellite constants (mpc_b200_atmo.cu only)
};

size_t mpc_units_sizeof(int which);   // 0 DiscParams, 1 DstTab, 2 PropParams, 3 CtrlParams, 4 Rk45Opts
cudaError_t mpc_units_launch_disc(const MpcUnitsDisc *a);
cudaError_t mpc_units_launch_rk45(const MpcUnitsProp *a);
// x [n_sats][7][K], u [n_sats][3][K]; first == NULL: rectangular (n_units = n_sats K threads), else ragged (live intervals)
cudaError_t mpc_units_launch_cterms(const double *x, const double *u, int n_sats, int K, long long n_units,
                                    const long long *first, const double *mu_sat, double *rbar, double *ubar, double *fin,
                                    cudaStream_t stream);
