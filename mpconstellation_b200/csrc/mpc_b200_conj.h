// mpc_b200_conj.h -- interface between mpc_b200.cu and mpc_b200_conj.cu (the translation unit of the conjunction
// screening kernels, conjunction_kernel.cuh).  The argument checks and the derivation of the scale table stay in
// mpc_b200.cu.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

struct MpcConjLaunch {
    const double *y;           // device [n_sats][7][T], normalized
    double *scratch;           // device, mpc_conj_scratch_doubles(n_sats, T): X, S, then the scale table [n_sats][2]
    const double *scale_host;  // host [n_sats][2] = (R0_s, R0_s / s0_s), copied to the tail of scratch
    int n_sats, T;
    double h, threshold;       // sample spacing (s), threshold (m)
    void *events;              // device mpc::ConjRecord [capacity]
    long long capacity;
    unsigned long long *counters;   // device [2]: events found, events flagged
    int32_t *skipped;          // device [n_sats]
    cudaStream_t stream;
};

long long mpc_conj_scratch_doubles(int n_sats, int T);
size_t mpc_conj_record_size();   // sizeof(mpc::ConjRecord)
// counters and skipped zeroed, the pre-pass, the pair kernel: 2 launches
cudaError_t mpc_conj_launch(const MpcConjLaunch *a);
