// mpc_b200_conj.cu -- the conjunction screening kernels (conjunction_kernel.cuh) in their OWN translation unit, for the
// reason the drag, units, shard, atmosphere and RK23 kernels have theirs: ptxas's register allocation of the hot kernels
// depends on what else the module holds, and the kernels of the other units keep the code generation they were measured
// with.  As there, the kernel header is included under another namespace name and the interface to mpc_b200.cu is plain
// C (mpc_b200_conj.h).
#include <cuda_runtime.h>
#include <stdint.h>

#define mpc mpc_conjtu
#include "conjunction_kernel.cuh"
#include "mpc_b200_conj.h"

namespace {
constexpr int kPrepassBlock = 128;
}

long long mpc_conj_scratch_doubles(int n_sats, int T)
{
    return (long long)n_sats * (6LL * T + 4LL * (T - 1) + 2);
}

size_t mpc_conj_record_size() { return sizeof(mpc::ConjRecord); }

cudaError_t mpc_conj_launch(const MpcConjLaunch *a)
{
    const long long n = a->n_sats;
    double *X = a->scratch, *S = X + n * 6 * a->T, *scale = S + n * 4 * (a->T - 1);
    cudaError_t e = cudaMemcpyAsync(scale, a->scale_host, (size_t)n * 2 * sizeof(double), cudaMemcpyHostToDevice, a->stream);
    if (e != cudaSuccess) return e;
    if ((e = cudaMemsetAsync(a->counters, 0, 2 * sizeof(unsigned long long), a->stream)) != cudaSuccess) return e;
    if ((e = cudaMemsetAsync(a->skipped, 0, (size_t)n * sizeof(int32_t), a->stream)) != cudaSuccess) return e;
    const long long n_thr = n * a->T;
    mpc::conj_prepass_kernel<kPrepassBlock><<<(unsigned)((n_thr + kPrepassBlock - 1) / kPrepassBlock), kPrepassBlock, 0, a->stream>>>(
        a->y, scale, a->n_sats, a->T, a->h, X, S, a->skipped);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    const unsigned nb = (unsigned)((n + mpc::kConjTile - 1) / mpc::kConjTile);
    mpc::conj_pair_kernel<<<dim3(nb, nb), mpc::kConjThreads, 0, a->stream>>>(
        X, S, a->n_sats, a->T, a->h, a->threshold, (mpc::ConjRecord *)a->events, a->capacity, a->counters);
    return cudaGetLastError();
}
