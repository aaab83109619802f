// mpc_b200_rk23.cu -- the default quadrature mode with scipy's RK23 (discretize_rk23_kernel) in its OWN translation unit,
// for the reason the drag, units, shard and atmosphere kernels have theirs: ptxas's register allocation of the hot
// kernels depends on what else the module holds, and the kernels of mpc_b200.cu keep the code generation they were
// measured with.  As there, the kernel headers are included under another namespace name and the interface to
// mpc_b200.cu is plain C (mpc_b200_rk23.h).
#include <cuda_runtime.h>
#include <math_constants.h>
#include <stdint.h>

#define mpc mpc_rk23tu
#include "discretize_rk23_kernel.cuh"
#include "mpc_b200_rk23.h"

namespace {

// One set of 16 kernels: J2 x BLOCK (32 / 256) x ragged x per-satellite constants.
template <bool J2, int BLOCK, bool RAG, bool PSC>
cudaError_t rk23(const MpcRk23Disc &a)
{
    auto kern = mpc::discretize_rk23_kernel<J2, BLOCK, RAG, PSC>;
    const size_t smem = (size_t)mpc::kRkSlots * BLOCK * sizeof(double);
    static thread_local int configured_dev = -1;
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    if (configured_dev != dev) {
        e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        e = cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
        if (e != cudaSuccess) return e;
        configured_dev = dev;
    }
    const unsigned grid = (unsigned)((a.n_units + BLOCK - 1) / BLOCK);
    // (with PSC the launch-wide P is not read: every thread takes psc[s])
    const mpc::DiscParams P = PSC ? mpc::DiscParams{} : *(const mpc::DiscParams *)a.P;
    kern<<<grid, BLOCK, smem, a.stream>>>(a.x, a.u, a.tf, P, (const mpc::DiscParams *)a.psc, a.n_sats, a.K, a.rtol, a.atol,
                                          a.max_step, a.out, a.pitch, a.offset, a.status, a.n_nodes, a.first);
    return cudaGetLastError();
}

template <bool J2, bool RAG, bool PSC>
cudaError_t rk23_b(const MpcRk23Disc &a)
{
    return a.block == 32 ? rk23<J2, 32, RAG, PSC>(a) : rk23<J2, 256, RAG, PSC>(a);
}

template <bool J2>
cudaError_t rk23_j(const MpcRk23Disc &a)
{
    if (a.first) return a.psc ? rk23_b<J2, true, true>(a) : rk23_b<J2, true, false>(a);
    return a.psc ? rk23_b<J2, false, true>(a) : rk23_b<J2, false, false>(a);
}

}  // namespace

size_t mpc_rk23_sizeof() { return sizeof(mpc::DiscParams); }

cudaError_t mpc_rk23_launch_disc(const MpcRk23Disc *a)
{
    return a->include_j2 ? rk23_j<true>(*a) : rk23_j<false>(*a);
}
