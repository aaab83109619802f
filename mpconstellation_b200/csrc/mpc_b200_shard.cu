// mpc_b200_shard.cu -- the multi-destination (NDST = 2, 4, 8) instantiations of the ragged discretization kernels, with
// and without per-satellite constants, in their OWN translation unit.
//
// A rank of a sharded constellation discretizes its satellites and stores every result into every rank's gathered buffer
// (mpc_discretize_batch_ragged_gather).  The kernels are the ragged ones of the single-GPU path with NDST > 1.  They live
// here for the reason the per-satellite-constants kernels live in mpc_b200_units.cu: ptxas's register allocation of the
// 254-register hot kernels depends on what else the module holds, and the kernels of mpc_b200.cu and mpc_b200_units.cu
// keep the code generation they were measured with.  As there, the kernel headers are included under another namespace
// name and the interface to mpc_b200.cu is plain C.
#include <cuda_runtime.h>
#include <math_constants.h>
#include <stdint.h>

#define mpc mpc_shardtu
#include "discretize_kernel.cuh"
#include "discretize_adaptive_kernel.cuh"
#include "discretize_default_kernel.cuh"
#include "discretize_pair_kernel.cuh"
#include "mpc_b200_shard.h"

namespace {

template <typename Kern>
cudaError_t configure(Kern kern, size_t smem, int &configured_dev)
{
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
    return cudaSuccess;
}

template <bool J2, int BLOCK, int NDST, bool PSC>
cudaError_t pair(const MpcUnitsDisc &a, const mpc::DiscParams &P)
{
    auto kern = mpc::discretize_pair_kernel<J2, BLOCK, 255, NDST, true, PSC>;
    const size_t smem = (size_t)(mpc::kDiscSlots + (PSC ? 1 : 0)) * BLOCK * sizeof(double);   // PSC: + the slot of 1/(G0 ISP)
    static thread_local int configured_dev = -1;
    cudaError_t e = configure(kern, smem, configured_dev);
    if (e != cudaSuccess) return e;
    const unsigned grid = (unsigned)((a.n_units + BLOCK - 1) / BLOCK);
    kern<<<grid, BLOCK, smem, a.stream>>>(a.x, a.u, a.tf, P, a.n_sats, a.K, a.n_sub, *(const mpc::DstTab *)a.dst_tab, a.pitch,
                                          a.offset, a.status, 0, a.K - 1, a.first, (const mpc::DiscParams *)a.psc);
    return cudaGetLastError();
}

template <bool J2, int BLOCK, int NDST>
cudaError_t dflt_one(const MpcUnitsDisc &a, const mpc::DiscParams &P)
{
    auto kern = mpc::discretize_default_ragged_multi_kernel<J2, BLOCK, NDST>;
    const size_t smem = (size_t)mpc::kDfSlots * BLOCK * sizeof(double);
    static thread_local int configured_dev = -1;
    cudaError_t e = configure(kern, smem, configured_dev);
    if (e != cudaSuccess) return e;
    const unsigned grid = (unsigned)((a.n_units + BLOCK - 1) / BLOCK);
    kern<<<grid, BLOCK, smem, a.stream>>>(a.x, a.u, a.tf, P, a.n_sats, a.K, a.rtol, a.atol, a.max_step,
                                          *(const mpc::DstTab *)a.dst_tab, a.pitch, a.offset, a.status, a.n_nodes, a.first);
    return cudaGetLastError();
}

template <bool J2, int BLOCK, int NDST>
cudaError_t dflt_units(const MpcUnitsDisc &a)
{
    auto kern = mpc::discretize_default_units_multi_kernel<J2, BLOCK, NDST>;
    const size_t smem = (size_t)mpc::kDfSlots * BLOCK * sizeof(double);
    static thread_local int configured_dev = -1;
    cudaError_t e = configure(kern, smem, configured_dev);
    if (e != cudaSuccess) return e;
    const unsigned grid = (unsigned)((a.n_units + BLOCK - 1) / BLOCK);
    kern<<<grid, BLOCK, smem, a.stream>>>(a.x, a.u, a.tf, (const mpc::DiscParams *)a.psc, a.n_sats, a.K, a.rtol, a.atol,
                                          a.max_step, *(const mpc::DstTab *)a.dst_tab, a.pitch, a.offset, a.status, a.n_nodes,
                                          a.first);
    return cudaGetLastError();
}

template <int NDST, bool J2>
cudaError_t disc(const MpcUnitsDisc &a, const mpc::DiscParams &P)
{
    if (a.adaptive) {
        if (a.block == 32) return a.psc ? dflt_units<J2, 32, NDST>(a) : dflt_one<J2, 32, NDST>(a, P);
        return a.psc ? dflt_units<J2, 256, NDST>(a) : dflt_one<J2, 256, NDST>(a, P);
    }
    if (a.block == 32) return a.psc ? pair<J2, 32, NDST, true>(a, P) : pair<J2, 32, NDST, false>(a, P);
    return a.psc ? pair<J2, 128, NDST, true>(a, P) : pair<J2, 128, NDST, false>(a, P);
}

template <int NDST>
cudaError_t disc_n(const MpcUnitsDisc &a, const mpc::DiscParams &P)
{
    return a.include_j2 ? disc<NDST, true>(a, P) : disc<NDST, false>(a, P);
}

}  // namespace

cudaError_t mpc_shard_launch_disc(const MpcUnitsDisc *a, const void *P, int n_dst)
{
    if (!a->first) return cudaErrorInvalidValue;
    const mpc::DiscParams &p = *(const mpc::DiscParams *)P;
    switch (n_dst) {
        case 2: return disc_n<2>(*a, p);
        case 4: return disc_n<4>(*a, p);
        case 8: return disc_n<8>(*a, p);
        default: return cudaErrorInvalidValue;
    }
}
