// mpc_b200_units.cu -- the per-satellite-constants instantiations (PSC = true) in their OWN translation unit.
//
// Each satellite of a constellation that mixes altitudes and masses is linearized in the designer units of its own
// SatelliteScale (its own MU, R_E, 1/(G0 ISP), S, RHO), as N separate controllers of the reference would do.  The kernels
// are the production ones with a template flag (or an entry of their own) that makes thread -> satellite s read its
// constants from a device table [n_sats] instead of the launch-wide parameter.  They live here for the reason the drag kernels live in
// mpc_b200_drag.cu: ptxas's register allocation of the 254-register hot kernels depends on what else the module holds,
// and the kernels of mpc_b200.cu keep the code generation they were measured with.  As there, the kernel headers are
// included under another namespace name (their __constant__ tables would otherwise be defined twice in the library) and
// the interface to mpc_b200.cu is plain C.
#include <cuda_runtime.h>
#include <math_constants.h>
#include <stdint.h>

#define mpc mpc_unitstu
#include "discretize_kernel.cuh"
#include "discretize_adaptive_kernel.cuh"
#include "discretize_default_kernel.cuh"
#include "discretize_pair_kernel.cuh"
#include "propagate_kernel.cuh"
#include "propagate_rk45_kernel.cuh"
#include "constraint_terms_kernel.cuh"
#include "mpc_b200_units.h"

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

// ragged only: a rectangular batch comes as one with equal counts (launch_units_disc in mpc_b200.cu)
template <bool J2, int BLOCK>
cudaError_t pair(const MpcUnitsDisc &a)
{
    auto kern = mpc::discretize_pair_kernel<J2, BLOCK, 255, 1, true, true>;
    const size_t smem = (size_t)(mpc::kDiscSlots + 1) * BLOCK * sizeof(double);   // + the slot of 1/(G0 ISP)
    static thread_local int configured_dev = -1;
    cudaError_t e = configure(kern, smem, configured_dev);
    if (e != cudaSuccess) return e;
    const unsigned grid = (unsigned)((a.n_units + BLOCK - 1) / BLOCK);
    const mpc::DiscParams *psc = (const mpc::DiscParams *)a.psc;
    // (the launch-wide P is not read: every thread takes psc[s])
    kern<<<grid, BLOCK, smem, a.stream>>>(a.x, a.u, a.tf, mpc::DiscParams{}, a.n_sats, a.K, a.n_sub,
                                          *(const mpc::DstTab *)a.dst_tab, a.pitch, a.offset, a.status, 0, a.K - 1, a.first, psc);
    return cudaGetLastError();
}

template <bool J2, int BLOCK, bool RAG>
cudaError_t dflt(const MpcUnitsDisc &a)
{
    auto kern = mpc::discretize_default_units_kernel<J2, BLOCK, RAG>;
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

template <bool J2, bool RAG>
cudaError_t disc(const MpcUnitsDisc &a)
{
    if (a.adaptive) {
        if (a.block == 256) return dflt<J2, 256, RAG>(a);
        if (a.block == 128) return dflt<J2, 128, RAG>(a);
        return dflt<J2, 32, RAG>(a);
    }
    if constexpr (RAG) return a.block == 32 ? pair<J2, 32>(a) : pair<J2, 128>(a);
    else return cudaErrorInvalidValue;
}

// The rectangular propagation is the ragged form without counts (T_sat = Ku_sat = NULL: every lane samples all T columns
// of its whole table), the same steps and samples as a rectangular run: one set of 16 kernels, not two.  The speculative
// first stage is always on (it changes the schedule, not the result; mpc_set_tuning(11) is an A/B knob of the
// single-constant kernels).
template <int KIND, bool DRAG, bool J2>
void rk45(const MpcUnitsProp &a)
{
    constexpr int BLOCK = 32;
    // (the table of per-satellite constants goes in the place of the progress words, see the kernel)
    mpc::propagate_rk45_kernel<BLOCK, KIND, DRAG, J2, true, true, true><<<a.n_warps, BLOCK, 0, a.stream>>>(
        a.y0, a.tf, mpc::PropParams{}, *(const mpc::CtrlParams *)a.ctrl, *(const mpc::Rk45Opts *)a.opts, a.n_sats, a.T, a.lpw,
        a.y, a.u_out, a.status, a.n_steps, (unsigned int *)a.psc, 0, a.T_sat, a.ku);
}

template <int KIND>
void rk45_k(const MpcUnitsProp &a)
{
    if (a.include_drag) {
        if (a.include_j2) rk45<KIND, true, true>(a);
        else rk45<KIND, true, false>(a);
    } else {
        if (a.include_j2) rk45<KIND, false, true>(a);
        else rk45<KIND, false, false>(a);
    }
}

}  // namespace

size_t mpc_units_sizeof(int which)
{
    switch (which) {
        case 0: return sizeof(mpc::DiscParams);
        case 1: return sizeof(mpc::DstTab);
        case 2: return sizeof(mpc::PropParams);
        case 3: return sizeof(mpc::CtrlParams);
        default: return sizeof(mpc::Rk45Opts);
    }
}

cudaError_t mpc_units_launch_disc(const MpcUnitsDisc *a)
{
    if (a->first) return a->include_j2 ? disc<true, true>(*a) : disc<false, true>(*a);
    return a->include_j2 ? disc<true, false>(*a) : disc<false, false>(*a);
}

cudaError_t mpc_units_launch_rk45(const MpcUnitsProp *a)
{
    switch (a->kind) {
        case 0: rk45_k<0>(*a); break;
        case 1: rk45_k<1>(*a); break;
        case 2: rk45_k<2>(*a); break;
        default: rk45_k<3>(*a); break;
    }
    return cudaGetLastError();
}

cudaError_t mpc_units_launch_cterms(const double *x, const double *u, int n_sats, int K, long long n_units,
                                    const long long *first, const double *mu_sat, double *rbar, double *ubar, double *fin,
                                    cudaStream_t stream)
{
    const unsigned grid = (unsigned)((n_units + 255) / 256);
    if (first)
        mpc::constraint_terms_units_kernel<true><<<grid, 256, 0, stream>>>(x, u, n_sats, K, mu_sat, 2.220446049250313e-16, rbar,
                                                                          ubar, fin, first);
    else
        mpc::constraint_terms_units_kernel<false><<<grid, 256, 0, stream>>>(x, u, n_sats, K, mu_sat, 2.220446049250313e-16, rbar,
                                                                           ubar, fin, nullptr);
    return cudaGetLastError();
}
