// mpc_b200_atmo.cu -- the RK45 replay with drag under an altitude-dependent atmosphere (propagate_rk45_atmo_kernel) in
// its OWN translation unit, for the reason the drag, units and shard kernels have theirs: ptxas's register allocation of
// the hot kernels depends on what else the module holds, and the kernels of mpc_b200.cu keep the code generation they
// were measured with.  As there, the kernel headers are included under another namespace name and the interface to
// mpc_b200.cu is plain C (mpc_b200_atmo.h).
#include <cuda_runtime.h>
#include <math_constants.h>
#include <stdint.h>

#define mpc mpc_atmotu
#include "propagate_kernel.cuh"
#include "propagate_rk45_kernel.cuh"
#include "mpc_b200_atmo.h"

namespace {

// One set of 16 kernels (law x J2 x per-satellite constants): a rectangular batch is the ragged form without counts
// (T_sat = Ku_sat = NULL), the same steps and samples as a rectangular run.
template <int KIND, bool J2, bool PSC>
void rk45(const MpcUnitsProp &a, const mpc::AtmoParams &A)
{
    mpc::propagate_rk45_atmo_kernel<KIND, J2, PSC><<<a.n_warps, 32, 0, a.stream>>>(
        a.y0, a.tf, *(const mpc::PropParams *)a.prop, *(const mpc::CtrlParams *)a.ctrl, *(const mpc::Rk45Opts *)a.opts,
        a.n_sats, a.T, a.lpw, a.y, a.u_out, a.status, a.n_steps, a.T_sat, a.ku, A, (const mpc::AtmoSat *)a.psc);
}

template <int KIND>
void rk45_k(const MpcUnitsProp &a, const mpc::AtmoParams &A)
{
    if (a.psc) {
        if (a.include_j2) rk45<KIND, true, true>(a, A);
        else rk45<KIND, false, true>(a, A);
    } else {
        if (a.include_j2) rk45<KIND, true, false>(a, A);
        else rk45<KIND, false, false>(a, A);
    }
}

}  // namespace

size_t mpc_atmo_sizeof(int which)
{
    switch (which) {
        case 0: return sizeof(mpc::PropParams);
        case 1: return sizeof(mpc::CtrlParams);
        case 2: return sizeof(mpc::Rk45Opts);
        case 3: return sizeof(mpc::AtmoParams);
        default: return sizeof(mpc::AtmoSat);
    }
}

cudaError_t mpc_atmo_launch_rk45(const MpcUnitsProp *a, const void *atmo)
{
    const mpc::AtmoParams &A = *(const mpc::AtmoParams *)atmo;
    switch (a->kind) {
        case 0: rk45_k<0>(*a, A); break;
        case 1: rk45_k<1>(*a, A); break;
        case 2: rk45_k<2>(*a, A); break;
        default: rk45_k<3>(*a, A); break;
    }
    return cudaGetLastError();
}
