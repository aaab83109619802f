// mpc_b200_atmo.h -- interface between mpc_b200.cu and mpc_b200_atmo.cu (the translation unit of the RK45 replay under an
// altitude-dependent atmosphere).  The launch policy (validation, lanes per warp, the constants tables) stays in mpc_b200.cu.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>

#include "mpc_b200_units.h"

size_t mpc_atmo_sizeof(int which);   // 0 PropParams, 1 CtrlParams, 2 Rk45Opts, 3 AtmoParams, 4 AtmoSat
// a->prop: the launch-wide mpc::PropParams; a->psc: device mpc::AtmoSat [n_sats] or NULL (one constants bag);
// atmo: mpc::AtmoParams (passed to the kernel by value); include_drag is implied
cudaError_t mpc_atmo_launch_rk45(const MpcUnitsProp *a, const void *atmo);
