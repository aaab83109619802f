// mpc_b200_shard.h -- interface between mpc_b200.cu and mpc_b200_shard.cu (the translation unit of the multi-destination
// ragged discretization kernels: one rank's shard of a ragged batch stored into every rank's gathered buffer).  The
// launch policy (block size, validation, the constants table, the prefix sums) stays in mpc_b200.cu.
#pragma once
#include "mpc_b200_units.h"

// a: a ragged launch (a->first != NULL) as mpc_units_launch_disc takes it; a->psc == NULL: one constants bag, *P (an
// mpc::DiscParams).  n_dst: 2, 4 or 8 destinations in the DstTab.  Default mode: CTA 32 or 256; fixed step: 32 or 128.
cudaError_t mpc_shard_launch_disc(const MpcUnitsDisc *a, const void *P, int n_dst);
