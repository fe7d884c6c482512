// The TRAJ instantiations of mppi_mlp_rollout_kernel (the trajectory viewers' replays), compiled apart from the tick's
// instantiations (see mlp_traj_kernels in mppi_mlp.cu).
#define MPPI_MLP_TRAJ_UNIT
#include "mppi_mlp.cu"
