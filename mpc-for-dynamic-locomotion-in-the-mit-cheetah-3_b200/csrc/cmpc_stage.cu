// cmpc_stage.cu - per-robot stage weights (cmpc_set_stage_weights): the BODY + WEIGHTS + FORCE + STAGE and
// BODY + CONTACT + WEIGHTS + FORCE + STAGE solve kernels (solve_rows<true, false, true, true, true> and
// <true, true, true, true, true>).  The kernels that store the weights are those of cmpc_set_weights
// (cmpc_weights.cu).  A translation unit of its own so that the kernels of the other modules compile exactly as they
// do without these (see solve_rows in cmpc_launch.cuh).
#define CMPC_SOLVE_KERNELS_ONLY   // the other kernels of cmpc_kernels.cuh are defined in cmpc.cu
#include "cmpc_launch.cuh"

namespace cmpc {

template const SolveRow* solve_rows<true, false, true, true, true>();
template const SolveRow* solve_rows<true, true, true, true, true>();

}  // namespace cmpc
