// cmpc_body.cu - the BODY solve kernels (solve_rows<true, false, false>): the same template arguments as the plain
// kernels, reading each problem's mass and inverse inertia from its slot (cmpc_set_body).  A translation unit of its
// own so that the kernels of cmpc.cu compile exactly as they do without these (see solve_rows in cmpc_launch.cuh).
#define CMPC_SOLVE_KERNELS_ONLY   // the other kernels of cmpc_kernels.cuh are defined in cmpc.cu
#include "cmpc_launch.cuh"

namespace cmpc {

template const SolveRow* solve_rows<true, false, false>();

}  // namespace cmpc
