// cmpc_body.cu - the BODY twins of every solve kernel cmpc.cu launches: the same template arguments, reading
// each problem's mass and inverse inertia from its slot (cmpc_set_body).  A translation unit of its own so
// that the kernels of cmpc.cu compile exactly as they do without the twins (see cmpc_launch.cuh).
#define CMPC_SOLVE_KERNELS_ONLY   // the other kernels of cmpc_kernels.cuh are defined in cmpc.cu
#include "cmpc_launch.cuh"

namespace cmpc {

// one entry per row of kHorizons (cmpc.cu), same kernels with BODY = true
const BodyTwins kBodyTwins[] = {
    {4, launch_solve<4, 1, 8, 1, false, false, false, true>, nullptr, nullptr},
    {5, launch_solve<5, 1, 8, 1, false, false, false, true>, nullptr, nullptr},
    {8, launch_solve<8, 1, 8, 1, false, false, false, true>, nullptr, nullptr},
    {10, launch_solve<10, 1, 6, 1, false, true, true, true>, launch_solve_riccati<10, 8, true>,
     launch_solve<10, 1, 6, 1, true, true, true, true>},
    {12, launch_solve<12, 2, 4, 1, false, false, false, true>, launch_solve_riccati<12, 8, true>, nullptr},
    {16, launch_solve<16, 2, 3, 1, false, false, false, true>, launch_solve_riccati<16, 8, true>, nullptr},
    {20, launch_solve_riccati<20, 6, true>, launch_solve<20, 2, 2, 1, false, false, false, true>, nullptr},
    {30, launch_solve_riccati<30, 4, true>, launch_solve<30, 6, 1, 3, false, false, false, true>,
     launch_solve<30, 6, 1, 3, true, false, false, true>},
    {40, launch_solve_riccati<40, 3, true>, nullptr, nullptr},
    {60, launch_solve_riccati<60, 2, true>, nullptr, nullptr},
};
const int kBodyTwinCount = sizeof kBodyTwins / sizeof kBodyTwins[0];

}  // namespace cmpc
