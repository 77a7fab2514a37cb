// Instantiates the shared-scene variants of vfk_solve (SOLVE = true, SHARED = true) of the fused cycle kernel for double, every
// joint count (own translation unit: compiles in parallel with the other kernels).
#include "vfk_launch.cuh"

int vfk_solve_shared_f64(vfk_ctx* h, const CycleCall& call) { return launch_family<double, true, true, 6, 7, 10, 17>(h, call); }
