// Instantiates the vfk_solve variants (SOLVE = true) of the fused cycle kernel for double, every joint count (own
// translation unit: compiles in parallel with the step kernels).
#include "vfk_launch.cuh"

int vfk_solve_f64(vfk_ctx* h, const CycleCall& call) { return launch_family<double, true, false, 6, 7, 10, 17>(h, call); }
