// Instantiates the fused cycle kernel for double, N in {6, 7} (own translation unit: compiles in parallel).
#include "vfk_launch.cuh"

int vfk_launch_f64_small(vfk_ctx* h, const CycleCall& call) { return launch_family<double, false, false, 6, 7>(h, call); }
