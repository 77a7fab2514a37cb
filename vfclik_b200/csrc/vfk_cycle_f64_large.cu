// Instantiates the fused cycle kernel for double, N in {10, 17} (own translation unit: compiles in parallel).
#include "vfk_launch.cuh"

int vfk_launch_f64_large(vfk_ctx* h, const CycleCall& call) { return launch_family<double, false, false, 10, 17>(h, call); }
