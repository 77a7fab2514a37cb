// Instantiates the fused cycle kernel for float, N in {6, 7} (own translation unit: compiles in parallel).
#include "vfk_launch.cuh"

int vfk_launch_f32_small(vfk_ctx* h, const CycleCall& call) { return launch_family<float, false, false, 6, 7>(h, call); }
