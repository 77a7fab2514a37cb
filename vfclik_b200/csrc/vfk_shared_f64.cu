// Instantiates the shared-scene variants (SHARED = true, vfk_buffers.obst_shared) of the fused cycle kernel's step for double,
// every joint count (own translation unit: compiles in parallel with the per-instance kernels).
#include "vfk_launch.cuh"

int vfk_launch_shared_f64(vfk_ctx* h, const CycleCall& call) { return launch_family<double, false, true, 6, 7, 10, 17>(h, call); }
