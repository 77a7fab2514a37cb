// Instantiates the shared-scene variants (SHARED = true, vfk_buffers.obst_shared) of the fused cycle kernel's step for double,
// every joint count (own translation unit: compiles in parallel with the per-instance kernels).
#include "vfk_launch.cuh"

int vfk_launch_shared_f64(vfk_ctx* h, const vfk_buffers* b, int64_t n, int n_obst, const vfk_shared_scene* sh, int k_cycles, cudaStream_t st,
                          const vfk_io* io) {
    const KConst<double>& c = h->cd;
    switch (h->n_kernel) {
        case 6: return dispatch_ext<double, 6, false, true>(h, c, b, n, n_obst, k_cycles, st, io, nullptr, sh);
        case 7: return dispatch_ext<double, 7, false, true>(h, c, b, n, n_obst, k_cycles, st, io, nullptr, sh);
        case 10: return dispatch_ext<double, 10, false, true>(h, c, b, n, n_obst, k_cycles, st, io, nullptr, sh);
        case 17: return dispatch_ext<double, 17, false, true>(h, c, b, n, n_obst, k_cycles, st, io, nullptr, sh);
    }
    return fail(h, VFK_ERR_UNSUPPORTED, "no kernel for n_joints = %d", h->chain.n_joints);
}
