// Instantiates the shared-scene variants of vfk_solve (SOLVE = true, SHARED = true) of the fused cycle kernel for double, every
// joint count (own translation unit: compiles in parallel with the other kernels).
#include "vfk_launch.cuh"

int vfk_solve_shared_f64(vfk_ctx* h, const vfk_buffers* b, int64_t n, int n_obst, const vfk_shared_scene* sh, int max_cycles, cudaStream_t st,
                         const vfk_solve_io* sv) {
    const KConst<double>& c = h->cd;
    switch (h->n_kernel) {
        case 6: return dispatch_ext<double, 6, true, true>(h, c, b, n, n_obst, max_cycles, st, nullptr, sv, sh);
        case 7: return dispatch_ext<double, 7, true, true>(h, c, b, n, n_obst, max_cycles, st, nullptr, sv, sh);
        case 10: return dispatch_ext<double, 10, true, true>(h, c, b, n, n_obst, max_cycles, st, nullptr, sv, sh);
        case 17: return dispatch_ext<double, 17, true, true>(h, c, b, n, n_obst, max_cycles, st, nullptr, sv, sh);
    }
    return fail(h, VFK_ERR_UNSUPPORTED, "no kernel for n_joints = %d", h->chain.n_joints);
}
