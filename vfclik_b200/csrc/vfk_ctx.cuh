// vfk_ctx.cuh -- the handle behind vfk_handle, shared by the translation units of libvfk.so.
#pragma once
#include <cuda_runtime.h>

#include <cstdarg>
#include <cstdio>
#include <string>

#include "../../include/vfk.h"
#include "vfk_kernels.cuh"

// Direct host I/O request of the host-buffer session (see KArgs::q_src): dense [N][ld] arrays in mapped page-locked host
// memory that the cycle kernel reads q from / writes qdot to instead of the blocked device buffers.
struct vfk_io {
    const void* q_src = nullptr;
    int64_t q_src_ld = 0;
    void* qdot = nullptr;
    int64_t qdot_ld = 0;
};

// Stop rule and result buffers of vfk_solve, handed to the SOLVE instantiations of the cycle kernel.
struct vfk_solve_io {
    double tol_trans, tol_rot;  // metres, radians (>= pi: orientation not checked)
    int32_t* cycles;            // [1] blocked
    void* dist;                 // [2] blocked, or null
};

struct vfk_ctx {
    vfk_chain_desc chain;       // as given
    vfk_chain_desc canon;       // every joint about / along Z
    vfk_params params;
    int precision;
    int device;
    int sm_count;
    int pattern;                // 0: GenericPattern, 1: LwrPattern, 2: DhPattern (structure of the canonical chain)
    int dh_chain;               // all joints revolute, all tip rotations RotX(alpha): what DhPattern and the lane-split kernel take
    int n_kernel;               // joint count of the instantiation that runs this chain: the smallest of 6, 7, 10, 17 that is
                                // >= n_joints (shorter chains run padded: KArgs::n_comp)
    uint64_t generation;        // bumped by vfk_set_params: captured CUDA graphs bake the constants in
    vfk::KConst<float> cf;
    vfk::KConst<double> cd;
    std::string err;
};

inline thread_local std::string g_create_err;

inline int fail(vfk_ctx* h, int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    if (h) h->err = buf; else g_create_err = buf;
    return code;
}

#define VFK_CUDA(h, call)                                                                   \
    do {                                                                                    \
        cudaError_t e_ = (call);                                                            \
        if (e_ != cudaSuccess)                                                              \
            return fail((h), VFK_ERR_CUDA, "%s failed: %s", #call, cudaGetErrorString(e_)); \
    } while (0)


// One obstacle list of a scene (m = 0: empty).
struct vfk_obst_list {
    const void* obst;          // own list: blocked pairs (vfk.h); shared list: dense [m][4]
    const void* obst_ext;      // own list: blocked [m][2]; shared list: dense [m][2]; or null
    int m;
};

// The scene of a call, resolved once from vfk_buffers by the ABI layer (resolve_scene in vfk_api.cu): the instances' own
// lists, which run through the obstacle ring, and the list shared by the whole batch, which the SHARED kernels stage into
// shared memory.  Mode 0 has only own lists, mode 1 only the shared list, mode 2 both.
struct vfk_scene {
    vfk_obst_list own, shared;
};

// One cycle-kernel call, from the ABI down to the launch.
struct CycleCall {
    const vfk_buffers* b;
    int64_t n;
    int k_cycles;               // vfk_solve: max_cycles
    cudaStream_t stream;
    const vfk_io* io;           // direct host I/O of a session, or null
    const vfk_solve_io* sv;     // vfk_solve's stop rule and results; null for a step
    vfk_scene scene;
};

// Cycle-kernel launchers, one translation unit each so they compile in parallel: the step kernels per (precision, joint-count
// group), and per precision the vfk_solve kernels and the SHARED step and solve kernels (a non-empty shared list).
int vfk_launch_f32_small(vfk_ctx* h, const CycleCall& call);   // N = 6, 7
int vfk_launch_f32_large(vfk_ctx* h, const CycleCall& call);   // N = 10, 17
int vfk_launch_f64_small(vfk_ctx* h, const CycleCall& call);
int vfk_launch_f64_large(vfk_ctx* h, const CycleCall& call);
int vfk_solve_f32(vfk_ctx* h, const CycleCall& call);
int vfk_solve_f64(vfk_ctx* h, const CycleCall& call);
int vfk_launch_shared_f32(vfk_ctx* h, const CycleCall& call);
int vfk_launch_shared_f64(vfk_ctx* h, const CycleCall& call);
int vfk_solve_shared_f32(vfk_ctx* h, const CycleCall& call);
int vfk_solve_shared_f64(vfk_ctx* h, const CycleCall& call);
