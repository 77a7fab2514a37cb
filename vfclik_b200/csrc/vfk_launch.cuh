// vfk_launch.cuh -- launch plan and feature dispatch of the fused cycle kernel (included by the ten launcher units).
#pragma once
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <mutex>

#include "vfk_ctx.cuh"
#include "vfk_split.cuh"

using namespace vfk;

// Launch plan: every warp is a persistent worker with its own obstacle ring (n_stages stages of kChunk
// obstacles x 32 instances) and two q/goal buffers.  Two stages measured best on B200 for both K = 1
// (106 us vs 110 us with three at the headline shape) and K = 100 (streaming the ring from L2 every cycle at
// full occupancy beats keeping four chunks resident at 2 CTAs/SM): gpurun_out t03, DESIGN.md section 4.1.
// Long FP32 chains run 2 CTAs per SM on registers, so a third stage is free: config 5 0.684 -> 0.708 of the HBM roofline
// (4: 0.697; 6 and 8 cost a resident CTA: 0.44); everywhere else a third stage costs occupancy (config 4: 1.009 -> 0.988).
template <typename T, int N>
constexpr int kRingStages = (sizeof(T) == 4 && N >= 10) ? 3 : 2;

// Launch plan of one kernel instantiation: resident CTAs per SM for a given dynamic shared-memory size, per device.  One
// instance per instantiation (function-local static at the call site); a handful of (device, smem) entries behind a mutex, so
// concurrent host threads and sessions with different obstacle counts neither race nor evict one another.
struct PlanCache {
    std::mutex mu;
    struct Entry { int device; size_t smem; int per_sm; } e[16];
    int used = 0;
    template <typename K>
    cudaError_t get(K kern, int device, size_t smem, int* per_sm) {
        std::lock_guard<std::mutex> lock(mu);
        for (int i = 0; i < used; ++i)
            if (e[i].device == device && e[i].smem == smem) { *per_sm = e[i].per_sm; return cudaSuccess; }
        cudaError_t err = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 << 10);
        if (err == cudaSuccess) err = cudaOccupancyMaxActiveBlocksPerMultiprocessor(per_sm, kern, kBlock, smem);
        if (err != cudaSuccess) return err;
        const int slot = used < 16 ? used++ : 15;
        e[slot] = Entry{device, smem, *per_sm};
        return cudaSuccess;
    }
};

constexpr int64_t kCoopMaxInstances = 4096;      // <= 128 tiles: 1024 cooperative warps instead of 128 solo ones

template <typename T>
static const KConst<T>& kconst(const vfk_ctx* h) {
    if constexpr (sizeof(T) == 4) return h->cf; else return h->cd;
}

// Chunk plan of a list of m obstacles, as KArgs holds it for the own list and for the shared list.
static ChunkPlan chunk_plan(int m) {
    return ChunkPlan{m, (m + 1) & ~1, (m + kChunk - 1) / kChunk, m / kChunk, m % kChunk};
}

// The launch of every cycle-kernel shape: `units` warp-sized work units, each warp a persistent worker, so at most as many
// CTAs as fit the SMs at once.  One plan cache per kernel instantiation: opt in to > 48 KB of dynamic shared memory and ask
// the occupancy once per (device, smem size).
template <auto kern, typename... Args>
static int launch_persistent(vfk_ctx* h, int64_t units, size_t smem, cudaStream_t st, const Args&... args) {
    static PlanCache plans;
    int per_sm = 0;
    VFK_CUDA(h, plans.get(kern, h->device, smem, &per_sm));
    if (per_sm < 1) return fail(h, VFK_ERR_CUDA, "kernel does not fit an SM with %zu bytes of shared memory", smem);
    const int64_t want = (units + kBlock / 32 - 1) / (kBlock / 32);
    const int64_t cap = (int64_t)h->sm_count * per_sm;
    kern<<<(unsigned)(want < cap ? want : cap), kBlock, smem, st>>>(args...);
    VFK_CUDA(h, cudaGetLastError());
    return 1;
}

// The LEAN kernel's preconditions (see vfk_kernels.cuh): on the constants and inputs (all a solve has to meet, since it
// has no per-cycle outputs), and for a step also on the outputs.
template <typename T>
static bool lean_inputs(const KConst<T>& c, const vfk_buffers* b) {
    return c.tool_identity && c.unit_weights && c.share_factor && c.ik_mode == 0 && c.ns_mode == VFK_NS_PROJECTOR && !c.need_jp && !b->ns_in &&
           !c.shoulder_clamp &&
           !b->jp_ref && !b->jp_lo && !b->q_cmded && !b->ext_cmd[0] && !b->ext_cmd[1] && !b->ext_cmd[2] && !(b->aux && b->n_aux > 0);
}

template <typename T>
static bool is_lean(const KConst<T>& c, const vfk_buffers* b) {
    return lean_inputs<T>(c, b) && !b->qdot_vf && !b->qdot_ns && !b->qdot_jp && !b->cmd && !b->pose && !b->twist && !b->flags && b->qdot;
}

// HIOCC: the single-cycle lean FP32 launch asks for one more resident CTA per SM (4 x 128 threads at 128 registers, no
// spills).  Measured on B200, 1 M instances: 109.5 us vs 111.2 us per launch at K = 1 (more warps hide more HBM latency),
// but 1.6 % slower at K = 100, where the kernel is issue-bound and the tighter register budget costs instructions.
// SOLVE: the vfk_solve variant (vfk_kernels.cuh), with its stop rule and result buffers in `call.sv`.
// SHARED: the scene's shared list, staged into shared memory per CTA; the own list (a mixed scene; empty in a shared-only
// call) runs through the ring as usual.
template <typename T, int N, class PAT, bool EXT, bool LEAN, int G = 1, bool HIOCC = false, bool SOLVE = false, bool SHARED = false>
static int launch_cycle(vfk_ctx* h, const CycleCall& call) {
    const vfk_buffers* b = call.b;
    const vfk_scene& sc = call.scene;
    const vfk_io* io = call.io;
    KArgs<T> a;
    memset(&a, 0, sizeof a);
    a.q = static_cast<T*>(b->q);
    a.goal = static_cast<const T*>(b->goal);
    a.obst = static_cast<const Vec4<T>*>(sc.own.obst);
    a.obst_ext = static_cast<const Vec2<T>*>(sc.own.obst_ext);
    a.aux = b->n_aux > 0 ? static_cast<const T*>(b->aux) : nullptr;
    a.n_aux = a.aux ? b->n_aux : 0;
    a.jp_ref = static_cast<T*>(b->jp_ref);
    a.jp_lo = static_cast<const T*>(b->jp_lo);
    a.jp_hi = static_cast<const T*>(b->jp_hi);
    a.ns_in = static_cast<const T*>(b->ns_in);
    a.ns_lastvec = static_cast<T*>(b->ns_lastvec);
    a.q_cmded = static_cast<const T*>(b->q_cmded);
    for (int e = 0; e < 3; ++e) a.ext_cmd[e] = static_cast<const T*>(b->ext_cmd[e]);
    a.qdot_vf = static_cast<T*>(b->qdot_vf);
    a.qdot_ns = static_cast<T*>(b->qdot_ns);
    a.qdot_jp = static_cast<T*>(b->qdot_jp);
    a.qdot = static_cast<T*>(b->qdot);
    a.cmd = static_cast<T*>(b->cmd);
    a.pose = static_cast<T*>(b->pose);
    a.twist = static_cast<T*>(b->twist);
    a.flags = b->flags;
    if (io && io->q_src) { a.q_src = static_cast<const T*>(io->q_src); a.q_src_ld = io->q_src_ld; }
    if (io && io->qdot) { a.qdot = static_cast<T*>(io->qdot); a.qdot_ld = io->qdot_ld; a.qdot_dev = static_cast<T*>(b->qdot); }
    a.n = call.n;
    a.n_comp = h->chain.n_joints;
    a.k_cycles = call.k_cycles;
    if constexpr (SOLVE) {
        // thresholds in T: |dp|^2 against tol_trans^2, and |xyz|^2 = sin^2(angle / 2) of the error quaternion against
        // sin^2(tol_rot / 2) -- exact and monotone on [0, pi], no transcendental in the kernel
        const vfk_solve_io* sv = call.sv;
        a.tol_d2 = (T)(sv->tol_trans * sv->tol_trans);
        const double sh_rot = std::sin(0.5 * sv->tol_rot);
        a.tol_q2 = sv->tol_rot >= 3.14159265358979323846 ? (T)INFINITY : (T)(sh_rot * sh_rot);
        a.cycles = sv->cycles;
        a.dist = static_cast<T*>(sv->dist);
    }
    a.own = chunk_plan(sc.own.m);
    a.n_stages = a.own.chunks < kRingStages<T, N> ? a.own.chunks : kRingStages<T, N>;
    size_t smem = kSmemHeader + kTabBytes<T> + (size_t)(kBlock / 32) * WarpStage<T, N, EXT>::warp_bytes(a.n_stages);
    if constexpr (SHARED) {
        // Shared memory: the own ring (its usual plan on the own count; no stages without one), the staged shared list and
        // the q / goal buffers.  Every instantiation fits an SM with an own list at the largest stage count and a shared
        // list at the cap: FP64 + EXT with 17 joints takes 204.5 KiB there (one CTA per SM, as its MINB asks).
        static_assert(kSmemHeader + kTabBytes<T> + shared_scene_bytes<T, EXT>(VFK_MAX_SHARED_OBSTACLES, VFK_MAX_SHARED_OBSTACLES) +
                          (kBlock / 32) * WarpStage<T, N, EXT>::warp_bytes(kRingStages<T, N>) <= (227u << 10),
                      "a mixed scene at the shared-list cap does not fit an SM");
        a.sh_obst = static_cast<const T*>(sc.shared.obst);
        a.sh_obst_ext = static_cast<const T*>(sc.shared.obst_ext);
        a.sh = chunk_plan(sc.shared.m);
        smem += shared_scene_bytes<T, EXT>(a.sh.np, a.sh.n);
    }
    // resident CTAs per SM that the register allocation aims for.  The shared-scene FP32 lean solve kernels of N <= 7 ask for
    // four: at three the LWR one took 130 registers where its per-instance twin takes 128, one resident CTA fewer (at four it
    // takes 127 without spilling; the 7-joint generic one spills 24 bytes, as its HIOCC step twin does)
    constexpr int MINB = (HIOCC || (SHARED && SOLVE && LEAN && sizeof(T) == 4 && N <= 7)) ? 4
                         : (sizeof(T) == 4 ? (N <= 10 ? 3 : 2) : (N <= 7 ? 2 : 1));
    // G = 8: a tile is spread over 8 warps (4 instances each)
    return launch_persistent<vfk_cycle_kernel<T, N, PAT, EXT, LEAN, MINB, G, SOLVE, SHARED>>(h, (call.n + 31) / 32 * G, smem, call.stream,
                                                                                           kconst<T>(h), a);
}

// ------------------------------------------------------------------------------ lane-split shape (vfk_split.cuh)
typedef CUresult (*vfk_encode_tiled_fn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                        const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                        CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static vfk_encode_tiled_fn encode_tiled_entry() {
    static vfk_encode_tiled_fn fn = [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult qr;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qr) != cudaSuccess || qr != cudaDriverEntryPointSuccess)
            p = nullptr;
        return reinterpret_cast<vfk_encode_tiled_fn>(p);
    }();
    return fn;
}

// [tiles][rows][inner] array of T, box {box_inner, box_rows, 1}: the 32 / L lanes a warp takes of `box_rows` rows of one tile
template <typename T>
static int encode_map3(vfk_ctx* h, CUtensorMap* m, const void* base, uint64_t inner, uint64_t rows, uint64_t tiles, uint32_t box_inner,
                       uint32_t box_rows) {
    vfk_encode_tiled_fn enc = encode_tiled_entry();
    if (!enc) return fail(h, VFK_ERR_CUDA, "cuTensorMapEncodeTiled is not available from this driver");
    const cuuint64_t gdim[3] = {inner, rows, tiles};
    const cuuint64_t gstr[2] = {inner * sizeof(T), inner * rows * sizeof(T)};
    const cuuint32_t box[3] = {box_inner, box_rows, 1};
    const cuuint32_t estr[3] = {1, 1, 1};
    const CUresult r = enc(m, sizeof(T) == 4 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 3, const_cast<void*>(base),
                           gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(h, VFK_ERR_CUDA, "cuTensorMapEncodeTiled failed (%d)", (int)r);
    return VFK_OK;
}

// The lane-split shape is instantiated for the FP64 17-joint kernel only: there the one-thread-per-instance kernel cannot
// hold its Jacobian (102 doubles for 17 joints) and runs 1 CTA per SM with 568 B of spills, while two lanes per instance fit
// 255 registers without spills at 2 CTAs per SM: 173 us against 217 us per launch (256 k x 17 joints x 64 obstacles, 0.60
// against 0.48 of the HBM roofline).  Everywhere else it measured slower and was removed (FP32 config 5: 184 vs 154 us;
// 10 joints: 98 vs 70 us in FP64, 95 vs 70 us in FP32; FP64 config 2: 29.6 vs 23.4 us; DESIGN.md section 4.2), and so were
// four lanes per instance (231 us on the FP64 17-joint shape: every lane repeats the attractor, the Cholesky and the solves).
template <typename T, int N>
constexpr bool kSplit = sizeof(T) == 8 && N == 17;

// May this call run in the lane-split shape?  Lean call on blocked device buffers, DH-form chain of exactly the instantiated
// length.  VFK_NO_SPLIT=1 runs the one-thread-per-instance kernel instead (the reference the tests compare against).
template <typename T>
static bool split_ok(vfk_ctx* h, int n_kernel, const CycleCall& call) {
    const vfk_io* io = call.io;
    return !getenv("VFK_NO_SPLIT") && h->dh_chain && h->chain.n_joints == n_kernel && is_lean<T>(kconst<T>(h), call.b) &&
           !(io && (io->q_src || io->qdot));
}

template <typename T, int N>
static int launch_split(vfk_ctx* h, const CycleCall& call) {
    using SH = SplitShape<T, N>;
    const vfk_buffers* b = call.b;
    KArgs<T> a;
    memset(&a, 0, sizeof a);
    a.q = static_cast<T*>(b->q);
    a.qdot = static_cast<T*>(b->qdot);
    a.n = call.n;
    a.n_comp = h->chain.n_joints;
    a.k_cycles = call.k_cycles;
    a.own = chunk_plan(call.scene.own.m);
    a.n_stages = a.own.chunks < 2 ? a.own.chunks : 2;
    const size_t smem = kSmemHeader + SH::kTab + (size_t)(kBlock / 32) * SH::warp_bytes(a.n_stages);
    const uint64_t tiles = (uint64_t)((call.n + 31) / 32);
    SplitMaps maps;
    memset(&maps, 0, sizeof maps);
    int rc;
    if ((rc = encode_map3<T>(h, &maps.q, b->q, 32, (uint64_t)a.n_comp, tiles, SH::SUB, (uint32_t)a.n_comp)) != VFK_OK) return rc;
    if ((rc = encode_map3<T>(h, &maps.goal, b->goal, 32, 13, tiles, SH::SUB, 13)) != VFK_OK) return rc;
    if (a.own.n > 0) {
        const uint64_t rows = (uint64_t)a.own.np / 2 * ObstPairs<T>::kPlanes;                   // plane rows of 32 lanes x 16 bytes per tile
        if ((rc = encode_map3<T>(h, &maps.obst, call.scene.own.obst, 32 * 16 / sizeof(T), rows, tiles, SH::kRowBytes / sizeof(T),
                                 SH::kRowsPerChunk)) != VFK_OK)
            return rc;
    }
    return launch_persistent<vfk_split_kernel<T, N>>(h, (call.n + 31) / 32 * SH::L, smem, call.stream, kconst<T>(h), a, maps);
}

// SOLVE: the same choice of shape for vfk_solve, except that the lane-split shape has no solve variant (those calls run
// the one-thread-per-instance kernel) and the lean kernel's output conditions do not apply.
// SHARED (a non-empty shared list): the same choices among the one-thread-per-instance kernels -- EXT, lean / general, HIOCC --
// but neither the cooperative shape (FP64, n <= 4096) nor the lane-split shape (FP64, 17 joints) has a shared variant:
// those calls run the one-thread kernel, whose field they match bit for bit (DESIGN.md section 4.5).
// A mixed scene (own list and shared list) takes the same SHARED kernels; with ext rows both lists carry them.
template <typename T, int N, class PAT, bool SOLVE, bool SHARED>
static int dispatch_feat(vfk_ctx* h, const CycleCall& call) {
    const KConst<T>& c = kconst<T>(h);
    const vfk_buffers* b = call.b;
    const vfk_scene& sc = call.scene;
    const bool ext = (sc.own.obst_ext && sc.own.m > 0) || (sc.shared.obst_ext && sc.shared.m > 0);
    // Small FP64 batches cannot fill the GPU with one thread per instance: switch to the cooperative latency shape.
    // Measured (scripts/latency.py, one robot, 1000 fused cycles): FP64 M = 32: 6.4 vs 7.1 us per cycle, M = 256: 23.6 vs
    // 36.3 us.  In FP32 the repeller is three MUFU instructions and the shape only adds ring overhead (3.7 vs 2.7 us),
    // so it is neither selected nor instantiated there.
    if constexpr (sizeof(T) == 8 && !SHARED) {
        const bool coop = call.n <= kCoopMaxInstances && sc.own.m >= 2 * kChunk && !getenv("VFK_NO_COOP");
        if (coop) return ext ? launch_cycle<T, N, PAT, true, false, kChunk, false, SOLVE>(h, call)
                             : launch_cycle<T, N, PAT, false, false, kChunk, false, SOLVE>(h, call);
    }
    if (ext) return launch_cycle<T, N, PAT, true, false, 1, false, SOLVE, SHARED>(h, call);
    // Two lanes per instance (vfk_split.cuh) for the FP64 17-joint kernel.
    if constexpr (kSplit<T, N> && !SOLVE && !SHARED) {
        if (sc.own.m > 0 && split_ok<T>(h, N, call)) return launch_split<T, N>(h, call);
    }
    if ((SOLVE ? lean_inputs<T>(c, b) : is_lean<T>(c, b)) && h->chain.n_joints == N) {
        if constexpr (sizeof(T) == 4 && N <= 7 && !SOLVE) {
            if (call.k_cycles == 1) return launch_cycle<T, N, PAT, false, true, 1, true, false, SHARED>(h, call);
        }
        return launch_cycle<T, N, PAT, false, true, 1, false, SOLVE, SHARED>(h, call);
    }
    return launch_cycle<T, N, PAT, false, false, 1, false, SOLVE, SHARED>(h, call);
}

template <typename T, int N, bool SOLVE, bool SHARED>
static int dispatch_ext(vfk_ctx* h, const CycleCall& call) {
    if constexpr (N == 7) {
        if (h->pattern == 1) return dispatch_feat<T, N, LwrPattern, SOLVE, SHARED>(h, call);
    }
    if constexpr (N >= 10) {
        if (h->pattern == 2) return dispatch_feat<T, N, DhPattern, SOLVE, SHARED>(h, call);
    }
    return dispatch_feat<T, N, GenericPattern, SOLVE, SHARED>(h, call);
}

// The body of every launcher: the kernels of one precision, step or solve, per-instance or SHARED, for the joint counts Ns
// its translation unit instantiates, picked by the chain's kernel joint count.
template <typename T, bool SOLVE, bool SHARED, int... Ns>
static int launch_family(vfk_ctx* h, const CycleCall& call) {
    int rc = 0;
    if (((h->n_kernel == Ns && (rc = dispatch_ext<T, Ns, SOLVE, SHARED>(h, call), true)) || ...)) return rc;
    return fail(h, VFK_ERR_UNSUPPORTED, "no kernel for n_joints = %d", h->chain.n_joints);
}
