// vfk_kernels.cuh -- the fused vfclik control-cycle kernel for sm_100a.
//
// One thread = one manipulator instance; a warp is a persistent worker over tiles of 32
// consecutive instances.  All per-instance state (q, frame, the 6xN Jacobian, the 6x6
// normal matrix) lives in registers across the K fused cycles.  Global arrays are
// tile-blocked SoA (include/vfk.h): element (component c, instance i) of a C-component
// array lives at ((i/32)*C + c)*32 + i%32; obstacles {x,y,z,radius} are stored in pairs, each
// lane's 16-byte vectors holding the same component(s) of both (ObstPairs below), so
// everything a warp needs for a tile -- q (N rows), goal (13 rows), every chunk of 8
// obstacles -- is ONE contiguous burst.  Those bursts are moved global -> shared with
// cp.async.bulk (TMA), one copy each, into per-warp buffers guarded by mbarriers, one tile
// AHEAD of the arithmetic, so HBM latency is hidden behind the previous tile's FK / Cholesky
// work; the repulsor loop reads two conflict-free LDS.128 per obstacle PAIR and runs on the
// packed FP32 instructions (FFMA2 / FMUL2 / FADD2).  Robot constants (chain, limits, gains,
// the sin / cos table) arrive as a __grid_constant__ kernel parameter (constant bank 0),
// indexed at compile time.
//
// Reference mapping (see include/vfk.h and SURVEY.md App. C.2):
//   fk_jacobian()   scripts/vf:316-318, scripts/nullspace:175  (Lafik / KDL FK + Jacobian)
//   attractor/repulsor  scripts/vf:276-293,344-347              (vfl type 1 + type 2 fields)
//   dls             scripts/vf:461                              (Lafik.getIKV)
//   nullspace       scripts/nullspace:75-131,159-184
//   jp controller   scripts/joint_p_controller:79-89,126-146
//   mixer / clamp   src/command_mixer.py:71-82, scripts/bridge:188-203
#pragma once
#include <stdint.h>
#include "vfk_math.cuh"
#include "vfk_tma.cuh"
#include "vfk_nullspace.cuh"

namespace vfk {

constexpr int kMaxJ = 17;
#ifndef VFK_BLOCK
#define VFK_BLOCK 128
#endif
constexpr int kBlock = VFK_BLOCK;    // threads per CTA of the cycle kernel (warps are independent workers; 64 measured 0.3 % slower, must divide 128)
constexpr int kSmallBlock = 128;     // threads per CTA of the small one-element-per-thread kernels
#ifndef VFK_CHUNK
#define VFK_CHUNK 8
#endif
constexpr int kChunk = VFK_CHUNK;            // obstacles per shared-memory stage (4 measured: FP64 config 2 -13 %, -30 % with 3 CTAs/SM; FP32 headline -14 %)
constexpr int kMaxStages = 8;
constexpr int kSmemHeader = 512;     // per-warp mbarriers live in the first 512 bytes of dynamic smem
// TAB (kernel template parameter): the FP32 mode's wide kinematic chain takes sin / cos from a 128-entry table in shared
// memory (sincos_table, vfk_math.cuh: 13 FP64 operations per joint instead of 23, a dependent chain half as long); the
// table sits between the header and the per-warp regions and is built once per CTA behind the first tile's copies.
// Measured on B200 (same-box A/Bs, profiles/r02t_sincos_table_ab.txt): 17 joints K = 1 126.7 -> 123.6 us, K = 100 +3.2 %;
// the headline shape K = 100 +4.7 - 5.3 % (1.34 -> 1.40e10 inst-cycles/s) and 0.983 instead of 0.960 of the HBM roofline
// over 1000 launches (less FP64 work, later power cap).  Its HBM-bound single-cycle launch lost 3.4 % with the table while
// every chunk still waited for DRAM (the table's random 16-byte reads are ~10 shared-memory wavefronts each, +45 % on the
// L1 data pipe that also takes the TMA deliveries); with the L2 prefetch in place it is unchanged, so the host turns the
// table on for every FP32 instantiation (launch_cycle).  -DVFK_NO_SINCOS_TABLE turns it off everywhere.
#ifdef VFK_NO_SINCOS_TABLE
constexpr bool kSinCosTable = false;
#else
constexpr bool kSinCosTable = true;
#endif
template <typename T>
constexpr bool kCanTab = kSinCosTable && sizeof(T) == 4 && sizeof(typename WideOf<T>::type) == 8;
template <typename T, bool TAB>
constexpr uint32_t kTabBytes = (TAB && kCanTab<T>) ? kSinCosTabEntries * 16 : 0;
// FP32 decay order 20 (the reference's typical value, old/README.old:75) by five multiplications instead of MUFU lg2 / ex2:
// two more instructions per obstacle but two fewer on the quarter-rate XU pipe, which also carries rsqrt and the
// FP64 <-> FP32 conversions.  Measured on B200 (1 M instances): 109.1 us vs 110.3 us per launch at K = 1, -0.6 % at
// K = 100; also the more accurate of the two.  -DVFK_NO_F32_POWCHAIN restores the MUFU form.
#ifdef VFK_NO_F32_POWCHAIN
constexpr bool kF32PowChain = false;
#else
constexpr bool kF32PowChain = true;
#endif

// Kernel-side constants in the kernel's arithmetic type.  Joints are canonicalised on
// the host (vfk_api.cu: canonicalise_chain) so that every joint acts about / along its
// local Z axis: RotX/RotY/TransX/TransY are conjugated into the neighbouring tips.
template <typename T>
struct KConst {
    using W = typename WideOf<T>::type;
    SinCosTab sincos;          // reduction constants and polynomial coefficients of sincos_wide
    W base[12];
    W tip[kMaxJ][12];
    T q_lo[kMaxJ], q_hi[kMaxJ];
    T ns_q0_scale[kMaxJ];      // -k / (hi - lo)^2
    T ns_mid[kMaxJ];
    T w_joint[kMaxJ];
    T jp_ref[kMaxJ];
    T w_task[6];
    T mixer_w[6];
    T tool[12];
    T ns_control[4];
    typename WideNE<T>::type ik_lambda2, ns_lambda2;
    T dt, speed_scale, max_vel, jp_kp, jp_delta;
    T ns_gain, ns_lookahead, rot_slowdown_inv, goal_force, obst_force, obst_safe_inv, obst_order;
    int32_t prismatic_mask;    // bit j set: joint j is TransZ, else RotZ
    int32_t xtwist_mask;       // bit j set: tip j's rotation is RotX(alpha) (every DH-specified chain), alpha in tip[j][4], [7]
    int32_t tipident_mask;     // bit j set: tip j's rotation is the identity
    int32_t ns_mode;
    int32_t direct_control;    // resolved 0/1 (1 for the Powercube / iCub back-ends: they command qdot_lim itself)
    int32_t shoulder_clamp;    // Powercube_Bridge.set_vel's second clamp on joint 0 (scripts/bridge:295-303)
    T shoulder_pos, shoulder_neg;
    int32_t integrate;
    int32_t unit_weights;      // w_task and w_joint are all ones
    int32_t share_factor;      // nullspace can reuse the IK Cholesky factor
    int32_t tool_identity;
    int32_t need_jp;           // joint P controller observable (weight != 0 or an output wants it)
    int32_t asin_series;       // rot_slowdown <= 0.3 rad: small-angle series replaces atan2 in FP32
    int32_t order_int;         // obst_order when it is a small integer, else 0
    int32_t all_xtwist;        // every tip rotation is the identity or RotX(alpha): the lane-split kernel's uniform fast path
    int32_t ik_mode;           // VFK_IK_*: 1 = truncated (KDL-wdls-style) form through a one-sided Jacobi SVD, FP64 general kernel only
    double ik_eps, ik_lambda2_d;
    int32_t ns_qr;             // nullspace through the Householder basis of null(J): control mode, or the projector with ns_lambda = 0
};

template <typename T>
struct KArgs {
    T* q;
    const T* goal;
    const Vec4<T>* obst;       // pair-interleaved blocked [tile][Mp / 2][planes][32 x 16 B], Mp = M rounded up to even (ObstPairs)
    const Vec2<T>* obst_ext;   // blocked [tile][M][32] {safe, order} or null
    const T* aux;              // blocked [n_aux * 12] auxiliary field records or null
    T* jp_ref;
    const T* jp_lo;            // per-instance limits of the joint controller (both or neither), see vfk_buffers
    const T* jp_hi;
    const T* ns_in;
    T* ns_lastvec;
    const T* q_cmded;
    const T* ext_cmd[3];
    T* qdot_vf;
    T* qdot_ns;
    T* qdot_jp;
    T* qdot;
    T* cmd;
    T* pose;
    T* twist;                  // [6] commanded tool twist (velPos, velRot of scripts/vf:346-347)
    int32_t* flags;
    // Direct host I/O of the host-buffer session (zero-copy): when q_src is set the q tile is read from a DENSE [N][q_src_ld]
    // array (page-locked host memory mapped into the device address space) instead of the blocked `q`; when qdot_ld is
    // non-zero `qdot` is such a dense array too.  The integrated q still goes to the blocked `q`.
    const T* q_src;
    int64_t q_src_ld;
    int64_t qdot_ld;
    T* qdot_dev;               // direct host I/O: the blocked device mirror of qdot (kept current for vfk_session_read), or null
    int64_t n;
    int32_t n_obst;
    int32_t n_obst_p;          // n_obst rounded up to even: rows of 32 Vec4<T> per tile in `obst`
    int32_t n_chunks;          // ceil(n_obst / kChunk)
    int32_t n_full;            // n_obst / kChunk (chunks with all kChunk obstacles)
    int32_t n_rem;             // n_obst % kChunk
    int32_t n_stages;          // shared-memory stages (<= kMaxStages); >= n_chunks means resident
    int32_t k_cycles;
    int32_t n_aux;
    int32_t n_comp;            // joint components per instance in memory (<= N: generic chains of fewer joints run padded, see nc below)
};

// ------------------------------------------------------------------------------ chain patterns
// A chain pattern fixes, at compile time, the *structure* of the tip frames: which tips have a
// signed-permutation rotation (every DH chain with twists in {0, +-pi/2, pi}) and which tip
// translation components are zero.  The numeric values still come from KConst; the pattern only
// lets the compiler turn R * R_tip into register renaming and drop the multiplies by 0.
// GenericPattern makes no assumption (full 3x3 products, runtime prismatic mask).
struct GenericPattern {
    static constexpr bool generic = true;
    static constexpr bool dh = false;
    static constexpr bool base_identity = false;
    __host__ __device__ static constexpr int perm(int, int) { return 0; }
    __host__ __device__ static constexpr int sign(int, int) { return 1; }
    __host__ __device__ static constexpr bool pnz(int, int) { return true; }
};

// KUKA LWR-style 7R chain: base rotation identity, tips RotX(+90), RotX(-90), RotX(-90), RotX(+90),
// RotX(+90), RotX(-90), identity; translations only along y (tips 1, 3) and z (tip 6); all revolute.
// new column k of (R * R_tip) = sign(j,k) * old column perm(j,k).
struct LwrPattern {
    static constexpr bool generic = false;
    static constexpr bool dh = false;
    static constexpr bool base_identity = true;
    __host__ __device__ static constexpr int kind(int j) {       // +1: RotX(+90), -1: RotX(-90), 0: identity
        return (j == 0 || j == 3 || j == 4) ? 1 : (j == 6 ? 0 : -1);
    }
    __host__ __device__ static constexpr int perm(int j, int k) { return kind(j) == 0 ? k : (k == 0 ? 0 : (k == 1 ? 2 : 1)); }
    __host__ __device__ static constexpr int sign(int j, int k) {
        return kind(j) == 0 ? 1 : (k == 0 ? 1 : (k == 1 ? (kind(j) > 0 ? 1 : -1) : (kind(j) > 0 ? -1 : 1)));
    }
    __host__ __device__ static constexpr bool pnz(int j, int k) { return ((j == 1 || j == 3) && k == 1) || (j == 6 && k == 2); }
};

// Any chain given in Denavit-Hartenberg form: every joint revolute (about its local Z after the host's canonicalisation), every
// tip rotation RotX(alpha) -- alpha = 0, i.e. the identity, included -- and any tip translation.  Values come from KConst; what
// the pattern removes is every per-joint run-time decision of GenericPattern (prismatic?, identity / X-twist / general tip?,
// padding joint?) together with the register copies their join points cost: the tip product is 12 operations in place.
struct DhPattern {
    static constexpr bool generic = false;
    static constexpr bool dh = true;
    static constexpr bool base_identity = false;
    __host__ __device__ static constexpr int perm(int, int) { return 0; }
    __host__ __device__ static constexpr int sign(int, int) { return 1; }
    __host__ __device__ static constexpr bool pnz(int, int) { return true; }
};

// ------------------------------------------------------------------------------ FK + J
// T_{j+1} = T_j * RotZ(q_j) * tip_j, carried in the wide type W (double in both modes: an FP32 chain leaves ~1e-7 m in the
// tool position, which the order-20 repeller decay turns into 1e-4 relative field errors near obstacles).  Records the
// joint axis z_j = R_j[:,2] and origin p_j before each joint, then forms J = [z x (p_e - p_j); z] (revolute) or [z; 0]
// in T.  Outputs: R, and the tool-less flange position as hi + lo parts in T (lo = 0 when T is already wide).
template <typename T, int N, class PAT, bool TAB = false>
__device__ __forceinline__ void fk_jacobian(const KConst<T>& c, const T (&q)[N], typename WideOf<T>::type (&R)[9],
                                            typename WideOf<T>::type (&p)[3], T (&Jl)[N][3], T (&Ja)[N][3], int nc,
                                            [[maybe_unused]] const double2* sctab) {
    using W = typename WideOf<T>::type;
    if constexpr (PAT::base_identity) {
#pragma unroll
        for (int k = 0; k < 9; ++k) R[k] = (k % 4 == 0) ? W(1) : W(0);
    } else {
#pragma unroll
        for (int k = 0; k < 9; ++k) R[k] = c.base[k];
    }
#pragma unroll
    for (int k = 0; k < 3; ++k) p[k] = c.base[9 + k];
    static_for<0, N>([&](auto jc) {
        constexpr int j = decltype(jc)::value;
        if (PAT::generic && j >= nc) {                                  // padding joint of a shorter chain: no motion, zero column
            Ja[j][0] = Ja[j][1] = Ja[j][2] = T(0);
            Jl[j][0] = Jl[j][1] = Jl[j][2] = T(0);
            return;
        }
        Ja[j][0] = (T)R[2]; Ja[j][1] = (T)R[5]; Ja[j][2] = (T)R[8];
        Jl[j][0] = (T)p[0]; Jl[j][1] = (T)p[1]; Jl[j][2] = (T)p[2];      // holds p_j until p_e is known
        const W qj = (W)q[j];
        if (PAT::generic && (c.prismatic_mask & (1 << j))) {
            p[0] = fma(R[2], qj, p[0]); p[1] = fma(R[5], qj, p[1]); p[2] = fma(R[8], qj, p[2]);
        } else {
            W s, co;
            // FP32 mode's wide chain: the quarter-angle form (no quadrant logic, ~10 instructions fewer per joint; measured on B200
            // against sincos_wide<5>: K = 1 headline 109.5 vs 109.9 us, K = 100 +3.2 %, 17 joints +2.6 % / +3.3 %)
            if constexpr (kTabBytes<T, TAB> != 0) sincos_table(c.sincos, sctab, qj, &s, &co);
            else if constexpr (sizeof(T) == 4 && sizeof(W) == 8) sincos_quarter<5>(c.sincos, qj, &s, &co);
            else sincos_wide<(sizeof(T) == sizeof(W)) ? 7 : 5>(c.sincos, qj, &s, &co);
#pragma unroll
            for (int r = 0; r < 3; ++r) {
                const W a = R[3 * r + 0], b = R[3 * r + 1];
                R[3 * r + 0] = fma(co, a, s * b);
                R[3 * r + 1] = fma(co, b, -s * a);
            }
        }
        const W* tp = c.tip[j];
        static_for<0, 3>([&](auto kc) {
            constexpr int k = decltype(kc)::value;
            if constexpr (PAT::pnz(j, k)) {
#pragma unroll
                for (int r = 0; r < 3; ++r) p[r] = fma(R[3 * r + k], tp[9 + k], p[r]);
            }
        });
        if constexpr (PAT::dh) {
            const W ca = tp[4], sa = tp[7];
#pragma unroll
            for (int r = 0; r < 3; ++r) {
                const W a = R[3 * r + 1], b = R[3 * r + 2];
                R[3 * r + 1] = fma(ca, a, sa * b);
                R[3 * r + 2] = fma(ca, b, -sa * a);
            }
            return;
        }
        W Rn[9];
        if constexpr (PAT::generic) {
            // warp-uniform choice on the robot's constants: identity tip (nothing), X-twist tip (12 ops), general (27)
            if (c.tipident_mask & (1 << j)) {
#pragma unroll
                for (int k = 0; k < 9; ++k) Rn[k] = R[k];
            } else if (c.xtwist_mask & (1 << j)) {
                const W ca = tp[4], sa = tp[7];
#pragma unroll
                for (int r = 0; r < 3; ++r) {
                    const W a = R[3 * r + 1], b = R[3 * r + 2];
                    Rn[3 * r + 0] = R[3 * r + 0];
                    Rn[3 * r + 1] = fma(ca, a, sa * b);
                    Rn[3 * r + 2] = fma(ca, b, -sa * a);
                }
            } else {
#pragma unroll
                for (int r = 0; r < 3; ++r)
#pragma unroll
                    for (int cc = 0; cc < 3; ++cc)
                        Rn[3 * r + cc] = fma(R[3 * r + 0], tp[cc], fma(R[3 * r + 1], tp[3 + cc], R[3 * r + 2] * tp[6 + cc]));
            }
        } else {
            static_for<0, 3>([&](auto kc) {
                constexpr int k = decltype(kc)::value;
#pragma unroll
                for (int r = 0; r < 3; ++r)
                    Rn[3 * r + k] = PAT::sign(j, k) > 0 ? R[3 * r + PAT::perm(j, k)] : -R[3 * r + PAT::perm(j, k)];
            });
        }
#pragma unroll
        for (int k = 0; k < 9; ++k) R[k] = Rn[k];
    });
    const T pe[3] = {(T)p[0], (T)p[1], (T)p[2]};
    const T pel[3] = {(T)(p[0] - (W)pe[0]), (T)(p[1] - (W)pe[1]), (T)(p[2] - (W)pe[2])};
    static_for<0, N>([&](auto jc) {
        constexpr int j = decltype(jc)::value;
        if (PAT::generic && (c.prismatic_mask & (1 << j))) {
            Jl[j][0] = Ja[j][0]; Jl[j][1] = Ja[j][1]; Jl[j][2] = Ja[j][2];
            Ja[j][0] = Ja[j][1] = Ja[j][2] = T(0);
        } else {
            const T dx = (pe[0] - Jl[j][0]) + pel[0], dy = (pe[1] - Jl[j][1]) + pel[1], dz = (pe[2] - Jl[j][2]) + pel[2];
            Jl[j][0] = Ja[j][1] * dz - Ja[j][2] * dy;
            Jl[j][1] = Ja[j][2] * dx - Ja[j][0] * dz;
            Jl[j][2] = Ja[j][0] * dy - Ja[j][1] * dx;
        }
    });
}

// Tool position as a sum of two T values (hi + lo): differences against it are accurate to an ulp of the difference
// even though T alone cannot represent the position to better than 6e-8 m.  lo is identically zero when T is wide.
template <typename T>
struct Pos {
    T hi[3], lo[3];
    template <typename W>
    __device__ __forceinline__ void set(const W (&p)[3]) {
#pragma unroll
        for (int k = 0; k < 3; ++k) { hi[k] = (T)p[k]; lo[k] = (T)(p[k] - (W)hi[k]); }
    }
    // x - position_k
    __device__ __forceinline__ T from(T x, int k) const {
        if constexpr (sizeof(T) == sizeof(typename WideOf<T>::type)) return x - hi[k];
        else return (x - hi[k]) - lo[k];
    }
};

// ------------------------------------------------------------------------------ obstacle storage
// Obstacles are stored in PAIRS so that one 16-byte vector per lane holds the same component(s) of two obstacles:
//   FP32: pair p of a tile = 2 planes of 32 lanes x float4:  {x0, x1, y0, y1}, {z0, z1, r0, r1}
//   FP64: pair p of a tile = 4 planes of 32 lanes x double2: {x0, x1}, {y0, y1}, {z0, z1}, {r0, r1}
// (obstacle 2p in slot 0, obstacle 2p + 1 in slot 1; an odd obstacle count is padded with a zero-radius slot).  A pair takes
// the bytes of two {x, y, z, radius} vectors per lane, so a chunk of kChunk obstacles is still one contiguous burst.  What
// it buys: every shared-memory read is a conflict-free 16-byte access in both precisions (a lane-strided 32-byte FP64 vector
// was a 2-way bank conflict), and in FP32 the two obstacles of a pair sit in adjacent registers exactly as sm_100's packed
// FP32 instructions (fma / mul / add .f32x2 -> SASS FFMA2 / FMUL2 / FADD2) want their operands: the repulsor of TWO
// obstacles issues as ~25 instructions instead of 2 x 22.
template <typename T> struct ObstPairs;
template <> struct ObstPairs<float> {
    static constexpr int kPlanes = 2;
    // obstacle `s` (0 / 1) of the pair whose first plane starts at `pair` (lane 0), for `lane`
    static __device__ __forceinline__ Vec4<float> load(const Vec4<float>* pair, int lane, int s) {
        const float* f = reinterpret_cast<const float*>(pair) + lane * 4 + s;
        Vec4<float> o;
        o.x = f[0]; o.y = f[2]; o.z = f[128]; o.w = f[130];
        return o;
    }
    static __device__ __forceinline__ void store(Vec4<float>* pair, int lane, int s, const Vec4<float>& o) {
        float* f = reinterpret_cast<float*>(pair) + lane * 4 + s;
        f[0] = o.x; f[2] = o.y; f[128] = o.z; f[130] = o.w;
    }
};
template <> struct ObstPairs<double> {
    static constexpr int kPlanes = 4;
    static __device__ __forceinline__ Vec4<double> load(const Vec4<double>* pair, int lane, int s) {
        const double* f = reinterpret_cast<const double*>(pair) + lane * 2 + s;
        Vec4<double> o;
        o.x = f[0]; o.y = f[64]; o.z = f[128]; o.w = f[192];
        return o;
    }
    static __device__ __forceinline__ void store(Vec4<double>* pair, int lane, int s, const Vec4<double>& o) {
        double* f = reinterpret_cast<double*>(pair) + lane * 2 + s;
        f[0] = o.x; f[64] = o.y; f[128] = o.z; f[192] = o.w;
    }
};

// ------------------------------------------------------------------------------ field pieces
// One decay repeller (vfl type 2): acc += (o - p)/d * (radius / max(d, safe))^order.
// d^2 carries a 1e-30 (1e-300 in FP64) bias so that d = 0 gives a finite 1/d and a zero contribution
// (0 * finite) without a branch; radius = 0 (empty slot) gives lg2(0) = -inf -> decay = 0 since order > 0.
template <typename T, int ORDER = 0>
__device__ __forceinline__ void repel(const Vec4<T>& o, T safe_inv, T order, const Pos<T>& pt, T (&acc)[3]) {
    const T dx = pt.from(o.x, 0), dy = pt.from(o.y, 1), dz = pt.from(o.z, 2);
    const T dd = fma(dx, dx, fma(dy, dy, fma(dz, dz, Prec<T>::tiny())));
    const T inv = Prec<T>::rsqrt_pos(dd);                                       // 1/d
    const T ratio = o.w * Prec<T>::fmin_(inv, safe_inv);                        // radius / max(d, safe)
    T wgt = pow_fixed<ORDER, T>(ratio, order) * inv;
    // FP32: (radius / d)^order / d passes 3.4e38 once the tool is within ~radius/75 of an obstacle centre (order 20) --
    // one instance in a few million at 256 random obstacles.  Saturating the weight keeps the sum finite; such an
    // obstacle still outweighs everything else by > 1e15, and normCart only keeps the direction.
    if constexpr (sizeof(T) == 4) wgt = Prec<T>::fmin_(wgt, T(1e30));
    acc[0] = fma(wgt, dx, acc[0]); acc[1] = fma(wgt, dy, acc[1]); acc[2] = fma(wgt, dz, acc[2]);
}

// The same for the two obstacles of a pair at once in FP32, on sm_100's packed instructions.  A = {x0, x1, y0, y1},
// B = {z0, z1, r0, r1} as they come out of shared memory; np = the tool position as negated, lane-duplicated hi / lo pairs;
// acc = {sum over slot-0 obstacles, sum over slot-1 obstacles} per axis (added together after the loop).  Every packed
// instruction is the IEEE operation on each half, so one obstacle's contribution is bit-identical to repel<float>().
struct NegPos2 {
    float2 hi[3], lo[3];
    __device__ __forceinline__ void set(const Pos<float>& p) {
#pragma unroll
        for (int k = 0; k < 3; ++k) { hi[k] = make_float2(-p.hi[k], -p.hi[k]); lo[k] = make_float2(-p.lo[k], -p.lo[k]); }
    }
};

template <int ORDER>
__device__ __forceinline__ void repel2(const float4& A, const float4& B, float safe_inv, float order, const NegPos2& np,
                                       float2 (&acc)[3]) {
    const float2 dx = __fadd2_rn(__fadd2_rn(make_float2(A.x, A.y), np.hi[0]), np.lo[0]);
    const float2 dy = __fadd2_rn(__fadd2_rn(make_float2(A.z, A.w), np.hi[1]), np.lo[1]);
    const float2 dz = __fadd2_rn(__fadd2_rn(make_float2(B.x, B.y), np.hi[2]), np.lo[2]);
    const float2 tiny = make_float2(1e-30f, 1e-30f);
    const float2 dd = __ffma2_rn(dx, dx, __ffma2_rn(dy, dy, __ffma2_rn(dz, dz, tiny)));
    const float2 inv = make_float2(Prec<float>::rsqrt_pos(dd.x), Prec<float>::rsqrt_pos(dd.y));
    const float2 ratio = __fmul2_rn(make_float2(B.z, B.w), make_float2(fminf(inv.x, safe_inv), fminf(inv.y, safe_inv)));
    float2 pw;
    if constexpr (ORDER == 20) {
        const float2 x2 = __fmul2_rn(ratio, ratio), x4 = __fmul2_rn(x2, x2), x5 = __fmul2_rn(x4, ratio), x10 = __fmul2_rn(x5, x5);
        pw = __fmul2_rn(x10, x10);
    } else {
        pw = make_float2(Prec<float>::pow_pos(ratio.x, order), Prec<float>::pow_pos(ratio.y, order));
    }
    float2 wgt = __fmul2_rn(pw, inv);
    wgt = make_float2(fminf(wgt.x, 1e30f), fminf(wgt.y, 1e30f));          // see repel(): saturate instead of overflowing
    acc[0] = __ffma2_rn(wgt, dx, acc[0]); acc[1] = __ffma2_rn(wgt, dy, acc[1]); acc[2] = __ffma2_rn(wgt, dz, acc[2]);
}

// Goal attractor (vfl type 1) at tool frame (Rt, pt): unit direction to the goal, unit rotation
// axis of R_g Rt^T scaled by the rotational slowdown, and the translational slowdown scalar.
template <typename T>
__device__ __forceinline__ void attract(const KConst<T>& c, const T (&g)[13], const T (&Rt)[9], const Pos<T>& pt,
                                        T (&V)[3], T& S0, T (&w)[3]) {
    const T ex = pt.from(g[9], 0), ey = pt.from(g[10], 1), ez = pt.from(g[11], 2);
    const T d2 = fma(ex, ex, fma(ey, ey, fma(ez, ez, Prec<T>::tiny())));
    const T invd = Prec<T>::rsqrt_pos(d2);
    const T dist = d2 * invd;
    const T gi = c.goal_force * invd;
    V[0] = gi * ex; V[1] = gi * ey; V[2] = gi * ez;
    S0 = g[12] > T(0) ? Prec<T>::fmin_(T(1), Prec<T>::div(dist, g[12])) : T(1);
    T E[9];                                                     // R_err = R_g * Rt^T
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
        for (int cc = 0; cc < 3; ++cc)
            E[3 * r + cc] = fma(g[3 * r + 0], Rt[3 * cc + 0], fma(g[3 * r + 1], Rt[3 * cc + 1], g[3 * r + 2] * Rt[3 * cc + 2]));
    T qw, qx, qy, qz;
    rot_to_quat<T>(E, qw, qx, qy, qz);
    const T n2 = fma(qx, qx, fma(qy, qy, qz * qz));
    const T invn = n2 > T(0) ? Prec<T>::rsqrt_pos(n2) : T(0);
    // angle = 2 atan2(|xyz|, w) in [0, pi].  It only matters below rot_slowdown (above it S1 saturates at 1), so
    // when the slowdown angle is small the FP32 path uses angle = 2 asin(n) through its series (error < 5e-7
    // relative for n <= 0.15); larger n just has to stay above the threshold, which the series does.
    const T nrm = n2 * invn;
    T angle;
    if (Prec<T>::kSeriesAsin && c.asin_series) {
        const T n2c = Prec<T>::fmin_(n2, T(0.25));
        angle = T(2) * nrm * fma(n2c, fma(n2c, T(0.075), T(1.0 / 6.0)), T(1));
    } else {
        angle = T(2) * Prec<T>::atan2_(nrm, qw);
    }
    // rot_slowdown_inv = +inf when off.  The product goes first: at angle = 0 it is 0 * inf = NaN, and fmin_ then selects 1
    // (FP64's fmin_ is `a < b ? a : b`, which returns its second operand when the first is NaN).
    const T S1 = Prec<T>::fmin_(angle * c.rot_slowdown_inv, T(1));
    const T sr = c.speed_scale * S1 * c.goal_force * invn;
    w[0] = sr * qx; w[1] = sr * qy; w[2] = sr * qz;
}

// Auxiliary fields (SURVEY.md section 8 row f2): records of VFK_AUX_COMPS = 12 scalars {type, force, p0..p9} in slots of a
// blocked per-instance array.  type 4 = hemisphere repeller (scripts/object_feeder:335-354: xyz, normal, safe, order),
// type 5 = funnel attractor (:262-280: goal xyz, axis, cut angle, angle-decay order, cut distance, distance-decay order);
// any other type code = empty slot.  Functional forms: oracle.batch.ORACLE_CHOICES (vfl is un-vendored).
template <typename T>
__device__ __forceinline__ void aux_fields(const T* __restrict__ aux, int n_aux, int64_t tile, int lane, const Pos<T>& pt, T (&V)[3]) {
    for (int s = 0; s < n_aux; ++s) {
        const T* r = aux + (tile * (n_aux * 12) + s * 12) * 32 + lane;
        const int type = (int)__ldg(r);
        if (type != 4 && type != 5) continue;
        const T force = __ldg(r + 32);
        T p[10];
#pragma unroll
        for (int k = 0; k < 10; ++k) p[k] = __ldg(r + (2 + k) * 32);
        const T rx = -pt.from(p[0], 0), ry = -pt.from(p[1], 1), rz = -pt.from(p[2], 2);
        const T an2 = p[3] * p[3] + p[4] * p[4] + p[5] * p[5];
        if (!(an2 > T(0))) continue;
        const T ian = Prec<T>::rsqrt_pos(an2);
        const T ax = p[3] * ian, ay = p[4] * ian, az = p[5] * ian;
        const T s_ax = rx * ax + ry * ay + rz * az;                       // height above the plane / distance along the axis
        if (type == 4) {
            const T safe = p[6], order = p[7];
            const T ratio = Prec<T>::div(safe, Prec<T>::fmax_(s_ax, safe));
            const T mag = -force * Prec<T>::pow_pos(ratio, order);        // field points toward the surface (-normal)
            V[0] = fma(mag, ax, V[0]); V[1] = fma(mag, ay, V[1]); V[2] = fma(mag, az, V[2]);
        } else {
            const T cut_a = p[6], ord_a = p[7], cut_d = p[8], ord_d = p[9];
            const T px = rx - s_ax * ax, py = ry - s_ax * ay, pz = rz - s_ax * az;   // radial offset from the approach axis
            const T rho2 = px * px + py * py + pz * pz;
            if (!(rho2 > T(0))) continue;
            const T rho = Prec<T>::sqrt_(rho2);
            const T theta = Prec<T>::atan2_(rho, s_ax);
            const T R = Prec<T>::sqrt_(rx * rx + ry * ry + rz * rz);
            const T wa = theta <= cut_a ? T(1) : Prec<T>::pow_pos(Prec<T>::div(cut_a, theta), ord_a);
            const T wd = R <= cut_d ? T(1) : Prec<T>::pow_pos(Prec<T>::div(cut_d, R), ord_d);
            const T mag = -force * wa * wd * Prec<T>::rcp(rho);           // unit vector toward the axis
            V[0] = fma(mag, px, V[0]); V[1] = fma(mag, py, V[1]); V[2] = fma(mag, pz, V[2]);
        }
    }
}

// normCart + saturation: unit translational part (zero stays zero), pre-scaled by its largest
// component so the squared norm cannot overflow in FP32; v = speed * S0 * V.
template <typename T>
__device__ __forceinline__ void saturate(const KConst<T>& c, T (&V)[3], T S0, T (&v)[3]) {
    const T big = Prec<T>::fmax_(Prec<T>::fabs_(V[0]), Prec<T>::fmax_(Prec<T>::fabs_(V[1]), Prec<T>::fabs_(V[2])));
    T scale = T(0);
    if (big > T(0)) {
        const T ib = Prec<T>::rcp(big);
        V[0] *= ib; V[1] *= ib; V[2] *= ib;
        scale = Prec<T>::rsqrt_pos(fma(V[0], V[0], fma(V[1], V[1], V[2] * V[2])));
    }
    const T sl = c.speed_scale * S0 * scale;
    v[0] = sl * V[0]; v[1] = sl * V[1]; v[2] = sl * V[2];
}

// ------------------------------------------------------------------------------ per-warp staging
// Every warp is an independent persistent worker over tiles of 32 consecutive instances.  It owns
//   * a ring of `n_stages` obstacle stages (kChunk obstacles x 32 instances each), and
//   * two q/goal buffers ((N + 13) rows x 32 instances),
// each guarded by its own mbarrier and filled by cp.async.bulk (TMA).  The ring runs ahead of the
// arithmetic across tile boundaries: while a warp works on tile t its lanes have already requested
// q/goal of tile t+1 and, stage by stage, the obstacles of tile t+1.  No CTA-wide barrier exists.
template <typename T, int N, bool EXT>
struct WarpStage {
    static constexpr uint32_t kRow = 32 * sizeof(Vec4<T>);                 // one obstacle, 32 instances
    static constexpr uint32_t kRowExt = EXT ? 32 * sizeof(Vec2<T>) : 0;
    static constexpr uint32_t kStage = kChunk * (kRow + kRowExt);
    static constexpr uint32_t kQgRow = 32 * sizeof(T);
    static constexpr uint32_t kQgRows = N + 13;
    static constexpr uint32_t kQg = kQgRows * kQgRow;
    static constexpr int kBars = kMaxStages + 2;                            // full[stage], qg[2]
    __host__ __device__ static constexpr uint32_t warp_bytes(int n_stages) { return n_stages * kStage + 2 * kQg; }
};

// One bulk copy per obstacle chunk (and one for its ext rows): the chunk's kChunk x 32 vectors are contiguous.
// Called by all lanes after a __syncwarp(); lane 0 issues.
template <typename T, int N, bool EXT>
__device__ __forceinline__ void issue_obst(const KArgs<T>& a, int64_t tile, int chunk, int stage, uint32_t region,
                                           uint32_t bars, int lane) {
    using WS = WarpStage<T, N, EXT>;
    if (lane == 0) {
        const int m0 = chunk * kChunk;
        const uint32_t cnt = (uint32_t)min(kChunk, a.n_obst - m0);
        const uint32_t cntp = (cnt + 1u) & ~1u;                           // whole pairs (the odd one out carries a zero-radius slot)
        const uint32_t dst = region + (uint32_t)stage * WS::kStage, bar = bars + 8u * (uint32_t)stage;
        mbar_arrive_expect_tx_a(bar, cntp * WS::kRow + cnt * WS::kRowExt);
        bulk_g2s_a(dst, a.obst + (tile * a.n_obst_p + m0) * 32, cntp * WS::kRow, bar);
        if (EXT) bulk_g2s_a(dst + kChunk * WS::kRow, a.obst_ext + (tile * a.n_obst + m0) * 32, cnt * WS::kRowExt, bar);
    }
}

// q tile (N rows) + goal tile (13 rows): two bulk copies into q/goal buffer `buf`.
template <typename T, int N, bool EXT>
__device__ __forceinline__ void issue_qg(const KArgs<T>& a, int64_t tile, int buf, uint32_t region, uint32_t bars,
                                         int lane, int nc) {
    using WS = WarpStage<T, N, EXT>;
    if (lane == 0) {
        const uint32_t dst = region + (uint32_t)a.n_stages * WS::kStage + (uint32_t)buf * WS::kQg;
        const uint32_t bar = bars + 8u * (uint32_t)(kMaxStages + buf);
        mbar_arrive_expect_tx_a(bar, (uint32_t)(nc + 13) * WS::kQgRow);
        if (a.q_src) {
#pragma unroll
            for (int j = 0; j < N; ++j)
                if (j < nc) bulk_g2s_a(dst + j * WS::kQgRow, a.q_src + j * a.q_src_ld + (tile << 5), WS::kQgRow, bar);
        } else {
            bulk_g2s_a(dst, a.q + tile * (nc * 32), (uint32_t)nc * WS::kQgRow, bar);
        }
        bulk_g2s_a(dst + N * WS::kQgRow, a.goal + tile * (13 * 32), 13 * WS::kQgRow, bar);
    }
}

// ------------------------------------------------------------------------------ the fused kernel
// LEAN = compile-time promise of the common production shape (checked on the host, vfk_api.cu:is_lean): identity
// tool frame and IK weights, projector-mode nullspace on the built-in limit-avoidance gradient sharing the IK
// factor, joint P controller unobserved, no extra mixer ports, and q / qdot as the only outputs.  It removes every
// runtime feature branch from the hot loop (fewer instructions, registers and I-cache lines); the general
// instantiation keeps them all.
// G = lanes cooperating on one instance.  G = 1: one thread per instance (throughput shape).  G = 8: latency shape for
// small batches -- a warp takes 4 instances of a tile, the 8 lanes of a group split each chunk of 8 obstacles between
// them and combine their partial repulsor sums with __shfl_xor_sync; the rest of the cycle is computed redundantly by
// the group and lane 0 of the group stores.  A tile is then spread over 8 warps instead of one.
template <typename T, int N, class PAT, bool EXT, bool LEAN, int MINB, int G = 1, bool TAB = false>
__global__ void __launch_bounds__(kBlock, MINB)
vfk_cycle_kernel(const __grid_constant__ KConst<T> c, const __grid_constant__ KArgs<T> a) {
    using WS = WarpStage<T, N, EXT>;
    extern __shared__ __align__(128) unsigned char smem[];
    const int lane = threadIdx.x & 31;
    // read through a shuffle so that the compiler knows it is warp-uniform: tile numbers, ring positions and the addresses of
    // the bulk copies then live in uniform registers, and the copies issue without an elect-one loop around them
    const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem) + warp * WS::kBars;
    unsigned char* region = smem + kSmemHeader + kTabBytes<T, TAB> + (size_t)warp * WS::warp_bytes(a.n_stages);
    [[maybe_unused]] const double2* sctab = reinterpret_cast<const double2*>(smem + kSmemHeader);
    const uint32_t bars_a = smem_u32(bars), region_a = smem_u32(region);       // shared-window addresses, once per warp
    static_assert(G == 1 || G == kChunk, "a cooperative group takes one obstacle of a chunk per lane");
    constexpr int kSub = G == 1 ? 1 : G;                        // work units per tile (G == 8: 8 units of 4 instances)
    const int64_t n_tiles = (a.n + 31) >> 5;
    const int64_t n_units = n_tiles * kSub;
    const int64_t stride = (int64_t)gridDim.x * (kBlock / 32);
    int64_t unit = (int64_t)blockIdx.x * (kBlock / 32) + warp;
    if constexpr (kTabBytes<T, TAB> == 0) {
        if (unit >= n_units) return;
    }
    const int ol = lane & (G - 1);                              // obstacle lane within the group
    // Joint components in memory.  Chains with a joint count that has no instantiation of its own run in the next larger
    // generic one: joints >= nc are padding (zero Jacobian column, no motion, nothing loaded or stored for them).
    const int nc = (PAT::generic && !LEAN) ? a.n_comp : N;        // the lean instantiations only take chains of exactly N joints

    // Ring bookkeeping.  A "use" is one consumption of one chunk; a tile has U uses and the ring S slots.
    // resident: S = n_chunks, every chunk is loaded once per tile and reused by all K cycles (U = n_chunks);
    // streaming: S < n_chunks, chunks are re-requested every cycle (U = K * n_chunks).
    // The producer cursor (p_*) is always exactly S uses ahead of the consumer, so a refill targets the slot
    // the consumer has just finished with.  Everything advances by increments (no integer division).
    const bool resident = a.n_chunks <= a.n_stages;
    const int S = resident ? a.n_chunks : a.n_stages;
    const int U = resident ? a.n_chunks : a.n_chunks * a.k_cycles;

    if (lane == 0) {
        for (int s = 0; s < kMaxStages + 2; ++s) mbar_init(&bars[s], 1);
        mbar_fence_init();
    }
    __syncwarp();
    int64_t p_unit = unit;
    int p_u = 0, p_chunk = 0;
    if (kTabBytes<T, TAB> == 0 || unit < n_units) {
        issue_qg<T, N, EXT>(a, unit / kSub, 0, region_a, bars_a, lane, nc);
        for (int u = 0; u < S; ++u) {
            issue_obst<T, N, EXT>(a, p_unit / kSub, p_chunk, u, region_a, bars_a, lane);
            if (++p_chunk == a.n_chunks) p_chunk = 0;
            if (++p_u == U) { p_u = 0; p_unit += stride; }
        }
    }
    if constexpr (kTabBytes<T, TAB> != 0) {
        // the sin / cos table is built behind the first tile's copies; the only CTA-wide barrier, passed once by every warp
        // (those without work included) before any can leave
        sincos_table_fill(c.sincos, reinterpret_cast<double2*>(smem + kSmemHeader), (int)threadIdx.x, kBlock);
        __syncthreads();
    }
    int c_stage = 0;
    uint32_t c_phase = 0;

    for (int it = 0; unit < n_units; unit += stride, ++it) {
        const int64_t tile = unit / kSub;
        const int slot = G == 1 ? lane : (int)(unit % kSub) * (32 / G) + (lane / G);     // instance within the tile
        const bool active = (tile << 5) + slot < a.n && ol == 0;     // padding / helper lanes compute, never store
        const int64_t tN = tile * (nc * 32) + slot;             // this instance's slot in a blocked array of nc joint components
        __syncwarp();
        if (unit + stride < n_units) issue_qg<T, N, EXT>(a, (unit + stride) / kSub, (it + 1) & 1, region_a, bars_a, lane, nc);
        // L2 prefetch of the rest of THIS tile.  The two-stage ring can request chunk c + S only when chunk c has been consumed,
        // one chunk-time (~0.4 us) before it is needed -- less than the loaded DRAM latency, so every chunk from S onwards used to
        // stall its warp (long-scoreboard 1.19 per issue on the headline launch).  One cp.async.bulk.prefetch.L2 (SASS UBLKPF.L2)
        // per tile, issued before the tile's arithmetic starts, brings those chunks (contiguous: 8 KB at M = 32) into L2 2 - 3 us
        // ahead, and the ring's copies hit there.  No shared memory, no extra DRAM traffic.  Measured on B200, same-box A/B
        // (profiles/r02u_l2_prefetch_ab.txt): headline launch 110.1 -> 105.4 us (0.955 -> 0.998 of the HBM roofline), 17 joints
        // 127.6 -> 119.1 us (0.815 -> 0.873).  Distance matters: the same instruction one TILE ahead (~7 us) cost 19 % -- the lines
        // were evicted before use and read twice; after the previous tile's repulsor loop (~5 us) it gains nothing, after this
        // tile's kinematic chain (~1.5 us) a third of what it gains here.  Blocks over 32 KB (M = 256) are left to the ring,
        // which is at the copy peak there; a launch of fewer than four tiles per warp is dominated by its start, where every
        // warp's demand copies are queued at once, and skips the prefetch on its first tile (FP64 config 2: -3 % otherwise).
#ifndef VFK_NO_PREFETCH
        if constexpr (G == 1) {
            const int first = S * kChunk;
            const uint32_t bytes = a.n_obst_p > first ? (uint32_t)(a.n_obst_p - first) * 32u * (uint32_t)sizeof(Vec4<T>) : 0u;
            if (!resident && bytes != 0 && bytes <= 32768u && (it > 0 || n_units >= 4 * stride) && lane == 0)
                bulk_prefetch_l2(a.obst + (tile * a.n_obst_p + first) * 32, bytes);
        }
#endif
        mbar_wait_a(bars_a + 8u * (uint32_t)(kMaxStages + (it & 1)), (uint32_t)(it >> 1) & 1u);
        const T* qg = reinterpret_cast<const T*>(region + (size_t)a.n_stages * WS::kStage + (size_t)(it & 1) * WS::kQg) + slot;

    T q[N];
#pragma unroll
    for (int j = 0; j < N; ++j) q[j] = j < nc ? qg[j * 32] : T(0);
    // Long chains (N >= 10) live at the register limit: the lean instantiation re-reads the goal from the staging buffer when
    // the attractor needs it, never materialises the nullspace input or the per-controller velocity vectors, and takes the
    // all-or-nothing limit check as a pass of its own (two cheap dot products per joint recomputed instead of 3 N live values).
    constexpr bool kSlim = LEAN && N >= 10;
    T g[13];
    if constexpr (!kSlim) {
#pragma unroll
        for (int k = 0; k < 13; ++k) g[k] = qg[(N + k) * 32];
    }

    for (int cyc = 0; cyc < a.k_cycles; ++cyc) {
        const bool last = (cyc == a.k_cycles - 1);
        int flags = 0;

        // 1. FK, Jacobian, tool frame
        using W = typename WideOf<T>::type;
        T Jl[N][3], Ja[N][3];
        T Rt[9], dp[3];
        Pos<T> pt;
        {
            W Rw[9], pw[3];
            fk_jacobian<T, N, PAT, TAB>(c, q, Rw, pw, Jl, Ja, nc, sctab);
            if (LEAN || c.tool_identity) {
#pragma unroll
                for (int k = 0; k < 9; ++k) Rt[k] = (T)Rw[k];
                pt.set(pw);
#pragma unroll
                for (int k = 0; k < 3; ++k) dp[k] = T(0);
            } else {
                W ptw[3];
#pragma unroll
                for (int r = 0; r < 3; ++r) {
                    const W off = fma(Rw[3 * r + 0], (W)c.tool[9], fma(Rw[3 * r + 1], (W)c.tool[10], Rw[3 * r + 2] * (W)c.tool[11]));
                    ptw[r] = pw[r] + off;
                    dp[r] = (T)(-off);
#pragma unroll
                    for (int cc = 0; cc < 3; ++cc)
                        Rt[3 * r + cc] = (T)fma(Rw[3 * r + 0], (W)c.tool[cc], fma(Rw[3 * r + 1], (W)c.tool[3 + cc], Rw[3 * r + 2] * (W)c.tool[6 + cc]));
                }
                pt.set(ptw);
            }
        }

        // 2-4. field: attractor, repulsor sum over the staged obstacles, saturation, shift to the flange
        T tw[6];
        {
            T V[3], S0, w[3], acc[3] = {T(0), T(0), T(0)};
            if constexpr (kSlim) {
#pragma unroll
                for (int k = 0; k < 13; ++k) g[k] = qg[(N + k) * 32];
            }
            attract<T>(c, g, Rt, pt, V, S0, w);
            [[maybe_unused]] NegPos2 np2;                               // FP32 packed repulsor: duplicated tool position, paired sums
            [[maybe_unused]] float2 acc2[3] = {make_float2(0.f, 0.f), make_float2(0.f, 0.f), make_float2(0.f, 0.f)};
            if constexpr (sizeof(T) == 4 && !EXT && G == 1) np2.set(pt);
            for (int ch = 0; ch < a.n_chunks; ++ch) {
                const int stage = resident ? ch : c_stage;
                mbar_wait_a(bars_a + 8u * (uint32_t)stage, resident ? (uint32_t)(it & 1) : c_phase);
                const unsigned char* sb = region + (size_t)stage * WS::kStage;
                const Vec4<T>* sp = reinterpret_cast<const Vec4<T>*>(sb);                      // pair p starts at sp + p * 64
                const Vec2<T>* se = reinterpret_cast<const Vec2<T>*>(sb + kChunk * WS::kRow) + slot;
                const int n_here = ch < a.n_full ? kChunk : a.n_rem;                           // obstacles in this chunk
                // one obstacle by its index in the chunk: scalar form (FP64, per-obstacle {safe, order}, cooperative shape)
                auto one = [&](int m, auto order_c) {
                    constexpr int ORD = decltype(order_c)::value;
                    const Vec4<T> o = ObstPairs<T>::load(sp + (m >> 1) * 64, slot, m & 1);
                    T safe_inv = c.obst_safe_inv, order = c.obst_order;
                    if (EXT) { const Vec2<T> e = se[m * 32]; safe_inv = Prec<T>::rcp(e.x); order = e.y; }
                    repel<T, ORD>(o, safe_inv, order, pt, acc);
                };
                if constexpr (G > 1) {
                    // cooperative shape: lane ol of the group takes obstacle ol of this chunk
                    if (ol < n_here) one(ol, std::integral_constant<int, 0>{});
                } else if constexpr (sizeof(T) == 4 && !EXT) {
                    // FP32: two obstacles per step on the packed FP32 pipe; a zero-radius padding slot contributes exactly 0
                    const float4* pl = reinterpret_cast<const float4*>(sb) + slot;
                    if (ch < a.n_full) {
                        auto full_chunk = [&](auto order_c) {
#pragma unroll
                            for (int p = 0; p < kChunk / 2; ++p)
                                repel2<decltype(order_c)::value>(pl[p * 64], pl[p * 64 + 32], c.obst_safe_inv, c.obst_order, np2, acc2);
                        };
                        if (kF32PowChain && c.order_int == 20) full_chunk(std::integral_constant<int, 20>{});
                        else full_chunk(std::integral_constant<int, 0>{});
                    } else {
                        for (int p = 0; p < (a.n_rem + 1) >> 1; ++p)
                            repel2<0>(pl[p * 64], pl[p * 64 + 32], c.obst_safe_inv, c.obst_order, np2, acc2);
                    }
                } else if (ch < a.n_full) {
                    // FP64 with a uniform small-integer decay order: fixed multiplication chain instead of pow()
                    auto full_chunk = [&](auto order_c) {
#pragma unroll
                        for (int m = 0; m < kChunk; ++m) one(m, order_c);
                    };
                    if (sizeof(T) == 8 && !EXT && c.order_int == 20) full_chunk(std::integral_constant<int, 20>{});
                    else if (sizeof(T) == 8 && !EXT && c.order_int == 5) full_chunk(std::integral_constant<int, 5>{});
                    else if (sizeof(T) == 8 && !EXT && c.order_int == 2) full_chunk(std::integral_constant<int, 2>{});
                    else full_chunk(std::integral_constant<int, 0>{});
                } else {
                    for (int m = 0; m < a.n_rem; ++m) one(m, std::integral_constant<int, 0>{});
                }
                // this slot is free again: request the chunk that will occupy it S uses from now
                if (!resident || last) {
                    __syncwarp();
                    if (p_unit < n_units) issue_obst<T, N, EXT>(a, p_unit / kSub, p_chunk, stage, region_a, bars_a, lane);
                    if (++p_chunk == a.n_chunks) p_chunk = 0;
                    if (++p_u == U) { p_u = 0; p_unit += stride; }
                }
                if (!resident && ++c_stage == S) { c_stage = 0; c_phase ^= 1u; }
            }
            if constexpr (sizeof(T) == 4 && !EXT && G == 1) {
#pragma unroll
                for (int k = 0; k < 3; ++k) acc[k] = acc2[k].x + acc2[k].y;
            }
            if constexpr (G > 1) {                          // combine the group's partial repulsor sums
#pragma unroll
                for (int off = 1; off < G; off <<= 1) {
#pragma unroll
                    for (int k = 0; k < 3; ++k) acc[k] += __shfl_xor_sync(0xffffffffu, acc[k], off);
                }
            }
            V[0] = fma(c.obst_force, acc[0], V[0]); V[1] = fma(c.obst_force, acc[1], V[1]); V[2] = fma(c.obst_force, acc[2], V[2]);
            if (!LEAN && a.aux) aux_fields<T>(a.aux, a.n_aux, tile, slot, pt, V);
            T v[3];
            saturate<T>(c, V, S0, v);
            if (!LEAN && last && active && a.twist) {
#pragma unroll
                for (int k = 0; k < 3; ++k) {
                    a.twist[tile * (6 * 32) + k * 32 + slot] = v[k];
                    a.twist[tile * (6 * 32) + (3 + k) * 32 + slot] = w[k];
                }
            }
            tw[0] = v[0] + (w[1] * dp[2] - w[2] * dp[1]);
            tw[1] = v[1] + (w[2] * dp[0] - w[0] * dp[2]);
            tw[2] = v[2] + (w[0] * dp[1] - w[1] * dp[0]);
            tw[3] = w[0]; tw[4] = w[1]; tw[5] = w[2];
        }

        // 5. weighted damped least squares: qdot = Wj Jw^T (Jw Jw^T + l^2 I)^-1 Wt t.  The normal matrix, its Cholesky
        // factor and the triangular solves are carried in W: formed in FP32, A's rounding error (~1e-6 absolute) is 1e-4
        // of lambda^2 = 0.01 and lands directly in the joints' weakest direction.  J itself stays in T.
        using WN = typename WideNE<T>::type;
        const bool unitw = LEAN || c.unit_weights;
        const bool ns_on = LEAN || c.ns_mode != 0;
        const bool ns_proj = LEAN || c.ns_mode == 1;
        const bool share = LEAN || c.share_factor;
        T x[N];                                             // nullspace input (projector mode): known before the factorisation
        auto x_slim = [&](int j) { return c.ns_q0_scale[j] * (q[j] - c.ns_mid[j]); };
        if (ns_proj && !kSlim) {
            if (!LEAN && a.ns_in) {
#pragma unroll
                for (int j = 0; j < N; ++j) x[j] = j < nc ? __ldg(a.ns_in + tN + j * 32) : T(0);
            } else {
#pragma unroll
                for (int j = 0; j < N; ++j) x[j] = c.ns_q0_scale[j] * (q[j] - c.ns_mid[j]);
            }
        }
        WN A[21], invd[6], Jx[6];
#pragma unroll
        for (int r = 0; r < 6; ++r) {
            Jx[r] = WN(0);
#pragma unroll
            for (int s = 0; s <= r; ++s) A[tri(r, s)] = (r == s) ? c.ik_lambda2 : WN(0);
        }
        static_for<0, N>([&](auto jc) {
            constexpr int j = decltype(jc)::value;
            WN col[6] = {(WN)Jl[j][0], (WN)Jl[j][1], (WN)Jl[j][2], (WN)Ja[j][0], (WN)Ja[j][1], (WN)Ja[j][2]};
            // (the short-chain lean tail wants the projector's right-hand side negated: -J x, see dot6x2 there)
            if (ns_proj && share) axpy6(Jx, col, kSlim ? (WN)x_slim(j) : ((LEAN && !kSlim) ? -(WN)x[j] : (WN)x[j]));
            if (!unitw) {
#pragma unroll
                for (int r = 0; r < 6; ++r) col[r] *= (WN)c.w_task[r] * (WN)c.w_joint[j];
            }
            syr6(A, col);
        });
        // FP64 accepts ik_lambda = 0 (the reference's undamped pinv): at a singular posture a pivot of J J^T is zero or, by
        // rounding, negative.  Flooring it relative to the trace keeps the factor finite (the step is then clamped like any
        // other); FP32 requires lambda > 0, whose pivots are >= lambda^2.
        [[maybe_unused]] WN pivot_floor = WN(0);
        if constexpr (sizeof(WN) == 8)
            pivot_floor = WN(1e-28) * (A[tri(0, 0)] + A[tri(1, 1)] + A[tri(2, 2)] + A[tri(3, 3)] + A[tri(4, 4)] + A[tri(5, 5)]) + WN(1e-300);
        chol6<WN>(A, invd, pivot_floor);
        T mix[N];
        [[maybe_unused]] T qd_vf[N], qd_ns[N], qd_jp[N];
        bool nan = false;
        if constexpr (kSlim) {
            T yv[6], yn[6];
            {
                WN y[6];
#pragma unroll
                for (int r = 0; r < 6; ++r) y[r] = (WN)tw[r];
                chol6_fwd<WN>(A, invd, y);                 // (chol6_solve2's register pairs cost ~150 moves at this register count)
                chol6_bwd<WN>(A, invd, y);
                chol6_fwd<WN>(A, invd, Jx);
                chol6_bwd<WN>(A, invd, Jx);
#pragma unroll
                for (int r = 0; r < 6; ++r) { yv[r] = (T)y[r]; yn[r] = (T)Jx[r]; }
            }
            bool bad = false;                               // pass 1: the lookahead check over ALL joints decides for all
#pragma unroll
            for (int j = 0; j < N; ++j) {
                const T cj[6] = {Jl[j][0], Jl[j][1], Jl[j][2], Ja[j][0], Ja[j][1], Ja[j][2]};
                const T d = fma(c.ns_lookahead, dot6_packed(cj, yn, x_slim(j), true), q[j]);
                bad = bad || (d < c.q_lo[j]) || (d > c.q_hi[j]);
            }
            if (bad) flags |= 2;
            const T w1 = bad ? T(0) : c.ns_gain * c.mixer_w[1];
#pragma unroll
            for (int j = 0; j < N; ++j) {                   // pass 2: both controllers' velocities straight into the mixer sum
                const T cj[6] = {Jl[j][0], Jl[j][1], Jl[j][2], Ja[j][0], Ja[j][1], Ja[j][2]};
                mix[j] = fma(dot6_packed(cj, yn, x_slim(j), true), w1, dot6_packed(cj, yv, T(0), false) * c.mixer_w[0]);
            }
        } else if constexpr (LEAN) {
            // Short chains: both solves first, then per joint BOTH products J_j . y (IK) and x_j - J_j . y' (projector) from one
            // packed chain (dot6x2).  Same operations in the same order as the general instantiation below, so asking for one
            // more output never changes a bit of qdot; measured: FP64 config 2 21.2 against 21.8 us per launch, FP32 unchanged.
            T yv[6], yn[6];
            {
                WN y[6];
#pragma unroll
                for (int r = 0; r < 6; ++r) y[r] = (WN)tw[r];
                chol6_solve2(A, invd, y, Jx);
#pragma unroll
                for (int r = 0; r < 6; ++r) { yv[r] = (T)y[r]; yn[r] = (T)Jx[r]; }        // Jx holds -(J x) here
            }
            T raw[N];
            bool bad = false;
#pragma unroll
            for (int j = 0; j < N; ++j) {
                const T cj[6] = {Jl[j][0], Jl[j][1], Jl[j][2], Ja[j][0], Ja[j][1], Ja[j][2]};
                dot6x2(cj, yv, yn, T(0), x[j], &mix[j], &raw[j]);
                const T d = fma(c.ns_lookahead, raw[j], q[j]);
                bad = bad || (d < c.q_lo[j]) || (d > c.q_hi[j]);
            }
            if (bad) flags |= 2;
            const T gain = bad ? T(0) : c.ns_gain;
#pragma unroll
            for (int j = 0; j < N; ++j) mix[j] = fma(raw[j] * gain, c.mixer_w[1], mix[j] * c.mixer_w[0]);
        } else {
            {
                WN y[6];
    #pragma unroll
                for (int r = 0; r < 6; ++r) y[r] = unitw ? (WN)tw[r] : (WN)tw[r] * (WN)c.w_task[r];
                chol6_fwd<WN>(A, invd, y);
                chol6_bwd<WN>(A, invd, y);
                T yt[6];
    #pragma unroll
                for (int r = 0; r < 6; ++r) yt[r] = unitw ? (T)y[r] : (T)(y[r] * (WN)c.w_task[r]);
    #pragma unroll
                for (int j = 0; j < N; ++j) {
                    const T cj[6] = {Jl[j][0], Jl[j][1], Jl[j][2], Ja[j][0], Ja[j][1], Ja[j][2]};
                    const T acc = dot6(cj, yt, T(0), false);
                    qd_vf[j] = unitw ? acc : acc * c.w_joint[j] * c.w_joint[j];
                }
            }
            if constexpr (!LEAN && sizeof(T) == 8) {
                if (c.ik_mode == 1) {
                    // VFK_IK_TRUNCATED: qdot = Wj V diag(f(sigma)) U^T Wt t through a one-sided Jacobi SVD of Jw = Wt J Wj
                    double G[6 * N], yw[6], qdw[N];
    #pragma unroll
                    for (int j = 0; j < N; ++j)
    #pragma unroll
                        for (int r = 0; r < 6; ++r)
                            G[r * N + j] = (double)(r < 3 ? Jl[j][r] : Ja[j][r - 3]) * (unitw ? 1.0 : (double)c.w_task[r] * (double)c.w_joint[j]);
    #pragma unroll
                    for (int r = 0; r < 6; ++r) yw[r] = unitw ? (double)tw[r] : (double)tw[r] * (double)c.w_task[r];
                    ik_truncated(G, N, yw, c.ik_lambda2_d, c.ik_eps, qdw);
    #pragma unroll
                    for (int j = 0; j < N; ++j) qd_vf[j] = unitw ? (T)qdw[j] : (T)(qdw[j] * (double)c.w_joint[j]);
                }
            }

            // 6. nullspace
    #pragma unroll
            for (int j = 0; j < N; ++j) qd_ns[j] = T(0);
            if (ns_on) {
                T raw[N];
                const bool qr = !LEAN && c.ns_qr;
                if (!qr) {
                    // damped projector through the normal equations: raw = x - J^T (J J^T + l^2 I)^-1 (J x)
                    if (!share) {                               // own damping or weighted IK: factor J J^T + ns_lambda^2 I
    #pragma unroll
                        for (int r = 0; r < 6; ++r) {
                            Jx[r] = WN(0);
    #pragma unroll
                            for (int s = 0; s <= r; ++s) A[tri(r, s)] = (r == s) ? c.ns_lambda2 : WN(0);
                        }
                        static_for<0, N>([&](auto jc) {
                            constexpr int j = decltype(jc)::value;
                            const WN col[6] = {(WN)Jl[j][0], (WN)Jl[j][1], (WN)Jl[j][2], (WN)Ja[j][0], (WN)Ja[j][1], (WN)Ja[j][2]};
                            axpy6(Jx, col, (WN)x[j]);
                            syr6(A, col);
                        });
                        if constexpr (sizeof(WN) == 8)
                            pivot_floor = WN(1e-28) * (A[tri(0, 0)] + A[tri(1, 1)] + A[tri(2, 2)] + A[tri(3, 3)] + A[tri(4, 4)] + A[tri(5, 5)]) + WN(1e-300);
                        chol6<WN>(A, invd, pivot_floor);
                    }
                    chol6_fwd<WN>(A, invd, Jx);
                    chol6_bwd<WN>(A, invd, Jx);
                    T yt[6];
    #pragma unroll
                    for (int r = 0; r < 6; ++r) yt[r] = (T)Jx[r];
    #pragma unroll
                    for (int j = 0; j < N; ++j) {
                        const T cj[6] = {Jl[j][0], Jl[j][1], Jl[j][2], Ja[j][0], Ja[j][1], Ja[j][2]};
                        raw[j] = dot6(cj, yt, x[j], true);
                    }
                } else {
                    // the reference's own form (scripts/nullspace:75-117): orthonormal basis u_i of null(J) -- Householder QR of
                    // J^T, error cond(J) * eps, no damping (vfk_nullspace.cuh) -- then either the projector
                    // (I - pinv(J) J) x = sum_i u_i (u_i . x), or the control interface sum_{i < min(4, k)} control_i u_i with
                    // every u_i's sign kept continuous against the previous cycle's vector (ns_lastvec, [min(4, k)][N]).
    #pragma unroll
                    for (int j = 0; j < N; ++j) raw[j] = T(0);
                    if constexpr (!LEAN && ns_null_vectors(N) > 0) {
                        double At[N * 6], tau[6], wv[N];
    #pragma unroll
                        for (int j = 0; j < N; ++j)
    #pragma unroll
                            for (int r = 0; r < 6; ++r) At[j * 6 + r] = (double)(r < 3 ? Jl[j][r] : Ja[j][r - 3]);
                        ns_qr_factor(At, nc, tau);
                        if (ns_proj) {
    #pragma unroll
                            for (int j = 0; j < N; ++j) wv[j] = (double)x[j];
                            ns_qr_project(At, tau, nc, wv);
    #pragma unroll
                            for (int j = 0; j < N; ++j) raw[j] = j < nc ? (T)wv[j] : T(0);
                        } else {
                            const int kk = ns_ctrl_vectors(nc);                      // rows of ns_lastvec
                            double rawd[N];
    #pragma unroll
                            for (int j = 0; j < N; ++j) rawd[j] = 0.0;
    #pragma unroll 1
                            for (int i = 0; i < kk; ++i) {
                                ns_qr_column(At, tau, nc, 6 + i, wv);
                                T* lv = a.ns_lastvec + tile * (kk * nc * 32) + i * (nc * 32) + slot;
                                double dotl = 0.0;
    #pragma unroll
                                for (int j = 0; j < N; ++j) if (j < nc) dotl = fma(wv[j], (double)lv[j * 32], dotl);
                                const double sgn = dotl < 0.0 ? -1.0 : 1.0;      // |s u - last| > |s u + last|  <=>  s u . last < 0
                                const double ci = a.ns_in ? (double)__ldg(a.ns_in + tile * (4 * 32) + i * 32 + slot) : (double)c.ns_control[i];
                                if (active) {
    #pragma unroll
                                    for (int j = 0; j < N; ++j) if (j < nc) lv[j * 32] = (T)(sgn * wv[j]);
                                }
    #pragma unroll
                                for (int j = 0; j < N; ++j) if (j < nc) rawd[j] = fma(sgn * ci, wv[j], rawd[j]);
                            }
                            if (G > 1) __syncwarp();             // a group's lanes re-read what its lane 0 stored
    #pragma unroll
                            for (int j = 0; j < N; ++j) raw[j] = (T)rawd[j];
                        }
                    }
                }
                // all-or-nothing lookahead limit check, then gain
                bool bad = false;
    #pragma unroll
                for (int j = 0; j < N; ++j) {
                    const T d = fma(c.ns_lookahead, raw[j], q[j]);
                    bad = bad || (d < c.q_lo[j]) || (d > c.q_hi[j]);
                }
                if (bad) flags |= 2;
    #pragma unroll
                for (int j = 0; j < N; ++j) qd_ns[j] = bad ? T(0) : raw[j] * c.ns_gain;
            }

            // 7. joint P controller (skipped when nothing can observe it)
    #pragma unroll
            for (int j = 0; j < N; ++j) qd_jp[j] = T(0);
            if (!LEAN && (c.need_jp || a.qdot_jp || a.flags)) {
                bool all_reached = true;
    #pragma unroll
                for (int j = 0; j < N; ++j) {
                    T ref = (a.jp_ref && j < nc) ? a.jp_ref[tN + j * 32] : c.jp_ref[j];
                    const T lo = (a.jp_lo && j < nc) ? __ldg(a.jp_lo + tN + j * 32) : c.q_lo[j];
                    const T hi = (a.jp_lo && j < nc) ? __ldg(a.jp_hi + tN + j * 32) : c.q_hi[j];
                    ref = ref < lo ? lo : (ref > hi ? hi : ref);
                    if (a.jp_lo && a.jp_ref && last && active && j < nc) a.jp_ref[tN + j * 32] = ref;      // the clamp persists
                    const T err = ref - q[j];
                    qd_jp[j] = err * c.jp_kp;
                    all_reached = all_reached && (err < c.jp_delta);
                }
                if (all_reached) flags |= 1;
            }

            // 8-9. mixer, clamp
    #pragma unroll
            for (int j = 0; j < N; ++j) {
                T m = T(0);
                m = fma(qd_vf[j], c.mixer_w[0], m);
                m = fma(qd_ns[j], c.mixer_w[1], m);
                m = fma(qd_jp[j], c.mixer_w[2], m);
                if (!LEAN) nan = nan || (qd_vf[j] != qd_vf[j]) || (qd_ns[j] != qd_ns[j]) || (qd_jp[j] != qd_jp[j]);
                mix[j] = m;
            }
    #pragma unroll
            for (int e = 0; e < 3; ++e)
                if (!LEAN && a.ext_cmd[e]) {
    #pragma unroll
                    for (int j = 0; j < N; ++j) {
                        const T x = j < nc ? __ldg(a.ext_cmd[e] + tN + j * 32) : T(0);
                        nan = nan || (x != x);
                        mix[j] = fma(x, c.mixer_w[3 + e], mix[j]);
                    }
                }
        }
        T lead = T(0);
#pragma unroll
        for (int j = 0; j < N; ++j) lead = Prec<T>::fmax_(lead, Prec<T>::fabs_(mix[j]));
        if constexpr (!LEAN || sizeof(T) == 8) {
            // never integrate a non-finite step (a NaN in q or in an input port, an overflow): command zero and say so
            T z = T(0);
#pragma unroll
            for (int j = 0; j < N; ++j) z = fma(mix[j], T(0), z);
            if (z != T(0)) {
                nan = true;
                lead = T(0);
#pragma unroll
                for (int j = 0; j < N; ++j) mix[j] = T(0);
            }
        }
        if (nan) flags |= 4;
        T ratio = T(1);
        if (lead > c.max_vel) { ratio = Prec<T>::div(c.max_vel, lead); flags |= 8; }
        if (!LEAN && c.shoulder_clamp) {
            // the reference keeps one `ratio` variable for both clamps: without a shoulder hit the leading ratio is
            // applied twice (bug-compatible, see include/vfk.h)
            const T sh = mix[0] * ratio;
            T r2 = ratio;
            if (sh > c.shoulder_pos) r2 = Prec<T>::fabs_(Prec<T>::div(c.shoulder_pos, sh));
            else if (sh < c.shoulder_neg) r2 = Prec<T>::fabs_(Prec<T>::div(c.shoulder_neg, sh));
            ratio *= r2;
        }

        if (last && active) {
            if (!LEAN && a.qdot_vf) {
#pragma unroll
                for (int j = 0; j < N; ++j) if (j < nc) a.qdot_vf[tN + j * 32] = qd_vf[j];
            }
            if (!LEAN && a.qdot_ns) {
#pragma unroll
                for (int j = 0; j < N; ++j) if (j < nc) a.qdot_ns[tN + j * 32] = qd_ns[j];
            }
            if (!LEAN && a.qdot_jp) {
#pragma unroll
                for (int j = 0; j < N; ++j) if (j < nc) a.qdot_jp[tN + j * 32] = qd_jp[j];
            }
            if (LEAN || a.qdot) {
                T* o = a.qdot_ld ? a.qdot + (tile << 5) + slot : a.qdot + tN;
                const int64_t rs = a.qdot_ld ? a.qdot_ld : 32;
#pragma unroll
                for (int j = 0; j < N; ++j) if (j < nc) o[j * rs] = mix[j] * ratio;
                if (a.qdot_ld && a.qdot_dev) {
#pragma unroll
                    for (int j = 0; j < N; ++j) if (j < nc) a.qdot_dev[tN + j * 32] = mix[j] * ratio;
                }
            }
            if (!LEAN && a.cmd) {
#pragma unroll
                for (int j = 0; j < N; ++j) {
                    if (j >= nc) continue;
                    const T qd = mix[j] * ratio;
                    const T qc = a.q_cmded ? __ldg(a.q_cmded + tN + j * 32) : q[j];
                    a.cmd[tN + j * 32] = c.direct_control ? qd : (-qc + q[j] + qd);
                }
            }
            if (!LEAN && a.pose) {
#pragma unroll
                for (int k = 0; k < 9; ++k) a.pose[tile * (12 * 32) + k * 32 + slot] = Rt[k];
#pragma unroll
                for (int k = 0; k < 3; ++k) a.pose[tile * (12 * 32) + (9 + k) * 32 + slot] = pt.hi[k];
            }
            if (!LEAN && a.flags) a.flags[(tile << 5) + slot] = flags;
        }
        // 10. plant
        if (c.integrate) {
#pragma unroll
            for (int j = 0; j < N; ++j) q[j] = fma(c.dt, mix[j] * ratio, q[j]);
        }
    }
    if (active) {
        if (c.integrate || a.q_src) {                  // direct host I/O: the session's device copy of q follows the caller's
#pragma unroll
            for (int j = 0; j < N; ++j) if (j < nc) a.q[tN + j * 32] = q[j];
        }
    }
    }   // tile loop
}

// ------------------------------------------------------------------------------ small kernels
// Field query at given tool poses (scripts/vf:469-503); low-rate visualisation path, plain loads.
template <typename T>
__global__ void __launch_bounds__(kSmallBlock)
vfk_field_kernel(const __grid_constant__ KConst<T> c, const T* __restrict__ pose, const T* __restrict__ goal,
                 const Vec4<T>* __restrict__ obst, const Vec2<T>* __restrict__ obst_ext, const T* __restrict__ aux, int n_aux,
                 T* __restrict__ twist, int64_t n, int n_obst) {
    const int64_t i = (int64_t)blockIdx.x * kSmallBlock + threadIdx.x;
    if (i >= n) return;
    const int64_t tile = i >> 5;
    const int lane = (int)(i & 31);
    T Rt[9], g[13];
    Pos<T> pt;
#pragma unroll
    for (int k = 0; k < 9; ++k) Rt[k] = pose[(tile * 12 + k) * 32 + lane];
#pragma unroll
    for (int k = 0; k < 3; ++k) { pt.hi[k] = pose[(tile * 12 + 9 + k) * 32 + lane]; pt.lo[k] = T(0); }
#pragma unroll
    for (int k = 0; k < 13; ++k) g[k] = goal[(tile * 13 + k) * 32 + lane];
    T V[3], S0, w[3], acc[3] = {T(0), T(0), T(0)}, v[3];
    attract<T>(c, g, Rt, pt, V, S0, w);
    const int n_obst_p = (n_obst + 1) & ~1;
    for (int m = 0; m < n_obst; ++m) {
        const Vec4<T> o = ObstPairs<T>::load(obst + (tile * n_obst_p + (m & ~1)) * 32, lane, m & 1);
        T safe_inv = c.obst_safe_inv, order = c.obst_order;
        if (obst_ext) { const Vec2<T> e = obst_ext[(tile * n_obst + m) * 32 + lane]; safe_inv = Prec<T>::rcp(e.x); order = e.y; }
        repel<T>(o, safe_inv, order, pt, acc);
    }
    V[0] = fma(c.obst_force, acc[0], V[0]); V[1] = fma(c.obst_force, acc[1], V[1]); V[2] = fma(c.obst_force, acc[2], V[2]);
    if (aux) aux_fields<T>(aux, n_aux, tile, lane, pt, V);
    saturate<T>(c, V, S0, v);
#pragma unroll
    for (int k = 0; k < 3; ++k) { twist[(tile * 6 + k) * 32 + lane] = v[k]; twist[(tile * 6 + 3 + k) * 32 + lane] = w[k]; }
}

struct MixArgs {
    const void* cmds[8];
    double w[8];
    int n_ports;
};

// out(c, i) = sum_p w_p * cmds[p](c, i)  (src/command_mixer.py:78-82), NaN report (:71-75).  All arrays
// share one blocked layout, so the sum is element-wise over the flat buffers (n_channels * 32 * tiles elements).
template <typename T>
__global__ void __launch_bounds__(256)
vfk_mix_kernel(const __grid_constant__ MixArgs m, T* __restrict__ out, int32_t* __restrict__ nan_flags,
               int n_channels, int64_t n_tiles) {
    const int64_t e = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (e >= n_tiles * n_channels * 32) return;
    T acc = T(0);
    bool nan = false;
#pragma unroll
    for (int p = 0; p < 8; ++p) {
        if (p < m.n_ports && m.cmds[p]) {
            const T x = static_cast<const T*>(m.cmds[p])[e];
            nan = nan || (x != x);
            acc = fma(x, (T)m.w[p], acc);
        }
    }
    out[e] = acc;
    if (nan_flags && nan) {
        const int64_t tile = e / (n_channels * 32);
        atomicOr(&nan_flags[(tile << 5) + (e & 31)], 4);
    }
}

// LWR_Bridge.set_vel (scripts/bridge:188-203) on blocked arrays: leading-joint clamp and command forming.
template <typename T>
__global__ void __launch_bounds__(256)
vfk_set_vel_kernel(const T* __restrict__ qdot, const T* __restrict__ q, const T* __restrict__ q_cmded, T* __restrict__ cmd,
                   T* __restrict__ qdot_lim, T max_vel, int direct, int shoulder_clamp, T shoulder_pos, T shoulder_neg,
                   int n_channels, int64_t n) {
    const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (i >= n) return;
    const int64_t base = (i >> 5) * (n_channels * 32) + (i & 31);
    T lead = T(0);
    for (int c = 0; c < n_channels; ++c) lead = Prec<T>::fmax_(lead, Prec<T>::fabs_(qdot[base + c * 32]));
    T ratio = lead > max_vel ? max_vel / lead : T(1);
    if (shoulder_clamp) {                      // Powercube_Bridge.set_vel (scripts/bridge:295-303), see the cycle kernel
        const T sh = qdot[base] * ratio;
        T r2 = ratio;
        if (sh > shoulder_pos) r2 = Prec<T>::fabs_(shoulder_pos / sh);
        else if (sh < shoulder_neg) r2 = Prec<T>::fabs_(shoulder_neg / sh);
        ratio *= r2;
    }
    for (int c = 0; c < n_channels; ++c) {
        const T v = qdot[base + c * 32] * ratio;
        if (qdot_lim) qdot_lim[base + c * 32] = v;
        const T qc = q_cmded ? q_cmded[base + c * 32] : q[base + c * 32];
        cmd[base + c * 32] = direct ? v : (-qc + q[base + c * 32] + v);
    }
}

// ------------------------------------------------------------------------------ monitoring (SURVEY.md section 8, row f1)
// Tracking-error diagnostics of scripts/vf:349-428 and the distance monitor of scripts/monitor_distance:76-84,148-219,
// one thread per instance, state carried between calls in two blocked arrays:
//   sf [32]: previous tool pose (12), the three previous commanded twists (3 x 6, oldest first), last track errors (2)
//   si [6] : cycles seen, xyz state ring (2 x 32 bits), rot state ring (2 x 32 bits), votes in the ring
// Outputs: track [8] = the 7 doubles + the arm_tracking int of /vectorField/track_error;
//          dist [2]  = distance to the goal in metres and degrees (/dmonitor/distOut, object 0);
//          state [2] = majority tracking state over the last 20 cycles (0 on goal, 1 follow, 2 not follow) for xyz / rot,
//                      -1 until 21 samples have been seen.
template <typename T>
__device__ __forceinline__ void rotvec_between(const T (&Ra)[9], const T (&Rb)[9], T (&out)[3]) {
    // KDL diff(Fa, Fb).rot = Ra * rotvec(Ra^T Rb)
    T E[9];
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
        for (int cc = 0; cc < 3; ++cc)
            E[3 * r + cc] = Ra[r] * Rb[cc] + Ra[3 + r] * Rb[3 + cc] + Ra[6 + r] * Rb[6 + cc];
    T qw, qx, qy, qz;
    rot_to_quat<T>(E, qw, qx, qy, qz);
    const T n2 = qx * qx + qy * qy + qz * qz;
    const T n = Prec<T>::sqrt_(n2);
    const T ang = T(2) * Prec<T>::atan2_(n, qw);
    const T sc = n > T(0) ? Prec<T>::div(ang, n) : T(0);
    const T lx = qx * sc, ly = qy * sc, lz = qz * sc;
    out[0] = Ra[0] * lx + Ra[1] * ly + Ra[2] * lz;
    out[1] = Ra[3] * lx + Ra[4] * ly + Ra[5] * lz;
    out[2] = Ra[6] * lx + Ra[7] * ly + Ra[8] * lz;
}

__device__ __forceinline__ int ring_majority(uint32_t lo, uint32_t hi) {
    // 20 two-bit states packed from bit 0; first maximum in the order on goal, follow, not follow
    int cnt[3] = {0, 0, 0};
    uint64_t bits = ((uint64_t)hi << 32) | lo;
#pragma unroll
    for (int k = 0; k < 20; ++k) { const int s = (int)((bits >> (2 * k)) & 3u); if (s < 3) ++cnt[s]; }
    int best = 0;
    if (cnt[1] > cnt[best]) best = 1;
    if (cnt[2] > cnt[best]) best = 2;
    return best;
}

template <typename T>
__global__ void __launch_bounds__(kSmallBlock)
vfk_monitor_kernel(const T* __restrict__ pose, const T* __restrict__ twist, const T* __restrict__ goal, T* __restrict__ sf,
                   int32_t* __restrict__ si, T* __restrict__ track, T* __restrict__ dist, int32_t* __restrict__ state, int64_t n) {
    const int64_t i = (int64_t)blockIdx.x * kSmallBlock + threadIdx.x;
    if (i >= n) return;
    const int64_t tile = i >> 5;
    const int lane = (int)(i & 31);
    auto F = [&](const T* base, int comps, int c) -> const T& { return base[(tile * comps + c) * 32 + lane]; };
    T R[9], p[3], cmd[6], g[13];
#pragma unroll
    for (int k = 0; k < 9; ++k) R[k] = F(pose, 12, k);
#pragma unroll
    for (int k = 0; k < 3; ++k) p[k] = F(pose, 12, 9 + k);
#pragma unroll
    for (int k = 0; k < 6; ++k) cmd[k] = F(twist, 6, k);
#pragma unroll
    for (int k = 0; k < 13; ++k) g[k] = F(goal, 13, k);
    T* sfi = sf + tile * (32 * 32) + lane;
    int32_t* sii = si + tile * (6 * 32) + lane;
    const int seen = sii[0] + 1;                       // frames appended so far, this one included (scripts/vf:354)

    // ---- tracking diagnostics (scripts/vf:349-428): needs 6 frames and the command of 3 cycles ago
    T te_xyz = T(0), te_rot = T(0);
    bool have_te = false;
    if (seen > 5) {
        T Rp[9], pp[3], old[6];
#pragma unroll
        for (int k = 0; k < 9; ++k) Rp[k] = sfi[k * 32];
#pragma unroll
        for (int k = 0; k < 3; ++k) pp[k] = sfi[(9 + k) * 32];
#pragma unroll
        for (int k = 0; k < 6; ++k) old[k] = sfi[(12 + k) * 32];       // oldest of the 4 buffered commands
        const T ev[3] = {p[0] - pp[0], p[1] - pp[1], p[2] - pp[2]};
        T er[3];
        rotvec_between<T>(Rp, R, er);
        auto unit_dot = [&](const T (&a3)[3], const T* b3, T& amag, T& bmag) {
            amag = Prec<T>::sqrt_(a3[0] * a3[0] + a3[1] * a3[1] + a3[2] * a3[2]);
            bmag = Prec<T>::sqrt_(b3[0] * b3[0] + b3[1] * b3[1] + b3[2] * b3[2]);
            T ua[3] = {T(1), T(0), T(0)}, ub[3] = {T(1), T(0), T(0)};
            if (amag > T(0)) { ua[0] = Prec<T>::div(a3[0], amag); ua[1] = Prec<T>::div(a3[1], amag); ua[2] = Prec<T>::div(a3[2], amag); }
            if (bmag > T(0)) { ub[0] = Prec<T>::div(b3[0], bmag); ub[1] = Prec<T>::div(b3[1], bmag); ub[2] = Prec<T>::div(b3[2], bmag); }
            T d = ub[0] * ua[0] + ub[1] * ua[1] + ub[2] * ua[2];
            return Prec<T>::fmin_(T(1), Prec<T>::fmax_(T(-1), d));
        };
        T ext_vel_mag, cmd_vel_mag, ext_rot_mag, cmd_rot_mag;
        const T vel_dot = unit_dot(ev, old, ext_vel_mag, cmd_vel_mag);
        const T rot_dot = unit_dot(er, old + 3, ext_rot_mag, cmd_rot_mag);
        te_xyz = Prec<T>::fabs_((T)acos((double)vel_dot));
        te_rot = Prec<T>::fabs_((T)acos((double)rot_dot));
        const T loop_freq = T(150), tracking_th = T(0.10);
        const T ext_vel_corr = ext_vel_mag * loop_freq, ext_rot_corr = ext_rot_mag * loop_freq;
        const T cmd_rot_corr = cmd_rot_mag / T(5), cmd_vel_corr = cmd_vel_mag;
        const T ext_int_diff = Prec<T>::fabs_((cmd_vel_corr + cmd_rot_corr) - (ext_vel_corr + ext_rot_corr));
        have_te = true;
        if (track) {
            T* t = track + tile * (8 * 32) + lane;
            t[0] = te_xyz; t[32] = te_rot; t[64] = ext_vel_corr; t[96] = ext_rot_corr; t[128] = cmd_vel_corr;
            t[160] = cmd_rot_corr; t[192] = ext_int_diff; t[224] = ext_int_diff < tracking_th ? T(1) : T(0);
        }
    } else if (track) {
        T* t = track + tile * (8 * 32) + lane;
#pragma unroll
        for (int k = 0; k < 8; ++k) t[k * 32] = T(0);
    }
    // the monitor keeps the last track error it received (scripts/monitor_distance:156-159): carry it in sf[30..31]
    if (have_te) { sfi[30 * 32] = te_xyz; sfi[31 * 32] = te_rot; } else { te_xyz = sfi[30 * 32]; te_rot = sfi[31 * 32]; }

    // ---- distance monitor (scripts/monitor_distance:160-219), object 0 = the goal
    const T dx = p[0] - g[9], dy = p[1] - g[10], dz = p[2] - g[11];
    const T dxyz = Prec<T>::sqrt_(dx * dx + dy * dy + dz * dz);
    T gr[9];
#pragma unroll
    for (int k = 0; k < 9; ++k) gr[k] = g[k];
    T rv[3];
    rotvec_between<T>(R, gr, rv);
    const T ddeg = T(180.0 / 3.14159265358979323846) * Prec<T>::sqrt_(rv[0] * rv[0] + rv[1] * rv[1] + rv[2] * rv[2]);
    if (dist) { dist[tile * (2 * 32) + lane] = dxyz; dist[tile * (2 * 32) + 32 + lane] = ddeg; }
    int xs = 0, rs = 0;                                                // 0 on goal, 1 follow, 2 not follow
    if (dxyz > T(0.02) && te_xyz > T(0.1)) xs = 2;
    if (dxyz > T(0.02) && te_xyz < T(0.1)) xs = 1;
    if (dxyz < T(0.02)) xs = 0;
    if (ddeg > T(1.0) && te_rot > T(0.1)) rs = 2;
    if (ddeg > T(1.0) && te_rot < T(0.1)) rs = 1;
    if (ddeg < T(1.0)) rs = 0;
    uint64_t xr = ((uint64_t)(uint32_t)sii[2 * 32] << 32) | (uint32_t)sii[1 * 32];
    uint64_t rr = ((uint64_t)(uint32_t)sii[4 * 32] << 32) | (uint32_t)sii[3 * 32];
    const uint64_t mask40 = (1ull << 40) - 1;
    xr = ((xr << 2) | (uint64_t)xs) & mask40;                          // newest state in the low bits, 20 states kept
    rr = ((rr << 2) | (uint64_t)rs) & mask40;
    const int votes = sii[5 * 32] + 1;
    if (state) {
        int sx = -1, sr = -1;
        if (votes > 20) { sx = ring_majority((uint32_t)xr, (uint32_t)(xr >> 32)); sr = ring_majority((uint32_t)rr, (uint32_t)(rr >> 32)); }
        state[tile * (2 * 32) + lane] = sx;
        state[tile * (2 * 32) + 32 + lane] = sr;
    }
    // ---- state update: shift the command ring, store the pose
    sii[0] = seen; sii[1 * 32] = (int32_t)(uint32_t)xr; sii[2 * 32] = (int32_t)(uint32_t)(xr >> 32);
    sii[3 * 32] = (int32_t)(uint32_t)rr; sii[4 * 32] = (int32_t)(uint32_t)(rr >> 32); sii[5 * 32] = votes;
#pragma unroll
    for (int k = 0; k < 9; ++k) sfi[k * 32] = R[k];
#pragma unroll
    for (int k = 0; k < 3; ++k) sfi[(9 + k) * 32] = p[k];
#pragma unroll
    for (int k = 0; k < 12; ++k) sfi[(12 + k) * 32] = sfi[(18 + k) * 32];
#pragma unroll
    for (int k = 0; k < 6; ++k) sfi[(24 + k) * 32] = cmd[k];
}

// ------------------------------------------------------------------------------ layout conversion
// dense SoA [C][dense_ld >= n] (element: scalar, Vec2 or Vec4 of T)  <->  tile-blocked [tile][C][32].
template <typename V>
__global__ void __launch_bounds__(256)
vfk_pack_kernel(const V* __restrict__ dense, int64_t dense_ld, V* __restrict__ blocked, int C, int64_t n, int64_t n_tiles) {
    const int64_t e = (int64_t)blockIdx.x * 256 + threadIdx.x;          // index into the blocked array
    if (e >= n_tiles * C * 32) return;
    const int lane = (int)(e & 31);
    const int64_t tc = e >> 5;
    const int64_t tile = tc / C;
    const int cidx = (int)(tc - tile * C);
    const int64_t i = (tile << 5) + lane;
    V zero;
    memset(&zero, 0, sizeof zero);
    blocked[e] = i < n ? dense[(int64_t)cidx * dense_ld + i] : zero;
}

template <typename V>
__global__ void __launch_bounds__(256)
vfk_unpack_kernel(const V* __restrict__ blocked, V* __restrict__ dense, int64_t dense_ld, int C, int64_t n, int64_t n_tiles) {
    const int64_t e = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (e >= n_tiles * C * 32) return;
    const int lane = (int)(e & 31);
    const int64_t tc = e >> 5;
    const int64_t tile = tc / C;
    const int cidx = (int)(tc - tile * C);
    const int64_t i = (tile << 5) + lane;
    if (i < n) dense[(int64_t)cidx * dense_ld + i] = blocked[e];
}

// Obstacles: dense [M][dense_ld >= n] of {x, y, z, radius}  <->  the pair-interleaved blocked array (ObstPairs), one thread
// per (tile, pair, lane).  Packing zero-fills the padding lanes of the last tile and the padding slot of an odd M.
template <typename T>
__global__ void __launch_bounds__(256)
vfk_pack_obst_kernel(const Vec4<T>* __restrict__ dense, int64_t dense_ld, Vec4<T>* __restrict__ blocked, int M, int64_t n, int64_t n_tiles) {
    const int M2 = (M + 1) >> 1;
    const int64_t e = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (e >= n_tiles * M2 * 32) return;
    const int lane = (int)(e & 31);
    const int64_t tp = e >> 5;
    const int64_t tile = tp / M2;
    const int p = (int)(tp - tile * M2);
    const int64_t i = (tile << 5) + lane;
    Vec4<T> zero;
    memset(&zero, 0, sizeof zero);
#pragma unroll
    for (int s = 0; s < 2; ++s) {
        const int m = 2 * p + s;
        ObstPairs<T>::store(blocked + (tile * M2 + p) * 64, lane, s, (i < n && m < M) ? dense[(int64_t)m * dense_ld + i] : zero);
    }
}

template <typename T>
__global__ void __launch_bounds__(256)
vfk_unpack_obst_kernel(const Vec4<T>* __restrict__ blocked, Vec4<T>* __restrict__ dense, int64_t dense_ld, int M, int64_t n, int64_t n_tiles) {
    const int M2 = (M + 1) >> 1;
    const int64_t e = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (e >= n_tiles * M2 * 32) return;
    const int lane = (int)(e & 31);
    const int64_t tp = e >> 5;
    const int64_t tile = tp / M2;
    const int p = (int)(tp - tile * M2);
    const int64_t i = (tile << 5) + lane;
    if (i >= n) return;
#pragma unroll
    for (int s = 0; s < 2; ++s) {
        const int m = 2 * p + s;
        if (m < M) dense[(int64_t)m * dense_ld + i] = ObstPairs<T>::load(blocked + (tile * M2 + p) * 64, lane, s);
    }
}

}  // namespace vfk
