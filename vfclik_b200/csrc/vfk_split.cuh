// vfk_split.cuh -- the lane-split shape of the fused control-cycle kernel: L lanes cooperate on ONE instance.
//
// The one-thread-per-instance kernel (vfk_kernels.cuh) keeps the whole 6 x N Jacobian of its instance in registers.  For a
// 17-joint chain that is 102 registers before anything else (248 in all: 2 CTAs per SM, 8 warps, latency-bound at 0.58 of
// the HBM roofline), and in FP64 even 7 joints cost 234.  Here the JOINTS of an instance are split over L = 2 lanes:
//
//   * lane h of an instance owns joints [h * NL, (h + 1) * NL), NL = ceil(N / L): their angles, their Jacobian columns,
//     their share of J J^T, J x and J^T y, their limits, their outputs -- a warp takes 32 / L instances of a tile;
//   * forward kinematics runs as L partial chains in parallel, each from the identity (lane 0: from the base frame); one
//     shuffle exchange of the partial frames hands lane 1 the frame its partial chain starts from and both lanes the
//     flange frame; joint axes and origins are then moved to the base frame;
//   * the 21 + 6 partial sums of J J^T and J x are added across the L lanes by xor-shuffles; the 6 x 6 Cholesky and the
//     triangular solves are repeated by every lane (same instructions whether one lane or 32 execute them);
//   * the obstacle pairs of a chunk are dealt round-robin to the L lanes and the three partial repulsor sums shuffled
//     together (north_star's "reduced with warp shuffles"); the all-or-nothing limit check and the leading-joint clamp
//     combine their per-lane verdicts the same way.
//
// The shape runs the FP64 17-joint chain only (vfk_launch.cuh: split_ok): every other chain and the FP32 mode measured
// slower here than in the one-thread-per-instance kernel, and four lanes per instance slower than two (DESIGN.md 4.2).
//
// Staging: a warp needs the rows of HALF a tile -- 32 / L lanes of every 32-lane row.  Those are strided
// pieces, so the 1-D bulk copies of the full-tile kernel would become one copy per row; instead the arrays are described to
// the TMA unit as 3-D tensors [tile][row][lane] (cuTensorMapEncodeTiled on the host, one descriptor per array per launch)
// and ONE cp.async.bulk.tensor (SASS UTMALDG) per stage gathers the box {32 / L lanes, rows of the chunk, 1 tile} into a
// dense shared-memory tile.  Same mbarrier ring as the full-tile kernel, one tile-part ahead of the arithmetic.
//
// Scope: the production ("lean") shape -- identity tool frame and IK weights, projector nullspace on the built-in
// limit-avoidance gradient sharing the IK factor, q / qdot the only outputs -- for chains in the generic pattern.  Anything
// else runs the one-thread-per-instance kernel.  Robot constants are indexed by a lane-dependent joint number here, which
// the constant bank serialises; they are copied once per CTA into a shared-memory table instead.
#pragma once
#include <cuda.h>

#include "vfk_kernels.cuh"

namespace vfk {

struct alignas(64) SplitMaps {
    CUtensorMap q, goal, obst;
};

constexpr int kSplitTabJoints = kMaxJ + 3;       // L * NL can exceed N by up to L - 1 padding joints
constexpr int kSplitLanes = 2;                   // L: lanes per instance

// Per-joint constants of a DH chain: tip = {cos alpha, sin alpha, tx, ty, tz} (RotX(alpha) and the translation), limits and
// the limit-avoidance gradient's scale / centre.  Padding joints (index >= N): identity tip, zeros.
template <typename T>
struct SplitTab {
    T tip[kSplitTabJoints][6];
    T lim[kSplitTabJoints][4];                   // q_lo, q_hi, ns_scale, ns_mid
};

__host__ __device__ constexpr uint32_t round128(uint32_t x) { return (x + 127u) & ~127u; }

template <typename T, int N>
struct SplitShape {
    static constexpr int L = kSplitLanes;
    static constexpr int NL = (N + L - 1) / L;                                  // joints per lane
    static constexpr int SUB = 32 / L;                                          // instances per warp
    static constexpr uint32_t kRowBytes = SUB * 16;                             // one obstacle plane row of the warp's instances
    static constexpr int kRowsPerChunk = kChunk / 2 * ObstPairs<T>::kPlanes;    // FP32: 8, FP64: 16
    static constexpr uint32_t kStage = kRowsPerChunk * kRowBytes;
    static constexpr uint32_t kQ = round128(N * SUB * sizeof(T));
    static constexpr uint32_t kG = round128(13 * SUB * sizeof(T));
    static constexpr uint32_t kQg = kQ + kG;
    static constexpr int kBars = kMaxStages + 2;
    static constexpr uint32_t kTab = round128(sizeof(SplitTab<T>));
    __host__ __device__ static constexpr uint32_t warp_bytes(int n_stages) { return n_stages * kStage + 2 * kQg; }
};

// One box of a 3-D tensor, global -> shared, completing on an mbarrier (SASS UTMALDG).
__device__ __forceinline__ void tma_box3(void* dst_smem, const CUtensorMap* map, int c0, int c1, int c2, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];" ::"r"(
            smem_u32(dst_smem)),
        "l"(map), "r"(c0), "r"(c1), "r"(c2), "r"(smem_u32(bar))
        : "memory");
}

template <typename T>
__device__ __forceinline__ void frame_mul(const T (&Ra)[9], const T (&pa)[3], const T (&Rb)[9], const T (&pb)[3], T (&R)[9], T (&p)[3]) {
#pragma unroll
    for (int r = 0; r < 3; ++r) {
#pragma unroll
        for (int cc = 0; cc < 3; ++cc)
            R[3 * r + cc] = fma(Ra[3 * r + 0], Rb[cc], fma(Ra[3 * r + 1], Rb[3 + cc], Ra[3 * r + 2] * Rb[6 + cc]));
        p[r] = fma(Ra[3 * r + 0], pb[0], fma(Ra[3 * r + 1], pb[1], fma(Ra[3 * r + 2], pb[2], pa[r])));
    }
}

// 2 resident CTAs per SM: 255 registers, no spills for 17 joints (3 CTAs / 168 registers spill and measured equal to the solo kernel)
template <typename T, int N>
__global__ void __launch_bounds__(kBlock, 2)
vfk_split_kernel(const __grid_constant__ KConst<T> c, const __grid_constant__ KArgs<T> a, const __grid_constant__ SplitMaps maps) {
    static_assert(sizeof(T) == 8, "the lane-split shape is FP64 only");
    using SH = SplitShape<T, N>;
    constexpr int L = SH::L, NL = SH::NL, SUB = SH::SUB;
    extern __shared__ __align__(128) unsigned char smem[];
    const int lane = threadIdx.x & 31;
    const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);     // tells the compiler it is warp-uniform: no divergence guards around the shuffles
    const int h = lane / SUB;                                    // which part of the chain this lane owns
    const int sl = lane % SUB;                                   // instance within the warp
    const int j0 = h * NL;                                       // first joint of this lane
    constexpr int nc = N;                                        // chains of exactly N joints only (the host checks)
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem) + warp * SH::kBars;
    SplitTab<T>* tab = reinterpret_cast<SplitTab<T>*>(smem + kSmemHeader);
    unsigned char* region = smem + kSmemHeader + SH::kTab + (size_t)warp * SH::warp_bytes(a.n_stages);

    // per-joint robot constants -> shared memory
    for (int j = threadIdx.x; j < L * NL; j += kBlock) {
        const bool real = j < N;
        tab->tip[j][0] = real ? c.tip[j][4] : T(1);
        tab->tip[j][1] = real ? c.tip[j][7] : T(0);
        tab->tip[j][2] = real ? c.tip[j][9] : T(0);
        tab->tip[j][3] = real ? c.tip[j][10] : T(0);
        tab->tip[j][4] = real ? c.tip[j][11] : T(0);
        tab->tip[j][5] = T(0);
        tab->lim[j][0] = real ? c.q_lo[j] : T(0);
        tab->lim[j][1] = real ? c.q_hi[j] : T(0);
        tab->lim[j][2] = real ? c.ns_q0_scale[j] : T(0);
        tab->lim[j][3] = real ? c.ns_mid[j] : T(0);
    }
    __syncthreads();
    const T (*tipb)[6] = tab->tip + j0;   // this lane's joints: compile-time offsets from here on
    const T (*limb)[4] = tab->lim + j0;
    // joint k of this lane exists unless it is one of the last lane's padding slots (N is not a multiple of L)
    auto real_joint = [&](int k) { return k < N - (L - 1) * NL || h != L - 1; };

    const int64_t n_tiles = (a.n + 31) >> 5;
    const int64_t n_units = n_tiles * L;                         // a unit = the 32 / L instances one warp takes at a time
    const int64_t stride = (int64_t)gridDim.x * (kBlock / 32);
    int64_t unit = (int64_t)blockIdx.x * (kBlock / 32) + warp;
    if (unit >= n_units) return;

    const bool resident = a.own.chunks <= a.n_stages;
    const int S = resident ? a.own.chunks : a.n_stages;
    const int U = resident ? a.own.chunks : a.own.chunks * a.k_cycles;
    const uint32_t qg_bytes = (uint32_t)(nc + 13) * SUB * sizeof(T);

    auto issue_qg = [&](int64_t u, int buf) {
        if (lane == 0) {
            unsigned char* dst = region + (size_t)a.n_stages * SH::kStage + (size_t)buf * SH::kQg;
            const int tile = (int)(u / L), col = (int)(u % L) * SUB;
            mbar_arrive_expect_tx(&bars[kMaxStages + buf], qg_bytes);
            tma_box3(dst, &maps.q, col, 0, tile, &bars[kMaxStages + buf]);
            tma_box3(dst + SH::kQ, &maps.goal, col, 0, tile, &bars[kMaxStages + buf]);
        }
    };
    auto issue_obst = [&](int64_t u, int chunk, int stage) {
        if (lane == 0) {
            const int tile = (int)(u / L), col = (int)(u % L) * (int)(SH::kRowBytes / sizeof(T));
            mbar_arrive_expect_tx(&bars[stage], SH::kStage);     // the box is always whole: rows past the tile's last are zero-filled
            tma_box3(region + (size_t)stage * SH::kStage, &maps.obst, col, chunk * SH::kRowsPerChunk, tile, &bars[stage]);
        }
    };

    if (lane == 0) {
        for (int s = 0; s < kMaxStages + 2; ++s) mbar_init(&bars[s], 1);
        mbar_fence_init();
    }
    __syncwarp();
    issue_qg(unit, 0);
    int64_t p_unit = unit;
    int p_u = 0, p_chunk = 0;
    for (int u = 0; u < S; ++u) {
        issue_obst(p_unit, p_chunk, u);
        if (++p_chunk == a.own.chunks) p_chunk = 0;
        if (++p_u == U) { p_u = 0; p_unit += stride; }
    }
    int c_stage = 0;
    uint32_t c_phase = 0;

    for (int it = 0; unit < n_units; unit += stride, ++it) {
        const int64_t tile = unit / L;
        const int slot = (int)(unit % L) * SUB + sl;             // instance within the tile
        const bool active = (tile << 5) + slot < a.n;
        const int64_t tN = tile * (nc * 32) + slot;
        __syncwarp();
        if (unit + stride < n_units) issue_qg(unit + stride, (it + 1) & 1);
        mbar_wait(&bars[kMaxStages + (it & 1)], (uint32_t)(it >> 1) & 1u);
        const unsigned char* qgb = region + (size_t)a.n_stages * SH::kStage + (size_t)(it & 1) * SH::kQg;
        const T* qs = reinterpret_cast<const T*>(qgb) + sl;
        const T* gs = reinterpret_cast<const T*>(qgb + SH::kQ) + sl;

        T q[NL];
#pragma unroll
        for (int k = 0; k < NL; ++k) q[k] = real_joint(k) ? qs[(j0 + k) * SUB] : T(0);
        T g[13];
#pragma unroll
        for (int k = 0; k < 13; ++k) g[k] = gs[k * SUB];

        for (int cyc = 0; cyc < a.k_cycles; ++cyc) {
            const bool last = (cyc == a.k_cycles - 1);

            // 1. forward kinematics of this lane's part of the chain, from the identity (lane 0: from the base frame)
            T Jl[NL][3], Ja[NL][3];                              // first: joint origin / axis in the part's own frame
            T Rt[9];
            Pos<T> pt;
            {
                T R[9], p[3];
#pragma unroll
                for (int k = 0; k < 9; ++k) R[k] = (h == 0) ? c.base[k] : ((k % 4 == 0) ? T(1) : T(0));
#pragma unroll
                for (int k = 0; k < 3; ++k) p[k] = (h == 0) ? c.base[9 + k] : T(0);
                static_for<0, NL>([&](auto kc) {
                    constexpr int k = decltype(kc)::value;
                    Ja[k][0] = (T)R[2]; Ja[k][1] = (T)R[5]; Ja[k][2] = (T)R[8];
                    Jl[k][0] = (T)p[0]; Jl[k][1] = (T)p[1]; Jl[k][2] = (T)p[2];
                    const T* tp = tipb[k];
                    T s, co;
                    sincos_wide(c.sincos, q[k], &s, &co);
                    const T ca = tp[0], sa = tp[1], t0 = tp[2], t1 = tp[3], t2 = tp[4];
#pragma unroll
                    for (int r = 0; r < 3; ++r) {
                        const T x0 = R[3 * r + 0], y0 = R[3 * r + 1], z0 = R[3 * r + 2];
                        const T x = fma(co, x0, s * y0), y = fma(co, y0, -s * x0);            // RotZ(q)
                        p[r] = fma(x, t0, fma(y, t1, fma(z0, t2, p[r])));                     // tip translation
                        R[3 * r + 0] = x;
                        R[3 * r + 1] = fma(ca, y, sa * z0);                                   // tip rotation RotX(alpha)
                        R[3 * r + 2] = fma(ca, z0, -sa * y);
                    }
                });

                // Combine the partial frames.  Lane 1 needs the frame its part starts from (lane 0 began at the base) and both
                // need the flange frame.  One exchange: lane 0 holds X0 and receives X1, lane 1 the other way round; flange = X0 X1.
                T Rs[9], ps[3], pe[3];
                {
                    T Ry[9], py[3];
#pragma unroll
                    for (int k = 0; k < 9; ++k) Ry[k] = __shfl_xor_sync(0xffffffffu, R[k], SUB);
#pragma unroll
                    for (int k = 0; k < 3; ++k) py[k] = __shfl_xor_sync(0xffffffffu, p[k], SUB);
                    T Ra[9], pa[3], Rb[9], pb[3], Re[9];
#pragma unroll
                    for (int k = 0; k < 9; ++k) { Ra[k] = h ? Ry[k] : R[k]; Rb[k] = h ? R[k] : Ry[k]; }
#pragma unroll
                    for (int k = 0; k < 3; ++k) { pa[k] = h ? py[k] : p[k]; pb[k] = h ? p[k] : py[k]; }
                    frame_mul<T>(Ra, pa, Rb, pb, Re, pe);
#pragma unroll
                    for (int k = 0; k < 9; ++k) { Rt[k] = Re[k]; Rs[k] = h ? Ry[k] : ((k % 4 == 0) ? T(1) : T(0)); }
#pragma unroll
                    for (int k = 0; k < 3; ++k) ps[k] = h ? py[k] : T(0);
                }
                pt.set(pe);
                // joint axes and origins to the base frame, then the Jacobian columns [z x (p_e - p_j); z]
                static_for<0, NL>([&](auto kc) {
                    constexpr int k = decltype(kc)::value;
                    const T zx = Ja[k][0], zy = Ja[k][1], zz = Ja[k][2], ox = Jl[k][0], oy = Jl[k][1], oz = Jl[k][2];
                    T z[3], o[3];
#pragma unroll
                    for (int r = 0; r < 3; ++r) {
                        z[r] = fma(Rs[3 * r + 0], zx, fma(Rs[3 * r + 1], zy, Rs[3 * r + 2] * zz));
                        o[r] = fma(Rs[3 * r + 0], ox, fma(Rs[3 * r + 1], oy, fma(Rs[3 * r + 2], oz, ps[r])));
                    }
                    const T ex = (pt.hi[0] - o[0]) + pt.lo[0], ey = (pt.hi[1] - o[1]) + pt.lo[1], ez = (pt.hi[2] - o[2]) + pt.lo[2];   // p_e - o
                    if constexpr (k >= N - (L - 1) * NL) {           // a padding slot on the last lane: zero column
                        const bool real = h != L - 1;
#pragma unroll
                        for (int r = 0; r < 3; ++r) z[r] = real ? z[r] : T(0);
                    }
                    Jl[k][0] = z[1] * ez - z[2] * ey; Jl[k][1] = z[2] * ex - z[0] * ez; Jl[k][2] = z[0] * ey - z[1] * ex;
                    Ja[k][0] = z[0]; Ja[k][1] = z[1]; Ja[k][2] = z[2];
                });
            }

            // 2-4. field: attractor (every lane), this lane's share of the repulsor sum, saturation
            T tw[6];
            {
                T V[3], S0, w[3], acc[3] = {T(0), T(0), T(0)};
                attract<T>(c, g, Rt, pt, V, S0, w);
                for (int ch = 0; ch < a.own.chunks; ++ch) {
                    const int stage = resident ? ch : c_stage;
                    mbar_wait(&bars[stage], resident ? (uint32_t)(it & 1) : c_phase);
                    const unsigned char* sb = region + (size_t)stage * SH::kStage;
                    const int n_here = ch < a.own.full ? kChunk : a.own.rem;
                    const int n_pairs = (n_here + 1) >> 1;
                    // stage = [pair][4 planes][SUB lanes] of double2 {slot 0, slot 1}
                    const double2* pl = reinterpret_cast<const double2*>(sb) + sl;
                    auto deal = [&](auto order_c) {
                        constexpr int ORD = decltype(order_c)::value;
                        const bool full = ch < a.own.full;
#pragma unroll
                        for (int i = 0; i < (kChunk / 2 + L - 1) / L; ++i) {
                            const int pr = i * L + h;
                            if (full || pr < n_pairs) {
                                const double2 X = pl[(4 * pr) * SUB], Y = pl[(4 * pr + 1) * SUB], Z = pl[(4 * pr + 2) * SUB], Rr = pl[(4 * pr + 3) * SUB];
                                Vec4<T> o0, o1;
                                o0.x = X.x; o0.y = Y.x; o0.z = Z.x; o0.w = Rr.x;
                                o1.x = X.y; o1.y = Y.y; o1.z = Z.y; o1.w = Rr.y;
                                repel<T, ORD>(o0, c.obst_safe_inv, c.obst_order, pt, acc);
                                repel<T, ORD>(o1, c.obst_safe_inv, c.obst_order, pt, acc);       // zero radius in a padding slot: adds 0
                            }
                        }
                    };
                    with_order<T, false>(c.order_int, deal);
                    if (!resident || last) {
                        __syncwarp();
                        if (p_unit < n_units) issue_obst(p_unit, p_chunk, stage);
                        if (++p_chunk == a.own.chunks) p_chunk = 0;
                        if (++p_u == U) { p_u = 0; p_unit += stride; }
                    }
                    if (!resident && ++c_stage == S) { c_stage = 0; c_phase ^= 1u; }
                }
#pragma unroll
                for (int off = SUB; off < 32; off <<= 1) {
#pragma unroll
                    for (int k = 0; k < 3; ++k) acc[k] += __shfl_xor_sync(0xffffffffu, acc[k], off);
                }
                V[0] = fma(c.obst_force, acc[0], V[0]); V[1] = fma(c.obst_force, acc[1], V[1]); V[2] = fma(c.obst_force, acc[2], V[2]);
                T v[3];
                saturate<T>(c, V, S0, v);
                tw[0] = v[0]; tw[1] = v[1]; tw[2] = v[2]; tw[3] = w[0]; tw[4] = w[1]; tw[5] = w[2];
            }

            // 5. damped least squares: this lane's columns into J J^T and J x, summed over the instance's lanes
            T x[NL];
#pragma unroll
            for (int k = 0; k < NL; ++k) x[k] = limb[k][2] * (q[k] - limb[k][3]);
            T A[21], invd[6], Jx[6];
#pragma unroll
            for (int r = 0; r < 6; ++r) {
                Jx[r] = T(0);
#pragma unroll
                for (int s = 0; s <= r; ++s) A[tri(r, s)] = T(0);
            }
            static_for<0, NL>([&](auto kc) {
                constexpr int k = decltype(kc)::value;
                const T col[6] = {Jl[k][0], Jl[k][1], Jl[k][2], Ja[k][0], Ja[k][1], Ja[k][2]};
                axpy6(Jx, col, x[k]);
                syr6(A, col);
            });
#pragma unroll
            for (int off = SUB; off < 32; off <<= 1) {
#pragma unroll
                for (int i = 0; i < 21; ++i) A[i] += __shfl_xor_sync(0xffffffffu, A[i], off);
#pragma unroll
                for (int r = 0; r < 6; ++r) Jx[r] += __shfl_xor_sync(0xffffffffu, Jx[r], off);
            }
#pragma unroll
            for (int r = 0; r < 6; ++r) A[tri(r, r)] += c.ik_lambda2;
            // see vfk_cycle_kernel: FP64 accepts ik_lambda = 0
            const T pivot_floor = T(1e-28) * (A[tri(0, 0)] + A[tri(1, 1)] + A[tri(2, 2)] + A[tri(3, 3)] + A[tri(4, 4)] + A[tri(5, 5)]) + T(1e-300);
            chol6<T>(A, invd, pivot_floor);
            T yv[6], yn[6];
            {
                T y[6];
#pragma unroll
                for (int r = 0; r < 6; ++r) y[r] = tw[r];
                chol6_fwd<T>(A, invd, y);
                chol6_bwd<T>(A, invd, y);
                chol6_fwd<T>(A, invd, Jx);
                chol6_bwd<T>(A, invd, Jx);
#pragma unroll
                for (int r = 0; r < 6; ++r) { yv[r] = y[r]; yn[r] = Jx[r]; }
            }

            // 6. nullspace projector on the limit-avoidance gradient, all-or-nothing lookahead check over ALL joints; 8-9. mixer, clamp
            T mix[NL];
            bool bad = false;
#pragma unroll
            for (int k = 0; k < NL; ++k) {
                const T cj[6] = {Jl[k][0], Jl[k][1], Jl[k][2], Ja[k][0], Ja[k][1], Ja[k][2]};
                const T raw = dot6_packed(cj, yn, x[k], true);
                const T d = fma(c.ns_lookahead, raw, q[k]);
                bad = bad || (d < limb[k][0]) || (d > limb[k][1]);
                x[k] = raw;                                              // x is not needed any more
                mix[k] = dot6_packed(cj, yv, T(0), false) * c.mixer_w[0];
            }
            {
                int b = bad ? 1 : 0;
#pragma unroll
                for (int off = SUB; off < 32; off <<= 1) b |= __shfl_xor_sync(0xffffffffu, b, off);
                bad = b != 0;
            }
            T lead = T(0);
#pragma unroll
            for (int k = 0; k < NL; ++k) {
                const T ns = bad ? T(0) : x[k] * c.ns_gain;
                mix[k] = fma(ns, c.mixer_w[1], mix[k]);
                lead = Prec<T>::fmax_(lead, Prec<T>::fabs_(mix[k]));
            }
#pragma unroll
            for (int off = SUB; off < 32; off <<= 1) lead = Prec<T>::fmax_(lead, __shfl_xor_sync(0xffffffffu, lead, off));
            T ratio = T(1);
            if (lead > c.max_vel) ratio = Prec<T>::div(c.max_vel, lead);
            {                                                        // never integrate a non-finite step
                T z = T(0);
#pragma unroll
                for (int k = 0; k < NL; ++k) z = fma(mix[k], T(0), z);
                int nf = (z != T(0)) ? 1 : 0;                        // NaN or inf anywhere in this lane's part
#pragma unroll
                for (int off = SUB; off < 32; off <<= 1) nf |= __shfl_xor_sync(0xffffffffu, nf, off);
                if (nf) {
                    ratio = T(0);
#pragma unroll
                    for (int k = 0; k < NL; ++k) mix[k] = T(0);
                }
            }

            if (last && active) {
#pragma unroll
                for (int k = 0; k < NL; ++k)
                    if (real_joint(k)) a.qdot[tN + (j0 + k) * 32] = mix[k] * ratio;
            }
            // 10. plant
            if (c.integrate) {
#pragma unroll
                for (int k = 0; k < NL; ++k) q[k] = fma(c.dt, mix[k] * ratio, q[k]);
            }
        }
        if (active && c.integrate) {
#pragma unroll
            for (int k = 0; k < NL; ++k)
                if (real_joint(k)) a.q[tN + (j0 + k) * 32] = q[k];
        }
    }
}

}  // namespace vfk
