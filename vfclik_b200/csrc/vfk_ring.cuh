// vfk_ring.cuh -- cursor arithmetic of the cycle kernel's per-warp obstacle ring (vfk_kernels.cuh).
//
// A "use" is one consumption of one obstacle chunk; a unit (a warp's share of a tile) has U uses, the ring S slots.
// The producer cursor (p_unit, p_u, p_chunk) names the next use to request, and is always exactly S uses ahead of the
// consumer, whose slot and phase are (c_stage, c_phase) on a streaming ring.  Plain integer code, compiled for the host as
// well so that a CPU test can drive the same arithmetic the kernel runs (tests/test_solve_cpu.py).
#pragma once
#include <stdint.h>

#ifdef __CUDACC__
#define VFK_HD __host__ __device__ __forceinline__
#else
#define VFK_HD inline
#endif

namespace vfk {

// The producer has requested one more use.
VFK_HD void ring_produced(int64_t& p_unit, int& p_u, int& p_chunk, int n_chunks, int U, int64_t stride) {
    if (++p_chunk == n_chunks) p_chunk = 0;
    if (++p_u == U) { p_u = 0; p_unit += stride; }
}

// The consumer is done with its slot (streaming ring: slots are taken in turn, the phase flips on every wrap).
VFK_HD void ring_consumed(int& c_stage, uint32_t& c_phase, int S) {
    if (++c_stage == S) { c_stage = 0; c_phase ^= 1u; }
}

// A streaming ring's warp leaves its unit with `left` uses not consumed (vfk_solve: every instance of the unit has stopped).
// The first min(left, S) of them are in flight; the rest were never requested and never will be.  Moves the producer past
// those to the next unit's first use and returns how many in-flight slots the caller must still wait, in order, refilling
// each one as the ring always does (wait, request the producer's use into the freed slot, ring_produced, ring_consumed).
// Afterwards every requested copy has been waited exactly once, and the producer is again exactly S uses ahead of the
// consumer, which stands at the next unit's first use.  When left <= S the producer is already inside the next unit and
// the uses it requested there stay as they are.
VFK_HD int ring_leave(int64_t& p_unit, int& p_u, int& p_chunk, int left, int S, int64_t stride) {
    if (left <= S) return left;
    p_u = 0;
    p_chunk = 0;
    p_unit += stride;
    return S;
}

}  // namespace vfk
