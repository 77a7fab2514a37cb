// Host model of one warp of the cycle kernel walking its obstacle ring (vfk_kernels.cuh), driven through the cursor
// arithmetic of vfk_ring.cuh over random shapes and random early exits (vfk_solve).  mbarriers and bulk copies are modelled
// per slot: a copy is in flight from its request until a wait on the slot's current phase lands it.  Fails (exit 1, with a
// message) when a copy is requested into a slot whose previous copy was never waited, a wait finds no copy (a hang on the
// GPU), a wait returns on an older phase while a copy is in flight or returns another chunk than the consumer expects, the
// producer is not exactly S uses ahead when a unit starts, or a copy is left unwaited at the end.  Prints "ok <cases>".
#include <cstdio>
#include <cstdlib>
#include <random>
#include <vector>

#include "vfk_ring.cuh"

using namespace vfk;

#define CHECK(c, ...) do { if (!(c)) { std::printf(__VA_ARGS__); std::printf("\n"); std::exit(1); } } while (0)

struct Slot {
    int completed = 0;        // phases completed
    bool inflight = false;    // a requested copy that no wait has landed yet
    int64_t unit = -1;
    int chunk = -1;
};

struct Warp {
    int n_chunks, S, K, stride;
    int64_t n_units;
    bool resident;
    std::vector<Slot> slot;
    int64_t issued = 0, landed = 0;
    const char* ctx;

    void issue(int s, int64_t unit, int chunk) {
        Slot& x = slot[s];
        CHECK(!x.inflight, "%s: request into slot %d while its copy of (%lld, %d) was never waited", ctx, s, (long long)x.unit, x.chunk);
        x.inflight = true;
        x.unit = unit;
        x.chunk = chunk;
        ++issued;
    }
    // rewait: a resident ring's later cycles wait the phase the first cycle already saw complete
    void wait(int s, uint32_t parity, int64_t unit, int chunk, bool rewait) {
        Slot& x = slot[s];
        if ((uint32_t)(x.completed & 1) != parity) {            // the phase of this parity has completed: returns at once
            CHECK(!x.inflight, "%s: wait on slot %d returned on an older phase while a copy is in flight", ctx, s);
            CHECK(rewait, "%s: slot %d waited twice for the same copy (unit %lld chunk %d)", ctx, s, (long long)unit, chunk);
        } else {
            CHECK(x.inflight, "%s: wait on slot %d (parity %u) with no copy outstanding: the warp would hang", ctx, s, parity);
            x.inflight = false;
            ++x.completed;
            ++landed;
        }
        CHECK(x.unit == unit && x.chunk == chunk, "%s: slot %d holds (unit %lld, chunk %d), the consumer expects (%lld, %d)", ctx, s,
              (long long)x.unit, x.chunk, (long long)unit, chunk);
    }
};

// One warp over units unit0, unit0 + stride, ...  exit_use[u]: the use index at which unit u's instances have all stopped
// (streaming: any index 0..U, the kernel itself stops only at cycle boundaries; resident: a multiple of n_chunks); U = none.
static void run(int n_chunks, int n_stages, int K, int stride, int64_t n_units, int64_t unit0, const std::vector<int>& exit_use,
                const char* ctx) {
    Warp w;
    w.n_chunks = n_chunks;
    w.resident = n_chunks <= n_stages;
    w.S = w.resident ? n_chunks : n_stages;
    w.K = K;
    w.stride = stride;
    w.n_units = n_units;
    w.slot.assign(w.S, Slot());
    w.ctx = ctx;
    const int S = w.S, U = w.resident ? n_chunks : n_chunks * K;
    int64_t p_unit = unit0;
    int p_u = 0, p_chunk = 0;
    if (unit0 < n_units)
        for (int u = 0; u < S; ++u) {
            w.issue(u, p_unit, p_chunk);
            ring_produced(p_unit, p_u, p_chunk, n_chunks, U, stride);
        }
    int c_stage = 0;
    uint32_t c_phase = 0;
    int it = 0;
    for (int64_t unit = unit0; unit < n_units; unit += stride, ++it) {
        CHECK((p_unit - unit) / stride * U + p_u == S, "%s: unit %lld starts with the producer %lld uses ahead, not %d", ctx,
              (long long)unit, (long long)((p_unit - unit) / stride * U + p_u), S);
        const int e = exit_use[unit];
        int cu = 0;                                             // consumer's use index within the unit
        bool left_unit = false;
        for (int cyc = 0; cyc <= K && !left_unit; ++cyc) {
            const bool last = cyc == K - 1;
            for (int ch = 0; ch <= n_chunks; ++ch) {
                // the kernel checks at the start of a cycle (ch == 0); the streaming model also leaves between chunks
                const bool leave = cyc == K || (w.resident ? (ch == 0 && e == cyc * n_chunks) : cu == e);
                if (leave) {
                    const int left = w.resident ? (cyc < K ? n_chunks : 0) : ring_leave(p_unit, p_u, p_chunk, U - cu, S, stride);
                    for (int i = 0; i < left; ++i) {
                        const int stage = w.resident ? i : c_stage;
                        w.wait(stage, w.resident ? (uint32_t)(it & 1) : c_phase, unit, w.resident ? i : (cu + i) % n_chunks, w.resident && cyc > 0);
                        if (p_unit < n_units) w.issue(stage, p_unit, p_chunk);
                        ring_produced(p_unit, p_u, p_chunk, n_chunks, U, stride);
                        if (!w.resident) ring_consumed(c_stage, c_phase, S);
                    }
                    left_unit = true;
                    break;
                }
                if (ch == n_chunks) break;
                const int stage = w.resident ? ch : c_stage;
                w.wait(stage, w.resident ? (uint32_t)(it & 1) : c_phase, unit, ch, w.resident && cyc > 0);
                if (!w.resident || last) {
                    if (p_unit < n_units) w.issue(stage, p_unit, p_chunk);
                    ring_produced(p_unit, p_u, p_chunk, n_chunks, U, stride);
                }
                if (!w.resident) ring_consumed(c_stage, c_phase, S);
                ++cu;
            }
        }
    }
    for (int s = 0; s < S; ++s) CHECK(!w.slot[s].inflight, "%s: slot %d still has a copy in flight at the end", ctx, s);
    CHECK(w.issued == w.landed, "%s: %lld copies requested, %lld waited", ctx, (long long)w.issued, (long long)w.landed);
}

int main(int argc, char** argv) {
    const int n_cases = argc > 1 ? std::atoi(argv[1]) : 20000;
    std::mt19937 rng(12345);
    auto uni = [&](int lo, int hi) { return std::uniform_int_distribution<int>(lo, hi)(rng); };
    char ctx[256];
    int cases = 0;
    for (int t = 0; t < n_cases; ++t) {
        const int n_chunks = uni(1, 9), n_stages = uni(1, 3), K = uni(1, 5), stride = uni(1, 4);
        const int64_t n_units = uni(1, 24), unit0 = uni(0, stride - 1);
        const bool resident = n_chunks <= n_stages;
        const int S = resident ? n_chunks : n_stages, U = resident ? n_chunks : n_chunks * K;
        std::vector<int> exit_use(n_units);
        const int mode = t % 6;     // 0 random, 1 none stop, 2 all at cycle 0, 3 at the last cycle, 4 fewer than S uses left, 5 mixed
        for (auto& e : exit_use) {
            int cyc_exit = uni(0, K);
            if (mode == 1) cyc_exit = K;
            if (mode == 2) cyc_exit = 0;
            if (mode == 3) cyc_exit = K - 1;
            e = resident ? cyc_exit * n_chunks : (mode == 0 || mode == 5 ? uni(0, U) : cyc_exit * n_chunks);
            if (mode == 4 && !resident) e = U - uni(0, S < U ? S : U);
            if (resident && mode == 0) e = uni(0, K) * n_chunks;
        }
        std::snprintf(ctx, sizeof ctx, "case %d (n_chunks %d, stages %d, K %d, stride %d, units %lld, first %lld, mode %d)", t, n_chunks,
                      n_stages, K, stride, (long long)n_units, (long long)unit0, mode);
        run(n_chunks, n_stages, K, stride, n_units, unit0, exit_use, ctx);
        ++cases;
    }
    std::printf("ok %d\n", cases);
    return 0;
}
