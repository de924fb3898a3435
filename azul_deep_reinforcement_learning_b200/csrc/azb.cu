// azb.cu -- sm_100a kernels and the C ABI (include/azb.h) of the batched Azul engine.
//
// One game per thread: the whole packed state (17 / 22 / 27 words for 2 / 3 / 4 players) lives in
// registers, loads and stores of the structure-of-arrays state are fully coalesced (a warp touches
// 32 consecutive words per state word), and all rule arithmetic is SWAR on bit-planes
// (azb_rules.cuh).  The path is integer work bounded by HBM traffic for the single-step entry
// points and by the issue rate for the fused K-step rollout; there is nothing GEMM-shaped here.
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "azb_internal.h"
#include "azb_rules.cuh"
#include "azb_queue.cuh"

using namespace azb;

// ------------------------------------------------------------------------------------------
// error plumbing
// ------------------------------------------------------------------------------------------
static thread_local char g_err[512] = "";

int azb_fail(int code, const char* fmt, const char* detail)
{
    snprintf(g_err, sizeof(g_err), fmt, detail);
    return code;
}

// ------------------------------------------------------------------------------------------
// kernels
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ void store_mask(uint32_t* __restrict__ mask6, int64_t n, int64_t g, const uint32_t m[6])
{
#pragma unroll
    for (int p = 0; p < 6; p++) mask6[p * n + g] = m[p];
}

// K6: fresh game in the selected slots
template <int P, int POOL>
__global__ void k_reset(Launch L, const uint8_t* __restrict__ which)
{
    const int64_t g = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (g >= L.n) return;
    if (which && which[g] == 0) return;
    Game<P> gm;
    gm.steps = L.state[6 * L.n + g];
    const Philox rng{L.k0, L.k1};
    reset_game<P, POOL>(gm, rng, L.gid0 + (uint32_t)g, L.first_rule);
    gm.store(L.state, L.n, g);
}

// K2: legal mask only -- reads the 4 shared words and the mover's pattern + wall words
template <int P>
__global__ void k_legal_mask(const uint32_t* __restrict__ s, int64_t n, uint32_t* __restrict__ mask6)
{
    const int64_t g = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (g >= n) return;
    Game<P> gm;
    gm.pl0 = s[g]; gm.pl1 = s[n + g]; gm.pl2 = s[2 * n + g]; gm.set_misc_word(s[3 * n + g]);
    const int seat = gm.seat();
#pragma unroll
    for (int p = 0; p < P; p++) { gm.pat[p] = 0; gm.wall[p] = 0; }
    const uint32_t pat = s[(7 + 5 * seat) * n + g], wall = s[(8 + 5 * seat) * n + g];
    gm.put(gm.pat, seat, pat);
    gm.put(gm.wall, seat, wall);
    uint32_t m[6];
    legal_mask(gm, m);
    store_mask(mask6, n, g, m);
}

// K1 (+K2, K5): one Azul.step per game.
// The move is cheap and uniform; the end-of-round work (count_score, game-over test, new_round) hits ~10 % of
// the games of a launch, i.e. ~3 of a warp's 32 lanes.  Each warp therefore walks several rows of 32 games and
// parks the games whose round just ended in a warp-private shared-memory queue (packed state + game index);
// once STEP_DRAIN_AT are waiting, the warp finishes them together with (nearly) every lane busy.  No block barrier is
// involved; the finished games are written back with per-lane (scattered) 4-byte stores that merge in L2 with the
// whole-line row stores of the same 128-byte lines (which carry an L2 evict_last policy for that reason).
struct StepOut {
    uint32_t* __restrict__ mask6;
    int16_t* __restrict__ preview;
    uint8_t* __restrict__ done;
    uint8_t* __restrict__ status;
};

__device__ __forceinline__ void st_global_hint(uint32_t* dst, uint32_t v, uint64_t policy)
{
    asm volatile("st.global.L2::cache_hint.b32 [%0], %1, %2;" ::"l"(dst), "r"(v), "l"(policy) : "memory");
}

// state (when the game moved) and the per-game outputs of azb_step; `policy` != 0: L2 cache hint for the state and mask
// words (the queue drain's patches are the last writes to their lines: evict first)
template <int P, int POOL>
__device__ __forceinline__ void step_finish(const Launch& L, const StepOut& O, Game<P>& gm, int64_t g, uint32_t status, bool moved,
                                            uint64_t policy = 0)
{
    if (moved) {
        if (policy) {
            uint32_t w[Game<P>::WORDS];
            gm.store(w, 1, 0);
#pragma unroll
            for (int i = 0; i < Game<P>::WORDS; i++) st_global_hint(L.state + i * L.n + g, w[i], policy);
        } else {
            gm.store(L.state, L.n, g);
        }
    }
    if (O.mask6 || O.status) {
        uint32_t m[6];
        legal_mask(gm, m);
        if (!gm.ended() && m[0] == 0u /* words 1..5 are subsets of word 0 */ && gm.current_player() != 0u)
            status |= ST_STUCK;
        if (O.mask6) {
            if (policy) {
#pragma unroll
                for (int p = 0; p < 6; p++) st_global_hint(O.mask6 + p * L.n + g, m[p], policy);
            } else {
                store_mask(O.mask6, L.n, g, m);
            }
        }
    }
    if (O.preview) {
        Game<P> cp = gm;
        count_score<P, POOL>(cp);
#pragma unroll
        for (int p = 0; p < P; p++) O.preview[p * L.n + g] = (int16_t)(cp.scf[p] & 0xFFFFu);
    }
    if (O.done) O.done[g] = gm.ended() ? 1 : 0;
    if (O.status) O.status[g] = (uint8_t)(status | gm.status());
}

// ---- k_step: staged, persistent-warp implementation ----
// Each warp owns (in dynamic shared memory) a ring of STAGES row tiles [word][lane], one output tile for the legal
// mask and its queue of finished rounds.  Rows are fetched NSTAGE-1 iterations ahead with 16-byte cp.async copies
// (no registers are held by loads in flight), read from the tile with conflict-free 4-byte shared loads, and --
// on the aligned path -- written back through the tile with 16-byte global stores, so that a row costs
// ceil(W/4) + 2 global store instructions instead of W + 6 and every 128-byte line is written whole.

constexpr int STEP_CLAIM = 4;                      // consecutive rows a warp takes from the device-wide counter at a time
constexpr int STEP_SCHED_WORDS = 16;               // row counter, exit counter
// games waiting in a warp's queue that trigger a pass: fuller passes cost fewer instructions, earlier passes patch lines that
// are still in L2 (measured 16 / 20 / 24 / 28 / 32: 201 / 191 / 183 / 186 / 196 us for 4.2 M two-player games)
constexpr int STEP_DRAIN_AT = 24;
constexpr int STEP_QCAP = 56;                      // a row that would overflow the queue drains it first
constexpr int STEP_WARPS = 2;                      // warps per block (fine-grained shared-memory occupancy)
constexpr int STEP_MINBLOCKS = 8;

template <int P, int STAGES>
struct StepSmem {
    static constexpr int W = 7 + 5 * P;
    static constexpr int QUEUE = (W + 2) * STEP_QCAP;
    static constexpr int TILE = W * 32 + 8;                                  // + the row's 32 action bytes
    static constexpr int MASK = 6 * 32;
    static constexpr int WORDS_PER_WARP = QUEUE + STAGES * TILE + MASK;      // multiple of 4 words: 16-byte aligned parts
    static constexpr size_t bytes(int warps) { return (size_t)warps * WORDS_PER_WARP * sizeof(uint32_t); }
};

__device__ __forceinline__ void cp_async16(uint32_t* smem_dst, const uint32_t* gsrc)
{
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(gsrc) : "memory");
}
// L2 residency hints: a row's lines are read once, rewritten whole a few rows later and -- for the games whose round
// ended -- patched once more when their warp's queue drains; keeping the rewritten lines in L2 until then avoids
// partial-sector writes to lines that already left for DRAM.
__device__ __forceinline__ uint64_t l2_policy_evict_last()
{
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ uint64_t l2_policy_evict_first()
{
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ void cp_async16_hint(uint32_t* smem_dst, const uint32_t* gsrc, uint64_t policy)
{
    asm volatile("cp.async.cg.shared.global.L2::cache_hint [%0], [%1], 16, %2;\n" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(gsrc), "l"(policy) : "memory");
}
__device__ __forceinline__ void st_global_v4_hint(uint32_t* dst, const uint4& v, uint64_t policy)
{
    asm volatile("st.global.L2::cache_hint.v4.b32 [%0], {%1, %2, %3, %4}, %5;" ::"l"(dst), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w), "l"(policy) : "memory");
}
__device__ __forceinline__ void cp_async4(uint32_t* smem_dst, const uint32_t* gsrc)
{
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;\n" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N) : "memory"); }

// global [word][n] row of 32 games (+ its 32 action bytes on the aligned path) -> tile [word][32] (+ 8 words).
// The actions travel with the row: a separate register load issued after the copies would return behind them
// (a warp's memory operations complete in order) and cut the prefetch distance to one row.
// Lane l moves the 16-byte chunks l, l + 32, ...: chunk c is part (c & 7) of word (c >> 3), so consecutive chunks of a
// lane are 4 words apart: `lane_off` = (l >> 3) * n + 4 * (l & 7) is fixed per thread and `n4` = 4 * n steps to the next.
template <int LINES>
__device__ __forceinline__ void row_fetch(uint32_t* tile, const uint32_t* __restrict__ s, const uint8_t* __restrict__ action,
                                          int64_t n, int64_t g0, int lane, bool fast, int64_t lane_off, int64_t n4, uint64_t policy)
{
    if (fast) {
        const uint32_t* src = s + lane_off + g0;
        uint32_t* dst = tile + 4 * lane;
#pragma unroll
        for (int k = 0; k < (LINES * 8 + 31) / 32; k++, src += n4, dst += 128)
            if (32 * k + 32 <= LINES * 8 || lane < LINES * 8 - 32 * k) cp_async16_hint(dst, src, policy);
        if (lane < 2) cp_async16(tile + LINES * 32 + 4 * lane, reinterpret_cast<const uint32_t*>(action + g0) + 4 * lane);
    } else if (g0 + lane < n) {
#pragma unroll
        for (int w = 0; w < LINES; w++) cp_async4(tile + 32 * w + lane, s + (int64_t)w * n + g0 + lane);
    }
}
// tile [word][32] -> global [word][n], 16 bytes per lane (aligned, full rows only)
template <int LINES>
__device__ __forceinline__ void row_flush(const uint32_t* tile, uint32_t* __restrict__ s, int64_t g0, int lane, int64_t lane_off, int64_t n4, uint64_t policy)
{
    uint32_t* dst = s + lane_off + g0;
    const uint32_t* src = tile + 4 * lane;
#pragma unroll
    for (int k = 0; k < (LINES * 8 + 31) / 32; k++, dst += n4, src += 128)
        if (32 * k + 32 <= LINES * 8 || lane < LINES * 8 - 32 * k) st_global_v4_hint(dst, *reinterpret_cast<const uint4*>(src), policy);
}

template <int P, int POOL, int STAGES>
__global__ void __launch_bounds__(32 * STEP_WARPS, STEP_MINBLOCKS) k_step(Launch L, const uint8_t* __restrict__ action,
                                                           const int8_t* __restrict__ draws, StepOut O, int aligned,
                                                           unsigned int* __restrict__ sched)
{
    using S = StepSmem<P, STAGES>;
    constexpr int W = S::W, QCAP = STEP_QCAP;
    static_assert(QCAP >= STEP_DRAIN_AT - 1 + 32, "a row must fit behind a queue that is just below the drain threshold");
    extern __shared__ __align__(16) uint32_t step_smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t* q = step_smem + (size_t)warp * S::WORDS_PER_WARP;
    uint32_t* tiles = q + S::QUEUE;
    uint32_t* mask_tile = tiles + STAGES * S::TILE;
    const int64_t n_rows = (L.n + 31) / 32;
    const Philox rng{L.k0, L.k1};
    int waiting = 0;                                        // warp-uniform: entries in this warp's queue
    const uint64_t pol_first = l2_policy_evict_first(), pol_last = l2_policy_evict_last();
    const int64_t lane_off = (int64_t)(lane >> 3) * L.n + 4 * (lane & 7), n4 = 4 * L.n;

    // Rows are claimed from a device-wide counter (sched[0]), not assigned by stride: a warp's time depends on how many of
    // its games end their round, and with a fixed assignment the slowest warp set the kernel's tail.  Results do not
    // depend on which warp steps a game.  The last warp to leave resets the counters for the next launch.
    // One atomic per ROW bounds the kernel (131,072 atomics on one address per launch of 4.2 M games: 0.59 of the HBM peak,
    // the memory path alone 0.69), so a ticket is STEP_CLAIM consecutive rows: 2 / 4 / 8 rows 0.68 / 0.70 / 0.69 (larger
    // tickets bring the tail back; the memory path alone reaches 0.87 with 4).  Measured and rejected: tickets that
    // shrink towards the end (0.67: the single-row tail is atomic-bound again) and one counter per group of 8 blocks
    // (0.63 - 0.65: a group's blocks share an SM, so nothing balances the SMs any more).
    const uint32_t n_rows32 = (uint32_t)n_rows, fast_rows = aligned ? (uint32_t)(L.n / 32) : 0u;   // n_games <= 2^31
    uint32_t claim_next = 0, claim_end = 0;
    auto claim = [&]() -> uint32_t {
        if (claim_next == claim_end) {
            unsigned int r = 0;
            if (lane == 0) r = atomicAdd(&sched[0], (unsigned int)STEP_CLAIM);
            claim_next = __shfl_sync(0xFFFFFFFFu, r, 0);
            claim_end = claim_next + STEP_CLAIM;
        }
        return claim_next++;
    };
    // rows in flight, in the order they were claimed = the order they are consumed (rows >= n_rows mean "none");
    // the row at the head was loaded into tile `stage`
    uint32_t in_flight[STAGES - 1];
    // prologue: STAGES-1 rows of this warp in flight
#pragma unroll
    for (int k = 0; k < STAGES - 1; k++) {
        const uint32_t r = claim();
        in_flight[k] = r;
        if (r < n_rows32) row_fetch<W>(tiles + k * S::TILE, L.state, action, L.n, (int64_t)r * 32, lane, r < fast_rows, lane_off, n4, pol_first);
        cp_async_commit();
    }
    int stage = 0;
    for (;;) {
        const uint32_t row = in_flight[0];
        const bool have_row = row < n_rows32;
        if (have_row) {
            const int64_t g = (int64_t)row * 32 + lane;
            const bool valid = g < L.n;
            const bool fast = row < fast_rows;
            uint32_t* tile = tiles + stage * S::TILE;
            {   // refill the tile consumed by the previous iteration; every lane is past its reads of it
                __syncwarp();
                const uint32_t r = claim();
#pragma unroll
                for (int k = 0; k + 1 < STAGES - 1; k++) in_flight[k] = in_flight[k + 1];
                in_flight[STAGES - 2] = r;
                const int st_fill = stage == 0 ? STAGES - 1 : stage - 1;
                if (r < n_rows32) row_fetch<W>(tiles + st_fill * S::TILE, L.state, action, L.n, (int64_t)r * 32, lane, r < fast_rows, lane_off, n4, pol_first);
                cp_async_commit();
            }
            cp_async_wait<STAGES - 1>();
            __syncwarp();
            Game<P> gm;
            uint32_t a = AZB_ACTION_SKIP;
            if (valid) {
                gm.load(tile, 32, lane);
                a = fast ? reinterpret_cast<const uint8_t*>(tile + W * 32)[lane] : action[g];
            }
            bool round_over = false, moved = false;
            uint32_t status = 0;
            if (valid && a != AZB_ACTION_SKIP) {
                if (gm.ended()) {
                    status = ST_ENDED;                                        // azul.py:298-299
                } else {
                    if (!move_if_legal<P, POOL>(gm, a)) {                     // azul.py:301-304
                        status = ST_ILLEGAL;
                    } else {
                        gm.steps += 1u;
                        moved = true;
                        round_over = is_end_of_round(gm);                     // azul.py:306
                        if (!round_over) next_player(gm);                     // azul.py:313
                    }
                }
            }
            if (fast) {
                // whole lines through the tile; the lanes whose round ended write their interim state and outputs here
                // and the final ones in the drain -- later in program order of this warp, ordered by __syncwarp.  (Parking only
                // (game index, status) and letting the drain read the interim state back from L2 was measured: 0.63 against
                // 0.71 of the HBM peak -- 17 more registers for the loads in flight and an L2 round trip in every pass)
                const bool any_moved = __any_sync(0xFFFFFFFFu, moved);
                uint32_t m[6];
                legal_mask(gm, m);
                if (!round_over && !gm.ended() && m[0] == 0u /* words 1..5 are subsets of word 0 */ && gm.current_player() != 0u)
                    status |= ST_STUCK;
                if (any_moved) gm.store(tile, 32, lane);
                if (O.mask6) {
#pragma unroll
                    for (int p = 0; p < 6; p++) mask_tile[32 * p + lane] = m[p];
                }
                __syncwarp();
                if (any_moved) row_flush<W>(tile, L.state, (int64_t)row * 32, lane, lane_off, n4, pol_last);
                if (O.mask6) row_flush<6>(mask_tile, O.mask6, (int64_t)row * 32, lane, lane_off, n4, pol_last);
                if (!round_over) {
                    if (O.preview) {
                        Game<P> cp = gm;
                        count_score<P, POOL>(cp);
#pragma unroll
                        for (int p = 0; p < P; p++) O.preview[p * L.n + g] = (int16_t)(cp.scf[p] & 0xFFFFu);
                    }
                    if (O.done) O.done[g] = gm.ended() ? 1 : 0;
                    if (O.status) O.status[g] = (uint8_t)(status | gm.status());
                }
            } else if (valid && !round_over) {
                step_finish<P, POOL>(L, O, gm, g, status, moved);
            }
            const uint32_t over = __ballot_sync(0xFFFFFFFFu, round_over);
            if (over) {                                                       // waiting < STEP_DRAIN_AT here: the row fits
                if (round_over) queue_put<P, QCAP>(q, waiting + __popc(over & ((1u << lane) - 1u)), gm, (uint32_t)g, status);
                waiting += __popc(over);
                __syncwarp();
            }
            stage = stage + 1 == STAGES ? 0 : stage + 1;
        }
        // ONE drain site (the pass is ~2 k instructions; three inlined copies did not fit the instruction cache):
        // a pass runs once STEP_DRAIN_AT games wait, and for whatever is left when the rows have run out
        if (waiting >= STEP_DRAIN_AT || (!have_row && waiting > 0)) {
            const int count = waiting < 32 ? waiting : 32;                    // finish `count` games from the tail of the queue
            if (lane < count) {
                Game<P> h;
                uint32_t gidx, st;
                queue_get<P, QCAP>(q, waiting - count + lane, h, gidx, st);
                count_score<P, POOL>(h);                                      // azul.py:307
                if (is_end_of_game(h)) {                                      // azul.py:308-309
                    h.misc |= 1u << 12;
                } else if (draws) {                                           // azul.py:311
                    const int8_t* d = draws + 20 * (int64_t)gidx;
                    new_round_injected<P, POOL>(h, [&](int k) { return (int)d[k]; });
                } else {
                    new_round_philox<P, POOL>(h, rng, L.gid0 + gidx, PURPOSE_REFILL);
                }
                step_finish<P, POOL>(L, O, h, (int64_t)gidx, st, true, pol_first);
            }
            waiting -= count;
            __syncwarp();
        } else if (!have_row) {
            break;
        }
    }
    cp_async_wait<0>();
    if (lane == 0) {
        const unsigned int warps_total = gridDim.x * STEP_WARPS;
        __threadfence();
        if (atomicAdd(&sched[1], 1u) == warps_total - 1u) { sched[0] = 0u; sched[1] = 0u; __threadfence(); }
    }
}

// K1+K2+K3+K6 fused: k_steps random-agent env steps per game in one launch
struct BlockSink {
    unsigned long long* c;             // the block's counters in shared memory
    uint32_t r[AZB_N_COUNTERS];        // this lane's share of the game statistics since the last flush
    uint32_t passes;
    __device__ __forceinline__ explicit BlockSink(unsigned long long* shared) : c(shared), passes(0u)
    {
#pragma unroll
        for (int i = 0; i < AZB_N_COUNTERS; i++) r[i] = 0u;
    }
    // rare events and the per-launch totals: straight to the block's counters
    __device__ __forceinline__ void add(int i, uint32_t v)
    {
        if (v) atomicAdd(&c[i], (unsigned long long)v);
    }
    // the statistics of finished games: a register add per counter.  (One REDUX + one 64-bit shared atomic per counter
    // and end-of-round pass cost 17 instructions per env step and 5 % of the kernel's stall samples.)
    __device__ __forceinline__ void add_group(int i, uint32_t v) { r[i] += v; }
    // whole warp, after every end-of-round pass: flush before a 32-bit warp sum could overflow (a pass adds at most
    // 4 * 65,535 per lane: 256 passes * 32 lanes stay below 2^32)
    __device__ __forceinline__ void pass_done()
    {
        if ((++passes & 255u) == 0u) flush();
    }
    __device__ __forceinline__ void flush()
    {
#pragma unroll
        for (int i = 0; i < AZB_N_COUNTERS; i++) {
            const uint32_t tot = __reduce_add_sync(0xFFFFFFFFu, r[i]);
            if (tot && (threadIdx.x & 31) == 0) atomicAdd(&c[i], (unsigned long long)tot);
            r[i] = 0u;
        }
    }
};

// Action words of a whole round, computed by the full warp during the end-of-round pass (when all of its games
// are at the same point) and parked in shared memory: ROUND_WORDS words per game, [word][thread] so that a warp
// reads 32 consecutive banks.  A round that outlasts them falls back to computing a block in place.
constexpr int ROUND_WORDS = 16;          // 12 / 16 / 20 words: 3.61 / 3.70 / 3.67e10 env steps/s (rounds last ~10.5 steps; longer ones fall back)
struct RoundWords {
    uint32_t base;           // shared-window byte address of buf[threadIdx.x] (a generic pointer costs an address conversion per read)
    uint32_t stride;         // 4 * blockDim.x
    uint32_t first_block;
    uint32_t w[4];
    uint32_t block;
    __device__ __forceinline__ void prefetch(const Philox& rng, uint32_t gid, uint32_t T)
    {
        first_block = T >> 2;
#pragma unroll 1
        for (uint32_t j = 0; j < ROUND_WORDS / 4; j++) {
            uint32_t r[4];
            rng(gid, first_block + j, PURPOSE_ACTION, 0u, r);
#pragma unroll
            for (uint32_t i = 0; i < 4; i++)
                asm volatile("st.shared.b32 [%0], %1;" ::"r"(base + (4 * j + i) * stride), "r"(r[i]) : "memory");
        }
        block = 0xFFFFFFFFu;
    }
    __device__ __forceinline__ uint32_t get(const Philox& rng, uint32_t gid, uint32_t T)
    {
        const uint32_t idx = T - 4u * first_block;
        if (idx < (uint32_t)ROUND_WORDS) {
            uint32_t v;
            asm volatile("ld.shared.b32 %0, [%1];" : "=r"(v) : "r"(base + idx * stride) : "memory");
            return v;
        }
        if (block != (T >> 2)) { block = T >> 2; rng(gid, block, PURPOSE_ACTION, 0u, w); }
        const uint32_t i = T & 3u;
        return i == 0u ? w[0] : i == 1u ? w[1] : i == 2u ? w[2] : w[3];
    }
};

template <int P, int POOL>
__global__ void k_rollout_random(Launch L, int k_steps, int defer, uint32_t* __restrict__ mask6_out,
                                 unsigned long long* __restrict__ counters)
{
    extern __shared__ uint32_t round_words[];          // [ROUND_WORDS][blockDim.x]
    __shared__ unsigned long long cnt[AZB_N_COUNTERS];
    if (threadIdx.x < AZB_N_COUNTERS) cnt[threadIdx.x] = 0ull;
    __syncthreads();
    const int64_t g = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    const bool valid = g < L.n;
    const int64_t gl = valid ? g : L.n - 1;            // whole warps stay in the loop: they vote together
    Game<P> gm;
    gm.load(L.state, L.n, gl);
    const Philox rng{L.k0, L.k1};
    BlockSink sink(cnt);
    RoundWords words;
    words.base = (uint32_t)__cvta_generic_to_shared(round_words + threadIdx.x);
    words.stride = 4u * blockDim.x;
    rollout_steps<P, POOL>(gm, rng, L.gid0 + (uint32_t)gl, L.first_rule, k_steps, sink, WarpLanes{}, valid, defer, words);
    sink.flush();
    if (valid) {
        gm.store(L.state, L.n, g);
        if (mask6_out) {
            uint32_t m[6];
            legal_mask(gm, m);
            store_mask(mask6_out, L.n, g, m);
        }
    }
    __syncthreads();
    if (counters && threadIdx.x < AZB_N_COUNTERS && cnt[threadIdx.x]) atomicAdd(&counters[threadIdx.x], cnt[threadIdx.x]);
}

// ---- k_rollout_rotate: the same rollout with the 32-game batches ROTATING through the warps of the block ----
// A batch resident in one wave gives every SM one block; with 14 batches per block (65,536 games on 148 SMs) the four warp
// schedulers of an SM hold 4, 4, 3 and 3 warps, every game runs the same number of steps, and the warps on the fuller
// schedulers set the kernel's time (8.7 % of all warp samples sat at the barrier before EXIT; per warp the 14-warp block is no
// faster than a 16-warp one).  No static placement fixes 14 on 4.  Here the block has two warps more than batches: a warp
// plays its batch for `passes_per_turn` end-of-round passes, then -- if the next warp of the ring is idle -- parks the batch
// (packed states, steps left) in that warp's shared-memory slot and becomes idle itself.  The two idle slots travel backwards
// round the ring, the batches forwards: every batch spends its time on fuller and emptier schedulers alike, and so does
// every scheduler.  Results cannot depend on it: a game's trajectory depends on its id and step counter only.
__device__ __forceinline__ uint32_t ld_shared_volatile(const uint32_t* p) { return *reinterpret_cast<const volatile uint32_t*>(p); }
__device__ __forceinline__ void st_shared_volatile(uint32_t* p, uint32_t v) { *reinterpret_cast<volatile uint32_t*>(p) = v; }

template <int P, int POOL>
__global__ void __launch_bounds__(512) k_rollout_rotate(Launch L, int k_steps, int defer, uint32_t* __restrict__ mask6_out,
                                                        unsigned long long* __restrict__ counters, int batches_per_block,
                                                        int passes_per_turn)
{
    constexpr int W = Game<P>::WORDS;
    extern __shared__ uint32_t rot_smem[];             // [ROUND_WORDS][blockDim.x] action words, then [warps][W + 1][32] parked batches
    __shared__ unsigned long long cnt[AZB_N_COUNTERS];
    __shared__ uint32_t slot_state[16];                // 0 playing, 1 idle, 3 a batch is parked in this warp's slot
    __shared__ uint32_t slot_batch[16];
    __shared__ uint32_t n_done;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, warps = (int)(blockDim.x >> 5);
    uint32_t* park = rot_smem + ROUND_WORDS * blockDim.x;
    const int64_t block_g0 = blockIdx.x * (int64_t)(32 * batches_per_block);
    const int64_t games_here = L.n - block_g0 < 32 * batches_per_block ? L.n - block_g0 : 32 * batches_per_block;
    const uint32_t n_batches = (uint32_t)((games_here + 31) / 32);
    if (threadIdx.x < AZB_N_COUNTERS) cnt[threadIdx.x] = 0ull;
    if (threadIdx.x < 16) slot_state[threadIdx.x] = (uint32_t)threadIdx.x < n_batches ? 0u : 1u;
    if (threadIdx.x == 0) n_done = 0u;
    __syncthreads();
    const Philox rng{L.k0, L.k1};
    BlockSink sink(cnt);
    RoundWords words;
    words.base = (uint32_t)__cvta_generic_to_shared(rot_smem + threadIdx.x);
    words.stride = 4u * blockDim.x;
    Game<P> gm;
    bool have = (uint32_t)warp < n_batches;
    uint32_t batch = (uint32_t)warp;
    int remaining = 0;
    int64_t g = block_g0 + 32 * (int64_t)batch + lane;
    bool valid = have && g < L.n;
    int64_t gl = g < L.n ? g : L.n - 1;
    if (have) { gm.load(L.state, L.n, gl); remaining = valid ? k_steps : 0; }
    const int succ = warp + 1 == warps ? 0 : warp + 1;
    for (;;) {
        if (have) {
            remaining = rollout_steps<P, POOL, true>(gm, rng, L.gid0 + (uint32_t)gl, L.first_rule, remaining, sink, WarpLanes{}, valid, defer,
                                                     words, passes_per_turn);
            if (!__any_sync(0xFFFFFFFFu, remaining > 0)) {                    // the batch has run all its steps
                if (valid) {
                    gm.store(L.state, L.n, g);
                    if (mask6_out) {
                        uint32_t m[6];
                        legal_mask(gm, m);
                        store_mask(mask6_out, L.n, g, m);
                    }
                }
                have = false;
                __syncwarp();
                if (lane == 0) { atomicAdd(&n_done, 1u); __threadfence_block(); st_shared_volatile(&slot_state[warp], 1u); }
            } else if (ld_shared_volatile(&slot_state[succ]) == 1u) {         // the next warp is idle: the batch moves on
                uint32_t* dst = park + (size_t)succ * (W + 1) * 32;
                gm.store(dst, 32, lane);
                dst[W * 32 + lane] = (uint32_t)remaining;
                if (lane == 0) slot_batch[succ] = batch;
                __threadfence_block();
                __syncwarp();
                have = false;
                if (lane == 0) { st_shared_volatile(&slot_state[succ], 3u); st_shared_volatile(&slot_state[warp], 1u); }
            }
        } else {
            uint32_t s = 0u;
            if (lane == 0) {
                for (;;) {
                    s = ld_shared_volatile(&slot_state[warp]);
                    if (s == 3u) break;
                    if (ld_shared_volatile(&n_done) >= n_batches) break;      // every batch has finished: none can arrive
                    __nanosleep(400);
                }
            }
            s = __shfl_sync(0xFFFFFFFFu, s, 0);
            if (s != 3u) break;
            __threadfence_block();
            const uint32_t* src = park + (size_t)warp * (W + 1) * 32;
            gm.load(src, 32, lane);
            remaining = (int)src[W * 32 + lane];
            batch = slot_batch[warp];
            g = block_g0 + 32 * (int64_t)batch + lane;
            valid = g < L.n;
            gl = valid ? g : L.n - 1;
            __syncwarp();
            if (lane == 0) st_shared_volatile(&slot_state[warp], 0u);
            have = true;
        }
    }
    sink.flush();
    __syncthreads();
    if (counters && threadIdx.x < AZB_N_COUNTERS && cnt[threadIdx.x]) atomicAdd(&counters[threadIdx.x], cnt[threadIdx.x]);
}

// K5: score preview on a copy
template <int P, int POOL>
__global__ void k_score_preview(const uint32_t* __restrict__ s, int64_t n, int16_t* __restrict__ out)
{
    const int64_t g = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (g >= n) return;
    Game<P> gm;
    gm.load(s, n, g);
    count_score<P, POOL>(gm);
#pragma unroll
    for (int p = 0; p < P; p++) out[p * n + g] = (int16_t)(gm.scf[p] & 0xFFFFu);
}

// K7: unpacked records <-> packed state
template <int P>
__global__ void k_import(const int32_t* __restrict__ rec, uint32_t* __restrict__ s, int64_t n, uint8_t* __restrict__ ok_out)
{
    const int64_t g = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (g >= n) return;
    const int32_t* r = rec + g * (48 + 58 * P);
    Game<P> gm;
    const bool ok = import_record<P>(gm, [&](int i) { return r[i]; });
    gm.store(s, n, g);
    if (ok_out) ok_out[g] = ok ? 1 : 0;
}

template <int P>
__global__ void k_export(const uint32_t* __restrict__ s, int32_t* __restrict__ rec, int64_t n)
{
    const int64_t g = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (g >= n) return;
    int32_t* r = rec + g * (48 + 58 * P);
    Game<P> gm;
    gm.load(s, n, g);
    export_record<P>(gm, [&](int i, int32_t v) { r[i] = v; });
}

// GameRunner.get_state (game_runner.py:56-72)
__device__ __forceinline__ void obs_store(float* o, int i, float v) { o[i] = v; }
__device__ __forceinline__ void obs_store(__nv_bfloat16* o, int i, float v) { o[i] = __float2bfloat16_rn(v); }

// GameRunner.get_state (game_runner.py:56-72) of one game: D = 32 + 52P values written to o[0..D)
template <int P, typename T>
__device__ __forceinline__ void observe_row(const Game<P>& gm, int perspective, T* o)
{
    const int persp = perspective >= 0 ? perspective : gm.seat();
    for (int i = 0; i < 5; i++)
        for (int c = 0; c < 5; c++) {
            const uint32_t b = (uint32_t)(i + 1 + 6 * c);
            obs_store(o, i * 5 + c, (float)(((gm.pl0 >> b) & 1u) | (((gm.pl1 >> b) & 1u) << 1) | (((gm.pl2 >> b) & 1u) << 2)));
        }
    for (int c = 0; c < 5; c++) {
        const uint32_t b = (uint32_t)(6 * c);
        obs_store(o, 25 + c, (float)(((gm.pl0 >> b) & 1u) | (((gm.pl1 >> b) & 1u) << 1) | (((gm.pl2 >> b) & 1u) << 2) |
                            (((gm.pl3 >> b) & 1u) << 3)));
    }
    obs_store(o, 30, (float)((gm.misc >> 5) & 1u));
    // order = [perspective] + ascending others (game_runner.py:57)
#pragma unroll
    for (int slot = 0; slot < P; slot++) {
        const int p = slot == 0 ? persp : (slot - 1 < persp ? slot - 1 : slot);
        const uint32_t pat = gm.sel(gm.pat, p), wall = gm.sel(gm.wall, p), scf = gm.sel(gm.scf, p);
        for (int r = 0; r < 5; r++) {
            const uint32_t cnt = (pat >> (6 * r + 3)) & 7u, col = (pat >> (6 * r)) & 7u;
            for (int c = 0; c < 5; c++) {
                obs_store(o, 31 + 25 * slot + 5 * r + c, (float)((cnt && col == (uint32_t)c) ? cnt : 0u));
                obs_store(o, 31 + 25 * P + 25 * slot + 5 * r + c, (float)((wall >> (5 * r + c)) & 1u));
            }
        }
        obs_store(o, 31 + 50 * P + slot, (float)((scf >> 16) & 7u));
        obs_store(o, 31 + 51 * P + slot, (float)(scf & 0xFFFFu));
    }
    const int nf = (int)gm.next_first_player();
    obs_store(o, 31 + 52 * P, nf > 0 ? (float)(((nf - 1 - persp) % P + P) % P + 1) : 0.0f);     // game_runner.py:58-61
}

// A warp's 32 observation rows ([lane][D + 1] in shared memory) -> the output, where they are contiguous: coalesced
// stores (a thread writing its own row directly touches 32 different sectors per store instruction).
template <int P, typename T>
__device__ __forceinline__ void observe_flush(const T* tile, T* __restrict__ out, int64_t rows, int lane)
{
    constexpr int D = 32 + 52 * P;
    __syncwarp();
    int row = 0, col = lane;
    for (int64_t idx = lane; idx < rows * D; idx += 32) {
        out[idx] = tile[row * (D + 1) + col];
        col += 32;
        if (col >= D) { col -= D; row++; }
    }
}

// One warp per block and 32 games per warp
template <int P, typename T>
__global__ void __launch_bounds__(32) k_observe(const uint32_t* __restrict__ s, int64_t n, int perspective, T* __restrict__ obs_out)
{
    constexpr int D = 32 + 52 * P;
    __shared__ T tile[32 * (D + 1)];
    const int lane = threadIdx.x;
    const int64_t g0 = (int64_t)blockIdx.x * 32, g = g0 + lane;
    Game<P> gm;
    gm.load(s, n, g < n ? g : n - 1);
    observe_row<P, T>(gm, perspective, tile + lane * (D + 1));
    observe_flush<P, T>(tile, obs_out + g0 * D, n - g0 < 32 ? n - g0 : 32, lane);
}

// Azul.get_statistics raw integers (azul.py:314-315)
template <int P>
__global__ void k_stats(const uint32_t* __restrict__ s, int64_t n, int32_t* __restrict__ out)
{
    const int64_t g = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (g >= n) return;
    Game<P> gm;
    gm.load(s, n, g);
    int32_t* o = out + g * 10;
    uint32_t fps = 0;
#pragma unroll
    for (int p = 0; p < P; p++) fps += gm.sta[p] & 0xFFFu;
    o[0] = (int32_t)(gm.scf[0] & 0xFFFFu);
    o[1] = (int32_t)(gm.scf[1] & 0xFFFFu);
    o[2] = (int32_t)gm.turn_counter();
    o[3] = (int32_t)(gm.sta[0] & 0xFFFu);
    o[4] = (int32_t)fps;
    o[5] = (int32_t)((gm.sta[0] >> 12) & 0xFFFFu);
    o[6] = (int32_t)(gm.sta[0] >> 28);
    o[7] = (int32_t)(gm.stb[0] & 255u);
    o[8] = (int32_t)((gm.stb[0] >> 16) & 255u);
    o[9] = (int32_t)((gm.stb[0] >> 8) & 255u);
}

// the reference's per-function entry points (façade): 0 move, 1 next_player, 2 count_score, 3 new_round
template <int P, int POOL, int OP>
__global__ void k_op(Launch L, const uint8_t* __restrict__ action, const int8_t* __restrict__ draws)
{
    const int64_t g = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (g >= L.n) return;
    Game<P> gm;
    gm.load(L.state, L.n, g);
    if (OP == 0) {
        const uint32_t a = action[g];
        if (a >= 180u) return;
        apply_move<P, POOL>(gm, a);
    } else if (OP == 1) {
        next_player(gm);
    } else if (OP == 2) {
        count_score<P, POOL>(gm);
    } else {
        if (draws) {
            const int8_t* d = draws + 20 * g;
            new_round_injected<P, POOL>(gm, [&](int k) { return (int)d[k]; });
        } else {
            const Philox rng{L.k0, L.k1};
            new_round_philox<P, POOL>(gm, rng, L.gid0 + (uint32_t)g, PURPOSE_REFILL);
        }
    }
    gm.store(L.state, L.n, g);
}

// a14: GameRunner.step after the agent's own move: opponent loop, reward, done, next mask -- and, optionally, the
// observation of the resulting state from seat 1's perspective (the next decision's network input) in bfloat16, so
// that a training rollout needs no separate observation launch.  Blocks are whole warps.  GREEDY: the greedy agent is
// the opponent (k_opponent_greedy), else the random agent (k_opponent_random).
template <int P, int POOL, bool GREEDY>
__device__ __forceinline__ void opponent_turns(Launch L, int require_two, int16_t* __restrict__ player_score,
                                               int16_t* __restrict__ reward_out, uint8_t* __restrict__ done_out,
                                               uint8_t* __restrict__ status_out, uint32_t* __restrict__ mask6_out,
                                               __nv_bfloat16* __restrict__ obs_out)
{
    constexpr int D = 32 + 52 * P;
    extern __shared__ __align__(16) unsigned char opp_smem[];          // [warp][32][D + 1] bf16 when obs_out
    const int64_t g = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    const bool valid = g < L.n;
    Game<P> gm;
    gm.load(L.state, L.n, valid ? g : L.n - 1);
    if (valid) {
        const Philox rng{L.k0, L.k1};
        uint32_t m[6];
        const int32_t diff = opponent_random<P, POOL, GREEDY>(gm, rng, L.gid0 + (uint32_t)g, require_two != 0, m);
        gm.store(L.state, L.n, g);
        if (player_score) {
            if (reward_out) reward_out[g] = (int16_t)(diff - (int32_t)player_score[g]);    // game_runner.py:51
            player_score[g] = (int16_t)diff;                                                // game_runner.py:52
        }
        if (done_out) done_out[g] = gm.ended() ? 1 : 0;
        if (status_out) status_out[g] = (uint8_t)gm.status();
        if (mask6_out) store_mask(mask6_out, L.n, g, m);
    }
    if (obs_out) {
        const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
        __nv_bfloat16* tile = reinterpret_cast<__nv_bfloat16*>(opp_smem) + (size_t)warp * 32 * (D + 1);
        const int64_t g0 = g - lane;
        observe_row<P, __nv_bfloat16>(gm, 0, tile + lane * (D + 1));
        if (g0 < L.n) observe_flush<P, __nv_bfloat16>(tile, obs_out + g0 * D, L.n - g0 < 32 ? L.n - g0 : 32, lane);
    }
}

template <int P, int POOL>
__global__ void k_opponent_random(Launch L, int require_two, int16_t* __restrict__ player_score,
                                  int16_t* __restrict__ reward_out, uint8_t* __restrict__ done_out,
                                  uint8_t* __restrict__ status_out, uint32_t* __restrict__ mask6_out,
                                  __nv_bfloat16* __restrict__ obs_out)
{
    opponent_turns<P, POOL, false>(L, require_two, player_score, reward_out, done_out, status_out, mask6_out, obs_out);
}

template <int P, int POOL>
__global__ void k_opponent_greedy(Launch L, int require_two, int16_t* __restrict__ player_score,
                                  int16_t* __restrict__ reward_out, uint8_t* __restrict__ done_out,
                                  uint8_t* __restrict__ status_out, uint32_t* __restrict__ mask6_out,
                                  __nv_bfloat16* __restrict__ obs_out)
{
    opponent_turns<P, POOL, true>(L, require_two, player_score, reward_out, done_out, status_out, mask6_out, obs_out);
}

// the greedy agent's action for the seat to move (greedy_action, the word of the game's current env step); state untouched
template <int P, int POOL>
__global__ void k_greedy_action(Launch L, uint8_t* __restrict__ action_out)
{
    const int64_t g = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (g >= L.n) return;
    Game<P> gm;
    gm.load(L.state, L.n, g);
    uint32_t a = 180u;
    if (!gm.ended()) {
        uint32_t m[6], w[4];
        legal_mask(gm, m);
        const Philox rng{L.k0, L.k1};
        rng(L.gid0 + (uint32_t)g, gm.steps >> 2, PURPOSE_ACTION, 0u, w);
        const uint32_t idx = gm.steps & 3u;
        a = greedy_action<P, POOL>(gm, m, idx == 0u ? w[0] : idx == 1u ? w[1] : idx == 2u ? w[2] : w[3]);
    }
    action_out[g] = a < 180u ? (uint8_t)a : (uint8_t)AZB_ACTION_SKIP;
}

template <int P>
__global__ void k_round_flags(const uint32_t* __restrict__ s, int64_t n, uint8_t* __restrict__ flags)
{
    const int64_t g = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (g >= n) return;
    Game<P> gm;
    gm.load(s, n, g);
    flags[g] = (uint8_t)((is_end_of_round(gm) ? 1 : 0) | (is_end_of_game(gm) ? 2 : 0));
}

// ------------------------------------------------------------------------------------------
// C ABI
// ------------------------------------------------------------------------------------------
#define DISPATCH_P(h, EXPR)                         \
    switch ((h)->players) {                         \
    case 2: { constexpr int P = 2; EXPR; } break;   \
    case 3: { constexpr int P = 3; EXPR; } break;   \
    default: { constexpr int P = 4; EXPR; } break;  \
    }

#define DISPATCH_PP(h, EXPR)                                                   \
    if ((h)->tile_pool == AZB_POOL_LID) { constexpr int POOL = 1; DISPATCH_P(h, EXPR) } \
    else { constexpr int POOL = 0; DISPATCH_P(h, EXPR) }

static inline dim3 grid_of(const azb_t* h) { return dim3((unsigned)((h->n_games + h->block_threads - 1) / h->block_threads)); }

// persistent warps: each walks many rows of 32 games so that its queue of finished rounds fills up; as many blocks
// as fit (shared memory decides), never more than there are rows
template <int P, int POOL>
static int launch_step(const azb_t* h, const Launch& L, const uint8_t* action, const int8_t* draws, const StepOut& O,
                       int aligned, cudaStream_t stream)
{
    constexpr int STAGES = P == 2 ? 4 : 3;       // 2 / 3 / 4 / 5 stages: 183 / 192 / 183 / 198 us for 4.2 M two-player games
    auto kern = k_step<P, POOL, STAGES>;
    constexpr int WARPS = STEP_WARPS;
    const size_t smem = StepSmem<P, STAGES>::bytes(STEP_WARPS);
    static thread_local int per_sm_cached[64] = {0};      // function attributes are per device
    int uncached = 0;
    int& per_sm = h->device < 64 ? per_sm_cached[h->device] : uncached;
    if (per_sm == 0) {
        AZB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        AZB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
        AZB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, 32 * WARPS, smem));
        if (per_sm < 1) per_sm = 1;
    }
    const int64_t rows = (h->n_games + 31) / 32;
    int64_t blocks = (rows + WARPS - 1) / WARPS;
    const int64_t resident = (int64_t)h->sm_count * per_sm;
    if (blocks > resident) blocks = resident;
    kern<<<dim3((unsigned)blocks), 32 * WARPS, smem, stream>>>(L, action, draws, O, aligned, h->sched);
    return 0;
}

// azb_opponent_random / azb_opponent_greedy
template <bool GREEDY>
static int launch_opponent(azb_t* h, uint32_t* state, int require_two, int16_t* player_score, int16_t* reward_out,
                           uint8_t* done_out, uint8_t* status_out, uint32_t* mask6_out, void* obs_bf16_out, void* stream)
{
    CHECK_HANDLE(h);
    if (!state) return azb_fail(AZB_E_INVALID, "state is null%s");
    const Launch L = make_launch(h, state);
    // with the observation output every warp stages 32 rows in shared memory (32 x (33 + 52P) bf16 per warp): 128-thread
    // blocks for 2 / 3 players (35 / 47 KB), 64-thread blocks for 4 players (31 KB) stay under the 48 KB default limit
    const int threads = obs_bf16_out ? (h->players == 4 ? 64 : 128) : h->block_threads;
    const size_t smem = obs_bf16_out ? (size_t)(threads / 32) * 32 * (32 + 52 * h->players + 1) * sizeof(__nv_bfloat16) : 0;
    const dim3 grid((unsigned)((h->n_games + threads - 1) / threads));
    __nv_bfloat16* obs = (__nv_bfloat16*)obs_bf16_out;
    if (GREEDY)
        DISPATCH_PP(h, (k_opponent_greedy<P, POOL><<<grid, threads, smem, (cudaStream_t)stream>>>(
                           L, require_two, player_score, reward_out, done_out, status_out, mask6_out, obs)))
    else
        DISPATCH_PP(h, (k_opponent_random<P, POOL><<<grid, threads, smem, (cudaStream_t)stream>>>(
                           L, require_two, player_score, reward_out, done_out, status_out, mask6_out, obs)))
    CHECK_LAUNCH();
    return 0;
}

extern "C" {

int azb_abi_version(void) { return AZB_ABI_VERSION; }
int azb_state_words(int players) { return (players >= 2 && players <= 4) ? 7 + 5 * players : AZB_E_INVALID; }
int azb_record_size(int players) { return (players >= 2 && players <= 4) ? 48 + 58 * players : AZB_E_INVALID; }
int azb_obs_size(int players) { return (players >= 2 && players <= 4) ? 32 + 52 * players : AZB_E_INVALID; }
const char* azb_last_error(void) { return g_err; }

int azb_create(azb_t** out, int device, int64_t n_games, int players, int tile_pool, int first_player,
               uint64_t seed, uint64_t game_id_base)
{
    if (!out) return azb_fail(AZB_E_INVALID, "out is null%s");
    *out = nullptr;
    if (players < 2 || players > 4) return azb_fail(AZB_E_INVALID, "players must be 2..4%s");
    if (tile_pool != AZB_POOL_RANDOM && tile_pool != AZB_POOL_LID) return azb_fail(AZB_E_INVALID, "tile_pool must be 0 (Random) or 1 (Lid)%s");
    if (first_player < 0 || first_player > players) return azb_fail(AZB_E_INVALID, "first_player must be 0 (Random) or 1..players%s");   // IllegalRule, azul.py:40-41
    if (n_games < 1 || n_games > (int64_t)1 << 31) return azb_fail(AZB_E_INVALID, "n_games out of range%s");
    // the Philox counter carries a 32-bit global game id: ids beyond 2^32 would alias streams
    if (game_id_base > 0xFFFFFFFFull || game_id_base + (uint64_t)n_games > (1ull << 32))
        return azb_fail(AZB_E_INVALID, "game_id_base + n_games exceeds the 32-bit global game id of the draw schedule%s");
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0)
        return azb_fail(AZB_E_NODEVICE, "no CUDA device (%s); this library has no CPU path", e != cudaSuccess ? cudaGetErrorString(e) : "device count 0");
    if (device < 0 || device >= count) return azb_fail(AZB_E_INVALID, "device index out of range%s");
    AZB_CUDA(cudaSetDevice(device));
    azb_t* h = new azb_handle();
    h->device = device; h->n_games = n_games; h->players = players; h->tile_pool = tile_pool;
    h->first_player = first_player; h->seed = seed; h->game_id_base = game_id_base; h->block_threads = 128; h->block_threads_set = 0; h->defer = 32;
    AZB_CUDA(cudaDeviceGetAttribute(&h->sm_count, cudaDevAttrMultiProcessorCount, device));
    // row counter + exit counter of azb_step's dynamic row schedule (reset by the kernel itself after every launch)
    e = cudaMalloc(&h->sched, STEP_SCHED_WORDS * sizeof(unsigned int));
    if (e == cudaSuccess) e = cudaMemset(h->sched, 0, STEP_SCHED_WORDS * sizeof(unsigned int));
    if (e != cudaSuccess) { delete h; return azb_fail(AZB_E_CUDA, "scheduler counters: %s", cudaGetErrorString(e)); }
    *out = h;
    return 0;
}

int azb_destroy(azb_t* h)
{
    if (h && h->sched) { cudaSetDevice(h->device); cudaFree(h->sched); }
    delete h;
    return 0;
}

int azb_set_block_threads(azb_t* h, int threads)
{
    if (!h) return azb_fail(AZB_E_INVALID, "null handle%s");
    h->block_threads_set = threads != 0;
    if (threads == 0) threads = 128;
    if (threads < 32 || threads > 1024 || threads % 32) return azb_fail(AZB_E_INVALID, "block threads must be a multiple of 32 in 32..1024%s");
    h->block_threads = threads;
    return 0;
}

int azb_set_rollout_defer(azb_t* h, int games)
{
    if (!h) return azb_fail(AZB_E_INVALID, "null handle%s");
    if (games == 0) games = 32;
    if (games < 1 || games > 32) return azb_fail(AZB_E_INVALID, "defer must be 1..32%s");
    h->defer = games;
    return 0;
}

int azb_reset(azb_t* h, uint32_t* state, const uint8_t* which, void* stream)
{
    CHECK_HANDLE(h);
    if (!state) return azb_fail(AZB_E_INVALID, "state is null%s");
    const Launch L = make_launch(h, state);
    DISPATCH_PP(h, (k_reset<P, POOL><<<grid_of(h), h->block_threads, 0, (cudaStream_t)stream>>>(L, which)));
    CHECK_LAUNCH();
    return 0;
}

int azb_legal_mask(azb_t* h, const uint32_t* state, uint32_t* mask6, void* stream)
{
    CHECK_HANDLE(h);
    if (!state || !mask6) return azb_fail(AZB_E_INVALID, "null buffer%s");
    DISPATCH_P(h, (k_legal_mask<P><<<grid_of(h), h->block_threads, 0, (cudaStream_t)stream>>>(state, h->n_games, mask6)));
    CHECK_LAUNCH();
    return 0;
}

int azb_step(azb_t* h, uint32_t* state, const uint8_t* action, const int8_t* draws20, uint32_t* mask6_out,
             int16_t* preview_out, uint8_t* done_out, uint8_t* status_out, void* stream)
{
    CHECK_HANDLE(h);
    if (!state || !action) return azb_fail(AZB_E_INVALID, "null buffer%s");
    const Launch L = make_launch(h, state);
    if (h->n_games > (int64_t)0xFFFFFFFFll) return azb_fail(AZB_E_INVALID, "n_games exceeds the step kernel's 32-bit game index%s");
    StepOut O{mask6_out, preview_out, done_out, status_out};
    // 16-byte copies need every [word] plane (offset w * n_games words), the mask planes and the actions 16-byte aligned
    const int aligned = h->n_games % 4 == 0 && (((uintptr_t)state | (uintptr_t)mask6_out | (uintptr_t)action) & 15u) == 0;
    int rc = 0;
    DISPATCH_PP(h, (rc = launch_step<P, POOL>(h, L, action, draws20, O, aligned, (cudaStream_t)stream)));
    if (rc) return rc;
    CHECK_LAUNCH();
    return 0;
}

int azb_rollout_random(azb_t* h, uint32_t* state, int k_steps, uint32_t* mask6_out, unsigned long long* counters,
                       void* stream)
{
    CHECK_HANDLE(h);
    if (!state) return azb_fail(AZB_E_INVALID, "state is null%s");
    if (k_steps < 0) return azb_fail(AZB_E_INVALID, "k_steps < 0%s");
    const Launch L = make_launch(h, state);
    // Grid sizing: the kernel is issue-bound and every game runs for the whole launch, so the slowest SM sets the time.
    // Unless the caller fixed the block size: when the whole batch is resident at once give every SM the same number
    // of equally sized blocks, k = ceil(n / (SMs * 512)) blocks per SM of ceil(n / (SMs * k)) threads (rounded to a warp).
    int threads = h->block_threads;
    if (!h->block_threads_set) {
        // single wave (everything resident at once, e.g. 65,536 or 131,072 games): equal blocks per SM;
        // several waves: small blocks, so that the tail of the last wave is short
        int blocks64 = 0;
        DISPATCH_PP(h, AZB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&blocks64, k_rollout_random<P, POOL>, 64,
                                                                             (size_t)ROUND_WORDS * 64 * sizeof(uint32_t))));
        const int64_t per_sm = (h->n_games + h->sm_count - 1) / h->sm_count;
        if (per_sm <= (int64_t)blocks64 * 64) {
            const int64_t k = (per_sm + 511) / 512;
            threads = (int)(((per_sm + k - 1) / k + 31) / 32 * 32);
            threads = threads < 64 ? 64 : threads > 512 ? 512 : threads;
        } else {
            threads = 128;
        }
    }
    constexpr int ROTATE_PASSES = 32;      // 1 / 2 / 4 / 8 / 16 / 24 / 32 / 64 / 128 passes per turn: 2.96 / 4.06 / 4.54 / 4.75 / 4.82 / 4.87 / 4.85 / 4.84 / 4.88e10 env steps/s (never: 4.67)
    // one block per SM whose 32-game batches spread 4, 4, 3, 3 (or 3, 3, 2, 2, ...) over the warp schedulers: two warps more than
    // batches, and the batches rotate (k_rollout_rotate)
    if (!h->block_threads_set && h->defer >= 32 && (threads / 32) % 4 == 2 && threads + 64 <= 512 && k_steps > 0 &&
        (h->n_games + threads - 1) / threads <= h->sm_count) {
        const int launch_threads = threads + 64;
        const size_t smem = ((size_t)ROUND_WORDS * launch_threads + (size_t)(launch_threads / 32) * (7 + 5 * h->players + 1) * 32) * sizeof(uint32_t);
        const dim3 rgrid((unsigned)((h->n_games + threads - 1) / threads));
        DISPATCH_PP(h, AZB_CUDA(cudaFuncSetAttribute(k_rollout_rotate<P, POOL>, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024)));
        DISPATCH_PP(h, (k_rollout_rotate<P, POOL><<<rgrid, launch_threads, smem, (cudaStream_t)stream>>>(
                           L, k_steps, h->defer, mask6_out, counters, threads / 32, ROTATE_PASSES)));
        CHECK_LAUNCH();
        return 0;
    }
    const size_t words_bytes = (size_t)ROUND_WORDS * threads * sizeof(uint32_t);
    if (words_bytes > 48 * 1024) return azb_fail(AZB_E_INVALID, "block threads too large for the rollout kernel's word buffer%s");
    const dim3 grid((unsigned)((h->n_games + threads - 1) / threads));
    DISPATCH_PP(h, (k_rollout_random<P, POOL><<<grid, threads, words_bytes, (cudaStream_t)stream>>>(
                       L, k_steps, h->defer, mask6_out, counters)));
    CHECK_LAUNCH();
    return 0;
}

int azb_score_preview(azb_t* h, const uint32_t* state, int16_t* score_out, void* stream)
{
    CHECK_HANDLE(h);
    if (!state || !score_out) return azb_fail(AZB_E_INVALID, "null buffer%s");
    DISPATCH_PP(h, (k_score_preview<P, POOL><<<grid_of(h), h->block_threads, 0, (cudaStream_t)stream>>>(state, h->n_games, score_out)));
    CHECK_LAUNCH();
    return 0;
}

int azb_import_state(azb_t* h, const int32_t* records, uint32_t* state, uint8_t* ok_out, void* stream)
{
    CHECK_HANDLE(h);
    if (!state || !records) return azb_fail(AZB_E_INVALID, "null buffer%s");
    DISPATCH_P(h, (k_import<P><<<grid_of(h), h->block_threads, 0, (cudaStream_t)stream>>>(records, state, h->n_games, ok_out)));
    CHECK_LAUNCH();
    return 0;
}

int azb_export_state(azb_t* h, const uint32_t* state, int32_t* records, void* stream)
{
    CHECK_HANDLE(h);
    if (!state || !records) return azb_fail(AZB_E_INVALID, "null buffer%s");
    DISPATCH_P(h, (k_export<P><<<grid_of(h), h->block_threads, 0, (cudaStream_t)stream>>>(state, records, h->n_games)));
    CHECK_LAUNCH();
    return 0;
}

int azb_observe(azb_t* h, const uint32_t* state, int perspective, float* obs, void* stream)
{
    CHECK_HANDLE(h);
    if (!state || !obs) return azb_fail(AZB_E_INVALID, "null buffer%s");
    if (perspective < -1 || perspective >= h->players) return azb_fail(AZB_E_INVALID, "perspective out of range%s");
    DISPATCH_P(h, (k_observe<P, float><<<dim3((unsigned)((h->n_games + 31) / 32)), 32, 0, (cudaStream_t)stream>>>(state, h->n_games, perspective, obs)));
    CHECK_LAUNCH();
    return 0;
}

int azb_observe_bf16(azb_t* h, const uint32_t* state, int perspective, void* obs_bf16, void* stream)
{
    CHECK_HANDLE(h);
    if (!state || !obs_bf16) return azb_fail(AZB_E_INVALID, "null buffer%s");
    if (perspective < -1 || perspective >= h->players) return azb_fail(AZB_E_INVALID, "perspective out of range%s");
    DISPATCH_P(h, (k_observe<P, __nv_bfloat16><<<dim3((unsigned)((h->n_games + 31) / 32)), 32, 0, (cudaStream_t)stream>>>(
                      state, h->n_games, perspective, (__nv_bfloat16*)obs_bf16)));
    CHECK_LAUNCH();
    return 0;
}

int azb_stats(azb_t* h, const uint32_t* state, int32_t* stats10, void* stream)
{
    CHECK_HANDLE(h);
    if (!state || !stats10) return azb_fail(AZB_E_INVALID, "null buffer%s");
    DISPATCH_P(h, (k_stats<P><<<grid_of(h), h->block_threads, 0, (cudaStream_t)stream>>>(state, h->n_games, stats10)));
    CHECK_LAUNCH();
    return 0;
}

int azb_move(azb_t* h, uint32_t* state, const uint8_t* action, void* stream)
{
    CHECK_HANDLE(h);
    if (!state || !action) return azb_fail(AZB_E_INVALID, "null buffer%s");
    const Launch L = make_launch(h, state);
    DISPATCH_PP(h, (k_op<P, POOL, 0><<<grid_of(h), h->block_threads, 0, (cudaStream_t)stream>>>(L, action, nullptr)));
    CHECK_LAUNCH();
    return 0;
}

int azb_next_player(azb_t* h, uint32_t* state, void* stream)
{
    CHECK_HANDLE(h);
    if (!state) return azb_fail(AZB_E_INVALID, "state is null%s");
    const Launch L = make_launch(h, state);
    DISPATCH_PP(h, (k_op<P, POOL, 1><<<grid_of(h), h->block_threads, 0, (cudaStream_t)stream>>>(L, nullptr, nullptr)));
    CHECK_LAUNCH();
    return 0;
}

int azb_count_score(azb_t* h, uint32_t* state, void* stream)
{
    CHECK_HANDLE(h);
    if (!state) return azb_fail(AZB_E_INVALID, "state is null%s");
    const Launch L = make_launch(h, state);
    DISPATCH_PP(h, (k_op<P, POOL, 2><<<grid_of(h), h->block_threads, 0, (cudaStream_t)stream>>>(L, nullptr, nullptr)));
    CHECK_LAUNCH();
    return 0;
}

int azb_new_round(azb_t* h, uint32_t* state, const int8_t* draws20, void* stream)
{
    CHECK_HANDLE(h);
    if (!state) return azb_fail(AZB_E_INVALID, "state is null%s");
    const Launch L = make_launch(h, state);
    DISPATCH_PP(h, (k_op<P, POOL, 3><<<grid_of(h), h->block_threads, 0, (cudaStream_t)stream>>>(L, nullptr, draws20)));
    CHECK_LAUNCH();
    return 0;
}

int azb_opponent_random(azb_t* h, uint32_t* state, int require_two, int16_t* player_score, int16_t* reward_out,
                        uint8_t* done_out, uint8_t* status_out, uint32_t* mask6_out, void* obs_bf16_out, void* stream)
{
    return launch_opponent<false>(h, state, require_two, player_score, reward_out, done_out, status_out, mask6_out,
                                  obs_bf16_out, stream);
}

int azb_opponent_greedy(azb_t* h, uint32_t* state, int require_two, int16_t* player_score, int16_t* reward_out,
                        uint8_t* done_out, uint8_t* status_out, uint32_t* mask6_out, void* obs_bf16_out, void* stream)
{
    return launch_opponent<true>(h, state, require_two, player_score, reward_out, done_out, status_out, mask6_out,
                                 obs_bf16_out, stream);
}

int azb_greedy_action(azb_t* h, const uint32_t* state, uint8_t* action_out, void* stream)
{
    CHECK_HANDLE(h);
    if (!state || !action_out) return azb_fail(AZB_E_INVALID, "null buffer%s");
    const Launch L = make_launch(h, const_cast<uint32_t*>(state));
    DISPATCH_PP(h, (k_greedy_action<P, POOL><<<grid_of(h), h->block_threads, 0, (cudaStream_t)stream>>>(L, action_out)));
    CHECK_LAUNCH();
    return 0;
}

int azb_round_flags(azb_t* h, const uint32_t* state, uint8_t* flags, void* stream)
{
    CHECK_HANDLE(h);
    if (!state || !flags) return azb_fail(AZB_E_INVALID, "null buffer%s");
    DISPATCH_P(h, (k_round_flags<P><<<grid_of(h), h->block_threads, 0, (cudaStream_t)stream>>>(state, h->n_games, flags)));
    CHECK_LAUNCH();
    return 0;
}

}  // extern "C"
