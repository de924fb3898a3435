// azb_policy.cu -- K4: the ActorCritic MLP (reference azulnet/model.py:12-41) fused with the
// observation builder (game_runner.py:56-72), masked softmax / log-softmax (model.py:37-40),
// action sampling (agent.py:64-81), the entropy term of nn_runner.py:36-40 and, optionally, the
// env step, for a batch of 2-player games.
//
// Shape of the work: 128 games per tile, one tile per pass of a persistent CTA of 512 threads: thread t
// works on game (row) t & 127 and on column part t >> 7 (four threads share a game and split the
// epilogue columns 4 x 48, so that an SM holds 16 warps although shared memory allows one CTA).
//   layer 1   [128 x 144] x [144 x 368]   obs (136, zero-padded to 144) times [W1_actor ; W1_critic]^T
//             (180 + 180 hidden units back to back, padded to 368; two MMAs of N = 192 + 176)
//                                                                              -> TMEM columns [0,368)
//   layer 2   [128 x 192] x [192 x 192]   relu(hidden_actor) times W2_actor^T   -> TMEM columns [0,192)
//   critic    value = w2c . relu(hidden_critic) + b2c on CUDA cores straight from the TMEM row
// Both dense layers run on the 5th-generation tensor cores: tcgen05.mma (kind::f16, fp16 inputs, fp32
// accumulate in TMEM), issued by one thread, operands in shared memory in the canonical K-major
// no-swizzle core-matrix layout, accumulators read back with tcgen05.ld 32x32b (thread t <- TMEM lane t,
// i.e. every thread receives exactly the row of its own game, so softmax and sampling need no
// cross-thread traffic).  The fp16 weights (180 KB) stay resident in shared memory for the lifetime of
// the CTA; the observation tile is generated in-kernel from the packed state and never touches HBM.
#include <cuda_fp16.h>
#include <stdlib.h>

#include "azb_internal.h"
#include "azb_rules.cuh"
#include "azb_tc.cuh"

namespace pol {

struct PolicyArgs {
    const uint32_t* __restrict__ state_in;   // packed state (read)
    uint32_t* __restrict__ state;            // packed state (written when apply_step)
    int64_t n;
    const unsigned char* __restrict__ packed;
    uint32_t k0, k1, gid0;
    int mode;            // 0 sample from the masked policy, 1 argmax (agent.py action_selection)
    int apply_step;      // 1: also execute Azul.step with the chosen action (Philox refill); 2: and start a fresh game when it ends
    int first_rule;
    int act_filter;      // 0 every game decides; 1 only games where it is NOT (seat 1 to move with >= 2 legal actions),
                         // i.e. the opponent's turns of GameRunner.step (game_runner.py:46); 2 only the agent's turns
    unsigned long long* __restrict__ counters;   // rollout counters (apply_step == 2), may be null
    float* __restrict__ logits_out;          // [n][180] raw logits (debug / parity), may be null
    float* __restrict__ value_out;           // [n]
    uint8_t* __restrict__ action_out;        // [n]
    float* __restrict__ logp_out;            // [n] log pi(action)
    float* __restrict__ entropy_out;         // [n] -mean(log pi over legal actions) (nn_runner.py:36-40)
    uint8_t* __restrict__ done_out;          // [n]
    uint8_t* __restrict__ status_out;        // [n]
    uint32_t* __restrict__ mask6_out;        // [6][n] legal mask used for the decision
    // ---- persistent form (azb_policy_rollout): k_decisions decisions per game in one launch, state resident ----
    int k_decisions;     // >= 1; the per-game outputs above then hold the LAST decision
    int runner_mode;     // 0 self-play (every seat decides); 1 GameRunner.step semantics (game_runner.py:43-55): after each
                         // decision the random opponent moves until seat 1 is to move with >= 2 legal actions, the reward is taken
                         // and the decision is recorded; an ended game stays ended (one episode per slot)
    int16_t* __restrict__ player_score;      // [n] runner mode: GameRunner.player_score (game_runner.py:52)
    // decision records of the runner mode.  Compact: slot = atomic counter n_dec (device), capacity rec_cap
    uint32_t* __restrict__ n_dec;            // [1]
    int64_t rec_cap;
    uint32_t* __restrict__ state_rec;        // [17][rec_cap] packed state the decision was taken on (update kernel input)
    uint8_t* __restrict__ action_rec;        // [rec_cap]
    float* __restrict__ logp_rec;            // [rec_cap] optional
    float* __restrict__ value_rec;           // [rec_cap] optional
    // per (decision index, game): [k_decisions][n]
    int32_t* __restrict__ slot_rec;          // compact slot of the decision, -1 when the game took none
    int16_t* __restrict__ reward_rec;        // GameRunner.step reward (game_runner.py:51)
    uint8_t* __restrict__ flags_rec;         // bit 0 a decision was taken, bit 1 game over after it
    uint32_t* __restrict__ steps_used;       // [1] optional: max over CTAs of the decision iterations actually run
    // ---- runner mode against a frozen policy opponent (azb_policy_rollout_vs_policy, k_policy<..., OPP = true>) ----
    const unsigned char* __restrict__ opponent_packed;   // the opponent's weight image (seat 2 and seat 1's forced moves)
    uint32_t* __restrict__ opp_passes;       // [1] optional: max over CTAs and decisions of the opponent passes in one decision
};

constexpr uint32_t PURPOSE_POLICY = 4;
constexpr int TM_H = 384;                    // tensor-memory columns [384, 480): the fp16 hidden tile, layer 2's A operand
static_assert(CRITIC_SHIFT + 16 * 10 + 16 <= 192 && TM_H >= N1 + 8 && TM_H + K2 / 2 <= (int)TMEM_COLS, "tensor-memory map");
// transient MISC bits between k_policy's tile loop and its finishing phase (never visible outside azb_policy_step)
constexpr uint32_t FLAG_ROUND_OVER = 1u << 28, FLAG_FRESH_GAME = 1u << 29;

struct SmemSink {
    unsigned long long* c;
    __device__ __forceinline__ void add(int i, uint32_t v)
    {
        if (v) atomicAdd(&c[i], (unsigned long long)v);
    }
    __device__ __forceinline__ void add_group(int i, uint32_t v) { add(i, v); }
};

// Completes the step of one game whose move k_policy applied: count_score, game-over test and new_round (azul.py:307-311)
// when its round ended, a fresh game for a finished / stuck slot in self-play mode; finalises done / status.
template <int POOL>
__device__ __forceinline__ void finish_game(Game<2>& h, uint32_t gidx, uint32_t flags, const Philox& rng, uint32_t gid0,
                                            int first_rule, bool auto_reset, uint32_t* __restrict__ state, int64_t n,
                                            uint8_t* __restrict__ done_out, uint8_t* __restrict__ status_out, SmemSink& sink)
{
    const uint32_t gid = gid0 + gidx;
    bool over = false, fresh = (flags & FLAG_FRESH_GAME) != 0u;
    if (flags & FLAG_ROUND_OVER) {
        count_score<2, POOL>(h);                                  // azul.py:307
        over = is_end_of_game(h);                                 // azul.py:308-309
        if (over) h.misc |= 1u << 12;
    }
    if (done_out) done_out[gidx] = h.ended() ? 1 : 0;
    if (over && auto_reset) { tally_finished(h, sink); fresh = true; }
    if (fresh) {
        reset_game<2, POOL>(h, rng, gid, first_rule);
        if (auto_reset) sink.add(2, 1);
    } else if (!over) {
        new_round_philox<2, POOL>(h, rng, gid, PURPOSE_REFILL);   // azul.py:311
        if (auto_reset) sink.add(2, 1);
    }
    h.store(state, n, (int64_t)gidx);
    if (status_out) status_out[gidx] |= (uint8_t)h.status();
}

// GameRunner.step's opponent loop (game_runner.py:46-52; opponent_random() / opponent_greedy() in azb_rules.cuh are the one-game
// forms) for the 32 games of a warp TOGETHER, with the random agent's or -- GREEDY -- the greedy agent's pick: every lane makes the same sequence of rule calls on its own game as the one-game form, but a game
// whose round ended -- by the agent's move (`pending`) or by an opponent move -- waits until no lane of the warp can move any
// more, and ONE count_score + refill pass serves all of them (the rollout kernel's light / heavy split).  Run one game at a
// time under divergence, the ~1,300-instruction pass was walked by the warp once for the agent's move and again at every
// loop iteration in which some lane's opponent move ended a round.  Inactive lanes take part in the votes only.
template <int POOL, bool GREEDY>
__device__ __forceinline__ int32_t opponent_warp(Game<2>& h, const Philox& rng, uint32_t gid, bool active, bool pending,
                                                 uint32_t m[6])
{
    int phase = !active ? 2 : pending ? 1 : 0;            // 0 to move, 1 round over: waits for the pass, 2 handed back
    for (;;) {
        if (phase == 0) {
            legal_mask(h, m);
            if (h.ended()) {
                phase = 2;
            } else {
                const int n_valid = popc(m[0]) + popc(m[1]) + popc(m[2]) + popc(m[3]) + popc(m[4]) + popc(m[5]);
                if (h.current_player() == 1u && n_valid >= 2) {
                    phase = 2;                                             // seat 1 decides again (game_runner.py:46)
                } else if (n_valid == 0) {
                    h.add_status(ST_STUCK);
                    phase = 2;
                } else {
                    uint32_t w[4];
                    rng(gid, h.steps >> 2, PURPOSE_ACTION, 0u, w);
                    const uint32_t idx = h.steps & 3u;
                    const uint32_t word = idx == 0u ? w[0] : idx == 1u ? w[1] : idx == 2u ? w[2] : w[3];
                    apply_move<2, POOL>(h, opponent_pick<2, POOL, GREEDY>(h, m, word));   // azul.py:304
                    h.steps += 1u;
                    if (is_end_of_round(h)) phase = 1;                     // azul.py:306
                    else next_player(h);                                   // azul.py:313
                }
            }
        }
        if (__any_sync(0xFFFFFFFFu, phase == 0)) continue;
        if (!__any_sync(0xFFFFFFFFu, phase == 1)) break;
        if (phase == 1) {
            count_score<2, POOL>(h);                                       // azul.py:307
            if (is_end_of_game(h)) h.misc |= 1u << 12;                     // azul.py:308-309
            else new_round_philox<2, POOL>(h, rng, gid, PURPOSE_REFILL);   // azul.py:311
            phase = 0;
        }
    }
    Game<2> cp = h;                                                        // game_runner.py:48-50: score preview on a copy
    count_score<2, POOL>(cp);
    return (int32_t)(cp.scf[0] & 0xFFFFu) - (int32_t)(cp.scf[1] & 0xFFFFu);
}

// The loop condition of GameRunner.step (game_runner.py:46) for a game whose round is not pending: the opponent is to move
// (or seat 1 has a single legal action), the game is not over and has a legal action, and no earlier bound froze it.
__device__ __forceinline__ bool opponent_to_move(const Game<2>& h)
{
    if (h.ended() || (h.status() & ST_STUCK)) return false;
    uint32_t m[6];
    legal_mask(h, m);
    const int n_valid = popc(m[0]) + popc(m[1]) + popc(m[2]) + popc(m[3]) + popc(m[4]) + popc(m[5]);
    return n_valid > 0 && !(h.current_player() == 1u && n_valid >= 2);
}

// Thread 0: the fp16 weight image `src` -> shared memory [0, PACKED_BYTES) as chunked bulk async copies completing on bar_w.
__device__ __forceinline__ void issue_image_copy(unsigned char* smem, const unsigned char* src, uint32_t bar_w)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar_w), "r"((uint32_t)PACKED_BYTES) : "memory");
    constexpr uint32_t CHUNK = 32768;
    for (uint32_t off = 0; off < (uint32_t)PACKED_BYTES; off += CHUNK) {
        const uint32_t bytes = (uint32_t)PACKED_BYTES - off < CHUNK ? (uint32_t)PACKED_BYTES - off : CHUNK;
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                     ::"r"(smem_u32(smem) + off), "l"(src + off), "r"(bytes), "r"(bar_w) : "memory");
    }
}

// bits [start, start + 48) of the 180-bit linear mask; start is 0, 48, 96 or 144
__device__ __forceinline__ uint64_t mask_window(const uint32_t (&lin)[6], int start)
{
    const int w = start >> 5, sh = start & 31;
    const uint64_t x = (((uint64_t)pick6(lin, w + 1) << 32) | pick6(lin, w)) >> sh;
    return x & 0xFFFFFFFFFFFFull;
}

// cross-part scratch: lives in the tail of the A region (dead once the layer-2 MMA has read the hidden tile), behind
// the first 36,864 bytes that the NEXT tile's observation is written to while the owner threads play this tile's moves
struct RowPart { float m, s, sl, value; int amax, n; };
constexpr int OBS_TILE_BYTES = K1_CHUNKS * M_GROUPS * 128;
constexpr int OFF_PARTS = OBS_TILE_BYTES;                                // RowPart[PARTS][TILE_M] as 5 words each
constexpr int PART_WORDS = 5;                                            // m, s, sl, value, amax | n << 8
constexpr int OFF_RESULT = OFF_PARTS + PARTS * TILE_M * PART_WORDS * 4;  // int2[TILE_M]: sampled action, logit bits
constexpr int OFF_SAMPLE = OFF_RESULT + TILE_M * 8;                      // uint32[TILE_M]: the row's Philox word (computed by part 0)
static_assert(OFF_SAMPLE + TILE_M * 4 <= A_BYTES, "scratch exceeds the A tile");

__device__ __forceinline__ RowPart load_part(const float* parts, int slot)
{
    RowPart rp;
    rp.m = parts[0 * THREADS + slot]; rp.s = parts[1 * THREADS + slot]; rp.sl = parts[2 * THREADS + slot];
    rp.value = parts[3 * THREADS + slot];
    const int an = __float_as_int(parts[4 * THREADS + slot]);
    rp.amax = an & 255; rp.n = an >> 8;
    return rp;
}

// FULL: the single-step entry point (azb_policy_step) with its optional diagnostics -- raw logits and the entropy term;
// the persistent rollouts (azb_policy_rollout) never ask for either, and the sum of the legal logits that the entropy
// needs is 2 of the 6.5 instructions per logit of the softmax pass (measured: 31 % of that pass).
// OPP: the runner mode against a frozen policy opponent (azb_policy_rollout_vs_policy).  Each decision iteration is a pass of
// the tile loop with the agent's image resident (act_filter 0, records), then -- with the opponent's image copied over it --
// passes with act_filter 1 and no records until no game of the CTA is in the opponent's hands, then the runner block, whose
// random opponent then has nothing to play; the agent's image comes back for the next decision.
// GREEDY: the runner mode against the greedy agent (azb_policy_rollout_vs_greedy): the runner block's opponent loop picks the
// greedy agent's moves instead of the random agent's; nothing else differs.
constexpr int MAX_OPP_PASSES = 64;           // the bound of the eager loop (selfplay.py _opponent_policy_moves)
template <int POOL, int MODE, bool FULL, bool OPP = false, bool GREEDY = false>
__global__ void __launch_bounds__(THREADS, 1) k_policy(PolicyArgs A)
{
    static_assert(!(GREEDY && OPP), "one opponent per launch: a frozen network or the greedy agent");
    extern __shared__ __align__(128) unsigned char smem[];
    const int tid = threadIdx.x, warp = tid >> 5, row = tid & (TILE_M - 1), part = tid >> 7;
    unsigned char* a_tile = smem + OFF_A;
    const float* vec = reinterpret_cast<const float*>(smem + OFF_VEC);
    const uint32_t bar1 = smem_u32(smem + OFF_BAR), bar2 = bar1 + 8;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + OFF_BAR + 16);
    float* parts = reinterpret_cast<float*>(a_tile + OFF_PARTS);     // [word][part][row]: conflict-free
    int2* result = reinterpret_cast<int2*>(a_tile + OFF_RESULT);
    uint32_t* sample = reinterpret_cast<uint32_t*>(a_tile + OFF_SAMPLE);
    __shared__ unsigned long long cnt[AZB_N_COUNTERS];
    __shared__ uint64_t bar3_storage;                      // layer 1, critic half (bar1: actor half)
    __shared__ uint32_t n_list;                            // length of the finishing phase's list
    const uint32_t bar3 = smem_u32(&bar3_storage);
    if (tid < AZB_N_COUNTERS) cnt[tid] = 0ull;
    SmemSink sink{cnt};

    // one-time: barriers, tensor memory, and the weight image -> shared memory as bulk async copies (TMA, no registers
    // and no thread time: the first observation tile is built while the 180 KB arrive)
    const uint32_t bar_w = bar1 + 24;
    // Programmatic dependent launch: this grid may be scheduled while the previous kernel of the stream is still draining
    // (its launch latency, barrier setup and TMEM allocation then overlap that tail); nothing the previous kernel may have
    // written -- game state, the weight image -- is read before this point.  The next grid is released right away: it
    // cannot get an SM before one of this grid's CTAs exits, and it waits here too.
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    if (tid == 0) {
        mbar_init(bar1, 1);
        mbar_init(bar2, 1);
        mbar_init(bar3, 1);
        mbar_init(bar_w, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    asm volatile("griddepcontrol.wait;" ::: "memory");
    if (tid == 0) issue_image_copy(smem, A.packed, bar_w);
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    const uint32_t tmem_row = tmem_base + ((uint32_t)((warp & 3) * 32) << 16);   // a warp reaches TMEM lanes 32*(warp%4)..+31
    // The critic head reads 16-column chunks up to column HID + 191 = 371; layer 1 writes [0, 368).  Zero the tail once so
    // that the (zero-weight) products of those columns are 0 and not NaN.
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %1, %1, %1, %1, %1, %1, %1};" ::"r"(tmem_row + N1), "r"(0u) : "memory");
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");

    const uint32_t w1_addr = smem_u32(smem + OFF_W1), w2_addr = smem_u32(smem + OFF_W2), a_addr = smem_u32(a_tile);
    const Philox rng{A.k0, A.k1};
    uint32_t phase = 0;
    const int64_t tiles = (A.n + TILE_M - 1) / TILE_M;
    const int col0 = part * PART_COLS;                 // this thread's 48 epilogue columns
    auto quad_sync = [&]() { asm volatile("bar.sync %0, %1;" ::"r"(3 + (warp & 3)), "n"(TILE_M) : "memory"); };

    // Persistent form: a CTA owns the tiles blockIdx.x + j * gridDim.x for the whole launch and takes k_decisions decisions for
    // each of their games; between decisions the packed state stays in global memory (L2-resident: 68 B per game), written and
    // re-read by this CTA only, so block barriers order everything.
    const int64_t my_tiles = (int64_t)blockIdx.x < tiles ? (tiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;

    // ---- the rare, long part of Azul.step for this CTA's own games: the ones flagged by the tile loop (round over / fresh
    // game) are collected into a dense list (the A region is free then) and finished 32 per warp with every lane busy,
    // instead of under divergence inside the tile loop or in a second kernel launch.  OPP: `need` collects whether a
    // finished game is in the opponent's hands in its new round ----
    auto finish_flagged = [&](uint8_t* __restrict__ done_o, uint8_t* __restrict__ status_o, bool& need) {
        // the list holds at most FINISH_GROUP tiles' worth of games (every game of a tile can be flagged, e.g. when a whole
        // batch asks for fresh games), so a CTA with more tiles than that works through them in groups
        constexpr int FINISH_GROUP = A_BYTES / 4 / TILE_M / PARTS * PARTS;         // 96 tiles = 12,288 entries
        static_assert(FINISH_GROUP >= PARTS && FINISH_GROUP * TILE_M * 4 <= A_BYTES, "finish list exceeds the A region");
        uint32_t* list = reinterpret_cast<uint32_t*>(a_tile);
        for (int64_t j0 = 0; j0 < my_tiles; j0 += FINISH_GROUP) {
            if (tid == 0) n_list = 0u;
            __syncthreads();
            const int64_t j1 = j0 + FINISH_GROUP < my_tiles ? j0 + FINISH_GROUP : my_tiles;
            for (int64_t j = j0 + part; j < j1; j += PARTS) {
                const int64_t g = ((int64_t)blockIdx.x + j * gridDim.x) * TILE_M + row;
                if (g < A.n && (A.state[3 * A.n + g] & (FLAG_ROUND_OVER | FLAG_FRESH_GAME))) list[atomicAdd(&n_list, 1u)] = (uint32_t)g;
            }
            __syncthreads();
            const uint32_t total = n_list;
            for (uint32_t i = (uint32_t)tid; i < total; i += THREADS) {
                const uint32_t gidx = list[i];
                Game<2> h;
                h.load(A.state, A.n, (int64_t)gidx);
                const uint32_t flags = h.misc & (FLAG_ROUND_OVER | FLAG_FRESH_GAME);
                h.misc &= ~(FLAG_ROUND_OVER | FLAG_FRESH_GAME);
                finish_game<POOL>(h, gidx, flags, rng, A.gid0, A.first_rule, A.apply_step == 2, A.state, A.n, done_o, status_o, sink);
                if (OPP) need |= opponent_to_move(h);
            }
            __syncthreads();                           // the list is reused by the next group
        }
    };

    int it = 0;
    uint32_t w_phase = 0u, max_opp = 0u;               // OPP: parity of bar_w's next completion; most opponent passes
    bool w_pending = true, opp_image = false;          // OPP: an image copy to wait for; the opponent's image is resident
    for (; it < A.k_decisions; it++) {
    for (int pass = 0;; pass++) {                      // OPP: pass 0 takes the agent's decisions, passes >= 1 the opponent's
    const bool record = !OPP || pass == 0;             // decision records and per-game outputs: the agent's pass only
    bool need = false;                                 // OPP: a game this thread moved is (still) in the opponent's hands
    // software pipeline over tiles: the next tile's state is loaded during this tile's epilogues and its observation
    // is built by parts 1..3 while part 0 plays this tile's moves
    // (the next tile's state is held as the 17 RAW words: Game::load unpacks the MISC word on the spot, and that first use
    // made every thread sit out the L2 round trip right behind the loads -- 3 % of the kernel's stall samples)
    uint32_t nraw[Game<2>::WORDS];
    auto load_raw = [&](int64_t g1) {
#pragma unroll
        for (int i = 0; i < Game<2>::WORDS; i++) nraw[i] = A.state_in[i * A.n + g1];
    };
    if ((int64_t)blockIdx.x < tiles) {
        const int64_t g0 = (int64_t)blockIdx.x * TILE_M + row;
        load_raw(g0 < A.n ? g0 : A.n - 1);
        Game<2> first;
        first.load(nraw, 1, 0);
        build_obs_tile(first, a_tile, row, part);
    }
    if (OPP ? w_pending : it == 0) {                       // weights and vectors have landed (every thread reads the vectors)
        mbar_wait(bar_w, OPP ? w_phase : 0u);
        if (OPP) { w_phase ^= 1u; w_pending = false; }
    }
    for (int64_t tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
        const int64_t g = tile * TILE_M + row;
        const bool valid = g < A.n;
        const int64_t gl = valid ? g : A.n - 1;
        Game<2> gm;
        gm.load(nraw, 1, 0);
        const bool has_next = tile + gridDim.x < tiles;

        // ---- layer 1 on the tensor cores.  For the first tile of a decision round the observation was built by all four
        // parts in the prologue: one block barrier, then thread 0 issues.  For every later tile parts 1..3 built it during
        // the previous tile's last epilogue and thread 128 issued the MMAs right there (see the end of the loop body): the
        // MMAs start while part 0 still plays the previous tile's moves (+1.4 % decisions/s; building the observation even
        // earlier -- right after layer 2, by all four parts -- and issuing before epilogue 2c was measured and is no faster) ----
        // (descriptors: the start-address field advances by a constant per k-step and never carries out of its 14 bits -- shared
        // memory ends below 2^18 bytes -- so the loop is unrolled into one add per descriptor; the rolled loop rebuilt each
        // descriptor from the byte address, ~35 dependent uniform-datapath instructions per k-step on the one issuing thread)
        auto issue_layer1 = [&]() {
            tc_fence_after();
            const uint64_t ad0 = smem_desc(a_addr, M_GROUPS * 128, 128);
            const uint64_t ba0 = smem_desc(w1_addr, N1_GROUPS * 128, 128);
            const uint64_t bc0 = smem_desc(w1_addr + (N1A / 8) * 128, N1_GROUPS * 128, 128);
            // the actor half first, with its own commit: epilogue 1 only needs that half, and since the hidden tile goes to
            // tensor memory (below) it no longer overwrites the observation tile that the critic half is still reading
#pragma unroll
            for (int s = 0; s < K1 / 16; s++)
                umma(tmem_base, ad0 + (uint64_t)(s * ((2 * M_GROUPS * 128) >> 4)), ba0 + (uint64_t)(s * ((2 * N1_GROUPS * 128) >> 4)),
                     instr_desc(N1A), s > 0);
            umma_commit(bar1);
#pragma unroll
            for (int s = 0; s < K1 / 16; s++)
                umma(tmem_base + N1A, ad0 + (uint64_t)(s * ((2 * M_GROUPS * 128) >> 4)), bc0 + (uint64_t)(s * ((2 * N1_GROUPS * 128) >> 4)),
                     instr_desc(N1C), s > 0);
            umma_commit(bar3);
        };
        if (tile == (int64_t)blockIdx.x) {
            fence_async_smem();
            tc_fence_before();
            __syncthreads();
            if (tid == 0) issue_layer1();
        }
        if (has_next) {                                    // in flight while the epilogues run
            const int64_t g2 = (tile + gridDim.x) * TILE_M + row;
            load_raw(g2 < A.n ? g2 : A.n - 1);
        }
        mbar_wait(bar1, phase);
        tc_fence_after();

        // ---- epilogue 1: actor hidden -> relu -> fp16 -> TENSOR memory columns [TM_H, TM_H + 96): the layer-2 A operand
        // (row = lane, two hidden units per column).  Shared memory could only hold it on top of the observation tile ----
#pragma unroll 1
        for (int c0 = col0; c0 < col0 + PART_COLS; c0 += 16) {
            float v[16];
            tmem_ld16(tmem_row + c0, v);                               // b1 is already in the accumulator (BIAS_K1)
            uint32_t o[8];
#pragma unroll
            for (int e = 0; e < 8; e++) {
                const int j = c0 + 2 * e;                              // hidden unit (even, so j and j + 1 are both < or >= 180)
                o[e] = j < HID ? pack_relu_f16(v[2 * e], v[2 * e + 1])
                               : (j == BIAS_K2 ? 0x3C003C00u : 0u);    // the two constant-one units that carry b2
            }
            tmem_st8(tmem_row + TM_H + (c0 >> 1), o);
        }
        // ---- critic head, partial sum over this part's units.  Critic units 176..179 sit in columns 180..183 of the ACTOR
        // half (which layer 2 overwrites): part 0 reads them now; units 0..175 are columns [192,368) of the critic half, read
        // in eleven 16-column chunks WHILE the layer-2 MMAs run (part 0 two, parts 1..3 three each) ----
        float value_p = 0.0f;
        auto critic_chunk = [&](int k) {                               // columns 192 + 16 k .. + 15 = units 16 k .. + 15
            float v[16], ww[16];
            tmem_ld16(tmem_row + N1A + 16 * k, v);
            ld16f(vec + V_W2C + CRITIC_SHIFT + 16 * k, ww);
#pragma unroll
            for (int i = 0; i < 16; i++) value_p = fmaf(fmaxf(v[i], 0.0f), ww[i], value_p);
        };
        if (part == 0) {
            float v[16];
            tmem_ld16(tmem_row + HID - 4, v);                          // columns 176..191: [4..7] are critic units 176..179
#pragma unroll
            for (int i = 0; i < 4; i++) value_p = fmaf(fmaxf(v[4 + i], 0.0f), vec[V_W2C + i], value_p);
        }
        tc_wait_st();
        tc_fence_before();
        __syncthreads();

        // ---- layer 2 on the tensor cores: A from tensor memory ----
        if (tid == 2 * TILE_M) {                           // a warp of part 2: part 0 has the Philox word, warp 4 the layer-1 issue
            tc_fence_after();
            const uint64_t bd0 = smem_desc(w2_addr, N2_GROUPS * 128, 128);
#pragma unroll
            for (int s = 0; s < K2 / 16; s++)
                umma_ts(tmem_base, tmem_base + TM_H + 8 * s, bd0 + (uint64_t)(s * ((2 * N2_GROUPS * 128) >> 4)), instr_desc(N2), s > 0);
            umma_commit(bar2);
        }
        // while the layer-2 MMAs run: everything the epilogue needs that does not depend on the logits -- the legal
        // mask of the game, this part's 48-bit window of it, and the Philox word of the sampling step
        uint32_t m[6], lin[6];
        legal_mask(gm, m);
        linear_mask(m, lin);
        const uint64_t mybits = mask_window(lin, col0);
        uint32_t sample_word = 0u;
        if (MODE == 0 && part == 0) {                     // one Philox per game, not four: the other parts read it from the scratch
            uint32_t w[4];
            rng(A.gid0 + (uint32_t)gl, gm.steps >> 2, PURPOSE_POLICY, 0u, w);
            const uint32_t idx = gm.steps & 3u;
            sample_word = idx == 0u ? w[0] : idx == 1u ? w[1] : idx == 2u ? w[2] : w[3];
        }
        mbar_wait(bar3, phase);                            // the critic half of layer 1 (long done: it ran under epilogue 1)
        tc_fence_after();
#pragma unroll 1
        for (int k = part == 0 ? 0 : 3 * part - 1; k < 3 * part + 2; k++) critic_chunk(k);
        mbar_wait(bar2, phase);
        tc_fence_after();
        phase ^= 1;

        // ---- epilogue 2a: per part -- critic partial sum and online softmax over its 48 columns ----
        // online softmax statistics over this part's legal logits, one 16-column chunk at a time and without
        // per-column branches (32 different games share a warp): chunk maximum first, one rescale, then the sum.
        // The chunk sums (relative to the running maximum at that chunk) are kept for the sampling step.
        float mx = -INFINITY, se = 0.0f, sl = 0.0f;
        float cs[3], cms[3];
        int amax = 0;
#pragma unroll
        for (int c = 0; c < PART_COLS / 16; c++) {
            const int c0 = col0 + 16 * c;
            float v[16];
            tmem_ld16(tmem_row + c0, v);                               // b2 is already in the accumulator (BIAS_K2)
            const uint32_t bits = (uint32_t)(mybits >> (16 * c)) & 0xFFFFu;
            if (FULL && A.logits_out && valid) {
#pragma unroll
                for (int i = 0; i < 16; i++)
                    if (c0 + i < ACT) A.logits_out[g * ACT + c0 + i] = v[i];
            }
            float cm = -INFINITY;
            int ci = 0;
#pragma unroll
            for (int i = 0; i < 16; i++) {
                const bool legal = (bits >> i) & 1u;
                const float l = v[i];
                v[i] = legal ? l : -INFINITY;
                if (FULL) sl += legal ? l : 0.0f;
                if (MODE == 1) { if (v[i] > cm) { cm = v[i]; ci = i; } }      // argmax mode tracks the index
                else cm = fmaxf(cm, v[i]);
            }
            if (MODE == 1) amax = cm > mx ? c0 + ci : amax;
            const float nm = fmaxf(mx, cm);
            const float ms = nm == -INFINITY ? 0.0f : nm;          // no legal action so far: every term below is 2^-inf = 0
            const float ms2 = ms * LOG2E;
            float sum = 0.0f;
#pragma unroll
            for (int i = 0; i < 16; i++) { v[i] = ex2f(fmaf(v[i], LOG2E, -ms2)); sum += v[i]; }
            // sampling mode: the weights 2^(logit - chunk maximum) -- exactly 0 for an illegal action -- replace the logits in
            // TMEM, so that the inverse-CDF scan below neither repeats the exponentials nor looks at the mask again
            if (MODE == 0) tmem_st16(tmem_row + c0, v);
            se = se * ex2f(fmaf(mx, LOG2E, -ms2)) + sum;
            cs[c] = sum; cms[c] = ms;
            mx = nm;
        }
        if (MODE == 0) tc_wait_st();
        {
            const int slot = part * TILE_M + row;
            parts[0 * THREADS + slot] = mx; parts[1 * THREADS + slot] = se; parts[2 * THREADS + slot] = sl;
            parts[3 * THREADS + slot] = value_p;
            parts[4 * THREADS + slot] = __int_as_float(amax | (__popcll(mybits) << 8));
            if (part == 0) { result[row] = make_int2(-1, 0); sample[row] = sample_word; }
        }
        tc_fence_before();
        // the scratch is exchanged between the four threads of a ROW only: the four warps that share rows 32 q .. 32 q + 31
        // (warps q, q + 4, q + 8, q + 12) meet at a named barrier of their own instead of waiting for all sixteen
        quad_sync();

        // ---- epilogue 2b: merge the four parts of the row (every thread of the row computes the same numbers) ----
        float gmx = -INFINITY, gsl = 0.0f, value = vec[V_B2C];
        int n_valid = 0, gamax = 0;
#pragma unroll
        for (int q = 0; q < PARTS; q++) {
            const RowPart rp = load_part(parts, q * TILE_M + row);
            if (rp.n > 0 && rp.m > gmx) { gmx = rp.m; gamax = rp.amax; }
            gsl += rp.sl; value += rp.value; n_valid += rp.n;
        }
        // slices of the cumulative distribution: part q owns [run_{q-1}, run_q); every thread of the row adds the
        // same numbers in the same order, so the four threads agree on the owner bit for bit
        float gse = 0.0f, prefix = 0.0f;
        float wq[PARTS];
        int last_part = 0;
#pragma unroll
        for (int q = 0; q < PARTS; q++) {
            const RowPart rp = load_part(parts, q * TILE_M + row);
            wq[q] = rp.n > 0 ? rp.s * ex2f((rp.m - gmx) * LOG2E) : 0.0f;
            if (rp.n > 0) last_part = q;
            if (q < part) prefix += wq[q];
            gse += wq[q];
        }
        const float lse = gmx + __logf(gse);
        if (MODE == 0) {
            // inverse-CDF sampling with one Philox word (agent.py:69 np.random.choice(p = policy)): the part that owns the
            // target, then the 16-column chunk inside it (from the chunk sums), then a branch-free scan of that chunk only.
            // tcgen05.ld is warp-collective and the chunk differs from lane to lane, so every lane loads its three chunks
            // and keeps the one it needs by selects.
            const float target = (float)(sample[row] >> 8) * (1.0f / 16777216.0f) * gse;
            int owner = -1;
            float run = 0.0f;
#pragma unroll
            for (int q = 0; q < PARTS; q++) {
                run += wq[q];
                if (owner < 0 && target < run) owner = q;
            }
            if (owner < 0) owner = last_part;
            const bool mine = owner == part && n_valid > 0;
            const float gm2 = (n_valid > 0 ? gmx : 0.0f) * LOG2E;
            // chunk k: the first whose cumulative weight passes the target; `base` = weight before it (<= target)
            float sc[3], wc[3];
#pragma unroll
            for (int c = 0; c < 3; c++) { sc[c] = ex2f(fmaf(cms[c], LOG2E, -gm2)); wc[c] = cs[c] * sc[c]; }
            int k = -1;
            float base = prefix, acc = prefix;
#pragma unroll
            for (int c = 0; c < 3; c++) {
                const float nacc = acc + wc[c];
                const bool hit = k < 0 && target < nacc;
                base = hit ? acc : base;
                k = hit ? c : k;
                acc = nacc;
            }
            if (k < 0) {                                   // rounding left the target beyond the part: its last legal chunk
                k = (mybits >> 32) ? 2 : ((mybits >> 16) & 0xFFFFull) ? 1 : 0;
                base = prefix + (k > 0 ? wc[0] : 0.0f) + (k > 1 ? wc[1] : 0.0f);
            }
            const float sk = k == 0 ? sc[0] : k == 1 ? sc[1] : sc[2], mk = k == 0 ? cms[0] : k == 1 ? cms[1] : cms[2];
            float vs[16];                                  // the chunk's weights relative to its own maximum mk (epilogue 2a)
#pragma unroll
            for (int c = 0; c < 3; c++) {
                float v[16];
                tmem_ld16(tmem_row + col0 + 16 * c, v);
                const bool take = c == 0 || c == k;
#pragma unroll
                for (int i = 0; i < 16; i++) vs[i] = take ? v[i] : vs[i];
            }
            float cum = base, chosen_e = 1.0f;
            int chosen = -1;
#pragma unroll
            for (int i = 0; i < 16; i++) {
                // an action with weight 0 (illegal, or underflowed) is never chosen; rounding may leave cum <= target to the
                // end: then the chunk's last action of positive weight
                const bool upd = vs[i] > 0.0f && cum <= target;
                chosen = upd ? i : chosen;
                chosen_e = upd ? vs[i] : chosen_e;
                cum = fmaf(vs[i], sk, cum);
            }
            const float chosen_l = fmaf(lg2f(chosen_e), LN2, mk);        // the logit back from its weight: l = mk + ln(e)
            if (mine && chosen >= 0) result[row] = make_int2(col0 + 16 * k + chosen, __float_as_int(chosen_l));
        }
        tc_fence_before();
        quad_sync();                                       // (the layer-1 issue below still follows a barrier of ALL part 1..3 warps,
                                                           // each of which has met its part-0 warp here: every TMEM read is over)

        // ---- epilogue 2c: one thread per game publishes the decision and plays the move ----
        bool issuer = false;                               // warp-uniform: this warp issues the next tile's layer 1 (below)
        if (part == 0) {
            uint32_t action = (uint32_t)gamax;
            float la = gmx;                             // argmax mode, and the fallback if rounding left no part a winner
            if (MODE == 0) {
                const int2 r = result[row];
                if (r.x >= 0) { action = (uint32_t)r.x; la = __int_as_float(r.y); }
            }
            const float logp = n_valid > 0 ? la - lse : 0.0f;
            const float entropy = n_valid > 0 ? -(gsl / (float)n_valid - lse) : 0.0f;
            uint32_t status = n_valid > 0 ? 0u : (gm.ended() ? (uint32_t)ST_ENDED : (uint32_t)ST_STUCK);
            const bool agent_turn = gm.current_player() == 1u && n_valid >= 2;
            // OPP: the agent's pass decides every game (act_filter 0), the opponent's passes the games outside seat 1's turn
            // (act_filter 1); a game frozen at the opponent-pass bound (ST_STUCK in its state) takes no move from either network
            const bool acts = OPP ? !(gm.status() & ST_STUCK) && (pass == 0 || !agent_turn)
                                  : A.act_filter == 0 || (A.act_filter == 1 ? !agent_turn : agent_turn);
            if (!acts) { n_valid = 0; status = 0u; }      // filtered out: reported as AZB_ACTION_SKIP, state untouched
            if (valid && record) {
                if (A.mask6_out) {
#pragma unroll
                    for (int p = 0; p < 6; p++) A.mask6_out[p * A.n + g] = m[p];
                }
                if (A.value_out) A.value_out[g] = value;
                if (A.action_out) A.action_out[g] = n_valid > 0 ? (uint8_t)action : (uint8_t)AZB_ACTION_SKIP;
                if (A.logp_out) A.logp_out[g] = logp;
                if (FULL && A.entropy_out) A.entropy_out[g] = entropy;
            }
            if (A.runner_mode && record) {
                // NNRunner.run_episode's per-decision record (nn_runner.py:27-45) in compact form: the warp's deciding games take
                // consecutive slots (one atomic per warp); the packed state the decision was taken on is what the update
                // kernel rebuilds observation and mask from
                const bool decides = valid && n_valid > 0 && !gm.ended();
                const uint32_t votes = __ballot_sync(0xFFFFFFFFu, decides);
                uint32_t base = 0;
                if (votes && (tid & 31) == 0) base = atomicAdd(A.n_dec, (uint32_t)__popc(votes));
                base = __shfl_sync(0xFFFFFFFFu, base, 0);
                const int64_t slot = (int64_t)base + __popc(votes & ((1u << (tid & 31)) - 1u));
                const bool fits = decides && slot < A.rec_cap;
                if (fits) {
                    gm.store(A.state_rec, A.rec_cap, slot);
                    A.action_rec[slot] = (uint8_t)action;
                    if (A.logp_rec) A.logp_rec[slot] = logp;
                    if (A.value_rec) A.value_rec[slot] = value;
                }
                if (valid) {
                    A.slot_rec[(int64_t)it * A.n + g] = fits ? (int32_t)slot : -1;
                    A.flags_rec[(int64_t)it * A.n + g] = decides ? 1 : 0;         // bit 1 (done) is added by the opponent phase
                }
            }
            // Only the cheap, uniform part of Azul.step runs here (move, next player).  Games whose round just ended --
            // and, in self-play mode, slots that need a fresh game -- are flagged in MISC and completed by
            // the finishing phase at the end of this kernel, 32 per warp with every lane busy.
            const bool ended_before = gm.ended();
            const bool stuck = acts && status == (uint32_t)ST_STUCK;
            uint32_t flags = 0u;
            bool stepped = false;
            if (A.apply_step && n_valid > 0 && !ended_before) {
                apply_move<2, POOL>(gm, action);                          // azul.py:304
                gm.steps += 1u;
                if (is_end_of_round(gm)) flags = FLAG_ROUND_OVER;         // azul.py:306 -> finishing phase
                else {
                    next_player(gm);                                      // azul.py:313
                    if (OPP) need |= valid && opponent_to_move(gm);
                }
                stepped = valid && A.apply_step == 2;
            } else if (A.apply_step == 2 && acts && (ended_before || stuck)) {
                flags = FLAG_FRESH_GAME;                                  // GameRunner.reset, game_runner.py:76-80
                if (valid && stuck) sink.add(6, 1);
            }
            {   // env steps executed by this warp's 32 games: one shared-memory atomic per warp (part 0 = whole warps)
                const uint32_t n_stepped = (uint32_t)__popc(__ballot_sync(0xFFFFFFFFu, stepped));
                if ((tid & 31) == 0) sink.add(0, n_stepped);
            }
            gm.misc |= flags;
            if (valid && A.apply_step) gm.store(A.state, A.n, g);
            if (valid && record) {
                if (A.done_out) A.done_out[g] = ended_before ? 1 : 0;      // finalised by the finishing phase for flagged games
                if (A.status_out) A.status_out[g] = (uint8_t)(status | gm.status());
            }
        }
        else if (has_next) {
            Game<2> nxt;
            nxt.load(nraw, 1, 0);
            build_obs_tile_3(nxt, a_tile, row, part);      // writes [0, OBS_TILE_BYTES): the scratch above it stays intact
            // Layer 1 of the NEXT tile starts now, while part 0 still publishes and plays this tile's moves: nobody reads
            // TMEM any more (every thread passed the barrier after epilogue 2b behind a tcgen05 fence; part 0 works from
            // registers and the scratch behind the observation tile), and the observation's writers are exactly the 384
            // threads of parts 1..3, which meet at a named barrier of their own.
            fence_async_smem();
            asm volatile("bar.sync 1, %0;" ::"n"(THREADS - TILE_M) : "memory");
            if (warp == TILE_M / 32) {
                // the issuing warp only ARRIVES at the end-of-tile barrier: nobody waits for the ~300 uniform-datapath
                // instructions of the issue loop (the other warps go on to the next tile's state loads and meet the MMAs at
                // their mbarrier), and the warp itself is done with this tile's TMEM and scratch
                asm volatile("bar.arrive 2, %0;" ::"n"(THREADS) : "memory");
                if (tid == TILE_M) issue_layer1();
                issuer = true;
            }
        }
        // all TMEM reads and scratch reads of this tile are complete before the next tile overwrites them
        if (!issuer) asm volatile("bar.sync 2, %0;" ::"n"(THREADS) : "memory");
    }
    if (!OPP) break;
    // ---- OPP: finish the rounds this pass ended (the opponent network must see the new round, as after
    // azb_policy_step(apply_step = 1)), then vote: is any game of this CTA still in the opponent's hands? ----
    __syncthreads();                                   // every state / done / status write of the tile loop is visible to the CTA
    finish_flagged(record ? A.done_out : nullptr, record ? A.status_out : nullptr, need);
    const bool more = __syncthreads_or(need ? 1 : 0) != 0;
    if (pass > 0 && (uint32_t)pass > max_opp) max_opp = (uint32_t)pass;
    if (!more) break;
    if (pass == MAX_OPP_PASSES) {
        // only a bug gets here (a round is at most 20 takes long): freeze the games the opponent still holds -- ST_STUCK
        // ends their episode for the alive vote and azb_train_stats, and no later pass moves them
        for (int64_t j = part; j < my_tiles; j += PARTS) {
            const int64_t g = ((int64_t)blockIdx.x + j * gridDim.x) * TILE_M + row;
            if (g >= A.n) continue;
            Game<2> h;
            h.load(A.state, A.n, g);
            if (opponent_to_move(h)) { h.add_status(ST_STUCK); h.store(A.state, A.n, g); }
        }
        break;
    }
    if (pass == 0) {
        // swap in the opponent's image: the barrier above closed every generic read of the agent's image (the critic vector),
        // and every MMA that read it was waited for at bar1 / bar2 / bar3.  The next pass builds its first observation tile
        // while the copy runs and waits for it before its first layer-1 issue.
        if (tid == 0) { fence_async_smem(); issue_image_copy(smem, A.opponent_packed, bar_w); }
        w_pending = opp_image = true;
    }
    }   // passes

    // ---- the rare, long part of Azul.step, or the runner mode's closing of the decision ----
    __syncthreads();                                   // every state / done / status write of the tile loop is visible to the CTA
    bool any_alive = true;
    if (A.runner_mode) {
        // GameRunner.step after the agent's move (game_runner.py:46-55), one thread per game of this CTA's tiles: finish the
        // round the move may have ended, let the random opponent (GREEDY: the greedy agent) play until seat 1 is to move with
        // >= 2 legal actions (or the game is over), take the reward from a score preview, and close the decision's record.
        // OPP: the policy opponent's
        // passes already restored that invariant, so the random opponent plays no move (as the eager path's trailing
        // azb_opponent_random(require_two = 1))
        bool alive = false;
        // (spreading a tile's 128 games over all 16 warps, 8 lanes each, was measured slower: 1.07 vs 0.97 ms per rollout of
        // 16,384 episodes -- the state loads lose their coalescing and every warp still walks the union of its games' paths)
        for (int64_t j = part; j < my_tiles; j += PARTS) {                 // warp-uniform trip count: the opponent loop votes
            const int64_t g = ((int64_t)blockIdx.x + j * gridDim.x) * TILE_M + row;
            const bool in_range = g < A.n;
            const int64_t gl2 = in_range ? g : A.n - 1;
            const bool decided = in_range && (A.flags_rec[(int64_t)it * A.n + gl2] & 1);
            if (in_range && !decided) A.reward_rec[(int64_t)it * A.n + g] = 0;
            Game<2> h;
            h.load(A.state, A.n, gl2);
            const uint32_t gid = A.gid0 + (uint32_t)gl2;
            const bool pending = (h.misc & FLAG_ROUND_OVER) != 0u;
            if (decided) h.misc &= ~(FLAG_ROUND_OVER | FLAG_FRESH_GAME);
            uint32_t m2[6];
            // OPP: a game frozen at the pass bound gets no random move either (its mask is reported empty)
            const bool frozen = OPP && (h.status() & ST_STUCK) != 0u;
            if (frozen) for (int p = 0; p < 6; p++) m2[p] = 0u;
            const int32_t diff = opponent_warp<POOL, GREEDY>(h, rng, gid, decided && !frozen, pending, m2);
            if (!decided) continue;
            h.store(A.state, A.n, g);
            const int32_t before = (int32_t)A.player_score[g];
            A.player_score[g] = (int16_t)diff;                            // game_runner.py:52
            A.reward_rec[(int64_t)it * A.n + g] = (int16_t)(diff - before);   // game_runner.py:51
            const bool over = h.ended();
            A.flags_rec[(int64_t)it * A.n + g] = (uint8_t)(1 | (over ? 2 : 0));
            if (A.done_out) A.done_out[g] = over ? 1 : 0;
            if (A.status_out) A.status_out[g] |= (uint8_t)h.status();
            if (A.mask6_out) {
#pragma unroll
                for (int p = 0; p < 6; p++) A.mask6_out[p * A.n + g] = m2[p];
            }
            alive |= !over && !(h.status() & ST_STUCK);
        }
        any_alive = __syncthreads_or(alive ? 1 : 0) != 0;
    } else if (A.apply_step) {
        bool unused = false;
        finish_flagged(A.done_out, A.status_out, unused);
    }
    __syncthreads();                                   // the next decision reads the states written above
    if (OPP && opp_image && any_alive && it + 1 < A.k_decisions) {
        // swap the agent's image back for the next decision (the barrier above closed every read of the opponent's; no
        // copy is left in flight when the CTA exits)
        if (tid == 0) { fence_async_smem(); issue_image_copy(smem, A.packed, bar_w); }
        w_pending = true;
        opp_image = false;
    }
    if (!any_alive) { it++; break; }                   // runner mode: every episode of this CTA is over
    }   // decision loop
    if (OPP && A.opp_passes && tid == 0) atomicMax(A.opp_passes, max_opp);
    if (A.steps_used && tid == 0) atomicMax(A.steps_used, (uint32_t)it);
    __syncthreads();
    if (A.counters && tid < AZB_N_COUNTERS && cnt[tid]) atomicAdd(&A.counters[tid], cnt[tid]);
    if (warp == 0) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
    }
}

// fp32 torch-layout weights -> the fp16 shared-memory image
__global__ void k_pack_weights(const float* __restrict__ w1a, const float* __restrict__ b1a, const float* __restrict__ w2a,
                               const float* __restrict__ b2a, const float* __restrict__ w1c, const float* __restrict__ b1c,
                               const float* __restrict__ w2c, const float* __restrict__ b2c, unsigned char* __restrict__ out)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    // one thread per fp16 element of W1 / W2, then the fp32 vectors
    // bias b as two fp16 inputs: hi = half(b), lo = half(b - hi)
    auto split = [](float b, bool low) {
        const float hi = __half2float(__float2half_rn(b));
        return low ? b - hi : b;
    };
    auto to_half = [](float v) { return __float2half_rn(fminf(fmaxf(v, -65504.0f), 65504.0f)); };
    if (i < N1 * K1) {
        const int n = i / K1, k = i % K1;
        float v = 0.0f;
        const int cu = n < HID ? -1 : critic_unit(n - HID);      // critic unit of this layer-1 output row (see critic_unit)
        if (k < OBS) {
            if (n < HID) v = w1a[n * OBS + k];
            else if (cu >= 0) v = w1c[cu * OBS + k];
        } else if (k == BIAS_K1 || k == BIAS_K1 + 1) {
            if (n < HID) v = split(b1a[n], k != BIAS_K1);
            else if (cu >= 0) v = split(b1c[cu], k != BIAS_K1);
        }
        *reinterpret_cast<__half*>(out + OFF_W1 + ((k >> 3) * N1_GROUPS + (n >> 3)) * 128 + (n & 7) * 16 + (k & 7) * 2) = to_half(v);
    } else if (i < N1 * K1 + N2 * K2) {
        const int j = i - N1 * K1, n = j / K2, k = j % K2;
        float v = 0.0f;
        if (n < ACT) {
            if (k < HID) v = w2a[n * HID + k];
            else if (k == BIAS_K2 || k == BIAS_K2 + 1) v = split(b2a[n], k != BIAS_K2);
        }
        *reinterpret_cast<__half*>(out + OFF_W2 + ((k >> 3) * N2_GROUPS + (n >> 3)) * 128 + (n & 7) * 16 + (k & 7) * 2) = to_half(v);
    } else if (i < N1 * K1 + N2 * K2 + VEC_FLOATS) {
        const int j = i - N1 * K1 - N2 * K2;
        float v = 0.0f;
        if (j < V_B2C) { const int cu = critic_unit(j - V_W2C); if (cu >= 0) v = w2c[cu]; }   // indexed like the TMEM columns
        else if (j == V_B2C) v = b2c[0];
        reinterpret_cast<float*>(out + OFF_VEC)[j] = v;
    }
}

template <int POOL, int MODE, bool FULL, bool OPP = false, bool GREEDY = false>
static int launch_policy(const PolicyArgs& A, int grid, cudaStream_t stream)
{
    AZB_CUDA(cudaFuncSetAttribute(k_policy<POOL, MODE, FULL, OPP, GREEDY>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)grid); cfg.blockDim = dim3(THREADS); cfg.dynamicSmemBytes = SMEM_BYTES; cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;       // see griddepcontrol in k_policy
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    AZB_CUDA(cudaLaunchKernelEx(&cfg, k_policy<POOL, MODE, FULL, OPP, GREEDY>, A));
    return 0;
}

}  // namespace pol

extern "C" {

int azb_policy_packed_bytes(void) { return pol::PACKED_BYTES; }

int azb_policy_pack_weights(azb_t* h, const float* w1a, const float* b1a, const float* w2a, const float* b2a,
                            const float* w1c, const float* b1c, const float* w2c, const float* b2c, void* packed,
                            void* stream)
{
    CHECK_HANDLE(h);
    if (!w1a || !b1a || !w2a || !b2a || !w1c || !b1c || !w2c || !b2c || !packed) return azb_fail(AZB_E_INVALID, "null buffer%s");
    const int total = pol::N1 * pol::K1 + pol::N2 * pol::K2 + pol::VEC_FLOATS;
    pol::k_pack_weights<<<(total + 255) / 256, 256, 0, (cudaStream_t)stream>>>(w1a, b1a, w2a, b2a, w1c, b1c, w2c, b2c,
                                                                              (unsigned char*)packed);
    CHECK_LAUNCH();
    return 0;
}

int azb_policy_step(azb_t* h, uint32_t* state, const void* packed, int mode, int apply_step, uint8_t* action_out,
                    float* logp_out, float* value_out, float* entropy_out, uint32_t* mask6_out, uint8_t* done_out,
                    uint8_t* status_out, float* logits_out, unsigned long long* counters, int act_filter, void* stream)
{
    CHECK_HANDLE(h);
    if (!state || !packed) return azb_fail(AZB_E_INVALID, "null buffer%s");
    if (h->players != 2) return azb_fail(AZB_E_INVALID, "the policy network is defined for 2 players (136 inputs, agent.py:29)%s");
    if (mode != 0 && mode != 1) return azb_fail(AZB_E_INVALID, "mode must be 0 (sample) or 1 (argmax)%s");
    pol::PolicyArgs A;
    A.state_in = state; A.state = state; A.n = h->n_games; A.packed = (const unsigned char*)packed;
    A.k0 = (uint32_t)h->seed; A.k1 = (uint32_t)(h->seed >> 32); A.gid0 = (uint32_t)h->game_id_base;
    if (apply_step < 0 || apply_step > 2) return azb_fail(AZB_E_INVALID, "apply_step must be 0, 1 or 2%s");
    A.mode = mode; A.apply_step = apply_step; A.first_rule = h->first_player; A.counters = counters;
    if (act_filter < 0 || act_filter > 2) return azb_fail(AZB_E_INVALID, "act_filter must be 0, 1 or 2%s");
    A.act_filter = act_filter;
    A.logits_out = logits_out; A.value_out = value_out; A.action_out = action_out; A.logp_out = logp_out;
    A.entropy_out = entropy_out; A.done_out = done_out; A.status_out = status_out; A.mask6_out = mask6_out;
    A.k_decisions = 1; A.runner_mode = 0; A.player_score = nullptr; A.n_dec = nullptr; A.rec_cap = 0; A.state_rec = nullptr;
    A.action_rec = nullptr; A.logp_rec = nullptr; A.value_rec = nullptr; A.slot_rec = nullptr; A.reward_rec = nullptr;
    A.flags_rec = nullptr; A.steps_used = nullptr; A.opponent_packed = nullptr; A.opp_passes = nullptr;
    const int64_t tiles = (h->n_games + pol::TILE_M - 1) / pol::TILE_M;
    const int grid = (int)(tiles < h->sm_count ? tiles : h->sm_count);
    int rc = 0;
    if (h->tile_pool == AZB_POOL_LID) rc = mode == 0 ? pol::launch_policy<1, 0, true>(A, grid, (cudaStream_t)stream) : pol::launch_policy<1, 1, true>(A, grid, (cudaStream_t)stream);
    else rc = mode == 0 ? pol::launch_policy<0, 0, true>(A, grid, (cudaStream_t)stream) : pol::launch_policy<0, 1, true>(A, grid, (cudaStream_t)stream);
    if (rc) return rc;
    CHECK_LAUNCH();
    return 0;
}

int azb_policy_rollout(azb_t* h, uint32_t* state, const void* packed, int mode, int k_decisions, int runner_mode,
                       int16_t* player_score, uint32_t* n_dec, int64_t rec_cap, uint32_t* state_rec, uint8_t* action_rec,
                       float* logp_rec, float* value_rec, int32_t* slot_rec, int16_t* reward_rec, uint8_t* flags_rec,
                       uint32_t* steps_used, uint8_t* action_out, float* logp_out, float* value_out, uint32_t* mask6_out,
                       uint8_t* done_out, uint8_t* status_out, unsigned long long* counters, void* stream)
{
    CHECK_HANDLE(h);
    if (!state || !packed) return azb_fail(AZB_E_INVALID, "null buffer%s");
    if (h->players != 2) return azb_fail(AZB_E_INVALID, "the policy network is defined for 2 players (136 inputs, agent.py:29)%s");
    if (mode != 0 && mode != 1) return azb_fail(AZB_E_INVALID, "mode must be 0 (sample) or 1 (argmax)%s");
    if (k_decisions < 1) return azb_fail(AZB_E_INVALID, "k_decisions must be >= 1%s");
    if (runner_mode != 0 && runner_mode != 1) return azb_fail(AZB_E_INVALID, "runner_mode must be 0 (self-play) or 1 (GameRunner)%s");
    if (runner_mode && (!player_score || !n_dec || rec_cap < 1 || !state_rec || !action_rec || !slot_rec || !reward_rec || !flags_rec))
        return azb_fail(AZB_E_INVALID, "runner mode needs player_score, n_dec, rec_cap and the state / action / slot / reward / flags records%s");
    pol::PolicyArgs A;
    A.state_in = state; A.state = state; A.n = h->n_games; A.packed = (const unsigned char*)packed;
    A.k0 = (uint32_t)h->seed; A.k1 = (uint32_t)(h->seed >> 32); A.gid0 = (uint32_t)h->game_id_base;
    A.mode = mode; A.apply_step = runner_mode ? 1 : 2; A.first_rule = h->first_player; A.counters = counters; A.act_filter = 0;
    A.logits_out = nullptr; A.value_out = value_out; A.action_out = action_out; A.logp_out = logp_out; A.entropy_out = nullptr;
    A.done_out = done_out; A.status_out = status_out; A.mask6_out = mask6_out;
    A.k_decisions = k_decisions; A.runner_mode = runner_mode; A.player_score = player_score; A.n_dec = n_dec; A.rec_cap = rec_cap;
    A.state_rec = state_rec; A.action_rec = action_rec; A.logp_rec = logp_rec; A.value_rec = value_rec; A.slot_rec = slot_rec;
    A.reward_rec = reward_rec; A.flags_rec = flags_rec; A.steps_used = steps_used;
    A.opponent_packed = nullptr; A.opp_passes = nullptr;
    const int64_t tiles = (h->n_games + pol::TILE_M - 1) / pol::TILE_M;
    const int grid = (int)(tiles < h->sm_count ? tiles : h->sm_count);
    int rc = 0;
    if (h->tile_pool == AZB_POOL_LID) rc = mode == 0 ? pol::launch_policy<1, 0, false>(A, grid, (cudaStream_t)stream) : pol::launch_policy<1, 1, false>(A, grid, (cudaStream_t)stream);
    else rc = mode == 0 ? pol::launch_policy<0, 0, false>(A, grid, (cudaStream_t)stream) : pol::launch_policy<0, 1, false>(A, grid, (cudaStream_t)stream);
    if (rc) return rc;
    CHECK_LAUNCH();
    return 0;
}

int azb_policy_rollout_vs_policy(azb_t* h, uint32_t* state, const void* packed, const void* opponent_packed, int mode,
                                 int k_decisions, int16_t* player_score, uint32_t* n_dec, int64_t rec_cap,
                                 uint32_t* state_rec, uint8_t* action_rec, float* logp_rec, float* value_rec,
                                 int32_t* slot_rec, int16_t* reward_rec, uint8_t* flags_rec, uint32_t* steps_used,
                                 uint32_t* opp_passes, uint32_t* mask6_out, uint8_t* done_out, uint8_t* status_out,
                                 void* stream)
{
    CHECK_HANDLE(h);
    if (!state || !packed || !opponent_packed) return azb_fail(AZB_E_INVALID, "null buffer%s");
    if (h->players != 2) return azb_fail(AZB_E_INVALID, "the policy network is defined for 2 players (136 inputs, agent.py:29)%s");
    if (mode != 0 && mode != 1) return azb_fail(AZB_E_INVALID, "mode must be 0 (sample) or 1 (argmax)%s");
    if (k_decisions < 1) return azb_fail(AZB_E_INVALID, "k_decisions must be >= 1%s");
    if (!player_score || !n_dec || rec_cap < 1 || !state_rec || !action_rec || !slot_rec || !reward_rec || !flags_rec)
        return azb_fail(AZB_E_INVALID, "runner mode needs player_score, n_dec, rec_cap and the state / action / slot / reward / flags records%s");
    pol::PolicyArgs A;
    A.state_in = state; A.state = state; A.n = h->n_games; A.packed = (const unsigned char*)packed;
    A.k0 = (uint32_t)h->seed; A.k1 = (uint32_t)(h->seed >> 32); A.gid0 = (uint32_t)h->game_id_base;
    A.mode = mode; A.apply_step = 1; A.first_rule = h->first_player; A.counters = nullptr; A.act_filter = 0;
    A.logits_out = nullptr; A.value_out = nullptr; A.action_out = nullptr; A.logp_out = nullptr; A.entropy_out = nullptr;
    A.done_out = done_out; A.status_out = status_out; A.mask6_out = mask6_out;
    A.k_decisions = k_decisions; A.runner_mode = 1; A.player_score = player_score; A.n_dec = n_dec; A.rec_cap = rec_cap;
    A.state_rec = state_rec; A.action_rec = action_rec; A.logp_rec = logp_rec; A.value_rec = value_rec; A.slot_rec = slot_rec;
    A.reward_rec = reward_rec; A.flags_rec = flags_rec; A.steps_used = steps_used;
    A.opponent_packed = (const unsigned char*)opponent_packed; A.opp_passes = opp_passes;
    const int64_t tiles = (h->n_games + pol::TILE_M - 1) / pol::TILE_M;
    const int grid = (int)(tiles < h->sm_count ? tiles : h->sm_count);
    int rc = 0;
    if (h->tile_pool == AZB_POOL_LID) rc = mode == 0 ? pol::launch_policy<1, 0, false, true>(A, grid, (cudaStream_t)stream) : pol::launch_policy<1, 1, false, true>(A, grid, (cudaStream_t)stream);
    else rc = mode == 0 ? pol::launch_policy<0, 0, false, true>(A, grid, (cudaStream_t)stream) : pol::launch_policy<0, 1, false, true>(A, grid, (cudaStream_t)stream);
    if (rc) return rc;
    CHECK_LAUNCH();
    return 0;
}

int azb_policy_rollout_vs_greedy(azb_t* h, uint32_t* state, const void* packed, int mode, int k_decisions,
                                 int16_t* player_score, uint32_t* n_dec, int64_t rec_cap, uint32_t* state_rec,
                                 uint8_t* action_rec, float* logp_rec, float* value_rec, int32_t* slot_rec, int16_t* reward_rec,
                                 uint8_t* flags_rec, uint32_t* steps_used, uint8_t* action_out, float* logp_out,
                                 float* value_out, uint32_t* mask6_out, uint8_t* done_out, uint8_t* status_out, void* stream)
{
    CHECK_HANDLE(h);
    if (!state || !packed) return azb_fail(AZB_E_INVALID, "null buffer%s");
    if (h->players != 2) return azb_fail(AZB_E_INVALID, "the policy network is defined for 2 players (136 inputs, agent.py:29)%s");
    if (mode != 0 && mode != 1) return azb_fail(AZB_E_INVALID, "mode must be 0 (sample) or 1 (argmax)%s");
    if (k_decisions < 1) return azb_fail(AZB_E_INVALID, "k_decisions must be >= 1%s");
    if (!player_score || !n_dec || rec_cap < 1 || !state_rec || !action_rec || !slot_rec || !reward_rec || !flags_rec)
        return azb_fail(AZB_E_INVALID, "runner mode needs player_score, n_dec, rec_cap and the state / action / slot / reward / flags records%s");
    pol::PolicyArgs A;
    A.state_in = state; A.state = state; A.n = h->n_games; A.packed = (const unsigned char*)packed;
    A.k0 = (uint32_t)h->seed; A.k1 = (uint32_t)(h->seed >> 32); A.gid0 = (uint32_t)h->game_id_base;
    A.mode = mode; A.apply_step = 1; A.first_rule = h->first_player; A.counters = nullptr; A.act_filter = 0;
    A.logits_out = nullptr; A.value_out = value_out; A.action_out = action_out; A.logp_out = logp_out; A.entropy_out = nullptr;
    A.done_out = done_out; A.status_out = status_out; A.mask6_out = mask6_out;
    A.k_decisions = k_decisions; A.runner_mode = 1; A.player_score = player_score; A.n_dec = n_dec; A.rec_cap = rec_cap;
    A.state_rec = state_rec; A.action_rec = action_rec; A.logp_rec = logp_rec; A.value_rec = value_rec; A.slot_rec = slot_rec;
    A.reward_rec = reward_rec; A.flags_rec = flags_rec; A.steps_used = steps_used;
    A.opponent_packed = nullptr; A.opp_passes = nullptr;
    const int64_t tiles = (h->n_games + pol::TILE_M - 1) / pol::TILE_M;
    const int grid = (int)(tiles < h->sm_count ? tiles : h->sm_count);
    int rc = 0;
    if (h->tile_pool == AZB_POOL_LID) rc = mode == 0 ? pol::launch_policy<1, 0, false, false, true>(A, grid, (cudaStream_t)stream) : pol::launch_policy<1, 1, false, false, true>(A, grid, (cudaStream_t)stream);
    else rc = mode == 0 ? pol::launch_policy<0, 0, false, false, true>(A, grid, (cudaStream_t)stream) : pol::launch_policy<0, 1, false, false, true>(A, grid, (cudaStream_t)stream);
    if (rc) return rc;
    CHECK_LAUNCH();
    return 0;
}

}  // extern "C"
