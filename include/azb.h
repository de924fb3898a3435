/*
 * azb.h -- C ABI of the B200-native batched Azul engine (libazb.so).
 *
 * The reference (patello/azul_deep_reinforcement_learning) has NO native / FFI interface: its
 * boundary for this path is the Python surface re-exported by azulnet/__init__.py:1-5.  The entry
 * points below are what a binding for that surface needs; each one names the reference
 * function(s) it replaces for a whole batch of independent games.  The Python package
 * azul_deep_reinforcement_learning_b200 binds them with ctypes (see INTEGRATION.md for the stub a
 * reference maintainer would add).
 *
 * Conventions
 *   - every function returns 0 on success or a negative AZB_E_* code; nothing throws across the
 *     ABI; azb_last_error() returns a thread-local message for the last failure.
 *   - the CALLER owns every device buffer (plain device pointers, e.g. torch tensor data_ptr());
 *     the handle owns only configuration.  All launches are asynchronous on `stream`
 *     (a cudaStream_t passed as void*, NULL = default stream); no hidden synchronisation.
 *   - one handle per (device, batch shape); thread-compatible, not thread-safe.
 *   - per-game status bits replace the reference's exceptions:
 *       AZB_ST_ILLEGAL  IllegalMove (azul.py:301-302), state untouched
 *       AZB_ST_ENDED    GameEnded   (azul.py:298-299), state untouched
 *       AZB_ST_STUCK    no legal action although the round is not over (reference crashes)
 *       AZB_ST_BAG_EMPTY  Lid pool ran out of tiles during a refill (azul.py:86 TODO)
 *       AZB_ST_BAD_IMPORT record not representable in the packed state
 *
 * Buffers (G = n_games, P = players, W = azb_state_words(P), U = azb_record_size(P)):
 *   state    uint32 [W][G]   packed structure-of-arrays game state (DESIGN.md "HBM layout")
 *   mask6    uint32 [6][G]   legal mask; word p bit (d + 6c) <=> action d + 6c + 30p legal
 *                            (action codec of game_runner.py:102-111)
 *   action   uint8  [G]      0..179; AZB_ACTION_SKIP leaves that game untouched (status 0)
 *   draws20  int8   [G][20]  tile colours for the next new_round in (display, slot) order
 *                            (azul.py:74-75); NULL = counter-based Philox4x32-10 schedule
 *   records  int32  [G][U]   unpacked interchange records mirroring the reference Azul object
 */
#ifndef AZB_H
#define AZB_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define AZB_ABI_VERSION 1

#define AZB_POOL_RANDOM 0          /* rules["tile_pool"] == "Random", azul.py:45-47 */
#define AZB_POOL_LID 1             /* rules["tile_pool"] == "Lid",    azul.py:48-52 */
#define AZB_FIRST_PLAYER_RANDOM 0  /* rules["first_player"] == "Random", azul.py:36-37; 1..P fixed */

#define AZB_ST_ILLEGAL 1
#define AZB_ST_ENDED 2
#define AZB_ST_STUCK 4
#define AZB_ST_BAG_EMPTY 8
#define AZB_ST_BAD_IMPORT 16

#define AZB_ACTION_SKIP 255
#define AZB_N_ACTIONS 180
#define AZB_N_COUNTERS 16

#define AZB_E_INVALID (-1)         /* bad argument */
#define AZB_E_CUDA (-2)            /* CUDA runtime error (message in azb_last_error) */
#define AZB_E_NODEVICE (-3)        /* no usable CUDA device: there is no CPU fallback */

typedef struct azb_handle azb_t;

int azb_abi_version(void);
int azb_state_words(int players);           /* 7 + 5P */
int azb_record_size(int players);           /* 48 + 58P */
int azb_obs_size(int players);              /* 32 + 52P (136 for P = 2, agent.py:29) */
const char* azb_last_error(void);

/* Azul.__init__ configuration for a batch (azul.py:18-61): players 2..4, rules as integers,
 * Philox key `seed`; game g of this handle has global id game_id_base + g (multi-GPU sharding:
 * results do not depend on how the id range is split over devices). */
int azb_create(azb_t** out, int device, int64_t n_games, int players, int tile_pool, int first_player,
               uint64_t seed, uint64_t game_id_base);
int azb_destroy(azb_t* h);
/* threads per block for the kernels of this handle (multiple of 32, <= 1024); 0 = default (128, and an
 * SM-balanced choice for azb_rollout_random: equal blocks per SM, see DESIGN.md) */
int azb_set_block_threads(azb_t* h, int threads);
/* azb_rollout_random tuning: how many of a warp's 32 games must have reached the end of their round
 * before the warp runs the scoring / refill pass for them (1..32, 0 = default 32).  Results do not
 * depend on it. */
int azb_set_rollout_defer(azb_t* h, int games);

/* GameRunner.reset / Azul(rules) + new_round() (game_runner.py:76-80, azul.py:18-89): fresh
 * game in every slot with which[g] != 0 (which == NULL: all slots).  total_steps is preserved. */
int azb_reset(azb_t* h, uint32_t* state, const uint8_t* which, void* stream);

/* check_all_valid (game_runner.py:113-117) over Azul.is_legal_move (azul.py:162-176) */
int azb_legal_mask(azb_t* h, const uint32_t* state, uint32_t* mask6, void* stream);

/* Azul.step (azul.py:296-313) for every game.  Outputs are optional (NULL to skip):
 *   mask6_out   legal mask of the resulting state
 *   preview_out int16 [P][G] score after a non-mutating count_score (game_runner.py:48-50)
 *   done_out    uint8 [G] end_of_game after the step
 *   status_out  uint8 [G] AZB_ST_* bits of this call plus the sticky ones
 * Any n_games and any buffer alignment work; with n_games % 4 == 0 and 16-byte aligned state / mask6_out / action
 * pointers the rows of 32 games move as 16-byte asynchronous copies and whole-line stores (the fast path).
 * The kernel's warps take their rows from a small counter block owned by the handle (allocated by azb_create, reset by
 * the kernel itself): launch azb_step on ONE stream at a time per handle; other entry points are unaffected. */
int azb_step(azb_t* h, uint32_t* state, const uint8_t* action, const int8_t* draws20, uint32_t* mask6_out,
             int16_t* preview_out, uint8_t* done_out, uint8_t* status_out, void* stream);

/* k_steps env steps per game with the random agent on every seat (RandomAgent, game_runner.py:87-97:
 * weight 0.01 for straight-to-floor actions, 1.0 otherwise), Philox draws and auto-reset, fused in
 * one launch; counters: device uint64[AZB_N_COUNTERS], accumulated (see DESIGN.md). */
int azb_rollout_random(azb_t* h, uint32_t* state, int k_steps, uint32_t* mask6_out,
                       unsigned long long* counters, void* stream);

/* score after count_score on a copy (game_runner.py:48-50): int16 [P][G]; state untouched */
int azb_score_preview(azb_t* h, const uint32_t* state, int16_t* score_out, void* stream);

/* Azul.import_JSON / export_JSON / __eq__ field set (azul.py:63,90-117) plus box/lid, end_of_game
 * and the statistics arrays, as unpacked int32 records.  ok_out (uint8 [G], optional) is 0 for
 * records that cannot be packed (those slots also carry AZB_ST_BAD_IMPORT). */
int azb_import_state(azb_t* h, const int32_t* records, uint32_t* state, uint8_t* ok_out, void* stream);
int azb_export_state(azb_t* h, const uint32_t* state, int32_t* records, void* stream);

/* GameRunner.get_state (game_runner.py:56-72): float32 [G][32 + 52P]; perspective 0..P-1, or -1
 * for the seat to move in each game (opponent_move, game_runner.py:38). */
int azb_observe(azb_t* h, const uint32_t* state, int perspective, float* obs, void* stream);

/* Azul.get_statistics (azul.py:314-315) as int32 [G][10]: player_score, opponent_score, rounds,
 * first_player_stats[0], sum(first_player_stats), -floor_penalty[0], max_combo[0], completed rows,
 * completed columns, completed colours (seat 0). */
int azb_stats(azb_t* h, const uint32_t* state, int32_t* stats10, void* stream);

/* azb_observe with bfloat16 output (uint16 bit patterns, [G][32 + 52P]): what the policy kernel feeds its first
 * layer and what the training loop records per decision.  Counts <= 256 are exact in bf16. */
int azb_observe_bf16(azb_t* h, const uint32_t* state, int perspective, void* obs_bf16, void* stream);

/* The reference's public per-function entry points, batched (used by the azulnet façade):
 *   azb_move         Azul.move            azul.py:118-161 (no legality check, like the reference)
 *   azb_next_player  Azul.next_player     azul.py:177-181
 *   azb_count_score  Azul.count_score     azul.py:192-295
 *   azb_new_round    Azul.new_round       azul.py:64-89 (draws20 NULL = Philox schedule)
 *   azb_round_flags  uint8 [G]: bit 0 Azul.is_end_of_round (azul.py:182-183),
 *                                bit 1 Azul.is_end_of_game (azul.py:184-191, recomputed from walls) */
int azb_move(azb_t* h, uint32_t* state, const uint8_t* action, void* stream);
int azb_next_player(azb_t* h, uint32_t* state, void* stream);
int azb_count_score(azb_t* h, uint32_t* state, void* stream);
int azb_new_round(azb_t* h, uint32_t* state, const int8_t* draws20, void* stream);
int azb_round_flags(azb_t* h, const uint32_t* state, uint8_t* flags, void* stream);

/* GameRunner.step after the agent's own move (game_runner.py:46-55), random-agent opponent
 * (RandomAgent, :87-97, Philox words): opponent moves until it is seat 1's turn with >= 2 legal actions
 * (require_two != 0, :46) or just seat 1's turn (require_two == 0, GameRunner.reset :84-85) or the game
 * is over; then reward = (score1 - score2 after count_score on a copy) - player_score, player_score updated
 * in place (int16 [G], :48-52), done = is_end_of_game, mask6 = legal mask of the resulting state.
 * obs_bf16_out (optional): GameRunner.get_state of the resulting state from seat 1's perspective, bfloat16 [G][32 + 52P]
 * (what azb_observe_bf16(perspective 0) would write) -- the next decision's network input, recorded by training. */
int azb_opponent_random(azb_t* h, uint32_t* state, int require_two, int16_t* player_score, int16_t* reward_out,
                        uint8_t* done_out, uint8_t* status_out, uint32_t* mask6_out, void* obs_bf16_out, void* stream);

/* The greedy agent (no counterpart in the reference; DESIGN.md "Greedy agent"): for the seat to move, the legal action
 * whose move followed by count_score on a copy leaves the mover's score highest -- without the clamp at zero of
 * azul.py:294-295 -- ties broken by the random agent's Philox word of that env step over the tied actions in ascending
 * action index.  Deterministic given (seed, game id, step count), like every agent here.
 *   azb_greedy_action    uint8 [G]: the greedy agent's action in every game (AZB_ACTION_SKIP when the game is over or no
 *                        action is legal); the state is not touched.
 *   azb_opponent_greedy  azb_opponent_random with the greedy agent as the opponent: the same arguments, loop rule
 *                        (require_two), reward, outputs and optional bf16 observation. */
int azb_greedy_action(azb_t* h, const uint32_t* state, uint8_t* action_out, void* stream);
int azb_opponent_greedy(azb_t* h, uint32_t* state, int require_two, int16_t* player_score, int16_t* reward_out,
                        uint8_t* done_out, uint8_t* status_out, uint32_t* mask6_out, void* obs_bf16_out, void* stream);

/* ---- K4: the policy/value network of azulnet/model.py:12-41 fused with its callers ------------
 * ActorCritic(136, 180, hidden 180): actor 136 -> 180 -> ReLU -> 180 logits, critic 136 -> 180 -> ReLU -> 1.
 * azb_policy_pack_weights converts the eight fp32 parameter tensors (torch layout [out][in], device
 * pointers) into the fp16 image (azb_policy_packed_bytes() bytes, device; biases as fp16 hi + lo pairs) the kernel keeps in shared
 * memory.  azb_policy_step then does, for every 2-player game of the batch, in ONE launch:
 *   observation from the seat to move        GameRunner.get_state            game_runner.py:56-72
 *   both dense layers on tcgen05 tensor cores ActorCritic.forward_actor/critic model.py:23-41
 *   logits[~mask] = -inf, softmax/log_softmax  model.py:37-40
 *   action ~ policy (mode 0) or argmax (mode 1) Agent.get_ac_output          agent.py:64-81
 *   log pi(action), -mean(log pi over legal)   NNRunner.run_episode          nn_runner.py:32-40
 *   and, when apply_step != 0, Azul.step with that action (Philox refill)   azul.py:296-313;
 *   apply_step == 2 additionally starts a fresh game in slots whose game ended (self-play rollouts) and
 *   accumulates the rollout counters (device uint64[AZB_N_COUNTERS], optional).
 * act_filter selects which games decide in this launch: 0 all; 1 only the opponent's turns of GameRunner.step
 * (not "seat 1 to move with >= 2 legal actions", game_runner.py:46: a frozen Agent as opponent_move); 2 only the
 * agent's turns.  Games filtered out report AZB_ACTION_SKIP and are left untouched.
 * Outputs (device, each optional / NULL): action uint8 [G] (AZB_ACTION_SKIP when no action is legal),
 * logp, value, entropy float [G], mask6 uint32 [6][G] (the mask the decision used), done / status uint8 [G]
 * (AZB_ST_ENDED / AZB_ST_STUCK instead of model.py:33-34 IllegalMask), logits float [G][180] (unmasked). */
int azb_policy_packed_bytes(void);
int azb_policy_pack_weights(azb_t* h, const float* w1a, const float* b1a, const float* w2a, const float* b2a,
                            const float* w1c, const float* b1c, const float* w2c, const float* b2c, void* packed,
                            void* stream);
int azb_policy_step(azb_t* h, uint32_t* state, const void* packed, int mode, int apply_step, uint8_t* action_out,
                    float* logp_out, float* value_out, float* entropy_out, uint32_t* mask6_out, uint8_t* done_out,
                    uint8_t* status_out, float* logits_out, unsigned long long* counters, int act_filter, void* stream);

/* ---- K4, persistent form: k_decisions decisions per game in ONE launch, the packed state resident on the device in
 * between (each CTA owns its games for the whole launch; no launch, no host copy per env step).
 * runner_mode 0 -- self-play (BASELINE.json configs[3]): every seat's move is sampled from the policy, Azul.step
 *   (azul.py:296-313) with Philox refills, finished games are tallied in `counters` and replaced by fresh ones.
 * runner_mode 1 -- NNRunner.run_episode (nn_runner.py:17-47) over GameRunner.step (game_runner.py:43-55) for one episode
 *   per slot: seat 1 decides; after each decision the random opponent (RandomAgent, :87-97) moves until seat 1 is to move
 *   with >= 2 legal actions or the game is over, the reward is (score1 - score2 after count_score on a copy) -
 *   player_score (int16 [G], updated in place).  The caller starts the episodes (azb_reset + azb_opponent_random with
 *   require_two = 0 = GameRunner.reset, :76-85).  Ended games take no further decisions; a CTA whose episodes are all over
 *   stops early.  Decision records:
 *     compact, slot = old value of the device counter n_dec[0] (uint32, zeroed by the caller), capacity rec_cap:
 *       state_rec uint32 [W][rec_cap] (packed state the decision was taken on: observation and legal mask are functions of
 *       it), action_rec uint8 [rec_cap], logp_rec / value_rec float [rec_cap] (optional)
 *     per (decision index t, game g), [k_decisions][G]: slot_rec int32 (-1: no decision / record full), reward_rec int16,
 *       flags_rec uint8 (bit 0 decision taken, bit 1 game over after it)
 *     steps_used uint32 [1] (optional, zeroed by the caller): decision iterations actually run (max over CTAs).
 * action_out / logp_out / value_out / mask6_out / done_out / status_out ([G], optional) hold the LAST decision's outputs
 * (runner mode: mask6_out / done_out describe the state after the opponent loop). */
int azb_policy_rollout(azb_t* h, uint32_t* state, const void* packed, int mode, int k_decisions, int runner_mode,
                       int16_t* player_score, uint32_t* n_dec, int64_t rec_cap, uint32_t* state_rec, uint8_t* action_rec,
                       float* logp_rec, float* value_rec, int32_t* slot_rec, int16_t* reward_rec, uint8_t* flags_rec,
                       uint32_t* steps_used, uint8_t* action_out, float* logp_out, float* value_out, uint32_t* mask6_out,
                       uint8_t* done_out, uint8_t* status_out, unsigned long long* counters, void* stream);

/* ---- K4, persistent runner mode against a frozen policy opponent: GameRunner(opponent=Agent(base_net_file=...))
 * (game_runner.py:26-30, scripts/run_batch.py) for one episode per slot in ONE launch.  As azb_policy_rollout's runner mode
 * (same records, outputs and checks), but seat 2 -- and seat 1 when it has a single legal action -- is played by the
 * network in `opponent_packed` (azb_policy_pack_weights image; may be `packed` itself) with the same `mode` as the agent:
 * after each agent decision the opponent takes one move per game that is in its hands, pass after pass, until seat 1 is
 * to move with >= 2 legal actions or the game is over; then the reward.  The decisions equal those of azb_policy_step
 * (act_filter 0 for the agent, then act_filter 1 with the opponent's image until no game acts) followed by
 * azb_opponent_random(require_two = 1): the sampling word depends only on the game and its step count.
 * The caller starts the episodes with azb_reset, then ONE azb_policy_step(opponent_packed, the same mode, apply_step = 1,
 * act_filter = 1) -- on a fresh board the opponent moves at most once before seat 1 is to move with >= 2 legal actions --
 * then azb_opponent_random(require_two = 0), and zeroes player_score; no host synchronisation is needed.
 * opp_passes uint32 [1] (optional, zeroed by the caller): the most opponent passes one decision needed (max over CTAs and
 * decisions).  At most 64 passes are run per decision; a game still in the opponent's hands then (only a bug can cause
 * it) gets AZB_ST_STUCK, takes no further move and counts as unfinished. */
int azb_policy_rollout_vs_policy(azb_t* h, uint32_t* state, const void* packed, const void* opponent_packed, int mode,
                                 int k_decisions, int16_t* player_score, uint32_t* n_dec, int64_t rec_cap,
                                 uint32_t* state_rec, uint8_t* action_rec, float* logp_rec, float* value_rec,
                                 int32_t* slot_rec, int16_t* reward_rec, uint8_t* flags_rec, uint32_t* steps_used,
                                 uint32_t* opp_passes, uint32_t* mask6_out, uint8_t* done_out, uint8_t* status_out,
                                 void* stream);

/* ---- K4, persistent runner mode against the greedy agent: azb_policy_rollout's runner mode (the same records, outputs and
 * checks; always runner mode, no counters) with azb_greedy_action's agent as the opponent in place of the random agent:
 * after each agent decision the greedy agent moves until seat 1 is to move with >= 2 legal actions or the game is over, then
 * the reward.  The decisions equal those of azb_policy_step(apply_step = 1) followed by azb_opponent_greedy(require_two = 1).
 * The caller starts the episodes with azb_reset + azb_opponent_greedy(require_two = 0) and zeroes player_score; no host
 * synchronisation is needed. */
int azb_policy_rollout_vs_greedy(azb_t* h, uint32_t* state, const void* packed, int mode, int k_decisions,
                                 int16_t* player_score, uint32_t* n_dec, int64_t rec_cap, uint32_t* state_rec,
                                 uint8_t* action_rec, float* logp_rec, float* value_rec, int32_t* slot_rec, int16_t* reward_rec,
                                 uint8_t* flags_rec, uint32_t* steps_used, uint8_t* action_out, float* logp_out,
                                 float* value_out, uint32_t* mask6_out, uint8_t* done_out, uint8_t* status_out, void* stream);

/* ---- K4, persistent two-seat self-play: one network plays both seats of every game for one episode per slot in ONE launch,
 * and every decision with a choice is recorded -- seat 2's as well as seat 1's.  Seats are 1 and 2 (current_player 1 is seat
 * 1); for a state, d_s = seat s's score preview (count_score on a copy, azb_score_preview) minus the other seat's.
 *   Decision: in every iteration each live game's mover plays the network's move (mode 0 samples, 1 takes the argmax; the
 *   Philox word is keyed by game and env step).  It is recorded only when the mover has >= 2 legal actions
 *   (game_runner.py:46 applied to either seat); a single legal action is played unrecorded.  Rounds are then finished as in
 *   azb_policy_step(apply_step = 1): the decisions equal those of repeated azb_policy_step(apply_step = 1, act_filter = 0).
 *   Reward: player_score int16 [2][G] (seat s at [s - 1][g]) is zeroed by the caller when the episodes start (azb_reset;
 *   there are no opening moves).  A seat's open decision is closed when that seat is next to move with >= 2 legal actions,
 *   or when the game is over or stuck (then both seats' are): reward = d_s - player_score[s], then player_score[s] = d_s.
 *   For a finished episode seat s's rewards therefore sum to d_s of the final state, and the two seats' sums negate each
 *   other.  A game with no legal action gets AZB_ST_STUCK.  A reward is 0 until its decision is closed: a decision still
 *   open when k_decisions stops the launch keeps 0, and its game counts as unfinished.
 *   Records: those of azb_policy_rollout's runner mode, at most one decision per (iteration t, game g) cell; flags_rec bit 0
 *   decision recorded, bit 1 game over when it was closed, bit 2 seat 2's decision.  The reward of iteration t is written
 *   at a later iteration, when the decision is closed.
 *   pending int32 [2][G]: device scratch (the open decision's iteration per seat), initialised by the kernel.
 * mask6_out / done_out / status_out ([G], optional) describe the final state.  Checks as azb_policy_rollout_vs_greedy; no
 * host synchronisation is needed, so a training batch stays one CUDA graph. */
int azb_policy_rollout_selfplay(azb_t* h, uint32_t* state, const void* packed, int mode, int k_decisions,
                                int16_t* player_score, int32_t* pending, uint32_t* n_dec, int64_t rec_cap, uint32_t* state_rec,
                                uint8_t* action_rec, float* logp_rec, float* value_rec, int32_t* slot_rec, int16_t* reward_rec,
                                uint8_t* flags_rec, uint32_t* steps_used, uint32_t* mask6_out, uint8_t* done_out,
                                uint8_t* status_out, void* stream);

/* Discounted returns of NNRunner.train (nn_runner.py:72-75) over the records of azb_policy_rollout's runner mode:
 * q_t = r_t + gamma * q_{t+1} over each game's decisions (accumulated in double like the reference's numpy loop), written
 * as float to qval[slot] (float [rec_cap]); reward_sum (double [1], optional) += the sum of all rewards; steps_used
 * (device uint32 [1], optional: azb_policy_rollout's output) bounds the walk to the decision iterations actually run.
 * One running return per seat, picked by flags bit 2: two-seat self-play (azb_policy_rollout_selfplay) discounts each
 * seat's decisions separately; the runner modes never set the bit. */
int azb_discounted_returns(azb_t* h, int k_decisions, double gamma, const int16_t* reward_rec, const uint8_t* flags_rec,
                           const int32_t* slot_rec, float* qval, double* reward_sum, const uint32_t* steps_used, void* stream);

/* The statistics of one training batch in one launch (what Agent.update and GameRunner's GameStatistics report,
 * agent.py:58-59, game_runner.py:10-22, azul.py:314-315), from the final packed states of the batch's games and the
 * device-side results of the rollout / update: out18 double [18] = decision count (clamped to rec_cap), the three loss
 * sums, sum of rewards, games, the sums of Azul.get_statistics' ten raw values (azb_stats order), games seat 1 won, games
 * not finished (+ 1e9 when n_dec > rec_cap: the decision records overflowed).  Sums, so that ranks can all-reduce them. */
int azb_train_stats(azb_t* h, const uint32_t* state, const uint32_t* n_dec, int64_t rec_cap, const double* loss_sums,
                    const double* reward_sum, double* out18, void* stream);

/* ---- a19: the loss of Agent.update and its gradient at the network outputs --------------------
 * For n recorded agent decisions (device arrays): logits float [n][180] (raw actor outputs), value float [n],
 * mask_rows uint32 [n][6] (the legal-mask words of each decision), action int64 [n], qval float [n]
 * (discounted returns, nn_runner.py:72-75).  Per decision, exactly as the reference:
 *   log_prob  = log_softmax(logits with illegal = -inf)[action]          nn_runner.py:32, model.py:37-40
 *   entropy   = -mean(log_softmax over the legal actions)                nn_runner.py:36-40
 *   advantage = qval - value (not detached in the actor term)            agent.py:45
 *   loss      = scale * sum(actor_coeff * -log_prob * advantage + critic_coeff * advantage^2
 *                           + entropy_coeff * entropy)                   agent.py:47-56 (means: scale = 1/N)
 * Writes dlogits float [n][180] = d loss / d logits, dvalue float [n] = d loss / d value, and ADDS the unscaled sums
 * of the three terms to sums double [3] (optional).  The caller back-propagates (dlogits, dvalue) through the
 * network (torch.autograd.backward) -- the dense layers stay in the caller's framework.
 * Excluded decisions (here and in azb_a2c_update_gradients): a decision whose action is not legal in its mask -- no legal
 * action at all, an action outside [0, 180), or a masked-out action -- contributes nothing: its dlogits row and dvalue
 * are 0, and it adds nothing to sums or to the parameter gradients. */
int azb_a2c_loss_grad(azb_t* h, int64_t n, const float* logits, const float* value, const uint32_t* mask_rows,
                      const int64_t* action, const float* qval, float scale, float actor_coeff, float critic_coeff,
                      float entropy_coeff, float* dlogits, float* dvalue, double* sums, void* stream);

/* ---- a19 on the tensor cores: the whole of Agent.update's gradient (agent.py:39-62) for recorded decisions, no library
 * GEMM and no autograd.  Inputs: the decision records of azb_policy_rollout's runner mode -- state_rec uint32 [W][capacity]
 * (packed state each decision was taken on; observation and legal mask are rebuilt from it), action uint8 [capacity], qval
 * float [capacity] (azb_discounted_returns) -- and the decision count, either on the device (n_dec uint32 [1], clamped to
 * capacity; no host synchronisation) or n_fixed when n_dec is NULL; `packed` = the current parameters' image
 * (azb_policy_pack_weights).  Forward recomputation (model.py:23-41), masked log-softmax, the three loss terms with the
 * reference's non-detached advantage, and the backward pass through both heads run as tcgen05 GEMMs (fp16 operands, fp32
 * accumulation); decisions are excluded as for azb_a2c_loss_grad.  The gradient SUMS over the decisions are ADDED to
 * the eight fp32 buffers in torch layout ([out][in]): grad_w1a [180][136], grad_b1a [180], grad_w2a [180][180], grad_b2a [180], grad_w1c [180][136], grad_b1c [180],
 * grad_w2c [180], grad_b2c [1]; sums double [3] += the unscaled actor / critic / entropy loss terms.  workspace: device
 * scratch of azb_update_workspace_bytes(capacity) bytes.  logits_out float [n][180] / value_out float [n] (optional): the
 * recomputed network outputs. */
int64_t azb_update_workspace_bytes(int64_t capacity);
/* The update works through the decisions in chunks so that the workspace stays bounded however large `capacity` is
 * (default 2^20 decisions = 1.9 GB); process-wide tuning / test hook: rows must be a positive multiple of 128 and be set
 * before azb_update_workspace_bytes is asked for the size. */
int azb_update_set_chunk_rows(int64_t rows);
int azb_a2c_update_gradients(azb_t* h, const uint32_t* state_rec, int64_t capacity, const uint8_t* action, const float* qval,
                             const uint32_t* n_dec, int64_t n_fixed, const void* packed, float actor_coeff, float critic_coeff,
                             float entropy_coeff, void* workspace, float* grad_w1a, float* grad_b1a, float* grad_w2a,
                             float* grad_b2a, float* grad_w1c, float* grad_b1c, float* grad_w2c, float* grad_b2c, double* sums,
                             float* logits_out, float* value_out, void* stream);

/* ---- opt-in rule variant: factory count by player count (SURVEY §8f rank 4; the reference's azul.py:72 TODO) --------
 * The reference always builds five factory displays (azul.py:19).  With `factories` = 2 * players + 1 (7 for three
 * players, 9 for four, as in the board game) a round draws 4 * factories tiles and the action space grows to
 * 30 * (factories + 1) = 240 / 300: action a = d + S*c + 5*S*p with S = factories + 1 sources (game_runner.py:102-103 with
 * 6 -> S), legal mask = six 64-bit words (word p bit d + S*c), actions are uint16 (0xFFFF = skip), draws int8
 * [G][4 * factories], records int32 [G][azb_v_record_size] (the default record with `factories` display rows in front),
 * state uint32 [azb_v_state_words][G].  The handle comes from azb_create; `factories` = 5 runs the reference's rule
 * through the same code (it reproduces the default engine bit for bit: tests).  Everything else -- scoring, floor, lid,
 * Philox schedule (display i draws from word i resp. words 2i, 2i + 1), status bits, counters -- is as in the default path. */
int azb_v_state_words(int players, int factories);
int azb_v_record_size(int players, int factories);
int azb_v_n_actions(int factories);
int azb_v_reset(azb_t* h, int factories, uint32_t* state, const uint8_t* which, void* stream);
int azb_v_legal_mask(azb_t* h, int factories, const uint32_t* state, uint64_t* mask6, void* stream);
int azb_v_step(azb_t* h, int factories, uint32_t* state, const uint16_t* action, const int8_t* draws, uint64_t* mask6_out,
               uint8_t* done_out, uint8_t* status_out, void* stream);
int azb_v_rollout_random(azb_t* h, int factories, uint32_t* state, int k_steps, unsigned long long* counters, void* stream);
int azb_v_import_state(azb_t* h, int factories, const int32_t* records, uint32_t* state, uint8_t* ok_out, void* stream);
int azb_v_export_state(azb_t* h, int factories, const uint32_t* state, int32_t* records, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* AZB_H */
