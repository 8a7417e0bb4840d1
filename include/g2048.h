/* libg2048 -- C ABI of the B200 (sm_100a) rollout engine for 2048.
 *
 * This is the drop-in boundary for the one hot path of michaelriedl/2048-ppo-agent: the batched
 * 2048 env step fused with action selection, rollout-buffer writes and GAE.  The reference has no
 * FFI of its own (it is pure Python on Pgx/JAX); each entry point below names the reference code
 * it replaces (paths relative to the reference repo root).  INTEGRATION.md shows the ctypes
 * binding a maintainer adds on the reference side.
 *
 * Conventions
 *   - Plain pointers and sizes only; no torch / jax types.  Every `d_` pointer is DEVICE memory
 *     on the current CUDA device, every `h_` pointer is HOST memory.  Nothing is allocated or
 *     freed by `d_` entry points; work is enqueued on `stream` (a cudaStream_t passed as void*,
 *     NULL = legacy default stream) and the call returns without synchronising.
 *     `*_host` entry points take host buffers, do their own device allocation + H2D/D2H copies
 *     and synchronise before returning.
 *   - Return value: 0 on success, G2048_ERR_INVALID (-1) for a bad argument, otherwise the
 *     cudaError_t that was raised.  g2048_last_error() gives the text.  There is no CPU
 *     fallback: without a CUDA device every compute entry point fails.
 *   - Board: uint64 nibble bitboard, cell i = 4*row + col in bits [4i, 4i+4), value = exponent
 *     (0 empty, e = tile 2^e, Pgx's own encoding).  Status byte per env: bits 0-3 = legal-action
 *     mask as Pgx exposes it (bit a = action a legal; all four set on a terminal state),
 *     bit 4 = terminated, bit 5 = sticky "tile 2^16 needed" overflow flag.
 *   - Actions: 0 = Left, 1 = Up, 2 = Right, 3 = Down (src/actions/act_drul.py:8,39-40).
 *   - Keys: a jax.random key is two uint32 words (hi, lo).  `rng_mode` selects the Threefry
 *     counter layout: G2048_RNG_ORIGINAL (jax_threefry_partitionable=False) or
 *     G2048_RNG_PARTITIONABLE (=True, default of the pinned jax==0.5.3).
 *   - Env indices are GLOBAL: a shard owns envs [env_lo, env_lo + n) of a batch of
 *     `batch_global` envs, and per-env keys are split(sub, batch_global)[env index], so results
 *     do not depend on how the batch is sharded over GPUs.  Entry points that take one sub key
 *     (`d_sub`) also accept batch_global == 0 (with env_lo == 0): `d_sub` is then an explicit
 *     (n,2) array of per-env keys, exactly what jax.vmap(act_fn)(keys, obs, mask) receives.
 *     The fused loops (g2048_play, g2048_rollout_steps) need batch_global > 0.
 */
#ifndef G2048_H_
#define G2048_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define G2048_OK 0
#define G2048_ERR_INVALID (-1)

#define G2048_RNG_ORIGINAL 0
#define G2048_RNG_PARTITIONABLE 1

#define G2048_POLICY_RANDOM 0 /* src/actions/act_randomly.py:40-56 */
#define G2048_POLICY_DRUL 1   /* src/actions/act_drul.py:40-49 */

#define G2048_STATUS_MASK 0x0F
#define G2048_STATUS_DONE 0x10
#define G2048_STATUS_OVERFLOW 0x20

#define G2048_OBS_BOOL 0 /* uint8 0/1, the layout of pgx State.observation (4,4,31) bool */
#define G2048_OBS_F32 1  /* float32, what RolloutBuffer.get_buffer_data / PPOAgent consume */
#define G2048_OBS_BF16 2

/* number of uint64 slots of the play statistics block, see g2048_play */
#define G2048_PLAY_STATS_WORDS 32

int g2048_version(void);
const char* g2048_last_error(void);
/* SM count of the current device, or a negative error */
int g2048_device_sm_count(void);

/* ---- RNG (replaces jax.random.key/split at src/runs/batch_runner.py:32,105-106,118-119,126-127) */

/* Threefry-2x32-20 blocks: out[i] = TF(key[i]; ctr[i]); all (n,2) uint32.  Test hook / KATs. */
int g2048_threefry2x32(const uint32_t* d_keys, const uint32_t* d_ctrs, int64_t n, uint32_t* d_out, void* stream);

/* The runner's chain `key, sub = split(key)` advanced n_sub times on the device:
 * d_subs[(n_sub,2)] receives the successive sub keys, d_key_io[2] the advanced chain key. */
int g2048_chain_advance(uint32_t* d_key_io, int rng_mode, int64_t n_sub, uint32_t* d_subs, void* stream);

/* keys[i] = split(*d_sub, batch_global)[env_lo + i], i < n: the per-env keys the reference hands
 * to vmap(act_fn) / vmap(env.step).  Only needed when a caller-supplied policy wants real keys. */
int g2048_split_keys(const uint32_t* d_sub, int64_t batch_global, int64_t env_lo, int64_t n, int rng_mode,
                     uint32_t* d_keys, void* stream);

/* ---- env (replaces pgx "2048" init/step via jit(vmap(...)) at src/runs/batch_runner.py:34-35,107,128) */

/* env.init(split(*d_sub, batch_global)[env_lo + i]) -> board, status (rewards 0, not terminated) */
int g2048_env_init(const uint32_t* d_sub, int64_t batch_global, int64_t env_lo, int64_t n, int rng_mode,
                   uint64_t* d_boards, uint8_t* d_status, void* stream);

/* env.step(state, action, split(*d_sub, batch_global)[env_lo + i]) in place.
 * d_rewards (n) float32 as pgx State.rewards[:,0]; frozen envs get 0, an action illegal under the
 * pre-step mask gets -1 and terminates.  d_actions int32. */
int g2048_env_step(uint64_t* d_boards, uint8_t* d_status, const int32_t* d_actions, const uint32_t* d_sub,
                   int64_t batch_global, int64_t env_lo, int64_t n, int rng_mode, float* d_rewards, void* stream);

/* Same step with the spawn's two 32-bit draws supplied per env (position draw, value draw) instead
 * of a key: the "identical actions and spawn draws" form the bit-exactness contract is stated in. */
int g2048_env_step_draws(uint64_t* d_boards, uint8_t* d_status, const int32_t* d_actions,
                         const uint32_t* d_bits_pos, const uint32_t* d_bits_val, int64_t n, float* d_rewards,
                         void* stream);

/* vmap(act_randomly | act_drul)(split(*d_sub, batch_global)[env_lo + i], obs, mask):
 * d_actions int32 (n); d_log_probs float32 (n) or NULL (act_drul returns None). */
int g2048_act(int policy, const uint8_t* d_status, const uint32_t* d_sub, int64_t batch_global, int64_t env_lo,
              int64_t n, int rng_mode, int32_t* d_actions, float* d_log_probs, void* stream);

/* ---- fused loops */

/* Play envs [env_lo, env_lo+n) of BatchRunner(seed).run_*(batch_global) to termination inside ONE
 * persistent kernel (src/runs/batch_runner.py:105-136 with act_randomly / act_drul, and the
 * max-tile reduction of src/runs/run_actions_max_tile.py:61-69).  Lanes that finish an episode
 * pull the next env, so no lane idles on a frozen env.
 *   d_subs: chain sub keys, [0] = init, [1+2t] = act keys of loop step t, [2+2t] = step keys;
 *           n_subs of them are valid (episodes longer than (n_subs-1)/2 set stats[3]).
 *   d_work: uint64[2] scratch, zeroed by the caller: [0] = env queue head, [1] unused.
 *   d_final_boards / d_lengths / d_scores: per-env outputs (n), each may be NULL.
 *           length = loop steps until terminated (first done index + 1), score = sum of rewards.
 *   d_stats: uint64[G2048_PLAY_STATS_WORDS], ACCUMULATED into (caller zeroes):
 *           [0] episodes, [1] env-steps, [2] sum of scores, [3] envs cut short by n_subs,
 *           [4] envs with the overflow flag, [5] longest episode, [6] sum max_tile, [7] sum max_tile^2,
 *           [16+e] episodes whose max tile is 2^e (e = 0..15). */
int g2048_play(int policy, const uint32_t* d_subs, int64_t n_subs, int64_t batch_global, int64_t env_lo, int64_t n,
               int rng_mode, uint64_t* d_work, uint64_t* d_final_boards, uint32_t* d_lengths, uint32_t* d_scores,
               uint64_t* d_stats, void* stream);

/* The two kernels behind g2048_play, each with the same arguments and results: `_tables` keeps the
 * row move / legality tables in shared memory (192 KiB per CTA; used for n >= 32768), `_swar` does
 * the board logic with SWAR arithmetic in registers (no tables; small batches). */
int g2048_play_tables(int policy, const uint32_t* d_subs, int64_t n_subs, int64_t batch_global, int64_t env_lo,
                      int64_t n, int rng_mode, uint64_t* d_work, uint64_t* d_final_boards, uint32_t* d_lengths,
                      uint32_t* d_scores, uint64_t* d_stats, void* stream);
int g2048_play_swar(int policy, const uint32_t* d_subs, int64_t n_subs, int64_t batch_global, int64_t env_lo,
                    int64_t n, int rng_mode, uint64_t* d_work, uint64_t* d_final_boards, uint32_t* d_lengths,
                    uint32_t* d_scores, uint64_t* d_stats, void* stream);

/* Per-env results of a play-to-termination run as one 16-byte record (little-endian; a numpy structured dtype
 * {"board": "<u8", "length": "<u4", "score": "<u4"} views an array of them). */
typedef struct G2048EpisodeResult {
    uint64_t board;  /* final bitboard */
    uint32_t length; /* env-steps played */
    uint32_t score;  /* sum of the merge rewards */
} G2048EpisodeResult;

/* g2048_play with the per-env results as ONE record per env instead of three arrays (d_results: n records, 16-byte
 * aligned, may be NULL): a finished episode is a single 16-byte store.  Same dispatch, statistics and key usage. */
int g2048_play_packed(int policy, const uint32_t* d_subs, int64_t n_subs, int64_t batch_global, int64_t env_lo, int64_t n,
                      int rng_mode, uint64_t* d_work, G2048EpisodeResult* d_results, uint64_t* d_stats, void* stream);

/* ---- recorded play to termination: g2048_play that also keeps every env's trajectory (the rollout-buffer write of
 * src/runs/batch_runner.py:117-154 + src/ppo/rollout_buffer.py:164-187 fused into the persistent table kernel).
 * A lane plays its envs one after the other, so it appends their records to its own region of an ARENA
 * (d_arena_boards: uint64 per slot, d_arena_meta: uint8 per slot; arena_slots slots, at least
 * g2048_play_record_arena_slots(n, n_subs, mean_steps) of them, mean_steps = the caller's estimate of the mean episode
 * length -- it only sizes the lanes' regions).  Per env-step one slot: the pre-step board and a meta byte (bits 0-1
 * action, 2-5 pre-step legal mask, 6 post-step done, 7 "the spawn of this step was a 4-tile"); after an env's last
 * step one more slot with its final board.  d_env_slot[i] (uint64, n) = slot of step 0 of env env_lo + i, so its
 * episode is slots [d_env_slot[i], d_env_slot[i] + d_lengths[i]].  d_lengths is required; the other per-env outputs
 * and d_stats are those of g2048_play.  If the arena is too small for the batch some envs are not played:
 * d_stats[0] (episodes) < n then, and the caller retries with more slots.
 *
 * g2048_play_record_compact turns the arena into the env-major flat buffer RolloutBuffer keeps (what
 * g2048_rollout_steps + g2048_compact_records produce, bit for bit): flat index = out_base + d_offsets[i] + t for
 * t < d_lengths[i] (d_offsets = exclusive scan of d_lengths).  d_boards pre-step boards, d_meta bits 0-6 of the meta
 * byte, d_rewards = potential(board t+1) - potential(board t) - 4 * bit 7 (= the sum of the merged tiles' values,
 * Pgx's reward), d_log_probs = log(1 / #legal actions) for G2048_POLICY_RANDOM and 0 for DRUL, d_values = 0.
 * d_max_reward (n, float32) = max over the env's steps of the reward (the trainer's "episode reward",
 * src/ppo/ppo_trainer.py:218-227).  Any output may be NULL.  out_capacity = the number of steps of this batch the flat output
 * arrays have room for: a step with d_offsets[i] + t >= out_capacity is not written, so a caller may launch the compaction into arrays
 * sized from an ESTIMATE of the total before it has read the statistics back, and repeat it only if the estimate was
 * short (d_offsets[n] is the exact total).  d_max_reward is always complete. */
int64_t g2048_play_record_arena_slots(int64_t n, int64_t n_subs, int64_t mean_steps);
int g2048_play_record(int policy, const uint32_t* d_subs, int64_t n_subs, int64_t batch_global, int64_t env_lo, int64_t n,
                      int rng_mode, uint64_t* d_work, uint64_t* d_arena_boards, uint8_t* d_arena_meta, int64_t arena_slots,
                      uint64_t* d_env_slot, uint64_t* d_final_boards, uint32_t* d_lengths, uint32_t* d_scores,
                      uint64_t* d_stats, void* stream);
int g2048_play_record_compact(int policy, const uint64_t* d_arena_boards, const uint8_t* d_arena_meta,
                              const uint64_t* d_env_slot, const uint32_t* d_lengths, const int64_t* d_offsets, int64_t n,
                              int64_t out_base, int64_t out_capacity, uint64_t* d_boards, uint8_t* d_meta, float* d_rewards,
                              float* d_log_probs, float* d_values, float* d_max_reward, void* stream);

/* Test hook for the shared-memory tables of g2048_play_tables: for each 16-bit row (four nibbles, nibble 0 =
 * column 0) the row slid/merged toward column 0 and the flags (bit 0: moves left, bit 2: moves right). */
int g2048_row_table_lookup(const uint16_t* d_rows, int64_t n, uint16_t* d_left, uint8_t* d_flags, void* stream);

/* ---- Monte-Carlo playout values of caller-given boards: for every (board, action) pair, K games played to the end
 * with a built-in rollout policy after that action (the play kernel of g2048_play_tables started from a given board
 * with a forced first move).
 *   d_boards (n): start bitboards.  Board i has the GLOBAL id d_board_ids[i] (int64, each in [0, n_boards_global)),
 *           or board_lo + i when d_board_ids is NULL (board_lo must be 0 with an id list).
 *   playouts = K >= 1.  Playout p = (id * 4 + a) * K + k, k < K, belongs to a batch of P = n_boards_global * 4 * K
 *           playouts (P <= 2^31 - 1, else G2048_ERR_INVALID), and starts from board `id`:
 *           at t = 0 it plays action a and spawns with split(d_subs[2], P)[p]; at t >= 1 the policy acts with
 *           split(d_subs[1 + 2t], P)[p] and the step spawns with split(d_subs[2 + 2t], P)[p] -- g2048_play's per-env
 *           derivations, so the draws do not depend on how the boards are sharded or ordered.
 *   d_subs: n_subs >= 3 sub keys laid out as for g2048_play ([0] unused, [1+2t] act, [2+2t] step keys);
 *           max_steps = (n_subs - 1) / 2 steps per playout, a playout still running then is cut short.
 *   d_work: uint64[2] scratch, zeroed by the caller (queue head).
 *   d_records (n * 4, 8-byte aligned): record 4 i + a, OVERWRITTEN: sums over the K playouts of (board i, action a) of
 *           the score (merge rewards from the start board on, the forced move's included), its square and the steps
 *           (the forced move included); `playouts` = K if a is legal on board i, else 0 (an illegal pair is not
 *           played); `cut_short` = playouts that reached max_steps.
 *   d_stats: NULL, or uint64[G2048_PLAY_STATS_WORDS] ACCUMULATED as g2048_play's, playouts counted as episodes.
 * A start board that holds a 2^15 tile is outside the contract (as for g2048_play); such playouts are counted in
 * d_stats[4]. */
typedef struct G2048PlayoutStats {
    uint64_t score_sum;
    uint64_t score_sq_sum;
    uint64_t steps_sum;
    uint32_t playouts;
    uint32_t cut_short;
} G2048PlayoutStats;
int g2048_playout_values(int policy, const uint64_t* d_boards, int64_t n, const int64_t* d_board_ids, int64_t board_lo,
                         int64_t n_boards_global, int64_t playouts, const uint32_t* d_subs, int64_t n_subs, int rng_mode,
                         uint64_t* d_work, G2048PlayoutStats* d_records, uint64_t* d_stats, void* stream);

/* ---- Depth-limited expectimax values of caller-given boards over a row heuristic (no pruning, no transposition
 * table; all arithmetic float32 in exactly this order, so the values are bit-exact):
 *   H(b)      = T[row0] + T[row1] + T[row2] + T[row3] + T[col0] + T[col1] + T[col2] + T[col3], left to right
 *               (row r = bits [16r, 16r+16); column c = row c of the transpose: nibble k is cell 4k + c);
 *   Q_1(b, a) = w * r + H(b_a);  Q_k(b, a) = w * r + C_{k-1}(b_a) for k >= 2, where (b_a, r) = move(b, a), a legal,
 *               and r = potential(b_a) - potential(b) is the merge reward (no spawn);
 *   C_k(s)    = acc / (float)n_empty, acc = 0 then acc = acc + (0.9f * V_k(s + 2@c) + 0.1f * V_k(s + 4@c)) for the
 *               empty cells c of s in increasing index;
 *   V_k(b)    = max over the legal a of Q_k(b, a); 0 for a board without a legal action.
 *   d_boards (n): bitboards; n >= 0 (n = 0 is a no-op).  depth = d in 1..4 counts moves.
 *   d_row_values: T, float[65536] (device).  reward_weight: w.
 *   d_q (n * 4, 4-byte aligned): OVERWRITTEN with Q_d(board i, a) at 4 i + a, NaN where a is illegal on board i.
 *   d_counters: NULL, or uint64[2] ACCUMULATED: [0] H evaluations (leaves), [1] chance nodes expanded.  Both depend on
 *           the tree alone.
 * A board that holds a 2^15 tile is outside the contract (as for g2048_play). */
int g2048_expectimax_values(const uint64_t* d_boards, int64_t n, int depth, const float* d_row_values, float reward_weight,
                            float* d_q, uint64_t* d_counters, void* stream);

/* ---- Batched TD(0) afterstate learning of the row table T that g2048_expectimax_values reads (H as above).
 * Synchronous: every env of a step reads the same frozen T_t, the TD errors are summed in fixed point with integer
 * atomics, and T_{t+1} is applied after the whole batch has made the step -- so the result is bit-exact and does not
 * depend on how the work is spread over the GPU.
 * State of env e < n: d_boards (uint64), d_after (uint64: the previous afterstate, 0 = none -- no afterstate is the
 * empty board), d_scores and d_lengths (uint32).  Step t uses k = split(d_subs[t], n)[e] and does for every env:
 *   1. s = board.  If s has a legal action: q_a = (float)r_a + H_t(s_a) for each legal a in action order,
 *      (s_a, r_a) = move(s, a); a* = the first legal action, replaced by every strictly larger q; target = q_{a*}
 *      (Q_1 of g2048_expectimax_values with w = 1, the same tie rule).  Without a legal action target = 0.
 *   2. If after != 0: delta = target - H_t(after) (float32, no contraction); for each of the 8 lines of after in H's
 *      order acc[idx] += fx(delta) and cnt[idx] += 1, where fx(d) = rint(clamp(d, -2^24, 2^24) * 4096) as int64,
 *      rounded to nearest even (clamp(d, lo, hi) = fminf(fmaxf(d, lo), hi)).
 *   3. Without a legal action the episode ends: it is counted in d_stats, board = init(k) (g2048_env_init with the
 *      explicit key k) and after = score = length = 0; the env makes no move this step.  Otherwise
 *      board = step(s, a*, k) (g2048_env_step: the same spawn draws), after = s_{a*}, score += r_{a*}, length += 1.
 *   4. After all envs: for every i with cnt[i] > 0, T[i] = T[i] + alpha * (float)((double)acc[i] / (4096.0 *
 *      (double)cnt[i])) (float multiply and add, not fused); then acc[i] = cnt[i] = 0.  The per-entry mean makes the
 *      learning rate independent of the batch size and of how common a row is: a row seen once gets alpha * delta.
 *   d_row_values: T, float[65536], updated in place.  d_subs: n_steps sub keys (n_steps >= 0; 0 is a no-op).
 *   d_scratch: g2048_td_scratch_bytes() bytes (acc int64[65536], then cnt uint32[65536]), zeroed by the caller once;
 *           every call leaves it zeroed.
 *   d_stats: NULL, or uint64[G2048_PLAY_STATS_WORDS] ACCUMULATED in g2048_play's layout over the episodes that end
 *           in the call: [0] episodes, [1] their moves, [2] their scores, [4] those whose final board holds a 2^15
 *           tile, [5] longest, [6] / [7] sum of max tile / its square, [16 + e] episodes whose max tile is 2^e.
 * G2048_ERR_INVALID for n outside [1, 2^20], n_steps < 0, a negative or non-finite alpha, NULL or misaligned
 * pointers (8 bytes for boards, after, subs, scratch and stats; 4 for the others).  The launch is cooperative: it
 * fails with an error, rather than waiting, if its grid cannot be resident at once.  A board that holds a 2^15 tile
 * is outside the contract (as for g2048_play). */
int64_t g2048_td_scratch_bytes(void);
int g2048_td_train(uint64_t* d_boards, uint64_t* d_after, uint32_t* d_scores, uint32_t* d_lengths, int64_t n,
                   float* d_row_values, float alpha, const uint32_t* d_subs, int64_t n_steps, int rng_mode,
                   void* d_scratch, uint64_t* d_stats, void* stream);

/* ---- N-tuple networks: a value function V over one flat float32 weight array W (n_weights entries), given as an
 * ordered list of placements.  Placement p reads the k = n_cells cells cells[0..k) of the board:
 *   idx_p(b) = sum over j < k of exp(b, cells[j]) << 4j        (cell = 4 * row + col, exp(b, c) = nibble c of b)
 *   V(b)     = W[off_0 + idx_0(b)] + W[off_1 + idx_1(b)] + ... + W[off_{P-1} + idx_{P-1}(b)], float32, left to right
 *              from the first term (no leading 0).
 * Several placements with the same offset share one table (symmetric sharing).  The row heuristic H above is the
 * network of one 65 536-entry table at offset 0 with the 8 placements (4r, 4r+1, 4r+2, 4r+3) for r = 0..3, then
 * (c, c+4, c+8, c+12) for c = 0..3: V == H bit for bit.
 * The placement list is a HOST array of 1..G2048_NTUPLE_MAX_PLACEMENTS entries, checked before any launch:
 * G2048_ERR_INVALID for n_cells outside 1..6, a cell >= 16 or repeated within a placement, a nonzero reserved byte,
 * off + 16^k > n_weights, or n_weights outside [1, 2^28]. */
typedef struct G2048TuplePlacement {
    uint32_t offset;  /* first entry of this placement's table in W */
    uint8_t n_cells;  /* k, 1..6 */
    uint8_t cells[6]; /* cell = 4*row + col; nibble j of the index is the exponent in cells[j] */
    uint8_t reserved; /* 0 */
} G2048TuplePlacement; /* 12 bytes */
#define G2048_NTUPLE_MAX_PLACEMENTS 64
#define G2048_NTUPLE_MAX_WEIGHTS (1ll << 28)

/* Batched TD(0) afterstate learning of an n-tuple network: g2048_td_train's contract word for word, with V in place of
 * H and, in step 2, for each placement p in order acc[off_p + idx_p(after)] += fx(delta) and cnt[...] += 1.  With
 * P <= 64 and n <= 2^20, |acc[i]| <= 2^20 * 64 * 2^36 = 2^62: the int64 sums cannot overflow.  Step 4 is the same
 * per-entry mean for every entry with cnt[i] > 0, so the result is bit-exact whatever the grid or the atomics' order.
 *   d_weights: W, float[n_weights], updated in place (4-byte aligned).
 *   d_scratch: g2048_ntuple_td_scratch_bytes(n, n_placements, n_weights) bytes, zeroed by the caller once; every call
 *           leaves it zeroed.  The size grows with n_weights (the per-entry sums), and with n * n_placements (the
 *           list of the entries touched in one step: the update after each step costs work proportional to those
 *           entries, not to n_weights).  g2048_ntuple_td_scratch_bytes returns -1 for invalid sizes.
 * G2048_ERR_INVALID for everything g2048_td_train rejects and for an invalid network (above). */
int64_t g2048_ntuple_td_scratch_bytes(int64_t n, int n_placements, int64_t n_weights);
int g2048_ntuple_td_train(uint64_t* d_boards, uint64_t* d_after, uint32_t* d_scores, uint32_t* d_lengths, int64_t n,
                          const G2048TuplePlacement* h_placements, int n_placements, float* d_weights, int64_t n_weights,
                          float alpha, const uint32_t* d_subs, int64_t n_steps, int rng_mode,
                          void* d_scratch, uint64_t* d_stats, void* stream);

/* Batched temporal coherence (TC) learning of an n-tuple network (Beal & Smith 1999; Jaskowski 2018): every weight
 * has its own step size, scaled by how consistently its errors agree in sign.  Steps 1 to 3 are g2048_ntuple_td_train
 * word for word, and step 2 also adds |fx(delta)| into abs[off_p + idx_p(after)] for each placement p (int64, the same
 * 2^62 bound as acc).  Step 4, for every i with cnt[i] > 0, in double unless stated otherwise:
 *     m    = (double)acc[i] / (4096.0 * (double)cnt[i])
 *     beta = A[i] > 0 ? fmin(fabs(E[i]) / A[i], 1.0) : 1.0          (E and A as they were before this step)
 *     W[i] = W[i] + alpha * (float)(beta * m)                       (float multiply and add, not fused)
 *     E[i] = E[i] + (double)acc[i] / 4096.0
 *     A[i] = A[i] + (double)abs[i] / 4096.0
 * then acc[i] = abs[i] = cnt[i] = 0.  A weight whose errors keep one sign keeps beta near 1; one whose errors cancel
 * stops moving.  |E| <= A holds exactly; the fmin absorbs the rounding of the two double sums.  From E = A = 0 one
 * step equals one g2048_ntuple_td_train step with the same alpha, bit for bit.  With alpha = 0 W stays fixed while E
 * and A still accumulate.
 *   d_err_sum, d_abs_err_sum: E and A, float64[n_weights] each, 8-byte aligned, updated in place (zero at the start of
 *           a run).  They are float64 because A only grows: by an estimate from the sizes, a hot entry at n = 2^16
 *           can gain about 2^41 a step, so an int64 fixed-point A would reach 2^63 after a few million steps, and a
 *           float32 A would stop absorbing increments long before that.
 *   d_scratch: g2048_ntuple_tc_scratch_bytes(n, n_placements, n_weights) bytes (acc int64[n_weights], abs
 *           int64[n_weights], cnt uint32[n_weights], the touched list, the two list lengths), zeroed by the caller
 *           once; every call leaves it zeroed.  g2048_ntuple_tc_scratch_bytes returns -1 for invalid sizes.
 * G2048_ERR_INVALID for everything g2048_ntuple_td_train rejects and for NULL or misaligned d_err_sum / d_abs_err_sum.
 * The `lines` network through this entry point is TC learning of the row table. */
int64_t g2048_ntuple_tc_scratch_bytes(int64_t n, int n_placements, int64_t n_weights);
int g2048_ntuple_tc_train(uint64_t* d_boards, uint64_t* d_after, uint32_t* d_scores, uint32_t* d_lengths, int64_t n,
                          const G2048TuplePlacement* h_placements, int n_placements, float* d_weights, int64_t n_weights,
                          double* d_err_sum, double* d_abs_err_sum, float alpha, const uint32_t* d_subs,
                          int64_t n_steps, int rng_mode, void* d_scratch, uint64_t* d_stats, void* stream);

/* g2048_expectimax_values with V of an n-tuple network in place of H at the leaves: the same tree, float order, NaN
 * for illegal actions and counters.  d_weights: W, float[n_weights] (device, read-only while the call runs).  Depth 1
 * with reward_weight 1 is g2048_ntuple_td_train's greedy move. */
int g2048_expectimax_values_ntuple(const uint64_t* d_boards, int64_t n, int depth,
                                   const G2048TuplePlacement* h_placements, int n_placements,
                                   const float* d_weights, int64_t n_weights, float reward_weight,
                                   float* d_q, uint64_t* d_counters, void* stream);

/* ---- Multi-stage n-tuple networks (Yeh et al. 2016; Jaskowski 2018): the game is split into S = n_thresholds + 1
 * stages by the largest tile on the board, and each stage has its own copy of every table, `stride` entries after the
 * previous stage's.
 *   stage(b) = the number of j < n_thresholds with max_exponent(b) >= thresholds[j]    (the empty board: stage 0)
 *   V_S(b)   = W[stage(b) * stride + off_0 + idx_0(b)] + ... + W[stage(b) * stride + off_{P-1} + idx_{P-1}(b)],
 *              float32, left to right from the first term: V's float order, and V itself when S = 1.
 * The stage is that of the board being valued: a TD target r + V_S(s'') may lie in a higher stage than V_S(after), so
 * errors cross stage borders, and all stages learn in one launch.  The stages are a HOST struct, checked with the
 * placements before any launch: G2048_ERR_INVALID for a NULL pointer, n_thresholds > 15, thresholds that are not
 * strictly increasing in 1..15, a nonzero unused threshold byte, stride != 0 when S = 1 or stride == 0 when S > 1, or
 * (S - 1) * stride + off_p + 16^k > n_weights for some placement.  n_weights stays at most 2^28, so the 4x6 network
 * (2^26 weights a stage) has at most 4 stages. */
typedef struct G2048TupleStages {
    uint32_t stride;         /* entries from one stage's tables to the next stage's; 0 when n_thresholds == 0 */
    uint8_t n_thresholds;    /* S - 1, 0..15 */
    uint8_t thresholds[15];  /* tile exponents, strictly increasing, each in 1..15; unused bytes 0 */
} G2048TupleStages;          /* 20 bytes */
#define G2048_NTUPLE_MAX_STAGES 16

/* The three n-tuple entry points above, word for word, with V_S in place of V.  The scratch sizes are those of the
 * unstaged calls (g2048_ntuple_td_scratch_bytes, g2048_ntuple_tc_scratch_bytes): they depend on n, P and n_weights
 * only, and one step still touches at most min(n * P, n_weights) entries.  The results are bit-exact and independent
 * of the grid, as for the unstaged calls: each entry still receives one integer sum (and count) per step.  With
 * S = 1 each call equals its unstaged form bit for bit. */
int g2048_ntuple_staged_td_train(uint64_t* d_boards, uint64_t* d_after, uint32_t* d_scores, uint32_t* d_lengths,
                                 int64_t n, const G2048TuplePlacement* h_placements, int n_placements,
                                 const G2048TupleStages* h_stages, float* d_weights, int64_t n_weights, float alpha,
                                 const uint32_t* d_subs, int64_t n_steps, int rng_mode, void* d_scratch,
                                 uint64_t* d_stats, void* stream);
int g2048_ntuple_staged_tc_train(uint64_t* d_boards, uint64_t* d_after, uint32_t* d_scores, uint32_t* d_lengths,
                                 int64_t n, const G2048TuplePlacement* h_placements, int n_placements,
                                 const G2048TupleStages* h_stages, float* d_weights, int64_t n_weights,
                                 double* d_err_sum, double* d_abs_err_sum, float alpha, const uint32_t* d_subs,
                                 int64_t n_steps, int rng_mode, void* d_scratch, uint64_t* d_stats, void* stream);
int g2048_expectimax_values_ntuple_staged(const uint64_t* d_boards, int64_t n, int depth,
                                          const G2048TuplePlacement* h_placements, int n_placements,
                                          const G2048TupleStages* h_stages, const float* d_weights, int64_t n_weights,
                                          float reward_weight, float* d_q, uint64_t* d_counters, void* stream);

/* ---- Delayed TD(lambda) and TC(lambda) learning of an n-tuple network (Jaskowski 2018, delayed temporal coherence):
 * each env keeps a window of its last h = horizon afterstates and their errors, and an afterstate is updated h - 1
 * steps late with the lambda-weighted sum of its h errors (a truncated lambda-return).  g2048_ntuple_td_train's contract
 * (g2048_ntuple_tc_train's for the TC form; V_S of h_stages, or V when h_stages is NULL) word for word except step 2.
 *   c_k (k < h): computed on the host in double by repeated multiplication, d_0 = 1, d_k = d_{k-1} * (double)lambda,
 *           c_k = (float)d_k (no pow).
 *   d_hist_after: uint64[h * n], the afterstates; d_hist_delta: float[h * n], their errors.  Slot-major: entry (j, e)
 *           is at j * n + e.  Caller-owned, updated in place; zeros are a valid start.
 * Let L = lengths[e] at the start of the step.  x_m (m = 1..L) is the afterstate of the episode's m-th move and lives in
 * slot (m - 1) mod h with its error delta_m.  The window is defined by L alone: slots of an earlier episode are never
 * read.  Step 2 becomes: if after != 0 (after = x_L) and 1 <= L < 2^31 (an env with an afterstate and L outside that
 * range is outside the contract; it stores and releases nothing):
 *   a. delta_L = target - V_t(x_L) as in step 2 of g2048_ntuple_td_train; it is stored in hist_delta slot (L - 1) mod h.
 *   b. Released afterstates: if the env moves, x_{L-h+1} when L >= h; if the episode ends, every x_m with
 *      max(1, L - h + 1) <= m <= L (their missing later errors count as 0).
 *   c. A released x_m carries e_m = delta_m, then e_m = e_m + c_k * delta_{m+k} for k = 1, 2, ... while m + k <= L
 *      (so k <= h - 1), float32, the product rounded before the add (no contraction).
 *   d. For each released x_m and each placement p in order: fx(e_m) into acc, 1 into cnt (TC: |fx(e_m)| into abs) at
 *      stage(x_m) * stride + off_p + idx_p(x_m).
 * Step 3 also stores the new afterstate x_{L+1} in hist_after slot L mod h (the slot just released) when the env moves.
 * Step 4 (TC: beta, E and A) is unchanged.  The errors of a window were computed with the weights of their own steps,
 * not with the weights at the release ("delayed" lambda-returns).  With h = 1 (any lambda) each call equals
 * g2048_ntuple_td_train / g2048_ntuple_tc_train (staged: their staged forms) bit for bit.  An env releases at most h
 * afterstates a step, so |acc[i]| <= n * h * 64 * 2^36; n * h <= 2^20 keeps the 2^62 bound.  The results are bit-exact
 * and independent of the grid: each entry still receives one integer (sum, |sum|, count) per step.
 *   d_scratch: g2048_ntuple_td_scratch_bytes(n * h, n_placements, n_weights) bytes (TC: g2048_ntuple_tc_scratch_bytes),
 *           zeroed by the caller once; every call leaves it zeroed (a step touches at most n * h * P entries).
 * G2048_ERR_INVALID before any launch for everything the corresponding call rejects, lambda not finite or outside
 * [0, 1], horizon outside 1..G2048_NTUPLE_MAX_HORIZON, n * horizon > 2^20, and NULL or misaligned hist pointers (8 bytes
 * for d_hist_after, 4 for d_hist_delta). */
#define G2048_NTUPLE_MAX_HORIZON 8
int g2048_ntuple_lambda_td_train(uint64_t* d_boards, uint64_t* d_after, uint32_t* d_scores, uint32_t* d_lengths,
                                 int64_t n, const G2048TuplePlacement* h_placements, int n_placements,
                                 const G2048TupleStages* h_stages, float* d_weights, int64_t n_weights, float alpha,
                                 float lambda, int horizon, uint64_t* d_hist_after, float* d_hist_delta,
                                 const uint32_t* d_subs, int64_t n_steps, int rng_mode, void* d_scratch,
                                 uint64_t* d_stats, void* stream);
int g2048_ntuple_lambda_tc_train(uint64_t* d_boards, uint64_t* d_after, uint32_t* d_scores, uint32_t* d_lengths,
                                 int64_t n, const G2048TuplePlacement* h_placements, int n_placements,
                                 const G2048TupleStages* h_stages, float* d_weights, int64_t n_weights,
                                 double* d_err_sum, double* d_abs_err_sum, float alpha, float lambda, int horizon,
                                 uint64_t* d_hist_after, float* d_hist_delta, const uint32_t* d_subs, int64_t n_steps,
                                 int rng_mode, void* d_scratch, uint64_t* d_stats, void* stream);

/* ---- Carousel shaping of a multi-stage network (Jaskowski 2018): episodes take turns starting at the opening and
 * from the boards at which earlier episodes entered stage 1, 2, ..., so that the later stages get a fair share of the
 * training.  g2048_ntuple_lambda_td_train / _tc_train word for word (h = 1: TD(0) / TC), with d_hist_after and
 * d_hist_delta allowed to be NULL when horizon == 1, h_stages required with S >= 2, and two caller-owned arrays:
 *   d_start_stage: uint32[n], per env the stage its current episode began in (4-byte aligned).
 *   d_stage_pool:  uint64[(S - 1) * n], stage-major (8-byte aligned): entry (l - 1, e) at (l - 1) * n + e is the board
 *           at which env e most recently entered stage l; 0 is none.
 * Zeroed arrays are a valid start: such a run is the staged learner's until the first stage entry.  Only step 3 and
 * the statistics change:
 *   Recording (an env that moves): s is the board at the start of the step, s' = spawn(best) its new board.  If
 *           stage(s') > stage(s) (by 1: the thresholds are strictly increasing and the largest exponent grows by at
 *           most 1 a move), s' is written to pool entry (stage(s') - 1, e).  The write is visible from step t + 1:
 *           every draw of step t reads the pool as it was at the start of step t, which keeps the results bit-exact
 *           and independent of the grid.
 *   Restart (an env without a legal move): c = start_stage[e], l = c + 1 if c + 1 < S, else 0 (c >= S - 1 wraps to 0).
 *           If l >= 1: split2(k, k1, k2) with the env's step key k, j = (uint32)(((uint64)bits_scalar(k1) * n) >> 32),
 *           b = pool entry (l - 1, j) as it was at the start of the step; if b != 0 the env restarts from b with
 *           start_stage[e] = l.  Otherwise (l = 0 or an empty entry) it restarts from init(k) as before, with
 *           start_stage[e] = 0.  In both cases after, score and length go to 0.  Pool boards that hold a 2^15 tile are
 *           outside the contract, as for d_boards.
 *   Statistics: words [0..7] and [16 + e] count only the episodes that began at the opening (start_stage == 0), so
 *           summaries stay comparable with the other learners'; the episodes that began from a pool board add 1 to
 *           word [12] and their length to word [13].
 * Equivalence: if no env enters a stage during a call, the pool stays as it was, and with an empty pool every restart
 * takes init(k): the call then equals g2048_ntuple_staged_td_train / _tc_train (h = 1) or
 * g2048_ntuple_lambda_td_train / _tc_train (h > 1) bit for bit -- W, E, A, the env state, the rings and the
 * statistics.
 *   d_scratch: g2048_ntuple_carousel_scratch_bytes(n, horizon, n_placements, n_weights, tc) bytes: the lambda form's
 *           scratch for n * h envs, then one pending board per env (uint64[n]) that holds a stage entry until the
 *           pool takes it after the step's draws.  Zeroed by the caller once; every call leaves it zeroed.  -1 for
 *           invalid sizes.
 * G2048_ERR_INVALID before any launch for everything the lambda entry points reject, NULL h_stages or S = 1, and NULL
 * or misaligned d_start_stage / d_stage_pool. */
int64_t g2048_ntuple_carousel_scratch_bytes(int64_t n, int horizon, int n_placements, int64_t n_weights, int tc);
int g2048_ntuple_carousel_td_train(uint64_t* d_boards, uint64_t* d_after, uint32_t* d_scores, uint32_t* d_lengths,
                                   int64_t n, const G2048TuplePlacement* h_placements, int n_placements,
                                   const G2048TupleStages* h_stages, float* d_weights, int64_t n_weights, float alpha,
                                   float lambda, int horizon, uint64_t* d_hist_after, float* d_hist_delta,
                                   uint32_t* d_start_stage, uint64_t* d_stage_pool, const uint32_t* d_subs,
                                   int64_t n_steps, int rng_mode, void* d_scratch, uint64_t* d_stats, void* stream);
int g2048_ntuple_carousel_tc_train(uint64_t* d_boards, uint64_t* d_after, uint32_t* d_scores, uint32_t* d_lengths,
                                   int64_t n, const G2048TuplePlacement* h_placements, int n_placements,
                                   const G2048TupleStages* h_stages, float* d_weights, int64_t n_weights,
                                   double* d_err_sum, double* d_abs_err_sum, float alpha, float lambda, int horizon,
                                   uint64_t* d_hist_after, float* d_hist_delta, uint32_t* d_start_stage,
                                   uint64_t* d_stage_pool, const uint32_t* d_subs, int64_t n_steps, int rng_mode,
                                   void* d_scratch, uint64_t* d_stats, void* stream);

/* Host-buffer form of the same call (the reference-facing entry: run_actions_max_tile's inner
 * run).  seed -> jax.random.key(seed); h_key_io (2 words, may be NULL) overrides the seed with an
 * explicit chain key and receives the key the reference's runner would hold afterwards.
 * h_* outputs may be NULL.  Copies H2D/D2H and synchronises.  A result array in pinned (page-locked, mapped) host
 * memory is written by the kernel itself while the batch runs; pageable arrays are filled by staged copies after it. */
int g2048_play_host(int policy, uint64_t seed, uint32_t* h_key_io, int64_t batch_global, int64_t env_lo, int64_t n,
                    int rng_mode, uint64_t* h_final_boards, uint32_t* h_lengths, uint32_t* h_scores,
                    uint64_t* h_stats);

/* g2048_play_host with the per-env results as one G2048EpisodeResult per env (h_results: n records, may be NULL).
 * In pinned host memory the records are written by the kernel as episodes end -- one 16-byte PCIe write per episode
 * instead of three small ones, which is what keeps eight GPUs behind shared PCIe uplinks from slowing each other. */
int g2048_play_host_packed(int policy, uint64_t seed, uint32_t* h_key_io, int64_t batch_global, int64_t env_lo, int64_t n,
                           int rng_mode, G2048EpisodeResult* h_results, uint64_t* h_stats);

/* Lock-step recorded rollout: `n_steps` loop steps of src/runs/batch_runner.py:117-136 for
 * act_randomly / act_drul in one kernel, state kept in registers in between.
 * Records are time-major (row t_local of each array has n entries):
 *   d_rec_boards uint64  pre-step board            (observation stored at :121,130)
 *   d_rec_meta   uint8   bits 0-1 action, 2-5 pre-step legal mask, 6 post-step done
 *   d_rec_rewards float32 post-step reward; d_rec_log_probs float32 (random only, else NULL)
 * d_subs points at the act sub key of the first of these steps (pairs act, step).
 * d_counters uint64[4] accumulated: [0] envs that terminated in this call, [1] max over envs of
 * (first-done loop step + 1) (atomicMax), [2] env-steps of live envs, [3] sum of rewards > 0.
 * t0 = loop step index of the first step (for [1]). */
int g2048_rollout_steps(int policy, uint64_t* d_boards, uint8_t* d_status, const uint32_t* d_subs, int64_t n_steps,
                        int64_t t0, int64_t batch_global, int64_t env_lo, int64_t n, int rng_mode,
                        uint64_t* d_rec_boards, uint8_t* d_rec_meta, float* d_rec_rewards, float* d_rec_log_probs,
                        uint64_t* d_counters, void* stream);
/* The same steps for a compact list of live envs (local indices, int64): an env that finishes leaves the loop and
 * the record slots of the steps after its end are not written, so the work is proportional to the live env-steps
 * instead of (loop steps) x (batch size).  Envs not listed are not touched. */
int g2048_rollout_steps_live(int policy, uint64_t* d_boards, uint8_t* d_status, const uint32_t* d_subs, int64_t n_steps,
                             int64_t t0, int64_t batch_global, int64_t env_lo, int64_t n, int rng_mode,
                             const int64_t* d_env_ids, int64_t n_live, uint64_t* d_rec_boards, uint8_t* d_rec_meta,
                             float* d_rec_rewards, float* d_rec_log_probs, uint64_t* d_counters, void* stream);

/* State of m listed envs (d_env_ids: GLOBAL env indices, int64) of the run BatchRunner(seed).run_*(batch_global) after
 * d_steps[i] loop steps of the built-in policy (d_subs as for g2048_play; each env needs 1 + 2 * d_steps[i] <= n_subs sub
 * keys).  One thread per listed env; meant for a handful of envs -- e.g. the board an env held BEFORE its last step,
 * which is what the reference's run_actions_max_tile reads for the envs that live until the last loop step
 * (src/runs/run_actions_max_tile.py:61-64 with src/runs/batch_runner.py:121,130).  d_status may be NULL. */
int g2048_replay_envs(int policy, const uint32_t* d_subs, int64_t n_subs, int64_t batch_global, const int64_t* d_env_ids,
                      const uint32_t* d_steps, int64_t m, int rng_mode, uint64_t* d_boards, uint8_t* d_status, void* stream);

/* ---- policy-logit sampling fused with the step and the rollout-buffer write
 * (src/ppo/torch_action_wrapper.py:84-102 + src/ppo/ppo_agent.py:117-121 + env.step + the
 * bookkeeping of src/runs/batch_runner.py:130-136).  One loop step:
 *   logits (n,4) f32 straight from the network; if use_mask: logits - 1e8*(1-mask);
 *   clip to >= -FLT_MAX; action = categorical(split(*d_sub_act,B)[e], logits) or argmax;
 *   log_prob = logits[a] - logsumexp(logits); step with split(*d_sub_step,B)[e];
 *   record row: pre-step board, meta, reward, log_prob, value (copied from d_values, may be NULL).
 * auto_reset != 0: a finished env is re-initialised with init(split(step_key)[1]) after the step
 * (pgx.experimental.auto_reset semantics: done/reward of the finishing step are kept). */
int g2048_policy_step(uint64_t* d_boards, uint8_t* d_status, const float* d_logits, const float* d_values,
                      int use_mask, int sample, int auto_reset, const uint32_t* d_sub_act, const uint32_t* d_sub_step,
                      int64_t batch_global, int64_t env_lo, int64_t n, int rng_mode, uint64_t* d_rec_boards,
                      uint8_t* d_rec_meta, float* d_rec_rewards, float* d_rec_log_probs, float* d_rec_values,
                      int32_t* d_actions_out, void* stream);

/* The same step with the step number read from device memory, so that ONE captured CUDA graph (observation ->
 * network forward -> this kernel -> g2048_counter_add) can be replayed for every step of a rollout (SURVEY 8f
 * rank 3).  t = *d_step_index; d_subs points at the chunk's first act sub key in the layout g2048_chain_advance
 * writes (act key of step t at words [4t, 4t+2), step key at [4t+2, 4t+4)); the record pointers are the chunk's
 * bases and slot t*n is written. */
int g2048_policy_step_at(uint64_t* d_boards, uint8_t* d_status, const float* d_logits, const float* d_values,
                         int use_mask, int sample, int auto_reset, const uint32_t* d_subs,
                         const int32_t* d_step_index, int64_t batch_global, int64_t env_lo, int64_t n, int rng_mode,
                         uint64_t* d_rec_boards, uint8_t* d_rec_meta, float* d_rec_rewards, float* d_rec_log_probs,
                         float* d_rec_values, int32_t* d_actions_out, void* stream);

/* The same step for a COMPACT list of live envs (what the reference's loop would not need to feed to the network:
 * finished envs only repeat their frozen state, src/runs/batch_runner.py:117-136).  Row i < n_live of d_logits /
 * d_values belongs to env d_env_ids[i] (local index in [0, n)); state, RNG counter and record slot are the env's own,
 * so the live envs' trajectories do not depend on who else is still alive.  Records of envs not listed stay as
 * they are. */
int g2048_policy_step_live(uint64_t* d_boards, uint8_t* d_status, const float* d_logits, const float* d_values,
                           int use_mask, int sample, int auto_reset, const uint32_t* d_sub_act, const uint32_t* d_sub_step,
                           const int64_t* d_env_ids, int64_t n_live, int64_t batch_global, int64_t env_lo, int64_t n,
                           int rng_mode, uint64_t* d_rec_boards, uint8_t* d_rec_meta, float* d_rec_rewards,
                           float* d_rec_log_probs, float* d_rec_values, int32_t* d_actions_out, void* stream);

/* One launch per loop step of the network-policy rollout: g2048_policy_step_at for step t = *d_step_index (NULL: t = 0,
 * d_subs then points at this step's act sub key) FUSED with g2048_expand_obs of the stepped boards -- d_obs_next
 * (n,16,31) in obs_dtype (G2048_OBS_*) receives the observation of the NEXT forward pass, written from registers: the
 * new boards are handed from lane to lane by shuffles and go through the same shared-memory image ring and bulk stores
 * as g2048_expand_obs.  Same records, state and draws as g2048_policy_step_at.  d_counters (uint64[2], may be NULL,
 * ACCUMULATED): [0] envs that terminated on this step, [1] sum of the rewards > 0 -- so the host can test "all done"
 * without a reduction kernel.  advance_step != 0 (with d_step_index): the kernel adds 1 to *d_step_index once all its
 * CTAs are done, so a captured graph of {network forward, this launch} can be replayed step after step with nothing
 * else in it (one such launch at a time per device: the CTA ticket is a library global). */
int g2048_policy_step_obs(uint64_t* d_boards, uint8_t* d_status, const float* d_logits, const float* d_values, int use_mask,
                          int sample, int auto_reset, const uint32_t* d_subs, int32_t* d_step_index, int advance_step,
                          int64_t batch_global, int64_t env_lo, int64_t n, int rng_mode, uint64_t* d_rec_boards,
                          uint8_t* d_rec_meta, float* d_rec_rewards, float* d_rec_log_probs, float* d_rec_values,
                          int32_t* d_actions_out, int obs_dtype, void* d_obs_next, uint64_t* d_counters, void* stream);

/* *d_counter += delta on the stream (one thread): advances the device-resident step number between replays. */
int g2048_counter_add(int32_t* d_counter, int32_t delta, void* stream);

/* Only the sampling part (A6/A7), for parity tests and for callers that step separately. */
int g2048_sample_logits(const float* d_logits, const uint8_t* d_status, int use_mask, int sample,
                        const uint32_t* d_sub_act, int64_t batch_global, int64_t env_lo, int64_t n, int rng_mode,
                        int32_t* d_actions, float* d_log_probs, float* d_entropy, void* stream);

/* log_prob / entropy of GIVEN actions under (masked) logits: PPOAgent.evaluate_actions'
 * Categorical part (src/ppo/ppo_agent.py:182-189). */
int g2048_evaluate_logits(const float* d_logits, const uint8_t* d_mask_bits, int use_mask, const int32_t* d_actions,
                          int64_t n, float* d_log_probs, float* d_entropy, void* stream);

/* ---- observation / record materialisation (HBM-bound) */

/* One-hot observation of n boards: out[i, cell, c] = (exponent(cell) == c), (n,16,31) = pgx
 * observe() flattened as src/runs/run_actions_max_tile.py:61 and RolloutBuffer do.  dtype = G2048_OBS_*.
 * If row_stride_boards > 0 the boards are read as a (rows, n_cols) time-major record matrix and
 * written env-major: out index = col * rows + row (the (B,T,...) stacking of batch_runner.py:138). */
int g2048_expand_obs(const uint64_t* d_boards, int64_t n, int dtype, void* d_out, int64_t rows, int64_t n_cols,
                     void* stream);

/* d_out[i] = one-hot observation of d_boards[d_indices[i]], i < m (int64 indices) */
int g2048_expand_obs_gather(const uint64_t* d_boards, const int64_t* d_indices, int64_t m, int dtype, void* d_out,
                            void* stream);

/* Inverse of g2048_expand_obs: argmax over the 31 channels of every cell (the
 * `observations.argmax(-1)` of src/runs/run_actions_max_tile.py:61-63).  dtype BOOL or F32. */
int g2048_pack_obs(const void* d_obs, int dtype, int64_t n, uint64_t* d_boards, void* stream);

/* status byte -> pgx State.legal_action_mask (n,4) uint8 and State.terminated (n) uint8 */
int g2048_unpack_status(const uint8_t* d_status, int64_t n, uint8_t* d_masks, uint8_t* d_terminated, void* stream);

/* Unpack time-major (T,B) record rows into the reference's env-major (B,T) arrays
 * (src/runs/batch_runner.py:138-144): actions int32, masks uint8 (B,T,4), terminations uint8,
 * rewards / log_probs / values float32 transposed.  Any output may be NULL. */
int g2048_unpack_records(const uint8_t* d_rec_meta, const float* d_rec_rewards, const float* d_rec_log_probs,
                         const float* d_rec_values, int64_t t_steps, int64_t n, int32_t* d_actions, uint8_t* d_masks,
                         uint8_t* d_terminations, float* d_rewards, float* d_log_probs, float* d_values,
                         void* stream);

/* RolloutBuffer.store_batch (src/ppo/rollout_buffer.py:164-187): per-env kept length
 * (first done + 1, or 0 if the env never terminated in t_steps) from the time-major meta. */
int g2048_episode_lengths(const uint8_t* d_rec_meta, int64_t t_steps, int64_t n, uint32_t* d_lengths, void* stream);

/* exclusive prefix sum of n uint32 into int64 offsets (n+1 entries, last = total) */
int g2048_exclusive_scan(const uint32_t* d_in, int64_t n, int64_t* d_out, void* stream);

/* Ragged env-major compaction of time-major records into flat packed arrays (what
 * store_batch + get_buffer_data produce, src/ppo/rollout_buffer.py:164-206, minus the one-hot
 * expansion): flat index = d_offsets[e] + t for t < d_lengths[e].  out_base is added to every
 * flat index (appending after earlier batches).  Outputs may be NULL. */
int g2048_compact_records(const uint64_t* d_rec_boards, const uint8_t* d_rec_meta, const float* d_rec_rewards,
                          const float* d_rec_log_probs, const float* d_rec_values, int64_t t_steps, int64_t n,
                          const uint32_t* d_lengths, const int64_t* d_offsets, int64_t out_base,
                          uint64_t* d_boards, uint8_t* d_meta, float* d_rewards, float* d_log_probs, float* d_values,
                          void* stream);

/* RolloutBuffer.store_batch for arbitrary per-step rows (src/ppo/rollout_buffer.py:128-187 does not depend on the
 * observation or action shape; g2048_compact_records is the form for packed 2048 records).
 * g2048_first_done_rows: d_terminations (n_envs, t_steps) uint8 env-major -> d_lengths[e] = index of the first nonzero
 * flag + 1, or 0 when the env never terminates (:168-175: such an env stores nothing).
 * g2048_compact_rows: d_src (n_envs, t_steps, row_bytes) env-major; the rows t < d_lengths[e] of env e are copied to
 * d_dst + (out_base + d_offsets[e]) * row_bytes (d_offsets = exclusive scan of d_lengths).  One call per field. */
int g2048_first_done_rows(const uint8_t* d_terminations, int64_t n_envs, int64_t t_steps, uint32_t* d_lengths, void* stream);
int g2048_compact_rows(const void* d_src, int64_t n_envs, int64_t t_steps, int64_t row_bytes, const uint32_t* d_lengths,
                       const int64_t* d_offsets, int64_t out_base, void* d_dst, void* stream);

/* flat packed meta -> reference-format columns: actions one-hot f32 (N,4), masks uint8 (N,4),
 * terminations uint8 (N) (src/ppo/ppo_trainer.py:197-202, rollout_buffer.py:199-205) */
int g2048_unpack_flat_meta(const uint8_t* d_meta, int64_t n, float* d_actions_onehot, uint8_t* d_masks,
                           uint8_t* d_terminations, void* stream);

/* Minibatch gather from the flat packed buffer (SURVEY 8f rank 1; replaces PPODataset.__getitem__ and the
 * DataLoader's collation, src/ppo/data_loader.py:132-166,217-223): for i < m, s = d_indices[i]:
 *   d_obs[i]  = one-hot (16,31) of d_boards[s] in obs_dtype (G2048_OBS_*), 16-byte aligned, may be NULL
 *   d_actions[i] int64 action index, d_masks[i] uint8 (4), d_old_log_probs / d_old_values /
 *   d_out_adv / d_out_ret float32 gathered from the corresponding source arrays, d_out_boards[i] = d_boards[s]
 *   (for callers that embed the bitboards directly instead of reading observations).  Any output may be NULL.
 *   One launch either way: the observation kernel gathers the scalars itself; without d_obs a small kernel does. */
int g2048_gather_minibatch(const int64_t* d_indices, int64_t m, const uint64_t* d_boards, const uint8_t* d_meta,
                           const float* d_log_probs, const float* d_values, const float* d_adv, const float* d_ret,
                           int obs_dtype, void* d_obs, int64_t* d_actions, uint8_t* d_masks, float* d_old_log_probs,
                           float* d_old_values, float* d_out_adv, float* d_out_ret, uint64_t* d_out_boards, void* stream);

/* Sample records: the training view of the flat buffer with every field of a sample in ONE 32-byte sector, so that a
 * random minibatch costs one sector per sample instead of one per source array (six).  g2048_pack_samples builds them
 * in one pass that also applies the global normalisation of src/ppo/data_loader.py:61-67 to advantages and returns
 * (d_moments as written by g2048_gae_flat; NULL = store d_adv / d_ret as they are), replacing the two g2048_normalize
 * passes; g2048_gather_samples is g2048_gather_minibatch reading them.  d_rewards / d_log_probs / d_values / d_adv /
 * d_ret may be NULL (stored as 0). */
typedef struct G2048SampleRecord {
    uint64_t board;   /* pre-step bitboard */
    uint32_t meta;    /* low byte: action | legal mask << 2 | done << 6 */
    float reward;
    float log_prob, value, advantage, ret; /* second 16-byte half */
} G2048SampleRecord;
int g2048_pack_samples(const uint64_t* d_boards, const uint8_t* d_meta, const float* d_rewards, const float* d_log_probs,
                       const float* d_values, const float* d_adv, const float* d_ret, int64_t n, const double* d_moments,
                       G2048SampleRecord* d_records, void* stream);
int g2048_gather_samples(const int64_t* d_indices, int64_t m, const G2048SampleRecord* d_records, int obs_dtype, void* d_obs,
                         int64_t* d_actions, uint8_t* d_masks, float* d_old_log_probs, float* d_old_values, float* d_out_adv,
                         float* d_out_ret, uint64_t* d_out_boards, void* stream);

/* Random subset / shuffle of buffer positions (replaces torch.randperm(total_length)[:length] and the DataLoader's
 * shuffle, src/ppo/data_loader.py:73-101,217-223): d_out[i] = P(first + i) for i < m, where P is a pseudo-random
 * bijection of [0, n) selected by the key -- a 4-round Feistel network over 2h bits (4^h >= n) whose round function
 * is Threefry-2x32(key; (right half, round)), restricted to [0, n) by cycle walking.  Distinct inputs give distinct
 * positions, so first = 0, m = n is a full shuffle and m < n a subset without replacement, in O(m) work.
 * first + m <= n <= 2^62. */
int g2048_random_subset(uint32_t key0, uint32_t key1, int64_t n, int64_t first, int64_t m, int64_t* d_out, void* stream);

/* ---- packed boards -> input embedding (SURVEY 8f rank 1; src/ppo/ppo_agent.py:60,108) */

/* out[i, c, :] = table[exponent of cell c of board i, :] -- what Linear(31 -> d_model, bias=False) returns for the
 * one-hot observation of the board, without the observation.  d_table: (31, d_model) row-major = the Linear's
 * weight transposed, in `dtype` (G2048_OBS_F32 or G2048_OBS_BF16); d_out: (n, 16, d_model) in `dtype`.
 * d_indices (int64, may be NULL): row i uses d_boards[d_indices[i]] (minibatch gather).  d_model * itemsize must
 * be a multiple of 16 and the table must fit in shared memory (31 * d_model * itemsize <= 200 KiB).
 * Two kernels: _bulk issues one shared->global bulk copy (cp.async.bulk) per cell straight from the table,
 * _plain copies a row per warp with 16-byte stores; g2048_embed_boards is the bulk form (as fast with a warm L2,
 * 25-45 % faster once L2 holds another kernel's dirty lines -- measured on B200); _plain stays for A/B runs. */
int g2048_embed_boards(const uint64_t* d_boards, int64_t n, const int64_t* d_indices, const void* d_table,
                       int d_model, int dtype, void* d_out, void* stream);
int g2048_embed_boards_bulk(const uint64_t* d_boards, int64_t n, const int64_t* d_indices, const void* d_table,
                            int d_model, int dtype, void* d_out, void* stream);
int g2048_embed_boards_plain(const uint64_t* d_boards, int64_t n, const int64_t* d_indices, const void* d_table,
                             int d_model, int dtype, void* d_out, void* stream);

/* Gradient of the table: d_grad_table[r, :] (float32 (31, d_model), overwritten) = sum over cells whose exponent
 * is r of d_grad_out[cell, :] (d_grad_out: (n, 16, d_model) in `dtype`); rows 16..30 are zero.  Deterministic:
 * per-CTA partial tables in d_scratch (g2048_embed_grad_scratch_bytes(n, d_model, dtype) bytes, 16-byte aligned,
 * need not be zeroed) are added in a fixed order.  The scratch size query returns -1 for an unsupported d_model. */
int64_t g2048_embed_grad_scratch_bytes(int64_t n, int d_model, int dtype);
int g2048_embed_boards_grad(const uint64_t* d_boards, int64_t n, const int64_t* d_indices, const void* d_grad_out,
                            int d_model, int dtype, float* d_grad_table, void* d_scratch, void* stream);

/* ---- GAE (src/ppo/data_loader.py:103-130) and normalisation (:61-67) */

/* Flat buffer, reverse segmented scan: if done[t]: last_v = last_gae = 0;
 * delta = r[t] + gamma*last_v - V[t]; gae = delta + gamma*lambda*gae; adv[t]=gae; ret[t]=gae+V[t].
 * Single pass over the buffer in tiles (one lane per episode, decoupled look-back of depth one across
 * tiles); bit-identical to the reference loop.  d_scan_state: scratch of
 * g2048_gae_flat_scratch_bytes(n) bytes, zeroed by the caller.  d_moments (double[6], may be NULL,
 * ACCUMULATED): [0] n, [1] sum adv, [2] sum adv^2, [3] sum ret, [4] sum ret^2, [5] unused. */
int64_t g2048_gae_flat_scratch_bytes(int64_t n);
int g2048_gae_flat(const float* d_rewards, const float* d_values, const uint8_t* d_dones, int64_t n, double gamma,
                   double lambda_gae, float* d_adv, float* d_ret, void* d_scan_state, double* d_moments, void* stream);

/* The two current kernels behind g2048_gae_flat (same arguments, same scratch, bit-identical outputs):
 *   _tiled      one 6 144-step tile per CTA, phases one after the other; used below 2^23 steps
 *   _pipelined  persistent CTAs holding two 8 192-step tiles: walker warps on tile i while streamer warps store tile
 *               i-1 and load tile i+1; used from 2^23 steps on
 * (the first-generation kernel lives in the tests' own build of the library, tests/legacy/g2048_legacy.h). */
int g2048_gae_flat_tiled(const float* d_rewards, const float* d_values, const uint8_t* d_dones, int64_t n, double gamma,
                         double lambda_gae, float* d_adv, float* d_ret, void* d_scan_state, double* d_moments,
                         void* stream);
int g2048_gae_flat_pipelined(const float* d_rewards, const float* d_values, const uint8_t* d_dones, int64_t n,
                             double gamma, double lambda_gae, float* d_adv, float* d_ret, void* d_scan_state,
                             double* d_moments, void* stream);

/* g2048_gae_flat as a segmented affine REVERSE SCAN (north_star's "warp shuffles handle the reverse-scan GAE"): same
 * arguments and moments, its own scratch (g2048_gae_scan_scratch_bytes(n) bytes, 16-byte aligned, need not be zeroed).
 * The recurrence is re-associated (thread / warp-shuffle / CTA scan of 2 048-step tiles, one contiguous range of tiles
 * per persistent CTA with the carry in registers, a second small launch for the range boundaries), so the
 * results agree with the reference loop within the 1e-5 relative tolerance north_star states for GAE, NOT bit for bit --
 * opt-in; g2048_gae_flat stays the bit-identical default.  A pure stream: no lane ever walks an episode. */
int64_t g2048_gae_scan_scratch_bytes(int64_t n);
int g2048_gae_flat_scan(const float* d_rewards, const float* d_values, const uint8_t* d_dones, int64_t n, double gamma,
                        double lambda_gae, float* d_adv, float* d_ret, void* d_scan_state, double* d_moments, void* stream);

/* Time-major (T,B) buffer, one lane per env, exactly the reference's operation order per env;
 * d_bootstrap (n) float32 or NULL is V(s_T) for envs whose last step is not done (fixed-horizon
 * rollouts with auto-reset; the reference itself never bootstraps). */
int g2048_gae_time_major(const float* d_rewards, const float* d_values, const uint8_t* d_rec_meta, int64_t t_steps,
                         int64_t n, const float* d_bootstrap, double gamma, double lambda_gae, float* d_adv,
                         float* d_ret, double* d_moments, void* stream);

/* x = (x - mean) / (std + 1e-8) in place with mean / unbiased std from the moments block
 * (sum at d_moments[which], sum of squares at [which+1], count at [0]); which = 1 (adv) or 3 (ret). */
int g2048_normalize(float* d_x, int64_t n, const double* d_moments, int which, void* stream);

/* Host-buffer GAE + normalisation (the PPODataset.__init__ path) */
int g2048_gae_host(const float* h_rewards, const float* h_values, const uint8_t* h_dones, int64_t n, double gamma,
                   double lambda_gae, int normalize, float* h_adv, float* h_ret);

/* The *_host entry points keep, per calling thread, a stream, a grow-only device buffer and 2 x 16 MiB of pinned staging
 * memory between calls (re-created when the thread switches device).  This frees the calling thread's; a thread that
 * used *_host entry points should call it before it ends. */
int g2048_release_host_workspace(void);

/* ---- statistics (src/stats/running_stats_vec.py:55-87) */

/* per feature row of x (F, n) float64: count, mean, population variance -> d_out (F,3) double */
int g2048_row_moments(const double* d_x, int64_t n_features, int64_t n, double* d_out, void* stream);

/* ---- measurement helpers */

/* Integer-issue roofline probe: every thread runs `iters` dependent-chain rounds of the Threefry
 * instruction mix (ADD / SHF.L.W / LOP3) on `chains` independent chains; writes one word per
 * thread so nothing is optimised away.  Instructions executed = blocks*threads*iters*chains*3. */
int g2048_int_peak_probe(int blocks, int threads, int iters, uint32_t* d_sink, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* G2048_H_ */
