// Persistent play-to-termination kernel, third generation: row tables in shared memory.
//
// ncu on the SWAR kernel (g2048_play.cu): ALU pipe 95 % busy, ~870 ALU instructions per env-step of
// which only 400 are Threefry (the ROTATE and XOR of each round; the ADD goes to the FMA pipe) -- the
// rest is board logic on 64-bit words, where every shift costs two ALU instructions.  This kernel
// moves that logic off the ALU pipe:
//   * the slide/merge of a row is ONE 16-bit load from a 65 536-entry table held in shared memory
//     (128 KiB, built once per process, copied per CTA), as BASELINE.json's north_star suggests;
//   * the exact legal-action mask is 8 byte loads from a second table (64 KiB): "this row can move
//     left / right", looked up for the four rows of the board and the four rows of its transpose;
//   * the lane keeps the board AND its transpose in registers, so a vertical move is a horizontal
//     move on the transpose and every step pays exactly one transpose (8 ALU-pipe instructions).
// Shared-memory loads issue on the LSU pipe, which the kernel otherwise leaves idle.
// 192 KiB of tables -> one CTA per SM, of 768 threads (512 for small batches: play3_block_threads).  Same lane
// scheduling, init-as-two-iterations trick, score-from-potential and results as g2048_play.cu (bit-identical; tested).
#include "g2048_play3.cuh"

namespace g2048 {

#ifndef G2048_PLAY3_TAIL_STEPS
#define G2048_PLAY3_TAIL_STEPS 8
#endif
#ifndef G2048_PLAY3_TAIL
// 1: tail compaction (play3_tail below).  Off in the shipped build: it shortens the fixed cost of a launch (2^18 envs:
// 1.53 -> 1.47 ms) but its presence costs the main loop 0.9 % at 2^24 envs (69.84 -> 70.44 ms) and the recording form
// more (DRUL, 2^18 envs: 1.91 -> 2.07 ms); the headline workload is the large batch.  A/B: tools/ab_variants.py.
#define G2048_PLAY3_TAIL 0
#endif
#ifndef G2048_PLAY3_TAIL_REC
// 1: tail compaction in the RECORDING form only, inlined (that form runs at C4-like sizes, 3-4 episodes per lane, where
// the drain is a third of the launch): 2^18 envs, random policy 1.64 -> 1.55 ms, DRUL unchanged, and the plain form's code is
// not touched (A/B on one box, profiles/r02_ab_variants.jsonl)
#define G2048_PLAY3_TAIL_REC 1
#endif

[[maybe_unused]] constexpr int PLAY3_TAIL_STEPS = G2048_PLAY3_TAIL_STEPS;  // steps between two compactions of the CTA's live envs in the tail
// what moves with an env when the tail compaction hands it to another lane (32 bytes)
struct TailEntry {
    unsigned long long board;
    unsigned long long slot;  // recording: the env's next arena slot (it keeps writing into its first lane's region)
    uint32_t e, t, fours, flags;  // flags: bits 0-1 phase, bit 2 seen15
};
constexpr int PLAY3_STATS_BYTES = G2048_PLAY_STATS_WORDS * 8;
constexpr int PLAY3_CTL_BYTES = 16;  // tail flag, two alternating live-env counters
// the shared memory of a CTA of THREADS threads: row tables, statistics, tail control, tail pool, spawn masks, action table
template <int THREADS>
struct Play3Smem {
    static constexpr int POOL_BYTES = THREADS * (int)sizeof(TailEntry);
    static constexpr int SPAWN_OFFSET = PLAY3_TABLE_BYTES + PLAY3_STATS_BYTES + PLAY3_CTL_BYTES + POOL_BYTES;
    static constexpr int ACT_OFFSET = SPAWN_OFFSET + PLAY3_SPAWN_BYTES;
    static constexpr int BYTES = ACT_OFFSET + PLAY3_ACT_BYTES;
};

__device__ __forceinline__ void play3_epilogue(Play3Lane& L, const Play3Ctx& c) {
    if (L.pk_has) {
        const uint32_t score = board_potential(L.pk_board) - 4u * L.pk_fours;
        if (c.final_boards) c.final_boards[L.pk_e] = L.pk_board;
        if (c.lengths) c.lengths[L.pk_e] = L.pk_t;
        if (c.scores) c.scores[L.pk_e] = score;
        if (c.results) c.results[L.pk_e] = make_uint4((uint32_t)L.pk_board, (uint32_t)(L.pk_board >> 32), L.pk_t, score);  // G2048EpisodeResult
        const uint32_t me = max_exponent(L.pk_board);
        const unsigned long long tile = 1ull << me;
        L.st_episodes += 1;
        L.st_steps += L.pk_t;
        L.st_score += score;
        L.st_cut += L.pk_cut ? 1u : 0u;
        L.st_ovf += (L.pk_seen15 || has_max_nibble(L.pk_board)) ? 1u : 0u;
        L.st_longest = max(L.st_longest, L.pk_t);
        L.st_tile += tile;
        L.st_tile2 += tile * tile;
        atomicAdd(&c.s_stats[16 + me], 1ull);
        L.pk_has = false;
    }
}

// park what the lanes that just finished still hold (call converged)
__device__ __forceinline__ void play3_park(Play3Lane& L, const Play3Ctx& c) {
    const unsigned fresh = __ballot_sync(0xFFFFFFFFu, L.fin_live);
    if (fresh) {
        const unsigned parked = __ballot_sync(0xFFFFFFFFu, L.pk_has);
        if ((fresh & parked) != 0u || __popc(fresh | parked) >= PLAY3_EPILOGUE_BATCH) play3_epilogue(L, c);
        if (L.fin_live) {
            L.pk_board = L.board;
            L.pk_t = L.t;
            L.pk_fours = L.fours;
            L.pk_e = L.e;
            L.pk_cut = L.fin_cut;
            L.pk_seen15 = L.seen15;
            L.pk_has = true;
            L.fin_live = false;
        }
    }
}


// Tail of the launch.  Once the queue is empty no lane gets a new env and the warps thin out: a warp with one live lane
// costs as many issue slots per step as a full one.  The CTA therefore plays the rest in rounds of PLAY3_TAIL_STEPS
// steps with a CTA-wide compaction in between: the live envs move through shared memory into the lowest lanes of the
// CTA, warps without envs only wait at the barrier, and the cost of a step follows the number of live envs.  The fixed
// cost of a launch (what does not shrink with the batch) drops from 0.49 to 0.37 ms: 2^18 envs (C4) 1.54 -> 1.44 ms
// inlined, 1.47 ms out of line.  Out of line because inlined the same source cost the main loop 2 % (2^24 envs:
// 69.8 -> 71.3 ms; A/B on one box, tools/ab_variants.py); see G2048_PLAY3_TAIL above for why it is still off.
#if G2048_PLAY3_TAIL_REC
#define G2048_TAIL_INLINE __forceinline__
#else
#define G2048_TAIL_INLINE __noinline__
#endif
template <int MODE, int POLICY, bool REC>
__device__ G2048_TAIL_INLINE void play3_tail(Play3Lane& lane_state, const Play3Ctx& c, unsigned* s_tail_cnt, TailEntry* s_pool) {
    Play3Lane L = lane_state;  // work on a copy in registers: stores through the context's pointers cannot alias it
    const unsigned lane = threadIdx.x & 31u;
    unsigned round = 0;
    while (true) {
        play3_park(L, c);
        // ---- compaction: live envs -> pool -> lanes 0 .. total-1 of the CTA ----------------------------------------
        unsigned* cnt = &s_tail_cnt[round & 1u];
        const unsigned livemask = __ballot_sync(0xFFFFFFFFu, L.phase != PHASE_NONE);
        unsigned base = 0;
        if (livemask) {
            if (lane == 0) base = atomicAdd(cnt, (unsigned)__popc(livemask));
            base = __shfl_sync(0xFFFFFFFFu, base, 0);
        }
        race_jitter();
        if (L.phase != PHASE_NONE) {
            const unsigned at = base + (unsigned)__popc(livemask & ((1u << lane) - 1u));
            s_pool[at] = TailEntry{L.board, L.slot, L.e, L.t, L.fours, L.phase | (L.seen15 ? 4u : 0u)};
        }
        __syncthreads();
        const unsigned total = *(volatile unsigned*)cnt;
        if (threadIdx.x == 0) s_tail_cnt[(round + 1u) & 1u] = 0u;  // next round's counter: untouched until after the barrier below
        if (total == 0u) break;  // uniform over the CTA
        race_jitter();
        if (threadIdx.x < total) {
            const TailEntry en = s_pool[threadIdx.x];
            L.board = en.board;
            L.slot = en.slot;
            L.e = en.e;
            L.t = en.t;
            L.fours = en.fours;
            L.phase = en.flags & 3u;
            L.seen15 = (en.flags & 4u) != 0u;
            L.boardT = transpose_board(L.board);
            L.lm = play3_legal(c.s_flags, L.board, L.boardT);
        } else {
            L.phase = PHASE_NONE;
        }
        __syncthreads();  // every entry has been read before the next round writes the pool
        ++round;
        for (int it = 0; it < PLAY3_TAIL_STEPS; ++it) {
            if (__ballot_sync(0xFFFFFFFFu, L.phase != PHASE_NONE) == 0u) break;  // nothing left in this warp: wait at the barrier
            if (L.phase != PHASE_NONE) play3_step<MODE, POLICY, REC>(L, c);
            if (__ballot_sync(0xFFFFFFFFu, L.fin_live)) play3_park(L, c);
        }
    }
    lane_state = L;
}

template <int MODE, int POLICY, bool REC, int THREADS>
__global__ void __launch_bounds__(THREADS, 1)
play3_kernel(const uint2* __restrict__ subs, int64_t n_subs, uint32_t batch_global, uint32_t env_lo, uint32_t n,
             unsigned long long* __restrict__ work, u64* __restrict__ final_boards, uint32_t* __restrict__ lengths,
             uint32_t* __restrict__ scores, unsigned long long* __restrict__ stats, uint4* __restrict__ results,
             const PlayRecordArena rec) {
    extern __shared__ __align__(16) uint8_t smem_raw[];
    unsigned long long* s_stats = reinterpret_cast<unsigned long long*>(smem_raw + PLAY3_TABLE_BYTES);
#if G2048_PLAY3_TAIL || G2048_PLAY3_TAIL_REC
    volatile unsigned* s_tail_flag = reinterpret_cast<volatile unsigned*>(smem_raw + PLAY3_TABLE_BYTES + PLAY3_STATS_BYTES);
    unsigned* s_tail_cnt = reinterpret_cast<unsigned*>(smem_raw + PLAY3_TABLE_BYTES + PLAY3_STATS_BYTES) + 1;  // [2]
    TailEntry* s_pool = reinterpret_cast<TailEntry*>(smem_raw + PLAY3_TABLE_BYTES + PLAY3_STATS_BYTES + PLAY3_CTL_BYTES);
#endif

    {
        play3_copy_row_tables<THREADS>(smem_raw);
        for (int i = threadIdx.x; i < G2048_PLAY_STATS_WORDS; i += THREADS) s_stats[i] = 0ull;
        if (threadIdx.x < 4) reinterpret_cast<unsigned*>(smem_raw + PLAY3_TABLE_BYTES + PLAY3_STATS_BYTES)[threadIdx.x] = 0u;
        // the spawn masks, as play3_fill_spawn_masks writes them (spelt out here: through the helper ptxas masks one
        // address differently, and this kernel's code is kept instruction for instruction)
        if (threadIdx.x < 16) {
            const unsigned cell = threadIdx.x, cellT = ((cell & 3u) << 2) | (cell >> 2);
            const u64 m = 1ull << (4 * cell), mT = 1ull << (4 * cellT);
            reinterpret_cast<uint4*>(smem_raw + Play3Smem<THREADS>::SPAWN_OFFSET)[cell] =
                make_uint4((uint32_t)m, (uint32_t)(m >> 32), (uint32_t)mT, (uint32_t)(mT >> 32));
        }
        play3_fill_act_table(reinterpret_cast<ActEntry*>(smem_raw + Play3Smem<THREADS>::ACT_OFFSET));
    }
    __syncthreads();

    const unsigned lane = threadIdx.x & 31u;
    Play3Ctx c;
    c.subs = subs;
    c.init_sub = subs[0];
    c.max_steps = (uint32_t)((n_subs - 1) / 2);
    c.batch_global = batch_global;
    c.env_lo = env_lo;
    c.s_left = reinterpret_cast<const uint16_t*>(smem_raw);
    c.s_flags = smem_raw + 65536 * 2;
    c.s_spawn = reinterpret_cast<const uint4*>(smem_raw + Play3Smem<THREADS>::SPAWN_OFFSET);
    c.s_act = reinterpret_cast<const ActEntry*>(smem_raw + Play3Smem<THREADS>::ACT_OFFSET);
    c.s_stats = s_stats;
    c.final_boards = final_boards;
    c.lengths = lengths;
    c.scores = scores;
    c.results = results;
    c.rec = rec;

    Play3Lane L = {};
    L.phase = PHASE_NONE;
    if (REC) {
        L.slot = ((unsigned long long)blockIdx.x * THREADS + threadIdx.x) * rec.cap;
        L.slot_end = L.slot + rec.cap;
    }
    bool exhausted = false;  // warp-uniform

    // ---- main phase: every lane that finishes an episode takes the next env of the queue at once ---------------------
    bool tail_seen = false;  // warp-uniform
    while (true) {
        const unsigned idle = __ballot_sync(0xFFFFFFFFu, L.phase == PHASE_NONE);
        // a recording lane takes a new env only while a whole episode still fits into its arena region
        const bool can_take = !REC || L.slot + (unsigned long long)c.max_steps + 1ull <= L.slot_end;
        const unsigned want = REC ? __ballot_sync(0xFFFFFFFFu, L.phase == PHASE_NONE && can_take) : idle;
        if (idle) {
            play3_park(L, c);
            if (!exhausted && want) {
                const int cnt = __popc(want);
                unsigned long long base = 0;
                race_jitter();
                if (lane == 0) base = atomicAdd(work, (unsigned long long)cnt);
                base = __shfl_sync(0xFFFFFFFFu, base, 0);
                if (base + (unsigned long long)cnt >= (unsigned long long)n) exhausted = true;
                if (L.phase == PHASE_NONE && (!REC || can_take)) {
                    const unsigned long long mine = base + (unsigned long long)__popc(want & ((1u << lane) - 1u));
                    if (mine < (unsigned long long)n) {
                        L.e = (uint32_t)mine;
                        L.board = 0ull;
                        L.boardT = 0ull;
                        L.lm = 0;
                        L.t = 0;
                        L.fours = 0;
                        L.seen15 = false;
                        L.phase = PHASE_INIT0;
                    }
                }
            }
            constexpr bool TAIL = G2048_PLAY3_TAIL || (G2048_PLAY3_TAIL_REC && REC);
            if (TAIL) {
#if G2048_PLAY3_TAIL || G2048_PLAY3_TAIL_REC
                // The queue is empty (or, recording, no idle lane of this warp can take an env any more): tell the CTA.
                if (exhausted || (REC && want == 0u && idle == 0xFFFFFFFFu)) {
                    *s_tail_flag = 1;
                    tail_seen = true;
                }
#endif
            } else {
                if (__ballot_sync(0xFFFFFFFFu, L.phase != PHASE_NONE) == 0u && (exhausted || want == 0u)) tail_seen = true;
            }
        }
#if G2048_PLAY3_TAIL || G2048_PLAY3_TAIL_REC
        // once any warp of the CTA has seen the queue empty, all of them (each looks at the flag once per iteration)
        // leave for the tail phase together
        if ((G2048_PLAY3_TAIL || REC) && *s_tail_flag) tail_seen = true;
#endif
        if (tail_seen) break;
        if (L.phase != PHASE_NONE) play3_step<MODE, POLICY, REC>(L, c);
    }
#if G2048_PLAY3_TAIL || G2048_PLAY3_TAIL_REC
    if (G2048_PLAY3_TAIL || REC) {
        Play3Lane handed = L;  // only this copy has its address taken: the main loop's state stays in registers
        play3_tail<MODE, POLICY, REC>(handed, c, s_tail_cnt, s_pool);
        L = handed;
    }
#endif
    play3_epilogue(L, c);  // whatever is still parked (a finished lane always passes a park, and is parked, before the loops end)

    atomicAdd(&s_stats[0], (unsigned long long)L.st_episodes);
    atomicAdd(&s_stats[1], L.st_steps);
    atomicAdd(&s_stats[2], L.st_score);
    atomicAdd(&s_stats[3], (unsigned long long)L.st_cut);
    atomicAdd(&s_stats[4], (unsigned long long)L.st_ovf);
    atomicMax(&s_stats[5], (unsigned long long)L.st_longest);
    atomicAdd(&s_stats[6], L.st_tile);
    atomicAdd(&s_stats[7], L.st_tile2);
    __syncthreads();
    for (int i = threadIdx.x; i < G2048_PLAY_STATS_WORDS; i += blockDim.x) {
        const unsigned long long v = s_stats[i];
        if (v) {
            if (i == 5) atomicMax(&stats[i], v);
            else atomicAdd(&stats[i], v);
        }
    }
}


__global__ void build_row_tables_kernel() {
    const uint32_t row = blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= 65536u) return;
    build_row_table_entry(row);
}

static int ensure_row_tables(cudaStream_t st) { return ensure_row_tables_with<build_row_tables_kernel>(st); }

__global__ void row_table_lookup_kernel(const uint16_t* __restrict__ rows, int64_t n, uint16_t* __restrict__ left,
                                        uint8_t* __restrict__ flags) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    left[i] = g_row_left[rows[i]];
    flags[i] = g_row_flags[rows[i]];
}

// CTAs (one per SM, persistent) and threads per CTA of a table-kernel launch over n envs; the recording form sizes its
// arena by them
struct Play3Shape {
    int64_t grid;
    int threads;
    int64_t lanes() const { return grid * threads; }
};
static Play3Shape play3_shape(int64_t n, int sms) {
    const int threads = play3_block_threads(n, sms);
    const int64_t needed = (n + threads - 1) / threads;
    return Play3Shape{needed < sms ? needed : sms, threads};
}

template <int MODE, int POLICY, bool REC, int THREADS>
static int launch_play3_with(int64_t grid, const uint32_t* d_subs, int64_t n_subs, int64_t batch_global, int64_t env_lo,
                             int64_t n, uint64_t* d_work, uint64_t* d_final_boards, uint32_t* d_lengths, uint32_t* d_scores,
                             uint64_t* d_stats, cudaStream_t st, void* d_results, PlayRecordArena rec) {
    static bool configured_on[64] = {false};
    bool* configured = device_once_flag(configured_on);
    if (!configured) return fail_arg("no CUDA device");
    if (!*configured) {
        const int rc = check_cuda(cudaFuncSetAttribute(play3_kernel<MODE, POLICY, REC, THREADS>,
                                                       cudaFuncAttributeMaxDynamicSharedMemorySize, Play3Smem<THREADS>::BYTES),
                                  "play: shared memory attribute");
        if (rc) return rc;
        *configured = true;
    }
    play3_kernel<MODE, POLICY, REC, THREADS><<<(unsigned)grid, THREADS, Play3Smem<THREADS>::BYTES, st>>>(
        (const uint2*)d_subs, n_subs, (uint32_t)batch_global, (uint32_t)env_lo, (uint32_t)n,
        (unsigned long long*)d_work, (u64*)d_final_boards, d_lengths, d_scores, (unsigned long long*)d_stats,
        (uint4*)d_results, rec);
    return check_cuda(cudaGetLastError(), "play");
}

template <int MODE, int POLICY, bool REC>
static int launch_play3(const uint32_t* d_subs, int64_t n_subs, int64_t batch_global, int64_t env_lo, int64_t n,
                        uint64_t* d_work, uint64_t* d_final_boards, uint32_t* d_lengths, uint32_t* d_scores,
                        uint64_t* d_stats, cudaStream_t st, void* d_results, PlayRecordArena rec = PlayRecordArena{}) {
    const int rc = ensure_row_tables(st);
    if (rc) return rc;
    const int sms = sm_count();
    if (sms <= 0) return fail_arg("play: no device");
    const Play3Shape shape = play3_shape(n, sms);
    if (shape.threads == PLAY3_THREADS)
        return launch_play3_with<MODE, POLICY, REC, PLAY3_THREADS>(shape.grid, d_subs, n_subs, batch_global, env_lo, n, d_work,
                                                                   d_final_boards, d_lengths, d_scores, d_stats, st, d_results, rec);
    return launch_play3_with<MODE, POLICY, REC, PLAY3_SMALL_THREADS>(shape.grid, d_subs, n_subs, batch_global, env_lo, n, d_work,
                                                                     d_final_boards, d_lengths, d_scores, d_stats, st, d_results, rec);
}

// the table kernel with every output form (d_results: one 16-byte G2048EpisodeResult per env, may be NULL)
int play_tables_impl(int policy, const uint32_t* d_subs, int64_t n_subs, int64_t batch_global, int64_t env_lo, int64_t n,
                     int rng_mode, uint64_t* d_work, uint64_t* d_final_boards, uint32_t* d_lengths, uint32_t* d_scores,
                     uint64_t* d_stats, void* d_results, void* stream) {
    G2048_REQUIRE(policy == G2048_POLICY_RANDOM || policy == G2048_POLICY_DRUL, "play: policy");
    G2048_REQUIRE(rng_mode == G2048_RNG_ORIGINAL || rng_mode == G2048_RNG_PARTITIONABLE, "play: rng_mode");
    G2048_REQUIRE(batch_global > 0 && batch_global <= 0x7FFFFFFFll && env_lo >= 0 && n >= 0 && env_lo + n <= batch_global,
                  "play: batch");
    G2048_REQUIRE(n_subs >= 3 && d_subs && d_work && d_stats, "play: pointers");
    G2048_REQUIRE(((uintptr_t)d_results & 15u) == 0, "play: results must be 16-byte aligned");
    if (n == 0) return G2048_OK;
    cudaStream_t st = (cudaStream_t)stream;
#define ARGS d_subs, n_subs, batch_global, env_lo, n, d_work, d_final_boards, d_lengths, d_scores, d_stats, st, d_results
    if (policy == G2048_POLICY_RANDOM) {
        if (rng_mode == G2048_RNG_PARTITIONABLE) return launch_play3<G2048_RNG_PARTITIONABLE, G2048_POLICY_RANDOM, false>(ARGS);
        return launch_play3<G2048_RNG_ORIGINAL, G2048_POLICY_RANDOM, false>(ARGS);
    }
    if (rng_mode == G2048_RNG_PARTITIONABLE) return launch_play3<G2048_RNG_PARTITIONABLE, G2048_POLICY_DRUL, false>(ARGS);
    return launch_play3<G2048_RNG_ORIGINAL, G2048_POLICY_DRUL, false>(ARGS);
#undef ARGS
}

// ---- recording form: arena sizing, launch, compaction into the env-major flat buffer ---------------------------------

// slots per lane: room for one whole episode (max_steps + 1) beyond the lane's expected share of the batch's records
static int64_t play_record_lane_slots(int64_t n, int64_t max_steps, int64_t mean_steps, int sms) {
    const int64_t lanes = play3_shape(n, sms).lanes();
    const int64_t envs_per_lane = (n + lanes - 1) / lanes;
    // share: mean episode (+1 slot for its final board) x envs per lane, +25 % and two mean episodes of slack for the
    // imbalance between lanes (a lane that runs out retires; the others take its envs)
    const int64_t share = (envs_per_lane * (mean_steps + 1) * 5) / 4 + 2 * (mean_steps + 1);
    return share + max_steps + 1;
}

int play_record_impl(int policy, const uint32_t* d_subs, int64_t n_subs, int64_t batch_global, int64_t env_lo, int64_t n,
                     int rng_mode, uint64_t* d_work, uint64_t* d_arena_boards, uint8_t* d_arena_meta, int64_t arena_slots,
                     uint64_t* d_env_slot, uint64_t* d_final_boards, uint32_t* d_lengths, uint32_t* d_scores,
                     uint64_t* d_stats, void* stream) {
    G2048_REQUIRE(policy == G2048_POLICY_RANDOM || policy == G2048_POLICY_DRUL, "play_record: policy");
    G2048_REQUIRE(rng_mode == G2048_RNG_ORIGINAL || rng_mode == G2048_RNG_PARTITIONABLE, "play_record: rng_mode");
    G2048_REQUIRE(batch_global > 0 && batch_global <= 0x7FFFFFFFll && env_lo >= 0 && n >= 0 && env_lo + n <= batch_global,
                  "play_record: batch");
    G2048_REQUIRE(n_subs >= 3 && d_subs && d_work && d_stats, "play_record: pointers");
    if (n == 0) return G2048_OK;
    G2048_REQUIRE(d_arena_boards && d_arena_meta && d_env_slot && d_lengths, "play_record: record pointers");
    const int sms = sm_count();
    if (sms <= 0) return fail_arg("play_record: no device");
    const int64_t lanes = play3_shape(n, sms).lanes();
    const int64_t max_steps = (n_subs - 1) / 2;
    PlayRecordArena rec;
    rec.boards = (u64*)d_arena_boards;
    rec.meta = d_arena_meta;
    rec.cap = (unsigned long long)(arena_slots / lanes);
    rec.env_slot = (unsigned long long*)d_env_slot;
    G2048_REQUIRE((int64_t)rec.cap >= max_steps + 1, "play_record: arena smaller than one episode per lane");
    cudaStream_t st = (cudaStream_t)stream;
#define ARGS d_subs, n_subs, batch_global, env_lo, n, d_work, d_final_boards, d_lengths, d_scores, d_stats, st, nullptr, rec
    if (policy == G2048_POLICY_RANDOM) {
        if (rng_mode == G2048_RNG_PARTITIONABLE) return launch_play3<G2048_RNG_PARTITIONABLE, G2048_POLICY_RANDOM, true>(ARGS);
        return launch_play3<G2048_RNG_ORIGINAL, G2048_POLICY_RANDOM, true>(ARGS);
    }
    if (rng_mode == G2048_RNG_PARTITIONABLE) return launch_play3<G2048_RNG_PARTITIONABLE, G2048_POLICY_DRUL, true>(ARGS);
    return launch_play3<G2048_RNG_ORIGINAL, G2048_POLICY_DRUL, true>(ARGS);
#undef ARGS
}

// One warp per env: the episode's slot range -> its segment of the flat buffer (9 B read + up to 21 B written per
// env-step).  A warp takes 128 steps per iteration -- the mean episode is about that long -- with every load of the
// iteration issued before the first use.  The first form executed 171 instructions per lane-step (ncu), many of them
// predication (loads guarded by t <= len, five null tests per store group, shuffles inside divergent code); this one
// clamps the load indices instead (slot `len` holds the final board, so every address is valid), keeps the shuffles
// in uniform code, tests t < len once, and is compiled a second time for callers that want every output (ALL: the
// product path) without the pointer tests: 139 instructions per lane-step -- and 249 instead of 255 us for C4's
// 3.1e7 steps, so instructions were not what bounds it.  Neither are the three other things ncu
// (profiles/r02_compact_ncu.txt: l1tex 70 %, long_scoreboard 12.7 per issue, DRAM 45 %) suggested, each built and timed:
// see the notes in the body.  What is left is the access pattern itself -- seven streams of 0.1 - 1 KB chunks per
// env, the reads scattered over the lanes' arena regions -- at 3.7 TB/s.
template <int POLICY, bool ALL>
__global__ void __launch_bounds__(256)
play_record_compact_kernel(const u64* __restrict__ arena_boards, const uint8_t* __restrict__ arena_meta,
                           const unsigned long long* __restrict__ env_slot, const uint32_t* __restrict__ lengths,
                           const int64_t* __restrict__ offsets, int64_t n, int64_t out_base, int64_t out_capacity,
                           u64* __restrict__ o_boards, uint8_t* __restrict__ o_meta, float* __restrict__ o_rewards,
                           float* __restrict__ o_log_probs, float* __restrict__ o_values, float* __restrict__ o_max_reward) {
    constexpr int K = 4;  // 32-step groups per iteration
    const uint32_t lane = threadIdx.x & 31u;
    const int64_t warps = (int64_t)gridDim.x * (blockDim.x >> 5);
    // potential of a pair of cells (one byte of the board): 8 shared-memory lookups per board instead of 16 x 6
    // instructions; log(1 / #legal) by legal mask (the lock-step recorder's act_random_log_prob, bit for bit).
    // (One copy of the table per bank -- lookups of a warp never conflict, 32 KiB per CTA, one wave of resident CTAs --
    // was slower as well: 284 vs 249 us.)
    __shared__ uint32_t s_pot[256];
    __shared__ float s_lp[16];
    {
        const uint32_t lo = threadIdx.x & 15u, hi = (threadIdx.x >> 4) & 15u;
        s_pot[threadIdx.x & 255] = (lo ? ((lo - 1u) << lo) : 0u) + (hi ? ((hi - 1u) << hi) : 0u);
        if (threadIdx.x < 16) s_lp[threadIdx.x] = (POLICY == G2048_POLICY_RANDOM) ? act_random_log_prob(threadIdx.x) : 0.0f;
    }
    __syncthreads();
    const char* pot_base = reinterpret_cast<const char*>(s_pot);
    auto pair = [&](uint32_t byte_times_4) -> uint32_t { return *reinterpret_cast<const uint32_t*>(pot_base + byte_times_4); };
    auto potential = [&](u64 x) -> uint32_t {
        const uint32_t a = (uint32_t)x, c = (uint32_t)(x >> 32);
        return (pair((a << 2) & 0x3FCu) + pair((a >> 6) & 0x3FCu) + pair((a >> 14) & 0x3FCu) + pair((a >> 22) & 0x3FCu)) +
               (pair((c << 2) & 0x3FCu) + pair((c >> 6) & 0x3FCu) + pair((c >> 14) & 0x3FCu) + pair((c >> 22) & 0x3FCu));
    };
    // (A software pipeline over the warp's envs -- header two envs ahead, the first 128 steps' loads one env ahead --
    // needed 80 registers, three CTAs per SM instead of five, and was slower: 289 vs 249 us for C4's 3.1e7 steps.)
    struct Header {
        uint32_t len;
        int32_t fits;  // steps of the env that lie inside the output arrays (all of them unless the caller's estimate was short)
        const u64* boards;
        const uint8_t* meta;
        int64_t dst;
    };
    auto load_header = [&](int64_t e) -> Header {
        const unsigned long long slot = env_slot[e];
        const uint32_t len = lengths[e];
        const int64_t off = offsets[e], room = out_capacity - off;
        return Header{len, (int32_t)(room < 0 ? 0 : (room < (int64_t)len ? room : (int64_t)len)), arena_boards + slot, arena_meta + slot,
                      out_base + off};
    };
    // (Windows of 32 steps aligned in the DESTINATION -- every store a whole line -- were slower, 267 vs 249 us: the
    // partial first window costs more loads than the straddling stores cost lines.)
    // boards t0 .. t0 + 32 K (one more than steps: the reward of a step needs the next board's potential)
    auto load_records = [&](const Header& h, int32_t t0, u64 (&b)[K + 1], uint32_t (&m)[K]) {
        const int32_t len = (int32_t)h.len, last = max(len - 1, 0);
#pragma unroll
        for (int k = 0; k < K; ++k) {
            const int32_t t = t0 + 32 * k + (int32_t)lane;
            b[k] = __ldg(h.boards + min(t, len));
            m[k] = (uint32_t)__ldg(h.meta + min(t, last));
        }
        b[K] = __ldg(h.boards + min(t0 + 32 * K, len));  // the board after the iteration's last step: one address, broadcast
    };
    auto write_steps = [&](const Header& h, int32_t t0, const u64 (&b)[K + 1], const uint32_t (&m)[K], uint32_t& best) {
        uint32_t pot[K + 1];
#pragma unroll
        for (int k = 0; k <= K; ++k) pot[k] = potential(b[k]);
#pragma unroll
        for (int k = 0; k < K; ++k) {
            const int32_t t = t0 + 32 * k + (int32_t)lane;
            uint32_t p1 = __shfl_down_sync(0xFFFFFFFFu, pot[k], 1);
            const uint32_t first_of_next = (k + 1 < K) ? __shfl_sync(0xFFFFFFFFu, pot[k + 1], 0) : pot[K];
            if (lane == 31u) p1 = first_of_next;
            if (t < (int32_t)h.len) {
                const uint32_t gained = p1 - pot[k] - ((m[k] >> 5) & 4u);  // bit 7: the spawned tile was a 4
                const int64_t o = h.dst + t;
                best = max(best, gained);
                if (t < h.fits) {
                    if (ALL || o_boards) o_boards[o] = b[k];
                    if (ALL || o_meta) o_meta[o] = (uint8_t)(m[k] & 0x7Fu);
                    if (ALL || o_rewards) o_rewards[o] = (float)gained;
                    if (ALL || o_log_probs) o_log_probs[o] = s_lp[(m[k] >> 2) & 15u];
                    if (ALL || o_values) o_values[o] = 0.0f;
                }
            }
        }
    };
    for (int64_t e = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); e < n; e += warps) {
        const Header h = load_header(e);
        uint32_t best = 0;  // the trainer's "episode reward" = max_t reward (src/ppo/ppo_trainer.py:218-227)
        for (int32_t t0 = 0; t0 < (int32_t)h.len; t0 += 32 * K) {
            u64 b[K + 1];
            uint32_t m[K];
            load_records(h, t0, b, m);
            write_steps(h, t0, b, m, best);
        }
        if (o_max_reward) {
            for (int off = 16; off > 0; off >>= 1) best = max(best, __shfl_xor_sync(0xFFFFFFFFu, best, off));
            if (lane == 0) o_max_reward[e] = (float)best;
        }
    }
}

}  // namespace g2048

using namespace g2048;

// Test hook: the table entries of the given 16-bit rows (row = four nibbles, nibble 0 = column 0).
extern "C" int g2048_row_table_lookup(const uint16_t* d_rows, int64_t n, uint16_t* d_left, uint8_t* d_flags,
                                      void* stream) {
    G2048_REQUIRE(n >= 0 && (n == 0 || (d_rows && d_left && d_flags)), "row_table_lookup");
    if (n == 0) return G2048_OK;
    int rc = ensure_row_tables((cudaStream_t)stream);
    if (rc) return rc;
    row_table_lookup_kernel<<<blocks_for(n, 256), 256, 0, (cudaStream_t)stream>>>(d_rows, n, d_left, d_flags);
    G2048_CHECK_LAUNCH("row_table_lookup");
    return G2048_OK;
}

// Table kernel entry: same arguments and results as g2048_play.  g2048_play itself dispatches here
// for batches large enough to amortise the 192 KiB table copy per CTA.
extern "C" int g2048_play_tables(int policy, const uint32_t* d_subs, int64_t n_subs, int64_t batch_global,
                                 int64_t env_lo, int64_t n, int rng_mode, uint64_t* d_work, uint64_t* d_final_boards,
                                 uint32_t* d_lengths, uint32_t* d_scores, uint64_t* d_stats, void* stream) {
    return play_tables_impl(policy, d_subs, n_subs, batch_global, env_lo, n, rng_mode, d_work, d_final_boards, d_lengths,
                            d_scores, d_stats, nullptr, stream);
}

// ---- recording form (see PlayRecordArena above) ---------------------------------------------------------------------
extern "C" int64_t g2048_play_record_arena_slots(int64_t n, int64_t n_subs, int64_t mean_steps) {
    if (n <= 0 || n_subs < 3 || mean_steps < 0) return -1;
    const int sms = sm_count();
    if (sms <= 0) return -1;
    const int64_t lanes = play3_shape(n, sms).lanes();
    return lanes * play_record_lane_slots(n, (n_subs - 1) / 2, mean_steps, sms);
}

extern "C" int g2048_play_record(int policy, const uint32_t* d_subs, int64_t n_subs, int64_t batch_global, int64_t env_lo,
                                 int64_t n, int rng_mode, uint64_t* d_work, uint64_t* d_arena_boards, uint8_t* d_arena_meta,
                                 int64_t arena_slots, uint64_t* d_env_slot, uint64_t* d_final_boards, uint32_t* d_lengths,
                                 uint32_t* d_scores, uint64_t* d_stats, void* stream) {
    return play_record_impl(policy, d_subs, n_subs, batch_global, env_lo, n, rng_mode, d_work, d_arena_boards, d_arena_meta,
                            arena_slots, d_env_slot, d_final_boards, d_lengths, d_scores, d_stats, stream);
}

extern "C" int g2048_play_record_compact(int policy, const uint64_t* d_arena_boards, const uint8_t* d_arena_meta,
                                         const uint64_t* d_env_slot, const uint32_t* d_lengths, const int64_t* d_offsets,
                                         int64_t n, int64_t out_base, int64_t out_capacity, uint64_t* d_boards, uint8_t* d_meta,
                                         float* d_rewards, float* d_log_probs, float* d_values, float* d_max_reward, void* stream) {
    G2048_REQUIRE(policy == G2048_POLICY_RANDOM || policy == G2048_POLICY_DRUL, "play_record_compact: policy");
    G2048_REQUIRE(n >= 0 && out_base >= 0 && out_capacity >= 0, "play_record_compact: sizes");
    if (n == 0) return G2048_OK;
    G2048_REQUIRE(d_arena_boards && d_arena_meta && d_env_slot && d_lengths && d_offsets, "play_record_compact: pointers");
    const int sms = sm_count();
    if (sms <= 0) return fail_arg("play_record_compact: no device");
    const int64_t need = (n + 7) / 8;  // 8 warps (envs) per CTA
    const int64_t cap = (int64_t)sms * 32;  // grid-stride beyond 8 resident CTAs per SM x 4
    const unsigned grid = (unsigned)(need < cap ? need : cap);
    cudaStream_t st = (cudaStream_t)stream;
#define G2048_COMPACT_LAUNCH(P, A)                                                                                      \
    play_record_compact_kernel<P, A><<<grid, 256, 0, st>>>((const u64*)d_arena_boards, d_arena_meta,                    \
        (const unsigned long long*)d_env_slot, d_lengths, d_offsets, n, out_base, out_capacity, (u64*)d_boards, d_meta, \
        d_rewards, d_log_probs, d_values, d_max_reward)
    const bool all = d_boards && d_meta && d_rewards && d_log_probs && d_values;
    if (policy == G2048_POLICY_RANDOM) {
        if (all) G2048_COMPACT_LAUNCH(G2048_POLICY_RANDOM, true); else G2048_COMPACT_LAUNCH(G2048_POLICY_RANDOM, false);
    } else {
        if (all) G2048_COMPACT_LAUNCH(G2048_POLICY_DRUL, true); else G2048_COMPACT_LAUNCH(G2048_POLICY_DRUL, false);
    }
#undef G2048_COMPACT_LAUNCH
    G2048_CHECK_LAUNCH("play_record_compact");
    return G2048_OK;
}
