// Pieces of the shared-memory-table play kernel (g2048_play3.cu) that the playout kernel (g2048_playout.cu) is built
// from as well: the row tables, the lane state, the legal mask and the game step.
#pragma once
#include "g2048_board.cuh"
#include "g2048_common.cuh"
#include "g2048_env.cuh"
#include "g2048_play.cuh"

namespace g2048 {

#ifndef G2048_PLAY3_THREADS
#define G2048_PLAY3_THREADS 768
#endif
#ifndef G2048_PLAY3_SMALL_THREADS
#define G2048_PLAY3_SMALL_THREADS 512
#endif
#ifndef G2048_PLAY3_BIG_ENVS_PER_LANE
#define G2048_PLAY3_BIG_ENVS_PER_LANE 16
#endif
#ifndef G2048_PLAY3_EPILOGUE_BATCH
#define G2048_PLAY3_EPILOGUE_BATCH 16
#endif
constexpr int PLAY3_EPILOGUE_BATCH = G2048_PLAY3_EPILOGUE_BATCH;  // parked finished episodes per epilogue run
// One CTA per SM.  While the kernel was bound by the ALU pipe alone, 512 / 768 / 1024 threads were within 3 % and 512
// drained fastest.  With fewer ALU instructions per step latency matters more: 768 threads (24 warps, <= 80 registers,
// no spills) are 2.7 % faster at 2^24 envs, but the drain of the last episodes, longer with more lanes, makes them
// slower where a lane plays only a few envs (2^18 envs: +7 %; break-even between 2^20 and 2^21 envs on 148 SMs, 9 and
// 18 envs per lane).  So the kernels are compiled for both sizes, and a launch runs PLAY3_THREADS threads per CTA
// when every lane gets at least PLAY3_BIG_ENVS_PER_LANE envs on average, else PLAY3_SMALL_THREADS (profiles/README.md,
// round 5).  (One build for 768 threads launched with 512 where needed is as fast at small sizes, but the block size
// read at run time changes ptxas's schedule of the whole kernel: 2^24 envs 63.1 -> 63.8 ms.)
constexpr int PLAY3_THREADS = G2048_PLAY3_THREADS;
constexpr int PLAY3_SMALL_THREADS = G2048_PLAY3_SMALL_THREADS;

// threads per CTA of a launch over n envs (or playouts) on `sms` SMs
inline int play3_block_threads(int64_t n, int sms) {
    return n >= (int64_t)G2048_PLAY3_BIG_ENVS_PER_LANE * sms * PLAY3_THREADS ? PLAY3_THREADS : PLAY3_SMALL_THREADS;
}
constexpr int PLAY3_TABLE_BYTES = 65536 * 2 + 65536;

// (static: each translation unit that includes this file has its own tables)
static __device__ uint16_t g_row_left[65536];  // row slid and merged toward nibble 0
static __device__ uint8_t g_row_flags[65536];  // bit 0: the row changes when moved toward nibble 0, bit 2: toward nibble 3

__device__ __forceinline__ uint32_t row_left_scalar(uint32_t row) {
    uint32_t tiles[4];
    int n = 0;
    for (int c = 0; c < 4; ++c) {
        const uint32_t v = (row >> (4 * c)) & 15u;
        if (v) tiles[n++] = v;
    }
    uint32_t out = 0;
    int w = 0;
    for (int j = 0; j < n; ++w) {
        if (j + 1 < n && tiles[j] == tiles[j + 1]) {
            out |= ((tiles[j] + 1u) & 15u) << (4 * w);  // 2^15 + 2^15 wraps; such envs are flagged by the caller
            j += 2;
        } else {
            out |= tiles[j] << (4 * w);
            j += 1;
        }
    }
    return out;
}

__device__ __forceinline__ uint32_t row_mirror_scalar(uint32_t row) {
    return ((row & 0xFu) << 12) | ((row & 0xF0u) << 4) | ((row >> 4) & 0xF0u) | ((row >> 12) & 0xFu);
}

// the table entries of one row (a translation unit's build kernel runs this for rows 0 .. 65535)
__device__ __forceinline__ void build_row_table_entry(uint32_t row) {
    const uint32_t left = row_left_scalar(row);
    const uint32_t right = row_mirror_scalar(row_left_scalar(row_mirror_scalar(row)));
    g_row_left[row] = (uint16_t)left;
    g_row_flags[row] = (uint8_t)((left != row ? 1u : 0u) | (right != row ? 4u : 0u));  // bits 0 and 2: see the legal mask below
}

// tables: global (L2) -> shared (at smem_raw: left moves, then flags), by a CTA of THREADS threads
template <int THREADS>
__device__ __forceinline__ void play3_copy_row_tables(uint8_t* smem_raw) {
    const uint4* src_left = reinterpret_cast<const uint4*>(g_row_left);
    const uint4* src_flags = reinterpret_cast<const uint4*>(g_row_flags);
    uint4* dst = reinterpret_cast<uint4*>(smem_raw);
    for (int i = threadIdx.x; i < 65536 * 2 / 16; i += THREADS) dst[i] = __ldg(&src_left[i]);
    for (int i = threadIdx.x; i < 65536 / 16; i += THREADS) dst[65536 * 2 / 16 + i] = __ldg(&src_flags[i]);
}

// spawn masks: for each cell, a 1 in its nibble of the board and in its nibble of the transpose (uint4: lo, hi, lo, hi)
constexpr int PLAY3_SPAWN_BYTES = 16 * 16;
__device__ __forceinline__ void play3_fill_spawn_masks(uint4* s_spawn) {
    if (threadIdx.x < 16) {
        const unsigned cell = threadIdx.x, cellT = ((cell & 3u) << 2) | (cell >> 2);
        const u64 m = 1ull << (4 * cell), mT = 1ull << (4 * cellT);
        s_spawn[cell] = make_uint4((uint32_t)m, (uint32_t)(m >> 32), (uint32_t)mT, (uint32_t)(mT >> 32));
    }
}

// the random policy's action table (act_random_table, g2048_play.cuh), one entry per legal mask
constexpr int PLAY3_ACT_BYTES = 16 * (int)sizeof(ActEntry);
__device__ __forceinline__ void play3_fill_act_table(ActEntry* s_act) {
    if (threadIdx.x < 16) s_act[threadIdx.x] = act_entry_of(threadIdx.x);
}

// Recording form (REC = true; src/runs/batch_runner.py:117-154 + src/ppo/rollout_buffer.py:164-187): the lane also
// writes the trajectory of every env it plays.  A lane plays its envs one after the other, so its records are one
// sequential stream: lane L owns slots [L * cap, (L + 1) * cap) of an arena and appends, per env-step, the pre-step
// board (8 B) and a meta byte (action | pre-step legal mask << 2 | post-step done << 6 | "the spawn was a 4-tile" << 7),
// and after an env's last step its final board (one extra slot).  env_slot[e] is the slot of env e's step 0, so an
// episode is the contiguous slot range [env_slot[e], env_slot[e] + length[e]] -- what g2048_play_record_compact turns
// into the env-major flat buffer RolloutBuffer keeps, deriving the per-step reward from consecutive boards
// (reward_t = potential(board_{t+1}) - potential(board_t) - 4 * [4-tile spawned at t], see board_potential) so that
// the play loop itself computes no reward.  ~12 instructions and two stores per env-step on top of play3_kernel.
// A lane only takes a new env while a whole episode (max_steps + 1 slots) still fits into its region; a lane that
// cannot retires, and envs nobody could take are reported through stats[0] < n (the caller retries with a larger arena).
struct PlayRecordArena {
    u64* boards;                   // arena slots: pre-step boards (+ final board of each episode)
    uint8_t* meta;                 // arena slots: meta bytes
    unsigned long long cap;        // slots per lane
    unsigned long long* env_slot;  // (n) slot of step 0 of env i
};

// Everything a lane holds: its env, the finished episode it has parked, its share of the statistics.
struct Play3Lane {
    u64 board, boardT;  // the board and its transpose
    uint32_t lm, e, t, fours, phase;
    bool seen15;
    bool fin_live, fin_cut;  // the live fields hold a finished episode that is not parked yet
    // Episode epilogue (score from the final board, result stores, statistics: ~150 instructions).  Lanes finish
    // one at a time -- a warp meets a finished episode on roughly every fourth step -- so running the epilogue on the
    // spot means running it with one active lane, ~4 % of the kernel's instructions.  A finished lane parks its final
    // state in a second register set instead and takes the next env at once; the epilogue runs for all parked lanes
    // together when PLAY3_EPILOGUE_BATCH of them have gathered (or a parked lane finishes again, or at the end).
    // 2^21 envs, random policy: 25.76 G env-steps/s with the epilogue on the spot, 26.22 batched by 8, 26.32 by 16 or 32.
    u64 pk_board;
    uint32_t pk_t, pk_fours, pk_e;
    bool pk_has, pk_cut, pk_seen15;
    uint32_t st_episodes, st_cut, st_ovf, st_longest;
    unsigned long long st_steps, st_score, st_tile, st_tile2;
    unsigned long long slot, slot_end;  // recording: next free slot of the arena region being written, end of the lane's own region
};

// What is constant over the launch.
struct Play3Ctx {
    const uint2* subs;
    uint2 init_sub;
    uint32_t max_steps, batch_global, env_lo;
    const uint16_t* s_left;
    const uint8_t* s_flags;
    const uint4* s_spawn;
    const ActEntry* s_act;
    unsigned long long* s_stats;
    u64* final_boards;
    uint32_t* lengths;
    uint32_t* scores;
    uint4* results;
    PlayRecordArena rec;
};

// exact legal mask: "row can move left / right" for the 4 rows and the 4 columns
__device__ __forceinline__ uint32_t play3_legal(const uint8_t* s_flags, u64 b, u64 bT) {
    const uint32_t blo = (uint32_t)b, bhi = (uint32_t)(b >> 32);
    const uint32_t tlo = (uint32_t)bT, thi = (uint32_t)(bT >> 32);
    const uint32_t fb = s_flags[blo & 0xFFFFu] | s_flags[blo >> 16] | s_flags[bhi & 0xFFFFu] | s_flags[bhi >> 16];
    const uint32_t ft = s_flags[tlo & 0xFFFFu] | s_flags[tlo >> 16] | s_flags[thi & 0xFFFFu] | s_flags[thi >> 16];
    return fb | (ft << 1);  // rows give Left (bit 0) and Right (bit 2), columns the same bits one up: Up (1), Down (3)
}

// One loop iteration of a lane that holds an env: a game step, or one of the two init spawns.
// (The draws of an iteration are a pure function of (env, loop step, phase) -- never of the board -- so they can be made
// one iteration AHEAD, next to the game logic of the current one; in the drain of a launch, where a scheduler has few
// warps left, the three Threefry blocks that precede the first look at the board are most of a step's latency.  Built
// and A/B-timed in round 2, bit-exact, and 14 % slower at 2^24 envs (69.7 -> 81.2 ms), 9 % at 2^18: the env a lane has
// just claimed needs its first draws on the spot, one or two lanes of a warp at a time, every fourth step -- a whole
// RNG evaluation per claim at one lane's width.  An extra all-lanes "pre" iteration per episode would avoid that
// divergence for ~1.5 % more work in the dense phase, which is where the headline number lives; not pursued.)
template <int MODE, int POLICY, bool REC>
__device__ __forceinline__ void play3_step(Play3Lane& L, const Play3Ctx& c) {
    // keys: identical to g2048_play.cu
    const bool playing = L.phase == PHASE_PLAY;
    const uint2 ss = __ldg(&c.subs[2 + 2 * (int64_t)L.t]);
    int action;
    Key kstep;
    if (POLICY == G2048_POLICY_RANDOM) {
        const uint2 sa = __ldg(&c.subs[1 + 2 * (int64_t)L.t]);
        const Key head = playing ? Key{sa.x, sa.y} : Key{c.init_sub.x, c.init_sub.y};
        const KeyBlocks<MODE> kb = key_blocks<MODE>(split_at<MODE>(head, c.batch_global, c.env_lo + L.e));
        action = act_random_table(kb.bits, c.s_act[L.lm]);  // = argmax_bits_legal(kb.bits, L.lm)
        const Key kplay = split_at<MODE>(Key{ss.x, ss.y}, c.batch_global, c.env_lo + L.e);
        const Key kinit = (L.phase == PHASE_INIT0) ? kb.child[0] : kb.child[1];
        kstep = playing ? kplay : kinit;
    } else {
        action = act_drul(L.lm);
        const Key head = playing ? Key{ss.x, ss.y} : Key{c.init_sub.x, c.init_sub.y};
        kstep = split_at<MODE>(head, c.batch_global, c.env_lo + L.e);
        if (!playing) {  // r_phase = split(init key)[phase]
            Key c0, c1;
            split2<MODE>(kstep, c0, c1);
            kstep = (L.phase == PHASE_INIT0) ? c0 : c1;
        }
    }
    Key k1, k2;
    split2<MODE>(kstep, k1, k2);
    const uint32_t bits_pos = bits_scalar<MODE>(k1);
    const uint32_t bits_val = bits_scalar<MODE>(k2);

    // ---- move: four table lookups on the board (Left/Right) or its transpose (Up/Down) -----------------
    const u64 pre_board = L.board;   // REC: what the record of this step holds
    const uint32_t pre_lm = L.lm;
    const bool vertical = (action & 1) != 0, rev = action >= 2;
    u64 src = vertical ? L.boardT : L.board;
    if (rev) src = mirror_rows(src);
    const uint32_t slo = (uint32_t)src, shi = (uint32_t)(src >> 32);
    const uint32_t m0 = c.s_left[slo & 0xFFFFu], m1 = c.s_left[slo >> 16];
    const uint32_t m2 = c.s_left[shi & 0xFFFFu], m3 = c.s_left[shi >> 16];
    u64 moved = ((u64)(m2 | (m3 << 16)) << 32) | (u64)(m0 | (m1 << 16));
    if (rev) moved = mirror_rows(moved);
    const u64 movedT = transpose_board(moved);
    u64 nb = vertical ? movedT : moved;   // row-major board after the move
    u64 nbT = vertical ? moved : movedT;  // its transpose
    if (!playing) {  // the two init iterations only spawn
        nb = L.board;
        nbT = L.boardT;
    }
    // ---- spawn into both orientations -------------------------------------------------------------------
    int cell;
    u64 val;
    spawn_select(nb, bits_pos, bits_val, cell, val);
    // The chosen cell is empty (a legal move leaves one; a full board is only reachable through illegal actions, which
    // these policies never take), so setting it is an add: mask * val + board per 32-bit half, on the FMA pipe, with the
    // masks of the cell in both orientations from a 16-entry shared-memory table (LSU pipe).  Two 64-bit variable
    // shifts, the transposed cell index and four ORs on the ALU pipe cost more (2^24 envs, random policy: 1.8 % in an
    // A/B on one B200).
    {
        const uint4 m = c.s_spawn[cell];
        const uint32_t v = (uint32_t)val;
        L.board = ((u64)(m.y * v + (uint32_t)(nb >> 32)) << 32) | (u64)(m.x * v + (uint32_t)nb);
        L.boardT = ((u64)(m.w * v + (uint32_t)(nbT >> 32)) << 32) | (u64)(m.z * v + (uint32_t)nbT);
    }
    L.fours += (val == 2ull) ? 1u : 0u;
    L.lm = play3_legal(c.s_flags, L.board, L.boardT);

    if (!playing) {
        L.phase += 1;  // INIT0 -> INIT1 -> PLAY
        return;
    }
    ++L.t;
    const bool done = L.lm == 0u;
    const bool cut = !done && L.t >= c.max_steps;
    if ((L.t & 255u) == 0u) L.seen15 |= has_max_nibble(L.board);  // the final board is checked in the epilogue
    if (REC) {  // the lane's own sequential stream: consecutive steps fill consecutive bytes of the same sectors
        c.rec.boards[L.slot] = pre_board;
        c.rec.meta[L.slot] = (uint8_t)((uint32_t)action | (pre_lm << 2) | (done ? 0x40u : 0u) | ((uint32_t)(val & 2ull) << 6));
        ++L.slot;
    }
    if (done || cut) {  // the final state stays in board / t / fours / e / seen15 until it is parked at the loop top
        L.fin_live = true;
        L.fin_cut = cut;
        L.phase = PHASE_NONE;
        if (REC) {  // the episode's last board closes its slot range (the reward of the last step needs it)
            c.rec.boards[L.slot] = L.board;
            c.rec.env_slot[L.e] = L.slot - (unsigned long long)L.t;
            ++L.slot;
        }
    }
}

// tables are built once per device, the first time a table kernel is launched; BUILD is the translation unit's own
// build kernel (65536 threads, build_row_table_entry each)
template <void (*BUILD)()>
static int ensure_row_tables_with(cudaStream_t st) {
    static bool built[64] = {false};
    int dev = 0;
    int rc = check_cuda(cudaGetDevice(&dev), "play: device");
    if (rc) return rc;
    if (dev < 0 || dev >= 64) return fail_arg("play: device index");
    if (built[dev]) return G2048_OK;
    BUILD<<<65536 / 256, 256, 0, st>>>();
    rc = check_cuda(cudaGetLastError(), "play: build tables");
    if (rc) return rc;
    rc = check_cuda(cudaStreamSynchronize(st), "play: build tables");  // one-time: later launches may use other streams
    if (rc) return rc;
    built[dev] = true;
    return G2048_OK;
}

}  // namespace g2048
