// Monte-Carlo playout values of caller-given boards (g2048_playout_values, include/g2048.h): for every (board, action)
// K games played to the end with a built-in rollout policy, the first move forced.  The persistent play kernel of
// g2048_play3.cu with two changes: a lane that claims playout p loads its start board instead of running env.init, and
// plays the forced action at t = 0 by presenting it to the policy as the only legal one.  The step itself is
// play3_step (g2048_play3.cuh), so a playout draws exactly what g2048_play draws for env p of a batch of P.
#include "g2048_play3.cuh"

namespace g2048 {

constexpr int PLAYOUT_STATS_BYTES = G2048_PLAY_STATS_WORDS * 8;
constexpr int PLAYOUT_SPAWN_OFFSET = PLAY3_TABLE_BYTES + PLAYOUT_STATS_BYTES;
constexpr int PLAYOUT_ACT_OFFSET = PLAYOUT_SPAWN_OFFSET + PLAY3_SPAWN_BYTES;
constexpr int PLAYOUT_SMEM_BYTES = PLAYOUT_ACT_OFFSET + PLAY3_ACT_BYTES;

// A playout lane: the game as play3_step sees it (e = the global playout index p, which keys its draws) and what the
// epilogue needs besides -- the (board, action) record it adds to and the start board's potential -- live and parked.
struct PlayoutLane {
    Play3Lane g;
    uint32_t rec, pot0;
    uint32_t pk_rec, pk_pot0;
};

__device__ __forceinline__ void playout_epilogue(PlayoutLane& P, const Play3Ctx& c, G2048PlayoutStats* records) {
    Play3Lane& L = P.g;
    if (L.pk_has) {
        // merge rewards from the start board on: potential gained minus the 4 that every spawned 4-tile brings
        const uint32_t score = board_potential(L.pk_board) - P.pk_pot0 - 4u * L.pk_fours;
        G2048PlayoutStats* r = records + P.pk_rec;
        atomicAdd(reinterpret_cast<unsigned long long*>(&r->score_sum), (unsigned long long)score);
        atomicAdd(reinterpret_cast<unsigned long long*>(&r->score_sq_sum), (unsigned long long)score * score);
        atomicAdd(reinterpret_cast<unsigned long long*>(&r->steps_sum), (unsigned long long)L.pk_t);
        atomicAdd(&r->playouts, 1u);
        if (L.pk_cut) atomicAdd(&r->cut_short, 1u);
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

// play3_park with the playout epilogue (call converged)
__device__ __forceinline__ void playout_park(PlayoutLane& P, const Play3Ctx& c, G2048PlayoutStats* records) {
    Play3Lane& L = P.g;
    const unsigned fresh = __ballot_sync(0xFFFFFFFFu, L.fin_live);
    if (fresh) {
        const unsigned parked = __ballot_sync(0xFFFFFFFFu, L.pk_has);
        if ((fresh & parked) != 0u || __popc(fresh | parked) >= PLAY3_EPILOGUE_BATCH) playout_epilogue(P, c, records);
        if (L.fin_live) {
            L.pk_board = L.board;
            L.pk_t = L.t;
            L.pk_fours = L.fours;
            L.pk_cut = L.fin_cut;
            L.pk_seen15 = L.seen15;
            L.pk_has = true;
            P.pk_rec = P.rec;
            P.pk_pot0 = P.pot0;
            L.fin_live = false;
        }
    }
}

// Work item j < n * 4 * K is playout k = j % K of action a = (j / K) % 4 on board i = j / (4 K); its record is j / K.
template <int MODE, int POLICY, int THREADS>
__global__ void __launch_bounds__(THREADS, 1)
playout_kernel(const u64* __restrict__ boards, const int64_t* __restrict__ board_ids, uint32_t board_lo, uint32_t n_items,
               uint32_t playouts, const uint2* __restrict__ subs, int64_t n_subs, uint32_t batch_global,
               unsigned long long* __restrict__ work, G2048PlayoutStats* __restrict__ records,
               unsigned long long* __restrict__ stats) {
    extern __shared__ __align__(16) uint8_t smem_raw[];
    unsigned long long* s_stats = reinterpret_cast<unsigned long long*>(smem_raw + PLAY3_TABLE_BYTES);
    play3_copy_row_tables<THREADS>(smem_raw);
    for (int i = threadIdx.x; i < G2048_PLAY_STATS_WORDS; i += THREADS) s_stats[i] = 0ull;
    play3_fill_spawn_masks(reinterpret_cast<uint4*>(smem_raw + PLAYOUT_SPAWN_OFFSET));
    play3_fill_act_table(reinterpret_cast<ActEntry*>(smem_raw + PLAYOUT_ACT_OFFSET));
    __syncthreads();

    const unsigned lane = threadIdx.x & 31u;
    Play3Ctx c = {};
    c.subs = subs;
    c.init_sub = subs[0];  // unused: playouts have no init iterations
    c.max_steps = (uint32_t)((n_subs - 1) / 2);
    c.batch_global = batch_global;
    c.env_lo = 0;  // L.e is the global playout index itself
    c.s_left = reinterpret_cast<const uint16_t*>(smem_raw);
    c.s_flags = smem_raw + 65536 * 2;
    c.s_spawn = reinterpret_cast<const uint4*>(smem_raw + PLAYOUT_SPAWN_OFFSET);
    c.s_act = reinterpret_cast<const ActEntry*>(smem_raw + PLAYOUT_ACT_OFFSET);
    c.s_stats = s_stats;

    PlayoutLane P = {};
    Play3Lane& L = P.g;
    L.phase = PHASE_NONE;
    bool exhausted = false;  // warp-uniform
    while (true) {
        const unsigned idle = __ballot_sync(0xFFFFFFFFu, L.phase == PHASE_NONE);
        if (idle) {
            playout_park(P, c, records);
            if (!exhausted) {
                const int cnt = __popc(idle);
                unsigned long long base = 0;
                race_jitter();
                if (lane == 0) base = atomicAdd(work, (unsigned long long)cnt);
                base = __shfl_sync(0xFFFFFFFFu, base, 0);
                if (base + (unsigned long long)cnt >= (unsigned long long)n_items) exhausted = true;
                if (L.phase == PHASE_NONE) {
                    const unsigned long long mine = base + (unsigned long long)__popc(idle & ((1u << lane) - 1u));
                    if (mine < (unsigned long long)n_items) {
                        const uint32_t j = (uint32_t)mine, rec = j / playouts, i = rec >> 2, a = rec & 3u;
                        const u64 b = __ldg(&boards[i]);  // shared by the 4 K consecutive items of the board: a cache hit
                        const u64 bT = transpose_board(b);
                        const uint32_t lm = play3_legal(c.s_flags, b, bT);
                        if ((lm >> a) & 1u) {  // an illegal (board, action) pair is dropped here and costs no step
                            const uint32_t id = board_ids ? (uint32_t)__ldg(&board_ids[i]) : board_lo + i;
                            L.e = (id * 4u + a) * playouts + (j - rec * playouts);
                            L.board = b;
                            L.boardT = bT;
                            L.lm = 1u << a;  // the forced first move: the only action the policy may take at t = 0
                            L.t = 0;
                            L.fours = 0;
                            L.seen15 = has_max_nibble(b);  // a start board with a 2^15 tile is flagged as overflowed
                            L.phase = PHASE_PLAY;
                            P.rec = rec;
                            P.pot0 = board_potential(b);
                        }
                    }
                }
            }
            if (__ballot_sync(0xFFFFFFFFu, L.phase != PHASE_NONE) == 0u && exhausted) break;
        }
        if (L.phase != PHASE_NONE) play3_step<MODE, POLICY, false>(L, c);
    }
    playout_epilogue(P, c, records);  // whatever is still parked

    atomicAdd(&s_stats[0], (unsigned long long)L.st_episodes);
    atomicAdd(&s_stats[1], L.st_steps);
    atomicAdd(&s_stats[2], L.st_score);
    atomicAdd(&s_stats[3], (unsigned long long)L.st_cut);
    atomicAdd(&s_stats[4], (unsigned long long)L.st_ovf);
    atomicMax(&s_stats[5], (unsigned long long)L.st_longest);
    atomicAdd(&s_stats[6], L.st_tile);
    atomicAdd(&s_stats[7], L.st_tile2);
    __syncthreads();
    if (stats) {
        for (int i = threadIdx.x; i < G2048_PLAY_STATS_WORDS; i += blockDim.x) {
            const unsigned long long v = s_stats[i];
            if (v) {
                if (i == 5) atomicMax(&stats[i], v);
                else atomicAdd(&stats[i], v);
            }
        }
    }
}

// this translation unit's copy of the row tables
__global__ void build_playout_row_tables_kernel() {
    const uint32_t row = blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= 65536u) return;
    build_row_table_entry(row);
}

template <int MODE, int POLICY, int THREADS>
static int launch_playout_with(int64_t grid, const uint64_t* d_boards, const int64_t* d_board_ids, int64_t board_lo,
                               int64_t n_items, int64_t playouts, const uint32_t* d_subs, int64_t n_subs, int64_t batch_global,
                               uint64_t* d_work, G2048PlayoutStats* d_records, uint64_t* d_stats, cudaStream_t st) {
    static bool configured_on[64] = {false};
    bool* configured = device_once_flag(configured_on);
    if (!configured) return fail_arg("no CUDA device");
    if (!*configured) {
        const int rc = check_cuda(cudaFuncSetAttribute(playout_kernel<MODE, POLICY, THREADS>,
                                                       cudaFuncAttributeMaxDynamicSharedMemorySize, PLAYOUT_SMEM_BYTES),
                                  "playout_values: shared memory attribute");
        if (rc) return rc;
        *configured = true;
    }
    playout_kernel<MODE, POLICY, THREADS><<<(unsigned)grid, THREADS, PLAYOUT_SMEM_BYTES, st>>>(
        (const u64*)d_boards, d_board_ids, (uint32_t)board_lo, (uint32_t)n_items, (uint32_t)playouts, (const uint2*)d_subs,
        n_subs, (uint32_t)batch_global, (unsigned long long*)d_work, d_records, (unsigned long long*)d_stats);
    return check_cuda(cudaGetLastError(), "playout_values");
}

template <int MODE, int POLICY>
static int launch_playout(const uint64_t* d_boards, const int64_t* d_board_ids, int64_t board_lo, int64_t n_items,
                          int64_t playouts, const uint32_t* d_subs, int64_t n_subs, int64_t batch_global, uint64_t* d_work,
                          G2048PlayoutStats* d_records, uint64_t* d_stats, cudaStream_t st) {
    const int rc = ensure_row_tables_with<build_playout_row_tables_kernel>(st);
    if (rc) return rc;
    const int sms = sm_count();
    if (sms <= 0) return fail_arg("playout_values: no device");
    const int threads = play3_block_threads(n_items, sms);
    const int64_t needed = (n_items + threads - 1) / threads;
    const int64_t grid = needed < sms ? needed : sms;  // one CTA per SM, persistent
#define ARGS grid, d_boards, d_board_ids, board_lo, n_items, playouts, d_subs, n_subs, batch_global, d_work, d_records, d_stats, st
    if (threads == PLAY3_THREADS) return launch_playout_with<MODE, POLICY, PLAY3_THREADS>(ARGS);
    return launch_playout_with<MODE, POLICY, PLAY3_SMALL_THREADS>(ARGS);
#undef ARGS
}

}  // namespace g2048

using namespace g2048;

extern "C" int g2048_playout_values(int policy, const uint64_t* d_boards, int64_t n, const int64_t* d_board_ids,
                                    int64_t board_lo, int64_t n_boards_global, int64_t playouts, const uint32_t* d_subs,
                                    int64_t n_subs, int rng_mode, uint64_t* d_work, G2048PlayoutStats* d_records,
                                    uint64_t* d_stats, void* stream) {
    G2048_REQUIRE(policy == G2048_POLICY_RANDOM || policy == G2048_POLICY_DRUL, "playout_values: policy");
    G2048_REQUIRE(rng_mode == G2048_RNG_ORIGINAL || rng_mode == G2048_RNG_PARTITIONABLE, "playout_values: rng_mode");
    G2048_REQUIRE(playouts >= 1 && playouts <= 0x7FFFFFFFll, "playout_values: playouts must be >= 1");
    G2048_REQUIRE(n_boards_global >= 1 && n_boards_global <= 0x7FFFFFFFll / (4 * playouts),
                  "playout_values: n_boards_global * 4 * playouts must be in [1, 2^31 - 1]");
    G2048_REQUIRE(n >= 0 && n <= n_boards_global, "playout_values: n");
    G2048_REQUIRE(d_board_ids ? board_lo == 0 : (board_lo >= 0 && board_lo + n <= n_boards_global),
                  "playout_values: board_lo (0 with an id list, else board_lo + n <= n_boards_global)");
    G2048_REQUIRE(n_subs >= 3 && d_subs, "playout_values: sub keys (n_subs >= 3)");
    G2048_REQUIRE(((uintptr_t)d_records & 7u) == 0, "playout_values: records must be 8-byte aligned");
    if (n == 0) return G2048_OK;
    G2048_REQUIRE(d_boards && d_work && d_records, "playout_values: pointers");
    cudaStream_t st = (cudaStream_t)stream;
    int rc = check_cuda(cudaMemsetAsync(d_records, 0, (size_t)n * 4 * sizeof(G2048PlayoutStats), st), "playout_values: records");
    if (rc) return rc;
    const int64_t batch = n_boards_global * 4 * playouts, items = n * 4 * playouts;
#define ARGS d_boards, d_board_ids, board_lo, items, playouts, d_subs, n_subs, batch, d_work, d_records, d_stats, st
    if (policy == G2048_POLICY_RANDOM) {
        if (rng_mode == G2048_RNG_PARTITIONABLE) return launch_playout<G2048_RNG_PARTITIONABLE, G2048_POLICY_RANDOM>(ARGS);
        return launch_playout<G2048_RNG_ORIGINAL, G2048_POLICY_RANDOM>(ARGS);
    }
    if (rng_mode == G2048_RNG_PARTITIONABLE) return launch_playout<G2048_RNG_PARTITIONABLE, G2048_POLICY_DRUL>(ARGS);
    return launch_playout<G2048_RNG_ORIGINAL, G2048_POLICY_DRUL>(ARGS);
#undef ARGS
}
