// Batched TD(0) afterstate learning of the expectimax row table T (g2048_td_train, include/g2048.h).
//
// Step t, for every env e < n with its key k = split(subs[t], n)[e]:
//   greedy move over q_a = (float)r_a + H_t(s_a) (Q_1 of g2048_expectimax_values with w = 1, same tie rule);
//   if the env holds an afterstate: fx(target - H_t(after)) into acc[idx] and 1 into cnt[idx] for its 8 lines;
//   then a finished episode restarts from init(k), anything else moves and spawns with k.
// After the whole batch: T[i] += alpha * mean of the fixed-point errors of entry i, and acc / cnt go back to zero.
//
// Mapping: ONE cooperative persistent launch for all the steps.  Thread j of the grid owns envs j, j + G, j + 2G, ...
// (G = grid threads) for the whole launch, and each step has two phases separated by grid.sync(): the accumulate phase
// reads the frozen T_t and adds integer errors with atomics, the apply phase (the grid striding over the 65 536
// entries) folds them into T.  The sums are integers, so neither the grid shape nor the order of the atomics changes a
// bit.  A grid that could not be co-resident makes cudaLaunchCooperativeKernel fail; there is no hand-rolled barrier
// that could hang.
//
// Hot rows: early boards put the empty line 0x0000 into most of their 8 lines, so the naive form makes about 10^5
// atomics on one address per step at n = 2^16.  Each line index is first aggregated in the warp (__match_any_sync:
// the group's leader adds the group's sum), and index 0 is further summed per CTA in shared memory, with one global
// atomic per CTA and step.
#include <cooperative_groups.h>

#include "g2048_xm.cuh"

namespace g2048 {

namespace cg = cooperative_groups;

// G2048_TD_AGGREGATE=0 (A/B builds only: make EXTRA=-DG2048_TD_AGGREGATE=0) makes one global atomic pair per line
// instead.  Aggregation wins at every size measured on one B200: 1.58 vs 1.00 G learning steps/s at n = 2^16, 1.88 vs
// 1.15 G at 2^18 (profiles/README.md, round 7).
#ifndef G2048_TD_AGGREGATE
#define G2048_TD_AGGREGATE 1
#endif

constexpr int TD_THREADS = 512;
constexpr int TD_SMEM_BYTES = PLAY3_TABLE_BYTES;  // the row tables; the small arrays below are static
constexpr int64_t TD_ENTRIES = 65536;
constexpr int64_t TD_SCRATCH_BYTES = TD_ENTRIES * 8 + TD_ENTRIES * 4;  // acc int64[65536], then cnt uint32[65536]
constexpr float TD_FX_CLAMP = 16777216.0f;  // 2^24: 2^20 envs * 8 lines * 2^24 * 4096 stays inside int64
constexpr float TD_FX_ONE = 4096.0f;

struct TdArgs {
    u64* boards;
    u64* after;
    uint32_t* scores;
    uint32_t* lengths;
    uint32_t n;
    float* T;
    float alpha;
    const uint2* subs;
    int64_t n_steps;
    unsigned long long* acc;
    uint32_t* cnt;
    unsigned long long* stats;
};

// fx(d) = rint(clamp(d, -2^24, 2^24) * 4096) as int64, to nearest even (the multiply by a power of two is exact)
__device__ __forceinline__ long long td_fx(float d) {
    return __float2ll_rn(fminf(fmaxf(d, -TD_FX_CLAMP), TD_FX_CLAMP) * TD_FX_ONE);
}

template <int MODE>
__global__ void __launch_bounds__(TD_THREADS, 1) td_train_kernel(const TdArgs a) {
    extern __shared__ __align__(16) uint8_t smem_raw[];
    __shared__ unsigned long long s_stats[G2048_PLAY_STATS_WORDS];
    __shared__ long long s_fx[TD_THREADS];
    __shared__ unsigned long long s_acc0;
    __shared__ unsigned s_cnt0;
    play3_copy_row_tables<TD_THREADS>(smem_raw);
    for (int i = threadIdx.x; i < G2048_PLAY_STATS_WORDS; i += TD_THREADS) s_stats[i] = 0ull;
    if (threadIdx.x == 0) {
        s_acc0 = 0ull;
        s_cnt0 = 0u;
    }
    __syncthreads();

    cg::grid_group grid = cg::this_grid();
    XmCtx c;
    c.T = a.T;
    c.w = 1.0f;
    c.s_left = reinterpret_cast<const uint16_t*>(smem_raw);
    c.s_flags = smem_raw + 65536 * 2;
    const unsigned lane = threadIdx.x & 31u;
    long long* warp_fx = s_fx + (threadIdx.x & ~31u);
    const uint32_t stride = gridDim.x * TD_THREADS;

    for (int64_t t = 0; t < a.n_steps; ++t) {
        const uint2 sub = __ldg(&a.subs[t]);
        // ---- accumulate: the whole CTA walks the envs together, so every warp is converged at the matches
        for (uint32_t base = blockIdx.x * TD_THREADS; base < a.n; base += stride) {
            const uint32_t e = base + threadIdx.x;
            const bool active = e < a.n;
            u64 s = 0ull, aft = 0ull;
            uint32_t score = 0u, length = 0u;
            if (active) {
                s = a.boards[e];
                aft = a.after[e];
                score = a.scores[e];
                length = a.lengths[e];
            }
            const u64 sT = transpose_board(s);
            const uint32_t lm = active ? play3_legal(c.s_flags, s, sT) : 0u;
            float target = 0.0f;
            u64 best = 0ull;
            uint32_t best_r = 0u;
            bool any = false;
#pragma unroll 1
            for (int act = 0; act < 4; ++act) {
                if ((lm >> act) & 1u) {
                    u64 nb, nbT;
                    uint32_t r;
                    xm_move<true>(c, s, sT, act, nb, nbT, r);
                    const float q = (float)r + xm_heuristic<true>(c, nb, nbT);
                    if (!any || q > target) {
                        target = q;
                        best = nb;
                        best_r = r;
                    }
                    any = true;
                }
            }
            const bool update = aft != 0ull;  // inactive lanes hold after = 0
            const u64 aftT = transpose_board(aft);
            warp_fx[lane] = update ? td_fx(target - xm_heuristic<true>(c, aft, aftT)) : 0ll;
            __syncwarp();
#pragma unroll 1
            for (int l = 0; l < 8; ++l) {
                const u64 src = l < 4 ? aft : aftT;
                const uint32_t idx = (uint32_t)(src >> (16 * (l & 3))) & 0xFFFFu;
#if G2048_TD_AGGREGATE
                const unsigned group = __match_any_sync(0xFFFFFFFFu, update ? idx : 0xFFFFFFFFu);
#else  // A/B builds only: one global atomic pair per line
                const unsigned group = 1u << lane;
#endif
                if (update && lane == (unsigned)(__ffs((int)group) - 1)) {
                    long long sum = 0;
                    for (unsigned m = group; m; m &= m - 1u) sum += warp_fx[__ffs((int)m) - 1];
                    const unsigned count = (unsigned)__popc((int)group);
                    if (G2048_TD_AGGREGATE && idx == 0u) {
                        atomicAdd(&s_acc0, (unsigned long long)sum);
                        atomicAdd(&s_cnt0, count);
                    } else {
                        atomicAdd(&a.acc[idx], (unsigned long long)sum);
                        atomicAdd(&a.cnt[idx], count);
                    }
                }
            }
            __syncwarp();  // warp_fx is rewritten by the next env

            if (active) {
                const Key k = split_at<MODE>(Key{sub.x, sub.y}, a.n, e);
                if (lm == 0u) {  // the episode ends here: count it and start the next one
                    const uint32_t me = max_exponent(s);
                    const unsigned long long tile = 1ull << me;
                    atomicAdd(&s_stats[0], 1ull);
                    atomicAdd(&s_stats[1], (unsigned long long)length);
                    atomicAdd(&s_stats[2], (unsigned long long)score);
                    if (has_max_nibble(s)) atomicAdd(&s_stats[4], 1ull);
                    atomicMax(&s_stats[5], (unsigned long long)length);
                    atomicAdd(&s_stats[6], tile);
                    atomicAdd(&s_stats[7], tile * tile);
                    atomicAdd(&s_stats[16 + me], 1ull);
                    a.boards[e] = env_init<MODE>(k).board;
                    a.after[e] = 0ull;
                    a.scores[e] = 0u;
                    a.lengths[e] = 0u;
                } else {
                    Key k1, k2;
                    split2<MODE>(k, k1, k2);
                    a.boards[e] = spawn_tile(best, bits_scalar<MODE>(k1), bits_scalar<MODE>(k2));
                    a.after[e] = best;
                    a.scores[e] = score + best_r;
                    a.lengths[e] = length + 1u;
                }
            }
        }
        __syncthreads();
        if (threadIdx.x == 0 && s_cnt0) {
            atomicAdd(&a.acc[0], s_acc0);
            atomicAdd(&a.cnt[0], s_cnt0);
            s_acc0 = 0ull;
            s_cnt0 = 0u;
        }
        grid.sync();
        // ---- apply: every entry with errors moves by alpha times their mean, and its accumulators go back to zero
        for (uint32_t i = blockIdx.x * TD_THREADS + threadIdx.x; i < (uint32_t)TD_ENTRIES; i += stride) {
            const uint32_t count = __ldcg(&a.cnt[i]);
            if (count) {
                const long long sum = (long long)__ldcg(&a.acc[i]);
                const float mean = (float)((double)sum / (4096.0 * (double)count));
                a.T[i] = a.T[i] + a.alpha * mean;
                a.acc[i] = 0ull;
                a.cnt[i] = 0u;
            }
        }
        grid.sync();
    }

    if (a.stats) {
        __syncthreads();
        for (int i = threadIdx.x; i < G2048_PLAY_STATS_WORDS; i += TD_THREADS) {
            const unsigned long long v = s_stats[i];
            if (v) {
                if (i == 5) atomicMax(&a.stats[i], v);
                else atomicAdd(&a.stats[i], v);
            }
        }
    }
}

// this translation unit's copy of the row tables
__global__ void build_td_row_tables_kernel() {
    const uint32_t row = blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= 65536u) return;
    build_row_table_entry(row);
}

template <int MODE>
static int launch_td(const TdArgs& args, cudaStream_t st) {
    auto kernel = td_train_kernel<MODE>;
    static bool configured_on[64] = {false};
    bool* configured = device_once_flag(configured_on);
    if (!configured) return fail_arg("no CUDA device");
    int dev = 0;
    int rc = check_cuda(cudaGetDevice(&dev), "td_train: device");
    if (rc) return rc;
    if (!*configured) {
        int coop = 0;
        rc = check_cuda(cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, dev), "td_train: device attribute");
        if (rc) return rc;
        if (!coop) return fail_arg("td_train: the device does not support cooperative launches");
        rc = check_cuda(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, TD_SMEM_BYTES),
                        "td_train: shared memory attribute");
        if (rc) return rc;
        *configured = true;
    }
    rc = ensure_row_tables_with<build_td_row_tables_kernel>(st);
    if (rc) return rc;
    int per_sm = 0;
    rc = check_cuda(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, TD_THREADS, TD_SMEM_BYTES),
                    "td_train: occupancy");
    if (rc) return rc;
    const int sms = sm_count();
    if (sms <= 0 || per_sm <= 0) return fail_arg("td_train: the kernel does not fit on this device");
    const int64_t needed = ((int64_t)args.n + TD_THREADS - 1) / TD_THREADS;
    const int64_t resident = (int64_t)per_sm * sms;
    const unsigned grid = (unsigned)(needed < resident ? needed : resident);
    void* params[] = {const_cast<TdArgs*>(&args)};
    return check_cuda(cudaLaunchCooperativeKernel((const void*)kernel, dim3(grid), dim3(TD_THREADS), params,
                                                  (size_t)TD_SMEM_BYTES, st),
                      "td_train");
}

}  // namespace g2048

using namespace g2048;

extern "C" int64_t g2048_td_scratch_bytes(void) { return TD_SCRATCH_BYTES; }

extern "C" int g2048_td_train(uint64_t* d_boards, uint64_t* d_after, uint32_t* d_scores, uint32_t* d_lengths, int64_t n,
                              float* d_row_values, float alpha, const uint32_t* d_subs, int64_t n_steps, int rng_mode,
                              void* d_scratch, uint64_t* d_stats, void* stream) {
    G2048_REQUIRE(n >= 1 && n <= (1ll << 20), "td_train: n must be in [1, 2^20]");
    G2048_REQUIRE(n_steps >= 0, "td_train: n_steps must be >= 0");
    G2048_REQUIRE(alpha >= 0.0f && alpha <= 3.402823466e38f, "td_train: alpha must be finite and >= 0");
    G2048_REQUIRE(rng_mode == G2048_RNG_ORIGINAL || rng_mode == G2048_RNG_PARTITIONABLE, "td_train: rng_mode");
    G2048_REQUIRE(d_boards && d_after && d_scores && d_lengths && d_row_values && d_scratch, "td_train: pointers");
    G2048_REQUIRE(n_steps == 0 || d_subs, "td_train: pointers");
    G2048_REQUIRE(((uintptr_t)d_boards & 7u) == 0 && ((uintptr_t)d_after & 7u) == 0 && ((uintptr_t)d_scratch & 7u) == 0 &&
                      ((uintptr_t)d_subs & 7u) == 0 && ((uintptr_t)d_stats & 7u) == 0,
                  "td_train: d_boards, d_after, d_subs, d_scratch and d_stats must be 8-byte aligned");
    G2048_REQUIRE(((uintptr_t)d_scores & 3u) == 0 && ((uintptr_t)d_lengths & 3u) == 0 && ((uintptr_t)d_row_values & 3u) == 0,
                  "td_train: d_scores, d_lengths and d_row_values must be 4-byte aligned");
    if (n_steps == 0) return G2048_OK;
    TdArgs args;
    args.boards = (u64*)d_boards;
    args.after = (u64*)d_after;
    args.scores = d_scores;
    args.lengths = d_lengths;
    args.n = (uint32_t)n;
    args.T = d_row_values;
    args.alpha = alpha;
    args.subs = (const uint2*)d_subs;
    args.n_steps = n_steps;
    args.acc = (unsigned long long*)d_scratch;
    args.cnt = (uint32_t*)((uint8_t*)d_scratch + TD_ENTRIES * 8);
    args.stats = (unsigned long long*)d_stats;
    cudaStream_t st = (cudaStream_t)stream;
    if (rng_mode == G2048_RNG_PARTITIONABLE) return launch_td<G2048_RNG_PARTITIONABLE>(args, st);
    return launch_td<G2048_RNG_ORIGINAL>(args, st);
}
