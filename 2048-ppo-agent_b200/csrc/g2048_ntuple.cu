// Batched TD(0) afterstate learning of an n-tuple network (g2048_ntuple_td_train, include/g2048.h).
//
// Step t, for every env e < n with its key k = split(subs[t], n)[e]:
//   greedy move over q_a = (float)r_a + V_t(s_a) (Q_1 of g2048_expectimax_values_ntuple with w = 1, same tie rule);
//   if the env holds an afterstate: fx(target - V_t(after)) into acc[i] and 1 into cnt[i] for i = off_p + idx_p(after),
//   every placement p in order; then a finished episode restarts from init(k), anything else moves and spawns with k.
// After the whole batch: W[i] += alpha * mean of the fixed-point errors of entry i, and acc / cnt go back to zero.
//
// Mapping: the accumulate / grid.sync() / apply / grid.sync() structure of td_train_kernel (g2048_td.cu), one
// cooperative persistent launch for all the steps.  What differs is the size of W: the 4x6 network has 2^26 weights,
// so the apply phase cannot sweep the sums as the row learner does (12 bytes an entry, ~0.8 GB a step).  Instead the
// accumulate phase lists the entries it touches: the atomicAdd on cnt[i] that returns 0 is the entry's first touch of
// the step, and that lane appends i to a list (one list atomic per warp and placement).  The apply phase walks the
// list, so its cost follows the entries touched, not n_weights.  The new value of an entry depends only on its integer
// (sum, count), so neither the grid, the order of the atomics nor the order of the list changes a bit.
//
// V evaluations: the 4 candidate afterstates and the previous afterstate are evaluated together (nt_values), so 5
// gathers per placement are in flight at once; an illegal action's board is the unmoved board, whose value is unused.
//
// Hot entries: early boards give most placements index 0 (all cells empty).  Each entry is first aggregated in the warp
// (__match_any_sync: the group's leader adds the group's sum), and index 0 of every placement is further summed per CTA
// in shared memory, with one global atomic per CTA, placement and step.
//
// Temporal coherence (g2048_ntuple_tc_train, the TC instantiations): the same kernel, which also sums |fx| into
// abs[i] next to acc[i] (the same warp aggregation and per-CTA index-0 sums), and whose apply phase scales each
// entry's step by beta = |E[i]| / A[i] from the entry's float64 running sums, then adds the step's sums to E and A.
// Only the apply phase touches E and A, one thread per listed entry, and grid.sync() orders the steps, so they use
// ordinary loads and stores.  With TC = false none of it is compiled in.
//
// Multi-stage networks (g2048_ntuple_staged_td_train / _tc_train, the STAGED instantiations): each of the 5 boards
// valued per env gets its stage base stage(b) * stride once, before the placement loop, and every entry of that board
// is moved by it; the accumulate phase uses the previous afterstate's base.  Nothing else changes: the listing, the
// apply walk and the fixed-point sums work on entries, whatever stage they belong to.  With STAGED = false none of it
// is compiled in.
//
// Delayed TD(lambda) / TC(lambda) (g2048_ntuple_lambda_td_train / _tc_train, the LAMBDA instantiations): each env keeps
// its last h afterstates and errors in a slot-major ring.  After v[] is used, a lane stores delta_L, reads the errors of
// the afterstates it releases (one a step in steady state, up to h when its episode ends) and the released board, and
// forms each e_m with __fmul_rn / __fadd_rn.  The placement loop (match, per-CTA index-0 sums, listing) runs once per
// release round; the round count is the warp's largest release count, so it stays warp-uniform, and a lane with nothing
// to release in a round takes part with the "no update" key.  With LAMBDA = false none of it is compiled in.
//
// Carousel shaping (g2048_ntuple_carousel_td_train / _tc_train, the CAROUSEL instantiations, always STAGED): an env
// whose move raises the stage stores its new board in its pending word in the scratch; the apply phase, after the
// first grid.sync(), commits each pending word of the envs the thread owns to the pool and clears it, so no draw of
// the step sees it.  An env whose episode ends reads its start stage and draws one pool slot; it restarts from that
// board, or from init(k) when the slot is empty or the carousel is back at the opening.  With CAROUSEL = false none of
// it is compiled in.
#include <cooperative_groups.h>

#include "g2048_ntuple.cuh"
#include "g2048_xm.cuh"

namespace g2048 {

namespace cg = cooperative_groups;

// G2048_NTUPLE_PHASES (A/B builds only: make OUT=... BUILD=... EXTRA=-DG2048_NTUPLE_PHASES, as tools/bench_ntuple.py
// does) makes CTA 0 time both phases of every step with %globaltimer, each up to the grid.sync() that ends it, and
// ADD to d_stats[8] the accumulate nanoseconds, [9] the apply nanoseconds and [10] the entries listed (words the
// statistics layout leaves unused).  The default build has none of it.
#ifdef G2048_NTUPLE_PHASES
__device__ __forceinline__ unsigned long long nt_clock() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
#endif

constexpr int NT_THREADS = 512;
constexpr int NT_SMEM_BYTES = PLAY3_TABLE_BYTES;  // the row tables; the small arrays below are static
constexpr float NT_FX_CLAMP = 16777216.0f;        // 2^24: 2^20 envs * 64 placements * 2^24 * 4096 = 2^62
constexpr float NT_FX_ONE = 4096.0f;

// scratch: acc int64[n_weights], (TC: abs int64[n_weights],) cnt uint32[n_weights], list uint32[min(n * P,
// n_weights)], then list_len uint32[2]; the lambda forms lay it out for n * h envs, as an env releases up to h
// afterstates a step.  The carousel forms append the pending words, uint64[n], at `bytes`.
struct NtScratch {
    int64_t abs_off, cnt_off, list_off, len_off, bytes;
};

static NtScratch nt_scratch_layout(int64_t n, int n_placements, int64_t n_weights, bool tc) {
    const int64_t touched = n * n_placements < n_weights ? n * n_placements : n_weights;
    NtScratch s;
    s.abs_off = 8 * n_weights;
    s.cnt_off = (tc ? 16 : 8) * n_weights;
    s.list_off = s.cnt_off + 4 * n_weights;
    s.len_off = (s.list_off + 4 * touched + 7) & ~7ll;
    s.bytes = s.len_off + 8;
    return s;
}

struct NtTdArgs {
    u64* boards;
    u64* after;
    uint32_t* scores;
    uint32_t* lengths;
    uint32_t n;
    float* W;
    float alpha;
    const uint2* subs;
    int64_t n_steps;
    unsigned long long* acc;
    uint32_t* cnt;
    uint32_t* list;
    uint32_t* list_len;  // [2]: step t appends through list_len[t & 1]
    unsigned long long* stats;
    NtNet net;  // net.W == W
    // TC only (after net, so the TD instantiations see the parameter layout they always had)
    unsigned long long* abs_acc;  // the sums of |fx|, next to acc
    double* err_sum;              // E
    double* abs_err_sum;          // A
    // STAGED only (after the TC fields, so the unstaged instantiations see the parameter layout they always had)
    NtStages stages;
    // LAMBDA only (after the stages, for the same reason)
    float c[G2048_NTUPLE_MAX_HORIZON];  // c_0 .. c_{h-1}, 0 beyond
    uint32_t horizon;                   // h
    u64* hist_after;                    // [h * n], slot-major
    float* hist_delta;                  // [h * n], slot-major
    // CAROUSEL only (after the lambda fields, for the same reason)
    uint32_t* start_stage;  // [n]
    u64* pool;              // [(S - 1) * n], stage-major
    u64* pending;           // [n], in the scratch: the board with which the env entered a stage this step, or 0
};

// fx(d) = rint(clamp(d, -2^24, 2^24) * 4096) as int64, to nearest even (the multiply by a power of two is exact)
__device__ __forceinline__ long long nt_fx(float d) {
    return __float2ll_rn(fminf(fmaxf(d, -NT_FX_CLAMP), NT_FX_CLAMP) * NT_FX_ONE);
}

// the lanes with `first` append their entry i to the list: one list atomic per warp (all 32 lanes call this)
__device__ __forceinline__ void nt_append(bool first, uint32_t i, uint32_t* list, uint32_t* list_len, unsigned lane) {
    const unsigned firsts = __ballot_sync(0xFFFFFFFFu, first);
    if (firsts) {
        uint32_t pos = 0u;
        if (lane == 0u) pos = atomicAdd(list_len, (uint32_t)__popc((int)firsts));
        pos = __shfl_sync(0xFFFFFFFFu, pos, 0);
        if (first) list[pos + (uint32_t)__popc((int)(firsts & ((1u << lane) - 1u)))] = i;
    }
}

template <int MODE, bool TC, bool STAGED, bool LAMBDA, bool CAROUSEL>
__global__ void __launch_bounds__(NT_THREADS, 1) ntuple_td_kernel(const __grid_constant__ NtTdArgs a) {
    static_assert(!CAROUSEL || STAGED, "carousel shaping needs stages");
    extern __shared__ __align__(16) uint8_t smem_raw[];
    __shared__ unsigned long long s_stats[G2048_PLAY_STATS_WORDS];
    __shared__ long long s_fx[NT_THREADS];
    __shared__ unsigned long long s_acc0[G2048_NTUPLE_MAX_PLACEMENTS];
    __shared__ unsigned s_cnt0[G2048_NTUPLE_MAX_PLACEMENTS];
    __shared__ unsigned long long s_abs0[TC ? G2048_NTUPLE_MAX_PLACEMENTS : 1];
    play3_copy_row_tables<NT_THREADS>(smem_raw);
    for (int i = threadIdx.x; i < G2048_PLAY_STATS_WORDS; i += NT_THREADS) s_stats[i] = 0ull;
    if (threadIdx.x < G2048_NTUPLE_MAX_PLACEMENTS) {
        s_acc0[threadIdx.x] = 0ull;
        s_cnt0[threadIdx.x] = 0u;
        if constexpr (TC) s_abs0[threadIdx.x] = 0ull;
    }
    __syncthreads();

    cg::grid_group grid = cg::this_grid();
    XmCtx c;
    c.T = nullptr;
    c.w = 1.0f;
    c.s_left = reinterpret_cast<const uint16_t*>(smem_raw);
    c.s_flags = smem_raw + 65536 * 2;
    const unsigned lane = threadIdx.x & 31u;
    long long* warp_fx = s_fx + (threadIdx.x & ~31u);
    const uint32_t stride = gridDim.x * NT_THREADS;
    const uint32_t P = a.net.n_placements;
#ifdef G2048_NTUPLE_PHASES
    unsigned long long t_mark = nt_clock(), ns_acc = 0ull, ns_apply = 0ull, listed = 0ull;
#endif

    for (int64_t t = 0; t < a.n_steps; ++t) {
        const uint2 sub = __ldg(&a.subs[t]);
        uint32_t* list_len = a.list_len + (t & 1);
        // ---- accumulate: the whole CTA walks the envs together, so every warp is converged at the matches
        for (uint32_t base = blockIdx.x * NT_THREADS; base < a.n; base += stride) {
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
            u64 cand[5];
            uint32_t rew[4];
#pragma unroll
            for (int act = 0; act < 4; ++act) {
                u64 nbT;
                xm_move<true>(c, s, sT, act, cand[act], nbT, rew[act]);
            }
            cand[4] = aft;
            float v[5];
            uint32_t aft_base = 0u;  // the previous afterstate's stage base
            if constexpr (STAGED) {
                uint32_t base[5];
#pragma unroll
                for (int j = 0; j < 5; ++j) base[j] = nt_stage_base(a.stages, cand[j]);
                nt_values_at<true, 5>(a.net, cand, base, v);
                aft_base = base[4];
            } else {
                nt_values<true, 5>(a.net, cand, v);
            }
            float target = 0.0f;
            u64 best = 0ull;
            uint32_t best_r = 0u;
            bool any = false;
#pragma unroll
            for (int act = 0; act < 4; ++act) {
                if ((lm >> act) & 1u) {
                    const float q = (float)rew[act] + v[act];
                    if (!any || q > target) {
                        target = q;
                        best = cand[act];
                        best_r = rew[act];
                    }
                    any = true;
                }
            }
            const bool update = aft != 0ull;  // inactive lanes hold after = 0
            // the placement loop over board x (stage base xbase) of the lanes with upd, whose fx are in warp_fx
            auto accumulate = [&](bool upd, u64 x, uint32_t xbase) {
#pragma unroll 1
                for (uint32_t p = 0; p < P; ++p) {
                    const uint32_t i = xbase + nt_entry(a.net.pl[p], x);
                    const unsigned group = __match_any_sync(0xFFFFFFFFu, upd ? i : 0xFFFFFFFFu);  // i < 2^28
                    bool first = false;
                    if (upd && lane == (unsigned)(__ffs((int)group) - 1)) {
                        long long sum = 0, abs_sum = 0;
                        for (unsigned m = group; m; m &= m - 1u) {
                            const long long fx = warp_fx[__ffs((int)m) - 1];
                            sum += fx;
                            if constexpr (TC) abs_sum += fx < 0 ? -fx : fx;
                        }
                        const unsigned count = (unsigned)__popc((int)group);
                        // index 0 of placement p in stage 0.  The per-CTA sums are flushed to off_p, so this relies
                        // on no other entry of p equalling off_p: an entry of stage s >= 1 is at least stride + off_p
                        // with stride >= 1, so the later stages' index 0 goes through the global atomics.
                        if (i == a.net.pl[p].offset) {
                            atomicAdd(&s_acc0[p], (unsigned long long)sum);
                            if constexpr (TC) atomicAdd(&s_abs0[p], (unsigned long long)abs_sum);
                            atomicAdd(&s_cnt0[p], count);
                        } else {
                            atomicAdd(&a.acc[i], (unsigned long long)sum);
                            if constexpr (TC) atomicAdd(&a.abs_acc[i], (unsigned long long)abs_sum);
                            first = atomicAdd(&a.cnt[i], count) == 0u;
                        }
                    }
                    nt_append(first, i, a.list, list_len, lane);
                }
            };
            if constexpr (LAMBDA) {
                // L = length; delta_L goes to slot (L - 1) mod h.  Released: x_m for m0 <= m < m0 + n_rel.  An env
                // with an afterstate but L outside [1, 2^31) is outside the contract and stores and releases nothing.
                const int h = (int)a.horizon, L = (int)length;
                const float dL = target - v[4];
                int m0 = L - h + 1, n_rel = 0;
                if (update && L >= 1) {
                    a.hist_delta[(size_t)((L - 1) % h) * a.n + e] = dL;
                    if (lm == 0u) {
                        m0 = m0 > 1 ? m0 : 1;
                        n_rel = L - m0 + 1;
                    } else {
                        n_rel = L >= h ? 1 : 0;
                    }
                }
                // d[k] = delta_{m0 + k} while m0 + k <= L (the fresh delta_L in place of its slot)
                float d[G2048_NTUPLE_MAX_HORIZON];
                const int slot0 = n_rel ? (m0 - 1) % h : 0;
#pragma unroll
                for (int k = 0; k < G2048_NTUPLE_MAX_HORIZON; ++k) {
                    d[k] = 0.0f;
                    int slot = slot0 + k;
                    slot = slot >= h ? slot - h : slot;
                    if (n_rel && m0 + k < L) d[k] = a.hist_delta[(size_t)slot * a.n + e];
                    if (n_rel && m0 + k == L) d[k] = dL;
                }
                const uint32_t rounds = __reduce_max_sync(0xFFFFFFFFu, (unsigned)n_rel);
                int slot = slot0;
#pragma unroll 1
                for (uint32_t r = 0; r < rounds; ++r) {
                    const int m = m0 + (int)r;
                    const bool upd = (int)r < n_rel;
                    u64 x = 0ull;
                    float em = d[0];
                    if (upd) {
                        x = a.hist_after[(size_t)slot * a.n + e];
#pragma unroll
                        for (int k = 1; k < G2048_NTUPLE_MAX_HORIZON; ++k)
                            if (m + k <= L) em = __fadd_rn(em, __fmul_rn(a.c[k], d[k]));
                    }
#pragma unroll
                    for (int k = 0; k + 1 < G2048_NTUPLE_MAX_HORIZON; ++k) d[k] = d[k + 1];  // the next release's window
                    slot = slot + 1 == h ? 0 : slot + 1;
                    warp_fx[lane] = upd ? nt_fx(em) : 0ll;
                    __syncwarp();
                    accumulate(upd, x, STAGED && upd ? nt_stage_base(a.stages, x) : 0u);
                    __syncwarp();  // warp_fx is rewritten by the next round
                }
            } else {
                warp_fx[lane] = update ? nt_fx(target - v[4]) : 0ll;
                __syncwarp();
                accumulate(update, aft, aft_base);
                __syncwarp();  // warp_fx is rewritten by the next env
            }

            if (active) {
                const Key k = split_at<MODE>(Key{sub.x, sub.y}, a.n, e);
                if (lm == 0u) {  // the episode ends here: count it and start the next one
                    bool opening = true;  // the episode began at the opening (always, without the carousel)
                    u64 next = 0ull;      // the restart board; 0: init(k)
                    uint32_t next_stage = 0u;
                    if constexpr (CAROUSEL) {
                        // l = c + 1, or 0 when c + 1 >= S (the wrap); S - 1 is the stage of exponent 15
                        const uint32_t c0 = a.start_stage[e];
                        const uint32_t l = c0 + 1u <= (uint32_t)(a.stages.stage_of >> 60) ? c0 + 1u : 0u;
                        opening = c0 == 0u;
                        if (l) {
                            Key k1, k2;
                            split2<MODE>(k, k1, k2);
                            const uint32_t j = (uint32_t)(((u64)bits_scalar<MODE>(k1) * a.n) >> 32);
                            next = a.pool[(size_t)(l - 1u) * a.n + j];
                            next_stage = next ? l : 0u;
                        }
                        a.start_stage[e] = next_stage;
                    }
                    if (opening) {
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
                    } else {  // an episode that began from a pool board
                        atomicAdd(&s_stats[12], 1ull);
                        atomicAdd(&s_stats[13], (unsigned long long)length);
                    }
                    a.boards[e] = next ? next : env_init<MODE>(k).board;
                    a.after[e] = 0ull;
                    a.scores[e] = 0u;
                    a.lengths[e] = 0u;
                } else {
                    Key k1, k2;
                    split2<MODE>(k, k1, k2);
                    const u64 spawned = spawn_tile(best, bits_scalar<MODE>(k1), bits_scalar<MODE>(k2));
                    a.boards[e] = spawned;
                    // the stage rises by at most 1 a move; the apply phase commits the board to the pool
                    if constexpr (CAROUSEL)
                        if (nt_stage(a.stages, spawned) > nt_stage(a.stages, s)) a.pending[e] = spawned;
                    a.after[e] = best;
                    if constexpr (LAMBDA) a.hist_after[(size_t)(length % a.horizon) * a.n + e] = best;  // x_{L+1}
                    a.scores[e] = score + best_r;
                    a.lengths[e] = length + 1u;
                }
            }
        }
        __syncthreads();
        if (threadIdx.x < P && s_cnt0[threadIdx.x]) {  // the CTA's index-0 sums, one placement per thread
            const uint32_t i = a.net.pl[threadIdx.x].offset;
            atomicAdd(&a.acc[i], s_acc0[threadIdx.x]);
            if constexpr (TC) {
                atomicAdd(&a.abs_acc[i], s_abs0[threadIdx.x]);
                s_abs0[threadIdx.x] = 0ull;
            }
            if (atomicAdd(&a.cnt[i], s_cnt0[threadIdx.x]) == 0u) a.list[atomicAdd(list_len, 1u)] = i;
            s_acc0[threadIdx.x] = 0ull;
            s_cnt0[threadIdx.x] = 0u;
        }
        grid.sync();
#ifdef G2048_NTUPLE_PHASES
        {
            const unsigned long long now = nt_clock();
            ns_acc += now - t_mark;
            t_mark = now;
            listed += __ldcg(list_len);
        }
#endif
        // ---- apply: every listed entry moves by alpha times the mean of its errors (TC: times beta, from E and A
        // before this step, which then take the step's sums); its sums and its list slot go back to zero, and the
        // other list's length is cleared for the next step
        const uint32_t len = __ldcg(list_len);
        for (uint32_t j = blockIdx.x * NT_THREADS + threadIdx.x; j < len; j += stride) {
            const uint32_t i = __ldcg(&a.list[j]);
            const uint32_t count = __ldcg(&a.cnt[i]);
            const long long sum = (long long)__ldcg(&a.acc[i]);
            if constexpr (TC) {
                const long long abs_sum = (long long)__ldcg(&a.abs_acc[i]);
                const double m = (double)sum / (4096.0 * (double)count);
                const double e = a.err_sum[i], A = a.abs_err_sum[i];
                const double beta = A > 0.0 ? fmin(fabs(e) / A, 1.0) : 1.0;
                a.W[i] = a.W[i] + a.alpha * (float)(beta * m);
                a.err_sum[i] = e + (double)sum / 4096.0;
                a.abs_err_sum[i] = A + (double)abs_sum / 4096.0;
                a.abs_acc[i] = 0ull;
            } else {
                const float mean = (float)((double)sum / (4096.0 * (double)count));
                a.W[i] = a.W[i] + a.alpha * mean;
            }
            a.acc[i] = 0ull;
            a.cnt[i] = 0u;
            a.list[j] = 0u;
        }
        if constexpr (CAROUSEL) {  // the envs this thread stepped: their stage entries go to the pool
            for (uint32_t e = blockIdx.x * NT_THREADS + threadIdx.x; e < a.n; e += stride) {
                const u64 b = a.pending[e];
                if (b) {
                    a.pool[(size_t)(nt_stage(a.stages, b) - 1u) * a.n + e] = b;
                    a.pending[e] = 0ull;
                }
            }
        }
        if (blockIdx.x == 0 && threadIdx.x == 0) a.list_len[(t + 1) & 1] = 0u;
        grid.sync();
#ifdef G2048_NTUPLE_PHASES
        {
            const unsigned long long now = nt_clock();
            ns_apply += now - t_mark;
            t_mark = now;
        }
#endif
    }
#ifdef G2048_NTUPLE_PHASES
    if (blockIdx.x == 0 && threadIdx.x == 0 && a.stats) {
        atomicAdd(&a.stats[8], ns_acc);
        atomicAdd(&a.stats[9], ns_apply);
        atomicAdd(&a.stats[10], listed);
    }
#endif
    if (blockIdx.x == 0 && threadIdx.x == 0 && a.n_steps > 0) a.list_len[(a.n_steps - 1) & 1] = 0u;

    if (a.stats) {
        __syncthreads();
        for (int i = threadIdx.x; i < G2048_PLAY_STATS_WORDS; i += NT_THREADS) {
            const unsigned long long v = s_stats[i];
            if (v) {
                if (i == 5) atomicMax(&a.stats[i], v);
                else atomicAdd(&a.stats[i], v);
            }
        }
    }
}

// this translation unit's copy of the row tables
__global__ void build_ntuple_row_tables_kernel() {
    const uint32_t row = blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= 65536u) return;
    build_row_table_entry(row);
}

// who: the entry point's name, which prefixes every message
template <int MODE, bool TC, bool STAGED, bool LAMBDA, bool CAROUSEL>
static int launch_ntuple_td(const char* who, const NtTdArgs& args, cudaStream_t st) {
    auto kernel = ntuple_td_kernel<MODE, TC, STAGED, LAMBDA, CAROUSEL>;
    char msg[128];
    auto what = [&](const char* s) {
        snprintf(msg, sizeof(msg), "%s%s%s", who, *s ? ": " : "", s);
        return msg;
    };
    static bool configured_on[64] = {false};
    bool* configured = device_once_flag(configured_on);
    if (!configured) return fail_arg("no CUDA device");
    int dev = 0;
    int rc = check_cuda(cudaGetDevice(&dev), what("device"));
    if (rc) return rc;
    if (!*configured) {
        int coop = 0;
        rc = check_cuda(cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, dev), what("device attribute"));
        if (rc) return rc;
        if (!coop) return fail_arg(what("the device does not support cooperative launches"));
        rc = check_cuda(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, NT_SMEM_BYTES),
                        what("shared memory attribute"));
        if (rc) return rc;
        *configured = true;
    }
    rc = ensure_row_tables_with<build_ntuple_row_tables_kernel>(st);
    if (rc) return rc;
    int per_sm = 0;
    rc = check_cuda(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, NT_THREADS, NT_SMEM_BYTES),
                    what("occupancy"));
    if (rc) return rc;
    const int sms = sm_count();
    if (sms <= 0 || per_sm <= 0) return fail_arg(what("the kernel does not fit on this device"));
    const int64_t needed = ((int64_t)args.n + NT_THREADS - 1) / NT_THREADS;
    const int64_t resident = (int64_t)per_sm * sms;
    const unsigned grid = (unsigned)(needed < resident ? needed : resident);
    void* params[] = {const_cast<NtTdArgs*>(&args)};
    return check_cuda(cudaLaunchCooperativeKernel((const void*)kernel, dim3(grid), dim3(NT_THREADS), params,
                                                  (size_t)NT_SMEM_BYTES, st),
                      what(""));
}

}  // namespace g2048

using namespace g2048;

namespace {

int nt_fail(const char* who, const char* what) {
    char msg[160];
    snprintf(msg, sizeof(msg), "%s: %s", who, what);
    return fail_arg(msg);
}

int64_t nt_scratch_bytes(int64_t n, int n_placements, int64_t n_weights, bool tc) {
    if (n < 1 || n > (1ll << 20) || n_placements < 1 || n_placements > G2048_NTUPLE_MAX_PLACEMENTS || n_weights < 1 ||
        n_weights > G2048_NTUPLE_MAX_WEIGHTS)
        return -1;
    return nt_scratch_layout(n, n_placements, n_weights, tc).bytes;
}

template <bool TC, bool STAGED, bool LAMBDA, bool CAROUSEL = false>
int nt_launch(const char* who, int rng_mode, const NtTdArgs& args, cudaStream_t st) {
    if (rng_mode == G2048_RNG_PARTITIONABLE)
        return launch_ntuple_td<G2048_RNG_PARTITIONABLE, TC, STAGED, LAMBDA, CAROUSEL>(who, args, st);
    return launch_ntuple_td<G2048_RNG_ORIGINAL, TC, STAGED, LAMBDA, CAROUSEL>(who, args, st);
}

// the window of the lambda entry points
struct NtLambda {
    float lambda;
    int horizon;
    uint64_t* hist_after;
    float* hist_delta;
};

// the arrays of the carousel entry points
struct NtCarousel {
    uint32_t* start_stage;
    uint64_t* stage_pool;
};

// g2048_ntuple_td_train (tc = false; E and A unused) and g2048_ntuple_tc_train, their staged forms (h_stages not
// NULL; staged = false passes NULL), their lambda forms (lam not NULL; staged when h_stages is not NULL) and their
// carousel forms (lam and car not NULL, staged): the checks, then one launch
int nt_train(const char* who, bool tc, bool staged, uint64_t* d_boards, uint64_t* d_after, uint32_t* d_scores,
             uint32_t* d_lengths, int64_t n, const G2048TuplePlacement* h_placements, int n_placements,
             const G2048TupleStages* h_stages, float* d_weights, int64_t n_weights, double* d_err_sum,
             double* d_abs_err_sum, float alpha, const uint32_t* d_subs, int64_t n_steps, int rng_mode,
             void* d_scratch, uint64_t* d_stats, void* stream, const NtLambda* lam = nullptr,
             const NtCarousel* car = nullptr) {
    if (!(n >= 1 && n <= (1ll << 20))) return nt_fail(who, "n must be in [1, 2^20]");
    if (!(n_steps >= 0)) return nt_fail(who, "n_steps must be >= 0");
    if (!(alpha >= 0.0f && alpha <= 3.402823466e38f)) return nt_fail(who, "alpha must be finite and >= 0");
    if (!(rng_mode == G2048_RNG_ORIGINAL || rng_mode == G2048_RNG_PARTITIONABLE)) return nt_fail(who, "rng_mode");
    char invalid[64];
    snprintf(invalid, sizeof(invalid), "%s: invalid network", who);
    int rc = ntuple_check(h_placements, n_placements, n_weights, invalid);
    if (rc) return rc;
    if (staged) {
        snprintf(invalid, sizeof(invalid), "%s: invalid stages", who);
        rc = ntuple_stages_check(h_stages, h_placements, n_placements, n_weights, invalid);
        if (rc) return rc;
    }
    if (car && !(staged && h_stages->n_thresholds >= 1)) return nt_fail(who, "carousel shaping needs at least 2 stages");
    if (!(d_boards && d_after && d_scores && d_lengths && d_weights && d_scratch)) return nt_fail(who, "pointers");
    if (!(n_steps == 0 || d_subs)) return nt_fail(who, "pointers");
    if (tc && !(d_err_sum && d_abs_err_sum)) return nt_fail(who, "pointers");
    if (!(((uintptr_t)d_boards & 7u) == 0 && ((uintptr_t)d_after & 7u) == 0 && ((uintptr_t)d_scratch & 7u) == 0 &&
          ((uintptr_t)d_subs & 7u) == 0 && ((uintptr_t)d_stats & 7u) == 0))
        return nt_fail(who, "d_boards, d_after, d_subs, d_scratch and d_stats must be 8-byte aligned");
    if (tc && !(((uintptr_t)d_err_sum & 7u) == 0 && ((uintptr_t)d_abs_err_sum & 7u) == 0))
        return nt_fail(who, "d_err_sum and d_abs_err_sum must be 8-byte aligned");
    if (!(((uintptr_t)d_scores & 3u) == 0 && ((uintptr_t)d_lengths & 3u) == 0 && ((uintptr_t)d_weights & 3u) == 0))
        return nt_fail(who, "d_scores, d_lengths and d_weights must be 4-byte aligned");
    if (lam) {
        if (!(lam->lambda >= 0.0f && lam->lambda <= 1.0f)) return nt_fail(who, "lambda must be finite and in [0, 1]");
        if (!(lam->horizon >= 1 && lam->horizon <= G2048_NTUPLE_MAX_HORIZON))
            return nt_fail(who, "horizon must be in [1, G2048_NTUPLE_MAX_HORIZON]");
        if (n * lam->horizon > (1ll << 20)) return nt_fail(who, "n * horizon must be <= 2^20");
        // the carousel forms run h = 1 without the window, so they take NULL rings there
        if (!(lam->hist_after && lam->hist_delta) && !(car && lam->horizon == 1)) return nt_fail(who, "pointers");
        if (!(((uintptr_t)lam->hist_after & 7u) == 0 && ((uintptr_t)lam->hist_delta & 3u) == 0))
            return nt_fail(who, "d_hist_after must be 8-byte and d_hist_delta 4-byte aligned");
    }
    if (car) {
        if (!(car->start_stage && car->stage_pool)) return nt_fail(who, "pointers");
        if (!(((uintptr_t)car->start_stage & 3u) == 0 && ((uintptr_t)car->stage_pool & 7u) == 0))
            return nt_fail(who, "d_start_stage must be 4-byte and d_stage_pool 8-byte aligned");
    }
    if (n_steps == 0) return G2048_OK;
    const NtScratch lay = nt_scratch_layout(lam ? n * lam->horizon : n, n_placements, n_weights, tc);
    NtTdArgs args;
    args.boards = (u64*)d_boards;
    args.after = (u64*)d_after;
    args.scores = d_scores;
    args.lengths = d_lengths;
    args.n = (uint32_t)n;
    args.W = d_weights;
    args.alpha = alpha;
    args.subs = (const uint2*)d_subs;
    args.n_steps = n_steps;
    args.acc = (unsigned long long*)d_scratch;
    args.cnt = (uint32_t*)((uint8_t*)d_scratch + lay.cnt_off);
    args.list = (uint32_t*)((uint8_t*)d_scratch + lay.list_off);
    args.list_len = (uint32_t*)((uint8_t*)d_scratch + lay.len_off);
    args.stats = (unsigned long long*)d_stats;
    ntuple_net(args.net, h_placements, n_placements, d_weights);
    args.abs_acc = tc ? (unsigned long long*)((uint8_t*)d_scratch + lay.abs_off) : nullptr;
    args.err_sum = tc ? d_err_sum : nullptr;
    args.abs_err_sum = tc ? d_abs_err_sum : nullptr;
    args.stages = staged ? ntuple_stages(*h_stages) : NtStages{0ull, 0u};
    // c_k by repeated multiplication in double (no pow), so that the host-side restatements get the same bits
    double d = 1.0;
    for (int k = 0; k < G2048_NTUPLE_MAX_HORIZON; ++k) {
        args.c[k] = lam && k < lam->horizon ? (float)d : 0.0f;
        if (lam) d *= (double)lam->lambda;
    }
    args.horizon = lam ? (uint32_t)lam->horizon : 0u;
    args.hist_after = lam ? (u64*)lam->hist_after : nullptr;
    args.hist_delta = lam ? lam->hist_delta : nullptr;
    args.start_stage = car ? car->start_stage : nullptr;
    args.pool = car ? (u64*)car->stage_pool : nullptr;
    args.pending = car ? (u64*)((uint8_t*)d_scratch + lay.bytes) : nullptr;
    cudaStream_t st = (cudaStream_t)stream;
    if (car) {  // h = 1 is the staged TD(0) / TC step, without the ring traffic
        if (lam->horizon > 1) return tc ? nt_launch<true, true, true, true>(who, rng_mode, args, st)
                                        : nt_launch<false, true, true, true>(who, rng_mode, args, st);
        return tc ? nt_launch<true, true, false, true>(who, rng_mode, args, st)
                  : nt_launch<false, true, false, true>(who, rng_mode, args, st);
    }
    if (lam) {
        if (staged) return tc ? nt_launch<true, true, true>(who, rng_mode, args, st)
                              : nt_launch<false, true, true>(who, rng_mode, args, st);
        return tc ? nt_launch<true, false, true>(who, rng_mode, args, st)
                  : nt_launch<false, false, true>(who, rng_mode, args, st);
    }
    if (staged) return tc ? nt_launch<true, true, false>(who, rng_mode, args, st)
                          : nt_launch<false, true, false>(who, rng_mode, args, st);
    return tc ? nt_launch<true, false, false>(who, rng_mode, args, st) : nt_launch<false, false, false>(who, rng_mode, args, st);
}

}  // namespace

extern "C" int64_t g2048_ntuple_td_scratch_bytes(int64_t n, int n_placements, int64_t n_weights) {
    return nt_scratch_bytes(n, n_placements, n_weights, false);
}

extern "C" int g2048_ntuple_td_train(uint64_t* d_boards, uint64_t* d_after, uint32_t* d_scores, uint32_t* d_lengths,
                                     int64_t n, const G2048TuplePlacement* h_placements, int n_placements,
                                     float* d_weights, int64_t n_weights, float alpha, const uint32_t* d_subs,
                                     int64_t n_steps, int rng_mode, void* d_scratch, uint64_t* d_stats, void* stream) {
    return nt_train("ntuple_td_train", false, false, d_boards, d_after, d_scores, d_lengths, n, h_placements,
                    n_placements, nullptr, d_weights, n_weights, nullptr, nullptr, alpha, d_subs, n_steps, rng_mode,
                    d_scratch, d_stats, stream);
}

extern "C" int64_t g2048_ntuple_tc_scratch_bytes(int64_t n, int n_placements, int64_t n_weights) {
    return nt_scratch_bytes(n, n_placements, n_weights, true);
}

extern "C" int g2048_ntuple_tc_train(uint64_t* d_boards, uint64_t* d_after, uint32_t* d_scores, uint32_t* d_lengths,
                                     int64_t n, const G2048TuplePlacement* h_placements, int n_placements,
                                     float* d_weights, int64_t n_weights, double* d_err_sum, double* d_abs_err_sum,
                                     float alpha, const uint32_t* d_subs, int64_t n_steps, int rng_mode,
                                     void* d_scratch, uint64_t* d_stats, void* stream) {
    return nt_train("ntuple_tc_train", true, false, d_boards, d_after, d_scores, d_lengths, n, h_placements,
                    n_placements, nullptr, d_weights, n_weights, d_err_sum, d_abs_err_sum, alpha, d_subs, n_steps,
                    rng_mode, d_scratch, d_stats, stream);
}

extern "C" int g2048_ntuple_staged_td_train(uint64_t* d_boards, uint64_t* d_after, uint32_t* d_scores,
                                            uint32_t* d_lengths, int64_t n, const G2048TuplePlacement* h_placements,
                                            int n_placements, const G2048TupleStages* h_stages, float* d_weights,
                                            int64_t n_weights, float alpha, const uint32_t* d_subs, int64_t n_steps,
                                            int rng_mode, void* d_scratch, uint64_t* d_stats, void* stream) {
    return nt_train("ntuple_staged_td_train", false, true, d_boards, d_after, d_scores, d_lengths, n, h_placements,
                    n_placements, h_stages, d_weights, n_weights, nullptr, nullptr, alpha, d_subs, n_steps, rng_mode,
                    d_scratch, d_stats, stream);
}

extern "C" int g2048_ntuple_staged_tc_train(uint64_t* d_boards, uint64_t* d_after, uint32_t* d_scores,
                                            uint32_t* d_lengths, int64_t n, const G2048TuplePlacement* h_placements,
                                            int n_placements, const G2048TupleStages* h_stages, float* d_weights,
                                            int64_t n_weights, double* d_err_sum, double* d_abs_err_sum, float alpha,
                                            const uint32_t* d_subs, int64_t n_steps, int rng_mode, void* d_scratch,
                                            uint64_t* d_stats, void* stream) {
    return nt_train("ntuple_staged_tc_train", true, true, d_boards, d_after, d_scores, d_lengths, n, h_placements,
                    n_placements, h_stages, d_weights, n_weights, d_err_sum, d_abs_err_sum, alpha, d_subs, n_steps,
                    rng_mode, d_scratch, d_stats, stream);
}

extern "C" int g2048_ntuple_lambda_td_train(uint64_t* d_boards, uint64_t* d_after, uint32_t* d_scores,
                                            uint32_t* d_lengths, int64_t n, const G2048TuplePlacement* h_placements,
                                            int n_placements, const G2048TupleStages* h_stages, float* d_weights,
                                            int64_t n_weights, float alpha, float lambda, int horizon,
                                            uint64_t* d_hist_after, float* d_hist_delta, const uint32_t* d_subs,
                                            int64_t n_steps, int rng_mode, void* d_scratch, uint64_t* d_stats,
                                            void* stream) {
    const NtLambda lam{lambda, horizon, d_hist_after, d_hist_delta};
    return nt_train("ntuple_lambda_td_train", false, h_stages != nullptr, d_boards, d_after, d_scores, d_lengths, n,
                    h_placements, n_placements, h_stages, d_weights, n_weights, nullptr, nullptr, alpha, d_subs,
                    n_steps, rng_mode, d_scratch, d_stats, stream, &lam);
}

extern "C" int g2048_ntuple_lambda_tc_train(uint64_t* d_boards, uint64_t* d_after, uint32_t* d_scores,
                                            uint32_t* d_lengths, int64_t n, const G2048TuplePlacement* h_placements,
                                            int n_placements, const G2048TupleStages* h_stages, float* d_weights,
                                            int64_t n_weights, double* d_err_sum, double* d_abs_err_sum, float alpha,
                                            float lambda, int horizon, uint64_t* d_hist_after, float* d_hist_delta,
                                            const uint32_t* d_subs, int64_t n_steps, int rng_mode, void* d_scratch,
                                            uint64_t* d_stats, void* stream) {
    const NtLambda lam{lambda, horizon, d_hist_after, d_hist_delta};
    return nt_train("ntuple_lambda_tc_train", true, h_stages != nullptr, d_boards, d_after, d_scores, d_lengths, n,
                    h_placements, n_placements, h_stages, d_weights, n_weights, d_err_sum, d_abs_err_sum, alpha,
                    d_subs, n_steps, rng_mode, d_scratch, d_stats, stream, &lam);
}

extern "C" int64_t g2048_ntuple_carousel_scratch_bytes(int64_t n, int horizon, int n_placements, int64_t n_weights,
                                                       int tc) {
    if (!(horizon >= 1 && horizon <= G2048_NTUPLE_MAX_HORIZON) || n < 1 || n * horizon > (1ll << 20)) return -1;
    const int64_t bytes = nt_scratch_bytes(n * horizon, n_placements, n_weights, tc != 0);
    return bytes < 0 ? -1 : bytes + 8 * n;  // the pending words
}

extern "C" int g2048_ntuple_carousel_td_train(uint64_t* d_boards, uint64_t* d_after, uint32_t* d_scores,
                                              uint32_t* d_lengths, int64_t n, const G2048TuplePlacement* h_placements,
                                              int n_placements, const G2048TupleStages* h_stages, float* d_weights,
                                              int64_t n_weights, float alpha, float lambda, int horizon,
                                              uint64_t* d_hist_after, float* d_hist_delta, uint32_t* d_start_stage,
                                              uint64_t* d_stage_pool, const uint32_t* d_subs, int64_t n_steps,
                                              int rng_mode, void* d_scratch, uint64_t* d_stats, void* stream) {
    const NtLambda lam{lambda, horizon, d_hist_after, d_hist_delta};
    const NtCarousel car{d_start_stage, d_stage_pool};
    return nt_train("ntuple_carousel_td_train", false, h_stages != nullptr, d_boards, d_after, d_scores, d_lengths, n,
                    h_placements, n_placements, h_stages, d_weights, n_weights, nullptr, nullptr, alpha, d_subs,
                    n_steps, rng_mode, d_scratch, d_stats, stream, &lam, &car);
}

extern "C" int g2048_ntuple_carousel_tc_train(uint64_t* d_boards, uint64_t* d_after, uint32_t* d_scores,
                                              uint32_t* d_lengths, int64_t n, const G2048TuplePlacement* h_placements,
                                              int n_placements, const G2048TupleStages* h_stages, float* d_weights,
                                              int64_t n_weights, double* d_err_sum, double* d_abs_err_sum, float alpha,
                                              float lambda, int horizon, uint64_t* d_hist_after, float* d_hist_delta,
                                              uint32_t* d_start_stage, uint64_t* d_stage_pool, const uint32_t* d_subs,
                                              int64_t n_steps, int rng_mode, void* d_scratch, uint64_t* d_stats,
                                              void* stream) {
    const NtLambda lam{lambda, horizon, d_hist_after, d_hist_delta};
    const NtCarousel car{d_start_stage, d_stage_pool};
    return nt_train("ntuple_carousel_tc_train", true, h_stages != nullptr, d_boards, d_after, d_scores, d_lengths, n,
                    h_placements, n_placements, h_stages, d_weights, n_weights, d_err_sum, d_abs_err_sum, alpha,
                    d_subs, n_steps, rng_mode, d_scratch, d_stats, stream, &lam, &car);
}
