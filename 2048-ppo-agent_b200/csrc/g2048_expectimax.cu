// Depth-limited expectimax values of caller-given boards over a caller-supplied row heuristic
// (g2048_expectimax_values, include/g2048.h).
//
// The tree, with every sum in a fixed order so that the values are bit-exact:
//   H(b)      = T[row0] + .. + T[row3] + T[col0] + .. + T[col3]                       (left to right)
//   Q_1(b, a) = w r + H(b_a)            Q_k(b, a) = w r + C_{k-1}(b_a)   (b_a, r) = move(b, a), a legal
//   C_k(s)    = (sum over the empty cells c of s, in increasing index, of 0.9 V_k(s + 2@c) + 0.1 V_k(s + 4@c)) / n_empty
//   V_k(b)    = max over the legal a of Q_k(b, a) (the first legal action's value, replaced by every strictly larger
//               one in action order), 0 without a legal action
//
// Mapping: a work item is one (board, first action) pair, played by one warp.  The warp lists the children of the
// root chance node's afterstate together with their first move, j = (empty cell k, spawn v, action a1), and each lane
// evaluates Q_{d-1}(child, a1) for j = lane, lane + 32, ..., depth-first in registers.  The results go into the warp's
// shared-memory slots, indexed by j; lanes then take the max over a1 per child and lane 0 folds the children in cell
// order.  Every reduction runs in the order of the contract, whatever lane computed its terms, so the values do not
// depend on the mapping.  Subtree sizes differ by 100x from board to board, so the warps of a CTA claim items through a
// shared-memory counter, and the CTAs of the persistent grid take interleaved items (item = blockIdx + k * gridDim):
// no global scratch and no inter-CTA hand-over.
#include "g2048_ntuple.cuh"
#include "g2048_xm.cuh"

namespace g2048 {

// Moves and legal masks come from the shared-memory row tables of g2048_play3.cuh (192 KiB: one CTA per SM, and a small
// L1 for T).  The register SWAR moves of g2048_board.cuh leave shared memory empty and all of L1 for T, but were 1.8x
// slower at depth 3 and 2.2x at depth 4 on one B200, and 8 % faster only at depth 2, where a call over 4 096 boards
// takes 24 us (profiles/README.md, round 6).
constexpr int XM_THREADS = 768;
constexpr int XM_WARPS = XM_THREADS / 32;
constexpr int XM_SLOTS = 15 * 8;  // an afterstate has at most 15 empty cells: (cell, spawn, action) children
constexpr int XM_VALS = 15 * 2;
constexpr int XM_SMEM_BYTES = PLAY3_TABLE_BYTES + XM_WARPS * (XM_SLOTS + XM_VALS) * 4;

struct XmCount {
    unsigned long long leaves, chance;
};

template <int K, bool REWARD, class Leaf>
__device__ __forceinline__ float xm_chance(const XmCtx& c, const typename Leaf::Param& leaf, u64 s, u64 sT, XmCount& n);

// Q_K(b, a) for a legal a
template <int K, bool REWARD, class Leaf>
__device__ __forceinline__ float xm_q(const XmCtx& c, const typename Leaf::Param& leaf, u64 b, u64 bT, int a, XmCount& n) {
    u64 nb, nbT;
    uint32_t r;
    xm_move<REWARD>(c, b, bT, a, nb, nbT, r);
    float tail;
    if constexpr (K == 1) {
        ++n.leaves;
        tail = Leaf::value(c, leaf, nb, nbT);
    } else {
        tail = xm_chance<K - 1, REWARD, Leaf>(c, leaf, nb, nbT, n);
    }
    // w r with r = 0 when w == 0: w * r = w exactly (w = +0 or -0, r >= 0), so the reward-free form adds w itself
    return (REWARD ? c.w * (float)r : c.w) + tail;
}

template <int K, bool REWARD, class Leaf>
__device__ __forceinline__ float xm_value(const XmCtx& c, const typename Leaf::Param& leaf, u64 b, u64 bT, XmCount& n) {
    const uint32_t lm = play3_legal(c.s_flags, b, bT);
    float v = 0.0f;
    bool any = false;
#pragma unroll 1
    for (int a = 0; a < 4; ++a) {
        if ((lm >> a) & 1u) {
            const float q = xm_q<K, REWARD, Leaf>(c, leaf, b, bT, a, n);
            if (!any || q > v) v = q;
            any = true;
        }
    }
    return v;
}

// the spawn of exponent v into the empty nibble at bit p of s, in both orientations
__device__ __forceinline__ void xm_spawn(u64 s, u64 sT, int p, uint32_t v, u64& child, u64& childT) {
    const int cell = p >> 2, cellT = ((cell & 3) << 2) | (cell >> 2);
    child = s + ((u64)v << p);
    childT = sT + ((u64)v << (4 * cellT));
}

template <int K, bool REWARD, class Leaf>
__device__ __forceinline__ float xm_chance(const XmCtx& c, const typename Leaf::Param& leaf, u64 s, u64 sT, XmCount& n) {
    ++n.chance;
    u64 e = ~nonzero_lsb(s) & NIB_LSB;
    const int ne = __popcll(e);
    float acc = 0.0f;
#pragma unroll 1
    while (e) {
        const int p = __ffsll((long long)e) - 1;
        e &= e - 1;
        u64 ch, chT;
        xm_spawn(s, sT, p, 1u, ch, chT);
        const float v2 = xm_value<K, REWARD, Leaf>(c, leaf, ch, chT, n);
        xm_spawn(s, sT, p, 2u, ch, chT);
        const float v4 = xm_value<K, REWARD, Leaf>(c, leaf, ch, chT, n);
        acc = acc + (0.9f * v2 + 0.1f * v4);
    }
    return acc / (float)ne;
}

// The leaf of the search, a template parameter of the kernel.  Leaf::Param is the kernel parameter that carries it:
// the table T of the row heuristic H (g2048_expectimax_values), which the kernel puts into the search context ...
struct XmRowLeaf {
    using Param = const float* __restrict__;
    static __device__ __forceinline__ const float* table(const Param& T) { return T; }
    static __device__ __forceinline__ float value(const XmCtx& c, const Param&, u64 b, u64 bT) { return xm_heuristic(c, b, bT); }
};

// ... or an n-tuple network (g2048_expectimax_values_ntuple): V at the leaves, its placements read from the parameter's
// constant bank ...
struct XmTupleLeaf {
    using Param = NtNet;
    static __device__ __forceinline__ const float* table(const Param&) { return nullptr; }
    static __device__ __forceinline__ float value(const XmCtx&, const Param& net, u64 b, u64) { return nt_value<false>(net, b); }
};

// ... or a multi-stage n-tuple network (g2048_expectimax_values_ntuple_staged): V_S at the leaves, the stage taken
// from each leaf board
struct XmStagedTupleNet {
    NtNet net;
    NtStages stages;
};

struct XmStagedTupleLeaf {
    using Param = XmStagedTupleNet;
    static __device__ __forceinline__ const float* table(const Param&) { return nullptr; }
    static __device__ __forceinline__ float value(const XmCtx&, const Param& p, u64 b, u64) {
        return nt_value_staged<false>(p.net, p.stages, b);
    }
};

// Item j < n * 4 is (board j / 4, first action j % 4), one warp each.
template <int DEPTH, bool REWARD, class Leaf>
__global__ void __launch_bounds__(XM_THREADS, 1)
expectimax_kernel(const u64* __restrict__ boards, uint32_t n_items, const typename Leaf::Param leaf, float w,
                  float* __restrict__ q_out, unsigned long long* __restrict__ counters) {
    extern __shared__ __align__(16) uint8_t smem_raw[];
    __shared__ unsigned s_next;
    play3_copy_row_tables<XM_THREADS>(smem_raw);
    if (threadIdx.x == 0) s_next = 0;
    __syncthreads();

    const unsigned lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    float* slots = reinterpret_cast<float*>(smem_raw + PLAY3_TABLE_BYTES) + warp * (XM_SLOTS + XM_VALS);
    float* vals = slots + XM_SLOTS;
    XmCtx c;
    c.T = Leaf::table(leaf);
    c.w = w;
    c.s_left = reinterpret_cast<const uint16_t*>(smem_raw);
    c.s_flags = smem_raw + 65536 * 2;
    XmCount n = {0ull, 0ull};

    while (true) {
        unsigned k = 0;
        if (lane == 0) k = atomicAdd(&s_next, 1u);
        k = __shfl_sync(0xFFFFFFFFu, k, 0);
        const unsigned long long item = (unsigned long long)blockIdx.x + (unsigned long long)k * gridDim.x;
        if (item >= n_items) break;
        const u64 b = __ldg(&boards[item >> 2]);
        const int a0 = (int)(item & 3u);
        const u64 bT = transpose_board(b);
        if (!((play3_legal(c.s_flags, b, bT) >> a0) & 1u)) {
            if (lane == 0) q_out[item] = __int_as_float(0x7FC00000);  // NaN: illegal
            continue;
        }
        if constexpr (DEPTH == 1) {
            if (lane == 0) q_out[item] = xm_q<1, REWARD, Leaf>(c, leaf, b, bT, a0, n);
            continue;
        } else {
            u64 s, sT;
            uint32_t r0;
            xm_move<REWARD>(c, b, bT, a0, s, sT, r0);
            const u64 e = ~nonzero_lsb(s) & NIB_LSB;
            const int ne = __popcll(e);
            // children of the root chance node with their first move: j = (k-th empty cell) * 8 + (4-tile) * 4 + a1
            for (int j = (int)lane; j < ne * 8; j += 32) {
                const int p = 4 * kth_flag_cell(e, (j >> 3) + 1);
                u64 ch, chT;
                xm_spawn(s, sT, p, 1u + ((j >> 2) & 1u), ch, chT);
                const int a1 = j & 3;
                slots[j] = ((play3_legal(c.s_flags, ch, chT) >> a1) & 1u)
                               ? xm_q<DEPTH - 1, REWARD, Leaf>(c, leaf, ch, chT, a1, n)
                               : __int_as_float(0x7FC00000);  // NaN: a1 illegal
            }
            __syncwarp();
            for (int l = (int)lane; l < 2 * ne; l += 32) {  // V_{d-1} of child l: max over its legal a1 in order
                float v = 0.0f;
                bool any = false;
                for (int a = 0; a < 4; ++a) {
                    const float q = slots[4 * l + a];
                    if (q == q) {
                        if (!any || q > v) v = q;
                        any = true;
                    }
                }
                vals[l] = v;
            }
            __syncwarp();
            if (lane == 0) {
                ++n.chance;
                float acc = 0.0f;
                for (int k2 = 0; k2 < ne; ++k2) acc = acc + (0.9f * vals[2 * k2] + 0.1f * vals[2 * k2 + 1]);
                const float cv = acc / (float)ne;
                q_out[item] = (REWARD ? w * (float)r0 : w) + cv;
            }
            __syncwarp();  // the slots are reused by the next item
        }
    }

    if (counters) {
        unsigned long long leaves = n.leaves, chance = n.chance;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            leaves += __shfl_xor_sync(0xFFFFFFFFu, leaves, o);
            chance += __shfl_xor_sync(0xFFFFFFFFu, chance, o);
        }
        if (lane == 0) {
            if (leaves) atomicAdd(&counters[0], leaves);
            if (chance) atomicAdd(&counters[1], chance);
        }
    }
}

// this translation unit's copy of the row tables
__global__ void build_expectimax_row_tables_kernel() {
    const uint32_t row = blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= 65536u) return;
    build_row_table_entry(row);
}

template <int DEPTH, bool REWARD, class Leaf>
static int launch_expectimax(const uint64_t* d_boards, int64_t n_items, const typename Leaf::Param& leaf, float w, float* d_q,
                             uint64_t* d_counters, cudaStream_t st) {
    auto kernel = expectimax_kernel<DEPTH, REWARD, Leaf>;
    static bool configured_on[64] = {false};
    bool* configured = device_once_flag(configured_on);
    if (!configured) return fail_arg("no CUDA device");
    if (!*configured) {
        const int rc = check_cuda(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, XM_SMEM_BYTES),
                                  "expectimax_values: shared memory attribute");
        if (rc) return rc;
        *configured = true;
    }
    const int rc = ensure_row_tables_with<build_expectimax_row_tables_kernel>(st);
    if (rc) return rc;
    const int sms = sm_count();
    if (sms <= 0) return fail_arg("expectimax_values: no device");
    const int64_t needed = (n_items + XM_WARPS - 1) / XM_WARPS;
    const int64_t grid = needed < sms ? needed : sms;  // one CTA per SM, persistent
    kernel<<<(unsigned)grid, XM_THREADS, XM_SMEM_BYTES, st>>>((const u64*)d_boards, (uint32_t)n_items, leaf, w, d_q,
                                                             (unsigned long long*)d_counters);
    return check_cuda(cudaGetLastError(), "expectimax_values");
}

template <bool REWARD, class Leaf>
static int launch_expectimax_depth(int depth, const uint64_t* d_boards, int64_t n_items, const typename Leaf::Param& leaf, float w,
                                   float* d_q, uint64_t* d_counters, cudaStream_t st) {
    switch (depth) {
        case 1: return launch_expectimax<1, REWARD, Leaf>(d_boards, n_items, leaf, w, d_q, d_counters, st);
        case 2: return launch_expectimax<2, REWARD, Leaf>(d_boards, n_items, leaf, w, d_q, d_counters, st);
        case 3: return launch_expectimax<3, REWARD, Leaf>(d_boards, n_items, leaf, w, d_q, d_counters, st);
        default: return launch_expectimax<4, REWARD, Leaf>(d_boards, n_items, leaf, w, d_q, d_counters, st);
    }
}

// the reward-free form when w == 0 (+0 or -0): no merge reward to compute
template <class Leaf>
static int launch_expectimax_leaf(int depth, const uint64_t* d_boards, int64_t n, const typename Leaf::Param& leaf, float w, float* d_q,
                                  uint64_t* d_counters, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    if (w == 0.0f) return launch_expectimax_depth<false, Leaf>(depth, d_boards, n * 4, leaf, w, d_q, d_counters, st);
    return launch_expectimax_depth<true, Leaf>(depth, d_boards, n * 4, leaf, w, d_q, d_counters, st);
}

}  // namespace g2048

using namespace g2048;

extern "C" int g2048_expectimax_values(const uint64_t* d_boards, int64_t n, int depth, const float* d_row_values,
                                       float reward_weight, float* d_q, uint64_t* d_counters, void* stream) {
    G2048_REQUIRE(depth >= 1 && depth <= 4, "expectimax_values: depth must be in 1..4");
    G2048_REQUIRE(n >= 0 && n < (1ll << 29), "expectimax_values: n must be in [0, 2^29)");
    G2048_REQUIRE(((uintptr_t)d_q & 3u) == 0, "expectimax_values: d_q must be 4-byte aligned");
    if (n == 0) return G2048_OK;
    G2048_REQUIRE(d_boards && d_row_values && d_q, "expectimax_values: pointers");
    return launch_expectimax_leaf<XmRowLeaf>(depth, d_boards, n, d_row_values, reward_weight, d_q, d_counters, stream);
}

extern "C" int g2048_expectimax_values_ntuple(const uint64_t* d_boards, int64_t n, int depth,
                                              const G2048TuplePlacement* h_placements, int n_placements,
                                              const float* d_weights, int64_t n_weights, float reward_weight,
                                              float* d_q, uint64_t* d_counters, void* stream) {
    G2048_REQUIRE(depth >= 1 && depth <= 4, "expectimax_values_ntuple: depth must be in 1..4");
    G2048_REQUIRE(n >= 0 && n < (1ll << 29), "expectimax_values_ntuple: n must be in [0, 2^29)");
    G2048_REQUIRE(((uintptr_t)d_q & 3u) == 0 && ((uintptr_t)d_weights & 3u) == 0,
                  "expectimax_values_ntuple: d_q and d_weights must be 4-byte aligned");
    const int rc = ntuple_check(h_placements, n_placements, n_weights, "expectimax_values_ntuple: invalid network");
    if (rc) return rc;
    if (n == 0) return G2048_OK;
    G2048_REQUIRE(d_boards && d_weights && d_q, "expectimax_values_ntuple: pointers");
    NtNet net;
    ntuple_net(net, h_placements, n_placements, d_weights);
    return launch_expectimax_leaf<XmTupleLeaf>(depth, d_boards, n, net, reward_weight, d_q, d_counters, stream);
}

extern "C" int g2048_expectimax_values_ntuple_staged(const uint64_t* d_boards, int64_t n, int depth,
                                                     const G2048TuplePlacement* h_placements, int n_placements,
                                                     const G2048TupleStages* h_stages, const float* d_weights,
                                                     int64_t n_weights, float reward_weight, float* d_q,
                                                     uint64_t* d_counters, void* stream) {
    G2048_REQUIRE(depth >= 1 && depth <= 4, "expectimax_values_ntuple_staged: depth must be in 1..4");
    G2048_REQUIRE(n >= 0 && n < (1ll << 29), "expectimax_values_ntuple_staged: n must be in [0, 2^29)");
    G2048_REQUIRE(((uintptr_t)d_q & 3u) == 0 && ((uintptr_t)d_weights & 3u) == 0,
                  "expectimax_values_ntuple_staged: d_q and d_weights must be 4-byte aligned");
    int rc = ntuple_check(h_placements, n_placements, n_weights, "expectimax_values_ntuple_staged: invalid network");
    if (rc) return rc;
    rc = ntuple_stages_check(h_stages, h_placements, n_placements, n_weights,
                             "expectimax_values_ntuple_staged: invalid stages");
    if (rc) return rc;
    if (n == 0) return G2048_OK;
    G2048_REQUIRE(d_boards && d_weights && d_q, "expectimax_values_ntuple_staged: pointers");
    XmStagedTupleNet p;
    ntuple_net(p.net, h_placements, n_placements, d_weights);
    p.stages = ntuple_stages(*h_stages);
    return launch_expectimax_leaf<XmStagedTupleLeaf>(depth, d_boards, n, p, reward_weight, d_q, d_counters, stream);
}
