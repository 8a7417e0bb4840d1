// N-tuple networks (include/g2048.h): the value V(b) = W[off_0 + idx_0(b)] + .. + W[off_{P-1} + idx_{P-1}(b)] (left to
// right from the first term) shared by the n-tuple TD learner (g2048_ntuple.cu) and the expectimax kernel's network
// leaf (g2048_expectimax.cu), and the host-side check of a placement list.  A multi-stage network (G2048TupleStages)
// adds stage(b) * stride to every entry of board b: nt_stage_base once per board, then the same gathers.
//
// The placement list travels by value in the kernel parameters, so every lane reads the
// same placement from the constant bank: the loop over placements is uniform, and only the W gathers diverge.
#pragma once
#include "g2048_board.cuh"
#include "g2048_common.cuh"

namespace g2048 {

struct NtNet {
    const float* W;
    uint32_t n_placements;
    G2048TuplePlacement pl[G2048_NTUPLE_MAX_PLACEMENTS];
};

// Host: G2048_OK, or fail_arg for an invalid network
inline int ntuple_check(const G2048TuplePlacement* pl, int n_placements, int64_t n_weights, const char* what) {
    if (!pl || n_placements < 1 || n_placements > G2048_NTUPLE_MAX_PLACEMENTS) return fail_arg(what);
    if (n_weights < 1 || n_weights > G2048_NTUPLE_MAX_WEIGHTS) return fail_arg(what);
    for (int p = 0; p < n_placements; ++p) {
        const G2048TuplePlacement& t = pl[p];
        if (t.n_cells < 1 || t.n_cells > 6 || t.reserved != 0) return fail_arg(what);
        unsigned seen = 0u;
        for (int j = 0; j < t.n_cells; ++j) {
            if (t.cells[j] >= 16 || ((seen >> t.cells[j]) & 1u)) return fail_arg(what);
            seen |= 1u << t.cells[j];
        }
        if ((int64_t)t.offset + (1ll << (4 * t.n_cells)) > n_weights) return fail_arg(what);
    }
    return G2048_OK;
}

inline void ntuple_net(NtNet& net, const G2048TuplePlacement* pl, int n_placements, const float* W) {
    net = NtNet{};
    net.W = W;
    net.n_placements = (uint32_t)n_placements;
    for (int p = 0; p < n_placements; ++p) net.pl[p] = pl[p];
}

// The stages as the kernels read them: nibble e of stage_of is the stage of a board whose largest exponent is e
// (S <= 16, so a stage fits a nibble), and a stage-s board reads its tables s * stride entries further on.
struct NtStages {
    unsigned long long stage_of;
    uint32_t stride;
};

// Host: G2048_OK, or fail_arg for invalid stages of a valid network (ntuple_check first)
inline int ntuple_stages_check(const G2048TupleStages* st, const G2048TuplePlacement* pl, int n_placements,
                               int64_t n_weights, const char* what) {
    if (!st || st->n_thresholds > G2048_NTUPLE_MAX_STAGES - 1) return fail_arg(what);
    for (int j = 0; j < G2048_NTUPLE_MAX_STAGES - 1; ++j) {
        const int t = st->thresholds[j];
        if (j >= st->n_thresholds) {
            if (t != 0) return fail_arg(what);
        } else if (t < 1 || t > 15 || (j > 0 && t <= st->thresholds[j - 1])) {
            return fail_arg(what);
        }
    }
    if ((st->n_thresholds == 0) != (st->stride == 0u)) return fail_arg(what);
    const int64_t last = (int64_t)st->n_thresholds * (int64_t)st->stride;
    for (int p = 0; p < n_placements; ++p)
        if (last + (int64_t)pl[p].offset + (1ll << (4 * pl[p].n_cells)) > n_weights) return fail_arg(what);
    return G2048_OK;
}

inline NtStages ntuple_stages(const G2048TupleStages& st) {
    NtStages s;
    s.stage_of = 0ull;
    for (int e = 0; e < 16; ++e) {
        unsigned long long stage = 0ull;
        for (int j = 0; j < st.n_thresholds; ++j) stage += e >= st.thresholds[j] ? 1ull : 0ull;
        s.stage_of |= stage << (4 * e);
    }
    s.stride = st.stride;
    return s;
}

#ifdef __CUDACC__
// off_p + idx_p(b) (< 2^28)
__device__ __forceinline__ uint32_t nt_entry(const G2048TuplePlacement& p, u64 b) {
    uint32_t idx = 0u;
#pragma unroll
    for (int j = 0; j < 6; ++j)
        if (j < p.n_cells) idx |= (uint32_t)(b >> (4 * p.cells[j]) & 15u) << (4 * j);
    return p.offset + idx;
}

// W[i] through the read-only path, or -- COHERENT -- through an ordinary load, for a kernel that changes W between the
// phases of one launch
template <bool COHERENT>
__device__ __forceinline__ float nt_weight(const float* W, uint32_t i) {
    if constexpr (COHERENT) return W[i];
    else return __ldg(&W[i]);
}

// v[j] = V(b[j] at entries base[j] further on) for NB boards at once: the gathers of the NB boards and of 4 placements
// are independent, so they are in flight together; each sum still runs over the placements in order.  base[j] is 0 for
// a single-stage network, and nt_stage_base(b[j]) for a multi-stage one.
template <bool COHERENT, int NB>
__device__ __forceinline__ void nt_values_at(const NtNet& net, const u64 (&b)[NB], const uint32_t (&base)[NB],
                                             float (&v)[NB]) {
#pragma unroll
    for (int j = 0; j < NB; ++j) v[j] = nt_weight<COHERENT>(net.W, base[j] + nt_entry(net.pl[0], b[j]));
#pragma unroll 4
    for (uint32_t p = 1; p < net.n_placements; ++p) {
        float w[NB];
#pragma unroll
        for (int j = 0; j < NB; ++j) w[j] = nt_weight<COHERENT>(net.W, base[j] + nt_entry(net.pl[p], b[j]));
#pragma unroll
        for (int j = 0; j < NB; ++j) v[j] = v[j] + w[j];
    }
}

template <bool COHERENT, int NB>
__device__ __forceinline__ void nt_values(const NtNet& net, const u64 (&b)[NB], float (&v)[NB]) {
    const uint32_t base[NB] = {};
    nt_values_at<COHERENT, NB>(net, b, base, v);
}

template <bool COHERENT>
__device__ __forceinline__ float nt_value(const NtNet& net, u64 b) {
    const u64 bb[1] = {b};
    float v[1];
    nt_values<COHERENT, 1>(net, bb, v);
    return v[0];
}

// stage(b) * stride (< 2^28: the stages check bounds (S - 1) * stride by n_weights)
__device__ __forceinline__ uint32_t nt_stage_base(const NtStages& st, u64 b) {
    return (uint32_t)(st.stage_of >> (4 * max_exponent(b)) & 15u) * st.stride;
}

// stage(b)
__device__ __forceinline__ uint32_t nt_stage(const NtStages& st, u64 b) {
    return (uint32_t)(st.stage_of >> (4 * max_exponent(b)) & 15u);
}

// V_S(b) of a multi-stage network
template <bool COHERENT>
__device__ __forceinline__ float nt_value_staged(const NtNet& net, const NtStages& st, u64 b) {
    const u64 bb[1] = {b};
    const uint32_t base[1] = {nt_stage_base(st, b)};
    float v[1];
    nt_values_at<COHERENT, 1>(net, bb, base, v);
    return v[0];
}
#endif

}  // namespace g2048
