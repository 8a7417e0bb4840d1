// The row heuristic and the table-driven move shared by the expectimax kernel (g2048_expectimax.cu) and the TD learner
// (g2048_td.cu), so that both use one H and one move:
//   H(b) = T[row0] + .. + T[row3] + T[col0] + .. + T[col3]   (left to right; include/g2048.h)
#pragma once
#include "g2048_play3.cuh"

namespace g2048 {

struct XmCtx {
    const float* T;
    float w;
    const uint16_t* s_left;
    const uint8_t* s_flags;
};

// T[i] through the read-only path (__ldg), or -- COHERENT -- through an ordinary load, for a kernel that changes T
// between the phases of one launch (ld.global.nc is only defined for data that stays read-only while the kernel runs)
template <bool COHERENT>
__device__ __forceinline__ float xm_row_value(const float* T, uint32_t i) {
    if constexpr (COHERENT) return T[i];
    else return __ldg(&T[i]);
}

// A board travels with its transpose bT: columns are rows of the transpose.
template <bool COHERENT = false>
__device__ __forceinline__ float xm_heuristic(const XmCtx& c, u64 b, u64 bT) {
    const uint32_t lo = (uint32_t)b, hi = (uint32_t)(b >> 32), tlo = (uint32_t)bT, thi = (uint32_t)(bT >> 32);
    float h = xm_row_value<COHERENT>(c.T, lo & 0xFFFFu);
    h = h + xm_row_value<COHERENT>(c.T, lo >> 16);
    h = h + xm_row_value<COHERENT>(c.T, hi & 0xFFFFu);
    h = h + xm_row_value<COHERENT>(c.T, hi >> 16);
    h = h + xm_row_value<COHERENT>(c.T, tlo & 0xFFFFu);
    h = h + xm_row_value<COHERENT>(c.T, tlo >> 16);
    h = h + xm_row_value<COHERENT>(c.T, thi & 0xFFFFu);
    h = h + xm_row_value<COHERENT>(c.T, thi >> 16);
    return h;
}

// (nb, nbT) = move(b, a); with REWARD also r = potential(nb) - potential(b), the merge reward
template <bool REWARD>
__device__ __forceinline__ void xm_move(const XmCtx& c, u64 b, u64 bT, int a, u64& nb, u64& nbT, uint32_t& r) {
    const bool vertical = (a & 1) != 0, rev = a >= 2;
    u64 src = vertical ? bT : b;
    if (rev) src = mirror_rows(src);
    const uint32_t slo = (uint32_t)src, shi = (uint32_t)(src >> 32);
    const uint32_t m0 = c.s_left[slo & 0xFFFFu], m1 = c.s_left[slo >> 16];
    const uint32_t m2 = c.s_left[shi & 0xFFFFu], m3 = c.s_left[shi >> 16];
    u64 moved = ((u64)(m2 | (m3 << 16)) << 32) | (u64)(m0 | (m1 << 16));
    if (rev) moved = mirror_rows(moved);
    const u64 movedT = transpose_board(moved);
    nb = vertical ? movedT : moved;
    nbT = vertical ? moved : movedT;
    if (REWARD) r = board_potential(nb) - board_potential(b);
}

}  // namespace g2048
