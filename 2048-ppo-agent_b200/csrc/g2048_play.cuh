// Pieces shared by the persistent play kernels (g2048_play.cu: SWAR board logic, g2048_play3.cu: row tables).
#pragma once
#include "g2048_board.cuh"
#include "g2048_env.cuh"

namespace g2048 {

// The blocks of one key that both bits4() and split2() are made of.
template <int MODE>
struct KeyBlocks {
    uint32_t bits[4];  // random_bits(key, (4,))
    Key child[2];      // split(key, 2)
};

template <int MODE>
__device__ __forceinline__ KeyBlocks<MODE> key_blocks(Key k) {
    KeyBlocks<MODE> o;
    if (MODE == G2048_RNG_PARTITIONABLE) {
        Key y[4];
#pragma unroll
        for (uint32_t i = 0; i < 4; ++i) {
            y[i] = threefry2x32(k, 0u, i);
            o.bits[i] = y[i].a ^ y[i].b;
        }
        o.child[0] = y[0];
        o.child[1] = y[1];
    } else {
        const Key y0 = threefry2x32(k, 0u, 2u);
        const Key y1 = threefry2x32(k, 1u, 3u);
        o.bits[0] = y0.a;
        o.bits[1] = y1.a;
        o.bits[2] = y0.b;
        o.bits[3] = y1.b;
        o.child[0] = Key{y0.a, y1.a};
        o.child[1] = Key{y0.b, y1.b};
    }
    return o;
}

__device__ __forceinline__ int argmax_bits_legal(const uint32_t bits[4], uint32_t legal) {
    const uint32_t allowed = (legal & 15u) ? (legal & 15u) : 15u;
    int best = 0, best_v = -1;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int v = ((allowed >> i) & 1u) ? (int)(bits[i] >> 9) : -1;
        if (v > best_v) {
            best_v = v;
            best = i;
        }
    }
    return best;
}

// argmax_bits_legal from a 16-entry table indexed by the legal mask: entry lm holds, per action i, a mask mm_i
// (0xFFFFFE00 if i is allowed, else 0) and a tie constant c_i (7 - i if allowed, else 0).  v_i = (bits_i & mm_i) + c_i
// orders the allowed actions by bits_i >> 9 and, on ties, the lower index first; a disallowed action has v_i = 0 below
// every allowed one (c_i >= 4).  The maximum's low three bits are 7 - i, so the action is ~max & 7.  (In the
// partitionable layout bits_i = y.a ^ y.b, and the XOR and the AND are one LOP3.)
struct ActEntry {
    uint4 mm, c;
};

__device__ __forceinline__ ActEntry act_entry_of(uint32_t lm) {
    const uint32_t allowed = lm ? lm : 15u;  // no legal action: all four, as argmax_bits_legal
    ActEntry e;
    uint32_t mm[4], c[4];
    for (uint32_t i = 0; i < 4; ++i) {
        mm[i] = ((allowed >> i) & 1u) ? 0xFFFFFE00u : 0u;
        c[i] = ((allowed >> i) & 1u) ? 7u - i : 0u;
    }
    e.mm = make_uint4(mm[0], mm[1], mm[2], mm[3]);
    e.c = make_uint4(c[0], c[1], c[2], c[3]);
    return e;
}

__device__ __forceinline__ int act_random_table(const uint32_t bits[4], const ActEntry& e) {
    const uint32_t v0 = add_fma(bits[0] & e.mm.x, e.c.x), v1 = add_fma(bits[1] & e.mm.y, e.c.y);
    const uint32_t v2 = add_fma(bits[2] & e.mm.z, e.c.z), v3 = add_fma(bits[3] & e.mm.w, e.c.w);
    return (int)(~max(max(v0, v1), max(v2, v3)) & 7u);
}

enum : uint32_t { PHASE_INIT0 = 0, PHASE_INIT1 = 1, PHASE_PLAY = 2, PHASE_NONE = 3 };

}  // namespace g2048
