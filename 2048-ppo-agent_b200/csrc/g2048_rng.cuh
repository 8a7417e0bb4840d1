// Counter-based RNG that reproduces jax.random (Threefry-2x32, 20 rounds) bit for bit, in both
// counter layouts jax has shipped:
//   G2048_RNG_ORIGINAL       jax_threefry_partitionable=False (default before jax 0.5)
//   G2048_RNG_PARTITIONABLE  jax_threefry_partitionable=True  (default of the pinned jax==0.5.3)
// Replaces the jax.random calls at src/runs/batch_runner.py:32,105-106,118-119,126-127,
// src/actions/act_randomly.py:48 and src/ppo/torch_action_wrapper.py:91 of the reference, and the
// key handling inside Pgx's 2048 _init/_step/_add_random_num.  Everything is integer work kept in
// registers; one Threefry block is 40 ALU-pipe instructions (SHF.L.W / LOP3) and ~42 FMA-pipe adds (IMAD).
#pragma once
#include <cstdint>

#define G2048_RNG_ORIGINAL 0
#define G2048_RNG_PARTITIONABLE 1

namespace g2048 {

struct Key {
    uint32_t a, b;
};

__device__ __forceinline__ uint32_t rotl32(uint32_t x, int r) { return __funnelshift_l(x, x, r); }

// The kernels that hash the most (play3_kernel above all) were bound by the ALU pipe, which takes the rotates (SHF.L.W)
// and XORs (LOP3) of Threefry.  Left to itself ptxas folds every key injection and the round add after it into one
// IADD3 -- also an ALU-pipe instruction -- and only the plain round adds become IMAD.IADD on the FMA pipe.  add_fma()
// keeps an add on the FMA pipe: a mad.lo.u32 by a 1 that ptxas cannot see as a constant (it is read from constant
// memory, so the multiplier is a uniform-register operand and costs no per-thread register).
// (Host builds of these headers -- the test shim -- get a plain add.)
#ifdef __CUDACC__
static __constant__ uint32_t c_fma_one = 1u;
#endif

__device__ __forceinline__ uint32_t add_fma(uint32_t a, uint32_t b) {
#ifdef __CUDA_ARCH__
    uint32_t d;
    asm("mad.lo.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(c_fma_one), "r"(b));
    return d;
#else
    return a + b;
#endif
}

// a * M + b on the FMA pipe, for constant M (a shift by a constant and an OR or XOR with bits it cannot overlap, in one
// instruction).  The multiplier is M times the constant-memory 1, so ptxas cannot turn the product back into a shift
// (SHF / LEA on the ALU pipe); the product of two uniform values is computed once, outside the loops.
template <uint32_t M>
__device__ __forceinline__ uint32_t mad_fma(uint32_t a, uint32_t b) {
#ifdef __CUDA_ARCH__
    uint32_t d;
    asm("mad.lo.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(c_fma_one * M), "r"(b));
    return d;
#else
    return a * M + b;
#endif
}

// One Threefry-2x32-20 block.  Every add runs on the FMA pipe (add_fma); the rotates and XORs stay on the ALU pipe.
// The key schedule (ks2 and the five `ks + c` sums of the injections) depends on the key alone: callers that hash
// several counters under one key get it computed once, because the asm statements are pure and common
// subexpressions after inlining.
__device__ __forceinline__ Key threefry2x32(Key k, uint32_t x0, uint32_t x1) {
    const uint32_t ks0 = k.a, ks1 = k.b, ks2 = k.a ^ k.b ^ 0x1BD11BDAu;
    const uint32_t ks2p1 = add_fma(ks2, 1u), ks0p2 = add_fma(ks0, 2u), ks1p3 = add_fma(ks1, 3u);
    const uint32_t ks2p4 = add_fma(ks2, 4u), ks0p5 = add_fma(ks0, 5u);
    x0 = add_fma(x0, ks0);
    x1 = add_fma(x1, ks1);
#define G2048_TF_ROUND(r)   \
    x0 = add_fma(x0, x1);   \
    x1 = rotl32(x1, r);     \
    x1 ^= x0;
    G2048_TF_ROUND(13) G2048_TF_ROUND(15) G2048_TF_ROUND(26) G2048_TF_ROUND(6)
    x0 = add_fma(x0, ks1);
    x1 = add_fma(x1, ks2p1);
    G2048_TF_ROUND(17) G2048_TF_ROUND(29) G2048_TF_ROUND(16) G2048_TF_ROUND(24)
    x0 = add_fma(x0, ks2);
    x1 = add_fma(x1, ks0p2);
    G2048_TF_ROUND(13) G2048_TF_ROUND(15) G2048_TF_ROUND(26) G2048_TF_ROUND(6)
    x0 = add_fma(x0, ks0);
    x1 = add_fma(x1, ks1p3);
    G2048_TF_ROUND(17) G2048_TF_ROUND(29) G2048_TF_ROUND(16) G2048_TF_ROUND(24)
    x0 = add_fma(x0, ks1);
    x1 = add_fma(x1, ks2p4);
    G2048_TF_ROUND(13) G2048_TF_ROUND(15) G2048_TF_ROUND(26) G2048_TF_ROUND(6)
    x0 = add_fma(x0, ks2);
    x1 = add_fma(x1, ks0p5);
#undef G2048_TF_ROUND
    return Key{x0, x1};
}

// jax.random.split(key, n)[i].
//   partitionable: both words of TF(key; (0, i)).
//   original:      the (n,2) result is concat(y0, y1) of TF(key; iota(n), n + iota(n)) reshaped, so
//                  key i is flat words 2i and 2i+1; word m is y0[m] for m < n, else y1[m - n].
template <int MODE>
__device__ __forceinline__ Key split_at(Key k, uint32_t n, uint32_t i) {
    if (MODE == G2048_RNG_PARTITIONABLE) return threefry2x32(k, 0u, i);
    const uint32_t m0 = 2u * i, m1 = 2u * i + 1u;
    Key out;
    // m0 and m1 fall on the same side of n unless n is odd and m0 == n - 1
    out.a = (m0 < n) ? threefry2x32(k, m0, n + m0).a : threefry2x32(k, m0 - n, m0).b;
    out.b = (m1 < n) ? threefry2x32(k, m1, n + m1).a : threefry2x32(k, m1 - n, m1).b;
    return out;
}

// split(key, 2) -> both children (2 blocks in either layout).
template <int MODE>
__device__ __forceinline__ void split2(Key k, Key& c0, Key& c1) {
    if (MODE == G2048_RNG_PARTITIONABLE) {
        c0 = threefry2x32(k, 0u, 0u);
        c1 = threefry2x32(k, 0u, 1u);
    } else {
        const Key y0 = threefry2x32(k, 0u, 2u);  // -> flat words 0 and 2
        const Key y1 = threefry2x32(k, 1u, 3u);  // -> flat words 1 and 3
        c0 = Key{y0.a, y1.a};
        c1 = Key{y0.b, y1.b};
    }
}

// random_bits(key, shape=()) : one 32-bit draw.
template <int MODE>
__device__ __forceinline__ uint32_t bits_scalar(Key k) {
    const Key y = threefry2x32(k, 0u, 0u);
    return (MODE == G2048_RNG_PARTITIONABLE) ? (y.a ^ y.b) : y.a;
}

// random_bits(key, shape=(4,)).
template <int MODE>
__device__ __forceinline__ void bits4(Key k, uint32_t out[4]) {
    if (MODE == G2048_RNG_PARTITIONABLE) {
#pragma unroll
        for (uint32_t i = 0; i < 4; ++i) {
            const Key y = threefry2x32(k, 0u, i);
            out[i] = y.a ^ y.b;
        }
    } else {
        const Key y0 = threefry2x32(k, 0u, 2u);
        const Key y1 = threefry2x32(k, 1u, 3u);
        out[0] = y0.a;
        out[1] = y1.a;
        out[2] = y0.b;
        out[3] = y1.b;
    }
}

// jax.random.uniform's bits -> [0, 1): mantissa fill of 1.xxx minus one.
__device__ __forceinline__ float unit_float(uint32_t bits) {
    return __fsub_rn(__uint_as_float((bits >> 9) | 0x3F800000u), 1.0f);
}

// uniform(key, (), minval=tiny, maxval=1) as jax.random.gumbel/categorical draw it:
// max(tiny, f * (1 - tiny) + tiny).  (1 - tiny) rounds to 1 and f + tiny rounds to f for f > 0.
__device__ __forceinline__ float unit_float_tiny(uint32_t bits) {
    const float tiny = 1.17549435e-38f;
    const float f = unit_float(bits);
    return fmaxf(tiny, __fadd_rn(__fmul_rn(f, 1.0f), tiny));
}

// ---- keyed pseudo-random bijection of [0, n) (g2048_random_subset, g2048_data.cu) ---------------------------------
// Balanced Feistel network, 4 rounds, over 2h bits with 4^h >= n; round function = low h bits of the first word of
// Threefry-2x32(key; (right half, round)); images >= n go through the network again (cycle walking).
inline int feistel_half_bits(uint64_t n) {
    int h = 1;
    while (h < 31 && (1ull << (2 * h)) < n) ++h;
    return h;
}

__device__ __forceinline__ uint64_t feistel_pass(Key k, uint64_t x, int h, uint32_t mask) {
    uint32_t left = (uint32_t)(x >> h), right = (uint32_t)x & mask;
#pragma unroll
    for (uint32_t r = 0; r < 4; ++r) {
        const uint32_t f = threefry2x32(k, right, r).a & mask;
        const uint32_t nl = right;
        right = left ^ f;
        left = nl;
    }
    return ((uint64_t)left << h) | (uint64_t)right;
}

__device__ __forceinline__ uint64_t feistel_position(Key k, uint64_t x, int h, uint64_t n) {
    const uint32_t mask = (h >= 32) ? 0xFFFFFFFFu : ((1u << h) - 1u);
    do {
        x = feistel_pass(k, x, h, mask);
    } while (x >= n);
    return x;
}

}  // namespace g2048
