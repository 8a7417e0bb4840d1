// 2048 board as a 64-bit nibble bitboard held in registers.
//
// Cell i = 4*row + col (row-major, same order as Pgx's flat board) lives in bits [4i, 4i+4) and
// stores the exponent e (0 = empty, e = tile 2^e).  Row r is bits [16r, 16r+16).  All four rows (or
// columns) of a move are processed at once with SWAR arithmetic on the whole word: a move toward
// lower cell indices ("Left": stride 4 bits, "Up": stride 16 bits) is three conditional one-cell
// shifts, one merge pass, two more shifts; Right/Down run the same code on the nibble-reversed
// board.  There is no lookup table: the shared-memory row table of classic bitboard 2048 costs
// 128 KiB + bank conflicts, while the SWAR move is ~140 integer instructions -- small next to the
// ~850 instructions of Threefry per env-step.
//
// Replaces Pgx 2.6.0's 2048 _step/_slide_and_merge/_can_slide_left/_add_random_num/observe as called
// from src/runs/batch_runner.py:34-35,107,128 of the reference (actions 0=Left 1=Up 2=Right 3=Down).
#pragma once
#include <cstdint>

#include "g2048_rng.cuh"

namespace g2048 {

typedef unsigned long long u64;

constexpr u64 NIB_LSB = 0x1111111111111111ull;

// bit 0 of every nibble = (nibble != 0)
__device__ __forceinline__ u64 nonzero_lsb(u64 x) {
    u64 t = x | (x >> 1);
    t |= t >> 2;
    return t & NIB_LSB;
}

// 0xF in every nibble whose lsb is set in t (t has only nibble lsbs)
__device__ __forceinline__ u64 spread_nibble(u64 t) { return (t << 4) - t; }

// reverse the 16 nibbles: cell i <-> cell 15 - i (a 180 degree turn of the board)
__device__ __forceinline__ u64 reverse_nibbles(u64 x) {
    uint32_t lo = (uint32_t)x, hi = (uint32_t)(x >> 32);
    lo = __byte_perm(lo, 0, 0x0123);
    hi = __byte_perm(hi, 0, 0x0123);
    lo = ((lo & 0x0F0F0F0Fu) << 4) | ((lo >> 4) & 0x0F0F0F0Fu);
    hi = ((hi & 0x0F0F0F0Fu) << 4) | ((hi >> 4) & 0x0F0F0F0Fu);
    return ((u64)lo << 32) | hi;
}

// Slide + merge toward lower cell indices along lines of stride `s` bits (4: rows, i.e. Left;
// 16: columns, i.e. Up).  `has_lower` marks the cells that have a neighbour at p - s in their line.
// Returns the moved board; `reward` gets sum of 2^(e+1) over merges (Pgx: the merged tile's value);
// `overflow` is set if a 2^15 pair merged (the result does not fit a nibble).
template <bool WANT_REWARD>
__device__ __forceinline__ u64 slide_merge_low(u64 x, int s, u64 has_lower, u64 line_ge2, u64 line_eq3,
                                               uint32_t& reward, bool& overflow) {
#define G2048_COMPRESS_ONCE()                                          \
    {                                                                  \
        const u64 empty = ~spread_nibble(nonzero_lsb(x));              \
        const u64 mv = x & (empty << s) & has_lower;                   \
        x = (x ^ mv) | (mv >> s);                                      \
    }
    G2048_COMPRESS_ONCE()
    G2048_COMPRESS_ONCE()
    G2048_COMPRESS_ONCE()
    // merge pass: pair (p, p+s) merges iff equal, non-empty and p was not consumed by (p-s, p)
    const u64 has_upper = has_lower >> s;
    const u64 nz = nonzero_lsb(x);
    const u64 eq = ~nonzero_lsb(x ^ (x >> s)) & nz & has_upper & NIB_LSB;  // lsb flags at p
    // position in line: line0 = cells with no lower neighbour
    const u64 line0 = ~has_lower & NIB_LSB;
    const u64 m0 = eq & line0;
    const u64 m1 = eq & (line0 << s) & ~(m0 << s);
    const u64 m2 = eq & (line0 << (2 * s)) & ~(m1 << s);
    const u64 m = m0 | m1 | m2;
    reward = 0;
    if (WANT_REWARD && m) {
        u64 mm = m;
        do {
            const int p = __ffsll((long long)mm) - 1;
            const uint32_t v = (uint32_t)(x >> p) & 15u;
            overflow |= (v == 15u);
            reward += 2u << v;
            mm &= mm - 1;
        } while (mm);
    }
    x += m;                                  // merged cell: e -> e + 1
    const u64 hole = m << s;                 // lsb flags where the partner disappears
    x &= ~spread_nibble(hole);
    // close the holes: a cell moves down by exactly one step iff a hole lies below it in its line
    // (holes sit at line positions 1..3; two holes are never both below a live cell)
    const u64 below = ((hole << s) & line_ge2) | ((hole << (2 * s)) & line_eq3);
    const u64 mv = x & spread_nibble(below);
    x = (x ^ mv) | (mv >> s);
#undef G2048_COMPRESS_ONCE
    return x;
}

// Pgx _step's board part: rot90(board, action) -> slide/merge left -> rotate back.
// WANT_REWARD = false skips the per-merge reward sum (the persistent play kernel derives the score
// from the final board instead, see board_potential) and leaves `reward` / `overflow` untouched.
template <bool WANT_REWARD = true>
__device__ __forceinline__ u64 move_board(u64 x, int action, uint32_t& reward, bool& overflow) {
    const bool rev = action >= 2;            // Right = Left on the reversed board, Down = Up on it
    if (rev) x = reverse_nibbles(x);
    const bool vertical = action & 1;
    const int s = vertical ? 16 : 4;
    const u64 has_lower = vertical ? 0xFFFFFFFFFFFF0000ull : 0xFFF0FFF0FFF0FFF0ull;
    const u64 line_ge2 = vertical ? 0x1111111100000000ull : 0x1100110011001100ull;  // lsb flags, line position >= 2
    const u64 line_eq3 = vertical ? 0x1111000000000000ull : 0x1000100010001000ull;  // line position == 3
    x = slide_merge_low<WANT_REWARD>(x, s, has_lower, line_ge2, line_eq3, reward, overflow);
    if (rev) x = reverse_nibbles(x);
    return x;
}

// true iff some cell holds exponent 15 (a 2^15 tile: the next merge would not fit a nibble)
__device__ __forceinline__ bool has_max_nibble(u64 x) {
    u64 t = x & (x >> 1);
    t &= t >> 2;
    return (t & NIB_LSB) != 0ull;
}

// Exact legal-action mask, bit a = (move(board, a) != board): a line can move toward a side iff
// some adjacent pair along it is (empty, tile) in that order, or two equal tiles.
__device__ __forceinline__ uint32_t legal_mask(u64 x) {
    const u64 nz = nonzero_lsb(x);
    const u64 H = 0x0111011101110111ull;     // pairs (p, p+1 col) for col 0..2
    const u64 V = 0x0000111111111111ull;     // pairs (p, p+1 row) for row 0..2
    const u64 nzr = nz >> 4, nzd = nz >> 16;
    const u64 eqh = ~nonzero_lsb(x ^ (x >> 4)) & nz;
    const u64 eqv = ~nonzero_lsb(x ^ (x >> 16)) & nz;
    const u64 left = ((~nz & nzr) | eqh) & H;
    const u64 right = ((nz & ~nzr) | eqh) & H;
    const u64 up = ((~nz & nzd) | eqv) & V;
    const u64 down = ((nz & ~nzd) | eqv) & V;
    return (left ? 1u : 0u) | (up ? 2u : 0u) | (right ? 4u : 0u) | (down ? 8u : 0u);
}

// index (0-based cell) of the k-th (1-based) set flag of `flags` (one flag per cell, at the nibble's lsb), 1 <= k <= number
// of flags.  Prefix counts by one multiply: nibble i of w * 0x11111111 is the number of flags among cells 0..i of that
// half (at most 8, so no carry crosses a nibble); adding 8 - k sets bit 3 of exactly the nibbles whose prefix count has
// reached k, and the lowest of them is the cell.  (13 instructions; the popcount bisection it replaces took 25.)
__device__ __forceinline__ int kth_flag_cell(u64 flags, int k) {
    const uint32_t lo = (uint32_t)flags, hi = (uint32_t)(flags >> 32);
    const int c = __popc(lo);
    const bool upper = k > c;
    const uint32_t w = upper ? hi : lo;
    const uint32_t kk = (uint32_t)(upper ? k - c : k);  // 1..8
    const uint32_t prefix = w * 0x11111111u;
    const uint32_t reached = (prefix + (8u - kk) * 0x11111111u) & 0x88888888u;
    return (upper ? 8 : 0) + ((__ffs((int)reached) - 1) >> 2);
}

// Pgx _add_random_num given the two 32-bit draws behind uniform(k1) and uniform(k2):
//   pos = choice(arange(16), p=(board==0)) = searchsorted_left(cumsum_f32(empty), n_empty*(1-u))
//       = the ceil(fl32(n_empty * (1-u)))-th empty cell in row-major order, 1-based;
//   val = 2 (a 4-tile) iff 1.0f*(1-u') > 0.9f, else 1.
// With u = f - 1 for f in [1,2): 1 - u = m * 2^-23 exactly, m = 2^23 - (bits >> 9).
// The spawn decision alone: which cell (row-major index) and which exponent (1 or 2).
__device__ __forceinline__ void spawn_select(u64 x, uint32_t bits_pos, uint32_t bits_val, int& cell, u64& val) {
    const u64 empties = ~nonzero_lsb(x) & NIB_LSB;
    const int n_empty = __popcll(empties);
    const float one_minus_u = __fsub_rn(1.0f, unit_float(bits_pos));
    const float r = __fmul_rn((float)n_empty, one_minus_u);
    const int k = (int)ceilf(r);
    // a full board (only reachable through the illegal-action path) leaves searchsorted at cell 0
    cell = (n_empty == 0) ? 0 : kth_flag_cell(empties, k);
    // m * 2^-23 > 0.9f = 15099494 * 2^-24  <=>  m = 2^23 - (bits >> 9) > 7549747  <=>  bits >> 9 < 838861
    //                                      <=>  bits < 838861 * 2^9 = 429496832 (tests/test_step_logic.py)
    val = (bits_val < 429496832u) ? 2ull : 1ull;
}

__device__ __forceinline__ u64 spawn_tile(u64 x, uint32_t bits_pos, uint32_t bits_val) {
    int cell;
    u64 val;
    spawn_select(x, bits_pos, bits_val, cell, val);
    return (x & ~(0xFull << (4 * cell))) | (val << (4 * cell));
}

// (a & m) | (b & ~m) as one LOP3 (left to itself, ptxas splits the mirror's select below into two)
__device__ __forceinline__ uint32_t bit_select(uint32_t a, uint32_t b, uint32_t m) {
#ifdef __CUDA_ARCH__
    uint32_t d;
    asm("lop3.b32 %0, %1, %2, %3, 0xE4;" : "=r"(d) : "r"(a), "r"(b), "r"(m));  // 0xE4 = (0xF0 & 0xAA) | (0xCC & ~0xAA)
    return d;
#else
    return (a & m) | (b & ~m);
#endif
}

// transpose of the 4x4 nibble matrix: cell (r, c) <-> cell (c, r), in 32-bit halves (the 64-bit form costs twice the
// ALU-pipe instructions: every 64-bit shift is two)
__device__ __forceinline__ u64 transpose_board(u64 x) {
    uint32_t lo = (uint32_t)x, hi = (uint32_t)(x >> 32);
    // 2x2 blocks of cells: swap the (0, 1) and (1, 0) cells of each, which lie in the same half (rows 0-1 / rows 2-3);
    // t and t << 12 cannot overlap, so t ^ (t << 12) = t * 4097
    const uint32_t tl = (lo ^ (lo >> 12)) & 0x0000F0F0u, th = (hi ^ (hi >> 12)) & 0x0000F0F0u;
    lo ^= mad_fma<4097u>(tl, 0u);
    hi ^= mad_fma<4097u>(th, 0u);
    // 2x2 blocks of blocks: the upper right block (bytes 1 and 3 of the low half) and the lower left one (bytes 0 and
    // 2 of the high half) change places
    const uint32_t nlo = __byte_perm(lo, hi, 0x6240), nhi = __byte_perm(lo, hi, 0x7351);
    return ((u64)nhi << 32) | nlo;
}

// reverse the nibble order inside each 16-bit row (mirror the board left <-> right)
__device__ __forceinline__ u64 mirror_rows(u64 x) {
    uint32_t lo = (uint32_t)x, hi = (uint32_t)(x >> 32);
    lo = __byte_perm(lo, 0, 0x2301);
    hi = __byte_perm(hi, 0, 0x2301);
    // the two nibbles of every byte change places: one bit-select between the word shifted up (on the FMA pipe) and
    // the word shifted down
    lo = bit_select(mad_fma<16u>(lo, 0u), lo >> 4, 0xF0F0F0F0u);
    hi = bit_select(mad_fma<16u>(hi, 0u), hi >> 4, 0xF0F0F0F0u);
    return ((u64)hi << 32) | lo;
}

__device__ __forceinline__ uint32_t max_exponent(u64 x) {
    uint32_t m = 0;
#pragma unroll
    for (int i = 0; i < 16; ++i) m = max(m, (uint32_t)(x >> (4 * i)) & 15u);
    return m;
}

// Pgx score bookkeeping without per-step rewards: sum over tiles of (e - 1) * 2^e equals the sum of
// all merge rewards that built the board from spawned 2-tiles; every spawned 4-tile overcounts by 4.
__device__ __forceinline__ uint32_t board_potential(u64 x) {
    uint32_t f = 0;
#pragma unroll
    for (int i = 0; i < 16; ++i) {
        const uint32_t e = (uint32_t)(x >> (4 * i)) & 15u;
        f += e ? ((e - 1u) << e) : 0u;
    }
    return f;
}

}  // namespace g2048
