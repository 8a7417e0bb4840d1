// TEST-ONLY: the play step's board and policy helpers (g2048_board.cuh, g2048_play.cuh) compiled for the host through
// cuda_shim.h, for tests/test_step_logic.py.
#include "cuda_shim.h"

struct uint4 { uint32_t x, y, z, w; };
static inline uint4 make_uint4(uint32_t x, uint32_t y, uint32_t z, uint32_t w) { return uint4{x, y, z, w}; }

#include "../../2048-ppo-agent_b200/csrc/g2048_play.cuh"

using namespace g2048;

extern "C" {

// the spawned exponent (1 or 2) of spawn_select for bits_val = (h << 9) | low, every h < 2^23
void step_spawn_val_all(uint32_t low, uint8_t* out /* [2^23] */) {
    for (uint32_t h = 0; h < (1u << 23); ++h) {
        int cell;
        u64 val;
        spawn_select(0ull, 0u, (h << 9) | low, cell, val);
        out[h] = (uint8_t)val;
    }
}

void step_transpose_mirror(const uint64_t* boards, int64_t n, uint64_t* transposed, uint64_t* mirrored) {
    for (int64_t i = 0; i < n; ++i) {
        transposed[i] = transpose_board(boards[i]);
        mirrored[i] = mirror_rows(boards[i]);
    }
}

// act_random_table with the table entry of lm, and argmax_bits_legal, for n (bits[4], lm) pairs
void step_act(const uint32_t* bits /* [n][4] */, const uint32_t* lm, int64_t n, int32_t* table, int32_t* reference) {
    for (int64_t i = 0; i < n; ++i) {
        table[i] = act_random_table(bits + 4 * i, act_entry_of(lm[i] & 15u));
        reference[i] = argmax_bits_legal(bits + 4 * i, lm[i]);
    }
}

}  // extern "C"
