/* Depth-limited expectimax restated on the CPU with the oracle's own move function.  TEST INFRASTRUCTURE ONLY.
 *
 * The oracle (oracle/pgx2048_oracle.c) is included whole, so this file uses its move_board (which returns the merge
 * reward) and exact_legal as they are and adds one entry point on top; tests/expectimax_oracle.py compiles it (gcc -O2
 * -fopenmp -shared -fPIC -ffp-contract=off, like oracle/Makefile).  Every float operation is written in the order of
 * the contract in include/g2048.h (g2048_expectimax_values).
 */
#include "../oracle/pgx2048_oracle.c"

typedef struct {
    const float* T;
    float w;
    uint64_t leaves, chance;
} xm_ctx;

static float xm_value(xm_ctx* c, const uint8_t* b, int k);

/* H(b): the 4 rows, then the 4 columns, left to right; row r = cells 4r..4r+3 (nibble j = column j), column c =
 * cells c, c+4, c+8, c+12 (nibble j = row j) */
static float xm_heuristic(const xm_ctx* c, const uint8_t* b) {
    float h = 0.0f;
    for (int line = 0; line < 8; ++line) {
        uint32_t idx = 0;
        for (int j = 0; j < 4; ++j) idx |= (uint32_t)b[line < 4 ? 4 * line + j : 4 * j + (line - 4)] << (4 * j);
        h = line == 0 ? c->T[idx] : h + c->T[idx];
    }
    return h;
}

static float xm_chance(xm_ctx* c, const uint8_t* s, int k) {
    c->chance += 1;
    float acc = 0.0f;
    int ne = 0;
    for (int cell = 0; cell < 16; ++cell) {
        if (s[cell]) continue;
        ++ne;
        uint8_t ch[16];
        memcpy(ch, s, 16);
        ch[cell] = 1;
        const float v2 = xm_value(c, ch, k);
        ch[cell] = 2;
        const float v4 = xm_value(c, ch, k);
        acc = acc + (0.9f * v2 + 0.1f * v4);
    }
    return acc / (float)ne;
}

/* Q_k(b, a) for a legal a */
static float xm_q(xm_ctx* c, const uint8_t* b, int a, int k) {
    uint8_t nb[16];
    memcpy(nb, b, 16);
    const int r = move_board(nb, a);
    float tail;
    if (k == 1) {
        c->leaves += 1;
        tail = xm_heuristic(c, nb);
    } else {
        tail = xm_chance(c, nb, k - 1);
    }
    return c->w * (float)r + tail;
}

static float xm_value(xm_ctx* c, const uint8_t* b, int k) {
    uint8_t mask[4];
    exact_legal(b, mask);
    float v = 0.0f;
    int any = 0;
    for (int a = 0; a < 4; ++a) {
        if (!mask[a]) continue;
        const float q = xm_q(c, b, a, k);
        if (!any || q > v) v = q;
        any = 1;
    }
    return v;
}

/* q (n*4): Q_depth(board i, a) at 4i + a, NaN where a is illegal; counters[0] += leaves, counters[1] += chance nodes */
void orc_expectimax(const uint8_t* boards, int64_t n, int depth, const float* T, float w, float* q, uint64_t* counters) {
    uint64_t leaves = 0, chance = 0;
#pragma omp parallel for schedule(dynamic, 1) reduction(+ : leaves, chance)
    for (int64_t j = 0; j < n * 4; ++j) {
        const uint8_t* b = boards + 16 * (j / 4);
        const int a = (int)(j % 4);
        uint8_t mask[4];
        exact_legal(b, mask);
        if (!mask[a]) {
            q[j] = NAN;
            continue;
        }
        xm_ctx c = {T, w, 0, 0};
        q[j] = xm_q(&c, b, a, depth);
        leaves += c.leaves;
        chance += c.chance;
    }
    if (counters) {
        counters[0] += leaves;
        counters[1] += chance;
    }
}
