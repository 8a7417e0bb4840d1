/* N-tuple networks restated on the CPU: the value V, expectimax with V at the leaves, and batched TD(0) learning of
 * the weights.  TEST INFRASTRUCTURE ONLY.
 *
 * tests/td_oracle.c is included whole (and with it the expectimax oracle and the C oracle), so the move, the legal
 * mask, the env init / step, fx and the statistics are the code the row-table oracles use.  tests/ntuple_oracle.py
 * compiles it (gcc -O2 -fopenmp -shared -fPIC -ffp-contract=off).  Every float operation is written in the order of
 * the contract in include/g2048.h (g2048_ntuple_td_train, g2048_expectimax_values_ntuple).
 */
#include "td_oracle.c"

/* G2048TuplePlacement */
typedef struct {
    uint32_t offset;
    uint8_t n_cells;
    uint8_t cells[6];
    uint8_t reserved;
} nt_placement;

typedef struct {
    const nt_placement* pl;
    int n_pl;
    const float* W;
    float w;
    uint64_t leaves, chance;
} nt_ctx;

/* the networks g2048_ntuple_td_train accepts: 0, or -1 */
static int nt_valid(const nt_placement* pl, int n_pl, int64_t n_weights) {
    if (n_pl < 1 || n_pl > 64 || n_weights < 1 || n_weights > (1ll << 28)) return -1;
    for (int p = 0; p < n_pl; ++p) {
        const int k = pl[p].n_cells;
        if (k < 1 || k > 6 || pl[p].reserved) return -1;
        for (int j = 0; j < k; ++j) {
            if (pl[p].cells[j] >= 16) return -1;
            for (int i = 0; i < j; ++i)
                if (pl[p].cells[i] == pl[p].cells[j]) return -1;
        }
        if ((int64_t)pl[p].offset + (1ll << (4 * k)) > n_weights) return -1;
    }
    return 0;
}

/* off_p + idx_p(b) */
static uint32_t nt_entry(const nt_placement* p, const uint8_t* b) {
    uint32_t idx = 0;
    for (int j = 0; j < p->n_cells; ++j) idx |= (uint32_t)b[p->cells[j]] << (4 * j);
    return p->offset + idx;
}

/* V(b): the placements in order, left to right from the first term */
static float nt_value(const nt_placement* pl, int n_pl, const float* W, const uint8_t* b) {
    float v = W[nt_entry(&pl[0], b)];
    for (int p = 1; p < n_pl; ++p) v = v + W[nt_entry(&pl[p], b)];
    return v;
}

/* out[i] = V(boards[i]) for packed boards; 0, or -1 for an invalid network */
int orc_ntuple_value(const uint64_t* boards, int64_t n, const nt_placement* pl, int n_pl, const float* W,
                     int64_t n_weights, float* out) {
    if (nt_valid(pl, n_pl, n_weights)) return -1;
    for (int64_t i = 0; i < n; ++i) {
        uint8_t b[16];
        td_unpack(boards[i], b);
        out[i] = nt_value(pl, n_pl, W, b);
    }
    return 0;
}

/* ---- expectimax with V at the leaves: orc_expectimax's tree and float order (tests/expectimax_oracle.c) */
static float nt_xm_value(nt_ctx* c, const uint8_t* b, int k);

static float nt_xm_chance(nt_ctx* c, const uint8_t* s, int k) {
    c->chance += 1;
    float acc = 0.0f;
    int ne = 0;
    for (int cell = 0; cell < 16; ++cell) {
        if (s[cell]) continue;
        ++ne;
        uint8_t ch[16];
        memcpy(ch, s, 16);
        ch[cell] = 1;
        const float v2 = nt_xm_value(c, ch, k);
        ch[cell] = 2;
        const float v4 = nt_xm_value(c, ch, k);
        acc = acc + (0.9f * v2 + 0.1f * v4);
    }
    return acc / (float)ne;
}

static float nt_xm_q(nt_ctx* c, const uint8_t* b, int a, int k) {
    uint8_t nb[16];
    memcpy(nb, b, 16);
    const int r = move_board(nb, a);
    float tail;
    if (k == 1) {
        c->leaves += 1;
        tail = nt_value(c->pl, c->n_pl, c->W, nb);
    } else {
        tail = nt_xm_chance(c, nb, k - 1);
    }
    return c->w * (float)r + tail;
}

static float nt_xm_value(nt_ctx* c, const uint8_t* b, int k) {
    uint8_t mask[4];
    exact_legal(b, mask);
    float v = 0.0f;
    int any = 0;
    for (int a = 0; a < 4; ++a) {
        if (!mask[a]) continue;
        const float q = nt_xm_q(c, b, a, k);
        if (!any || q > v) v = q;
        any = 1;
    }
    return v;
}

/* boards (n, 16) exponents; q (n*4): Q_depth(board i, a) at 4i + a, NaN where a is illegal; counters[0] += leaves,
 * counters[1] += chance nodes.  0, or -1 for an invalid network or depth. */
int orc_ntuple_expectimax(const uint8_t* boards, int64_t n, int depth, const nt_placement* pl, int n_pl, const float* W,
                          int64_t n_weights, float w, float* q, uint64_t* counters) {
    if (depth < 1 || depth > 4 || nt_valid(pl, n_pl, n_weights)) return -1;
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
        nt_ctx c = {pl, n_pl, W, w, 0, 0};
        q[j] = nt_xm_q(&c, b, a, depth);
        leaves += c.leaves;
        chance += c.chance;
    }
    if (counters) {
        counters[0] += leaves;
        counters[1] += chance;
    }
    return 0;
}

/* ---- g2048_ntuple_td_train over n envs for n_steps steps (subs: (n_steps, 2)): orc_td_train with V in place of H
 * and the placements in place of the 8 lines.  boards / after / scores / lengths and W are updated in place; stats (32
 * words, may be NULL) is accumulated in g2048_play's layout.  Returns 0, or -1 for the arguments the entry point
 * rejects. */
int orc_ntuple_td_train(uint64_t* boards, uint64_t* after, uint32_t* scores, uint32_t* lengths, int64_t n,
                        const nt_placement* pl, int n_pl, float* W, int64_t n_weights, float alpha, const uint32_t* subs,
                        int64_t n_steps, int mode, uint64_t* stats) {
    if (n < 1 || n > (1ll << 20) || n_steps < 0 || !(alpha >= 0.0f && alpha <= 3.402823466e38f)) return -1;
    if (nt_valid(pl, n_pl, n_weights)) return -1;
    int64_t* acc = calloc((size_t)n_weights, sizeof(int64_t));
    uint32_t* cnt = calloc((size_t)n_weights, sizeof(uint32_t));
    uint32_t* touched = malloc(sizeof(uint32_t) * (size_t)(n * n_pl));
    int64_t* fx = malloc(sizeof(int64_t) * n);
    uint8_t* ended = malloc(n);
    uint64_t* old_after = malloc(sizeof(uint64_t) * n);
    uint64_t* old_board = malloc(sizeof(uint64_t) * n);
    uint32_t* old_length = malloc(sizeof(uint32_t) * n);
    uint32_t* old_score = malloc(sizeof(uint32_t) * n);
    for (int64_t t = 0; t < n_steps; ++t) {
        const key_t2 sub = {subs[2 * t], subs[2 * t + 1]};
#pragma omp parallel for schedule(static)
        for (int64_t e = 0; e < n; ++e) {
            uint8_t s[16], mask[4];
            td_unpack(boards[e], s);
            exact_legal(s, mask);
            float target = 0.0f;
            int best = -1;
            uint8_t sbest[16];
            int rbest = 0;
            for (int a = 0; a < 4; ++a) {
                if (!mask[a]) continue;
                uint8_t nb[16];
                memcpy(nb, s, 16);
                const int r = move_board(nb, a);
                const float q = (float)r + nt_value(pl, n_pl, W, nb);
                if (best < 0 || q > target) {
                    target = q;
                    best = a;
                    memcpy(sbest, nb, 16);
                    rbest = r;
                }
            }
            old_after[e] = after[e];
            old_board[e] = boards[e];
            old_length[e] = lengths[e];
            old_score[e] = scores[e];
            fx[e] = 0;
            if (after[e] != 0) {
                uint8_t ab[16];
                td_unpack(after[e], ab);
                fx[e] = orc_td_fx(target - nt_value(pl, n_pl, W, ab));
            }
            const key_t2 k = split_at(sub, (uint32_t)n, (uint32_t)e, mode);
            ended[e] = best < 0;
            if (best < 0) {
                uint8_t b[16], m[4];
                init_one(k, mode, b, m);
                boards[e] = td_pack(b);
                after[e] = 0;
                scores[e] = 0;
                lengths[e] = 0;
            } else {
                uint8_t b[16], m[4], done = 0;
                memcpy(b, s, 16);
                memcpy(m, mask, 4);
                step_one(b, m, &done, best, k, mode);
                boards[e] = td_pack(b);
                after[e] = td_pack(sbest);
                scores[e] += (uint32_t)rbest;
                lengths[e] += 1;
            }
        }
        int64_t n_touched = 0;
        for (int64_t e = 0; e < n; ++e) {
            if (old_after[e] != 0) {
                uint8_t ab[16];
                td_unpack(old_after[e], ab);
                for (int p = 0; p < n_pl; ++p) {
                    const uint32_t i = nt_entry(&pl[p], ab);
                    if (cnt[i] == 0) touched[n_touched++] = i;
                    acc[i] += fx[e];
                    cnt[i] += 1;
                }
            }
            if (ended[e] && stats) {
                uint8_t b[16];
                td_unpack(old_board[e], b);
                int me = 0, has15 = 0;
                for (int i = 0; i < 16; ++i) {
                    if (b[i] > me) me = b[i];
                    has15 |= b[i] == 15;
                }
                const uint64_t tile = 1ull << me;
                stats[0] += 1;
                stats[1] += old_length[e];
                stats[2] += old_score[e];
                stats[4] += (uint64_t)has15;
                if (old_length[e] > stats[5]) stats[5] = old_length[e];
                stats[6] += tile;
                stats[7] += tile * tile;
                stats[16 + me] += 1;
            }
        }
        for (int64_t j = 0; j < n_touched; ++j) {  /* every entry with cnt > 0, once */
            const uint32_t i = touched[j];
            W[i] = W[i] + alpha * (float)((double)acc[i] / (4096.0 * (double)cnt[i]));
            acc[i] = 0;
            cnt[i] = 0;
        }
    }
    free(acc);
    free(cnt);
    free(touched);
    free(fx);
    free(ended);
    free(old_after);
    free(old_board);
    free(old_length);
    free(old_score);
    return 0;
}
