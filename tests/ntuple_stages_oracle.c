/* Multi-stage n-tuple networks restated on the CPU: V_S, expectimax with V_S at the leaves, and batched TD(0) and TC
 * learning of the weights (g2048_ntuple_staged_td_train, g2048_ntuple_staged_tc_train,
 * g2048_expectimax_values_ntuple_staged; include/g2048.h).  TEST INFRASTRUCTURE ONLY.
 *
 * tests/ntuple_tc_oracle.c is included whole (and with it the TD, expectimax and C oracles), so the move, the legal
 * mask, the env init / step, fx, nt_entry and the statistics are the code the unstaged oracles use.  What is repeated
 * here is only what computes an entry: every index of a board b is stage(b) * stride further on.  The step loop is
 * orc_ntuple_td_train's / orc_ntuple_tc_train's, with the stage base of each valued board.  tests/ntuple_stages_oracle.py
 * compiles it (gcc -O2 -fopenmp -shared -fPIC -ffp-contract=off).
 */
#include "ntuple_tc_oracle.c"

/* G2048TupleStages */
typedef struct {
    uint32_t stride;
    uint8_t n_thresholds;
    uint8_t thresholds[15];
} nt_stages;

/* the stages the staged entry points accept, for a valid network: 0, or -1 */
static int nt_stages_valid(const nt_stages* st, const nt_placement* pl, int n_pl, int64_t n_weights) {
    if (!st || st->n_thresholds > 15) return -1;
    for (int j = 0; j < 15; ++j) {
        const int t = st->thresholds[j];
        if (j >= st->n_thresholds) {
            if (t) return -1;
        } else if (t < 1 || t > 15 || (j > 0 && t <= st->thresholds[j - 1])) {
            return -1;
        }
    }
    if ((st->n_thresholds == 0) != (st->stride == 0)) return -1;
    for (int p = 0; p < n_pl; ++p)
        if ((int64_t)st->n_thresholds * st->stride + pl[p].offset + (1ll << (4 * pl[p].n_cells)) > n_weights) return -1;
    return 0;
}

/* stage(b) * stride: stage(b) = the number of thresholds that the largest exponent of b reaches */
static uint32_t nt_stage_base(const nt_stages* st, const uint8_t* b) {
    int me = 0;
    for (int c = 0; c < 16; ++c)
        if (b[c] > me) me = b[c];
    uint32_t stage = 0;
    for (int j = 0; j < st->n_thresholds; ++j) stage += me >= st->thresholds[j];
    return stage * st->stride;
}

/* V_S(b): nt_value's order, every entry at the board's stage base */
static float nt_s_value(const nt_placement* pl, int n_pl, const nt_stages* st, const float* W, const uint8_t* b) {
    const uint32_t base = nt_stage_base(st, b);
    float v = W[base + nt_entry(&pl[0], b)];
    for (int p = 1; p < n_pl; ++p) v = v + W[base + nt_entry(&pl[p], b)];
    return v;
}

/* out[i] = V_S(boards[i]) for packed boards; 0, or -1 for an invalid network or stages */
int orc_ntuple_staged_value(const uint64_t* boards, int64_t n, const nt_placement* pl, int n_pl, const nt_stages* st,
                            const float* W, int64_t n_weights, float* out) {
    if (nt_valid(pl, n_pl, n_weights) || nt_stages_valid(st, pl, n_pl, n_weights)) return -1;
    for (int64_t i = 0; i < n; ++i) {
        uint8_t b[16];
        td_unpack(boards[i], b);
        out[i] = nt_s_value(pl, n_pl, st, W, b);
    }
    return 0;
}

/* ---- expectimax with V_S at the leaves: orc_ntuple_expectimax's tree and float order */
typedef struct {
    nt_ctx c;
    const nt_stages* st;
} nt_s_ctx;

static float nt_s_xm_value(nt_s_ctx* c, const uint8_t* b, int k);

static float nt_s_xm_chance(nt_s_ctx* c, const uint8_t* s, int k) {
    c->c.chance += 1;
    float acc = 0.0f;
    int ne = 0;
    for (int cell = 0; cell < 16; ++cell) {
        if (s[cell]) continue;
        ++ne;
        uint8_t ch[16];
        memcpy(ch, s, 16);
        ch[cell] = 1;
        const float v2 = nt_s_xm_value(c, ch, k);
        ch[cell] = 2;
        const float v4 = nt_s_xm_value(c, ch, k);
        acc = acc + (0.9f * v2 + 0.1f * v4);
    }
    return acc / (float)ne;
}

static float nt_s_xm_q(nt_s_ctx* c, const uint8_t* b, int a, int k) {
    uint8_t nb[16];
    memcpy(nb, b, 16);
    const int r = move_board(nb, a);
    float tail;
    if (k == 1) {
        c->c.leaves += 1;
        tail = nt_s_value(c->c.pl, c->c.n_pl, c->st, c->c.W, nb);
    } else {
        tail = nt_s_xm_chance(c, nb, k - 1);
    }
    return c->c.w * (float)r + tail;
}

static float nt_s_xm_value(nt_s_ctx* c, const uint8_t* b, int k) {
    uint8_t mask[4];
    exact_legal(b, mask);
    float v = 0.0f;
    int any = 0;
    for (int a = 0; a < 4; ++a) {
        if (!mask[a]) continue;
        const float q = nt_s_xm_q(c, b, a, k);
        if (!any || q > v) v = q;
        any = 1;
    }
    return v;
}

/* orc_ntuple_expectimax with V_S: 0, or -1 for an invalid network, stages or depth */
int orc_ntuple_staged_expectimax(const uint8_t* boards, int64_t n, int depth, const nt_placement* pl, int n_pl,
                                 const nt_stages* st, const float* W, int64_t n_weights, float w, float* q,
                                 uint64_t* counters) {
    if (depth < 1 || depth > 4 || nt_valid(pl, n_pl, n_weights) || nt_stages_valid(st, pl, n_pl, n_weights)) return -1;
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
        nt_s_ctx c = {{pl, n_pl, W, w, 0, 0}, st};
        q[j] = nt_s_xm_q(&c, b, a, depth);
        leaves += c.c.leaves;
        chance += c.c.chance;
    }
    if (counters) {
        counters[0] += leaves;
        counters[1] += chance;
    }
    return 0;
}

/* ---- the staged learners over n envs for n_steps steps (subs: (n_steps, 2)): the step loop of orc_ntuple_td_train
 * (E == NULL) or orc_ntuple_tc_train (E and A given), every entry at its board's stage base */
static int nt_s_train(uint64_t* boards, uint64_t* after, uint32_t* scores, uint32_t* lengths, int64_t n,
                      const nt_placement* pl, int n_pl, const nt_stages* st, float* W, int64_t n_weights, double* E,
                      double* A, float alpha, const uint32_t* subs, int64_t n_steps, int mode, uint64_t* stats) {
    const int tc = E != NULL;
    int64_t* acc = calloc((size_t)n_weights, sizeof(int64_t));
    int64_t* abs_acc = calloc((size_t)n_weights, sizeof(int64_t));
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
                const float q = (float)r + nt_s_value(pl, n_pl, st, W, nb);
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
                fx[e] = orc_td_fx(target - nt_s_value(pl, n_pl, st, W, ab));
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
                const uint32_t base = nt_stage_base(st, ab);
                for (int p = 0; p < n_pl; ++p) {
                    const uint32_t i = base + nt_entry(&pl[p], ab);
                    if (cnt[i] == 0) touched[n_touched++] = i;
                    acc[i] += fx[e];
                    abs_acc[i] += fx[e] < 0 ? -fx[e] : fx[e];
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
        for (int64_t j = 0; j < n_touched; ++j) { /* every entry with cnt > 0, once */
            const uint32_t i = touched[j];
            if (tc) {
                const double m = (double)acc[i] / (4096.0 * (double)cnt[i]);
                const double beta = A[i] > 0.0 ? fmin(fabs(E[i]) / A[i], 1.0) : 1.0;
                W[i] = W[i] + alpha * (float)(beta * m);
                E[i] = E[i] + (double)acc[i] / 4096.0;
                A[i] = A[i] + (double)abs_acc[i] / 4096.0;
            } else {
                W[i] = W[i] + alpha * (float)((double)acc[i] / (4096.0 * (double)cnt[i]));
            }
            acc[i] = 0;
            abs_acc[i] = 0;
            cnt[i] = 0;
        }
    }
    free(acc);
    free(abs_acc);
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

static int nt_s_args_valid(int64_t n, const nt_placement* pl, int n_pl, const nt_stages* st, int64_t n_weights,
                           float alpha, int64_t n_steps) {
    if (n < 1 || n > (1ll << 20) || n_steps < 0 || !(alpha >= 0.0f && alpha <= 3.402823466e38f)) return -1;
    if (nt_valid(pl, n_pl, n_weights) || nt_stages_valid(st, pl, n_pl, n_weights)) return -1;
    return 0;
}

/* g2048_ntuple_staged_td_train: 0, or -1 for the arguments the entry point rejects */
int orc_ntuple_staged_td_train(uint64_t* boards, uint64_t* after, uint32_t* scores, uint32_t* lengths, int64_t n,
                               const nt_placement* pl, int n_pl, const nt_stages* st, float* W, int64_t n_weights,
                               float alpha, const uint32_t* subs, int64_t n_steps, int mode, uint64_t* stats) {
    if (nt_s_args_valid(n, pl, n_pl, st, n_weights, alpha, n_steps)) return -1;
    return nt_s_train(boards, after, scores, lengths, n, pl, n_pl, st, W, n_weights, NULL, NULL, alpha, subs, n_steps,
                      mode, stats);
}

/* g2048_ntuple_staged_tc_train (E and A: float64[n_weights], both required): 0, or -1 for the arguments the entry
 * point rejects */
int orc_ntuple_staged_tc_train(uint64_t* boards, uint64_t* after, uint32_t* scores, uint32_t* lengths, int64_t n,
                               const nt_placement* pl, int n_pl, const nt_stages* st, float* W, int64_t n_weights,
                               double* E, double* A, float alpha, const uint32_t* subs, int64_t n_steps, int mode,
                               uint64_t* stats) {
    if (nt_s_args_valid(n, pl, n_pl, st, n_weights, alpha, n_steps) || !E || !A) return -1;
    return nt_s_train(boards, after, scores, lengths, n, pl, n_pl, st, W, n_weights, E, A, alpha, subs, n_steps, mode,
                      stats);
}
