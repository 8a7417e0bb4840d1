/* Carousel shaping of a multi-stage n-tuple network (g2048_ntuple_carousel_td_train, g2048_ntuple_carousel_tc_train;
 * include/g2048.h) restated on the CPU.  TEST INFRASTRUCTURE ONLY.
 *
 * tests/ntuple_lambda_oracle.c is included whole (and with it the staged, TC, TD, expectimax and C oracles), so V_S, the
 * move, the legal mask, the env init / step, fx, the entries, the window and the statistics are the code the other
 * oracles use.  What is repeated here is only the step loop of nt_l_train, with the start stage, the pool draw against
 * the pool as it was at the start of the step, the recording of stage entries and their commit after the step, and
 * the two statistics words of the shaped episodes.  tests/ntuple_carousel_oracle.py compiles it (gcc -O2 -fopenmp
 * -shared -fPIC -ffp-contract=off).
 */
#include "ntuple_lambda_oracle.c"

/* stage(b): the number of thresholds that the largest exponent of b reaches */
static uint32_t nt_c_stage(const nt_stages* st, const uint8_t* b) {
    int me = 0;
    for (int i = 0; i < 16; ++i)
        if (b[i] > me) me = b[i];
    uint32_t stage = 0;
    for (int j = 0; j < st->n_thresholds; ++j) stage += me >= st->thresholds[j];
    return stage;
}

/* the carousel learners over n envs for n_steps steps (subs: (n_steps, 2)); E NULL is TD; the rings may be NULL when
 * h == 1 (they are then neither read nor written) */
static int nt_c_train(uint64_t* boards, uint64_t* after, uint32_t* scores, uint32_t* lengths, int64_t n,
                      const nt_placement* pl, int n_pl, const nt_stages* st, float* W, int64_t n_weights, double* E,
                      double* A, float alpha, float lambda, int h, uint64_t* hist_after, float* hist_delta,
                      uint32_t* start_stage, uint64_t* pool, const uint32_t* subs, int64_t n_steps, int mode,
                      uint64_t* stats) {
    const int tc = E != NULL;
    const uint32_t S = (uint32_t)st->n_thresholds + 1u;
    float c[NT_MAX_HORIZON];
    nt_l_coefficients(lambda, h, c);
    int64_t* acc = calloc((size_t)n_weights, sizeof(int64_t));
    int64_t* abs_acc = calloc((size_t)n_weights, sizeof(int64_t));
    uint32_t* cnt = calloc((size_t)n_weights, sizeof(uint32_t));
    uint32_t* touched = malloc(sizeof(uint32_t) * (size_t)(n * h * n_pl));
    int64_t* fx = malloc(sizeof(int64_t) * n * h);
    uint64_t* rel = malloc(sizeof(uint64_t) * n * h);
    int* n_rel = malloc(sizeof(int) * n);
    uint8_t* ended = malloc(n);
    uint8_t* shaped = malloc(n);                        /* the ended episode began from a pool board */
    uint64_t* pending = calloc((size_t)n, sizeof(uint64_t)); /* the stage entry of the step, committed after it */
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
            old_board[e] = boards[e];
            old_length[e] = lengths[e];
            old_score[e] = scores[e];
            n_rel[e] = 0;
            const int64_t L = lengths[e];
            /* h = 1 is TD(0) / TC, which updates every afterstate whatever the length */
            if (after[e] != 0 && (h == 1 || (L >= 1 && L < (1ll << 31)))) {
                uint8_t ab[16];
                td_unpack(after[e], ab);
                const float dL = target - nt_s_value(pl, n_pl, st, W, ab);
                if (h == 1) { /* TD(0) / TC: the afterstate itself with its error */
                    rel[e * h] = after[e];
                    fx[e * h] = orc_td_fx(dL);
                    n_rel[e] = 1;
                } else {
                    hist_delta[((L - 1) % h) * n + e] = dL;
                    int64_t lo = L + 1, hi = L;
                    if (best < 0) {
                        lo = L - h + 1 > 1 ? L - h + 1 : 1;
                    } else if (L >= h) {
                        lo = hi = L - h + 1;
                    }
                    for (int64_t m = lo; m <= hi; ++m) {
                        float em = hist_delta[((m - 1) % h) * n + e];
                        for (int k = 1; k < h && m + k <= L; ++k) {
                            const float term = c[k] * hist_delta[((m + k - 1) % h) * n + e];
                            em = em + term;
                        }
                        rel[e * h + n_rel[e]] = hist_after[((m - 1) % h) * n + e];
                        fx[e * h + n_rel[e]] = orc_td_fx(em);
                        n_rel[e] += 1;
                    }
                }
            }
            const key_t2 k = split_at(sub, (uint32_t)n, (uint32_t)e, mode);
            ended[e] = best < 0;
            if (best < 0) {
                const uint32_t c0 = start_stage[e];
                const uint32_t l = c0 + 1u < S ? c0 + 1u : 0u; /* uint32 arithmetic: c0 = 2^32 - 1 also wraps to 0 */
                shaped[e] = c0 != 0u;
                uint64_t b0 = 0;
                if (l >= 1u) {
                    const key_t2 k1 = split_at(k, 2, 0, mode);
                    const uint32_t j = (uint32_t)(((uint64_t)bits_at(k1, 1, 0, mode) * (uint64_t)n) >> 32);
                    b0 = pool[(int64_t)(l - 1u) * n + j]; /* not yet changed in this step: commits follow the loop */
                }
                if (b0) {
                    boards[e] = b0;
                    start_stage[e] = l;
                } else {
                    uint8_t b[16], m[4];
                    init_one(k, mode, b, m);
                    boards[e] = td_pack(b);
                    start_stage[e] = 0;
                }
                after[e] = 0;
                scores[e] = 0;
                lengths[e] = 0;
            } else {
                uint8_t b[16], m[4], done = 0;
                memcpy(b, s, 16);
                memcpy(m, mask, 4);
                step_one(b, m, &done, best, k, mode);
                boards[e] = td_pack(b);
                if (nt_c_stage(st, b) > nt_c_stage(st, s)) pending[e] = boards[e];
                after[e] = td_pack(sbest);
                if (h > 1) hist_after[(L % h) * n + e] = after[e]; /* x_{L+1} */
                scores[e] += (uint32_t)rbest;
                lengths[e] += 1;
            }
        }
        int64_t n_touched = 0;
        for (int64_t e = 0; e < n; ++e) {
            for (int j = 0; j < n_rel[e]; ++j) {
                uint8_t ab[16];
                td_unpack(rel[e * h + j], ab);
                const uint32_t base = nt_stage_base(st, ab);
                const int64_t f = fx[e * h + j];
                for (int p = 0; p < n_pl; ++p) {
                    const uint32_t i = base + nt_entry(&pl[p], ab);
                    if (cnt[i] == 0) touched[n_touched++] = i;
                    acc[i] += f;
                    abs_acc[i] += f < 0 ? -f : f;
                    cnt[i] += 1;
                }
            }
            if (ended[e] && stats && shaped[e]) {
                stats[12] += 1;
                stats[13] += old_length[e];
            } else if (ended[e] && stats) {
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
            if (pending[e]) { /* the commit: visible from the next step's draws */
                uint8_t b[16];
                td_unpack(pending[e], b);
                pool[(int64_t)(nt_c_stage(st, b) - 1u) * n + e] = pending[e];
                pending[e] = 0;
            }
        }
        for (int64_t j = 0; j < n_touched; ++j) {
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
    free(rel);
    free(n_rel);
    free(ended);
    free(shaped);
    free(pending);
    free(old_board);
    free(old_length);
    free(old_score);
    return 0;
}

static int nt_c_args_valid(int64_t n, const nt_placement* pl, int n_pl, const nt_stages* st, int64_t n_weights,
                           float alpha, float lambda, int h, const uint64_t* hist_after, const float* hist_delta,
                           const uint32_t* start_stage, const uint64_t* pool, int64_t n_steps) {
    if (n < 1 || n > (1ll << 20) || n_steps < 0 || !(alpha >= 0.0f && alpha <= 3.402823466e38f)) return -1;
    if (nt_valid(pl, n_pl, n_weights) || !st || nt_stages_valid(st, pl, n_pl, n_weights)) return -1;
    if (st->n_thresholds < 1) return -1;
    if (!(lambda >= 0.0f && lambda <= 1.0f) || h < 1 || h > NT_MAX_HORIZON || n * h > (1ll << 20)) return -1;
    if (h > 1 && (!hist_after || !hist_delta)) return -1;
    if (!start_stage || !pool) return -1;
    return 0;
}

/* g2048_ntuple_carousel_td_train: 0, or -1 for the arguments the entry point rejects */
int orc_ntuple_carousel_td_train(uint64_t* boards, uint64_t* after, uint32_t* scores, uint32_t* lengths, int64_t n,
                                 const nt_placement* pl, int n_pl, const nt_stages* st, float* W, int64_t n_weights,
                                 float alpha, float lambda, int h, uint64_t* hist_after, float* hist_delta,
                                 uint32_t* start_stage, uint64_t* pool, const uint32_t* subs, int64_t n_steps,
                                 int mode, uint64_t* stats) {
    if (nt_c_args_valid(n, pl, n_pl, st, n_weights, alpha, lambda, h, hist_after, hist_delta, start_stage, pool,
                        n_steps))
        return -1;
    return nt_c_train(boards, after, scores, lengths, n, pl, n_pl, st, W, n_weights, NULL, NULL, alpha, lambda, h,
                      hist_after, hist_delta, start_stage, pool, subs, n_steps, mode, stats);
}

/* g2048_ntuple_carousel_tc_train (E and A: float64[n_weights], both required): 0, or -1 for the arguments the entry
 * point rejects */
int orc_ntuple_carousel_tc_train(uint64_t* boards, uint64_t* after, uint32_t* scores, uint32_t* lengths, int64_t n,
                                 const nt_placement* pl, int n_pl, const nt_stages* st, float* W, int64_t n_weights,
                                 double* E, double* A, float alpha, float lambda, int h, uint64_t* hist_after,
                                 float* hist_delta, uint32_t* start_stage, uint64_t* pool, const uint32_t* subs,
                                 int64_t n_steps, int mode, uint64_t* stats) {
    if (nt_c_args_valid(n, pl, n_pl, st, n_weights, alpha, lambda, h, hist_after, hist_delta, start_stage, pool,
                        n_steps) || !E || !A)
        return -1;
    return nt_c_train(boards, after, scores, lengths, n, pl, n_pl, st, W, n_weights, E, A, alpha, lambda, h,
                      hist_after, hist_delta, start_stage, pool, subs, n_steps, mode, stats);
}
