/* Batched temporal coherence learning of an n-tuple network (g2048_ntuple_tc_train, include/g2048.h) restated on the
 * CPU.  TEST INFRASTRUCTURE ONLY.
 *
 * tests/ntuple_oracle.c is included whole, so V, the move, the legal mask, the env init / step, fx and the statistics
 * are the code the TD oracle uses.  orc_ntuple_tc_train is orc_ntuple_td_train's step loop with the second sum
 * (|fx| per entry) and the contract's step 4: beta from E and A before the step, the float update of W, then the
 * double sums E and A.  tests/ntuple_tc_oracle.py compiles it (gcc -O2 -fopenmp -shared -fPIC -ffp-contract=off).
 */
#include "ntuple_oracle.c"

/* g2048_ntuple_tc_train over n envs for n_steps steps (subs: (n_steps, 2)); E and A (float64[n_weights], both
 * required) are updated in place with W and the env state.  Returns 0, or -1 for the arguments the entry point
 * rejects. */
int orc_ntuple_tc_train(uint64_t* boards, uint64_t* after, uint32_t* scores, uint32_t* lengths, int64_t n,
                        const nt_placement* pl, int n_pl, float* W, int64_t n_weights, double* E, double* A,
                        float alpha, const uint32_t* subs, int64_t n_steps, int mode, uint64_t* stats) {
    if (n < 1 || n > (1ll << 20) || n_steps < 0 || !(alpha >= 0.0f && alpha <= 3.402823466e38f)) return -1;
    if (nt_valid(pl, n_pl, n_weights) || !E || !A) return -1;
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
        for (int64_t j = 0; j < n_touched; ++j) {  /* every entry with cnt > 0, once */
            const uint32_t i = touched[j];
            const double m = (double)acc[i] / (4096.0 * (double)cnt[i]);
            const double beta = A[i] > 0.0 ? fmin(fabs(E[i]) / A[i], 1.0) : 1.0;
            W[i] = W[i] + alpha * (float)(beta * m);
            E[i] = E[i] + (double)acc[i] / 4096.0;
            A[i] = A[i] + (double)abs_acc[i] / 4096.0;
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
