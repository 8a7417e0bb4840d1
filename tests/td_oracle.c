/* Batched TD(0) learning of the row table restated on the CPU.  TEST INFRASTRUCTURE ONLY.
 *
 * tests/expectimax_oracle.c is included whole (and with it the C oracle), so H, move_board and exact_legal are the
 * code the expectimax oracle uses, and env init / step are the oracle's own init_one / step_one with per-env keys.
 * tests/td_oracle.py compiles it (gcc -O2 -fopenmp -shared -fPIC -ffp-contract=off).  Every float operation is written
 * in the order of the contract in include/g2048.h (g2048_td_train).
 */
#include "expectimax_oracle.c"

static void td_unpack(uint64_t x, uint8_t* b) {
    for (int i = 0; i < 16; ++i) b[i] = (uint8_t)((x >> (4 * i)) & 15u);
}

static uint64_t td_pack(const uint8_t* b) {
    uint64_t x = 0;
    for (int i = 0; i < 16; ++i) x |= (uint64_t)(b[i] & 15u) << (4 * i);
    return x;
}

/* fx(d) = rint(clamp(d, -2^24, 2^24) * 4096) as int64, to nearest even (the default rounding mode) */
int64_t orc_td_fx(float d) {
    const float c = fminf(fmaxf(d, -16777216.0f), 16777216.0f);
    return (int64_t)rintf(c * 4096.0f);
}

/* the 8 line indices of b in H's order: rows 0..3, then columns 0..3 */
static void td_lines(const uint8_t* b, uint32_t* idx) {
    for (int line = 0; line < 8; ++line) {
        uint32_t v = 0;
        for (int j = 0; j < 4; ++j) v |= (uint32_t)b[line < 4 ? 4 * line + j : 4 * j + (line - 4)] << (4 * j);
        idx[line] = v;
    }
}

/* g2048_td_train over n envs for n_steps steps (subs: (n_steps, 2)).  boards / after / scores / lengths and T are
 * updated in place; stats (32 words, may be NULL) is accumulated in g2048_play's layout.  Returns 0, or -1 for the
 * arguments g2048_td_train rejects. */
int orc_td_train(uint64_t* boards, uint64_t* after, uint32_t* scores, uint32_t* lengths, int64_t n, float* T, float alpha,
                 const uint32_t* subs, int64_t n_steps, int mode, uint64_t* stats) {
    if (n < 1 || n > (1ll << 20) || n_steps < 0 || !(alpha >= 0.0f && alpha <= 3.402823466e38f)) return -1;
    int64_t* acc = calloc(65536, sizeof(int64_t));
    uint32_t* cnt = calloc(65536, sizeof(uint32_t));
    int64_t* fx = malloc(sizeof(int64_t) * n);
    uint8_t* ended = malloc(n);
    uint64_t* old_after = malloc(sizeof(uint64_t) * n);
    uint64_t* old_board = malloc(sizeof(uint64_t) * n);
    uint32_t* old_length = malloc(sizeof(uint32_t) * n);
    uint32_t* old_score = malloc(sizeof(uint32_t) * n);
    for (int64_t t = 0; t < n_steps; ++t) {
        const key_t2 sub = {subs[2 * t], subs[2 * t + 1]};
        xm_ctx c = {T, 1.0f, 0, 0};
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
                const float q = (float)r + xm_heuristic(&c, nb);
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
                fx[e] = orc_td_fx(target - xm_heuristic(&c, ab));
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
        for (int64_t e = 0; e < n; ++e) {
            if (old_after[e] != 0) {
                uint8_t ab[16];
                uint32_t idx[8];
                td_unpack(old_after[e], ab);
                td_lines(ab, idx);
                for (int l = 0; l < 8; ++l) {
                    acc[idx[l]] += fx[e];
                    cnt[idx[l]] += 1;
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
        for (int i = 0; i < 65536; ++i) {
            if (cnt[i]) {
                T[i] = T[i] + alpha * (float)((double)acc[i] / (4096.0 * (double)cnt[i]));
                acc[i] = 0;
                cnt[i] = 0;
            }
        }
    }
    free(acc);
    free(cnt);
    free(fx);
    free(ended);
    free(old_after);
    free(old_board);
    free(old_length);
    free(old_score);
    return 0;
}
