/* Monte-Carlo playouts restated on the CPU with the oracle's own game and policies.  TEST INFRASTRUCTURE ONLY.
 *
 * The oracle (oracle/pgx2048_oracle.c) is included whole, so this file uses its Threefry, Pgx step and policies as
 * they are and adds one entry point on top; tests/playout_oracle.py compiles it (gcc -O2 -fopenmp -shared -fPIC
 * -ffp-contract=off, like oracle/Makefile) and checks it against the numpy oracle composed by hand.
 */
#include "../oracle/pgx2048_oracle.c"

/* Monte-Carlo playouts (the contract of g2048_playout_values): for board i (n of them, (n,16) exponents; global id
 * ids[i], or board_lo + i when ids is NULL) and action a, K games.  Playout p = (id*4 + a)*K + k of a batch of
 * P = n_global*4*K: t = 0 plays a and steps with split(subs[2], P)[p]; t >= 1 acts with split(subs[1+2t], P)[p] and
 * steps with split(subs[2+2t], P)[p]; at most max_steps steps.  An action illegal on the start board is not played.
 * Per (i, a) the sums over its playouts of the score (rewards of the playout's steps), its square and the steps, the
 * number of playouts and of those that reached max_steps; all outputs (n*4) are overwritten. */
void orc_playout(const uint8_t* boards, int64_t n, const int64_t* ids, int64_t board_lo, int64_t n_global, int64_t K,
                 const uint32_t* subs, int64_t max_steps, int policy, int mode, uint64_t* score_sum,
                 uint64_t* score_sq_sum, uint64_t* steps_sum, uint32_t* playouts, uint32_t* cut_short) {
    const uint32_t P = (uint32_t)(n_global * 4 * K);
    memset(score_sum, 0, (size_t)n * 4 * sizeof(uint64_t));
    memset(score_sq_sum, 0, (size_t)n * 4 * sizeof(uint64_t));
    memset(steps_sum, 0, (size_t)n * 4 * sizeof(uint64_t));
    memset(playouts, 0, (size_t)n * 4 * sizeof(uint32_t));
    memset(cut_short, 0, (size_t)n * 4 * sizeof(uint32_t));
#pragma omp parallel for schedule(dynamic, 16)
    for (int64_t j = 0; j < n * 4 * K; ++j) {
        const int64_t rec = j / K, i = rec / 4, k = j % K;
        const int a = (int)(rec % 4);
        uint8_t b[16], mask[4], done = 0;
        memcpy(b, boards + 16 * i, 16);
        exact_legal(b, mask);
        if (!mask[a]) continue;
        const int64_t id = ids ? ids[i] : board_lo + i;
        const uint32_t p = (uint32_t)((id * 4 + a) * K + k);
        uint64_t score = 0;
        int64_t t = 0;
        for (; t < max_steps && !done; ++t) {
            key_t2 sa = {subs[2 * (1 + 2 * t)], subs[2 * (1 + 2 * t) + 1]};
            key_t2 ss = {subs[2 * (2 + 2 * t)], subs[2 * (2 + 2 * t) + 1]};
            int act = a;
            if (t > 0) act = policy == POLICY_RANDOM ? act_random_one(split_at(sa, P, p, mode), mask, mode, NULL) : act_drul_one(mask);
            float r = step_one(b, mask, &done, act, split_at(ss, P, p, mode), mode);
            if (r > 0) score += (uint64_t)r;
        }
#pragma omp atomic
        score_sum[rec] += score;
#pragma omp atomic
        score_sq_sum[rec] += score * score;
#pragma omp atomic
        steps_sum[rec] += (uint64_t)t;
#pragma omp atomic
        playouts[rec] += 1u;
        if (!done) {
#pragma omp atomic
            cut_short[rec] += 1u;
        }
    }
}
