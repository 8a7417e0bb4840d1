"""CPU checks of the TD(0) learner's contract (g2048_td_train): orc_td_train (tests/td_oracle.c, built on the expectimax
oracle and the C oracle) against a plain-Python float32 / int64 restatement, the no-update cases, the greedy move
against orc_expectimax, fx at the edges, and the argument checks of the entry point and of TDLearner, which run
before anything touches a device."""
import math

import numpy as np
import pytest

from oracle import c_oracle as CO
from oracle import pgx2048_oracle as O

import expectimax_oracle as XO
import td_oracle as TO
from test_expectimax_oracle import random_table

F = np.float32
ONE_LEGAL = [0, 1, 2, 3, 0, 2, 3, 1, 0, 1, 2, 3, 0, 2, 3, 1]
TERMINAL = [1, 2, 1, 2, 2, 1, 2, 1, 1, 2, 1, 2, 2, 1, 2, 1]
NEAR_END = [1, 2, 1, 2, 2, 1, 2, 1, 1, 2, 1, 2, 2, 1, 3, 3]  # one merge left


def _pack(b):
    return int((np.asarray(b, np.uint64) << (np.arange(16, dtype=np.uint64) * np.uint64(4))).sum())


def _unpack(x):
    return ((np.uint64(x) >> (np.arange(16, dtype=np.uint64) * np.uint64(4))) & np.uint64(15)).astype(np.int32)


def _lines(b):
    return [sum(int(b[4 * ln + j if ln < 4 else 4 * j + ln - 4]) << (4 * j) for j in range(4)) for ln in range(8)]


def _H(T, b):
    h = None
    for idx in _lines(b):
        h = T[idx] if h is None else F(h + T[idx])
    return h


def _fx(d):
    c = F(min(max(F(d), F(-(2.0 ** 24))), F(2.0 ** 24)))
    return int(np.rint(F(c * F(4096.0))))


def _py_train(st, alpha, subs, mode):
    """The contract step by step in plain Python with np.float32 scalars and Python ints; the game (init, spawn) is
    the C oracle's, keyed per env."""
    T = st.T.copy()
    boards, after = [int(x) for x in st.boards], [int(x) for x in st.after]
    scores, lengths = [int(x) for x in st.scores], [int(x) for x in st.lengths]
    stats = st.stats.astype(np.int64).copy()
    n = len(boards)
    for sub in np.asarray(subs, np.uint32).reshape(-1, 2):
        keys = CO.split(sub, n, mode)
        acc, cnt = {}, {}
        for e in range(n):
            s = _unpack(boards[e])
            legal = O.exact_legal(s[None])[0]
            target, best = F(0.0), None
            for a in range(4):
                if legal[a]:
                    nb, r = O.move(s[None], [a])
                    q = F(F(r[0]) + _H(T, nb[0]))
                    if best is None or q > target:
                        target, best = q, (a, nb[0], int(r[0]))
            if after[e]:
                fx = _fx(F(target - _H(T, _unpack(after[e]))))
                for idx in _lines(_unpack(after[e])):
                    acc[idx] = acc.get(idx, 0) + fx
                    cnt[idx] = cnt.get(idx, 0) + 1
            if best is None:
                me = int(s.max())
                stats[0] += 1
                stats[1] += lengths[e]
                stats[2] += scores[e]
                stats[4] += int(me == 15)
                stats[5] = max(stats[5], lengths[e])
                stats[6] += 1 << me
                stats[7] += (1 << me) ** 2
                stats[16 + me] += 1
                b, _ = CO.env_init(keys[e][None], mode)
                boards[e], after[e], scores[e], lengths[e] = _pack(b[0]), 0, 0, 0
            else:
                a, sa, r = best
                b, _, _, _ = CO.env_step(s[None].astype(np.uint8), legal[None].astype(np.uint8), np.zeros(1, np.uint8),
                                         [a], keys[e][None], mode)
                boards[e], after[e] = _pack(b[0]), _pack(sa)
                scores[e] += r
                lengths[e] += 1
        for i in sorted(cnt):
            T[i] = F(T[i] + F(F(alpha) * F(acc[i] / (4096.0 * cnt[i]))))
    return T, boards, after, scores, lengths, stats


def _start(mode, seed=4):
    """Envs in mid-game, one at the end of its game and one a move away from it, most with an afterstate."""
    key = np.array([0, seed], np.uint32)
    st = TO.fresh(key, 5, mode, random_table(seed) * F(1e-3))
    _, subs = CO.chain(key, mode, 30)
    TO.train(st, 0.01, subs, mode)  # play some moves so that afterstates exist
    st.boards[3], st.after[3] = _pack(TERMINAL), _pack(ONE_LEGAL)
    st.boards[4], st.after[4] = _pack(NEAR_END), _pack(TERMINAL)
    st.stats[:] = 0
    return st


@pytest.mark.parametrize("mode", [CO.PARTITIONABLE, CO.ORIGINAL])
@pytest.mark.parametrize("alpha", [1.0 / 1024, 0.05])
def test_orc_td_train_matches_python_restatement(mode, alpha):
    st = _start(mode)
    _, subs = CO.chain(np.array([3, 9], np.uint32), mode, 6)
    T, boards, after, scores, lengths, stats = _py_train(st, alpha, subs, mode)
    got = TO.train(st.copy(), alpha, subs, mode)
    np.testing.assert_array_equal(got.T.view(np.uint32), T.view(np.uint32))
    assert got.boards.tolist() == boards and got.after.tolist() == after
    assert got.scores.tolist() == scores and got.lengths.tolist() == lengths
    assert got.stats.astype(np.int64).tolist() == stats.tolist()
    assert stats[0] >= 1 and not np.array_equal(T, st.T)  # an episode ended and T moved


def test_alpha_zero_leaves_the_table_unchanged():
    st = _start(CO.PARTITIONABLE)
    _, subs = CO.chain(np.array([0, 1], np.uint32), CO.PARTITIONABLE, 12)
    got = TO.train(st.copy(), 0.0, subs, CO.PARTITIONABLE)
    np.testing.assert_array_equal(got.T.view(np.uint32), st.T.view(np.uint32))
    assert not np.array_equal(got.boards, st.boards)


def test_first_step_from_fresh_envs_makes_no_update():
    key = np.array([0, 17], np.uint32)
    T0 = random_table(2)
    st = TO.fresh(key, 64, CO.ORIGINAL, T0)
    _, subs = CO.chain(key, CO.ORIGINAL, 2)
    TO.train(st, 0.05, subs[:1], CO.ORIGINAL)
    np.testing.assert_array_equal(st.T.view(np.uint32), T0.view(np.uint32))
    assert (st.after != 0).all() and (st.lengths == 1).all()
    TO.train(st, 0.05, subs[1:], CO.ORIGINAL)
    assert not np.array_equal(st.T, T0)


def test_greedy_move_is_expectimax_depth_one_with_reward_weight_one():
    mode = CO.PARTITIONABLE
    st = _start(mode, seed=11)
    before = st.copy()
    _, subs = CO.chain(np.array([1, 2], np.uint32), mode, 1)
    TO.train(st, 0.05, subs, mode)
    boards = np.stack([_unpack(x) for x in before.boards]).astype(np.uint8)
    q, _ = XO.expectimax(boards, 1, before.T, 1.0)
    best = XO.best_actions(q)
    legal = O.exact_legal(boards)
    for e in range(boards.shape[0]):
        if legal[e].any():
            want, _ = O.move(boards[e][None], [best[e]])
            assert int(st.after[e]) == _pack(want[0]), e
        else:
            assert int(st.after[e]) == 0 and int(st.lengths[e]) == 0


def test_fx_clamps_and_rounds_to_nearest_even():
    u = 1.0 / 4096
    assert [TO.fx(k * u) for k in (0.5, 1.5, 2.5, -0.5, -1.5, -2.5, 3.0)] == [0, 2, 2, 0, -2, -2, 3]
    assert TO.fx(2.0 ** 24) == 2 ** 36 and TO.fx(-(2.0 ** 24)) == -(2 ** 36)
    assert TO.fx(3e38) == 2 ** 36 and TO.fx(-math.inf) == -(2 ** 36) and TO.fx(math.inf) == 2 ** 36
    below = float(np.nextafter(F(2.0 ** 24), F(0.0)))
    assert TO.fx(below) == int(below * 4096) == 2 ** 36 - 2 ** 12
    for d in (0.3, -7.77, 12345.678, -1e-7):
        assert TO.fx(d) == _fx(d)


def test_td_train_rejects_bad_arguments_before_any_launch():
    from g2048 import _native as N

    def rc(n=4, alpha=0.01, n_steps=3, boards=8, after=8, scores=8, lengths=8, T=8, subs=8, scratch=8, stats=None):
        return N.lib.g2048_td_train(boards, after, scores, lengths, n, T, alpha, subs, n_steps, 1, scratch, stats, None)

    assert rc(n=0) == -1 and "n must" in N.last_error()
    assert rc(n=(1 << 20) + 1) == -1 and "n must" in N.last_error()
    assert rc(n_steps=-1) == -1 and "n_steps" in N.last_error()
    for alpha in (-0.5, math.nan, math.inf):
        assert rc(alpha=alpha) == -1 and "alpha" in N.last_error()
    assert rc(boards=None) == -1 and "pointers" in N.last_error()
    assert rc(scratch=None) == -1 and "pointers" in N.last_error()
    assert rc(subs=None) == -1 and "pointers" in N.last_error()
    assert rc(after=12) == -1 and "aligned" in N.last_error()
    assert rc(stats=4) == -1 and "aligned" in N.last_error()
    assert rc(scores=10) == -1 and "aligned" in N.last_error()
    assert rc(n_steps=0, subs=None) == 0  # nothing to do
    assert N.lib.g2048_td_scratch_bytes() == 65536 * 12
    for n, alpha, steps in ((0, 0.1, 1), (1 << 21, 0.1, 1), (4, -1.0, 1), (4, math.nan, 1), (4, 0.1, -1)):
        assert TO.train_rc(n, alpha, steps) == -1
    assert TO.train_rc(4, 0.1, 0) == 0


def test_td_learner_checks_its_arguments_before_any_launch():
    import g2048

    for kw in (dict(batch_size=0), dict(batch_size=(1 << 20) + 1), dict(alpha=-0.1), dict(alpha=math.nan),
               dict(alpha=1e39), dict(table=np.zeros(100, np.float32)), dict(table=np.full(65536, np.inf, np.float32))):
        args = dict(init_seed=0, batch_size=8)
        args.update(kw)
        with pytest.raises(ValueError):
            g2048.TDLearner(**args)
