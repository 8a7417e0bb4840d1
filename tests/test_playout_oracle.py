"""CPU checks of the Monte-Carlo playout contract (g2048_playout_values): orc_playout (tests/playout_oracle.c, built on
the C oracle) against the numpy oracle's env_step / act_randomly / act_drul composed by hand, and the entry point's
argument checks, which run before anything touches a device."""
import numpy as np
import pytest

from oracle import c_oracle as CO
from oracle import pgx2048_oracle as O

import playout_oracle as PO


def _boards(seed, depths, mode):
    """Boards of real games: env.init and `depth` random-policy steps (the C oracle), one board per depth."""
    keys = CO.split(np.array([0, seed], np.uint32), 2 * len(depths) + 1, mode)
    boards, masks = CO.env_init(keys[:len(depths)], mode)
    done = np.zeros(len(depths), np.uint8)
    for t in range(max(depths)):
        step = CO.split(keys[len(depths) + t % len(depths)], 2 * len(depths), mode)
        acts, _ = CO.act(step[:len(depths)], masks, CO.RANDOM, mode)
        nb, nm, nd, _ = CO.env_step(boards, masks, done, acts, step[len(depths):], mode)
        live = np.array([t < d for d in depths])
        boards[live], masks[live], done[live] = nb[live], nm[live], nd[live]
    return boards


def _numpy_playouts(boards, ids, n_global, K, subs, policy, mode):
    """The contract restated with the numpy oracle, all playouts of the call as one batch."""
    n = boards.shape[0]
    P = n_global * 4 * K
    max_steps = (subs.shape[0] - 1) // 2
    i, a, k = np.meshgrid(np.arange(n), np.arange(4), np.arange(K), indexing="ij")
    i, a, k = i.ravel(), a.ravel(), k.ravel()
    legal0 = O.exact_legal(boards)
    keep = legal0[i, a]
    i, a, k = i[keep], a[keep], k[keep]
    p = (ids[i] * 4 + a) * K + k
    b = boards[i].astype(np.int32)
    m = b.shape[0]
    state = O.State(b, O.exact_legal(b), np.zeros((m, 1), np.float32), np.zeros(m, bool), np.zeros(m, bool))
    score = np.zeros(m, np.uint64)
    steps = np.zeros(m, np.uint64)
    for t in range(max_steps):
        alive = ~state.terminated
        if not alive.any():
            break
        if t == 0:
            acts = a.astype(np.int32)
        elif policy == CO.RANDOM:
            ka = O.split((subs[1 + 2 * t, 0], subs[1 + 2 * t, 1]), P, mode)
            acts, _ = O.act_randomly((ka[0][p], ka[1][p]), state.legal_action_mask, mode)
        else:
            acts = O.act_drul(state.legal_action_mask)
        ks = O.split((subs[2 + 2 * t, 0], subs[2 + 2 * t, 1]), P, mode)
        state = O.env_step(state, acts, (ks[0][p], ks[1][p]), mode)
        score += np.where(alive, state.rewards[:, 0], 0).astype(np.uint64)
        steps += alive.astype(np.uint64)
    rec = i * 4 + a
    out = {f: np.zeros(n * 4, np.uint64) for f in ("score_sum", "score_sq_sum", "steps_sum", "playouts", "cut_short")}
    np.add.at(out["score_sum"], rec, score)
    np.add.at(out["score_sq_sum"], rec, score * score)
    np.add.at(out["steps_sum"], rec, steps)
    np.add.at(out["playouts"], rec, 1)
    np.add.at(out["cut_short"], rec, (~state.terminated).astype(np.uint64))
    return {f: v.reshape(n, 4) for f, v in out.items()}


@pytest.mark.parametrize("mode", [CO.PARTITIONABLE, CO.ORIGINAL])
@pytest.mark.parametrize("policy", [CO.RANDOM, CO.DRUL])
def test_orc_playout_matches_numpy_oracle(mode, policy):
    boards = _boards(11 + policy, [0, 3, 20, 60], mode)
    # a board with one legal action (Left only) and a terminal one
    one_legal = np.array([0, 1, 2, 3, 0, 2, 3, 1, 0, 1, 2, 3, 0, 2, 3, 1], np.uint8)
    terminal = np.array([1, 2, 1, 2, 2, 1, 2, 1, 1, 2, 1, 2, 2, 1, 2, 1], np.uint8)
    boards = np.concatenate([boards, one_legal[None], terminal[None]])
    assert O.exact_legal(one_legal[None]).sum() == 1 and O.exact_legal(terminal[None]).sum() == 0
    ids = np.array([7, 2, 9, 0, 4, 5], np.int64)  # permuted, strided global ids in a batch of 10 boards
    K, max_steps = 3, 40
    _, subs = CO.chain(np.array([0, 5 + mode], np.uint32), mode, 1 + 2 * max_steps)
    got = PO.playout(boards, K, subs, policy, mode, ids=ids, n_global=10)
    want = _numpy_playouts(boards, ids, 10, K, subs, policy, mode)
    for f in want:
        np.testing.assert_array_equal(got[f].astype(np.uint64), want[f], err_msg=f)
    legal = O.exact_legal(boards)
    np.testing.assert_array_equal(got["playouts"], K * legal)
    assert got["cut_short"].sum() > 0  # playouts that reach max_steps ...
    if policy == CO.RANDOM:
        assert got["cut_short"].sum() < got["playouts"].sum()  # ... and, with the short random games, ones that end


def test_orc_playout_board_lo_equals_id_list():
    mode = CO.PARTITIONABLE
    boards = _boards(3, [5, 10, 15], mode)
    _, subs = CO.chain(np.array([0, 9], np.uint32), mode, 1 + 2 * 64)
    a = PO.playout(boards, 2, subs, CO.RANDOM, mode, board_lo=4, n_global=8)
    b = PO.playout(boards, 2, subs, CO.RANDOM, mode, ids=np.array([4, 5, 6]), n_global=8)
    for f in a:
        np.testing.assert_array_equal(a[f], b[f])


def test_playout_values_rejects_bad_arguments_before_any_launch():
    from g2048 import _native as N

    def rc(policy=0, n=4, ids=None, board_lo=0, n_global=16, K=8, n_subs=5, mode=1):
        return N.lib.g2048_playout_values(policy, None, n, ids, board_lo, n_global, K, 8, n_subs, mode, None, None, None, None)

    assert rc() == -1 and "pointers" in N.last_error()  # valid sizes: only the NULL pointers are wrong
    assert rc(n_global=1 << 29, K=1) == -1 and "2^31" in N.last_error()  # P = 2^31
    assert rc(n_global=(1 << 29) - 1, K=1, n=0) == 0  # P = 2^31 - 4 is allowed (nothing to do for n = 0)
    assert rc(K=0) == -1 and "playouts" in N.last_error()
    assert rc(policy=2) == -1 and "policy" in N.last_error()
    assert rc(mode=2) == -1 and "rng_mode" in N.last_error()
    assert rc(n_subs=2) == -1 and "n_subs" in N.last_error()
    assert rc(board_lo=13) == -1 and "board_lo" in N.last_error()
    assert rc(ids=8, board_lo=1) == -1 and "board_lo" in N.last_error()
