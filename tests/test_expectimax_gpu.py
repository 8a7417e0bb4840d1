"""Expectimax values (g2048_expectimax_values) and the expectimax player on the GPU: q and the counters bit for bit
against orc_expectimax (tests/expectimax_oracle.c, built on the C oracle) with the default and a random row table, a
recursion identity that checks depth 4 through the kernel's own depth-3 values, edge boards, splitting, guard bands
around the outputs, and the player against the oracle's game and a loop over the public API."""
import numpy as np
import pytest
import torch

import g2048
from g2048 import _native as N
from g2048 import engine as E
from oracle import pgx2048_oracle as O

import expectimax_oracle as XO
from test_expectimax_oracle import random_table

pytestmark = pytest.mark.gpu

# hand-built edges: terminal, one legal action (Left), near-full, one empty cell after the move, tiles up to 2^14
TERMINAL = [1, 2, 1, 2, 2, 1, 2, 1, 1, 2, 1, 2, 2, 1, 2, 1]
ONE_LEGAL = [0, 1, 2, 3, 0, 2, 3, 1, 0, 1, 2, 3, 0, 2, 3, 1]
EDGES = [TERMINAL, ONE_LEGAL,
         [1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 1, 2, 3, 4, 0], [0, 3, 1, 3, 2, 4, 2, 4, 3, 5, 3, 5, 4, 6, 4, 6],
         [11, 10, 9, 8, 7, 6, 5, 4, 3, 2, 1, 2, 3, 4, 1, 1],
         [1, 2, 1, 2, 2, 1, 2, 1, 1, 2, 1, 2, 2, 1, 3, 3],  # one merge on the last row: one empty cell after it
         [14, 13, 12, 11, 10, 9, 8, 7, 0, 0, 1, 2, 0, 0, 0, 1], [14, 14, 13, 0, 12, 0, 0, 0, 0, 0, 0, 1, 0, 0, 0, 0]]


def _game_boards(n, mode=E.RNG_PARTITIONABLE, seed=5):
    """Boards of real games at several depths: g2048_play_record's trajectories (DRUL), board t of env e with t spread
    over the episode."""
    subs = E.chain_advance(E.words_tensor([0, seed], "cuda"), mode, 1 + 2 * 2048)
    rec = E.play_record(E.POLICY_DRUL, subs, n, 0, n, mode)
    slot = rec["env_slot"].cpu().numpy()
    length = rec["lengths"].cpu().numpy().astype(np.int64)
    depth = (np.arange(n) * 37) % np.maximum(length, 1)
    return E.boards_numpy(rec["arena_boards"][torch.from_numpy(slot + depth).cuda()])


def _table(name):
    return g2048.expectimax.default_row_table_numpy() if name == "default" else random_table(7)


def _gpu(boards_u8, depth, T, w):
    boards = torch.from_numpy(E.pack_boards(boards_u8)).cuda()
    counters = torch.zeros(2, dtype=torch.int64, device="cuda")
    q = E.expectimax_values(boards, depth, torch.from_numpy(T).cuda(), w, counters)
    return q.cpu().numpy(), counters.cpu().numpy().astype(np.uint64)


def _bits(x):
    return np.asarray(x, np.float32).view(np.uint32)


@pytest.fixture(scope="module")
def boards_2k():
    return np.concatenate([_game_boards(2000), np.asarray(EDGES, np.uint8)])


@pytest.mark.parametrize("depth", [1, 2, 3])
@pytest.mark.parametrize("table", ["default", "random"])
@pytest.mark.parametrize("w", [0.0, 0.5, 1.0])
def test_values_bit_exact_against_oracle(boards_2k, depth, table, w):
    T = _table(table)
    got, counters = _gpu(boards_2k, depth, T, w)
    want, want_counters = XO.expectimax(boards_2k, depth, T, w)
    np.testing.assert_array_equal(_bits(got), _bits(want))
    assert counters.tolist() == want_counters.tolist()
    np.testing.assert_array_equal(~np.isnan(got), O.exact_legal(boards_2k))


@pytest.mark.parametrize("table,w", [("default", 0.0), ("random", 0.5), ("random", 1.0)])
def test_depth_four_bit_exact_against_oracle(table, w):
    boards = np.concatenate([_game_boards(56, seed=9), np.asarray(EDGES, np.uint8)])
    T = _table(table)
    got, counters = _gpu(boards, 4, T, w)
    want, want_counters = XO.expectimax(boards, 4, T, w)
    np.testing.assert_array_equal(_bits(got), _bits(want))
    assert counters.tolist() == want_counters.tolist()


@pytest.mark.parametrize("table,w", [("default", 0.0), ("random", 1.0)])
def test_depth_four_through_the_kernels_depth_three_values(table, w):
    """Q_4(b, a) = w r + fold over the children s + 2@c / s + 4@c of s = move(b, a) of V_3(child), where V_3 is the max
    of the kernel's own depth-3 q over the child's legal actions (0 without one)."""
    boards = _game_boards(300, seed=13)[::3]
    T = _table(table)
    q4, _ = _gpu(boards, 4, T, w)
    legal = O.exact_legal(boards)
    F = np.float32
    pairs = [(i, a) for i in range(boards.shape[0]) for a in range(4) if legal[i, a]][:120]
    children, index = [], []
    for i, a in pairs:
        s, r = O.move(boards[i][None], [a])
        s = s[0]
        cells = np.flatnonzero(s == 0)
        index.append((i, a, int(r[0]), len(children), len(cells)))
        for c in cells:
            for v in (1, 2):
                ch = s.copy()
                ch[c] = v
                children.append(ch)
    q3, _ = _gpu(np.asarray(children, np.uint8), 3, T, w)
    v3 = np.where(np.isnan(q3), -np.inf, q3).max(axis=1).astype(np.float32)
    v3[np.isnan(q3).all(axis=1)] = 0.0
    for i, a, r, first, ne in index:
        acc = F(0.0)
        for k in range(ne):
            acc = F(acc + F(F(F(0.9) * v3[first + 2 * k]) + F(F(0.1) * v3[first + 2 * k + 1])))
        want = F(F(F(w) * F(r)) + F(acc / F(ne)))
        assert _bits(q4[i, a]) == _bits(want), (i, a)


def test_illegal_terminal_and_empty_calls():
    T = torch.from_numpy(_table("default")).cuda()
    q = E.expectimax_values(torch.from_numpy(E.pack_boards(np.asarray(EDGES[:2], np.uint8))).cuda(), 2, T)
    assert torch.isnan(q[0]).all() and torch.isnan(q[1, 1:]).all() and not torch.isnan(q[1, 0])
    res = g2048.expectimax_values(torch.from_numpy(E.pack_boards(np.asarray(EDGES[:2], np.uint8))).cuda(), depth=2)
    assert res.best_action().tolist() == [0, 0] and res.legal.sum().item() == 1
    empty = E.expectimax_values(torch.zeros(0, dtype=torch.int64, device="cuda"), 3, T)
    assert empty.shape == (0, 4)
    counters = torch.zeros(2, dtype=torch.int64, device="cuda")
    E.expectimax_values(torch.zeros(0, dtype=torch.int64, device="cuda"), 3, T, 0.0, counters)
    assert counters.tolist() == [0, 0]


def test_split_calls_give_the_same_values(boards_2k):
    boards = torch.from_numpy(E.pack_boards(boards_2k[:600])).cuda()
    T = torch.from_numpy(_table("random")).cuda()
    c_whole = torch.zeros(2, dtype=torch.int64, device="cuda")
    c_parts = torch.zeros(2, dtype=torch.int64, device="cuda")
    whole = E.expectimax_values(boards, 2, T, 0.5, c_whole)
    parts = torch.cat([E.expectimax_values(boards[:217], 2, T, 0.5, c_parts), E.expectimax_values(boards[217:], 2, T, 0.5, c_parts)])
    assert torch.equal(whole.view(torch.int32), parts.view(torch.int32))
    assert torch.equal(c_whole, c_parts)


def test_outputs_are_surrounded_by_untouched_guard_bands(monkeypatch):
    from test_guard_bands_gpu import GuardedTorch

    guard = GuardedTorch()
    monkeypatch.setattr(E, "torch", guard)
    T = torch.from_numpy(_table("default")).cuda()
    boards = np.concatenate([_game_boards(64), np.asarray(EDGES, np.uint8)])
    for n in (1, 33, 72):
        b = torch.from_numpy(E.pack_boards(boards[:n])).cuda()
        for depth in (1, 2):
            counters = guard.zeros(2, dtype=torch.int64, device="cuda")
            E.expectimax_values(b, depth, T, 0.5, counters)
    assert len(guard.raw) >= 12
    assert guard.check() == []


# ---------------------------------------------------------------------------------------------- the expectimax player
def _own_loop(seed, B, depth, T, w, mode):
    """The player restated with the public expectimax_values and env_step: every env is searched at every move (a
    finished env has no legal action and gets action 0, which the step ignores)."""
    chain = g2048.keys.KeyChain(seed, mode, "cuda")
    subs = chain.peek(1 + 2 * 4096)
    boards, status = E.env_init(subs[0], B, 0, B, mode)
    lengths = torch.zeros(B, dtype=torch.int64, device="cuda")
    scores = torch.zeros(B, dtype=torch.int64, device="cuda")
    t = 0
    while bool(((status & N.STATUS_DONE) == 0).any()):
        res = g2048.expectimax_values(boards, depth=depth, row_values=T, reward_weight=w)
        alive = (status & N.STATUS_DONE) == 0
        rewards = E.env_step(boards, status, res.best_action().to(torch.int32), subs[2 + 2 * t], B, 0, mode)
        lengths += alive.to(torch.int64)
        scores += rewards.to(torch.int64)
        t += 1
    return boards, lengths, scores


@pytest.mark.parametrize("depth", [1, 2])
@pytest.mark.parametrize("mode", [E.RNG_PARTITIONABLE, E.RNG_ORIGINAL])
def test_expectimax_player_matches_oracle_and_own_loop(depth, mode):
    B, seed, w = 16, 12, 0.5
    T = torch.from_numpy(_table("default")).cuda()
    policy = g2048.ExpectimaxPolicy(depth=depth, row_values=T, reward_weight=w)
    runner = g2048.BatchRunner(seed, policy, rng_mode=mode)
    out = runner.run_eval_batch(B)
    want = XO.expectimax_games(seed, B, depth, _table("default"), w, mode)
    np.testing.assert_array_equal(E.boards_numpy(out["final_boards"]), want["final_boards"])
    np.testing.assert_array_equal(out["lengths"].cpu().numpy(), want["lengths"])
    np.testing.assert_array_equal(out["scores"].cpu().numpy(), want["scores"])
    boards, lengths, scores = _own_loop(seed, B, depth, T, w, mode)
    assert torch.equal(out["final_boards"], boards)
    assert torch.equal(out["lengths"].to(torch.int64), lengths) and torch.equal(out["scores"].to(torch.int64), scores)
    s = out["summary"]
    assert s["episodes"] == B and s["env_steps"] == int(lengths.sum()) and s["score_sum"] == int(scores.sum())
    assert sum(s["max_tile_hist"].values()) == B and s["loop_steps"] == s["longest"] == int(lengths.max())
    assert runner.chain.position == 1 + 2 * s["loop_steps"]


def test_expectimax_player_only_through_run_eval_batch():
    runner = g2048.BatchRunner(0, g2048.ExpectimaxPolicy(depth=1))
    for call in (runner.run_stats_batch, runner.run_flat_batch, runner.run_packed_batch, runner.run_actions_batch):
        with pytest.raises(ValueError, match="run_eval_batch"):
            call(8)


def test_expectimax_player_beats_drul():
    """Sanity, not parity: depth 2 over the default table plays far better than DRUL on the same seeds.  The oracle's
    own depth-2 games for this seed average 28 797 (computed on the CPU); the bound sits well below that."""
    B = 64
    ex = g2048.BatchRunner(3, g2048.ExpectimaxPolicy(depth=2)).run_eval_batch(B)
    drul = g2048.BatchRunner(3, g2048.act_drul).run_stats_batch(B)
    ex_mean = ex["summary"]["score_sum"] / B
    drul_mean = drul["summary"]["score_sum"] / B
    assert ex_mean > 4 * drul_mean and ex_mean > 10000, (ex_mean, drul_mean)
