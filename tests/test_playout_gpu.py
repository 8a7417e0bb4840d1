"""Monte-Carlo playout values (g2048_playout_values) and the playout-search player on the GPU: every record field bit
for bit against orc_playout (tests/playout_oracle.c, built on the C oracle), consistency with the statistics block,
invariance under splitting the boards over calls, the K = 1 records against a loop of the separately tested entry
points, guard bands around the outputs, and the Monte-Carlo player against the oracle's game."""
import numpy as np
import pytest
import torch

import g2048
from g2048 import _native as N
from g2048 import engine as E
from oracle import c_oracle as CO
from oracle import pgx2048_oracle as O

import playout_oracle as PO

pytestmark = pytest.mark.gpu

MODES = [E.RNG_PARTITIONABLE, E.RNG_ORIGINAL]
POLICIES = [E.POLICY_RANDOM, E.POLICY_DRUL]
# hand-built edges: terminal, one legal action (Left), near-full boards
TERMINAL = [1, 2, 1, 2, 2, 1, 2, 1, 1, 2, 1, 2, 2, 1, 2, 1]
ONE_LEGAL = [0, 1, 2, 3, 0, 2, 3, 1, 0, 1, 2, 3, 0, 2, 3, 1]
NEAR_FULL = [[1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 1, 2, 3, 4, 0], [0, 3, 1, 3, 2, 4, 2, 4, 3, 5, 3, 5, 4, 6, 4, 6],
             [11, 10, 9, 8, 7, 6, 5, 4, 3, 2, 1, 2, 3, 4, 1, 1]]


def _game_boards(n, mode, seed=5):
    """Boards of real games at several depths: g2048_play_record's trajectories (DRUL), board t of env e with
    t spread over the episode."""
    subs = E.chain_advance(E.words_tensor([0, seed], "cuda"), mode, 1 + 2 * 2048)
    rec = E.play_record(E.POLICY_DRUL, subs, n, 0, n, mode)
    slot = rec["env_slot"].cpu().numpy()
    length = rec["lengths"].cpu().numpy().astype(np.int64)
    depth = (np.arange(n) * 37) % np.maximum(length, 1)  # 0 .. length-1
    return rec["arena_boards"][torch.from_numpy(slot + depth).cuda()]


def _edge_boards():
    return np.stack([TERMINAL, ONE_LEGAL] + NEAR_FULL).astype(np.uint8)


def _all_boards(mode):
    game = E.boards_numpy(_game_boards(45, mode))
    return np.concatenate([game, _edge_boards()])  # 50 boards


def _subs(mode, max_steps, seed=3):
    return E.chain_advance(E.words_tensor([0, seed], "cuda"), mode, 1 + 2 * max_steps)


def _gpu(boards_u8, subs, K, policy, mode, **kw):
    boards = torch.from_numpy(E.pack_boards(boards_u8)).cuda()
    stats = torch.zeros(N.PLAY_STATS_WORDS, dtype=torch.int64, device="cuda")
    out = E.playout_values(policy, boards, subs, K, mode, stats=stats, **kw)
    return {k: (v.cpu().numpy() if isinstance(v, torch.Tensor) else v) for k, v in out.items()}


def _assert_records_equal(got, want):
    for f in ("score_sum", "score_sq_sum", "steps_sum", "playouts", "cut_short"):
        np.testing.assert_array_equal(got[f].astype(np.uint64), want[f].astype(np.uint64), err_msg=f)


@pytest.mark.parametrize("K", [1, 7, 64])
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("policy", POLICIES)
def test_records_bit_exact_against_oracle(policy, mode, K):
    boards = _all_boards(mode)
    max_steps = 2048 if K != 7 else 60  # K = 7: short keys, so that playouts are cut
    subs = _subs(mode, max_steps)
    got = _gpu(boards, subs, K, policy, mode)
    want = PO.playout(boards, K, E.words_numpy(subs), policy, mode)
    _assert_records_equal(got, want)
    np.testing.assert_array_equal(got["playouts"], K * O.exact_legal(boards))
    assert got["playouts"][45].sum() == 0 and got["playouts"][46].tolist() == [K, 0, 0, 0]  # terminal, Left only
    if K == 7:
        assert 0 < want["cut_short"].sum() < want["playouts"].sum()
    # the statistics block is the sum over the records
    st = E.play_stats_dict(torch.from_numpy(got["stats"]))
    assert st["episodes"] == int(got["playouts"].sum()) and st["env_steps"] == int(got["steps_sum"].sum())
    assert st["score_sum"] == int(got["score_sum"].sum()) and st["cut_short"] == int(got["cut_short"].sum())
    assert sum(st["max_tile_hist"].values()) == st["episodes"] and st["overflowed"] == 0


@pytest.mark.parametrize("mode", MODES)
def test_id_list_permuted_and_strided(mode):
    boards = _all_boards(mode)
    n = boards.shape[0]
    rng = np.random.default_rng(1)
    ids = rng.permutation(3 * n)[:n].astype(np.int64)  # distinct global ids in a batch of 3 n, in no order
    subs = _subs(mode, 2048)
    got = _gpu(boards, subs, 5, E.POLICY_RANDOM, mode, board_ids=torch.from_numpy(ids).cuda(), n_boards_global=3 * n)
    want = PO.playout(boards, 5, E.words_numpy(subs), E.POLICY_RANDOM, mode, ids=ids, n_global=3 * n)
    _assert_records_equal(got, want)


@pytest.mark.parametrize("policy", POLICIES)
def test_split_calls_give_the_same_records(policy):
    mode = E.RNG_PARTITIONABLE
    boards = _all_boards(mode)
    n, K = boards.shape[0], 9
    subs = _subs(mode, 2048)
    whole = _gpu(boards, subs, K, policy, mode)
    lo = _gpu(boards[:17], subs, K, policy, mode, board_lo=0, n_boards_global=n)
    hi = _gpu(boards[17:], subs, K, policy, mode, board_lo=17, n_boards_global=n)
    for f in ("score_sum", "score_sq_sum", "steps_sum", "playouts", "cut_short"):
        np.testing.assert_array_equal(np.concatenate([lo[f], hi[f]]), whole[f], err_msg=f)
    # by ids: the odd boards, then the even ones
    for part in (np.arange(1, n, 2), np.arange(0, n, 2)):
        ids = torch.from_numpy(part.astype(np.int64)).cuda()
        got = _gpu(boards[part], subs, K, policy, mode, board_ids=ids, n_boards_global=n)
        for f in ("score_sum", "score_sq_sum", "steps_sum", "playouts", "cut_short"):
            np.testing.assert_array_equal(got[f], whole[f][part], err_msg=f)


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("policy", POLICIES)
def test_single_playouts_equal_a_loop_of_env_step_and_act(policy, mode):
    """K = 1: playout p = 4 i + a is env p of a batch of P = 4 n, stepped with g2048_act / g2048_env_step."""
    boards = _all_boards(mode)[[3, 20, 44, 46, 47]]
    n = boards.shape[0]
    P, max_steps = 4 * n, 2048
    subs = _subs(mode, max_steps)
    got = _gpu(boards, subs, 1, policy, mode)
    legal = O.exact_legal(boards)
    mask_bits = (legal * (1 << np.arange(4))).sum(axis=1)
    start = np.repeat(E.pack_boards(boards), 4)
    legal_p = legal.reshape(-1)
    status = np.where(legal_p, np.repeat(mask_bits, 4), N.STATUS_MASK | N.STATUS_DONE).astype(np.uint8)
    b = torch.from_numpy(start).cuda()
    s = torch.from_numpy(status).cuda()
    score = torch.zeros(P, dtype=torch.int64, device="cuda")
    steps = torch.zeros(P, dtype=torch.int64, device="cuda")
    for t in range(max_steps):
        alive = (s & N.STATUS_DONE) == 0
        if not bool(alive.any()):
            break
        if t == 0:
            actions = torch.arange(P, dtype=torch.int32, device="cuda") % 4
        else:
            actions, _ = E.act(policy, s, subs[1 + 2 * t], P, 0, mode)
        rewards = E.env_step(b, s, actions, subs[2 + 2 * t], P, 0, mode)
        score += torch.where(alive, rewards.to(torch.int64), 0)
        steps += alive.to(torch.int64)
    score = score.cpu().numpy().reshape(n, 4)
    steps = steps.cpu().numpy().reshape(n, 4)
    np.testing.assert_array_equal(got["score_sum"], np.where(legal, score, 0))
    np.testing.assert_array_equal(got["steps_sum"], np.where(legal, steps, 0))
    np.testing.assert_array_equal(got["score_sq_sum"], np.where(legal, score * score, 0))


def test_outputs_are_surrounded_by_untouched_guard_bands(monkeypatch):
    from test_guard_bands_gpu import GuardedTorch

    guard = GuardedTorch()
    monkeypatch.setattr(E, "torch", guard)
    mode = E.RNG_PARTITIONABLE
    for n in (1, 33, 50):
        boards = torch.from_numpy(E.pack_boards(_all_boards(mode)[:n])).cuda()
        for policy in POLICIES:
            E.playout_values(policy, boards, _subs(mode, 256), 3, mode)
    assert len(guard.raw) >= 12
    assert guard.check() == []


def test_public_playout_values_summaries():
    boards = torch.from_numpy(E.pack_boards(_all_boards(E.RNG_PARTITIONABLE))).cuda()
    res = g2048.playout_values(boards, 16, key=7)
    want = E.playout_values(E.POLICY_RANDOM, boards, E.split_keys(E.words_tensor([0, 7], "cuda"), 4097, 0, 4097, 1), 16, 1)
    assert torch.equal(res.score_sum, want["score_sum"])
    legal = res.playouts > 0
    assert torch.isnan(res.mean_score[~legal]).all() and torch.isnan(res.std_score[~legal]).all()
    mean = res.score_sum.double() / 16
    assert torch.equal(res.mean_score[legal], mean[legal])
    assert torch.equal(res.mean_length[legal], (res.steps_sum.double() / 16)[legal])
    best = res.best_action()
    assert bool(legal[torch.arange(len(best)), best][legal.any(dim=1)].all())
    masked = torch.where(legal, res.score_sum, -1)
    assert torch.equal(masked.gather(1, best[:, None])[:, 0], masked.max(dim=1).values)
    assert torch.equal(res.best_action("length"), torch.where(legal, res.steps_sum, -1).argmax(dim=1))


# ---------------------------------------------------------------------------------------------- the Monte-Carlo player
def _own_loop(seed, B, K, rollout, criterion, mode, max_steps):
    """The player restated with the public playout_values and env_step: every env is evaluated at every move (a
    finished env has no legal action, so it plays no playout), with its env index as board id in a batch of B."""
    chain = g2048.keys.KeyChain(seed, mode, "cuda")
    subs = chain.peek(1 + 2 * 4096)
    boards, status = E.env_init(subs[0], B, 0, B, mode)
    lengths = torch.zeros(B, dtype=torch.int64, device="cuda")
    scores = torch.zeros(B, dtype=torch.int64, device="cuda")
    t = 0
    while bool(((status & N.STATUS_DONE) == 0).any()):
        res = g2048.playout_values(boards, K, subs[1 + 2 * t], rollout=rollout, max_steps=max_steps, rng_mode=mode)
        alive = (status & N.STATUS_DONE) == 0
        rewards = E.env_step(boards, status, res.best_action(criterion).to(torch.int32), subs[2 + 2 * t], B, 0, mode)
        lengths += alive.to(torch.int64)
        scores += rewards.to(torch.int64)
        t += 1
    return boards, lengths, scores


@pytest.mark.parametrize("rollout,criterion,mode", [(g2048.act_randomly, "score", E.RNG_PARTITIONABLE),
                                                    (g2048.act_drul, "length", E.RNG_ORIGINAL)])
def test_monte_carlo_player_matches_oracle_and_own_loop(rollout, criterion, mode):
    B, K, seed, max_steps = 5, 4, 12, 512
    policy = g2048.MonteCarloPolicy(playouts=K, rollout=rollout, criterion=criterion, max_steps=max_steps)
    runner = g2048.BatchRunner(seed, policy, rng_mode=mode)
    out = runner.run_eval_batch(B)
    again = g2048.BatchRunner(seed, policy, rng_mode=mode).run_eval_batch(B)
    for k in ("final_boards", "lengths", "scores"):
        assert torch.equal(out[k], again[k]), k
    assert out["summary"] == again["summary"]
    want = PO.monte_carlo_games(seed, B, K, rollout.policy_id, criterion, mode, max_steps=max_steps)
    np.testing.assert_array_equal(E.boards_numpy(out["final_boards"]), want["final_boards"])
    np.testing.assert_array_equal(out["lengths"].cpu().numpy(), want["lengths"])
    np.testing.assert_array_equal(out["scores"].cpu().numpy(), want["scores"])
    boards, lengths, scores = _own_loop(seed, B, K, rollout, criterion, mode, max_steps)
    assert torch.equal(out["final_boards"], boards)
    assert torch.equal(out["lengths"].to(torch.int64), lengths) and torch.equal(out["scores"].to(torch.int64), scores)
    s = out["summary"]
    assert s["episodes"] == B and s["env_steps"] == int(lengths.sum()) and s["score_sum"] == int(scores.sum())
    assert sum(s["max_tile_hist"].values()) == B and s["loop_steps"] == s["longest"] == int(lengths.max())
    # the chain moved on by the run's loop steps, as for every other run_eval_batch
    assert runner.chain.position == 1 + 2 * s["loop_steps"]


def test_monte_carlo_player_only_through_run_eval_batch():
    runner = g2048.BatchRunner(0, g2048.MonteCarloPolicy(playouts=2))
    for call in (runner.run_stats_batch, runner.run_flat_batch, runner.run_packed_batch, runner.run_actions_batch):
        with pytest.raises(ValueError, match="run_eval_batch"):
            call(8)


def test_monte_carlo_player_beats_drul():
    """Sanity, not parity: 16 random playouts per action play far better than DRUL on the same seeds."""
    B = 256
    mc = g2048.BatchRunner(3, g2048.MonteCarloPolicy(playouts=16)).run_eval_batch(B)
    drul = g2048.BatchRunner(3, g2048.act_drul).run_stats_batch(B)
    mc_mean = mc["summary"]["score_sum"] / B
    drul_mean = drul["summary"]["score_sum"] / B
    assert mc_mean > 3 * drul_mean, (mc_mean, drul_mean)
