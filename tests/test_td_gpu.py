"""TD(0) learning of the row table (g2048_td_train) and TDLearner on the GPU: table, env state and statistics bit for
bit against orc_td_train (tests/td_oracle.c), split runs and checkpoints, one step restated through the public API,
guard bands around the table and the scratch, and a learning sanity check."""
import numpy as np
import pytest
import torch

import g2048
from g2048 import engine as E
from oracle import c_oracle as CO
from oracle import pgx2048_oracle as O

import td_oracle as TO
from test_expectimax_oracle import random_table

pytestmark = pytest.mark.gpu

TABLES = ("zero", "default", "random")
ALPHAS = (0.0, 1.0 / 1024, 0.05)


def _table(name):
    if name == "zero":
        return np.zeros(65536, np.float32)
    if name == "default":
        return g2048.expectimax.default_row_table_numpy()
    return random_table(23) * np.float32(1e-4)  # mixed sign, up to ~2e2: the search still sees the game


def _words(x):
    return torch.from_numpy(np.ascontiguousarray(x, np.uint32).view(np.int32)).cuda()


def _run_both(n, n_steps, table, alpha, mode, seed=3):
    key = np.array([0, seed], np.uint32)
    _, subs = CO.chain(key, mode, 1 + n_steps)
    T = _table(table)
    want = TO.train(TO.fresh(subs[0], n, mode, T), alpha, subs[1:], mode)
    subs_t = _words(subs)
    boards, _ = E.env_init(subs_t[0], n, 0, n, mode)
    after = torch.zeros(n, dtype=torch.int64, device="cuda")
    scores = torch.zeros(n, dtype=torch.int32, device="cuda")
    lengths = torch.zeros(n, dtype=torch.int32, device="cuda")
    T_t = torch.from_numpy(T).cuda()
    scratch = E.td_scratch("cuda")
    stats = torch.zeros(32, dtype=torch.int64, device="cuda")
    E.td_train(boards, after, scores, lengths, T_t, alpha, subs_t[1:], mode, scratch, stats)
    got = dict(T=T_t.cpu().numpy(), boards=boards.cpu().numpy().view(np.uint64), after=after.cpu().numpy().view(np.uint64),
               scores=scores.cpu().numpy().view(np.uint32), lengths=lengths.cpu().numpy().view(np.uint32),
               stats=stats.cpu().numpy().view(np.uint64))
    return got, want, scratch


def _assert_same(got, want):
    np.testing.assert_array_equal(got["T"].view(np.uint32), want.T.view(np.uint32))
    np.testing.assert_array_equal(got["boards"], want.boards)
    np.testing.assert_array_equal(got["after"], want.after)
    np.testing.assert_array_equal(got["scores"], want.scores)
    np.testing.assert_array_equal(got["lengths"], want.lengths)
    np.testing.assert_array_equal(got["stats"], want.stats)


@pytest.mark.parametrize("mode", [E.RNG_PARTITIONABLE, E.RNG_ORIGINAL])
@pytest.mark.parametrize("n", [1, 33, 4096])
@pytest.mark.parametrize("n_steps", [1, 2, 17, 500])
def test_bit_exact_against_oracle(n, n_steps, mode):
    i = [1, 33, 4096].index(n) + [1, 2, 17, 500].index(n_steps)
    table, alpha = TABLES[i % 3], ALPHAS[(i + mode) % 3]  # all tables and step sizes over the grid (every pair below)
    got, want, scratch = _run_both(n, n_steps, table, alpha, mode)
    _assert_same(got, want)
    assert int(torch.count_nonzero(scratch)) == 0
    if n_steps == 500:
        assert want.stats[0] > 0  # episodes ended and restarted inside the run


@pytest.mark.parametrize("mode", [E.RNG_PARTITIONABLE, E.RNG_ORIGINAL])
@pytest.mark.parametrize("table", TABLES)
@pytest.mark.parametrize("alpha", ALPHAS)
def test_every_table_and_alpha_bit_exact(table, alpha, mode):
    got, want, _ = _run_both(33, 60, table, alpha, mode, seed=8)
    _assert_same(got, want)
    if alpha == 0.0:
        np.testing.assert_array_equal(got["T"].view(np.uint32), _table(table).view(np.uint32))


@pytest.mark.parametrize("mode", [E.RNG_PARTITIONABLE, E.RNG_ORIGINAL])
def test_several_env_passes_per_step_bit_exact(mode):
    """n = 2^17 is more than the co-resident grid holds threads (one 512-thread CTA per SM), so every thread walks
    several envs per step and the CTA's index-0 sum spans those passes."""
    got, want, scratch = _run_both(1 << 17, 6, "random", 0.05, mode, seed=12)
    _assert_same(got, want)
    assert int(torch.count_nonzero(scratch)) == 0


def _learner_state(lr):
    return [lr.table.clone(), lr.boards.clone(), lr.after.clone(), lr.scores.clone(), lr.lengths.clone()]


def _summary_sum(a, b):
    out = {k: a[k] + b[k] for k in E.STAT_NAMES}
    out["longest"] = max(a["longest"], b["longest"])
    out["max_tile_hist"] = {t: a["max_tile_hist"].get(t, 0) + b["max_tile_hist"].get(t, 0)
                            for t in set(a["max_tile_hist"]) | set(b["max_tile_hist"])}
    return out


@pytest.mark.parametrize("mode", [E.RNG_PARTITIONABLE, E.RNG_ORIGINAL])
def test_split_training_and_checkpoints_resume_bit_for_bit(mode):
    whole = g2048.TDLearner(5, 1000, alpha=0.01, rng_mode=mode)
    s_whole = whole.train(300)
    parts = g2048.TDLearner(5, 1000, alpha=0.01, rng_mode=mode)
    s1 = parts.train(120)
    ckpt = parts.state_dict()
    s2 = parts.train(180)
    for x, y in zip(_learner_state(whole), _learner_state(parts)):
        assert torch.equal(x, y)
    assert _summary_sum(s1, s2) == s_whole and s_whole["episodes"] > 0
    resumed = g2048.TDLearner(99, 1000, alpha=0.5, rng_mode=1 - mode)  # everything comes from the checkpoint
    resumed.load_state_dict(ckpt)
    assert resumed.train(180) == s2
    for x, y in zip(_learner_state(whole), _learner_state(resumed)):
        assert torch.equal(x, y)
    assert resumed.steps == whole.steps == 300 and np.array_equal(resumed.chain.key, whole.chain.key)


def test_load_state_dict_rejects_a_corrupt_checkpoint():
    lr = g2048.TDLearner(2, 64, alpha=0.01)
    lr.train(3)
    good = lr.state_dict()
    before = _learner_state(lr)
    for key, bad in (("table", torch.zeros(100)), ("table", torch.full((65536,), float("nan"))), ("rng_mode", 7),
                     ("alpha", -1.0), ("batch_size", 65)):
        state = dict(good)
        state[key] = bad
        with pytest.raises(ValueError):
            lr.load_state_dict(state)
    for x, y in zip(before, _learner_state(lr)):  # a rejected checkpoint changes nothing
        assert torch.equal(x, y)


@pytest.mark.parametrize("mode", [E.RNG_PARTITIONABLE, E.RNG_ORIGINAL])
def test_one_step_through_the_public_api(mode):
    n = 2048
    lr = g2048.TDLearner(11, n, alpha=0.02, table=_table("random"), rng_mode=mode)
    lr.train(40)
    T = lr.table.clone()
    boards = lr.boards.clone()
    sub = lr.chain.peek(1)[0].clone()
    legal = O.exact_legal(E.boards_numpy(boards))
    status = torch.from_numpy((legal * (1 << np.arange(4))).sum(axis=1).astype(np.uint8)).cuda()
    res = g2048.expectimax_values(boards, depth=1, row_values=T, reward_weight=1.0)
    actions = res.best_action()
    stepped = boards.clone()
    E.env_step(stepped, status, actions.to(torch.int32), sub, n, 0, mode)
    lr.train(1)
    moved = torch.from_numpy(legal.any(axis=1)).cuda()
    assert bool(moved.any()) and torch.equal(lr.boards[moved], stepped[moved])
    after, _ = O.move(E.boards_numpy(boards), actions.cpu().numpy())
    want_after = torch.from_numpy(E.pack_boards(after)).cuda()
    assert torch.equal(lr.after[moved], want_after[moved])
    assert bool((lr.after[~moved] == 0).all()) and bool((lr.lengths[~moved] == 0).all())


def test_table_and_scratch_are_surrounded_by_untouched_guard_bands():
    from test_guard_bands_gpu import GuardedTorch

    guard = GuardedTorch()
    mode = E.RNG_PARTITIONABLE
    subs = E.chain_advance(E.words_tensor([0, 4], "cuda"), mode, 41)
    for n in (1, 33, 4096):
        boards, _ = E.env_init(subs[0], n, 0, n, mode)
        b = guard.empty(n, dtype=torch.int64, device="cuda")
        b.copy_(boards)
        after = guard.zeros(n, dtype=torch.int64, device="cuda")
        scores = guard.zeros(n, dtype=torch.int32, device="cuda")
        lengths = guard.zeros(n, dtype=torch.int32, device="cuda")
        T = guard.empty(65536, dtype=torch.float32, device="cuda")
        T.copy_(torch.from_numpy(_table("random")).cuda())
        scratch = guard.zeros(int(g2048._native.lib.g2048_td_scratch_bytes()) // 8, dtype=torch.int64, device="cuda")
        stats = guard.zeros(32, dtype=torch.int64, device="cuda")
        E.td_train(b, after, scores, lengths, T, 0.05, subs[1:], mode, scratch, stats)
        assert int(torch.count_nonzero(scratch)) == 0
    assert len(guard.raw) == 21
    assert guard.check() == []


def test_learned_table_beats_drul_and_the_zero_table():
    """Sanity, not parity: a few seconds of training from zeros at n = 2^16, then the greedy player with the learned
    table against DRUL and against the greedy player with the zero table, over the same 1 024 seeded games."""
    lr = g2048.TDLearner(1, 1 << 16)
    lr.train(3000)
    B = 1024

    def greedy(T):
        out = g2048.BatchRunner(7, g2048.ExpectimaxPolicy(depth=1, row_values=T, reward_weight=1.0)).run_eval_batch(B)
        return out["summary"]["score_sum"] / B

    learned = greedy(lr.table)
    zero = greedy(torch.zeros(65536, dtype=torch.float32, device="cuda"))
    drul = g2048.BatchRunner(7, g2048.act_drul).run_stats_batch(B)["summary"]["score_sum"] / B
    assert learned > drul and learned > zero, (learned, zero, drul)
