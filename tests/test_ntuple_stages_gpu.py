"""Multi-stage n-tuple networks on the GPU (g2048_ntuple_staged_td_train, g2048_ntuple_staged_tc_train,
g2048_expectimax_values_ntuple_staged, NTupleNetwork.staged): W, E, A, boards, afterstates, scores, lengths and
statistics bit for bit against tests/ntuple_stages_oracle.c, one stage against the unstaged entry points, thresholds
never reached, expectimax against the oracle, checkpoints, guard bands, the player against the oracle's games, and a
learning sanity check."""
import numpy as np
import pytest
import torch

import g2048
from g2048 import _native as N
from g2048 import engine as E
from g2048.ntuple import NTupleNetwork, make_stages
from oracle import c_oracle as CO

import ntuple_oracle as NO
import ntuple_stages_oracle as SO
from test_ntuple_gpu import SMALL_WEIGHTS, _four_six_host, _game_boards, _words, random_weights, small_placements
from test_ntuple_tc_gpu import random_sums

pytestmark = pytest.mark.gpu

THRESHOLDS = ((3,), (3, 5), (4, 6, 8))  # low enough that envs cross them within a run


def _gpu_train(n, subs, mode, placements, stages, W, alpha, sums=None):
    """One launch of the staged learner (TD, or TC with sums = (E, A)) from fresh envs; stages None: the unstaged
    entry point."""
    subs_t = _words(subs)
    boards, _ = E.env_init(subs_t[0], n, 0, n, mode)
    after = torch.zeros(n, dtype=torch.int64, device="cuda")
    scores = torch.zeros(n, dtype=torch.int32, device="cuda")
    lengths = torch.zeros(n, dtype=torch.int32, device="cuda")
    W_t = torch.from_numpy(W).cuda()
    stats = torch.zeros(32, dtype=torch.int64, device="cuda")
    got = {}
    if sums is None:
        scratch = E.ntuple_td_scratch(n, placements, W.shape[0], "cuda")
        E.ntuple_td_train(boards, after, scores, lengths, placements, W_t, alpha, subs_t[1:], mode, scratch, stats,
                          stages=stages)
    else:
        E_t, A_t = torch.from_numpy(sums[0]).cuda(), torch.from_numpy(sums[1]).cuda()
        scratch = E.ntuple_tc_scratch(n, placements, W.shape[0], "cuda")
        E.ntuple_tc_train(boards, after, scores, lengths, placements, W_t, E_t, A_t, alpha, subs_t[1:], mode, scratch,
                          stats, stages=stages)
        got.update(E=E_t.cpu().numpy(), A=A_t.cpu().numpy())
    got.update(T=W_t.cpu().numpy(), boards=boards.cpu().numpy().view(np.uint64),
               after=after.cpu().numpy().view(np.uint64), scores=scores.cpu().numpy().view(np.uint32),
               lengths=lengths.cpu().numpy().view(np.uint32), stats=stats.cpu().numpy().view(np.uint64))
    assert int(torch.count_nonzero(scratch)) == 0
    return got


def _run_both(n, n_steps, placements, stages, W, alpha, mode, tc, seed=3):
    _, subs = CO.chain(np.array([0, seed], np.uint32), mode, 1 + n_steps)
    if tc:
        Es, As = random_sums(W.shape[0], seed) if W.shape[0] <= 1 << 26 else (np.zeros(W.shape[0]), np.zeros(W.shape[0]))
        got = _gpu_train(n, subs, mode, placements, stages, W, alpha, (Es, As))
        Es, As = Es.copy(), As.copy()
        want = SO.tc_train(NO.fresh(subs[0], n, mode, W), Es, As, placements, stages, alpha, subs[1:], mode)
        np.testing.assert_array_equal(got["E"].view(np.uint64), Es.view(np.uint64))
        np.testing.assert_array_equal(got["A"].view(np.uint64), As.view(np.uint64))
    else:
        got = _gpu_train(n, subs, mode, placements, stages, W, alpha)
        want = SO.train(NO.fresh(subs[0], n, mode, W), placements, stages, alpha, subs[1:], mode)
    np.testing.assert_array_equal(got["T"].view(np.uint32), want.T.view(np.uint32))
    for k in ("boards", "after", "scores", "lengths", "stats"):
        np.testing.assert_array_equal(got[k], getattr(want, k))
    return got, want


@pytest.mark.parametrize("mode", [E.RNG_PARTITIONABLE, E.RNG_ORIGINAL])
@pytest.mark.parametrize("tc", [False, True])
@pytest.mark.parametrize("n,n_steps", [(1, 500), (33, 200), (4096, 60)])
def test_staged_learning_bit_exact_against_oracle(n, n_steps, tc, mode):
    i = [1, 33, 4096].index(n)
    thresholds = THRESHOLDS[(i + mode) % 3]
    stages = make_stages(thresholds, SMALL_WEIGHTS)
    n_weights = (len(thresholds) + 1) * SMALL_WEIGHTS
    W = random_weights(n_weights, 23 + i) if (i + tc) % 2 else np.zeros(n_weights, np.float32)
    got, _ = _run_both(n, n_steps, small_placements(), stages, W, (0.05, 1.0 / 1024, 1.0)[i], mode, tc)
    assert not np.array_equal(got["T"][SMALL_WEIGHTS:], W[SMALL_WEIGHTS:])  # a later stage learned


@pytest.mark.parametrize("tc", [False, True])
def test_two_stage_four_six_bit_exact_against_oracle(tc):
    W = random_weights(1 << 27, 5) if tc else np.zeros(1 << 27, np.float32)
    got, _ = _run_both(33, 60, _four_six_host(), make_stages((4,), 1 << 26), W, 0.02, E.RNG_PARTITIONABLE, tc, seed=8)
    assert not np.array_equal(got["T"][1 << 26:], W[1 << 26:])


@pytest.mark.parametrize("tc", [False, True])
def test_staged_several_env_passes_per_step_bit_exact(tc):
    """n = 2^17: every thread walks several envs per step; stage 0's index-0 sums go through the CTA's shared sums."""
    W = random_weights(3 * SMALL_WEIGHTS, 12)
    _run_both(1 << 17, 6, small_placements(), make_stages((3, 5), SMALL_WEIGHTS), W, 0.05, E.RNG_ORIGINAL, tc, seed=12)


@pytest.mark.parametrize("tc", [False, True])
def test_one_stage_equals_the_unstaged_entry_points(tc):
    mode = E.RNG_PARTITIONABLE
    _, subs = CO.chain(np.array([0, 6], np.uint32), mode, 1 + 80)
    W = random_weights(SMALL_WEIGHTS, 4)
    sums = random_sums(SMALL_WEIGHTS, 4) if tc else None
    a = _gpu_train(2048, subs, mode, small_placements(), make_stages((), 0), W, 0.05,
                   None if sums is None else (sums[0].copy(), sums[1].copy()))
    b = _gpu_train(2048, subs, mode, small_placements(), None, W, 0.05, sums)
    for k in a:
        np.testing.assert_array_equal(a[k], b[k])
    boards = torch.from_numpy(E.pack_boards(_game_boards(64))).cuda()
    W_t = torch.from_numpy(W).cuda()
    for depth in (1, 2):
        q1 = E.expectimax_values_ntuple(boards, depth, small_placements(), W_t, 0.5, stages=make_stages((), 0))
        q2 = E.expectimax_values_ntuple(boards, depth, small_placements(), W_t, 0.5)
        assert torch.equal(q1.view(torch.int32), q2.view(torch.int32))


@pytest.mark.parametrize("tc", [False, True])
def test_thresholds_never_reached_leave_the_later_stages_alone(tc):
    """Threshold 15 (a 32768 tile) is never reached in these games: stage 0 learns what the unstaged network learns,
    bit for bit, and stage 1 keeps its values."""
    mode = E.RNG_ORIGINAL
    _, subs = CO.chain(np.array([0, 2], np.uint32), mode, 1 + 100)
    W0, W1 = random_weights(SMALL_WEIGHTS, 8), random_weights(SMALL_WEIGHTS, 9)
    sums = random_sums(SMALL_WEIGHTS, 8) if tc else None
    staged_sums = None if sums is None else (np.concatenate([sums[0], np.zeros(SMALL_WEIGHTS)]),
                                             np.concatenate([sums[1], np.zeros(SMALL_WEIGHTS)]))
    a = _gpu_train(4096, subs, mode, small_placements(), make_stages((15,), SMALL_WEIGHTS), np.concatenate([W0, W1]),
                   0.05, staged_sums)
    b = _gpu_train(4096, subs, mode, small_placements(), None, W0, 0.05, sums)
    np.testing.assert_array_equal(a["T"][:SMALL_WEIGHTS].view(np.uint32), b["T"].view(np.uint32))
    np.testing.assert_array_equal(a["T"][SMALL_WEIGHTS:].view(np.uint32), W1.view(np.uint32))
    for k in ("boards", "after", "scores", "lengths", "stats"):
        np.testing.assert_array_equal(a[k], b[k])
    if tc:
        np.testing.assert_array_equal(a["E"][:SMALL_WEIGHTS], b["E"])
        assert not a["E"][SMALL_WEIGHTS:].any() and not a["A"][SMALL_WEIGHTS:].any()


# --------------------------------------------------------------------------------------------------- expectimax
@pytest.fixture(scope="module")
def staged_boards():
    """Boards of real games: their largest exponents span the stages of (4, 6, 8)."""
    boards = _game_boards(256, seed=9)
    stages = np.array([sum(int(b.max()) >= t for t in (4, 6, 8)) for b in boards])
    assert len(set(stages)) >= 3
    return boards


@pytest.mark.parametrize("depth", [1, 2, 3])
@pytest.mark.parametrize("w", [0.0, 1.0])
def test_staged_expectimax_bit_exact_against_oracle(staged_boards, depth, w):
    boards = staged_boards if depth < 3 else staged_boards[::8]
    pl, st = small_placements(), make_stages((4, 6, 8), SMALL_WEIGHTS)
    W = random_weights(4 * SMALL_WEIGHTS, 17)
    counters = torch.zeros(2, dtype=torch.int64, device="cuda")
    q = E.expectimax_values_ntuple(torch.from_numpy(E.pack_boards(boards)).cuda(), depth, pl, torch.from_numpy(W).cuda(),
                                   w, counters, stages=st).cpu().numpy()
    want_q, want_c = SO.expectimax(boards, depth, pl, st, W, w)
    np.testing.assert_array_equal(q.view(np.uint32), want_q.view(np.uint32))
    np.testing.assert_array_equal(counters.cpu().numpy().astype(np.uint64), want_c)


@pytest.mark.parametrize("depth", [1, 2, 3])
def test_staged_network_searches_like_its_base(staged_boards, depth):
    base = NTupleNetwork(small_placements(), SMALL_WEIGHTS, random_weights(SMALL_WEIGHTS, 3))
    net = NTupleNetwork.staged(base, (4, 6, 8))
    boards = staged_boards if depth < 3 else staged_boards[::8]
    a = g2048.expectimax_values(boards, depth=depth, network=net, reward_weight=1.0)
    b = g2048.expectimax_values(boards, depth=depth, network=base, reward_weight=1.0)
    assert torch.equal(a.q.view(torch.int32), b.q.view(torch.int32)) and torch.equal(a.counters, b.counters)


# ------------------------------------------------------------------------------------------ learners, checkpoints
def _staged_net(thresholds=(3, 5), weights=None):
    base = NTupleNetwork(small_placements(), SMALL_WEIGHTS, weights)
    return NTupleNetwork.staged(base, thresholds)


def _state(lr):
    out = [lr.weights.clone(), lr.boards.clone(), lr.after.clone(), lr.scores.clone(), lr.lengths.clone()]
    if isinstance(lr, g2048.NTupleTCLearner):
        out += [lr.err_sum.clone(), lr.abs_err_sum.clone()]
    return out


@pytest.mark.parametrize("cls", [g2048.NTupleTDLearner, g2048.NTupleTCLearner])
def test_split_training_and_checkpoints_resume_bit_for_bit(cls):
    whole = cls(5, 1000, network=_staged_net(), alpha=0.5)
    s_whole = whole.train(300)
    parts = cls(5, 1000, network=_staged_net(), alpha=0.5)
    s1 = parts.train(120)
    ckpt = parts.state_dict()
    assert ckpt["stage_thresholds"] == [3, 5] and ckpt["stage_stride"] == SMALL_WEIGHTS
    s2 = parts.train(180)
    for x, y in zip(_state(whole), _state(parts)):
        assert torch.equal(x, y)
    assert s1["episodes"] + s2["episodes"] == s_whole["episodes"] > 0
    resumed = cls(99, 1000, network=_staged_net(), alpha=0.01)
    resumed.load_state_dict(ckpt)
    assert resumed.train(180) == s2
    for x, y in zip(_state(whole), _state(resumed)):
        assert torch.equal(x, y)


def test_a_checkpoint_with_other_stages_is_rejected():
    lr = g2048.NTupleTDLearner(2, 64, network=_staged_net(), alpha=0.1)
    lr.train(3)
    good = lr.state_dict()
    before = _state(lr)
    for key, bad in (("stage_thresholds", [3, 6]), ("stage_thresholds", [3]), ("stage_stride", SMALL_WEIGHTS - 1),
                     ("stage_thresholds", None)):
        state = dict(good)
        if bad is None:
            del state[key]
        else:
            state[key] = bad
        with pytest.raises(ValueError, match="stages"):
            lr.load_state_dict(state)
    for x, y in zip(before, _state(lr)):  # a rejected checkpoint changes nothing
        assert torch.equal(x, y)
    # a single-stage learner takes a checkpoint without stage entries (as written before stages existed), and rejects
    # a staged one of the same n_weights
    single = g2048.NTupleTDLearner(2, 64, network=NTupleNetwork(small_placements(), 3 * SMALL_WEIGHTS), alpha=0.1)
    old = {k: v for k, v in single.state_dict().items() if not k.startswith("stage_")}
    single.load_state_dict(old)
    with pytest.raises(ValueError, match="stages"):
        single.load_state_dict(good)


def test_learners_take_the_staged_path_only_for_several_stages(monkeypatch):
    calls = []
    for name in ("ntuple_td_train", "ntuple_tc_train"):
        orig = getattr(E, name)

        def spy(*args, _orig=orig, **kw):
            calls.append(kw.get("stages"))
            return _orig(*args, **kw)

        monkeypatch.setattr(E, name, spy)
    g2048.NTupleTDLearner(0, 32, network=NTupleNetwork(small_placements(), SMALL_WEIGHTS)).train(2)
    g2048.NTupleTCLearner(0, 32, network=_staged_net()).train(2)
    assert calls[0] is None and calls[1].dtype == g2048.ntuple.STAGES_DTYPE


def test_weights_sums_scratch_and_outputs_are_surrounded_by_untouched_guard_bands():
    from test_guard_bands_gpu import GuardedTorch

    guard = GuardedTorch()
    mode = E.RNG_PARTITIONABLE
    pl, st, nw = small_placements(), make_stages((3, 5), SMALL_WEIGHTS), 3 * SMALL_WEIGHTS
    subs = E.chain_advance(E.words_tensor([0, 4], "cuda"), mode, 41)
    for n in (1, 33, 4096):
        for tc in (False, True):
            boards, _ = E.env_init(subs[0], n, 0, n, mode)
            b = guard.empty(n, dtype=torch.int64, device="cuda")
            b.copy_(boards)
            after = guard.zeros(n, dtype=torch.int64, device="cuda")
            scores = guard.zeros(n, dtype=torch.int32, device="cuda")
            lengths = guard.zeros(n, dtype=torch.int32, device="cuda")
            W = guard.empty(nw, dtype=torch.float32, device="cuda")
            W.copy_(torch.from_numpy(random_weights(nw, 2)).cuda())
            stats = guard.zeros(32, dtype=torch.int64, device="cuda")
            if tc:
                Es = guard.zeros(nw, dtype=torch.float64, device="cuda")
                As = guard.zeros(nw, dtype=torch.float64, device="cuda")
                size = int(N.lib.g2048_ntuple_tc_scratch_bytes(n, pl.shape[0], nw))
                scratch = guard.zeros(size // 8, dtype=torch.int64, device="cuda")
                E.ntuple_tc_train(b, after, scores, lengths, pl, W, Es, As, 0.05, subs[1:], mode, scratch, stats,
                                  stages=st)
            else:
                size = int(N.lib.g2048_ntuple_td_scratch_bytes(n, pl.shape[0], nw))
                scratch = guard.zeros(size // 8, dtype=torch.int64, device="cuda")
                E.ntuple_td_train(b, after, scores, lengths, pl, W, 0.05, subs[1:], mode, scratch, stats, stages=st)
            assert int(torch.count_nonzero(scratch)) == 0
    assert guard.check() == []


# ----------------------------------------------------------------------------------------------------- the player
@pytest.mark.parametrize("mode", [E.RNG_PARTITIONABLE, E.RNG_ORIGINAL])
def test_staged_player_matches_oracle_games(mode):
    B, seed, depth, w = 16, 12, 1, 1.0
    W = random_weights(3 * SMALL_WEIGHTS, 41)
    net = NTupleNetwork(small_placements(), 3 * SMALL_WEIGHTS, W, stage_thresholds=(3, 5), stage_stride=SMALL_WEIGHTS)
    runner = g2048.BatchRunner(seed, g2048.ExpectimaxPolicy(depth=depth, network=net, reward_weight=w), rng_mode=mode)
    out = runner.run_eval_batch(B)
    want = SO.expectimax_games(seed, B, depth, net.placements, net.stages, W, w, mode)
    np.testing.assert_array_equal(E.boards_numpy(out["final_boards"]), want["final_boards"])
    np.testing.assert_array_equal(out["lengths"].cpu().numpy(), want["lengths"])
    np.testing.assert_array_equal(out["scores"].cpu().numpy(), want["scores"])
    assert int(want["final_boards"].max()) >= 5  # the games reached the last stage


def test_learned_staged_four_six_network_beats_drul():
    """Sanity, not parity: a short TD run of a 2-stage 4x6 network from zeros at n = 2^16, then its greedy player
    against DRUL over the same 1 024 seeded games."""
    lr = g2048.NTupleTDLearner(1, 1 << 16, network=NTupleNetwork.staged(NTupleNetwork.four_six(), (8,)))
    lr.train(1000)
    B = 1024
    out = g2048.BatchRunner(7, g2048.ExpectimaxPolicy(depth=1, network=lr.network, reward_weight=1.0)).run_eval_batch(B)
    learned = out["summary"]["score_sum"] / B
    drul = g2048.BatchRunner(7, g2048.act_drul).run_stats_batch(B)["summary"]["score_sum"] / B
    assert learned > drul, (learned, drul)
