"""N-tuple networks on the GPU: TD(0) learning (g2048_ntuple_td_train) and expectimax over a network
(g2048_expectimax_values_ntuple) bit for bit against tests/ntuple_oracle.c, the `lines` network against the row-table
kernels (g2048_td_train, g2048_expectimax_values), a network at high offsets of a larger weight array, split runs and
checkpoints, guard bands, one step restated through the public API, the player against the oracle's games and a
public-API loop, and a learning sanity check."""
import numpy as np
import pytest
import torch

import g2048
from g2048 import _native as N
from g2048 import engine as E
from g2048.ntuple import NTupleNetwork, make_placements
from oracle import c_oracle as CO
from oracle import pgx2048_oracle as O

import ntuple_oracle as NO

pytestmark = pytest.mark.gpu

ALPHAS = (0.0, 1.0 / 1024, 0.05)

# a small mixed network: k = 1..6, a shared table (two placements at offset 16), tables packed in order
SMALL_TUPLES = [(0, [(5,)]), (16, [(0, 1), (3, 2)]), (272, [(4, 8, 12)]), (4368, [(0, 5, 10, 15)]),
                (69904, [(1, 2, 6, 7, 11)]), (1118480, [(9, 10, 13, 14, 15, 12)])]
SMALL_WEIGHTS = 1118480 + (1 << 24)


MID_WEIGHTS = 1118480  # SMALL_TUPLES without the 6-cell table


def small_placements(shift=0, tuples=SMALL_TUPLES):
    return make_placements([(off + shift, cells) for off, group in tuples for cells in group])


def random_weights(n, seed, scale=1e-4):
    """float32 values of mixed sign over many binades (scaled so that a search still sees the game)."""
    rng = np.random.default_rng(seed)
    mag = np.exp2(rng.uniform(-20.0, 20.0, n).astype(np.float32))
    return (mag * rng.choice(np.array([-1.0, 1.0], np.float32), n) * np.float32(scale)).astype(np.float32)


def _four_six_host():
    return g2048.ntuple.make_placements(
        [(j << 24, im) for j, t in enumerate(g2048.ntuple.FOUR_SIX_TUPLES) for im in g2048.ntuple.symmetric_images(t)])


def _words(x):
    return torch.from_numpy(np.ascontiguousarray(x, np.uint32).view(np.int32)).cuda()


def _gpu_train(n, subs, mode, placements, W, alpha):
    subs_t = _words(subs)
    boards, _ = E.env_init(subs_t[0], n, 0, n, mode)
    after = torch.zeros(n, dtype=torch.int64, device="cuda")
    scores = torch.zeros(n, dtype=torch.int32, device="cuda")
    lengths = torch.zeros(n, dtype=torch.int32, device="cuda")
    W_t = torch.from_numpy(W).cuda()
    scratch = E.ntuple_td_scratch(n, placements, W.shape[0], "cuda")
    stats = torch.zeros(32, dtype=torch.int64, device="cuda")
    E.ntuple_td_train(boards, after, scores, lengths, placements, W_t, alpha, subs_t[1:], mode, scratch, stats)
    got = dict(T=W_t.cpu().numpy(), boards=boards.cpu().numpy().view(np.uint64), after=after.cpu().numpy().view(np.uint64),
               scores=scores.cpu().numpy().view(np.uint32), lengths=lengths.cpu().numpy().view(np.uint32),
               stats=stats.cpu().numpy().view(np.uint64))
    return got, scratch


def _run_both(n, n_steps, placements, W, alpha, mode, seed=3):
    key = np.array([0, seed], np.uint32)
    _, subs = CO.chain(key, mode, 1 + n_steps)
    want = NO.train(NO.fresh(subs[0], n, mode, W), placements, alpha, subs[1:], mode)
    got, scratch = _gpu_train(n, subs, mode, placements, W, alpha)
    return got, want, scratch


def _assert_same(got, want):
    np.testing.assert_array_equal(got["T"].view(np.uint32), want.T.view(np.uint32))
    np.testing.assert_array_equal(got["boards"], want.boards)
    np.testing.assert_array_equal(got["after"], want.after)
    np.testing.assert_array_equal(got["scores"], want.scores)
    np.testing.assert_array_equal(got["lengths"], want.lengths)
    np.testing.assert_array_equal(got["stats"], want.stats)


# ------------------------------------------------------------------------------------------------ TD learning
@pytest.mark.parametrize("mode", [E.RNG_PARTITIONABLE, E.RNG_ORIGINAL])
@pytest.mark.parametrize("n", [1, 33, 4096])
@pytest.mark.parametrize("n_steps", [1, 2, 17, 500])
def test_td_bit_exact_against_oracle(n, n_steps, mode):
    i = [1, 33, 4096].index(n) + [1, 2, 17, 500].index(n_steps)
    alpha = ALPHAS[(i + mode) % 3]
    W = np.zeros(SMALL_WEIGHTS, np.float32) if i % 2 else random_weights(SMALL_WEIGHTS, 23)
    got, want, scratch = _run_both(n, n_steps, small_placements(), W, alpha, mode)
    _assert_same(got, want)
    assert int(torch.count_nonzero(scratch)) == 0
    if n_steps == 500:
        assert want.stats[0] > 0  # episodes ended and restarted inside the run


@pytest.mark.parametrize("mode", [E.RNG_PARTITIONABLE, E.RNG_ORIGINAL])
@pytest.mark.parametrize("alpha", ALPHAS)
def test_td_four_six_bit_exact_against_oracle(alpha, mode):
    W = random_weights(1 << 26, 5) if alpha != ALPHAS[1] else np.zeros(1 << 26, np.float32)
    got, want, scratch = _run_both(33, 40, _four_six_host(), W, alpha, mode, seed=8)
    _assert_same(got, want)
    assert int(torch.count_nonzero(scratch)) == 0


@pytest.mark.parametrize("mode", [E.RNG_PARTITIONABLE, E.RNG_ORIGINAL])
def test_td_several_env_passes_per_step_bit_exact(mode):
    """n = 2^17 is more than the co-resident grid holds threads, so every thread walks several envs per step and the
    CTA's index-0 sums span those passes."""
    got, want, scratch = _run_both(1 << 17, 6, small_placements(), random_weights(SMALL_WEIGHTS, 12), 0.05, mode,
                                   seed=12)
    _assert_same(got, want)
    assert int(torch.count_nonzero(scratch)) == 0


@pytest.mark.parametrize("mode", [E.RNG_PARTITIONABLE, E.RNG_ORIGINAL])
def test_lines_network_equals_the_row_table_learner(mode):
    """The `lines` network through g2048_ntuple_td_train is g2048_td_train, bit for bit."""
    n, steps = 1 << 16, 300
    subs = E.chain_advance(E.words_tensor([0, 21], "cuda"), mode, 1 + steps)
    T0 = torch.from_numpy(g2048.expectimax.default_row_table_numpy() * np.float32(1e-3)).cuda()
    out = []
    for kind in ("row", "lines"):
        boards, _ = E.env_init(subs[0], n, 0, n, mode)
        after = torch.zeros(n, dtype=torch.int64, device="cuda")
        scores = torch.zeros(n, dtype=torch.int32, device="cuda")
        lengths = torch.zeros(n, dtype=torch.int32, device="cuda")
        stats = torch.zeros(32, dtype=torch.int64, device="cuda")
        T = T0.clone()
        if kind == "row":
            E.td_train(boards, after, scores, lengths, T, 0.05, subs[1:], mode, E.td_scratch("cuda"), stats)
        else:
            net = NTupleNetwork.lines()
            E.ntuple_td_train(boards, after, scores, lengths, net.placements, T, 0.05, subs[1:], mode,
                              E.ntuple_td_scratch(n, net.placements, 65536, "cuda"), stats)
        out.append([T, boards, after, scores, lengths, stats])
    assert int(out[0][5][0]) > 0
    for x, y in zip(*out):
        assert torch.equal(x.view(torch.int32) if x.dtype == torch.float32 else x,
                           y.view(torch.int32) if y.dtype == torch.float32 else y)


def test_tables_at_high_offsets_of_a_larger_array_learn_the_same():
    """The same network trained packed, and with its tables at high offsets of a weight array 16 times as large: the
    touched entries are identical and every other weight is untouched."""
    mode = E.RNG_PARTITIONABLE
    _, subs = CO.chain(np.array([0, 31], np.uint32), mode, 1 + 50)
    mid = SMALL_TUPLES[:-1]
    W = random_weights(MID_WEIGHTS, 3)
    packed, _ = _gpu_train(4096, subs, mode, small_placements(0, mid), W, 0.05)
    shift = 15 * MID_WEIGHTS
    big = np.full(16 * MID_WEIGHTS, np.float32(7.25))
    big[shift:] = W
    high, scratch = _gpu_train(4096, subs, mode, small_placements(shift, mid), big, 0.05)
    np.testing.assert_array_equal(high["T"][shift:].view(np.uint32), packed["T"].view(np.uint32))
    assert bool((high["T"][:shift] == np.float32(7.25)).all())
    for k in ("boards", "after", "scores", "lengths", "stats"):
        np.testing.assert_array_equal(high[k], packed[k])
    assert int(torch.count_nonzero(scratch)) == 0


def _learner_state(lr):
    return [lr.weights.clone(), lr.boards.clone(), lr.after.clone(), lr.scores.clone(), lr.lengths.clone()]


def _small_net(weights=None):
    return NTupleNetwork(small_placements(), SMALL_WEIGHTS, weights)


@pytest.mark.parametrize("mode", [E.RNG_PARTITIONABLE, E.RNG_ORIGINAL])
def test_split_training_and_checkpoints_resume_bit_for_bit(mode):
    whole = g2048.NTupleTDLearner(5, 1000, network=_small_net(), alpha=0.01, rng_mode=mode)
    s_whole = whole.train(300)
    parts = g2048.NTupleTDLearner(5, 1000, network=_small_net(), alpha=0.01, rng_mode=mode)
    s1 = parts.train(120)
    ckpt = parts.state_dict()
    s2 = parts.train(180)
    for x, y in zip(_learner_state(whole), _learner_state(parts)):
        assert torch.equal(x, y)
    assert s1["episodes"] + s2["episodes"] == s_whole["episodes"] > 0
    assert s1["score_sum"] + s2["score_sum"] == s_whole["score_sum"]
    resumed = g2048.NTupleTDLearner(99, 1000, network=_small_net(), alpha=0.5, rng_mode=1 - mode)
    resumed.load_state_dict(ckpt)
    assert resumed.train(180) == s2
    for x, y in zip(_learner_state(whole), _learner_state(resumed)):
        assert torch.equal(x, y)
    assert resumed.steps == whole.steps == 300 and np.array_equal(resumed.chain.key, whole.chain.key)


def test_learner_accepts_a_device_given_without_an_index():
    lr = g2048.NTupleTDLearner(4, 64, network=_small_net(), alpha=0.01, device="cuda")
    lr.train(2)
    default = g2048.NTupleTDLearner(4, 64, alpha=0.01, device=torch.device("cuda"))
    assert default.network.n_placements == 32
    with pytest.raises(ValueError):
        g2048.NTupleTDLearner(4, 64, network=NTupleNetwork.lines(device="cpu"), device="cuda")


def test_load_state_dict_rejects_a_checkpoint_for_another_network():
    lr = g2048.NTupleTDLearner(2, 64, network=_small_net(), alpha=0.01)
    lr.train(3)
    good = lr.state_dict()
    before = _learner_state(lr)
    other = small_placements()
    other[3]["cells"][0] = 7
    for key, bad in (("placements", other), ("placements", small_placements()[:-1]), ("n_weights", SMALL_WEIGHTS + 1),
                     ("weights", torch.zeros(100)), ("weights", torch.full((SMALL_WEIGHTS,), float("nan"))),
                     ("rng_mode", 7), ("alpha", -1.0), ("batch_size", 65)):
        state = dict(good)
        state[key] = bad
        with pytest.raises(ValueError):
            lr.load_state_dict(state)
    for x, y in zip(before, _learner_state(lr)):  # a rejected checkpoint changes nothing
        assert torch.equal(x, y)


@pytest.mark.parametrize("mode", [E.RNG_PARTITIONABLE, E.RNG_ORIGINAL])
def test_one_step_through_the_public_api(mode):
    n = 2048
    net = _small_net(random_weights(SMALL_WEIGHTS, 9))
    lr = g2048.NTupleTDLearner(11, n, network=net, alpha=0.02, rng_mode=mode)
    lr.train(40)
    boards = lr.boards.clone()
    sub = lr.chain.peek(1)[0].clone()
    legal = O.exact_legal(E.boards_numpy(boards))
    status = torch.from_numpy((legal * (1 << np.arange(4))).sum(axis=1).astype(np.uint8)).cuda()
    res = g2048.expectimax_values(boards, depth=1, network=net, reward_weight=1.0)
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


def test_weights_scratch_and_outputs_are_surrounded_by_untouched_guard_bands(monkeypatch):
    from test_guard_bands_gpu import GuardedTorch

    guard = GuardedTorch()
    mode = E.RNG_PARTITIONABLE
    pl = small_placements()
    subs = E.chain_advance(E.words_tensor([0, 4], "cuda"), mode, 41)
    for n in (1, 33, 4096):
        boards, _ = E.env_init(subs[0], n, 0, n, mode)
        b = guard.empty(n, dtype=torch.int64, device="cuda")
        b.copy_(boards)
        after = guard.zeros(n, dtype=torch.int64, device="cuda")
        scores = guard.zeros(n, dtype=torch.int32, device="cuda")
        lengths = guard.zeros(n, dtype=torch.int32, device="cuda")
        W = guard.empty(SMALL_WEIGHTS, dtype=torch.float32, device="cuda")
        W.copy_(torch.from_numpy(random_weights(SMALL_WEIGHTS, 2)).cuda())
        size = int(N.lib.g2048_ntuple_td_scratch_bytes(n, pl.shape[0], SMALL_WEIGHTS))
        scratch = guard.zeros(size // 8, dtype=torch.int64, device="cuda")
        stats = guard.zeros(32, dtype=torch.int64, device="cuda")
        E.ntuple_td_train(b, after, scores, lengths, pl, W, 0.05, subs[1:], mode, scratch, stats)
        assert int(torch.count_nonzero(scratch)) == 0
    monkeypatch.setattr(E, "torch", guard)
    Wx = torch.from_numpy(random_weights(SMALL_WEIGHTS, 2)).cuda()
    for n in (1, 33, 72):
        for depth in (1, 2):
            counters = guard.zeros(2, dtype=torch.int64, device="cuda")
            E.expectimax_values_ntuple(boards[:n], depth, pl, Wx, 0.5, counters)
    assert len(guard.raw) >= 21 + 12
    assert guard.check() == []


# --------------------------------------------------------------------------------------------------- expectimax
def _game_boards(n, mode=E.RNG_PARTITIONABLE, seed=5):
    """Boards of real games at several depths (DRUL trajectories of g2048_play_record)."""
    subs = E.chain_advance(E.words_tensor([0, seed], "cuda"), mode, 1 + 2 * 2048)
    rec = E.play_record(E.POLICY_DRUL, subs, n, 0, n, mode)
    slot = rec["env_slot"].cpu().numpy()
    length = rec["lengths"].cpu().numpy().astype(np.int64)
    depth = (np.arange(n) * 37) % np.maximum(length, 1)
    return E.boards_numpy(rec["arena_boards"][torch.from_numpy(slot + depth).cuda()])


@pytest.fixture(scope="module")
def four_six_weights():
    return random_weights(1 << 26, 17)


@pytest.fixture(scope="module")
def game_boards():
    return _game_boards(256)


def _gpu_xm(boards_u8, depth, placements, W_t, w):
    boards = torch.from_numpy(E.pack_boards(boards_u8)).cuda()
    counters = torch.zeros(2, dtype=torch.int64, device="cuda")
    q = E.expectimax_values_ntuple(boards, depth, placements, W_t, w, counters)
    return q.cpu().numpy(), counters.cpu().numpy().astype(np.uint64)


@pytest.mark.parametrize("depth", [1, 2, 3])
@pytest.mark.parametrize("w", [0.0, 0.5, 1.0])
def test_expectimax_four_six_bit_exact_against_oracle(game_boards, four_six_weights, depth, w):
    boards = game_boards if depth < 3 else game_boards[::8]
    pl = _four_six_host()
    q, c = _gpu_xm(boards, depth, pl, torch.from_numpy(four_six_weights).cuda(), w)
    want_q, want_c = NO.expectimax(boards, depth, pl, four_six_weights, w)
    np.testing.assert_array_equal(q.view(np.uint32), want_q.view(np.uint32))
    np.testing.assert_array_equal(c, want_c)


def test_expectimax_four_six_depth_four_bit_exact_against_oracle(game_boards, four_six_weights):
    full = game_boards[np.argsort((game_boards == 0).sum(axis=1))[:3]]  # the fullest boards: the smallest trees
    pl = _four_six_host()
    q, c = _gpu_xm(full, 4, pl, torch.from_numpy(four_six_weights).cuda(), 0.5)
    want_q, want_c = NO.expectimax(full, 4, pl, four_six_weights, 0.5)
    np.testing.assert_array_equal(q.view(np.uint32), want_q.view(np.uint32))
    np.testing.assert_array_equal(c, want_c)


@pytest.mark.parametrize("depth", [1, 2, 3, 4])
def test_lines_expectimax_equals_the_row_table_kernel(game_boards, depth):
    boards = game_boards[:64] if depth < 4 else game_boards[np.argsort((game_boards == 0).sum(axis=1))[:4]]
    T = torch.from_numpy(random_weights(65536, 29)).cuda()
    b = torch.from_numpy(E.pack_boards(boards)).cuda()
    for w in (0.0, 1.0):
        c_row = torch.zeros(2, dtype=torch.int64, device="cuda")
        c_net = torch.zeros(2, dtype=torch.int64, device="cuda")
        q_row = E.expectimax_values(b, depth, T, w, c_row)
        q_net = E.expectimax_values_ntuple(b, depth, NTupleNetwork.lines(device="cuda").placements, T, w, c_net)
        assert torch.equal(q_row.view(torch.int32), q_net.view(torch.int32))
        assert torch.equal(c_row, c_net)


def test_expectimax_api_rejects_a_row_table_and_a_network_together():
    net = _small_net()
    with pytest.raises(ValueError):
        g2048.expectimax_values(np.zeros(1, np.uint64), 1, row_values=torch.zeros(65536, device="cuda"), network=net)
    with pytest.raises(ValueError):
        g2048.ExpectimaxPolicy(depth=1, row_values=torch.zeros(65536, device="cuda"), network=net)


# ----------------------------------------------------------------------------------------------------- the player
def _own_loop(seed, B, depth, net, w, mode):
    chain = g2048.keys.KeyChain(seed, mode, "cuda")
    subs = chain.peek(1 + 2 * 4096)
    boards, status = E.env_init(subs[0], B, 0, B, mode)
    lengths = torch.zeros(B, dtype=torch.int64, device="cuda")
    scores = torch.zeros(B, dtype=torch.int64, device="cuda")
    t = 0
    while bool(((status & N.STATUS_DONE) == 0).any()):
        res = g2048.expectimax_values(boards, depth=depth, network=net, reward_weight=w)
        alive = (status & N.STATUS_DONE) == 0
        rewards = E.env_step(boards, status, res.best_action().to(torch.int32), subs[2 + 2 * t], B, 0, mode)
        lengths += alive.to(torch.int64)
        scores += rewards.to(torch.int64)
        t += 1
    return boards, lengths, scores


@pytest.mark.parametrize("mode", [E.RNG_PARTITIONABLE, E.RNG_ORIGINAL])
def test_player_matches_oracle_games_and_own_loop(mode):
    B, seed, depth, w = 16, 12, 1, 1.0
    W = random_weights(SMALL_WEIGHTS, 41)
    net = _small_net(W)
    runner = g2048.BatchRunner(seed, g2048.ExpectimaxPolicy(depth=depth, network=net, reward_weight=w), rng_mode=mode)
    out = runner.run_eval_batch(B)
    want = NO.expectimax_games(seed, B, depth, net.placements, W, w, mode)
    np.testing.assert_array_equal(E.boards_numpy(out["final_boards"]), want["final_boards"])
    np.testing.assert_array_equal(out["lengths"].cpu().numpy(), want["lengths"])
    np.testing.assert_array_equal(out["scores"].cpu().numpy(), want["scores"])
    boards, lengths, scores = _own_loop(seed, B, depth, net, w, mode)
    assert torch.equal(out["final_boards"], boards)
    assert torch.equal(out["lengths"].to(torch.int64), lengths) and torch.equal(out["scores"].to(torch.int64), scores)
    assert runner.chain.position == 1 + 2 * out["summary"]["loop_steps"]


def test_network_player_only_through_run_eval_batch():
    runner = g2048.BatchRunner(0, g2048.ExpectimaxPolicy(depth=1, network=_small_net()))
    for call in (runner.run_stats_batch, runner.run_flat_batch, runner.run_packed_batch, runner.run_actions_batch):
        with pytest.raises(ValueError, match="run_eval_batch"):
            call(8)


def test_learned_four_six_network_beats_drul_and_the_zero_network():
    """Sanity, not parity: a short run of the 4x6 network from zeros at n = 2^16, then its greedy player against DRUL
    and against the greedy player of the zero network, over the same 1 024 seeded games."""
    lr = g2048.NTupleTDLearner(1, 1 << 16)
    lr.train(1000)
    B = 1024

    def greedy(net):
        out = g2048.BatchRunner(7, g2048.ExpectimaxPolicy(depth=1, network=net, reward_weight=1.0)).run_eval_batch(B)
        return out["summary"]["score_sum"] / B

    learned = greedy(lr.network)
    zero = greedy(NTupleNetwork.four_six())
    drul = g2048.BatchRunner(7, g2048.act_drul).run_stats_batch(B)["summary"]["score_sum"] / B
    assert learned > drul and learned > zero, (learned, zero, drul)
