"""N-tuple temporal coherence learning on the GPU (g2048_ntuple_tc_train, NTupleTCLearner): W, E, A, boards,
afterstates, scores, lengths and statistics bit for bit against tests/ntuple_tc_oracle.c, one step from zero sums against
g2048_ntuple_td_train through the public API, alpha = 0, split runs and checkpoints, guard bands, and a learning
sanity check."""
import numpy as np
import pytest
import torch

import g2048
from g2048 import _native as N
from g2048 import engine as E
from g2048.ntuple import NTupleNetwork
from oracle import c_oracle as CO

import ntuple_oracle as NO
import ntuple_tc_oracle as TCO
from test_ntuple_gpu import SMALL_WEIGHTS, _four_six_host, _words, random_weights, small_placements

pytestmark = pytest.mark.gpu


def random_sums(n, seed):
    """E and A with |E| <= A, zero for about a third of the entries, so beta takes every branch from the first step."""
    rng = np.random.default_rng(seed)
    A = np.where(rng.random(n) < 0.3, 0.0, np.exp2(rng.uniform(-10.0, 20.0, n)))
    return A * rng.uniform(-1.0, 1.0, n), A


def _gpu_tc_train(n, subs, mode, placements, W, Es, As, alpha):
    subs_t = _words(subs)
    boards, _ = E.env_init(subs_t[0], n, 0, n, mode)
    after = torch.zeros(n, dtype=torch.int64, device="cuda")
    scores = torch.zeros(n, dtype=torch.int32, device="cuda")
    lengths = torch.zeros(n, dtype=torch.int32, device="cuda")
    W_t = torch.from_numpy(W).cuda()
    E_t, A_t = torch.from_numpy(Es).cuda(), torch.from_numpy(As).cuda()
    scratch = E.ntuple_tc_scratch(n, placements, W.shape[0], "cuda")
    stats = torch.zeros(32, dtype=torch.int64, device="cuda")
    E.ntuple_tc_train(boards, after, scores, lengths, placements, W_t, E_t, A_t, alpha, subs_t[1:], mode, scratch,
                      stats)
    got = dict(T=W_t.cpu().numpy(), E=E_t.cpu().numpy(), A=A_t.cpu().numpy(),
               boards=boards.cpu().numpy().view(np.uint64), after=after.cpu().numpy().view(np.uint64),
               scores=scores.cpu().numpy().view(np.uint32), lengths=lengths.cpu().numpy().view(np.uint32),
               stats=stats.cpu().numpy().view(np.uint64))
    return got, scratch


def _run_both(n, n_steps, placements, W, sums, alpha, mode, seed=3):
    _, subs = CO.chain(np.array([0, seed], np.uint32), mode, 1 + n_steps)
    Es, As = (np.zeros(W.shape[0]), np.zeros(W.shape[0])) if sums is None else sums
    got, scratch = _gpu_tc_train(n, subs, mode, placements, W, Es, As, alpha)
    Es, As = Es.copy(), As.copy()
    want = TCO.tc_train(NO.fresh(subs[0], n, mode, W), Es, As, placements, alpha, subs[1:], mode)
    return got, want, Es, As, scratch


def _assert_same(got, want, Es, As):
    np.testing.assert_array_equal(got["T"].view(np.uint32), want.T.view(np.uint32))
    np.testing.assert_array_equal(got["E"].view(np.uint64), Es.view(np.uint64))
    np.testing.assert_array_equal(got["A"].view(np.uint64), As.view(np.uint64))
    for k in ("boards", "after", "scores", "lengths", "stats"):
        np.testing.assert_array_equal(got[k], getattr(want, k))


@pytest.mark.parametrize("mode", [E.RNG_PARTITIONABLE, E.RNG_ORIGINAL])
@pytest.mark.parametrize("n", [1, 33, 4096])
@pytest.mark.parametrize("n_steps", [1, 17, 500])
def test_tc_bit_exact_against_oracle(n, n_steps, mode):
    i = [1, 33, 4096].index(n) + [1, 17, 500].index(n_steps)
    alpha = (1.0 / 1024, 0.05, 1.0)[(i + mode) % 3]
    W = np.zeros(SMALL_WEIGHTS, np.float32) if i % 2 else random_weights(SMALL_WEIGHTS, 23)
    sums = random_sums(SMALL_WEIGHTS, 7) if (i + mode) % 2 else None
    got, want, Es, As, scratch = _run_both(n, n_steps, small_placements(), W, sums, alpha, mode)
    _assert_same(got, want, Es, As)
    assert int(torch.count_nonzero(scratch)) == 0
    if n_steps == 500:
        assert want.stats[0] > 0  # episodes ended and restarted inside the run


@pytest.mark.parametrize("mode", [E.RNG_PARTITIONABLE, E.RNG_ORIGINAL])
@pytest.mark.parametrize("alpha", [0.02, 0.5])
def test_tc_four_six_bit_exact_against_oracle(alpha, mode):
    W = random_weights(1 << 26, 5) if alpha == 0.5 else np.zeros(1 << 26, np.float32)
    got, want, Es, As, scratch = _run_both(33, 40, _four_six_host(), W, None, alpha, mode, seed=8)
    _assert_same(got, want, Es, As)
    assert int(torch.count_nonzero(scratch)) == 0


@pytest.mark.parametrize("mode", [E.RNG_PARTITIONABLE, E.RNG_ORIGINAL])
def test_tc_several_env_passes_per_step_bit_exact(mode):
    """n = 2^17: every thread walks several envs per step, and the CTA's index-0 sums of acc and abs span them."""
    got, want, Es, As, scratch = _run_both(1 << 17, 6, small_placements(), random_weights(SMALL_WEIGHTS, 12), None,
                                           0.05, mode, seed=12)
    _assert_same(got, want, Es, As)
    assert int(torch.count_nonzero(scratch)) == 0


def test_alpha_zero_keeps_the_weights_and_accumulates_the_sums():
    mode = E.RNG_PARTITIONABLE
    W = random_weights(SMALL_WEIGHTS, 31)
    got, want, Es, As, scratch = _run_both(4096, 60, small_placements(), W, None, 0.0, mode, seed=5)
    _assert_same(got, want, Es, As)
    np.testing.assert_array_equal(got["T"].view(np.uint32), W.view(np.uint32))
    assert (got["A"] > 0).sum() > 1000 and bool((np.abs(got["E"]) <= got["A"]).all())


def _small_net(weights=None):
    return NTupleNetwork(small_placements(), SMALL_WEIGHTS, weights)


def _state(lr):
    out = [lr.weights.clone(), lr.boards.clone(), lr.after.clone(), lr.scores.clone(), lr.lengths.clone()]
    if isinstance(lr, g2048.NTupleTCLearner):
        out += [lr.err_sum.clone(), lr.abs_err_sum.clone()]
    return out


@pytest.mark.parametrize("mode", [E.RNG_PARTITIONABLE, E.RNG_ORIGINAL])
def test_one_tc_step_from_zero_sums_is_one_td_step_through_the_public_api(mode):
    """A network trained by NTupleTDLearner, handed to NTupleTCLearner with the TD learner's env state: TC starts from
    those weights with E = A = 0, and its first step is the TD learner's next step, bit for bit."""
    n = 2048
    td = g2048.NTupleTDLearner(11, n, network=_small_net(random_weights(SMALL_WEIGHTS, 9)), alpha=0.02, rng_mode=mode)
    td.train(40)
    tc = g2048.NTupleTCLearner(0, n, network=_small_net(td.weights), alpha=0.02, rng_mode=mode)
    assert tc.alpha == 0.02 and not bool(tc.err_sum.any()) and not bool(tc.abs_err_sum.any())
    ckpt = td.state_dict()
    ckpt.update(err_sum=torch.zeros(SMALL_WEIGHTS, dtype=torch.float64),
                abs_err_sum=torch.zeros(SMALL_WEIGHTS, dtype=torch.float64))
    tc.load_state_dict(ckpt)
    assert td.train(1) == tc.train(1)
    for x, y in zip(_state(td), _state(tc)):
        assert torch.equal(x, y)
    assert bool((tc.abs_err_sum > 0).any())
    td.train(5)
    tc.train(5)
    assert not torch.equal(td.weights, tc.weights)  # later steps scale the errors by beta


@pytest.mark.parametrize("mode", [E.RNG_PARTITIONABLE, E.RNG_ORIGINAL])
def test_split_training_and_checkpoints_resume_bit_for_bit(mode):
    whole = g2048.NTupleTCLearner(5, 1000, network=_small_net(), alpha=0.5, rng_mode=mode)
    s_whole = whole.train(300)
    parts = g2048.NTupleTCLearner(5, 1000, network=_small_net(), alpha=0.5, rng_mode=mode)
    s1 = parts.train(120)
    ckpt = parts.state_dict()
    assert ckpt["err_sum"].dtype == ckpt["abs_err_sum"].dtype == torch.float64
    s2 = parts.train(180)
    for x, y in zip(_state(whole), _state(parts)):
        assert torch.equal(x, y)
    assert s1["episodes"] + s2["episodes"] == s_whole["episodes"] > 0
    resumed = g2048.NTupleTCLearner(99, 1000, network=_small_net(), alpha=0.01, rng_mode=1 - mode)
    resumed.load_state_dict(ckpt)
    assert resumed.train(180) == s2
    for x, y in zip(_state(whole), _state(resumed)):
        assert torch.equal(x, y)
    assert resumed.steps == whole.steps == 300 and np.array_equal(resumed.chain.key, whole.chain.key)


def test_load_state_dict_rejects_a_malformed_checkpoint():
    lr = g2048.NTupleTCLearner(2, 64, network=_small_net(), alpha=0.1)
    lr.train(3)
    good = lr.state_dict()
    before = _state(lr)
    neg = good["abs_err_sum"].clone()
    neg[5] = -1.0
    nan = good["err_sum"].clone()
    nan[7] = float("nan")
    for key, bad in (("err_sum", good["err_sum"].float()), ("abs_err_sum", good["abs_err_sum"][:-1]),
                     ("err_sum", torch.zeros((SMALL_WEIGHTS, 1), dtype=torch.float64)), ("err_sum", nan),
                     ("abs_err_sum", torch.full((SMALL_WEIGHTS,), float("inf"), dtype=torch.float64)),
                     ("abs_err_sum", neg), ("err_sum", None), ("weights", torch.zeros(100)), ("alpha", -1.0)):
        state = dict(good)
        if bad is None:
            del state[key]
        else:
            state[key] = bad
        with pytest.raises(ValueError):
            lr.load_state_dict(state)
    for x, y in zip(before, _state(lr)):  # a rejected checkpoint changes nothing
        assert torch.equal(x, y)
    lr.load_state_dict(dict(good, err_sum=good["err_sum"].numpy(), abs_err_sum=good["abs_err_sum"].numpy()))


def test_weights_sums_scratch_and_outputs_are_surrounded_by_untouched_guard_bands():
    from test_guard_bands_gpu import GuardedTorch

    guard = GuardedTorch()
    mode = E.RNG_PARTITIONABLE
    pl = small_placements()
    subs = E.chain_advance(E.words_tensor([0, 4], "cuda"), mode, 41)
    Es0, As0 = random_sums(SMALL_WEIGHTS, 3)
    for n in (1, 33, 4096):
        boards, _ = E.env_init(subs[0], n, 0, n, mode)
        b = guard.empty(n, dtype=torch.int64, device="cuda")
        b.copy_(boards)
        after = guard.zeros(n, dtype=torch.int64, device="cuda")
        scores = guard.zeros(n, dtype=torch.int32, device="cuda")
        lengths = guard.zeros(n, dtype=torch.int32, device="cuda")
        W = guard.empty(SMALL_WEIGHTS, dtype=torch.float32, device="cuda")
        W.copy_(torch.from_numpy(random_weights(SMALL_WEIGHTS, 2)).cuda())
        Es = guard.empty(SMALL_WEIGHTS, dtype=torch.float64, device="cuda")
        Es.copy_(torch.from_numpy(Es0).cuda())
        As = guard.empty(SMALL_WEIGHTS, dtype=torch.float64, device="cuda")
        As.copy_(torch.from_numpy(As0).cuda())
        size = int(N.lib.g2048_ntuple_tc_scratch_bytes(n, pl.shape[0], SMALL_WEIGHTS))
        scratch = guard.zeros(size // 8, dtype=torch.int64, device="cuda")
        stats = guard.zeros(32, dtype=torch.int64, device="cuda")
        E.ntuple_tc_train(b, after, scores, lengths, pl, W, Es, As, 0.05, subs[1:], mode, scratch, stats)
        assert int(torch.count_nonzero(scratch)) == 0
    assert len(guard.raw) == 3 * 9
    assert guard.check() == []


def test_learned_four_six_tc_network_beats_drul_and_the_zero_network():
    """Sanity, not parity: a short TC run of the 4x6 network from zeros at n = 2^16 at the default alpha, then its
    greedy player against DRUL and against the greedy player of the zero network, over the same 1 024 seeded games."""
    lr = g2048.NTupleTCLearner(1, 1 << 16)
    lr.train(1000)
    B = 1024

    def greedy(net):
        out = g2048.BatchRunner(7, g2048.ExpectimaxPolicy(depth=1, network=net, reward_weight=1.0)).run_eval_batch(B)
        return out["summary"]["score_sum"] / B

    learned = greedy(lr.network)
    zero = greedy(NTupleNetwork.four_six())
    drul = g2048.BatchRunner(7, g2048.act_drul).run_stats_batch(B)["summary"]["score_sum"] / B
    assert learned > drul and learned > zero, (learned, zero, drul)
