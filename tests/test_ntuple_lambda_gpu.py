"""Delayed TD(lambda) / TC(lambda) on the GPU (g2048_ntuple_lambda_td_train, g2048_ntuple_lambda_tc_train, the
learners' lam / horizon): W, E, A, the env state, the statistics and both rings bit for bit against
tests/ntuple_lambda_oracle.c, h = 1 against the four existing entry points, split calls, checkpoints, guard bands and a
learning sanity check."""
import numpy as np
import pytest
import torch

import g2048
from g2048 import engine as E
from g2048.ntuple import NTupleNetwork, make_stages
from oracle import c_oracle as CO

import ntuple_lambda_oracle as LO
from test_ntuple_gpu import SMALL_WEIGHTS, _four_six_host, _words, random_weights, small_placements
from test_ntuple_lambda_oracle import windowed_state
from test_ntuple_tc_gpu import random_sums

pytestmark = pytest.mark.gpu


def _dev(state, ha, hd):
    t = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a).view(dt)).cuda()  # noqa: E731
    return dict(boards=t(state.boards, np.int64), after=t(state.after, np.int64), scores=t(state.scores, np.int32),
                lengths=t(state.lengths, np.int32), ha=t(ha, np.int64), hd=t(hd, np.float32))


def _host(d):
    return dict(boards=d["boards"].cpu().numpy().view(np.uint64), after=d["after"].cpu().numpy().view(np.uint64),
                scores=d["scores"].cpu().numpy().view(np.uint32), lengths=d["lengths"].cpu().numpy().view(np.uint32),
                hist_after=d["ha"].cpu().numpy().view(np.uint64), hist_delta=d["hd"].cpu().numpy())


def _gpu_lambda(d, subs, mode, placements, stages, W_t, alpha, lam, sums=None, scratch=None, stats=None):
    """One call of the lambda entry point on device state d (from _dev), in place."""
    n, h = d["boards"].shape[0], d["ha"].shape[0]
    nw = W_t.numel()
    if sums is None:
        scratch = E.ntuple_td_scratch(n * h, placements, nw, "cuda") if scratch is None else scratch
        E.ntuple_lambda_td_train(d["boards"], d["after"], d["scores"], d["lengths"], placements, W_t, alpha, lam,
                                 d["ha"], d["hd"], _words(subs), mode, scratch, stats, stages=stages)
    else:
        scratch = E.ntuple_tc_scratch(n * h, placements, nw, "cuda") if scratch is None else scratch
        E.ntuple_lambda_tc_train(d["boards"], d["after"], d["scores"], d["lengths"], placements, W_t, sums[0], sums[1],
                                 alpha, lam, d["ha"], d["hd"], _words(subs), mode, scratch, stats, stages=stages)
    return scratch


def _run_both(n, h, n_steps, placements, stages, W, alpha, lam, mode, tc, seed=3, start=None):
    state, ha, hd = windowed_state(n, h, seed, mode, W) if start is None else start
    _, subs = CO.chain(np.array([0, seed], np.uint32), mode, n_steps)
    d = _dev(state, ha, hd)
    W_t = torch.from_numpy(W).cuda()
    stats = torch.zeros(32, dtype=torch.int64, device="cuda")
    if tc:
        Es, As = random_sums(W.shape[0], seed) if W.shape[0] <= 1 << 26 else (np.zeros(W.shape[0]), np.zeros(W.shape[0]))
        sums = (torch.from_numpy(Es).cuda(), torch.from_numpy(As).cuda())
        scratch = _gpu_lambda(d, subs, mode, placements, stages, W_t, alpha, lam, sums, stats=stats)
        Es, As = Es.copy(), As.copy()
        want = LO.tc_train(state, Es, As, ha, hd, placements, stages, alpha, lam, subs, mode)
        np.testing.assert_array_equal(sums[0].cpu().numpy().view(np.uint64), Es.view(np.uint64))
        np.testing.assert_array_equal(sums[1].cpu().numpy().view(np.uint64), As.view(np.uint64))
    else:
        scratch = _gpu_lambda(d, subs, mode, placements, stages, W_t, alpha, lam, stats=stats)
        want = LO.train(state, ha, hd, placements, stages, alpha, lam, subs, mode)
    assert int(torch.count_nonzero(scratch)) == 0
    got = _host(d)
    np.testing.assert_array_equal(W_t.cpu().numpy().view(np.uint32), want.T.view(np.uint32))
    for k in ("boards", "after", "scores", "lengths"):
        np.testing.assert_array_equal(got[k], getattr(want, k))
    np.testing.assert_array_equal(stats.cpu().numpy().view(np.uint64), want.stats)
    np.testing.assert_array_equal(got["hist_after"], ha)
    np.testing.assert_array_equal(got["hist_delta"].view(np.uint32), hd.view(np.uint32))
    assert want.stats[0] > 0
    return want


@pytest.mark.parametrize("staged", [False, True])
@pytest.mark.parametrize("tc", [False, True])
@pytest.mark.parametrize("h", [2, 3, 8])
@pytest.mark.parametrize("lam", [0.0, 0.5, 1.0])
def test_lambda_bit_exact_against_oracle(lam, h, tc, staged):
    mode = (E.RNG_PARTITIONABLE, E.RNG_ORIGINAL)[(h + tc + staged) % 2]
    stages = make_stages((3, 5), SMALL_WEIGHTS) if staged else None
    nw = (3 if staged else 1) * SMALL_WEIGHTS
    W = random_weights(nw, 23 + h)
    _run_both(777, h, 40, small_placements(), stages, W, 0.05, lam, mode, tc, seed=h + 7)


@pytest.mark.parametrize("tc", [False, True])
def test_four_six_at_n_times_h_of_2_to_the_20_bit_exact(tc):
    """n = 2^17, h = 8: every thread walks several envs a step, and n * h is the largest the contract allows."""
    W = random_weights(1 << 26, 5) if tc else np.zeros(1 << 26, np.float32)
    _run_both(1 << 17, 8, 5, _four_six_host(), None, W, 0.02, 0.5, E.RNG_PARTITIONABLE, tc, seed=8)


def _full_windows(n, h, seed, mode, W):
    """windowed_state with every env at L = h .. h + 2 (a full window; every third env, env 0 included, on a board
    without a legal move, so it releases its whole window on the first step), and env 4 holding an afterstate with
    L = 0, which is outside the contract: it must store and release nothing."""
    state, ha, hd = windowed_state(n, h, seed, mode, W)
    L = h + np.arange(n) % 3
    state.lengths[:] = L
    state.after[:] = ha[(L - 1) % h, np.arange(n)]
    if n > 4:
        state.lengths[4] = 0
    return state, ha, hd


@pytest.mark.parametrize("tc", [False, True])
@pytest.mark.parametrize("n", [1, 5, 16])
def test_few_envs_releasing_whole_windows_bit_exact(n, tc):
    """The 4x6 network with few envs (n * P < n_weights) and h = 8: an env that ends its episode releases 8 afterstates
    at once, so one step lists up to n * 8 * 32 entries, more than the n * 32 a TD(0) step of n envs can touch."""
    h, mode = 8, (E.RNG_PARTITIONABLE, E.RNG_ORIGINAL)[n % 2]
    W = random_weights(1 << 26, 13) if tc else np.zeros(1 << 26, np.float32)
    start = _full_windows(n, h, 14 + n, mode, W)
    _run_both(n, h, 20, _four_six_host(), None, W, 0.02, 0.5, mode, tc, seed=14 + n, start=start)


@pytest.mark.parametrize("tc", [False, True])
def test_two_stage_four_six_bit_exact(tc):
    W = random_weights(1 << 27, 6) if tc else np.zeros(1 << 27, np.float32)
    _run_both(4096, 3, 30, _four_six_host(), make_stages((4,), 1 << 26), W, 0.02, 0.75, E.RNG_ORIGINAL, tc, seed=9)


@pytest.mark.parametrize("mode", [E.RNG_PARTITIONABLE, E.RNG_ORIGINAL])
@pytest.mark.parametrize("staged", [False, True])
@pytest.mark.parametrize("tc", [False, True])
def test_horizon_one_equals_the_existing_entry_points(tc, staged, mode):
    stages = make_stages((3, 5), SMALL_WEIGHTS) if staged else None
    nw = (3 if staged else 1) * SMALL_WEIGHTS
    W = random_weights(nw, 4)
    state, ha, hd = windowed_state(2048, 1, 4, mode, W)
    _, subs = CO.chain(np.array([0, 6], np.uint32), mode, 80)
    sums = random_sums(nw, 4) if tc else None
    out = []
    for lam in (None, 0.0, 0.7):
        d = _dev(state, ha, hd)
        W_t = torch.from_numpy(W).cuda()
        s = None if sums is None else (torch.from_numpy(sums[0]).cuda(), torch.from_numpy(sums[1]).cuda())
        stats = torch.zeros(32, dtype=torch.int64, device="cuda")
        args = (d["boards"], d["after"], d["scores"], d["lengths"], small_placements(), W_t)
        if lam is not None:
            _gpu_lambda(d, subs, mode, small_placements(), stages, W_t, 0.05, lam, s, stats=stats)
        elif tc:
            E.ntuple_tc_train(*args, s[0], s[1], 0.05, _words(subs), mode,
                              E.ntuple_tc_scratch(2048, small_placements(), nw, "cuda"), stats, stages=stages)
        else:
            E.ntuple_td_train(*args, 0.05, _words(subs), mode, E.ntuple_td_scratch(2048, small_placements(), nw, "cuda"),
                              stats, stages=stages)
        h = _host(d)
        h.update(W=W_t.cpu().numpy().view(np.uint32), stats=stats.cpu().numpy())
        if s is not None:
            h.update(E=s[0].cpu().numpy(), A=s[1].cpu().numpy())
        out.append(h)
    for other in out[1:]:
        for k in out[0]:
            if not k.startswith("hist_"):  # the existing entry points keep no rings
                np.testing.assert_array_equal(out[0][k], other[k], err_msg=k)
    for k in out[1]:  # with h = 1, lambda changes nothing, the rings included
        np.testing.assert_array_equal(out[1][k], out[2][k], err_msg=k)
    assert out[0]["stats"][0] > 0


@pytest.mark.parametrize("tc", [False, True])
def test_one_call_equals_two_half_calls(tc):
    mode = E.RNG_PARTITIONABLE
    W = random_weights(SMALL_WEIGHTS, 12)
    state, ha, hd = windowed_state(3000, 5, 12, mode, W)
    _, subs = CO.chain(np.array([0, 12], np.uint32), mode, 120)
    res = []
    for splits in ((0, 120), (0, 60, 120)):
        d = _dev(state, ha, hd)
        W_t = torch.from_numpy(W).cuda()
        s = None
        if tc:
            Es, As = random_sums(SMALL_WEIGHTS, 12)
            s = (torch.from_numpy(Es).cuda(), torch.from_numpy(As).cuda())
        scratch = None
        for a, b in zip(splits[:-1], splits[1:]):
            scratch = _gpu_lambda(d, subs[a:b], mode, small_placements(), None, W_t, 0.05, 0.6, s, scratch=scratch)
        res.append([W_t.cpu()] + [v.cpu() for v in d.values()] + ([] if s is None else [x.cpu() for x in s]))
    for x, y in zip(*res):
        assert torch.equal(x, y)


# ------------------------------------------------------------------------------------------ learners, checkpoints
def _small_net():
    return NTupleNetwork(small_placements(), SMALL_WEIGHTS)


def _state(lr):
    out = [lr.weights.clone(), lr.boards.clone(), lr.after.clone(), lr.scores.clone(), lr.lengths.clone(),
           lr.hist_after.clone(), lr.hist_delta.clone()]
    if isinstance(lr, g2048.NTupleTCLearner):
        out += [lr.err_sum.clone(), lr.abs_err_sum.clone()]
    return out


@pytest.mark.parametrize("cls", [g2048.NTupleTDLearner, g2048.NTupleTCLearner])
def test_checkpoint_mid_episode_resumes_bit_for_bit(cls):
    whole = cls(5, 1000, network=_small_net(), alpha=0.5, lam=0.5, horizon=4)
    s_whole = whole.train(301)
    parts = cls(5, 1000, network=_small_net(), alpha=0.5, lam=0.5, horizon=4)
    s1 = parts.train(121)
    ckpt = parts.state_dict()
    assert ckpt["horizon"] == 4 and ckpt["lam"] == 0.5 and tuple(ckpt["hist_after"].shape) == (4, 1000)
    lengths = ckpt["lengths"]
    assert bool(((lengths > 0) & (lengths < 4)).any()) and bool((lengths >= 4).any())  # windows partly and fully filled
    s2 = parts.train(180)
    for x, y in zip(_state(whole), _state(parts)):
        assert torch.equal(x, y)
    assert s1["episodes"] + s2["episodes"] == s_whole["episodes"] > 0
    resumed = cls(99, 1000, network=_small_net(), alpha=0.01, lam=0.9, horizon=4)
    resumed.load_state_dict(ckpt)
    assert resumed.lam == 0.5
    assert resumed.train(180) == s2
    for x, y in zip(_state(whole), _state(resumed)):
        assert torch.equal(x, y)


def test_a_checkpoint_with_another_window_is_rejected_before_anything_changes():
    lr = g2048.NTupleTDLearner(2, 64, network=_small_net(), alpha=0.1, lam=0.5, horizon=3)
    lr.train(5)
    good = lr.state_dict()
    before = _state(lr)
    bad_entries = [("horizon", 2), ("horizon", None), ("horizon", 3.5), ("horizon", "3"), ("lam", float("nan")),
                   ("lam", 1.5), ("lam", None),
                   ("hist_after", torch.zeros((2, 64), dtype=torch.int64)),
                   ("hist_after", torch.zeros((3, 64), dtype=torch.int32)),
                   ("hist_delta", torch.zeros((3, 65), dtype=torch.float32)),
                   ("hist_delta", torch.zeros((3, 64), dtype=torch.float64)), ("hist_delta", None)]
    for key, bad in bad_entries:
        state = dict(good)
        if bad is None:
            del state[key]
        else:
            state[key] = bad
        with pytest.raises(ValueError):
            lr.load_state_dict(state)
    for x, y in zip(before, _state(lr)):
        assert torch.equal(x, y)
    # a horizon-1 learner writes today's checkpoint, takes one without window entries, and rejects a windowed one
    single = g2048.NTupleTDLearner(2, 64, network=_small_net(), alpha=0.1)
    old = single.state_dict()
    assert not {"lam", "horizon", "hist_after", "hist_delta"} & set(old)
    single.load_state_dict(old)
    with pytest.raises(ValueError, match="horizon"):
        single.load_state_dict(good)


def test_learners_take_the_lambda_path_only_above_horizon_one(monkeypatch):
    calls = []
    for name in ("ntuple_td_train", "ntuple_tc_train", "ntuple_lambda_td_train", "ntuple_lambda_tc_train"):
        orig = getattr(E, name)

        def spy(*args, _orig=orig, _name=name, **kw):
            calls.append(_name)
            return _orig(*args, **kw)

        monkeypatch.setattr(E, name, spy)
    g2048.NTupleTDLearner(0, 32, network=_small_net(), lam=0.5).train(2)
    g2048.NTupleTCLearner(0, 32, network=_small_net(), lam=0.5).train(2)
    g2048.NTupleTDLearner(0, 32, network=_small_net(), lam=0.5, horizon=2).train(2)
    g2048.NTupleTCLearner(0, 32, network=_small_net(), lam=0.5, horizon=2).train(2)
    assert calls == ["ntuple_td_train", "ntuple_tc_train", "ntuple_lambda_td_train", "ntuple_lambda_tc_train"]


def test_rings_weights_sums_and_scratch_are_surrounded_by_untouched_guard_bands():
    from test_guard_bands_gpu import GuardedTorch

    guard = GuardedTorch()
    mode = E.RNG_PARTITIONABLE
    pl, nw = small_placements(), SMALL_WEIGHTS
    W0 = random_weights(nw, 2)
    for n, h in ((1, 8), (33, 3), (4096, 2)):
        state, ha, hd = windowed_state(n, h, 3, mode, W0)
        _, subs = CO.chain(np.array([0, 3], np.uint32), mode, 30)
        for tc in (False, True):
            src = _dev(state, ha, hd)
            d = {}
            for k, v in src.items():
                d[k] = guard.empty(*v.shape, dtype=v.dtype, device="cuda")
                d[k].copy_(v)
            W = guard.empty(nw, dtype=torch.float32, device="cuda")
            W.copy_(torch.from_numpy(W0).cuda())
            stats = guard.zeros(32, dtype=torch.int64, device="cuda")
            size_of = E.N.lib.g2048_ntuple_tc_scratch_bytes if tc else E.N.lib.g2048_ntuple_td_scratch_bytes
            scratch = guard.zeros(int(size_of(n * h, pl.shape[0], nw)) // 8, dtype=torch.int64, device="cuda")
            sums = (guard.zeros(nw, dtype=torch.float64, device="cuda"),
                    guard.zeros(nw, dtype=torch.float64, device="cuda")) if tc else None
            _gpu_lambda(d, subs, mode, pl, None, W, 0.05, 0.5, sums, scratch=scratch, stats=stats)
            assert int(torch.count_nonzero(scratch)) == 0
    assert guard.check() == []


def test_lambda_four_six_learner_beats_drul_by_a_wide_margin():
    """Sanity, not parity: a short TD(0.5) run with h = 3 of the 4x6 network from zeros at n = 2^16, then its greedy
    player against DRUL over the same 1 024 seeded games."""
    lr = g2048.NTupleTDLearner(1, 1 << 16, lam=0.5, horizon=3)
    lr.train(1000)
    B = 1024
    out = g2048.BatchRunner(7, g2048.ExpectimaxPolicy(depth=1, network=lr.network, reward_weight=1.0)).run_eval_batch(B)
    learned = out["summary"]["score_sum"] / B
    drul = g2048.BatchRunner(7, g2048.act_drul).run_stats_batch(B)["summary"]["score_sum"] / B
    assert learned > 3 * drul, (learned, drul)
