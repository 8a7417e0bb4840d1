"""Carousel shaping on the GPU (g2048_ntuple_carousel_td_train, g2048_ntuple_carousel_tc_train, the learners'
carousel): W, E, A, the env state, both rings, start_stage, stage_pool and the statistics bit for bit against
tests/ntuple_carousel_oracle.c; a threshold never reached against the staged and lambda entry points; split calls;
checkpoints; guard bands; and a deterministic learning check."""
import numpy as np
import pytest
import torch

import g2048
from g2048 import engine as E
from g2048.ntuple import NTupleNetwork, make_stages
from oracle import c_oracle as CO

import ntuple_carousel_oracle as KO
from test_ntuple_carousel_oracle import _packed, carousel_state, short_games
from test_ntuple_gpu import SMALL_WEIGHTS, _four_six_host, _words, random_weights, small_placements
from test_ntuple_tc_gpu import random_sums

pytestmark = pytest.mark.gpu


def _dev(state, ss, pool, ha, hd):
    t = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a).view(dt)).cuda()  # noqa: E731
    d = dict(boards=t(state.boards, np.int64), after=t(state.after, np.int64), scores=t(state.scores, np.int32),
             lengths=t(state.lengths, np.int32), ss=t(ss, np.int32), pool=t(pool, np.int64))
    if ha is not None:
        d.update(ha=t(ha, np.int64), hd=t(hd, np.float32))
    return d


def _host(d):
    out = {k: d[k].cpu().numpy() for k in d}
    for k, dt in (("boards", np.uint64), ("after", np.uint64), ("scores", np.uint32), ("lengths", np.uint32),
                  ("ss", np.uint32), ("pool", np.uint64), ("ha", np.uint64), ("hd", np.uint32)):
        if k in out:
            out[k] = out[k].view(dt)
    return out


def _gpu(d, subs, mode, placements, stages, W_t, alpha, lam=0.5, sums=None, scratch=None, stats=None):
    """One call of a carousel entry point on device state d (from _dev), in place; returns the scratch."""
    n, h = d["boards"].shape[0], (d["ha"].shape[0] if "ha" in d else 1)
    tc = sums is not None
    if scratch is None:
        scratch = E.ntuple_carousel_scratch(n, h, placements, W_t.numel(), tc, "cuda")
    args = (d["boards"], d["after"], d["scores"], d["lengths"], placements, W_t)
    rest = (lam, d.get("ha"), d.get("hd"), d["ss"], d["pool"], _words(subs), mode, scratch, stats)
    if tc:
        E.ntuple_carousel_tc_train(*args, sums[0], sums[1], alpha, *rest, stages=stages)
    else:
        E.ntuple_carousel_td_train(*args, alpha, *rest, stages=stages)
    return scratch


def _run_both(start, n_steps, placements, stages, W, alpha, mode, tc, seed):
    state, ss, pool, ha, hd = start
    _, subs = CO.chain(np.array([0, seed], np.uint32), mode, n_steps)
    d = _dev(state, ss, pool, ha, hd)
    W_t = torch.from_numpy(W).cuda()
    stats = torch.zeros(32, dtype=torch.int64, device="cuda")
    rings = {} if ha is None else dict(lam=0.5, hist_after=ha, hist_delta=hd)
    if tc:
        Es, As = random_sums(W.shape[0], seed)
        sums = (torch.from_numpy(Es).cuda(), torch.from_numpy(As).cuda())
        scratch = _gpu(d, subs, mode, placements, stages, W_t, alpha, sums=sums, stats=stats)
        Es, As = Es.copy(), As.copy()
        want = KO.tc_train(state, Es, As, ss, pool, placements, stages, alpha, subs, mode, **rings)
        np.testing.assert_array_equal(sums[0].cpu().numpy().view(np.uint64), Es.view(np.uint64))
        np.testing.assert_array_equal(sums[1].cpu().numpy().view(np.uint64), As.view(np.uint64))
    else:
        scratch = _gpu(d, subs, mode, placements, stages, W_t, alpha, stats=stats)
        want = KO.train(state, ss, pool, placements, stages, alpha, subs, mode, **rings)
    assert int(torch.count_nonzero(scratch)) == 0
    got = _host(d)
    np.testing.assert_array_equal(W_t.cpu().numpy().view(np.uint32), want.T.view(np.uint32))
    for k in ("boards", "after", "scores", "lengths"):
        np.testing.assert_array_equal(got[k], getattr(want, k), err_msg=k)
    np.testing.assert_array_equal(got["ss"], ss)
    np.testing.assert_array_equal(got["pool"], pool)
    np.testing.assert_array_equal(stats.cpu().numpy().view(np.uint64), want.stats)
    if ha is not None:
        np.testing.assert_array_equal(got["ha"], ha)
        np.testing.assert_array_equal(got["hd"], hd.view(np.uint32))
    return want


CASES = [(1, (3,)), (5, (3, 5)), (777, (3, 5)), (1 << 17, (3,))]  # 2^17: several env passes per CTA


@pytest.mark.parametrize("case", range(len(CASES)))
@pytest.mark.parametrize("h", [1, 3])
@pytest.mark.parametrize("tc", [False, True])
def test_carousel_bit_exact_against_oracle(tc, h, case):
    n, thresholds = CASES[case]
    mode = (E.RNG_PARTITIONABLE, E.RNG_ORIGINAL)[(h + tc + case) % 2]
    S = len(thresholds) + 1
    stages = make_stages(thresholds, SMALL_WEIGHTS)
    W = random_weights(S * SMALL_WEIGHTS, 23 + h)
    n_steps = 200 if n < 10 else 40
    want = _run_both(carousel_state(n, S, 31 + n, mode, W, h), n_steps, small_placements(), stages, W, 0.05, mode,
                     tc, seed=h + 7 + case)
    assert want.stats[12] > 0


def _four_six_start(n, mode, W, h, seed):
    """carousel_state with the 4x6 network's split at 13: half of the pool holds short games with an 8192 tile (the
    other half is empty), and a third of the envs play two adjacent 4096 tiles, which they merge into stage 1."""
    state, ss, pool, ha, hd = carousel_state(n, 2, seed, mode, W, h)
    rng = np.random.default_rng(seed)
    high = short_games(n, rng)
    high = (high & ~np.uint64(0xF)) | np.uint64(13)  # cell 0 holds the 8192 tile
    pool[0] = np.where(rng.random(n) < 0.5, high, np.uint64(0))
    state.boards[2::3] = _packed([12, 12] + [0] * 14)
    return state, ss, pool, ha, hd


@pytest.mark.parametrize("h", [1, 3])
@pytest.mark.parametrize("tc", [False, True])
def test_four_six_with_a_prefilled_pool_bit_exact(tc, h):
    mode = (E.RNG_PARTITIONABLE, E.RNG_ORIGINAL)[h % 2]
    W = random_weights(1 << 27, 6) if tc else np.zeros(1 << 27, np.float32)
    start = _four_six_start(4096, mode, W, h, 9 + h)
    want = _run_both(start, 30, _four_six_host(), make_stages((13,), 1 << 26), W, 0.02, mode, tc, seed=9)
    assert want.stats[12] > 0


@pytest.mark.parametrize("h", [1, 3])
@pytest.mark.parametrize("tc", [False, True])
def test_a_threshold_never_reached_equals_the_staged_and_lambda_entry_points(tc, h):
    mode = E.RNG_PARTITIONABLE
    stages = make_stages((15,), 1 << 26)
    W = random_weights(1 << 27, 4) if tc else np.zeros(1 << 27, np.float32)
    n = 4096
    state, _, _, ha, hd = carousel_state(n, 2, 4, mode, W, h)
    ss, pool = np.zeros(n, np.uint32), np.zeros((1, n), np.uint64)
    _, subs = CO.chain(np.array([0, 6], np.uint32), mode, 60)
    pl = _four_six_host()
    out = []
    for carousel in (False, True):
        d = _dev(state, ss, pool, ha, hd)
        W_t = torch.from_numpy(W).cuda()
        sums = None
        if tc:
            Es, As = random_sums(W.shape[0], 4)
            sums = (torch.from_numpy(Es).cuda(), torch.from_numpy(As).cuda())
        stats = torch.zeros(32, dtype=torch.int64, device="cuda")
        args = (d["boards"], d["after"], d["scores"], d["lengths"], pl, W_t)
        if carousel:
            _gpu(d, subs, mode, pl, stages, W_t, 0.02, sums=sums, stats=stats)
        elif h == 1 and tc:
            E.ntuple_tc_train(*args, *sums, 0.02, _words(subs), mode, E.ntuple_tc_scratch(n, pl, W_t.numel(), "cuda"),
                              stats, stages=stages)
        elif h == 1:
            E.ntuple_td_train(*args, 0.02, _words(subs), mode, E.ntuple_td_scratch(n, pl, W_t.numel(), "cuda"), stats,
                              stages=stages)
        elif tc:
            E.ntuple_lambda_tc_train(*args, *sums, 0.02, 0.5, d["ha"], d["hd"], _words(subs), mode,
                                     E.ntuple_tc_scratch(n * h, pl, W_t.numel(), "cuda"), stats, stages=stages)
        else:
            E.ntuple_lambda_td_train(*args, 0.02, 0.5, d["ha"], d["hd"], _words(subs), mode,
                                     E.ntuple_td_scratch(n * h, pl, W_t.numel(), "cuda"), stats, stages=stages)
        res = _host(d)
        res.update(W=W_t.cpu().numpy().view(np.uint32), stats=stats.cpu().numpy())
        if sums is not None:
            res.update(E=sums[0].cpu().numpy(), A=sums[1].cpu().numpy())
        out.append(res)
    for k in out[0]:
        np.testing.assert_array_equal(out[0][k], out[1][k], err_msg=k)
    assert out[0]["stats"][0] > 0 and not out[1]["pool"].any() and not out[1]["ss"].any()


@pytest.mark.parametrize("h", [1, 3])
@pytest.mark.parametrize("tc", [False, True])
def test_one_call_equals_two_calls(tc, h):
    """The stage entries recorded in a call's last step are committed before it returns."""
    mode = E.RNG_PARTITIONABLE
    stages = make_stages((3,), SMALL_WEIGHTS)
    W = random_weights(2 * SMALL_WEIGHTS, 12)
    start = carousel_state(3000, 2, 12, mode, W, h)
    _, subs = CO.chain(np.array([0, 12], np.uint32), mode, 120)
    res = []
    for splits in ((0, 120), (0, 37, 120)):
        d = _dev(*start)
        W_t = torch.from_numpy(W).cuda()
        s = None
        if tc:
            Es, As = random_sums(W.shape[0], 12)
            s = (torch.from_numpy(Es).cuda(), torch.from_numpy(As).cuda())
        scratch = None
        for a, b in zip(splits[:-1], splits[1:]):
            scratch = _gpu(d, subs[a:b], mode, small_placements(), stages, W_t, 0.05, sums=s, scratch=scratch)
        res.append([W_t.cpu()] + [v.cpu() for v in d.values()] + ([] if s is None else [x.cpu() for x in s]))
    for x, y in zip(*res):
        assert torch.equal(x, y)
    assert bool((res[0][1 + list(d).index("ss")] != 0).any())


# ------------------------------------------------------------------------------------------ learners, checkpoints
def _staged_net():
    return NTupleNetwork(small_placements(), 2 * SMALL_WEIGHTS, stage_thresholds=(3,), stage_stride=SMALL_WEIGHTS)


def _state(lr):
    out = [lr.weights.clone(), lr.boards.clone(), lr.after.clone(), lr.scores.clone(), lr.lengths.clone(),
           lr.start_stage.clone(), lr.stage_pool.clone()]
    if lr.horizon > 1:
        out += [lr.hist_after.clone(), lr.hist_delta.clone()]
    if isinstance(lr, g2048.NTupleTCLearner):
        out += [lr.err_sum.clone(), lr.abs_err_sum.clone()]
    return out


@pytest.mark.parametrize("h", [1, 3])
@pytest.mark.parametrize("cls", [g2048.NTupleTDLearner, g2048.NTupleTCLearner])
def test_checkpoint_mid_episode_resumes_bit_for_bit(cls, h):
    whole = cls(5, 1000, network=_staged_net(), alpha=0.5, lam=0.5, horizon=h, carousel=True)
    s_whole = whole.train(601)
    parts = cls(5, 1000, network=_staged_net(), alpha=0.5, lam=0.5, horizon=h, carousel=True)
    s1 = parts.train(321)
    ckpt = parts.state_dict()
    assert ckpt["carousel"] is True and tuple(ckpt["stage_pool"].shape) == (1, 1000)
    assert bool((ckpt["start_stage"] == 1).any()) and bool((ckpt["stage_pool"] != 0).any())
    s2 = parts.train(280)
    for x, y in zip(_state(whole), _state(parts)):
        assert torch.equal(x, y)
    assert s1["shaped_episodes"] + s2["shaped_episodes"] == s_whole["shaped_episodes"] > 0
    assert s1["episodes"] + s2["episodes"] == s_whole["episodes"] > 0
    resumed = cls(99, 1000, network=_staged_net(), alpha=0.01, lam=0.9, horizon=h, carousel=True)
    resumed.load_state_dict(ckpt)
    assert resumed.train(280) == s2
    for x, y in zip(_state(whole), _state(resumed)):
        assert torch.equal(x, y)


def test_a_checkpoint_that_does_not_fit_is_rejected_before_anything_changes():
    lr = g2048.NTupleTCLearner(2, 64, network=_staged_net(), alpha=0.1, carousel=True)
    lr.train(40)
    good = lr.state_dict()
    before = _state(lr)
    bad_entries = [("carousel", False), ("carousel", None), ("carousel", "yes"),
                   ("start_stage", torch.zeros(65, dtype=torch.int32)),
                   ("start_stage", torch.zeros(64, dtype=torch.int64)),
                   ("start_stage", torch.full((64,), 2, dtype=torch.int32)),
                   ("start_stage", torch.full((64,), -1, dtype=torch.int32)), ("start_stage", None),
                   ("stage_pool", torch.zeros((2, 64), dtype=torch.int64)),
                   ("stage_pool", torch.zeros((1, 64), dtype=torch.int32)),
                   ("stage_pool", torch.zeros(64, dtype=torch.int64)), ("stage_pool", None)]
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
    # a learner without the carousel writes today's checkpoint and rejects one with it
    plain = g2048.NTupleTCLearner(2, 64, network=_staged_net(), alpha=0.1)
    old = plain.state_dict()
    assert not {"carousel", "start_stage", "stage_pool"} & set(old)
    with pytest.raises(ValueError, match="carousel"):
        plain.load_state_dict(good)
    with pytest.raises(ValueError, match="carousel"):
        lr.load_state_dict(old)
    plain.load_state_dict(old)


def test_learners_take_the_carousel_path_for_every_horizon(monkeypatch):
    calls = []
    for name in ("ntuple_td_train", "ntuple_tc_train", "ntuple_lambda_td_train", "ntuple_lambda_tc_train",
                 "ntuple_carousel_td_train", "ntuple_carousel_tc_train"):
        orig = getattr(E, name)

        def spy(*args, _orig=orig, _name=name, **kw):
            calls.append(_name)
            return _orig(*args, **kw)

        monkeypatch.setattr(E, name, spy)
    for h in (1, 2):
        g2048.NTupleTDLearner(0, 32, network=_staged_net(), lam=0.5, horizon=h, carousel=True).train(2)
        g2048.NTupleTCLearner(0, 32, network=_staged_net(), lam=0.5, horizon=h, carousel=True).train(2)
    g2048.NTupleTDLearner(0, 32, network=_staged_net()).train(2)
    assert calls == ["ntuple_carousel_td_train", "ntuple_carousel_tc_train"] * 2 + ["ntuple_td_train"]


def test_carousel_arrays_scratch_and_outputs_are_surrounded_by_untouched_guard_bands():
    from test_guard_bands_gpu import GuardedTorch

    guard = GuardedTorch()
    mode = E.RNG_PARTITIONABLE
    pl, nw = small_placements(), 3 * SMALL_WEIGHTS
    stages = make_stages((3, 5), SMALL_WEIGHTS)
    W0 = random_weights(nw, 2)
    for n, h in ((1, 1), (33, 3), (4096, 1), (777, 8)):
        start = carousel_state(n, 3, 3, mode, W0, h)
        _, subs = CO.chain(np.array([0, 3], np.uint32), mode, 60)
        for tc in (False, True):
            src = _dev(*start)
            d = {}
            for k, v in src.items():
                d[k] = guard.empty(*v.shape, dtype=v.dtype, device="cuda")
                d[k].copy_(v)
            W = guard.empty(nw, dtype=torch.float32, device="cuda")
            W.copy_(torch.from_numpy(W0).cuda())
            stats = guard.zeros(32, dtype=torch.int64, device="cuda")
            size = int(E.N.lib.g2048_ntuple_carousel_scratch_bytes(n, h, pl.shape[0], nw, int(tc)))
            scratch = guard.zeros(size // 8, dtype=torch.int64, device="cuda")
            sums = (guard.zeros(nw, dtype=torch.float64, device="cuda"),
                    guard.zeros(nw, dtype=torch.float64, device="cuda")) if tc else None
            _gpu(d, subs, mode, pl, stages, W, 0.05, sums=sums, scratch=scratch, stats=stats)
            assert int(torch.count_nonzero(scratch)) == 0
    assert guard.check() == []


def test_carousel_trains_more_stage_one_entries():
    """Deterministic, not a score threshold: TC of the 4x6 network split at 11 (a 2048 tile) from zeros at n = 2^14,
    the same seed with and without the carousel.  Once envs reach the 2048 tile, the carousel restarts episodes from
    their stage entries, and more stage-1 entries are ever updated (A > 0)."""
    n, steps = 1 << 14, 3000
    runs = {}
    for carousel in (False, True):
        net = NTupleNetwork.staged(NTupleNetwork.four_six(), (11,))
        lr = g2048.NTupleTCLearner(0, n, network=net, carousel=carousel)
        s = lr.train(steps)
        runs[carousel] = dict(summary=s, updated=int((lr.abs_err_sum[1 << 26:] > 0).sum()), lr=lr)
    plain, shaped = runs[False], runs[True]
    reached = sum(v for k, v in plain["summary"]["max_tile_hist"].items() if k >= 2048)
    assert reached > 0 and bool((shaped["lr"].stage_pool != 0).any())
    assert shaped["summary"]["shaped_episodes"] > 0 and shaped["summary"]["shaped_env_steps"] > 0
    assert shaped["updated"] > plain["updated"] > 0, (shaped["updated"], plain["updated"])
