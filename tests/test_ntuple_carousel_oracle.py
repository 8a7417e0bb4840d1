"""CPU checks of carousel shaping (g2048_ntuple_carousel_td_train, g2048_ntuple_carousel_tc_train): the carousel oracle
(tests/ntuple_carousel_oracle.c) against a plain-Python restatement of the contract, the equivalence with the staged
and lambda oracles when no env enters a stage, and the argument checks of the C entry points, the engine wrappers and
the learners, which run before anything touches a device."""
import numpy as np
import pytest
import torch

from oracle import c_oracle as CO
from oracle import pgx2048_oracle as O

import ntuple_carousel_oracle as KO
import ntuple_lambda_oracle as LO
import ntuple_oracle as NO
import ntuple_stages_oracle as SO
from test_ntuple_oracle import TINY, TINY_WEIGHTS, _fx, _pack, _unpack, _weights
from test_ntuple_stages_oracle import _entries_s, _stage, _V_s

from g2048 import ntuple as NT

F = np.float32
_SHIFTS = np.arange(16, dtype=np.uint64) * np.uint64(4)


def _packed(cells):
    return (np.asarray(cells, np.uint64) << _SHIFTS).sum(axis=-1, dtype=np.uint64)


def short_games(n, rng):
    """(n,) packed boards a few moves from the end: a board without a legal move (neighbours differ in parity), exponents
    up to 6, with one or two cells emptied."""
    parity = np.array([(r + c) % 2 for r in range(4) for c in range(4)])
    cells = 1 + parity + 2 * rng.integers(0, 3, (n, 16))
    for i in range(n):
        cells[i, rng.choice(16, size=1 + i % 2, replace=False)] = 0
    return _packed(cells)


def carousel_state(n, S, seed, mode, W, h):
    """Envs whose episodes end every few steps and a part-filled pool: a third of the envs on boards without a legal
    move, a third a few moves from the end and a third on boards of two adjacent 4s, which enter stage 1 of threshold 3
    on their first move (so that envs which end in step 1 can draw the slot of an env that records an entry in it).
    Start stages cover every stage and the wrap (S - 1 and above, 2^32 - 1 included); about half of the pool entries
    hold short games, the rest are empty.  Returns (state, start_stage, pool, hist_after, hist_delta); the rings are
    None for h = 1."""
    rng = np.random.default_rng(seed)
    _, subs = CO.chain(np.array([1, seed], np.uint32), mode, 2)
    st = NO.fresh(subs[1], n, mode, W)
    parity = np.array([(r + c) % 2 for r in range(4) for c in range(4)])
    terminal = _packed(1 + parity + 2 * rng.integers(0, 3, (n, 16)))
    st.boards[0::3] = terminal[0::3]
    st.boards[1::3] = short_games(n, rng)[1::3]
    st.boards[2::3] = _packed([2, 2] + [0] * 14)
    start_stage = ((np.arange(n) // 3) % (S + 2)).astype(np.uint32)
    start_stage[start_stage == S + 1] = np.uint32(0xFFFFFFFF)
    pool = np.where(rng.random((S - 1, n)) < 0.5, short_games((S - 1) * n, rng).reshape(S - 1, n), np.uint64(0))
    pool = np.ascontiguousarray(pool, np.uint64)
    if h == 1:
        return st, start_stage, pool, None, None
    return st, start_stage, pool, np.zeros((h, n), np.uint64), np.zeros((h, n), np.float32)


def _draw_slot(key, n, mode):
    """j = (bits_scalar(k1) * n) >> 32 with split2(k) = (k1, k2), restated from the Threefry primitive."""
    k1 = CO.split(key, 2, mode)[0]
    a, b = CO.threefry2x32(int(k1[0]), int(k1[1]), 0, 0)
    bits = a ^ b if mode == CO.PARTITIONABLE else a
    return (bits * n) >> 32


def _py_train(st, start_stage, pool, ha, hd, rows, thresholds, stride, alpha, lam, subs, mode, sums=None):
    """The contract step by step in plain Python: np.float32 scalars for V, W, the errors and c_k, Python floats for E,
    A and beta, Python ints for the fixed-point sums; the game is the C oracle's.  h = 1 (``ha`` None) is TD(0) / TC.
    Also counts the draws of a slot that its env records in the same step (which must read the old board)."""
    W = st.T.copy()
    E, A = (None, None) if sums is None else ([float(x) for x in sums[0]], [float(x) for x in sums[1]])
    h = 1 if ha is None else ha.shape[0]
    ha = None if h == 1 else [[int(x) for x in row] for row in ha]
    hd = None if h == 1 else [[F(x) for x in row] for row in hd]
    c, d = [], 1.0
    for _ in range(h):
        c.append(F(d))
        d *= float(F(lam))
    S = len(thresholds) + 1
    boards, after = [int(x) for x in st.boards], [int(x) for x in st.after]
    scores, lengths = [int(x) for x in st.scores], [int(x) for x in st.lengths]
    start, pl = [int(x) for x in start_stage], [[int(x) for x in row] for row in pool]
    stats = [int(x) for x in st.stats]
    n = len(boards)
    events = dict(shaped_restarts=0, fallbacks=0, same_step=0, entries=0)
    for sub in np.asarray(subs, np.uint32).reshape(-1, 2):
        keys = CO.split(sub, n, mode)
        acc, absacc, cnt = {}, {}, {}
        draws, recorded = [], {}
        old_pool = [row[:] for row in pl]
        for e in range(n):
            s = _unpack(boards[e])
            legal = O.exact_legal(s[None])[0]
            best, target, sbest, rbest = -1, F(0.0), None, 0
            for a in range(4):
                if not legal[a]:
                    continue
                nb, r = O.move(s[None], np.array([a]))
                q = F(F(int(r[0])) + _V_s(W, rows, thresholds, stride, nb[0]))
                if best < 0 or q > target:
                    best, target, sbest, rbest = a, q, nb[0], int(r[0])
            L = lengths[e]
            released = []  # (board, error)
            if after[e] and h == 1:
                released = [(after[e], F(target - _V_s(W, rows, thresholds, stride, _unpack(after[e]))))]
            elif after[e] and 1 <= L < 1 << 31:
                hd[(L - 1) % h][e] = F(target - _V_s(W, rows, thresholds, stride, _unpack(after[e])))
                ms = range(max(1, L - h + 1), L + 1) if best < 0 else ([L - h + 1] if L >= h else [])
                for m in ms:
                    em = hd[(m - 1) % h][e]
                    k = 1
                    while k < h and m + k <= L:
                        em = F(em + F(c[k] * hd[(m + k - 1) % h][e]))
                        k += 1
                    released.append((ha[(m - 1) % h][e], em))
            for x, err in released:
                f = _fx(err)
                for i in _entries_s(rows, thresholds, stride, _unpack(x)):
                    acc[i] = acc.get(i, 0) + f
                    absacc[i] = absacc.get(i, 0) + abs(f)
                    cnt[i] = cnt.get(i, 0) + 1
            if best < 0:
                c0 = start[e]
                l = c0 + 1 if c0 + 1 < S else 0
                if c0 == 0:
                    b = _unpack(boards[e])
                    me = int(b.max())
                    stats[0] += 1
                    stats[1] += L
                    stats[2] += scores[e]
                    stats[4] += int(me == 15)
                    stats[5] = max(stats[5], L)
                    stats[6] += 1 << me
                    stats[7] += (1 << me) ** 2
                    stats[16 + me] += 1
                else:
                    stats[12] += 1
                    stats[13] += L
                board = 0
                if l >= 1:
                    j = _draw_slot(keys[e], n, mode)
                    board = old_pool[l - 1][j]
                    draws.append((l, j))
                if board:
                    boards[e], start[e] = board, l
                    events["shaped_restarts"] += 1
                else:
                    b, _ = CO.env_init(keys[e][None], mode)
                    boards[e], start[e] = _pack(b[0]), 0
                    events["fallbacks"] += l >= 1
                after[e], scores[e], lengths[e] = 0, 0, 0
            else:
                b, _, _, _ = CO.env_step(s[None].astype(np.uint8), legal[None].astype(np.uint8), np.zeros(1, np.uint8),
                                         [best], keys[e][None], mode)
                boards[e], after[e] = _pack(b[0]), _pack(sbest)
                if h > 1:
                    ha[L % h][e] = after[e]
                scores[e] += rbest
                lengths[e] = L + 1
                ls = _stage(thresholds, b[0])
                if ls > _stage(thresholds, s):
                    recorded[(ls, e)] = boards[e]
        for (l, e), b in recorded.items():  # the commits, after every draw of the step
            pl[l - 1][e] = b
            events["entries"] += 1
        events["same_step"] += sum(1 for l, j in draws if (l, j) in recorded)
        for i in sorted(acc):
            m = float(acc[i]) / (4096.0 * float(cnt[i]))
            if E is None:
                W[i] = F(W[i] + F(F(alpha) * F(m)))
            else:
                beta = min(abs(E[i]) / A[i], 1.0) if A[i] > 0.0 else 1.0
                W[i] = F(W[i] + F(F(alpha) * F(beta * m)))
                E[i] += float(acc[i]) / 4096.0
                A[i] += float(absacc[i]) / 4096.0
    out = dict(T=W, boards=boards, after=after, scores=scores, lengths=lengths, start_stage=start, pool=pl,
               stats=stats, E=E, A=A, events=events)
    if h > 1:
        out.update(hist_after=np.array(ha, np.uint64), hist_delta=np.array(hd, np.float32))
    return out


_EVENTS = {}


@pytest.mark.parametrize("n", [1, 3, 64])
@pytest.mark.parametrize("tc", [False, True])
@pytest.mark.parametrize("h", [1, 3])
@pytest.mark.parametrize("thresholds", [(3,), (3, 5)])
def test_oracle_matches_plain_python(thresholds, h, tc, n):
    mode = (CO.PARTITIONABLE, CO.ORIGINAL)[(h + tc + n) % 2]
    S, stride = len(thresholds) + 1, TINY_WEIGHTS
    n_weights = S * TINY_WEIGHTS
    W0 = _weights(n_weights, 3, 1e-2)
    pl, st = NT.make_placements(TINY), NT.make_stages(thresholds, stride)
    n_steps = {1: 300, 3: 200, 64: 40}[n]
    _, subs = CO.chain(np.array([0, 40 + h + n], np.uint32), mode, n_steps)
    state, ss, pool, ha, hd = carousel_state(n, S, 17 + n + h, mode, W0, h)
    rings = {} if h == 1 else dict(lam=0.5, hist_after=ha.copy(), hist_delta=hd.copy())
    alpha = 0.05
    got_ss, got_pool = ss.copy(), pool.copy()
    if tc:
        rng = np.random.default_rng(1)
        A0 = np.where(rng.random(n_weights) < 0.3, 0.0, rng.uniform(0.0, 5.0, n_weights))
        E0 = A0 * rng.uniform(-1.0, 1.0, n_weights)
        Es, As = E0.copy(), A0.copy()
        got = KO.tc_train(state.copy(), Es, As, got_ss, got_pool, pl, st, alpha, subs, mode, **rings)
        want = _py_train(state, ss, pool, ha, hd, TINY, thresholds, stride, alpha, 0.5, subs, mode, (E0, A0))
        np.testing.assert_array_equal(Es, np.array(want["E"]))
        np.testing.assert_array_equal(As, np.array(want["A"]))
    else:
        got = KO.train(state.copy(), got_ss, got_pool, pl, st, alpha, subs, mode, **rings)
        want = _py_train(state, ss, pool, ha, hd, TINY, thresholds, stride, alpha, 0.5, subs, mode)
    np.testing.assert_array_equal(got.T.view(np.uint32), want["T"].view(np.uint32))
    for k in ("boards", "after", "scores", "lengths"):
        assert [int(x) for x in getattr(got, k)] == want[k], k
    assert [int(x) for x in got_ss] == want["start_stage"]
    assert got_pool.tolist() == want["pool"]
    assert [int(x) for x in got.stats] == want["stats"]
    if h > 1:
        np.testing.assert_array_equal(rings["hist_after"], want["hist_after"])
        np.testing.assert_array_equal(rings["hist_delta"].view(np.uint32), want["hist_delta"].view(np.uint32))
    ev = want["events"]
    assert ev["entries"] > 0 and want["stats"][12] > 0, ev
    if n > 1:  # one env plays one long game from its fresh board
        assert ev["shaped_restarts"] > 0 and want["stats"][0] > 0, ev
    _EVENTS[(thresholds, h, tc, n)] = ev


def test_the_runs_above_draw_empty_slots_and_slots_recorded_in_the_same_step():
    """The runs above include restarts that fall back to init(k) from an empty slot, and draws of a slot whose env
    records a stage entry in the same step (they must read the old board); with few envs that happens often enough to
    be checked."""
    if len(_EVENTS) < 24:
        pytest.skip("needs the whole parametrized test above in this session")
    assert sum(ev["fallbacks"] for ev in _EVENTS.values()) > 0, _EVENTS
    assert sum(ev["same_step"] for (_, _, _, n), ev in _EVENTS.items() if n == 3) > 0, _EVENTS


@pytest.mark.parametrize("h", [1, 3])
@pytest.mark.parametrize("tc", [False, True])
def test_a_threshold_never_reached_equals_the_staged_and_lambda_oracles(tc, h):
    """Threshold 15 (a 2^15 tile) is never reached, so no env records an entry, the pool stays empty and every restart
    takes init(k): W, E, A, the env state, the rings and the statistics equal the entry point without the carousel."""
    mode = CO.PARTITIONABLE if h == 1 else CO.ORIGINAL
    thresholds = (15,)
    nw = 2 * TINY_WEIGHTS
    W0 = _weights(nw, 8, 1e-2)
    pl, st = NT.make_placements(TINY), NT.make_stages(thresholds, TINY_WEIGHTS)
    state, _, _, _, _ = carousel_state(40, 2, 5, mode, W0, h)
    ss, pool = KO.arrays(st, 40)
    _, subs = CO.chain(np.array([0, 23], np.uint32), mode, 40)
    ring = lambda: (np.zeros((h, 40), np.uint64), np.zeros((h, 40), np.float32))  # noqa: E731
    ha1, hd1 = ring()
    ha2, hd2 = ring()
    rings = {} if h == 1 else dict(lam=0.5, hist_after=ha1, hist_delta=hd1)
    E1 = A1 = E2 = A2 = None
    if tc:
        E1, A1, E2, A2 = (np.zeros(nw) for _ in range(4))
        a = KO.tc_train(state.copy(), E1, A1, ss, pool, pl, st, 0.1, subs, mode, **rings)
        b = (SO.tc_train(state.copy(), E2, A2, pl, st, 0.1, subs, mode) if h == 1
             else LO.tc_train(state.copy(), E2, A2, ha2, hd2, pl, st, 0.1, 0.5, subs, mode))
    else:
        a = KO.train(state.copy(), ss, pool, pl, st, 0.1, subs, mode, **rings)
        b = (SO.train(state.copy(), pl, st, 0.1, subs, mode) if h == 1
             else LO.train(state.copy(), ha2, hd2, pl, st, 0.1, 0.5, subs, mode))
    np.testing.assert_array_equal(a.T.view(np.uint32), b.T.view(np.uint32))
    for k in ("boards", "after", "scores", "lengths", "stats"):
        np.testing.assert_array_equal(getattr(a, k), getattr(b, k))
    if tc:
        np.testing.assert_array_equal(E1, E2)
        np.testing.assert_array_equal(A1, A2)
    if h > 1:
        np.testing.assert_array_equal(ha1, ha2)
        np.testing.assert_array_equal(hd1.view(np.uint32), hd2.view(np.uint32))
    assert not pool.any() and not ss.any() and a.stats[0] > 0 and a.stats[12] == 0


# ------------------------------------------------------------------------------------------------ argument checks
def _c_call(fn, tc, n=4, pl=None, stp=0, nw=2 * TINY_WEIGHTS, h=1, ha=8, hd=8, ss=8, pool=8, n_steps=3):
    """One call of a carousel C entry point with fake device pointers, for arguments it must reject before any launch
    (n_steps = 0 runs only the checks)."""
    pl = NT.make_placements(TINY) if pl is None else pl
    sums = (8, 8) if tc else ()
    return fn(8, 8, 8, 8, n, pl.ctypes.data, pl.shape[0], stp, 8, nw, *sums, 0.01, 0.5, h, ha, hd, ss, pool, 8, n_steps,
              1, 8, None, None)


def test_c_entry_points_reject_bad_carousel_arguments():
    from g2048 import _native as N

    st2 = NT.make_stages((3,), TINY_WEIGHTS)
    st1 = NT.make_stages((), 0)
    for fn, tc, who in ((N.lib.g2048_ntuple_carousel_td_train, False, "ntuple_carousel_td_train"),
                        (N.lib.g2048_ntuple_carousel_tc_train, True, "ntuple_carousel_tc_train")):
        ok = st2.ctypes.data
        assert _c_call(fn, tc, stp=None) == -1 and who in N.last_error()
        assert _c_call(fn, tc, stp=st1.ctypes.data) == -1 and "2 stages" in N.last_error()
        assert _c_call(fn, tc, stp=ok, ss=None) == -1 and "pointers" in N.last_error()
        assert _c_call(fn, tc, stp=ok, pool=None) == -1 and "pointers" in N.last_error()
        assert _c_call(fn, tc, stp=ok, ss=6) == -1 and "aligned" in N.last_error()
        assert _c_call(fn, tc, stp=ok, pool=12) == -1 and "aligned" in N.last_error()
        assert _c_call(fn, tc, stp=ok, h=3, ha=None, hd=None) == -1 and "pointers" in N.last_error()
        assert _c_call(fn, tc, stp=ok, h=9) == -1 and "horizon" in N.last_error()
        assert _c_call(fn, tc, stp=ok, h=4, n=(1 << 18) + 1) == -1 and "2^20" in N.last_error()
        # all checks pass: zero steps are a no-op; h = 1 takes NULL rings
        assert _c_call(fn, tc, stp=ok, ha=None, hd=None, n_steps=0) == 0
        assert _c_call(fn, tc, stp=ok, h=3, ss=4, n_steps=0) == 0
        if tc:
            assert fn(8, 8, 8, 8, 4, NT.make_placements(TINY).ctypes.data, 4, ok, 8, 2 * TINY_WEIGHTS, None, 8, 0.01,
                      0.5, 1, None, None, 8, 8, 8, 3, 1, 8, None, None) == -1
    # the existing checks still come first: an invalid network or stages
    bad = NT.make_placements([(2 * TINY_WEIGHTS, (0,))])
    assert _c_call(N.lib.g2048_ntuple_carousel_td_train, False, pl=bad, stp=st2.ctypes.data) == -1
    assert "invalid network" in N.last_error()
    big = NT.make_stages((3,), 4 * TINY_WEIGHTS)
    assert _c_call(N.lib.g2048_ntuple_carousel_td_train, False, stp=big.ctypes.data) == -1
    assert "invalid stages" in N.last_error()


def test_oracle_rejects_what_the_entry_points_reject():
    pl, nw = NT.make_placements(TINY), 2 * TINY_WEIGHTS
    st2 = NT.make_stages((3,), TINY_WEIGHTS)
    for tc in (False, True):
        assert KO.train_rc(pl, nw, None, tc=tc) == -1
        assert KO.train_rc(pl, nw, NT.make_stages((), 0), tc=tc) == -1
        assert KO.train_rc(pl, nw, st2, arrays_given=False, tc=tc) == -1
        assert KO.train_rc(pl, nw, st2, h=3, rings_given=False, tc=tc) == -1
        assert KO.train_rc(pl, nw, st2, h=9, tc=tc) == -1


def test_scratch_size_is_the_lambda_scratch_plus_the_pending_words():
    from g2048 import _native as N

    for n, h, tc in ((1, 1, 0), (777, 3, 1), (1 << 17, 8, 0), (1 << 20, 1, 1)):
        size_of = N.lib.g2048_ntuple_tc_scratch_bytes if tc else N.lib.g2048_ntuple_td_scratch_bytes
        want = int(size_of(n * h, 4, 2 * TINY_WEIGHTS)) + 8 * n
        assert int(N.lib.g2048_ntuple_carousel_scratch_bytes(n, h, 4, 2 * TINY_WEIGHTS, tc)) == want
    for n, h in ((0, 1), (1, 0), (1, 9), ((1 << 19) + 1, 2)):
        assert int(N.lib.g2048_ntuple_carousel_scratch_bytes(n, h, 4, 2 * TINY_WEIGHTS, 0)) == -1


def _host_args(n, h, nw, S=2, tc=False, scratch_bytes=None):
    from g2048 import engine as E

    z = lambda *s, dt=torch.int64: torch.zeros(*s, dtype=dt)  # noqa: E731
    scratch = (E.ntuple_carousel_scratch(n, h, NT.make_placements(TINY), nw, tc, "cpu") if scratch_bytes is None
               else z(scratch_bytes // 8))
    return dict(boards=z(n), after=z(n), scores=z(n, dt=torch.int32), lengths=z(n, dt=torch.int32),
                W=z(nw, dt=torch.float32), ss=z(n, dt=torch.int32), pool=z(S - 1, n), scratch=scratch,
                ha=None if h == 1 else z(h, n), hd=None if h == 1 else z(h, n, dt=torch.float32))


@pytest.mark.parametrize("h", [1, 3])
@pytest.mark.parametrize("tc", [False, True])
def test_engine_wrappers_reject_bad_carousel_arguments(tc, h):
    from g2048 import engine as E

    n, nw = 8, 2 * TINY_WEIGHTS
    pl = NT.make_placements(TINY)
    st2 = NT.make_stages((3,), TINY_WEIGHTS)
    subs = torch.zeros((1, 2), dtype=torch.int32)
    sums = (torch.zeros(nw, dtype=torch.float64), torch.zeros(nw, dtype=torch.float64))

    def run(stages=st2, lam=0.5, **kw):
        a = _host_args(n, h, nw, tc=tc)
        a.update(kw)
        if tc:
            E.ntuple_carousel_tc_train(a["boards"], a["after"], a["scores"], a["lengths"], pl, a["W"], *sums, 0.01, lam,
                                       a["ha"], a["hd"], a["ss"], a["pool"], subs, 1, a["scratch"], stages=stages)
        else:
            E.ntuple_carousel_td_train(a["boards"], a["after"], a["scores"], a["lengths"], pl, a["W"], 0.01, lam,
                                       a["ha"], a["hd"], a["ss"], a["pool"], subs, 1, a["scratch"], stages=stages)

    with pytest.raises(ValueError, match="multi-stage"):
        run(stages=None)
    with pytest.raises(ValueError, match="S >= 2"):
        run(stages=NT.make_stages((), 0))
    with pytest.raises(ValueError, match="stage"):
        run(stages=NT.make_stages((3,), 4 * TINY_WEIGHTS))
    for ss in (torch.zeros(n, dtype=torch.int64), torch.zeros(n + 1, dtype=torch.int32),
               torch.zeros((1, n), dtype=torch.int32), np.zeros(n, np.int32)):
        with pytest.raises(ValueError, match="start_stage"):
            run(ss=ss)
    for pool in (torch.zeros((1, n), dtype=torch.int32), torch.zeros((2, n), dtype=torch.int64),
                 torch.zeros(n, dtype=torch.int64), torch.zeros((1, n + 1), dtype=torch.int64)):
        with pytest.raises(ValueError, match="stage_pool"):
            run(pool=pool)
    with pytest.raises(ValueError, match="contiguous"):
        run(pool=torch.zeros((1, 2 * n), dtype=torch.int64)[:, ::2])
    with pytest.raises(ValueError, match="contiguous"):
        run(ss=torch.zeros(2 * n, dtype=torch.int32)[::2])
    for lam in (float("nan"), -0.5, 1.01):
        with pytest.raises(ValueError, match="lambda"):
            run(lam=lam)
    with pytest.raises(ValueError, match="scratch"):
        run(scratch=_host_args(n, h, nw, tc=tc)["scratch"][:-1])  # without the last pending word
    if h == 1:
        with pytest.raises(ValueError, match="both"):
            run(ha=torch.zeros((2, n), dtype=torch.int64))
    else:
        with pytest.raises(ValueError, match="hist"):
            run(ha=torch.zeros((h, n + 1), dtype=torch.int64))
        with pytest.raises(ValueError, match="int64"):
            run(hd=torch.zeros((h, n), dtype=torch.float64))


@pytest.mark.parametrize("cls_name", ["NTupleTDLearner", "NTupleTCLearner"])
def test_learners_reject_carousel_without_stages_before_touching_a_device(cls_name):
    import g2048

    cls = getattr(g2048, cls_name)
    one = g2048.NTupleNetwork(NT.make_placements(TINY), TINY_WEIGHTS, device="cpu")
    with pytest.raises(ValueError, match="multi-stage"):
        cls(0, 64, network=one, device="meta", carousel=True)
    with pytest.raises(ValueError, match="multi-stage"):
        cls(0, 64, device="meta", carousel=True)  # the default network has one stage
    two = g2048.NTupleNetwork.staged(one, (3,))
    for bad in ("yes", 1, None):
        with pytest.raises(ValueError, match="carousel"):
            cls(0, 64, network=two, device="meta", carousel=bad)
