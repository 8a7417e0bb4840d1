"""CPU checks of the delayed TD(lambda) / TC(lambda) contracts (g2048_ntuple_lambda_td_train,
g2048_ntuple_lambda_tc_train): the lambda oracle (tests/ntuple_lambda_oracle.c) against a plain-Python restatement of
the window, the oracle with h = 1 against the TD, TC and staged oracles, the rounding rule of the coefficients c_k, and
the argument checks of the C entry points, the engine wrappers and the learners, which run before anything touches a
device."""
import numpy as np
import pytest
import torch

from oracle import c_oracle as CO
from oracle import pgx2048_oracle as O

import ntuple_lambda_oracle as LO
import ntuple_oracle as NO
import ntuple_stages_oracle as SO
import ntuple_tc_oracle as TCO
from test_ntuple_oracle import TINY, TINY_WEIGHTS, _fx, _pack, _unpack, _weights
from test_ntuple_stages_oracle import _entries_s, _V_s

from g2048 import ntuple as NT

F = np.float32
LAMBDAS = (0.0, 0.5, 1.0)


def windowed_state(n, h, seed, mode, W):
    """Envs in every position of their window: lengths L over 0 .. h + 2 (L = 0 has no afterstate), rings of random
    afterstates and errors with after = x_L, and every third env on a board without a legal move, so that its episode
    ends on the first step with L below, at and above h.  The other envs play on from their fresh boards.  Returns
    (state, hist_after, hist_delta)."""
    rng = np.random.default_rng(seed)
    _, subs = CO.chain(np.array([1, seed], np.uint32), mode, 2)
    st = NO.fresh(subs[1], n, mode, W)
    shifts = np.arange(16, dtype=np.uint64) * np.uint64(4)
    hist_after = (rng.integers(0, 7, (h, n, 16)).astype(np.uint64) << shifts).sum(axis=2, dtype=np.uint64)
    hist_delta = rng.normal(0.0, 40.0, (h, n)).astype(np.float32)
    L = np.arange(n) % (h + 3)
    st.lengths[:] = L
    st.scores[:] = 4 * L
    st.after[:] = np.where(L > 0, hist_after[(L - 1) % h, np.arange(n)], np.uint64(0))
    parity = np.array([(r + c) % 2 for r in range(4) for c in range(4)])
    terminal = (1 + parity + 2 * rng.integers(0, 3, (n, 16))).astype(np.uint64)  # neighbours differ in parity
    st.boards[::3] = (terminal << shifts).sum(axis=1, dtype=np.uint64)[::3]
    return st, np.ascontiguousarray(hist_after), hist_delta


def _py_train(st, hist_after, hist_delta, rows, thresholds, stride, alpha, lam, subs, mode, sums=None):
    """The contract step by step in plain Python: np.float32 scalars for V, W, the errors and c_k, Python floats for E,
    A and beta, Python ints for the fixed-point sums; the game is the C oracle's."""
    W = st.T.copy()
    E, A = (None, None) if sums is None else ([float(x) for x in sums[0]], [float(x) for x in sums[1]])
    h = hist_after.shape[0]
    ha = [[int(x) for x in row] for row in hist_after]
    hd = [[F(x) for x in row] for row in hist_delta]
    c, d = [], 1.0
    for _ in range(h):
        c.append(F(d))
        d *= float(F(lam))
    boards, after, lengths = [int(x) for x in st.boards], [int(x) for x in st.after], [int(x) for x in st.lengths]
    n = len(boards)
    for sub in np.asarray(subs, np.uint32).reshape(-1, 2):
        keys = CO.split(sub, n, mode)
        acc, absacc, cnt = {}, {}, {}
        for e in range(n):
            s = _unpack(boards[e])
            legal = O.exact_legal(s[None])[0]
            best, target, sbest = -1, F(0.0), None
            for a in range(4):
                if not legal[a]:
                    continue
                nb, r = O.move(s[None], np.array([a]))
                q = F(F(int(r[0])) + _V_s(W, rows, thresholds, stride, nb[0]))
                if best < 0 or q > target:
                    best, target, sbest = a, q, nb[0]
            L = lengths[e]
            if after[e] and 1 <= L < 1 << 31:
                hd[(L - 1) % h][e] = F(target - _V_s(W, rows, thresholds, stride, _unpack(after[e])))
                if best < 0:
                    released = range(max(1, L - h + 1), L + 1)
                else:
                    released = [L - h + 1] if L >= h else []
                for m in released:
                    em = hd[(m - 1) % h][e]
                    k = 1
                    while k < h and m + k <= L:
                        em = F(em + F(c[k] * hd[(m + k - 1) % h][e]))
                        k += 1
                    f = _fx(em)
                    for i in _entries_s(rows, thresholds, stride, _unpack(ha[(m - 1) % h][e])):
                        acc[i] = acc.get(i, 0) + f
                        absacc[i] = absacc.get(i, 0) + abs(f)
                        cnt[i] = cnt.get(i, 0) + 1
            if best < 0:
                b, _ = CO.env_init(keys[e][None], mode)
                boards[e], after[e], lengths[e] = _pack(b[0]), 0, 0
            else:
                b, _, _, _ = CO.env_step(s[None].astype(np.uint8), legal[None].astype(np.uint8), np.zeros(1, np.uint8),
                                         [best], keys[e][None], mode)
                boards[e], after[e] = _pack(b[0]), _pack(sbest)
                ha[L % h][e] = after[e]
                lengths[e] = L + 1
        for i in sorted(acc):
            m = float(acc[i]) / (4096.0 * float(cnt[i]))
            if E is None:
                W[i] = F(W[i] + F(F(alpha) * F(m)))
            else:
                beta = min(abs(E[i]) / A[i], 1.0) if A[i] > 0.0 else 1.0
                W[i] = F(W[i] + F(F(alpha) * F(beta * m)))
                E[i] += float(acc[i]) / 4096.0
                A[i] += float(absacc[i]) / 4096.0
    return dict(T=W, boards=boards, after=after, lengths=lengths, hist_after=np.array(ha, np.uint64),
                hist_delta=np.array(hd, np.float32), E=E, A=A)


def _random_sums(n, seed):
    rng = np.random.default_rng(seed)
    A = np.where(rng.random(n) < 0.3, 0.0, rng.uniform(0.0, 5.0, n))
    return A * rng.uniform(-1.0, 1.0, n), A


@pytest.mark.parametrize("staged", [False, True])
@pytest.mark.parametrize("tc", [False, True])
@pytest.mark.parametrize("h", [2, 3])
@pytest.mark.parametrize("lam", LAMBDAS)
def test_oracle_matches_plain_python(lam, h, tc, staged):
    mode = CO.PARTITIONABLE if h == 2 else CO.ORIGINAL
    thresholds, stride = ((2, 4), TINY_WEIGHTS) if staged else ((), 0)
    n_weights = (len(thresholds) + 1) * TINY_WEIGHTS
    W0 = _weights(n_weights, 3, 1e-2)
    pl, st = NT.make_placements(TINY), NT.make_stages(thresholds, stride) if staged else None
    _, subs = CO.chain(np.array([0, 4 + h], np.uint32), mode, 25)
    alpha = 0.05
    state, ha, hd = windowed_state(9, h, 11 + h, mode, W0)
    ha0, hd0 = ha.copy(), hd.copy()
    if tc:
        E0, A0 = _random_sums(n_weights, 1)
        Es, As = E0.copy(), A0.copy()
        got = LO.tc_train(state.copy(), Es, As, ha, hd, pl, st, alpha, lam, subs, mode)
        want = _py_train(state, ha0, hd0, TINY, thresholds, stride, alpha, lam, subs, mode, (E0, A0))
        np.testing.assert_array_equal(Es, np.array(want["E"]))
        np.testing.assert_array_equal(As, np.array(want["A"]))
    else:
        got = LO.train(state.copy(), ha, hd, pl, st, alpha, lam, subs, mode)
        want = _py_train(state, ha0, hd0, TINY, thresholds, stride, alpha, lam, subs, mode)
    np.testing.assert_array_equal(got.T.view(np.uint32), want["T"].view(np.uint32))
    for k in ("boards", "after", "lengths"):
        assert [int(x) for x in getattr(got, k)] == want[k], k
    np.testing.assert_array_equal(ha, want["hist_after"])
    np.testing.assert_array_equal(hd.view(np.uint32), want["hist_delta"].view(np.uint32))
    assert not np.array_equal(got.T, W0)
    assert got.stats[0] >= 3  # the terminal envs ended their episodes


@pytest.mark.parametrize("tc", [False, True])
def test_an_afterstate_with_length_zero_stores_and_releases_nothing(tc):
    """Outside the contract (after != 0 with L = 0): the env's ring slots keep their values and nothing is released;
    the env still moves, and its next afterstate is x_1."""
    mode, h = CO.PARTITIONABLE, 3
    W0 = _weights(TINY_WEIGHTS, 4, 1e-2)
    pl = NT.make_placements(TINY)
    state, ha, hd = windowed_state(6, h, 9, mode, W0)
    state.lengths[1] = 0  # env 1 keeps its afterstate
    state.boards[1] = state.boards[2]  # and a board with a legal move
    _, subs = CO.chain(np.array([0, 9], np.uint32), mode, 1)
    ha0, hd0 = ha.copy(), hd.copy()
    sums = _random_sums(TINY_WEIGHTS, 3) if tc else None
    E, A = (sums[0].copy(), sums[1].copy()) if tc else (None, None)
    got = (LO.tc_train(state.copy(), E, A, ha, hd, pl, None, 0.05, 0.5, subs, mode) if tc
           else LO.train(state.copy(), ha, hd, pl, None, 0.05, 0.5, subs, mode))
    want = _py_train(state, ha0, hd0, TINY, (), 0, 0.05, 0.5, subs, mode, sums)
    np.testing.assert_array_equal(got.T.view(np.uint32), want["T"].view(np.uint32))
    np.testing.assert_array_equal(hd.view(np.uint32), want["hist_delta"].view(np.uint32))
    np.testing.assert_array_equal(hd[:, 1].view(np.uint32), hd0[:, 1].view(np.uint32))
    assert int(got.lengths[1]) == 1 and int(ha[0, 1]) == int(got.after[1]) != 0


@pytest.mark.parametrize("lam", [0.0, 0.3, 0.5, 1.0])
def test_horizon_one_equals_the_existing_oracles(lam):
    mode = CO.PARTITIONABLE
    pl = NT.make_placements(TINY)
    st2 = NT.make_stages((3,), TINY_WEIGHTS)
    _, subs = CO.chain(np.array([0, 21], np.uint32), mode, 30)
    for staged in (False, True):
        nw = (2 if staged else 1) * TINY_WEIGHTS
        W0 = _weights(nw, 8, 1e-2)
        state, ha, hd = windowed_state(10, 1, 5, mode, W0)
        a = LO.train(state.copy(), ha.copy(), hd.copy(), pl, st2 if staged else None, 0.1, lam, subs, mode)
        b = (SO.train(state.copy(), pl, st2, 0.1, subs, mode) if staged else NO.train(state.copy(), pl, 0.1, subs, mode))
        E0, A0 = _random_sums(nw, 2)
        E1, A1, E2, A2 = E0.copy(), A0.copy(), E0.copy(), A0.copy()
        c = LO.tc_train(state.copy(), E1, A1, ha.copy(), hd.copy(), pl, st2 if staged else None, 0.1, lam, subs, mode)
        d = (SO.tc_train(state.copy(), E2, A2, pl, st2, 0.1, subs, mode) if staged
             else TCO.tc_train(state.copy(), E2, A2, pl, 0.1, subs, mode))
        for x, y in ((a, b), (c, d)):
            np.testing.assert_array_equal(x.T.view(np.uint32), y.T.view(np.uint32))
            for k in ("boards", "after", "scores", "lengths", "stats"):
                np.testing.assert_array_equal(getattr(x, k), getattr(y, k))
        np.testing.assert_array_equal(E1, E2)
        np.testing.assert_array_equal(A1, A2)


@pytest.mark.parametrize("lam", [0.0, 0.1, 0.25, 1.0 / 3.0, 0.5, 0.7, 0.9, 0.99, 1.0])
def test_coefficients_are_rounded_products_in_double(lam):
    lam32 = float(np.float32(lam))
    for h in range(1, 9):
        d, want = 1.0, np.zeros(8, np.float32)
        for k in range(h):
            want[k] = np.float32(d)
            d *= lam32
        np.testing.assert_array_equal(LO.coefficients(lam, h).view(np.uint32), want.view(np.uint32))
    c = LO.coefficients(lam, 8)
    assert c[0] == 1.0 and all(c[k + 1] <= c[k] for k in range(7))


def test_coefficients_are_not_float_products():
    """Repeated multiplication in float32 would round at every step; the rule rounds once, from double."""
    lam = np.float32(0.3)  # the two rules differ from k = 5 on
    f, d = np.float32(1.0), 1.0
    for _ in range(5):
        f, d = np.float32(f * lam), d * float(lam)
    c = LO.coefficients(lam, 8)
    assert c[5] == np.float32(d) and c[5] != f


# ------------------------------------------------------------------------------------------------ argument checks
BAD_WINDOWS = [  # (lam, horizon, n): rejected for any valid network
    (float("nan"), 2, 4), (float("inf"), 2, 4), (-0.25, 2, 4), (1.5, 2, 4), (-1e-30, 2, 4),
    (0.5, 0, 4), (0.5, 9, 4), (0.5, -1, 4),
    (0.5, 2, (1 << 19) + 1), (0.5, 8, (1 << 17) + 1),
]


@pytest.mark.parametrize("i", range(len(BAD_WINDOWS)))
def test_bad_windows_are_rejected_before_any_launch(i):
    from g2048 import _native as N

    lam, h, n = BAD_WINDOWS[i]
    pl = NT.make_placements(TINY)
    for staged in (False, True):
        st = NT.make_stages((3,), TINY_WEIGHTS) if staged else None
        stp = st.ctypes.data if staged else None
        nw = 2 * TINY_WEIGHTS
        assert N.lib.g2048_ntuple_lambda_td_train(8, 8, 8, 8, n, pl.ctypes.data, 4, stp, 8, nw, 0.01, lam, h, 8, 8, 8,
                                                  3, 1, 8, None, None) == -1
        assert "ntuple_lambda_td_train" in N.last_error()
        assert N.lib.g2048_ntuple_lambda_tc_train(8, 8, 8, 8, n, pl.ctypes.data, 4, stp, 8, nw, 8, 8, 0.01, lam, h, 8,
                                                  8, 8, 3, 1, 8, None, None) == -1
        assert "ntuple_lambda_tc_train" in N.last_error()
        if n <= 8:
            assert LO.train_rc(pl, nw, lam, h, n, st) == -1 and LO.train_rc(pl, nw, lam, h, n, st, tc=True) == -1


def test_hist_pointers_are_checked_before_any_launch():
    from g2048 import _native as N

    pl = NT.make_placements(TINY)
    for fn, tc in ((N.lib.g2048_ntuple_lambda_td_train, False), (N.lib.g2048_ntuple_lambda_tc_train, True)):
        def call(ha, hd, n_steps=3, lam=0.5, h=3):
            sums = (8, 8) if tc else ()
            return fn(8, 8, 8, 8, 4, pl.ctypes.data, 4, None, 8, TINY_WEIGHTS, *sums, 0.01, lam, h, ha, hd, 8, n_steps,
                      1, 8, None, None)
        assert call(None, 8) == -1 and "pointers" in N.last_error()
        assert call(8, None) == -1 and "pointers" in N.last_error()
        assert call(12, 8) == -1 and "aligned" in N.last_error()
        assert call(8, 6) == -1 and "aligned" in N.last_error()
        assert call(8, 4, n_steps=0) == 0  # all checks pass: zero steps are a no-op
        assert call(8, 4, n_steps=0, lam=1.0, h=8) == 0
        assert call(8, 4, n_steps=0, lam=0.0, h=1) == 0
    assert LO.train_rc(pl, TINY_WEIGHTS, 0.5, 2, rings_given=False) == -1
    # the existing checks still come first: an invalid network or stages
    bad = NT.make_placements([(TINY_WEIGHTS, (0,))])
    assert N.lib.g2048_ntuple_lambda_td_train(8, 8, 8, 8, 4, bad.ctypes.data, 1, None, 8, TINY_WEIGHTS, 0.01, 0.5, 2,
                                              8, 8, 8, 3, 1, 8, None, None) == -1
    assert "invalid network" in N.last_error()
    st = NT.make_stages((3,), TINY_WEIGHTS)
    assert N.lib.g2048_ntuple_lambda_td_train(8, 8, 8, 8, 4, pl.ctypes.data, 4, st.ctypes.data, 8, TINY_WEIGHTS, 0.01,
                                              0.5, 2, 8, 8, 8, 3, 1, 8, None, None) == -1
    assert "invalid stages" in N.last_error()


def _host_args(n, h, nw, scratch_n=None, tc=False):
    from g2048 import _native as N

    boards, after = torch.zeros(n, dtype=torch.int64), torch.zeros(n, dtype=torch.int64)
    scores, lengths = torch.zeros(n, dtype=torch.int32), torch.zeros(n, dtype=torch.int32)
    W = torch.zeros(nw, dtype=torch.float32)
    size_of = N.lib.g2048_ntuple_tc_scratch_bytes if tc else N.lib.g2048_ntuple_td_scratch_bytes
    size = int(size_of(n * h if scratch_n is None else scratch_n, 4, nw))
    scratch = torch.zeros(size // 8, dtype=torch.int64)
    return boards, after, scores, lengths, W, scratch


@pytest.mark.parametrize("tc", [False, True])
def test_engine_wrappers_reject_bad_windows(tc):
    from g2048 import engine as E

    n, h, nw = 8, 3, TINY_WEIGHTS
    pl = NT.make_placements(TINY)
    boards, after, scores, lengths, W, scratch = _host_args(n, h, nw, tc=tc)
    subs = torch.zeros((1, 2), dtype=torch.int32)
    Es, As = torch.zeros(nw, dtype=torch.float64), torch.zeros(nw, dtype=torch.float64)

    def run(lam=0.5, ha=None, hd=None, scr=scratch):
        ha = torch.zeros((h, n), dtype=torch.int64) if ha is None else ha
        hd = torch.zeros((h, n), dtype=torch.float32) if hd is None else hd
        if tc:
            E.ntuple_lambda_tc_train(boards, after, scores, lengths, pl, W, Es, As, 0.01, lam, ha, hd, subs, 1, scr)
        else:
            E.ntuple_lambda_td_train(boards, after, scores, lengths, pl, W, 0.01, lam, ha, hd, subs, 1, scr)

    for lam in (float("nan"), float("inf"), -0.5, 1.01):
        with pytest.raises(ValueError, match="lambda"):
            run(lam=lam)
    for ha, hd in ((torch.zeros((h, n + 1), dtype=torch.int64), None), (None, torch.zeros((h + 1, n))),
                   (torch.zeros((0, n), dtype=torch.int64), torch.zeros((0, n))),
                   (torch.zeros((9, n), dtype=torch.int64), torch.zeros((9, n))),
                   (torch.zeros(h * n, dtype=torch.int64), None)):
        with pytest.raises(ValueError, match="hist"):
            run(ha=ha, hd=hd)
    for ha, hd in ((torch.zeros((h, n), dtype=torch.float64), None), (None, torch.zeros((h, n), dtype=torch.float64)),
                   (torch.zeros((h, n), dtype=torch.int32), None)):
        with pytest.raises(ValueError, match="int64"):
            run(ha=ha, hd=hd)
    with pytest.raises(ValueError, match="contiguous"):
        run(ha=torch.zeros((n, h), dtype=torch.int64).t())
    with pytest.raises(ValueError, match="scratch"):
        run(scr=_host_args(n, h, nw, scratch_n=n, tc=tc)[5])  # sized for n, not n * h
    big = (1 << 18) + 1
    bb, ba, bs, bl, _, _ = _host_args(big, 1, nw, scratch_n=1, tc=tc)
    with pytest.raises(ValueError, match="2\\^20"):
        fn = E.ntuple_lambda_tc_train if tc else E.ntuple_lambda_td_train
        sums = (Es, As) if tc else ()
        fn(bb, ba, bs, bl, pl, W, *sums, 0.01, 0.5, torch.zeros((4, big), dtype=torch.int64),
           torch.zeros((4, big), dtype=torch.float32), subs, 1, scratch)


@pytest.mark.parametrize("cls_name", ["NTupleTDLearner", "NTupleTCLearner"])
def test_learners_reject_bad_windows_before_touching_a_device(cls_name):
    import g2048

    cls = getattr(g2048, cls_name)
    for kw in ({"lam": float("nan")}, {"lam": -0.1}, {"lam": 2.0}, {"horizon": 0}, {"horizon": 9}, {"horizon": 2.5},
               {"horizon": None}, {"horizon": "2"}, {"horizon": float("nan")},
               {"horizon": 2, "batch_size": (1 << 19) + 1}, {"horizon": 8, "batch_size": (1 << 17) + 1}):
        kw = dict(kw)
        batch = kw.pop("batch_size", 64)
        with pytest.raises(ValueError, match="lam|horizon"):
            cls(0, batch, device="meta", **kw)
    assert NT.MAX_HORIZON == 8
