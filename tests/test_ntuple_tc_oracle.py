"""CPU checks of the n-tuple temporal coherence contract (g2048_ntuple_tc_train): the oracle (tests/ntuple_tc_oracle.c)
against a plain-Python float32 / float64 / int64 restatement, its first step from E = A = 0 against the TD oracle, the
edges of the step scale beta, and the argument checks of the C entry point, the engine wrapper and NTupleTCLearner,
which run before anything touches a device."""
import math

import numpy as np
import pytest

from oracle import c_oracle as CO
from oracle import pgx2048_oracle as O

import ntuple_oracle as NO
import ntuple_tc_oracle as TCO
from test_ntuple_oracle import SMALL, SMALL_WEIGHTS, TINY, TINY_WEIGHTS, _entries, _fx, _pack, _unpack, _V, _weights

from g2048 import ntuple as NT

F = np.float32


def _py_tc_train(st, E, A, rows, alpha, subs, mode):
    """The TC contract step by step in plain Python: np.float32 scalars for V and W, Python floats (IEEE double) for
    E, A and beta, Python ints for the fixed-point sums; the game (init, spawn) is the C oracle's, keyed per env."""
    W, E, A = st.T.copy(), [float(x) for x in E], [float(x) for x in A]
    boards, after = [int(x) for x in st.boards], [int(x) for x in st.after]
    scores, lengths = [int(x) for x in st.scores], [int(x) for x in st.lengths]
    n = len(boards)
    for sub in np.asarray(subs, np.uint32).reshape(-1, 2):
        keys = CO.split(sub, n, mode)
        acc, absacc, cnt = {}, {}, {}
        for e in range(n):
            s = _unpack(boards[e])
            legal = O.exact_legal(s[None])[0]
            best, target, sbest, rbest = -1, F(0.0), None, 0
            for a in range(4):
                if not legal[a]:
                    continue
                nb, r = O.move(s[None], np.array([a]))
                q = F(F(int(r[0])) + _V(W, rows, nb[0]))
                if best < 0 or q > target:
                    best, target, sbest, rbest = a, q, nb[0], int(r[0])
            if after[e]:
                d = _fx(F(target - _V(W, rows, _unpack(after[e]))))
                for i in _entries(rows, _unpack(after[e])):
                    acc[i] = acc.get(i, 0) + d
                    absacc[i] = absacc.get(i, 0) + abs(d)
                    cnt[i] = cnt.get(i, 0) + 1
            k = keys[e]
            if best < 0:
                b, _ = CO.env_init(k[None], mode)
                boards[e], after[e], scores[e], lengths[e] = _pack(b[0]), 0, 0, 0
            else:
                b, _, _, _ = CO.env_step(s[None].astype(np.uint8), legal[None].astype(np.uint8), np.zeros(1, np.uint8),
                                         [best], k[None], mode)
                boards[e], after[e] = _pack(b[0]), _pack(sbest)
                scores[e] += rbest
                lengths[e] += 1
        for i in sorted(acc):
            m = float(acc[i]) / (4096.0 * float(cnt[i]))
            beta = min(abs(E[i]) / A[i], 1.0) if A[i] > 0.0 else 1.0
            W[i] = F(W[i] + F(F(alpha) * F(beta * m)))
            E[i] = E[i] + float(acc[i]) / 4096.0
            A[i] = A[i] + float(absacc[i]) / 4096.0
    return W, np.array(E), np.array(A), boards, after, scores, lengths


def _sums(n, seed):
    """E and A with |E| <= A, zero for about a third of the entries, so beta takes every branch."""
    rng = np.random.default_rng(seed)
    A = np.where(rng.random(n) < 0.3, 0.0, np.exp2(rng.uniform(-10.0, 20.0, n)))
    return A * rng.uniform(-1.0, 1.0, n), A


@pytest.mark.parametrize("mode", [CO.PARTITIONABLE, CO.ORIGINAL])
@pytest.mark.parametrize("alpha", [0.0, 0.05, 1.0])
@pytest.mark.parametrize("start", ["zero", "random"])
def test_tc_oracle_matches_plain_python(alpha, mode, start):
    W0 = _weights(TINY_WEIGHTS, 3, 1e-2)
    E0, A0 = (np.zeros(TINY_WEIGHTS), np.zeros(TINY_WEIGHTS)) if start == "zero" else _sums(TINY_WEIGHTS, 4)
    pl = NT.make_placements(TINY)
    _, subs = CO.chain(np.array([0, 4], np.uint32), mode, 1 + 20)
    E, A = E0.copy(), A0.copy()
    st = TCO.tc_train(NO.fresh(subs[0], 6, mode, W0), E, A, pl, alpha, subs[1:], mode)
    W, E_py, A_py, boards, after, scores, lengths = _py_tc_train(NO.fresh(subs[0], 6, mode, W0), E0, A0, TINY, alpha,
                                                                 subs[1:], mode)
    np.testing.assert_array_equal(st.T.view(np.uint32), W.view(np.uint32))
    np.testing.assert_array_equal(E.view(np.uint64), E_py.view(np.uint64))
    np.testing.assert_array_equal(A.view(np.uint64), A_py.view(np.uint64))
    assert [int(x) for x in st.boards] == boards and [int(x) for x in st.after] == after
    assert [int(x) for x in st.scores] == scores and [int(x) for x in st.lengths] == lengths
    assert not np.array_equal(A, A0)  # the sums move whatever alpha is
    if alpha == 0.0:
        np.testing.assert_array_equal(st.T.view(np.uint32), W0.view(np.uint32))
    else:
        assert not np.array_equal(st.T, W0)


def _after_some_td_steps(mode, n=8, steps=30, seed=6):
    """A state whose envs hold afterstates (TD steps from random weights), and the next sub keys."""
    _, subs = CO.chain(np.array([0, seed], np.uint32), mode, 1 + steps + 3)
    st = NO.train(NO.fresh(subs[0], n, mode, _weights(SMALL_WEIGHTS, 9)), NT.make_placements(SMALL), 0.02,
                  subs[1:1 + steps], mode)
    return st, subs[1 + steps:]


def _same_state(a, b):
    np.testing.assert_array_equal(a.T.view(np.uint32), b.T.view(np.uint32))
    for k in ("boards", "after", "scores", "lengths", "stats"):
        np.testing.assert_array_equal(getattr(a, k), getattr(b, k))


@pytest.mark.parametrize("mode", [CO.PARTITIONABLE, CO.ORIGINAL])
def test_first_tc_step_from_zero_sums_is_a_td_step(mode):
    st, subs = _after_some_td_steps(mode)
    assert (st.after != 0).any()
    pl = NT.make_placements(SMALL)
    td = NO.train(st.copy(), pl, 0.05, subs[:1], mode)
    E, A = np.zeros(SMALL_WEIGHTS), np.zeros(SMALL_WEIGHTS)
    tc = TCO.tc_train(st.copy(), E, A, pl, 0.05, subs[:1], mode)
    _same_state(tc, td)
    assert (A > 0).any() and bool((np.abs(E) <= A).all())
    # a second step from the sums of the first is not a TD step any more (some entries' errors disagree in sign)
    td2 = NO.train(td, pl, 0.05, subs[1:3], mode)
    tc2 = TCO.tc_train(tc, E, A, pl, 0.05, subs[1:3], mode)
    assert not np.array_equal(tc2.T, td2.T)


@pytest.mark.parametrize("case", ["A zero", "clamped", "E zero"])
def test_beta_edges(case):
    """beta = 1 where A = 0 whatever E holds, beta = 1 where rounding lets |E| exceed A (the fmin), and beta = 0 where
    E = 0 < A: the first two make the step a TD step, the last leaves W where it was.  E and A move in every case."""
    mode = CO.PARTITIONABLE
    st, subs = _after_some_td_steps(mode)
    pl = NT.make_placements(SMALL)
    rng = np.random.default_rng(2)
    if case == "A zero":
        E, A = rng.uniform(-5.0, 5.0, SMALL_WEIGHTS), np.zeros(SMALL_WEIGHTS)
    elif case == "clamped":
        A = np.exp2(rng.uniform(-4.0, 30.0, SMALL_WEIGHTS))
        E = -np.nextafter(A, np.inf)  # |E| / A > 1 by an ulp
        assert (np.abs(E) / A > 1.0).all()
    else:
        E, A = np.zeros(SMALL_WEIGHTS), np.exp2(rng.uniform(-4.0, 30.0, SMALL_WEIGHTS))
    E0, A0 = E.copy(), A.copy()
    tc = TCO.tc_train(st.copy(), E, A, pl, 0.05, subs[:1], mode)
    if case == "E zero":
        want = st.copy()
        NO.train(want, pl, 0.0, subs[:1], mode)
    else:
        want = NO.train(st.copy(), pl, 0.05, subs[:1], mode)
    _same_state(tc, want)
    assert not np.array_equal(st.T, NO.train(st.copy(), pl, 0.05, subs[:1], mode).T)  # the TD step moves W
    assert not np.array_equal(A, A0) and not np.array_equal(E, E0)


def test_ntuple_tc_train_rejects_bad_arguments_before_any_launch():
    from g2048 import _native as N

    pl = NT.make_placements([(0, (0, 1, 2, 3))])

    def rc(n=4, alpha=0.01, n_steps=3, boards=8, after=8, scores=8, lengths=8, W=8, Es=8, As=8, subs=8, scratch=8,
           stats=None, placements=pl.ctypes.data, n_pl=1, n_weights=65536):
        return N.lib.g2048_ntuple_tc_train(boards, after, scores, lengths, n, placements, n_pl, W, n_weights, Es, As,
                                           alpha, subs, n_steps, 1, scratch, stats, None)

    assert rc(n=0) == -1 and "n must" in N.last_error()
    assert rc(n=(1 << 20) + 1) == -1 and "n must" in N.last_error()
    assert rc(n_steps=-1) == -1 and "n_steps" in N.last_error()
    for alpha in (-0.5, math.nan, math.inf):
        assert rc(alpha=alpha) == -1 and "alpha" in N.last_error()
    assert rc(placements=None) == -1 and "network" in N.last_error()
    assert rc(n_pl=65) == -1 and "network" in N.last_error()
    assert rc(n_weights=4096) == -1 and "network" in N.last_error()
    assert "ntuple_tc_train" in N.last_error()
    for kw in (dict(boards=None), dict(W=None), dict(subs=None), dict(scratch=None), dict(Es=None), dict(As=None)):
        assert rc(**kw) == -1 and "pointers" in N.last_error()
    assert rc(after=12) == -1 and "aligned" in N.last_error()
    assert rc(W=6) == -1 and "aligned" in N.last_error()
    for kw in (dict(Es=12), dict(As=4)):
        assert rc(**kw) == -1 and "d_err_sum and d_abs_err_sum must be 8-byte aligned" in N.last_error()
    assert rc(n_steps=0, subs=None) == 0  # nothing to do
    f = N.lib.g2048_ntuple_tc_scratch_bytes
    assert f(1, 1, 16) >= 16 * 20 + 4 + 8
    assert f(1 << 16, 32, 1 << 26) == ((1 << 26) * 20 + (1 << 21) * 4 + 7) // 8 * 8 + 8
    assert f(1 << 16, 32, 1 << 26) - N.lib.g2048_ntuple_td_scratch_bytes(1 << 16, 32, 1 << 26) == 8 << 26
    for args in ((0, 1, 16), (1 << 21, 1, 16), (4, 0, 16), (4, 65, 16), (4, 1, 0), (4, 1, (1 << 28) + 1)):
        assert f(*args) == -1
    for n, alpha, steps in ((0, 0.1, 1), (1 << 21, 0.1, 1), (4, -1.0, 1), (4, math.nan, 1), (4, 0.1, -1)):
        assert TCO.tc_train_rc(n, pl, 65536, alpha, steps) == -1
    assert TCO.tc_train_rc(4, pl, 4096) == -1  # the network's table does not fit
    assert TCO.tc_train_rc(4, pl, 65536, sums=False) == -1


def test_ntuple_tc_train_wrapper_rejects_a_td_scratch_and_bad_sums():
    import torch

    from g2048 import engine as E
    from g2048 import _native as N

    pl = NT.make_placements([(0, (0, 1, 2, 3))])
    n = 64
    boards, after = torch.zeros(n, dtype=torch.int64), torch.zeros(n, dtype=torch.int64)
    scores, lengths = torch.zeros(n, dtype=torch.int32), torch.zeros(n, dtype=torch.int32)
    W = torch.zeros(65536, dtype=torch.float32)
    Es, As = torch.zeros(65536, dtype=torch.float64), torch.zeros(65536, dtype=torch.float64)
    subs = torch.zeros((1, 2), dtype=torch.int32)
    need = int(N.lib.g2048_ntuple_tc_scratch_bytes(n, 1, 65536))
    for scratch in (torch.zeros(need // 8 - 1, dtype=torch.int64),  # one word short
                    torch.zeros(int(N.lib.g2048_ntuple_td_scratch_bytes(n, 1, 65536)) // 8, dtype=torch.int64)):
        with pytest.raises(ValueError, match="scratch"):
            E.ntuple_tc_train(boards, after, scores, lengths, pl, W, Es, As, 0.01, subs, 1, scratch)
    scratch = torch.zeros(need // 8, dtype=torch.int64)
    for bad in (torch.zeros(65536, dtype=torch.float32), torch.zeros(65535, dtype=torch.float64),
                torch.zeros((65536, 2), dtype=torch.float64)[:, 0]):
        for es, as_ in ((bad, As), (Es, bad)):
            with pytest.raises(AssertionError):
                E.ntuple_tc_train(boards, after, scores, lengths, pl, W, es, as_, 0.01, subs, 1, scratch)
    with pytest.raises(ValueError, match="invalid sizes"):
        E.ntuple_tc_scratch(0, pl, 65536, "cpu")


def test_ntuple_tc_learner_checks_its_arguments_before_any_launch():
    import g2048

    assert g2048.NTupleTCLearner.__mro__[1] is g2048.NTupleTDLearner
    for kw in (dict(batch_size=0), dict(batch_size=(1 << 20) + 1), dict(alpha=-0.1), dict(alpha=math.nan),
               dict(alpha=1e39), dict(network="four_six")):
        args = dict(init_seed=0, batch_size=8)
        args.update(kw)
        with pytest.raises(ValueError):
            g2048.NTupleTCLearner(**args)
