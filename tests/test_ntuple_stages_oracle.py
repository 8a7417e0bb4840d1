"""CPU checks of the multi-stage n-tuple contracts (g2048_ntuple_staged_td_train, g2048_ntuple_staged_tc_train,
g2048_expectimax_values_ntuple_staged): the staged oracle (tests/ntuple_stages_oracle.c) against a plain-Python
restatement of stage, the entry, V_S and the learning step, the staged oracle with one stage against the unstaged
oracles, NTupleNetwork.staged, and the stage checks of the C entry points, the engine wrappers and NTupleNetwork,
which run before anything touches a device."""
import numpy as np
import pytest
import torch

from oracle import c_oracle as CO
from oracle import pgx2048_oracle as O

import ntuple_oracle as NO
import ntuple_stages_oracle as SO
import ntuple_tc_oracle as TCO
from test_ntuple_oracle import TINY, TINY_WEIGHTS, _fx, _pack, _unpack, _weights

from g2048 import ntuple as NT

F = np.float32


def _stage(thresholds, b):
    return sum(1 for t in thresholds if max(int(x) for x in b) >= t)


def _entries_s(rows, thresholds, stride, b):
    base = _stage(thresholds, b) * stride
    return [base + off + sum(int(b[c]) << (4 * j) for j, c in enumerate(cells)) for off, cells in rows]


def _V_s(W, rows, thresholds, stride, b):
    v = None
    for i in _entries_s(rows, thresholds, stride, b):
        v = W[i] if v is None else F(v + W[i])
    return v


def _py_train(st, rows, thresholds, stride, alpha, subs, mode, sums=None):
    """The staged TD (sums None) or TC (sums = (E, A)) contract step by step in plain Python: np.float32 scalars for V
    and W, Python floats for E, A and beta, Python ints for the fixed-point sums; the game is the C oracle's."""
    W = st.T.copy()
    E, A = (None, None) if sums is None else ([float(x) for x in sums[0]], [float(x) for x in sums[1]])
    boards, after = [int(x) for x in st.boards], [int(x) for x in st.after]
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
            if after[e]:
                ab = _unpack(after[e])
                d = _fx(F(target - _V_s(W, rows, thresholds, stride, ab)))
                for i in _entries_s(rows, thresholds, stride, ab):
                    acc[i] = acc.get(i, 0) + d
                    absacc[i] = absacc.get(i, 0) + abs(d)
                    cnt[i] = cnt.get(i, 0) + 1
            if best < 0:
                b, _ = CO.env_init(keys[e][None], mode)
                boards[e], after[e] = _pack(b[0]), 0
            else:
                b, _, _, _ = CO.env_step(s[None].astype(np.uint8), legal[None].astype(np.uint8), np.zeros(1, np.uint8),
                                         [best], keys[e][None], mode)
                boards[e], after[e] = _pack(b[0]), _pack(sbest)
        for i in sorted(acc):
            m = float(acc[i]) / (4096.0 * float(cnt[i]))
            if E is None:
                W[i] = F(W[i] + F(F(alpha) * F(m)))
            else:
                beta = min(abs(E[i]) / A[i], 1.0) if A[i] > 0.0 else 1.0
                W[i] = F(W[i] + F(F(alpha) * F(beta * m)))
                E[i] += float(acc[i]) / 4096.0
                A[i] += float(absacc[i]) / 4096.0
    return W, boards, after, E, A


def _boards_of_every_stage(n, seed):
    """Random boards whose largest exponent runs over 0..15."""
    rng = np.random.default_rng(seed)
    out = []
    for i in range(n):
        me = i % 16
        b = rng.integers(0, me + 1, 16)
        b[rng.integers(0, 16)] = me
        out.append(b)
    return np.array(out)


@pytest.mark.parametrize("thresholds,stride", [((3,), TINY_WEIGHTS), ((3, 7, 11), TINY_WEIGHTS), ((1, 15), 1),
                                               ((2, 4, 6, 8, 10, 12, 14), 300)])
def test_value_matches_plain_python(thresholds, stride):
    n_weights = len(thresholds) * stride + TINY_WEIGHTS
    W = _weights(n_weights, 5)
    boards = _boards_of_every_stage(320, 1)
    got = SO.value(np.array([_pack(b) for b in boards], np.uint64), NT.make_placements(TINY),
                   NT.make_stages(thresholds, stride), W)
    want = np.array([_V_s(W, TINY, thresholds, stride, b) for b in boards], np.float32)
    np.testing.assert_array_equal(got.view(np.uint32), want.view(np.uint32))
    assert {_stage(thresholds, b) for b in boards} == set(range(len(thresholds) + 1))


def test_the_empty_board_is_in_stage_zero():
    W = _weights(3 * TINY_WEIGHTS, 2)
    got = SO.value(np.zeros(1, np.uint64), NT.make_placements(TINY), NT.make_stages((1, 2), TINY_WEIGHTS), W)
    want = NO.value(np.zeros(1, np.uint64), NT.make_placements(TINY), W[:TINY_WEIGHTS])
    np.testing.assert_array_equal(got.view(np.uint32), want.view(np.uint32))


@pytest.mark.parametrize("mode", [CO.PARTITIONABLE, CO.ORIGINAL])
@pytest.mark.parametrize("tc", [False, True])
def test_oracle_learning_matches_plain_python(tc, mode):
    """Low thresholds, so the envs cross them within the run and errors cross stage borders."""
    thresholds, stride = (2, 4), TINY_WEIGHTS
    W0 = _weights(3 * TINY_WEIGHTS, 3, 1e-2)
    pl, st = NT.make_placements(TINY), NT.make_stages(thresholds, stride)
    _, subs = CO.chain(np.array([0, 4], np.uint32), mode, 1 + 30)
    alpha = 0.05
    if tc:
        rng = np.random.default_rng(1)
        A0 = np.where(rng.random(W0.shape[0]) < 0.3, 0.0, rng.uniform(0.0, 5.0, W0.shape[0]))
        E0 = A0 * rng.uniform(-1.0, 1.0, W0.shape[0])
        E, A = E0.copy(), A0.copy()
        got = SO.tc_train(NO.fresh(subs[0], 6, mode, W0), E, A, pl, st, alpha, subs[1:], mode)
        W, boards, after, E_py, A_py = _py_train(NO.fresh(subs[0], 6, mode, W0), TINY, thresholds, stride, alpha,
                                                 subs[1:], mode, (E0, A0))
        np.testing.assert_array_equal(E, np.array(E_py))
        np.testing.assert_array_equal(A, np.array(A_py))
    else:
        got = SO.train(NO.fresh(subs[0], 6, mode, W0), pl, st, alpha, subs[1:], mode)
        W, boards, after, _, _ = _py_train(NO.fresh(subs[0], 6, mode, W0), TINY, thresholds, stride, alpha, subs[1:],
                                           mode)
    np.testing.assert_array_equal(got.T.view(np.uint32), W.view(np.uint32))
    assert [int(x) for x in got.boards] == boards and [int(x) for x in got.after] == after
    assert not np.array_equal(got.T[2 * stride:], W0[2 * stride:])  # the last stage learned


def test_one_stage_equals_the_unstaged_oracles():
    mode = CO.PARTITIONABLE
    W0 = _weights(TINY_WEIGHTS, 7, 1e-2)
    pl, st = NT.make_placements(TINY), NT.make_stages((), 0)
    boards = _boards_of_every_stage(64, 3)
    packed = np.array([_pack(b) for b in boards], np.uint64)
    np.testing.assert_array_equal(SO.value(packed, pl, st, W0).view(np.uint32), NO.value(packed, pl, W0).view(np.uint32))
    live = boards[:12] % 8
    for depth in (1, 2):
        q1, c1 = SO.expectimax(live, depth, pl, st, W0, 0.5)
        q2, c2 = NO.expectimax(live, depth, pl, W0, 0.5)
        np.testing.assert_array_equal(q1.view(np.uint32), q2.view(np.uint32))
        np.testing.assert_array_equal(c1, c2)
    _, subs = CO.chain(np.array([0, 9], np.uint32), mode, 1 + 40)
    a = SO.train(NO.fresh(subs[0], 5, mode, W0), pl, st, 0.1, subs[1:], mode)
    b = NO.train(NO.fresh(subs[0], 5, mode, W0), pl, 0.1, subs[1:], mode)
    E1, A1, E2, A2 = (np.zeros(TINY_WEIGHTS) for _ in range(4))
    c = SO.tc_train(NO.fresh(subs[0], 5, mode, W0), E1, A1, pl, st, 0.1, subs[1:], mode)
    d = TCO.tc_train(NO.fresh(subs[0], 5, mode, W0), E2, A2, pl, 0.1, subs[1:], mode)
    for x, y in ((a, b), (c, d)):
        np.testing.assert_array_equal(x.T.view(np.uint32), y.T.view(np.uint32))
        for k in ("boards", "after", "scores", "lengths", "stats"):
            np.testing.assert_array_equal(getattr(x, k), getattr(y, k))
    np.testing.assert_array_equal(E1, E2)
    np.testing.assert_array_equal(A1, A2)


def test_staged_network_starts_with_the_values_of_its_base():
    base = NT.NTupleNetwork(NT.make_placements(TINY), TINY_WEIGHTS, _weights(TINY_WEIGHTS, 11), device="cpu")
    net = NT.NTupleNetwork.staged(base, (3, 9))
    assert net.n_stages == 3 and net.stage_thresholds == (3, 9) and net.stage_stride == TINY_WEIGHTS
    assert net.n_weights == 3 * TINY_WEIGHTS and np.array_equal(net.placements, base.placements)
    assert base.n_stages == 1 and base.stage_thresholds == () and base.stage_stride == 0 and base.stages is None
    assert net.stages.dtype == NT.STAGES_DTYPE and net.stages.itemsize == 20
    boards = _boards_of_every_stage(160, 4)
    packed = np.array([_pack(b) for b in boards], np.uint64)
    got = SO.value(packed, net.placements, net.stages, net.weights.numpy())
    want = NO.value(packed, base.placements, base.weights.numpy())
    np.testing.assert_array_equal(got.view(np.uint32), want.view(np.uint32))
    q1, _ = SO.expectimax(boards[:8] % 10, 2, net.placements, net.stages, net.weights.numpy(), 1.0)
    q2, _ = NO.expectimax(boards[:8] % 10, 2, base.placements, base.weights.numpy(), 1.0)
    np.testing.assert_array_equal(q1.view(np.uint32), q2.view(np.uint32))
    assert NT.NTupleNetwork.staged(base, ()).n_weights == TINY_WEIGHTS
    with pytest.raises(ValueError):
        NT.NTupleNetwork.staged(net, (12,))  # already staged
    with pytest.raises(ValueError):
        NT.NTupleNetwork.staged(NT.NTupleNetwork.four_six(device="cpu"), (10, 11, 12, 13))  # 5 * 2^26 > 2^28


def _raw_stages(n_thresholds, thresholds, stride):
    st = np.zeros(1, NT.STAGES_DTYPE)
    st[0]["stride"] = stride
    st[0]["n_thresholds"] = n_thresholds
    st[0]["thresholds"][: len(thresholds)] = thresholds
    return st


# for TINY over 2 * TINY_WEIGHTS weights
BAD_STAGES = [
    _raw_stages(16, list(range(1, 16)), 1),                 # 17 stages
    _raw_stages(2, [5, 5], 1),                              # not strictly increasing
    _raw_stages(2, [6, 4], 1),
    _raw_stages(1, [0], 1),                                 # threshold 0
    _raw_stages(1, [16], 1),                                # threshold 16
    _raw_stages(1, [3, 7], TINY_WEIGHTS),                   # an unused byte set
    _raw_stages(0, [], 5),                                  # one stage with a stride
    _raw_stages(1, [3], 0),                                 # two stages without one
    _raw_stages(2, [3, 7], TINY_WEIGHTS),                   # the last stage's tables do not fit
    _raw_stages(1, [3], TINY_WEIGHTS + 1),
]


@pytest.mark.parametrize("i", range(len(BAD_STAGES)))
def test_bad_stages_are_rejected_everywhere_before_any_launch(i):
    from g2048 import _native as N
    from g2048 import engine as E

    st, pl, nw = BAD_STAGES[i], NT.make_placements(TINY), 2 * TINY_WEIGHTS
    q = np.zeros(4, np.float32)
    assert N.lib.g2048_expectimax_values_ntuple_staged(8, 1, 1, pl.ctypes.data, pl.shape[0], st.ctypes.data, 8, nw,
                                                       0.0, q.ctypes.data, None, None) == -1
    assert "stages" in N.last_error()
    assert N.lib.g2048_ntuple_staged_td_train(8, 8, 8, 8, 4, pl.ctypes.data, pl.shape[0], st.ctypes.data, 8, nw, 0.01,
                                              8, 3, 1, 8, None, None) == -1
    assert "ntuple_staged_td_train: invalid stages" in N.last_error()
    assert N.lib.g2048_ntuple_staged_tc_train(8, 8, 8, 8, 4, pl.ctypes.data, pl.shape[0], st.ctypes.data, 8, nw, 8, 8,
                                              0.01, 8, 3, 1, 8, None, None) == -1
    assert "ntuple_staged_tc_train: invalid stages" in N.last_error()
    assert SO.value_rc(pl, st, nw) == -1
    assert SO.train_rc(pl, st, nw) == -1 and SO.train_rc(pl, st, nw, tc=True) == -1
    with pytest.raises(ValueError):
        NT.check_stages(st, pl, nw)
    n = 8
    boards, after = torch.zeros(n, dtype=torch.int64), torch.zeros(n, dtype=torch.int64)
    scores, lengths = torch.zeros(n, dtype=torch.int32), torch.zeros(n, dtype=torch.int32)
    W = torch.zeros(nw, dtype=torch.float32)
    Es, As = torch.zeros(nw, dtype=torch.float64), torch.zeros(nw, dtype=torch.float64)
    subs = torch.zeros((1, 2), dtype=torch.int32)
    scratch = torch.zeros(int(N.lib.g2048_ntuple_tc_scratch_bytes(n, pl.shape[0], nw)) // 8, dtype=torch.int64)
    with pytest.raises(ValueError, match="stage"):
        E.ntuple_td_train(boards, after, scores, lengths, pl, W, 0.01, subs, 1, scratch, stages=st)
    with pytest.raises(ValueError, match="stage"):
        E.ntuple_tc_train(boards, after, scores, lengths, pl, W, Es, As, 0.01, subs, 1, scratch, stages=st)
    with pytest.raises(ValueError, match="stage"):
        E.expectimax_values_ntuple(boards, 1, pl, W, 0.0, stages=st)
    if st[0]["n_thresholds"] <= 15:
        k = int(st[0]["n_thresholds"])
        thresholds = [int(t) for t in st[0]["thresholds"][:k]]
        if not any(st[0]["thresholds"][k:]):
            with pytest.raises(ValueError):
                NT.NTupleNetwork(pl, nw, device="cpu", stage_thresholds=thresholds, stage_stride=int(st[0]["stride"]))


def test_null_stages_and_too_many_thresholds_are_rejected():
    from g2048 import _native as N

    pl = NT.make_placements(TINY)
    assert N.lib.g2048_ntuple_staged_td_train(8, 8, 8, 8, 4, pl.ctypes.data, 4, None, 8, TINY_WEIGHTS, 0.01, 8, 3, 1,
                                              8, None, None) == -1
    assert "invalid stages" in N.last_error()
    q = np.zeros(4, np.float32)
    assert N.lib.g2048_expectimax_values_ntuple_staged(8, 1, 1, pl.ctypes.data, 4, None, 8, TINY_WEIGHTS, 0.0,
                                                       q.ctypes.data, None, None) == -1
    with pytest.raises(ValueError):
        NT.make_stages(range(1, 17), 1)
    with pytest.raises(ValueError):
        NT.NTupleNetwork(pl, 17 * TINY_WEIGHTS, device="cpu", stage_thresholds=range(1, 17), stage_stride=TINY_WEIGHTS)


def test_good_stages_pass_every_check():
    from g2048 import _native as N

    pl = NT.make_placements(TINY)
    for thresholds, stride, nw in (((3,), TINY_WEIGHTS, 2 * TINY_WEIGHTS), ((1, 15), 1, TINY_WEIGHTS + 2),
                                   (tuple(range(1, 16)), TINY_WEIGHTS, 16 * TINY_WEIGHTS), ((), 0, TINY_WEIGHTS)):
        st = NT.make_stages(thresholds, stride)
        NT.check_stages(st, pl, nw)
        assert SO.value_rc(pl, st, nw) == 0
        # the staged entry point passes the stage checks and stops at the misaligned pointer that follows them
        assert N.lib.g2048_ntuple_staged_td_train(8, 12, 8, 8, 4, pl.ctypes.data, 4, st.ctypes.data, 8, nw, 0.01, 8, 3,
                                                  1, 8, None, None) == -1
        assert "aligned" in N.last_error()
        net = NT.NTupleNetwork(pl, nw, device="cpu", stage_thresholds=thresholds, stage_stride=stride)
        assert net.n_stages == len(thresholds) + 1
