"""CPU checks of the n-tuple contracts (g2048_ntuple_td_train, g2048_expectimax_values_ntuple): the oracle
(tests/ntuple_oracle.c) against a plain-Python float32 / int64 restatement for small mixed networks, the `lines`
network through the n-tuple oracle against the row-table oracles bit for bit, the symmetry expansion of the 4x6
network, and the placement and argument checks of the C entry points and of NTupleNetwork / NTupleTDLearner, which
run before anything touches a device."""
import math

import numpy as np
import pytest

from oracle import c_oracle as CO
from oracle import pgx2048_oracle as O

import expectimax_oracle as XO
import ntuple_oracle as NO
import td_oracle as TO
from test_expectimax_oracle import random_table

from g2048 import ntuple as NT

F = np.float32

# mixed k = 1..6 with a shared table; tables packed in order
SMALL = [(0, (5,)), (16, (0, 1)), (16, (3, 2)), (272, (4, 8, 12)), (4368, (0, 5, 10, 15)), (69904, (1, 2, 6, 7, 11)),
         (1118480, (9, 10, 13, 14, 15, 12))]
SMALL_WEIGHTS = 1118480 + (1 << 24)
TINY = [(0, (0, 1)), (256, (15,)), (0, (5, 10)), (272, (3, 6, 9))]  # 4368 weights: hot entries at every step
TINY_WEIGHTS = 272 + 4096


def _weights(n, seed, scale=1e-4):
    rng = np.random.default_rng(seed)
    mag = np.exp2(rng.uniform(-20.0, 20.0, n))
    return (mag * rng.choice([-1.0, 1.0], n) * scale).astype(np.float32)


def _unpack(x):
    return ((np.uint64(x) >> (np.arange(16, dtype=np.uint64) * np.uint64(4))) & np.uint64(15)).astype(np.int32)


def _pack(b):
    return int((np.asarray(b, np.uint64) << (np.arange(16, dtype=np.uint64) * np.uint64(4))).sum())


def _entries(rows, b):
    return [off + sum(int(b[c]) << (4 * j) for j, c in enumerate(cells)) for off, cells in rows]


def _V(W, rows, b):
    v = None
    for i in _entries(rows, b):
        v = W[i] if v is None else F(v + W[i])
    return v


def _fx(d):
    c = F(min(max(F(d), F(-(2.0 ** 24))), F(2.0 ** 24)))
    return int(np.rint(F(c * F(4096.0))))


def _py_train(st, rows, alpha, subs, mode):
    """The contract step by step in plain Python with np.float32 scalars and Python ints; the game (init, spawn) is
    the C oracle's, keyed per env."""
    W = st.T.copy()
    boards, after = [int(x) for x in st.boards], [int(x) for x in st.after]
    scores, lengths = [int(x) for x in st.scores], [int(x) for x in st.lengths]
    n = len(boards)
    for sub in np.asarray(subs, np.uint32).reshape(-1, 2):
        keys = CO.split(sub, n, mode)
        acc, cnt = {}, {}
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
            W[i] = F(W[i] + F(F(alpha) * F(np.float64(acc[i]) / (4096.0 * np.float64(cnt[i])))))
    return W, boards, after, scores, lengths


@pytest.mark.parametrize("mode", [CO.PARTITIONABLE, CO.ORIGINAL])
@pytest.mark.parametrize("alpha", [0.0, 0.05, 1.0])
def test_oracle_matches_plain_python(alpha, mode):
    W0 = _weights(TINY_WEIGHTS, 3, 1e-2)
    pl = NT.make_placements(TINY)
    _, subs = CO.chain(np.array([0, 4], np.uint32), mode, 1 + 25)
    st = NO.train(NO.fresh(subs[0], 6, mode, W0), pl, alpha, subs[1:], mode)
    W, boards, after, scores, lengths = _py_train(NO.fresh(subs[0], 6, mode, W0), TINY, alpha, subs[1:], mode)
    np.testing.assert_array_equal(st.T.view(np.uint32), W.view(np.uint32))
    assert [int(x) for x in st.boards] == boards and [int(x) for x in st.after] == after
    assert [int(x) for x in st.scores] == scores and [int(x) for x in st.lengths] == lengths
    if alpha == 0.0:
        np.testing.assert_array_equal(st.T.view(np.uint32), W0.view(np.uint32))
    else:
        assert not np.array_equal(st.T, W0)


def test_value_matches_plain_python_for_every_tuple_size():
    W = _weights(SMALL_WEIGHTS, 5)
    pl = NT.make_placements(SMALL)
    rng = np.random.default_rng(1)
    boards = rng.integers(0, 16, (200, 16))
    got = NO.value(np.array([_pack(b) for b in boards], np.uint64), pl, W)
    want = np.array([_V(W, SMALL, b) for b in boards], np.float32)
    np.testing.assert_array_equal(got.view(np.uint32), want.view(np.uint32))


def _lines_placements():
    rows = [(0, (4 * r, 4 * r + 1, 4 * r + 2, 4 * r + 3)) for r in range(4)]
    return NT.make_placements(rows + [(0, (c, c + 4, c + 8, c + 12)) for c in range(4)])


@pytest.mark.parametrize("mode", [CO.PARTITIONABLE, CO.ORIGINAL])
def test_lines_network_is_the_row_table_learner(mode):
    T = random_table(23) * np.float32(1e-4)
    _, subs = CO.chain(np.array([0, 9], np.uint32), mode, 1 + 120)
    a = TO.train(TO.fresh(subs[0], 200, mode, T), 0.05, subs[1:], mode)
    b = NO.train(NO.fresh(subs[0], 200, mode, T), _lines_placements(), 0.05, subs[1:], mode)
    np.testing.assert_array_equal(a.T.view(np.uint32), b.T.view(np.uint32))
    for k in ("boards", "after", "scores", "lengths", "stats"):
        np.testing.assert_array_equal(getattr(a, k), getattr(b, k))
    assert a.stats[0] > 0


@pytest.mark.parametrize("depth", [1, 2, 3])
def test_lines_network_is_the_row_table_expectimax(depth):
    T = random_table(7)
    rng = np.random.default_rng(depth)
    boards = np.where(rng.random((12, 16)) < 0.5, rng.integers(1, 12, (12, 16)), 0).astype(np.uint8)
    for w in (0.0, 1.0):
        q1, c1 = XO.expectimax(boards, depth, T, w)
        q2, c2 = NO.expectimax(boards, depth, _lines_placements(), T, w)
        np.testing.assert_array_equal(q1.view(np.uint32), q2.view(np.uint32))
        np.testing.assert_array_equal(c1, c2)


def test_four_six_symmetry_expansion():
    pl = NT.make_placements([(j << 24, im) for j, t in enumerate(NT.FOUR_SIX_TUPLES) for im in NT.symmetric_images(t)])
    assert pl.shape[0] == 32 and pl.dtype.itemsize == 12
    assert list(pl["offset"]) == [(p // 8) << 24 for p in range(32)]
    assert all(int(k) == 6 for k in pl["n_cells"]) and not pl["reserved"].any()
    assert NT.check_placements(pl, 1 << 26).shape[0] == 32
    for t in NT.FOUR_SIX_TUPLES:  # every image is a set of 6 distinct cells
        assert all(len(set(im)) == 6 and all(0 <= c < 16 for c in im) for im in NT.symmetric_images(t))
    # an asymmetric tuple has 8 distinct images, the first the tuple itself; (r, c) -> (c, r) is image 4
    ims = NT.symmetric_images((0, 1, 2, 4, 5, 6))
    assert ims[0] == (0, 1, 2, 4, 5, 6) and len({frozenset(i) for i in ims}) == 8
    assert ims[4] == (0, 4, 8, 1, 5, 9) and ims[1] == (3, 2, 1, 7, 6, 5)
    # the lines network
    lines = _lines_placements()
    assert list(lines["offset"]) == [0] * 8 and [list(p["cells"][:4]) for p in lines][4] == [0, 4, 8, 12]


def _set(field, value, j=None):
    def fix(p):
        if j is None:
            p[field][0] = value
        else:
            p[field][0, j] = value
    return fix


BAD_ROWS = [
    ("n_cells 0", _set("n_cells", 0), 1 << 16),
    ("n_cells 7", _set("n_cells", 7), 1 << 28),
    ("cell 16", _set("cells", 16, 1), 1 << 16),
    ("repeated cell", _set("cells", 0, 1), 1 << 16),
    ("reserved", _set("reserved", 1), 1 << 16),
    ("offset past the end", _set("offset", 1), 1 << 16),
    ("n_weights 0", lambda p: None, 0),
    ("n_weights 2^28 + 1", lambda p: None, (1 << 28) + 1),
]


def _bad(i):
    pl = NT.make_placements([(0, (0, 1, 2, 3))])
    _, fix, nw = BAD_ROWS[i]
    fix(pl)
    return pl, nw


@pytest.mark.parametrize("i", range(len(BAD_ROWS)))
def test_bad_networks_are_rejected_everywhere_before_any_launch(i):
    from g2048 import _native as N

    pl, nw = _bad(i)
    q = np.zeros(4, np.float32)
    assert N.lib.g2048_expectimax_values_ntuple(8, 1, 1, pl.ctypes.data, 1, 8, nw, 0.0, q.ctypes.data, None, None) == -1
    assert "network" in N.last_error()
    assert N.lib.g2048_ntuple_td_train(8, 8, 8, 8, 4, pl.ctypes.data, 1, 8, nw, 0.01, 8, 3, 1, 8, None, None) == -1
    assert "network" in N.last_error()
    assert NO.train_rc(4, pl, nw) == -1
    with pytest.raises(ValueError):
        NT.check_placements(pl, nw)
    with pytest.raises(ValueError):
        NT.NTupleNetwork(pl, nw, device="cpu")


def test_placement_count_and_pointer_are_checked():
    from g2048 import _native as N

    one = NT.make_placements([(0, (0,))])
    many = NT.make_placements([(0, (0,))] * 65)
    for pl, count in ((one, 0), (many, 65)):
        assert N.lib.g2048_ntuple_td_train(8, 8, 8, 8, 4, pl.ctypes.data, count, 8, 16, 0.01, 8, 3, 1, 8, None, None) == -1
        assert "network" in N.last_error()
    assert N.lib.g2048_ntuple_td_train(8, 8, 8, 8, 4, None, 1, 8, 16, 0.01, 8, 3, 1, 8, None, None) == -1
    with pytest.raises(ValueError):
        NT.NTupleNetwork(many, 16, device="cpu")
    with pytest.raises(ValueError):
        NT.NTupleNetwork.from_tuples([(0, 1)] * 9, symmetric=True, device="cpu")  # 72 placements
    with pytest.raises(ValueError):
        NT.NTupleNetwork.from_tuples([(0, 1, 2, 3, 4, 5, 6)], device="cpu")


def test_ntuple_td_train_rejects_bad_arguments_before_any_launch():
    from g2048 import _native as N

    pl = NT.make_placements([(0, (0, 1, 2, 3))])

    def rc(n=4, alpha=0.01, n_steps=3, boards=8, after=8, scores=8, lengths=8, W=8, subs=8, scratch=8, stats=None):
        return N.lib.g2048_ntuple_td_train(boards, after, scores, lengths, n, pl.ctypes.data, 1, W, 65536, alpha, subs,
                                           n_steps, 1, scratch, stats, None)

    assert rc(n=0) == -1 and "n must" in N.last_error()
    assert rc(n=(1 << 20) + 1) == -1 and "n must" in N.last_error()
    assert rc(n_steps=-1) == -1 and "n_steps" in N.last_error()
    for alpha in (-0.5, math.nan, math.inf):
        assert rc(alpha=alpha) == -1 and "alpha" in N.last_error()
    assert rc(boards=None) == -1 and "pointers" in N.last_error()
    assert rc(W=None) == -1 and "pointers" in N.last_error()
    assert rc(subs=None) == -1 and "pointers" in N.last_error()
    assert rc(after=12) == -1 and "aligned" in N.last_error()
    assert rc(W=6) == -1 and "aligned" in N.last_error()
    assert rc(n_steps=0, subs=None) == 0  # nothing to do
    f = N.lib.g2048_ntuple_td_scratch_bytes
    assert f(1, 1, 16) >= 16 * 12 + 4 + 8
    assert f(1 << 16, 32, 1 << 26) == ((1 << 26) * 12 + (1 << 21) * 4 + 7) // 8 * 8 + 8
    for args in ((0, 1, 16), (1 << 21, 1, 16), (4, 0, 16), (4, 65, 16), (4, 1, 0), (4, 1, (1 << 28) + 1)):
        assert f(*args) == -1
    for n, alpha, steps in ((0, 0.1, 1), (1 << 21, 0.1, 1), (4, -1.0, 1), (4, math.nan, 1), (4, 0.1, -1)):
        assert NO.train_rc(n, pl, 65536, alpha, steps) == -1


def test_ntuple_td_learner_checks_its_arguments_before_any_launch():
    import g2048

    for kw in (dict(batch_size=0), dict(batch_size=(1 << 20) + 1), dict(alpha=-0.1), dict(alpha=math.nan),
               dict(alpha=1e39), dict(network="four_six")):
        args = dict(init_seed=0, batch_size=8)
        args.update(kw)
        with pytest.raises(ValueError):
            g2048.NTupleTDLearner(**args)
    for w in (np.zeros(100, np.float32), np.full(65536, np.inf, np.float32)):
        with pytest.raises(ValueError):
            NT.NTupleNetwork.lines(weights=w, device="cpu")
    with pytest.raises(ValueError):
        g2048.expectimax_values(np.zeros(1, np.uint64), 1, network="lines")


def test_ntuple_td_train_rejects_a_scratch_made_for_another_batch_or_network():
    import torch

    from g2048 import engine as E
    from g2048 import _native as N

    pl = NT.make_placements([(0, (0, 1, 2, 3))])
    n = 64
    need = int(N.lib.g2048_ntuple_td_scratch_bytes(n, 1, 65536))
    boards, after = torch.zeros(n, dtype=torch.int64), torch.zeros(n, dtype=torch.int64)
    scores, lengths = torch.zeros(n, dtype=torch.int32), torch.zeros(n, dtype=torch.int32)
    W = torch.zeros(65536, dtype=torch.float32)
    subs = torch.zeros((1, 2), dtype=torch.int32)
    for scratch in (torch.zeros(need // 8 - 1, dtype=torch.int64),  # one word short
                    torch.zeros(int(N.lib.g2048_ntuple_td_scratch_bytes(n, 1, 4096)) // 8, dtype=torch.int64)):
        with pytest.raises(ValueError, match="scratch"):
            E.ntuple_td_train(boards, after, scores, lengths, pl, W, 0.01, subs, 1, scratch)
