"""CPU checks of the expectimax contract (g2048_expectimax_values): orc_expectimax (tests/expectimax_oracle.c, built on
the C oracle) against a plain-Python recursion over the numpy oracle's move function, closed forms, the tree sizes, the
default row table, and the entry point's argument checks, which run before anything touches a device."""
import numpy as np
import pytest

from oracle import c_oracle as CO
from oracle import pgx2048_oracle as O

import expectimax_oracle as XO

F = np.float32


def _default_table():
    from g2048.expectimax import default_row_table_numpy

    return default_row_table_numpy()


def random_table(seed):
    """float32 values of mixed sign spanning 2^-20 .. 2^20: any deviation from the contract's summation order changes
    bits."""
    rng = np.random.default_rng(seed)
    mag = np.exp2(rng.uniform(-20.0, 20.0, 65536))
    return (mag * rng.choice([-1.0, 1.0], 65536) * rng.uniform(1.0, 2.0, 65536)).astype(np.float32)


def _boards(seed, depths, mode=CO.PARTITIONABLE):
    """Boards of real games: env.init and `depth` random-policy steps (the C oracle), one board per depth."""
    keys = CO.split(np.array([0, seed], np.uint32), 2 * len(depths) + 1, mode)
    boards, masks = CO.env_init(keys[:len(depths)], mode)
    done = np.zeros(len(depths), np.uint8)
    for t in range(max(depths)):
        step = CO.split(keys[len(depths) + t % len(depths)], 2 * len(depths), mode)
        acts, _ = CO.act(step[:len(depths)], masks, CO.RANDOM, mode)
        nb, nm, nd, _ = CO.env_step(boards, masks, done, acts, step[len(depths):], mode)
        live = np.array([t < d for d in depths])
        boards[live], masks[live], done[live] = nb[live], nm[live], nd[live]
    return boards


ONE_LEGAL = [0, 1, 2, 3, 0, 2, 3, 1, 0, 1, 2, 3, 0, 2, 3, 1]
TERMINAL = [1, 2, 1, 2, 2, 1, 2, 1, 1, 2, 1, 2, 2, 1, 2, 1]


def _test_boards():
    game = _boards(21, [0, 2, 5, 9, 14, 20, 27, 35, 44, 54, 65, 77, 90, 104, 119, 135, 152, 170])
    return np.concatenate([game, np.array([ONE_LEGAL, TERMINAL], np.uint8)])  # 20 boards


class _PyTree:
    """The contract as a plain recursion with np.float32 scalars, over the numpy oracle's move."""

    def __init__(self, table, w):
        self.T, self.w = table, F(w)
        self.leaves = self.chance = 0

    def H(self, b):
        h = None
        for line in range(8):
            cells = [4 * line + j for j in range(4)] if line < 4 else [4 * j + line - 4 for j in range(4)]
            idx = sum(int(b[c]) << (4 * j) for j, c in enumerate(cells))
            h = self.T[idx] if h is None else F(h + self.T[idx])
        return h

    def Q(self, b, a, k):
        nb, r = O.move(b[None], [a])
        nb = nb[0]
        if k == 1:
            self.leaves += 1
            tail = self.H(nb)
        else:
            tail = self.C(nb, k - 1)
        return F(F(self.w * F(r[0])) + tail)

    def C(self, s, k):
        self.chance += 1
        acc, ne = F(0.0), 0
        for cell in range(16):
            if s[cell]:
                continue
            ne += 1
            ch = s.copy()
            ch[cell] = 1
            v2 = self.V(ch, k)
            ch[cell] = 2
            v4 = self.V(ch, k)
            acc = F(acc + F(F(F(0.9) * v2) + F(F(0.1) * v4)))
        return F(acc / F(ne))

    def V(self, b, k):
        legal = O.exact_legal(b[None])[0]
        v, any_ = F(0.0), False
        for a in range(4):
            if legal[a]:
                q = self.Q(b, a, k)
                if not any_ or q > v:
                    v = q
                any_ = True
        return v

    def q(self, boards, depth):
        out = np.full((boards.shape[0], 4), np.nan, np.float32)
        legal = O.exact_legal(boards)
        for i, b in enumerate(boards.astype(np.int32)):
            for a in range(4):
                if legal[i, a]:
                    out[i, a] = self.Q(b, a, depth)
        return out


def _bits(x):
    return np.asarray(x, np.float32).view(np.uint32)


@pytest.mark.parametrize("depth", [1, 2])
@pytest.mark.parametrize("table,w", [("default", 0.0), ("random", 0.5), ("random", 1.0)])
def test_orc_expectimax_matches_python_recursion(depth, table, w):
    boards = _test_boards()
    T = _default_table() if table == "default" else random_table(3)
    got, counters = XO.expectimax(boards, depth, T, w)
    py = _PyTree(T, w)
    want = py.q(boards, depth)
    np.testing.assert_array_equal(_bits(got), _bits(want))
    assert counters.tolist() == [py.leaves, py.chance]
    legal = O.exact_legal(boards)
    assert np.array_equal(~np.isnan(got), legal)
    assert np.isnan(got[-1]).all() and (~np.isnan(got[-2])).sum() == 1  # terminal, Left only


def test_closed_forms_depth_one():
    boards = _test_boards()
    legal = O.exact_legal(boards)
    # zero table, w = 1: the merge reward itself
    q, _ = XO.expectimax(boards, 1, np.zeros(65536, np.float32), 1.0)
    for a in range(4):
        _, r = O.move(boards, np.full(boards.shape[0], a))
        np.testing.assert_array_equal(q[legal[:, a], a], r[legal[:, a]].astype(np.float32))
    # constant table 1.5, w = 0: eight lines
    q, counters = XO.expectimax(boards, 1, np.full(65536, 1.5, np.float32), 0.0)
    assert (q[legal] == 12.0).all() and np.isnan(q[~legal]).all()
    assert counters.tolist() == [int(legal.sum()), 0]


def test_counters_accumulate_and_count_the_tree():
    boards = _test_boards()[:6]
    T = random_table(5)
    _, c1 = XO.expectimax(boards, 2, T, 0.0)
    # depth 2: one chance node per legal (board, a0), one leaf per legal action of every child of it
    legal = O.exact_legal(boards)
    leaves = chance = 0
    for i, b in enumerate(boards.astype(np.int32)):
        for a in np.flatnonzero(legal[i]):
            s = O.move(b[None], [a])[0][0]
            chance += 1
            for cell in np.flatnonzero(s == 0):
                for v in (1, 2):
                    ch = s.copy()
                    ch[cell] = v
                    leaves += int(O.exact_legal(ch[None]).sum())
    assert c1.tolist() == [leaves, chance]


def test_default_row_values_spot_values():
    T = _default_table()
    assert T.dtype == np.float32 and T.shape == (65536,)
    assert T[0x0000] == 201080.0  # four empty cells
    assert T[0x0001] == 200799.0  # [1,0,0,0]: 3 empty, sum 1, mono_left 1, mono_right 0
    assert T[0x1111] == 202756.0  # one run of four: merges 4, sum 4
    # [1,2,3,4]: no empty cell, no merge, mono_left 0 (min), sum = 1 + 2^3.5 + 3^3.5 + 4^3.5
    assert T[0x4321] == np.float32(200000.0 - 11.0 * (1.0 + 2.0 ** 3.5 + 3.0 ** 3.5 + 4.0 ** 3.5))
    # [2,2,0,2]: one empty, a run of three over the gap (merges 3), sum 3 * 2^3.5, mono_left = mono_right = 16
    assert T[0x2022] == np.float32(200000.0 + 270.0 + 2100.0 - 47.0 * 16.0 - 11.0 * 3 * 2.0 ** 3.5)
    # [3,1,3,1]: mono_left (81-1) + (81-1) = 160, mono_right 80; min 80
    assert T[0x1313] == np.float32(200000.0 - 47.0 * 80.0 - 11.0 * (2 * 3.0 ** 3.5 + 2.0))


def test_expectimax_values_rejects_bad_arguments_before_any_launch():
    from g2048 import _native as N

    def rc(n=4, depth=2, boards=None, table=None, q=None):
        return N.lib.g2048_expectimax_values(boards, n, depth, table, 0.0, q, None, None)

    assert rc() == -1 and "pointers" in N.last_error()  # valid sizes: only the NULL pointers are wrong
    assert rc(depth=0) == -1 and "depth" in N.last_error()
    assert rc(depth=5) == -1 and "depth" in N.last_error()
    assert rc(n=-1) == -1 and "n must" in N.last_error()
    assert rc(boards=8, table=8, q=10) == -1 and "aligned" in N.last_error()
    assert rc(n=0) == 0  # nothing to do
