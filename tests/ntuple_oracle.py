"""ctypes binding of tests/ntuple_oracle.c: n-tuple networks (V, expectimax over V, TD(0) learning of the weights)
restated with the row-table oracles' game, move and fixed point, and the games of the expectimax player over a
network.  TEST INFRASTRUCTURE ONLY.

The library is compiled on first use into a temporary directory (the tree may be read-only where the tests run)."""
from __future__ import annotations

import ctypes as C
import subprocess
import tempfile
from pathlib import Path

import numpy as np

from oracle import c_oracle as CO

import td_oracle as TO

_SRC = Path(__file__).resolve().parent / "ntuple_oracle.c"
_LIB = None
_P = C.c_void_p


def _lib():
    global _LIB
    if _LIB is None:
        out = Path(tempfile.mkdtemp(prefix="g2048_ntuple_oracle_")) / "libntuple_oracle.so"
        subprocess.run(["gcc", "-O2", "-fopenmp", "-fPIC", "-shared", "-ffp-contract=off", "-fno-fast-math", "-Wall",
                        "-o", str(out), str(_SRC), "-lm"], check=True, capture_output=True)
        _LIB = C.CDLL(str(out))
        _LIB.orc_ntuple_value.restype = C.c_int
        _LIB.orc_ntuple_value.argtypes = [_P, C.c_int64, _P, C.c_int, _P, C.c_int64, _P]
        _LIB.orc_ntuple_expectimax.restype = C.c_int
        _LIB.orc_ntuple_expectimax.argtypes = [_P, C.c_int64, C.c_int, _P, C.c_int, _P, C.c_int64, C.c_float, _P, _P]
        _LIB.orc_ntuple_td_train.restype = C.c_int
        _LIB.orc_ntuple_td_train.argtypes = [_P, _P, _P, _P, C.c_int64, _P, C.c_int, _P, C.c_int64, C.c_float, _P,
                                             C.c_int64, C.c_int, _P]
    return _LIB


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def _pl(placements):
    pl = np.ascontiguousarray(placements)
    assert pl.dtype.itemsize == 12
    return pl


def value(packed_boards, placements, W) -> np.ndarray:
    """V of (n,) packed boards (float32)."""
    b = np.ascontiguousarray(packed_boards, np.uint64)
    W = np.ascontiguousarray(W, np.float32)
    pl = _pl(placements)
    out = np.zeros(b.shape[0], np.float32)
    rc = _lib().orc_ntuple_value(_p(b), b.shape[0], _p(pl), pl.shape[0], _p(W), W.shape[0], _p(out))
    if rc != 0:
        raise ValueError("orc_ntuple_value rejected the network")
    return out


def expectimax(boards, depth, placements, W, w=0.0):
    """orc_ntuple_expectimax on (n,16) exponent boards: (q (n,4) float32 with NaN where illegal, counters (2,) uint64)."""
    boards = np.ascontiguousarray(boards, np.uint8).reshape(-1, 16)
    W = np.ascontiguousarray(W, np.float32)
    pl = _pl(placements)
    n = boards.shape[0]
    q = np.zeros((n, 4), np.float32)
    counters = np.zeros(2, np.uint64)
    rc = _lib().orc_ntuple_expectimax(_p(boards), n, int(depth), _p(pl), pl.shape[0], _p(W), W.shape[0],
                                      float(np.float32(w)), _p(q), _p(counters))
    if rc != 0:
        raise ValueError("orc_ntuple_expectimax rejected its arguments")
    return q, counters


def fresh(key, n, mode, W):
    """Envs initialised with split(key, n)[e] and no afterstate; the weights travel in the state's ``T`` slot."""
    return TO.fresh(key, n, mode, W)


def train(state: TO.State, placements, alpha, subs, mode) -> TO.State:
    """orc_ntuple_td_train on the state (its ``T`` holds W), in place (returns it)."""
    subs = np.ascontiguousarray(subs, np.uint32).reshape(-1, 2)
    pl = _pl(placements)
    rc = _lib().orc_ntuple_td_train(_p(state.boards), _p(state.after), _p(state.scores), _p(state.lengths),
                                    state.boards.shape[0], _p(pl), pl.shape[0], _p(state.T), state.T.shape[0],
                                    float(np.float32(alpha)), _p(subs), subs.shape[0], int(mode), _p(state.stats))
    if rc != 0:
        raise ValueError("orc_ntuple_td_train rejected its arguments")
    return state


def train_rc(n, placements, n_weights, alpha=0.01, n_steps=1) -> int:
    """orc_ntuple_td_train's return code on a one-env state (the weight array is only allocated when it is valid)."""
    pl = _pl(placements)
    st = TO.State(np.zeros(1), np.zeros(1), np.zeros(1), np.zeros(1), np.zeros(1))
    subs = np.zeros((1, 2), np.uint32)
    return int(_lib().orc_ntuple_td_train(_p(st.boards), _p(st.after), _p(st.scores), _p(st.lengths), int(n), _p(pl),
                                          pl.shape[0], None, int(n_weights), float(alpha), _p(subs), int(n_steps), 0,
                                          None))


def expectimax_games(seed, batch, depth, placements, W, w, mode):
    """BatchRunner(seed, ExpectimaxPolicy(depth, network=(placements, W), reward_weight=w)).run_eval_batch(batch)
    restated as expectimax_oracle.expectimax_games restates the row-table player.  Returns dict(final_boards (n,16) u8,
    lengths, scores)."""
    import expectimax_oracle as XO

    key = np.array([(int(seed) >> 32) & 0xFFFFFFFF, int(seed) & 0xFFFFFFFF], np.uint32)
    n_sub = 1 + 2 * 1024
    _, subs = CO.chain(key, mode, n_sub)
    boards, masks = CO.env_init(CO.split(subs[0], batch, mode), mode)
    done = np.zeros(batch, np.uint8)
    lengths = np.zeros(batch, np.int64)
    scores = np.zeros(batch, np.int64)
    t = 0
    while not done.all():
        if 2 + 2 * t >= subs.shape[0]:
            n_sub = 2 * n_sub + 1
            _, subs = CO.chain(key, mode, n_sub)
        live = np.flatnonzero(done == 0)
        q, _ = expectimax(boards[live], depth, placements, W, w)
        actions = np.zeros(batch, np.int32)
        actions[live] = XO.best_actions(q)
        alive = done == 0
        keys = CO.split(subs[2 + 2 * t], batch, mode)
        boards, masks, done, rewards = CO.env_step(boards, masks, done, actions, keys, mode)
        lengths += alive
        scores += rewards.astype(np.int64)
        t += 1
    return dict(final_boards=boards, lengths=lengths, scores=scores)
