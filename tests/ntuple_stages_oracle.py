"""ctypes binding of tests/ntuple_stages_oracle.c: multi-stage n-tuple networks (V_S, expectimax over V_S, TD(0) and TC
learning of the weights) restated on the CPU, and the games of the expectimax player over such a network.
TEST INFRASTRUCTURE ONLY.

``stages`` is a (1,) ``g2048.ntuple.STAGES_DTYPE`` record (``g2048.ntuple.make_stages``).  The library is compiled on
first use into a temporary directory (the tree may be read-only where the tests run)."""
from __future__ import annotations

import ctypes as C
import subprocess
import tempfile
from pathlib import Path

import numpy as np

from oracle import c_oracle as CO

import td_oracle as TO

_SRC = Path(__file__).resolve().parent / "ntuple_stages_oracle.c"
_LIB = None
_P = C.c_void_p


def _lib():
    global _LIB
    if _LIB is None:
        out = Path(tempfile.mkdtemp(prefix="g2048_ntuple_stages_oracle_")) / "libntuple_stages_oracle.so"
        subprocess.run(["gcc", "-O2", "-fopenmp", "-fPIC", "-shared", "-ffp-contract=off", "-fno-fast-math", "-Wall",
                        "-o", str(out), str(_SRC), "-lm"], check=True, capture_output=True)
        _LIB = C.CDLL(str(out))
        _LIB.orc_ntuple_staged_value.restype = C.c_int
        _LIB.orc_ntuple_staged_value.argtypes = [_P, C.c_int64, _P, C.c_int, _P, _P, C.c_int64, _P]
        _LIB.orc_ntuple_staged_expectimax.restype = C.c_int
        _LIB.orc_ntuple_staged_expectimax.argtypes = [_P, C.c_int64, C.c_int, _P, C.c_int, _P, _P, C.c_int64,
                                                      C.c_float, _P, _P]
        _LIB.orc_ntuple_staged_td_train.restype = C.c_int
        _LIB.orc_ntuple_staged_td_train.argtypes = [_P, _P, _P, _P, C.c_int64, _P, C.c_int, _P, _P, C.c_int64,
                                                    C.c_float, _P, C.c_int64, C.c_int, _P]
        _LIB.orc_ntuple_staged_tc_train.restype = C.c_int
        _LIB.orc_ntuple_staged_tc_train.argtypes = [_P, _P, _P, _P, C.c_int64, _P, C.c_int, _P, _P, C.c_int64, _P, _P,
                                                    C.c_float, _P, C.c_int64, C.c_int, _P]
    return _LIB


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _pl(placements):
    pl = np.ascontiguousarray(placements)
    assert pl.dtype.itemsize == 12
    return pl


def _st(stages):
    st = np.ascontiguousarray(stages).reshape(-1)
    assert st.dtype.itemsize == 20 and st.shape[0] == 1
    return st


def value(packed_boards, placements, stages, W) -> np.ndarray:
    """V_S of (n,) packed boards (float32)."""
    b = np.ascontiguousarray(packed_boards, np.uint64)
    W = np.ascontiguousarray(W, np.float32)
    pl, st = _pl(placements), _st(stages)
    out = np.zeros(b.shape[0], np.float32)
    rc = _lib().orc_ntuple_staged_value(_p(b), b.shape[0], _p(pl), pl.shape[0], _p(st), _p(W), W.shape[0], _p(out))
    if rc != 0:
        raise ValueError("orc_ntuple_staged_value rejected the network or its stages")
    return out


def value_rc(placements, stages, n_weights) -> int:
    """orc_ntuple_staged_value's return code on no boards (the weights are never read)."""
    pl, st = _pl(placements), _st(stages)
    return int(_lib().orc_ntuple_staged_value(None, 0, _p(pl), pl.shape[0], _p(st), None, int(n_weights), None))


def expectimax(boards, depth, placements, stages, W, w=0.0):
    """orc_ntuple_staged_expectimax on (n,16) exponent boards: (q (n,4) float32, NaN where illegal; counters (2,))."""
    boards = np.ascontiguousarray(boards, np.uint8).reshape(-1, 16)
    W = np.ascontiguousarray(W, np.float32)
    pl, st = _pl(placements), _st(stages)
    n = boards.shape[0]
    q = np.zeros((n, 4), np.float32)
    counters = np.zeros(2, np.uint64)
    rc = _lib().orc_ntuple_staged_expectimax(_p(boards), n, int(depth), _p(pl), pl.shape[0], _p(st), _p(W), W.shape[0],
                                             float(np.float32(w)), _p(q), _p(counters))
    if rc != 0:
        raise ValueError("orc_ntuple_staged_expectimax rejected its arguments")
    return q, counters


def train(state: TO.State, placements, stages, alpha, subs, mode) -> TO.State:
    """orc_ntuple_staged_td_train on the state (its ``T`` holds W), in place (returns it)."""
    subs = np.ascontiguousarray(subs, np.uint32).reshape(-1, 2)
    pl, st = _pl(placements), _st(stages)
    rc = _lib().orc_ntuple_staged_td_train(_p(state.boards), _p(state.after), _p(state.scores), _p(state.lengths),
                                           state.boards.shape[0], _p(pl), pl.shape[0], _p(st), _p(state.T),
                                           state.T.shape[0], float(np.float32(alpha)), _p(subs), subs.shape[0],
                                           int(mode), _p(state.stats))
    if rc != 0:
        raise ValueError("orc_ntuple_staged_td_train rejected its arguments")
    return state


def tc_train(state: TO.State, E, A, placements, stages, alpha, subs, mode) -> TO.State:
    """orc_ntuple_staged_tc_train on the state (its ``T`` holds W) and on E / A (float64, the weights' length), in
    place (returns the state)."""
    subs = np.ascontiguousarray(subs, np.uint32).reshape(-1, 2)
    pl, st = _pl(placements), _st(stages)
    assert E.dtype == A.dtype == np.float64 and E.flags.c_contiguous and A.flags.c_contiguous
    assert E.shape == A.shape == state.T.shape
    rc = _lib().orc_ntuple_staged_tc_train(_p(state.boards), _p(state.after), _p(state.scores), _p(state.lengths),
                                           state.boards.shape[0], _p(pl), pl.shape[0], _p(st), _p(state.T),
                                           state.T.shape[0], _p(E), _p(A), float(np.float32(alpha)), _p(subs),
                                           subs.shape[0], int(mode), _p(state.stats))
    if rc != 0:
        raise ValueError("orc_ntuple_staged_tc_train rejected its arguments")
    return state


def train_rc(placements, stages, n_weights, tc=False) -> int:
    """The staged learner's return code for arguments it must reject, on a 4-env state with valid scalars.  The state
    arrays are sized for the 4 envs, and W and the sums are never allocated, so the helper asserts the rejection: a
    call that went on to run would read W."""
    pl, st = _pl(placements), _st(stages)
    n = 4
    s = TO.State(np.zeros(n, np.uint64), np.zeros(n, np.uint64), np.zeros(n, np.uint32), np.zeros(n, np.uint32),
                 np.zeros(1, np.float32))
    subs = np.zeros((1, 2), np.uint32)
    if tc:
        E = A = np.zeros(1)
        rc = int(_lib().orc_ntuple_staged_tc_train(_p(s.boards), _p(s.after), _p(s.scores), _p(s.lengths), n, _p(pl),
                                                   pl.shape[0], _p(st), None, int(n_weights), _p(E), _p(A), 0.01,
                                                   _p(subs), 1, 0, None))
    else:
        rc = int(_lib().orc_ntuple_staged_td_train(_p(s.boards), _p(s.after), _p(s.scores), _p(s.lengths), n, _p(pl),
                                                   pl.shape[0], _p(st), None, int(n_weights), 0.01, _p(subs), 1, 0,
                                                   None))
    assert rc == -1, "train_rc takes only arguments the staged learner rejects"
    return rc


def expectimax_games(seed, batch, depth, placements, stages, W, w, mode):
    """BatchRunner(seed, ExpectimaxPolicy(depth, network=<the staged network>, reward_weight=w)).run_eval_batch(batch)
    restated as ntuple_oracle.expectimax_games restates the unstaged player.  Returns dict(final_boards (n,16) u8,
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
        q, _ = expectimax(boards[live], depth, placements, stages, W, w)
        actions = np.zeros(batch, np.int32)
        actions[live] = XO.best_actions(q)
        alive = done == 0
        keys = CO.split(subs[2 + 2 * t], batch, mode)
        boards, masks, done, rewards = CO.env_step(boards, masks, done, actions, keys, mode)
        lengths += alive
        scores += rewards.astype(np.int64)
        t += 1
    return dict(final_boards=boards, lengths=lengths, scores=scores)
