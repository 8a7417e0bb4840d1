"""ctypes binding of tests/td_oracle.c: the TD(0) row-table learner (g2048_td_train) restated with the C oracle's game
and the expectimax oracle's H and move.  TEST INFRASTRUCTURE ONLY.

The library is compiled on first use into a temporary directory (the tree may be read-only where the tests run)."""
from __future__ import annotations

import ctypes as C
import subprocess
import tempfile
from pathlib import Path

import numpy as np

from oracle import c_oracle as CO

_SRC = Path(__file__).resolve().parent / "td_oracle.c"
_LIB = None
STATS_WORDS = 32


def _lib():
    global _LIB
    if _LIB is None:
        out = Path(tempfile.mkdtemp(prefix="g2048_td_oracle_")) / "libtd_oracle.so"
        subprocess.run(["gcc", "-O2", "-fopenmp", "-fPIC", "-shared", "-ffp-contract=off", "-fno-fast-math", "-Wall",
                        "-o", str(out), str(_SRC), "-lm"], check=True, capture_output=True)
        _LIB = C.CDLL(str(out))
        _LIB.orc_td_train.restype = C.c_int
        _LIB.orc_td_train.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_float,
                                      C.c_void_p, C.c_int64, C.c_int, C.c_void_p]
        _LIB.orc_td_fx.restype = C.c_int64
        _LIB.orc_td_fx.argtypes = [C.c_float]
    return _LIB


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def fx(d) -> int:
    return int(_lib().orc_td_fx(float(np.float32(d))))


class State:
    """The learner's state as host arrays: boards / after (n,) uint64, scores / lengths (n,) uint32, T (65536,) float32,
    stats (32,) uint64 accumulated."""

    def __init__(self, boards, after, scores, lengths, T):
        self.boards = np.ascontiguousarray(boards, np.uint64).copy()
        self.after = np.ascontiguousarray(after, np.uint64).copy()
        self.scores = np.ascontiguousarray(scores, np.uint32).copy()
        self.lengths = np.ascontiguousarray(lengths, np.uint32).copy()
        self.T = np.ascontiguousarray(T, np.float32).copy()
        self.stats = np.zeros(STATS_WORDS, np.uint64)

    def copy(self):
        s = State(self.boards, self.after, self.scores, self.lengths, self.T)
        s.stats = self.stats.copy()
        return s


def fresh(key, n, mode, T):
    """Envs initialised with split(key, n)[e] and no afterstate (what TDLearner's sub key 0 does)."""
    boards, _ = CO.env_init(CO.split(np.asarray(key, np.uint32), n, mode), mode)
    packed = (boards.astype(np.uint64) << (np.arange(16, dtype=np.uint64) * np.uint64(4))).sum(axis=1).astype(np.uint64)
    return State(packed, np.zeros(n, np.uint64), np.zeros(n, np.uint32), np.zeros(n, np.uint32), T)


def train(state: State, alpha, subs, mode) -> State:
    """orc_td_train on the state, in place (returns it)."""
    subs = np.ascontiguousarray(subs, np.uint32).reshape(-1, 2)
    rc = _lib().orc_td_train(_p(state.boards), _p(state.after), _p(state.scores), _p(state.lengths), state.boards.shape[0],
                             _p(state.T), float(np.float32(alpha)), _p(subs), subs.shape[0], int(mode), _p(state.stats))
    if rc != 0:
        raise ValueError("orc_td_train rejected its arguments")
    return state


def train_rc(n, alpha, n_steps) -> int:
    """orc_td_train's return code for the given sizes and alpha (on a one-env state, nothing allocated beyond it)."""
    st = State(np.zeros(1), np.zeros(1), np.zeros(1), np.zeros(1), np.zeros(65536))
    subs = np.zeros((1, 2), np.uint32)
    return int(_lib().orc_td_train(_p(st.boards), _p(st.after), _p(st.scores), _p(st.lengths), int(n), _p(st.T),
                                   float(alpha), _p(subs), int(n_steps), 0, None))
