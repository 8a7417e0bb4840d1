"""ctypes binding of tests/ntuple_carousel_oracle.c: carousel shaping of multi-stage n-tuple networks, learned by TD /
TC with a window of h afterstates (h = 1: TD(0) / TC), restated on the CPU.  TEST INFRASTRUCTURE ONLY.

``stages`` is a (1,) ``g2048.ntuple.STAGES_DTYPE`` record with S >= 2.  ``start_stage`` (uint32, (n,)) and ``pool``
(uint64, (S - 1, n)) are updated in place, as are the rings ``hist_after`` / ``hist_delta`` ((h, n) arrays, or None for
h = 1).  The library is compiled on first use into a temporary directory (the tree may be read-only where the tests
run)."""
from __future__ import annotations

import ctypes as C
import subprocess
import tempfile
from pathlib import Path

import numpy as np

import td_oracle as TO

_SRC = Path(__file__).resolve().parent / "ntuple_carousel_oracle.c"
_LIB = None
_P = C.c_void_p


def _lib():
    global _LIB
    if _LIB is None:
        out = Path(tempfile.mkdtemp(prefix="g2048_ntuple_carousel_oracle_")) / "libntuple_carousel_oracle.so"
        subprocess.run(["gcc", "-O2", "-fopenmp", "-fPIC", "-shared", "-ffp-contract=off", "-fno-fast-math", "-Wall",
                        "-o", str(out), str(_SRC), "-lm"], check=True, capture_output=True)
        _LIB = C.CDLL(str(out))
        _LIB.orc_ntuple_carousel_td_train.restype = C.c_int
        _LIB.orc_ntuple_carousel_td_train.argtypes = [_P, _P, _P, _P, C.c_int64, _P, C.c_int, _P, _P, C.c_int64,
                                                      C.c_float, C.c_float, C.c_int, _P, _P, _P, _P, _P, C.c_int64,
                                                      C.c_int, _P]
        _LIB.orc_ntuple_carousel_tc_train.restype = C.c_int
        _LIB.orc_ntuple_carousel_tc_train.argtypes = [_P, _P, _P, _P, C.c_int64, _P, C.c_int, _P, _P, C.c_int64, _P,
                                                      _P, C.c_float, C.c_float, C.c_int, _P, _P, _P, _P, _P, C.c_int64,
                                                      C.c_int, _P]
    return _LIB


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _pl(placements):
    pl = np.ascontiguousarray(placements)
    assert pl.dtype.itemsize == 12
    return pl


def _st(stages):
    if stages is None:
        return None
    st = np.ascontiguousarray(stages).reshape(-1)
    assert st.dtype.itemsize == 20 and st.shape[0] == 1
    return st


def arrays(stages, n):
    """Zeroed (start_stage, pool) for n envs of a network with these stages."""
    S = int(_st(stages)["n_thresholds"][0]) + 1
    return np.zeros(n, np.uint32), np.zeros((S - 1, n), np.uint64)


def _check(state, start_stage, pool, hist_after, hist_delta):
    n = state.boards.shape[0]
    assert start_stage.dtype == np.uint32 and start_stage.shape == (n,) and start_stage.flags.c_contiguous
    assert pool.dtype == np.uint64 and pool.ndim == 2 and pool.shape[1] == n and pool.flags.c_contiguous
    if hist_after is None:
        assert hist_delta is None
        return 1
    assert hist_after.dtype == np.uint64 and hist_delta.dtype == np.float32
    assert hist_after.flags.c_contiguous and hist_delta.flags.c_contiguous
    assert hist_after.shape == hist_delta.shape and hist_after.shape[1] == n
    return hist_after.shape[0]


def train(state: TO.State, start_stage, pool, placements, stages, alpha, subs, mode, lam=0.0, hist_after=None,
          hist_delta=None) -> TO.State:
    """orc_ntuple_carousel_td_train on the state (its ``T`` holds W), the carousel arrays and the rings, in place."""
    subs = np.ascontiguousarray(subs, np.uint32).reshape(-1, 2)
    pl, st = _pl(placements), _st(stages)
    h = _check(state, start_stage, pool, hist_after, hist_delta)
    rc = _lib().orc_ntuple_carousel_td_train(_p(state.boards), _p(state.after), _p(state.scores), _p(state.lengths),
                                             state.boards.shape[0], _p(pl), pl.shape[0], _p(st), _p(state.T),
                                             state.T.shape[0], float(np.float32(alpha)), float(np.float32(lam)), h,
                                             _p(hist_after), _p(hist_delta), _p(start_stage), _p(pool), _p(subs),
                                             subs.shape[0], int(mode), _p(state.stats))
    if rc != 0:
        raise ValueError("orc_ntuple_carousel_td_train rejected its arguments")
    return state


def tc_train(state: TO.State, E, A, start_stage, pool, placements, stages, alpha, subs, mode, lam=0.0,
             hist_after=None, hist_delta=None) -> TO.State:
    """orc_ntuple_carousel_tc_train on the state, E / A (float64, the weights' length), the carousel arrays and the
    rings, in place."""
    subs = np.ascontiguousarray(subs, np.uint32).reshape(-1, 2)
    pl, st = _pl(placements), _st(stages)
    h = _check(state, start_stage, pool, hist_after, hist_delta)
    assert E.dtype == A.dtype == np.float64 and E.flags.c_contiguous and A.flags.c_contiguous
    assert E.shape == A.shape == state.T.shape
    rc = _lib().orc_ntuple_carousel_tc_train(_p(state.boards), _p(state.after), _p(state.scores), _p(state.lengths),
                                             state.boards.shape[0], _p(pl), pl.shape[0], _p(st), _p(state.T),
                                             state.T.shape[0], _p(E), _p(A), float(np.float32(alpha)),
                                             float(np.float32(lam)), h, _p(hist_after), _p(hist_delta),
                                             _p(start_stage), _p(pool), _p(subs), subs.shape[0], int(mode),
                                             _p(state.stats))
    if rc != 0:
        raise ValueError("orc_ntuple_carousel_tc_train rejected its arguments")
    return state


def train_rc(placements, n_weights, stages, h=1, n=4, tc=False, arrays_given=True, rings_given=True) -> int:
    """The learner's return code for arguments it must reject, on an n-env state with valid scalars.  W and the sums
    are never allocated, so the helper asserts the rejection: a call that went on to run would read W."""
    pl, st = _pl(placements), _st(stages)
    s = TO.State(np.zeros(n, np.uint64), np.zeros(n, np.uint64), np.zeros(n, np.uint32), np.zeros(n, np.uint32),
                 np.zeros(1, np.float32))
    ha, hd = (np.zeros(8 * n, np.uint64), np.zeros(8 * n, np.float32)) if rings_given else (None, None)
    ss, pool = (np.zeros(n, np.uint32), np.zeros(16 * n, np.uint64)) if arrays_given else (None, None)
    subs = np.zeros((1, 2), np.uint32)
    if tc:
        E = A = np.zeros(1)
        rc = int(_lib().orc_ntuple_carousel_tc_train(_p(s.boards), _p(s.after), _p(s.scores), _p(s.lengths), n,
                                                     _p(pl), pl.shape[0], _p(st), None, int(n_weights), _p(E), _p(A),
                                                     0.01, 0.5, int(h), _p(ha), _p(hd), _p(ss), _p(pool), _p(subs), 1,
                                                     0, None))
    else:
        rc = int(_lib().orc_ntuple_carousel_td_train(_p(s.boards), _p(s.after), _p(s.scores), _p(s.lengths), n,
                                                     _p(pl), pl.shape[0], _p(st), None, int(n_weights), 0.01, 0.5,
                                                     int(h), _p(ha), _p(hd), _p(ss), _p(pool), _p(subs), 1, 0, None))
    assert rc == -1, "train_rc takes only arguments the carousel learner rejects"
    return rc
