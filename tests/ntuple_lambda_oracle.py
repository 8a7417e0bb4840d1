"""ctypes binding of tests/ntuple_lambda_oracle.c: delayed TD(lambda) and TC(lambda) learning of n-tuple networks,
staged or not, restated on the CPU.  TEST INFRASTRUCTURE ONLY.

``stages`` is None (one stage) or a (1,) ``g2048.ntuple.STAGES_DTYPE`` record.  The rings ``hist_after`` (uint64) and
``hist_delta`` (float32) are (h, n) arrays, updated in place.  The library is compiled on first use into a temporary
directory (the tree may be read-only where the tests run)."""
from __future__ import annotations

import ctypes as C
import subprocess
import tempfile
from pathlib import Path

import numpy as np

import td_oracle as TO

_SRC = Path(__file__).resolve().parent / "ntuple_lambda_oracle.c"
_LIB = None
_P = C.c_void_p


def _lib():
    global _LIB
    if _LIB is None:
        out = Path(tempfile.mkdtemp(prefix="g2048_ntuple_lambda_oracle_")) / "libntuple_lambda_oracle.so"
        subprocess.run(["gcc", "-O2", "-fopenmp", "-fPIC", "-shared", "-ffp-contract=off", "-fno-fast-math", "-Wall",
                        "-o", str(out), str(_SRC), "-lm"], check=True, capture_output=True)
        _LIB = C.CDLL(str(out))
        _LIB.orc_ntuple_lambda_coefficients.restype = None
        _LIB.orc_ntuple_lambda_coefficients.argtypes = [C.c_float, C.c_int, _P]
        _LIB.orc_ntuple_lambda_td_train.restype = C.c_int
        _LIB.orc_ntuple_lambda_td_train.argtypes = [_P, _P, _P, _P, C.c_int64, _P, C.c_int, _P, _P, C.c_int64,
                                                    C.c_float, C.c_float, C.c_int, _P, _P, _P, C.c_int64, C.c_int, _P]
        _LIB.orc_ntuple_lambda_tc_train.restype = C.c_int
        _LIB.orc_ntuple_lambda_tc_train.argtypes = [_P, _P, _P, _P, C.c_int64, _P, C.c_int, _P, _P, C.c_int64, _P, _P,
                                                    C.c_float, C.c_float, C.c_int, _P, _P, _P, C.c_int64, C.c_int, _P]
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


def coefficients(lam, h) -> np.ndarray:
    """c_0 .. c_7 as the entry points compute them (zero from h on), float32."""
    c = np.zeros(8, np.float32)
    _lib().orc_ntuple_lambda_coefficients(float(np.float32(lam)), int(h), _p(c))
    return c


def rings(h, n):
    """Zeroed (hist_after, hist_delta) rings of h slots for n envs."""
    return np.zeros((h, n), np.uint64), np.zeros((h, n), np.float32)


def _check_rings(state, hist_after, hist_delta):
    n = state.boards.shape[0]
    assert hist_after.dtype == np.uint64 and hist_delta.dtype == np.float32
    assert hist_after.flags.c_contiguous and hist_delta.flags.c_contiguous
    assert hist_after.shape == hist_delta.shape and hist_after.shape[1] == n
    return hist_after.shape[0]


def train(state: TO.State, hist_after, hist_delta, placements, stages, alpha, lam, subs, mode) -> TO.State:
    """orc_ntuple_lambda_td_train on the state (its ``T`` holds W) and the rings, in place (returns the state)."""
    subs = np.ascontiguousarray(subs, np.uint32).reshape(-1, 2)
    pl, st = _pl(placements), _st(stages)
    h = _check_rings(state, hist_after, hist_delta)
    rc = _lib().orc_ntuple_lambda_td_train(_p(state.boards), _p(state.after), _p(state.scores), _p(state.lengths),
                                           state.boards.shape[0], _p(pl), pl.shape[0], _p(st), _p(state.T),
                                           state.T.shape[0], float(np.float32(alpha)), float(np.float32(lam)), h,
                                           _p(hist_after), _p(hist_delta), _p(subs), subs.shape[0], int(mode),
                                           _p(state.stats))
    if rc != 0:
        raise ValueError("orc_ntuple_lambda_td_train rejected its arguments")
    return state


def tc_train(state: TO.State, E, A, hist_after, hist_delta, placements, stages, alpha, lam, subs, mode) -> TO.State:
    """orc_ntuple_lambda_tc_train on the state, E / A (float64, the weights' length) and the rings, in place."""
    subs = np.ascontiguousarray(subs, np.uint32).reshape(-1, 2)
    pl, st = _pl(placements), _st(stages)
    h = _check_rings(state, hist_after, hist_delta)
    assert E.dtype == A.dtype == np.float64 and E.flags.c_contiguous and A.flags.c_contiguous
    assert E.shape == A.shape == state.T.shape
    rc = _lib().orc_ntuple_lambda_tc_train(_p(state.boards), _p(state.after), _p(state.scores), _p(state.lengths),
                                           state.boards.shape[0], _p(pl), pl.shape[0], _p(st), _p(state.T),
                                           state.T.shape[0], _p(E), _p(A), float(np.float32(alpha)),
                                           float(np.float32(lam)), h, _p(hist_after), _p(hist_delta), _p(subs),
                                           subs.shape[0], int(mode), _p(state.stats))
    if rc != 0:
        raise ValueError("orc_ntuple_lambda_tc_train rejected its arguments")
    return state


def train_rc(placements, n_weights, lam, h, n=4, stages=None, tc=False, rings_given=True) -> int:
    """The learner's return code for arguments it must reject, on an n-env state with valid scalars.  W and the sums
    are never allocated, so the helper asserts the rejection: a call that went on to run would read W."""
    pl, st = _pl(placements), _st(stages)
    s = TO.State(np.zeros(n, np.uint64), np.zeros(n, np.uint64), np.zeros(n, np.uint32), np.zeros(n, np.uint32),
                 np.zeros(1, np.float32))
    ha, hd = (np.zeros(8, np.uint64), np.zeros(8, np.float32)) if rings_given else (None, None)
    subs = np.zeros((1, 2), np.uint32)
    lam = float(np.float32(lam)) if np.isfinite(lam) else float(lam)
    if tc:
        E = A = np.zeros(1)
        rc = int(_lib().orc_ntuple_lambda_tc_train(_p(s.boards), _p(s.after), _p(s.scores), _p(s.lengths), n, _p(pl),
                                                   pl.shape[0], _p(st), None, int(n_weights), _p(E), _p(A), 0.01, lam,
                                                   int(h), _p(ha), _p(hd), _p(subs), 1, 0, None))
    else:
        rc = int(_lib().orc_ntuple_lambda_td_train(_p(s.boards), _p(s.after), _p(s.scores), _p(s.lengths), n, _p(pl),
                                                   pl.shape[0], _p(st), None, int(n_weights), 0.01, lam, int(h),
                                                   _p(ha), _p(hd), _p(subs), 1, 0, None))
    assert rc == -1, "train_rc takes only arguments the lambda learner rejects"
    return rc
