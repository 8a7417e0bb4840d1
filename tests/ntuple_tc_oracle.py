"""ctypes binding of tests/ntuple_tc_oracle.c: temporal coherence learning of n-tuple networks restated on the CPU.
TEST INFRASTRUCTURE ONLY.

The library is compiled on first use into a temporary directory (the tree may be read-only where the tests run)."""
from __future__ import annotations

import ctypes as C
import subprocess
import tempfile
from pathlib import Path

import numpy as np

import td_oracle as TO

_SRC = Path(__file__).resolve().parent / "ntuple_tc_oracle.c"
_LIB = None
_P = C.c_void_p


def _lib():
    global _LIB
    if _LIB is None:
        out = Path(tempfile.mkdtemp(prefix="g2048_ntuple_tc_oracle_")) / "libntuple_tc_oracle.so"
        subprocess.run(["gcc", "-O2", "-fopenmp", "-fPIC", "-shared", "-ffp-contract=off", "-fno-fast-math", "-Wall",
                        "-o", str(out), str(_SRC), "-lm"], check=True, capture_output=True)
        _LIB = C.CDLL(str(out))
        _LIB.orc_ntuple_tc_train.restype = C.c_int
        _LIB.orc_ntuple_tc_train.argtypes = [_P, _P, _P, _P, C.c_int64, _P, C.c_int, _P, C.c_int64, _P, _P, C.c_float,
                                             _P, C.c_int64, C.c_int, _P]
    return _LIB


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _pl(placements):
    pl = np.ascontiguousarray(placements)
    assert pl.dtype.itemsize == 12
    return pl


def tc_train(state: TO.State, E, A, placements, alpha, subs, mode) -> TO.State:
    """orc_ntuple_tc_train on the state (its ``T`` holds W) and on E / A (float64 arrays of the weights' length), all in
    place (returns the state)."""
    subs = np.ascontiguousarray(subs, np.uint32).reshape(-1, 2)
    pl = _pl(placements)
    assert E.dtype == A.dtype == np.float64 and E.flags.c_contiguous and A.flags.c_contiguous
    assert E.shape == A.shape == state.T.shape
    rc = _lib().orc_ntuple_tc_train(_p(state.boards), _p(state.after), _p(state.scores), _p(state.lengths),
                                    state.boards.shape[0], _p(pl), pl.shape[0], _p(state.T), state.T.shape[0], _p(E),
                                    _p(A), float(np.float32(alpha)), _p(subs), subs.shape[0], int(mode), _p(state.stats))
    if rc != 0:
        raise ValueError("orc_ntuple_tc_train rejected its arguments")
    return state


def tc_train_rc(n, placements, n_weights, alpha=0.01, n_steps=1, sums=True) -> int:
    """orc_ntuple_tc_train's return code on a one-env state (``sums=False`` passes NULL for E and A; the weight array is
    never allocated, so only arguments the entry point rejects may be given)."""
    pl = _pl(placements)
    st = TO.State(np.zeros(1), np.zeros(1), np.zeros(1), np.zeros(1), np.zeros(1))
    subs = np.zeros((1, 2), np.uint32)
    E = np.zeros(1) if sums else None
    A = np.zeros(1) if sums else None
    return int(_lib().orc_ntuple_tc_train(_p(st.boards), _p(st.after), _p(st.scores), _p(st.lengths), int(n), _p(pl),
                                          pl.shape[0], None, int(n_weights), _p(E), _p(A), float(alpha), _p(subs),
                                          int(n_steps), 0, None))
