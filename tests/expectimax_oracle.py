"""ctypes binding of tests/expectimax_oracle.c: the expectimax contract (g2048_expectimax_values) and the expectimax
player restated with the C oracle's game.  TEST INFRASTRUCTURE ONLY.

The library is compiled on first use into a temporary directory (the tree may be read-only where the tests run)."""
from __future__ import annotations

import ctypes as C
import subprocess
import tempfile
from pathlib import Path

import numpy as np

from oracle import c_oracle as CO

_SRC = Path(__file__).resolve().parent / "expectimax_oracle.c"
_LIB = None


def _lib():
    global _LIB
    if _LIB is None:
        out = Path(tempfile.mkdtemp(prefix="g2048_expectimax_oracle_")) / "libexpectimax_oracle.so"
        subprocess.run(["gcc", "-O2", "-fopenmp", "-fPIC", "-shared", "-ffp-contract=off", "-fno-fast-math", "-Wall",
                        "-o", str(out), str(_SRC), "-lm"], check=True, capture_output=True)
        _LIB = C.CDLL(str(out))
        _LIB.orc_expectimax.argtypes = [C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_float, C.c_void_p, C.c_void_p]
    return _LIB


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def expectimax(boards, depth, table, w=0.0):
    """orc_expectimax on (n,16) exponent boards: returns (q (n,4) float32 with NaN where illegal, counters (2,) uint64
    = leaves, chance nodes)."""
    boards = np.ascontiguousarray(boards, np.uint8).reshape(-1, 16)
    table = np.ascontiguousarray(table, np.float32)
    assert table.shape == (65536,)
    n = boards.shape[0]
    q = np.zeros((n, 4), np.float32)
    counters = np.zeros(2, np.uint64)
    _lib().orc_expectimax(_p(boards), n, int(depth), _p(table), float(w), _p(q), _p(counters))
    return q, counters


def best_actions(q):
    """Per board the legal action with the largest value, ties to the lowest index; 0 without a legal action."""
    return np.where(np.isnan(q), -np.inf, q).argmax(axis=1).astype(np.int32)


def expectimax_games(seed, batch, depth, table, w, mode, env_lo=0, env_hi=None, key=None):
    """Envs [env_lo, env_hi) of BatchRunner(seed, ExpectimaxPolicy(depth, table, w)).run_eval_batch(batch): at loop
    step t the live envs play their best action and are stepped with split(step sub key of t, batch)[env].  Returns
    dict(final_boards (n,16) u8, lengths, scores)."""
    env_hi = batch if env_hi is None else env_hi
    n = env_hi - env_lo
    if key is None:
        key = np.array([(int(seed) >> 32) & 0xFFFFFFFF, int(seed) & 0xFFFFFFFF], np.uint32)
    n_sub = 1 + 2 * 1024
    _, subs = CO.chain(key, mode, n_sub)
    boards, masks = CO.env_init(CO.split(subs[0], batch, mode)[env_lo:env_hi], mode)
    done = np.zeros(n, np.uint8)
    lengths = np.zeros(n, np.int64)
    scores = np.zeros(n, np.int64)
    t = 0
    while not done.all():
        if 2 + 2 * t >= subs.shape[0]:
            n_sub = 2 * n_sub + 1
            _, subs = CO.chain(key, mode, n_sub)
        live = np.flatnonzero(done == 0)
        q, _ = expectimax(boards[live], depth, table, w)
        actions = np.zeros(n, np.int32)
        actions[live] = best_actions(q)
        alive = done == 0
        keys = CO.split(subs[2 + 2 * t], batch, mode)[env_lo:env_hi]
        boards, masks, done, rewards = CO.env_step(boards, masks, done, actions, keys, mode)
        lengths += alive
        scores += rewards.astype(np.int64)
        t += 1
    return dict(final_boards=boards, lengths=lengths, scores=scores)
