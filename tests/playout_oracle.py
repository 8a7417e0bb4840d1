"""ctypes binding of tests/playout_oracle.c: the Monte-Carlo playout contract (g2048_playout_values) and the
Monte-Carlo player restated with the C oracle's game and policies.  TEST INFRASTRUCTURE ONLY.

The library is compiled on first use into a temporary directory (the tree may be read-only where the tests run)."""
from __future__ import annotations

import ctypes as C
import subprocess
import tempfile
from pathlib import Path

import numpy as np

from oracle import c_oracle as CO

_SRC = Path(__file__).resolve().parent / "playout_oracle.c"
_LIB = None


def _lib():
    global _LIB
    if _LIB is None:
        out = Path(tempfile.mkdtemp(prefix="g2048_playout_oracle_")) / "libplayout_oracle.so"
        subprocess.run(["gcc", "-O2", "-fopenmp", "-fPIC", "-shared", "-ffp-contract=off", "-fno-fast-math", "-Wall",
                        "-o", str(out), str(_SRC), "-lm"], check=True, capture_output=True)
        _LIB = C.CDLL(str(out))
    return _LIB


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def playout(boards, playouts, subs, policy, mode, ids=None, board_lo=0, n_global=None):
    """orc_playout: K = `playouts` Monte-Carlo games per (board, action) of the (n,16) exponent boards (global ids `ids`
    or board_lo + i, in a batch of n_global boards); subs (1 + 2*max_steps, 2) as for `oracle.c_oracle.play`.
    Returns dict of (n,4) arrays score_sum, score_sq_sum, steps_sum (uint64), playouts, cut_short (uint32)."""
    boards = np.ascontiguousarray(boards, np.uint8).reshape(-1, 16)
    subs = np.ascontiguousarray(subs, np.uint32)
    n = boards.shape[0]
    n_global = board_lo + n if n_global is None else n_global
    ids = None if ids is None else np.ascontiguousarray(ids, np.int64)
    out = {k: np.zeros((n, 4), np.uint64) for k in ("score_sum", "score_sq_sum", "steps_sum")}
    out.update({k: np.zeros((n, 4), np.uint32) for k in ("playouts", "cut_short")})
    _lib().orc_playout(
        _p(boards), C.c_int64(n), _p(ids) if ids is not None else None, C.c_int64(board_lo), C.c_int64(n_global),
        C.c_int64(playouts), _p(subs), C.c_int64((subs.shape[0] - 1) // 2), C.c_int(policy), C.c_int(mode),
        _p(out["score_sum"]), _p(out["score_sq_sum"]), _p(out["steps_sum"]), _p(out["playouts"]),
        _p(out["cut_short"]),
    )
    return out


def best_actions(rec, criterion="score"):
    """Per board the legal action with the largest sum of the criterion over its playouts, ties to the lowest index."""
    sums = rec["score_sum" if criterion == "score" else "steps_sum"].astype(np.int64)
    return np.where(rec["playouts"] > 0, sums, -1).argmax(axis=1).astype(np.int32)


def monte_carlo_games(seed, batch, playouts, policy, criterion, mode, max_steps=2048, env_lo=0, env_hi=None, key=None):
    """Envs [env_lo, env_hi) of BatchRunner(seed, MonteCarloPolicy(playouts, rollout, criterion, max_steps))
    .run_eval_batch(batch): at loop step t the live envs' playouts use split(act sub key of t, 1 + 2*max_steps), the
    chosen actions are stepped with split(step sub key of t, batch)[env].  Returns dict(final_boards (n,16) u8, lengths,
    scores)."""
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
        psubs = CO.split(subs[1 + 2 * t], 1 + 2 * max_steps, mode)
        rec = playout(boards[live], playouts, psubs, policy, mode, ids=live + env_lo, n_global=batch)
        actions = np.zeros(n, np.int32)
        actions[live] = best_actions(rec, criterion)
        alive = done == 0
        keys = CO.split(subs[2 + 2 * t], batch, mode)[env_lo:env_hi]
        boards, masks, done, rewards = CO.env_step(boards, masks, done, actions, keys, mode)
        lengths += alive
        scores += rewards.astype(np.int64)
        t += 1
    return dict(final_boards=boards, lengths=lengths, scores=scores)
