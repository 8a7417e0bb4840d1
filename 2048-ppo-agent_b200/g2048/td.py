"""TD(0) afterstate learning of the expectimax row table on the GPU.

    learner = g2048.TDLearner(0, batch_size=1 << 16)
    summary = learner.train(2000)                                   # the episodes that ended in these steps
    player = g2048.ExpectimaxPolicy(depth=1, row_values=learner.table, reward_weight=1.0)

The learned table ``T`` is the one ``expectimax_values`` / ``ExpectimaxPolicy`` read: ``H(b) = sum of T[line]`` over the
4 rows and 4 columns.  Every env plays the greedy afterstate move (``ExpectimaxPolicy(depth=1, row_values=T,
reward_weight=1.0)``), and ``T`` moves toward ``r' + H(s'')`` at the lines of the previous afterstate.  All
``batch_size`` envs of a step read the same ``T``, the errors are summed in fixed point, and the update follows the
whole step, so training is bit-exact and a run is a function of (seed, batch size, alpha, initial table, rng_mode,
steps).  A call of ``train`` is one launch of ``g2048_td_train`` (include/g2048.h).
"""
from __future__ import annotations

import math

import numpy as np
import torch

from . import _native as N
from . import engine as E
from .keys import KeyChain

# the step size of the round-7 sweep on one B200 whose greedy player scored best (profiles/README.md, round 7)
DEFAULT_ALPHA = 0.1
MAX_BATCH = 1 << 20
_FLT_MAX = float(np.finfo(np.float32).max)


def _check_alpha(alpha) -> float:
    alpha = float(alpha)
    if not (math.isfinite(alpha) and 0.0 <= alpha <= _FLT_MAX):
        raise ValueError(f"alpha must be a finite float32 >= 0, got {alpha}")
    return alpha


def _check_table(table) -> torch.Tensor:
    """A host or device copy of 65 536 finite values as a float32 (65536,) tensor, or ValueError."""
    table = table.detach() if isinstance(table, torch.Tensor) else torch.from_numpy(np.asarray(table, np.float32))
    if table.numel() != 65536:
        raise ValueError("table must hold 65536 values")
    table = table.reshape(65536).to(torch.float32)
    if not bool(torch.isfinite(table).all()):
        raise ValueError("table must be finite")
    return table


class TDLearner:
    """Learns the row table by synchronous batched TD(0) over ``batch_size`` envs (1 .. 2^20).

    ``table``: the float32 (65536,) device tensor being learned (zeros, or a copy of the given finite table).
    ``train(n_steps)`` makes ``n_steps`` steps and returns the summary of the episodes that ended in them
    (``engine.play_stats_dict`` form).  Keys come from the runner's chain of ``init_seed``: sub key 0 initialises the
    envs, and every step consumes one more.  ``state_dict`` / ``load_state_dict`` resume a run bit for bit."""

    def __init__(self, init_seed: int, batch_size: int, alpha: float = DEFAULT_ALPHA, table=None, rng_mode=None,
                 device=None):
        batch_size = int(batch_size)
        if not 1 <= batch_size <= MAX_BATCH:
            raise ValueError(f"batch_size must be in [1, 2^20], got {batch_size}")
        self.alpha = _check_alpha(alpha)
        if table is not None:
            table = _check_table(table)
        self.rng_mode = E.resolve_rng_mode(rng_mode)
        self.device = N.require_cuda() if device is None else torch.device(device)
        self.batch_size = batch_size
        if table is None:
            self.table = torch.zeros(65536, dtype=torch.float32, device=self.device)
        else:
            self.table = table.to(self.device).clone()
        self.chain = KeyChain(init_seed, self.rng_mode, self.device)
        n = batch_size
        self.boards, _ = E.env_init(self.chain.peek(1)[0], n, 0, n, self.rng_mode)
        self.chain.consume(1)
        self.after = torch.zeros(n, dtype=torch.int64, device=self.device)
        self.scores = torch.zeros(n, dtype=torch.int32, device=self.device)
        self.lengths = torch.zeros(n, dtype=torch.int32, device=self.device)
        self._scratch = E.td_scratch(self.device)
        self.steps = 0

    def train(self, n_steps: int) -> dict:
        """``n_steps`` learning steps in one launch; returns the summary of the episodes that ended in them."""
        n_steps = int(n_steps)
        if n_steps < 0:
            raise ValueError(f"n_steps must be >= 0, got {n_steps}")
        stats = torch.zeros(N.PLAY_STATS_WORDS, dtype=torch.int64, device=self.device)
        if n_steps:
            subs = self.chain.peek(n_steps)
            E.td_train(self.boards, self.after, self.scores, self.lengths, self.table, self.alpha, subs, self.rng_mode,
                       self._scratch, stats)
            self.chain.consume(n_steps)
            self.steps += n_steps
        return E.play_stats_dict(stats)

    # -- checkpointing: key chain, env state and table ---------------------------------------------------------
    def state_dict(self) -> dict:
        return {"key": [int(w) for w in self.chain.key], "position": int(self.chain.position), "rng_mode": int(self.rng_mode),
                "batch_size": self.batch_size, "alpha": self.alpha, "steps": self.steps, "table": self.table.cpu().clone(),
                "boards": self.boards.cpu().clone(), "after": self.after.cpu().clone(),
                "scores": self.scores.cpu().clone(), "lengths": self.lengths.cpu().clone()}

    def load_state_dict(self, state: dict) -> None:
        if int(state["batch_size"]) != self.batch_size or state["boards"].shape[0] != self.batch_size:
            raise ValueError("checkpoint was written for a different batch size")
        alpha = _check_alpha(state["alpha"])
        table = _check_table(state["table"])
        if int(state["rng_mode"]) not in (E.RNG_ORIGINAL, E.RNG_PARTITIONABLE):
            raise ValueError(f"checkpoint has an unknown rng_mode {state['rng_mode']!r}")
        self.alpha = alpha
        self.rng_mode = int(state["rng_mode"])
        self.chain = KeyChain(np.asarray(state["key"], dtype=np.uint32), self.rng_mode, self.device)
        self.chain._base_pos = int(state["position"])
        self.steps = int(state["steps"])
        self.table.copy_(table.to(self.device))
        for name in ("boards", "after", "scores", "lengths"):
            getattr(self, name).copy_(state[name].to(self.device))
