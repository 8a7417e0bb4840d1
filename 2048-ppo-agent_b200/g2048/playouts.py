"""Monte-Carlo playout values of given boards, and the playout-search player built on them.

    res = g2048.playout_values(boards, playouts=256, key=g2048.keys.key(0))   # K games per (board, action)
    res.mean_score, res.best_action()

    runner = g2048.BatchRunner(0, g2048.MonteCarloPolicy(playouts=64))
    out = runner.run_eval_batch(1024)                                          # every move chosen by playouts

The playouts run in one launch of the persistent play kernel (``g2048_playout_values``): for each (board, action) pair
K games are played to the end with a built-in rollout policy after that action.  ``score`` is the sum of the merge
rewards from the board on (the first move's included), ``length`` the number of moves (the first one included).
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np
import torch

from . import _native as N
from . import engine as E
from .actions import act_randomly
from .keys import as_key_tensor

CRITERIA = ("score", "length")


def _sums(records: dict, criterion: str) -> torch.Tensor:
    if criterion not in CRITERIA:
        raise ValueError(f"criterion must be one of {CRITERIA}, got {criterion!r}")
    return records["score_sum"] if criterion == "score" else records["steps_sum"]


def best_actions(records: dict, criterion: str = "score") -> torch.Tensor:
    """(n,) int64: per board the legal action with the largest sum of ``criterion`` over its playouts (every legal
    action has the same number of playouts, so this is the largest mean), ties to the lowest action index; 0 for a
    board without a legal action."""
    sums = _sums(records, criterion)
    legal = records["playouts"] > 0
    return torch.where(legal, sums, torch.full_like(sums, -1)).argmax(dim=1)


def _rollout_policy(rollout) -> int:
    policy = getattr(rollout, "policy_id", None)
    if policy is None:
        raise ValueError("the rollout policy must be g2048.act_randomly or g2048.act_drul")
    return policy


class PlayoutValues:
    """Result of ``playout_values``: per (board, action) the integer sums over its playouts (device tensors, (n, 4)
    int64: ``score_sum``, ``score_sq_sum``, ``steps_sum``, ``playouts``, ``cut_short``) and the float64 summaries
    ``mean_score``, ``std_score`` (population), ``mean_length`` -- NaN where the action is illegal."""

    def __init__(self, records: dict):
        self.records = records
        for k in ("score_sum", "score_sq_sum", "steps_sum", "playouts", "cut_short"):
            setattr(self, k, records[k])
        self.stats = records["stats"]
        count = self.playouts.double()
        legal = self.playouts > 0
        nan = torch.full_like(count, float("nan"))
        self.mean_score = torch.where(legal, self.score_sum.double() / count, nan)
        self.mean_length = torch.where(legal, self.steps_sum.double() / count, nan)
        var = self.score_sq_sum.double() / count - self.mean_score ** 2
        self.std_score = torch.where(legal, var.clamp(min=0.0).sqrt(), nan)

    @property
    def legal(self) -> torch.Tensor:
        return self.playouts > 0

    def best_action(self, criterion: str = "score") -> torch.Tensor:
        """(n,) int64 argmax over the legal actions of the integer sums; ties go to the lowest action index."""
        return best_actions(self.records, criterion)


def playout_values(boards, playouts: int, key, rollout=act_randomly, max_steps: int = 2048, rng_mode=None,
                   device=None) -> PlayoutValues:
    """Play ``playouts`` games per (board, action) to the end with ``rollout`` (act_randomly / act_drul) after that
    action, at most ``max_steps`` moves each.  ``boards``: (n,) int64 bitboards (a tensor, or anything numpy reads as
    such); ``key``: a jax.random-style key (two uint32 words, or an int seed).  Board i is board i of a batch of n,
    and the playouts use the sub keys ``split(key, 1 + 2 * max_steps)``, so the result is a function of (boards, key,
    playouts, rollout, max_steps, rng_mode)."""
    if playouts < 1:
        raise ValueError(f"playouts must be >= 1, got {playouts}")
    if max_steps < 1:
        raise ValueError(f"max_steps must be >= 1, got {max_steps}")
    policy = _rollout_policy(rollout)
    mode = E.resolve_rng_mode(rng_mode)
    if isinstance(boards, torch.Tensor):
        device = boards.device if device is None else torch.device(device)
        boards = boards.to(device=device, dtype=torch.int64).contiguous()
    else:
        device = N.require_cuda() if device is None else torch.device(device)
        boards = torch.from_numpy(np.ascontiguousarray(np.asarray(boards, dtype=np.uint64).reshape(-1)).view(np.int64)).to(device)
    if isinstance(key, (int, np.integer)):
        key = list(E.key_words(int(key)))
    n_subs = 1 + 2 * max_steps
    subs = E.split_keys(as_key_tensor(key, device), n_subs, 0, n_subs, mode)
    stats = torch.zeros(N.PLAY_STATS_WORDS, dtype=torch.int64, device=device)
    return PlayoutValues(E.playout_values(policy, boards, subs, playouts, mode, stats=stats))


@dataclass(frozen=True)
class MonteCarloPolicy:
    """The pure Monte-Carlo player: at every move, ``playouts`` games per legal action played to the end with
    ``rollout`` (at most ``max_steps`` moves each); the action with the best mean ``criterion`` ("score" or "length")
    is played.  An act_fn for ``BatchRunner.run_eval_batch``: at loop step t the runner's act sub key is the key of that
    move's playouts (sub keys ``split(act_key, 1 + 2 * max_steps)``), only the envs still alive are evaluated, with
    their global env ids as board ids, and the chosen actions are stepped with the step sub key like any policy's --
    so a game is a function of (seed, batch size, playouts, rollout, criterion, rng_mode, max_steps) and does not
    depend on sharding."""

    playouts: int = 64
    rollout: object = act_randomly
    criterion: str = "score"
    max_steps: int = 2048

    def __post_init__(self):
        if int(self.playouts) < 1:
            raise ValueError(f"playouts must be >= 1, got {self.playouts}")
        if int(self.max_steps) < 1:
            raise ValueError(f"max_steps must be >= 1, got {self.max_steps}")
        if self.criterion not in CRITERIA:
            raise ValueError(f"criterion must be one of {CRITERIA}, got {self.criterion!r}")
        _rollout_policy(self.rollout)

    @property
    def rollout_policy(self) -> int:
        return _rollout_policy(self.rollout)
