"""Depth-limited expectimax values of given boards over a row heuristic, and the expectimax player built on them.

    res = g2048.expectimax_values(boards, depth=3)                        # (n, 4) Q values, NaN where illegal
    res.best_action()

    runner = g2048.BatchRunner(0, g2048.ExpectimaxPolicy(depth=2))
    out = runner.run_eval_batch(1024)                                     # every move chosen by expectimax

The search runs in one launch of ``g2048_expectimax_values``: max nodes over the legal moves, chance nodes over every
empty cell with a 2 (probability 0.9) or a 4 (0.1), and at depth ``depth`` (counted in moves) the heuristic
``H(b) = sum of T[row] over the 4 rows and 4 columns``.  A move's value adds ``reward_weight`` times its merge reward.
All arithmetic is float32 in a fixed order (include/g2048.h), so the values are bit-exact and a game is deterministic
given the spawns.  With ``network=`` (a ``g2048.NTupleNetwork``) the leaves are the network's value V instead of H
(``g2048_expectimax_values_ntuple``), with the same tree and float order; a multi-stage network takes each leaf's
stage from the leaf board (``g2048_expectimax_values_ntuple_staged``).
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np
import torch

from . import _native as N
from . import engine as E

_DEFAULT_TABLES = {}  # device -> the default row table on it


def default_row_table_numpy() -> np.ndarray:
    """The default row heuristic (nneonneo/2048-ai's), computed in float64 and rounded once to float32.  For a row with
    exponents l[0..3] (nibble k = column k): empty = zero cells; merges = over the nonzero cells in order, every run of
    m + 1 equal neighbours adds 1 + m; sum = sum of l^3.5; mono_left = sum over i of [l[i-1] > l[i]] (l[i-1]^4 - l[i]^4),
    mono_right the same for l[i-1] < l[i];  T = 200000 + 270 empty + 700 merges - 47 min(mono_left, mono_right) - 11 sum."""
    rows = np.arange(65536, dtype=np.int64)
    ls = [((rows >> (4 * k)) & 15).astype(np.float64) for k in range(4)]
    empty = sum((x == 0).astype(np.float64) for x in ls)
    merges = np.zeros(65536, np.float64)
    prev = np.zeros(65536, np.float64)
    counter = np.zeros(65536, np.float64)
    for x in ls:
        nz = x != 0
        same = nz & (prev == x)
        close = nz & ~same & (counter > 0)
        merges += np.where(close, 1 + counter, 0.0)
        counter = np.where(same, counter + 1, np.where(close, 0.0, counter))
        prev = np.where(nz, x, prev)
    merges += np.where(counter > 0, 1 + counter, 0.0)
    total = sum(x ** 3.5 for x in ls)
    mono_left = sum(np.where(ls[i - 1] > ls[i], ls[i - 1] ** 4 - ls[i] ** 4, 0.0) for i in range(1, 4))
    mono_right = sum(np.where(ls[i - 1] < ls[i], ls[i] ** 4 - ls[i - 1] ** 4, 0.0) for i in range(1, 4))
    t = 200000.0 + 270.0 * empty + 700.0 * merges - 47.0 * np.minimum(mono_left, mono_right) - 11.0 * total
    return t.astype(np.float32)


def default_row_values(device=None) -> torch.Tensor:
    """The default row table as a float32 device tensor of 65 536 values, computed once per device."""
    device = N.require_cuda() if device is None else torch.device(device)
    if device.type == "cuda" and device.index is None:
        device = torch.device("cuda", torch.cuda.current_device())
    t = _DEFAULT_TABLES.get(device)
    if t is None:
        t = torch.from_numpy(default_row_table_numpy()).to(device)
        _DEFAULT_TABLES[device] = t
    return t


def _check(depth: int, row_values, network=None) -> None:
    if not 1 <= int(depth) <= 4:
        raise ValueError(f"depth must be in 1..4, got {depth}")
    if row_values is not None and (not isinstance(row_values, torch.Tensor) or row_values.numel() != 65536):
        raise ValueError("row_values must be a tensor of 65536 float32 values")
    if network is not None:
        from .ntuple import NTupleNetwork

        if not isinstance(network, NTupleNetwork):
            raise ValueError("network must be an NTupleNetwork")
        if row_values is not None:
            raise ValueError("pass row_values or network, not both")


def best_actions(q: torch.Tensor) -> torch.Tensor:
    """(n,) int64: per board the legal action with the largest value, ties to the lowest action index; 0 for a board
    without a legal action."""
    return torch.where(torch.isnan(q), torch.full_like(q, -float("inf")), q).argmax(dim=1)


class ExpectimaxValues:
    """Result of ``expectimax_values``: ``q`` (n, 4) float32 (NaN where the action is illegal), ``legal`` (n, 4) bool,
    and ``counters`` (2 int64: leaves, chance nodes of this search)."""

    def __init__(self, q: torch.Tensor, counters: torch.Tensor):
        self.q = q
        self.counters = counters

    @property
    def legal(self) -> torch.Tensor:
        return ~torch.isnan(self.q)

    @property
    def leaves(self) -> int:
        return int(self.counters[0].item())

    @property
    def chance_nodes(self) -> int:
        return int(self.counters[1].item())

    def best_action(self) -> torch.Tensor:
        """(n,) int64 arg-max over the legal actions, ties to the lowest index; 0 for a board without a legal action."""
        return best_actions(self.q)


def _table_on(row_values, device) -> torch.Tensor:
    if row_values is None:
        return default_row_values(device)
    return row_values.to(device=device, dtype=torch.float32).contiguous()


def expectimax_values(boards, depth: int = 2, row_values=None, reward_weight: float = 0.0, device=None,
                      network=None) -> ExpectimaxValues:
    """Depth-``depth`` expectimax (1 <= depth <= 4, counted in moves) of every (board, action).  ``boards``: (n,) int64
    bitboards (a tensor, or anything numpy reads as such); ``row_values``: the row table T (65 536 values, default
    ``default_row_values()``); ``reward_weight``: w, the weight of a move's merge reward; ``network``: an
    ``NTupleNetwork`` whose V replaces H at the leaves (not together with ``row_values``)."""
    _check(depth, row_values, network)
    if isinstance(boards, torch.Tensor):
        device = boards.device if device is None else torch.device(device)
        boards = boards.to(device=device, dtype=torch.int64).contiguous()
    else:
        device = N.require_cuda() if device is None else torch.device(device)
        boards = torch.from_numpy(np.ascontiguousarray(np.asarray(boards, dtype=np.uint64).reshape(-1)).view(np.int64)).to(device)
    counters = torch.zeros(2, dtype=torch.int64, device=device)
    if network is not None:
        q = E.expectimax_values_ntuple(boards, int(depth), network.placements, network.weights_on(device),
                                       float(reward_weight), counters, stages=network.stages)
    else:
        q = E.expectimax_values(boards, int(depth), _table_on(row_values, device), float(reward_weight), counters)
    return ExpectimaxValues(q, counters)


@dataclass(frozen=True, eq=False)  # eq=False: the table is a tensor
class ExpectimaxPolicy:
    """The expectimax player: at every move the legal action with the largest depth-``depth`` expectimax value over
    ``row_values`` (default: ``default_row_values()``) and ``reward_weight``.  An act_fn for
    ``BatchRunner.run_eval_batch``: per move one search over the envs still alive, then ``g2048_env_step`` with that
    move's step sub key.  The act sub key is not used, so a game is a function of (seed, batch size, depth, table,
    reward_weight, rng_mode).  With ``network`` (an ``NTupleNetwork``, not together with ``row_values``) the leaves
    are the network's V."""

    depth: int = 2
    row_values: torch.Tensor | None = None
    reward_weight: float = 0.0
    network: object | None = None

    def __post_init__(self):
        _check(self.depth, self.row_values, self.network)

    def table(self, device) -> torch.Tensor:
        return _table_on(self.row_values, device)
