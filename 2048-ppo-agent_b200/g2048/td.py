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

``NTupleTDLearner`` learns an n-tuple network (``g2048.NTupleNetwork``) the same way, through
``g2048_ntuple_td_train``: V in place of H, and the update at every placement of the previous afterstate.
``NTupleTCLearner`` learns it by temporal coherence (``g2048_ntuple_tc_train``): the same step, with every weight's
step scaled by |E| / A, its running sum of errors over the sum of their absolute values.  A multi-stage network
(``NTupleNetwork.staged``) is learned by the staged entry points, all its stages in one launch; a single-stage network
takes the unstaged ones.

Both n-tuple learners take ``lam`` and ``horizon`` (h, 1..8) for delayed TD(lambda) / TC(lambda)
(``g2048_ntuple_lambda_td_train`` / ``_tc_train``): every env keeps its last h afterstates and their errors, and an
afterstate is updated h - 1 steps late with the lambda-weighted sum of its h errors (each computed with the weights of
its own step).  ``horizon=1`` (the default) is TD(0) / TC exactly, through the entry points above.  On the 4x6
network TC(lambda) learned better players than TC and TD(0), and TD(lambda) worse ones than TD(0) after 40 000 steps
(profiles/README.md, round 11):

    learner = g2048.NTupleTCLearner(0, batch_size=1 << 16, lam=0.5, horizon=3)

With ``carousel=True`` a multi-stage network is learned with carousel shaping (``g2048_ntuple_carousel_td_train`` /
``_tc_train``, any horizon): an episode that ends restarts, in turn, at the opening or from a board at which an
earlier episode entered stage 1, 2, ..., so that the later stages' tables see a fair share of the training.  The
summary of ``train`` then also counts those shaped episodes (``shaped_episodes``, ``shaped_env_steps``); the other
entries count only the episodes that began at the opening (profiles/README.md, round 12):

    net = g2048.NTupleNetwork.staged(g2048.NTupleNetwork.four_six(), (13,))
    learner = g2048.NTupleTCLearner(0, batch_size=1 << 16, network=net, lam=0.5, horizon=3, carousel=True)
"""
from __future__ import annotations

import math

import numpy as np
import torch

from . import _native as N
from . import engine as E
from .keys import KeyChain
from .ntuple import MAX_HORIZON, NTupleNetwork, check_placements, _check_weights

# the step size of the round-7 sweep on one B200 whose greedy player scored best (profiles/README.md, round 7)
DEFAULT_ALPHA = 0.1
# the step size of the round-8 sweep on one B200 whose greedy 4x6 player scored best (profiles/README.md, round 8)
DEFAULT_NTUPLE_ALPHA = 0.02
# round 9: TD's default, so that no TC step is larger than the TD step it starts as (beta <= 1, and from E = A = 0 a TC
# step is a TD step with the same alpha; profiles/README.md, round 9)
DEFAULT_NTUPLE_TC_ALPHA = DEFAULT_NTUPLE_ALPHA
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


def _check_lam(lam) -> float:
    lam = float(lam)
    if not (math.isfinite(lam) and 0.0 <= lam <= 1.0):
        raise ValueError(f"lam must be finite and in [0, 1], got {lam}")
    return lam


def _check_horizon(horizon) -> int:
    try:
        h = int(horizon)
    except (TypeError, ValueError, OverflowError):
        h = None
    if h is None or isinstance(horizon, bool) or h != horizon or not 1 <= h <= MAX_HORIZON:
        raise ValueError(f"horizon must be an integer in [1, {MAX_HORIZON}], got {horizon!r}")
    return h


def _check_ring(ring, shape, dtype, name) -> torch.Tensor:
    """A checkpoint's window ring: a (h, n) tensor of the given dtype, or ValueError."""
    if not isinstance(ring, torch.Tensor) or ring.dtype != dtype or tuple(ring.shape) != shape:
        got = (ring.dtype, tuple(ring.shape)) if isinstance(ring, torch.Tensor) else type(ring).__name__
        raise ValueError(f"{name} must be a {dtype} tensor of shape {shape}, got {got}")
    return ring


def _check_start_stage(t, n: int, n_stages: int) -> torch.Tensor:
    """A checkpoint's start_stage: an int32 (n,) tensor with values in [0, n_stages), or ValueError."""
    if not isinstance(t, torch.Tensor) or t.dtype != torch.int32 or tuple(t.shape) != (n,):
        got = (t.dtype, tuple(t.shape)) if isinstance(t, torch.Tensor) else type(t).__name__
        raise ValueError(f"start_stage must be a torch.int32 tensor of shape ({n},), got {got}")
    if bool(((t < 0) | (t >= n_stages)).any()):
        raise ValueError(f"start_stage values must lie in [0, {n_stages})")
    return t


def _resolved(device) -> torch.device:
    """``device`` with the current CUDA device filled in for a bare "cuda"."""
    device = torch.device(device)
    if device.type == "cuda" and device.index is None:
        device = torch.device("cuda", torch.cuda.current_device())
    return device


class _BatchTDLearner:
    """What the two learners share: ``batch_size`` envs (1 .. 2^20) with their afterstates, scores and lengths, the key
    chain of ``init_seed`` (sub key 0 initialises the envs, every step consumes one more), ``train`` and the
    checkpoint.  A subclass holds the value function and launches the steps (``_launch``); its checkpoint entries
    come from ``_values_state`` and are checked by ``_check_values_state`` before a load changes anything."""

    def _check_common(self, batch_size, alpha) -> tuple[int, float]:
        batch_size = int(batch_size)
        if not 1 <= batch_size <= MAX_BATCH:
            raise ValueError(f"batch_size must be in [1, 2^20], got {batch_size}")
        return batch_size, _check_alpha(alpha)

    def _start(self, rng_mode, device) -> None:
        """rng_mode and device, after the arguments are checked and before anything is allocated."""
        self.rng_mode = E.resolve_rng_mode(rng_mode)
        self.device = N.require_cuda() if device is None else torch.device(device)

    def _init_envs(self, init_seed) -> None:
        self.chain = KeyChain(init_seed, self.rng_mode, self.device)
        n = self.batch_size
        self.boards, _ = E.env_init(self.chain.peek(1)[0], n, 0, n, self.rng_mode)
        self.chain.consume(1)
        self.after = torch.zeros(n, dtype=torch.int64, device=self.device)
        self.scores = torch.zeros(n, dtype=torch.int32, device=self.device)
        self.lengths = torch.zeros(n, dtype=torch.int32, device=self.device)
        self.steps = 0

    def _launch(self, subs: torch.Tensor, stats: torch.Tensor) -> None:
        raise NotImplementedError

    def train(self, n_steps: int) -> dict:
        """``n_steps`` learning steps in one launch; returns the summary of the episodes that ended in them."""
        n_steps = int(n_steps)
        if n_steps < 0:
            raise ValueError(f"n_steps must be >= 0, got {n_steps}")
        stats = torch.zeros(N.PLAY_STATS_WORDS, dtype=torch.int64, device=self.device)
        if n_steps:
            subs = self.chain.peek(n_steps)
            self._launch(subs, stats)
            self.chain.consume(n_steps)
            self.steps += n_steps
        return self._summary(stats)

    def _summary(self, stats: torch.Tensor) -> dict:
        return E.play_stats_dict(stats)

    # -- checkpointing: key chain, env state and the value function ----------------------------------------------
    def _values_state(self) -> dict:
        raise NotImplementedError

    def _check_values_state(self, state: dict):
        raise NotImplementedError

    def _load_values(self, values) -> None:
        raise NotImplementedError

    def state_dict(self) -> dict:
        out = {"key": [int(w) for w in self.chain.key], "position": int(self.chain.position), "rng_mode": int(self.rng_mode),
               "batch_size": self.batch_size, "alpha": self.alpha, "steps": self.steps}
        out.update(self._values_state())
        out.update({"boards": self.boards.cpu().clone(), "after": self.after.cpu().clone(),
                    "scores": self.scores.cpu().clone(), "lengths": self.lengths.cpu().clone()})
        return out

    def load_state_dict(self, state: dict) -> None:
        if int(state["batch_size"]) != self.batch_size or state["boards"].shape[0] != self.batch_size:
            raise ValueError("checkpoint was written for a different batch size")
        alpha = _check_alpha(state["alpha"])
        values = self._check_values_state(state)
        if int(state["rng_mode"]) not in (E.RNG_ORIGINAL, E.RNG_PARTITIONABLE):
            raise ValueError(f"checkpoint has an unknown rng_mode {state['rng_mode']!r}")
        self.alpha = alpha
        self.rng_mode = int(state["rng_mode"])
        self.chain = KeyChain(np.asarray(state["key"], dtype=np.uint32), self.rng_mode, self.device)
        self.chain._base_pos = int(state["position"])
        self.steps = int(state["steps"])
        self._load_values(values)
        for name in ("boards", "after", "scores", "lengths"):
            getattr(self, name).copy_(state[name].to(self.device))


class TDLearner(_BatchTDLearner):
    """Learns the row table by synchronous batched TD(0) over ``batch_size`` envs (1 .. 2^20).

    ``table``: the float32 (65536,) device tensor being learned (zeros, or a copy of the given finite table).
    ``train(n_steps)`` makes ``n_steps`` steps and returns the summary of the episodes that ended in them
    (``engine.play_stats_dict`` form).  Keys come from the runner's chain of ``init_seed``: sub key 0 initialises the
    envs, and every step consumes one more.  ``state_dict`` / ``load_state_dict`` resume a run bit for bit."""

    def __init__(self, init_seed: int, batch_size: int, alpha: float = DEFAULT_ALPHA, table=None, rng_mode=None,
                 device=None):
        self.batch_size, self.alpha = self._check_common(batch_size, alpha)
        if table is not None:
            table = _check_table(table)
        self._start(rng_mode, device)
        if table is None:
            self.table = torch.zeros(65536, dtype=torch.float32, device=self.device)
        else:
            self.table = table.to(self.device).clone()
        self._init_envs(init_seed)
        self._scratch = E.td_scratch(self.device)

    def _launch(self, subs, stats) -> None:
        E.td_train(self.boards, self.after, self.scores, self.lengths, self.table, self.alpha, subs, self.rng_mode,
                   self._scratch, stats)

    def _values_state(self) -> dict:
        return {"table": self.table.cpu().clone()}

    def _check_values_state(self, state):
        return _check_table(state["table"])

    def _load_values(self, table) -> None:
        self.table.copy_(table.to(self.device))


class NTupleTDLearner(_BatchTDLearner):
    """Learns an n-tuple network by synchronous batched TD(0) over ``batch_size`` envs (1 .. 2^20), as ``TDLearner``
    learns the row table: the same greedy move, fixed-point update, key chain and statistics.

    ``network``: the ``NTupleNetwork`` whose ``weights`` are learned in place (default: a zero ``four_six()``).
    ``lam`` / ``horizon``: delayed TD(lambda) over a window of each env's last ``horizon`` afterstates (1..8;
    ``batch_size * horizon <= 2^20``), held in ``hist_after`` / ``hist_delta`` ((horizon, batch_size) device tensors)
    when ``horizon > 1``.  ``horizon=1`` is TD(0), whatever ``lam``.
    ``state_dict`` / ``load_state_dict`` resume a run bit for bit; the checkpoint holds the placements and the stages,
    and a load whose placements, n_weights or stages differ from the learner's network is rejected before anything
    changes (a checkpoint without stages is a single-stage network's).  With ``horizon > 1`` it also holds ``lam``,
    ``horizon`` and both rings; a load with another horizon or with rings of the wrong shape or dtype is rejected, and
    a checkpoint without them is a ``horizon=1`` learner's.
    ``carousel``: carousel shaping of a multi-stage network (a single-stage one is a ValueError), through
    ``g2048_ntuple_carousel_td_train`` for every horizon.  The learner then holds ``start_stage`` (int32 (batch_size,))
    and ``stage_pool`` (int64 (S - 1, batch_size)), zeros at construction, and its checkpoint holds ``carousel`` and
    both; a load with another carousel setting, arrays of the wrong shape or dtype, or a start stage outside [0, S)
    is rejected before anything changes."""

    def __init__(self, init_seed: int, batch_size: int, network: NTupleNetwork | None = None,
                 alpha: float = DEFAULT_NTUPLE_ALPHA, rng_mode=None, device=None, lam: float = 0.0, horizon: int = 1,
                 carousel: bool = False):
        self.batch_size, self.alpha = self._check_common(batch_size, alpha)
        self.lam = _check_lam(lam)
        self.horizon = _check_horizon(horizon)
        if self.batch_size * self.horizon > MAX_BATCH:
            raise ValueError(f"batch_size * horizon must be <= 2^20, got {self.batch_size} * {self.horizon}")
        if network is not None and not isinstance(network, NTupleNetwork):
            raise ValueError("network must be an NTupleNetwork")
        if not isinstance(carousel, (bool, np.bool_)):
            raise ValueError(f"carousel must be a bool, got {carousel!r}")
        self.carousel = bool(carousel)
        if self.carousel and (network is None or network.n_stages < 2):
            raise ValueError("carousel shaping needs a multi-stage network (NTupleNetwork.staged)")
        self._start(rng_mode, device)
        self.network = NTupleNetwork.four_six(device=self.device) if network is None else network
        if _resolved(self.network.weights.device) != _resolved(self.device):
            raise ValueError(f"the network's weights are on {self.network.weights.device}, the learner runs on {self.device}")
        self._init_envs(init_seed)
        if self.horizon > 1:
            shape = (self.horizon, self.batch_size)
            self.hist_after = torch.zeros(shape, dtype=torch.int64, device=self.device)
            self.hist_delta = torch.zeros(shape, dtype=torch.float32, device=self.device)
        if self.carousel:
            self.start_stage = torch.zeros(self.batch_size, dtype=torch.int32, device=self.device)
            self.stage_pool = torch.zeros((self.network.n_stages - 1, self.batch_size), dtype=torch.int64,
                                          device=self.device)
        self._scratch = self._new_scratch()

    def _new_scratch(self) -> torch.Tensor:
        if self.carousel:
            return E.ntuple_carousel_scratch(self.batch_size, self.horizon, self.network.placements,
                                             self.network.n_weights, False, self.device)
        return E.ntuple_td_scratch(self.batch_size * self.horizon, self.network.placements, self.network.n_weights,
                                   self.device)

    def _rings(self) -> tuple:
        return (self.hist_after, self.hist_delta) if self.horizon > 1 else (None, None)

    def _summary(self, stats: torch.Tensor) -> dict:
        out = E.play_stats_dict(stats)
        if self.carousel:
            words = stats.cpu()
            out.update(shaped_episodes=int(words[12]), shaped_env_steps=int(words[13]))
        return out

    @property
    def weights(self) -> torch.Tensor:
        return self.network.weights

    def _launch(self, subs, stats) -> None:
        net = self.network
        if self.carousel:
            E.ntuple_carousel_td_train(self.boards, self.after, self.scores, self.lengths, net.placements, net.weights,
                                       self.alpha, self.lam, *self._rings(), self.start_stage, self.stage_pool, subs,
                                       self.rng_mode, self._scratch, stats, stages=net.stages)
            return
        if self.horizon > 1:
            E.ntuple_lambda_td_train(self.boards, self.after, self.scores, self.lengths, net.placements, net.weights,
                                     self.alpha, self.lam, self.hist_after, self.hist_delta, subs, self.rng_mode,
                                     self._scratch, stats, stages=net.stages)
            return
        E.ntuple_td_train(self.boards, self.after, self.scores, self.lengths, net.placements, net.weights, self.alpha,
                          subs, self.rng_mode, self._scratch, stats, stages=net.stages)

    def _values_state(self) -> dict:
        net = self.network
        out = {"placements": net.placements.copy(), "n_weights": net.n_weights,
               "stage_thresholds": list(net.stage_thresholds), "stage_stride": net.stage_stride,
               "weights": net.weights.cpu().clone()}
        if self.horizon > 1:
            out.update({"lam": self.lam, "horizon": self.horizon, "hist_after": self.hist_after.cpu().clone(),
                        "hist_delta": self.hist_delta.cpu().clone()})
        if self.carousel:
            out.update({"carousel": True, "start_stage": self.start_stage.cpu().clone(),
                        "stage_pool": self.stage_pool.cpu().clone()})
        return out

    def _check_carousel_state(self, state):
        """The checkpoint's carousel arrays: None without carousel, else (start_stage, stage_pool); ValueError if they
        do not fit this learner."""
        carousel = state.get("carousel", False)
        if not isinstance(carousel, (bool, np.bool_)) or bool(carousel) != self.carousel:
            raise ValueError(f"checkpoint was written with carousel={carousel!r}, this learner has "
                             f"carousel={self.carousel}")
        if not self.carousel:
            return None
        S = self.network.n_stages
        start_stage = _check_start_stage(state.get("start_stage"), self.batch_size, S)
        return start_stage, _check_ring(state.get("stage_pool"), (S - 1, self.batch_size), torch.int64, "stage_pool")

    def _check_window_state(self, state):
        """The checkpoint's window: None for horizon 1, else (lam, hist_after, hist_delta); ValueError if it does not
        fit this learner."""
        horizon = _check_horizon(state.get("horizon", 1))
        if horizon != self.horizon:
            raise ValueError(f"checkpoint was written with horizon {horizon}, this learner's is {self.horizon}")
        if self.horizon == 1:
            return None
        if "lam" not in state:
            raise ValueError("checkpoint has no lam")
        lam = _check_lam(state["lam"])
        shape = (self.horizon, self.batch_size)
        return (lam, _check_ring(state.get("hist_after"), shape, torch.int64, "hist_after"),
                _check_ring(state.get("hist_delta"), shape, torch.float32, "hist_delta"))

    def _check_values_state(self, state):
        net = self.network
        if int(state["n_weights"]) != net.n_weights:
            raise ValueError("checkpoint was written for a network with a different n_weights")
        placements = check_placements(state["placements"], net.n_weights)
        if not np.array_equal(placements, net.placements):
            raise ValueError("checkpoint was written for a network with different placements")
        thresholds = tuple(int(t) for t in state.get("stage_thresholds", ()))
        if thresholds != net.stage_thresholds or int(state.get("stage_stride", 0)) != net.stage_stride:
            raise ValueError("checkpoint was written for a network with different stages")
        window = self._check_window_state(state)
        carousel = self._check_carousel_state(state)
        return _check_weights(state["weights"], net.n_weights), window, carousel

    def _load_values(self, values) -> None:
        weights, window, carousel = values
        self.network.weights.copy_(weights.to(self.device))
        if window is not None:
            self.lam = window[0]
            self.hist_after.copy_(window[1].to(self.device))
            self.hist_delta.copy_(window[2].to(self.device))
        if carousel is not None:
            self.start_stage.copy_(carousel[0].to(self.device))
            self.stage_pool.copy_(carousel[1].to(self.device))


def _check_sums(sums, n_weights: int, name: str) -> torch.Tensor:
    """A checkpoint's E or A: float64 (n_weights,) finite values as a tensor, or ValueError."""
    if sums is None:
        raise ValueError(f"checkpoint has no {name} (it was not written by NTupleTCLearner)")
    t = sums.detach() if isinstance(sums, torch.Tensor) else torch.from_numpy(np.asarray(sums))
    if t.dtype != torch.float64 or tuple(t.shape) != (n_weights,):
        raise ValueError(f"{name} must be a float64 array of n_weights = {n_weights} values, got {t.dtype} {tuple(t.shape)}")
    if not bool(torch.isfinite(t).all()):
        raise ValueError(f"{name} must be finite")
    return t


class NTupleTCLearner(NTupleTDLearner):
    """Learns an n-tuple network by synchronous batched temporal coherence (TC) learning: ``NTupleTDLearner``'s
    greedy move, fixed-point errors, key chain and statistics, with every weight's step scaled by
    ``beta = |E| / A`` (1 while A is 0).  ``err_sum`` (E) and ``abs_err_sum`` (A) are the float64 (n_weights,) device
    sums of each weight's errors and of their absolute values, zero at construction; weights whose errors keep one
    sign keep a large step, weights whose errors cancel stop moving (g2048_ntuple_tc_train, include/g2048.h).

    ``network`` may hold weights learned before (for example by ``NTupleTDLearner``): TC starts from them with
    E = A = 0.  ``lam`` / ``horizon``: delayed TC(lambda), the window of ``NTupleTDLearner``; ``carousel``: its carousel
    shaping (``g2048_ntuple_carousel_tc_train``).  ``state_dict`` /
    ``load_state_dict`` resume a run bit for bit, E and A included."""

    def __init__(self, init_seed: int, batch_size: int, network: NTupleNetwork | None = None,
                 alpha: float = DEFAULT_NTUPLE_TC_ALPHA, rng_mode=None, device=None, lam: float = 0.0,
                 horizon: int = 1, carousel: bool = False):
        super().__init__(init_seed, batch_size, network=network, alpha=alpha, rng_mode=rng_mode, device=device,
                         lam=lam, horizon=horizon, carousel=carousel)
        n_weights = self.network.n_weights
        self.err_sum = torch.zeros(n_weights, dtype=torch.float64, device=self.device)
        self.abs_err_sum = torch.zeros(n_weights, dtype=torch.float64, device=self.device)

    def _new_scratch(self) -> torch.Tensor:
        if self.carousel:
            return E.ntuple_carousel_scratch(self.batch_size, self.horizon, self.network.placements,
                                             self.network.n_weights, True, self.device)
        return E.ntuple_tc_scratch(self.batch_size * self.horizon, self.network.placements, self.network.n_weights,
                                   self.device)

    def _launch(self, subs, stats) -> None:
        net = self.network
        if self.carousel:
            E.ntuple_carousel_tc_train(self.boards, self.after, self.scores, self.lengths, net.placements, net.weights,
                                       self.err_sum, self.abs_err_sum, self.alpha, self.lam, *self._rings(),
                                       self.start_stage, self.stage_pool, subs, self.rng_mode, self._scratch, stats,
                                       stages=net.stages)
            return
        if self.horizon > 1:
            E.ntuple_lambda_tc_train(self.boards, self.after, self.scores, self.lengths, net.placements, net.weights,
                                     self.err_sum, self.abs_err_sum, self.alpha, self.lam, self.hist_after,
                                     self.hist_delta, subs, self.rng_mode, self._scratch, stats, stages=net.stages)
            return
        E.ntuple_tc_train(self.boards, self.after, self.scores, self.lengths, net.placements, net.weights,
                          self.err_sum, self.abs_err_sum, self.alpha, subs, self.rng_mode, self._scratch, stats,
                          stages=net.stages)

    def _values_state(self) -> dict:
        out = super()._values_state()
        out.update({"err_sum": self.err_sum.cpu().clone(), "abs_err_sum": self.abs_err_sum.cpu().clone()})
        return out

    def _check_values_state(self, state):
        base = super()._check_values_state(state)  # (weights, window)
        n_weights = self.network.n_weights
        err_sum = _check_sums(state.get("err_sum"), n_weights, "err_sum")
        abs_err_sum = _check_sums(state.get("abs_err_sum"), n_weights, "abs_err_sum")
        if bool((abs_err_sum < 0).any()):
            raise ValueError("abs_err_sum must be >= 0")
        return base, err_sum, abs_err_sum

    def _load_values(self, values) -> None:
        base, err_sum, abs_err_sum = values
        super()._load_values(base)
        self.err_sum.copy_(err_sum.to(self.device))
        self.abs_err_sum.copy_(abs_err_sum.to(self.device))
