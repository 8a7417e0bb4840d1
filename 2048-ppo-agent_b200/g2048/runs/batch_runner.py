"""BatchRunner -- same surface as the reference's src/runs/batch_runner.py:10-195, with the
host `while` loop (three jitted dispatches and one blocking readback per step) replaced by
libg2048 kernels that keep every env in registers.

    runner = BatchRunner(init_seed=0, act_fn=act_randomly)
    obs, actions, masks, log_probs, values, rewards, terminations = runner.run_actions_batch(1024)

Which kernels run depends on the policy handed in as ``act_fn``:
  * ``act_randomly`` / ``act_drul`` (objects with ``policy_id``): the fused lock-step kernel
    ``g2048_rollout_steps`` records whole chunks of steps per launch; ``run_stats_batch`` uses the
    persistent ``g2048_play`` kernel when only per-episode results are wanted.
  * ``TorchActionFunction``: one network forward (PyTorch) + one ``g2048_policy_step`` launch per
    step (mask, categorical sample, log-prob, env step and record write fused).
  * any other callable ``(keys (B,2), obs (B,4,4,31) bool, mask (B,4) bool) -> (action, log_prob,
    value)`` on torch tensors: per-step ``g2048_split_keys`` / ``g2048_env_step`` launches around it.

Differences from the reference that a caller can see (SURVEY section 5, "defects"):
  * tensors are torch / numpy instead of jax arrays, keys are uint32 word pairs;
  * ``log_probs`` / ``values`` are returned as ``None`` when the policy yields ``None`` (the
    reference's np.stack on a list of None raises);
  * ``rng_mode`` selects jax's Threefry counter layout (default: partitionable, as in jax 0.5.3).
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Callable

import numpy as np
import torch

from .. import _native as N
from .. import engine as E
from ..expectimax import ExpectimaxPolicy
from ..expectimax import best_actions as expectimax_best_actions
from ..keys import KeyChain
from ..playouts import MonteCarloPolicy, best_actions
from ..state import State

ENV_ID = "2048"
CHUNK_STEPS = 64
GRAPH_SYNC_STEPS = 8  # graph replays between `all done` tests; divides CHUNK_STEPS
NET_SYNC_STEPS = 8    # eager network-policy loop: steps per chunk; the host looks at the device's done counter once per chunk


@dataclass
class PackedRollout:
    """A finished run in the engine's own format: time-major (T, B) device records.

    boards  int64  pre-step bitboards          meta   uint8  action | mask << 2 | done << 6
    rewards float32 post-step                  log_probs / values float32 or None
    final_boards / final_status: the state after the last step.
    """

    boards: torch.Tensor
    meta: torch.Tensor
    rewards: torch.Tensor
    log_probs: torch.Tensor | None
    values: torch.Tensor | None
    final_boards: torch.Tensor
    final_status: torch.Tensor
    t_steps: int
    batch_size: int
    env_steps: int  # steps taken by live envs (what the reference's RolloutBuffer keeps)

    def lengths(self) -> torch.Tensor:
        return E.episode_lengths(self.meta, self.t_steps, self.batch_size)


@dataclass
class FlatRollout:
    """A finished run of a built-in policy as the env-major ragged buffer ``RolloutBuffer`` keeps: the steps
    0..first_done of env 0, then those of env 1, ... (``offsets[e]`` = first flat index of env e, ``lengths[e]`` its
    number of steps).  Produced by ONE launch of the recording play kernel + one compaction kernel; identical, bit
    for bit, to ``RolloutBuffer.store_packed(run_packed_batch(...))``.

    boards int64 pre-step bitboards, meta uint8 (action | mask << 2 | done << 6), rewards / log_probs / values float32
    (log_probs of act_drul and all values are zero, as ``store_packed`` stores them).
    """

    boards: torch.Tensor
    meta: torch.Tensor
    rewards: torch.Tensor
    log_probs: torch.Tensor
    values: torch.Tensor
    lengths: torch.Tensor
    offsets: torch.Tensor
    final_boards: torch.Tensor
    scores: torch.Tensor
    max_rewards: torch.Tensor  # per env: max_t reward (the trainer's "episode reward")
    t_steps: int  # loop steps of the reference's run = the longest episode (over all shards)
    batch_size: int
    env_steps: int
    summary: dict


class BatchRunner:
    """Runs batches of 2048 envs with an action function (reference: batch_runner.py:10-37)."""

    def __init__(self, init_seed: int, act_fn: Callable = None, rng_mode=None, device=None,
                 shard: tuple[int, int] | None = None, cuda_graph: bool = False, compact_live: bool = False,
                 pinned_outputs: bool = False):
        """
        init_seed : seed of the runner's key chain (jax.random.key(seed), batch_runner.py:32)
        act_fn    : policy, see the module docstring; may be set later through ``.act_fn``
        rng_mode  : None / "partitionable" / "original"
        shard     : (rank, world) -- this process owns a contiguous slice of every batch; env
                    indices stay global, so the union over ranks equals the single-GPU run.
        cuda_graph: with a ``TorchActionFunction`` whose network runs on this GPU, capture one loop step
                    (observation -> network forward -> sample + env.step + record) as a CUDA graph and replay it,
                    with one host synchronisation per CHUNK_STEPS steps instead of one per step (SURVEY 8f
                    rank 3).  Same records as the eager loop.
        compact_live: ``run_packed_batch`` steps only the envs that are still alive -- with a ``TorchActionFunction`` only
                    they go through the network, with the built-in policies the recording kernel's work follows the
                    live env-steps (the reference pushes the finished ones through it until the last env ends,
                    batch_runner.py:117-136 -- about two thirds of the rows of a run to termination).  Env state, RNG
                    counters and record slots stay per env, so a live env's trajectory does not depend on who else
                    is alive; records of steps after an env's end are zero instead of repeating its frozen state
                    (``RolloutBuffer`` never reads them).  The reference-format calls ignore the flag.
        pinned_outputs: the numpy arrays ``run_actions_batch`` returns are page-locked memory (torch's caching host
                    allocator) written by one transfer each, instead of ordinary arrays filled by a second, page-faulting
                    copy: C1's 133 MB of outputs in 4 instead of 10 ms.  Off by default: page-locked memory is a
                    finite resource, and a caller that keeps many batches alive would hoard it.
        """
        self.device = N.require_cuda() if device is None else torch.device(device)
        self.rng_mode = E.resolve_rng_mode(rng_mode)
        self.chain = KeyChain(init_seed, self.rng_mode, self.device)
        self.shard = shard
        self._act_fn = act_fn
        self.cuda_graph = cuda_graph
        self.compact_live = compact_live
        self.pinned_outputs = pinned_outputs
        self._graphs = {}  # (batch_size, lo, n, steps, auto_reset) -> captured step of the current act_fn
        self._mean_steps = {}  # policy id -> mean episode length of the last recorded batch (sizes the next arena)

    # -- reference surface ---------------------------------------------------------------------
    @property
    def key(self) -> np.ndarray:
        """The chain key as two uint32 words (the reference's ``self.key``)."""
        return self.chain.key

    @property
    def act_fn(self):
        return self._act_fn

    @act_fn.setter
    def act_fn(self, act_fn: Callable):
        self._act_fn = act_fn

    # -- checkpointing (SURVEY 8f rank 4: the reference saves no env / RNG state, src/ppo/ppo_trainer.py:511-530) --
    def state_dict(self) -> dict:
        """Everything needed to continue the key chain exactly where it stands: two uint32 words."""
        return {"key": [int(w) for w in self.chain.key], "position": int(self.chain.position), "rng_mode": int(self.rng_mode)}

    def load_state_dict(self, state: dict) -> None:
        self.rng_mode = int(state["rng_mode"])
        self.chain = KeyChain(np.asarray(state["key"], dtype=np.uint32), self.rng_mode, self.device)
        self.chain._base_pos = int(state.get("position", 0))

    def run_actions_batch(self, batch_size: int):
        """-> (observations (B,T,4,4,31) bool, actions (B,T) int32, action_masks (B,T,4) bool,
        log_probs (B,T) f32 | None, values (B,T) f32 | None, rewards (B,T) f32, terminations (B,T) bool),
        numpy arrays stacked like batch_runner.py:138-154."""
        ro = self._run(batch_size, full_records=True)
        t, b = ro.t_steps, ro.batch_size
        obs = E.expand_obs(ro.boards, torch.bool, rows=t, n_cols=b)
        un = E.unpack_records(ro.meta, ro.rewards, ro.log_probs, ro.values, t, b)
        to_np = lambda x: None if x is None else E.to_host(x, self.pinned_outputs)  # noqa: E731
        return (
            to_np(obs).reshape(b, t, 4, 4, 31),
            to_np(un["actions"]),
            to_np(un["action_masks"]),
            to_np(un["log_probs"]),
            to_np(un["values"]),
            to_np(un["rewards"]),
            to_np(un["terminations"]),
        )

    def run_rollout_batch(self, batch_size: int) -> list:
        """-> list[State], the init state first (batch_runner.py:156-195).  The run itself is the recorded one of
        ``run_actions_batch`` (whole chunks of steps per launch); the states are views of its records: the board after
        step t is the pre-step board of step t + 1 (a finished env keeps its frozen board), its legal mask the pre-step
        mask of step t + 1, its terminated flag and reward those of step t."""
        ro = self._run(batch_size, full_records=True)
        t = ro.t_steps
        mask = (ro.meta >> 2) & N.STATUS_MASK
        done = ((ro.meta >> 6) & 1) << 4
        status = torch.cat([mask[:1], mask[1:] | done[:-1], ro.final_status.unsqueeze(0)])  # (T + 1, n)
        zero = torch.zeros(ro.batch_size, dtype=torch.float32, device=self.device)
        states = [State(ro.boards[0], status[0], zero)] if t else [State(ro.final_boards, ro.final_status, zero)]
        for k in range(t):
            states.append(State(ro.boards[k + 1] if k + 1 < t else ro.final_boards, status[k + 1], ro.rewards[k]))
        return states

    # -- engine-native results -----------------------------------------------------------------
    def run_packed_batch(self, batch_size: int) -> PackedRollout:
        """Same run as ``run_actions_batch`` but the records stay packed on the device (with ``compact_live`` the
        slots of steps after an env's end are zero)."""
        return self._run(batch_size, full_records=False)

    def run_stats_batch(self, batch_size: int, per_env: bool = True, last_stored_boards: bool = False) -> dict:
        """Play to termination and return only per-episode results (final boards, lengths, scores)
        and the reduced statistics block.  Built-in policies only: this is the persistent
        ``g2048_play`` kernel.
        last_stored_boards: also return ``last_stored_boards`` -- what the reference's ``observations[:, -1]`` shows
        (src/runs/run_actions_max_tile.py:61-64): an env's final board, except for the envs that live until the last
        loop step, whose last STORED observation is the board before that step (``g2048_replay_envs`` replays just
        those envs, usually one)."""
        self._check(batch_size)
        policy = getattr(self._act_fn, "policy_id", None)
        if policy is None:
            raise ValueError("run_stats_batch needs act_randomly or act_drul")
        lo, n = self._range(batch_size)
        max_steps = 2048
        while True:
            subs = self.chain.peek(1 + 2 * max_steps)
            out = E.play(policy, subs, batch_size, lo, n, self.rng_mode, per_env=per_env)
            stats = self._reduce_stats(out["stats"])
            st = E.play_stats_dict(stats)
            if st["cut_short"] == 0:
                break
            max_steps *= 4  # an episode outlived the keys that were generated: replay with more
        if last_stored_boards and per_env:
            longest = st["longest"]  # over all shards: the reference's number of loop steps
            ids = torch.nonzero(out["lengths"] == longest).flatten()
            stored = out["final_boards"].clone()
            if ids.numel():
                steps = torch.full((ids.numel(),), longest - 1, dtype=torch.int32, device=self.device)
                before, _ = E.replay_envs(policy, subs, batch_size, ids + lo, steps, self.rng_mode)
                stored[ids] = before
            out["last_stored_boards"] = stored
        self.chain.consume(1 + 2 * st["longest"])
        out["stats"] = stats
        out["summary"] = st
        return out

    def run_flat_batch(self, batch_size: int) -> FlatRollout:
        """``run_packed_batch`` + ``RolloutBuffer.store_packed`` for act_randomly / act_drul in two launches: the
        persistent table kernel plays every env to termination and appends its records to the playing lane's own
        arena region (``g2048_play_record``; no lane ever steps a finished env), and one HBM-bound pass lays the
        episodes out env after env (``g2048_play_record_compact``)."""
        self._check(batch_size)
        policy = getattr(self._act_fn, "policy_id", None)
        if policy is None:
            raise ValueError("run_flat_batch needs act_randomly or act_drul; use run_packed_batch for other policies")
        lo, n = self._range(batch_size)
        max_steps, mean_steps = 2048, self._mean_steps.get(policy)
        while True:
            subs = self.chain.peek(1 + 2 * max_steps)
            rec = E.play_record(policy, subs, batch_size, lo, n, self.rng_mode, mean_steps)
            # The scan and the compaction are queued behind the play kernel BEFORE the host waits for its statistics:
            # the flat arrays are sized from the previous batch's mean episode length plus a margin (six standard
            # deviations of the total), the kernel drops what would not fit, and only a short estimate costs a second
            # compaction.  (Waiting for the exact total first left the GPU idle for the ~70 us the host needs to come
            # back from the synchronisation, allocate and launch.)
            offsets = E.exclusive_scan(rec["lengths"])
            mean_guess = E.MEAN_STEPS_HINT[policy] if mean_steps is None else mean_steps
            room = int(n * mean_guess * 1.01) + 600 * int(n ** 0.5) + 4096
            flat = E.play_record_compact(rec, offsets, room)
            local = E.play_stats_dict(rec["stats"])
            if local["cut_short"]:
                max_steps *= 4  # an episode outlived the keys that were generated: replay with more
                continue
            if local["episodes"] < n:  # some lane regions filled up before the queue was empty: a larger arena
                mean_steps = 2 * (E.MEAN_STEPS_HINT[policy] if mean_steps is None else mean_steps)
                continue
            break
        if n:
            self._mean_steps[policy] = max(16, -(-local["env_steps"] // n))
        stats = self._reduce_stats(rec["stats"])
        st = local if stats is rec["stats"] else E.play_stats_dict(stats)  # one read-back per batch unless it is sharded
        self.chain.consume(1 + 2 * st["longest"])
        total = local["env_steps"]
        if total > room:
            flat = E.play_record_compact(rec, offsets, total)
        else:  # prefixes of the roomier arrays (views: the margin stays allocated as long as the rollout lives)
            flat = {k: (v if k == "max_rewards" else v[:total]) for k, v in flat.items()}
        return FlatRollout(flat["boards"], flat["meta"], flat["rewards"], flat["log_probs"], flat["values"], rec["lengths"],
                           offsets, rec["final_boards"], rec["scores"], flat["max_rewards"], st["longest"], n, total, st)

    def run_eval_batch(self, batch_size: int) -> dict:
        """Network policy, results only: play ``batch_size`` envs to termination with the ``TorchActionFunction`` and
        return per-episode ``final_boards`` / ``lengths`` / ``scores`` and a ``summary`` like ``run_stats_batch`` -- no
        records are kept (evaluating an agent over many games, run/viz_ppo_agent.py style, needs none), and only the
        envs that are still alive go through the network.  Same trajectories and key chain as ``run_packed_batch``."""
        self._check(batch_size, eval_batch=True)
        fn = self._act_fn
        if isinstance(fn, MonteCarloPolicy):
            return self._run_eval_monte_carlo(batch_size)
        if isinstance(fn, ExpectimaxPolicy):
            return self._run_eval_expectimax(batch_size)
        if not hasattr(fn, "forward_logits"):
            raise ValueError("run_eval_batch needs a TorchActionFunction; use run_stats_batch for act_randomly / act_drul")
        lo, n = self._range(batch_size)
        dev, mode = self.device, self.rng_mode
        boards, status = E.env_init(self.chain.peek(1)[0], batch_size, lo, n, mode)
        lengths = torch.zeros(n, dtype=torch.int32, device=dev)
        scores = torch.zeros(n, dtype=torch.float32, device=dev)
        t0 = 0
        while True:
            # chunks of NET_SYNC_STEPS steps: the live list is built once per chunk, the chunk's rewards and metas are
            # the only records kept (5 bytes per env-step, dropped after the chunk), one host read per chunk
            steps = NET_SYNC_STEPS
            subs = self.chain.peek(1 + 2 * (t0 + steps))
            live_ids = torch.nonzero((status & N.STATUS_DONE) == 0).flatten()
            rm = torch.zeros((steps, n), dtype=torch.uint8, device=dev)
            rr = torch.zeros((steps, n), dtype=torch.float32, device=dev)
            alive_before = (status & N.STATUS_DONE) == 0
            if live_ids.shape[0]:
                for k in range(steps):
                    t = t0 + k
                    obs = E.expand_obs_gather(boards, live_ids, fn.obs_dtype)
                    logits, values = fn.forward_logits(obs)
                    E.policy_step_live(boards, status, logits, values, fn.use_mask, fn.sample_actions, False, subs[1 + 2 * t],
                                       subs[2 + 2 * t], live_ids, batch_size, lo, mode, None, rm[k], rr[k])
            # per env: steps played in this chunk = first done + 1 (or all of them), for the envs alive at its start
            first = E.episode_lengths(rm, steps, n)
            played = torch.where(first > 0, first, torch.full_like(first, steps))
            lengths += torch.where(alive_before, played, torch.zeros_like(played))
            scores += rr.clamp_(min=0.0).sum(dim=0)  # the illegal-action penalty (-1) is not part of the game score
            t0 += steps
            done_now = int(((status & N.STATUS_DONE) != 0).sum().item())
            if self._all_done(done_now, n):
                break
        t = int(lengths.max().item()) if n else 0  # the reference's number of loop steps: the longest episode
        if self.shard is not None and self.shard[1] > 1:
            from ..dist import allreduce_max_int

            t = allreduce_max_int(t, self.device)
        self.chain.consume(1 + 2 * t)
        exps = torch.stack([(boards >> (4 * c)) & 15 for c in range(16)], dim=1).amax(dim=1)
        hist = torch.bincount(exps, minlength=16)
        tiles = (2.0 ** exps.double())
        summary = {"episodes": n, "env_steps": int(lengths.sum().item()), "score_sum": int(scores.double().sum().item()),
                   "longest": int(lengths.max().item()) if n else 0, "loop_steps": t,
                   "max_tile_hist": {1 << e: int(c) for e, c in enumerate(hist.tolist()) if c},
                   "mean_max_tile": float(tiles.mean().item()) if n else 0.0}
        return {"final_boards": boards, "lengths": lengths, "scores": scores.to(torch.int32), "summary": summary}

    def _run_eval_monte_carlo(self, batch_size: int) -> dict:
        """run_eval_batch with a ``MonteCarloPolicy``: per loop step t one ``g2048_playout_values`` launch over the envs
        alive at the start of the chunk (global env ids as board ids; sub keys split(act key of step t, 1 + 2 max_steps)),
        the best action per env, and ``g2048_env_step`` with the step key of step t.  An env that finishes inside a
        chunk is still listed until the chunk ends: it has no legal action, so none of its playouts is played, and the
        step leaves a finished env as it is.  The host reads the done count once per NET_SYNC_STEPS steps."""
        fn = self._act_fn
        mode = self.rng_mode
        policy, n_subs = fn.rollout_policy, 1 + 2 * int(fn.max_steps)

        def choose(live_boards, board_ids, sub_act):
            psubs = E.split_keys(sub_act, n_subs, 0, n_subs, mode)
            rec = E.playout_values(policy, live_boards, psubs, int(fn.playouts), mode, board_ids=board_ids,
                                   n_boards_global=batch_size)
            return best_actions(rec, fn.criterion)

        return self._run_eval_search(batch_size, choose)

    def _run_eval_expectimax(self, batch_size: int) -> dict:
        """run_eval_batch with an ``ExpectimaxPolicy``: per loop step one ``g2048_expectimax_values`` launch over the
        envs alive at the start of the chunk and the best action per env (an env that finished inside the chunk has no
        legal action and gets action 0, which the step ignores); the act sub key is not used."""
        fn = self._act_fn
        if fn.network is not None:
            net = fn.network
            placements, weights, stages = net.placements, net.weights_on(self.device), net.stages

            def choose(live_boards, board_ids, sub_act):
                return expectimax_best_actions(E.expectimax_values_ntuple(live_boards, int(fn.depth), placements, weights,
                                                                          float(fn.reward_weight), stages=stages))

            return self._run_eval_search(batch_size, choose)
        table = fn.table(self.device)

        def choose(live_boards, board_ids, sub_act):
            return expectimax_best_actions(E.expectimax_values(live_boards, int(fn.depth), table, float(fn.reward_weight)))

        return self._run_eval_search(batch_size, choose)

    def _run_eval_search(self, batch_size: int, choose) -> dict:
        """The per-move loop of the search players: per loop step t, ``choose(boards of the envs alive at the start of
        the chunk, their global env ids, act sub key of step t)`` gives their actions, and ``g2048_env_step`` steps
        every env with the step key of step t (a finished env stays as it is).  The live list is built once per
        chunk of NET_SYNC_STEPS steps, and the host reads the done count once per chunk."""
        lo, n = self._range(batch_size)
        dev, mode = self.device, self.rng_mode
        boards, status = E.env_init(self.chain.peek(1)[0], batch_size, lo, n, mode)
        lengths = torch.zeros(n, dtype=torch.int32, device=dev)
        scores = torch.zeros(n, dtype=torch.int64, device=dev)
        actions = torch.zeros(n, dtype=torch.int32, device=dev)
        t0 = 0
        while True:
            steps = NET_SYNC_STEPS
            subs = self.chain.peek(1 + 2 * (t0 + steps))
            live_ids = torch.nonzero((status & N.STATUS_DONE) == 0).flatten()
            if live_ids.shape[0]:
                board_ids = live_ids + lo
                for k in range(steps):
                    t = t0 + k
                    actions[live_ids] = choose(boards[live_ids], board_ids, subs[1 + 2 * t]).to(torch.int32)
                    alive = (status & N.STATUS_DONE) == 0
                    rewards = E.env_step(boards, status, actions, subs[2 + 2 * t], batch_size, lo, mode)
                    lengths += alive.to(torch.int32)
                    scores += rewards.to(torch.int64)  # a best action is legal: no -1 penalties, finished envs get 0
            t0 += steps
            done_now = int(((status & N.STATUS_DONE) != 0).sum().item())
            if self._all_done(done_now, n):
                break
        t = int(lengths.max().item()) if n else 0  # the reference's number of loop steps: the longest episode
        if self.shard is not None and self.shard[1] > 1:
            from ..dist import allreduce_max_int

            t = allreduce_max_int(t, self.device)
        self.chain.consume(1 + 2 * t)
        exps = torch.stack([(boards >> (4 * c)) & 15 for c in range(16)], dim=1).amax(dim=1)
        hist = torch.bincount(exps, minlength=16)
        tiles = (2.0 ** exps.double())
        summary = {"episodes": n, "env_steps": int(lengths.sum().item()), "score_sum": int(scores.sum().item()),
                   "longest": int(lengths.max().item()) if n else 0, "loop_steps": t,
                   "max_tile_hist": {1 << e: int(c) for e, c in enumerate(hist.tolist()) if c},
                   "mean_max_tile": float(tiles.mean().item()) if n else 0.0}
        return {"final_boards": boards, "lengths": lengths, "scores": scores.to(torch.int32), "summary": summary}

    # -- internals -----------------------------------------------------------------------------
    def _check(self, batch_size: int, eval_batch: bool = False) -> None:
        if self._act_fn is None:
            raise ValueError("The action function is not set.")
        if isinstance(self._act_fn, MonteCarloPolicy) and not eval_batch:
            raise ValueError("a MonteCarloPolicy plays through run_eval_batch only (it keeps no records)")
        if isinstance(self._act_fn, ExpectimaxPolicy) and not eval_batch:
            raise ValueError("an ExpectimaxPolicy plays through run_eval_batch only (it keeps no records)")
        if not isinstance(batch_size, (int, np.integer)) or batch_size <= 0:
            raise ValueError(f"batch_size must be a positive integer, got {batch_size!r}")

    def _range(self, batch_size: int) -> tuple[int, int]:
        if self.shard is None:
            return 0, batch_size
        rank, world = self.shard
        lo = batch_size * rank // world
        hi = batch_size * (rank + 1) // world
        return lo, hi - lo

    def _reduce_stats(self, stats: torch.Tensor) -> torch.Tensor:
        if self.shard is None or self.shard[1] == 1:
            return stats
        from ..dist import allreduce_play_stats

        return allreduce_play_stats(stats)

    def _all_done(self, done_count: int, n: int) -> bool:
        if self.shard is None or self.shard[1] == 1:
            return done_count == n
        from ..dist import all_ranks_true

        return all_ranks_true(done_count == n, self.device)

    def _run(self, batch_size: int, keep_states: bool = False, full_records: bool = True) -> PackedRollout:
        """A recorded run.  full_records: the caller reads the records of finished envs too (reference-format outputs)."""
        self._check(batch_size)
        lo, n = self._range(batch_size)
        dev, mode = self.device, self.rng_mode
        init_sub = self.chain.peek(1)[0]
        boards, status = E.env_init(init_sub, batch_size, lo, n, mode)
        policy = getattr(self._act_fn, "policy_id", None)
        is_net = hasattr(self._act_fn, "forward_logits")
        if self.cuda_graph and is_net:
            return self._run_net_graphed(batch_size, lo, n, boards, status)
        if is_net:
            return self._run_net(batch_size, lo, n, boards, status, compact=self.compact_live and not full_records)
        if policy is None:
            return self._run_callable(batch_size, lo, n, boards, status)
        # built-in policies: whole chunks of loop steps per launch (lock-step recorder); the kernel keeps the number of
        # finished envs and the longest episode on the device, read once per chunk
        compact = self.compact_live and not full_records
        counters = torch.zeros(4, dtype=torch.int64, device=dev)
        chunks, t0 = [], 0
        want_lp = policy != E.POLICY_DRUL
        while True:
            # a run whose envs are all finished at init cannot happen (two tiles on an empty board)
            steps = CHUNK_STEPS
            subs = self.chain.peek(1 + 2 * (t0 + steps))
            alloc = torch.zeros if compact else torch.empty  # compact mode leaves finished envs' slots untouched
            rb = alloc((steps, n), dtype=torch.int64, device=dev)
            rm = alloc((steps, n), dtype=torch.uint8, device=dev)
            rr = alloc((steps, n), dtype=torch.float32, device=dev)
            rl = alloc((steps, n), dtype=torch.float32, device=dev) if want_lp else None
            if compact:  # the envs alive at the start of the chunk; one that finishes inside it leaves the loop
                live_ids = torch.nonzero((status & N.STATUS_DONE) == 0).flatten()
                E.rollout_steps_live(policy, boards, status, subs[1 + 2 * t0:], steps, t0, batch_size, lo, mode,
                                     live_ids, rb, rm, rr, rl, counters)
            else:
                E.rollout_steps(policy, boards, status, subs[1 + 2 * t0:], steps, t0, batch_size, lo, mode,
                                rb, rm, rr, rl, counters)
            chunks.append((rb, rm, rr, rl))
            t0 += steps
            if self._all_done(int(counters[0].item()), n):
                break
        t_total = int(counters[1].item())
        if self.shard is not None and self.shard[1] > 1:
            from ..dist import allreduce_max_int

            t_total = allreduce_max_int(t_total, self.device)
        self.chain.consume(1 + 2 * t_total)
        cat = lambda i: None if chunks[0][i] is None else torch.cat([c[i] for c in chunks])[:t_total].contiguous()  # noqa: E731
        rb, rm, rr, rl = (cat(i) for i in range(4))
        return PackedRollout(rb, rm, rr, rl, None, boards, status, t_total, n, int(counters[2].item()))

    def _run_callable(self, batch_size: int, lo: int, n: int, boards, status) -> PackedRollout:
        """Any Python callable ``(keys, obs, mask) -> (action, log_prob, value)`` (the reference's act_fn contract,
        src/runs/batch_runner.py:120-124): the policy runs on the host side of every step, so this path keeps the
        reference's structure -- per step ``g2048_split_keys``, the callable, ``g2048_env_step`` -- and its per-step
        ``all done`` test."""
        dev, mode = self.device, self.rng_mode
        rows, t = [], 0
        has_lp = has_v = True
        while True:
            subs = self.chain.peek(1 + 2 * (t + 1))
            rb = torch.empty(n, dtype=torch.int64, device=dev)
            rm = torch.empty(n, dtype=torch.uint8, device=dev)
            rr, rl, rv = (torch.empty(n, dtype=torch.float32, device=dev) for _ in range(3))
            rl_k, rv_k = self._callable_step(boards, status, subs[1 + 2 * t], subs[2 + 2 * t], batch_size, lo, mode, rb, rm, rr, rl, rv)
            has_lp &= rl_k is not None  # the policy returns no log-probs (like act_drul)
            has_v &= rv_k is not None
            rows.append((rb, rm, rr, rl, rv))
            t += 1
            # the reference checks `all done` after every step (batch_runner.py:117)
            if self._all_done(int(((status & N.STATUS_DONE) != 0).sum().item()), n):
                break
        self.chain.consume(1 + 2 * t)
        rb, rm, rr, rl, rv = (torch.stack([r[i] for r in rows]) for i in range(5))
        env_steps = int(E.episode_lengths(rm, t, n).sum().item())
        return PackedRollout(rb, rm, rr, rl if has_lp else None, rv if has_v else None, boards, status, t, n, env_steps)

    # -- eager network-policy loop: one fused launch per step, one host synchronisation per chunk ----------------------
    def _run_net(self, batch_size: int, lo: int, n: int, boards, status, compact: bool) -> PackedRollout:
        """src/runs/batch_runner.py:117-136 with a ``TorchActionFunction``: per loop step the network forward (PyTorch)
        and ONE kernel -- ``g2048_policy_step_obs``: mask rule, categorical draw, log-prob, env.step, record write and the
        observation of the next forward pass, written from registers.  The reference tests ``all done`` after every
        step (a blocking read-back); here the kernel keeps the count of finished envs on the device and the host reads
        it once per NET_SYNC_STEPS steps -- stepping a finished batch is a no-op (frozen envs), and the loop steps past
        the last env's end are cut off afterwards.  compact: only the envs alive at the start of a chunk go through
        the network (``g2048_expand_obs_gather`` + ``g2048_policy_step_live``, which skips envs that finished inside
        the chunk)."""
        fn, dev, mode = self._act_fn, self.device, self.rng_mode
        counters = torch.zeros(2, dtype=torch.int64, device=dev)
        obs = None if compact else E.expand_obs(boards, fn.obs_dtype)
        alloc = torch.zeros if compact else torch.empty  # compact mode leaves the slots of finished envs untouched
        chunks, t0 = [], 0
        while True:
            steps = NET_SYNC_STEPS
            subs = self.chain.peek(1 + 2 * (t0 + steps))
            rb = alloc((steps, n), dtype=torch.int64, device=dev)
            rm = alloc((steps, n), dtype=torch.uint8, device=dev)
            rr, rl, rv = (alloc((steps, n), dtype=torch.float32, device=dev) for _ in range(3))
            if compact:
                live_ids = torch.nonzero((status & N.STATUS_DONE) == 0).flatten()  # once per chunk
            for k in range(steps):
                t = t0 + k
                if compact:
                    self._net_step_live(boards, status, live_ids, subs[1 + 2 * t], subs[2 + 2 * t], batch_size, lo, mode,
                                        rb[k], rm[k], rr[k], rl[k], rv[k])
                else:
                    logits, values = fn.forward_logits(obs)
                    E.policy_step_obs(boards, status, logits, values, fn.use_mask, fn.sample_actions, False, subs[1 + 2 * t:],
                                      None, batch_size, lo, mode, obs, rb[k], rm[k], rr[k], rl[k], rv[k], counters=counters)
            chunks.append((rb, rm, rr, rl, rv))
            t0 += steps
            if compact:
                done_now = int(((status & N.STATUS_DONE) != 0).sum().item())
            else:
                done_now = int(counters[0].item())  # maintained by the kernel: the one read-back of the chunk
            if self._all_done(done_now, n):
                break
        rb, rm, rr, rl, rv = (torch.cat([c[i] for c in chunks]) for i in range(5))
        lengths = E.episode_lengths(rm, t0, n)
        t_total = int(lengths.max().item()) if n else 0
        if self.shard is not None and self.shard[1] > 1:
            from ..dist import allreduce_max_int

            t_total = allreduce_max_int(t_total, self.device)
        self.chain.consume(1 + 2 * t_total)
        rb, rm, rr, rl, rv = (x[:t_total].contiguous() for x in (rb, rm, rr, rl, rv))
        return PackedRollout(rb, rm, rr, rl, rv, boards, status, t_total, n, int(lengths.sum().item()))

    # -- CUDA-graph form of the network-policy loop (SURVEY 8f rank 3) ---------------------------
    def _captured_step(self, batch_size: int, lo: int, n: int, steps: int = CHUNK_STEPS, auto_reset: bool = False) -> dict:
        """Static buffers + one captured graph: expand_obs -> forward -> policy_step_at -> counter_add.
        `steps` record slots per chunk; auto_reset: pgx.experimental.auto_reset semantics (fixed-horizon rollouts)."""
        fn = self._act_fn
        cache_key = (batch_size, lo, n, steps, auto_reset)
        g = self._graphs.get(cache_key)
        if g is not None and g["fn"] is fn:  # the entry keeps `fn` alive, so identity cannot be a recycled id
            return g
        dev, mode = self.device, self.rng_mode
        net_dev, run_dev = torch.device(fn.device), torch.device(dev)
        same_index = net_dev.index is None or run_dev.index is None or net_dev.index == run_dev.index
        if net_dev.type != "cuda" or not same_index:
            raise ValueError("cuda_graph=True needs the TorchActionFunction's network on the runner's GPU")
        g = dict(
            fn=fn,
            boards=torch.zeros(n, dtype=torch.int64, device=dev), status=torch.zeros(n, dtype=torch.uint8, device=dev),
            obs=torch.empty((n, 16, 31), dtype=fn.obs_dtype, device=dev),
            subs=torch.zeros((2 * steps, 2), dtype=torch.int32, device=dev),
            step_index=torch.zeros((), dtype=torch.int32, device=dev),
            rb=torch.empty((steps, n), dtype=torch.int64, device=dev), rm=torch.empty((steps, n), dtype=torch.uint8, device=dev),
            rr=torch.empty((steps, n), dtype=torch.float32, device=dev), rl=torch.empty((steps, n), dtype=torch.float32, device=dev),
            rv=torch.empty((steps, n), dtype=torch.float32, device=dev),
        )

        def step():
            # g["obs"] holds the observation of the current state (refresh_obs() before the first replay): the fused
            # kernel writes the next one from registers and moves the device-resident step number on itself
            logits, values = fn.forward_logits(g["obs"])
            E.policy_step_obs(g["boards"], g["status"], logits, values, fn.use_mask, fn.sample_actions, auto_reset, g["subs"],
                              g["step_index"], batch_size, lo, mode, g["obs"], g["rb"], g["rm"], g["rr"], g["rl"], g["rv"],
                              counters=g["counters"], advance_step=True)

        g["counters"] = torch.zeros(2, dtype=torch.int64, device=dev)
        g["refresh_obs"] = lambda: E.expand_obs(g["boards"], fn.obs_dtype, out=g["obs"])

        # warm-up on a side stream (lazy module loading, cuBLAS workspaces, autotuning) before the capture
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            g["refresh_obs"]()
            for _ in range(3):
                g["step_index"].zero_()
                step()
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize(dev)
        graph = torch.cuda.CUDAGraph()
        g["step_index"].zero_()
        with torch.cuda.graph(graph):
            step()
        g["graph"] = graph
        self._graphs[cache_key] = g
        return g

    def _run_net_graphed(self, batch_size: int, lo: int, n: int, boards, status) -> PackedRollout:
        g = self._captured_step(batch_size, lo, n)
        g["boards"].copy_(boards)
        g["status"].copy_(status)
        g["refresh_obs"]()
        g["counters"].zero_()
        chunks, t0 = [], 0
        while True:
            subs = self.chain.peek(1 + 2 * (t0 + CHUNK_STEPS))
            g["subs"].copy_(subs[1 + 2 * t0: 1 + 2 * (t0 + CHUNK_STEPS)])
            g["step_index"].zero_()
            # frozen envs do not change (env.step on a finished env is a no-op), so running past the reference's
            # per-step `all done` test only appends records that are cut off below; the test (one host
            # synchronisation) runs every GRAPH_SYNC_STEPS replays
            finished, used = False, 0
            while used < CHUNK_STEPS and not finished:
                for _ in range(GRAPH_SYNC_STEPS):
                    g["graph"].replay()
                used += GRAPH_SYNC_STEPS
                done_now = int(g["counters"][0].item())  # kept by the kernel: no reduction kernels on the loop's path
                finished = self._all_done(done_now, n)
            chunks.append(tuple(g[k][:used].clone() for k in ("rb", "rm", "rr", "rl", "rv")))
            t0 += used
            if finished:
                break
        rb, rm, rr, rl, rv = (torch.cat([c[i] for c in chunks]) for i in range(5))
        lengths = E.episode_lengths(rm, t0, n)
        t_total = int(lengths.max().item())
        if self.shard is not None and self.shard[1] > 1:
            from ..dist import allreduce_max_int

            t_total = allreduce_max_int(t_total, self.device)
        self.chain.consume(1 + 2 * t_total)
        rb, rm, rr, rl, rv = (x[:t_total].contiguous() for x in (rb, rm, rr, rl, rv))
        return PackedRollout(rb, rm, rr, rl, rv, g["boards"].clone(), g["status"].clone(), t_total, n,
                             int(lengths.sum().item()))

    def _net_step_live(self, boards, status, live_ids, sub_act, sub_step, batch_size, lo, mode, rb, rm, rr, rl, rv):
        fn = self._act_fn
        if live_ids.shape[0]:  # a shard whose envs are all finished waits for the other ranks
            obs = E.expand_obs_gather(boards, live_ids, fn.obs_dtype)
            logits, values = fn.forward_logits(obs)
            E.policy_step_live(boards, status, logits, values, fn.use_mask, fn.sample_actions, False, sub_act, sub_step,
                               live_ids, batch_size, lo, mode, rb, rm, rr, rl, rv)
        return rl, rv

    def _net_step(self, boards, status, sub_act, sub_step, batch_size, lo, mode, rb, rm, rr, rl, rv):
        fn = self._act_fn
        obs = E.expand_obs(boards, fn.obs_dtype)
        logits, values = fn.forward_logits(obs)
        E.policy_step(boards, status, logits, values, fn.use_mask, fn.sample_actions, False, sub_act, sub_step,
                      batch_size, lo, mode, rb, rm, rr, rl, rv)
        return rl, rv

    def _callable_step(self, boards, status, sub_act, sub_step, batch_size, lo, mode, rb, rm, rr, rl, rv):
        n = boards.shape[0]
        keys = E.split_keys(sub_act, batch_size, lo, n, mode)
        obs = E.expand_obs(boards, torch.bool).view(n, 4, 4, 31)
        mask, _ = E.unpack_status(status)
        action, log_prob, value = self._act_fn(keys, obs, mask)
        action = torch.as_tensor(action, device=boards.device).to(torch.int32).reshape(n).contiguous()
        rb.copy_(boards)
        pre_mask = status & N.STATUS_MASK
        rewards = E.env_step(boards, status, action, sub_step, batch_size, lo, mode)
        rr.copy_(rewards)
        done = (status & N.STATUS_DONE) != 0
        rm.copy_((action & 3).to(torch.uint8) | (pre_mask << 2) | (done.to(torch.uint8) << 6))
        if log_prob is not None and rl is not None:
            rl.copy_(torch.as_tensor(log_prob, device=boards.device).to(torch.float32).reshape(n))
        if value is not None and rv is not None:
            rv.copy_(torch.as_tensor(value, device=boards.device).to(torch.float32).reshape(n))
        return (rl if log_prob is not None else None), (rv if value is not None else None)
