"""Tensor-level wrappers over the C ABI: each function launches exactly one libg2048 kernel on
torch's current stream.  PyTorch is used for device memory and streams only.

Boards travel as ``torch.int64`` tensors holding the uint64 bitboard bits; keys and sub keys as
``torch.int32`` tensors holding uint32 words (shape (..., 2)).
"""
from __future__ import annotations

import math
import os
import threading

import numpy as np
import torch

from . import _native as N
from ._native import call, ptr, stream_ptr

RNG_ORIGINAL = N.RNG_ORIGINAL
RNG_PARTITIONABLE = N.RNG_PARTITIONABLE
POLICY_RANDOM = N.POLICY_RANDOM
POLICY_DRUL = N.POLICY_DRUL


def resolve_rng_mode(mode=None) -> int:
    """None -> $G2048_THREEFRY_PARTITIONABLE (default 1, like the pinned jax 0.5.3)."""
    if mode is None:
        env = os.environ.get("G2048_THREEFRY_PARTITIONABLE", os.environ.get("JAX_THREEFRY_PARTITIONABLE", "1"))
        return RNG_PARTITIONABLE if env.strip().lower() not in ("0", "false", "off", "no") else RNG_ORIGINAL
    if isinstance(mode, str):
        m = mode.lower()
        if m in ("partitionable", "1", "true"):
            return RNG_PARTITIONABLE
        if m in ("original", "0", "false"):
            return RNG_ORIGINAL
        raise ValueError(f"unknown rng_mode {mode!r}")
    return RNG_PARTITIONABLE if int(mode) else RNG_ORIGINAL


def key_words(seed: int) -> tuple[int, int]:
    """jax.random.key(seed) -> (hi, lo) uint32 words, as the reference gets them (src/runs/batch_runner.py:32 with jax's
    default 32-bit mode): the seed becomes an int32 array, so the high word -- a logical shift by 32 -- is always 0 and
    the low word is the seed's two's-complement bits (seed=-1 -> (0, 0xFFFFFFFF)); a seed outside [-2^31, 2^32) does
    not fit and raises OverflowError there, so it does here."""
    seed = int(seed)
    if not -(1 << 31) <= seed < (1 << 32):
        raise OverflowError(f"seed {seed} does not fit in 32 bits (jax.random.key without x64 rejects it too)")
    return 0, seed & 0xFFFFFFFF


def words_tensor(words, device) -> torch.Tensor:
    """uint32 words -> int32 device tensor with the same bits."""
    arr = np.asarray(words, dtype=np.uint32)
    return torch.from_numpy(arr.view(np.int32).copy()).to(device)


def words_numpy(t: torch.Tensor) -> np.ndarray:
    return t.detach().cpu().numpy().view(np.uint32)


def boards_numpy(t: torch.Tensor) -> np.ndarray:
    """int64 bitboards -> (..., 16) uint8 exponents (host)."""
    x = t.detach().cpu().numpy().view(np.uint64)
    return ((x[..., None] >> (np.arange(16, dtype=np.uint64) * np.uint64(4))) & np.uint64(15)).astype(np.uint8)


def pack_boards(exponents) -> np.ndarray:
    """(..., 16) exponents -> uint64 bitboards viewed as int64 (host)."""
    b = np.asarray(exponents, dtype=np.uint64)
    return (b << (np.arange(16, dtype=np.uint64) * np.uint64(4))).sum(axis=-1).astype(np.uint64).view(np.int64)


_STAGE = {}  # device index -> pinned uint8 staging buffer of to_host(), grown on demand
_STAGE_LOCK = threading.Lock()  # one staged copy at a time: the buffer is shared by every caller of the process


def to_host(x: torch.Tensor, pinned: bool = False) -> np.ndarray:
    """A fresh numpy array with the tensor's contents.  Large tensors go through a pinned staging buffer kept per
    device: a pageable device-to-host copy of C1's 130 MB of observations ran at 2 GB/s and was 80 % of
    run_actions_batch; staged, the transfer takes 2.5 ms and the copy into the caller's array the rest.
    pinned=True: the array IS page-locked memory from torch's caching host allocator (one transfer, no second copy, no
    first-touch page faults); it goes back to the allocator's cache when the array is released."""
    nbytes = x.numel() * x.element_size()
    if not x.is_cuda or nbytes < (1 << 20):
        return x.cpu().numpy()
    if pinned:
        out = torch.empty(x.shape, dtype=x.dtype, pin_memory=True)
        out.copy_(x, non_blocking=True)
        torch.cuda.current_stream(x.device).synchronize()
        return out.numpy()
    key = x.device.index
    with _STAGE_LOCK:
        stage = _STAGE.get(key)
        if stage is None or stage.numel() < nbytes:
            stage = _STAGE[key] = torch.empty(max(nbytes, 1 << 24), dtype=torch.uint8, pin_memory=True)
        view = stage[:nbytes].view(x.dtype).view(x.shape)
        view.copy_(x.contiguous(), non_blocking=True)
        torch.cuda.current_stream(x.device).synchronize()
        if torch.get_num_threads() > 1:
            out = torch.empty(x.shape, dtype=x.dtype)  # the caller's array; torch's CPU copy is multi-threaded,
            out.copy_(view)                            # which also spreads the first-touch page faults (C1: 44 -> 19 ms)
            return out.numpy()
        return view.numpy().copy()  # one thread (e.g. OMP_NUM_THREADS=1 under torchrun): numpy's memcpy is the faster one


def _i32(t):
    assert t.dtype == torch.int32, t.dtype
    return t


# ------------------------------------------------------------------------------------------- RNG
def threefry2x32(keys: torch.Tensor, ctrs: torch.Tensor) -> torch.Tensor:
    N.require_cuda()
    out = torch.empty_like(keys)
    call("g2048_threefry2x32", ptr(_i32(keys)), ptr(_i32(ctrs)), keys.shape[0], ptr(out), stream_ptr())
    return out


def chain_advance(key_io: torch.Tensor, rng_mode: int, n_sub: int, out: torch.Tensor | None = None) -> torch.Tensor:
    """Advances key_io (2 words, in place) n_sub times; returns the (n_sub, 2) sub keys."""
    N.require_cuda()
    if out is None:
        out = torch.empty((n_sub, 2), dtype=torch.int32, device=key_io.device)
    call("g2048_chain_advance", ptr(_i32(key_io)), rng_mode, n_sub, ptr(out), stream_ptr())
    return out


def split_keys(sub: torch.Tensor, batch_global: int, env_lo: int, n: int, rng_mode: int) -> torch.Tensor:
    N.require_cuda()
    out = torch.empty((n, 2), dtype=torch.int32, device=sub.device)
    call("g2048_split_keys", ptr(_i32(sub)), batch_global, env_lo, n, rng_mode, ptr(out), stream_ptr())
    return out


# ------------------------------------------------------------------------------------------- env
def env_init(sub: torch.Tensor, batch_global: int, env_lo: int, n: int, rng_mode: int):
    """-> boards (n,) int64, status (n,) uint8.  batch_global=0: `sub` is an explicit (n,2) key array."""
    dev = N.require_cuda() if not sub.is_cuda else sub.device
    boards = torch.empty(n, dtype=torch.int64, device=dev)
    status = torch.empty(n, dtype=torch.uint8, device=dev)
    call("g2048_env_init", ptr(_i32(sub)), batch_global, env_lo, n, rng_mode, ptr(boards), ptr(status), stream_ptr())
    return boards, status


def env_step(boards, status, actions, sub, batch_global: int, env_lo: int, rng_mode: int) -> torch.Tensor:
    """In place on boards/status; returns rewards (n,) float32."""
    n = boards.shape[0]
    rewards = torch.empty(n, dtype=torch.float32, device=boards.device)
    call("g2048_env_step", ptr(boards), ptr(status), ptr(_i32(actions)), ptr(_i32(sub)), batch_global, env_lo, n,
         rng_mode, ptr(rewards), stream_ptr())
    return rewards


def env_step_draws(boards, status, actions, bits_pos, bits_val) -> torch.Tensor:
    n = boards.shape[0]
    rewards = torch.empty(n, dtype=torch.float32, device=boards.device)
    call("g2048_env_step_draws", ptr(boards), ptr(status), ptr(_i32(actions)), ptr(_i32(bits_pos)), ptr(_i32(bits_val)),
         n, ptr(rewards), stream_ptr())
    return rewards


def act(policy: int, status, sub, batch_global: int, env_lo: int, rng_mode: int):
    """-> actions int32 (n,), log_probs float32 (n,) or None (act_drul)."""
    n = status.shape[0]
    actions = torch.empty(n, dtype=torch.int32, device=status.device)
    log_probs = torch.empty(n, dtype=torch.float32, device=status.device) if policy == POLICY_RANDOM else None
    call("g2048_act", policy, ptr(status), ptr(sub), batch_global, env_lo, n, rng_mode, ptr(actions), ptr(log_probs),
         stream_ptr())
    return actions, log_probs


# ------------------------------------------------------------------------------------------- fused loops
STAT_NAMES = ("episodes", "env_steps", "score_sum", "cut_short", "overflowed", "longest", "tile_sum", "tile_sq_sum")


def play(policy: int, subs: torch.Tensor, batch_global: int, env_lo: int, n: int, rng_mode: int,
         per_env: bool = True, stats: torch.Tensor | None = None, entry: str = "g2048_play"):
    """Persistent play-to-termination kernel.  Returns dict(final_boards, lengths, scores, stats).
    entry: another entry point with g2048_play's signature (g2048_play_tables, g2048_play_swar; tests also pass the
    first-generation g2048_play_v1 of their own legacy build, see _native.register_entry_points)."""
    dev = subs.device
    work = torch.zeros(2, dtype=torch.int64, device=dev)
    if stats is None:
        stats = torch.zeros(N.PLAY_STATS_WORDS, dtype=torch.int64, device=dev)
    boards = lengths = scores = None
    if per_env:
        boards = torch.empty(n, dtype=torch.int64, device=dev)
        lengths = torch.empty(n, dtype=torch.int32, device=dev)
        scores = torch.empty(n, dtype=torch.int32, device=dev)
    call(entry, policy, ptr(_i32(subs)), subs.shape[0], batch_global, env_lo, n, rng_mode, ptr(work),
         ptr(boards), ptr(lengths), ptr(scores), ptr(stats), stream_ptr())
    return dict(final_boards=boards, lengths=lengths, scores=scores, stats=stats)


def replay_envs(policy: int, subs: torch.Tensor, batch_global: int, env_ids: torch.Tensor, steps: torch.Tensor, rng_mode: int):
    """Boards and status of the listed envs (global indices, int64) after steps[i] (int32) loop steps of the built-in
    policy.  -> boards (m,) int64, status (m,) uint8."""
    m = env_ids.shape[0]
    assert env_ids.dtype == torch.int64 and steps.dtype == torch.int32 and steps.shape[0] == m
    boards = torch.empty(m, dtype=torch.int64, device=subs.device)
    status = torch.empty(m, dtype=torch.uint8, device=subs.device)
    call("g2048_replay_envs", policy, ptr(_i32(subs)), subs.shape[0], batch_global, ptr(env_ids), ptr(steps), m, rng_mode,
         ptr(boards), ptr(status), stream_ptr())
    return boards, status


def row_table_lookup(rows: torch.Tensor):
    """Test hook: table entries (row moved left, move flags) of int16 rows."""
    n = rows.shape[0]
    left = torch.empty(n, dtype=torch.int16, device=rows.device)
    flags = torch.empty(n, dtype=torch.uint8, device=rows.device)
    call("g2048_row_table_lookup", ptr(rows), n, ptr(left), ptr(flags), stream_ptr())
    return left, flags


def play_stats_dict(stats: torch.Tensor) -> dict:
    s = stats.detach().cpu().numpy().astype(np.uint64)
    out = {k: int(s[i]) for i, k in enumerate(STAT_NAMES)}
    out["max_tile_hist"] = {1 << e: int(s[16 + e]) for e in range(16) if s[16 + e]}
    return out


EPISODE_RESULT = np.dtype([("board", "<u8"), ("length", "<u4"), ("score", "<u4")])  # G2048EpisodeResult (include/g2048.h)


def play_packed(policy: int, subs: torch.Tensor, batch_global: int, env_lo: int, n: int, rng_mode: int,
                stats: torch.Tensor | None = None):
    """g2048_play with one 16-byte record per env: returns dict(results (n, 2) int64 device tensor -- word 0 the final
    bitboard, word 1 = length | score << 32 --, stats)."""
    dev = subs.device
    work = torch.zeros(2, dtype=torch.int64, device=dev)
    if stats is None:
        stats = torch.zeros(N.PLAY_STATS_WORDS, dtype=torch.int64, device=dev)
    results = torch.empty((n, 2), dtype=torch.int64, device=dev)
    call("g2048_play_packed", policy, ptr(_i32(subs)), subs.shape[0], batch_global, env_lo, n, rng_mode, ptr(work),
         ptr(results), ptr(stats), stream_ptr())
    return dict(results=results, stats=stats)


MEAN_STEPS_HINT = {POLICY_RANDOM: 128, POLICY_DRUL: 224}  # only sizes the recording arena (observed means: ~118 / ~207)


def play_record(policy: int, subs: torch.Tensor, batch_global: int, env_lo: int, n: int, rng_mode: int,
                mean_steps: int | None = None, stats: torch.Tensor | None = None) -> dict:
    """g2048_play that also records every env's trajectory into a per-lane arena (one launch of the persistent table
    kernel).  Returns dict(arena_boards, arena_meta, env_slot, final_boards, lengths, scores, stats); pass it to
    play_record_compact for the env-major flat buffer.  If stats["episodes"] < n the arena was too small (raise
    mean_steps)."""
    dev = subs.device
    mean = MEAN_STEPS_HINT[policy] if mean_steps is None else int(mean_steps)
    if n == 0:  # an empty shard (more ranks than envs): nothing to launch, empty results, zero statistics
        empty = lambda dt: torch.empty(0, dtype=dt, device=dev)  # noqa: E731
        return dict(arena_boards=empty(torch.int64), arena_meta=empty(torch.uint8), env_slot=empty(torch.int64),
                    final_boards=empty(torch.int64), lengths=empty(torch.int32), scores=empty(torch.int32),
                    stats=torch.zeros(N.PLAY_STATS_WORDS, dtype=torch.int64, device=dev) if stats is None else stats, policy=policy)
    with torch.cuda.device(dev):  # the arena follows the SM count of the GPU that will run the kernel
        slots = int(N.lib.g2048_play_record_arena_slots(n, subs.shape[0], mean))
    if slots <= 0:
        raise RuntimeError(f"g2048_play_record_arena_slots({n}, {subs.shape[0]}, {mean}) failed")
    work = torch.zeros(2, dtype=torch.int64, device=dev)
    if stats is None:
        stats = torch.zeros(N.PLAY_STATS_WORDS, dtype=torch.int64, device=dev)
    out = dict(
        arena_boards=torch.empty(slots, dtype=torch.int64, device=dev), arena_meta=torch.empty(slots, dtype=torch.uint8, device=dev),
        env_slot=torch.empty(n, dtype=torch.int64, device=dev), final_boards=torch.empty(n, dtype=torch.int64, device=dev),
        lengths=torch.zeros(n, dtype=torch.int32, device=dev), scores=torch.empty(n, dtype=torch.int32, device=dev),
        stats=stats, policy=policy)
    call("g2048_play_record", policy, ptr(_i32(subs)), subs.shape[0], batch_global, env_lo, n, rng_mode, ptr(work),
         ptr(out["arena_boards"]), ptr(out["arena_meta"]), slots, ptr(out["env_slot"]), ptr(out["final_boards"]),
         ptr(out["lengths"]), ptr(out["scores"]), ptr(stats), stream_ptr())
    return out


def play_record_compact(rec: dict, offsets: torch.Tensor, total: int) -> dict:
    """Arena of play_record -> flat env-major packed buffer (boards, meta, rewards, log_probs, values; max_rewards per
    env) with room for `total` steps; offsets = exclusive_scan(rec["lengths"]).  `total` is normally offsets[-1]; it may
    also be an estimate made before the statistics are read back -- steps beyond it are dropped (never written out of
    bounds), a larger one leaves the tail of the arrays unwritten: compare with the exact total afterwards."""
    dev = offsets.device
    n = rec["lengths"].shape[0]
    flat = dict(boards=torch.empty(total, dtype=torch.int64, device=dev), meta=torch.empty(total, dtype=torch.uint8, device=dev),
                rewards=torch.empty(total, dtype=torch.float32, device=dev),
                log_probs=torch.empty(total, dtype=torch.float32, device=dev),
                values=torch.empty(total, dtype=torch.float32, device=dev),
                max_rewards=torch.empty(n, dtype=torch.float32, device=dev))
    if n == 0:
        return flat
    call("g2048_play_record_compact", rec["policy"], ptr(rec["arena_boards"]), ptr(rec["arena_meta"]), ptr(rec["env_slot"]),
         ptr(rec["lengths"]), ptr(offsets), n, 0, total, ptr(flat["boards"]), ptr(flat["meta"]), ptr(flat["rewards"]),
         ptr(flat["log_probs"]), ptr(flat["values"]), ptr(flat["max_rewards"]), stream_ptr())
    return flat


PLAYOUT_STATS = np.dtype([("score_sum", "<u8"), ("score_sq_sum", "<u8"), ("steps_sum", "<u8"), ("playouts", "<u4"),
                          ("cut_short", "<u4")])  # G2048PlayoutStats (include/g2048.h)


def playout_values(policy: int, boards: torch.Tensor, subs: torch.Tensor, playouts: int, rng_mode: int,
                   board_ids: torch.Tensor | None = None, board_lo: int = 0, n_boards_global: int | None = None,
                   stats: torch.Tensor | None = None) -> dict:
    """Monte-Carlo playouts of the given bitboards (g2048_playout_values): for every (board, action) ``playouts`` games
    played to the end with the built-in ``policy`` after that action.  Board i has the global id ``board_ids[i]``
    (int64) or ``board_lo + i``; ``n_boards_global`` (default: ``board_lo + n``) sizes the batch the playouts' keys are
    split over.  ``subs``: sub keys as for ``play`` ([1+2t] act, [2+2t] step keys of playout step t).
    Returns dict(records (n, 4, 4) int64 -- the raw G2048PlayoutStats --, score_sum, score_sq_sum, steps_sum (n, 4)
    int64, playouts, cut_short (n, 4) int64, stats); ``stats`` (optional) accumulates g2048_play's statistics block."""
    dev = boards.device
    n = boards.shape[0]
    if n_boards_global is None:
        n_boards_global = max(board_lo + n, 1)
    if board_ids is not None:
        assert board_ids.dtype == torch.int64 and board_ids.shape[0] == n
    work = torch.zeros(2, dtype=torch.int64, device=dev)
    records = torch.empty((n, 4, 4), dtype=torch.int64, device=dev)
    call("g2048_playout_values", policy, ptr(boards), n, ptr(board_ids), board_lo, n_boards_global, playouts,
         ptr(_i32(subs)), subs.shape[0], rng_mode, ptr(work), ptr(records), ptr(stats), stream_ptr())
    last = records[..., 3]
    return dict(records=records, score_sum=records[..., 0], score_sq_sum=records[..., 1], steps_sum=records[..., 2],
                playouts=last & 0xFFFFFFFF, cut_short=last >> 32, stats=stats)


def expectimax_values(boards: torch.Tensor, depth: int, row_values: torch.Tensor, reward_weight: float = 0.0,
                      counters: torch.Tensor | None = None) -> torch.Tensor:
    """Depth-``depth`` expectimax values of the given bitboards over the row heuristic ``row_values`` (65 536 float32)
    (g2048_expectimax_values): (n, 4) float32 Q values, NaN where the action is illegal.  ``counters`` (optional, 2
    int64) accumulates the number of leaves (heuristic evaluations) and of chance nodes."""
    assert row_values.dtype == torch.float32 and row_values.numel() == 65536
    q = torch.empty((boards.shape[0], 4), dtype=torch.float32, device=boards.device)
    call("g2048_expectimax_values", ptr(boards), boards.shape[0], depth, ptr(row_values), float(reward_weight), ptr(q),
         ptr(counters), stream_ptr())
    return q


def td_scratch(device) -> torch.Tensor:
    """Zeroed scratch of g2048_td_train (every call leaves it zeroed, so one serves a whole training run)."""
    return torch.zeros(int(N.lib.g2048_td_scratch_bytes()) // 8, dtype=torch.int64, device=device)


def td_train(boards: torch.Tensor, after: torch.Tensor, scores: torch.Tensor, lengths: torch.Tensor,
             row_values: torch.Tensor, alpha: float, subs: torch.Tensor, rng_mode: int, scratch: torch.Tensor,
             stats: torch.Tensor | None = None) -> None:
    """``subs.shape[0]`` synchronous TD(0) steps of the row table (g2048_td_train), in place on the env state (boards /
    after int64, scores / lengths int32, n of each) and on ``row_values`` (65 536 float32).  ``scratch``: from
    ``td_scratch``.  ``stats`` (optional, 32 int64) accumulates the finished episodes in g2048_play's layout."""
    n = boards.shape[0]
    assert boards.dtype == after.dtype == torch.int64 and scores.dtype == lengths.dtype == torch.int32
    assert after.shape[0] == scores.shape[0] == lengths.shape[0] == n
    assert row_values.dtype == torch.float32 and row_values.numel() == 65536
    call("g2048_td_train", ptr(boards), ptr(after), ptr(scores), ptr(lengths), n, ptr(row_values), float(alpha),
         ptr(_i32(subs)), subs.shape[0], rng_mode, ptr(scratch), ptr(stats), stream_ptr())


def _placements_ptr(placements: np.ndarray) -> int:
    """Host pointer of an n-tuple placement array (G2048TuplePlacement[], 12 bytes each, C-contiguous)."""
    assert placements.dtype.itemsize == 12 and placements.flags.c_contiguous
    return placements.ctypes.data


def _stages_ptr(stages: np.ndarray, placements: np.ndarray, n_weights: int) -> tuple[np.ndarray, int]:
    """A checked copy of a G2048TupleStages record (``g2048.ntuple.STAGES_DTYPE``, ValueError when the staged entry
    points would reject it) and its host pointer; keep the copy alive over the call."""
    from .ntuple import check_stages

    st = check_stages(stages, placements, n_weights)
    return st, st.ctypes.data


def ntuple_td_scratch(n: int, placements: np.ndarray, n_weights: int, device) -> torch.Tensor:
    """Zeroed scratch of g2048_ntuple_td_train for n envs and this network (every call leaves it zeroed)."""
    size = int(N.lib.g2048_ntuple_td_scratch_bytes(n, placements.shape[0], n_weights))
    if size < 0:
        raise ValueError("ntuple_td_scratch: invalid sizes")
    return torch.zeros(size // 8, dtype=torch.int64, device=device)


def ntuple_td_train(boards: torch.Tensor, after: torch.Tensor, scores: torch.Tensor, lengths: torch.Tensor,
                    placements: np.ndarray, weights: torch.Tensor, alpha: float, subs: torch.Tensor, rng_mode: int,
                    scratch: torch.Tensor, stats: torch.Tensor | None = None, stages: np.ndarray | None = None) -> None:
    """``subs.shape[0]`` synchronous TD(0) steps of an n-tuple network (g2048_ntuple_td_train), in place on the env
    state (as ``td_train``) and on ``weights`` (float32, the network's n_weights).  ``placements``: the host
    G2048TuplePlacement array (``g2048.ntuple.PLACEMENT_DTYPE``).  ``scratch``: from ``ntuple_td_scratch``.
    ``stages``: None, or a G2048TupleStages record (``g2048.ntuple.STAGES_DTYPE``) for a multi-stage network
    (g2048_ntuple_staged_td_train)."""
    n = boards.shape[0]
    assert boards.dtype == after.dtype == torch.int64 and scores.dtype == lengths.dtype == torch.int32
    assert after.shape[0] == scores.shape[0] == lengths.shape[0] == n
    assert weights.dtype == torch.float32 and weights.is_contiguous()
    need = int(N.lib.g2048_ntuple_td_scratch_bytes(n, placements.shape[0], weights.numel()))
    if need < 0 or scratch.numel() * scratch.element_size() < need:
        raise ValueError(f"ntuple_td_train: scratch holds {scratch.numel() * scratch.element_size()} bytes, this batch "
                         f"and network need {need} (ntuple_td_scratch)")
    if stages is not None:
        st, st_ptr = _stages_ptr(stages, placements, weights.numel())
        call("g2048_ntuple_staged_td_train", ptr(boards), ptr(after), ptr(scores), ptr(lengths), n,
             _placements_ptr(placements), placements.shape[0], st_ptr, ptr(weights), weights.numel(), float(alpha),
             ptr(_i32(subs)), subs.shape[0], rng_mode, ptr(scratch), ptr(stats), stream_ptr())
        return
    call("g2048_ntuple_td_train", ptr(boards), ptr(after), ptr(scores), ptr(lengths), n, _placements_ptr(placements),
         placements.shape[0], ptr(weights), weights.numel(), float(alpha), ptr(_i32(subs)), subs.shape[0], rng_mode,
         ptr(scratch), ptr(stats), stream_ptr())


def ntuple_tc_scratch(n: int, placements: np.ndarray, n_weights: int, device) -> torch.Tensor:
    """Zeroed scratch of g2048_ntuple_tc_train for n envs and this network (every call leaves it zeroed)."""
    size = int(N.lib.g2048_ntuple_tc_scratch_bytes(n, placements.shape[0], n_weights))
    if size < 0:
        raise ValueError("ntuple_tc_scratch: invalid sizes")
    return torch.zeros(size // 8, dtype=torch.int64, device=device)


def ntuple_tc_train(boards: torch.Tensor, after: torch.Tensor, scores: torch.Tensor, lengths: torch.Tensor,
                    placements: np.ndarray, weights: torch.Tensor, err_sum: torch.Tensor, abs_err_sum: torch.Tensor,
                    alpha: float, subs: torch.Tensor, rng_mode: int, scratch: torch.Tensor,
                    stats: torch.Tensor | None = None, stages: np.ndarray | None = None) -> None:
    """``subs.shape[0]`` synchronous temporal-coherence steps of an n-tuple network (g2048_ntuple_tc_train): as
    ``ntuple_td_train``, and in place on ``err_sum`` / ``abs_err_sum`` (E and A: float64, the network's n_weights
    each; zeros at the start of a run).  ``scratch``: from ``ntuple_tc_scratch``.  ``stages``: as for
    ``ntuple_td_train`` (g2048_ntuple_staged_tc_train)."""
    n = boards.shape[0]
    assert boards.dtype == after.dtype == torch.int64 and scores.dtype == lengths.dtype == torch.int32
    assert after.shape[0] == scores.shape[0] == lengths.shape[0] == n
    assert weights.dtype == torch.float32 and weights.is_contiguous()
    for s in (err_sum, abs_err_sum):
        assert s.dtype == torch.float64 and s.is_contiguous() and s.numel() == weights.numel()
    need = int(N.lib.g2048_ntuple_tc_scratch_bytes(n, placements.shape[0], weights.numel()))
    if need < 0 or scratch.numel() * scratch.element_size() < need:
        raise ValueError(f"ntuple_tc_train: scratch holds {scratch.numel() * scratch.element_size()} bytes, this batch "
                         f"and network need {need} (ntuple_tc_scratch)")
    if stages is not None:
        st, st_ptr = _stages_ptr(stages, placements, weights.numel())
        call("g2048_ntuple_staged_tc_train", ptr(boards), ptr(after), ptr(scores), ptr(lengths), n,
             _placements_ptr(placements), placements.shape[0], st_ptr, ptr(weights), weights.numel(), ptr(err_sum),
             ptr(abs_err_sum), float(alpha), ptr(_i32(subs)), subs.shape[0], rng_mode, ptr(scratch), ptr(stats),
             stream_ptr())
        return
    call("g2048_ntuple_tc_train", ptr(boards), ptr(after), ptr(scores), ptr(lengths), n, _placements_ptr(placements),
         placements.shape[0], ptr(weights), weights.numel(), ptr(err_sum), ptr(abs_err_sum), float(alpha),
         ptr(_i32(subs)), subs.shape[0], rng_mode, ptr(scratch), ptr(stats), stream_ptr())


def _lambda_checks(who: str, boards: torch.Tensor, placements: np.ndarray, weights: torch.Tensor, lam: float,
                   hist_after: torch.Tensor, hist_delta: torch.Tensor, scratch: torch.Tensor, tc: bool) -> int:
    """The checks of the lambda wrappers (ValueError); returns the horizon h = hist_after.shape[0].  ``scratch`` None
    skips the scratch size (the carousel wrappers check their own)."""
    from .ntuple import MAX_HORIZON

    n = boards.shape[0]
    lam = float(lam)
    if not (math.isfinite(lam) and 0.0 <= lam <= 1.0):
        raise ValueError(f"{who}: lambda must be finite and in [0, 1], got {lam}")
    if hist_after.dim() != 2 or not 1 <= hist_after.shape[0] <= MAX_HORIZON:
        raise ValueError(f"{who}: hist_after must be (h, n) with h in [1, {MAX_HORIZON}], got {tuple(hist_after.shape)}")
    h = hist_after.shape[0]
    if tuple(hist_after.shape) != (h, n) or tuple(hist_delta.shape) != (h, n):
        raise ValueError(f"{who}: hist_after and hist_delta must be ({h}, {n}), got {tuple(hist_after.shape)} and "
                         f"{tuple(hist_delta.shape)}")
    if hist_after.dtype != torch.int64 or hist_delta.dtype != torch.float32:
        raise ValueError(f"{who}: hist_after must be int64 and hist_delta float32, got {hist_after.dtype} and "
                         f"{hist_delta.dtype}")
    for t in (hist_after, hist_delta):
        if t.device != boards.device or not t.is_contiguous():
            raise ValueError(f"{who}: the rings must be contiguous and on {boards.device}")
    if n * h > 1 << 20:
        raise ValueError(f"{who}: n * h must be <= 2^20, got {n} * {h}")
    if scratch is None:
        return h
    size_of = N.lib.g2048_ntuple_tc_scratch_bytes if tc else N.lib.g2048_ntuple_td_scratch_bytes
    need = int(size_of(n * h, placements.shape[0], weights.numel()))
    if need < 0 or scratch.numel() * scratch.element_size() < need:
        raise ValueError(f"{who}: scratch holds {scratch.numel() * scratch.element_size()} bytes, this batch, horizon "
                         f"and network need {need} (ntuple_{'tc' if tc else 'td'}_scratch(n * h, ...))")
    return h


def ntuple_lambda_td_train(boards: torch.Tensor, after: torch.Tensor, scores: torch.Tensor, lengths: torch.Tensor,
                           placements: np.ndarray, weights: torch.Tensor, alpha: float, lam: float,
                           hist_after: torch.Tensor, hist_delta: torch.Tensor, subs: torch.Tensor, rng_mode: int,
                           scratch: torch.Tensor, stats: torch.Tensor | None = None,
                           stages: np.ndarray | None = None) -> None:
    """``subs.shape[0]`` synchronous delayed TD(lambda) steps of an n-tuple network (g2048_ntuple_lambda_td_train): as
    ``ntuple_td_train``, with every afterstate updated h - 1 steps late by the lambda-weighted sum of its h errors.
    ``hist_after`` (int64) and ``hist_delta`` (float32) are the (h, n) window rings, updated in place (zeros at the
    start of a run); h = ``hist_after.shape[0]``, 1..8.  ``scratch``: ``ntuple_td_scratch(n * h, ...)``.  ``stages``:
    None for one stage, or a G2048TupleStages record."""
    n = boards.shape[0]
    assert boards.dtype == after.dtype == torch.int64 and scores.dtype == lengths.dtype == torch.int32
    assert after.shape[0] == scores.shape[0] == lengths.shape[0] == n
    assert weights.dtype == torch.float32 and weights.is_contiguous()
    h = _lambda_checks("ntuple_lambda_td_train", boards, placements, weights, lam, hist_after, hist_delta, scratch,
                       False)
    st, st_ptr = _stages_ptr(stages, placements, weights.numel()) if stages is not None else (None, None)
    call("g2048_ntuple_lambda_td_train", ptr(boards), ptr(after), ptr(scores), ptr(lengths), n,
         _placements_ptr(placements), placements.shape[0], st_ptr, ptr(weights), weights.numel(), float(alpha),
         float(lam), h, ptr(hist_after), ptr(hist_delta), ptr(_i32(subs)), subs.shape[0], rng_mode, ptr(scratch),
         ptr(stats), stream_ptr())


def ntuple_lambda_tc_train(boards: torch.Tensor, after: torch.Tensor, scores: torch.Tensor, lengths: torch.Tensor,
                           placements: np.ndarray, weights: torch.Tensor, err_sum: torch.Tensor,
                           abs_err_sum: torch.Tensor, alpha: float, lam: float, hist_after: torch.Tensor,
                           hist_delta: torch.Tensor, subs: torch.Tensor, rng_mode: int, scratch: torch.Tensor,
                           stats: torch.Tensor | None = None, stages: np.ndarray | None = None) -> None:
    """``subs.shape[0]`` synchronous delayed TC(lambda) steps (g2048_ntuple_lambda_tc_train): ``ntuple_tc_train``'s
    E / A update with ``ntuple_lambda_td_train``'s window.  ``scratch``: ``ntuple_tc_scratch(n * h, ...)``."""
    n = boards.shape[0]
    assert boards.dtype == after.dtype == torch.int64 and scores.dtype == lengths.dtype == torch.int32
    assert after.shape[0] == scores.shape[0] == lengths.shape[0] == n
    assert weights.dtype == torch.float32 and weights.is_contiguous()
    for s in (err_sum, abs_err_sum):
        assert s.dtype == torch.float64 and s.is_contiguous() and s.numel() == weights.numel()
    h = _lambda_checks("ntuple_lambda_tc_train", boards, placements, weights, lam, hist_after, hist_delta, scratch,
                       True)
    st, st_ptr = _stages_ptr(stages, placements, weights.numel()) if stages is not None else (None, None)
    call("g2048_ntuple_lambda_tc_train", ptr(boards), ptr(after), ptr(scores), ptr(lengths), n,
         _placements_ptr(placements), placements.shape[0], st_ptr, ptr(weights), weights.numel(), ptr(err_sum),
         ptr(abs_err_sum), float(alpha), float(lam), h, ptr(hist_after), ptr(hist_delta), ptr(_i32(subs)),
         subs.shape[0], rng_mode, ptr(scratch), ptr(stats), stream_ptr())


def ntuple_carousel_scratch(n: int, horizon: int, placements: np.ndarray, n_weights: int, tc: bool,
                            device) -> torch.Tensor:
    """Zeroed scratch of g2048_ntuple_carousel_td_train (tc False) / _tc_train (tc True) for n envs, window h =
    ``horizon`` and this network (every call leaves it zeroed)."""
    size = int(N.lib.g2048_ntuple_carousel_scratch_bytes(n, int(horizon), placements.shape[0], n_weights, int(bool(tc))))
    if size < 0:
        raise ValueError("ntuple_carousel_scratch: invalid sizes")
    return torch.zeros(size // 8, dtype=torch.int64, device=device)


def _carousel_checks(who: str, boards: torch.Tensor, placements: np.ndarray, weights: torch.Tensor, lam: float,
                     hist_after, hist_delta, start_stage: torch.Tensor, stage_pool: torch.Tensor, stages,
                     scratch: torch.Tensor, tc: bool) -> tuple[int, int, int, np.ndarray, int]:
    """The checks of the carousel wrappers (ValueError): the lambda wrappers' when h > 1, the stages (S >= 2) and the
    carousel arrays.  Returns (h, hist_after pointer, hist_delta pointer, the stages' checked copy, its pointer);
    ``hist_after`` / ``hist_delta`` None means h = 1 without rings."""
    n = boards.shape[0]
    if stages is None:
        raise ValueError(f"{who}: carousel shaping needs a multi-stage network (stages with S >= 2)")
    st, st_ptr = _stages_ptr(stages, placements, weights.numel())
    if int(st["n_thresholds"][0]) < 1:
        raise ValueError(f"{who}: carousel shaping needs a multi-stage network (stages with S >= 2), got one stage")
    S = int(st["n_thresholds"][0]) + 1
    if (hist_after is None) != (hist_delta is None):
        raise ValueError(f"{who}: hist_after and hist_delta must both be given or both be None")
    if hist_after is None:
        lam = float(lam)
        if not (math.isfinite(lam) and 0.0 <= lam <= 1.0):
            raise ValueError(f"{who}: lambda must be finite and in [0, 1], got {lam}")
        h, ha_ptr, hd_ptr = 1, None, None
    else:
        h = _lambda_checks(who, boards, placements, weights, lam, hist_after, hist_delta, None, tc)
        ha_ptr, hd_ptr = ptr(hist_after), ptr(hist_delta)
    if not (isinstance(start_stage, torch.Tensor) and start_stage.dtype == torch.int32
            and tuple(start_stage.shape) == (n,)):
        raise ValueError(f"{who}: start_stage must be an int32 tensor of shape ({n},)")
    if not (isinstance(stage_pool, torch.Tensor) and stage_pool.dtype == torch.int64
            and tuple(stage_pool.shape) == (S - 1, n)):
        raise ValueError(f"{who}: stage_pool must be an int64 tensor of shape ({S - 1}, {n})")
    for t in (start_stage, stage_pool):
        if t.device != boards.device or not t.is_contiguous():
            raise ValueError(f"{who}: start_stage and stage_pool must be contiguous and on {boards.device}")
    need = int(N.lib.g2048_ntuple_carousel_scratch_bytes(n, h, placements.shape[0], weights.numel(), int(tc)))
    if need < 0 or scratch.numel() * scratch.element_size() < need:
        raise ValueError(f"{who}: scratch holds {scratch.numel() * scratch.element_size()} bytes, this batch, horizon "
                         f"and network need {need} (ntuple_carousel_scratch)")
    return h, ha_ptr, hd_ptr, st, st_ptr


def ntuple_carousel_td_train(boards: torch.Tensor, after: torch.Tensor, scores: torch.Tensor, lengths: torch.Tensor,
                             placements: np.ndarray, weights: torch.Tensor, alpha: float, lam: float,
                             hist_after: torch.Tensor | None, hist_delta: torch.Tensor | None,
                             start_stage: torch.Tensor, stage_pool: torch.Tensor, subs: torch.Tensor, rng_mode: int,
                             scratch: torch.Tensor, stats: torch.Tensor | None = None,
                             stages: np.ndarray | None = None) -> None:
    """``subs.shape[0]`` synchronous TD steps of a multi-stage network with carousel shaping
    (g2048_ntuple_carousel_td_train): ``ntuple_lambda_td_train`` (``hist_after`` / ``hist_delta`` None: h = 1, TD(0)),
    where an episode that ends restarts, in turn, at the opening or from a board at which an earlier episode entered
    the next stage.  ``start_stage`` (int32, (n,)) and ``stage_pool`` (int64, (S - 1, n)) are updated in place (zeros
    at the start of a run).  ``stages``: the network's G2048TupleStages record, S >= 2, required.  ``scratch``:
    ``ntuple_carousel_scratch(n, h, ..., tc=False)``."""
    n = boards.shape[0]
    assert boards.dtype == after.dtype == torch.int64 and scores.dtype == lengths.dtype == torch.int32
    assert after.shape[0] == scores.shape[0] == lengths.shape[0] == n
    assert weights.dtype == torch.float32 and weights.is_contiguous()
    h, ha, hd, st, st_ptr = _carousel_checks("ntuple_carousel_td_train", boards, placements, weights, lam, hist_after,
                                             hist_delta, start_stage, stage_pool, stages, scratch, False)
    call("g2048_ntuple_carousel_td_train", ptr(boards), ptr(after), ptr(scores), ptr(lengths), n,
         _placements_ptr(placements), placements.shape[0], st_ptr, ptr(weights), weights.numel(), float(alpha),
         float(lam), h, ha, hd, ptr(start_stage), ptr(stage_pool), ptr(_i32(subs)), subs.shape[0], rng_mode,
         ptr(scratch), ptr(stats), stream_ptr())


def ntuple_carousel_tc_train(boards: torch.Tensor, after: torch.Tensor, scores: torch.Tensor, lengths: torch.Tensor,
                             placements: np.ndarray, weights: torch.Tensor, err_sum: torch.Tensor,
                             abs_err_sum: torch.Tensor, alpha: float, lam: float, hist_after: torch.Tensor | None,
                             hist_delta: torch.Tensor | None, start_stage: torch.Tensor, stage_pool: torch.Tensor,
                             subs: torch.Tensor, rng_mode: int, scratch: torch.Tensor,
                             stats: torch.Tensor | None = None, stages: np.ndarray | None = None) -> None:
    """``subs.shape[0]`` synchronous TC steps with carousel shaping (g2048_ntuple_carousel_tc_train):
    ``ntuple_lambda_tc_train``'s E / A update with ``ntuple_carousel_td_train``'s restarts.  ``scratch``:
    ``ntuple_carousel_scratch(n, h, ..., tc=True)``."""
    n = boards.shape[0]
    assert boards.dtype == after.dtype == torch.int64 and scores.dtype == lengths.dtype == torch.int32
    assert after.shape[0] == scores.shape[0] == lengths.shape[0] == n
    assert weights.dtype == torch.float32 and weights.is_contiguous()
    for s in (err_sum, abs_err_sum):
        assert s.dtype == torch.float64 and s.is_contiguous() and s.numel() == weights.numel()
    h, ha, hd, st, st_ptr = _carousel_checks("ntuple_carousel_tc_train", boards, placements, weights, lam, hist_after,
                                             hist_delta, start_stage, stage_pool, stages, scratch, True)
    call("g2048_ntuple_carousel_tc_train", ptr(boards), ptr(after), ptr(scores), ptr(lengths), n,
         _placements_ptr(placements), placements.shape[0], st_ptr, ptr(weights), weights.numel(), ptr(err_sum),
         ptr(abs_err_sum), float(alpha), float(lam), h, ha, hd, ptr(start_stage), ptr(stage_pool), ptr(_i32(subs)),
         subs.shape[0], rng_mode, ptr(scratch), ptr(stats), stream_ptr())


def expectimax_values_ntuple(boards: torch.Tensor, depth: int, placements: np.ndarray, weights: torch.Tensor,
                             reward_weight: float = 0.0, counters: torch.Tensor | None = None,
                             stages: np.ndarray | None = None) -> torch.Tensor:
    """``expectimax_values`` with V of an n-tuple network at the leaves (g2048_expectimax_values_ntuple): (n, 4)
    float32 Q values, NaN where the action is illegal.  ``stages``: as for ``ntuple_td_train``
    (g2048_expectimax_values_ntuple_staged)."""
    assert weights.dtype == torch.float32 and weights.is_contiguous()
    if stages is not None:
        st, st_ptr = _stages_ptr(stages, placements, weights.numel())
        q = torch.empty((boards.shape[0], 4), dtype=torch.float32, device=boards.device)
        call("g2048_expectimax_values_ntuple_staged", ptr(boards), boards.shape[0], depth, _placements_ptr(placements),
             placements.shape[0], st_ptr, ptr(weights), weights.numel(), float(reward_weight), ptr(q), ptr(counters),
             stream_ptr())
        return q
    q = torch.empty((boards.shape[0], 4), dtype=torch.float32, device=boards.device)
    call("g2048_expectimax_values_ntuple", ptr(boards), boards.shape[0], depth, _placements_ptr(placements),
         placements.shape[0], ptr(weights), weights.numel(), float(reward_weight), ptr(q), ptr(counters), stream_ptr())
    return q


def play_host(policy: int, seed: int, batch_global: int, rng_mode: int, env_lo: int = 0, n: int | None = None,
              key: np.ndarray | None = None, per_env: bool = True, pinned: bool = False):
    """The host-buffer C entry point (numpy in / numpy out; copies and syncs inside the call).
    pinned=True: the per-env results are one array of 16-byte records (EPISODE_RESULT) in page-locked host memory,
    which the play kernel writes directly, one PCIe write per finished episode and no copies after the kernel
    (g2048_play_host_packed); final_boards / lengths / scores are strided views of it and stay valid as long as they
    are referenced."""
    N.require_cuda()
    n = batch_global - env_lo if n is None else n
    stats = np.zeros(N.PLAY_STATS_WORDS, np.uint64)
    key_io = None if key is None else np.ascontiguousarray(key, np.uint32)
    as_p = lambda a: None if a is None else a.ctypes.data  # noqa: E731
    if pinned and per_env:
        records = torch.empty((n, 2), dtype=torch.int64, pin_memory=True).numpy().view(EPISODE_RESULT).reshape(n)
        call("g2048_play_host_packed", policy, key_words(seed)[1], as_p(key_io), batch_global, env_lo, n, rng_mode,
             as_p(records), as_p(stats))
        return dict(final_boards=records["board"], lengths=records["length"], scores=records["score"], stats=stats,
                    key=key_io, records=records)
    boards = np.empty(n, np.uint64) if per_env else None
    lengths = np.empty(n, np.uint32) if per_env else None
    scores = np.empty(n, np.uint32) if per_env else None
    call("g2048_play_host", policy, key_words(seed)[1], as_p(key_io), batch_global, env_lo, n, rng_mode,
         as_p(boards), as_p(lengths), as_p(scores), as_p(stats))
    return dict(final_boards=boards, lengths=lengths, scores=scores, stats=stats, key=key_io)


def rollout_steps(policy: int, boards, status, subs, n_steps: int, t0: int, batch_global: int, env_lo: int,
                  rng_mode: int, rec_boards, rec_meta, rec_rewards, rec_log_probs, counters) -> None:
    n = boards.shape[0]
    call("g2048_rollout_steps", policy, ptr(boards), ptr(status), ptr(_i32(subs)), n_steps, t0, batch_global, env_lo, n,
         rng_mode, ptr(rec_boards), ptr(rec_meta), ptr(rec_rewards), ptr(rec_log_probs), ptr(counters), stream_ptr())


def rollout_steps_live(policy: int, boards, status, subs, n_steps: int, t0: int, batch_global: int, env_lo: int,
                       rng_mode: int, env_ids: torch.Tensor, rec_boards, rec_meta, rec_rewards, rec_log_probs, counters) -> None:
    """rollout_steps for the envs listed in env_ids (int64 local indices) only; a finished env leaves the loop."""
    n = boards.shape[0]
    assert env_ids.dtype == torch.int64
    call("g2048_rollout_steps_live", policy, ptr(boards), ptr(status), ptr(_i32(subs)), n_steps, t0, batch_global, env_lo, n,
         rng_mode, ptr(env_ids), env_ids.shape[0], ptr(rec_boards), ptr(rec_meta), ptr(rec_rewards), ptr(rec_log_probs),
         ptr(counters), stream_ptr())


# ------------------------------------------------------------------------------------------- policy logits
def policy_step(boards, status, logits, values, use_mask: bool, sample: bool, auto_reset: bool, sub_act, sub_step,
                batch_global: int, env_lo: int, rng_mode: int, rec_boards=None, rec_meta=None, rec_rewards=None,
                rec_log_probs=None, rec_values=None, actions_out=None) -> None:
    n = boards.shape[0]
    assert logits.dtype == torch.float32 and logits.shape == (n, 4)
    if values is not None:
        assert values.dtype == torch.float32 and values.numel() == n
    call("g2048_policy_step", ptr(boards), ptr(status), ptr(logits), ptr(values), int(use_mask), int(sample),
         int(auto_reset), ptr(sub_act), ptr(sub_step), batch_global, env_lo, n, rng_mode, ptr(rec_boards),
         ptr(rec_meta), ptr(rec_rewards), ptr(rec_log_probs), ptr(rec_values), ptr(actions_out), stream_ptr())


def policy_step_at(boards, status, logits, values, use_mask: bool, sample: bool, auto_reset: bool, subs, step_index,
                   batch_global: int, env_lo: int, rng_mode: int, rec_boards=None, rec_meta=None, rec_rewards=None,
                   rec_log_probs=None, rec_values=None, actions_out=None) -> None:
    """policy_step whose step number t is read from `step_index` (int32 device scalar): sub keys subs[2t], subs[2t+1]
    and record slot t of the (steps, n) record tensors.  Every argument is replay-stable, so the launch can sit in
    a captured CUDA graph; follow it with counter_add(step_index)."""
    n = boards.shape[0]
    assert logits.dtype == torch.float32 and logits.shape == (n, 4)
    assert step_index.dtype == torch.int32 and subs.dtype == torch.int32
    if values is not None:
        assert values.dtype == torch.float32 and values.numel() == n
    call("g2048_policy_step_at", ptr(boards), ptr(status), ptr(logits), ptr(values), int(use_mask), int(sample),
         int(auto_reset), ptr(subs), ptr(step_index), batch_global, env_lo, n, rng_mode, ptr(rec_boards),
         ptr(rec_meta), ptr(rec_rewards), ptr(rec_log_probs), ptr(rec_values), ptr(actions_out), stream_ptr())


def policy_step_live(boards, status, logits, values, use_mask: bool, sample: bool, auto_reset: bool, sub_act, sub_step,
                     env_ids: torch.Tensor, batch_global: int, env_lo: int, rng_mode: int, rec_boards=None, rec_meta=None,
                     rec_rewards=None, rec_log_probs=None, rec_values=None, actions_out=None) -> None:
    """policy_step for the live envs only: logits / values have one row per entry of env_ids (int64 local env
    indices); state, RNG counters and record slots are the envs' own."""
    m, n = env_ids.shape[0], boards.shape[0]
    assert env_ids.dtype == torch.int64 and logits.dtype == torch.float32 and logits.shape == (m, 4)
    if values is not None:
        assert values.dtype == torch.float32 and values.numel() == m
    call("g2048_policy_step_live", ptr(boards), ptr(status), ptr(logits), ptr(values), int(use_mask), int(sample),
         int(auto_reset), ptr(sub_act), ptr(sub_step), ptr(env_ids), m, batch_global, env_lo, n, rng_mode, ptr(rec_boards),
         ptr(rec_meta), ptr(rec_rewards), ptr(rec_log_probs), ptr(rec_values), ptr(actions_out), stream_ptr())


def policy_step_obs(boards, status, logits, values, use_mask: bool, sample: bool, auto_reset: bool, subs, step_index,
                    batch_global: int, env_lo: int, rng_mode: int, obs_next: torch.Tensor, rec_boards=None, rec_meta=None,
                    rec_rewards=None, rec_log_probs=None, rec_values=None, actions_out=None, counters=None,
                    advance_step: bool = False) -> None:
    """policy_step_at fused with expand_obs of the stepped boards: `obs_next` (n,16,31) receives the observation the
    network reads on the next step.  step_index None: t = 0 -- `subs` starts at this step's act sub key and the record
    tensors are this step's rows.  counters: int64[2] (accumulated): envs that terminated on this step, reward sum.
    advance_step: the kernel itself adds 1 to step_index when it is done (graph replay without a counter kernel)."""
    n = boards.shape[0]
    assert logits.dtype == torch.float32 and logits.shape == (n, 4) and subs.dtype == torch.int32
    assert obs_next.shape == (n, 16, 31) and obs_next.is_contiguous()
    if values is not None:
        assert values.dtype == torch.float32 and values.numel() == n
    if step_index is not None:
        assert step_index.dtype == torch.int32
    call("g2048_policy_step_obs", ptr(boards), ptr(status), ptr(logits), ptr(values), int(use_mask), int(sample),
         int(auto_reset), ptr(subs), ptr(step_index), int(advance_step), batch_global, env_lo, n, rng_mode, ptr(rec_boards),
         ptr(rec_meta), ptr(rec_rewards), ptr(rec_log_probs), ptr(rec_values), ptr(actions_out), _OBS_DTYPES[obs_next.dtype], ptr(obs_next),
         ptr(counters), stream_ptr())


def counter_add(counter: torch.Tensor, delta: int = 1) -> None:
    """counter (int32 device scalar) += delta, on the stream."""
    assert counter.dtype == torch.int32
    call("g2048_counter_add", ptr(counter), int(delta), stream_ptr())


def sample_logits(logits, status, use_mask: bool, sample: bool, sub_act, batch_global: int, env_lo: int,
                  rng_mode: int, want_entropy: bool = False):
    n = logits.shape[0]
    assert logits.dtype == torch.float32 and logits.shape == (n, 4)
    actions = torch.empty(n, dtype=torch.int32, device=logits.device)
    log_probs = torch.empty(n, dtype=torch.float32, device=logits.device)
    entropy = torch.empty(n, dtype=torch.float32, device=logits.device) if want_entropy else None
    call("g2048_sample_logits", ptr(logits), ptr(status), int(use_mask), int(sample), ptr(sub_act), batch_global,
         env_lo, n, rng_mode, ptr(actions), ptr(log_probs), ptr(entropy), stream_ptr())
    return actions, log_probs, entropy


def evaluate_logits(logits, mask_bits, use_mask: bool, actions):
    n = logits.shape[0]
    assert logits.dtype == torch.float32 and logits.shape == (n, 4)
    log_probs = torch.empty(n, dtype=torch.float32, device=logits.device)
    entropy = torch.empty(n, dtype=torch.float32, device=logits.device)
    call("g2048_evaluate_logits", ptr(logits), ptr(mask_bits), int(use_mask), ptr(_i32(actions)), n, ptr(log_probs),
         ptr(entropy), stream_ptr())
    return log_probs, entropy


# ------------------------------------------------------------------------------------------- records
_OBS_DTYPES = {torch.bool: N.OBS_BOOL, torch.uint8: N.OBS_BOOL, torch.float32: N.OBS_F32, torch.bfloat16: N.OBS_BF16}


def expand_obs(boards: torch.Tensor, dtype=torch.float32, rows: int = 0, n_cols: int = 0, out=None,
               entry: str = "g2048_expand_obs") -> torch.Tensor:
    """One-hot (n,16,31).  rows/n_cols > 0: boards are (rows, n_cols) time-major, output is env-major.
    entry: another entry point with the same signature (the tests' legacy build has g2048_expand_obs_v1)."""
    n = boards.numel()
    if out is None:
        out = torch.empty((n, 16, 31), dtype=dtype, device=boards.device)
    call(entry, ptr(boards), n, _OBS_DTYPES[dtype], ptr(out), rows, n_cols, stream_ptr())
    return out


def expand_obs_gather(boards: torch.Tensor, indices: torch.Tensor, dtype=torch.float32, out=None) -> torch.Tensor:
    """One-hot (m,16,31) of boards[indices] (int64 indices) without materialising the gathered boards."""
    m = indices.shape[0]
    if out is None:
        out = torch.empty((m, 16, 31), dtype=dtype, device=boards.device)
    call("g2048_expand_obs_gather", ptr(boards), ptr(indices), m, _OBS_DTYPES[dtype], ptr(out), stream_ptr())
    return out


def pack_obs(obs: torch.Tensor) -> torch.Tensor:
    """One-hot (n,16,31) bool/uint8/float32 -> (n,) int64 bitboards (argmax over channels)."""
    n = obs.numel() // 496
    code = N.OBS_F32 if obs.dtype == torch.float32 else _OBS_DTYPES[obs.dtype]
    if code == N.OBS_BF16:
        raise ValueError("pack_obs takes bool/uint8/float32 observations")
    boards = torch.empty(n, dtype=torch.int64, device=obs.device)
    call("g2048_pack_obs", ptr(obs), code, n, ptr(boards), stream_ptr())
    return boards


def unpack_status(status: torch.Tensor):
    """status bytes -> (legal_action_mask (n,4) bool, terminated (n,) bool)."""
    n = status.shape[0]
    masks = torch.empty((n, 4), dtype=torch.bool, device=status.device)
    term = torch.empty(n, dtype=torch.bool, device=status.device)
    call("g2048_unpack_status", ptr(status), n, ptr(masks), ptr(term), stream_ptr())
    return masks, term


def unpack_records(rec_meta, rec_rewards, rec_log_probs, rec_values, t_steps: int, n: int):
    """(T,B) time-major records -> dict of (B,T) env-major reference arrays (device)."""
    dev = rec_meta.device
    out = dict(
        actions=torch.empty((n, t_steps), dtype=torch.int32, device=dev),
        action_masks=torch.empty((n, t_steps, 4), dtype=torch.bool, device=dev),
        terminations=torch.empty((n, t_steps), dtype=torch.bool, device=dev),
        rewards=torch.empty((n, t_steps), dtype=torch.float32, device=dev),
        log_probs=torch.empty((n, t_steps), dtype=torch.float32, device=dev) if rec_log_probs is not None else None,
        values=torch.empty((n, t_steps), dtype=torch.float32, device=dev) if rec_values is not None else None,
    )
    call("g2048_unpack_records", ptr(rec_meta), ptr(rec_rewards), ptr(rec_log_probs), ptr(rec_values), t_steps, n,
         ptr(out["actions"]), ptr(out["action_masks"]), ptr(out["terminations"]), ptr(out["rewards"]),
         ptr(out["log_probs"]), ptr(out["values"]), stream_ptr())
    return out


def episode_lengths(rec_meta, t_steps: int, n: int) -> torch.Tensor:
    out = torch.empty(n, dtype=torch.int32, device=rec_meta.device)
    call("g2048_episode_lengths", ptr(rec_meta), t_steps, n, ptr(out), stream_ptr())
    return out


def exclusive_scan(x: torch.Tensor) -> torch.Tensor:
    out = torch.empty(x.shape[0] + 1, dtype=torch.int64, device=x.device)
    call("g2048_exclusive_scan", ptr(_i32(x)), x.shape[0], ptr(out), stream_ptr())
    return out


def compact_records(rec_boards, rec_meta, rec_rewards, rec_log_probs, rec_values, t_steps: int, n: int, lengths,
                    offsets, out_base: int, boards, meta, rewards, log_probs, values) -> None:
    call("g2048_compact_records", ptr(rec_boards), ptr(rec_meta), ptr(rec_rewards), ptr(rec_log_probs),
         ptr(rec_values), t_steps, n, ptr(lengths), ptr(offsets), out_base, ptr(boards), ptr(meta), ptr(rewards),
         ptr(log_probs), ptr(values), stream_ptr())


def first_done_rows(terminations: torch.Tensor) -> torch.Tensor:
    """(n_envs, t_steps) uint8/bool env-major -> int32 (n_envs,): first done + 1, 0 if the env never terminates."""
    n_envs, t_steps = terminations.shape
    term = terminations if terminations.dtype == torch.uint8 else terminations.to(torch.uint8)
    out = torch.empty(n_envs, dtype=torch.int32, device=terminations.device)
    call("g2048_first_done_rows", ptr(term.contiguous()), n_envs, t_steps, ptr(out), stream_ptr())
    return out


def compact_rows(src: torch.Tensor, lengths: torch.Tensor, offsets: torch.Tensor, total: int) -> torch.Tensor:
    """Env-major (n_envs, t_steps, *row) -> flat (total, *row): the rows t < lengths[e] of every env, env after env."""
    n_envs, t_steps = src.shape[:2]
    row_bytes = src[0, 0].numel() * src.element_size() if src.dim() > 2 else src.element_size()
    out = torch.empty((total, *src.shape[2:]), dtype=src.dtype, device=src.device)
    if total:
        call("g2048_compact_rows", ptr(src.contiguous()), n_envs, t_steps, row_bytes, ptr(lengths), ptr(offsets), 0, ptr(out),
             stream_ptr())
    return out


def meta_dones(meta: torch.Tensor) -> torch.Tensor:
    """Packed meta bytes -> uint8 done flags only (no one-hot actions / masks are materialised)."""
    n = meta.shape[0]
    term = torch.empty(n, dtype=torch.uint8, device=meta.device)
    call("g2048_unpack_flat_meta", ptr(meta), n, None, None, ptr(term), stream_ptr())
    return term


def unpack_flat_meta(meta: torch.Tensor):
    n = meta.shape[0]
    dev = meta.device
    actions = torch.empty((n, 4), dtype=torch.float32, device=dev)
    masks = torch.empty((n, 4), dtype=torch.bool, device=dev)
    term = torch.empty(n, dtype=torch.bool, device=dev)
    call("g2048_unpack_flat_meta", ptr(meta), n, ptr(actions), ptr(masks), ptr(term), stream_ptr())
    return actions, masks, term


def random_subset(n: int, m: int, key, device, first: int = 0, out: torch.Tensor | None = None) -> torch.Tensor:
    """P(first), ..., P(first + m - 1) for the keyed pseudo-random bijection P of [0, n) (g2048_random_subset):
    m distinct random buffer positions in O(m) -- torch.randperm(n)[:m] without sorting n keys.  key: two uint32
    words (or one int seed)."""
    N.require_cuda()
    k0, k1 = (0, int(key)) if isinstance(key, int) else (int(key[0]), int(key[1]))
    if out is None:
        out = torch.empty(m, dtype=torch.int64, device=device)
    call("g2048_random_subset", k0 & 0xFFFFFFFF, k1 & 0xFFFFFFFF, n, first, m, ptr(out), stream_ptr())
    return out


def minibatch_buffers(m: int, device, obs_dtype=torch.float32, with_gae: bool = True) -> dict:
    """Output tensors of gather_minibatch for m samples (pass them back through `out=` to reuse them)."""
    dev = device
    return dict(
        observations=torch.empty((m, 16, 31), dtype=obs_dtype, device=dev) if obs_dtype is not None else None,
        actions=torch.empty(m, dtype=torch.int64, device=dev),
        action_masks=torch.empty((m, 4), dtype=torch.bool, device=dev),
        log_probs=torch.empty(m, dtype=torch.float32, device=dev),
        values=torch.empty(m, dtype=torch.float32, device=dev),
        advantages=torch.empty(m, dtype=torch.float32, device=dev) if with_gae else None,
        returns=torch.empty(m, dtype=torch.float32, device=dev) if with_gae else None,
        boards=torch.empty(m, dtype=torch.int64, device=dev) if obs_dtype is None else None,
    )


def gather_minibatch(indices: torch.Tensor, packed: dict, adv: torch.Tensor | None, ret: torch.Tensor | None,
                     obs_dtype=torch.float32, out: dict | None = None) -> dict:
    """Minibatch `indices` (int64, device) of a flat packed buffer (RolloutBuffer.get_packed()) as the
    tensors a PPO update consumes, in one launch (the observation kernel gathers the scalars too).  obs_dtype=None: no
    observations -- the batch carries the gathered bitboards under "boards" for ppo.board_embedding.
    out: tensors from minibatch_buffers() of the same size to write into instead of allocating."""
    m = indices.shape[0]
    if out is None:
        out = minibatch_buffers(m, indices.device, obs_dtype, adv is not None)
    else:
        out = dict(out)
    call("g2048_gather_minibatch", ptr(indices), m, ptr(packed["boards"]), ptr(packed["meta"]), ptr(packed["log_probs"]),
         ptr(packed["values"]), ptr(adv), ptr(ret), _OBS_DTYPES[obs_dtype or torch.float32], ptr(out["observations"]), ptr(out["actions"]),
         ptr(out["action_masks"]), ptr(out["log_probs"]), ptr(out["values"]), ptr(out["advantages"]), ptr(out["returns"]),
         ptr(out["boards"]) if obs_dtype is None else None, stream_ptr())
    return {k: v for k, v in out.items() if v is not None}


SAMPLE_RECORD = np.dtype([("board", "<u8"), ("meta", "<u4"), ("reward", "<f4"), ("log_prob", "<f4"), ("value", "<f4"),
                          ("advantage", "<f4"), ("ret", "<f4")])  # G2048SampleRecord (include/g2048.h), 32 bytes


def pack_samples(packed: dict, adv: torch.Tensor | None, ret: torch.Tensor | None, moments: torch.Tensor | None = None,
                 out: torch.Tensor | None = None) -> torch.Tensor:
    """Flat packed buffer (+ advantages / returns) -> (n, 4) int64 tensor of 32-byte sample records
    (G2048SampleRecord).  moments (the fp64 block gae_flat fills): normalise advantages and returns on the way, exactly as
    normalize_ would."""
    n = packed["boards"].shape[0]
    if out is None:
        out = torch.empty((n, 4), dtype=torch.int64, device=packed["boards"].device)
    call("g2048_pack_samples", ptr(packed["boards"]), ptr(packed["meta"]), ptr(packed.get("rewards")), ptr(packed.get("log_probs")),
         ptr(packed.get("values")), ptr(adv), ptr(ret), n, ptr(moments), ptr(out), stream_ptr())
    return out


def gather_samples(indices: torch.Tensor, records: torch.Tensor, obs_dtype=torch.float32, out: dict | None = None,
                   with_gae: bool = True) -> dict:
    """gather_minibatch reading 32-byte sample records (pack_samples): one sector per sample."""
    m = indices.shape[0]
    if out is None:
        out = minibatch_buffers(m, indices.device, obs_dtype, with_gae)
    else:
        out = dict(out)
    call("g2048_gather_samples", ptr(indices), m, ptr(records), _OBS_DTYPES[obs_dtype or torch.float32], ptr(out["observations"]),
         ptr(out["actions"]), ptr(out["action_masks"]), ptr(out["log_probs"]), ptr(out["values"]), ptr(out["advantages"]),
         ptr(out["returns"]), ptr(out["boards"]) if obs_dtype is None else None, stream_ptr())
    return {k: v for k, v in out.items() if v is not None}


# ------------------------------------------------------------------------------------------- embedding
def embed_boards(boards: torch.Tensor, table: torch.Tensor, indices: torch.Tensor | None = None, out=None,
                 entry: str = "g2048_embed_boards") -> torch.Tensor:
    """(n,16,d_model) = table[exponent of every cell]: Linear(31->d_model, bias=False) on the one-hot
    observation without the observation.  table: (31, d_model) float32/bfloat16 contiguous (weight.T);
    indices (int64): embed boards[indices].  entry="g2048_embed_boards_bulk" | "g2048_embed_boards_plain" pins the kernel."""
    if table.dim() != 2 or table.shape[0] != 31 or not table.is_contiguous():
        raise ValueError("table must be a contiguous (31, d_model) tensor")
    n = boards.numel() if indices is None else indices.numel()
    d_model = table.shape[1]
    if out is None:
        out = torch.empty((n, 16, d_model), dtype=table.dtype, device=boards.device)
    call(entry, ptr(boards), n, ptr(indices), ptr(table), d_model, _OBS_DTYPES[table.dtype], ptr(out), stream_ptr())
    return out


def embed_boards_grad(boards: torch.Tensor, grad_out: torch.Tensor, indices: torch.Tensor | None = None) -> torch.Tensor:
    """Gradient of embed_boards' table: (31, d_model) float32 (deterministic summation order)."""
    n = boards.numel() if indices is None else indices.numel()
    d_model = grad_out.shape[-1]
    code = _OBS_DTYPES[grad_out.dtype]
    nbytes = int(N.lib.g2048_embed_grad_scratch_bytes(n, d_model, code))
    if nbytes < 0:
        raise ValueError(f"embed_boards_grad: unsupported d_model {d_model} for {grad_out.dtype}")
    scratch = torch.empty(max(nbytes, 16), dtype=torch.uint8, device=boards.device)
    grad_table = torch.empty((31, d_model), dtype=torch.float32, device=boards.device)
    call("g2048_embed_boards_grad", ptr(boards), n, ptr(indices), ptr(grad_out), d_model, code, ptr(grad_table),
         ptr(scratch), stream_ptr())
    return grad_table


# ------------------------------------------------------------------------------------------- GAE
def gae_flat(rewards, values, dones, gamma: float, lambda_gae: float, want_moments: bool = True,
             entry: str = "g2048_gae_flat"):
    """-> adv, ret (n,) float32, moments (6,) float64 or None.  dones: uint8/bool (n,).
    entry: g2048_gae_flat_tiled / _pipelined pin a kernel; entry="g2048_gae_flat_scan" is the re-associated reverse
    scan (a pure stream; within 1e-5 relative of the reference loop instead of bit-identical)."""
    n = rewards.shape[0]
    dev = rewards.device
    adv = torch.empty(n, dtype=torch.float32, device=dev)
    ret = torch.empty(n, dtype=torch.float32, device=dev)
    size_fn = N.lib.g2048_gae_scan_scratch_bytes if entry == "g2048_gae_flat_scan" else N.lib.g2048_gae_flat_scratch_bytes
    scratch = torch.zeros(int(size_fn(n)), dtype=torch.uint8, device=dev)
    moments = torch.zeros(6, dtype=torch.float64, device=dev) if want_moments else None
    call(entry, ptr(rewards), ptr(values), ptr(dones), n, float(gamma), float(lambda_gae), ptr(adv),
         ptr(ret), ptr(scratch), ptr(moments), stream_ptr())
    return adv, ret, moments


def gae_time_major(rec_rewards, rec_values, rec_meta, t_steps: int, n: int, bootstrap, gamma: float,
                   lambda_gae: float, want_moments: bool = True):
    dev = rec_rewards.device
    adv = torch.empty((t_steps, n), dtype=torch.float32, device=dev)
    ret = torch.empty((t_steps, n), dtype=torch.float32, device=dev)
    moments = torch.zeros(6, dtype=torch.float64, device=dev) if want_moments else None
    call("g2048_gae_time_major", ptr(rec_rewards), ptr(rec_values), ptr(rec_meta), t_steps, n, ptr(bootstrap),
         float(gamma), float(lambda_gae), ptr(adv), ptr(ret), ptr(moments), stream_ptr())
    return adv, ret, moments


def normalize_(x: torch.Tensor, moments: torch.Tensor, which: int) -> torch.Tensor:
    call("g2048_normalize", ptr(x), x.numel(), ptr(moments), which, stream_ptr())
    return x


def gae_host(rewards: np.ndarray, values: np.ndarray, dones: np.ndarray, gamma: float, lambda_gae: float,
             normalize: bool):
    N.require_cuda()
    r = np.ascontiguousarray(rewards, np.float32)
    v = np.ascontiguousarray(values, np.float32)
    d = np.ascontiguousarray(dones, np.uint8)
    adv = np.empty_like(r)
    ret = np.empty_like(r)
    call("g2048_gae_host", r.ctypes.data, v.ctypes.data, d.ctypes.data, r.shape[0], float(gamma), float(lambda_gae),
         int(normalize), adv.ctypes.data, ret.ctypes.data)
    return adv, ret


def row_moments(x: torch.Tensor) -> torch.Tensor:
    """(F, n) float64 -> (F, 3): count, mean, population variance."""
    assert x.dtype == torch.float64 and x.dim() == 2
    out = torch.empty((x.shape[0], 3), dtype=torch.float64, device=x.device)
    call("g2048_row_moments", ptr(x), x.shape[0], x.shape[1], ptr(out), stream_ptr())
    return out


def int_peak_probe(blocks: int, threads: int, iters: int, sink: torch.Tensor) -> None:
    call("g2048_int_peak_probe", blocks, threads, iters, ptr(sink), stream_ptr())
