"""Throughput of the Monte-Carlo playout kernel (g2048_playout_values) and of the Monte-Carlo player; prints one JSON line.

  * playouts: P = 2^24 (4 096 mid-game boards x 4 actions x 1 024 random-policy playouts).  The boards are those of a
    DRUL run of the recording play kernel at step 100 (or the last board of a shorter episode).  Reported next to
    g2048_play (random policy) at 2^24 envs in the same process; both device-timed with CUDA events, L2 flushed
    (512 MiB write) before every timed launch, as bench.py does.  Also: the share of illegal (board, action) pairs
    and the time with and without the statistics block.
  * the player: BatchRunner(seed, MonteCarloPolicy(K)).run_eval_batch(B) for B in {1 024, 16 384}, K in {16, 64}, whole
    games, wall time: moves (env-steps of the games) per second and the mean score.

    python tools/bench_playout.py [--reps 5] [--out FILE]
"""
import argparse
import json
import statistics
import subprocess
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path[:0] = [str(ROOT), str(ROOT / "2048-ppo-agent_b200")]

import torch  # noqa: E402

import g2048  # noqa: E402
from g2048 import _native as N  # noqa: E402
from g2048 import engine as E  # noqa: E402


def gpu_info() -> dict:
    q = "name,power.limit,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=30).stdout.strip().splitlines()
        return dict(zip(q.split(","), (s.strip() for s in out[torch.cuda.current_device()].split(","))))
    except (OSError, IndexError, subprocess.TimeoutExpired):
        return {"name": torch.cuda.get_device_name()}


def mid_game_boards(n: int, step: int, mode: int) -> torch.Tensor:
    subs = E.chain_advance(E.words_tensor([0, 2024], "cuda"), mode, 1 + 2 * 2048)
    rec = E.play_record(E.POLICY_DRUL, subs, n, 0, n, mode)
    at = torch.minimum(rec["lengths"].to(torch.int64) - 1, torch.full((n,), step, dtype=torch.int64, device="cuda"))
    return rec["arena_boards"][rec["env_slot"] + at.clamp(min=0)]


def device_times(fn, reps: int, flush_buf) -> list:
    fn()
    torch.cuda.synchronize()
    times = []
    for i in range(reps):
        flush_buf.fill_(i & 0xFF)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        times.append(a.elapsed_time(b) * 1e-3)
    return times


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    mode = E.RNG_PARTITIONABLE
    flush_buf = torch.empty(512 << 20, dtype=torch.uint8, device="cuda")
    result = {"gpu": gpu_info(), "rng_mode": "partitionable", "l2": "flushed (512 MiB write) before every timed launch"}

    # ---- playouts at P = 2^24 next to g2048_play at 2^24 envs
    n_boards, K, max_steps = 4096, 1024, 2048
    boards = mid_game_boards(n_boards, 100, mode)
    subs = E.chain_advance(E.words_tensor([0, 99], "cuda"), mode, 1 + 2 * max_steps)
    out = {}

    def playouts(with_stats: bool):
        stats = torch.zeros(N.PLAY_STATS_WORDS, dtype=torch.int64, device="cuda") if with_stats else None
        out["rec"] = E.playout_values(E.POLICY_RANDOM, boards, subs, K, mode, stats=stats)

    t_stats = device_times(lambda: playouts(True), args.reps, flush_buf)
    st = E.play_stats_dict(out["rec"]["stats"])
    t_plain = device_times(lambda: playouts(False), args.reps, flush_buf)
    played = int(out["rec"]["playouts"].sum().item())
    n_play = 1 << 24
    play_out = {}

    def play():
        play_out["r"] = E.play(E.POLICY_RANDOM, subs, n_play, 0, n_play, mode, per_env=False)

    t_play = device_times(play, args.reps, flush_buf)
    pst = E.play_stats_dict(play_out["r"]["stats"])
    med = statistics.median
    result["playouts"] = {
        "boards": n_boards, "playouts_per_action": K, "P": n_boards * 4 * K, "rollout": "random",
        "board_source": "DRUL run of g2048_play_record, board at step 100",
        "illegal_pair_share": 1.0 - played / (n_boards * 4 * K), "playouts_played": played,
        "env_steps": st["env_steps"], "mean_playout_steps": st["env_steps"] / max(played, 1),
        "cut_short": st["cut_short"],
        "ms_with_stats": [round(t * 1e3, 3) for t in t_stats], "ms_without_stats": [round(t * 1e3, 3) for t in t_plain],
        "env_steps_per_s": st["env_steps"] / med(t_plain), "env_steps_per_s_with_stats": st["env_steps"] / med(t_stats),
        "playouts_per_s": played / med(t_plain),
    }
    result["play_2p24"] = {"envs": n_play, "env_steps": pst["env_steps"], "mean_episode_steps": pst["env_steps"] / n_play,
                           "ms": [round(t * 1e3, 3) for t in t_play], "env_steps_per_s": pst["env_steps"] / med(t_play)}
    result["playout_vs_play_env_steps_per_s"] = result["playouts"]["env_steps_per_s"] / result["play_2p24"]["env_steps_per_s"]
    del flush_buf
    torch.cuda.empty_cache()

    # ---- the Monte-Carlo player, whole games
    player = []
    g2048.BatchRunner(1, g2048.MonteCarloPolicy(playouts=4)).run_eval_batch(64)  # warm-up: module loads, tables
    for B in (1024, 16384):
        for K in (16, 64):
            runner = g2048.BatchRunner(0, g2048.MonteCarloPolicy(playouts=K))
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            res = runner.run_eval_batch(B)
            torch.cuda.synchronize()
            wall = time.perf_counter() - t0
            s = res["summary"]
            player.append({"B": B, "K": K, "seconds": round(wall, 3), "moves": s["env_steps"], "loop_steps": s["loop_steps"],
                           "moves_per_s": s["env_steps"] / wall, "mean_score": s["score_sum"] / B,
                           "max_tile_hist": {str(k): v for k, v in sorted(s["max_tile_hist"].items())}})
            print(json.dumps(player[-1]), file=sys.stderr, flush=True)
    result["monte_carlo_player"] = player
    line = json.dumps(result)
    print(line)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(line + "\n")


if __name__ == "__main__":
    main()
