"""Throughput of the expectimax kernel (g2048_expectimax_values) and strength of the expectimax player; prints one JSON
line.

  * search: depth 2, 3 and 4 over the default row table (w = 0) on 4 096 mid-game boards -- those of a DRUL run of the
    recording play kernel at step 100 (or the last board of a shorter episode).  Device-timed with CUDA events, L2
    flushed (512 MiB write) before every timed launch; leaves (heuristic evaluations) per second from the kernel's own
    counters.
  * the oracle's leaves/s on this host's cores (tests/expectimax_oracle.c, OpenMP) at depth 3 on the same boards.
  * the player: BatchRunner(seed, ExpectimaxPolicy(depth)).run_eval_batch(B) for depth in {2, 3}, B in {256, 4 096},
    whole games, wall time: moves per second, mean score and the share of games that reach 2048, 4096 and 8192.

    python tools/bench_expectimax.py [--reps 5] [--skip-player] [--out FILE]
"""
import argparse
import json
import os
import statistics
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path[:0] = [str(ROOT), str(ROOT / "2048-ppo-agent_b200"), str(ROOT / "tests")]

import torch  # noqa: E402

import g2048  # noqa: E402
from g2048 import engine as E  # noqa: E402

from bench_playout import device_times, gpu_info, mid_game_boards  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--skip-player", action="store_true")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    mode = E.RNG_PARTITIONABLE
    flush_buf = torch.empty(512 << 20, dtype=torch.uint8, device="cuda")
    result = {"gpu": gpu_info(), "l2": "flushed (512 MiB write) before every timed launch"}

    n_boards = 4096
    boards = mid_game_boards(n_boards, 100, mode)
    table = g2048.default_row_values()
    search = []
    for depth in (2, 3, 4):
        counters = torch.zeros(2, dtype=torch.int64, device="cuda")
        E.expectimax_values(boards, depth, table, 0.0, counters)
        leaves, chance = (int(x) for x in counters.tolist())
        times = device_times(lambda: E.expectimax_values(boards, depth, table, 0.0), args.reps, flush_buf)
        med = statistics.median(times)
        search.append({"depth": depth, "boards": n_boards, "leaves": leaves, "chance_nodes": chance,
                       "ms": [round(t * 1e3, 3) for t in times], "leaves_per_s": leaves / med})
        print(json.dumps(search[-1]), file=sys.stderr, flush=True)
    result["search"] = search
    del flush_buf
    torch.cuda.empty_cache()

    # ---- the oracle on the host cores
    import expectimax_oracle as XO

    host_boards = E.boards_numpy(boards)
    host_table = table.cpu().numpy()
    XO.expectimax(host_boards[:8], 2, host_table)  # compile
    t0 = time.perf_counter()
    _, c = XO.expectimax(host_boards, 3, host_table)
    wall = time.perf_counter() - t0
    result["oracle_host"] = {"depth": 3, "boards": n_boards, "cores": os.cpu_count(), "leaves": int(c[0]),
                             "seconds": round(wall, 3), "leaves_per_s": int(c[0]) / wall}
    print(json.dumps(result["oracle_host"]), file=sys.stderr, flush=True)

    # ---- the expectimax player, whole games
    if not args.skip_player:
        player = []
        g2048.BatchRunner(1, g2048.ExpectimaxPolicy(depth=1)).run_eval_batch(64)  # warm-up: module loads
        for depth in (2, 3):
            for B in (256, 4096):
                runner = g2048.BatchRunner(0, g2048.ExpectimaxPolicy(depth=depth))
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                res = runner.run_eval_batch(B)
                torch.cuda.synchronize()
                wall = time.perf_counter() - t0
                s = res["summary"]
                hist = s["max_tile_hist"]
                reach = {str(t): sum(v for k, v in hist.items() if k >= t) / B for t in (2048, 4096, 8192)}
                player.append({"depth": depth, "B": B, "seconds": round(wall, 3), "moves": s["env_steps"],
                               "loop_steps": s["loop_steps"], "moves_per_s": s["env_steps"] / wall,
                               "mean_score": s["score_sum"] / B, "reach": reach,
                               "max_tile_hist": {str(k): v for k, v in sorted(hist.items())}})
                print(json.dumps(player[-1]), file=sys.stderr, flush=True)
        result["expectimax_player"] = player
    line = json.dumps(result)
    print(line)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(line + "\n")


if __name__ == "__main__":
    main()
