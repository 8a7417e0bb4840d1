"""Speed and learning of the TD(0) row-table learner (g2048_td_train, g2048.TDLearner); prints one JSON line.

  * speed: learning steps (env-steps) per second and microseconds per batch step at n = 2^14, 2^16 and 2^18, device-timed
    with CUDA events around one launch of `steps` steps after a warm-up launch (the table and the env state, 0.8 MB +
    24 bytes per env, stay in L2, as they do in training).  --ab-lib LIB times a second build of the library (loaded in
    a subprocess through G2048_LIB) at the same sizes.  Next to it, the same steps as a CUDA graph of one-step launches.
  * an alpha sweep from the zero table at n = 2^16: the learning curve (mean score of the episodes that ended in each
    block of steps), then the greedy player (ExpectimaxPolicy(depth=1, row_values=T, reward_weight=1.0)) with each
    learned table over the same B seeded games.
  * the player with the table the sweep liked best at depth 1, 2 and 3, next to default_row_values() (w = 0, the
    expectimax player's default) and to DRUL: mean score and the share of games that reach 2048 and 4096.

    python tools/bench_td.py [--steps 2000] [--sweep-steps 4000] [--games 1024] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path[:0] = [str(ROOT), str(ROOT / "2048-ppo-agent_b200"), str(ROOT / "tools")]

import torch  # noqa: E402

import g2048  # noqa: E402
from g2048 import engine as E  # noqa: E402

from bench_playout import gpu_info  # noqa: E402

SIZES = (1 << 14, 1 << 16, 1 << 18)
ALPHAS = (0.001, 0.0025, 0.01, 0.025, 0.1)


def speed(steps: int, reps: int = 3) -> list:
    mode = E.RNG_PARTITIONABLE
    out = []
    for n in SIZES:
        lr = g2048.TDLearner(0, n, alpha=0.0025, rng_mode=mode)
        subs = E.chain_advance(E.words_tensor([0, 1], "cuda"), mode, steps)
        run = lambda: E.td_train(lr.boards, lr.after, lr.scores, lr.lengths, lr.table, lr.alpha, subs, mode,  # noqa: E731
                                 lr._scratch)
        run()  # warm-up: module load, row tables, and games in progress rather than fresh envs
        torch.cuda.synchronize()
        times = []
        for _ in range(reps):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            run()
            b.record()
            torch.cuda.synchronize()
            times.append(a.elapsed_time(b) * 1e-3)
        best = min(times)
        out.append({"n": n, "steps": steps, "seconds": [round(t, 4) for t in times], "us_per_step": best / steps * 1e6,
                    "learning_steps_per_s": n * steps / best})
        print(json.dumps(out[-1]), file=sys.stderr, flush=True)
    return out


def per_step_graph(steps: int, reps: int = 3) -> list:
    """The launch-per-step alternative, approximated: a CUDA graph of `steps` one-step launches of the same kernel (each
    launch copies the row tables into shared memory again and ends its step with the apply phase) against the one
    launch for all steps that speed() times."""
    mode = E.RNG_PARTITIONABLE
    out = []
    for n in SIZES:
        lr = g2048.TDLearner(0, n, alpha=0.0025, rng_mode=mode)
        subs = E.chain_advance(E.words_tensor([0, 1], "cuda"), mode, steps)

        def run():
            for t in range(steps):
                E.td_train(lr.boards, lr.after, lr.scores, lr.lengths, lr.table, lr.alpha, subs[t:t + 1], mode, lr._scratch)

        try:
            run()  # warm-up outside the capture
            torch.cuda.synchronize()
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                run()
            times = []
            for _ in range(reps):
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                graph.replay()
                b.record()
                torch.cuda.synchronize()
                times.append(a.elapsed_time(b) * 1e-3)
            best = min(times)
            out.append({"n": n, "steps": steps, "seconds": [round(t, 4) for t in times], "us_per_step": best / steps * 1e6,
                        "learning_steps_per_s": n * steps / best})
        except RuntimeError as exc:  # a capture the driver refuses is a result too
            out.append({"n": n, "error": str(exc)[:300]})
        print(json.dumps(out[-1]), file=sys.stderr, flush=True)
    return out


def _reach(summary, B):
    hist = summary["max_tile_hist"]
    return {str(t): sum(v for k, v in hist.items() if k >= t) / B for t in (2048, 4096)}


def play(policy, B, seed=7) -> dict:
    runner = g2048.BatchRunner(seed, policy)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    s = runner.run_eval_batch(B)["summary"] if isinstance(policy, g2048.ExpectimaxPolicy) else runner.run_stats_batch(B)["summary"]
    torch.cuda.synchronize()
    return {"mean_score": s["score_sum"] / B, "reach": _reach(s, B), "mean_moves": s["env_steps"] / B,
            "seconds": round(time.perf_counter() - t0, 2)}


def sweep(n: int, total: int, block: int, B: int) -> tuple:
    rows, tables = [], {}
    for alpha in ALPHAS:
        lr = g2048.TDLearner(0, n, alpha=alpha)
        curve = []
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(total // block):
            s = lr.train(block)
            curve.append(round(s["score_sum"] / max(s["episodes"], 1), 1))
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        greedy = play(g2048.ExpectimaxPolicy(depth=1, row_values=lr.table, reward_weight=1.0), B)
        rows.append({"alpha": alpha, "n": n, "steps": total, "block": block, "train_seconds": round(wall, 2),
                     "curve_mean_score": curve, "greedy": greedy})
        tables[alpha] = lr.table.clone()
        print(json.dumps(rows[-1]), file=sys.stderr, flush=True)
    return rows, tables


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=2000, help="batch steps per timed launch")
    ap.add_argument("--sweep-steps", type=int, default=4000)
    ap.add_argument("--block", type=int, default=250)
    ap.add_argument("--games", type=int, default=1024)
    ap.add_argument("--ab-lib", default=None)
    ap.add_argument("--speed-only", action="store_true")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    result = {"gpu": gpu_info(), "l2": "warm: T, the scratch and the env state stay resident", "speed": speed(args.steps)}
    if not args.speed_only:
        result["per_step_graph"] = per_step_graph(args.steps)
    if args.ab_lib:
        env = dict(os.environ, G2048_LIB=str(Path(args.ab_lib).resolve()))
        cmd = [sys.executable, __file__, "--speed-only", "--steps", str(args.steps)]
        res = subprocess.run(cmd, env=env, capture_output=True, text=True, check=True)
        result["speed_ab"] = {"lib": Path(args.ab_lib).name, "speed": json.loads(res.stdout.strip().splitlines()[-1])["speed"]}
    if not args.speed_only:
        B = args.games
        rows, tables = sweep(1 << 16, args.sweep_steps, args.block, B)
        result["sweep"] = rows
        best = max(rows, key=lambda r: r["greedy"]["mean_score"])["alpha"]
        T = tables[best]
        players = {"drul": play(g2048.act_drul, B),
                   "greedy_zero_table": play(g2048.ExpectimaxPolicy(depth=1, row_values=torch.zeros_like(T), reward_weight=1.0), B)}
        for depth in (1, 2, 3):
            players[f"learned_alpha{best}_depth{depth}"] = play(g2048.ExpectimaxPolicy(depth=depth, row_values=T, reward_weight=1.0), B)
            players[f"default_table_depth{depth}"] = play(g2048.ExpectimaxPolicy(depth=depth), B)
            print(json.dumps({k: v for k, v in players.items() if k.endswith(f"depth{depth}")}), file=sys.stderr, flush=True)
        result["players"] = {"games": B, "seed": 7, "best_alpha": best, "results": players}
    line = json.dumps(result)
    print(line)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(line + "\n")


if __name__ == "__main__":
    main()
