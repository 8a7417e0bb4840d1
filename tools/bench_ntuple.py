"""Speed and learning of the n-tuple TD(0) learner (g2048_ntuple_td_train, g2048.NTupleTDLearner) and of expectimax
over a network (g2048_expectimax_values_ntuple); prints one JSON line.

  * speed: learning steps (env-steps) per second and microseconds per batch step for the 4x6 network at n = 2^14, 2^16
    and 2^18, device-timed with CUDA events around one launch of `steps` steps after a warm-up launch.
  * the accumulate / apply split per step and the entries touched per step, from a
    second build of the library with -DG2048_NTUPLE_PHASES (compiled into a temporary directory, run in a subprocess).
  * the `lines` network through g2048_ntuple_td_train next to g2048_td_train at n = 2^16 (the same computation).
  * the step time with n_weights: a 2.2 M-weight network packed, and the same tables at high offsets of an array 16
    times as large, at n = 2^16.
  * an alpha sweep of the 4x6 network from zeros at n = 2^16: the learning curve (mean score of the episodes that
    ended in each block of steps) and the greedy player over the same B seeded games.
  * players: greedy / depth 2 / depth 3 with the learned 4x6 network, the learned row table (TDLearner, alpha 0.1) at
    the same number of learning steps and at the same training wall time, and default_row_values(): mean score and
    the share of games that reach 2048 / 4096 / 8192.
  * search: expectimax leaves/s at depth 2 and 3 on bench_expectimax.py's 4 096 mid-game boards with the 4x6 network
    leaf next to the row table (L2 flushed before every timed launch).

With --tc, the temporal coherence learner (g2048_ntuple_tc_train, g2048.NTupleTCLearner) instead:
  * speed: TC and TD for the 4x6 network at n = 2^14, 2^16 and 2^18, their timed launches alternated in one process;
  * the accumulate / apply split of both from the -DG2048_NTUPLE_PHASES build;
  * an alpha sweep of TC from the zero 4x6 network at n = 2^16 (learning curves, greedy player on the seed-7 games);
  * TC at its best alpha against TD at its default alpha 0.02 at equal steps (--sweep-steps and --long-steps): greedy
    and depth-2 mean scores, the 2048 / 4096 / 8192 / 16384 reach rates, and the training wall time.

With --stages, multi-stage networks (g2048_ntuple_staged_td_train, NTupleNetwork.staged) instead:
  * speed: at n = 2^14, 2^16 and 2^18, the 4x6 network trained for --pretrain-steps untimed steps, against 2-stage
    copies of it split at 11 (a 2048 tile) and at 13 (an 8192 tile) that carry on from the same envs, so that the
    timed window has a real share of envs in each stage; their timed launches alternated in one process, with the
    rate ratio and the time-averaged share of envs per stage;
  * search: expectimax leaves/s at depth 2 and 3 with the staged leaves next to the unstaged one, on the same values
    (the trained network of the n = 2^16 run and its staged copies) and 4 096 boards of that run's envs;
  * quality at n = 2^16, --long-steps steps of TD at alpha 0.02 from zeros (seed 0): unstaged; staged with thresholds
    (13,) and (14,); and half the steps unstaged, then staged((13,)), then the other half.  For each, the training wall
    time and the greedy and depth-2 players on the seed-7 games: mean score and the 4096 / 8192 / 16384 reach rates.

With --lambda, delayed TD(lambda) / TC(lambda) (g2048_ntuple_lambda_td_train / _tc_train, the learners' lam and
horizon) instead:
  * speed: at n = 2^14, 2^16 and 2^18, the 4x6 network trained by TD for --pretrain-steps untimed steps; then TD(0), TC
    and TD(lambda) / TC(lambda) at h = 2, 3, 5 (h capped so that n * h <= 2^20), each on its own copy of the weights
    and env state, their timed launches alternated in one process, with each rate over TD(0)'s (TC(lambda) also over
    TC's);
  * the accumulate / apply split of TD(0), TC, TD(lambda) and TC(lambda) at h = 3 from the -DG2048_NTUPLE_PHASES build,
    from the same pretrained start;
  * quality from the zero 4x6 network at n = 2^16 (seed 0): TD(0), TC and TD / TC(lambda) over lambda in {0.25, 0.5,
    0.75} x h in {2, 3, 5}, evaluated after --sweep-steps and after --long-steps steps (one run each: the second
    evaluation continues the first): learning curve, training wall time, greedy and depth-2 players on the seed-7 games;
    then one staged (13,) run of the best setting at --long-steps, next to staged TD(0).

With --carousel, carousel shaping of multi-stage networks (g2048_ntuple_carousel_td_train / _tc_train, the learners'
carousel) instead:
  * speed of the mechanism: at n = 2^14, 2^16 and 2^18, the 4x6 network trained by TD for --carousel-pretrain-steps
    untimed steps, then staged (14,) copies of it with and without the carousel (TD(0)), carrying on from the same envs,
    their timed launches alternated; few envs reach a 16384 tile, so the pool stays (nearly) empty and the ratio
    isolates the mechanism.  Each carousel row reports the non-zero pool entries after timing;
  * speed with a real mix: the same after --pretrain-steps untimed steps with (13,) copies, with the time-averaged
    share of envs per stage and (carousel) per start stage;
  * quality from the zero 4x6 network at n = 2^16 (seed 0), TC(lambda = 0.5, h = 3) at alpha 0.02: unstaged, staged
    (13,), staged (13,) with the carousel, and half of --sweep-steps unstaged then staged((13,)) with the carousel;
    evaluated after --sweep-steps and, continuing the same runs, after --long-steps steps: greedy and depth-2 players
    on the seed-7 games, the share of env-steps in stage 1 (of (13,), sampled after every block) and the stage-1
    entries ever updated (A > 0).

    python tools/bench_ntuple.py [--tc | --stages | --lambda | --carousel] [--long-steps 40000] [--steps 500] [--sweep-steps 4000] [--games 1024] [--deep-games 128] [--speed-only | --skip-speed] [--out FILE]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path[:0] = [str(ROOT), str(ROOT / "2048-ppo-agent_b200"), str(ROOT / "tools")]

import torch  # noqa: E402

import g2048  # noqa: E402
from g2048 import engine as E  # noqa: E402
from g2048.ntuple import NTupleNetwork, make_placements  # noqa: E402

from bench_playout import device_times, gpu_info, mid_game_boards  # noqa: E402

SIZES = (1 << 14, 1 << 16, 1 << 18)
ALPHAS = (0.001, 0.0025, 0.005, 0.01, 0.02, 0.03)
TC_ALPHAS = (0.01, 0.02, 0.05, 0.1, 0.2, 0.5, 1.0)
MODE = E.RNG_PARTITIONABLE


def _timed(run, reps):
    run()  # warm-up: module load, row tables, and games in progress rather than fresh envs
    torch.cuda.synchronize()
    return [_timed_once(run) for _ in range(reps)]


def _timed_once(run) -> float:
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    run()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) * 1e-3


def _row(name, n, steps, times, **extra):
    best = min(times)
    row = {"what": name, "n": n, "steps": steps, "seconds": [round(t, 4) for t in times],
           "us_per_step": best / steps * 1e6, "learning_steps_per_s": n * steps / best}
    row.update(extra)
    print(json.dumps(row), file=sys.stderr, flush=True)
    return row


def _ntuple_run(lr, subs):
    net = lr.network
    return lambda: E.ntuple_td_train(lr.boards, lr.after, lr.scores, lr.lengths, net.placements, net.weights, lr.alpha,
                                     subs, MODE, lr._scratch)


def _tc_run(lr, subs):
    net = lr.network
    return lambda: E.ntuple_tc_train(lr.boards, lr.after, lr.scores, lr.lengths, net.placements, net.weights,
                                     lr.err_sum, lr.abs_err_sum, lr.alpha, subs, MODE, lr._scratch)


def tc_speed(steps: int, reps: int = 3) -> list:
    """TD and TC at each size: both warmed up, then their timed launches alternated."""
    out = []
    subs = E.chain_advance(E.words_tensor([0, 1], "cuda"), MODE, steps)
    for n in SIZES:
        td = g2048.NTupleTDLearner(0, n, alpha=0.0025, rng_mode=MODE)
        tc = g2048.NTupleTCLearner(0, n, alpha=0.0025, rng_mode=MODE)
        runs = {"four_six_td": _ntuple_run(td, subs), "four_six_tc": _tc_run(tc, subs)}
        for run in runs.values():
            run()
        torch.cuda.synchronize()
        times = {k: [] for k in runs}
        for _ in range(reps):
            for k, run in runs.items():
                times[k].append(_timed_once(run))
        out += [_row(k, n, steps, times[k]) for k in runs]
        del td, tc, runs
        torch.cuda.empty_cache()
    return out


def speed(steps: int, reps: int = 3) -> list:
    out = []
    subs = E.chain_advance(E.words_tensor([0, 1], "cuda"), MODE, steps)
    for n in SIZES:
        lr = g2048.NTupleTDLearner(0, n, alpha=0.0025, rng_mode=MODE)
        out.append(_row("four_six", n, steps, _timed(_ntuple_run(lr, subs), reps)))
        del lr
        torch.cuda.empty_cache()
    return out


def phase_probe(steps: int, tc: bool = False) -> list:
    """In a build with -DG2048_NTUPLE_PHASES: the accumulate / apply split of one launch of `steps` steps after a
    warm-up launch, as CTA 0 timed it (%globaltimer up to each phase's closing grid.sync()), and the entries listed
    (touched) per step.  With tc, the TC learner at each size after the TD learner."""
    out = []
    subs = E.chain_advance(E.words_tensor([0, 1], "cuda"), MODE, steps)
    for n, kind in [(n, k) for n in SIZES for k in (("td", "tc") if tc else ("td",))]:
        lr = (g2048.NTupleTCLearner if kind == "tc" else g2048.NTupleTDLearner)(0, n, alpha=0.0025, rng_mode=MODE)
        net = lr.network
        stats = torch.zeros(32, dtype=torch.int64, device="cuda")
        if kind == "tc":
            run = lambda st=None: E.ntuple_tc_train(lr.boards, lr.after, lr.scores, lr.lengths, net.placements,  # noqa: E731
                                                    net.weights, lr.err_sum, lr.abs_err_sum, lr.alpha, subs, MODE,
                                                    lr._scratch, st)
        else:
            run = lambda st=None: E.ntuple_td_train(lr.boards, lr.after, lr.scores, lr.lengths, net.placements,  # noqa: E731
                                                    net.weights, lr.alpha, subs, MODE, lr._scratch, st)
        run()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        run(stats)
        b.record()
        torch.cuda.synchronize()
        acc_ns, apply_ns, listed = (int(x) for x in stats[8:11].tolist())
        out.append({"n": n, "steps": steps, "us_per_step": a.elapsed_time(b) * 1e3 / steps,
                    **({"learner": kind} if tc else {}),
                    "accumulate_us_per_step": acc_ns / 1e3 / steps, "apply_us_per_step": apply_ns / 1e3 / steps,
                    "entries_listed_per_step": listed / steps})
        print(json.dumps(out[-1]), file=sys.stderr, flush=True)
        del lr, net
        torch.cuda.empty_cache()
    return out


def phases(steps: int, tc: bool = False) -> dict:
    """Builds the library with -DG2048_NTUPLE_PHASES into a temporary directory and runs phase_probe on it."""
    tmp = Path(tempfile.mkdtemp(prefix="g2048_ntuple_phases_"))
    lib = tmp / "libg2048_phases.so"
    subprocess.run(["make", "-C", str(ROOT / "2048-ppo-agent_b200" / "csrc"), "-j16", f"OUT={lib}", f"BUILD={tmp / 'build'}",
                    "EXTRA=-DG2048_NTUPLE_PHASES"], check=True, capture_output=True)
    env = dict(os.environ, G2048_LIB=str(lib))
    res = subprocess.run([sys.executable, __file__, "--phase-probe", "--steps", str(steps)] + (["--tc"] if tc else []),
                         env=env, capture_output=True, text=True, check=True)
    return {"build": "-DG2048_NTUPLE_PHASES", "rows": json.loads(res.stdout.strip().splitlines()[-1])}


def lines_vs_row(steps: int, reps: int = 3) -> list:
    n = 1 << 16
    subs = E.chain_advance(E.words_tensor([0, 1], "cuda"), MODE, steps)
    row = g2048.TDLearner(0, n, alpha=0.1, rng_mode=MODE)
    run_row = lambda: E.td_train(row.boards, row.after, row.scores, row.lengths, row.table, row.alpha, subs, MODE,  # noqa: E731
                                 row._scratch)
    lines = g2048.NTupleTDLearner(0, n, network=NTupleNetwork.lines(), alpha=0.1, rng_mode=MODE)
    return [_row("row_table_td_train", n, steps, _timed(run_row, reps)),
            _row("lines_ntuple_td_train", n, steps, _timed(_ntuple_run(lines, subs), reps))]


def weights_size(steps: int, reps: int = 3) -> list:
    """A network of two 5-cell and two 4-cell tuples under the 8 symmetries (2.2 M weights), packed and at the top of
    an array 16 times as large."""
    n = 1 << 16
    tuples = [(0, 1, 2, 3, 4), (4, 5, 6, 7, 8), (0, 1, 4, 5), (8, 9, 12, 13)]
    sizes = [16 ** len(t) for t in tuples]
    total = sum(sizes)
    subs = E.chain_advance(E.words_tensor([0, 1], "cuda"), MODE, steps)
    out = []
    for name, shift in (("packed", 0), ("high_offsets", 15 * total)):
        rows = [(shift + sum(sizes[:j]), im) for j, t in enumerate(tuples) for im in g2048.ntuple.symmetric_images(t)]
        net = NTupleNetwork(make_placements(rows), shift + total)
        lr = g2048.NTupleTDLearner(0, n, network=net, alpha=0.0025, rng_mode=MODE)
        out.append(_row(name, n, steps, _timed(_ntuple_run(lr, subs), reps), n_weights=shift + total))
        del lr, net
        torch.cuda.empty_cache()
    return out


def _reach(summary, B):
    hist = summary["max_tile_hist"]
    return {str(t): sum(v for k, v in hist.items() if k >= t) / B for t in (2048, 4096, 8192, 16384)}


def play(policy, B, seed=7) -> dict:
    runner = g2048.BatchRunner(seed, policy)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    s = runner.run_eval_batch(B)["summary"] if isinstance(policy, g2048.ExpectimaxPolicy) else runner.run_stats_batch(B)["summary"]
    torch.cuda.synchronize()
    return {"games": B, "mean_score": s["score_sum"] / B, "reach": _reach(s, B), "mean_moves": s["env_steps"] / B,
            "seconds": round(time.perf_counter() - t0, 2)}


def _train(lr, total, block):
    curve = []
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(total // block):
        s = lr.train(block)
        curve.append(round(s["score_sum"] / max(s["episodes"], 1), 1))
    torch.cuda.synchronize()
    return curve, time.perf_counter() - t0


def sweep(n: int, total: int, block: int, B: int, alphas=ALPHAS, learner=g2048.NTupleTDLearner) -> tuple:
    rows, best = [], None
    for alpha in alphas:
        lr = learner(0, n, alpha=alpha)
        curve, wall = _train(lr, total, block)
        greedy = play(g2048.ExpectimaxPolicy(depth=1, network=lr.network, reward_weight=1.0), B)
        rows.append({"alpha": alpha, "n": n, "steps": total, "block": block, "train_seconds": round(wall, 2),
                     "curve_mean_score": curve, "greedy": greedy})
        print(json.dumps(rows[-1]), file=sys.stderr, flush=True)
        if best is None or greedy["mean_score"] > best[0]:
            best = (greedy["mean_score"], alpha, lr.network, wall)
        del lr
        torch.cuda.empty_cache()
    return rows, best


def search(reps: int, net) -> list:
    flush_buf = torch.empty(512 << 20, dtype=torch.uint8, device="cuda")
    boards = mid_game_boards(4096, 100, MODE)
    table = g2048.default_row_values()
    out = []
    for depth in (2, 3):
        for leaf in ("row_table", "four_six"):
            if leaf == "row_table":
                fn = lambda c=None: E.expectimax_values(boards, depth, table, 0.0, c)  # noqa: E731
            else:
                fn = lambda c=None: E.expectimax_values_ntuple(boards, depth, net.placements, net.weights, 0.0, c)  # noqa: E731
            counters = torch.zeros(2, dtype=torch.int64, device="cuda")
            fn(counters)
            leaves = int(counters[0].item())
            times = device_times(fn, reps, flush_buf)
            med = statistics.median(times)
            out.append({"depth": depth, "leaf": leaf, "boards": 4096, "leaves": leaves,
                        "ms": [round(t * 1e3, 3) for t in times], "leaves_per_s": leaves / med})
            print(json.dumps(out[-1]), file=sys.stderr, flush=True)
    return out


def equal_steps(tc_alpha: float, lengths, block: int, B: int, deep: int) -> list:
    """TD at its default alpha against TC at tc_alpha, from the zero 4x6 network at n = 2^16 (seed 0), for each number
    of steps: training wall time, learning curve, and the greedy and depth-2 players on the seed-7 games."""
    out = []
    for steps in lengths:
        for name, learner, alpha in (("td", g2048.NTupleTDLearner, g2048.td.DEFAULT_NTUPLE_ALPHA),
                                     ("tc", g2048.NTupleTCLearner, tc_alpha)):
            lr = learner(0, 1 << 16, alpha=alpha)
            curve, wall = _train(lr, steps, block)
            row = {"learner": name, "alpha": alpha, "n": 1 << 16, "steps": steps, "block": block,
                   "train_seconds": round(wall, 2), "curve_mean_score": curve}
            for depth, games in ((1, B), (2, deep)):
                row[f"depth{depth}"] = play(g2048.ExpectimaxPolicy(depth=depth, network=lr.network, reward_weight=1.0),
                                            games)
            out.append(row)
            print(json.dumps(row), file=sys.stderr, flush=True)
            del lr
            torch.cuda.empty_cache()
    return out


def _staged_run(lr, subs):
    net = lr.network
    return lambda: E.ntuple_td_train(lr.boards, lr.after, lr.scores, lr.lengths, net.placements, net.weights, lr.alpha,
                                     subs, MODE, lr._scratch, stages=net.stages)


def _promoted(lr, thresholds, carousel=False):
    """A learner of lr's class of staged(lr.network, thresholds) that carries on from lr's env state, window and key
    chain: at the start it has exactly lr's values, so it plays lr's games.  A TC learner's E and A are copied into
    every stage, as the weights are.  ``carousel``: the new learner shapes, from an empty pool."""
    promoted = type(lr)(0, lr.batch_size, network=NTupleNetwork.staged(lr.network, thresholds), alpha=lr.alpha,
                        rng_mode=lr.rng_mode, lam=lr.lam, horizon=lr.horizon, carousel=carousel)
    ckpt = lr.state_dict()
    for k in ("placements", "n_weights", "weights", "stage_thresholds", "stage_stride", "err_sum", "abs_err_sum"):
        ckpt.pop(k, None)
    for k, v in promoted._values_state().items():
        ckpt.setdefault(k, v)  # lr's window stays
    if isinstance(lr, g2048.NTupleTCLearner):
        S = len(thresholds) + 1
        ckpt["err_sum"], ckpt["abs_err_sum"] = lr.err_sum.cpu().repeat(S), lr.abs_err_sum.cpu().repeat(S)
    promoted.load_state_dict(ckpt)
    return promoted


def _stage_shares(boards, thresholds) -> list:
    """The share of the boards in each stage of these thresholds."""
    me = E.boards_numpy(boards).max(axis=1)
    stage = sum((me >= t).astype(int) for t in thresholds)
    return [round(float((stage == s).mean()), 4) for s in range(len(thresholds) + 1)]


STAGE_SPLITS = ((11,), (13,))


def stages_speed(steps: int, pretrain: int, reps: int = 3) -> tuple:
    """At each size, the 4x6 network trained by TD (alpha 0.02, seed 0) for `pretrain` untimed steps, so that the envs
    play the long games of a trained player; then staged copies of it at each split of STAGE_SPLITS, which carry on from
    the same env state and key chain.  The unstaged and staged learners' timed launches are alternated.  Each staged row
    carries its rate over the unstaged one and the share of envs in each stage, averaged over samples taken before and
    after every timed launch.  Also returns the network and 4 096 env boards of the n = 2^16 run, for the search."""
    out, search_net, search_boards = [], None, None
    subs = E.chain_advance(E.words_tensor([0, 1], "cuda"), MODE, steps)
    for n in SIZES:
        flat = g2048.NTupleTDLearner(0, n, alpha=g2048.td.DEFAULT_NTUPLE_ALPHA, rng_mode=MODE)
        flat.train(pretrain)
        learners = {"four_six": flat}
        for t in STAGE_SPLITS:
            learners["four_six_2_stages_t%d" % t[0]] = _promoted(flat, t)
        runs = {k: (_ntuple_run if k == "four_six" else _staged_run)(lr, subs) for k, lr in learners.items()}
        for run in runs.values():
            run()
        torch.cuda.synchronize()
        times = {k: [] for k in runs}
        shares = {k: [] for k in runs if k != "four_six"}
        for _ in range(reps):
            for k, run in runs.items():
                if k in shares:
                    shares[k].append(_stage_shares(learners[k].boards, learners[k].network.stage_thresholds))
                times[k].append(_timed_once(run))
                if k in shares:
                    shares[k].append(_stage_shares(learners[k].boards, learners[k].network.stage_thresholds))
        rows = [_row(k, n, steps, times[k], pretrain_steps=pretrain) for k in runs]
        for row in rows[1:]:
            row["rate_over_unstaged"] = row["learning_steps_per_s"] / rows[0]["learning_steps_per_s"]
            samples = shares[row["what"]]
            row["mean_share_of_envs_per_stage"] = [round(sum(x[s] for x in samples) / len(samples), 4)
                                                   for s in range(len(samples[0]))]
            print(json.dumps(row), file=sys.stderr, flush=True)
        out += rows
        if n == 1 << 16:
            search_net = NTupleNetwork(flat.network.placements, flat.network.n_weights, flat.network.weights)
            search_boards = flat.boards[:4096].clone()
        del flat, learners, runs
        torch.cuda.empty_cache()
    return out, search_net, search_boards


def stages_search(reps: int, net, boards) -> list:
    """Leaves/s of the staged leaf next to the unstaged one, on the same values (staged copies of `net`) and on boards
    of the trained learner's own games, whose stages are reported per split."""
    flush_buf = torch.empty(512 << 20, dtype=torch.uint8, device="cuda")
    leaves_nets = [("four_six", net, None)]
    leaves_nets += [("four_six_2_stages_t%d" % t[0], NTupleNetwork.staged(net, t), _stage_shares(boards, t))
                    for t in STAGE_SPLITS]
    out = []
    for depth in (2, 3):
        for leaf, nw, share in leaves_nets:
            fn = lambda c=None, nw=nw: E.expectimax_values_ntuple(boards, depth, nw.placements, nw.weights, 0.0, c,  # noqa: E731
                                                                   stages=nw.stages)
            counters = torch.zeros(2, dtype=torch.int64, device="cuda")
            fn(counters)
            leaves = int(counters[0].item())
            times = device_times(fn, reps, flush_buf)
            med = statistics.median(times)
            out.append({"depth": depth, "leaf": leaf, "boards": int(boards.shape[0]), "leaves": leaves,
                        "share_of_boards_per_stage": share, "ms": [round(t * 1e3, 3) for t in times],
                        "leaves_per_s": leaves / med})
            print(json.dumps(out[-1]), file=sys.stderr, flush=True)
    del leaves_nets
    torch.cuda.empty_cache()
    return out


def stages_quality(total: int, block: int, B: int, deep: int) -> list:
    """TD at alpha 0.02 from zeros at n = 2^16 (seed 0) for `total` steps: unstaged, staged (13,) and (14,), and half
    unstaged then staged((13,)); each with its training wall time and its greedy and depth-2 players on the seed-7
    games."""
    alpha, n = g2048.td.DEFAULT_NTUPLE_ALPHA, 1 << 16
    out = []
    for name in ("unstaged", "staged_t13", "staged_t14", "half_unstaged_then_staged_t13"):
        if name == "unstaged" or name.startswith("half"):
            net = NTupleNetwork.four_six()
        else:
            net = NTupleNetwork.staged(NTupleNetwork.four_six(), (13,) if name.endswith("13") else (14,))
        lr = g2048.NTupleTDLearner(0, n, network=net, alpha=alpha)
        if name.startswith("half"):
            curve, wall = _train(lr, total // 2, block)
            promoted = _promoted(lr, (13,))
            del lr
            torch.cuda.empty_cache()
            lr = promoted
            curve2, wall2 = _train(lr, total - total // 2, block)
            curve, wall = curve + curve2, wall + wall2
        else:
            curve, wall = _train(lr, total, block)
        row = {"run": name, "alpha": alpha, "n": n, "steps": total, "block": block, "train_seconds": round(wall, 2),
               "curve_mean_score": curve}
        for depth, games in ((1, B), (2, deep)):
            row[f"depth{depth}"] = play(g2048.ExpectimaxPolicy(depth=depth, network=lr.network, reward_weight=1.0),
                                        games)
        out.append(row)
        print(json.dumps(row), file=sys.stderr, flush=True)
        del lr
        torch.cuda.empty_cache()
    return out


def main_stages(args) -> None:
    result = {"gpu": gpu_info(), "l2": "warm for learning (the touched weights stay resident); flushed for search"}
    if not args.skip_speed:
        result["speed"], net, boards = stages_speed(args.steps, args.pretrain_steps)
        result["search"] = stages_search(args.reps, net, boards)
        del net, boards
        torch.cuda.empty_cache()
    if not args.speed_only:
        result["quality"] = stages_quality(args.long_steps, args.block, args.games, args.deep_games)
    _emit(result, args.out)


LAMBDA_HS = (2, 3, 5)
LAMBDA_GRID = tuple((lam, h) for lam in (0.25, 0.5, 0.75) for h in LAMBDA_HS)


def _lambda_learner(kind, n, lam, h, network=None):
    cls = g2048.NTupleTCLearner if kind == "tc" else g2048.NTupleTDLearner
    alpha = g2048.td.DEFAULT_NTUPLE_TC_ALPHA if kind == "tc" else g2048.td.DEFAULT_NTUPLE_ALPHA
    return cls(0, n, network=network, alpha=alpha, rng_mode=MODE, lam=lam, horizon=h)


def _lambda_run(lr, subs, stats=None):
    net = lr.network
    tc = isinstance(lr, g2048.NTupleTCLearner)
    if lr.horizon == 1:
        if tc:
            return lambda st=stats: E.ntuple_tc_train(lr.boards, lr.after, lr.scores, lr.lengths, net.placements,
                                                      net.weights, lr.err_sum, lr.abs_err_sum, lr.alpha, subs, MODE,
                                                      lr._scratch, st)
        return lambda st=stats: E.ntuple_td_train(lr.boards, lr.after, lr.scores, lr.lengths, net.placements,
                                                  net.weights, lr.alpha, subs, MODE, lr._scratch, st)
    if tc:
        return lambda st=stats: E.ntuple_lambda_tc_train(lr.boards, lr.after, lr.scores, lr.lengths, net.placements,
                                                         net.weights, lr.err_sum, lr.abs_err_sum, lr.alpha, lr.lam,
                                                         lr.hist_after, lr.hist_delta, subs, MODE, lr._scratch, st)
    return lambda st=stats: E.ntuple_lambda_td_train(lr.boards, lr.after, lr.scores, lr.lengths, net.placements,
                                                     net.weights, lr.alpha, lr.lam, lr.hist_after, lr.hist_delta,
                                                     subs, MODE, lr._scratch, st)


def _lambda_learners(n, pretrain, hs):
    """The 4x6 network trained by TD (alpha 0.02, seed 0) for `pretrain` steps at n envs, and learners that carry on
    from its weights and env state: name -> learner, for TD(0), TC and TD / TC(lambda = 0.5) at each h of hs."""
    flat = g2048.NTupleTDLearner(0, n, alpha=g2048.td.DEFAULT_NTUPLE_ALPHA, rng_mode=MODE)
    flat.train(pretrain)
    specs = [("td", "td", 0.0, 1), ("tc", "tc", 0.0, 1)]
    specs += [(f"{kind}_lambda_h{h}", kind, 0.5, h) for h in hs for kind in ("td", "tc")]
    out = {}
    for name, kind, lam, h in specs:
        net = NTupleNetwork(flat.network.placements, flat.network.n_weights, flat.network.weights.clone())
        lr = _lambda_learner(kind, n, lam, h, net)
        for k in ("boards", "after", "scores", "lengths"):
            getattr(lr, k).copy_(getattr(flat, k))
        out[name] = lr
    del flat
    torch.cuda.empty_cache()
    return out


def lambda_speed(steps: int, pretrain: int, reps: int = 3) -> list:
    """At each size: the learners of _lambda_learners (h capped so that n * h <= 2^20), all warmed up, then their timed
    launches alternated on the same sub keys."""
    out = []
    subs = E.chain_advance(E.words_tensor([0, 1], "cuda"), MODE, steps)
    for n in SIZES:
        learners = _lambda_learners(n, pretrain, [h for h in LAMBDA_HS if n * h <= 1 << 20])
        runs = {k: _lambda_run(lr, subs) for k, lr in learners.items()}
        for run in runs.values():
            run()
        torch.cuda.synchronize()
        times = {k: [] for k in runs}
        for _ in range(reps):
            for k, run in runs.items():
                times[k].append(_timed_once(run))
        rows = [_row(k, n, steps, times[k], pretrain_steps=pretrain, horizon=learners[k].horizon) for k in runs]
        rate = {r["what"]: r["learning_steps_per_s"] for r in rows}
        for row in rows:
            row["rate_over_td0"] = row["learning_steps_per_s"] / rate["td"]
            if row["what"].startswith("tc"):
                row["rate_over_tc"] = row["learning_steps_per_s"] / rate["tc"]
            print(json.dumps(row), file=sys.stderr, flush=True)
        out += rows
        del learners, runs
        torch.cuda.empty_cache()
    return out


def lambda_phase_probe(steps: int, pretrain: int) -> list:
    """In a build with -DG2048_NTUPLE_PHASES: the accumulate / apply split of TD(0), TC and TD / TC(lambda) at h = 3,
    one launch of `steps` steps after a warm-up launch, from the pretrained start of lambda_speed."""
    out = []
    subs = E.chain_advance(E.words_tensor([0, 1], "cuda"), MODE, steps)
    for n in SIZES:
        learners = _lambda_learners(n, pretrain, (3,))
        for name, lr in learners.items():
            stats = torch.zeros(32, dtype=torch.int64, device="cuda")
            run = _lambda_run(lr, subs)
            run()
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            run(stats)
            b.record()
            torch.cuda.synchronize()
            acc_ns, apply_ns, listed = (int(x) for x in stats[8:11].tolist())
            out.append({"n": n, "learner": name, "steps": steps, "us_per_step": a.elapsed_time(b) * 1e3 / steps,
                        "accumulate_us_per_step": acc_ns / 1e3 / steps, "apply_us_per_step": apply_ns / 1e3 / steps,
                        "entries_listed_per_step": listed / steps})
            print(json.dumps(out[-1]), file=sys.stderr, flush=True)
        del learners
        torch.cuda.empty_cache()
    return out


def lambda_phases(steps: int, pretrain: int) -> dict:
    tmp = Path(tempfile.mkdtemp(prefix="g2048_ntuple_phases_"))
    lib = tmp / "libg2048_phases.so"
    subprocess.run(["make", "-C", str(ROOT / "2048-ppo-agent_b200" / "csrc"), "-j16", f"OUT={lib}", f"BUILD={tmp / 'build'}",
                    "EXTRA=-DG2048_NTUPLE_PHASES"], check=True, capture_output=True)
    env = dict(os.environ, G2048_LIB=str(lib))
    res = subprocess.run([sys.executable, __file__, "--phase-probe", "--lambda", "--steps", str(steps),
                          "--pretrain-steps", str(pretrain)], env=env, capture_output=True, text=True, check=True)
    return {"build": "-DG2048_NTUPLE_PHASES", "rows": json.loads(res.stdout.strip().splitlines()[-1])}


def _players(net, B, deep) -> dict:
    return {f"depth{depth}": play(g2048.ExpectimaxPolicy(depth=depth, network=net, reward_weight=1.0), games)
            for depth, games in ((1, B), (2, deep))}


def lambda_quality(short: int, long: int, block: int, B: int, deep: int) -> list:
    """From the zero 4x6 network at n = 2^16: every setting evaluated after `short` steps and, continuing the same
    run, after `long` steps; then the best lambda setting at `long` (greedy mean) as a staged (13,) run next to staged
    TD(0)."""
    n = 1 << 16
    out = []
    settings = [("td", 0.0, 1), ("tc", 0.0, 1)] + [(k, lam, h) for k in ("td", "tc") for lam, h in LAMBDA_GRID]
    for kind, lam, h in settings:
        lr = _lambda_learner(kind, n, lam, h)
        curve, wall = _train(lr, short, block)
        row = {"learner": kind, "lam": lam, "horizon": h, "alpha": lr.alpha, "n": n, "block": block}
        row[f"steps{short}"] = {"train_seconds": round(wall, 2), **_players(lr.network, B, deep)}
        curve2, wall2 = _train(lr, long - short, block)
        row[f"steps{long}"] = {"train_seconds": round(wall + wall2, 2), **_players(lr.network, B, deep)}
        row["curve_mean_score"] = curve + curve2
        out.append(row)
        print(json.dumps(row), file=sys.stderr, flush=True)
        del lr
        torch.cuda.empty_cache()
    best = max((r for r in out if r["horizon"] > 1), key=lambda r: r[f"steps{long}"]["depth1"]["mean_score"])
    for kind, lam, h in (("td", 0.0, 1), (best["learner"], best["lam"], best["horizon"])):
        lr = _lambda_learner(kind, n, lam, h, NTupleNetwork.staged(NTupleNetwork.four_six(), (13,)))
        curve, wall = _train(lr, long, block)
        row = {"learner": kind, "lam": lam, "horizon": h, "alpha": lr.alpha, "n": n, "block": block,
               "stage_thresholds": [13], f"steps{long}": {"train_seconds": round(wall, 2), **_players(lr.network, B, deep)},
               "curve_mean_score": curve}
        out.append(row)
        print(json.dumps(row), file=sys.stderr, flush=True)
        del lr
        torch.cuda.empty_cache()
    return out


def main_lambda(args) -> None:
    result = {"gpu": gpu_info(), "l2": "warm for learning (the touched weights stay resident)"}
    if not args.skip_speed:
        result["speed"] = lambda_speed(args.steps, args.pretrain_steps)
        result["phases"] = lambda_phases(args.steps, args.pretrain_steps)
    if not args.speed_only:
        result["quality"] = lambda_quality(args.sweep_steps, args.long_steps, args.block, args.games, args.deep_games)
    _emit(result, args.out)


def _carousel_run(lr, subs):
    net = lr.network
    return lambda: E.ntuple_carousel_td_train(lr.boards, lr.after, lr.scores, lr.lengths, net.placements, net.weights,
                                              lr.alpha, 0.0, None, None, lr.start_stage, lr.stage_pool, subs, MODE,
                                              lr._scratch, stages=net.stages)


def _start_shares(lr) -> list:
    return [round(float((lr.start_stage == s).float().mean()), 4) for s in range(lr.network.n_stages)]


def carousel_speed(steps: int, pretrain: int, thresholds, reps: int = 3) -> list:
    """At each size, the 4x6 network trained by TD (alpha 0.02, seed 0) for `pretrain` untimed steps, then staged
    copies at `thresholds` with and without the carousel, which carry on from the same envs; their timed launches
    alternated.  The carousel row carries its rate over the staged one, the non-zero pool entries after timing, and
    (both) the share of envs per stage and, for the carousel, per start stage, averaged over samples taken before and
    after every timed launch."""
    out = []
    subs = E.chain_advance(E.words_tensor([0, 1], "cuda"), MODE, steps)
    for n in SIZES:
        flat = g2048.NTupleTDLearner(0, n, alpha=g2048.td.DEFAULT_NTUPLE_ALPHA, rng_mode=MODE)
        flat.train(pretrain)
        learners = {"staged": _promoted(flat, thresholds), "carousel": _promoted(flat, thresholds, carousel=True)}
        del flat
        torch.cuda.empty_cache()
        runs = {"staged": _staged_run(learners["staged"], subs), "carousel": _carousel_run(learners["carousel"], subs)}
        for run in runs.values():
            run()
        torch.cuda.synchronize()
        times = {k: [] for k in runs}
        shares = {k: [] for k in runs}
        starts = []
        for _ in range(reps):
            for k, run in runs.items():
                sample = lambda lr=learners[k]: (shares[k].append(_stage_shares(lr.boards, thresholds)),  # noqa: E731
                                                 lr.carousel and starts.append(_start_shares(lr)))
                sample()
                times[k].append(_timed_once(run))
                sample()
        rows = [_row(k, n, steps, times[k], pretrain_steps=pretrain, stage_thresholds=list(thresholds)) for k in runs]
        for row in rows:
            samples = shares[row["what"]]
            row["mean_share_of_envs_per_stage"] = [round(sum(x[s] for x in samples) / len(samples), 4)
                                                   for s in range(len(samples[0]))]
        rows[1]["rate_over_staged"] = rows[1]["learning_steps_per_s"] / rows[0]["learning_steps_per_s"]
        rows[1]["mean_share_of_envs_per_start_stage"] = [round(sum(x[s] for x in starts) / len(starts), 4)
                                                         for s in range(len(starts[0]))]
        rows[1]["pool_entries_nonzero"] = int((learners["carousel"].stage_pool != 0).sum())
        for row in rows:
            print(json.dumps(row), file=sys.stderr, flush=True)
        out += rows
        del learners, runs
        torch.cuda.empty_cache()
    return out


def _train_sampled(lr, total, block, shares):
    """_train, appending the share of envs in stage 1 of (13,) after every block to `shares`; also returns the shaped
    episodes and env-steps of a carousel learner."""
    curve, wall, shaped = [], 0.0, [0, 0]
    for _ in range(total // block):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        s = lr.train(block)
        torch.cuda.synchronize()
        wall += time.perf_counter() - t0
        curve.append(round(s["score_sum"] / max(s["episodes"], 1), 1))
        shares.append(_stage_shares(lr.boards, (13,))[1])
        shaped[0] += s.get("shaped_episodes", 0)
        shaped[1] += s.get("shaped_env_steps", 0)
    return curve, wall, shaped


CAROUSEL_RUNS = ("unstaged", "staged_t13", "staged_t13_carousel", "half_unstaged_then_staged_t13_carousel")


def carousel_quality(short: int, long: int, block: int, B: int, deep: int, runs=CAROUSEL_RUNS) -> list:
    """TC(lambda = 0.5, h = 3) at alpha 0.02 from the zero 4x6 network at n = 2^16 (seed 0): unstaged, staged (13,),
    staged (13,) with the carousel, and short / 2 steps unstaged then staged((13,)) with the carousel; each evaluated
    after `short` steps and, continuing, after `long`."""
    n, lam, h, alpha = 1 << 16, 0.5, 3, g2048.td.DEFAULT_NTUPLE_TC_ALPHA
    out = []
    for name in runs:
        net = NTupleNetwork.four_six()
        if name.startswith("staged"):
            net = NTupleNetwork.staged(net, (13,))
        lr = g2048.NTupleTCLearner(0, n, network=net, alpha=alpha, lam=lam, horizon=h,
                                   carousel=name == "staged_t13_carousel")
        row = {"run": name, "learner": "tc", "lam": lam, "horizon": h, "alpha": alpha, "n": n, "block": block}
        shares, curve, wall, shaped, done = [], [], 0.0, [0, 0], 0
        for upto in (short, long):
            if name.startswith("half") and done == 0:
                c, w, _ = _train_sampled(lr, short // 2, block, shares)
                curve, wall, done = curve + c, wall + w, short // 2
                promoted = _promoted(lr, (13,), carousel=True)
                del lr
                torch.cuda.empty_cache()
                lr = promoted
            c, w, sh = _train_sampled(lr, upto - done, block, shares)
            curve, wall, done = curve + c, wall + w, upto
            shaped = [shaped[0] + sh[0], shaped[1] + sh[1]]
            stage1 = None
            if lr.network.n_stages > 1:
                stage1 = int((lr.abs_err_sum[lr.network.stage_stride:] > 0).sum())
            row[f"steps{upto}"] = {"train_seconds": round(wall, 2), **_players(lr.network, B, deep),
                                   "share_of_env_steps_in_stage1_of_t13": round(sum(shares) / len(shares), 4),
                                   "stage1_entries_updated": stage1, "shaped_episodes": shaped[0],
                                   "shaped_env_steps": shaped[1]}
            print(json.dumps(row), file=sys.stderr, flush=True)
        row["curve_mean_score"] = curve
        out.append(row)
        del lr
        torch.cuda.empty_cache()
    return out


def main_carousel(args) -> None:
    result = {"gpu": gpu_info(), "l2": "warm for learning (the touched weights stay resident)"}
    if not args.skip_speed:
        result["speed_mechanism"] = carousel_speed(args.steps, args.carousel_pretrain_steps, (14,))
        result["speed_mix"] = carousel_speed(args.steps, args.pretrain_steps, (13,))
    if not args.speed_only:
        result["quality"] = carousel_quality(args.sweep_steps, args.long_steps, args.block, args.games, args.deep_games,
                                             args.carousel_runs.split(","))
    _emit(result, args.out)


def main_tc(args) -> None:
    result = {"gpu": gpu_info(), "l2": "warm for learning (the touched weights stay resident)"}
    if not args.skip_speed:
        result["speed"] = tc_speed(args.steps)
        result["phases"] = phases(args.steps, tc=True)
    if not args.speed_only:
        rows, (_, alpha, _, _) = sweep(1 << 16, args.sweep_steps, args.block, args.games, TC_ALPHAS,
                                       g2048.NTupleTCLearner)
        result["tc_sweep"] = rows
        result["equal_steps"] = equal_steps(alpha, (args.sweep_steps, args.long_steps), args.block, args.games,
                                            args.deep_games)
    _emit(result, args.out)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=500, help="batch steps per timed launch")
    ap.add_argument("--sweep-steps", type=int, default=4000)
    ap.add_argument("--block", type=int, default=250)
    ap.add_argument("--games", type=int, default=1024)
    ap.add_argument("--deep-games", type=int, default=128, help="games for the depth-2 and depth-3 players")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--speed-only", action="store_true", help="speed, phases, lines and n_weights only")
    ap.add_argument("--skip-speed", action="store_true", help="the sweep, search and players only")
    ap.add_argument("--tc", action="store_true", help="the temporal coherence learner against TD (see above)")
    ap.add_argument("--stages", action="store_true", help="multi-stage networks against the unstaged one (see above)")
    ap.add_argument("--lambda", dest="lam", action="store_true",
                    help="delayed TD(lambda) / TC(lambda) against TD(0) and TC (see above)")
    ap.add_argument("--carousel", action="store_true", help="carousel shaping of staged networks (see above)")
    ap.add_argument("--pretrain-steps", type=int, default=20000,
                    help="untimed training before the --stages, --lambda and --carousel (real mix) speed runs")
    ap.add_argument("--carousel-runs", default=",".join(CAROUSEL_RUNS),
                    help="comma-separated quality runs of --carousel (default: all four)")
    ap.add_argument("--carousel-pretrain-steps", type=int, default=2000,
                    help="untimed training before the --carousel speed run of the mechanism")
    ap.add_argument("--long-steps", type=int, default=40000,
                    help="the longer equal-steps comparison of --tc, and the runs of --stages")
    ap.add_argument("--phase-probe", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if args.phase_probe:
        probe = lambda_phase_probe(args.steps, args.pretrain_steps) if args.lam else phase_probe(args.steps, args.tc)
        print(json.dumps(probe))
        return
    if args.lam:
        main_lambda(args)
        return
    if args.carousel:
        main_carousel(args)
        return
    if args.tc:
        main_tc(args)
        return
    if args.stages:
        main_stages(args)
        return
    result = {"gpu": gpu_info(), "l2": "warm for learning (the touched weights stay resident); flushed for search"}
    if not args.skip_speed:
        result["speed"] = speed(args.steps)
        result["phases"] = phases(args.steps)
        result["lines_vs_row"] = lines_vs_row(args.steps)
        result["n_weights"] = weights_size(args.steps)
    if args.speed_only:
        _emit(result, args.out)
        return
    B = args.games
    rows, (_, alpha, net, wall) = sweep(1 << 16, args.sweep_steps, args.block, B)
    result["sweep"] = rows
    result["search"] = search(args.reps, net)
    # the row table: the same learning steps, and the same training wall time as the chosen 4x6 run
    row = g2048.TDLearner(0, 1 << 16)
    _, row_wall = _train(row, args.sweep_steps, args.block)
    row_time = g2048.TDLearner(0, 1 << 16)
    steps_in_wall = max(args.block, int(args.sweep_steps * wall / row_wall) // args.block * args.block)
    _train(row_time, steps_in_wall, args.block)
    players = {"drul": play(g2048.act_drul, B)}
    for depth in (1, 2, 3):
        g = B if depth == 1 else args.deep_games
        players[f"four_six_alpha{alpha}_depth{depth}"] = play(
            g2048.ExpectimaxPolicy(depth=depth, network=net, reward_weight=1.0), g)
        players[f"row_table_same_steps_depth{depth}"] = play(
            g2048.ExpectimaxPolicy(depth=depth, row_values=row.table, reward_weight=1.0), g)
        players[f"row_table_same_wall_depth{depth}"] = play(
            g2048.ExpectimaxPolicy(depth=depth, row_values=row_time.table, reward_weight=1.0), g)
        players[f"default_table_depth{depth}"] = play(g2048.ExpectimaxPolicy(depth=depth), g)
        print(json.dumps({k: v for k, v in players.items() if k.endswith(f"depth{depth}")}), file=sys.stderr, flush=True)
    result["players"] = {"seed": 7, "alpha": alpha, "four_six_train_seconds": round(wall, 2),
                         "row_train_seconds": round(row_wall, 2), "row_steps_in_same_wall": steps_in_wall,
                         "results": players}
    _emit(result, args.out)


def _emit(result: dict, out) -> None:
    line = json.dumps(result)
    print(line)
    if out:
        Path(out).parent.mkdir(parents=True, exist_ok=True)
        Path(out).write_text(line + "\n")


if __name__ == "__main__":
    main()
