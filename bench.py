#!/usr/bin/env python
"""Benchmark of the rollout hot path (contract: python bench.py --gpus N --steps K --warmup W).

A "step" is one pass of the hot path over one batch: BASELINE.json's C5 workload -- a batch of 2^24
(16 M) 2048 envs is played to termination under the random policy (act_randomly) by the persistent
`g2048_play` kernel (key chain generated on the device inside the step), followed by the episode
statistics reduction (one NCCL collective when N > 1).  The batch is sharded over the ranks with
global env indices: the default is C5 as BASELINE.json states it -- the SAME 16 M envs at N = 1, 2,
4, 8 ("scaling": "strong"); `--scaling weak --envs-per-gpu E` keeps the per-GPU work fixed instead,
and every line also carries a short weak-scaling measurement (`weak_scaling`, 2^21 envs per GPU --
round 1's configuration).  At every N each rank checks a window of its own shard against the
oracle and the pass flags are all-reduced into `parity`.

Prints ONE JSON line.  `value` is device-timed with everything resident in HBM; `e2e` is the same
metric through the host-buffer C entry point `g2048_play_host` (its own allocations, H2D/D2H copies
and synchronisation inside the timed region).  `roofline` is the dominant kernel (integer-issue
bound), `roofline_hbm` lists the HBM-bound rollout-write / GAE kernels, `cpu_baseline` is the
oracle's C port of the same workload on the host cores.

`--impl reference` times the reference's CPU path.  The reference itself (Pgx on JAX) cannot be
installed here (jax / pgx / torch2jax are not in the image and there is no network), so this arm
runs the oracle's C restatement of it -- pinned to the reference's golden artefacts -- with all host
threads, on a bounded sample of the same workload.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
for _p in (str(ROOT), str(ROOT / "2048-ppo-agent_b200")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

TOTAL_ENVS = 1 << 24   # C5: 16 M envs, sharded over the ranks (strong scaling, the default)
ENVS_PER_GPU = 1 << 21  # --scaling weak, and the `weak_scaling` leg of every line
SEED = 2048
MAX_STEPS = 2048  # loop steps of keys generated per batch (random episodes stay below ~700; checked via cut_short)
# SURVEY 8(d)'s paper count (74 int instr per Threefry block x 10 (5) + ~250 game logic); the roofline uses the
# MEASURED thread instructions per env-step of the shipped kernels instead when profiles/inst_counts.json is there
ALG_INSTR = {"random": 990, "drul": 620}
CPU_SAMPLE_ENVS = 1 << 17
REF_SAMPLE_ENVS = 1 << 16
PARITY_WINDOW = 4096  # envs of its own shard that every rank checks against the oracle


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="g2048", choices=["g2048", "reference"])
    ap.add_argument("--policy", default="random", choices=["random", "drul"])
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"],
                    help="strong: --envs envs in all, sharded over the GPUs (C5); weak: --envs-per-gpu envs on every GPU")
    ap.add_argument("--envs", type=int, default=TOTAL_ENVS)
    ap.add_argument("--envs-per-gpu", type=int, default=ENVS_PER_GPU)
    ap.add_argument("--no-extras", action="store_true", help="skip the secondary kernel measurements")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned to DIR/play_stats.npy (float64): the reduced statistics "
                         "block of g2048_play (include/g2048.h), so that two builds can be compared on the same inputs")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


# ------------------------------------------------------------------------------------------ helpers
class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    QUERY = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.rows = []  # (arrival time, fields)
        self.proc = None
        self.gpu_index = gpu_index
        self.t_begin = self.t_end = None

    def start(self):
        """Started BEFORE the warm-up steps: nvidia-smi needs a few hundred ms to produce its first line, more than a
        short timed region lasts."""
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.gpu_index), f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits", "-lms", "20"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [c.strip() for c in line.split(",")]))

    def begin(self):
        self.t_begin = time.perf_counter()

    def end(self):
        self.t_end = time.perf_counter()

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.05)
        self.proc.terminate()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

        def parse(rows):
            sm, mx, reasons, power = [], [], set(), []
            for _, r in rows:
                try:
                    sm.append(float(r[0]))
                    mx.append(float(r[1]))
                    power.append(float(r[2]))
                    for name, v in zip(names, r[3:7]):
                        if v.lower().startswith("active"):
                            reasons.add(name)
                except (ValueError, IndexError):
                    continue
            return sm, mx, reasons, power

        # a line printed at time t was sampled just before t: take the lines that arrived inside the timed region
        # (plus one sampling period); if the region was too short to catch two, widen to the warm-up steps before
        # it, which run the same kernels
        inside = [row for row in self.rows if self.t_begin is not None and self.t_begin <= row[0] <= self.t_end + 0.03]
        window = "timed region"
        if len(inside) < 2:
            inside = [row for row in self.rows if self.t_end is None or row[0] <= self.t_end + 0.03]
            window = "warm-up + timed region"
        sm, mx, reasons, power = parse(inside)
        if sm:
            cut = statistics.median(power)  # samples under load only: the top half of the observed power draw
            loaded = [x for x, pw in zip(sm, power) if pw >= cut] or sm
            return {"sm_mhz": statistics.median(loaded), "sm_max_mhz": max(mx), "reasons": sorted(reasons),
                    "samples": len(sm), "window": window, "power_w_max": max(power)}
        return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}


def measured_hbm_peak():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except (KeyError, ValueError):
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def oracle_play_rate(seed: int, batch_global: int, n_sample: int, policy: int, mode: int, min_seconds: float):
    """Times the oracle's C port (OpenMP, all host threads) on envs [0, n_sample) of the batch."""
    from oracle import c_oracle as CO

    CO.set_num_threads(os.cpu_count() or 1)  # torchrun exports OMP_NUM_THREADS=1; the baseline uses every host core
    threads = CO.num_threads()
    total_steps, t0, reps = 0, time.perf_counter(), 0
    out = None
    while True:
        out = CO.play(seed, batch_global, policy, mode, env_lo=0, env_hi=n_sample, max_steps=MAX_STEPS)
        total_steps += int(out["lengths"].sum())
        reps += 1
        if time.perf_counter() - t0 >= min_seconds:
            break
    dt = time.perf_counter() - t0
    return total_steps / dt, threads, reps, out


# ------------------------------------------------------------------------------------------ workload
def batch_shape(args, world: int, rank: int):
    """-> (batch_global, env_lo, n): the envs of the global batch this rank plays."""
    if args.scaling == "strong":
        batch_global = args.envs
        lo, hi = batch_global * rank // world, batch_global * (rank + 1) // world
        return batch_global, lo, hi - lo
    return args.envs_per_gpu * world, args.envs_per_gpu * rank, args.envs_per_gpu


def workload_config(args, world: int):
    batch_global, _, n0 = batch_shape(args, world, 0)
    how = (f"{batch_global} envs in all, sharded over {world} GPU(s) (BASELINE.json configs[4]: 16M envs across 1/2/4/8 B200)"
           if args.scaling == "strong" else f"{args.envs_per_gpu} envs per GPU")
    return {
        "workload": f"C5 throughput sweep: {args.policy}-policy 2048 envs played to termination + episode-stats reduction; {how}",
        "policy": args.policy, "scaling": args.scaling, "global_batch": batch_global, "envs_per_gpu": n0,
        "rng": "threefry2x32 partitionable (jax 0.5.3 default)", "seed": SEED,
        "l2": "L2 flushed (512 MiB write) between timed steps; the kernel's inputs are 32 KiB of keys, env state lives in registers",
    }


# ------------------------------------------------------------------------------------------ reference arm
def run_reference(args, rank: int):
    if rank != 0:
        return
    policy = 0 if args.policy == "random" else 1
    batch_global, _, _ = batch_shape(args, args.gpus, 0)
    n_sample = min(REF_SAMPLE_ENVS, batch_global)
    from oracle import c_oracle as CO

    CO.set_num_threads(os.cpu_count() or 1)  # torchrun exports OMP_NUM_THREADS=1; the reference arm uses every host core
    times, steps_done = [], []
    for i in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        out = CO.play(SEED + i, batch_global, policy, 1, env_lo=0, env_hi=n_sample, max_steps=MAX_STEPS)
        dt = time.perf_counter() - t0
        if i >= args.warmup:
            times.append(dt)
            steps_done.append(int(out["lengths"].sum()))
    value = sum(steps_done) / sum(times)
    sample = (f"envs [0,{n_sample}) of the {batch_global}-env batch per step, played to termination by the oracle's C "
              f"restatement of the Pgx/JAX path (jax, pgx, torch2jax absent from the image: the reference itself cannot run)")
    line = {
        "impl": "reference", "metric": "env_steps_per_sec", "value": value, "unit": "env-steps/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * sum(times) / len(times),
        "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "u8/u32 integer", "data": "synthetic",
        "config": workload_config(args, args.gpus),
        "cpu_baseline": {"value": value, "unit": "env-steps/s", "cores": CO.num_threads(), "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def measured_inst_counts():
    """profiles/inst_counts.json: smsp__thread_inst_executed.sum per env-step of the shipped play kernels (ncu)."""
    try:
        return json.loads((ROOT / "profiles" / "inst_counts.json").read_text())
    except Exception:  # noqa: BLE001 -- evidence, not a dependency
        return {}


# ------------------------------------------------------------------------------------------ our arm
def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    if world != args.gpus and not (world == 1 and args.gpus == 1):
        raise SystemExit(f"--gpus {args.gpus} needs WORLD_SIZE {args.gpus} (launch with torch.distributed.run); got {world}")

    import numpy as np
    import torch
    import torch.distributed as dist

    from g2048 import _native as N
    from g2048 import engine as E

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    # stdout carries exactly ONE line, the JSON: whatever libraries print there meanwhile (NCCL's version banner does, at
    # the first collective) goes to stderr instead -- file descriptor 1 is pointed at stderr until the line is written
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)
    if world > 1:
        # keep stdout for the one JSON line: NCCL's version / debug banner goes to stderr
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        import datetime

        # a collective that some rank never joins should fail within minutes, not after NCCL's default 10
        dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(seconds=300))

    policy_id = E.POLICY_RANDOM if args.policy == "random" else E.POLICY_DRUL
    mode = E.RNG_PARTITIONABLE
    n_subs = 1 + 2 * MAX_STEPS
    flush_buf = torch.empty(512 << 20, dtype=torch.uint8, device=dev)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def reduce_stats(stats):
        """ONE collective per step: all-gather the 256-byte statistics blocks, reduce locally (sum; slot 5 is a max)."""
        if world == 1:
            return stats
        flat = torch.empty(world * N.PLAY_STATS_WORDS, dtype=torch.int64, device=dev)
        dist.all_gather_into_tensor(flat, stats)
        gathered = flat.view(world, N.PLAY_STATS_WORDS)
        out = gathered.sum(dim=0)
        out[5] = gathered[:, 5].max()
        return out

    def timed_play_loop(batch_global, lo, n, warmup, steps, sampler=None):
        """warmup + steps batches; per step: key chain (prefetched on a side stream one batch ahead) + persistent play
        kernel + statistics reduction, device-timed with CUDA events (L2 flushed before each step).  Returns
        (seconds of the timed steps (max over ranks), reduced statistics of the timed steps, launches, seconds inside
        the play kernel, the last timed step's reduced statistics block as the device tensor it returned)."""
        # the inputs of a step (one 8-byte chain key per batch) are resident in HBM before the timed region
        step_keys = [E.words_tensor(list(E.key_words(SEED + i)), dev) for i in range(warmup + steps)]
        side = torch.cuda.Stream(device=dev)
        chains, launches = {}, {"n": 0}

        def prefetch_chain(i: int):
            # The key chain of a batch is sequential (one thread, ~0.14 us per split): it is generated on a side stream
            # one batch ahead, overlapping the previous batch's play kernel; the first batch waits for it.
            if i < len(step_keys) and i not in chains:
                with torch.cuda.stream(side):  # depends only on step_keys, which were ready before the timed region
                    subs_i = E.chain_advance(step_keys[i], mode, n_subs)
                    ev = torch.cuda.Event()
                    ev.record(side)
                chains[i] = (subs_i, ev)
                launches["n"] += 1

        kernel_events = []

        def one_step(i: int):
            prefetch_chain(i)
            subs, ev = chains.pop(i)
            torch.cuda.current_stream().wait_event(ev)
            k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            k0.record()
            out = E.play(policy_id, subs, batch_global, lo, n, mode, per_env=False)
            k1.record()
            kernel_events.append((k0, k1))
            subs.record_stream(torch.cuda.current_stream())
            launches["n"] += 1
            prefetch_chain(i + 1)
            return reduce_stats(out["stats"])

        for i in range(warmup):
            one_step(i)
        barrier()
        launches["n"] = 0
        kernel_events.clear()
        events, stats_all = [], []
        barrier()
        if sampler is not None:
            sampler.begin()
        for i in range(steps):
            flush_buf.fill_(i & 0xFF)  # L2 flush, outside the timed events
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            stats_all.append(one_step(warmup + i))
            b.record()
            events.append((a, b))
        barrier()
        if sampler is not None:
            sampler.end()
        elapsed = sum(a.elapsed_time(b) for a, b in events) * 1e-3
        t = torch.tensor([elapsed], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        kernel_s = sum(a.elapsed_time(b) for a, b in kernel_events) * 1e-3
        return float(t.item()), [E.play_stats_dict(s) for s in stats_all], launches["n"], kernel_s, stats_all[-1]

    # ---- the timed region -----------------------------------------------------------------------------------------
    batch_global, lo, n = batch_shape(args, world, rank)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    elapsed, summaries, gpu_launches, kernel_s, last_stats = timed_play_loop(batch_global, lo, n, args.warmup, args.steps, sampler)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:  # the block is reduced over the ranks: every rank holds the same one
        words = last_stats.cpu().numpy().view(np.uint64)
        assert int(words.max()) < (1 << 53), "a statistics word does not fit a float64 exactly"
        dump_dir = Path(args.dump_outputs)
        dump_dir.mkdir(parents=True, exist_ok=True)
        np.save(dump_dir / "play_stats.npy", words.astype(np.float64))
    total_env_steps = sum(s["env_steps"] for s in summaries)  # after the reduction: whole-job totals
    assert all(s["episodes"] == batch_global and s["cut_short"] == 0 and s["overflowed"] == 0 for s in summaries), summaries[0]
    value = total_env_steps / elapsed

    # ---- parity of THIS rank's shard against the oracle, at every N -------------------------------------------------
    from oracle import c_oracle as CO

    CO.set_num_threads(max(1, (os.cpu_count() or 1) // world))
    key0 = E.words_tensor(list(E.key_words(SEED)), dev)
    subs0 = E.chain_advance(key0, mode, n_subs)
    win = min(PARITY_WINDOW, n)
    w_lo = lo + (n - win) // 2  # a window in the middle of the shard: its env indices are the GLOBAL ones
    chk = E.play(policy_id, subs0, batch_global, w_lo, win, mode, per_env=True)
    ref = CO.play(SEED, batch_global, policy_id, 1, env_lo=w_lo, env_hi=w_lo + win, max_steps=MAX_STEPS)
    same = bool(np.array_equal(chk["lengths"].cpu().numpy(), ref["lengths"])
                and np.array_equal(E.boards_numpy(chk["final_boards"]), ref["final_boards"])
                and np.array_equal(chk["scores"].cpu().numpy(), ref["scores"]))
    flags = torch.tensor([int(same), win], dtype=torch.int64, device=dev)
    per_rank = [flags.clone() for _ in range(world)]
    if world > 1:
        dist.all_gather(per_rank, flags)
    parity = {"ok": all(int(f[0]) == 1 for f in per_rank), "ranks_ok": [bool(int(f[0])) for f in per_rank],
              "parity_checked_envs": [int(f[1]) for f in per_rank],
              "what": "final boards, lengths and scores of a window of each rank's own shard (global env indices), first timed "
                      "batch's seed, CUDA kernel vs the oracle's C restatement"}
    assert parity["ok"], f"a shard differs from the oracle: {parity}"

    # ---- dominant kernel (play), timed INSIDE the step loop above; instruction count per env-step as measured ---------
    steps_per_launch = total_env_steps / args.steps / world  # this is the whole job's mean; shards are equal to <0.1 %
    k_time = kernel_s / args.steps
    counts = measured_inst_counts()

    def instr_per_step(policy_name):
        c = counts.get(policy_name, {})
        if "thread_inst_per_env_step" in c:
            return float(c["thread_inst_per_env_step"]), f"measured: {c.get('source', 'profiles/inst_counts.json')}"
        return float(ALG_INSTR[policy_name]), "SURVEY 8(d) paper count (profiles/inst_counts.json absent)"

    # integer-issue peak: Threefry instruction mix, 4 independent chains per thread, full occupancy
    sms = N.lib.g2048_device_sm_count()
    blocks, threads, iters = sms * 8, 256, 20000
    sink = torch.empty(blocks * threads, dtype=torch.int32, device=dev)
    E.int_peak_probe(blocks, threads, iters, sink)
    torch.cuda.synchronize()
    p_times = []
    for _ in range(3):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        E.int_peak_probe(blocks, threads, iters, sink)
        b.record()
        torch.cuda.synchronize()
        p_times.append(a.elapsed_time(b) * 1e-3)
    int_peak = blocks * threads * iters * 48 / min(p_times) / 1e12  # 16 rounds x 3 instr per iteration
    ipe, ipe_src = instr_per_step(args.policy)
    achieved = ipe * steps_per_launch / k_time / 1e12
    roofline = {
        "kernel": "play3_kernel (g2048_play: row tables in shared memory)", "bound": "int_issue", "achieved": achieved, "peak": int_peak,
        "unit": "Tinstr/s", "frac": achieved / int_peak,
        # dram__bytes_read.sum + dram__bytes_write.sum of one launch of the shipped kernel (ncu --set full), if committed
        "traffic": counts.get(args.policy, {}).get("dram_bytes_per_launch"),
        "instr_per_env_step": ipe, "instr_source": ipe_src,
        "paper_count_frac": ALG_INSTR[args.policy] * steps_per_launch / k_time / 1e12 / int_peak,
        "note": (f"{ipe:.1f} thread instructions per env-step x {steps_per_launch:.0f} env-steps per launch / {k_time * 1e3:.3f} ms "
                 "(CUDA events around the play launch inside the timed step loop, mean over the timed steps); peak = live probe "
                 "of the ADD/SHF/LOP3 Threefry mix on this GPU, measured in this run; the kernel keeps env state in registers, "
                 "so HBM traffic is ~16 B per episode and not the bound"),
        "kernel_ms": k_time * 1e3, "kernel_env_steps": steps_per_launch,
    }

    # ---- end to end through the host-buffer C entry point ------------------------------------------
    e2e_times, e2e_steps = [], 0
    # host result buffer in pinned memory (what a caller that cares about transfer time passes): one 16-byte record per
    # env (G2048EpisodeResult: board, length, score), written by the play kernel itself as episodes end
    records = torch.empty((n, 2), dtype=torch.int64, pin_memory=True).numpy().view(E.EPISODE_RESULT).reshape(n)
    h_len, h_score = records["length"], records["score"]
    h_stats = np.zeros(N.PLAY_STATS_WORDS, np.uint64)
    for i in range(2 + min(args.steps, 5)):
        barrier()
        t0 = time.perf_counter()
        N.call("g2048_play_host_packed", policy_id, SEED + i, None, batch_global, lo, n, mode, records.ctypes.data,
               h_stats.ctypes.data)
        dt = time.perf_counter() - t0
        if i >= 2:
            e2e_times.append(dt)
            e2e_steps += int(h_stats[1])
    te = torch.tensor([sum(e2e_times)], dtype=torch.float64, device=dev)
    se = torch.tensor([e2e_steps], dtype=torch.int64, device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
        dist.all_reduce(se, op=dist.ReduceOp.SUM)
    e2e = {
        "value": float(se.item()) / float(te.item()), "unit": "env-steps/s",
        "h2d_bytes_per_step": 8, "d2h_bytes_per_step": int(16 * n + 8 * N.PLAY_STATS_WORDS),
        "api": "g2048_play_host_packed (C ABI, host buffers): key H2D + chain kernel + play kernel + device-to-host transfer of "
               "every env's final board, length and score (one 16-byte record per env) and the statistics block + synchronise, "
               "per call; the record array is pinned host memory, which the kernel writes directly over PCIe as episodes end "
               "(g2048_play_host with three pageable numpy arrays, copied after the kernel through staging buffers: "
               "e2e.pageable_results); device workspace cached by the library; bytes are per rank",
        # the host arrays really hold the batch: their lengths add up to the statistics block's env-step count
        "results_checked": bool(int(h_len.sum(dtype=np.uint64)) == int(h_stats[1]) and int(h_score.sum(dtype=np.uint64)) == int(h_stats[2])),
    }
    del records, h_len, h_score
    if rank == 0 and world == 1:  # the same call with ordinary numpy result arrays
        p_boards, p_len, p_score = np.empty(n, np.uint64), np.empty(n, np.uint32), np.empty(n, np.uint32)
        pg_times, pg_steps = [], 0
        for i in range(3):
            t0 = time.perf_counter()
            N.call("g2048_play_host", policy_id, SEED + i, None, batch_global, lo, n, mode, p_boards.ctypes.data,
                   p_len.ctypes.data, p_score.ctypes.data, h_stats.ctypes.data)
            dt = time.perf_counter() - t0
            if i >= 1:
                pg_times.append(dt)
                pg_steps += int(h_stats[1])
        e2e["pageable_results"] = {"value": pg_steps / sum(pg_times), "unit": "env-steps/s",
                                   "results_checked": bool(int(p_len.sum(dtype=np.uint64)) == int(h_stats[1]))}
        del p_boards, p_len, p_score
    # the same call when only the episode statistics are wanted (what run_actions_max_tile returns): 256 B come back
    so_times, so_steps = [], 0
    for i in range(1 + min(args.steps, 5)):
        barrier()
        t0 = time.perf_counter()
        N.call("g2048_play_host", policy_id, SEED + i, None, batch_global, lo, n, mode, None, None, None, h_stats.ctypes.data)
        dt = time.perf_counter() - t0
        if i >= 1:
            so_times.append(dt)
            so_steps += int(h_stats[1])
    ts = torch.tensor([sum(so_times)], dtype=torch.float64, device=dev)
    ss = torch.tensor([so_steps], dtype=torch.int64, device=dev)
    if world > 1:
        dist.all_reduce(ts, op=dist.ReduceOp.MAX)
        dist.all_reduce(ss, op=dist.ReduceOp.SUM)
    e2e["statistics_only"] = {"value": float(ss.item()) / float(ts.item()), "unit": "env-steps/s",
                              "d2h_bytes_per_step": int(8 * N.PLAY_STATS_WORDS)}

    # ---- the other scaling mode, short: per-GPU work fixed at 2^21 envs (round 1's bench line) -----------------------
    other = None
    if not args.no_extras and args.scaling == "strong":
        w_global, w_lo2, w_n = ENVS_PER_GPU * world, ENVS_PER_GPU * rank, ENVS_PER_GPU
        w_steps = min(args.steps, 10)
        w_elapsed, w_sum, _, w_kernel, _ = timed_play_loop(w_global, w_lo2, w_n, 3, w_steps)
        w_env_steps = sum(s_["env_steps"] for s_ in w_sum)
        assert all(s_["episodes"] == w_global and s_["cut_short"] == 0 for s_ in w_sum)
        other = {"scaling": "weak", "envs_per_gpu": ENVS_PER_GPU, "global_batch": w_global, "steps": w_steps,
                 "value": w_env_steps / w_elapsed, "unit": "env-steps/s", "ms_per_step": 1e3 * w_elapsed / w_steps,
                 "kernel_ms": 1e3 * w_kernel / w_steps}

    extras = {}
    if not args.no_extras and rank == 0:
        try:
            extras = secondary_measurements(E, N, torch, dev, flush_buf)
        except Exception as exc:  # noqa: BLE001 -- the secondary legs must not cost the headline line
            import traceback

            traceback.print_exc(file=sys.stderr)
            extras = {"extras_error": repr(exc)}
        # the DRUL row of the integer roofline (C2's kernel), same probe peak
        try:
            d_ipe, d_src = instr_per_step("drul")
            c2 = extras["c2_drul"]
            d_ach = d_ipe * c2["env_steps_per_sec"] / 1e12
            extras["roofline_drul"] = {"kernel": "play3_kernel<DRUL> (C2: 2^20 envs)", "bound": "int_issue", "achieved": d_ach,
                                       "peak": int_peak, "unit": "Tinstr/s", "frac": d_ach / int_peak,
                                       "instr_per_env_step": d_ipe, "instr_source": d_src,
                                       "traffic": counts.get("drul", {}).get("dram_bytes_per_launch")}
        except Exception as exc:  # noqa: BLE001
            extras["roofline_drul"] = {"error": repr(exc)}
        try:
            extras["c4_iteration"] = c4_iteration(E, N, torch, dev, measured_hbm_peak()[0])
        except Exception as exc:  # noqa: BLE001 -- an extra leg must not cost the bench line
            extras["c4_iteration"] = {"error": repr(exc)}

    cpu_baseline = None
    if rank == 0 and world == 1:
        n_sample = min(CPU_SAMPLE_ENVS, batch_global)
        rate, threads_used, reps, ref = oracle_play_rate(SEED, batch_global, n_sample, policy_id, 1, 10.0)
        cpu_baseline = {
            "value": rate, "unit": "env-steps/s", "cores": threads_used, "kind": "port",
            "sample": f"envs [0,{n_sample}) of the same {batch_global}-env batch (seed {SEED}), {reps} repetitions, "
                      "oracle C restatement with OpenMP on all host threads (Pgx/JAX not installable here)",
        }
        # the sample doubles as a second parity check of the benchmarked workload itself
        chk = E.play(policy_id, subs0, batch_global, 0, n_sample, mode, per_env=True)
        assert np.array_equal(chk["lengths"].cpu().numpy(), ref["lengths"]), "bench workload differs from the oracle"
        assert np.array_equal(E.boards_numpy(chk["final_boards"]), ref["final_boards"]), "bench workload differs from the oracle"
        cpu_baseline["parity_checked_envs"] = n_sample

    if rank == 0:
        line = {
            "metric": "env_steps_per_sec", "value": value, "unit": "env-steps/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * elapsed / args.steps, "higher_is_better": True,
            "scaling": args.scaling, "vs_baseline": None, "dtype": "u64 bitboard / u32 Threefry (integer)", "data": "synthetic",
            "config": workload_config(args, world), "clocks": clocks, "e2e": e2e, "gpu_launches": gpu_launches,
            "roofline": roofline, "cpu_baseline": cpu_baseline, "parity": parity,
            "env_steps_per_step": total_env_steps / args.steps, "mean_episode_length": total_env_steps / args.steps / batch_global,
            "weak_scaling": other,
        }
        line.update(extras)
        sys.stdout.flush()
        os.write(json_fd, (json.dumps(line) + "\n").encode())
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def secondary_measurements(E, N, torch, dev, flush_buf) -> dict:
    """HBM-bound kernels of the path (rollout write / observation / GAE) and the PPO-rollout step."""
    hbm_peak, peak_src = measured_hbm_peak()

    def timed(fn, reps=5):
        fn()
        torch.cuda.synchronize()
        ts = []
        for _ in range(reps):
            flush_buf.fill_(3)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            torch.cuda.synchronize()
            ts.append(a.elapsed_time(b) * 1e-3)
        return statistics.mean(ts)

    rows = []
    # dram bytes per launch of the same rows, from the committed ncu --set full capture (tools/profile_hbm.py)
    try:
        traffic = json.loads((ROOT / "profiles" / "hbm_traffic.json").read_text())["rows"]
    except Exception:  # noqa: BLE001 -- the capture is evidence, not a dependency
        traffic = {}

    def add(name, bytes_per_launch, seconds, note):
        gbs = bytes_per_launch / seconds / 1e9
        rows.append({"kernel": name, "bound": "hbm", "achieved": gbs, "peak": hbm_peak, "unit": "GB/s",
                     "frac": gbs / hbm_peak, "traffic": traffic.get(name, {}).get("traffic"),
                     "algorithmic_bytes": bytes_per_launch, "us": seconds * 1e6, "note": note})

    # observation expansion: C3-sized rollout record (65536 envs x 16 steps of boards -> float32 one-hot)
    n_b = 1 << 20
    boards = torch.randint(0, 1 << 62, (n_b,), dtype=torch.int64, device=dev)
    out_f32 = torch.empty((n_b, 16, 31), dtype=torch.float32, device=dev)
    t = timed(lambda: N.call("g2048_expand_obs", N.ptr(boards), n_b, N.OBS_F32, N.ptr(out_f32), 0, 0, N.stream_ptr()))
    add("expand_obs_tma_kernel<float>", n_b * (8 + 1984), t, "2^20 boards -> (n,16,31) f32; 8 B read + 1984 B written per board; bulk-copy (UBLKCP) stores")
    del out_f32

    # minibatch gather (SURVEY 8f rank 1): 65536 random samples of a 2^22-step packed buffer -> float32 observations etc.
    n_buf, m = 1 << 22, 1 << 16
    packed = dict(boards=torch.randint(0, 1 << 62, (n_buf,), dtype=torch.int64, device=dev),
                  meta=torch.randint(0, 127, (n_buf,), dtype=torch.uint8, device=dev),
                  log_probs=torch.rand(n_buf, device=dev), values=torch.rand(n_buf, device=dev))
    g_adv, g_ret = torch.rand(n_buf, device=dev), torch.rand(n_buf, device=dev)
    idx = torch.randperm(n_buf, device=dev)[:m].contiguous()
    mb_out = E.minibatch_buffers(m, dev)
    # sample records: every field of a sample in one 32-byte sector (g2048_pack_samples, once per iteration)
    packed["rewards"] = g_adv
    mom_p = torch.tensor([n_buf, 0.5 * n_buf, 0.34 * n_buf, 0.5 * n_buf, 0.34 * n_buf, 0.0], dtype=torch.float64, device=dev)
    records = torch.empty((n_buf, 4), dtype=torch.int64, device=dev)
    t = timed(lambda: E.pack_samples(packed, g_adv, g_ret, mom_p, out=records))
    add("pack_samples_kernel", n_buf * (25 + 32), t, "2^22 steps: 25 B read (board, meta, reward, log-prob, value, advantage, return) + one 32 B sample record written per step, normalisation applied on the way")
    per_sample = 8 + 32 + 1984 + 8 + 4 + 16
    t = timed(lambda: E.gather_samples(idx, records, out=mb_out))
    add("gather_samples (gather_samples_tile_kernel<float>)", m * per_sample, t,
        "65536 random samples: 8 B index + ONE 32 B record read + 2012 B written per sample; one launch into reused output tensors; 134 MB in all, a launch-bound size")
    t = timed(lambda: E.gather_minibatch(idx, packed, g_adv, g_ret, out=mb_out))
    add("gather_minibatch (round 1: one source array per field)", m * (8 + 8 + 1 + 16 + 1984 + 8 + 4 + 16), t,
        "the same minibatch gathered from the six flat arrays (one sector per array and sample)")
    del mb_out
    # the same at a size that is not launch-bound (2^19 samples, 1.07 GB): what the kernel does once it is busy
    m_big = 1 << 19
    idx_big = torch.randint(0, n_buf, (m_big,), device=dev)
    mb_big = E.minibatch_buffers(m_big, dev)
    t = timed(lambda: E.gather_samples(idx_big, records, out=mb_big))
    add("gather_samples, 2^19 samples", m_big * per_sample, t, "same kernel, 8 x the samples: 1.07 GB written")
    del mb_big, idx_big, records
    del packed, g_adv, g_ret, idx

    # packed boards -> input embedding (SURVEY 8f rank 1): 2^18 boards, d_model 256 (configs/model/transformer_combined.yaml)
    n_e, d_model = 1 << 18, 256
    e_boards = boards[:n_e].contiguous()
    for dt, item in ((torch.float32, 4), (torch.bfloat16, 2)):
        table = torch.randn(31, d_model, device=dev).to(dt)
        emb = torch.empty((n_e, 16, d_model), dtype=dt, device=dev)
        name = str(dt).split(".")[-1]
        t = timed(lambda: E.embed_boards(e_boards, table, out=emb))
        add(f"embed_boards ({name})", n_e * (8 + 16 * d_model * item), t,
            f"2^18 boards -> (n,16,256) {name}: the Linear(31,256) of the one-hot observation as a row gather; write-only traffic")
        t = timed(lambda: E.embed_boards_grad(e_boards, emb))
        add(f"embed_grad_partial_kernel + reduce ({name})", n_e * (8 + 16 * d_model * item), t,
            "table gradient of the same; read-only traffic, deterministic two-kernel reduction")
        del emb
    del boards, e_boards

    # GAE on a flat buffer: C4-sized (2^26 steps), episodes ~300 steps
    n_g = 1 << 26
    r = torch.rand(n_g, device=dev)
    v = torch.rand(n_g, device=dev)
    d = (torch.rand(n_g, device=dev) < 1 / 300).to(torch.uint8)
    adv = torch.empty(n_g, dtype=torch.float32, device=dev)
    ret = torch.empty(n_g, dtype=torch.float32, device=dev)
    scratch = torch.zeros(int(N.lib.g2048_gae_flat_scratch_bytes(n_g)), dtype=torch.uint8, device=dev)
    mom = torch.zeros(6, dtype=torch.float64, device=dev)

    def gae():
        scratch.zero_()
        N.call("g2048_gae_flat", N.ptr(r), N.ptr(v), N.ptr(d), n_g, 0.99, 0.95, N.ptr(adv), N.ptr(ret), N.ptr(scratch),
               N.ptr(mom), N.stream_ptr())

    t = timed(gae)
    add("gae_flat4_kernel (pipelined)", n_g * 17, t, "2^26 steps, done rate 1/300 (episodes ~300 steps); 9 B read + 8 B written per step (SURVEY 8d); includes zeroing the scratch; walks hidden behind the neighbouring tiles' traffic, see DESIGN.md")
    scan_scratch = torch.zeros(int(N.lib.g2048_gae_scan_scratch_bytes(n_g)), dtype=torch.uint8, device=dev)

    def gae_scan():
        N.call("g2048_gae_flat_scan", N.ptr(r), N.ptr(v), N.ptr(d), n_g, 0.99, 0.95, N.ptr(adv), N.ptr(ret), N.ptr(scan_scratch),
               N.ptr(mom), N.stream_ptr())

    t = timed(gae_scan)
    add("gae_scan_kernel (opt-in: re-associated reverse scan, 1e-5 relative)", n_g * 17, t,
        "same buffer and bytes as gae_flat4_kernel above; warp-shuffle affine scan over 2 048-step tiles, one contiguous range of tiles per persistent CTA "
        "(north_star's own design); within 1e-5 relative of the reference loop instead of bit-identical; two launches (scan + range fix-up)")
    t = timed(lambda: N.call("g2048_normalize", N.ptr(adv), n_g, N.ptr(mom), 1, N.stream_ptr()))
    add("normalize_kernel", n_g * 8, t, "2^26 steps in place; 4 B read + 4 B written per step")
    # the same buffer size with the episode lengths of real play instead of a constant done rate (whose geometric
    # lengths have a long tail: the longest of a tile's ~27 episodes is ~4 x the mean, and a tile's walk lasts as
    # long as its longest episode): lengths of 2^18 DRUL games (C2's policy, mean ~207 steps), tiled to 2^26 steps
    try:
        key_g = E.words_tensor([0, 2048], dev)
        subs_g = E.chain_advance(key_g, E.RNG_PARTITIONABLE, 1 + 2 * 2048)
        lens = E.play(N.POLICY_DRUL, subs_g, 1 << 18, 0, 1 << 18, E.RNG_PARTITIONABLE)["lengths"].to(torch.int64)
        ends = torch.cumsum(lens, 0) - 1
        period = int(ends[-1].item()) + 1
        reps_g = (n_g + period - 1) // period
        d_real = torch.zeros(reps_g * period, dtype=torch.uint8, device=dev)
        d_real.view(reps_g, period)[:, ends] = 1
        d_real = d_real[:n_g].contiguous()

        def gae_real():
            scratch.zero_()
            N.call("g2048_gae_flat", N.ptr(r), N.ptr(v), N.ptr(d_real), n_g, 0.99, 0.95, N.ptr(adv), N.ptr(ret), N.ptr(scratch),
                   N.ptr(mom), N.stream_ptr())

        t = timed(gae_real)
        add("gae_flat4_kernel, episode lengths of real play", n_g * 17, t,
            f"2^26 steps; episode lengths of 2^18 DRUL games (mean {float(lens.float().mean()):.0f}, longest {int(lens.max())} steps) "
            "repeated; same kernel and bytes as the row above, which draws dones at a constant rate (geometric lengths)")
        del d_real, lens, ends
    except Exception as exc:  # noqa: BLE001 -- an extra row must not cost the bench line
        rows.append({"kernel": "gae_flat4_kernel, episode lengths of real play", "error": repr(exc)})
    del r, v, d, adv, ret

    # GAE on time-major records: C3 (128 steps x 65536 envs)
    t_steps, b = 128, 1 << 16
    rr = torch.rand((t_steps, b), device=dev)
    vv = torch.rand((t_steps, b), device=dev)
    mm = ((torch.rand((t_steps, b), device=dev) < 1 / 300).to(torch.uint8) << 6)
    adv2 = torch.empty((t_steps, b), dtype=torch.float32, device=dev)
    ret2 = torch.empty((t_steps, b), dtype=torch.float32, device=dev)
    t = timed(lambda: N.call("g2048_gae_time_major", N.ptr(rr), N.ptr(vv), N.ptr(mm), t_steps, b, None, 0.99, 0.95,
                             N.ptr(adv2), N.ptr(ret2), N.ptr(mom), N.stream_ptr()))
    add("gae_time_major_kernel", t_steps * b * 17, t, "C3: 128 x 65536 steps; launch-bound size (143 MB), also reported in us")
    del rr, vv, mm, adv2, ret2
    b4 = 4 * b
    rr = torch.rand((t_steps, b4), device=dev)
    vv = torch.rand((t_steps, b4), device=dev)
    mm = ((torch.rand((t_steps, b4), device=dev) < 1 / 300).to(torch.uint8) << 6)
    adv2 = torch.empty((t_steps, b4), dtype=torch.float32, device=dev)
    ret2 = torch.empty((t_steps, b4), dtype=torch.float32, device=dev)
    t = timed(lambda: N.call("g2048_gae_time_major", N.ptr(rr), N.ptr(vv), N.ptr(mm), t_steps, b4, None, 0.99, 0.95,
                             N.ptr(adv2), N.ptr(ret2), N.ptr(mom), N.stream_ptr()))
    add("gae_time_major_kernel, 4 x C3", t_steps * b4 * 17, t, "128 x 262144 steps (570 MB): the same kernel once the launch is amortised")

    # PPO rollout step (C3): synthetic logits stand in for the policy network, which is outside the product path
    mode = E.RNG_PARTITIONABLE
    key = E.words_tensor([0, 3], dev)
    subs = E.chain_advance(key, mode, 1 + 2 * t_steps)
    pb, ps = E.env_init(subs[0], b, 0, b, mode)
    logits = torch.randn((b, 4), device=dev)
    values = torch.randn(b, device=dev)
    rec_b = torch.empty((t_steps, b), dtype=torch.int64, device=dev)
    rec_m = torch.empty((t_steps, b), dtype=torch.uint8, device=dev)
    rec_r, rec_l, rec_v = (torch.empty((t_steps, b), dtype=torch.float32, device=dev) for _ in range(3))
    obs = torch.empty((b, 16, 31), dtype=torch.float32, device=dev)

    def ppo_rollout():
        # one launch per step: sample + env.step + auto-reset + record + the observation of the next forward pass
        N.call("g2048_expand_obs", N.ptr(pb), b, N.OBS_F32, N.ptr(obs), 0, 0, N.stream_ptr())
        for k in range(t_steps):
            E.policy_step_obs(pb, ps, logits, values, True, True, True, subs[1 + 2 * k:], None, b, 0, mode, obs,
                              rec_b[k], rec_m[k], rec_r[k], rec_l[k], rec_v[k])
        N.call("g2048_gae_time_major", N.ptr(rec_r), N.ptr(rec_v), N.ptr(rec_m), t_steps, b, None, 0.99, 0.95,
               N.ptr(adv2), N.ptr(ret2), N.ptr(mom), N.stream_ptr())

    def ppo_rollout_two_launches():  # round 1's form: expand_obs + policy_step per step
        for k in range(t_steps):
            N.call("g2048_expand_obs", N.ptr(pb), b, N.OBS_F32, N.ptr(obs), 0, 0, N.stream_ptr())
            E.policy_step(pb, ps, logits, values, True, True, True, subs[1 + 2 * k], subs[2 + 2 * k], b, 0, mode,
                          rec_b[k], rec_m[k], rec_r[k], rec_l[k], rec_v[k])
        N.call("g2048_gae_time_major", N.ptr(rec_r), N.ptr(rec_v), N.ptr(rec_m), t_steps, b, None, 0.99, 0.95,
               N.ptr(adv2), N.ptr(ret2), N.ptr(mom), N.stream_ptr())

    t = timed(ppo_rollout, reps=3)
    t_two = timed(ppo_rollout_two_launches, reps=3)
    # the same loop writing bfloat16 observations (one-hot values are exact in bf16; what TorchActionFunction(obs_dtype=
    # torch.bfloat16) feeds a network that runs under bf16 autocast anyway): half the bytes per step
    obs16 = torch.empty((b, 16, 31), dtype=torch.bfloat16, device=dev)

    def ppo_rollout_bf16():
        N.call("g2048_expand_obs", N.ptr(pb), b, N.OBS_BF16, N.ptr(obs16), 0, 0, N.stream_ptr())
        for k in range(t_steps):
            E.policy_step_obs(pb, ps, logits, values, True, True, True, subs[1 + 2 * k:], None, b, 0, mode, obs16,
                              rec_b[k], rec_m[k], rec_r[k], rec_l[k], rec_v[k])
        N.call("g2048_gae_time_major", N.ptr(rec_r), N.ptr(rec_v), N.ptr(rec_m), t_steps, b, None, 0.99, 0.95,
               N.ptr(adv2), N.ptr(ret2), N.ptr(mom), N.stream_ptr())

    t_bf16 = timed(ppo_rollout_bf16, reps=3)
    t_bf16_graph = None
    try:
        side16 = torch.cuda.Stream()
        side16.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side16):
            ppo_rollout_bf16()
        torch.cuda.current_stream().wait_stream(side16)
        torch.cuda.synchronize()
        graph16 = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph16):
            ppo_rollout_bf16()
        t_bf16_graph = timed(graph16.replay, reps=3)
        del graph16
    except Exception as exc:  # noqa: BLE001
        t_bf16_graph = f"unavailable: {exc!r}"

    # the same 257 launches replayed as ONE CUDA graph: what the kernels cost once the Python / ctypes launch overhead
    # (two launches per step from the interpreter) is out of the way -- how FixedHorizonRunner(cuda_graph=True) runs them
    t_graph = None
    try:
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            ppo_rollout()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            ppo_rollout()
        t_graph = timed(graph.replay, reps=3)
        del graph
    except Exception as exc:  # noqa: BLE001 -- an extra number must not cost the bench line
        t_graph = f"unavailable: {exc!r}"

    # the policy network's forward pass at the same batch (PyTorch / cuBLAS, outside the product path): a stand-in
    # with the reference's default layer shapes (configs/model/transformer_combined.yaml: d_model 256, 8 heads,
    # 4 layers, ff 1024, hidden 512, CLS reduction, 17 tokens), bf16 autocast as in configs/trainer/default.yaml
    fwd_ms = None
    try:
        nn = torch.nn

        class PolicyStandIn(nn.Module):
            def __init__(self):
                super().__init__()
                self.embed = nn.Linear(31, 256, bias=False)
                self.cls = nn.Parameter(torch.zeros(1, 1, 256))
                layer = nn.TransformerEncoderLayer(256, 8, 1024, dropout=0.0, batch_first=True, norm_first=True)
                self.encoder = nn.TransformerEncoder(layer, 4, enable_nested_tensor=False)
                self.actor = nn.Sequential(nn.Linear(256, 512), nn.ReLU(), nn.Linear(512, 512), nn.ReLU(), nn.Linear(512, 4, bias=False))
                self.critic = nn.Sequential(nn.Linear(256, 512), nn.ReLU(), nn.Linear(512, 512), nn.ReLU(), nn.Linear(512, 1, bias=False))

            def forward(self, x):
                h = self.embed(x)
                h = torch.cat([self.cls.expand(h.shape[0], -1, -1), h], dim=1)
                h = self.encoder(h)[:, 0]
                return self.actor(h), self.critic(h)

        net = PolicyStandIn().to(dev).eval()

        def forward_all():  # chunks of 8192 envs keep the attention kernels inside their supported batch range
            for c in range(0, b, 8192):
                net(obs[c:c + 8192])

        with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):
            fwd = timed(forward_all, reps=3)
        fwd_ms = fwd * 1e3
        del net
    except Exception as exc:  # the stand-in is context, not part of the product
        fwd_ms = f"unavailable: {exc}"
    ppo = {
        "config": "C3: 65536 envs x 128 steps, auto-reset, masked categorical sampling from synthetic logits "
                  "(policy network = PyTorch/cuBLAS, outside the product path and not timed)",
        "env_steps_per_sec": t_steps * b / t, "ms_per_rollout": t * 1e3,
        "per_step_us": t * 1e6 / t_steps, "launches_per_rollout": t_steps + 2,
        "per_step_us_two_launches_per_step": t_two * 1e6 / t_steps,
        "bf16_observations": {"per_step_us": t_bf16 * 1e6 / t_steps,
                              "per_step_us_graph_replay": (t_bf16_graph * 1e6 / t_steps if isinstance(t_bf16_graph, float) else t_bf16_graph),
                              "hbm_floor_us_per_step": (b * (992 + 21 + 20 + 18)) / measured_hbm_peak()[0] / 1e3,
                              "note": "the same fused step writing bfloat16 observations (exact for one-hot values): half the bytes"},
        "hbm_floor_us_per_step": (b * (1984 + 21 + 20 + 18)) / measured_hbm_peak()[0] / 1e3,
        "algorithmic_bytes_per_step": b * (1984 + 21 + 20 + 18),
        "traffic_per_step": traffic.get("c3: policy_step_obs_kernel<float>", {}).get("traffic"),
        "graph_replay": ({"ms_per_rollout": t_graph * 1e3, "per_step_us": t_graph * 1e6 / t_steps,
                          "env_steps_per_sec": t_steps * b / t_graph,
                          "note": "the same launches captured once and replayed as a CUDA graph (no interpreter between them)"}
                         if isinstance(t_graph, float) else t_graph),
        "policy_forward_ms_per_step": fwd_ms,
        "policy_forward_note": "same-shaped PyTorch Transformer (3.96 M parameters, bf16 autocast, 65536 x 17 tokens), for scale only",
        "kernels": "per step ONE launch: policy_step_obs (mask, sample, log-prob, env step, auto-reset, record write, and the float32 "
                   "observation of the next forward pass written from registers); then gae_time_major",
    }
    # C2: DRUL corner policy, 2^20 envs to termination, score / max-tile statistics reduced on the device
    import g2048

    n2 = 1 << 20
    key2 = E.words_tensor([0, 0], dev)
    subs2 = E.chain_advance(key2, mode, 1 + 2 * 2048)
    st2 = {}
    t = timed(lambda: st2.update(stats=E.play(E.POLICY_DRUL, subs2, n2, 0, n2, mode, per_env=False)["stats"]), reps=3)
    s2 = E.play_stats_dict(st2["stats"])
    c2 = {"config": "C2: act_drul, 2^20 envs to termination, seed 0", "env_steps_per_sec": s2["env_steps"] / t,
          "ms": t * 1e3, "mean_episode_length": s2["env_steps"] / n2, "mean_score": s2["score_sum"] / n2,
          "mean_max_tile": s2["tile_sum"] / n2, "max_tile_hist": {str(k): v for k, v in s2["max_tile_hist"].items()}}

    # C1 through the reference-format API: BatchRunner(0, act_randomly).run_actions_batch(1024), numpy arrays out
    # (observations (B,T,4,4,31) bool etc., i.e. including the one-hot materialisation and the D2H copies)
    runner = g2048.BatchRunner(init_seed=0, act_fn=g2048.act_randomly)
    runner.run_actions_batch(1024)
    runner = g2048.BatchRunner(init_seed=0, act_fn=g2048.act_randomly)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = runner.run_actions_batch(1024)
    dt = time.perf_counter() - t0
    first_done = out[6].argmax(axis=1) + 1
    c1 = {"config": "C1: BatchRunner(0, act_randomly).run_actions_batch(1024), reference-format numpy outputs",
          "seconds": dt, "loop_steps": int(out[0].shape[1]), "env_steps": int(first_done.sum()),
          "env_steps_per_sec": float(first_done.sum() / dt), "output_bytes": int(sum(a.nbytes for a in out if a is not None))}
    pin_runner = lambda: g2048.BatchRunner(init_seed=0, act_fn=g2048.act_randomly, pinned_outputs=True)  # noqa: E731
    keep = pin_runner().run_actions_batch(1024)
    del keep  # the page-locked blocks are in the host allocator's cache now, as in any loop over batches
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out_p = pin_runner().run_actions_batch(1024)
    dt_p = time.perf_counter() - t0
    c1["pinned_outputs"] = {"seconds": dt_p, "env_steps_per_sec": float(first_done.sum() / dt_p),
                            "identical": bool(all((a is None and b_ is None) or np.array_equal(a, b_) for a, b_ in zip(out, out_p))),
                            "note": "BatchRunner(pinned_outputs=True): the returned arrays are page-locked memory written by one transfer each"}
    del out_p
    # the other reference-API calls at C1's size: run_rollout_batch (list of States, built from the records of a chunked
    # run) and run_actions_max_tile (persistent play kernel + replay of the longest envs for the reference's quirk)
    from g2048.runs.run_actions_max_tile import run_actions_max_tile

    def wall(fn):
        fn()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        res = fn()
        torch.cuda.synchronize()
        return res, time.perf_counter() - t0

    states, t_states = wall(lambda: g2048.BatchRunner(init_seed=0, act_fn=g2048.act_randomly).run_rollout_batch(1024))
    stats_q, t_mt = wall(lambda: run_actions_max_tile(0, 1024, 4096, g2048.act_randomly))
    _, t_mt_exact = wall(lambda: run_actions_max_tile(0, 1024, 4096, g2048.act_randomly, exact_reference_quirk=False))
    c1["run_rollout_batch_1024"] = {"seconds": t_states, "states": len(states), "env_steps_per_sec": float(first_done.sum() / t_states)}
    c1["run_actions_max_tile_4096_envs_in_batches_of_1024"] = {
        "seconds": t_mt, "seconds_without_the_reference_quirk": t_mt_exact, "mean_max_tile": float(torch.as_tensor(stats_q.mean).reshape(-1)[0])}
    return {"roofline_hbm": rows, "hbm_peak_source": peak_src, "ppo_rollout": ppo, "c2_drul": c2, "c1_reference_api": c1}


def c4_iteration(E, N, torch, dev, hbm_peak) -> dict:
    """BASELINE.json configs[3]: the data path of one full PPO iteration at 262 144 envs, phase by phase (the learner's
    GEMMs are PyTorch/cuBLAS and outside the product path; a random policy stands in for the network so that the
    rollout is the product's own kernels): recorded rollout to termination + rollout-buffer write, GAE + normalisation,
    4 epochs of 2048-sample minibatches (300 000 samples per epoch, configs/trainer/default.yaml), and the bit-exact
    board check on a 4 096-env sample."""
    import numpy as np

    import g2048
    from oracle import c_oracle as CO

    n_envs, epochs, minibatch, max_samples = 1 << 18, 4, 2048, 300_000
    mode = E.RNG_PARTITIONABLE

    def wall(fn):
        # from an idle device to the call's results being complete on the caller's stream.  (Not a device-wide
        # synchronisation at the end: the runner's key chain tops itself up on a side stream after every batch -- one
        # thread, ~0.1 ms, next to whatever the caller launches next -- and that is not part of this call's latency.)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = fn()
        torch.cuda.current_stream().synchronize()
        return out, time.perf_counter() - t0

    def dev_time(fn, reps=3):
        fn()
        torch.cuda.synchronize()
        ts = []
        for _ in range(reps):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            torch.cuda.synchronize()
            ts.append(a.elapsed_time(b) * 1e-3)
        return min(ts)

    report = {"config": f"C4: {n_envs} envs to termination (random policy records), GAE, {epochs} epochs x {max_samples} samples in "
                        f"minibatches of {minibatch}"}
    # -- rollout + store: the recording play kernel writes the buffer's own layout (run_flat_batch -> store_flat) --------
    runner = g2048.BatchRunner(init_seed=4, act_fn=g2048.act_randomly)
    for _ in range(3):  # warm-up at full size: allocator, table build, arena sizing hint, key chain a block ahead, torch's lazily loaded kernels
        runner.run_flat_batch(n_envs)
    key_before = runner.key  # the chain key the timed batch starts from (for the oracle replay below)
    buf = g2048.RolloutBuffer(31, 16, 4)
    flat, t_flat = wall(lambda: runner.run_flat_batch(n_envs))
    _, t_store = wall(lambda: buf.store_flat(flat))
    steps = flat.env_steps
    # the two kernels alone, device-timed
    subs = E.chain_advance(E.words_tensor(key_before, dev), mode, 1 + 2 * 2048)
    rec = {}
    t_rec = dev_time(lambda: rec.update(E.play_record(E.POLICY_RANDOM, subs, n_envs, 0, n_envs, mode, mean_steps=steps // n_envs + 1)))
    offsets = E.exclusive_scan(rec["lengths"])
    t_cmp = dev_time(lambda: E.play_record_compact(rec, offsets, steps))
    t_plain = dev_time(lambda: E.play(E.POLICY_RANDOM, subs, n_envs, 0, n_envs, mode, per_env=True))
    cmp_bytes = steps * (9 + 21)
    try:  # dram bytes of one launch from the committed ncu capture (tools/profile_hbm.py)
        captured = json.loads((ROOT / "profiles" / "hbm_traffic.json").read_text())["rows"]
    except Exception:  # noqa: BLE001 -- evidence, not a dependency
        captured = {}
    report["rollout_and_store"] = {
        "seconds": t_flat + t_store, "env_steps": steps, "env_steps_per_sec": steps / (t_flat + t_store),
        "api": "BatchRunner.run_flat_batch + RolloutBuffer.store_flat (wall clock; one host read-back of the statistics, the compaction is queued before it)",
        "play_record_kernel_ms": t_rec * 1e3, "play_record_env_steps_per_sec": steps / t_rec,
        "play_kernel_without_records_ms": t_plain * 1e3, "recording_overhead": t_rec / t_plain - 1.0,
        "compact_kernel_ms": t_cmp * 1e3,
        "compact_roofline": {"bound": "hbm", "achieved": cmp_bytes / t_cmp / 1e9, "peak": hbm_peak, "unit": "GB/s",
                             "frac": cmp_bytes / t_cmp / 1e9 / hbm_peak, "algorithmic_bytes": cmp_bytes,
                             "traffic": captured.get("c4: play_record_compact_kernel", {}).get("traffic"),
                             "note": "9 B read (board + meta) + 21 B written (board, meta, reward, log-prob, value) per kept step"},
        "arena_bytes": int(rec["arena_boards"].numel() * 9),
    }
    del rec
    # round 1's path for the same batch: lock-step recorder (every env stepped until the last one ends) + store_packed
    r1 = g2048.BatchRunner(init_seed=4, act_fn=g2048.act_randomly)
    for _ in range(3):  # the same three batches as the warm-up above, so the fourth one is the timed batch's twin
        r1.run_packed_batch(n_envs)
    ro, t_lock = wall(lambda: r1.run_packed_batch(n_envs))
    b1 = g2048.RolloutBuffer(31, 16, 4)
    _, t_store1 = wall(lambda: b1.store_packed(ro))
    p0, p1 = buf.get_packed(), b1.get_packed()
    report["lock_step_recorder_plus_store_packed"] = {
        "seconds": t_lock + t_store1, "env_steps_per_sec": steps / (t_lock + t_store1), "loop_steps": ro.t_steps,
        "live_fraction": steps / (ro.t_steps * n_envs),
        "flat_buffer_identical": bool(all(torch.equal(p0[k], p1[k]) for k in p0))}
    del ro, b1, p1, r1
    # -- GAE + normalisation + the epoch's subset ---------------------------------------------------------------------------
    packed = buf.get_packed()
    packed["values"].copy_(torch.randn_like(packed["values"]))  # stand-in critic outputs
    kw = dict(batch_size=minibatch, max_samples_per_epoch=max_samples, shuffle_on_reset=True, reuse_buffers=True)
    g2048.DevicePPOBatches(packed, 0.99, 0.95, **kw)
    batches, t_gae = wall(lambda: g2048.DevicePPOBatches(packed, 0.99, 0.95, **kw))
    report["gae_normalise"] = {"seconds": t_gae, "steps_per_sec": steps / t_gae,
                               "algorithmic_bytes_per_step": 17 + 25 + 32,
                               "achieved_gbs": steps * (17 + 25 + 32) / t_gae / 1e9, "frac_of_hbm": steps * (17 + 25 + 32) / t_gae / 1e9 / hbm_peak,
                               "note": "g2048_gae_flat (9 B read + 8 B written per step) + g2048_pack_samples (25 B read, 32 B sample "
                                       "record written, normalisation applied on the way) + the first epoch's g2048_random_subset; wall clock"}

    def run_epochs(source):
        k = 0
        for _ in range(epochs):
            source.reset_epoch()
            for b in source:
                k += b["actions"].shape[0]
        return k

    run_epochs(batches)
    n_samples, t_feed_each = wall(lambda: run_epochs(batches))
    batches_e = g2048.DevicePPOBatches(packed, 0.99, 0.95, epoch_prefetch=True, **kw)
    run_epochs(batches_e)
    _, t_feed = wall(lambda: run_epochs(batches_e))
    per_sample = 8 + 32 + 1984 + 8 + 4 + 16
    report["minibatches"] = {"seconds": t_feed, "samples": n_samples, "samples_per_sec": n_samples / t_feed,
                             "achieved_gbs": n_samples * per_sample / t_feed / 1e9, "frac_of_hbm": n_samples * per_sample / t_feed / 1e9 / hbm_peak,
                             "seconds_one_launch_per_minibatch": t_feed_each,
                             "note": "float32 observations; per epoch one g2048_random_subset + ONE g2048_gather_samples launch for all "
                                     "of the epoch's samples (DevicePPOBatches(epoch_prefetch=True)), minibatches are views; "
                                     "seconds_one_launch_per_minibatch = the same with a gather launch per minibatch"}
    batches_b = g2048.DevicePPOBatches(packed, 0.99, 0.95, obs_dtype=None, epoch_prefetch=True, **kw)
    run_epochs(batches_b)
    _, t_feed_b = wall(lambda: run_epochs(batches_b))
    report["minibatches_boards"] = {"seconds": t_feed_b, "note": "bitboards instead of observations (embedding as a row gather)"}
    # -- bit-exact board check on a 4 096-env sample: replay the recorded actions through the oracle's step, with the
    #    oracle's own spawn draws from the same keys; every recorded pre-step board, reward and done flag must agree
    sample, t_chk = 4096, 200
    _, o_subs = CO.chain(np.asarray(key_before, np.uint32), 1, 1 + 2 * t_chk)
    boards, masks = CO.env_init(CO.split(o_subs[0], n_envs, 1)[:sample], 1)
    done = np.zeros(sample, np.uint8)
    offs = flat.offsets[: sample + 1].cpu().numpy()
    lens = flat.lengths[:sample].cpu().numpy().astype(np.int64)
    hi = int(offs[-1])
    f_boards = E.boards_numpy(flat.boards[:hi])
    f_meta = flat.meta[:hi].cpu().numpy()
    f_rew = flat.rewards[:hi].cpu().numpy()
    ok = True
    for t in range(t_chk):
        live = lens > t
        pos = offs[:-1][live] + t
        ok &= bool(np.array_equal(f_boards[pos], boards[live]))
        actions = np.zeros(sample, np.int32)
        actions[live] = f_meta[pos] & 3
        step_keys = CO.split(o_subs[2 + 2 * t], n_envs, 1)[:sample]
        boards, masks, done, rew = CO.env_step(boards, masks, done, actions, step_keys, 1)
        ok &= bool(np.array_equal(rew[live], f_rew[pos]) and np.array_equal(done[live], (f_meta[pos] >> 6) & 1))
        ok &= bool(done[~live].all())  # an env whose record has ended is finished in the oracle too
    report["bit_exact_board_check"] = {"envs": sample, "steps": t_chk, "identical": bool(ok),
                                       "what": "pre-step boards, rewards and done flags of the flat buffer vs the oracle's env.step "
                                               "replayed with the recorded actions and its own spawn draws"}
    total = t_flat + t_store + t_gae + t_feed
    report["product_path_seconds"] = total
    report["share"] = {k: round(v / total, 3) for k, v in (("rollout_and_store", t_flat + t_store), ("gae", t_gae), ("minibatches", t_feed))}
    return report


if __name__ == "__main__":
    main()
