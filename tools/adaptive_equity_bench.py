"""Monte-Carlo equity to a target precision (get_equity_batch_adaptive) against the fixed-trial call, one JSON line on stdout.

    python tools/adaptive_equity_bench.py [--reps 7] [--out file.json]

Workloads (queries as bench.py makes them):
    cfg3  4,096 six-player flop queries, max 10,000 trials, uniform dealing
    cfg5  the queries of one step of 65,536 six-max self-play tables (after 100 warm-up steps), max 1,000, reference dealer
    cfg4  169 starting-hand classes, nine players preflop, max 1,000,000, uniform dealing
each at three stderr values, the largest 0.5 / sqrt(max_trials) (the worst-case standard error of the fixed count).
Per (workload, stderr): trials executed as a fraction of Q x max_trials, rounds (checkpoints from min_trials = 256), and the
median over `reps` calls of the adaptive call's time (CUDA events around the Python call on the stream) against the fixed
call at max_trials through the same all-shapes kernel (and, for the uniform-shape workloads, through the shape's own kernel,
bench.py's path).  The card's name, power limit and maximum SM clock are read in the same run."""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import bench  # noqa: E402
import neuron_poker_b200 as npk  # noqa: E402
from neuron_poker_b200.equity import adaptive_checkpoints  # noqa: E402


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power, clock = [x.strip() for x in q.split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def timed(fn, reps):
    fn()                                                  # warm-up (module load, allocator)
    ms = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = fn()
        e1.record()
        torch.cuda.synchronize()
        ms.append(e0.elapsed_time(e1))
    return statistics.median(ms), out


def selfplay_queries(dev):
    from neuron_poker_b200.holdem import EquityAgents, HoldemTables
    tb = HoldemTables(65536, n_players=6, seed=7, autoplay=[1] * 6, device=dev)
    agents = EquityAgents.equity_vs_random()
    for _ in range(100):
        tb.selfplay_step(agents, runs=1000, deal_mode="reference")
    return [t.clone() for t in tb.queries()[:3]]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--out")
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    res = {"gpu": gpu_info(), "min_trials": 256, "workloads": []}
    for name, deal, shape in (("cfg3", "uniform", (6, 3)), ("cfg5", "reference", None), ("cfg4", "uniform", (9, 0))):
        wl = bench.workload(name)
        max_trials = wl["trials"]
        if name == "cfg5":
            q = selfplay_queries(dev)
        else:
            q = [torch.as_tensor(x).to(dev) for x in bench.make_queries(wl, 1, 0)]
        Q = q[0].shape[0]
        reps = 3 if name == "cfg4" else args.reps
        fixed_ms, _ = timed(lambda: npk.get_equity_batch(*q, max_trials, seed_value=1, deal_mode=deal, validate=False), reps)
        row = {"workload": name, "queries": Q, "max_trials": max_trials, "deal_mode": deal,
               "rounds": len(adaptive_checkpoints(256, max_trials)), "fixed_ms": round(fixed_ms, 4), "runs": []}
        if shape is not None:
            ms, _ = timed(lambda: npk.get_equity_batch(*q, max_trials, seed_value=1, deal_mode=deal, uniform_shape=shape,
                                                       validate=False), reps)
            row["fixed_uniform_shape_ms"] = round(ms, 4)
        worst = 0.5 / max_trials ** 0.5
        for stderr in (worst, worst / 2 ** 0.5, worst / 2):
            ms, out = timed(lambda: npk.get_equity_batch_adaptive(*q, max_trials, stderr, seed_value=1, deal_mode=deal,
                                                                  validate=False), reps)
            trials = out["trials"].cpu()
            row["runs"].append({"stderr": stderr, "adaptive_ms": round(ms, 4), "time_vs_fixed": round(ms / fixed_ms, 4),
                                "trials_fraction": round(float(trials.sum()) / (Q * max_trials), 4),
                                "queries_at_max": int((trials == max_trials).sum()),
                                "queries_without_trials": int((trials == 0).sum())})
        res["workloads"].append(row)
        print(json.dumps(row), file=sys.stderr)
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
