"""Monte-Carlo equity with ranges to a target precision (get_equity_ranges_batch_adaptive) against the fixed-trial range call,
one JSON line on stdout.

    python tools/adaptive_ranges_bench.py [--reps 5] [--out file.json]

Workloads:
    ranges   bench.py's: 4,096 six-player flop queries, opponents in the top 30 %, reference dealer; max 1,000 and 10,000
    classes  the 1,326 hero hands, heads-up preflop against a top-20 % range, reference dealer; max 100,000
each at three stderr values, the largest 0.5 / sqrt(max_trials) (the worst-case standard error of the fixed count), and with
both samplers (the pair-list sampler, and the generic kernel that counts passes).  Per (workload, max, stderr, sampler): the
rounds (checkpoints from min_trials = 256), the trials run as a fraction of Q x max_trials, the queries that ran to max, and
the median over `reps` calls of the adaptive call's time (CUDA events around the unvalidated Python call on the stream)
against the fixed call at max_trials with the same sampler.  The card's name, power limit and maximum SM clock are read in
the same run."""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402
import neuron_poker_b200 as npk  # noqa: E402
from adaptive_equity_bench import gpu_info, timed  # noqa: E402
from neuron_poker_b200.equity import adaptive_checkpoints  # noqa: E402

MIN_TRIALS = 256


def class_queries(dev):
    """The 1,326 two-card hero hands, heads-up preflop."""
    hole = np.array([(a, b) for b in range(52) for a in range(b)], dtype=np.uint8)
    board = np.full((len(hole), 5), 0xFF, dtype=np.uint8)
    npl = np.full(len(hole), 2, dtype=np.uint8)
    return [torch.as_tensor(x).to(dev) for x in (hole, board, npl)]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out")
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    res = {"gpu": gpu_info(), "min_trials": MIN_TRIALS, "deal_mode": "reference", "workloads": []}
    ranges_q = [torch.as_tensor(x).to(dev) for x in bench.make_queries(bench.workload("ranges"), 1, 0)]
    for name, q, opp, max_trials in (("ranges", ranges_q, 0.3, 1000), ("ranges", ranges_q, 0.3, 10000),
                                     ("classes", class_queries(dev), 0.2, 100000)):
        Q = q[0].shape[0]
        for sampler in ("pair_list", "generic"):
            kw = dict(opponent_range=opp, seed_value=1, deal_mode="reference", validate=False, passes=sampler == "generic")
            fixed_ms, _ = timed(lambda: npk.get_equity_ranges_batch(*q, max_trials, **kw), args.reps)
            row = {"workload": name, "queries": Q, "players": int(q[2][0]), "opponent_range": opp, "max_trials": max_trials,
                   "sampler": sampler, "rounds": len(adaptive_checkpoints(MIN_TRIALS, max_trials)),
                   "fixed_ms": round(fixed_ms, 4), "runs": []}
            worst = 0.5 / max_trials ** 0.5
            for stderr in (worst, worst / 2 ** 0.5, worst / 2):
                ms, out = timed(lambda: npk.get_equity_ranges_batch_adaptive(*q, max_trials, stderr, min_trials=MIN_TRIALS,
                                                                             **kw), args.reps)
                trials = out["trials"].cpu()
                stops = trials.unique().tolist()
                row["runs"].append({"stderr": stderr, "adaptive_ms": round(ms, 4), "time_vs_fixed": round(ms / fixed_ms, 4),
                                    "rounds_run": len(adaptive_checkpoints(MIN_TRIALS, max(stops))),
                                    "trials_fraction": round(float(trials.sum()) / (Q * max_trials), 4),
                                    "queries_at_max": int((trials == max_trials).sum())})
            res["workloads"].append(row)
            print(json.dumps(row), file=sys.stderr)
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
