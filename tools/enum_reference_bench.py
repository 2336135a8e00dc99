"""Exact enumeration under the reference's dealer against uniform dealing (enumerate_equity, deal_mode "reference" and
"uniform"), one JSON line on stdout.

    python tools/enum_reference_bench.py [--reps 5] [--preflop-reps 1] [--workloads river,turn,flop,river3,preflop]
                                         [--out profiles/enum_reference_bench.json]

Workloads (seed 0, distinct cards, uniform):
    river    4,096 heads-up river spots            fast path, 990 opponent hands per spot
    turn     4,096 heads-up turn spots             fast path, 46 completions x C(45,2)
    flop     4,096 heads-up flop spots             fast path, C(47,2) completions x C(45,2)
    preflop  the 169 starting-hand classes, heads-up, no board   generic walk, C(50,5) completions x C(45,2)
    river3   4,096 three-player river spots        ordered pairs of disjoint opponent hands
Per workload and mode: the median over `reps` calls (CUDA events around the call on device tensors, without validation, after
one warm-up call; the preflop calls are timed without a warm-up: one call takes minutes, and the kernel's module is loaded
by an earlier workload or by the uniform call), the (completion, hand) pairs
per second -- the pairs of the uniform enumeration in both modes, the work the kernel walks -- and the REFERENCE / UNIFORM
throughput ratio (uniform time / reference time).  The totals of both modes are checked against their closed forms.  The
card's name, power limit and maximum SM clock are read in the same run."""
import argparse
import json
import math
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import neuron_poker_b200 as npk  # noqa: E402
from adaptive_equity_bench import gpu_info  # noqa: E402

Q = 4096


def random_spots(known, players, dev, seed=0):
    rng = np.random.default_rng(seed)
    cards = np.stack([rng.permutation(52)[:2 + known] for _ in range(Q)]).astype(np.uint8)
    board = np.full((Q, 5), 0xFF, dtype=np.uint8)
    board[:, :known] = cards[:, 2:]
    return [torch.as_tensor(x).to(dev) for x in (cards[:, :2].copy(), board, np.full(Q, players, dtype=np.uint8))]


def class_spots(dev):
    """One hand of each of the 169 classes: suited hi/lo of spades, offsuit and pairs as a spade and a heart."""
    hole = []
    for hi in range(13):
        for lo in range(hi + 1):
            hole.append((4 * hi + 3, 4 * lo + 2))                 # offsuit (a pair when lo == hi)
            if lo < hi:
                hole.append((4 * hi + 3, 4 * lo + 3))             # suited
    hole = np.array(hole, dtype=np.uint8)
    n = len(hole)
    return [torch.as_tensor(x).to(dev) for x in (hole, np.full((n, 5), 0xFF, dtype=np.uint8), np.full(n, 2, dtype=np.uint8))]


def pairs_per_spot(known, players):
    """(completion, hand) pairs of the uniform enumeration, and the totals of both modes."""
    n, m = 50 - known, 5 - known
    if players == 3:
        return math.comb(n, 2) * math.comb(n - 2, 2), math.comb(n, 2) * math.comb(n - 2, 2), (n - 1) ** 2 * (n - 3) ** 2
    uniform = math.comb(n, m) * math.comb(n - m, 2)
    return uniform, uniform, (n - 1) ** 2 * math.comb(n - 3, m)


def timed(fn, reps, warmup):
    if warmup:
        fn()
    ms, out = [], None
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = fn()
        e1.record()
        torch.cuda.synchronize()
        ms.append(e0.elapsed_time(e1))
    return statistics.median(ms), ms, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--preflop-reps", type=int, default=1)
    ap.add_argument("--workloads", default="river,turn,flop,river3,preflop")
    ap.add_argument("--out")
    args = ap.parse_args()
    wanted = args.workloads.split(",")
    dev = torch.device("cuda", 0)
    res = {"tool": "enum_reference_bench", "gpu": gpu_info(), "sm_count": torch.cuda.get_device_properties(dev).multi_processor_count,
           "workloads": []}
    loads = [("river", lambda: random_spots(5, 2, dev), 5, 2), ("turn", lambda: random_spots(4, 2, dev), 4, 2),
             ("flop", lambda: random_spots(3, 2, dev), 3, 2), ("river3", lambda: random_spots(5, 3, dev), 5, 3),
             ("preflop", lambda: class_spots(dev), 0, 2)]
    for name, make, known, players in loads:
        if name not in wanted:
            continue
        q = make()
        spots = q[0].shape[0]
        pairs, uniform_total, reference_total = pairs_per_spot(known, players)
        row = {"workload": name, "spots": spots, "players": players, "known_board_cards": known,
               "pairs_per_spot": pairs, "pairs_per_call": pairs * spots}
        for mode, want in (("uniform", uniform_total), ("reference", reference_total)):
            reps = args.preflop_reps if name == "preflop" else args.reps
            med, all_ms, out = timed(lambda: npk.enumerate_equity(*q, deal_mode=mode), reps, warmup=name != "preflop")
            totals = (out[0] + out[1] + out[2]).cpu()
            assert bool((totals == want).all()), (name, mode, totals[:4], want)
            eq = ((out[0] + out[1]).double() / totals.double().to(dev)).mean().item()
            row[mode] = {"ms_median": round(med, 4), "ms_all": [round(x, 4) for x in all_ms],
                         "pairs_per_s": pairs * spots / (med * 1e-3), "total_per_spot": want, "mean_equity": round(eq, 6)}
            print(name, mode, "%.4f ms" % med, file=sys.stderr, flush=True)
        row["reference_over_uniform_throughput"] = round(row["uniform"]["ms_median"] / row["reference"]["ms_median"], 4)
        res["workloads"].append(row)
        print(json.dumps(row), file=sys.stderr, flush=True)
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
