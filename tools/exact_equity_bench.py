"""Exact equity against one or two unknown opponents (exact_equity_batch) against the per-query enumeration
(enumerate_equity, enum_kernel) where that has the shape, one JSON line on stdout.

    python tools/exact_equity_bench.py [--reps 5] [--slow-reps 3] [--workloads ...] [--out profiles/exact_equity_bench.json]

Workloads (seed 0, distinct cards, no known hands, no dead cards):
    preflop1   one heads-up preflop spot (AsKs)                     C(50,5) completions x C(45,2) hands
    preflop169 the 169 starting-hand classes, heads-up, no board
    river, turn, flop      4,096 heads-up spots                    also timed through enumerate_equity
    river3     4,096 three-handed rivers                           also timed through enumerate_equity
    turn3      4,096 three-handed turns                            46 completions x unordered pairs of disjoint hands
    flop3      1,024 three-handed flops
    t3         AsKs, three players, preflop (the reference's test t3)
Per workload and mode: the median over the repetitions (CUDA events around the call on device tensors, without validation,
after one warm-up call), the (completion, unknown tuple) steps per second -- ordered tuples of the uniform enumeration in both
modes -- and, where enumerate_equity has the shape, its median and the ratio enum time / exact time (above 1: the new engine is
faster).  enum_kernel's preflop walk is not re-run: about 112 s per spot and 223 s for the 169 classes on a B200 (DESIGN.md
section 4.4).  The totals of both modes are checked against their closed forms, and the counts against enumerate_equity's.  The
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
from enum_reference_bench import class_spots, timed  # noqa: E402

AS, KS = 51, 47


def random_spots(q, known, players, dev, seed=0):
    rng = np.random.default_rng(seed)
    cards = np.stack([rng.permutation(52)[:2 + known] for _ in range(q)]).astype(np.uint8)
    board = np.full((q, 5), 0xFF, dtype=np.uint8)
    board[:, :known] = cards[:, 2:]
    return [torch.as_tensor(x).to(dev) for x in (cards[:, :2].copy(), board, np.full(q, players, dtype=np.uint8))]


def fixed_spot(hole, players, dev):
    return [torch.as_tensor(x).to(dev) for x in (np.array([hole], dtype=np.uint8), np.full((1, 5), 0xFF, dtype=np.uint8),
                                                 np.array([players], dtype=np.uint8))]


def sizes(known, players):
    """(completion, unknown tuple) steps per spot, and the totals of both modes."""
    n, m = 50 - known, 5 - known
    if players == 2:
        return (math.comb(n, m) * math.comb(n - m, 2), math.comb(n, 2) * math.comb(n - 2, m),
                (n - 1) ** 2 * math.comb(n - 3, m))
    steps = math.comb(n, m) * math.comb(n - m, 2) * math.comb(n - m - 2, 2)
    return steps, steps, (n - 1) ** 2 * (n - 3) ** 2 * math.comb(n - 5, m)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--slow-reps", type=int, default=3)
    ap.add_argument("--workloads", default="preflop1,preflop169,river,turn,flop,river3,turn3,flop3,t3")
    ap.add_argument("--out")
    args = ap.parse_args()
    wanted = args.workloads.split(",")
    dev = torch.device("cuda", 0)
    res = {"tool": "exact_equity_bench", "gpu": gpu_info(),
           "sm_count": torch.cuda.get_device_properties(dev).multi_processor_count,
           "enum_kernel_preflop_s": {"one_spot": 112, "classes_169": 223, "source": "DESIGN.md section 4.4"}, "workloads": []}
    loads = [("preflop1", lambda: fixed_spot([AS, KS], 2, dev), 0, 2, False, True),
             ("preflop169", lambda: class_spots(dev), 0, 2, False, True),
             ("river", lambda: random_spots(4096, 5, 2, dev), 5, 2, True, False),
             ("turn", lambda: random_spots(4096, 4, 2, dev), 4, 2, True, False),
             ("flop", lambda: random_spots(4096, 3, 2, dev), 3, 2, True, False),
             ("river3", lambda: random_spots(4096, 5, 3, dev), 5, 3, True, False),
             ("turn3", lambda: random_spots(4096, 4, 3, dev), 4, 3, False, True),
             ("flop3", lambda: random_spots(1024, 3, 3, dev), 3, 3, False, True),
             ("t3", lambda: fixed_spot([AS, KS], 3, dev), 0, 3, False, True)]
    for name, make, known, players, vs_enum, slow in loads:
        if name not in wanted:
            continue
        hole, board, npl = make()
        spots = hole.shape[0]
        holes = hole.view(spots, 1, 2)
        n_known = torch.ones(spots, dtype=torch.uint8, device=dev)
        n_random = npl - 1
        steps, uniform_total, reference_total = sizes(known, players)
        row = {"workload": name, "spots": spots, "players": players, "known_board_cards": known,
               "steps_per_spot": steps, "steps_per_call": steps * spots}
        for mode, want in (("uniform", uniform_total), ("reference", reference_total)):
            reps = args.slow_reps if slow else args.reps
            med, all_ms, out = timed(lambda: npk.exact_equity_batch(holes, n_known, n_random, board, deal_mode=mode), reps, True)
            totals = (out["win"] + out["tie"] + out["lose"]).cpu()
            assert bool((totals == want).all()), (name, mode, totals[:4], want)
            eq = ((out["win"] + out["tie"]).double() / totals.double().to(dev)).mean().item()
            r = {"ms_median": round(med, 4), "ms_all": [round(x, 4) for x in all_ms], "steps_per_s": steps * spots / (med * 1e-3),
                 "total_per_spot": want, "mean_equity": round(eq, 6)}
            if spots == 1:
                r["counts"] = [int(out[k][0]) for k in ("win", "tie", "lose")]
            if vs_enum:
                emed, eall, eout = timed(lambda: npk.enumerate_equity(hole, board, npl, deal_mode=mode), args.reps, True)
                assert all(bool((eout[i] == out[k]).all()) for i, k in enumerate(("win", "tie", "lose"))), (name, mode)
                r["enum_ms_median"] = round(emed, 4)
                r["enum_ms_all"] = [round(x, 4) for x in eall]
                r["enum_over_exact_time"] = round(emed / med, 4)
            row[mode] = r
            print(name, mode, "%.4f ms" % med, file=sys.stderr, flush=True)
        res["workloads"].append(row)
        print(json.dumps(row), file=sys.stderr, flush=True)
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
