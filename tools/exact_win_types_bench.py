"""Cost of the win-type histograms: the exact engines' workloads timed with and without win_types, one JSON line on stdout.

    python tools/exact_win_types_bench.py [--reps 3] [--plain-only] [--out file.json]

Exact equity (exact_equity_batch, both dealing modes; the workloads of tools/exact_equity_bench.py): one heads-up preflop spot,
the 169 heads-up preflop classes, 4,096 heads-up rivers / turns / flops, 4,096 three-handed rivers / turns, 1,024 three-handed
flops and AsKs three-handed preflop (t3).  Showdown equity (showdown_equity_batch, uniform; the workloads of
tools/showdown_equity_bench.py): W1 4,096 heads-up preflop spots, W2 65,536 six-player flops, W3 4,096 nine-player preflop spots.
Per workload: the median over `reps` calls (CUDA events around the call on device tensors, without validation, after one
warm-up call) of the plain call and, unless --plain-only, of the call with win_types=True, whose win / tie / lose (or win / tie /
share / completions) are checked equal to the plain call's and whose bins are checked to sum to win + tie.  --plain-only uses
only arguments the engines had before win_types, so the same script times an older tree.  The card's name, power limit and
maximum SM clock are read in the same run."""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import torch  # noqa: E402

import neuron_poker_b200 as npk  # noqa: E402
from adaptive_equity_bench import gpu_info  # noqa: E402
from enum_reference_bench import class_spots, timed  # noqa: E402
from exact_equity_bench import AS, KS, fixed_spot, random_spots  # noqa: E402
from showdown_equity_bench import spots as showdown_spots  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--plain-only", action="store_true")
    ap.add_argument("--out")
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    res = {"tool": "exact_win_types_bench", "gpu": gpu_info(), "plain_only": args.plain_only, "exact": [], "showdown": []}
    loads = [("preflop1", lambda: fixed_spot([AS, KS], 2, dev)), ("preflop169", lambda: class_spots(dev)),
             ("river", lambda: random_spots(4096, 5, 2, dev)), ("turn", lambda: random_spots(4096, 4, 2, dev)),
             ("flop", lambda: random_spots(4096, 3, 2, dev)), ("river3", lambda: random_spots(4096, 5, 3, dev)),
             ("turn3", lambda: random_spots(4096, 4, 3, dev)), ("flop3", lambda: random_spots(1024, 3, 3, dev)),
             ("t3", lambda: fixed_spot([AS, KS], 3, dev))]
    for name, make in loads:
        hole, board, npl = make()
        n = hole.shape[0]
        holes, n_known, n_random = hole.view(n, 1, 2), torch.ones(n, dtype=torch.uint8, device=dev), npl - 1
        row = {"workload": name, "spots": n}
        for mode in ("uniform", "reference"):
            call = lambda **kw: npk.exact_equity_batch(holes, n_known, n_random, board, deal_mode=mode, **kw)
            med, all_ms, plain = timed(call, args.reps, True)
            r = {"plain_ms_median": round(med, 4), "plain_ms_all": [round(x, 4) for x in all_ms]}
            if not args.plain_only:
                tmed, tall, typed = timed(lambda: call(win_types=True), args.reps, True)
                for k in ("win", "tie", "lose"):
                    assert torch.equal(plain[k], typed[k]), (name, mode, k)
                assert torch.equal(typed["win_types"].sum(1), typed["win"] + typed["tie"]), (name, mode)
                r.update({"win_types_ms_median": round(tmed, 4), "win_types_ms_all": [round(x, 4) for x in tall],
                          "win_types_over_plain": round(tmed / med, 4)})
            row[mode] = r
            print(name, mode, r, file=sys.stderr, flush=True)
        res["exact"].append(row)
    gen = torch.Generator().manual_seed(0)
    for name, P, nb, n in (("W1_hu_preflop", 2, 0, 4096), ("W2_sixway_flop", 6, 3, 65536), ("W3_ninefold_preflop", 9, 0, 4096)):
        holes, npl, board = showdown_spots(n, P, nb, gen, dev)
        call = lambda **kw: npk.showdown_equity_batch(holes, npl, board, **kw)
        med, all_ms, plain = timed(call, args.reps, True)
        row = {"workload": name, "spots": n, "plain_ms_median": round(med, 4), "plain_ms_all": [round(x, 4) for x in all_ms]}
        if not args.plain_only:
            tmed, tall, typed = timed(lambda: call(win_types=True), args.reps, True)
            for k in plain:
                assert torch.equal(plain[k], typed[k]), (name, k)
            assert torch.equal(typed["win_types"].sum(2), typed["win"] + typed["tie"]), name
            row.update({"win_types_ms_median": round(tmed, 4), "win_types_ms_all": [round(x, 4) for x in tall],
                        "win_types_over_plain": round(tmed / med, 4)})
        res["showdown"].append(row)
        print(name, row, file=sys.stderr, flush=True)
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
