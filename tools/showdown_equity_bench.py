"""Throughput of the exact showdown-equity enumeration (npk_showdown_equity_batch), one JSON line on stdout.

    python tools/showdown_equity_bench.py [--launches 20] [--out file.json]

Workloads (spots seeded with torch.Generator(0), distinct cards per spot):
    W1 hu_preflop        4,096 heads-up spots, no board      (1,712,304 completions each)
    W2 sixway_flop       65,536 six-player flops             (666 completions each)
    W3 ninefold_preflop  4,096 nine-player spots, no board   (278,256 completions each)
    W4 one_spot          one heads-up preflop spot through the blocking showdown_equity() call, and the single-core CPU
                         enumeration of tests/showdown_oracle.c on the same spot
Per batch workload: the median over `launches` timed calls (CUDA events around each call on the stream: the three kernels of
the call, outputs and workspace allocated once), completions/s and showdown evals/s (= completions x players / time).
The card's name, power limit and maximum SM clock are read in the same run."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import neuron_poker_b200 as npk  # noqa: E402
from neuron_poker_b200 import _lib  # noqa: E402


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power, clock = [x.strip() for x in q.split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def spots(n, players, board_cards, gen, dev):
    cards = torch.rand((n, 52), generator=gen).argsort(dim=1)[:, :2 * players + board_cards].to(torch.uint8)
    holes = cards[:, :2 * players].reshape(n, players, 2).contiguous().to(dev)
    board = torch.full((n, 5), 0xFF, dtype=torch.uint8)
    board[:, :board_cards] = cards[:, 2 * players:]
    return holes, torch.full((n,), players, dtype=torch.uint8, device=dev), board.to(dev)


def time_batch(L, holes, npl, board, launches, dev):
    N, maxp = holes.shape[0], holes.shape[1]
    outs = [torch.empty((N, maxp), dtype=torch.int64, device=dev) for _ in range(3)]
    comp = torch.empty(N, dtype=torch.int64, device=dev)
    ws = torch.empty(int(L.npk_showdown_equity_workspace_bytes(N)), dtype=torch.uint8, device=dev)
    stream = torch.cuda.current_stream(dev).cuda_stream

    def call():
        _lib.check(L.npk_showdown_equity_batch(holes.data_ptr(), npl.data_ptr(), board.data_ptr(), None, N, maxp,
                                               _lib.NPK_DEAL_UNIFORM, 0, outs[0].data_ptr(), outs[1].data_ptr(),
                                               outs[2].data_ptr(), comp.data_ptr(), ws.data_ptr(), stream))

    for _ in range(3):
        call()
    torch.cuda.synchronize(dev)
    ms = []
    for _ in range(launches):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        call()
        b.record()
        b.synchronize()
        ms.append(a.elapsed_time(b))
    t = statistics.median(ms) / 1e3
    completions = int(comp.sum())
    assert (outs[2].sum(dim=1) == 2520 * comp).all()
    return {"spots": N, "players": maxp, "completions": completions, "kernel_ms_median": round(t * 1e3, 4),
            "kernel_ms_min": round(min(ms), 4), "kernel_ms_max": round(max(ms), 4),
            "completions_per_s": completions / t, "showdown_evals_per_s": completions * maxp / t}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--launches", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("showdown_equity_bench needs a CUDA device")
    dev = torch.device("cuda", 0)
    L = _lib.ensure_init(0)
    gen = torch.Generator().manual_seed(0)
    res = {"tool": "showdown_equity_bench", "gpu": gpu_info(), "launches": args.launches}
    res["W1_hu_preflop"] = time_batch(L, *spots(4096, 2, 0, gen, dev), args.launches, dev)
    res["W2_sixway_flop"] = time_batch(L, *spots(65536, 6, 3, gen, dev), args.launches, dev)
    res["W3_ninefold_preflop"] = time_batch(L, *spots(4096, 9, 0, gen, dev), args.launches, dev)

    hands = [["AS", "KS"], ["QH", "QD"]]
    npk.showdown_equity(hands)
    calls = []
    for _ in range(args.launches):
        t0 = time.perf_counter()
        r = npk.showdown_equity(hands)
        calls.append(time.perf_counter() - t0)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import showdown_oracle
    showdown_oracle.lib()
    t0 = time.perf_counter()
    o = showdown_oracle.showdown_equity(hands, [])
    cpu = time.perf_counter() - t0
    assert o["win"] == r["win"] and o["tie"] == r["tie"] and o["completions"] == r["completions"]
    res["W4_one_spot"] = {"hands": hands, "completions": r["completions"], "call_ms_median": round(statistics.median(calls) * 1e3, 4),
                          "call_ms_min": round(min(calls) * 1e3, 4), "cpu_oracle_ms_single_core": round(cpu * 1e3, 2)}
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
