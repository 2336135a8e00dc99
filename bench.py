#!/usr/bin/env python3
"""bench.py -- headline benchmark of the equity hot path (BASELINE.json: "showdown evals/s ...; get_equity calls/s").

    python bench.py [--gpus N] [--steps K] [--warmup W]          # the default line: cfg3 headline + every other config
    python bench.py --dump-outputs DIR ...      # also write the counters of the headline's last timed step to DIR/*.npy
    python bench.py --workload cfg1|cfg2|cfg3|cfg4|cfg5|ranges [--deal uniform|reference]    # one workload alone
    python bench.py --impl reference ...        # the reference's own C++ calculator on the host cores (oracle/_ref)
    torchrun --nproc-per-node N bench.py --gpus N ...   (one rank per GPU)

A "step" is one pass of the hot path over one batch of synthetic queries.  The headline (`value`, `e2e`, `roofline`) is
  cfg3: 4,096 six-player flop queries x 10,000 trials per GPU = 245.76 M showdown evals per step per GPU; N GPUs: every
        rank owns its own 4,096 queries (weak scaling, no data-path collective; global query ids in the Philox counter).
The same JSON line carries, measured in the same run (BASELINE.json `configs`, SURVEY 8d):
  `sustained`  the cfg3 step looped for >= 3 s with its own clock samples (the K-step figure is a burst of a few ms)
  `workloads`  cfg1 (one heads-up preflop call: latency, CPU vs GPU), cfg2 (exact enumeration + rank ids of 64 M hands
               against the HBM roofline), cfg3 with the reference's dealer, cfg4 (169 classes x 1 M trials x 9 players,
               trials split over the N ranks with the count all-reduce INSIDE the timed step: strong scaling, efficiency
               against the unsharded job on one GPU, counters asserted bit-identical to the unsharded run on the device),
               cfg5 (65,536 six-max tables in self-play, both dealers) and an opponent-range workload
  `cpu_baseline`  the reference's C++, Python and numpy2 calculators on this box's host cores (N = 1 only)
`value` = showdown evals (trials x players, all ranks) / device time of the K steps (CUDA events, max over ranks), with
the queries already resident in HBM.  `e2e` = the same metric through the host-buffer API (equity_counts_batch ->
npk_equity_host): queries start in host memory, H2D + kernels + D2H inside the timed region.
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "showdown_evals_per_s"
UNIT = "showdown evals/s"


def algorithmic_instr(players, known):
    """SURVEY.md 8(d): integer thread-instructions one trial needs, A(P,b) = 64*ceil(D/8) + 8*D + 14*P + (P+3)."""
    d = 2 * (players - 1) + (5 - known)
    return 64 * -(-d // 8) + 8 * d + 14 * players + (players + 3)


def workload(name):
    if name == "cfg3":
        return dict(name="cfg3: 4096 six-player flop queries x 10000 trials per GPU", queries=4096, trials=10000,
                    players=6, known=3, shard="query")
    if name == "cfg4":
        return dict(name="cfg4: 169 starting-hand classes x 1000000 trials, 9 players, preflop", queries=169,
                    trials=1000000, players=9, known=0, shard="trial")
    if name == "cfg2":
        return dict(name="cfg2: exact enumeration of 4096 heads-up turn spots + 4096 river spots; rank ids of 64 M hands",
                    queries=4096, trials=0, players=2, known=4, shard="query")
    if name == "cfg5":
        return dict(name="cfg5: 65536 six-max HoldemTable self-play steps, get_equity (1000 runs) for every action",
                    queries=65536, trials=1000, players=6, known=-1, shard="query")
    if name == "cfg1":
        return dict(name="cfg1: AsKs heads-up preflop x 10000 trials", queries=1, trials=10000, players=2, known=0,
                    shard="query")
    if name == "ranges":
        return dict(name="ranges: 4096 six-player flop queries x 1000 trials, opponents in the top 30 % of the reference's "
                         "preflop ranking", queries=4096, trials=1000, players=6, known=3, shard="query")
    raise SystemExit("unknown workload " + name)


def make_queries(wl, world, rank):
    """Synthetic queries (numpy uint8).  cfg3: seed-0 torch generator, 5 distinct uniform cards per query (SURVEY 8d)."""
    import numpy as np
    import torch
    q = wl["queries"]
    if wl["name"].startswith("cfg3") or wl["name"].startswith("ranges"):
        g = torch.Generator().manual_seed(0)
        cards = torch.rand(q * world, 52, generator=g).argsort(1)[:, :5].to(torch.uint8).numpy()
        cards = cards[rank * q:(rank + 1) * q]
        hole = cards[:, :2].copy()
        board = np.full((q, 5), 255, dtype=np.uint8)
        board[:, :3] = cards[:, 2:5]
    elif wl["name"].startswith("cfg4"):
        hole = []
        for hi in range(13):
            for lo in range(hi + 1):
                if hi == lo:
                    hole.append([4 * hi + 0, 4 * hi + 1])            # pair: xC xD
                else:
                    hole.append([4 * hi + 3, 4 * lo + 3])            # suited: xS yS
                    hole.append([4 * hi + 3, 4 * lo + 2])            # offsuit: xS yH
        hole = np.array(hole, dtype=np.uint8)
        assert len(hole) == 169
        board = np.full((169, 5), 255, dtype=np.uint8)
    else:
        hole = np.array([[51, 47]], dtype=np.uint8)
        board = np.full((1, 5), 255, dtype=np.uint8)
    npl = np.full(len(hole), wl["players"], dtype=np.uint8)
    return hole, board, npl


class ClockSampler(threading.Thread):
    """SM clock / throttle reasons during the timed region (NVML, 10 ms period)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz, self._halt = index, [], set(), None, threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None or os.environ.get("NPK_BENCH_NO_SAMPLER") == "1":      # (debugging aid: no NVML calls at all)
            return
        nv = self.nv
        names = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20,
                 "hw_power_brake_slowdown": 0x80, "applications_clocks_setting": 0x2}
        while not self._halt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for n, bit in names.items():
                    if r & bit:
                        self.reasons.add(n)
            except Exception:
                pass
            time.sleep(0.01)

    def stop(self):
        self._halt.set()
        self.join(timeout=1)
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_min_mhz": s[0] if s else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(s)}


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


# ---------------------------------------------------------------------------------------------------------------------
# CPU legs: the reference's own implementations on the host cores
# ---------------------------------------------------------------------------------------------------------------------
def reference_sample(wl, hole, board, npl, n_queries, threads):
    """Time the reference's own C++ montecarlo() (oracle/_ref) on `n_queries` queries of the workload, `threads` threads."""
    import oracle
    hs = [[int(c) for c in hole[i % len(hole)]] for i in range(n_queries)]
    bs = [[int(c) for c in board[i % len(board)] if c != 255] for i in range(n_queries)]
    ps = [int(npl[i % len(npl)]) for i in range(n_queries)]
    t0 = time.perf_counter()
    eq = oracle.ref_montecarlo_batch(hs, bs, ps, wl["trials"], threads)
    dt = time.perf_counter() - t0
    assert all(0.0 <= e <= 1.0 for e in eq)
    return n_queries * wl["trials"] * wl["players"] / dt, dt


def port_sample(wl, hole, board, npl, n_queries):
    """Fallback when oracle/_ref was never built: the C port of the same loop (oracle/npk_oracle.c), one thread."""
    import oracle
    t0 = time.perf_counter()
    for i in range(n_queries):
        oracle.mc_uniform([int(c) for c in hole[i % len(hole)]], [int(c) for c in board[i % len(board)] if c != 255],
                          int(npl[i % len(npl)]), wl["trials"], 1 + i)
    dt = time.perf_counter() - t0
    return n_queries * wl["trials"] * wl["players"] / dt, dt


def cpu_baselines(wl, hole, board, npl, budget_cpp=12.0):
    """SURVEY 8d: the reference's C++ sibling, its Python run_montecarlo (1-s cut-off disabled), get_equity as shipped
    (cut-off active) and the numpy2 sibling (results wrong post-flop upstream: timed, flagged), each on one core and
    fanned out over all host cores, on queries of the workload.  Bounded to about 30 s of wall clock."""
    import oracle
    cores = host_cores()
    Q, T, P = len(hole), wl["trials"], wl["players"]
    out = {}
    if oracle.ref_available():
        v1, dt1 = reference_sample(wl, hole, board, npl, 1, 1)
        n = min(max(1, Q), 2 * cores)
        v, dt = reference_sample(wl, hole, board, npl, n, cores)
        n = int(max(n, min(Q if Q > 1 else 64, n * budget_cpp / max(dt, 1e-3))))
        v, dt = reference_sample(wl, hole, board, npl, n, cores)
        out = {"value": v, "unit": UNIT, "cores": cores, "kind": "reference",
               "sample": "%d queries x %d trials through the reference C++ montecarlo() (oracle/_ref), %d threads, %.1f s"
                         % (n, T, cores, dt),
               "cpp": {"one_core": v1, "all_cores": v, "cores": cores, "unit": UNIT,
                       "sample": "1 query / %d queries x %d trials, Montecarlo.cpp:240-259 compiled in place" % (n, T)}}
    else:
        v, dt = port_sample(wl, hole, board, npl, 2)
        out = {"value": v, "unit": UNIT, "cores": 1, "kind": "port",
               "sample": "2 queries x %d trials through oracle/npk_oracle.c, %.1f s" % (T, dt)}
    try:
        from oracle import ref_python
        if not ref_python.available():
            raise RuntimeError("baseline/_ref not built")
        q0 = (hole[0], board[0], int(npl[0]))
        eq, dt, ran = ref_python.python_run_montecarlo(*q0, T)
        py1 = ran * P / dt
        eqs, dts, rans = ref_python.python_get_equity_as_shipped(*q0, T)
        procs = min(cores, 32)
        qs = [(hole[i % Q], board[i % Q], int(npl[i % Q])) for i in range(procs)]
        res, wall = ref_python.fan_out("python", qs, T, procs)
        pyn = sum(r[2] for r in res) * P / wall
        eq2, dt2, ran2 = ref_python.numpy2_montecarlo(*q0, T)
        res2, wall2 = ref_python.fan_out("numpy2", qs * 4, T, procs)
        out["python"] = {"one_core": py1, "all_cores": pyn, "processes": procs, "unit": UNIT,
                         "sample": "MonteCarlo.run_montecarlo (montecarlo_python.py:191-252), timeout=+inf: 1 query x %d "
                                   "trials in %.2f s (equity %.3f); %d processes x 1 query in %.2f s" % (T, dt, eq, procs, wall),
                         "get_equity_as_shipped": {"seconds_per_call": dts, "trials_requested": T, "trials_run": rans,
                                                   "calls_per_s_per_core": 1.0 / dts, "equity": eqs,
                                                   "note": "montecarlo_python.py:401-406 stops after 1 s of wall clock"}}
        out["numpy2"] = {"one_core": ran2 * P / dt2, "all_cores": sum(r[2] for r in res2) * P / wall2, "processes": procs,
                         "unit": UNIT, "incorrect_results": True,
                         "sample": "numpy_montecarlo (montecarlo_numpy2.py:333-346): 1 query x %d trials in %.2f s, equity "
                                   "%.3f (wrong post-flop upstream, all its tests are skipped); %d processes x 4 queries in "
                                   "%.2f s" % (T, dt2, eq2, procs, wall2)}
    except Exception as exc:                                     # the GPU line must not die on a host-side baseline
        out["python"] = {"unavailable": repr(exc)[:200]}
    return out


def run_reference_arm(args, wl, rank):
    if rank != 0:
        return
    import oracle
    hole, board, npl = make_queries(wl, 1, 0)
    cores = host_cores()
    have_ref = oracle.ref_available()
    if have_ref:
        _, t1 = reference_sample(wl, hole, board, npl, 1, 1)
    else:
        _, t1 = port_sample(wl, hole, board, npl, 1)
    budget = 150.0
    n = int(max(1, min(4 * cores, budget * (cores if have_ref else 1) / ((args.steps + args.warmup) * t1))))
    n = min(n, max(1, wl["queries"]))
    times = []
    for i in range(args.warmup + args.steps):
        if have_ref:
            _, dt = reference_sample(wl, hole, board, npl, n, cores)
        else:
            _, dt = port_sample(wl, hole, board, npl, n)
        if i >= args.warmup:
            times.append(dt)
    total = sum(times)
    value = n * wl["trials"] * wl["players"] * args.steps / total
    sample = "%d of the workload's %d queries x %d trials per step" % (n, wl["queries"], wl["trials"])
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "int", "data": "synthetic",
            "config": {"workload": wl["name"], "players": wl["players"], "known_board_cards": wl["known"],
                       "trials": wl["trials"], "deal_mode": "uniform", "sample": sample},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores if have_ref else 1,
                             "kind": "reference" if have_ref else "port", "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------------------------
# GPU legs.  Every leg returns a dict; all ranks run it, timings are the max over ranks.
# ---------------------------------------------------------------------------------------------------------------------
class Ctx(object):
    def __init__(self, rank, world, local_rank, dev, L):
        self.rank, self.world, self.local_rank, self.dev, self.L = rank, world, local_rank, dev, L

    def max_over_ranks(self, x):
        import torch
        import torch.distributed as dist
        t = torch.tensor(x if isinstance(x, (list, tuple)) else [x], dtype=torch.float64, device=self.dev)
        if self.world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        v = [float(a) for a in t.tolist()]
        return v if isinstance(x, (list, tuple)) else v[0]

    def sum_over_ranks(self, t):
        import torch.distributed as dist
        if self.world > 1:
            dist.all_reduce(t)
        return t

    def barrier(self):
        import torch
        import torch.distributed as dist
        torch.cuda.synchronize()
        if self.world > 1:
            dist.barrier()


def int_issue_peak(L):
    """Integer-issue peak of this GPU, measured in this run (roofline denominator)."""
    import ctypes
    from neuron_poker_b200 import _lib
    peak, detail = 0.0, {}
    for variant, nm in ((0, "lop3"), (1, "imad"), (2, "imad+lop3")):
        v = ctypes.c_double(0)
        ms = ctypes.c_float(0)
        _lib.check(L.npk_int_peak(variant, 2000, ctypes.byref(v), ctypes.byref(ms)))
        detail[nm] = v.value / 1e12
        peak = max(peak, v.value)
    return peak, detail


def run_exact(args, wl, cx, steps=None):
    """cfg2 (SURVEY 8d): the exact kernels.  K3 enumerates every opponent hand x board completion of 4,096 heads-up turn
    spots and 4,096 river spots (seed-0 synthetic: 2 hole + 4 / 5 board cards, distinct, uniform); K2 ranks 64 M random
    7-card hands (7 B in, 2 B out per hand).  value = showdown evals/s of the enumeration (two hands per matchup)."""
    import torch
    import neuron_poker_b200 as npk
    rank, world, dev = cx.rank, cx.world, cx.dev
    Q = wl["queries"]
    g = torch.Generator().manual_seed(rank)
    cards = torch.rand(2 * Q, 52, generator=g).argsort(1)[:, :7].to(torch.uint8)
    hole = cards[:, :2].contiguous().to(dev)
    board = cards[:, 2:7].clone()
    board[:Q, 4] = 255                                      # first half: turn spots (one card to come)
    board = board.to(dev)
    npl = torch.full((2 * Q,), 2, dtype=torch.uint8, device=dev)
    matchups = Q * 46 * (45 * 44 // 2) + Q * (45 * 44 // 2)  # turn: 46 rivers x C(45,2) opponent hands; river: C(45,2)
    n_hands = 64 << 20
    hands = torch.rand(1 << 20, 52, generator=g).argsort(1)[:, :7].to(torch.uint8).to(dev).repeat(64, 1).contiguous()
    for _ in range(max(3, args.warmup)):
        w, t, l = npk.enumerate_equity(hole, board, npl)
        r = npk.rank7(hands)
    torch.cuda.synchronize()
    assert int((w + t + l).sum().item()) == matchups
    cx.barrier()
    steps = args.steps if steps is None else steps
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    sampler = ClockSampler(cx.local_rank)
    sampler.start()
    ev[0].record()
    for _ in range(steps):
        npk.enumerate_equity(hole, board, npl)
    ev[1].record()
    for _ in range(steps):
        npk.rank7(hands)
    ev[2].record()
    torch.cuda.synchronize()
    clocks = sampler.stop()
    enum_ms, rank_ms = (x / steps for x in cx.max_over_ranks([ev[0].elapsed_time(ev[1]), ev[1].elapsed_time(ev[2])]))
    # end to end: host arrays in, host arrays out
    hole_h, board_h, npl_h = hole.cpu().numpy(), board.cpu().numpy(), npl.cpu().numpy()
    t0 = time.perf_counter()
    for _ in range(3):
        w, t, l = npk.enumerate_equity(hole_h, board_h, npl_h)
        w.cpu(); t.cpu(); l.cpu()
    e2e_s = (time.perf_counter() - t0) / 3
    del hands
    peaks = {}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peaks = json.load(f)
    except Exception:
        pass
    hbm = float(peaks.get("hbm_gbs", 6544.3))
    rank_gbs = n_hands * 9 / (rank_ms * 1e-3) / 1e9
    return {"metric": METRIC, "value": 2 * matchups * world / (enum_ms * 1e-3), "unit": UNIT, "n_gpus": world, "steps": steps,
            "warmup": max(3, args.warmup), "ms_per_step": enum_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u32", "data": "synthetic",
            "config": {"workload": wl["name"], "spots_per_gpu": 2 * Q, "matchups_per_step": matchups,
                       "matchups_per_s": matchups * world / (enum_ms * 1e-3), "rank7_hands_per_s": n_hands * world / (rank_ms * 1e-3),
                       "rank7_ms": rank_ms, "l2": "rank7 input 448 MiB > L2; enumeration inputs are 64 KB"},
            "clocks": clocks,
            "e2e": {"value": 2 * matchups * world / e2e_s, "unit": UNIT, "h2d_bytes_per_step": 16 * Q, "d2h_bytes_per_step": 48 * Q,
                    "steps": 3, "api": "neuron_poker_b200.enumerate_equity (numpy in, counters read back)"},
            "gpu_launches": 2 * steps,
            "roofline": {"bound": "hbm", "kernel": "rank7_kernel", "achieved": rank_gbs, "peak": hbm, "unit": "GB/s",
                         "frac": rank_gbs / hbm, "traffic": None,
                         "algorithmic_bytes_per_hand": 9, "peak_source": "MEASURED_PEAKS.json hbm_gbs" if peaks else "fallback 6544.3"}}


def run_selfplay(args, wl, cx, deal, steps=None):
    """cfg5: every rank owns 65,536 six-max tables (4 equity agents + 2 random ones, main.py:136-150).  One step = one
    action on every table: equity query of the current player (1,000 runs, all players alive, env.py:262-264) -> Monte-Carlo
    kernels -> agent decisions -> betting state machine -> finished games restarted; nothing leaves the device."""
    import torch
    from neuron_poker_b200.holdem import EquityAgents, HoldemTables
    rank, world, dev = cx.rank, cx.world, cx.dev
    steps = args.steps if steps is None else steps
    N, runs = wl["queries"], wl["trials"]
    tb = HoldemTables(N, n_players=6, seed=7, table_offset=rank * N, autoplay=[1] * 6, device=dev)
    agents = EquityAgents.equity_vs_random()
    # what every step asked for is recorded (one small copy kernel per step) and summed after the timed region
    n_e2e = max(3, min(steps, 50))
    rec = torch.zeros((steps + n_e2e, N), dtype=torch.uint8, device=dev)
    cursor = [0]

    def step(count):
        tb.selfplay_step(agents, runs=runs, deal_mode=deal)
        _, _, npl, active = tb._q
        # players of the query, 0 for a table without a query.  Warm-up steps do the same into the last row (overwritten
        # later): the first launch of this torch kernel in a process loads its module, which on a freshly started box cost
        # the timed window 8 ms when only timed steps recorded (1.10 instead of 1.03 ms per step in the first process)
        torch.mul(npl, active, out=rec[cursor[0] if count else -1])
        if count:
            cursor[0] += 1

    def totals(lo, hi):
        r = rec[lo:hi].to(torch.int64)
        return torch.stack([r.sum() * runs, (r > 0).sum()])

    sampler = ClockSampler(cx.local_rank)            # (NVML initialisation happens here, before anything is timed)
    for _ in range(max(args.warmup, 100)):          # reach a steady mix of streets and player counts (and let whatever the
        step(False)                                 # process still pages in settle: 0.1 s)
    cx.barrier()
    sampler.start()
    for _ in range(5):                              # the GPU's queue is full when the clock starts: no idle gap in front of
        step(False)                                 # the first timed step (a 60-step leg is 70 ms long)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    h0 = time.perf_counter()
    for _ in range(steps):
        step(True)
    e1.record()
    host_ms = 1e3 * (time.perf_counter() - h0)      # what the host needed to enqueue the timed steps
    torch.cuda.synchronize()
    clocks = sampler.stop()
    dev_ms = cx.max_over_ranks(e0.elapsed_time(e1))
    tot = cx.sum_over_ranks(totals(0, steps).to(torch.float64))
    st = tb.state()
    # end to end: the same loop with the rewards of every step copied to the host
    w0 = time.perf_counter()
    for _ in range(n_e2e):
        step(True)
        tb.rewards.cpu()
    e2e_s = cx.max_over_ranks(time.perf_counter() - w0)
    e2e_evals = float(cx.sum_over_ranks(totals(steps, steps + n_e2e).to(torch.float64))[0].item())
    return {
        "metric": METRIC, "value": float(tot[0].item()) / (dev_ms * 1e-3), "unit": UNIT, "n_gpus": world, "steps": steps,
        "warmup": max(args.warmup, 100) + 5, "ms_per_step": dev_ms / steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u32", "data": "synthetic",
        "config": {"workload": wl["name"], "tables_per_gpu": N, "runs_per_action": runs, "deal_mode": deal,
                   "agents": "4 x agent_consider_equity + 2 x agent_random (main.py:136-150)",
                   "table_actions_per_s": float(tot[1].item()) / (dev_ms * 1e-3),
                   "mean_players_per_query": float(tot[0].item()) / max(1.0, float(tot[1].item()) * runs),
                   "hands_played_per_table": float(st["hands_played"].mean()), "table_errors": int((st["error"] != 0).sum()),
                   "host_enqueue_ms_per_step": host_ms / steps,
                   "l2": "state (50 MB per rank) streams through L2 every step; not flushed"},
        "clocks": clocks,
        "e2e": {"value": e2e_evals / e2e_s, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 8 * N,
                "steps": n_e2e, "api": "HoldemTables.selfplay_step + rewards.cpu()"},
        "gpu_launches": steps * tb.launches_per_step,
    }


def run_ranges(args, wl, cx, steps=None):
    """Opponent ranges (SURVEY 8f-2, montecarlo_python.py:136-181): 4,096 six-player flop queries x 1,000 trials, every
    opponent restricted to the top 30 % of the reference's preflop ranking, reference dealer.  `value` = the pair-list
    sampler (equity_ranges_fast_kernel, what a call without `passes` runs); the generic kernel that plays the reference's
    attempt loop literally (and counts `passes`) is timed beside it."""
    import torch
    import neuron_poker_b200 as npk
    dev = cx.dev
    steps = args.steps if steps is None else steps
    hole_h, board_h, npl_h = make_queries(wl, cx.world, cx.rank)
    hole, board, npl = (torch.as_tensor(x).to(dev) for x in (hole_h, board_h, npl_h))
    Q, T, P = len(hole_h), wl["trials"], wl["players"]
    out = {"wins": torch.zeros(Q, dtype=torch.int64, device=dev), "ties": torch.zeros(Q, dtype=torch.int64, device=dev),
           "passes": torch.zeros(Q, dtype=torch.int64, device=dev)}

    def timed(with_passes):
        def step(i):
            for v in out.values():
                if isinstance(v, torch.Tensor):
                    v.zero_()
            npk.get_equity_ranges_batch(hole, board, npl, T, opponent_range=0.3, seed_value=300 + i, deal_mode=args.deal_ranges,
                                        query_offset=cx.rank * Q, validate=False, passes=with_passes, out=out)
        for i in range(3):
            step(i)
        cx.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            step(3 + i)
        e1.record()
        torch.cuda.synchronize()
        return cx.max_over_ranks(e0.elapsed_time(e1)) / steps, float((out["wins"] + out["ties"]).double().mean().item() / T)

    ms_generic, eq_generic = timed(True)
    attempts = float(out["passes"].double().sum().item()) / (Q * T * (P - 1))
    ms, eq = timed(False)
    mode = 1 if args.deal_ranges == "reference" else 0
    return {"metric": METRIC, "value": Q * T * P * cx.world / (ms * 1e-3), "unit": UNIT, "n_gpus": cx.world, "steps": steps,
            "ms_per_step": ms, "scaling": "weak", "dtype": "u32", "data": "synthetic",
            "config": {"workload": wl["name"], "queries_per_gpu": Q, "trials": T, "players": P, "opponent_range": 0.3,
                       "deal_mode": args.deal_ranges, "mean_equity": eq,
                       "generic_kernel": {"kernel": "equity_ranges_kernel<%d>" % mode, "ms_per_step": ms_generic,
                                          "value": Q * T * P * cx.world / (ms_generic * 1e-3), "mean_equity": eq_generic,
                                          "attempts_per_opponent_hand": attempts,
                                          "note": "plays the reference's attempt loop literally; the only variant that "
                                                  "can count `passes`"}},
            "gpu_launches": steps, "kernel": "equity_ranges_fast_kernel<%d>" % mode}


def run_latency(args, wl, cx, with_cpu):
    """cfg1 (BASELINE config 1): get_equity({'AS','KS'}, set(), 2, 10000) -- one blocking call from Python, string parsing,
    launch, synchronisation and result read-back inside.  GPU through the drop-in; CPU through the reference's own
    tools/montecarlo_python.get_equity (as shipped, 1-s cut-off) and run_montecarlo without the cut-off."""
    import neuron_poker_b200 as npk
    res = {"workload": wl["name"]}
    for name, fn in (("get_equity", lambda: npk.get_equity({"AS", "KS"}, set(), 2, 10000)),
                     ("montecarlo", lambda: npk.montecarlo({"AS", "KS"}, {"null"}, 2, 10000))):
        for _ in range(30):
            fn()
        n = 400
        t0 = time.perf_counter()
        vals = [fn() for _ in range(n)]
        dt = time.perf_counter() - t0
        res[name] = {"us_per_call": 1e6 * dt / n, "calls_per_s": n / dt, "mean_equity": sum(vals) / n, "calls": n,
                     "dealer": "reference (montecarlo_python.py:165-189)" if name == "get_equity" else "uniform (Montecarlo.cpp:293-312)"}
    # the other half of BASELINE.json's metric: get_equity calls/s at 10,000 trials, 6 players
    fn = lambda: npk.get_equity({"AS", "KS"}, {"2C", "7D", "KH"}, 6, 10000)      # noqa: E731
    for _ in range(30):
        fn()
    n = 400
    t0 = time.perf_counter()
    vals = [fn() for _ in range(n)]
    dt = time.perf_counter() - t0
    res["get_equity_6_players_flop"] = {"us_per_call": 1e6 * dt / n, "calls_per_s": n / dt, "mean_equity": sum(vals) / n}
    # resident mode (opt-in, npk_resident_start): a persistent kernel serves the calls from a mailbox in mapped host memory,
    # no kernel launch per call; same results bit for bit
    npk.resident(True, idle_us=1000)
    try:
        for _ in range(30):
            fn()
        n = 2000
        t0 = time.perf_counter()
        vals = [fn() for _ in range(n)]
        dt = time.perf_counter() - t0
        res["get_equity_6_players_flop"]["resident"] = {"us_per_call": 1e6 * dt / n, "calls_per_s": n / dt,
                                                        "mean_equity": sum(vals) / n, "calls": n,
                                                        "mode": "neuron_poker_b200.resident(True): persistent server kernel on all "
                                                                "SMs, idle limit 1 ms"}
        f1 = lambda: npk.get_equity({"AS", "KS"}, set(), 2, 10000)      # noqa: E731
        for _ in range(30):
            f1()
        t0 = time.perf_counter()
        vals = [f1() for _ in range(n)]
        dt = time.perf_counter() - t0
        res["get_equity"]["resident"] = {"us_per_call": 1e6 * dt / n, "calls_per_s": n / dt, "mean_equity": sum(vals) / n}
    finally:
        npk.resident(False)
    # the same call from several host threads at once (the host entry point is re-entrant: every thread owns its stream and
    # result block inside libnpk, ctypes releases the GIL during the call): aggregate calls/s of the process
    import threading
    for nt in (2, 4):
        n_each = 1500
        gate = threading.Barrier(nt + 1)

        def worker():
            for _ in range(30):
                fn()
            gate.wait()
            for _ in range(n_each):
                fn()
            gate.wait()

        ts = [threading.Thread(target=worker) for _ in range(nt)]
        for t in ts:
            t.start()
        gate.wait()
        t0 = time.perf_counter()
        gate.wait()
        dt = time.perf_counter() - t0
        for t in ts:
            t.join()
        res["get_equity_6_players_flop"]["calls_per_s_%d_host_threads" % nt] = nt * n_each / dt
    if with_cpu:
        try:
            from oracle import ref_python
            h, b = [51, 47], [255] * 5
            eq, dt, ran = ref_python.python_get_equity_as_shipped(h, b, 2, 10000)
            eq2, dt2, ran2 = ref_python.python_run_montecarlo(h, b, 2, 10000)
            res["cpu_reference"] = {"get_equity_as_shipped": {"seconds": dt, "trials_run": ran, "equity": eq},
                                    "run_montecarlo_no_cutoff": {"seconds": dt2, "trials_run": ran2, "equity": eq2},
                                    "cores": 1, "source": "baseline/_ref/tools/montecarlo_python.py (unmodified copy)"}
            res["speedup_vs_python_full_10k"] = dt2 / (res["get_equity"]["us_per_call"] * 1e-6)
        except Exception as exc:
            res["cpu_reference"] = {"unavailable": repr(exc)[:200]}
    return res


def run_mc(args, wl, cx, deal, steps, warmup, peak=None, peak_detail=None, e2e=True, flush=True):
    """The Monte-Carlo kernels on a uniform-shape batch: cfg3 (query blocks per rank, no collective) and cfg4 (trial ranges
    per rank, the [2,Q] count all-reduce inside the timed step)."""
    import torch
    import neuron_poker_b200 as npk
    rank, world, dev = cx.rank, cx.world, cx.dev
    hole_h, board_h, npl_h = make_queries(wl, world, rank)
    Q, T, P, B = len(hole_h), wl["trials"], wl["players"], wl["known"]
    hole, board, npl = (torch.as_tensor(x).to(dev) for x in (hole_h, board_h, npl_h))
    by_trial = wl["shard"] == "trial" and world > 1
    t_off, t_cnt = npk.dist.trial_shard(T, rank, world) if by_trial else (0, T)
    q_off = 0 if wl["shard"] == "trial" else rank * Q
    both = torch.zeros((2, Q), dtype=torch.int64, device=dev)              # wins row, ties row: one tensor to all-reduce
    out = {"wins": both[0], "ties": both[1]}
    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device=dev) if flush else None      # > 126 MB L2
    job = npk.dist.TrialShardedJob(hole, board, npl, (P, B), rank, world, deal_mode=deal) if by_trial else None

    def step(i):
        if by_trial:
            return job.step(T, 1000 + i)                 # kernel on this rank's trial range + the count reduction
        both.zero_()
        npk.get_equity_batch(hole, board, npl, T, seed_value=1000 + i, deal_mode=deal, query_offset=q_off,
                             uniform_shape=(P, B), validate=False, out=out)
        return both

    for i in range(warmup):
        step(i)
    cx.barrier()
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
    ends = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
    sampler = ClockSampler(cx.local_rank)
    sampler.start()
    if by_trial:
        # The ranks leave the host-side set-up above milliseconds apart, and a sharded step is a barrier between the GPUs:
        # without this the early ranks' first timed step would be charged the late ranks' set-up.  One untimed step after a
        # host barrier lines the GPUs' queues up on the device.
        cx.barrier()
        step(warmup)
    torch.cuda.synchronize()
    wall0 = time.perf_counter()
    res = both
    for i in range(steps):
        if flush:
            flush_buf.fill_(i & 0xFF)                      # evict L2 between timed steps (outside the events)
        starts[i].record()
        res = step(warmup + i)
        ends[i].record()
    torch.cuda.synchronize()
    wall = time.perf_counter() - wall0
    clocks = sampler.stop()
    cx.barrier()
    dev_ms = cx.max_over_ranks(sum(s.elapsed_time(e) for s, e in zip(starts, ends)))
    last = res.cpu().numpy()          # [2, Q] wins / ties of the last timed step, read before the e2e leg reuses the job's buffers
    check_eq = float((res[0] + res[1]).double().mean().item() / T)
    evals_per_step = Q * T * P * (1 if by_trial else world)      # whole job, all ranks
    value = evals_per_step * steps / (dev_ms * 1e-3)
    kernel_ms = dev_ms / steps
    a_instr = algorithmic_instr(P, B)
    kname = ("equity_uniform_kernel<%d,%d>" if deal == "uniform" else "equity_refdeal_kernel<%d,%d>") % (P - 1, 5 - B)
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": warmup,
        "ms_per_step": kernel_ms, "higher_is_better": True, "scaling": "strong" if wl["shard"] == "trial" else "weak",
        "vs_baseline": None, "dtype": "u32", "data": "synthetic",
        "config": {"workload": wl["name"], "queries_per_gpu": Q, "trials": T, "players": P, "known_board_cards": B,
                   "deal_mode": deal, "sharding": ((job.describe() if by_trial else "one rank: the whole trial range")
                                                   if wl["shard"] == "trial" else "query blocks, no collective"),
                   "l2": ("flushed (256 MiB fill) between timed steps; " if flush else "not flushed; ") + "inputs are %d B" % (8 * Q),
                   "mean_equity": check_eq, "wall_s_timed_loop": wall,
                   "device_timed_call": "get_equity_batch(uniform_shape=(P,B), validate=False): query validation and shape "
                                        "classification are skipped in `value`; the e2e leg validates every query on the host"},
        "clocks": clocks, "gpu_launches": steps * (job.launches_per_step if by_trial else 1),
    }
    if peak:
        achieved = Q * t_cnt * a_instr / (kernel_ms * 1e-3)          # per GPU
        line["roofline"] = {"bound": "int_issue", "achieved": achieved / 1e12, "peak": peak / 1e12, "unit": "Tthread-instr/s",
                            "frac": achieved / peak, "traffic": None, "kernel": kname, "algorithmic_instr_per_trial": a_instr,
                            "peak_source": "npk_int_peak measured in this run", "peak_variants": peak_detail,
                            "nominal_issue_peak": 148 * 128 * 1.965e9 / 1e12}
    if e2e:
        # end to end through the host-buffer API: queries in host memory, counters back in host memory, every step
        # (for query-sharded workloads: two batches in flight per rank -- submit batch i+1, then collect batch i -- so the
        # staging and the copies overlap the previous kernel; every step still copies its queries H2D from pinned staging
        # and its counters D2H inside the timed region; the blocking one-call-per-step figure is reported next to it)
        e2e_steps = 100 if steps >= 10 else max(3, steps)        # 50 ms per leg: a 10 ms window is at the mercy of host jitter
        for i in range(5):                                # every staging slot of the library allocated before the clock starts
            npk.equity_counts_batch(hole_h, board_h, npl_h, t_cnt, seed_value=5000 + i, deal_mode=deal)
        cx.barrier()
        pinned = [torch.as_tensor(x).pin_memory() for x in (hole_h, board_h, npl_h)]
        e0 = time.perf_counter()
        for i in range(e2e_steps):
            if by_trial:
                # a trial shard of a larger job: host queries -> device, this rank's trial range, the count reduction,
                # totals back to the host (the host-buffer C entry point has no trial offset)
                job.load(*(x.to(dev, non_blocking=True) for x in pinned))
                r = job.step(T, 6000 + i).cpu()
            else:
                r = npk.equity_counts_batch(hole_h, board_h, npl_h, t_cnt, seed_value=6000 + i, deal_mode=deal)
        e2e_s = cx.max_over_ranks(time.perf_counter() - e0)
        line["e2e"] = {"value": Q * t_cnt * P * world * e2e_steps / e2e_s, "unit": UNIT, "h2d_bytes_per_step": int(8 * Q),
                       "d2h_bytes_per_step": int(16 * Q), "steps": e2e_steps,
                       "api": ("pinned host queries -> TrialShardedJob.step (trial shard + count reduction) -> host" if by_trial
                               else "neuron_poker_b200.equity_counts_batch -> npk_equity_host")}
        if not by_trial:
            for w in [npk.equity_counts_batch(hole_h, board_h, npl_h, t_cnt, seed_value=5100 + i, deal_mode=deal, block=False)
                      for i in range(npk.equity.MAX_IN_FLIGHT)]:
                w.result()                                # every staging slot allocated before the clock starts
            cx.barrier()
            pend, check = [], None
            e0 = time.perf_counter()
            for i in range(e2e_steps):
                pend.append(npk.equity_counts_batch(hole_h, board_h, npl_h, t_cnt, seed_value=6000 + i, deal_mode=deal,
                                                    block=False))
                if len(pend) > 1:
                    check = pend.pop(0).result()
            while pend:
                check = pend.pop(0).result()
            piped_s = cx.max_over_ranks(time.perf_counter() - e0)
            assert (check["wins"] == r["wins"]).all() and (check["ties"] == r["ties"]).all()     # same seed as the last blocking step
            line["e2e"].update({"blocking_value": line["e2e"]["value"], "value": Q * t_cnt * P * world * e2e_steps / piped_s,
                                "in_flight": 2,
                                "note": "can exceed `value`: the steps of this leg run back to back (no L2 flush between them) "
                                        "and the kernels of consecutive batches, on two streams, fill each other's tails",
                                "api": "neuron_poker_b200.equity_counts_batch(block=False) -> npk_equity_host_submit / "
                                       "npk_equity_host_wait, two batches in flight; blocking_value = one blocking "
                                       "npk_equity_host call per step"})
    return line, (hole_h, board_h, npl_h), last


def run_strong(args, cx, deal="uniform", steps=10):
    """cfg4 at this world size: strong scaling.  Times (a) the trial-sharded step with the count reduction inside,
    (b) the unsharded job on one GPU (every rank runs it, nothing is exchanged), and asserts on the device that the reduced
    counters of the sharded run equal the unsharded ones bit for bit for the same seed."""
    import torch
    import neuron_poker_b200 as npk
    wl = workload("cfg4")
    sharded, _, _ = run_mc(args, wl, cx, deal, steps, 3, e2e=False, flush=False)
    one = Ctx(0, 1, cx.local_rank, cx.dev, cx.L)                # the same job, whole trial range, this GPU alone
    alone, _, _ = run_mc(args, wl, one, deal, max(3, steps // 2), 2, e2e=False, flush=False)
    t1 = cx.max_over_ranks(alone["ms_per_step"])
    hole_h, board_h, npl_h = make_queries(wl, 1, 0)
    hole, board, npl = (torch.as_tensor(x).to(cx.dev) for x in (hole_h, board_h, npl_h))
    T, P, B = wl["trials"] // 10, wl["players"], wl["known"]
    ref = npk.get_equity_batch(hole, board, npl, T, seed_value=77, deal_mode=deal, uniform_shape=(P, B), validate=False)
    job = npk.dist.TrialShardedJob(hole, board, npl, (P, B), cx.rank, cx.world, deal_mode=deal)
    got = job.step(T, 77)
    same = bool(torch.equal(got[0], ref["wins"]) and torch.equal(got[1], ref["ties"]))
    same = cx.max_over_ranks(0.0 if same else 1.0) == 0.0
    assert same, "trial-sharded counters differ from the unsharded run"
    # where the time of a sharded step goes: this rank's trial range through the plain entry point (memset + kernel, no
    # exchange), timed the same way
    t_off, t_cnt = npk.dist.trial_shard(wl["trials"], cx.rank, cx.world)
    both = torch.zeros((2, len(hole_h)), dtype=torch.int64, device=cx.dev)
    share = {"wins": both[0], "ties": both[1]}
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    for i in range(steps + 2):
        if i == 2:
            ev[0].record()
        npk.get_equity_batch(hole, board, npl, t_cnt, seed_value=500 + i, deal_mode=deal, trial_offset=t_off,
                             uniform_shape=(P, B), validate=False, out=share)
    ev[1].record()
    torch.cuda.synchronize()
    share_ms = cx.max_over_ranks(ev[0].elapsed_time(ev[1])) / steps
    sharded["strong_scaling"] = {"ms_per_step_one_gpu_unsharded": t1, "ms_per_step_sharded": sharded["ms_per_step"],
                                 "efficiency": t1 / (cx.world * sharded["ms_per_step"]), "n_gpus": cx.world,
                                 "ms_per_step_share_without_exchange": share_ms,
                                 "exchange_and_skew_ms": sharded["ms_per_step"] - share_ms,
                                 "sharded_equals_unsharded_bit_exact": same,
                                 "check": "169 classes x %d trials, seed 77: reduced [2,169] counters of the %d-way trial "
                                          "split == one-GPU counters (torch.equal on the device, all ranks)" % (T, cx.world),
                                 "reduction": job.describe()}
    return sharded


def run_sustained(args, cx, deal="uniform", seconds=3.0):
    """The cfg3 step launched back to back for >= `seconds` of device time (no L2 flush, no host synchronisation inside):
    what the part sustains once power and thermals have settled, with its own clock samples."""
    import torch
    import neuron_poker_b200 as npk
    wl = workload("cfg3")
    hole_h, board_h, npl_h = make_queries(wl, cx.world, cx.rank)
    Q, T, P, B = len(hole_h), wl["trials"], wl["players"], wl["known"]
    hole, board, npl = (torch.as_tensor(x).to(cx.dev) for x in (hole_h, board_h, npl_h))
    both = torch.zeros((2, Q), dtype=torch.int64, device=cx.dev)
    out = {"wins": both[0], "ties": both[1]}

    def step(i):
        npk.get_equity_batch(hole, board, npl, T, seed_value=9000 + i, deal_mode=deal, query_offset=cx.rank * Q,
                             uniform_shape=(P, B), validate=False, out=out)

    for i in range(5):
        step(i)
    cx.barrier()
    n = int(seconds / 0.5e-3 * 1.15)
    sampler = ClockSampler(cx.local_rank)
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(n):
        step(i)
    e1.record()
    torch.cuda.synchronize()
    clocks = sampler.stop()
    ms = cx.max_over_ranks(e0.elapsed_time(e1))
    total = int(both.sum().item())
    assert 0 < total <= (5 + n) * Q * T
    return {"value": Q * T * P * cx.world * n / (ms * 1e-3), "unit": UNIT, "steps": n, "seconds": ms * 1e-3,
            "ms_per_step": ms / n, "clocks": clocks, "deal_mode": deal,
            "note": "back-to-back launches of the cfg3 step, counters accumulate (no reset, no L2 flush: the step reads 28 KB "
                    "of queries and 131 KB of tables per CTA)"}


def dump_outputs(directory, last):
    """What get_equity_batch handed back in the headline's last timed step: wins [Q] and ties [Q] of every query, as
    float64 (exact: the counts are far below 2**53).  The queries and the step's seed follow from the arguments alone."""
    import numpy as np
    os.makedirs(directory, exist_ok=True)
    for name, row in zip(("wins", "ties"), last):
        np.save(os.path.join(directory, name + ".npy"), row.astype(np.float64))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=300)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="all")
    ap.add_argument("--deal", default="uniform", choices=["uniform", "reference"])
    ap.add_argument("--deal-ranges", dest="deal_ranges", default="reference", choices=["uniform", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="cfg3 headline only (profiling runs)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write wins.npy and ties.npy (float64, one entry per query of rank 0) of the headline's last timed "
                         "step to DIR, to compare two builds output for output")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "b200" or args.workload not in ("all", "cfg3")):
        ap.error("--dump-outputs writes the counters of the cfg3 headline: use it with --workload all or cfg3")
    everything = args.workload == "all"
    wl = workload("cfg3" if everything else args.workload)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference_arm(args, wl, rank)
        return

    import torch
    import torch.distributed as dist
    from neuron_poker_b200 import _lib

    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    torch.cuda.set_device(local_rank)
    os.environ["NPK_DEVICE"] = str(local_rank)
    dev = torch.device("cuda", local_rank)
    L = _lib.ensure_init(local_rank)
    cx = Ctx(rank, world, local_rank, dev, L)
    with_cpu = rank == 0 and world == 1 and not args.no_cpu_baseline

    def finish(line):
        if rank == 0:
            print(json.dumps(line), flush=True)
        if world > 1:
            dist.destroy_process_group()

    if args.workload == "cfg2":
        return finish(run_exact(args, wl, cx))
    if args.workload == "cfg5":
        return finish(run_selfplay(args, wl, cx, args.deal))
    if args.workload == "ranges":
        return finish(run_ranges(args, wl, cx))
    if args.workload == "cfg1":
        return finish({"metric": "get_equity_latency", "config": {"workload": wl["name"]}, **run_latency(args, wl, cx, with_cpu)})
    if args.workload == "cfg4":
        line = run_strong(args, cx, args.deal, steps=args.steps)
        return finish(line)

    peak, peak_detail = int_issue_peak(L)
    line, (hole_h, board_h, npl_h), last = run_mc(args, wl, cx, args.deal, args.steps, max(3, args.warmup), peak, peak_detail)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last)
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            t_rec = json.load(f).get(line["roofline"]["kernel"])
        if t_rec:
            line["roofline"]["traffic"] = t_rec["dram_bytes_read"] + t_rec["dram_bytes_write"]
            line["roofline"]["traffic_note"] = ("DRAM bytes per launch from the committed ncu --set full capture "
                                                "(profiles/ncu_traffic.json); the kernel is bound by integer issue and shared "
                                                "memory, not HBM")
    except Exception:
        pass
    if not (everything and not args.no_extras):
        if with_cpu:
            line["cpu_baseline"] = cpu_baselines(wl, hole_h, board_h, npl_h)
        return finish(line)

    # ---- everything else BASELINE.json names, in the same run -------------------------------------------------------
    line["sustained"] = run_sustained(args, cx, args.deal)
    extras = {}
    lat = run_latency(args, workload("cfg1"), cx, with_cpu) if rank == 0 else None
    line["get_equity_calls_per_s"] = lat["get_equity_6_players_flop"]["calls_per_s"] if lat else None
    line["get_equity_calls_per_s_resident_mode"] = lat["get_equity_6_players_flop"]["resident"]["calls_per_s"] if lat else None
    extras["cfg1"] = lat
    cx.barrier()

    def brief(rec, keep=("value", "unit", "ms_per_step", "steps", "scaling", "config", "roofline", "e2e", "strong_scaling",
                         "gpu_launches", "clocks", "kernel")):
        return {k: rec[k] for k in keep if k in rec}

    extras["cfg2"] = brief(run_exact(args, workload("cfg2"), cx, steps=10))
    ref3, _, _ = run_mc(args, workload("cfg3"), cx, "reference", 20, 3, peak, peak_detail, e2e=False)
    extras["cfg3_reference_dealer"] = brief(ref3)
    extras["cfg4"] = brief(run_strong(args, cx, "uniform", steps=20))
    extras["cfg4_reference_dealer"] = brief(run_strong(args, cx, "reference", steps=10))
    extras["cfg5_uniform"] = brief(run_selfplay(args, workload("cfg5"), cx, "uniform", steps=120))
    extras["cfg5_reference_dealer"] = brief(run_selfplay(args, workload("cfg5"), cx, "reference", steps=120))
    extras["ranges"] = brief(run_ranges(args, workload("ranges"), cx, steps=5))
    line["workloads"] = extras
    if with_cpu:
        line["cpu_baseline"] = cpu_baselines(wl, hole_h, board_h, npl_h)
    finish(line)


if __name__ == "__main__":
    main()
