"""Every kernel of libnpk once, at sizes compute-sanitizer finishes in minutes (SURVEY 5: racecheck / memcheck / synccheck
on the shared-memory staging, the per-warp decks and the reductions).  Run as
    compute-sanitizer --tool memcheck|racecheck|synccheck|initcheck python tools/sanitizer_workload.py
or, where compute-sanitizer is not available (it is closed on the pool this was built on, profiles/r02_compute_sanitizer_closed.txt),
against the library's own checked build:
    bash tools/checked_build.sh && NPK_LIBRARY=$PWD/neuron_poker_b200/build/libnpk_checked.so python tools/sanitizer_workload.py
The results are checked for self-consistency only (wins + ties <= trials, enumeration totals); parity is tests/'s job."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import neuron_poker_b200 as npk
from neuron_poker_b200.holdem import EquityAgents, HoldemTables

QUICK = os.environ.get("NPK_SANITIZE_QUICK") == "1"
rng = np.random.default_rng(5)


def deal(n, k):
    return np.stack([rng.permutation(52)[:k] for _ in range(n)]).astype(np.uint8)


def queries(n, known, players):
    c = deal(n, 2 + known)
    board = np.full((n, 5), 255, dtype=np.uint8)
    board[:, :known] = c[:, 2:]
    return c[:, :2].copy(), board, np.full(n, players, dtype=np.uint8)


def check(out, trials, what):
    torch.cuda.synchronize()
    w, t = out["wins"].cpu().numpy(), out["ties"].cpu().numpy()
    assert ((w + t) <= trials).all() and (w + t).sum() > 0, what
    print("ok", what, flush=True)


# K2 / K4
h = deal(1031, 7)
r = npk.rank7(h).cpu().numpy()
assert (r == npk.host_rank7(h)).all()
r2 = npk.rank7_colex(1000, 3000).cpu().numpy()
assert r2.shape == (3000,)
holes = deal(257, 12).reshape(257, 6, 2)
npl = rng.integers(2, 7, 257).astype(np.uint8)
brd = np.stack([np.setdiff1d(np.arange(52, dtype=np.uint8), holes[i].ravel())[:5] for i in range(257)])
win, ty = npk.showdown(holes, npl, brd)[:2]
torch.cuda.synchronize()
print("ok rank7 / rank7_colex / showdown", flush=True)

# K3: river, turn, flop (generic walk), three players on the river
for known, players, n in ((5, 2, 9), (4, 2, 5), (3, 2, 1 if QUICK else 2), (5, 3, 2)):
    ho, bo, pl = queries(n, known, players)
    w, t, l = npk.enumerate_equity(ho, bo, pl)
    torch.cuda.synchronize()
    assert int((w + t + l).min()) > 0
print("ok enumerate_equity", flush=True)

# K1 / K1': a few shapes, odd trial counts, offsets, win types, passes
for mode in ("uniform", "reference"):
    for players, known in ((6, 3), (2, 0), (9, 0), (3, 5), (1, 4), (10, 3)):
        ho, bo, pl = queries(7, known, players)
        out = npk.get_equity_batch(ho, bo, pl, 777, seed_value=3, deal_mode=mode, uniform_shape=(players, known),
                                   win_types=True, passes=mode == "reference", trial_offset=5, query_offset=11)
        check(out, 777, "%s P=%d known=%d" % (mode, players, known))
    # mixed batch, classified on the host and sync-free
    parts = [queries(5, k, p) for p, k in ((2, 0), (6, 3), (3, 4), (4, 5), (6, 0))]
    ho, bo, pl = (np.concatenate([x[i] for x in parts]) for i in range(3))
    check(npk.get_equity_batch(ho, bo, pl, 300, seed_value=4, deal_mode=mode), 300, mode + " mixed")
    check(npk.get_equity_batch(ho, bo, pl, 300, seed_value=4, deal_mode=mode,
                               shapes=npk.equity.shape_mask(range(2, 7))), 300, mode + " mixed sync-free")
    # to a target precision: rounds of the all-shapes kernel on the queries still active, retired on the device
    ad = npk.get_equity_batch_adaptive(ho, bo, pl, 700, 0.03, min_trials=64, seed_value=4, deal_mode=mode, win_types=True,
                                       passes=mode == "reference")
    torch.cuda.synchronize()
    tr = ad["trials"].cpu().numpy()
    assert ((tr >= 64) & (tr <= 700)).all() and ((ad["wins"] + ad["ties"]).cpu().numpy() <= tr).all(), mode + " adaptive"
    print("ok", mode, "adaptive", flush=True)
    # host-buffer entry point: one-query fast path and the staged path
    for _ in range(3):
        c = npk.equity_counts({"AS", "KS"}, {"2C", "7D", "KH"}, 6, 1000, deal_mode=mode, win_types=True, passes=True)
        assert 0 < c["wins"] + c["ties"] <= 1000
    o = npk.equity_counts_batch(ho, bo, pl, 200, seed_value=9, deal_mode=mode, win_types=True)
    assert ((o["wins"] + o["ties"]) <= 200).all()
    # the launched one-query call with the packed hand-over, the resident server (same counters), batches in flight
    one = [npk.equity_counts({"AS", "KS"}, {"2C", "7D", "KH"}, p_, 3000, deal_mode=mode, seed_value=8) for p_ in (2, 6, 10)]
    npk.resident(True, idle_us=500)
    res = [npk.equity_counts({"AS", "KS"}, {"2C", "7D", "KH"}, p_, 3000, deal_mode=mode, seed_value=8) for p_ in (2, 6, 10)]
    npk.resident(False)
    assert one == res, (one, res)
    pend = [npk.equity_counts_batch(ho, bo, pl, 200, seed_value=9, deal_mode=mode, win_types=True, block=False) for _ in range(3)]
    for pnd in pend:
        r_ = pnd.result()
        assert (r_["wins"] == o["wins"]).all() and (r_["win_types"] == o["win_types"]).all()
    print("ok host entry points", mode, flush=True)

# K1'': ranges, hero range, ghost cards
ho, bo, pl = queries(6, 3, 4)
for mode in ("reference", "uniform"):
    check(npk.get_equity_ranges_batch(ho, bo, pl, 400, opponent_range=0.3, seed_value=2, deal_mode=mode, win_types=True,
                                      passes=True), 400, "ranges " + mode)
    gh = np.full((6, 2), 255, dtype=np.uint8)
    check(npk.get_equity_ranges_batch(None, bo, pl, 400, opponent_range={"AKS", "QQ", "77", "T9O"}, hero_range={"AA", "KK", "AKO"},
                                      ghost=gh, seed_value=2, deal_mode=mode), 400, "hero range " + mode)
mc = npk.MonteCarlo()
mc.run_montecarlo([["AS", "KS"]], ["2C", "7D", "KH"], 3, 1, 500, 0, ghost_cards=["2D", "3D"], opponent_range=0.2)
print("ok run_montecarlo with ranges", mc.equity, flush=True)
mc.run_montecarlo([["AS", "KS"], ["QH", "QD"], ["7C", "2D"]], ["2C", "7D", "KH"], 5, 1, 500, 0, ghost_cards='', opponent_range=0.5)
kn = np.tile(np.array([[[40, 41], [2, 7]]], dtype=np.uint8), (6, 1, 1))
ho2 = np.tile(np.array([[51, 47]], dtype=np.uint8), (6, 1)); bo2 = np.full((6, 5), 255, dtype=np.uint8)
for mode in ("reference", "uniform"):
    check(npk.get_equity_ranges_batch(ho2, bo2, np.full(6, 4, dtype=np.uint8), 400, opponent_range=0.4, seed_value=6,
                                      deal_mode=mode, known_opponents=kn, passes=mode == "reference"), 400, "known hands " + mode)
print("ok known opponent hands", mc.equity, flush=True)
# ranges to a target precision: rounds of both range kernels on the device-listed queries still active
ho3, bo3, pl3 = queries(64, 4, 5)
pl3[::4] = 1                                                        # retire at T_0: later rounds list a subset
for mode in ("reference", "uniform"):
    for passes in (True, False):
        ad = npk.get_equity_ranges_batch_adaptive(ho3, bo3, pl3, 700, 0.03, min_trials=64, opponent_range=0.3, seed_value=8,
                                                  deal_mode=mode, win_types=True, passes=passes)
        torch.cuda.synchronize()
        tr = ad["trials"].cpu().numpy()
        assert ((tr >= 64) & (tr <= 700)).all() and ((ad["wins"] + ad["ties"]).cpu().numpy() <= tr).all(), mode
        assert (tr[::4] == 64).all() and (tr > 64).any(), mode
print("ok adaptive ranges", flush=True)

# exact showdown equity of known hands: every player count and board size, dead cards, both dealers, garbage bytes
se_h = np.full((40, 10, 2), 255, dtype=np.uint8); se_b = np.full((40, 5), 255, dtype=np.uint8)
se_d = np.full((40, 2), 255, dtype=np.uint8); se_n = np.zeros(40, dtype=np.uint8)
for i in range(40):
    P, nb = 1 + i % 10, (3, 4, 5, 3)[i // 10]
    c = rng.permutation(52)[:2 * P + nb + 2]
    se_h[i, :P] = c[:2 * P].reshape(P, 2); se_b[i, :nb] = c[2 * P:2 * P + nb]; se_d[i] = c[2 * P + nb:]; se_n[i] = P
for mode in ("uniform", "reference"):
    o = npk.showdown_equity_batch(se_h, se_n, se_b, se_d, deal_mode=mode)
    assert (o["share"].sum(dim=1) == 2520 * o["completions"]).all()
npk.showdown_equity([["AS", "KS"], ["QH", "QD"], ["7C", "2D"]], ["2C"])
npk.showdown_equity_batch(torch.randint(0, 256, (256, 10, 2), dtype=torch.uint8, device="cuda"),
                          torch.randint(0, 256, (256,), dtype=torch.uint8, device="cuda"),
                          torch.randint(0, 256, (256, 5), dtype=torch.uint8, device="cuda"),
                          torch.randint(0, 256, (256, 3), dtype=torch.uint8, device="cuda"))
torch.cuda.synchronize()
print("ok showdown equity", flush=True)

# exact equity against one or two unknown opponents: known hands, every board size, dead cards, both dealers, garbage bytes
ee_h = np.full((48, 4, 2), 255, dtype=np.uint8); ee_b = np.full((48, 5), 255, dtype=np.uint8)
ee_d = np.full((48, 2), 255, dtype=np.uint8); ee_k = np.zeros(48, dtype=np.uint8); ee_r = np.zeros(48, dtype=np.uint8)
for i in range(48):
    K, k, nb = 1 + i % 4, 1 + (i // 4) % 2, (5, 4, 3, 5, 4, 0)[i // 8]
    k = 1 if nb < 4 else k
    c = rng.permutation(52)[:2 * K + nb + 2]
    ee_h[i, :K] = c[:2 * K].reshape(K, 2); ee_b[i, :nb] = c[2 * K:2 * K + nb]; ee_d[i] = c[2 * K + nb:]
    ee_k[i], ee_r[i] = K, k
for mode in ("uniform", "reference"):
    o = npk.exact_equity_batch(ee_h, ee_k, ee_r, ee_b, ee_d, deal_mode=mode)
    assert ((o["win"] + o["tie"] + o["lose"]) > 0).all()
npk.exact_equity_batch(torch.randint(0, 256, (256, 8, 2), dtype=torch.uint8, device="cuda"),
                       torch.randint(0, 256, (256,), dtype=torch.uint8, device="cuda"),
                       torch.randint(0, 4, (256,), dtype=torch.uint8, device="cuda"),
                       torch.randint(0, 256, (256, 5), dtype=torch.uint8, device="cuda"),
                       torch.randint(0, 256, (256, 3), dtype=torch.uint8, device="cuda"))
torch.cuda.synchronize()
print("ok exact equity", flush=True)

# win-type histograms of both exact engines: the same spots and garbage bytes
for mode in ("uniform", "reference"):
    o = npk.exact_equity_batch(ee_h, ee_k, ee_r, ee_b, ee_d, deal_mode=mode, win_types=True)
    assert (o["win_types"].sum(dim=1) == o["win"] + o["tie"]).all()
    o = npk.showdown_equity_batch(se_h, se_n, se_b, se_d, deal_mode=mode, win_types=True)
    assert (o["win_types"].sum(dim=2) == o["win"] + o["tie"]).all()
npk.exact_equity_batch(torch.randint(0, 256, (256, 8, 2), dtype=torch.uint8, device="cuda"),
                       torch.randint(0, 256, (256,), dtype=torch.uint8, device="cuda"),
                       torch.randint(0, 4, (256,), dtype=torch.uint8, device="cuda"),
                       torch.randint(0, 256, (256, 5), dtype=torch.uint8, device="cuda"),
                       torch.randint(0, 256, (256, 3), dtype=torch.uint8, device="cuda"), win_types=True)
npk.showdown_equity_batch(torch.randint(0, 256, (256, 10, 2), dtype=torch.uint8, device="cuda"),
                          torch.randint(0, 256, (256,), dtype=torch.uint8, device="cuda"),
                          torch.randint(0, 256, (256, 5), dtype=torch.uint8, device="cuda"),
                          torch.randint(0, 256, (256, 3), dtype=torch.uint8, device="cuda"), win_types=True)
torch.cuda.synchronize()
print("ok exact win types", flush=True)

# vectorised HoldemTable: self-play with both dealers, observation vector, showdowns
tb = HoldemTables(96, n_players=6, seed=3, autoplay=[1] * 6)
tb.enable_observations()
agents = EquityAgents.equity_vs_random()
for i in range(6 if QUICK else 25):
    tb.selfplay_step(agents, runs=64, deal_mode="reference" if i & 1 else "uniform", stderr=0.05 if i % 3 == 2 else None)
    tb.observe()
torch.cuda.synchronize()
st = tb.state()
assert int((st["error"] != 0).sum()) == 0
print("ok holdem self-play", flush=True)
import ctypes
from neuron_poker_b200 import _lib
L = _lib.ensure_init(0)
checked, code = ctypes.c_int(0), ctypes.c_uint32(0)
_lib.check(L.npk_checked_status(ctypes.byref(checked), ctypes.byref(code)))
print("checked build: %d   first failed NPK_CHECK: %d" % (checked.value, code.value))
assert code.value == 0
print("sanitizer workload finished")
