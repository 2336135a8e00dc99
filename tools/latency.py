"""Latency of one blocking get_equity call (10,000 runs, 6 players, flop), launched per call and through the resident server."""
import sys, os, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import neuron_poker_b200 as npk
for mode, fn in (("reference", lambda: npk.get_equity({"AS", "KS"}, {"2C", "7D", "KH"}, 6, 10000)),
                 ("uniform", lambda: npk.montecarlo({"AS", "KS"}, {"2C", "7D", "KH"}, 6, 10000))):
    for _ in range(50): fn()
    t0 = time.perf_counter(); n = 2000
    vals = [fn() for _ in range(n)]
    dt = time.perf_counter() - t0
    print(mode, "%.1f us/call  %.0f calls/s  mean equity %.4f" % (1e6 * dt / n, n / dt, sum(vals) / n), flush=True)
# the same calls with the resident server (no kernel launch per call)
import ctypes
for sms in (0, 64, 16):
    npk.resident(True, sms=sms, idle_us=1000)
    for mode, fn in (("reference", lambda: npk.get_equity({"AS", "KS"}, {"2C", "7D", "KH"}, 6, 10000)),
                     ("uniform", lambda: npk.montecarlo({"AS", "KS"}, {"2C", "7D", "KH"}, 6, 10000))):
        for _ in range(50): fn()
        t0 = time.perf_counter(); n = 4000
        vals = [fn() for _ in range(n)]
        dt = time.perf_counter() - t0
        print("resident sms=%d" % sms, mode, "%.1f us/call  %.0f calls/s  mean equity %.4f" % (1e6 * dt / n, n / dt, sum(vals) / n), flush=True)
    L = npk._lib.lib()
    out = (ctypes.c_uint64 * 12)()
    packed = npk.equity._pack_query({"AS", "KS"}, {"2C", "7D", "KH"})
    for trials in (10000, 1000, 64):
        for _ in range(50): L.npk_equity_one(packed, 6, trials, 1, 1, 0, out)
        t0 = time.perf_counter(); n = 4000
        for i in range(n): L.npk_equity_one(packed, 6, trials, i, 1, 0, out)
        dt = time.perf_counter() - t0
        print("resident sms=%d npk_equity_one via ctypes, %5d trials: %.2f us/call" % (sms, trials, 1e6 * dt / n), flush=True)
    npk.resident(False)
