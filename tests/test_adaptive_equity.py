"""Monte-Carlo equity to a target precision (npk_equity_batch_adaptive / get_equity_batch_adaptive).

A query of an adaptive call stops at the first checkpoint T_k (T_0 = min_trials, doubling, capped at max_trials) where the
add-one variance p (1 - p) / T_k, p = (wins + ties + 1) / (T_k + 2), is at most stderr^2.  Since trial t of query q is the
same Philox stream in every Monte-Carlo call, its counters must be EXACTLY those of get_equity_batch(trials=T_stop) with the
same seed: that is what the GPU tests check, bit for bit, together with the decision itself (restated on the host in double
arithmetic, in the device's order of operations), its boundary, its independence from the rest of the batch, the device-side
item plan at production item sizes, graph capture, and the self-play consumer.
"""
import ctypes
import math

import numpy as np
import pytest

from neuron_poker_b200 import _lib, cards
from neuron_poker_b200.equity import adaptive_checkpoints, adaptive_stops

NO = 0xFF


# ---- CPU ---------------------------------------------------------------------------------------------------------------
def test_checkpoint_schedule():
    assert adaptive_checkpoints(256, 256) == [256]
    assert adaptive_checkpoints(256, 1000) == [256, 512, 1000]                  # max not min * 2^k: the last step is short
    assert adaptive_checkpoints(256, 1024) == [256, 512, 1024]
    assert adaptive_checkpoints(1, 10) == [1, 2, 4, 8, 10]
    assert adaptive_checkpoints(1, 1) == [1]
    assert adaptive_checkpoints(3, 7) == [3, 6, 7]
    t = adaptive_checkpoints(1, 2**62 + 1)
    assert t[-1] == 2**62 + 1 and t[-2] == 2**62 and len(t) == 64
    for bad in ((0, 10), (11, 10), (-1, 5)):
        with pytest.raises(ValueError):
            adaptive_checkpoints(*bad)


def test_host_rule_restates_the_formula():
    """adaptive_stops is var <= s*s with var = p (1 - p) / T, p = (x + 1) / (T + 2): against exact rationals away from the
    boundary, and the known answer of x = T (players = 1, a made royal flush): var = (T + 1) / ((T + 2)^2 T)."""
    from fractions import Fraction
    rng = np.random.default_rng(3)
    for _ in range(2000):
        T = int(rng.integers(1, 10**7))
        x = int(rng.integers(0, T + 1))
        s = float(rng.uniform(1e-4, 0.2))
        p = Fraction(x + 1, T + 2)
        var = p * (1 - p) / T
        s2 = Fraction(s) * Fraction(s)
        if abs(var - s2) > s2 * Fraction(1, 10**9):                          # far from the boundary: no rounding question
            assert adaptive_stops(x, T, s) == (var <= s2), (x, T, s)
    for T in (1, 64, 256, 1000, 2**20):          # (1 - p in doubles loses about eps / (1 - p) relative: 2e-10 at T = 2^20)
        var = (T + 1) / ((T + 2) ** 2 * T)
        assert adaptive_stops(T, T, math.sqrt(var) * (1 + 1e-6))
        assert not adaptive_stops(T, T, math.sqrt(var) * (1 - 1e-6))
        assert adaptive_stops(0, T, math.sqrt(var) * (1 + 1e-6))             # symmetric: x = 0 has the same variance


def _adaptive_call(stderr, min_trials, max_trials):
    L = _lib.lib()
    rc = L.npk_equity_batch_adaptive(None, None, None, 1, int(min_trials), int(max_trials), ctypes.c_double(stderr),
                                     ctypes.c_uint64(2**60 - 1), ctypes.c_uint64(0), 0, 0, 0, None, None, None, None, None,
                                     None, None)
    return rc, L.npk_last_error().decode()


def test_argument_errors_need_no_device():
    """The rule's arguments are checked before the device is touched: each error has its own message."""
    msgs = set()
    for args in ((float("nan"), 64, 128), (float("inf"), 64, 128), (0.0, 64, 128), (-0.01, 64, 128), (-0.0, 64, 128)):
        rc, msg = _adaptive_call(*args)
        assert rc == -2 and "stderr" in msg, (args, rc, msg)
        msgs.add(msg)
    rc, msg = _adaptive_call(0.01, 0, 128)
    assert rc == -2 and "min_trials must be >= 1" in msg, msg
    msgs.add(msg)
    rc, msg = _adaptive_call(0.01, 129, 128)
    assert rc == -2 and "exceed max_trials" in msg, msg
    msgs.add(msg)
    assert len(msgs) == 3


def test_workspace_covers_the_fixed_call():
    L = _lib.lib()
    for Q in (0, 1, 4096, 65536):
        assert L.npk_equity_adaptive_workspace_bytes(Q) >= L.npk_equity_workspace_bytes(Q) + Q


# ---- GPU ---------------------------------------------------------------------------------------------------------------
def _mixed_batch(per_shape, seed):
    """per_shape random queries of every (players, known board cards) shape, then known answers: players = 1 (x = T) and a
    made royal flush for the hero (x = T) on every street and player count."""
    rng = np.random.default_rng(seed)
    hole, board, npl = [], [], []
    for players in range(1, 11):
        for known in range(6):
            for _ in range(per_shape):
                c = rng.permutation(52)[:2 + known]
                hole.append(c[:2])
                board.append(list(c[2:]) + [NO] * (5 - known))
                npl.append(players)
    royal = [cards.card_id(c) for c in ("AS", "KS", "QS", "JS", "TS", "2C", "3D")]
    for players in range(1, 11):
        for known in (3, 4, 5):
            hole.append(royal[:2])
            board.append(royal[2:2 + known] + [NO] * (5 - known))
            npl.append(players)
    return (np.array(hole, dtype=np.uint8), np.array(board, dtype=np.uint8), np.array(npl, dtype=np.uint8))


N_ROYAL = 30                                   # the last rows of _mixed_batch


def _x_equals_t(q):
    """Queries whose hero wins every trial: players = 1 and the made royal flushes."""
    m = q[2] == 1
    m[-N_ROYAL:] = True
    return m


def _np(t):
    return t.cpu().numpy()


def _fixed(q, T, seed, mode, query_offset=0):
    import neuron_poker_b200 as npk
    out = npk.get_equity_batch(*q, T, seed_value=seed, deal_mode=mode, win_types=True, passes=True, query_offset=query_offset)
    return {k: _np(out[k]) for k in ("wins", "ties", "win_types", "passes")}


def _adaptive(q, max_trials, stderr, min_trials, seed, mode, **kw):
    import neuron_poker_b200 as npk
    out = npk.get_equity_batch_adaptive(*q, max_trials, stderr, min_trials=min_trials, seed_value=seed, deal_mode=mode,
                                        win_types=True, passes=True, **kw)
    return {k: _np(v) for k, v in out.items()}


def _check_exact(ad, q, seed, mode, checkpoints, stderr):
    """Every query equals the fixed-trial run at its T_stop (wins, ties, win types, passes), and the host rule on the fixed
    counters continues at every earlier checkpoint and stops at T_stop (or T_stop = max_trials)."""
    fixed = {T: _fixed(q, T, seed, mode) for T in checkpoints}
    stops = ad["trials"]
    assert set(np.unique(stops)) <= set(checkpoints), np.unique(stops)
    for T in np.unique(stops):
        sel = stops == T
        for k in ("wins", "ties", "win_types", "passes"):
            assert (ad[k][sel] == fixed[T][k][sel]).all(), (mode, int(T), k)
    for i in range(len(stops)):
        for T in checkpoints:
            x = int(fixed[T]["wins"][i] + fixed[T]["ties"][i])
            stop = adaptive_stops(x, T, stderr) or T == checkpoints[-1]
            if T < stops[i]:
                assert not stop, (i, T, int(stops[i]))
            else:
                assert stop and T == stops[i], (i, T, int(stops[i]))
                break
    return fixed


# min 64, max 1024, stderr 0.02: x = T stops at T_0 (var = 65 / (66^2 * 64) = 2.33e-4 <= 4e-4); an equity of 0.5 reaches
# max_trials (0.25 / 512 > 4e-4); equities below about 0.05 / 0.12 / 0.29 (or above 1 minus those) stop by 128 / 256 / 512.
MIX = dict(min_trials=64, max_trials=1024, stderr=0.02)


@pytest.fixture(scope="module")
def mixed(cuda_device):
    return _mixed_batch(per_shape=20, seed=5)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["uniform", "reference"])
def test_bit_exact_against_fixed_trial_runs_and_rule_applied_exactly(mixed, mode):
    seed = 0x5eed0001 if mode == "uniform" else 0x5eed0002
    cps = adaptive_checkpoints(MIX["min_trials"], MIX["max_trials"])
    ad = _adaptive(mixed, MIX["max_trials"], MIX["stderr"], MIX["min_trials"], seed, mode)
    for T in cps:                                                         # the batch exercises every checkpoint
        assert (ad["trials"] == T).any(), (mode, T, np.unique(ad["trials"], return_counts=True))
    assert (ad["trials"][_x_equals_t(mixed)] == cps[0]).all()             # x = T stops at T_0
    _check_exact(ad, mixed, seed, mode, cps, MIX["stderr"])


def _predicted_stops(fixed, checkpoints, stderr, n):
    out = np.zeros(n, dtype=np.int64)
    for i in range(n):
        for T in checkpoints:
            if T == checkpoints[-1] or adaptive_stops(int(fixed[T]["wins"][i] + fixed[T]["ties"][i]), T, stderr):
                out[i] = T
                break
    return out


@pytest.mark.gpu
def test_boundary_of_the_rule(mixed):
    """s = sqrt(var) of a chosen query at a checkpoint, and the two doubles next to it: for every s the device stops every
    query exactly where the host rule var <= s*s says.  Known answers: x = T stops at T_0 iff s^2 >= (T_0+1)/((T_0+2)^2 T_0)."""
    mode, seed = "reference", 77
    cps = adaptive_checkpoints(MIX["min_trials"], MIX["max_trials"])
    fixed = {T: _fixed(mixed, T, seed, mode) for T in cps}
    n = len(mixed[0])
    T0 = cps[0]
    v_known = (T0 + 1.0) / float((T0 + 2) ** 2) / float(T0)
    p = (T0 + 1.0) / float(T0 + 2)
    v_known_host = p * (1.0 - p) / float(T0)                             # the rule's own order of operations
    chosen = [v_known_host]
    x2 = fixed[cps[2]]["wins"] + fixed[cps[2]]["ties"]
    i = int(np.argmin(np.abs(x2 / cps[2] - 0.1)))                         # a query near an equity of 0.1 at the third checkpoint
    p = (float(x2[i]) + 1.0) / float(cps[2] + 2)
    chosen.append(p * (1.0 - p) / float(cps[2]))
    seen_sides = set()
    for var in chosen:
        s = math.sqrt(var)
        for sv in (np.nextafter(s, 0.0), s, np.nextafter(s, 1.0)):
            sv = float(sv)
            want = _predicted_stops(fixed, cps, sv, n)
            ad = _adaptive(mixed, MIX["max_trials"], sv, MIX["min_trials"], seed, mode)
            assert (ad["trials"] == want).all(), (sv, np.nonzero(ad["trials"] != want)[0][:5])
            seen_sides.add(var <= sv * sv)
            known = _x_equals_t(mixed)
            assert (ad["trials"][known] == (T0 if v_known_host <= sv * sv else cps[1])).all()
    assert seen_sides == {True, False}                                    # the neighbours fall on both sides of the boundary
    assert abs(v_known - v_known_host) <= 1e-15


@pytest.mark.gpu
def test_independent_of_the_rest_of_the_batch(mixed):
    """The batch split in two with query_offset equals the whole batch; a query keeps its counts when every other query of
    the batch is replaced by one that retires at T_0 (players = 1)."""
    mode, seed = "uniform", 1234
    args = (MIX["max_trials"], MIX["stderr"], MIX["min_trials"], seed, mode)
    whole = _adaptive(mixed, *args)
    h = len(mixed[0]) // 3
    a = _adaptive(tuple(x[:h] for x in mixed), *args)
    b = _adaptive(tuple(x[h:] for x in mixed), *args, query_offset=h)
    for k in whole:
        assert (np.concatenate([a[k], b[k]]) == whole[k]).all(), k
    keep = np.arange(len(mixed[0])) % 7 == 3
    hole, board, npl = (x.copy() for x in mixed)
    npl[~keep] = 1
    lone = _adaptive((hole, board, npl), *args)
    assert (lone["trials"][~keep] == MIX["min_trials"]).all()
    for k in whole:
        assert (lone[k][keep] == whole[k][keep]).all(), k


def _item_plan(queries, trials, sm_count):
    """npk::item_plan (csrc/npk_kernels.h): trials per work item of a launch."""
    c = (queries * trials) // (8 * sm_count * 16)
    c = max(64, min(2048, (c + 63) // 64 * 64))
    return trials if trials <= c else c


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["uniform", "reference"])
def test_production_item_sizes(cuda_device, mode):
    """A batch sized from the SM count: most queries (players = 1) retire at T_0 = 2,048, about 8 x SMs heads-up preflop
    queries run on, so that the device-planned later rounds cut 2,048-trial items -- and test 1 holds there too."""
    sm = _lib.ensure_init(0).npk_sm_count()
    rng = np.random.default_rng(8)
    n_run = 8 * sm + 64
    n_one = 4 * n_run
    hole = np.stack([rng.permutation(52)[:2] for _ in range(n_run + n_one)]).astype(np.uint8)
    board = np.full((n_run + n_one, 5), NO, dtype=np.uint8)
    npl = np.array([2] * n_run + [1] * n_one, dtype=np.uint8)
    perm = rng.permutation(len(npl))
    q = (hole[perm], board[perm], npl[perm])
    stderr, lo, hi = 0.001, 2048, 2**18
    cps = adaptive_checkpoints(lo, hi)
    seed = 99 if mode == "uniform" else 100
    ad = _adaptive(q, hi, stderr, lo, seed, mode)
    stops = ad["trials"]
    assert (stops[q[2] == 1] == lo).all()
    plans = []
    for k in range(1, len(cps)):
        active = int((stops > cps[k - 1]).sum())
        plans.append(_item_plan(active, cps[k] - cps[k - 1], sm))
    assert plans[-1] == 2048 and plans[-2] == 2048, plans
    stopped = sorted(set(np.unique(stops)))
    fixed = {T: _fixed(q, T, seed, mode) for T in stopped}
    for T in stopped:
        sel = stops == T
        for k in ("wins", "ties", "win_types", "passes"):
            assert (ad[k][sel] == fixed[T][k][sel]).all(), (mode, T, k)


@pytest.mark.gpu
def test_graph_capture(mixed):
    """The call without validation captured once: two replays give identical results, equal to the eager call."""
    import torch
    import neuron_poker_b200 as npk
    hole, board, npl = (torch.as_tensor(x).cuda() for x in mixed)
    args = dict(min_trials=MIX["min_trials"], seed_value=31, deal_mode="reference", validate=False, win_types=True,
                passes=True)
    eager = npk.get_equity_batch_adaptive(hole, board, npl, MIX["max_trials"], MIX["stderr"], **args)
    eager = {k: v.clone() for k, v in eager.items()}
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        npk.get_equity_batch_adaptive(hole, board, npl, MIX["max_trials"], MIX["stderr"], **args)
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        cap = npk.get_equity_batch_adaptive(hole, board, npl, MIX["max_trials"], MIX["stderr"], **args)
    results = []
    for _ in range(2):
        for v in cap.values():
            v.fill_(-1)                        # the call zeroes its outputs itself
        g.replay()
        torch.cuda.synchronize()
        results.append({k: v.clone() for k, v in cap.items()})
    for k in eager:
        assert torch.equal(results[0][k], results[1][k]), k
        assert torch.equal(results[0][k], eager[k]), k


@pytest.mark.gpu
def test_validation(mixed):
    import neuron_poker_b200 as npk
    hole, board, npl = (x.copy() for x in mixed)
    hole[5] = hole[5][0]                      # duplicate card
    with pytest.raises(_lib.NpkError, match="1 invalid query"):
        npk.get_equity_batch_adaptive(hole, board, npl, 256, 0.01, min_trials=64)
    out = npk.get_equity_batch_adaptive(hole, board, npl, 256, 0.01, min_trials=64, validate=False)
    t = _np(out["trials"])
    assert t[5] == 0 and _np(out["wins"])[5] == 0 and _np(out["ties"])[5] == 0
    assert (np.delete(t, 5) > 0).all()
    only = npk.equity.shape_mask([2], known_board_cards=(0,))
    out = npk.get_equity_batch_adaptive(*mixed, 256, 0.01, min_trials=64, shapes=only)
    t = _np(out["trials"])
    in_mask = (mixed[2] == 2) & ((mixed[1] != NO).sum(1) == 0)
    assert (t[in_mask] > 0).all() and (t[~in_mask] == 0).all() and (_np(out["wins"])[~in_mask] == 0).all()


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["uniform", "reference"])
def test_selfplay_step_decides_on_adaptive_equity(cuda_device, mode):
    """selfplay_step(stderr=e) takes the actions decide(equity=(w + t) / trials) gives from the same adaptive counters."""
    import torch
    import neuron_poker_b200 as npk
    from neuron_poker_b200.holdem import EquityAgents, HoldemTables
    agents = EquityAgents.equity_vs_random()
    a = HoldemTables(2048, n_players=6, seed=21, autoplay=[1] * 6)
    b = HoldemTables(2048, n_players=6, seed=21, autoplay=[1] * 6)
    stderr, runs = 0.02, 1000
    short = 0
    for _ in range(40):
        got = a.selfplay_step(agents, runs=runs, deal_mode=mode, stderr=stderr)
        hole, board, npl, _ = b.queries()
        out = npk.get_equity_batch_adaptive(hole, board, npl, runs, stderr, min_trials=256,
                                            seed_value=(b.seed << 20) + b.decisions, deal_mode=mode,
                                            query_offset=b.table_offset, validate=False, device=b.device)
        eq = (out["wins"] + out["ties"]).double() / out["trials"].clamp(min=1).double()
        want = b.decide(agents, equity=eq)
        b.step(want, restart_finished=True)
        assert torch.equal(got, want)
        short += int((out["trials"] < runs).sum())
    assert short > 0                                                   # some equities stopped before `runs`
    assert (a.state()["error"] == 0).all()
    assert (a.state().view(np.uint8) == b.state().view(np.uint8)).all()
