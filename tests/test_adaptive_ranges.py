"""Monte-Carlo equity with ranges to a target precision (npk_equity_ranges_batch_adaptive / get_equity_ranges_batch_adaptive).

The contract is get_equity_batch_adaptive's (tests/test_adaptive_equity.py) applied to the range call: checkpoints T_0 =
min_trials, doubling, capped at max_trials; a query stops when p (1 - p) / T_k <= stderr^2, p = (wins + ties + 1) / (T_k + 2).
Both range kernels draw Philox per (seed, query, trial), so the counters of a query must be EXACTLY those of
get_equity_ranges_batch(trials=T_stop) with the same seed, query_offset, ranges, ghost cards, known hands and sampler (the
generic kernel with passes, the pair-list sampler without).  The GPU tests check that bit for bit over opponent and hero
ranges, ghost cards and known opponents, together with the rule, its boundary, independence from the rest of the batch, the
device-planned rounds at production item sizes, graph capture, validation and the attempt limit.
"""
import ctypes
import math

import numpy as np
import pytest

from neuron_poker_b200 import _lib, cards
from neuron_poker_b200.equity import adaptive_checkpoints, adaptive_stops

NO = 0xFF
FIELDS = ("wins", "ties", "win_types", "passes")


def _ids(*names):
    return [cards.card_id(c) for c in names]


# ---- CPU ---------------------------------------------------------------------------------------------------------------
def _adaptive_call(stderr, min_trials, max_trials, Q=1):
    L = _lib.lib()
    rc = L.npk_equity_ranges_batch_adaptive(None, None, None, None, None, 0, Q, int(min_trials), int(max_trials),
                                            ctypes.c_double(stderr), None, None, ctypes.c_uint64(0), 0, 1, 0, None, None,
                                            None, None, None, None, None)
    return rc, L.npk_last_error().decode()


def test_rule_argument_errors_need_no_device():
    """The rule's arguments are checked first, with the messages of npk_equity_batch_adaptive, whatever the other arguments."""
    for args in ((float("nan"), 64, 128), (float("inf"), 64, 128), (0.0, 64, 128), (-0.01, 64, 128)):
        rc, msg = _adaptive_call(*args)
        assert rc == -2 and "stderr must be a finite number > 0" in msg, (args, rc, msg)
    rc, msg = _adaptive_call(0.01, 0, 128)
    assert rc == -2 and "min_trials must be >= 1" in msg, msg
    rc, msg = _adaptive_call(0.01, 129, 128)
    assert rc == -2 and "min_trials must not exceed max_trials" in msg, msg


# ---- GPU ---------------------------------------------------------------------------------------------------------------
def _np(t):
    return t.cpu().numpy()


# min 64, max 1024, stderr 0.02 (as tests/test_adaptive_equity.py): x = T or x = 0 stops at T_0 = 64; an equity of 0.5 runs
# to max_trials; equities below about 0.05 / 0.12 / 0.29 (or above 1 minus those) stop by 128 / 256 / 512.
MIX = dict(min_trials=64, max_trials=1024, stderr=0.02)
CPS = adaptive_checkpoints(MIX["min_trials"], MIX["max_trials"])
SET_RANGE = {"AA", "KK", "QQ", "JJ", "TT", "99", "AKS", "AKO", "AQS", "KQS", "JTS", "76S"}
HERO_SET = {"AKO", "72O", "T9S", "55", "QJO"}
ROYAL = _ids("AS", "KS", "QS", "JS", "TS")
AA_VS_72 = dict(hero=_ids("7C", "2D"), known=_ids("AS", "AH"), board=_ids("KD", "QC", "9S", "4H", "3C"))   # x = 0


def _range_batch(n_known, hero_range, ghost, seed, per_shape=3):
    """Random queries of every players (n_known + 1..10) x known board cards (0, 3, 4, 5), then known answers: players = 1
    (x = T, when there are no known opponents), a made royal flush of a fixed hero (x = T) and, with known opponents, hero
    7-2 against a known pair of aces on a river where the 7-2 cannot improve (x = 0)."""
    rng = np.random.default_rng(seed)
    hole, board, npl, gh, kn, answer = [], [], [], [], [], []

    def add(h, b, p, g, k, x=None):
        hole.append(h); board.append(list(b) + [NO] * (5 - len(b))); npl.append(p); gh.append(g); kn.append(k)
        answer.append(x)

    for players in range(max(1, n_known + 1), 11):
        for known in (0, 3, 4, 5):
            for _ in range(per_shape):
                c = rng.permutation(52)
                add(c[:2], c[2:2 + known], players, c[10:12] if ghost else [NO, NO],
                    c[12:12 + 2 * n_known].reshape(n_known, 2))
    if n_known == 0:
        for known in (0, 3, 5):
            c = rng.permutation(52)
            add(c[:2], c[2:2 + known], 1, c[10:12] if ghost else [NO, NO], np.zeros((0, 2), dtype=np.int64), "T")
    spare = [c for c in range(52) if c not in ROYAL + AA_VS_72["hero"] + AA_VS_72["known"] + AA_VS_72["board"]]
    if hero_range is None:
        for players in range(n_known + 1 + (n_known == 0), 11, 3):
            for known in (3, 4, 5):
                b = ROYAL[2:2 + known] if known == 3 else ROYAL[2:] + spare[:known - 3]
                k = np.array(spare[2:2 + 2 * n_known]).reshape(n_known, 2)
                add(ROYAL[:2], b, players, spare[20:22] if ghost else [NO, NO], k, "T")
        if n_known >= 1:
            for players in range(n_known + 1, 11, 2):
                k = np.array(AA_VS_72["known"] + spare[2:2 * n_known]).reshape(n_known, 2)
                add(AA_VS_72["hero"], AA_VS_72["board"], players, spare[20:22] if ghost else [NO, NO], k, "0")
    q = dict(hole=np.array(hole, dtype=np.uint8), board=np.array(board, dtype=np.uint8),
             n_players=np.array(npl, dtype=np.uint8), ghost=np.array(gh, dtype=np.uint8) if ghost else None,
             known_opponents=np.array(kn, dtype=np.uint8).reshape(len(hole), n_known, 2) if n_known else None)
    return q, np.array([x == "T" for x in answer]), np.array([x == "0" for x in answer])


def _fixed(q, T, kw):
    import neuron_poker_b200 as npk
    out = npk.get_equity_ranges_batch(q["hole"], q["board"], q["n_players"], T, ghost=q["ghost"],
                                      known_opponents=q["known_opponents"], win_types=True, **kw)
    return {k: _np(out[k]) for k in FIELDS if k in out}


def _adaptive(q, kw, max_trials=MIX["max_trials"], stderr=MIX["stderr"], min_trials=MIX["min_trials"], **extra):
    import neuron_poker_b200 as npk
    out = npk.get_equity_ranges_batch_adaptive(q["hole"], q["board"], q["n_players"], max_trials, stderr,
                                               min_trials=min_trials, ghost=q["ghost"],
                                               known_opponents=q["known_opponents"], win_types=True, **kw, **extra)
    return {k: _np(v) for k, v in out.items()}


def _check_exact(ad, fixed, checkpoints, stderr):
    """Every query equals the fixed-trial run at its T_stop, and the host rule on the fixed counters continues at every
    earlier checkpoint and stops at T_stop (or T_stop = max_trials)."""
    stops = ad["trials"]
    assert set(np.unique(stops)) <= set(checkpoints), np.unique(stops)
    for T in np.unique(stops):
        sel = stops == T
        for k in fixed[T]:
            assert (ad[k][sel] == fixed[T][k][sel]).all(), (int(T), k)
    for i in range(len(stops)):
        for T in checkpoints:
            stop = adaptive_stops(int(fixed[T]["wins"][i] + fixed[T]["ties"][i]), T, stderr) or T == checkpoints[-1]
            if T < stops[i]:
                assert not stop, (i, T, int(stops[i]))
            else:
                assert stop and T == stops[i], (i, T, int(stops[i]))
                break


# (opponent range, hero range, ghost cards, known opponents): every argument of the range call
CONFIGS = [(0.3, None, False, 0), (SET_RANGE, HERO_SET, True, 0), (0.2, None, True, 1), (SET_RANGE, None, False, 2),
           (0.3, None, True, 3)]


@pytest.mark.gpu
@pytest.mark.parametrize("sampler", ["generic", "pair_list"])
@pytest.mark.parametrize("mode", ["uniform", "reference"])
@pytest.mark.parametrize("config", range(len(CONFIGS)))
def test_bit_exact_against_fixed_trial_runs_and_rule_applied_exactly(cuda_device, config, mode, sampler):
    opp, hero, ghost, n_known = CONFIGS[config]
    q, x_t, x_0 = _range_batch(n_known, hero, ghost, seed=40 + config)
    kw = dict(opponent_range=opp, hero_range=hero, seed_value=0xada0 + 2 * config + (mode == "reference"), deal_mode=mode,
              passes=sampler == "generic")
    ad = _adaptive(q, kw)
    assert ("passes" in ad) == (sampler == "generic")
    for T in CPS:                                                           # the batch stops queries at every checkpoint
        assert (ad["trials"] == T).any(), (T, np.unique(ad["trials"], return_counts=True))
    assert x_t.any() and (ad["trials"][x_t] == CPS[0]).all() and (ad["wins"][x_t] == CPS[0]).all()
    assert (x_0.any() or n_known == 0) and (ad["trials"][x_0] == CPS[0]).all()
    assert (ad["wins"][x_0] + ad["ties"][x_0] == 0).all()
    fixed = {T: _fixed(q, T, kw) for T in CPS}
    _check_exact(ad, fixed, CPS, MIX["stderr"])


def _predicted_stops(fixed, checkpoints, stderr, n):
    out = np.zeros(n, dtype=np.int64)
    for i in range(n):
        for T in checkpoints:
            if T == checkpoints[-1] or adaptive_stops(int(fixed[T]["wins"][i] + fixed[T]["ties"][i]), T, stderr):
                out[i] = T
                break
    return out


@pytest.mark.gpu
def test_boundary_of_the_rule(cuda_device):
    """s = sqrt(var) of chosen queries at a checkpoint, and the two doubles next to it: for every s the device stops every
    query exactly where the host rule says.  x = T and x = 0 stop at T_0 iff s^2 >= (T_0 + 1) / ((T_0 + 2)^2 T_0), each as
    rounded in the rule's order of operations (the two roundings differ in the last bit)."""
    q, x_t, x_0 = _range_batch(1, None, True, seed=77)
    kw = dict(opponent_range=0.3, seed_value=77, deal_mode="reference")
    fixed = {T: _fixed(q, T, kw) for T in CPS}
    n = len(q["hole"])
    T0 = CPS[0]
    p = (T0 + 1.0) / float(T0 + 2)
    v_t = p * (1.0 - p) / float(T0)                                         # x = T, in the rule's order of operations
    p = 1.0 / float(T0 + 2)
    v_0 = p * (1.0 - p) / float(T0)                                         # x = 0: the same rational, rounded apart
    chosen = [v_t, v_0]
    x2 = fixed[CPS[2]]["wins"] + fixed[CPS[2]]["ties"]
    i = int(np.argmin(np.abs(x2 / CPS[2] - 0.1)))                          # a query near an equity of 0.1 at T_2
    p = (float(x2[i]) + 1.0) / float(CPS[2] + 2)
    chosen.append(p * (1.0 - p) / float(CPS[2]))
    seen_sides = set()
    for var in chosen:
        s = math.sqrt(var)
        for sv in (float(np.nextafter(s, 0.0)), s, float(np.nextafter(s, 1.0))):
            ad = _adaptive(q, kw, stderr=sv)
            want = _predicted_stops(fixed, CPS, sv, n)
            assert (ad["trials"] == want).all(), (sv, np.nonzero(ad["trials"] != want)[0][:5])
            assert (ad["trials"][x_t] == (T0 if v_t <= sv * sv else CPS[1])).all()
            assert (ad["trials"][x_0] == (T0 if v_0 <= sv * sv else CPS[1])).all()
            seen_sides.add(var <= sv * sv)
    assert seen_sides == {True, False}


def _take(q, sel):
    return {k: (None if v is None else v[sel]) for k, v in q.items()}


@pytest.mark.gpu
@pytest.mark.parametrize("sampler", ["generic", "pair_list"])
def test_independent_of_the_rest_of_the_batch(cuda_device, sampler):
    """The batch split in two with query_offset equals the whole batch; a query keeps its counts when every other query of
    the batch is replaced by one that retires at T_0 (players = 1)."""
    q, _, _ = _range_batch(0, None, True, seed=9)
    kw = dict(opponent_range=0.3, seed_value=1234, deal_mode="uniform", passes=sampler == "generic")
    whole = _adaptive(q, kw)
    n = len(q["hole"])
    h = n // 3
    a = _adaptive(_take(q, slice(0, h)), kw)
    b = _adaptive(_take(q, slice(h, n)), kw, query_offset=h)
    for k in whole:
        assert (np.concatenate([a[k], b[k]]) == whole[k]).all(), k
    keep = np.arange(n) % 7 == 3
    lone = dict(q)
    lone["n_players"] = q["n_players"].copy()
    lone["n_players"][~keep] = 1
    out = _adaptive(lone, kw)
    assert (out["trials"][~keep] == MIX["min_trials"]).all()
    for k in whole:
        assert (out[k][keep] == whole[k][keep]).all(), k


def _item_plan(queries, trials, sm_count, lanes_worth=32):
    """npk::item_plan (csrc/npk_kernels.h): (trials per item, items per query)."""
    c = (queries * trials) // (8 * sm_count * 16)
    c = max(lanes_worth, min(2048, (c + lanes_worth - 1) // lanes_worth * lanes_worth))
    if trials <= c:
        return trials, 1
    return c, (trials + c - 1) // c


@pytest.mark.gpu
@pytest.mark.parametrize("sampler", ["generic", "pair_list"])
def test_production_item_sizes(cuda_device, sampler):
    """A batch sized from the SM count: most queries (players = 1) retire at T_0 = 2,048, about 8 x SMs heads-up preflop
    queries against a range run on, so that the device plans the later rounds in 2,048-trial items.  Called through the C
    entry point with a caller-owned workspace, whose work counter shows the last round's item count; every query equals
    the fixed-trial run at its T_stop."""
    import torch
    from neuron_poker_b200 import ranges
    L = _lib.ensure_init(0)
    sm = L.npk_sm_count()
    rng = np.random.default_rng(8)
    n_run = 8 * sm + 64
    n_one = 4 * n_run
    Q = n_run + n_one
    hole = np.stack([rng.permutation(52)[:2] for _ in range(Q)]).astype(np.uint8)
    board = np.full((Q, 5), NO, dtype=np.uint8)
    npl = np.array([2] * n_run + [1] * n_one, dtype=np.uint8)[rng.permutation(Q)]
    stderr, lo, hi = 0.001, 2048, 2**17
    cps = adaptive_checkpoints(lo, hi)
    mode, seed, generic = "reference", 99, sampler == "generic"
    dev = torch.device("cuda", 0)
    t_hole, t_board, t_npl = (torch.as_tensor(x).to(dev) for x in (hole, board, npl))
    out = {k: torch.full((Q, 9) if k == "win_types" else (Q,), -1, dtype=torch.int64, device=dev)
           for k in ("wins", "ties", "win_types", "passes", "trials")}
    ws = torch.zeros(int(L.npk_equity_adaptive_workspace_bytes(Q)), dtype=torch.uint8, device=dev)
    opp = ranges.opponent_mask(0.2)
    _lib.check(L.npk_equity_ranges_batch_adaptive(t_hole.data_ptr(), t_board.data_ptr(), t_npl.data_ptr(), None, None, 0, Q,
                                                  lo, hi, ctypes.c_double(stderr), opp.ctypes.data_as(ctypes.c_void_p), None,
                                                  ctypes.c_uint64(seed), 0, 1, _lib.NPK_FLAG_VALIDATE,
                                                  out["wins"].data_ptr(), out["ties"].data_ptr(), out["win_types"].data_ptr(),
                                                  out["passes"].data_ptr() if generic else None, out["trials"].data_ptr(),
                                                  ws.data_ptr(), torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    ad = {k: _np(v) for k, v in out.items() if generic or k != "passes"}
    stops = ad["trials"]
    assert (stops[npl == 1] == lo).all() and (stops[npl == 2] > lo).all()
    plans = []
    for k in range(1, len(cps)):
        plans.append(_item_plan(int((stops > cps[k - 1]).sum()), cps[k] - cps[k - 1], sm))
    assert plans[-1][0] == 2048 and plans[-2][0] == 2048, plans
    # the work counter of the last round: every item once, then one failed pull per warp of the grid (16 warps a CTA)
    last_active = int((stops > cps[-2]).sum())
    _, host_chunks = _item_plan(Q, cps[-1] - cps[-2], sm)
    grid = max(1, min(sm, -(-Q * host_chunks // 16)))
    counter = int(ws[:8].cpu().numpy().view(np.uint64)[0])
    assert counter == last_active * plans[-1][1] + 16 * grid, (counter, last_active, plans[-1], grid)
    kw = dict(opponent_range=0.2, seed_value=seed, deal_mode=mode, passes=generic)
    qd = dict(hole=hole, board=board, n_players=npl, ghost=None, known_opponents=None)
    for T in sorted(set(np.unique(stops))):
        fixed = _fixed(qd, int(T), kw)
        sel = stops == T
        for k in fixed:
            assert (ad[k][sel] == fixed[k][sel]).all(), (int(T), k)


@pytest.mark.gpu
@pytest.mark.parametrize("sampler", ["generic", "pair_list"])
def test_graph_capture(cuda_device, sampler):
    """The call without validation captured once: two replays give identical results, equal to the eager call."""
    import torch
    import neuron_poker_b200 as npk
    q, _, _ = _range_batch(1, None, True, seed=31)
    t = {k: (None if v is None else torch.as_tensor(v).cuda()) for k, v in q.items()}
    args = dict(min_trials=MIX["min_trials"], opponent_range=0.3, ghost=t["ghost"], known_opponents=t["known_opponents"],
                seed_value=31, deal_mode="reference", validate=False, win_types=True, passes=sampler == "generic")

    def call():
        return npk.get_equity_ranges_batch_adaptive(t["hole"], t["board"], t["n_players"], MIX["max_trials"], MIX["stderr"],
                                                    **args)
    eager = {k: v.clone() for k, v in call().items()}
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        call()
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        cap = call()
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
def test_validation(cuda_device):
    """An invalid query (a ghost card on the board) is NPK_ERR_INVALID_CARDS with the fixed call's message, before any trial
    runs: the caller's counters are zeroed and stay zero.  Without validation the query is left at 0 with trials = 0."""
    import torch
    import neuron_poker_b200 as npk
    from neuron_poker_b200 import ranges
    q, _, _ = _range_batch(1, None, True, seed=5)
    i = int(np.nonzero((q["board"] != NO).sum(1) == 5)[0][0])
    q["ghost"][i] = [q["board"][i][0], q["ghost"][i][1]]
    with pytest.raises(_lib.NpkError) as fixed_err:
        npk.get_equity_ranges_batch(q["hole"], q["board"], q["n_players"], 64, opponent_range=0.3, ghost=q["ghost"],
                                    known_opponents=q["known_opponents"])
    with pytest.raises(_lib.NpkError, match="1 invalid query") as err:
        _adaptive(q, dict(opponent_range=0.3))
    assert str(err.value) == str(fixed_err.value) and err.value.code == -5
    L = _lib.ensure_init(0)
    Q = len(q["hole"])
    dev = torch.device("cuda", 0)
    t = {k: torch.as_tensor(v).to(dev) for k, v in q.items()}
    out = {k: torch.full((Q,), -1, dtype=torch.int64, device=dev) for k in ("wins", "ties", "trials")}
    ws = torch.empty(int(L.npk_equity_adaptive_workspace_bytes(Q)), dtype=torch.uint8, device=dev)
    opp = ranges.opponent_mask(0.3)
    rc = L.npk_equity_ranges_batch_adaptive(t["hole"].data_ptr(), t["board"].data_ptr(), t["n_players"].data_ptr(),
                                            t["ghost"].data_ptr(), t["known_opponents"].data_ptr(), 1, Q, 64, 1024,
                                            ctypes.c_double(0.01), opp.ctypes.data_as(ctypes.c_void_p), None,
                                            ctypes.c_uint64(3), 0, 1, _lib.NPK_FLAG_VALIDATE, out["wins"].data_ptr(),
                                            out["ties"].data_ptr(), None, None, out["trials"].data_ptr(), ws.data_ptr(),
                                            torch.cuda.current_stream().cuda_stream)
    assert rc == -5
    torch.cuda.synchronize()
    for k in out:
        assert (_np(out[k]) == 0).all(), k                                  # zeroed, and no trial has run
    ad = _adaptive(q, dict(opponent_range=0.3), validate=False)
    assert ad["trials"][i] == 0 and ad["wins"][i] == 0 and ad["ties"][i] == 0
    assert (np.delete(ad["trials"], i) >= MIX["min_trials"]).all()


@pytest.mark.gpu
@pytest.mark.parametrize("sampler", ["generic", "pair_list"])
def test_unsatisfiable_range_is_an_error_and_the_call_returns(cuda_device, sampler):
    """Hero AS AH on an AD board against {'AA'}: no opponent hand is left, a draw hits the attempt limit, and the validated
    call reports NPK_ERR_RANGE with the fixed call's message -- also when that query retires at T_0 (x = 0) while the other
    queries run on to max_trials: the abort flag is cleared once per call, not per round."""
    import neuron_poker_b200 as npk
    rng = np.random.default_rng(2)
    n = 64
    hole = np.stack([rng.permutation(52)[:2] for _ in range(n)]).astype(np.uint8)
    board = np.full((n, 5), NO, dtype=np.uint8)
    npl = np.full(n, 2, dtype=np.uint8)
    hole[0] = _ids("AS", "AH")
    board[0, :3] = _ids("AD", "7C", "2H")
    kw = dict(opponent_range={"AA"}, deal_mode="reference", passes=sampler == "generic")
    with pytest.raises(_lib.NpkError) as fixed_err:
        npk.get_equity_ranges_batch(hole, board, npl, 64, **kw)
    for lo, hi in ((64, 64), (64, 4096)):
        with pytest.raises(_lib.NpkError) as err:
            npk.get_equity_ranges_batch_adaptive(hole, board, npl, hi, 0.02, min_trials=lo, **kw)
        assert err.value.code == -6 and str(err.value) == str(fixed_err.value)


@pytest.mark.gpu
def test_range_argument_errors_are_the_fixed_calls(cuda_device):
    """Null pointers, n_known, a hero range with known hands, the dealing mode and empty ranges: the same codes and messages
    as npk_equity_ranges_known_batch (one shared check)."""
    import torch
    from neuron_poker_b200 import ranges
    L = _lib.ensure_init(0)
    dev = torch.device("cuda", 0)
    Q = 4
    u8 = torch.zeros((Q, 8), dtype=torch.uint8, device=dev)
    o64 = torch.zeros((Q, 16), dtype=torch.int64, device=dev)
    ws = torch.zeros(int(L.npk_equity_adaptive_workspace_bytes(Q)), dtype=torch.uint8, device=dev)
    full, empty = ranges.opponent_mask(1.0), np.zeros(3, dtype=np.uint64)
    ptr = lambda a: a.ctypes.data_as(ctypes.c_void_p)                        # noqa: E731
    P = u8.data_ptr()
    cases = [  # hole, board, players, known, n_known, opp, hero, deal_mode, wins
        (P, None, P, None, 0, ptr(full), None, 1, o64.data_ptr()),
        (None, P, P, None, 0, ptr(full), None, 1, o64.data_ptr()),
        (P, P, P, None, 0, ptr(full), None, 1, None),
        (P, P, P, None, 0, None, None, 1, o64.data_ptr()),
        (P, P, P, None, 1, ptr(full), None, 1, o64.data_ptr()),
        (P, P, P, P, 10, ptr(full), None, 1, o64.data_ptr()),
        (P, P, P, P, 1, ptr(full), ptr(full), 1, o64.data_ptr()),
        (P, P, P, None, 0, ptr(full), None, 7, o64.data_ptr()),
        (P, P, P, None, 0, ptr(empty), None, 1, o64.data_ptr()),
        (P, P, P, None, 0, ptr(full), ptr(empty), 1, o64.data_ptr()),
    ]
    stream = torch.cuda.current_stream().cuda_stream
    for hole, board, npl, known, n_known, opp, hero, mode, wins in cases:
        rc_f = L.npk_equity_ranges_known_batch(hole, board, npl, None, known, n_known, Q, 64, opp, hero, ctypes.c_uint64(0),
                                               0, 0, mode, 0, wins, o64.data_ptr(), None, None, ws.data_ptr(), stream)
        msg_f = L.npk_last_error().decode()
        rc_a = L.npk_equity_ranges_batch_adaptive(hole, board, npl, None, known, n_known, Q, 64, 128, ctypes.c_double(0.01),
                                                  opp, hero, ctypes.c_uint64(0), 0, mode, 0, wins, o64.data_ptr(), None,
                                                  None, o64.data_ptr(), ws.data_ptr(), stream)
        msg_a = L.npk_last_error().decode()
        assert rc_f < 0 and (rc_a, msg_a) == (rc_f, msg_f), (rc_f, msg_f, rc_a, msg_a)
    torch.cuda.synchronize()
