"""GPU parity tests: libnpk's CUDA kernels, called through the C ABI, against the oracle and the golden fixtures.

Bar: bit-exact for rank ids, showdown winners, enumerated (win, tie, lose) counts AND for Monte-Carlo counts against
the executable sampler specification (tests/sampler_model.py scored by the oracle); statistical (3 sigma of the binomial
standard error, as BASELINE.json's north_star states) only where two different random streams are compared.
"""
import ctypes
import math

import numpy as np
import pytest

import neuron_poker_b200 as npk
import oracle
import sampler_model
from neuron_poker_b200 import _lib

pytestmark = pytest.mark.gpu

NO = 0xFF


def ids(cards):
    return [npk.card_id(c) for c in cards]


def pad_board(b):
    return list(b) + [NO] * (5 - len(b))


def sigma(p, n):
    return math.sqrt(max(p * (1 - p), 1e-12) / n)


@pytest.fixture(scope="module")
def torch_mod(cuda_device):
    import torch
    _lib.ensure_init(0)
    return torch


def test_philox_known_answers(torch_mod):
    torch = torch_mod
    ctrs = [(0, 0, 0, 0), (0xffffffff,) * 4, (0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (5, 0, 77, 1)]
    keys = [(0, 0), (0xffffffff, 0xffffffff), (0xa4093822, 0x299f31d0), (123, 456)]
    for c, k in zip(ctrs, keys):
        ctr = torch.tensor(np.array(c, dtype=np.uint32).view(np.int32), device="cuda")
        out = torch.zeros(4, dtype=torch.int32, device="cuda")
        _lib.check(_lib.lib().npk_philox_debug(ctr.data_ptr(), k[0], k[1], 1, out.data_ptr(), None))
        torch.cuda.synchronize()
        got = out.cpu().numpy().view(np.uint32).tolist()
        assert got == sampler_model.philox4x32_10(c, k)
    assert sampler_model.philox4x32_10((0, 0, 0, 0), (0, 0)) == [0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8]


def test_rank7_golden_and_oracle(torch_mod, golden_cases, golden_tables):
    hands = golden_cases["random_hands"] + golden_cases["rare_hands"]
    cards = np.array([h["cards"] for h in hands], dtype=np.uint8)
    got = npk.rank7(cards).cpu().numpy()
    assert (got == np.array([h["rank_id"] for h in hands])).all()
    rng = np.random.default_rng(3)
    big = np.stack([rng.permutation(52)[:7] for _ in range(200000)]).astype(np.uint8)
    assert (npk.rank7(big).cpu().numpy() == oracle.rank7_batch(big)).all()
    # every rank histogram (non-flush suits) and every flush mask: the whole key space of the evaluator
    hist = golden_tables["hist"]
    hc = np.zeros((len(hist), 7), dtype=np.uint8)
    for i, h in enumerate(hist):
        k = 0
        for r in range(13):
            for _ in range(h[r]):
                hc[i, k] = 4 * r + (k & 3)
                k += 1
    assert (npk.rank7(hc).cpu().numpy() == golden_tables["nonflush"]).all()
    fl = golden_tables["flush"]
    masks = [m for m in range(8192) if fl[m] != 0xFFFF]
    for suit in range(4):
        fc = []
        for m in masks:
            c = [4 * r + suit for r in range(13) if m >> r & 1]
            pad = 0
            while len(c) < 7:
                c.append(4 * pad + (suit + 1) % 4)
                pad += 1
            fc.append(c)
        assert (npk.rank7(np.array(fc, dtype=np.uint8)).cpu().numpy() == fl[masks]).all()


def test_rank7_exhaustive_all_133784560_hands(torch_mod):
    """Every 7-card hand (colexicographic enumeration on the GPU, no input traffic): per-chunk sum, position-weighted
    sum and hand-type census equal the oracle's golden checksums; three chunks are also compared id by id."""
    import json
    import os
    torch = torch_mod
    gold = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "colex_checksums.json")))
    chunk, n = gold["chunk"], gold["n_hands"]
    ts = torch.tensor([0, 407, 1877, 2640, 3215, 3225, 4502, 4658, 4736, 5034], device="cuda")
    for ci, start in enumerate(range(0, n, chunk)):
        cnt = min(chunk, n - start)
        r = npk.rank7_colex(start, cnt).to(torch.int64)
        idx = torch.arange(start, start + cnt, device="cuda", dtype=torch.int64)
        census = torch.bucketize(r, ts[1:9], right=True).bincount(minlength=9)
        got = [int(r.sum()), int((r * (idx % 65521 + 1)).sum())] + census.tolist()
        assert got == gold["chunks"][ci], ci
        if ci in (0, 31, 63):
            assert (r.cpu().numpy() == oracle.colex_range(start, cnt)[0]).all()


def test_rank7_empty_and_ragged(torch_mod):
    torch = torch_mod
    assert npk.rank7(np.zeros((0, 7), dtype=np.uint8)).numel() == 0
    one = npk.rank7(np.array([[0, 4, 8, 12, 16, 21, 25]], dtype=np.uint8)).cpu().numpy()   # 2C 3C 4C 5C 6C 7D 8D
    assert one[0] == oracle.rank7([0, 4, 8, 12, 16, 21, 25])


def test_known_answer_showdowns(torch_mod, golden_cases):
    for case in golden_cases["known"]:
        if case["name"] in ("3", "6b"):
            continue        # duplicate physical cards: expressible only at table level (SURVEY A.3), see test below
        best, ty = npk.eval_best_hand(case["hands"])
        assert best == case["hands"][case["winner"]] and ty == case["winner_type"], case["name"]


def test_duplicate_card_cases_at_table_level(golden_cases):
    """Cases 3 and 6b of tests/test_evaluator.py hold duplicate cards; their values are still (histogram, flush mask)
    keys of the lookup tables, which is what is compared here (host copy of the device tables)."""
    t = npk.host_tables()
    for case in golden_cases["known"]:
        if case["name"] not in ("3", "6b"):
            continue
        vals = []
        for hand in case["hands"]:
            cid = ids(hand)
            suits = [c & 3 for c in cid]
            fs = [s for s in range(4) if suits.count(s) >= 5]
            if fs:
                mask = 0
                for c in cid:
                    if (c & 3) == fs[0]:
                        mask |= 1 << (c >> 2)
                if bin(mask).count("1") >= 5:
                    vals.append(int(t["flush"][mask]))
                    continue
            mk = sum(int(t["desc"][4 * (c >> 2)]) >> 9 for c in cid) & ((1 << 23) - 1)
            vals.append(int(t["value"][int(t["rowoff"][mk >> 10]) + (mk & 1023)]))
        exp = [oracle.rank_of_tuple(tuple(tp[0]), tuple(tp[1])) for tp in case["tuples"]]
        if case["name"] == "3":
            assert vals == exp
        assert vals.index(max(vals)) == case["winner"]


def test_showdown_batch(torch_mod, golden_cases):
    sds = golden_cases["showdowns"]
    maxp = 9
    holes = np.zeros((len(sds), maxp, 2), dtype=np.uint8)
    npl = np.zeros(len(sds), dtype=np.uint8)
    board = np.zeros((len(sds), 5), dtype=np.uint8)
    for i, s in enumerate(sds):
        npl[i] = len(s["holes"])
        holes[i, :npl[i]] = s["holes"]
        board[i] = s["board"]
    w, t, r = npk.showdown(holes, npl, board, return_ranks=True)
    assert (w.cpu().numpy() == np.array([s["winner"] for s in sds])).all()
    assert (t.cpu().numpy() == np.array([s["type"] for s in sds])).all()
    s0 = sds[0]
    assert npk.get_winner([[npk.card_str(c) for c in h] for h in s0["holes"]],
                          [npk.card_str(c) for c in s0["board"]])[0] == s0["winner"]
    rk = r.cpu().numpy()
    for i in range(0, len(sds), 50):
        for p in range(npl[i]):
            assert rk[i, p] == oracle.rank7(list(sds[i]["holes"][p]) + list(sds[i]["board"]))


def test_enumeration_bit_exact(torch_mod, golden_enum):
    spots = [s for s in golden_enum["spots"] if "uniform" in s]
    hole = np.array([ids(s["hero"]) for s in spots], dtype=np.uint8)
    board = np.array([pad_board(ids(s["board"])) for s in spots], dtype=np.uint8)
    npl = np.array([s["players"] for s in spots], dtype=np.uint8)
    w, t, l = npk.enumerate_equity(hole, board, npl)
    got = np.stack([w.cpu().numpy(), t.cpu().numpy(), l.cpu().numpy()], 1).tolist()
    for s, g in zip(spots, got):
        assert g == s["uniform"], (s["name"], g)
    rnd = golden_enum["random_spots"]
    hole = np.array([ids(s["hero"]) for s in rnd], dtype=np.uint8)
    board = np.array([pad_board(ids(s["board"])) for s in rnd], dtype=np.uint8)
    w, t, l = npk.enumerate_equity(hole, board)
    got = np.stack([w.cpu().numpy(), t.cpu().numpy(), l.cpu().numpy()], 1).tolist()
    assert got == [s["uniform"] for s in rnd]


def test_enumeration_synthetic_batch_vs_oracle(torch_mod):
    """cfg 2: seeded random heads-up river and turn spots, GPU counts == CPU enumeration with the oracle evaluator."""
    rng = np.random.default_rng(0)
    hole, board = [], []
    for i in range(192):
        nb = 5 if i % 2 == 0 else 4
        c = rng.permutation(52)[:2 + nb].tolist()
        hole.append(c[:2])
        board.append(pad_board(c[2:]))
    w, t, l = npk.enumerate_equity(np.array(hole, dtype=np.uint8), np.array(board, dtype=np.uint8))
    w, t, l = w.cpu().numpy(), t.cpu().numpy(), l.cpu().numpy()
    for i in range(192):
        b = [c for c in board[i] if c != NO]
        assert (int(w[i]), int(t[i]), int(l[i])) == oracle.enum_headsup(hole[i], b)
        assert w[i] + t[i] + l[i] == (990 if len(b) == 5 else 45540)


def _run_batch(torch, hole, board, npl, trials, seed, mode, **kw):
    out = npk.get_equity_batch(np.array(hole, dtype=np.uint8), np.array(board, dtype=np.uint8),
                               np.array(npl, dtype=np.uint8), trials, seed_value=seed, deal_mode=mode, **kw)
    torch.cuda.synchronize()
    return {k: (v.cpu().numpy() if hasattr(v, "cpu") else v) for k, v in out.items()}


MODEL_QUERIES = [
    (["AS", "KS"], [], 2), (["AS", "KS"], [], 3), (["8S", "TS"], [], 5), (["7D", "7C"], [], 10),
    (["3S", "QH"], ["2C", "5H", "7C"], 2), (["AS", "KS"], ["2C", "7D", "KH"], 6), (["TC", "TH"], ["4D", "QD", "KC"], 9),
    (["5H", "KD"], ["KH", "JS", "2C", "QS"], 2), (["5H", "KD"], ["KH", "JS", "2C", "QS"], 4),
    (["3H", "3S"], ["8S", "4S", "QH", "8C", "4H"], 2), (["JD", "JS"], ["8C", "TC", "JC", "5H", "QC"], 3),
    (["8S", "2S"], ["5S", "3S", "4S", "KS", "AS"], 7), (["2H", "2D"], ["2C"], 3), (["9H", "9D"], ["2C", "3D"], 4),
    (["AH", "KH"], ["QH", "JH", "2C"], 6), (["AS", "AD"], [], 1),
]


@pytest.mark.parametrize("mode", ["uniform", "reference"])
def test_montecarlo_counts_equal_sampler_specification(torch_mod, mode):
    """Mixed-shape batch: wins / ties / win types (/ passes) bit-identical to the Python specification + oracle."""
    torch = torch_mod
    hole = [ids(q[0]) for q in MODEL_QUERIES]
    board = [pad_board(ids(q[1])) for q in MODEL_QUERIES]
    npl = [q[2] for q in MODEL_QUERIES]
    trials, seed = 150, 0x1234567890ABCDEF
    out = _run_batch(torch, hole, board, npl, trials, seed, mode, win_types=True, passes=(mode == "reference"))
    for qi, (h, b, p) in enumerate(MODEL_QUERIES):
        m = sampler_model.run_model(oracle, mode, seed, qi, ids(h), ids(b), p, trials)
        assert (int(out["wins"][qi]), int(out["ties"][qi])) == (m["wins"], m["ties"]), (mode, qi)
        assert out["win_types"][qi].tolist() == m["win_types"], (mode, qi)
        if mode == "reference":
            assert int(out["passes"][qi]) == m["passes"], qi


def test_every_kernel_instantiation_matches_specification(torch_mod):
    """All 60 template instantiations of the uniform kernel (0..9 opponents x 0..5 known board cards) and the same shapes
    through the reference-dealer kernel, each launched on its own (uniform_shape) and bit-exact against the specification,
    win types and passes included.  (This is the test that caught a ptxas miscompile of the last Fisher-Yates draw during
    bring-up.)  The persistent mixed kernel runs the same shapes in test_montecarlo_counts_equal_sampler_specification and
    test_mc_at_scale.py."""
    torch = torch_mod
    rng = np.random.default_rng(5)
    trials, seed = 40, 77
    for players in range(1, 11):
        for known in range(6):
            c = rng.permutation(52)[:2 + known].tolist()
            for mode in ("uniform", "reference"):
                out = _run_batch(torch, [c[:2]], [pad_board(c[2:])], [players], trials, seed, mode, uniform_shape=(players, known),
                                 win_types=True, passes=(mode == "reference"))
                m = sampler_model.run_model(oracle, mode, seed, 0, c[:2], c[2:], players, trials)
                assert (int(out["wins"][0]), int(out["ties"][0])) == (m["wins"], m["ties"]), (mode, players, known)
                assert out["win_types"][0].tolist() == m["win_types"], (mode, players, known)
                if mode == "reference":
                    assert int(out["passes"][0]) == m["passes"], (players, known)


def test_partition_invariance(torch_mod):
    """Counts depend only on (seed, query, trial): splitting the trials over calls (trial_offset) or running a query
    alone gives bit-identical totals.  This is what makes multi-GPU sharding exact."""
    torch = torch_mod
    hole = [ids(["AS", "KS"]), ids(["7D", "7C"])]
    board = [pad_board(ids(["2C", "7D", "KH"])), pad_board(ids(["2C", "7S", "KH"]))]
    npl = [6, 6]
    for mode in ("uniform", "reference"):
        whole = _run_batch(torch, hole, board, npl, 5000, 99, mode, uniform_shape=(6, 3))
        acc_w = np.zeros(2, dtype=np.int64)
        acc_t = np.zeros(2, dtype=np.int64)
        for off, n in ((0, 1777), (1777, 1200), (2977, 2023)):
            part = _run_batch(torch, hole, board, npl, n, 99, mode, trial_offset=off, uniform_shape=(6, 3))
            acc_w += part["wins"]
            acc_t += part["ties"]
        assert (acc_w == whole["wins"]).all() and (acc_t == whole["ties"]).all(), mode
        mixed = _run_batch(torch, hole, board, npl, 5000, 99, mode)           # classified path, same numbers
        assert (mixed["wins"] == whole["wins"]).all() and (mixed["ties"] == whole["ties"]).all()


def test_uniform_mode_matches_exact_enumeration(torch_mod, golden_enum):
    """UNIFORM dealing vs exact combinatorics (SURVEY A.3), 3 sigma at 4M trials (fixed seed; across seeds the
    z-scores of these spots behave like N(0,1), see profiles/r01_zscores.txt)."""
    torch = torch_mod
    spots = [s for s in golden_enum["spots"] if "uniform" in s]
    hole = [ids(s["hero"]) for s in spots]
    board = [pad_board(ids(s["board"])) for s in spots]
    npl = [s["players"] for s in spots]
    trials = 4000000
    out = _run_batch(torch, hole, board, npl, trials, 8, "uniform")
    for i, s in enumerate(spots):
        w, t, l = s["uniform"]
        tot = w + t + l
        for got, exact in ((out["wins"][i], w / tot), (out["ties"][i], t / tot)):
            assert abs(got / trials - exact) <= 3 * sigma(exact, trials) + 1e-9, (s["name"], got / trials, exact)


def test_reference_mode_matches_reference_dealer_expectation(torch_mod, golden_enum):
    """REFERENCE dealing vs the exact expectation of the reference's own dealer (weighted enumeration, SURVEY A.3)."""
    torch = torch_mod
    spots = [s for s in golden_enum["spots"] if "reference_mode" in s]
    hole = [ids(s["hero"]) for s in spots]
    board = [pad_board(ids(s["board"])) for s in spots]
    trials = 4000000
    out = _run_batch(torch, hole, board, [2] * len(spots), trials, 8, "reference")
    for i, s in enumerate(spots):
        num, den = s["reference_mode"]
        p = num / den
        got = (out["wins"][i] + out["ties"][i]) / trials
        assert abs(got - p) <= 3 * sigma(p, trials) + 1e-9, (s["name"], got, p)


def test_reference_mode_within_3_sigma_of_reference_runs(torch_mod, golden_mc):
    """Sampled equities vs the reference's own seeded runs (mc_seeded.json): |p_gpu - p_ref| <= 3 sigma of the
    reference's binomial standard error at ITS trial count (the GPU runs 400k trials, so its own error is negligible)."""
    torch = torch_mod
    by_name = {}
    for r in golden_mc["runs"]:
        e = by_name.setdefault(r["name"], {"hero": r["hero"], "board": r["board"], "players": r["players"], "w": 0, "n": 0})
        e["w"] += r["wins"]
        e["n"] += r["runs"]
    names = sorted(by_name)
    hole = [ids(by_name[n]["hero"]) for n in names]
    board = [pad_board(ids(by_name[n]["board"])) for n in names]
    npl = [by_name[n]["players"] for n in names]
    trials = 400000
    out = _run_batch(torch, hole, board, npl, trials, 31337, "reference")
    for i, n in enumerate(names):
        e = by_name[n]
        p_ref = e["w"] / e["n"]
        p_gpu = (out["wins"][i] + out["ties"][i]) / trials
        assert abs(p_gpu - p_ref) <= 3 * math.sqrt(sigma(p_gpu, e["n"]) ** 2 + sigma(p_gpu, trials) ** 2), (n, p_gpu, p_ref)


def test_dropin_api(torch_mod):
    """get_equity / montecarlo / MonteCarlo mirror the reference's signatures, types and argument handling."""
    npk.seed(5)
    eq = npk.get_equity({"AS", "KS"}, set(), np.int64(2), 20000)          # env passes sets and numpy.int64 (env.py:261-262)
    assert isinstance(eq, float) and abs(eq - 0.6608) < 0.015             # reference dealer: 0.661 (SURVEY A.2)
    eq = npk.montecarlo({"AS", "KS"}, {"null"}, 2, 20000)                  # C++ call site convention for "no board"
    assert isinstance(eq, float) and abs(eq - 0.6795) < 0.015             # uniform dealing: 0.679
    assert npk.get_equity(["8S", "2S"], ["5S", "3S", "4S", "KS", "AS"], 2, 2000) == 1.0     # test_montecarlo7
    assert npk.get_equity({"AS", "KS"}, set(), 1, 500) == 1.0             # players == 1 -> 1.0 (SURVEY 8b)
    mc = npk.MonteCarlo()
    equity, win_types = mc.run_montecarlo([["3H", "3S"]], ["8S", "4S", "QH", "8C", "4H"], 2, 1, maxRuns=15000,
                                          timeout=0, ghost_cards="", opponent_range=1)
    assert abs(equity * 100 - 40.2) < 3                                    # tests/test_montecarlo_python.py:44-50, :40
    assert abs(sum(mc.winnerCardTypeList.values()) - equity) < 1e-4       # :32
    assert mc.runs == 15000 and mc.passes >= 15000 and dict(win_types) == dict(mc.winnerCardTypeList)
    with pytest.raises(ValueError):
        npk.get_equity({"AS", "XX"}, set(), 2, 10)
    npk.seed(5)
    a = npk.get_equity({"AS", "KS"}, set(), 2, 3000)
    npk.seed(5)
    assert npk.get_equity({"AS", "KS"}, set(), 2, 3000) == a              # reproducible under a fixed seed
    np.random.seed(11); npk.seed(None)
    b = npk.get_equity({"AS", "KS"}, set(), 2, 3000)
    np.random.seed(11)
    assert npk.get_equity({"AS", "KS"}, set(), 2, 3000) == b              # np.random.seed governs it like the reference


def test_reference_montecarlo_test_spots(torch_mod, golden_enum):
    """The reference's own 19 non-range Monte-Carlo spots with its own acceptance rule:
    |mean of 5 runs - expected| < 3 points and stdev < 3 (tests/test_montecarlo_python.py:15-41)."""
    npk.seed(1)
    for s in golden_enum["spots"]:
        res = [100 * npk.get_equity(s["hero"], s["board"], s["players"], 15000) for _ in range(5)]
        assert abs(np.mean(res) - s["test_expected_pct"]) < 3 and np.std(res) < 3, (s["name"], res)


def test_numpy_sibling_call_form(torch_mod, golden_enum):
    """numpy_montecarlo(my_cards, table, iterations, player_amount) -> per cent (tools/montecarlo_numpy2.py:333-346): the 19
    spots of the sibling's own (upstream skipped) tests/test_montecarlo_numpy.py with their +-1 point rule, at 200,000 runs."""
    npk.seed(2)
    for s in golden_enum["spots"]:
        got = npk.numpy_montecarlo([list(s["hero"])], list(s["board"]), 200000, s["players"])
        assert abs(got - s["test_expected_pct"]) < 1.0, (s["name"], got, s["test_expected_pct"])
        if s.get("uniform"):                                   # exact (win, tie, lose) counts under uniform dealing
            w, t, l = s["uniform"]
            exact = (w + t) / (w + t + l)
            assert abs(got / 100 - exact) < 4 * sigma(exact, 200000) + 1e-9, (s["name"], got, exact)


def test_invalid_queries_are_reported(torch_mod):
    torch = torch_mod
    with pytest.raises(_lib.NpkError) as e:
        _run_batch(torch, [[51, 51]], [pad_board([])], [2], 10, 0, "uniform")
    assert e.value.code == -5
    with pytest.raises(_lib.NpkError):
        _run_batch(torch, [[0, 1]], [[2, NO, 3, NO, NO]], [2], 10, 0, "uniform")
    with pytest.raises(_lib.NpkError):
        _run_batch(torch, [[0, 1]], [pad_board([])], [11], 10, 0, "reference")
    out = _run_batch(torch, np.zeros((0, 2)), np.zeros((0, 5)), np.zeros((0,)), 10, 0, "uniform")
    assert out["wins"].shape == (0,)


def test_evaluator_entry_points_validate_their_inputs(torch_mod):
    """npk_rank7_batch / npk_showdown_batch / npk_enum_batch with NPK_FLAG_VALIDATE (the default for host arrays): a card id
    >= 52 -- including the 0xFF pad -- a duplicate card, n_players out of range or an enumeration shape the kernel does not
    implement is an error, not an out-of-bounds gather (the reference raises ValueError / RuntimeError there).  Without the
    flag the call is the caller's responsibility but must stay memory-safe."""
    torch = torch_mod
    good = np.array([[0, 5, 9, 13, 22, 37, 51]], dtype=np.uint8)
    assert int(npk.rank7(good)[0]) == int(npk.host_rank7(good)[0])
    for bad in ([[0, 5, 9, 13, 22, 37, 52]], [[0, 5, 9, 13, 22, 37, 255]], [[0, 5, 9, 13, 22, 37, 37]]):
        with pytest.raises(_lib.NpkError) as e:
            npk.rank7(np.array(bad, dtype=np.uint8))
        assert e.value.code == -5
    junk = torch.randint(0, 256, (4096, 7), dtype=torch.uint8, device="cuda")
    npk.rank7(junk, validate=False)                      # garbage in, garbage out -- but no fault
    torch.cuda.synchronize()
    hole, board = np.array([[0, 1]], dtype=np.uint8), np.array([[2, 3, 4, 5, 6]], dtype=np.uint8)
    with pytest.raises(_lib.NpkError) as e:
        npk.enumerate_equity(hole, board, np.array([4], dtype=np.uint8))          # four players: not implemented
    assert e.value.code == -2
    with pytest.raises(_lib.NpkError) as e:
        npk.enumerate_equity(hole, np.array([[2, 3, 4, NO, NO]], dtype=np.uint8), np.array([3], dtype=np.uint8))
    assert e.value.code == -2
    with pytest.raises(_lib.NpkError) as e:
        npk.enumerate_equity(np.array([[0, 60]], dtype=np.uint8), board)
    assert e.value.code == -5
    with pytest.raises(_lib.NpkError) as e:
        npk.enumerate_equity(hole, np.array([[2, NO, 4, NO, NO]], dtype=np.uint8))  # gap in the board
    assert e.value.code == -5
    w, t, l = npk.enumerate_equity(torch.randint(0, 256, (64, 2), dtype=torch.uint8, device="cuda"),
                                   torch.randint(0, 256, (64, 5), dtype=torch.uint8, device="cuda"), validate=False)
    torch.cuda.synchronize()
    holes = np.array([[[0, 1], [2, 3], [255, 255]]], dtype=np.uint8)
    brd = np.array([[10, 20, 30, 40, 50]], dtype=np.uint8)
    npk.showdown(holes, np.array([2], dtype=np.uint8), brd)                       # unused third seat may hold anything
    with pytest.raises(_lib.NpkError) as e:
        npk.showdown(holes, np.array([3], dtype=np.uint8), brd)
    assert e.value.code == -5
    with pytest.raises(_lib.NpkError) as e:
        npk.showdown(holes, np.array([4], dtype=np.uint8), brd)
    assert e.value.code == -2
    with pytest.raises(_lib.NpkError):
        npk.showdown(np.array([[[0, 1], [1, 3], [4, 5]]], dtype=np.uint8), np.array([2], dtype=np.uint8), brd)


def test_mixed_batch_status_reports_skipped_and_invalid_queries(torch_mod):
    """npk_equity_batch_async validates nothing by itself; npk_equity_batch_status tells afterwards how many queries of the
    last call were invalid or outside the shape mask (their counters are untouched)."""
    import ctypes
    torch = torch_mod
    hole = torch.tensor([[0, 1], [2, 3], [4, 4], [6, 7]], dtype=torch.uint8, device="cuda")
    board = torch.full((4, 5), NO, dtype=torch.uint8, device="cuda")
    npl = torch.tensor([2, 3, 2, 2], dtype=torch.uint8, device="cuda")
    L = _lib.ensure_init(0)
    ws = torch.empty(int(L.npk_equity_workspace_bytes(4)), dtype=torch.uint8, device="cuda")
    wins = torch.zeros(4, dtype=torch.int64, device="cuda")
    ties = torch.zeros(4, dtype=torch.int64, device="cuda")
    mask = npk.equity.shape_mask([2], [0])
    _lib.check(L.npk_equity_batch_async(hole.data_ptr(), board.data_ptr(), npl.data_ptr(), 4, 500, ctypes.c_uint64(mask),
                                        ctypes.c_uint64(5), 0, 0, 0, wins.data_ptr(), ties.data_ptr(), None, None,
                                        ws.data_ptr(), torch.cuda.current_stream().cuda_stream))
    inv, skp = ctypes.c_uint32(0), ctypes.c_uint32(0)
    _lib.check(L.npk_equity_batch_status(ws.data_ptr(), torch.cuda.current_stream().cuda_stream, ctypes.byref(inv), ctypes.byref(skp)))
    assert (inv.value, skp.value) == (1, 1)
    tot = (wins + ties).cpu().tolist()
    assert tot[0] > 0 and tot[3] > 0 and tot[1] == 0 and tot[2] == 0


def test_one_query_fast_path_equals_the_batched_path(torch_mod):
    """npk_equity_host with one query takes a copy-free path (query in the kernel parameters, counters resident on the
    device and reset by the last warp, results in mapped host memory).  Same seed, same query => the same counters as
    the batched path, call after call, in both dealing modes and with win types / passes.  The last spot asks for wins and
    ties only, with more trials (2**28) than the packed hand-over of the one-shot kernel can count."""
    import neuron_poker_b200 as npk
    spots = [(["AS", "KS"], ["2C", "7D", "KH"], 6, 10000), (["3H", "3S"], ["8S", "4S", "QH", "8C", "4H"], 2, 777),
             (["7D", "7C"], [], 10, 4097), (["AS", "AD"], [], 1, 100), (["JD", "JS"], ["8C", "TC", "JC", "5H"], 3, 31),
             (["AH", "KD"], [], 2, 2**28)]
    for rep in range(3):
        for mode in ("uniform", "reference"):
            for h, b, p, runs in spots:
                types = runs < 2**28
                one = npk.equity_counts(h, b, p, runs, deal_mode=mode, seed_value=99 + rep, win_types=types,
                                        passes=types and mode == "reference")
                two = npk.equity_counts_batch(np.array([ids(h), ids(h)], dtype=np.uint8),
                                              np.array([pad_board(ids(b))] * 2, dtype=np.uint8),
                                              np.array([p, p], dtype=np.uint8), runs, seed_value=99 + rep, deal_mode=mode,
                                              win_types=types, passes=types and mode == "reference")
                assert (one["wins"], one["ties"]) == (int(two["wins"][0]), int(two["ties"][0])), (mode, h, b, p)
                if types:
                    assert one["win_types"] == [int(x) for x in two["win_types"][0]]
                if types and mode == "reference":
                    assert one["passes"] == int(two["passes"][0])
                assert one["wins"] + one["ties"] <= runs


def test_mixed_kernel_equals_the_per_shape_kernels(torch_mod):
    """A mixed batch runs through ONE persistent kernel for all shapes (csrc/npk_mixed.cu, via npk_equity_batch and via
    npk_equity_batch_async with a shape mask): same counters, win types and passes as the shape-specialised kernels give query
    by query (uniform_shape hint, the query's own number in the Philox counter), in both dealing modes; queries whose shape is
    not in the mask are left untouched."""
    import neuron_poker_b200 as npk
    from neuron_poker_b200.equity import shape_mask
    rng = np.random.default_rng(11)
    Q = 300
    hole, board, npl = [], [], []
    for q in range(Q):
        known = [0, 3, 4, 5][rng.integers(0, 4)]
        c = rng.permutation(52)[:2 + known].tolist()
        hole.append(c[:2]); board.append(pad_board(c[2:])); npl.append(int(rng.integers(1, 8)))
    hole, board, npl = (np.array(x, dtype=np.uint8) for x in (hole, board, npl))
    for mode in ("uniform", "reference"):
        a = npk.get_equity_batch(hole, board, npl, 777, seed_value=21, deal_mode=mode, win_types=True, passes=(mode == "reference"),
                                 trial_offset=3, query_offset=9)
        b = npk.get_equity_batch(hole, board, npl, 777, seed_value=21, deal_mode=mode, win_types=True, passes=(mode == "reference"),
                                 trial_offset=3, query_offset=9, shapes=shape_mask(range(1, 8)))
        for k in ("wins", "ties", "win_types") + (("passes",) if mode == "reference" else ()):
            assert (a[k] == b[k]).all(), (mode, k)
        for q in range(Q):
            known = int((board[q] != NO).sum())
            one = npk.get_equity_batch(hole[q:q + 1], board[q:q + 1], npl[q:q + 1], 777, seed_value=21, deal_mode=mode,
                                       win_types=True, passes=(mode == "reference"), trial_offset=3, query_offset=9 + q,
                                       uniform_shape=(int(npl[q]), known), validate=False)
            for k in ("wins", "ties", "win_types") + (("passes",) if mode == "reference" else ()):
                assert (one[k][0] == a[k][q]).all(), (mode, k, q, int(npl[q]), known)
        c = npk.get_equity_batch(hole, board, npl, 777, seed_value=21, deal_mode=mode, shapes=shape_mask([2, 3]),
                                 trial_offset=3, query_offset=9)
        sel = torch_mod.as_tensor((npl == 2) | (npl == 3)).to(c["wins"].device)
        assert (c["wins"][sel] == a["wins"][sel]).all() and (c["wins"][~sel] == 0).all() and (c["ties"][~sel] == 0).all()


def test_host_entry_points_are_reentrant(torch_mod):
    """npk_equity_one / npk_equity_host from several host threads at once (ctypes releases the GIL): every thread owns its
    stream, staging and one-query scratch inside libnpk, so concurrent calls return exactly what the same calls return alone."""
    import threading
    spots = [({"AS", "KS"}, {"2C", "7D", "KH"}, 6), ({"3H", "3S"}, {"8S", "4S", "QH", "8C", "4H"}, 2), ({"TD", "7D"}, set(), 4),
             ({"QC", "QD"}, {"2C", "7D", "KH", "9S"}, 3)]
    want = {}
    for i, (h, b, n) in enumerate(spots):
        for mode in ("uniform", "reference"):
            r = npk.equity_counts(h, b, n, 5000, deal_mode=mode, seed_value=100 + i, win_types=(i & 1) == 1)
            want[(i, mode)] = (r["wins"], r["ties"], tuple(r.get("win_types", ())))
    rng = np.random.default_rng(4)
    cards = np.stack([rng.permutation(52)[:5] for _ in range(33)]).astype(np.uint8)
    bh, bb = cards[:, :2].copy(), np.full((33, 5), NO, dtype=np.uint8)
    bb[:, :3] = cards[:, 2:]
    bn = np.full(33, 5, dtype=np.uint8)
    batch_want = npk.equity_counts_batch(bh, bb, bn, 640, seed_value=9)
    errors = []

    def worker(tid):
        try:
            for rep in range(60):
                i = (tid + rep) % len(spots)
                mode = "reference" if (tid + rep) & 1 else "uniform"
                h, b, n = spots[i]
                r = npk.equity_counts(h, b, n, 5000, deal_mode=mode, seed_value=100 + i, win_types=(i & 1) == 1)
                got = (r["wins"], r["ties"], tuple(r.get("win_types", ())))
                if got != want[(i, mode)]:
                    errors.append((tid, rep, got, want[(i, mode)]))
                if rep % 15 == 0:
                    o = npk.equity_counts_batch(bh, bb, bn, 640, seed_value=9)
                    if not ((o["wins"] == batch_want["wins"]).all() and (o["ties"] == batch_want["ties"]).all()):
                        errors.append((tid, rep, "batch"))
        except Exception as exc:          # noqa: BLE001
            errors.append((tid, repr(exc)))

    threads = [threading.Thread(target=worker, args=(t,)) for t in range(6)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errors, errors[:3]


def test_pipelined_host_batches_equal_blocking_calls(torch_mod):
    """npk_equity_host_submit / npk_equity_host_wait (equity_counts_batch(block=False)): batches kept in flight give exactly
    the counters of the blocking call with the same arguments -- uniform-shape and mixed batches, both dealers, win types and
    passes, collected out of order; a fifth outstanding ticket, a ticket waited for twice and bad cards are errors."""
    from neuron_poker_b200._lib import NpkError
    rng = np.random.default_rng(21)
    jobs = []
    for k in range(7):
        Q = int(rng.integers(3, 400))
        cards = np.stack([rng.permutation(52)[:7] for _ in range(Q)]).astype(np.uint8)
        known = rng.choice([0, 3, 4, 5], size=Q) if k % 2 else np.full(Q, [3, 0, 4, 5][k // 2 % 4])
        board = cards[:, 2:].copy()
        for q in range(Q):
            board[q, known[q]:] = NO
        npl = rng.integers(2, 8, size=Q).astype(np.uint8) if k % 2 else np.full(Q, 2 + k, dtype=np.uint8)
        mode = "reference" if k % 3 == 0 else "uniform"
        kw = dict(seed_value=300 + k, deal_mode=mode, win_types=k % 2 == 0, passes=(mode == "reference"))
        jobs.append((cards[:, :2].copy(), board, npl, 500 + 37 * k, kw))
    want = [npk.equity_counts_batch(h, b, n, t, **kw) for h, b, n, t, kw in jobs]
    pend, got = [], {}
    for i, (h, b, n, t, kw) in enumerate(jobs):
        pend.append((i, npk.equity_counts_batch(h, b, n, t, block=False, **kw)))
        h[:] = 0                                     # the queries were copied at submission
        if len(pend) == npk.equity.MAX_IN_FLIGHT:
            j, p = pend.pop(1)                       # out of order
            got[j] = p.result()
    for j, p in pend:
        got[j] = p.result()
    for i, w in enumerate(want):
        assert set(got[i]) == set(w)
        for k in w:
            assert (got[i][k] == w[k]).all(), (i, k)
    h, b, n, t, kw = jobs[1]
    h[:] = 5                                         # the same card twice: rejected at submission
    with pytest.raises(NpkError):
        npk.equity_counts_batch(h, b, n, t, block=False)
    h2, b2, n2, t2, kw2 = jobs[2]
    h2[:] = 50
    h2[:, 1] = 51
    b2[:] = NO
    many = [npk.equity_counts_batch(h2, b2, n2, 64, block=False) for _ in range(npk.equity.MAX_IN_FLIGHT)]
    with pytest.raises(NpkError):
        npk.equity_counts_batch(h2, b2, n2, 64, block=False)
    first = many[0].result()
    again = npk.equity_counts_batch(h2, b2, n2, 64, block=False)        # a slot is free again
    for p in many[1:] + [again]:
        r = p.result()
        assert (r["wins"] == first["wins"]).all()
    L = npk._lib.lib()
    assert L.npk_equity_host_wait(10**6, None, None, None, None) < 0


def test_resident_server_equals_launch_per_call(torch_mod):
    """Resident mode (npk_resident_start): a persistent kernel serves the one-query calls of this thread from a mailbox in
    mapped host memory.  Same counters as the launch-per-call path for every shape and both dealers; the server leaves after its
    idle limit and the next call starts it again; calls it does not serve (win types, batches) stop it first; errors as before."""
    import time
    spots = [({"AS", "KS"}, {"2C", "7D", "KH"}, 6), ({"3H", "3S"}, {"8S", "4S", "QH", "8C", "4H"}, 2), ({"TD", "7D"}, set(), 4),
             ({"QC", "QD"}, {"2C", "7D", "KH", "9S"}, 3), ({"2C", "2D"}, set(), 10), ({"AH", "KD"}, {"2C", "7D", "KH"}, 1)]
    runs = [10000, 777, 64, 1, 130000, 0]
    want = {}
    for i, (h, b, n) in enumerate(spots):
        for mode in ("uniform", "reference"):
            for t in runs:
                r = npk.equity_counts(h, b, n, t, deal_mode=mode, seed_value=100 + i)
                want[(i, mode, t)] = (r["wins"], r["ties"])
    try:
        npk.resident(True, idle_us=300)
        for rep in range(3):
            for i, (h, b, n) in enumerate(spots):
                for mode in ("uniform", "reference"):
                    for t in runs:
                        r = npk.equity_counts(h, b, n, t, deal_mode=mode, seed_value=100 + i)
                        assert (r["wins"], r["ties"]) == want[(i, mode, t)], (rep, i, mode, t)
            time.sleep(0.02)                               # the server has left by now: the next call restarts it
        eq = npk.get_equity({"AS", "KS"}, {"2C", "7D", "KH"}, 6, 10000)
        assert 0.3 < eq < 0.9
        h, b, n = spots[0]
        a = npk.equity_counts(h, b, n, 5000, deal_mode="reference", seed_value=5, win_types=True, passes=True)   # launch path
        npk.resident(False)
        c = npk.equity_counts(h, b, n, 5000, deal_mode="reference", seed_value=5, win_types=True, passes=True)
        assert a == c
        npk.resident(True, sms=16, idle_us=100000)         # a server on 16 SMs that stays
        r = npk.equity_counts(h, b, n, 10000, deal_mode="uniform", seed_value=100)
        assert (r["wins"], r["ties"]) == want[(0, "uniform", 10000)]
        hole = np.array([[50, 51]] * 40, dtype=np.uint8)
        board = np.full((40, 5), NO, dtype=np.uint8)
        npl = np.full(40, 3, dtype=np.uint8)
        b1 = npk.equity_counts_batch(hole, board, npl, 640, seed_value=9)            # stops the server, runs, returns
        r = npk.equity_counts(h, b, n, 10000, deal_mode="uniform", seed_value=100)   # and the server comes back
        assert (r["wins"], r["ties"]) == want[(0, "uniform", 10000)]
        with pytest.raises(ValueError):
            npk.get_equity({"AS", "AS"}, set(), 2, 100)
        npk.resident(False)
        b2 = npk.equity_counts_batch(hole, board, npl, 640, seed_value=9)
        assert (b1["wins"] == b2["wins"]).all() and (b1["ties"] == b2["ties"]).all()
    finally:
        npk.resident(False)


def test_one_resident_server_per_device(torch_mod):
    """A second host thread cannot start a resident server on a device that already has one (its kernel could not get the SMs
    the first one holds); it can once the first thread has stopped its own; its launched calls work throughout."""
    import threading
    from neuron_poker_b200._lib import NpkError
    want = npk.equity_counts({"AS", "KS"}, {"2C", "7D", "KH"}, 6, 5000, deal_mode="uniform", seed_value=1)
    res = {}

    def other(tag):
        try:
            npk.resident(True)
            res[tag] = "started"
            res[tag + "_counts"] = npk.equity_counts({"AS", "KS"}, {"2C", "7D", "KH"}, 6, 5000, deal_mode="uniform", seed_value=1)
            npk.resident(False)
        except NpkError as exc:
            res[tag] = exc.code
            res[tag + "_counts"] = npk.equity_counts({"AS", "KS"}, {"2C", "7D", "KH"}, 6, 5000, deal_mode="uniform", seed_value=1)

    try:
        npk.resident(True, idle_us=2000)
        t = threading.Thread(target=other, args=("while",))
        t.start(); t.join()
        assert res["while"] == -2 and res["while_counts"] == want
        assert npk.equity_counts({"AS", "KS"}, {"2C", "7D", "KH"}, 6, 5000, deal_mode="uniform", seed_value=1) == want
    finally:
        npk.resident(False)
    t = threading.Thread(target=other, args=("after",))
    t.start(); t.join()
    assert res["after"] == "started" and res["after_counts"] == want


def test_rank7_quad_path_agrees_with_the_scalar_path_and_the_oracle(torch_mod):
    """rank7_kernel evaluates four hands per thread from seven aligned words (the quad loop) and falls back to one hand per
    thread for an unaligned batch and for the last n % 4 hands.  One million hands through both, a flush-heavy batch included
    (every third hand: the divergent flush branch in nearly every lane), and a sample against the oracle."""
    torch = torch_mod
    rng = np.random.default_rng(12)
    n = 1_000_003
    base = rng.random((n, 52)).argsort(1)[:, :7].astype(np.uint8)
    # every third hand gets five cards of one suit
    suits = rng.integers(0, 4, n)
    ranks = rng.random((n, 13)).argsort(1)[:, :5]
    fl = (4 * ranks + suits[:, None]).astype(np.uint8)
    heavy = base.copy()
    sel = np.arange(n) % 3 == 0
    other = np.array([[(4 * r + (s + 1) % 4) for r in (0, 1)] for s in range(4)], dtype=np.uint8)      # two cards of the next suit
    heavy[sel, :5] = fl[sel]
    heavy[sel, 5:] = other[suits[sel]]
    for cards in (base, heavy):
        dev = torch.as_tensor(cards).cuda()
        quad = npk.rank7(dev).cpu().numpy()
        flat = torch.zeros(7 * n + 1, dtype=torch.uint8, device="cuda")
        flat[1:] = dev.reshape(-1)
        scalar = npk.rank7(flat[1:].view(n, 7)).cpu().numpy()                  # pointer % 4 == 1: the scalar path
        assert (quad == scalar).all()
        idx = rng.integers(0, n, 60000)
        assert (quad[idx] == oracle.rank7_batch(cards[idx])).all()
        assert (quad >= 3225).sum() >= (n // 3 if cards is heavy else n // 50)  # flushes and better are really in there
