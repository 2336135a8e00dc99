"""Exact enumeration under the reference's dealer (npk_enum_dealer_batch / enumerate_equity(deal_mode="reference") /
exact_equity): the value get_equity converges to.

CPU: tests/enum_reference_oracle.c plays the dealer of montecarlo_python.py:165-189 literally over every index sequence it can
draw; it reproduces the eleven REFERENCE-mode fractions of enum_golden.json, it equals the weight formulation of include/npk.h
(numerators and totals, and the totals equal their closed forms), and it equals the sum over opponent hands of the weight
times the REFERENCE-mode showdown equity of hero + that hand (tests/showdown_oracle.c) -- the identity the preflop GPU check
uses.
GPU: the kernel bit-exact against the literal dealer on every non-preflop shape and against the golden fractions; preflop and
one / two known board cards against the weighted sum of showdown_equity_batch(deal_mode="reference") over every opponent hand;
the UNIFORM mode against npk_enum_batch; independence of the batch; validation; get_equity's AsKs heads-up preflop value; and
every REFERENCE-mode Monte-Carlo path within 4 sigma of the exact values.
"""
import ctypes
import math
import os
import shutil
import subprocess
import tempfile

import numpy as np
import pytest

import oracle
import showdown_oracle

HERE = os.path.dirname(os.path.abspath(__file__))
NO = 0xFF
# exact_equity({'AS','KS'}, set(), 2): (win + tie) / total of the weighted enumeration, total = 49^2 C(47,5)
ASKS_PREFLOP = (2369128797, 61048101, 1252810641)

_lib = None


def ref_lib():
    """tests/enum_reference_oracle.c, compiled with the C compiler into a temporary directory on first use."""
    global _lib
    if _lib is None:
        cc = os.environ.get("CC") or shutil.which("gcc") or shutil.which("cc")
        if not cc:
            raise RuntimeError("no C compiler for tests/enum_reference_oracle.c")
        tmp = tempfile.mkdtemp(prefix="npk_enum_reference_oracle_")
        try:
            out = os.path.join(tmp, "libenum_reference_oracle.so")
            subprocess.check_call([cc, "-O2", "-std=c11", "-fPIC", "-shared", "-Wall",
                                   os.path.join(HERE, "enum_reference_oracle.c"), "-o", out])
            L = ctypes.CDLL(out)                   # stays mapped after the file is gone
        finally:
            shutil.rmtree(tmp, ignore_errors=True)
        u8p = ctypes.POINTER(ctypes.c_uint8)
        for name in ("enum_reference_literal", "enum_reference_weighted"):
            getattr(L, name).argtypes = [ctypes.c_void_p, u8p, u8p, ctypes.c_int, ctypes.c_int, ctypes.POINTER(ctypes.c_int64)]
        O = oracle.lib()
        O.oracle_fast_init()
        L.rank7 = ctypes.cast(O.oracle_rank7_fast, ctypes.c_void_p)
        _lib = L
    return _lib


def _call(name, hero, board, players):
    L = ref_lib()
    h, b = oracle.ids(hero), oracle.ids(board)
    out = (ctypes.c_int64 * 3)()
    p = lambda a: a.ctypes.data_as(ctypes.POINTER(ctypes.c_uint8))
    rc = getattr(L, name)(L.rank7, p(h), p(b) if len(b) else None, len(b), int(players), out)
    assert rc == 0, (name, rc)
    return tuple(out)


def literal(hero, board, players=2):
    return _call("enum_reference_literal", hero, board, players)


def weighted(hero, board, players=2):
    return _call("enum_reference_weighted", hero, board, players)


def total(nb, players):
    n = 50 - nb
    return (n - 1) ** 2 * (math.comb(n - 3, 5 - nb) if players == 2 else (n - 3) ** 2)


def spots(seed, count, nb, players=2):
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(count):
        c = [int(x) for x in rng.permutation(52)[:2 + nb]]
        out.append((c[:2], c[2:], players))
    return out


def opponent_hands(hero, board):
    """(hand, weight) of every opponent hand: slots a < b of the unseen cards, weight 2 - [b == a + 1]."""
    r = sorted(set(range(52)) - set(hero) - set(board))
    return [((r[a], r[b]), 2 - (b == a + 1)) for a in range(len(r)) for b in range(a + 1, len(r))]


# ---- CPU ---------------------------------------------------------------------------------------------------------------
def test_literal_dealer_reproduces_the_golden_fractions(golden_enum):
    n = 0
    for s in golden_enum["spots"]:
        if "reference_mode" in s:
            w, t, l = literal(s["hero"], s["board"], s["players"])
            assert [w + t, w + t + l] == s["reference_mode"], s["name"]
            n += 1
    assert n == 11


@pytest.mark.parametrize("nb,players,count,seed", [(5, 2, 8, 1), (4, 2, 4, 2), (3, 2, 2, 3), (5, 3, 2, 4)])
def test_weights_equal_the_literal_dealer(nb, players, count, seed):
    for hero, board, p in spots(seed, count, nb, players):
        lit = literal(hero, board, p)
        assert weighted(hero, board, p) == lit, (hero, board, p)
        assert sum(lit) == total(nb, p)
    # the highest unseen ids in the hand or on the board move the excluded slot: hero / board holding 51, 50, 49
    for hero, board in (([51, 50], [49, 0, 1, 2, 3]), ([0, 50], [51, 7, 9, 11]), ([51, 1], [48, 47, 46])):
        lit = literal(hero, board)
        assert weighted(hero, board) == lit and sum(lit) == total(len(board), 2), (hero, board)


def test_showdown_sum_equals_the_literal_dealer():
    """sum over opponent hands of w * (REFERENCE-mode showdown equity of hero + that hand) = the literal dealer."""
    for hero, board, _ in spots(5, 2, 5) + spots(6, 1, 4) + spots(7, 1, 3):
        acc = [0, 0, 0]
        for hand, w in opponent_hands(hero, board):
            r = showdown_oracle.showdown_equity([hero, list(hand)], board, deal_mode="reference")
            acc[0] += w * r["win"][0]
            acc[1] += w * r["tie"][0]
            acc[2] += w * (r["completions"] - r["win"][0] - r["tie"][0])
        assert tuple(acc) == literal(hero, board), (hero, board)


def test_bad_deal_mode_needs_no_device():
    """deal_mode is checked before the device is touched (null pointers are never looked at)."""
    from neuron_poker_b200 import _lib as nl
    L = nl.lib()
    for mode in (-1, 2, 99):
        rc = L.npk_enum_dealer_batch(None, None, None, 1, mode, None, None, None, nl.NPK_FLAG_VALIDATE, None)
        assert rc == -2 and "deal_mode" in L.npk_last_error().decode(), (mode, rc)


def test_exact_equity_rejects_bad_input_before_the_device():
    import neuron_poker_b200 as npk
    for args in ((["AS", "XX"], [], 2), (["AS", "AS"], [], 2), (["AS", "KS"], ["AS", "2C", "3C"], 2),
                 (["AS"], [], 2), (["AS", "KS"], ["2C", "3C", "4C", "5C", "6C", "7C"], 2)):
        with pytest.raises(ValueError):
            npk.exact_equity(*args)
    for hand, board, players in ((["AS", "KS"], ["2C", "3C", "4C", "5C"], 3), (["AS", "KS"], [], 4), (["AS", "KS"], [], 1)):
        with pytest.raises(ValueError, match="two players with 0..5 table cards or three players with five"):
            npk.exact_equity(hand, board, players)
    with pytest.raises(ValueError, match="deal_mode"):
        npk.exact_equity(["AS", "KS"], [], 2, deal_mode="biased")


# ---- GPU ---------------------------------------------------------------------------------------------------------------
def _arrays(batch):
    hole = np.array([h for h, _, _ in batch], dtype=np.uint8)
    board = np.array([b + [NO] * (5 - len(b)) for _, b, _ in batch], dtype=np.uint8)
    npl = np.array([p for _, _, p in batch], dtype=np.uint8)
    return hole, board, npl


def _enum(batch, device, deal_mode="reference"):
    import neuron_poker_b200 as npk
    w, t, l = npk.enumerate_equity(*_arrays(batch), device=device, deal_mode=deal_mode)
    return list(zip(w.tolist(), t.tolist(), l.tolist()))


def _showdown_sum(hero, board, device):
    """sum over opponent hands of w * showdown_equity_batch(deal_mode="reference") of hero + that hand, on the GPU."""
    import neuron_poker_b200 as npk
    opp = opponent_hands(hero, board)
    holes = np.array([[hero, list(h)] for h, _ in opp], dtype=np.uint8)
    brd = np.tile(np.array(board + [NO] * (5 - len(board)), dtype=np.uint8), (len(opp), 1))
    out = npk.showdown_equity_batch(holes, np.full(len(opp), 2, dtype=np.uint8), brd, deal_mode="reference", device=device)
    w = np.array([x for _, x in opp], dtype=np.int64)
    win, tie = out["win"][:, 0].cpu().numpy(), out["tie"][:, 0].cpu().numpy()
    comp = out["completions"].cpu().numpy()
    return int((w * win).sum()), int((w * tie).sum()), int((w * (comp - win - tie)).sum())


NON_PREFLOP = spots(11, 16, 5) + spots(12, 8, 4) + spots(13, 3, 3) + spots(14, 6, 5, 3) + \
    [([51, 50], [49, 0, 1, 2, 3], 2), ([0, 50], [51, 7, 9, 11], 2), ([51, 1], [48, 47, 46], 2), ([51, 50], [49, 48, 0, 1, 2], 3)]


@pytest.mark.gpu
def test_gpu_bitexact_vs_the_literal_dealer(cuda_device, golden_enum):
    got = _enum(NON_PREFLOP, cuda_device)
    for (hero, board, p), g in zip(NON_PREFLOP, got):
        assert g == literal(hero, board, p), (hero, board, p)
    gold = [s for s in golden_enum["spots"] if "reference_mode" in s]
    got = _enum([(oracle.ids(s["hero"]).tolist(), oracle.ids(s["board"]).tolist(), s["players"]) for s in gold], cuda_device)
    for s, (w, t, l) in zip(gold, got):
        assert [w + t, w + t + l] == s["reference_mode"], s["name"]


@pytest.mark.gpu
@pytest.mark.slow
def test_gpu_preflop_and_early_boards_vs_weighted_showdown(cuda_device):
    """Preflop (the generic walk's main case) and one or two known board cards: the kernel equals the weighted sum of the
    REFERENCE-mode showdown equity of hero + every opponent hand, which is pinned to the literal pops.  A preflop query is
    one CTA walking 2.1 G completion x hand pairs: about 112 s on a B200 (DESIGN.md section 4.4)."""
    batch = [([51, 47], [], 2), ([0, 1], [], 2)] + spots(15, 1, 1) + spots(16, 2, 2)
    got = _enum(batch, cuda_device)
    for (hero, board, p), g in zip(batch, got):
        assert g == _showdown_sum(hero, board, cuda_device), (hero, board)
        assert sum(g) == total(len(board), 2)
    assert got[0] == ASKS_PREFLOP


@pytest.mark.gpu
def test_gpu_uniform_mode_is_npk_enum_batch(cuda_device):
    import torch
    import neuron_poker_b200 as npk
    from neuron_poker_b200 import _lib as nl
    batch = NON_PREFLOP + spots(17, 2, 2)
    hole, board, npl = (torch.as_tensor(a).to(cuda_device) for a in _arrays(batch))
    Q = len(batch)
    L = nl.ensure_init(cuda_device.index)
    outs = []
    for call in ("npk_enum_batch", "npk_enum_dealer_batch"):
        o = [torch.zeros(Q, dtype=torch.int64, device=cuda_device) for _ in range(3)]
        mode = () if call == "npk_enum_batch" else (nl.NPK_DEAL_UNIFORM,)
        nl.check(getattr(L, call)(hole.data_ptr(), board.data_ptr(), npl.data_ptr(), Q, *mode, *(x.data_ptr() for x in o),
                                  nl.NPK_FLAG_VALIDATE, torch.cuda.current_stream(cuda_device).cuda_stream))
        outs.append([x.tolist() for x in o])
    default = [x.tolist() for x in npk.enumerate_equity(hole, board, npl)]
    assert outs[0] == outs[1] == default
    ref = _enum(batch, cuda_device)
    assert [tuple(x) for x in zip(*outs[0])] != ref          # the two dealers differ on these spots


@pytest.mark.gpu
def test_gpu_counts_do_not_depend_on_the_batch(cuda_device):
    batch = NON_PREFLOP + spots(18, 2, 2)
    full = _enum(batch, cuda_device)
    assert _enum(batch[::-1], cuda_device) == full[::-1]
    assert _enum(batch * 12, cuda_device) == full * 12          # more queries than SMs: CTAs take several
    for i in (0, 16, 27, 30, len(batch) - 1):
        assert _enum([batch[i]], cuda_device) == [full[i]]


@pytest.mark.gpu
def test_gpu_validation(cuda_device):
    """The REFERENCE mode returns npk_enum_batch's errors, code and message, for the same bad rows."""
    import torch
    import neuron_poker_b200 as npk
    from neuron_poker_b200 import _lib as nl
    L = nl.ensure_init(cuda_device.index)
    stream = torch.cuda.current_stream(cuda_device).cuda_stream
    dev = lambda x: torch.as_tensor(np.ascontiguousarray(x, dtype=np.uint8)).to(cuda_device)
    h, b = [51, 47], [0, 1, 2, NO, NO]
    cases = [([h], [b], [4]),                              # four players
             ([h], [[0, 1, 2, 3, NO]], [3]),               # three players before the river
             ([[0, 60]], [b], [2]),                        # card id >= 52
             ([[0, 0]], [b], [2]),                         # duplicate
             ([h], [[0, 1, 51, NO, NO]], [2]),             # duplicate between hand and board
             ([h], [[2, NO, 4, NO, NO]], [2])]             # gap in the board
    o = [torch.zeros(1, dtype=torch.int64, device=cuda_device) for _ in range(3)]
    outs = [x.data_ptr() for x in o]
    for hole, board, npl in cases:
        ins = [dev(x) for x in (hole, board, npl)]
        res = []
        for mode in (None, nl.NPK_DEAL_UNIFORM, nl.NPK_DEAL_REFERENCE):
            args = [x.data_ptr() for x in ins] + [1] + ([] if mode is None else [mode]) + outs + [nl.NPK_FLAG_VALIDATE, stream]
            rc = (L.npk_enum_batch if mode is None else L.npk_enum_dealer_batch)(*args)
            res.append((rc, L.npk_last_error().decode()))
        assert res[0][0] < 0 and res[0] == res[1] == res[2], (hole, board, npl, res)
    good = [dev(x) for x in ([h], [b], [2])]
    for mode in (-1, 2):
        rc = L.npk_enum_dealer_batch(*(x.data_ptr() for x in good), 1, mode, *outs, nl.NPK_FLAG_VALIDATE, stream)
        assert rc == -2 and "deal_mode" in L.npk_last_error().decode()
    rc = L.npk_enum_dealer_batch(*(x.data_ptr() for x in good), -1, nl.NPK_DEAL_REFERENCE, *outs, 0, stream)
    assert rc == -2 and "negative Q" in L.npk_last_error().decode()
    with pytest.raises(nl.NpkError, match="deal_mode"):
        npk.enumerate_equity(*good, device=cuda_device, deal_mode="biased")


@pytest.mark.gpu
@pytest.mark.slow
def test_gpu_exact_equity_of_asks_preflop(cuda_device):
    """get_equity({'AS','KS'}, set(), 2, runs) converges to the exact value: within 3 sigma of the reference's own 400,000-trial
    estimate (0.6608, SURVEY A.2), and pinned."""
    import neuron_poker_b200 as npk
    e = npk.exact_equity({"AS", "KS"}, set(), 2)
    w, t, l = ASKS_PREFLOP
    assert e == (w + t) / (w + t + l)
    assert abs(e - 0.6608) < 3 * math.sqrt(e * (1 - e) / 400_000)


# Monte-Carlo paths of the REFERENCE dealer against the exact values: one spot per street, and three players on the river
MC_SPOTS = [([51, 47], [], 2)] + spots(21, 1, 3) + spots(22, 1, 4) + spots(23, 1, 5) + spots(24, 1, 5, 3)
MC_TRIALS = 1 << 20


@pytest.fixture(scope="module")
def mc_exact(cuda_device):
    got = [ASKS_PREFLOP] + _enum(MC_SPOTS[1:], cuda_device)
    return [(w + t) / (w + t + l) for w, t, l in got]


def _z(wins_ties, trials, p):
    return (wins_ties / trials - p) / math.sqrt(p * (1 - p) / trials)


@pytest.mark.gpu
def test_gpu_monte_carlo_paths_converge_to_the_exact_values(cuda_device, mc_exact):
    import torch
    import neuron_poker_b200 as npk
    from neuron_poker_b200.cards import card_str
    hole, board, npl = _arrays(MC_SPOTS)
    T = MC_TRIALS
    zs = {}
    for i, (h, b, p) in enumerate(MC_SPOTS):                 # per-shape kernels (K1')
        out = npk.get_equity_batch(hole[i:i + 1], board[i:i + 1], npl[i:i + 1], T, seed_value=101 + i,
                                   deal_mode="reference", uniform_shape=(p, len(b)), device=cuda_device)
        zs[("shape", i)] = _z(int(out["wins"][0] + out["ties"][0]), T, mc_exact[i])
    out = npk.get_equity_batch(hole, board, npl, T, seed_value=202, deal_mode="reference", device=cuda_device)   # mixed
    for i in range(len(MC_SPOTS)):
        zs[("mixed", i)] = _z(int(out["wins"][i] + out["ties"][i]), T, mc_exact[i])
    for passes in (True, False):                             # generic range kernel / pair-list sampler, full range
        out = npk.get_equity_ranges_batch(hole, board, npl, T, opponent_range=1, seed_value=303 + passes,
                                          deal_mode="reference", passes=passes, device=cuda_device)
        for i in range(len(MC_SPOTS)):
            zs[("ranges", passes, i)] = _z(int(out["wins"][i] + out["ties"][i]), T, mc_exact[i])
    torch.cuda.synchronize()
    npk.seed(404)                                            # the one-query drop-in
    try:
        for i, (h, b, p) in enumerate(MC_SPOTS):
            e = npk.get_equity({card_str(c) for c in h}, {card_str(c) for c in b}, p, T)
            zs[("get_equity", i)] = _z(round(e * T), T, mc_exact[i])
    finally:
        npk.seed(None)
    bad = {k: z for k, z in zs.items() if abs(z) > 4}
    assert not bad, (bad, mc_exact)
    assert len(zs) == 5 * len(MC_SPOTS)
