"""Exact showdown equity of known hands (npk_showdown_equity_batch / showdown_equity).

CPU: the literal enumeration of tests/showdown_oracle.c pinned to the existing heads-up / three-player enumerations and
goldens, its REFERENCE mode to the reference dealer's pop sequences and seeded runs, and its invariants.
GPU: the kernel bit-exact against that oracle, against enumerate_equity, independent of the batch it runs in, and at 3 sigma
against the known-hands Monte-Carlo path."""
import itertools
import math

import numpy as np
import pytest

import oracle
import showdown_oracle

NO = 0xFF
SHARE = 2520


def _deck_minus(*groups):
    used = {c for g in groups for c in g}
    return [c for c in range(52) if c not in used]


def _ids(cards):
    return [int(c) for c in oracle.ids(cards)]


def _unseen(hands, board, dead, mode):
    u = _deck_minus(*hands, board, dead)
    return u[:-1] if mode == "reference" and len(board) < 5 else u


# ---------------------------------------------------------------------------------------------------------------- CPU --
def _headsup_sum(hero, board):
    """(win, tie, lose) of the hero summed over every opponent hand, one exact showdown_equity per opponent."""
    win = tie = total = 0
    for a, b in itertools.combinations(_deck_minus(hero, board), 2):
        r = showdown_oracle.showdown_equity([hero, [a, b]], board)
        win += r["win"][0]
        tie += r["tie"][0]
        total += r["completions"]
    return win, tie, total - win - tie


def test_oracle_headsup_sums_to_enum_golden(golden_enum):
    spots = [s for s in golden_enum["spots"] if len(s["board"]) in (4, 5) and s["players"] == 2]
    assert spots
    for s in spots:
        hero, board = _ids(s["hero"]), _ids(s["board"])
        got = _headsup_sum(hero, board)
        assert got == oracle.enum_headsup(hero, board), s["name"]
        if "uniform" in s:
            assert list(got) == s["uniform"], s["name"]
    for s in golden_enum["random_spots"][:4]:
        assert list(_headsup_sum(_ids(s["hero"]), _ids(s["board"]))) == s["uniform"]


def test_oracle_headsup_flops_sum_to_enum_headsup():
    rng = np.random.default_rng(5)
    for _ in range(2):
        cards = [int(c) for c in rng.permutation(52)[:5]]
        hero, board = cards[:2], cards[2:]
        assert _headsup_sum(hero, board) == oracle.enum_headsup(hero, board)


def test_oracle_three_players_river_sums_to_enum_river_multi():
    hero, board = _ids(["AH", "TD"]), _ids(["TC", "7S", "2H", "KD", "7H"])
    rest = _deck_minus(hero, board)
    hands = list(itertools.combinations(rest, 2))
    win = tie = lose = 0
    for i, h1 in enumerate(hands):
        for h2 in hands[i + 1:]:
            if set(h1) & set(h2):
                continue
            r = showdown_oracle.showdown_equity([hero, list(h1), list(h2)], board)
            win += 2 * r["win"][0]
            tie += 2 * r["tie"][0]
            lose += 2 * (1 - r["win"][0] - r["tie"][0])
    assert (win, tie, lose) == oracle.enum_river_multi(hero, board, 3)


def _pop_sequences(hands, board, dead):
    """Totals over the reference dealer's literal pop sequences: a board card is list.pop(j), j in [0, len-1), from the
    id-ordered deck left after the dead cards, the board and every hand have been removed (montecarlo_python.py:185-189)."""
    tot = {"win": [0] * len(hands), "tie": [0] * len(hands), "share": [0] * len(hands), "sequences": 0}

    def rec(deck, table):
        if len(table) == 5:
            r = showdown_oracle.showdown_equity(hands, table)
            for k in ("win", "tie", "share"):
                tot[k] = [x + y for x, y in zip(tot[k], r[k])]
            tot["sequences"] += 1
            return
        for j in range(len(deck) - 1):
            d = list(deck)
            c = d.pop(j)
            rec(d, table + [c])

    rec(_deck_minus(*hands, board, dead), list(board))
    return tot


@pytest.mark.parametrize("nb", [5, 4, 3])
def test_reference_mode_is_the_reference_dealer(nb):
    rng = np.random.default_rng(10 + nb)
    for players, ndead in ((2, 0), (3, 2), (4, 1)):
        cards = [int(c) for c in rng.permutation(52)[:2 * players + nb + ndead]]
        hands = [cards[2 * p:2 * p + 2] for p in range(players)]
        board, dead = cards[2 * players:2 * players + nb], cards[2 * players + nb:]
        exact = showdown_oracle.showdown_equity(hands, board, dead, deal_mode="reference")
        seq = _pop_sequences(hands, board, dead)
        scale = math.factorial(5 - nb)                    # each unordered completion is dealt in (5 - nb)! orders
        assert seq["sequences"] == scale * exact["completions"]
        for k in ("win", "tie", "share"):
            assert seq[k] == [scale * x for x in exact[k]], k


@pytest.mark.parametrize("board,ghost", [((), None), (("2C", "7D", "KH"), ("5S", "9C")), (("2C", "7D", "KH", "QS"), None)])
def test_reference_mode_matches_seeded_reference_runs(board, ghost):
    hands = [["AS", "KS"], ["QH", "QD"], ["7C", "8C"]]
    runs = 100000
    for players in (2, 3):
        got = oracle.mc_reference_ranges(hands[0], list(board), players, runs, 17, (), ghost=list(ghost) if ghost else None,
                                         known=hands[1:players])
        exact = showdown_oracle.showdown_equity(hands[:players], list(board), list(ghost or ()), deal_mode="reference")
        p = (exact["win"][0] + exact["tie"][0]) / exact["completions"]      # get_winner: the hero wins his ties
        sigma = math.sqrt(p * (1 - p) / runs)
        assert abs(got["wins"] / runs - p) <= 3 * sigma, (players, got["wins"] / runs, p)
        assert got["passes"] == 0


def test_oracle_invariants():
    rng = np.random.default_rng(3)
    for players, nb, ndead, mode in ((2, 3, 0, "uniform"), (5, 4, 3, "reference"), (9, 3, 1, "uniform"), (1, 4, 0, "reference")):
        cards = [int(c) for c in rng.permutation(52)[:2 * players + nb + ndead]]
        hands = [cards[2 * p:2 * p + 2] for p in range(players)]
        board, dead = cards[2 * players:2 * players + nb], cards[2 * players + nb:]
        r = showdown_oracle.showdown_equity(hands, board, dead, deal_mode=mode)
        assert r["completions"] == math.comb(len(_unseen(hands, board, dead, mode)), 5 - nb)
        assert sum(r["share"]) == SHARE * r["completions"]
        for p in range(players):
            assert SHARE * r["win"][p] <= r["share"][p] <= SHARE * (r["win"][p] + r["tie"][p])
        perm = list(rng.permutation(players))
        q = showdown_oracle.showdown_equity([hands[i] for i in perm], board, dead, deal_mode=mode)
        for k in ("win", "tie", "share"):
            assert q[k] == [r[k][i] for i in perm]
    # the board plays (royal flush): every completion is split between all hands
    r = showdown_oracle.showdown_equity([["2C", "3D"], ["4H", "5C"], ["6D", "7H"]], ["TS", "JS", "QS", "KS", "AS"])
    assert r == {"win": [0, 0, 0], "tie": [1, 1, 1], "share": [840, 840, 840], "completions": 1}
    # equal hands on a flop: every completion without a flush for one of them is split
    r = showdown_oracle.showdown_equity([["AC", "KD"], ["AD", "KC"]], ["2H", "7H", "9S"])
    assert r["win"][0] == r["win"][1] and r["share"][0] == r["share"][1] == SHARE * r["completions"] // 2


# ---------------------------------------------------------------------------------------------------------------- GPU --
def _spots(seed, count, players, nb, ndead, maxp=10):
    rng = np.random.default_rng(seed)
    holes = np.full((count, maxp, 2), NO, dtype=np.uint8)
    board = np.full((count, 5), NO, dtype=np.uint8)
    dead = np.full((count, 3), NO, dtype=np.uint8)
    npl = np.zeros(count, dtype=np.uint8)
    for i in range(count):
        P = players[i % len(players)] if isinstance(players, (list, tuple)) else players
        b = nb[i % len(nb)] if isinstance(nb, (list, tuple)) else nb
        d = ndead[i % len(ndead)] if isinstance(ndead, (list, tuple)) else ndead
        c = rng.permutation(52)[:2 * P + b + d]
        holes[i, :P] = c[:2 * P].reshape(P, 2)
        board[i, :b] = c[2 * P:2 * P + b]
        dead[i, :d] = c[2 * P + b:]
        npl[i] = P
    return holes, npl, board, dead


def _oracle_row(holes, npl, board, dead, i, mode):
    P = int(npl[i])
    return showdown_oracle.showdown_equity([list(h) for h in holes[i, :P]], [int(c) for c in board[i] if c != NO],
                                  [int(c) for c in dead[i] if c != NO], deal_mode=mode)


def _host(out):
    return {k: v.cpu().numpy() for k, v in out.items()}


def _assert_row(out, i, ref, maxp):
    P = len(ref["win"])
    assert out["completions"][i] == ref["completions"], i
    for k in ("win", "tie", "share"):
        assert list(out[k][i, :P]) == ref[k], (i, k)
        assert not out[k][i, P:maxp].any(), (i, k)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["uniform", "reference"])
def test_gpu_bitexact_vs_oracle(cuda_device, mode):
    import neuron_poker_b200 as npk
    shapes = [(P, b, d) for P in range(1, 11) for b in (0, 3, 4, 5) for d in (0, 2)]
    parts = [_spots(100 + k, 1, P, b, d) for k, (P, b, d) in enumerate(shapes)]
    parts.append(_spots(7, 3, 2, 0, 0))                         # a few heads-up preflop spots
    holes, npl, board, dead = (np.concatenate([p[j] for p in parts]) for j in range(4))
    out = _host(npk.showdown_equity_batch(holes, npl, board, dead, deal_mode=mode, device=cuda_device))
    for i in range(len(npl)):
        _assert_row(out, i, _oracle_row(holes, npl, board, dead, i, mode), 10)


def _all_opponents(hero, board):
    opp = list(itertools.combinations(_deck_minus(hero, board), 2))
    holes = np.array([[hero, list(o)] for o in opp], dtype=np.uint8)
    brd = np.tile(np.array(list(board) + [NO] * (5 - len(board)), dtype=np.uint8), (len(opp), 1))
    return holes, np.full(len(opp), 2, dtype=np.uint8), brd


def _check_vs_enumerate_equity(hero, board, device):
    import neuron_poker_b200 as npk
    holes, npl, brd = _all_opponents(hero, board)
    out = _host(npk.showdown_equity_batch(holes, npl, brd, device=device))
    w, t, l = npk.enumerate_equity(np.array([hero], dtype=np.uint8), brd[:1], device=device)
    win, tie = int(out["win"][:, 0].sum()), int(out["tie"][:, 0].sum())
    assert (win, tie, int(out["completions"].sum()) - win - tie) == (int(w[0]), int(t[0]), int(l[0]))


@pytest.mark.gpu
def test_gpu_bitexact_vs_enumerate_equity(cuda_device):
    rng = np.random.default_rng(21)
    for nb in (3, 4, 5):
        c = [int(x) for x in rng.permutation(52)[:2 + nb]]
        _check_vs_enumerate_equity(c[:2], c[2:], cuda_device)


@pytest.mark.gpu
@pytest.mark.slow
def test_gpu_bitexact_vs_enumerate_equity_preflop(cuda_device):
    _check_vs_enumerate_equity(_ids(["JH", "TH"]), [], cuda_device)


@pytest.mark.gpu
def test_gpu_counts_do_not_depend_on_the_batch(cuda_device):
    import neuron_poker_b200 as npk
    probe = _spots(31, 8, [2, 6, 9, 10, 3, 1, 4, 2], [0, 3, 4, 5, 0, 3, 0, 0], [0, 1, 0, 2, 3, 0, 0, 1])
    alone = [_host(npk.showdown_equity_batch(*(a[i:i + 1] for a in probe[:3]), probe[3][i:i + 1], device=cuda_device))
             for i in range(8)]
    batches = [_spots(32, 4096, [2, 3, 6, 9, 10], [0, 3, 4, 5], [0, 1, 2]),      # mixed shapes
               _spots(33, 4096, 2, 0, 0),                                       # W1-sized: heads-up preflop
               _spots(34, 65536, 6, 3, 0)]                                      # W2-sized: six-player flops
    for bh, bn, bb, bd in batches:
        at = np.arange(0, 8) * (len(bn) // 8) + 3
        bh, bn, bb, bd = bh.copy(), bn.copy(), bb.copy(), bd.copy()
        for j, i in enumerate(at):
            bh[i], bn[i], bb[i], bd[i] = probe[0][j], probe[1][j], probe[2][j], probe[3][j]
        out = _host(npk.showdown_equity_batch(bh, bn, bb, bd, device=cuda_device))
        for j, i in enumerate(at):
            for k in ("win", "tie", "share", "completions"):
                assert (out[k][i] == alone[j][k][0]).all(), (len(bn), j, k)
        assert (out["share"].sum(axis=1) == SHARE * out["completions"]).all()


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["uniform", "reference"])
def test_gpu_exact_value_of_the_known_hands_monte_carlo_path(cuda_device, mode):
    import neuron_poker_b200 as npk
    runs = 3_000_000
    for hands, board in (([("AS", "KS"), ("QH", "QD")], ()), ([("AS", "KS"), ("QH", "QD"), ("7C", "8C")], ("2C", "7D", "KH")),
                         ([("9H", "9S"), ("AD", "JC"), ("KC", "QC"), ("5D", "4D")], ("TC", "2D", "6H", "JD"))):
        r = npk.equity_counts_ranges(list(hands[0]), list(board), len(hands), runs, deal_mode=mode, seed_value=5,
                                     known_opponents=[list(h) for h in hands[1:]])
        exact = npk.showdown_equity([set(h) for h in hands], list(board), deal_mode=mode)
        p = (exact["win"][0] + exact["tie"][0]) / exact["completions"]
        sigma = math.sqrt(p * (1 - p) / runs)
        assert abs((r["wins"] + r["ties"]) / runs - p) <= 3 * sigma, (mode, hands, (r["wins"] + r["ties"]) / runs, p)


@pytest.mark.gpu
def test_gpu_validation(cuda_device):
    import torch
    import neuron_poker_b200 as npk
    from neuron_poker_b200._lib import NpkError
    holes, npl, board, dead = _spots(41, 4, 3, 3, 1, maxp=4)

    def run(h=holes, n=npl, b=board, d=dead, mode="uniform"):
        return npk.showdown_equity_batch(h, n, b, d, deal_mode=mode, device=cuda_device, validate=True)

    run()
    cases = []
    h = holes.copy(); h[1, 0, 0] = 52; cases.append((dict(h=h), -5))                          # id >= 52
    h = holes.copy(); h[2, 1, 1] = h[2, 0, 0]; cases.append((dict(h=h), -5))                  # a card twice in the hands
    b = board.copy(); b[0, 0] = holes[0, 2, 1]; cases.append((dict(b=b), -5))                 # board card also in a hand
    d = dead.copy(); d[3, 1] = board[3, 1]; cases.append((dict(d=d), -5))                     # dead card also on the board
    b = board.copy(); b[1, 1] = NO; cases.append((dict(b=b), -5))                             # a gap in the board
    d = dead.copy(); d[0, 2] = 60; cases.append((dict(d=d), -5))                              # dead id >= 52
    n = npl.copy(); n[2] = 0; cases.append((dict(n=n), -2))
    n = npl.copy(); n[2] = 5; cases.append((dict(n=n), -2))                                   # more than maxp
    for kw, code in cases:
        with pytest.raises(NpkError) as e:
            run(**kw)
        assert e.value.code == code, kw
    # fewer cards left than missing board cards: 10 hands + 29 dead leave 3 for a 5-card board (4 in UNIFORM mode for 4 missing)
    c = list(range(52))
    h10 = np.array([[c[2 * p:2 * p + 2] for p in range(10)]], dtype=np.uint8)
    dd = np.array([c[20:49]], dtype=np.uint8)
    with pytest.raises(NpkError) as e:
        npk.showdown_equity_batch(h10, [10], [[NO] * 5], dd, device=cuda_device, validate=True)
    assert e.value.code == -2
    b1 = np.array([[49, NO, NO, NO, NO]], dtype=np.uint8)
    out = npk.showdown_equity_batch(h10, [10], b1, dd[:, :27], deal_mode="uniform", device=cuda_device, validate=True)
    assert int(out["completions"][0]) == 1                     # 47, 48, 50 and 51 left for four board cards
    with pytest.raises(NpkError) as e:                         # ... but the reference never deals 51
        npk.showdown_equity_batch(h10, [10], b1, dd[:, :27], deal_mode="reference", device=cuda_device, validate=True)
    assert e.value.code == -2
    # without the flag, garbage bytes give no fault (and a spot with too few cards gets nothing)
    g = torch.Generator().manual_seed(0)
    N = 2048
    gh = torch.randint(0, 256, (N, 10, 2), dtype=torch.uint8, generator=g).cuda()
    gn = torch.randint(0, 256, (N,), dtype=torch.uint8, generator=g).cuda()
    gb = torch.randint(0, 256, (N, 5), dtype=torch.uint8, generator=g).cuda()
    gd = torch.randint(0, 256, (N, 4), dtype=torch.uint8, generator=g).cuda()
    out = npk.showdown_equity_batch(gh, gn, gb, gd, device=cuda_device)
    torch.cuda.synchronize()
    out = npk.showdown_equity_batch(h10, [10], [[NO] * 5], dd, device=cuda_device, validate=False)
    assert int(out["completions"][0]) == 0 and not out["share"].any()


@pytest.mark.gpu
def test_gpu_one_spot_call(cuda_device):
    import neuron_poker_b200 as npk
    hands = [{"AS", "KS"}, {"QH", "QD"}, {"7C", "8C"}]
    for mode in ("uniform", "reference"):
        r = npk.showdown_equity(hands, {"2C", "7D", "KH"}, {"5S"}, deal_mode=mode)
        holes = np.array([[_ids(sorted(h)) for h in hands]], dtype=np.uint8)
        row = _host(npk.showdown_equity_batch(holes, [3], [_ids(["2C", "7D", "KH"]) + [NO, NO]], [[_ids(["5S"])[0]]],
                                              deal_mode=mode, device=cuda_device))
        assert r["win"] == list(row["win"][0]) and r["tie"] == list(row["tie"][0])
        assert r["completions"] == row["completions"][0]
        assert r["equity"] == [s / (SHARE * r["completions"]) for s in row["share"][0]]
        assert abs(sum(r["equity"]) - 1) < 1e-12
    for bad in ([{"AS", "KX"}, {"QH", "QD"}], [{"AS", "KS"}, {"AS", "QD"}]):
        with pytest.raises(ValueError):
            npk.showdown_equity(bad)
    with pytest.raises(ValueError):
        npk.showdown_equity([{"AS", "KS"}, {"QH", "QD"}], {"2C", "1D", "KH"})
