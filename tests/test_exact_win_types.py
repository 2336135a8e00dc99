"""Win-type histograms of the exact enumerations: exact_equity_batch / exact_equity_counts / showdown_equity_batch /
showdown_equity with win_types=True (npk_exact_equity_win_types_batch, npk_showdown_equity_win_types_batch).

CPU: tests/exact_win_types_oracle.c bins the hero's hand type in the two enumerators of tests/exact_equity_oracle.c; its literal
replay of the reference's dealer equals its weighted enumeration, bins included, its counts equal the existing checker's, and
the bins sum to win + tie.  Argument errors of the new arguments need no device.
GPU: bit-exact against the checker (both engines); win / tie / lose identical to the plain calls; the exact engine's bins equal
the weighted sum of showdown_equity_batch's player-0 bins; the Monte-Carlo win_types within 4 sigma of the exact fractions;
independence of the batch, graph capture and validation.
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
import test_exact_equity as ee
from test_exact_equity import NO, Spot, spots

HERE = os.path.dirname(os.path.abspath(__file__))
_lib = None


def wt_lib():
    """tests/exact_win_types_oracle.c, compiled with the C compiler into a temporary directory on first use."""
    global _lib
    if _lib is None:
        cc = os.environ.get("CC") or shutil.which("gcc") or shutil.which("cc")
        if not cc:
            raise RuntimeError("no C compiler for tests/exact_win_types_oracle.c")
        tmp = tempfile.mkdtemp(prefix="npk_exact_win_types_oracle_")
        try:
            out = os.path.join(tmp, "libexact_win_types_oracle.so")
            subprocess.check_call([cc, "-O2", "-std=c11", "-fPIC", "-shared", "-Wall",
                                   os.path.join(HERE, "exact_win_types_oracle.c"), "-o", out])
            L = ctypes.CDLL(out)                   # stays mapped after the file is gone
        finally:
            shutil.rmtree(tmp, ignore_errors=True)
        u8p, i, vp = ctypes.POINTER(ctypes.c_uint8), ctypes.c_int, ctypes.c_void_p
        i64p = ctypes.POINTER(ctypes.c_int64)
        L.exact_wt_literal.argtypes = [vp, vp, u8p, u8p, i, i, u8p, i, ctypes.c_uint64, i64p]
        L.exact_wt_weighted.argtypes = [vp, vp, u8p, u8p, i, i, u8p, i, ctypes.c_uint64, i, i64p]
        L.showdown_wt.argtypes = [vp, vp, u8p, i, u8p, i, ctypes.c_uint64, i, i64p, i64p, i64p]
        O = oracle.lib()
        O.oracle_fast_init()
        L.rank7 = ctypes.cast(O.oracle_rank7_fast, ctypes.c_void_p)
        import neuron_poker_b200 as npk
        L.type_start = np.ascontiguousarray(npk.host_tables()["type_start"], dtype=np.uint16)
        _lib = L
    return _lib


def _ts():
    return wt_lib().type_start.ctypes.data_as(ctypes.c_void_p)


def literal(sp):
    keep, args = ee._c_args(sp)
    out = (ctypes.c_int64 * 12)()
    rc = wt_lib().exact_wt_literal(wt_lib().rank7, _ts(), *args, out)
    assert rc == 0, (sp, rc)
    return tuple(out)


def weighted(sp, mode="reference"):
    """(win, tie, lose, bin 0, ..., bin 8)"""
    keep, args = ee._c_args(sp)
    out = (ctypes.c_int64 * 12)()
    rc = wt_lib().exact_wt_weighted(wt_lib().rank7, _ts(), *args, 1 if mode == "reference" else 0, out)
    assert rc == 0, (sp, rc)
    return tuple(out)


def showdown(hands, board, dead, mode):
    """every hand known: (win [P], tie [P], bins [P][9])"""
    P = len(hands)
    h = np.array(sum(hands, []), dtype=np.uint8)
    b = np.array(board or [0], dtype=np.uint8)
    mask = sum(1 << int(c) for c in dead)
    win, tie, bins = (ctypes.c_int64 * P)(), (ctypes.c_int64 * P)(), (ctypes.c_int64 * (9 * P))()
    p = lambda a: a.ctypes.data_as(ctypes.POINTER(ctypes.c_uint8))
    rc = wt_lib().showdown_wt(wt_lib().rank7, _ts(), p(h), P, p(b), len(board), mask, 1 if mode == "reference" else 0,
                              win, tie, bins)
    assert rc == 0
    return list(win), list(tie), [list(bins[9 * q:9 * q + 9]) for q in range(P)]


def known_spots(seed, count, nb, players, ndead):
    """(hands, board, dead) with every hand known"""
    rng = np.random.default_rng(seed)
    out = []
    for i in range(count):
        P = players[i % len(players)]
        c = [int(x) for x in rng.permutation(52)[:2 * P + nb + ndead]]
        out.append(([c[2 * q:2 * q + 2] for q in range(P)], c[2 * P:2 * P + nb], c[2 * P + nb:]))
    return out


# ---- CPU ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("nb,k,count,seed", [(5, 1, 4, 1), (4, 1, 3, 2), (3, 1, 2, 3), (5, 2, 3, 4), (4, 2, 1, 5)])
def test_checker_literal_dealer_equals_the_weighted_bins(nb, k, count, seed):
    """k = 1 and 2, 0-2 known hands, ghost cards, river / turn (and flop for k = 1), both dealing modes."""
    batch = spots(seed, count, nb, k, nknown=[0, 1, 2], ndead=2) if (nb, k) != (4, 2) else spots(seed, count, 4, 2, 2, 4)
    batch += [s for s in ee.HIGH if len(s.board) == nb and s.k == k]
    for sp in batch:
        lit = literal(sp)
        assert weighted(sp) == lit, sp
        assert lit[:3] == ee.weighted(sp), sp
        assert sum(lit[3:]) == lit[0] + lit[1], sp
        uni = weighted(sp, "uniform")
        assert uni[:3] == ee.weighted(sp, "uniform"), sp
        assert sum(uni[3:]) == uni[0] + uni[1], sp


def test_checker_showdown_bins_sum_to_win_and_tie():
    import showdown_oracle
    for hands, board, dead in known_spots(3, 6, 4, [2, 3, 6], 2) + known_spots(4, 4, 5, [2, 4, 10], 0):
        for mode in ("uniform", "reference"):
            win, tie, bins = showdown(hands, board, dead, mode)
            r = showdown_oracle.showdown_equity(hands, board, dead, deal_mode=mode)
            assert (win, tie) == (list(r["win"]), list(r["tie"])), (hands, board, mode)
            assert [sum(b) for b in bins] == [w + t for w, t in zip(win, tie)]


def test_win_types_argument_errors_need_no_device():
    import neuron_poker_b200 as npk
    from neuron_poker_b200 import _lib as nl
    for bad in (None, "yes", 1.5, [True]):
        with pytest.raises(ValueError, match="win_types"):
            npk.exact_equity_counts(["AS", "KS"], [], 2, win_types=bad)
        with pytest.raises(ValueError, match="win_types"):
            npk.showdown_equity([["AS", "KS"], ["QH", "QD"]], win_types=bad)
        with pytest.raises(ValueError, match="win_types"):
            npk.exact_equity_batch(None, None, None, None, win_types=bad)
        with pytest.raises(ValueError, match="win_types"):
            npk.showdown_equity_batch(None, None, None, win_types=bad)
    L = nl.lib()
    for mode, maxk, what in ((-1, 2, "deal_mode"), (2, 2, "deal_mode"), (1, 0, "maxk"), (0, 9, "maxk")):
        rc = L.npk_exact_equity_win_types_batch(None, None, None, None, None, 1, maxk, mode, nl.NPK_FLAG_VALIDATE, None, None,
                                                None, None, None, None)
        assert rc == -2 and what in L.npk_last_error().decode(), (mode, maxk, rc)


# ---- GPU ---------------------------------------------------------------------------------------------------------------
def _exact(batch, device, mode="reference", maxk=None, win_types=True):
    import neuron_poker_b200 as npk
    out = npk.exact_equity_batch(*ee._arrays(batch, maxk), deal_mode=mode, device=device, win_types=win_types)
    rows = list(zip(*(out[k].tolist() for k in ("win", "tie", "lose"))))
    return [r + tuple(b) for r, b in zip(rows, out["win_types"].tolist())] if win_types else rows


def _showdown_arrays(batch):
    P = max(len(h) for h, _, _ in batch)
    holes = np.full((len(batch), P, 2), NO, dtype=np.uint8)
    board = np.full((len(batch), 5), NO, dtype=np.uint8)
    dead = np.full((len(batch), max(1, max(len(d) for _, _, d in batch))), NO, dtype=np.uint8)
    for i, (h, b, d) in enumerate(batch):
        holes[i, :len(h)] = h
        board[i, :len(b)] = b
        dead[i, :len(d)] = d
    return holes, np.array([len(h) for h, _, _ in batch], dtype=np.uint8), board, dead


SHOWDOWN_SPOTS = (known_spots(71, 6, 5, [2, 3, 4, 5, 6], 2) + known_spots(72, 6, 4, [2, 3, 6], 3) +
                  known_spots(73, 4, 3, [2, 3, 4, 6], 2) + known_spots(74, 2, 0, [2, 6], 2))


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["uniform", "reference"])
def test_gpu_bitexact_vs_the_checker(cuda_device, mode):
    got = _exact(ee.GPU_SPOTS, cuda_device, mode)
    for sp, g in zip(ee.GPU_SPOTS, got):
        assert g == weighted(sp, mode), (sp, mode)
    import neuron_poker_b200 as npk
    out = npk.showdown_equity_batch(*_showdown_arrays(SHOWDOWN_SPOTS), deal_mode=mode, device=cuda_device, win_types=True)
    assert out["win_types"].shape == (len(SHOWDOWN_SPOTS), 6, 9)
    for i, (hands, board, dead) in enumerate(SHOWDOWN_SPOTS):
        win, tie, bins = showdown(hands, board, dead, mode)
        P = len(hands)
        assert out["win"][i, :P].tolist() == win and out["tie"][i, :P].tolist() == tie, (hands, board, mode)
        assert out["win_types"][i, :P].tolist() == bins, (hands, board, mode)
        assert not out["win_types"][i, P:].any()


def _plain_and_typed_showdown(batch, device, mode):
    import neuron_poker_b200 as npk
    arrs = _showdown_arrays(batch)
    plain = npk.showdown_equity_batch(*arrs, deal_mode=mode, device=device)
    typed = npk.showdown_equity_batch(*arrs, deal_mode=mode, device=device, win_types=True)
    return plain, typed


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["uniform", "reference"])
def test_gpu_same_counts_as_the_plain_calls(cuda_device, mode):
    batch = ee.GPU_SPOTS + ee._enum_shapes() + spots(41, 2, 3, 2) + spots(42, 1, 3, 2, 1, 2) + [Spot([51, 47], [], 1, [])]
    typed = _exact(batch, cuda_device, mode)
    assert [t[:3] for t in typed] == _exact(batch, cuda_device, mode, win_types=False)
    assert all(sum(t[3:]) == t[0] + t[1] for t in typed)
    sd = SHOWDOWN_SPOTS + known_spots(75, 64, 3, [2, 3, 4, 6, 9, 10], 0) + [([[51, 47], [40, 41]], [], [])]
    plain, typed = _plain_and_typed_showdown(sd, cuda_device, mode)
    assert set(typed) == set(plain) | {"win_types"}
    for k in plain:
        assert plain[k].tolist() == typed[k].tolist(), k
    assert (typed["win_types"].sum(2) == typed["win"] + typed["tie"]).all()


def _single_sum(sp, device, mode):
    """sum over the unknown hand o of w(o) * player 0's bins of showdown_equity_batch(hero, known, o)"""
    import neuron_poker_b200 as npk
    r = np.array(sorted(set(range(52)) - set(sp.hero) - set(sum(sp.known, [])) - set(sp.board) - set(sp.dead)))
    b, a = np.nonzero(np.tril(np.ones((len(r), len(r)), dtype=bool), -1))
    w = (2 - (b == a + 1)).astype(np.int64) if mode == "reference" else np.ones(len(a), dtype=np.int64)
    K = len(sp.known)
    holes = np.empty((len(a), K + 2, 2), dtype=np.uint8)
    holes[:, :K + 1] = np.array([sp.hero] + sp.known, dtype=np.uint8)
    holes[:, K + 1, 0], holes[:, K + 1, 1] = r[a], r[b]
    out = npk.showdown_equity_batch(holes, np.full(len(a), K + 2, dtype=np.uint8),
                                    np.tile(np.array(sp.board + [NO] * (5 - len(sp.board)), dtype=np.uint8), (len(a), 1)),
                                    np.tile(np.array(sp.dead or [NO], dtype=np.uint8), (len(a), 1)), deal_mode=mode,
                                    device=device, win_types=True)
    return [int(x) for x in (w[:, None] * out["win_types"][:, 0].cpu().numpy()).sum(0)]


def _pair_sum(sp, device, mode, chunk=1 << 18):
    """ee._pair_sum's construction with player 0's bins: sum over unordered pairs of unknown hands of both orders' weights"""
    import neuron_poker_b200 as npk
    r = np.array(sorted(set(range(52)) - set(sp.hero) - set(sum(sp.known, [])) - set(sp.board) - set(sp.dead)))
    n = len(r)
    b, a = np.nonzero(np.tril(np.ones((n, n), dtype=bool), -1))
    i1, i2 = np.nonzero(np.triu(np.ones((len(a), len(a)), dtype=bool), 1))
    ok = (a[i1] != a[i2]) & (a[i1] != b[i2]) & (b[i1] != a[i2]) & (b[i1] != b[i2])
    i1, i2 = i1[ok], i2[ok]
    A1, B1, A2, B2 = a[i1], b[i1], a[i2], b[i2]
    if mode == "reference":
        btw = lambda lo, hi, x: ((lo < x) & (x < hi)).astype(np.int64)
        w12 = (2 - (B1 == A1 + 1)) * (2 - (B2 - A2 - 1 == btw(A2, B2, A1) + btw(A2, B2, B1)))
        w21 = (2 - (B2 == A2 + 1)) * (2 - (B1 - A1 - 1 == btw(A1, B1, A2) + btw(A1, B1, B2)))
        w = (w12 + w21).astype(np.int64)
    else:
        w = np.full(len(i1), 2, dtype=np.int64)
    K = len(sp.known)
    fixed = np.array([sp.hero] + sp.known, dtype=np.uint8)
    brd = np.array(sp.board + [NO] * (5 - len(sp.board)), dtype=np.uint8)
    dead = np.array(sp.dead or [NO], dtype=np.uint8)
    acc = np.zeros(9, dtype=np.int64)
    for s in range(0, len(i1), chunk):
        e = min(len(i1), s + chunk)
        holes = np.empty((e - s, K + 3, 2), dtype=np.uint8)
        holes[:, :K + 1] = fixed
        holes[:, K + 1, 0], holes[:, K + 1, 1] = r[A1[s:e]], r[B1[s:e]]
        holes[:, K + 2, 0], holes[:, K + 2, 1] = r[A2[s:e]], r[B2[s:e]]
        out = npk.showdown_equity_batch(holes, np.full(e - s, K + 3, dtype=np.uint8), np.tile(brd, (e - s, 1)),
                                        np.tile(dead, (e - s, 1)), deal_mode=mode, device=device, win_types=True)
        acc += (w[s:e, None] * out["win_types"][:, 0].cpu().numpy()).sum(0)
    return [int(x) for x in acc]


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["uniform", "reference"])
def test_gpu_exact_bins_equal_the_weighted_showdown_bins(cuda_device, mode):
    """three-handed flops (with and without a known hand and ghost cards) and a heads-up preflop spot"""
    batch = spots(41, 2, 3, 2) + spots(42, 1, 3, 2, 1, 2)
    for sp, g in zip(batch, _exact(batch, cuda_device, mode)):
        assert list(g[3:]) == _pair_sum(sp, cuda_device, mode), (sp, mode)
    sp = Spot([51, 47], [], 1, [])
    g, = _exact([sp], cuda_device, mode)
    assert list(g[3:]) == _single_sum(sp, cuda_device, mode)


def _z_ok(counts, exact, total, T, label):
    bad = []
    for t in range(9):
        p = exact[t] / total
        if p == 0:
            if counts[t]:
                bad.append((label, t, counts[t], "impossible type sampled"))
            continue
        z = (counts[t] / T - p) / math.sqrt(p * (1 - p) / T)
        if abs(z) > 4:
            bad.append((label, t, z))
    return bad


@pytest.mark.gpu
def test_gpu_monte_carlo_win_types_land_on_the_exact_fractions(cuda_device):
    """get_equity_batch (reference dealer, 2^24 trials): AsKs heads-up preflop and the reference test t3 (AsKs three-handed
    preflop); equity_counts_ranges with a known opponent and ghost cards, both dealers."""
    import neuron_poker_b200 as npk
    bad = []
    T = 1 << 24
    for players, seed in ((2, 3), (3, 4)):
        ex = npk.exact_equity_counts(["AS", "KS"], [], players, win_types=True)
        assert sum(ex["win_types"]) == ex["win"] + ex["tie"]
        out = npk.get_equity_batch(np.array([[51, 47]], dtype=np.uint8), np.array([[NO] * 5], dtype=np.uint8),
                                   np.array([players], dtype=np.uint8), T, seed_value=seed, deal_mode="reference",
                                   win_types=True, device=cuda_device)
        bad += _z_ok(out["win_types"][0].tolist(), ex["win_types"], ex["win"] + ex["tie"] + ex["lose"], T, ("batch", players))
    T = 1 << 22
    cases = [(["AS", "KS"], [["QH", "QD"]], 3, ["2C", "7D", "KH"], ["AC", "3H"]),
             (["TD", "7D"], [["8C", "8H"]], 3, ["8D", "QD", "2C", "5S"], ["AH", "3S"]),
             (["9H", "9S"], [["AD", "JC"]], 3, [], ["2D", "2H"])]
    for mode in ("uniform", "reference"):
        for ci, (hero, known, players, board, ghost) in enumerate(cases):
            ex = npk.exact_equity_counts(hero, board, players, known_opponents=known, ghost_cards=ghost, deal_mode=mode,
                                         win_types=True)
            r = npk.equity_counts_ranges(hero, board, players, T, ghost_cards=ghost, deal_mode=mode, seed_value=21 + ci,
                                         known_opponents=known)
            bad += _z_ok(r["win_types"], ex["win_types"], ex["win"] + ex["tie"] + ex["lose"], T, (mode, ci))
    assert not bad, bad


@pytest.mark.gpu
def test_gpu_bins_do_not_depend_on_the_batch(cuda_device):
    probe = ee.GPU_SPOTS[::3]
    full = _exact(probe, cuda_device)
    assert _exact(probe[::-1], cuda_device) == full[::-1]
    big = spots(51, 2048, 5, 1, [0, 1, 2], 2)
    big[500:500] = probe
    assert _exact(big, cuda_device, maxk=4)[500:500 + len(probe)] == full
    for i in (0, 5, len(probe) - 1):
        assert _exact([probe[i]], cuda_device) == [full[i]]
    plain, typed = _plain_and_typed_showdown(SHOWDOWN_SPOTS, cuda_device, "reference")
    sd = known_spots(76, 1024, 4, [2, 6], 0)
    sd[100:100] = SHOWDOWN_SPOTS
    _, typed_big = _plain_and_typed_showdown(sd, cuda_device, "reference")
    P = typed["win_types"].shape[1]
    assert typed_big["win_types"][100:100 + len(SHOWDOWN_SPOTS), :P].tolist() == typed["win_types"].tolist()


@pytest.mark.gpu
def test_gpu_validation_matches_the_plain_calls(cuda_device):
    import neuron_poker_b200 as npk
    from neuron_poker_b200._lib import NpkError
    holes, nk, nr, board, dead = ee._arrays(spots(61, 4, 4, 1, 2, 2))
    cases = []
    h = holes.copy(); h[1, 0, 0] = 52; cases.append(dict(h=h))
    b = board.copy(); b[1, 1] = NO; cases.append(dict(b=b))
    k = nk.copy(); k[2] = 0; cases.append(dict(k=k))
    r = nr.copy(); r[1] = 3; cases.append(dict(r=r))
    for kw in cases:
        errs = []
        for wt in (False, True):
            with pytest.raises(NpkError) as e:
                npk.exact_equity_batch(kw.get("h", holes), kw.get("k", nk), kw.get("r", nr), kw.get("b", board), dead,
                                       device=cuda_device, validate=True, win_types=wt)
            errs.append((e.value.code, str(e.value)))
        assert errs[0] == errs[1], kw
    sh, sn, sb, sd = _showdown_arrays(SHOWDOWN_SPOTS[:4])
    for kw in (dict(sh=np.where(np.arange(sh.size).reshape(sh.shape) == 3, 60, sh).astype(np.uint8)),
               dict(sn=np.array([0, 2, 2, 2], dtype=np.uint8))):
        errs = []
        for wt in (False, True):
            with pytest.raises(NpkError) as e:
                npk.showdown_equity_batch(kw.get("sh", sh), kw.get("sn", sn), sb, sd, device=cuda_device, validate=True,
                                          win_types=wt)
            errs.append((e.value.code, str(e.value)))
        assert errs[0] == errs[1], kw


@pytest.mark.gpu
def test_gpu_graph_capture(cuda_device):
    import torch
    from neuron_poker_b200 import _lib as nl
    import neuron_poker_b200.evaluator as ev
    L = nl.ensure_init(cuda_device.index)
    batch = ee.GPU_SPOTS[:12]
    ins = ee._dev_inputs(batch, cuda_device)
    maxk = ins[0].shape[1]
    out = [torch.empty(len(batch), dtype=torch.int64, device=cuda_device) for _ in range(3)]
    wt = torch.empty((len(batch), 9), dtype=torch.int64, device=cuda_device)
    ws = torch.empty(int(L.npk_exact_equity_workspace_bytes(len(batch))), dtype=torch.uint8, device=cuda_device)
    sh, sn, sb, sd = _showdown_arrays(SHOWDOWN_SPOTS)
    sh, sn, sb = (torch.as_tensor(x).to(cuda_device) for x in (sh, sn, sb))
    sdm = ev._dead_masks(sd, len(SHOWDOWN_SPOTS), cuda_device)
    N, P = sh.shape[0], sh.shape[1]
    sout = [torch.empty((N, P), dtype=torch.int64, device=cuda_device) for _ in range(3)]
    scomp = torch.empty(N, dtype=torch.int64, device=cuda_device)
    swt = torch.empty((N, P, 9), dtype=torch.int64, device=cuda_device)
    sws = torch.empty(int(L.npk_showdown_equity_workspace_bytes(N)), dtype=torch.uint8, device=cuda_device)

    def calls():
        st = torch.cuda.current_stream(cuda_device).cuda_stream
        nl.check(L.npk_exact_equity_win_types_batch(*(t.data_ptr() for t in ins), len(batch), maxk, nl.NPK_DEAL_REFERENCE, 0,
                                                    *(o.data_ptr() for o in out), wt.data_ptr(), ws.data_ptr(), st))
        nl.check(L.npk_showdown_equity_win_types_batch(sh.data_ptr(), sn.data_ptr(), sb.data_ptr(), sdm.data_ptr(), N, P,
                                                       nl.NPK_DEAL_REFERENCE, 0, *(o.data_ptr() for o in sout),
                                                       scomp.data_ptr(), swt.data_ptr(), sws.data_ptr(), st))

    s = torch.cuda.Stream(cuda_device)
    s.wait_stream(torch.cuda.current_stream(cuda_device))
    with torch.cuda.stream(s):                                   # warm-up (module load, shared-memory attribute)
        calls()
    torch.cuda.current_stream(cuda_device).wait_stream(s)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        calls()
    for o in out + [wt, swt]:
        o.fill_(-1)
    g.replay()
    torch.cuda.synchronize()
    got = [r + tuple(b) for r, b in zip(zip(*(o.tolist() for o in out)), wt.tolist())]
    assert got == _exact(batch, cuda_device)
    import neuron_poker_b200 as npk
    ref = npk.showdown_equity_batch(*_showdown_arrays(SHOWDOWN_SPOTS), deal_mode="reference", device=cuda_device, win_types=True)
    assert swt.tolist() == ref["win_types"].tolist()


@pytest.mark.gpu
def test_gpu_one_spot_calls(cuda_device):
    """exact_equity_counts and showdown_equity with win_types: nine ints per result, summing to win + tie"""
    import neuron_poker_b200 as npk
    r = npk.exact_equity_counts(["AS", "KS"], ["2C", "7D", "KH"], 3, known_opponents=[["QH", "QD"]], ghost_cards=["5S", "9C"],
                                win_types=True)
    plain = npk.exact_equity_counts(["AS", "KS"], ["2C", "7D", "KH"], 3, known_opponents=[["QH", "QD"]],
                                    ghost_cards=["5S", "9C"])
    assert {k: v for k, v in r.items() if k != "win_types"} == plain
    assert len(r["win_types"]) == 9 and sum(r["win_types"]) == r["win"] + r["tie"]
    assert all(isinstance(x, int) for x in r["win_types"])
    s = npk.showdown_equity([["AS", "KS"], ["QH", "QD"], ["7C", "2D"]], ["2C", "9H"], ["5S"], win_types=True)
    assert {k: v for k, v in s.items() if k != "win_types"} == npk.showdown_equity([["AS", "KS"], ["QH", "QD"], ["7C", "2D"]],
                                                                                   ["2C", "9H"], ["5S"])
    assert [sum(b) for b in s["win_types"]] == [w + t for w, t in zip(s["win"], s["tie"])]
    assert len(s["win_types"]) == 3 and all(len(b) == 9 for b in s["win_types"])
