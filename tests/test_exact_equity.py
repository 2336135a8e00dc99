"""Exact equity against one or two unknown opponents, with known hands and ghost cards (npk_exact_equity_batch /
exact_equity_batch / exact_equity_counts).

CPU: tests/exact_equity_oracle.c replays the reference's dealer literally over every index sequence it can draw; it equals the
weighted enumeration of include/npk.h (numerators and totals, and the totals equal their closed forms).  The weighted enumeration
without known hands equals tests/enum_reference_oracle.c, and the sum over unknown hands of the weight times the REFERENCE-mode
showdown equity of tests/showdown_oracle.c.  Argument errors need no device.
GPU: the kernel bit-exact against the weighted checker, against npk_enum_dealer_batch on every shape that call has and against
enum_golden.json; three-handed flops against the weighted sum of showdown_equity_batch; AsKs three-handed preflop (the reference
test t3) pinned and against get_equity; the known-hands Monte-Carlo paths within 4 sigma; independence of the batch; validation;
graph capture.
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
import test_enum_reference as enum_ref

HERE = os.path.dirname(os.path.abspath(__file__))
NO = 0xFF
# exact_equity_counts({'AS','KS'}, set(), 3): the weighted enumeration, total = 49^2 47^2 C(45,5); equity 0.490814
T3_REFERENCE = (3058827209332, 121633079749, 3299516090950)

_lib = None


def ee_lib():
    """tests/exact_equity_oracle.c, compiled with the C compiler into a temporary directory on first use."""
    global _lib
    if _lib is None:
        cc = os.environ.get("CC") or shutil.which("gcc") or shutil.which("cc")
        if not cc:
            raise RuntimeError("no C compiler for tests/exact_equity_oracle.c")
        tmp = tempfile.mkdtemp(prefix="npk_exact_equity_oracle_")
        try:
            out = os.path.join(tmp, "libexact_equity_oracle.so")
            subprocess.check_call([cc, "-O2", "-std=c11", "-fPIC", "-shared", "-Wall",
                                   os.path.join(HERE, "exact_equity_oracle.c"), "-o", out])
            L = ctypes.CDLL(out)                   # stays mapped after the file is gone
        finally:
            shutil.rmtree(tmp, ignore_errors=True)
        u8p, i = ctypes.POINTER(ctypes.c_uint8), ctypes.c_int
        L.exact_equity_literal.argtypes = [ctypes.c_void_p, u8p, u8p, i, i, u8p, i, ctypes.c_uint64, ctypes.POINTER(ctypes.c_int64)]
        L.exact_equity_weighted.argtypes = [ctypes.c_void_p, u8p, u8p, i, i, u8p, i, ctypes.c_uint64, i,
                                            ctypes.POINTER(ctypes.c_int64)]
        O = oracle.lib()
        O.oracle_fast_init()
        L.rank7 = ctypes.cast(O.oracle_rank7_fast, ctypes.c_void_p)
        _lib = L
    return _lib


class Spot:
    def __init__(self, hero, known, k, board, dead=()):
        self.hero, self.known, self.k = list(hero), [list(h) for h in known], k
        self.board, self.dead = list(board), list(dead)

    def __repr__(self):
        return "Spot(%r, %r, %d, %r, %r)" % (self.hero, self.known, self.k, self.board, self.dead)

    @property
    def n(self):
        return 52 - 2 - 2 * len(self.known) - len(self.board) - len(self.dead)

    def total(self, mode):
        n, m = self.n, 5 - len(self.board)
        if mode == "uniform":
            return math.comb(n, 2) * (math.comb(n - 2, m) if self.k == 1 else math.comb(n - 2, 2) * math.comb(n - 4, m))
        return (n - 1) ** 2 * (math.comb(n - 3, m) if self.k == 1 else (n - 3) ** 2 * math.comb(n - 5, m))


def _c_args(sp):
    p = lambda a: a.ctypes.data_as(ctypes.POINTER(ctypes.c_uint8))
    h = np.array(sp.hero, dtype=np.uint8)
    kn = np.array(sum(sp.known, []) or [0], dtype=np.uint8)
    b = np.array(sp.board or [0], dtype=np.uint8)
    mask = 0
    for c in sp.dead:
        mask |= 1 << int(c)
    return (h, kn, b), (p(h), p(kn), len(sp.known), sp.k, p(b), len(sp.board), mask)


def literal(sp):
    keep, args = _c_args(sp)
    out = (ctypes.c_int64 * 3)()
    rc = ee_lib().exact_equity_literal(ee_lib().rank7, *args, out)
    assert rc == 0, (sp, rc)
    return tuple(out)


def weighted(sp, mode="reference"):
    keep, args = _c_args(sp)
    out = (ctypes.c_int64 * 3)()
    rc = ee_lib().exact_equity_weighted(ee_lib().rank7, *args, 1 if mode == "reference" else 0, out)
    assert rc == 0, (sp, rc)
    return tuple(out)


def spots(seed, count, nb, k, nknown=0, ndead=0):
    rng = np.random.default_rng(seed)
    out = []
    for i in range(count):
        K = nknown[i % len(nknown)] if isinstance(nknown, (list, tuple)) else nknown
        c = [int(x) for x in rng.permutation(52)[:2 + 2 * K + nb + ndead]]
        out.append(Spot(c[:2], [c[2 + 2 * j:4 + 2 * j] for j in range(K)], k, c[2 + 2 * K:2 + 2 * K + nb], c[2 + 2 * K + nb:]))
    return out


# spots whose highest unseen ids sit in a known hand, on the board or among the dead cards: the excluded slot moves
HIGH = [Spot([0, 4], [[51, 50]], 1, [49, 9, 13, 17, 21]), Spot([1, 5], [[51, 2]], 1, [50, 47, 30], [49, 48]),
        Spot([51, 3], [[50, 49]], 2, [48, 6, 10, 14, 18]), Spot([7, 11], [], 2, [51, 50, 12, 40], [49, 48])]


# ---- CPU ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("nb,k,count,seed", [(5, 1, 4, 1), (4, 1, 3, 2), (3, 1, 2, 3), (5, 2, 3, 4), (4, 2, 1, 5)])
def test_weights_equal_the_literal_dealer(nb, k, count, seed):
    # 0-2 known opponents and ghost cards; the two-opponent turn takes known hands and dead cards to keep the replay short
    batch = spots(seed, count, nb, k, nknown=[0, 1, 2], ndead=2) if (nb, k) != (4, 2) else spots(seed, count, 4, 2, 2, 4)
    batch += [s for s in HIGH if len(s.board) == nb and s.k == k]
    for sp in batch:
        lit = literal(sp)
        assert weighted(sp) == lit, sp
        assert sum(lit) == sp.total("reference"), sp
        assert sum(weighted(sp, "uniform")) == sp.total("uniform"), sp


def test_without_known_hands_equals_the_enumeration_checkers():
    """No known hand: the REFERENCE weights equal tests/enum_reference_oracle.c (heads-up on every street but preflop, three
    players on the river), and the UNIFORM counts equal the oracle's exhaustive enumerations."""
    for sp in spots(6, 3, 5, 1) + spots(7, 2, 4, 1) + spots(8, 1, 3, 1) + spots(9, 2, 5, 2):
        assert weighted(sp) == enum_ref.weighted(sp.hero, sp.board, 1 + sp.k), sp
        uni = oracle.enum_headsup(sp.hero, sp.board) if sp.k == 1 else oracle.enum_river_multi(sp.hero, sp.board, 3)
        assert weighted(sp, "uniform") == uni, sp


def _unknown_tuples(sp, mode):
    """(hands, weight) of every ordered tuple of unknown hands, with the weights of include/npk.h."""
    r = sorted(set(range(52)) - set(sp.hero) - set(sum(sp.known, [])) - set(sp.board) - set(sp.dead))
    ref = mode == "reference"
    pairs = [(a, b) for b in range(len(r)) for a in range(b)]
    for a1, b1 in pairs:
        w1 = 2 - (b1 == a1 + 1) if ref else 1
        if sp.k == 1:
            yield [[r[a1], r[b1]]], w1
            continue
        for a2, b2 in pairs:
            if {a1, b1} & {a2, b2}:
                continue
            gap = sum(1 for s in range(a2 + 1, b2) if s not in (a1, b1))
            yield [[r[a1], r[b1]], [r[a2], r[b2]]], w1 * ((2 - (gap == 0)) if ref else 1)


def test_showdown_sum_equals_the_weights():
    """sum over unknown tuples of w * (hero's win, tie, lose) of the showdown equity of every hand = the weighted enumeration:
    the REFERENCE showdown leaves the highest unseen id -- the excluded slot -- out of the board."""
    for sp in spots(10, 2, 4, 1, 1, 2) + spots(11, 1, 3, 1, 2, 0) + spots(12, 1, 5, 2, 1, 2) + HIGH[:2]:
        for mode in ("reference", "uniform"):
            acc = [0, 0, 0]
            for hands, w in _unknown_tuples(sp, mode):
                r = showdown_oracle.showdown_equity([sp.hero] + sp.known + hands, sp.board, sp.dead, deal_mode=mode)
                acc[0] += w * r["win"][0]
                acc[1] += w * r["tie"][0]
                acc[2] += w * (r["completions"] - r["win"][0] - r["tie"][0])
            assert tuple(acc) == weighted(sp, mode), (sp, mode)


def test_argument_errors_need_no_device():
    """deal_mode and maxk are checked before the device is touched (null pointers are never looked at)."""
    from neuron_poker_b200 import _lib as nl
    L = nl.lib()
    for mode, maxk, what in ((-1, 2, "deal_mode"), (2, 2, "deal_mode"), (1, 0, "maxk"), (0, 9, "maxk")):
        rc = L.npk_exact_equity_batch(None, None, None, None, None, 1, maxk, mode, nl.NPK_FLAG_VALIDATE, None, None, None,
                                      None, None)
        assert rc == -2 and what in L.npk_last_error().decode(), (mode, maxk, rc)


def test_exact_equity_counts_rejects_bad_input_before_the_device():
    import neuron_poker_b200 as npk
    for args, kw in (((["AS", "XX"], [], 2), {}), ((["AS", "AS"], [], 2), {}), ((["AS", "KS"], ["AS", "2C", "3C"], 2), {}),
                     ((["AS"], [], 2), {}), ((["AS", "KS"], ["2C", "3C", "4C", "5C", "6C", "7C"], 2), {}),
                     ((["AS", "KS"], [], 3), {"known_opponents": [["QH", "KS"]]}),
                     ((["AS", "KS"], [], 3), {"known_opponents": [["QH"]]}),
                     ((["AS", "KS"], ["2C"], 2), {"ghost_cards": ["2C", "3D"]}),
                     ((["AS", "KS"], [], 2), {"ghost_cards": ["2C"]}),
                     ((["AS", "KS"], [], 11), {}), ((["AS", "KS"], [], 2), {"deal_mode": "biased"})):
        with pytest.raises(ValueError):
            npk.exact_equity_counts(*args, **kw)
    with pytest.raises(IndexError):
        npk.exact_equity_counts(["AS", "KS"], [], 0)
    with pytest.raises(ValueError, match="showdown_equity"):
        npk.exact_equity_counts(["AS", "KS"], [], 2, known_opponents=[["QH", "QD"]])
    with pytest.raises(ValueError, match="one or two unknown opponents, not 3"):
        npk.exact_equity_counts(["AS", "KS"], [], 4)


# ---- GPU ---------------------------------------------------------------------------------------------------------------
def _arrays(batch, maxk=None):
    maxk = maxk or 1 + max(len(s.known) for s in batch)
    holes = np.full((len(batch), maxk, 2), NO, dtype=np.uint8)
    board = np.full((len(batch), 5), NO, dtype=np.uint8)
    dead = np.full((len(batch), max(1, max(len(s.dead) for s in batch))), NO, dtype=np.uint8)
    for i, s in enumerate(batch):
        holes[i, 0] = s.hero
        for j, h in enumerate(s.known):
            holes[i, 1 + j] = h
        board[i, :len(s.board)] = s.board
        dead[i, :len(s.dead)] = s.dead
    nk = np.array([1 + len(s.known) for s in batch], dtype=np.uint8)
    nr = np.array([s.k for s in batch], dtype=np.uint8)
    return holes, nk, nr, board, dead


def _exact(batch, device, mode="reference", maxk=None):
    import neuron_poker_b200 as npk
    out = npk.exact_equity_batch(*_arrays(batch, maxk), deal_mode=mode, device=device)
    return list(zip(*(out[k].tolist() for k in ("win", "tie", "lose"))))


GPU_SPOTS = (spots(21, 3, 3, 1, [1, 2, 3], 2) + spots(22, 3, 4, 1, [1, 2, 3], 2) + spots(23, 4, 5, 1, [0, 1, 2, 3], 2) +
             spots(24, 3, 4, 2, [1, 2, 3], 2) + spots(25, 4, 5, 2, [0, 1, 2, 3], 2) + spots(26, 1, 3, 2, 3, 10) + HIGH)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["uniform", "reference"])
def test_gpu_bitexact_vs_the_weighted_checker(cuda_device, mode):
    got = _exact(GPU_SPOTS, cuda_device, mode)
    for sp, g in zip(GPU_SPOTS, got):
        assert g == weighted(sp, mode), (sp, mode)
        assert sum(g) == sp.total(mode), (sp, mode)


def _enum_shapes():
    return (spots(31, 8, 5, 1) + spots(32, 6, 4, 1) + spots(33, 4, 3, 1) + spots(34, 2, 2, 1) +
            spots(35, 2, 1, 1) + spots(36, 8, 5, 2))


def _enum_dealer(batch, device, mode):
    import neuron_poker_b200 as npk
    hole = np.array([s.hero for s in batch], dtype=np.uint8)
    board = np.array([s.board + [NO] * (5 - len(s.board)) for s in batch], dtype=np.uint8)
    npl = np.array([1 + s.k for s in batch], dtype=np.uint8)
    w, t, l = npk.enumerate_equity(hole, board, npl, device=device, deal_mode=mode)
    return list(zip(w.tolist(), t.tolist(), l.tolist()))


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["uniform", "reference"])
def test_gpu_equals_enum_dealer_batch(cuda_device, golden_enum, mode):
    batch = _enum_shapes()
    assert _exact(batch, cuda_device, mode) == _enum_dealer(batch, cuda_device, mode)
    key = "uniform" if mode == "uniform" else "reference_mode"
    gold = [s for s in golden_enum["spots"] if key in s]
    got = _exact([Spot(oracle.ids(s["hero"]).tolist(), [], s["players"] - 1, oracle.ids(s["board"]).tolist()) for s in gold],
                 cuda_device, mode)
    assert any(s["name"] == "t17" for s in gold) or mode == "reference"
    for s, (w, t, l) in zip(gold, got):
        assert ([w, t, l] if mode == "uniform" else [w + t, w + t + l]) == s[key], s["name"]


@pytest.mark.gpu
@pytest.mark.slow
def test_gpu_equals_enum_dealer_batch_preflop(cuda_device):
    """A heads-up preflop spot: enum_kernel's generic walk takes about 112 s on a B200 (DESIGN.md section 4.4)."""
    batch = [Spot([51, 47], [], 1, [])]
    got = _exact(batch, cuda_device)
    assert got == _enum_dealer(batch, cuda_device, "reference") == [enum_ref.ASKS_PREFLOP]


def _pair_sum(sp, device, mode, chunk=1 << 18):
    """sum over ordered pairs of unknown hands of w(o1) w(o2|o1) (win + tie, lose) of showdown_equity_batch(hero, known, o1, o2):
    unordered pairs are scored once and weighted by both orders (the showdown is symmetric in o1 and o2)."""
    import neuron_poker_b200 as npk
    r = np.array(sorted(set(range(52)) - set(sp.hero) - set(sum(sp.known, [])) - set(sp.board) - set(sp.dead)))
    n = len(r)
    b, a = np.nonzero(np.tril(np.ones((n, n), dtype=bool), -1))          # hands a < b
    H = len(a)
    i1, i2 = np.nonzero(np.triu(np.ones((H, H), dtype=bool), 1))
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
    acc = np.zeros(2, dtype=np.int64)
    for s in range(0, len(i1), chunk):
        e = min(len(i1), s + chunk)
        holes = np.empty((e - s, K + 3, 2), dtype=np.uint8)
        holes[:, :K + 1] = fixed
        holes[:, K + 1, 0], holes[:, K + 1, 1] = r[A1[s:e]], r[B1[s:e]]
        holes[:, K + 2, 0], holes[:, K + 2, 1] = r[A2[s:e]], r[B2[s:e]]
        out = npk.showdown_equity_batch(holes, np.full(e - s, K + 3, dtype=np.uint8), np.tile(brd, (e - s, 1)),
                                        np.tile(dead, (e - s, 1)), deal_mode=mode, device=device)
        wt = (out["win"][:, 0] + out["tie"][:, 0]).cpu().numpy()
        comp = out["completions"].cpu().numpy()
        acc += [(w[s:e] * wt).sum(), (w[s:e] * (comp - wt)).sum()]
    return int(acc[0]), int(acc[1])


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["uniform", "reference"])
def test_gpu_three_handed_flops_vs_weighted_showdown(cuda_device, mode):
    batch = spots(41, 2, 3, 2) + spots(42, 1, 3, 2, 1, 2)
    for sp, (w, t, l) in zip(batch, _exact(batch, cuda_device, mode)):
        assert (w + t, l) == _pair_sum(sp, cuda_device, mode), (sp, mode)
        assert w + t + l == sp.total(mode)


@pytest.mark.gpu
@pytest.mark.slow
def test_gpu_three_handed_preflop_vs_weighted_showdown(cuda_device):
    sp = Spot([12, 33], [[40, 41]], 2, [], [5, 22])
    (w, t, l), = _exact([sp], cuda_device)
    assert (w + t, l) == _pair_sum(sp, cuda_device, "reference")
    assert w + t + l == sp.total("reference")


@pytest.mark.gpu
def test_gpu_t3_three_handed_preflop(cuda_device):
    """The reference's test t3: AsKs against two random hands preflop, expected 51.8 %."""
    import neuron_poker_b200 as npk
    r = npk.exact_equity_counts({"AS", "KS"}, set(), 3)
    assert r["win"] + r["tie"] + r["lose"] == Spot([0, 1], [], 2, []).total("reference")
    assert (r["win"], r["tie"], r["lose"]) == T3_REFERENCE
    assert abs(100 * r["equity"] - 51.8) < 3
    T = 1 << 22
    npk.seed(505)
    try:
        e = npk.get_equity({"AS", "KS"}, set(), 3, T)
    finally:
        npk.seed(None)
    p = r["equity"]
    assert abs(e - p) < 4 * math.sqrt(p * (1 - p) / T), (e, p)


@pytest.mark.gpu
def test_gpu_known_opponents_monte_carlo_paths(cuda_device):
    import neuron_poker_b200 as npk
    T = 1 << 20
    cases = [(["AS", "KS"], [["QH", "QD"]], 3, ["2C", "7D", "KH"], ""), (["9H", "9S"], [["AD", "JC"], ["KC", "QC"]], 5, [], ""),
             (["TD", "7D"], [["8C", "8H"]], 3, ["8D", "QD", "2C", "5S"], ["AC", "3H"])]
    zs = {}
    for mode in ("uniform", "reference"):
        for ci, (hero, known, players, board, ghost) in enumerate(cases):
            ex = npk.exact_equity_counts(hero, board, players, known_opponents=known, ghost_cards=ghost, deal_mode=mode)
            p = ex["equity"]
            z = lambda wt: (wt / T - p) / math.sqrt(p * (1 - p) / T)
            r = npk.equity_counts_ranges(hero, board, players, T, ghost_cards=ghost, deal_mode=mode, seed_value=7 + ci,
                                         known_opponents=known)
            zs[(mode, ci, "counts")] = z(r["wins"] + r["ties"])
            ids = lambda cs: [oracle.ids([c])[0] for c in cs]
            hole = np.array([ids(hero)], dtype=np.uint8)
            brd = np.array([ids(board) + [NO] * (5 - len(board))], dtype=np.uint8)
            gh = np.array([ids(ghost)], dtype=np.uint8) if ghost else None
            kn = np.array([[ids(h) for h in known]], dtype=np.uint8)
            for passes in (True, False):
                out = npk.get_equity_ranges_batch(hole, brd, np.array([players], dtype=np.uint8), T, opponent_range=1, ghost=gh,
                                                  seed_value=11 + ci + 100 * passes, deal_mode=mode, passes=passes,
                                                  known_opponents=kn, device=cuda_device)
                zs[(mode, ci, passes)] = z(int(out["wins"][0] + out["ties"][0]))
    bad = {k: v for k, v in zs.items() if abs(v) > 4}
    assert not bad, bad


def _call(L, nl, dev, tensors, N, maxk, mode, flags, out, ws):
    import torch
    return L.npk_exact_equity_batch(*(t.data_ptr() for t in tensors[:4]), tensors[4].data_ptr() if tensors[4] is not None else None,
                                    N, maxk, mode, flags, *(o.data_ptr() for o in out), ws.data_ptr(),
                                    torch.cuda.current_stream(dev).cuda_stream)


def _dev_inputs(batch, device, maxk=None):
    import torch
    import neuron_poker_b200.evaluator as ev
    holes, nk, nr, board, dead = _arrays(batch, maxk)
    t = [torch.as_tensor(x).to(device) for x in (holes, nk, nr, board)]
    return t + [ev._dead_masks(dead, len(batch), device)]


@pytest.mark.gpu
def test_gpu_counts_do_not_depend_on_the_batch(cuda_device):
    import torch
    from neuron_poker_b200 import _lib as nl
    L = nl.ensure_init(cuda_device.index)
    sm = torch.cuda.get_device_properties(cuda_device).multi_processor_count
    preflop = Spot([51, 47], [], 1, [])
    probe = GPU_SPOTS[::3]
    rivers = spots(51, 4096, 5, 1, [0, 1, 2], 2)
    rivers[::7] = spots(52, len(rivers[::7]), 5, 2, [0, 1], 0)

    def run(batch, mode=nl.NPK_DEAL_REFERENCE):
        ins = _dev_inputs(batch, cuda_device, maxk=4)
        out = [torch.empty(len(batch), dtype=torch.int64, device=cuda_device) for _ in range(3)]
        ws = torch.empty(int(L.npk_exact_equity_workspace_bytes(len(batch))), dtype=torch.uint8, device=cuda_device)
        nl.check(_call(L, nl, cuda_device, ins, len(batch), 4, mode, 0, out, ws))
        items = int(ws[:8].view(torch.int64)[0]) - sm                # every CTA takes one item number past the last
        return list(zip(*(o.tolist() for o in out))), items

    alone, items = run([preflop])
    assert items >= sm, items                                        # one preflop spot: items span every SM
    full, _ = run(probe)
    assert run(probe[::-1])[0] == full[::-1]
    for i in (0, 5, len(probe) - 1):
        assert run([probe[i]])[0] == [full[i]]
    big = list(rivers)
    big[1000:1000] = [preflop]
    big[3000:3000] = probe
    got, items = run(big)
    assert items >= sm
    assert got[1000] == alone[0]
    assert got[3000:3000 + len(probe)] == full
    assert got[:1000] == run(rivers[:1000])[0]


@pytest.mark.gpu
def test_gpu_validation(cuda_device):
    import torch
    import neuron_poker_b200 as npk
    from neuron_poker_b200._lib import NpkError
    batch = spots(61, 4, 4, 1, 2, 2)
    holes, nk, nr, board, dead = _arrays(batch)

    def run(h=holes, k=nk, r=nr, b=board, d=dead, mode="reference"):
        return npk.exact_equity_batch(h, k, r, b, d, deal_mode=mode, device=cuda_device, validate=True)

    run()
    msg = "n_known outside 1..maxk, n_random outside 1..2, more than 10 players or too few cards"
    cases = []
    h = holes.copy(); h[1, 0, 0] = 52; cases.append((dict(h=h), -5))                          # id >= 52
    h = holes.copy(); h[2, 1, 1] = h[2, 0, 0]; cases.append((dict(h=h), -5))                  # a card twice in the hands
    b = board.copy(); b[0, 0] = holes[0, 2, 1]; cases.append((dict(b=b), -5))                 # board card also in a hand
    d = dead.copy(); d[3, 1] = board[3, 1]; cases.append((dict(d=d), -5))                     # dead card also on the board
    b = board.copy(); b[1, 1] = NO; cases.append((dict(b=b), -5))                             # a gap in the board
    d = dead.copy(); d[0, 0] = 60; cases.append((dict(d=d), -5))                              # dead id >= 52
    k = nk.copy(); k[2] = 0; cases.append((dict(k=k), -2))
    k = nk.copy(); k[2] = 4; cases.append((dict(k=k), -2))                                    # more than maxk
    r = nr.copy(); r[1] = 0; cases.append((dict(r=r), -2))
    r = nr.copy(); r[1] = 3; cases.append((dict(r=r), -2))
    for kw, code in cases:
        with pytest.raises(NpkError) as e:
            run(**kw)
        assert e.value.code == code, kw
        assert ("card id >= 52" in str(e.value)) if code == -5 else (msg in str(e.value)), kw
    # ten players: the hero, seven known hands and two unknown ones
    h8 = np.array([[[2 * p, 2 * p + 1] for p in range(8)]], dtype=np.uint8)
    out = npk.exact_equity_batch(h8, [8], [2], [[NO] * 5], None, device=cuda_device, validate=True)
    assert int(out["win"][0] + out["tie"][0] + out["lose"][0]) == Spot([0, 1], [[0, 0]] * 7, 2, []).total("reference")
    # too few cards: 2 hands and 39 dead cards leave 9 = 2k + m for two opponents and five board cards, one short under
    # REFERENCE; one more dead card leaves too few in either mode
    h2 = np.array([[[0, 1], [2, 3]]], dtype=np.uint8)
    d39, d40 = np.array([list(range(4, 43))], dtype=np.uint8), np.array([list(range(4, 44))], dtype=np.uint8)
    out = npk.exact_equity_batch(h2, [2], [2], [[NO] * 5], d39, deal_mode="uniform", device=cuda_device, validate=True)
    assert int(out["win"][0] + out["tie"][0] + out["lose"][0]) == math.comb(9, 2) * math.comb(7, 2) * math.comb(5, 5)
    for d, mode in ((d39, "reference"), (d40, "uniform")):
        with pytest.raises(NpkError) as e:
            npk.exact_equity_batch(h2, [2], [2], [[NO] * 5], d, deal_mode=mode, device=cuda_device, validate=True)
        assert e.value.code == -2 and msg in str(e.value), mode
    # without the flag, garbage bytes give no fault and a spot with too few cards gets nothing
    g = torch.Generator().manual_seed(0)
    N = 2048
    npk.exact_equity_batch(torch.randint(0, 256, (N, 8, 2), dtype=torch.uint8, generator=g).cuda(),
                           torch.randint(0, 256, (N,), dtype=torch.uint8, generator=g).cuda(),
                           torch.randint(0, 4, (N,), dtype=torch.uint8, generator=g).cuda(),
                           torch.randint(0, 256, (N, 5), dtype=torch.uint8, generator=g).cuda(),
                           torch.randint(0, 256, (N, 3), dtype=torch.uint8, generator=g).cuda(), device=cuda_device)
    torch.cuda.synchronize()
    out = npk.exact_equity_batch(h2, [2], [2], [[NO] * 5], d40, deal_mode="uniform", device=cuda_device, validate=False)
    assert not any(int(out[k][0]) for k in ("win", "tie", "lose"))
    with pytest.raises(NpkError, match="deal_mode"):
        npk.exact_equity_batch(holes, nk, nr, board, dead, deal_mode="biased", device=cuda_device)


@pytest.mark.gpu
def test_gpu_graph_capture(cuda_device):
    import torch
    from neuron_poker_b200 import _lib as nl
    L = nl.ensure_init(cuda_device.index)
    batch = GPU_SPOTS[:12]
    ins = _dev_inputs(batch, cuda_device)
    maxk = ins[0].shape[1]
    out = [torch.empty(len(batch), dtype=torch.int64, device=cuda_device) for _ in range(3)]
    ws = torch.empty(int(L.npk_exact_equity_workspace_bytes(len(batch))), dtype=torch.uint8, device=cuda_device)
    s = torch.cuda.Stream(cuda_device)
    s.wait_stream(torch.cuda.current_stream(cuda_device))
    with torch.cuda.stream(s):                                   # warm-up (module load, shared-memory attribute)
        nl.check(_call(L, nl, cuda_device, ins, len(batch), maxk, nl.NPK_DEAL_REFERENCE, 0, out, ws))
    torch.cuda.current_stream(cuda_device).wait_stream(s)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        nl.check(_call(L, nl, cuda_device, ins, len(batch), maxk, nl.NPK_DEAL_REFERENCE, 0, out, ws))
    for o in out:
        o.fill_(-1)
    g.replay()
    torch.cuda.synchronize()
    assert list(zip(*(o.tolist() for o in out))) == _exact(batch, cuda_device)
