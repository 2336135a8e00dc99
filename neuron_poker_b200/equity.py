"""Drop-in equity calculators of the reference, backed by libnpk's sm_100a kernels.

Reference interfaces mirrored here (same names, positional arguments, return types and error behaviour):

  get_equity(player_cards, table_cards, players, runs) -> float
        tools/montecarlo_python.py:401-406.  Dealing = the Python reference's own dealer (NPK_DEAL_REFERENCE), ties
        count as wins.  Unlike the reference it always runs all `runs` trials (the reference silently stops after
        1 s of wall clock, :235-239, :405).
  montecarlo(my_cards, cards_on_table, number_of_players, iterations) -> float
        the pybind11 export tools/montecarlo_cpp/pymontecarlo.cpp:21-23 -> Montecarlo.cpp:240-259.  Uniform dealing,
        a table of fewer than 3 cards is treated as empty (:242-243), ties count as wins.
  MonteCarlo().run_montecarlo(...)   tools/montecarlo_python.py:191-252 with .equity/.runs/.passes/.winnerCardTypeList

Install into the environment by assigning the attribute the env binds in its constructor (gym_env/env.py:75-81):
    env.get_equity = neuron_poker_b200.get_equity          # or patch tools.montecarlo_python.get_equity before
                                                           # HoldemTable() is constructed
"""
import ctypes
import os
import threading
from collections import Counter

import numpy as np

from . import _lib, ranges
from .cards import HAND_TYPES, NO_CARD, _CARD_ID, card_ids, encode_query

DEAL_UNIFORM = _lib.NPK_DEAL_UNIFORM
DEAL_REFERENCE = _lib.NPK_DEAL_REFERENCE
_DEAL = {"uniform": DEAL_UNIFORM, "reference": DEAL_REFERENCE, DEAL_UNIFORM: DEAL_UNIFORM,
         DEAL_REFERENCE: DEAL_REFERENCE}

_seed_state = {"rng": None}


def seed(value=None):
    """Fix the stream of per-call Philox seeds.  Without it each call draws its seed from numpy's GLOBAL legacy RNG,
    the generator the reference itself consumes (montecarlo_python.py:169-170, 188), so np.random.seed(s) -- which is
    what HoldemTable.reset(seed) does (gym_env/env.py:141-142) -- makes a whole run reproducible, as in the reference."""
    _seed_state["rng"] = None if value is None else np.random.RandomState(int(value) & 0xFFFFFFFF)


_global_sample = np.random.random_sample       # bound method of numpy's global legacy RandomState (np.random.seed reseeds it)


def _next_seed():
    """53 random bits from the global legacy RandomState (one call; the reference's own generator)."""
    rng = _seed_state["rng"]
    return int((_global_sample() if rng is None else rng.random_sample()) * 9007199254740992.0)


_device_cache = {}


def _device():
    key = (os.environ.get("NPK_DEVICE"), os.environ.get("LOCAL_RANK"))
    d = _device_cache.get(key)
    if d is None:
        d = _device_cache[key] = int(key[0] if key[0] is not None else (key[1] if key[1] is not None else "0"))
    return d


def _u8(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def _seed(seed_value):
    """A Philox seed as libnpk takes it: the integer modulo 2^64."""
    return ctypes.c_uint64(int(seed_value) & (2**64 - 1))


class _CallBuffers(threading.local):
    """Per-thread result buffer of the one-query calls: allocated once and addressed by integer (a ctypes void* parameter
    accepts an int), so a get_equity call creates no arrays and no ctypes objects."""

    def __init__(self):
        self.out = (ctypes.c_uint64 * 12)()               # wins ties types[9] passes
        self.p_out = ctypes.addressof(self.out)


_buffers = _CallBuffers()
_PAD = tuple((((1 << (8 * m)) - 1) << (56 - 8 * m)) for m in range(6))      # 0xFF bytes for m MISSING board cards


def _pack_query(player_cards, table_cards):
    """hole[0] | hole[1] << 8 | board << 16 as one integer (0xFF for board cards not dealt yet).  Unknown card strings
    raise ValueError like list.index in the reference (montecarlo_python.py:127-128); duplicates are caught by the library."""
    ids = _CARD_ID
    try:
        hole = [ids[c] for c in player_cards]
        board = [ids[c] for c in table_cards]
    except (KeyError, TypeError):
        hole, board = card_ids(player_cards), card_ids(table_cards)      # card ids, or the reference's ValueError
    if len(hole) != 2:
        raise ValueError("player_cards must hold exactly two cards, got %d" % len(hole))
    nb = len(board)
    if nb > 5:
        raise ValueError("table_cards holds more than five cards")
    packed = hole[0] | hole[1] << 8 | _PAD[5 - nb]
    shift = 16
    for c in board:
        packed |= c << shift
        shift += 8
    return packed


def equity_counts(player_cards, table_cards, players, runs, deal_mode="uniform", seed_value=None, win_types=False,
                  passes=False):
    """One query through the one-query C entry point npk_equity_one: returns dict(wins, ties, runs[, win_types, passes]).
    `wins` = trials the hero strictly wins, `ties` = trials tied for best."""
    players = int(players)                      # numpy.int64 from sum(alive) is what the env passes (env.py:262)
    runs = int(runs)
    if players < 1:
        raise IndexError("list index out of range")     # reference: hands[winner] on an empty list
    if players > 10:
        raise ValueError("at most 10 players")
    packed = _pack_query(player_cards, table_cards)
    b = _buffers
    L = _lib.ensure_current(_device())
    s = _next_seed() if seed_value is None else int(seed_value) & (2**64 - 1)
    rc = L.npk_equity_one(packed, players, runs, s, _DEAL[deal_mode], (1 if win_types else 0) | (2 if passes else 0), b.p_out)
    if rc < 0:
        if rc == -5:
            raise ValueError("duplicate or invalid cards in player_cards / table_cards: " + L.npk_last_error().decode())
        _lib.check(rc)
    out = b.out
    res = {"wins": out[0], "ties": out[1], "runs": runs}
    if win_types:
        res["win_types"] = [out[i] for i in range(2, 11)]
    if passes:
        res["passes"] = out[11]
    return res


class PendingCounts(object):
    """A batch in flight (equity_counts_batch(..., block=False)): result() blocks until its counters are on the host."""

    def __init__(self, L, ticket, out):
        self._L, self._ticket, self._out = L, ticket, out

    def result(self):
        if self._ticket is not None:
            out = self._out
            rc = self._L.npk_equity_host_wait(self._ticket, _u8(out["wins"]), _u8(out["ties"]),
                                              _u8(out["win_types"]) if "win_types" in out else None,
                                              _u8(out["passes"]) if "passes" in out else None)
            self._ticket = None
            _lib.check(rc)
        return self._out


MAX_IN_FLIGHT = 4          # NPK_HOST_SLOTS


def equity_counts_batch(hole, board, n_players, trials, seed_value=0, deal_mode="uniform", win_types=False,
                        passes=False, block=True):
    """Host arrays in, host arrays out (numpy, uint8 [Q,2] / [Q,5] with 0xFF padding / [Q]): one blocking call of
    npk_equity_host = H2D copy of the queries from pinned staging, the kernels, D2H copy of the counters.
    Returns dict(wins [Q] uint64, ties [Q] uint64[, win_types [Q,9], passes [Q]]).
    block=False submits the batch (npk_equity_host_submit) and returns a PendingCounts whose result() gives the same dict:
    up to MAX_IN_FLIGHT batches per thread can be in flight, so the staging and the copies of one batch overlap the kernel
    of the previous one (the queries are copied at submission; the arrays may be reused at once)."""
    hole = np.ascontiguousarray(hole, dtype=np.uint8).reshape(-1, 2)
    board = np.ascontiguousarray(board, dtype=np.uint8).reshape(-1, 5)
    n_players = np.ascontiguousarray(n_players, dtype=np.uint8).reshape(-1)
    Q = len(hole)
    if not (len(board) == Q and len(n_players) == Q):
        raise ValueError("hole, board and n_players must describe the same number of queries")
    L = _lib.ensure_init(_device())
    out = {"wins": np.zeros(Q, dtype=np.uint64), "ties": np.zeros(Q, dtype=np.uint64)}
    if win_types:
        out["win_types"] = np.zeros((Q, 9), dtype=np.uint64)
    if passes:
        out["passes"] = np.zeros(Q, dtype=np.uint64)
    if not block:
        if Q == 0:
            return PendingCounts(L, None, out)
        ticket = L.npk_equity_host_submit(_u8(hole), _u8(board), _u8(n_players), Q, int(trials),
                                          _seed(seed_value), _DEAL[deal_mode],
                                          (1 if win_types else 0) | (2 if passes else 0))
        _lib.check(ticket)
        return PendingCounts(L, ticket, out)
    _lib.check(L.npk_equity_host(_u8(hole), _u8(board), _u8(n_players), Q, int(trials),
                                 _seed(seed_value), _DEAL[deal_mode], _u8(out["wins"]),
                                 _u8(out["ties"]), _u8(out["win_types"]) if win_types else None,
                                 _u8(out["passes"]) if passes else None))
    return out


def resident(on=True, sms=0, idle_us=200):
    """Resident mode of the one-query calls of THIS thread (get_equity, montecarlo, equity_counts without win types / passes):
    npk_resident_start keeps a persistent kernel with the tables staged on `sms` SMs (0 = all) that takes every call from a
    mailbox in mapped host memory instead of being launched per call; it leaves by itself after `idle_us` microseconds without
    a call and is restarted by the next one.  Same results bit for bit; while it is resident other GPU work waits for its SMs,
    hence opt-in (tight get_equity loops: single-environment stepping).  resident(False) returns to one launch per call."""
    L = _lib.ensure_current(_device())
    _lib.check(L.npk_resident_start(int(sms), int(idle_us)) if on else L.npk_resident_stop())


_fast_equity = None


def _fast_call(player_cards, table_cards, players, runs, mode):
    """The common case of a one-query call through the C binding (csrc/npk_pyfast.c): card strings -> npk_equity_one -> float
    without Python byte code in between.  None = not the common case, or an error: the caller runs the Python implementation,
    which raises the reference's exceptions."""
    global _fast_equity
    if getattr(_lib._current, "device", None) != _device():
        return None           # first call of this thread: the Python path validates the arguments, then initialises the device
    f = _fast_equity
    if f is None:
        f = _fast_equity = _lib.fast().equity
    rng = _seed_state["rng"]            # the call's Philox seed comes from the generator _next_seed uses
    return f(player_cards, table_cards, players, runs, mode, _global_sample if rng is None else rng.random_sample)


def get_equity(player_cards, table_cards, players, runs):
    """Get equity from a montecarlo run -- drop-in for tools/montecarlo_python.py:401-406 (reference dealing)."""
    e = _fast_call(player_cards, table_cards, players, runs, DEAL_REFERENCE)
    if e is not None:
        return e
    r = equity_counts(player_cards, table_cards, players, runs, "reference")
    return (r["wins"] + r["ties"]) / runs


def montecarlo(my_cards, cards_on_table, number_of_players, iterations):
    """Drop-in for the C++ calculator pymontecarlo.montecarlo (Montecarlo.cpp:240-259): uniform dealing; a table with
    fewer than 3 cards (the reference's callers pass {'null'}) is cleared (:242-243)."""
    table = list(cards_on_table)
    if len(table) < 3:
        table = []
    e = _fast_call(my_cards, table, number_of_players, iterations, DEAL_UNIFORM)
    if e is not None:
        return e
    try:
        r = equity_counts(my_cards, table, number_of_players, iterations, deal_mode="uniform")
    except ValueError as exc:                   # pybind11 surfaces std::runtime_error as RuntimeError
        raise RuntimeError("Card Type error!") from exc
    return (r["wins"] + r["ties"]) / iterations


def numpy_montecarlo(my_cards, table_cards_alpha_numeric, iterations, player_amount):
    """Call form of the numpy sibling, tools/montecarlo_numpy2.py:333-346: `my_cards` is [[card1, card2]], the argument order
    is (cards, table, iterations, players) and the result is the equity in PER CENT.  Uniform dealing like the sibling's
    argsort shuffle (:80-83), ties counted as wins -- i.e. what its (upstream skipped) tests expect
    (tests/test_montecarlo_numpy.py: the Python tests' values, +-1 point); its upstream defects (the first two board cards
    are dropped, :340; sole wins only, :309-313; results wrong post-flop) are NOT reproduced."""
    r = equity_counts(my_cards[0], table_cards_alpha_numeric, player_amount, iterations, "uniform")
    return 100.0 * (r["wins"] + r["ties"]) / int(iterations)


def equity_counts_ranges(player_cards, table_cards, players, runs, opponent_range=1, ghost_cards='',
                         deal_mode="reference", seed_value=None, known_opponents=()):
    """One run_montecarlo call with ranges through npk_equity_ranges_host (blocking).

    player_cards: two card strings, or a SET of class spellings ('AKO', 'AA', ...): the hero is then drawn from that
    range every trial (montecarlo_python.py:136-148).  opponent_range: a fraction of the reference's preflop ranking
    (:36-112) or a set of class spellings (:194-199).  ghost_cards: '' or two cards removed from the deck (:206-208).
    known_opponents: hands (two card strings each) of opponents whose cards are known -- the further entries of the
    reference's player_card_list (:132-163); they count among `players`.
    Returns dict(wins, ties, runs, win_types[9], passes)."""
    players, runs = int(players), int(runs)
    if players < 1:
        raise IndexError("list index out of range")
    if players > 10:
        raise ValueError("at most 10 players")
    hero_is_range = isinstance(player_cards, (set, frozenset))       # reference: `type(player_cards) == set` (:136)
    board = card_ids(table_cards)
    if len(board) > 5:
        raise ValueError("table_cards holds more than five cards")
    ghost = card_ids(ghost_cards) if ghost_cards not in ('', None) else []
    if ghost and len(ghost) != 2:
        raise ValueError("ghost_cards must be '' or two cards")
    hole = None
    if not hero_is_range:
        hole = card_ids(player_cards)
        if len(hole) != 2:
            raise ValueError("player_cards must hold exactly two cards, got %d" % len(hole))
    known = []
    for hand in known_opponents:
        if isinstance(hand, (set, frozenset)):
            raise NotImplementedError("a known opponent must be two cards, not a range")
        ids = card_ids(hand)
        if len(ids) != 2:
            raise ValueError("a known opponent's hand must hold exactly two cards, got %d" % len(ids))
        known += ids
    n_known = len(known) // 2
    if n_known and hero_is_range:
        raise NotImplementedError("a hero range together with known opponent hands (the reference draws the hero before it "
                                  "removes the known hands and deals duplicate cards, montecarlo_python.py:132-163)")
    if n_known > players - 1:
        raise ValueError("more known hands than players")
    opp_mask = ranges.opponent_mask(opponent_range)
    hero_mask = ranges.mask_from_classes(player_cards) if hero_is_range else None
    L = _lib.ensure_init(_device())
    hole_a = np.array(hole, dtype=np.uint8) if hole is not None else None
    board_a = np.array(board + [NO_CARD] * (5 - len(board)), dtype=np.uint8)
    ghost_a = np.array(ghost, dtype=np.uint8) if ghost else None
    npl = np.array([players], dtype=np.uint8)
    out_w, out_t = np.zeros(1, dtype=np.uint64), np.zeros(1, dtype=np.uint64)
    out_ty, out_p = np.zeros(9, dtype=np.uint64), np.zeros(1, dtype=np.uint64)
    s = _next_seed() if seed_value is None else int(seed_value)
    known_a = np.array(known, dtype=np.uint8) if n_known else None
    rc = L.npk_equity_ranges_known_host(_u8(hole_a) if hole_a is not None else None, _u8(board_a), _u8(npl),
                                        _u8(ghost_a) if ghost_a is not None else None,
                                        _u8(known_a) if known_a is not None else None, n_known, 1, runs, _u8(opp_mask),
                                        _u8(hero_mask) if hero_mask is not None else None,
                                        _seed(s), _DEAL[deal_mode], _u8(out_w), _u8(out_t),
                                        _u8(out_ty), _u8(out_p))
    _lib.check(rc)
    return {"wins": int(out_w[0]), "ties": int(out_t[0]), "runs": runs, "win_types": [int(x) for x in out_ty],
            "passes": int(out_p[0])}


class MonteCarlo(object):
    """Mirror of tools/montecarlo_python.py::MonteCarlo: the get_equity path (opponent_range=1) and the range / hero-range /
    ghost-card variants of run_montecarlo."""

    def create_card_deck(self):
        from .cards import DECK
        return list(DECK)

    def get_two_short_notation(self, input_cards, add_O_to_pairs=False):
        """montecarlo_python.py:24-34: both spellings of the starting-hand class of two cards."""
        card1, card2 = input_cards[0][0], input_cards[1][0]
        suited_str = 'S' if input_cards[0][1] == input_cards[1][1] else 'O'
        if card1 == card2:
            suited_str = "O" if add_O_to_pairs else ''
        return card1 + card2 + suited_str, card2 + card1 + suited_str

    def get_opponent_allowed_cards_list(self, opponent_ranges):
        """montecarlo_python.py:36-112: the top int(169 * range) classes of the reference's preflop ranking."""
        return ranges.allowed_classes(opponent_ranges)

    def run_montecarlo(self, original_player_card_list, original_table_card_list, player_amount, ui, maxRuns,
                       timeout, ghost_cards, opponent_range=1):
        """montecarlo_python.py:191-252.  `ui` and `timeout` are accepted and ignored (every run is executed).
        The plain case (opponent_range=1, one fixed hero, no ghost cards) runs equity_refdeal_kernel; anything else -- ranges,
        ghost cards, further known hands in the player list -- runs the range kernel.  A range no remaining hand can satisfy raises NpkError instead of looping forever."""
        if len(original_player_card_list) < 1:
            raise IndexError("list index out of range")
        hero = original_player_card_list[0]
        known = list(original_player_card_list[1:])       # further known hands: opponents whose cards are known (:132-163)
        plain = (ghost_cards == '' and not isinstance(opponent_range, (set, frozenset)) and
                 not isinstance(hero, (set, frozenset)) and not known and
                 len(ranges.allowed_classes(opponent_range)) == ranges.N_CLASSES)
        if plain:
            r = equity_counts(hero, original_table_card_list, player_amount, maxRuns, deal_mode="reference",
                              win_types=True, passes=True)
        else:
            r = equity_counts_ranges(hero, original_table_card_list, player_amount, maxRuns, opponent_range=opponent_range,
                                     ghost_cards=ghost_cards, deal_mode="reference", known_opponents=known)
        runs = r["runs"]
        self.equity = (r["wins"] + r["ties"]) / runs
        self.winnerCardTypeList = Counter({HAND_TYPES[i]: c / runs for i, c in enumerate(r["win_types"]) if c})
        self.winTypesDict = self.winnerCardTypeList.items()
        self.runs = runs
        self.passes = r["passes"]
        return self.equity, self.winTypesDict


# ---- batched API on device tensors -----------------------------------------------------------------------------------
def _batched_call(name, args, dev, Q, win_types, passes, adaptive=False, out=None):
    """libnpk's batched call `name`(*args, wins, ties, win_types, passes[, trials], workspace, stream) on the current torch
    stream of `dev`, with a workspace of its own.  Returns the outputs, int64 CUDA tensors viewing the u64 counters.  A fixed
    call adds to zeroed counters and uses those the caller's `out` already holds; an adaptive call zeroes its outputs itself
    and adds trials [Q]."""
    import torch
    L = _lib.ensure_init(dev.index)
    fields = [("wins", (Q,), True), ("ties", (Q,), True), ("win_types", (Q, 9), win_types), ("passes", (Q,), passes)]
    if adaptive:
        fields.append(("trials", (Q,), True))
    with torch.cuda.device(dev):
        out = {} if out is None else out
        for field, shape, want in fields:
            if want and field not in out:
                out[field] = (torch.empty if adaptive and Q else torch.zeros)(shape, dtype=torch.int64, device=dev)
        ws_bytes = L.npk_equity_adaptive_workspace_bytes if adaptive else L.npk_equity_workspace_bytes
        ws = torch.empty(int(ws_bytes(Q)), dtype=torch.uint8, device=dev)
        stream = torch.cuda.current_stream(dev)
        _lib.check(getattr(L, name)(*args, *(out[field].data_ptr() if want else None for field, _, want in fields),
                                    ws.data_ptr(), stream.cuda_stream))
        ws.record_stream(stream)
    return out


def get_equity_ranges_batch(hole, board, n_players, trials, opponent_range=1, hero_range=None, ghost=None, seed_value=0,
                            deal_mode="reference", trial_offset=0, query_offset=0, device=None, validate=True,
                            win_types=False, passes=False, out=None, known_opponents=None):
    """Batched Monte-Carlo counts with ranges (asynchronous on the current torch stream unless validate=True).
    known_opponents: None or [Q, n_known, 2] uint8 -- opponents whose cards are known (they count among n_players).

    opponent_range: fraction or set of class spellings shared by every query; hero_range: None (fixed `hole` [Q,2]) or a
    set of class spellings (the hero is drawn from it every trial, `hole` may be None); ghost: None or [Q,2] uint8
    (0xFF = none).  Returns dict of int64 CUDA tensors like get_equity_batch."""
    dev, a = _range_args(hole, board, n_players, opponent_range, hero_range, ghost, known_opponents, device)
    out = _batched_call("npk_equity_ranges_known_batch",
                        (a.hole, a.board, a.n_players, a.ghost, a.known, a.n_known, a.Q, int(trials), _u8(a.opp_mask),
                         a.hero_mask, _seed(seed_value), int(trial_offset), int(query_offset), _DEAL[deal_mode],
                         _lib.NPK_FLAG_VALIDATE if validate else 0),
                        dev, a.Q, win_types, passes, out=out)
    out["trials"] = int(trials)
    return out


def _range_args(hole, board, n_players, opponent_range, hero_range, ghost, known_opponents, device):
    """The arguments of the batched range calls as libnpk takes them: device pointers (or None), n_known, Q and the class
    masks.  The namespace holds the tensors and mask arrays too, so that the pointers stay valid while it lives."""
    import torch
    from types import SimpleNamespace
    dev = _resolve_device(device)
    a = SimpleNamespace()
    a.t_board = _as_cuda_u8(board, dev, (5,))
    a.t_players = _as_cuda_u8(n_players, dev, ())
    a.Q = Q = a.t_board.shape[0]
    a.t_hole = None if hero_range is not None else _as_cuda_u8(hole, dev, (2,))
    a.t_ghost = None if ghost is None else _as_cuda_u8(ghost, dev, (2,))
    a.n_known, a.t_known = 0, None
    if known_opponents is not None:
        a.t_known = torch.as_tensor(known_opponents, dtype=torch.uint8).to(dev).contiguous()
        if a.t_known.dim() != 3 or a.t_known.shape[0] != Q or a.t_known.shape[2] != 2:
            raise ValueError("known_opponents must have shape [Q, n_known, 2]")
        a.n_known = int(a.t_known.shape[1])
    a.opp_mask = ranges.opponent_mask(opponent_range)
    a.hero_mask_array = None if hero_range is None else ranges.mask_from_classes(hero_range)
    a.hole = a.t_hole.data_ptr() if a.t_hole is not None else None
    a.board, a.n_players = a.t_board.data_ptr(), a.t_players.data_ptr()
    a.ghost = a.t_ghost.data_ptr() if a.t_ghost is not None else None
    a.known = a.t_known.data_ptr() if a.n_known else None
    a.hero_mask = _u8(a.hero_mask_array) if a.hero_mask_array is not None else None
    return dev, a



def _resolve_device(device):
    """torch.device with an explicit index: 'cuda' (or None) means torch's CURRENT device, not device 0 -- libnpk selects the
    device by index, and the tensors must live where its kernels run."""
    import torch
    dev = torch.device("cuda") if device is None else torch.device(device)
    if dev.type != "cuda":
        raise ValueError("libnpk runs on CUDA devices only (there is no CPU fallback): got %r" % (device,))
    return dev if dev.index is not None else torch.device("cuda", torch.cuda.current_device())


def _as_cuda_u8(x, device, shape_tail):
    import torch
    if not isinstance(x, torch.Tensor):
        x = torch.as_tensor(np.ascontiguousarray(x, dtype=np.uint8))
    if x.dtype != torch.uint8:
        x = x.to(torch.uint8)
    x = x.to(device, non_blocking=True).contiguous()
    assert tuple(x.shape[1:]) == tuple(shape_tail), (x.shape, shape_tail)
    return x


def shape_mask(players, known_board_cards=(0, 3, 4, 5)):
    """Bit mask of the (players, known board cards) shapes a sync-free mixed batch may contain."""
    m = 0
    for p in players:
        for k in known_board_cards:
            m |= 1 << ((int(p) - 1) * 6 + int(k))
    return m


def get_equity_batch(hole, board, n_players, trials, seed_value=0, deal_mode="uniform", trial_offset=0, device=None,
                     uniform_shape=None, validate=True, win_types=False, passes=False, out=None, query_offset=0,
                     shapes=None):
    """Monte-Carlo counts for a batch of queries on the GPU (asynchronous on the current torch stream).

    hole [Q,2], board [Q,5] (0xFF padding), n_players [Q]: uint8 torch tensors (or array-likes, copied to the device).
    uniform_shape=(players, known_board_cards) promises every query has that shape: that shape's own kernel runs.
    Otherwise the batch may MIX shapes: the queries are sorted by shape on the device and one persistent kernel handles all
    of them (csrc/npk_mixed.cu) -- no host round trip unless validate=True.  shapes=shape_mask(...) restricts a mixed batch
    to some shapes (npk_equity_batch_async); queries of other shapes are skipped.
    trial_offset / query_offset shift the Philox counters, so shards of a larger job reproduce its exact numbers.
    Returns dict of int64 CUDA tensors: wins [Q], ties [Q] (+ win_types [Q,9], passes [Q]); the counters are u64 on
    the device and viewed as int64.  `out` may hold preallocated zeroed tensors to accumulate into.
    """
    dev = _resolve_device(device)
    hole = _as_cuda_u8(hole, dev, (2,))
    board = _as_cuda_u8(board, dev, (5,))
    n_players = _as_cuda_u8(n_players, dev, ())
    Q = hole.shape[0]
    queries = (hole.data_ptr(), board.data_ptr(), n_players.data_ptr(), Q, int(trials))
    if shapes is not None and uniform_shape is None:
        out = _batched_call("npk_equity_batch_async",
                            queries + (ctypes.c_uint64(int(shapes)), _seed(seed_value), int(trial_offset), int(query_offset),
                                       _DEAL[deal_mode]),
                            dev, Q, win_types, passes, out=out)
    else:
        up, uk = (-1, -1) if uniform_shape is None else (int(uniform_shape[0]), int(uniform_shape[1]))
        out = _batched_call("npk_equity_batch",
                            queries + (up, uk, _seed(seed_value), int(trial_offset), int(query_offset), _DEAL[deal_mode],
                                       _lib.NPK_FLAG_VALIDATE if validate else 0),
                            dev, Q, win_types, passes, out=out)
    out["trials"] = int(trials)
    return out


ALL_SHAPES = (1 << 60) - 1


def adaptive_checkpoints(min_trials, max_trials):
    """Checkpoints of get_equity_batch_adaptive: T_0 = min_trials, T_{k+1} = min(2 T_k, max_trials), up to max_trials."""
    min_trials, max_trials = int(min_trials), int(max_trials)
    if not 1 <= min_trials <= max_trials:
        raise ValueError("need 1 <= min_trials <= max_trials, got %d, %d" % (min_trials, max_trials))
    t = [min_trials]
    while t[-1] < max_trials:
        t.append(min(2 * t[-1], max_trials))
    return t


def adaptive_stops(wins_plus_ties, trials, stderr):
    """The stopping rule of get_equity_batch_adaptive after checkpoint `trials`, in the device's order of double operations:
    p = (x + 1) / (T + 2), var = p (1 - p) / T, stop when var <= stderr * stderr."""
    p = (float(wins_plus_ties) + 1.0) / float(trials + 2)
    return p * (1.0 - p) / float(trials) <= stderr * stderr


def get_equity_batch_adaptive(hole, board, n_players, max_trials, stderr, min_trials=256, seed_value=0, deal_mode="uniform",
                              query_offset=0, shapes=None, device=None, validate=True, win_types=False, passes=False):
    """Monte-Carlo counts to a target precision (npk_equity_batch_adaptive, asynchronous on the current torch stream unless
    validate=True): every query runs until the standard error of its equity (wins + ties) / trials is at most `stderr`,
    checked at the checkpoints adaptive_checkpoints(min_trials, max_trials), or until max_trials.  The counters of a query
    are exactly those of get_equity_batch(trials=T_stop) with the same seed and query_offset, whatever else is in the batch.
    Returns the dict of get_equity_batch, except that `trials` is an int64 CUDA tensor [Q] holding every query's T_stop
    (0 for a query outside `shapes`, or an invalid one when validate=False)."""
    dev = _resolve_device(device)
    hole = _as_cuda_u8(hole, dev, (2,))
    board = _as_cuda_u8(board, dev, (5,))
    n_players = _as_cuda_u8(n_players, dev, ())
    Q = hole.shape[0]
    return _batched_call("npk_equity_batch_adaptive",
                         (hole.data_ptr(), board.data_ptr(), n_players.data_ptr(), Q, int(min_trials), int(max_trials),
                          ctypes.c_double(float(stderr)),
                          ctypes.c_uint64(ALL_SHAPES if shapes is None else int(shapes) & ALL_SHAPES), _seed(seed_value),
                          int(query_offset), _DEAL[deal_mode], _lib.NPK_FLAG_VALIDATE if validate else 0),
                         dev, Q, win_types, passes, adaptive=True)


def get_equity_ranges_batch_adaptive(hole, board, n_players, max_trials, stderr, min_trials=256, opponent_range=1,
                                     hero_range=None, ghost=None, known_opponents=None, seed_value=0, deal_mode="reference",
                                     query_offset=0, device=None, validate=True, win_types=False, passes=False):
    """get_equity_batch_adaptive for the range calls (npk_equity_ranges_batch_adaptive, asynchronous on the current torch
    stream unless validate=True): every query runs until the standard error of its equity (wins + ties) / trials is at most
    `stderr`, checked at adaptive_checkpoints(min_trials, max_trials), or until max_trials.  The range arguments are those of
    get_equity_ranges_batch, and the counters of a query are exactly those of get_equity_ranges_batch(trials=T_stop) with the
    same seed, query_offset, ranges, ghost cards, known hands and sampler (passes=True: the generic kernel, else the pair-list
    sampler).  Returns the dict of get_equity_batch_adaptive: `trials` is an int64 CUDA tensor [Q] of every query's T_stop
    (0 for an invalid query when validate=False)."""
    dev, a = _range_args(hole, board, n_players, opponent_range, hero_range, ghost, known_opponents, device)
    return _batched_call("npk_equity_ranges_batch_adaptive",
                         (a.hole, a.board, a.n_players, a.ghost, a.known, a.n_known, a.Q, int(min_trials), int(max_trials),
                          ctypes.c_double(float(stderr)), _u8(a.opp_mask), a.hero_mask, _seed(seed_value),
                          int(query_offset), _DEAL[deal_mode], _lib.NPK_FLAG_VALIDATE if validate else 0),
                         dev, a.Q, win_types, passes, adaptive=True)
