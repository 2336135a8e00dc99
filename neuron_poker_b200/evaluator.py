"""Hand evaluation through the GPU rank tables: batched rank ids, showdown winners and exact enumeration.

Mirrors tools/hand_evaluator.py of the reference: `get_winner` (:9-17) and `eval_best_hand` (:20-24) keep their
signatures; the ordering is the reference's `_calc_score` ordering (:27-119) expressed as a rank id in [0, 5034).
"""
import ctypes

import numpy as np

from . import _lib
from .cards import HAND_TYPES, NO_CARD, card_ids, encode_query

N_HANDS_7 = 133784560  # C(52,7)


def _torch():
    import torch
    return torch


def _dev(device):
    from .equity import _resolve_device
    return _resolve_device(device)


def _want_check(x, validate):
    """Inputs are validated on the device (NPK_FLAG_VALIDATE: one extra pass + a synchronisation) unless the caller hands
    over CUDA tensors -- the batched hot-path form -- and does not ask for it."""
    if validate is None:
        torch = _torch()
        validate = not (isinstance(x, torch.Tensor) and x.is_cuda)
    return _lib.NPK_FLAG_VALIDATE if validate else 0


def rank7(cards, device=None, validate=None):
    """cards: [N,7] uint8 card ids (torch tensor or array-like) -> int16-viewable uint16 CUDA tensor of rank ids.
    validate: check ids / duplicates first (ValueError-like NpkError); default: yes unless `cards` is a CUDA tensor."""
    torch = _torch()
    dev = _dev(device)
    flags = _want_check(cards, validate)
    if not isinstance(cards, torch.Tensor):
        cards = torch.as_tensor(np.ascontiguousarray(cards, dtype=np.uint8))
    cards = cards.to(dev).contiguous().view(-1, 7)
    L = _lib.ensure_init(dev.index)
    out = torch.empty(cards.shape[0], dtype=torch.uint16, device=dev)
    with torch.cuda.device(dev):
        _lib.check(L.npk_rank7_batch(cards.data_ptr(), cards.shape[0], out.data_ptr(), flags,
                                     torch.cuda.current_stream(dev).cuda_stream))
    return out


def rank7_colex(first, count, device=None):
    """rank ids of hands number first..first+count-1 of the colexicographic enumeration of all C(52,7) hands."""
    torch = _torch()
    dev = _dev(device)
    L = _lib.ensure_init(dev.index)
    out = torch.empty(int(count), dtype=torch.uint16, device=dev)
    with torch.cuda.device(dev):
        _lib.check(L.npk_rank7_colex(int(first), int(count), out.data_ptr(), torch.cuda.current_stream(dev).cuda_stream))
    return out


def showdown(holes, n_players, board, device=None, return_ranks=False, validate=None):
    """Batched get_winner: holes [N,maxp,2], n_players [N], board [N,5] -> (winner int32 [N], type uint8 [N][, ranks])."""
    torch = _torch()
    dev = _dev(device)
    flags = _want_check(holes, validate)
    holes = torch.as_tensor(np.ascontiguousarray(holes, dtype=np.uint8)) if not isinstance(holes, torch.Tensor) else holes
    board = torch.as_tensor(np.ascontiguousarray(board, dtype=np.uint8)) if not isinstance(board, torch.Tensor) else board
    n_players = torch.as_tensor(np.ascontiguousarray(n_players, dtype=np.uint8)) if not isinstance(n_players, torch.Tensor) else n_players
    holes, board, n_players = holes.to(dev).contiguous(), board.to(dev).contiguous(), n_players.to(dev).contiguous()
    N, maxp = holes.shape[0], holes.shape[1]
    L = _lib.ensure_init(dev.index)
    winner = torch.empty(N, dtype=torch.int32, device=dev)
    wtype = torch.empty(N, dtype=torch.uint8, device=dev)
    ranks = torch.zeros((N, maxp), dtype=torch.uint16, device=dev) if return_ranks else None
    with torch.cuda.device(dev):
        _lib.check(L.npk_showdown_batch(holes.data_ptr(), n_players.data_ptr(), board.data_ptr(), N, maxp,
                                        winner.data_ptr(), wtype.data_ptr(), ranks.data_ptr() if return_ranks else None,
                                        flags, torch.cuda.current_stream(dev).cuda_stream))
    return (winner, wtype, ranks) if return_ranks else (winner, wtype)


def get_winner(player_hands, table_cards):
    """Determine the winning hand of multiple players -- drop-in for hand_evaluator.get_winner (:9-17):
    returns (index of the best hand, first index on ties; its hand type name)."""
    holes = np.array([card_ids(h) for h in player_hands], dtype=np.uint8)[None]
    board = np.array(card_ids(table_cards), dtype=np.uint8)[None]
    w, t = showdown(holes, np.array([holes.shape[1]], dtype=np.uint8), board)
    return int(w[0]), HAND_TYPES[int(t[0])]


def eval_best_hand(hands):
    """Evaluate the best hand -- drop-in for hand_evaluator.eval_best_hand (:20-24) for 7-card hands of distinct cards:
    returns (the winning hand, its hand type name)."""
    cards = np.array([card_ids(h) for h in hands], dtype=np.uint8)
    if cards.shape[1] != 7:
        raise ValueError("eval_best_hand on the GPU path takes 7-card hands")
    ids = rank7(cards).cpu().numpy()
    best = int(np.argmax(ids))            # argmax returns the first maximum = stable descending sort's first element
    L = _lib.lib()
    ts = (ctypes.c_uint16 * 10)()
    _lib.check(L.npk_get_tables(None, None, None, None, None, ts, None))
    ty = sum(int(ids[best]) >= ts[i] for i in range(1, 9))
    return hands[best], HAND_TYPES[ty]


def enumerate_equity(hole, board, n_players=None, device=None, validate=None, deal_mode="uniform"):
    """Exact enumeration (no sampling): hole [Q,2], board [Q,5] with 0xFF padding, n_players [Q] (2, or 3 on a complete
    board).  Returns int64 CUDA tensors (win, tie, lose) of hero-strictly-best / tied / beaten counts.
    deal_mode "uniform" counts every deal once; "reference" weights every deal by how often the reference's dealer makes it
    (include/npk.h, npk_enum_dealer_batch), so that (win + tie) / (win + tie + lose) is the value get_equity converges to."""
    from .equity import _DEAL
    torch = _torch()
    dev = _dev(device)
    flags = _want_check(hole, validate)
    hole = torch.as_tensor(np.ascontiguousarray(hole, dtype=np.uint8)) if not isinstance(hole, torch.Tensor) else hole
    board = torch.as_tensor(np.ascontiguousarray(board, dtype=np.uint8)) if not isinstance(board, torch.Tensor) else board
    hole, board = hole.to(dev).contiguous().view(-1, 2), board.to(dev).contiguous().view(-1, 5)
    Q = hole.shape[0]
    if n_players is None:
        n_players = torch.full((Q,), 2, dtype=torch.uint8, device=dev)
    elif not isinstance(n_players, torch.Tensor):
        n_players = torch.as_tensor(np.ascontiguousarray(n_players, dtype=np.uint8))
    n_players = n_players.to(dev).contiguous()
    L = _lib.ensure_init(dev.index)
    win = torch.zeros(Q, dtype=torch.int64, device=dev)
    tie = torch.zeros(Q, dtype=torch.int64, device=dev)
    lose = torch.zeros(Q, dtype=torch.int64, device=dev)
    with torch.cuda.device(dev):
        _lib.check(L.npk_enum_dealer_batch(hole.data_ptr(), board.data_ptr(), n_players.data_ptr(), Q,
                                           _DEAL.get(deal_mode, -1), win.data_ptr(), tie.data_ptr(), lose.data_ptr(), flags,
                                           torch.cuda.current_stream(dev).cuda_stream))
    return win, tie, lose


def exact_equity(player_cards, table_cards, players, deal_mode="reference"):
    """The exact value get_equity(player_cards, table_cards, players, runs) converges to as runs grows: every deal of the
    opponents' hands and the missing table cards enumerated on the GPU, weighted by how often the reference's dealer makes
    it (ties count as wins).  deal_mode="uniform" gives the value under uniform dealing instead.
    Enumerated shapes: two players with 0..5 table cards, three players with five.  Invalid or repeated cards raise
    ValueError, like get_equity; so does any other shape."""
    hole, board = encode_query(player_cards, table_cards)
    players, known = int(players), len(card_ids(table_cards))
    if not (players == 2 or (players == 3 and known == 5)):
        raise ValueError("exact_equity enumerates two players with 0..5 table cards or three players with five table cards, "
                         "not %d players with %d" % (players, known))
    if deal_mode not in ("uniform", "reference"):
        raise ValueError("deal_mode must be 'uniform' or 'reference'")
    w, t, l = enumerate_equity(hole[None], board[None], np.array([players], dtype=np.uint8), deal_mode=deal_mode,
                               validate=True)
    w, t, l = int(w[0]), int(t[0]), int(l[0])
    return (w + t) / (w + t + l)


SHARE_UNIT = 2520   # NPK_SHARE_UNIT: lcm(1..10), a pot split k ways gives each of the k players 2520 / k


def _u8_tensor(x, dev):
    torch = _torch()
    if not isinstance(x, torch.Tensor):
        x = torch.as_tensor(np.ascontiguousarray(x, dtype=np.uint8))
    return x.to(dev).contiguous()


def _dead_masks(dead, n, dev):
    """[N, k] card ids with 0xFF padding -> [N] int64 masks, one bit per id (ids 52..254 map to bits the validation rejects)."""
    torch = _torch()
    ids = _u8_tensor(dead, dev).view(n, -1).to(torch.int64)
    bits = torch.where(ids == 0xFF, torch.zeros_like(ids), torch.bitwise_left_shift(torch.ones_like(ids), ids.clamp(max=63)))
    mask = torch.zeros(n, dtype=torch.int64, device=dev)
    for j in range(bits.shape[1]):
        mask |= bits[:, j]
    return mask


def _check_win_types(win_types):
    if not isinstance(win_types, (bool, np.bool_)):
        raise ValueError("win_types must be True or False, not %r" % (win_types,))
    return bool(win_types)


def showdown_equity_batch(holes, n_players, board, dead=None, deal_mode="uniform", device=None, validate=None,
                          win_types=False):
    """Exact showdown equity of known hands: every completion of each spot's board, scored for every player.
    holes [N,maxp,2] (maxp 1..10), n_players [N], board [N,5] with 0xFF padding, dead [N,k] card ids removed from the deck
    (0xFF padding) or None.  deal_mode "uniform" enumerates every board completion from the unseen cards; "reference" leaves out
    the highest unseen id, which the reference's dealer never deals.  Returns a dict of int64 CUDA tensors: win, tie, share
    [N,maxp] (share in units of 1/2520 pot per completion) and completions [N]; entries of players >= n_players are 0.
    win_types=True adds win_types [N,maxp,9]: the completions in which each player holds the best rank, alone or tied, by the
    hand type of that rank (indexed like HAND_TYPES; the bins of a player sum to its win + tie).  With every hand known,
    {HAND_TYPES[t]: win_types[s,0,t] / completions[s]} is what run_montecarlo(...).winnerCardTypeList converges to."""
    from .equity import _DEAL
    want_types = _check_win_types(win_types)
    torch = _torch()
    dev = _dev(device)
    flags = _want_check(holes, validate)
    holes, board, n_players = _u8_tensor(holes, dev), _u8_tensor(board, dev), _u8_tensor(n_players, dev)
    N = holes.shape[0]
    maxp = holes.shape[1] if holes.dim() == 3 else 0
    if holes.dim() != 3 or holes.shape[2] != 2 or board.shape != (N, 5) or n_players.shape != (N,):
        raise ValueError("expected holes [N,maxp,2], n_players [N] and board [N,5]")
    masks = _dead_masks(dead, N, dev) if dead is not None and N else None
    L = _lib.ensure_init(dev.index)
    out = {k: torch.empty((N, maxp), dtype=torch.int64, device=dev) for k in ("win", "tie", "share")}
    out["completions"] = torch.empty(N, dtype=torch.int64, device=dev)
    if want_types:
        out["win_types"] = torch.empty((N, maxp, 9), dtype=torch.int64, device=dev)
    ws = torch.empty(int(L.npk_showdown_equity_workspace_bytes(N)), dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev):
        _lib.check(L.npk_showdown_equity_win_types_batch(holes.data_ptr(), n_players.data_ptr(), board.data_ptr(),
                                                         masks.data_ptr() if masks is not None else None, N, maxp,
                                                         _DEAL[deal_mode], flags, out["win"].data_ptr(), out["tie"].data_ptr(),
                                                         out["share"].data_ptr(), out["completions"].data_ptr(),
                                                         out["win_types"].data_ptr() if want_types else None, ws.data_ptr(),
                                                         torch.cuda.current_stream(dev).cuda_stream))
    return out


def showdown_equity(hands, table_cards=(), dead_cards=(), deal_mode="uniform", win_types=False):
    """Exact equity of one spot whose hands are all known -- run_montecarlo with every entry of player_card_list known,
    without sampling, for every player.  hands: two card strings per player (1..10 players, e.g. [{'AS','KS'}, {'QH','QD'}]),
    table_cards: 0..5 card strings, dead_cards: cards removed from the deck (the reference's ghost cards).
    Returns dict(equity = split-pot equity per player, win, tie = completions won alone / tied for best, completions).
    win_types=True adds win_types: one list of nine per player, the completions it wins or ties by the hand type of its rank
    (indexed like HAND_TYPES).  Player 0's bins divided by completions are what run_montecarlo(...).winnerCardTypeList
    converges to.  Invalid or repeated cards raise ValueError, like get_equity."""
    want_types = _check_win_types(win_types)
    holes = [card_ids(h) for h in hands]
    board, dead = card_ids(table_cards), card_ids(dead_cards)
    if not 1 <= len(holes) <= 10:
        raise ValueError("1..10 hands")
    if any(len(h) != 2 for h in holes):
        raise ValueError("every hand must hold exactly two cards")
    if len(board) > 5:
        raise ValueError("table_cards holds more than five cards")
    if len(set(sum(holes, []) + board + dead)) != 2 * len(holes) + len(board) + len(dead):
        raise ValueError("duplicate cards in hands / table_cards / dead_cards")
    P = len(holes)
    try:
        out = showdown_equity_batch(np.array([holes], dtype=np.uint8), np.array([P], dtype=np.uint8),
                                    np.array([board + [NO_CARD] * (5 - len(board))], dtype=np.uint8),
                                    np.array([dead or [NO_CARD]], dtype=np.uint8), deal_mode=deal_mode, validate=True,
                                    win_types=want_types)
    except _lib.NpkError as exc:
        raise ValueError(str(exc)) from None
    win, tie, share = (out[k][0].tolist() for k in ("win", "tie", "share"))
    comp = int(out["completions"][0])
    res = {"equity": [x / (SHARE_UNIT * comp) for x in share], "win": win, "tie": tie, "completions": comp}
    if want_types:
        res["win_types"] = out["win_types"][0].tolist()
    return res


def exact_equity_batch(holes, n_known, n_random, board, dead=None, deal_mode="reference", device=None, validate=None,
                       win_types=False):
    """Exact equity against one or two unknown opponents, with known opponent hands and dead cards: every deal of the unknown
    hands and every completion of the board enumerated on the GPU.
    holes [N,maxk,2] (maxk 1..8): the hero, then the known opponents; n_known [N]: hands of `holes` in the spot, hero included;
    n_random [N]: unknown opponents (1 or 2); board [N,5] with 0xFF padding; dead [N,k] card ids removed from the deck (0xFF
    padding) or None.  deal_mode "uniform" counts every deal once; "reference" weights it by how often the reference's dealer
    makes it (include/npk.h, npk_exact_equity_batch).  Returns a dict of int64 CUDA tensors win, tie, lose [N] (hero strictly
    best / tied for best / beaten); (win + tie) / (win + tie + lose) is the value run_montecarlo converges to.
    win_types=True adds win_types [N,9]: the part of win + tie (same weights) in which the hero's rank has each hand type, indexed
    like HAND_TYPES (the nine bins sum to win + tie); {HAND_TYPES[t]: win_types[s,t] / (win + tie + lose)} is what
    run_montecarlo(...).winnerCardTypeList converges to."""
    from .equity import _DEAL
    want_types = _check_win_types(win_types)
    torch = _torch()
    dev = _dev(device)
    flags = _want_check(holes, validate)
    holes, board = _u8_tensor(holes, dev), _u8_tensor(board, dev)
    n_known, n_random = _u8_tensor(n_known, dev), _u8_tensor(n_random, dev)
    N = holes.shape[0]
    maxk = holes.shape[1] if holes.dim() == 3 else 0
    if holes.dim() != 3 or holes.shape[2] != 2 or board.shape != (N, 5) or n_known.shape != (N,) or n_random.shape != (N,):
        raise ValueError("expected holes [N,maxk,2], n_known [N], n_random [N] and board [N,5]")
    masks = _dead_masks(dead, N, dev) if dead is not None and N else None
    L = _lib.ensure_init(dev.index)
    out = {k: torch.empty(N, dtype=torch.int64, device=dev) for k in ("win", "tie", "lose")}
    if want_types:
        out["win_types"] = torch.empty((N, 9), dtype=torch.int64, device=dev)
    ws = torch.empty(int(L.npk_exact_equity_workspace_bytes(N)), dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev):
        _lib.check(L.npk_exact_equity_win_types_batch(holes.data_ptr(), n_known.data_ptr(), n_random.data_ptr(),
                                                      board.data_ptr(), masks.data_ptr() if masks is not None else None, N,
                                                      maxk, _DEAL.get(deal_mode, -1), flags, out["win"].data_ptr(),
                                                      out["tie"].data_ptr(), out["lose"].data_ptr(),
                                                      out["win_types"].data_ptr() if want_types else None, ws.data_ptr(),
                                                      torch.cuda.current_stream(dev).cuda_stream))
    return out


def exact_equity_counts(player_cards, table_cards, players, known_opponents=(), ghost_cards='', deal_mode="reference",
                        win_types=False):
    """The exact value run_montecarlo(player_card_list = [player_cards] + known_opponents, table_cards, players, ghost_cards)
    converges to, for one or two unknown opponents: players - 1 - len(known_opponents) must be 1 or 2.  Argument names and
    checks follow equity_counts_ranges; player_cards and every known opponent are two cards (no ranges).
    Returns dict(equity = (win + tie) / (win + tie + lose), win, tie, lose).  win_types=True adds win_types: nine ints indexed
    like HAND_TYPES, the part of win + tie in which the hero's hand has each type (they sum to win + tie);
    {HAND_TYPES[t]: win_types[t] / (win + tie + lose)} is what run_montecarlo(...).winnerCardTypeList converges to."""
    want_types = _check_win_types(win_types)
    players = int(players)
    if players < 1:
        raise IndexError("list index out of range")
    if players > 10:
        raise ValueError("at most 10 players")
    if deal_mode not in ("uniform", "reference"):
        raise ValueError("deal_mode must be 'uniform' or 'reference'")
    board = card_ids(table_cards)
    if len(board) > 5:
        raise ValueError("table_cards holds more than five cards")
    ghost = card_ids(ghost_cards) if ghost_cards not in ('', None) else []
    if ghost and len(ghost) != 2:
        raise ValueError("ghost_cards must be '' or two cards")
    hole = card_ids(player_cards)
    if len(hole) != 2:
        raise ValueError("player_cards must hold exactly two cards, got %d" % len(hole))
    known = []
    for hand in known_opponents:
        ids = card_ids(hand)
        if len(ids) != 2:
            raise ValueError("a known opponent's hand must hold exactly two cards, got %d" % len(ids))
        known.append(ids)
    if len(set(hole + sum(known, []) + board + ghost)) != 2 + 2 * len(known) + len(board) + len(ghost):
        raise ValueError("duplicate cards in player_cards / known_opponents / table_cards / ghost_cards")
    k = players - 1 - len(known)
    if k == 0:
        raise ValueError("every opponent is known: showdown_equity gives the exact equity of known hands")
    if k not in (1, 2):
        raise ValueError("exact_equity_counts enumerates one or two unknown opponents, not %d" % k)
    holes = np.array([[hole] + known], dtype=np.uint8)
    try:
        out = exact_equity_batch(holes, [1 + len(known)], [k], [board + [NO_CARD] * (5 - len(board))],
                                 np.array([ghost or [NO_CARD]], dtype=np.uint8), deal_mode=deal_mode, validate=True,
                                 win_types=want_types)
    except _lib.NpkError as exc:
        raise ValueError(str(exc)) from None
    win, tie, lose = (int(out[x][0]) for x in ("win", "tie", "lose"))
    res = {"equity": (win + tie) / (win + tie + lose), "win": win, "tie": tie, "lose": lose}
    if want_types:
        res["win_types"] = out["win_types"][0].tolist()
    return res


def host_tables():
    """Host copies of the lookup tables built by libnpk (no GPU needed): dict of numpy arrays."""
    L = _lib.lib()
    n = ctypes.c_int64(0)
    _lib.check(L.npk_get_tables(None, ctypes.byref(n), None, None, None, None, None))
    value = np.zeros(n.value, dtype=np.uint16)
    rowoff = np.zeros(8192, dtype=np.uint16)
    flush = np.zeros(8192, dtype=np.uint16)
    desc = np.zeros(52, dtype=np.uint32)
    ts = np.zeros(10, dtype=np.uint16)
    keys = np.zeros(5034, dtype=np.uint64)
    p = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    _lib.check(L.npk_get_tables(p(value), ctypes.byref(n), p(rowoff), p(flush), p(desc), p(ts), p(keys)))
    return {"value": value, "rowoff": rowoff, "flush": flush, "desc": desc, "type_start": ts, "class_keys": keys}


def host_rank7(cards):
    """Rank ids through the HOST copy of the tables (table self-check for CPU-only tests; not a compute path)."""
    a = np.ascontiguousarray(cards, dtype=np.uint8).reshape(-1, 7)
    out = np.zeros(len(a), dtype=np.uint16)
    L = _lib.lib()
    _lib.check(L.npk_host_rank7(a.ctypes.data_as(ctypes.c_void_p), len(a), out.ctypes.data_as(ctypes.c_void_p)))
    return out
