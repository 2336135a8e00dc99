"""Hand evaluation through the GPU rank tables: batched rank ids, showdown winners and exact enumeration.

Mirrors tools/hand_evaluator.py of the reference: `get_winner` (:9-17) and `eval_best_hand` (:20-24) keep their
signatures; the ordering is the reference's `_calc_score` ordering (:27-119) expressed as a rank id in [0, 5034).
"""
import ctypes

import numpy as np

from . import _lib
from .cards import HAND_TYPES, NO_CARD, card_ids

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


def enumerate_equity(hole, board, n_players=None, device=None, validate=None):
    """Exact enumeration (no sampling): hole [Q,2], board [Q,5] with 0xFF padding, n_players [Q] (2, or 3 on a complete
    board).  Returns int64 CUDA tensors (win, tie, lose) of hero-strictly-best / tied / beaten counts."""
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
        _lib.check(L.npk_enum_batch(hole.data_ptr(), board.data_ptr(), n_players.data_ptr(), Q, win.data_ptr(),
                                    tie.data_ptr(), lose.data_ptr(), flags, torch.cuda.current_stream(dev).cuda_stream))
    return win, tie, lose


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


def showdown_equity_batch(holes, n_players, board, dead=None, deal_mode="uniform", device=None, validate=None):
    """Exact showdown equity of known hands: every completion of each spot's board, scored for every player.
    holes [N,maxp,2] (maxp 1..10), n_players [N], board [N,5] with 0xFF padding, dead [N,k] card ids removed from the deck
    (0xFF padding) or None.  deal_mode "uniform" enumerates every board completion from the unseen cards; "reference" leaves out
    the highest unseen id, which the reference's dealer never deals.  Returns a dict of int64 CUDA tensors: win, tie, share
    [N,maxp] (share in units of 1/2520 pot per completion) and completions [N]; entries of players >= n_players are 0."""
    from .equity import _DEAL
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
    ws = torch.empty(int(L.npk_showdown_equity_workspace_bytes(N)), dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev):
        _lib.check(L.npk_showdown_equity_batch(holes.data_ptr(), n_players.data_ptr(), board.data_ptr(),
                                               masks.data_ptr() if masks is not None else None, N, maxp, _DEAL[deal_mode],
                                               flags, out["win"].data_ptr(), out["tie"].data_ptr(), out["share"].data_ptr(),
                                               out["completions"].data_ptr(), ws.data_ptr(),
                                               torch.cuda.current_stream(dev).cuda_stream))
    return out


def showdown_equity(hands, table_cards=(), dead_cards=(), deal_mode="uniform"):
    """Exact equity of one spot whose hands are all known -- run_montecarlo with every entry of player_card_list known,
    without sampling, for every player.  hands: two card strings per player (1..10 players, e.g. [{'AS','KS'}, {'QH','QD'}]),
    table_cards: 0..5 card strings, dead_cards: cards removed from the deck (the reference's ghost cards).
    Returns dict(equity = split-pot equity per player, win, tie = completions won alone / tied for best, completions).
    Invalid or repeated cards raise ValueError, like get_equity."""
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
                                    np.array([dead or [NO_CARD]], dtype=np.uint8), deal_mode=deal_mode, validate=True)
    except _lib.NpkError as exc:
        raise ValueError(str(exc)) from None
    win, tie, share = (out[k][0].tolist() for k in ("win", "tie", "share"))
    comp = int(out["completions"][0])
    return {"equity": [x / (SHARE_UNIT * comp) for x in share], "win": win, "tie": tie, "completions": comp}


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
