"""The plain Monte-Carlo samplers of tests/sampler_model.py restated in NumPy, vectorised over trials (test infrastructure).

sampler_model deals one trial at a time in Python, about 10,000 trials per second.  Checking the kernels bit for bit at the
sizes they run in production -- work items of 2,048 trials, trial numbers past 2^33, query counters that wrap -- needs
hundreds of thousands of trials per check, so this module deals a whole block of trials at once with the same rules:

  uniform   (sampler_model.deal_uniform): partial Fisher-Yates over the unseen cards in ascending card id, two trials per
            Philox pair.
  reference (sampler_model.deal_reference): pops from the ordered list of unseen cards at the rejection-free indices of the
            reference's dealer, and `passes` from the law of its attempt counter.

Hands are scored with the oracle's rank ids (oracle.rank7_batch); the hand type of a rank id comes from TYPE_START, which
tests/test_mc_at_scale.py pins to oracle.type7 over every rank id.  tests/test_mc_at_scale.py also pins this module to
sampler_model.run_model bit for bit.
"""
import numpy as np

import oracle

M0, M1, W0, W1 = 0xD2511F53, 0xCD9E8D57, 0x9E3779B9, 0xBB67AE85
MASK = 0xFFFFFFFF
REFERENCE_BLOCK0 = 0x80000000
PASSES_BLOCK0 = 0x40000000
MAX_ATTEMPTS = 1 << 16
TYPE_START = (0, 407, 1877, 2640, 3215, 3225, 4502, 4658, 4736)   # first rank id of each hand type 0..8
BLOCK = 1 << 16                                                  # trials dealt at once (bounds the memory)

_U32 = np.uint64(MASK)
_S32 = np.uint64(32)


def philox4x32_10(c0, c1, c2, c3, k0, k1):
    """Philox4x32-10 of counters given as arrays (uint64 holding 32-bit values); returns the four output words."""
    c0, c1, c2, c3 = np.broadcast_arrays(*(np.asarray(c, dtype=np.uint64) & _U32 for c in (c0, c1, c2, c3)))
    k0, k1 = np.uint64(k0 & MASK), np.uint64(k1 & MASK)
    for _ in range(10):
        p0, p1 = c0 * np.uint64(M0), c2 * np.uint64(M1)
        c0, c1, c2, c3 = (p1 >> _S32) ^ c1 ^ k0, p1 & _U32, (p0 >> _S32) ^ c3 ^ k1, p0 & _U32
        k0, k1 = (k0 + np.uint64(W0)) & _U32, (k1 + np.uint64(W1)) & _U32
    return [c0, c1, c2, c3]


def _trial_words(seed, query, trials, block0, nblk, per_trial):
    """[T, per_trial] words of trials `trials` (uint64 array): pair P = t >> 1 draws blocks (P_lo, P_hi, query, block0 + b)
    for b < nblk, trial 2P reads words [0, per_trial), trial 2P+1 words [per_trial, 2 * per_trial)."""
    pair = trials >> np.uint64(1)
    half = (trials & np.uint64(1)).astype(np.int64)
    if per_trial == 0:                                           # one player, full board: nothing is dealt
        return np.zeros((len(trials), 0), dtype=np.uint64)
    w = []
    for b in range(nblk):
        w += philox4x32_10(pair & _U32, pair >> _S32, query & MASK, (block0 + b) & MASK, seed & MASK, seed >> 32)
    w = np.stack(w, 1)
    cols = half[:, None] * per_trial + np.arange(per_trial)[None, :]
    return np.take_along_axis(w, cols, 1)


def deal_uniform(seed, query, trials, hole, board, players):
    """sampler_model.deal_uniform for every trial number in `trials`: (opponent cards [T, 2 * opponents], board [T, 5])."""
    known = set(hole) | set(board)
    deck0 = np.array([c for c in range(52) if c not in known], dtype=np.uint8)
    n, nopp = len(deck0), players - 1
    d = 2 * nopp + 5 - len(board)
    nw = (d + 1) // 2
    T = len(trials)
    w = _trial_words(seed, query, trials, 0, (2 * nw + 3) // 4, nw)
    rows = np.arange(T)
    deck = np.tile(deck0, (T, 1))
    out = np.empty((T, d), dtype=np.uint8)
    rem = np.zeros(T, dtype=np.uint64)
    for k in range(d):
        x = rem if k & 1 else w[:, k >> 1]
        prod = x * np.uint64(n - k)
        idx = (prod >> _S32).astype(np.int64)
        rem = prod & _U32
        out[:, k] = deck[rows, idx]
        deck[rows, idx] = deck[:, n - 1 - k]
    full = np.concatenate([np.tile(np.array(board, dtype=np.uint8), (T, 1)), out[:, 2 * nopp:]], 1)
    return out[:, :2 * nopp], full


def _passes(seed, query, trials, n0, nopp):
    """The reference's attempt counter per trial: per opponent 1 + the number of times x < floor((2^32-1)/n) holds along
    x -> x*n mod 2^32, x the trial's word of that opponent in the blocks at PASSES_BLOCK0 (sampler_model.deal_reference)."""
    total = np.zeros(len(trials), dtype=np.int64)
    if nopp == 0:
        return total
    w = _trial_words(seed, query, trials, PASSES_BLOCK0, (2 * nopp + 3) // 4, nopp)
    for o in range(nopp):
        n = n0 - 2 * o
        x, tries = w[:, o].copy(), np.ones(len(trials), dtype=np.int64)
        live = (x < np.uint64(MASK // n)) & (tries < MAX_ATTEMPTS)
        while live.any():
            tries[live] += 1
            x[live] = (x[live] * np.uint64(n)) & _U32
            live &= (x < np.uint64(MASK // n)) & (tries < MAX_ATTEMPTS)
        total += tries
    return total


def deal_reference(seed, query, trials, hole, board, players):
    """sampler_model.deal_reference for every trial number in `trials`: (opponent cards [T, 2 * opponents], board [T, 5],
    passes [T]).  The pops are applied to the ordered list literally: pop i takes the i-th card still in it."""
    known = set(hole) | set(board)
    deck0 = np.array([c for c in range(52) if c not in known], dtype=np.uint8)
    n0, nopp, nb = len(deck0), players - 1, 5 - len(board)
    nwr = nopp + (nb + 1) // 2
    T = len(trials)
    w = _trial_words(seed, query, trials, REFERENCE_BLOCK0, (2 * nwr + 3) // 4, nwr)
    raw = []
    for o in range(nopp):
        m = np.uint64(n0 - 2 * o - 1)
        prod = w[:, o] * m
        a, b = prod >> _S32, ((prod & _U32) * m) >> _S32
        raw += [a + (a >= b), b]
    rem = np.zeros(T, dtype=np.uint64)
    for c in range(nb):
        m = np.uint64(n0 - 2 * nopp - c - 1)
        x = rem if c & 1 else w[:, nopp + (c >> 1)]
        prod = x * m
        raw.append(prod >> _S32)
        rem = prod & _U32
    live = np.ones((T, n0), dtype=bool)
    rows = np.arange(T)
    cards = np.empty((T, len(raw)), dtype=np.uint8)
    for k, i in enumerate(raw):
        slot = np.argmax(np.cumsum(live, 1) > i.astype(np.int64)[:, None], 1)       # the (i+1)-th card still in the list
        cards[:, k] = deck0[slot]
        live[rows, slot] = False
    full = np.concatenate([np.tile(np.array(board, dtype=np.uint8), (T, 1)), cards[:, 2 * nopp:]], 1)
    return cards[:, :2 * nopp], full, _passes(seed, query, trials, n0, nopp)


def hand_type(rank_ids):
    """Hand type 0..8 of rank ids (TYPE_START)."""
    return np.searchsorted(np.array(TYPE_START), np.asarray(rank_ids), side="right") - 1


def run(mode, seed, query, hole, board, players, trials, trial_offset=0):
    """dict(wins, ties, passes, win_types[9]) like sampler_model.run_model for the plain dealers.  `query` is the number in
    the Philox counter (the query's index plus the call's query_offset, modulo 2^32)."""
    hole, board = [int(c) for c in hole], [int(c) for c in board]
    wins = ties = passes = 0
    types = np.zeros(9, dtype=np.int64)
    nopp = players - 1
    for start in range(trial_offset, trial_offset + trials, BLOCK):
        t = np.arange(start, min(start + BLOCK, trial_offset + trials), dtype=np.uint64)
        if mode == "uniform":
            opp, full = deal_uniform(seed, query, t, hole, board, players)
        else:
            opp, full, p = deal_reference(seed, query, t, hole, board, players)
            passes += int(p.sum())
        hv = oracle.rank7_batch(np.concatenate([np.tile(np.array(hole, dtype=np.uint8), (len(t), 1)), full], 1)).astype(np.int32)
        best = np.full(len(t), -1, dtype=np.int32)
        for o in range(nopp):
            best = np.maximum(best, oracle.rank7_batch(np.concatenate([opp[:, 2 * o:2 * o + 2], full], 1)).astype(np.int32))
        wins += int((hv > best).sum())
        ties += int((hv == best).sum())
        types += np.bincount(hand_type(hv[hv >= best]), minlength=9)
    return {"wins": wins, "ties": ties, "passes": passes, "win_types": [int(x) for x in types]}
