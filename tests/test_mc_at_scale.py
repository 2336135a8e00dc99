"""Monte-Carlo kernels bit for bit against the sampler specification in the regime they run in production.

The planner (plan_items, csrc/npk_capi.cu) cuts a query into work items of up to 2,048 trials, but only when the batch is
large: Q*T >= 2,048 * 8 * 16 * SMs.  Small test batches get items of one warp iteration (64 trials), which leaves out what a
long item exercises -- the per-lane counters carried across iterations (wins, ties, packed win types, passes), the trial
window advancing by 64 per iteration, items that start at an odd trial.  These tests size their batches from the device's
SM count so that items are 2,048 trials long, put the trial numbers past 2^33 and let the query counter wrap past 2^32, and
compare with tests/sampler_vec.py, the vectorised restatement of tests/sampler_model.py (pinned to it by the CPU tests
here).  Known-answer spots (a royal flush for the hero, four aces on the board) fill the counter fields to their limits at sizes
no specification needs to score.
"""
import ctypes

import numpy as np
import pytest

import oracle
import sampler_model
import sampler_vec

NO = 0xFF
MASK = 0xFFFFFFFF
ITEM_CAP = 2048                       # plan_items' largest work item, in trials
ODD_FAR = (1 << 33) + 1               # an odd trial number past 2^33: the pair's high counter word is 2


# ---- CPU: the vectorised specification equals the scalar one ---------------------------------------------------------
OFFSETS = (0, 1, (1 << 32) - 1, (1 << 33) + 3)
QUERIES = (0, (1 << 32) - 1)


@pytest.mark.parametrize("mode", ["uniform", "reference"])
def test_vectorised_specification_equals_the_scalar_one(mode):
    """sampler_vec.run == sampler_model.run_model (wins, ties, passes, win types) for every player count 1..10 and known
    board 0..5; each shape at two of the eight (trial offset, query counter) pairs, so every pair meets several shapes."""
    rng = np.random.default_rng(17)
    combos = [(o, q) for o in OFFSETS for q in QUERIES]
    for i, (players, known) in enumerate((p, k) for p in range(1, 11) for k in range(6)):
        c = rng.permutation(52)[:2 + known].tolist()
        for off, query in (combos[i % 8], combos[(i + 3) % 8]):
            seed = int(rng.integers(0, 2**63)) * 2 + 1
            want = sampler_model.run_model(oracle, mode, seed, query, c[:2], c[2:], players, 120, trial_offset=off)
            got = sampler_vec.run(mode, seed, query, c[:2], c[2:], players, 120, trial_offset=off)
            assert got == want, (mode, players, known, off, query)


def test_hand_type_thresholds_equal_the_oracles_hand_types(golden_tables):
    """sampler_vec.TYPE_START against oracle.type7 for every rank id: one hand per rank histogram without a flush and
    one per flush mask (the evaluator's whole key space, as in test_gpu_parity.test_rank7_golden_and_oracle)."""
    hands = []
    for h in golden_tables["hist"]:
        cards, k = [], 0
        for r in range(13):
            for _ in range(h[r]):
                cards.append(4 * r + (k & 3))
                k += 1
        hands.append(cards)
    fl = golden_tables["flush"]
    for m in (m for m in range(8192) if fl[m] != 0xFFFF):
        cards = [4 * r for r in range(13) if m >> r & 1]
        pad = 0
        while len(cards) < 7:
            cards.append(4 * pad + 1)
            pad += 1
        hands.append(cards)
    hands = np.array(hands, dtype=np.uint8)
    ranks = oracle.rank7_batch(hands)
    assert (np.unique(ranks) == np.arange(5034)).all()                  # every rank id occurs
    types = np.array([oracle.type7(h.tolist()) for h in hands])
    assert (sampler_vec.hand_type(ranks) == types).all()


# ---- GPU helpers -------------------------------------------------------------------------------------------------------
def _lib():
    from neuron_poker_b200 import _lib as lib
    return lib


@pytest.fixture(scope="module")
def dev(cuda_device):
    import torch
    L = _lib().ensure_init(0)
    return {"torch": torch, "L": L, "sms": int(L.npk_sm_count())}


def cap_queries(sms, trials, factor=1):
    """Queries of `trials` trials that make plan_items choose its 2,048-trial cap (`factor` times over)."""
    return -(-factor * ITEM_CAP * 8 * 16 * sms // trials)


def pad(b):
    return list(b) + [NO] * (5 - len(b))


def random_queries(rng, Q, known):
    cards = rng.random((Q, 52)).argsort(1)[:, :2 + known].astype(np.uint8)
    board = np.full((Q, 5), NO, dtype=np.uint8)
    board[:, :known] = cards[:, 2:]
    return cards[:, :2].copy(), board


def launch(dev, hole, board, npl, trials, seed, mode, trial_offset=0, query_offset=0, shape=None, validate=False,
           shapes=None):
    """One npk_equity_batch (or, with `shapes`, npk_equity_batch_async) call with win types and, for the reference dealer,
    passes.  Returns the counters as numpy arrays and the work counter the kernel left in the workspace: every warp pulls
    items until one is past the end, so it holds items + warps of the grid."""
    torch, L = dev["torch"], dev["L"]
    lib = _lib()
    Q = len(hole)
    h, b, n = (torch.as_tensor(np.ascontiguousarray(x, dtype=np.uint8)).cuda() for x in (hole, board, npl))
    ws = torch.zeros(int(L.npk_equity_workspace_bytes(Q)), dtype=torch.uint8, device="cuda")
    wins, ties = (torch.zeros(Q, dtype=torch.int64, device="cuda") for _ in range(2))
    types = torch.zeros((Q, 9), dtype=torch.int64, device="cuda")
    passes = torch.zeros(Q, dtype=torch.int64, device="cuda") if mode == "reference" else None
    deal = lib.NPK_DEAL_REFERENCE if mode == "reference" else lib.NPK_DEAL_UNIFORM
    stream = torch.cuda.current_stream().cuda_stream
    common = (ctypes.c_uint64(seed), trial_offset, query_offset, deal)
    outs = (wins.data_ptr(), ties.data_ptr(), types.data_ptr(), passes.data_ptr() if passes is not None else None,
            ws.data_ptr(), stream)
    if shapes is not None:
        lib.check(L.npk_equity_batch_async(h.data_ptr(), b.data_ptr(), n.data_ptr(), Q, trials, ctypes.c_uint64(shapes),
                                           *common, *outs))
    else:
        up, uk = shape if shape else (-1, -1)
        lib.check(L.npk_equity_batch(h.data_ptr(), b.data_ptr(), n.data_ptr(), Q, trials, up, uk, *common,
                                     lib.NPK_FLAG_VALIDATE if validate else 0, *outs))
    torch.cuda.synchronize()
    counters = ws[:16].cpu().numpy().view(np.uint64)
    out = {"wins": wins.cpu().numpy(), "ties": ties.cpu().numpy(), "win_types": types.cpu().numpy()}
    if passes is not None:
        out["passes"] = passes.cpu().numpy()
    return out, int(counters[1] if (shape and validate) else counters[0])


def assert_items(counter, Q, per_query, dev):
    """The work counter of a per-shape launch: Q * per_query items plus one last pull per warp (at most 16 warps per SM)."""
    assert Q * per_query <= counter <= Q * per_query + 16 * dev["sms"], ("work items", counter, Q, per_query)


def check_query(out, q, mode, seed, hole, board, players, trials, trial_offset, query_offset, what=""):
    b = [int(c) for c in board if c != NO]
    m = sampler_vec.run(mode, seed, (q + query_offset) & MASK, hole, b, players, trials, trial_offset)
    got = {"wins": int(out["wins"][q]), "ties": int(out["ties"][q]), "win_types": [int(x) for x in out["win_types"][q]],
           "passes": int(out["passes"][q]) if "passes" in out else 0}
    assert got == m, (what, mode, q, players, len(b), trials, trial_offset)


SHAPES = [(p, k) for p in range(1, 11) for k in range(6)]
T_LONG = 2 * ITEM_CAP + 3              # two full items and a ragged one of three trials


# ---- GPU: every per-shape instance at production item size -------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["uniform", "reference"])
def test_every_per_shape_instance_at_production_item_size(dev, mode):
    """equity_uniform_kernel / equity_refdeal_kernel<NOPP, NB> for all 60 shapes (players 1..10 x known board 0..5): one
    uniform_shape batch each, sized for 2,048-trial items (asserted from the work counter), T = 2*2,048 + 3 trials from an
    odd trial number past 2^33, the query counter wrapping past 2^32 inside the batch.  First and last query bit for bit
    against the specification; odd shapes go through the validated launch."""
    rng = np.random.default_rng(100)
    Q = cap_queries(dev["sms"], T_LONG)
    for i, (players, known) in enumerate(SHAPES):
        hole, board = random_queries(rng, Q, known)
        npl = np.full(Q, players, dtype=np.uint8)
        seed, toff, qoff = 0x9E3779B97F4A7C15 + i, ODD_FAR + 2 * i, (1 << 32) - Q // 2 - i
        out, counter = launch(dev, hole, board, npl, T_LONG, seed, mode, toff, qoff, shape=(players, known),
                              validate=i % 2 == 1)
        assert_items(counter, Q, 3, dev)                  # items of 2,048, 2,048 and 3 trials
        for q in (0, Q - 1):
            check_query(out, q, mode, seed, hole[q].tolist(), board[q], players, T_LONG, toff, qoff, "per-shape")


# ---- GPU: the persistent mixed kernel at production item size ----------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["uniform", "reference"])
def test_mixed_kernel_at_production_item_size(dev, mode):
    """One batch holding all 60 shapes, sized for 2,048-trial items, through npk_equity_batch unvalidated and validated and
    through npk_equity_batch_async with a shape mask that leaves out two shapes.  One query per shape bit for bit against
    the specification, the three calls equal query for query, the masked-out shapes untouched."""
    from neuron_poker_b200.equity import shape_mask
    rng = np.random.default_rng(200)
    per = -(-cap_queries(dev["sms"], T_LONG) // len(SHAPES))
    hole, board, npl = [], [], []
    for players, known in SHAPES:
        h, b = random_queries(rng, per, known)
        hole.append(h); board.append(b); npl.append(np.full(per, players, dtype=np.uint8))
    perm = rng.permutation(per * len(SHAPES))
    hole, board, npl = (np.concatenate(x)[perm] for x in (hole, board, npl))
    Q = len(hole)
    seed, toff, qoff = 0xC0FFEE1234, ODD_FAR + 6, (1 << 32) - Q // 3
    a, counter = launch(dev, hole, board, npl, T_LONG, seed, mode, toff, qoff)
    assert counter == 3 * Q + 15 * dev["sms"], ("work items", counter, Q)    # 3 items per query + one last pull per warp
    b, _ = launch(dev, hole, board, npl, T_LONG, seed, mode, toff, qoff, validate=True)
    left_out = [(9, 2), (2, 1)]
    mask = 0
    for players, known in SHAPES:
        if (players, known) not in left_out:
            mask |= shape_mask([players], [known])
    c, _ = launch(dev, hole, board, npl, T_LONG, seed, mode, toff, qoff, shapes=mask)
    known_of = (board != NO).sum(1)
    out_mask = np.zeros(Q, dtype=bool)
    for players, known in left_out:
        out_mask |= (npl == players) & (known_of == known)
    for k in a:
        assert (a[k] == b[k]).all(), k
        assert (c[k][~out_mask] == a[k][~out_mask]).all() and (c[k][out_mask] == 0).all(), k
    for players, known in SHAPES:
        q = int(np.flatnonzero((npl == players) & (known_of == known))[-1])
        check_query(a, q, mode, seed, hole[q].tolist(), board[q], players, T_LONG, toff, qoff, "mixed")


# ---- GPU: small and ragged items -----------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("trials", [1, 63, 64, 65, 2047, 2048, 2049])
def test_small_and_ragged_items(dev, trials):
    """Trial counts around one warp iteration and around the item cap, from odd trial numbers: a lone query (items of 64)
    and the same query first in a batch large enough for the cap (one item per query up to 2,048 trials), per-shape and
    mixed kernels, both dealers."""
    rng = np.random.default_rng(trials)
    Q = cap_queries(dev["sms"], 2049)
    for mode in ("uniform", "reference"):
        for players, known in ((6, 3), (10, 0), (2, 5), (1, 4)):
            hole, board = random_queries(rng, Q, known)
            npl = np.full(Q, players, dtype=np.uint8)
            seed, toff = int(rng.integers(0, 2**62)), 2 * int(rng.integers(0, 2**40)) + 1
            big, _ = launch(dev, hole, board, npl, trials, seed, mode, toff, 5, shape=(players, known))
            one, _ = launch(dev, hole[:1], board[:1], npl[:1], trials, seed, mode, toff, 5, shape=(players, known))
            mixed, _ = launch(dev, hole[:1], board[:1], npl[:1], trials, seed, mode, toff, 5)
            check_query(big, 0, mode, seed, hole[0].tolist(), board[0], players, trials, toff, 5, "batch")
            check_query(big, Q - 1, mode, seed, hole[Q - 1].tolist(), board[Q - 1], players, trials, toff, 5, "batch")
            for k in big:
                assert (one[k][0] == big[k][0]).all() and (mixed[k][0] == big[k][0]).all(), (mode, k, players, known)


# ---- GPU: the one-query paths plan their own items ----------------------------------------------------------------------
def one_query(card_str, mode, seed, trials, **kw):
    import neuron_poker_b200 as npk
    h, b, p = card_str
    return npk.equity_counts(h, b, p, trials, deal_mode=mode, seed_value=seed, **kw)


def spec_one(card_str, mode, seed, trials):
    import neuron_poker_b200 as npk
    h, b, p = card_str
    return sampler_vec.run(mode, seed, 0, [npk.card_id(c) for c in h], [npk.card_id(c) for c in b], p, trials)


RIVER = (["AS", "KD"], ["KH", "JS", "2C", "QS", "7D"], 2)
FLOP3 = (["TC", "TH"], ["4D", "QD", "KC"], 3)


@pytest.mark.gpu
def test_one_shot_kernel_against_the_specification(dev):
    """equity_counts without win types (equity_oneshot_kernel, serve_request's own planner: trials / (8 * warps of the
    grid), rounded up to 64): trial counts on both sides of the switch from 4-warp to 15-warp CTAs and of the step from
    64- to 128-trial items."""
    sms = dev["sms"]
    warp_switch = 64 * 4 * sms                      # more items than 4 * SMs: 15 warps per CTA
    two_iter = 65 * 8 * 15 * min(sms, 255)          # from here on items of 128 trials
    for mode in ("uniform", "reference"):
        for trials in (warp_switch, warp_switch + 1, two_iter - 1, two_iter + 77):
            got = one_query(RIVER, mode, 4242, trials)
            m = spec_one(RIVER, mode, 4242, trials)
            assert (got["wins"], got["ties"]) == (m["wins"], m["ties"]), (mode, trials)


@pytest.mark.gpu
def test_one_query_per_shape_kernel_against_the_specification(dev):
    """equity_counts with win types / passes: the shape's own kernel planned for one query (items of 64 trials up to
    64 * 128 * SMs trials, 128 beyond) and finish_single_call's hand-over, against the specification."""
    two_iter = 65 * 128 * dev["sms"]
    for mode in ("uniform", "reference"):
        for trials in (5001, two_iter - 1, two_iter + 129):
            got = one_query(RIVER, mode, 77, trials, win_types=True, passes=mode == "reference")
            m = spec_one(RIVER, mode, 77, trials)
            assert (got["wins"], got["ties"], got["win_types"]) == (m["wins"], m["ties"], m["win_types"]), (mode, trials)
            if mode == "reference":
                assert got["passes"] == m["passes"], trials


@pytest.mark.gpu
def test_resident_server_on_one_sm_against_the_specification(dev):
    """The resident server started on one SM (15 warps): its planner reaches 128-trial items at 7,800 trials and the
    2,048-trial cap at 238,200; trial counts on both sides of both steps and one past the cap, both dealers."""
    import neuron_poker_b200 as npk
    try:
        npk.resident(True, sms=1, idle_us=100000)
        for mode in ("uniform", "reference"):
            for trials in (7799, 7800, 238199, 238200, 300001):
                got = one_query(FLOP3, mode, 31337, trials)
                m = spec_one(FLOP3, mode, 31337, trials)
                assert (got["wins"], got["ties"]) == (m["wins"], m["ties"]), (mode, trials)
    finally:
        npk.resident(False)


# ---- GPU: known answers that fill the counter fields --------------------------------------------------------------------
# (hole, board, hero wins every trial, hand type of every trial).  A royal flush on the board would not do for the ties: the
# reference's evaluator ranks a straight flush with a sixth card of its suit above one without (oracle.calc_score), so an
# opponent holding a spade beats it.  Four aces and a king on the board cannot be improved by any hole cards.
HERO_ROYAL = (["AS", "KS"], ["QS", "JS", "TS"], True, 8)
BOARD_QUADS = (["2C", "3D"], ["AS", "AH", "AD", "AC", "KS"], False, 7)


def saturation_spots():
    import neuron_poker_b200 as npk
    for h, b, hero_wins, ty in (HERO_ROYAL, BOARD_QUADS):
        for players in (2, 10):
            yield [npk.card_id(c) for c in h], [npk.card_id(c) for c in b], players, (hero_wins, ty)


def check_saturated(wins, ties, types, trials, answer, what):
    hero_wins, ty = answer
    assert (int(wins), int(ties)) == ((trials, 0) if hero_wins else (0, trials)), what
    assert [int(x) for x in types] == [trials if i == ty else 0 for i in range(9)], what


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["uniform", "reference"])
def test_known_answers_fill_the_per_lane_win_type_fields(dev, mode):
    """64 trials per lane of one hand type: the 7-bit win-type field of that type (straight flush, quads) is full in every
    lane.  Per-shape and mixed batches sized at four times the planner's cap threshold, so a larger cap would be used and
    overflow."""
    T = (1 << 20) + 1
    Q = cap_queries(dev["sms"], T, factor=4)
    spots = list(saturation_spots())
    for h, b, players, answer in spots:
        hole, board = np.array([h] * Q, dtype=np.uint8), np.array([pad(b)] * Q, dtype=np.uint8)
        out, counter = launch(dev, hole, board, np.full(Q, players, dtype=np.uint8), T, 3, mode, ODD_FAR, 0,
                              shape=(players, len(b)))
        for q in range(Q):
            check_saturated(out["wins"][q], out["ties"][q], out["win_types"][q], T, answer, ("per-shape", players, q))
        if mode == "reference":
            assert (out["passes"] >= (players - 1) * T).all()
        assert_items(counter, Q, -(-T // ITEM_CAP), dev)
    per = -(-Q // len(spots))
    hole = np.array([h for h, b, p, w in spots for _ in range(per)], dtype=np.uint8)
    board = np.array([pad(b) for h, b, p, w in spots for _ in range(per)], dtype=np.uint8)
    npl = np.array([p for h, b, p, w in spots for _ in range(per)], dtype=np.uint8)
    out, _ = launch(dev, hole, board, npl, T, 4, mode, ODD_FAR, 0)
    for i, (h, b, players, answer) in enumerate(spots):
        for q in range(i * per, (i + 1) * per):
            check_saturated(out["wins"][q], out["ties"][q], out["win_types"][q], T, answer, ("mixed", players, q))


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["uniform", "reference"])
def test_known_answers_at_the_limits_of_the_counters(dev, mode):
    """Counts at the edges of the packed hand-overs: 2^28 - 1 trials through the one-shot kernel and the resident server
    (28-bit fields), 2^28 through the launched per-shape path (the first count the packed hand-over cannot carry), and
    2^32 + 5 through a batch and a one-query call (counts past 32 bits)."""
    import neuron_poker_b200 as npk
    spots = list(saturation_spots())
    for h, b, players, answer in spots:
        hs, bs = [npk.card_str(c) for c in h], [npk.card_str(c) for c in b]
        for trials in ((1 << 28) - 1, (1 << 28), (1 << 32) + 5):
            r = npk.equity_counts(hs, bs, players, trials, deal_mode=mode, seed_value=trials, win_types=True,
                                  passes=mode == "reference")
            check_saturated(r["wins"], r["ties"], r["win_types"], trials, answer, ("one query", players, trials))
            if mode == "reference":
                assert r["passes"] >= (players - 1) * trials
        r = npk.equity_counts(hs, bs, players, (1 << 28) - 1, deal_mode=mode, seed_value=1)
        assert (r["wins"], r["ties"]) == (((1 << 28) - 1, 0) if answer[0] else (0, (1 << 28) - 1)), ("one-shot", players)
    try:
        npk.resident(True, idle_us=100000)
        for h, b, players, answer in spots:
            r = npk.equity_counts([npk.card_str(c) for c in h], [npk.card_str(c) for c in b], players, (1 << 28) - 1,
                                  deal_mode=mode, seed_value=2)
            assert (r["wins"], r["ties"]) == (((1 << 28) - 1, 0) if answer[0] else (0, (1 << 28) - 1)), ("resident", players)
    finally:
        npk.resident(False)
    T = (1 << 32) + 5
    hole = np.array([s[0] for s in spots], dtype=np.uint8)
    board = np.array([pad(s[1]) for s in spots], dtype=np.uint8)
    npl = np.array([s[2] for s in spots], dtype=np.uint8)
    out, _ = launch(dev, hole, board, npl, T, 6, mode, ODD_FAR, 0)
    for q, (h, b, players, answer) in enumerate(spots):
        check_saturated(out["wins"][q], out["ties"][q], out["win_types"][q], T, answer, ("batch", players))


# ---- GPU: the range kernels at production item size -------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["uniform", "reference"])
def test_range_kernels_at_production_item_size(dev, mode):
    """The generic range kernel (asked for passes) and the pair-list sampler, with and without a known opponent hand, in
    batches sized for 2,048-trial items (64 iterations of 32 trials), T = 2*2,048 + 3 from an odd trial number past 2^33,
    the query counter wrapping past 2^32: the last query against the scalar specification, the first one too for the
    generic kernel."""
    import neuron_poker_b200 as npk
    from neuron_poker_b200 import ranges
    rng = np.random.default_rng(300)
    Q, players = cap_queries(dev["sms"], T_LONG), 4
    mask = ranges.opponent_mask(0.3)
    for passes in (True, False):
        for n_known in (0, 1):
            cards = rng.random((Q, 52)).argsort(1)[:, :7].astype(np.uint8)
            hole, board = cards[:, :2].copy(), np.full((Q, 5), NO, dtype=np.uint8)
            board[:, :3] = cards[:, 2:5]
            known = cards[:, 5:7].reshape(Q, 1, 2).copy()
            seed, toff, qoff = int(rng.integers(0, 2**62)), ODD_FAR + 2 * int(rng.integers(0, 2**20)), (1 << 32) - Q // 2
            out = npk.get_equity_ranges_batch(hole, board, np.full(Q, players, dtype=np.uint8), T_LONG, opponent_range=0.3,
                                              seed_value=seed, deal_mode=mode, trial_offset=toff, query_offset=qoff,
                                              win_types=True, passes=passes, known_opponents=known if n_known else None)
            out = {k: v.cpu().numpy() for k, v in out.items() if k != "trials"}
            for q in ((0, Q - 1) if passes else (Q - 1,)):
                m = sampler_model.run_model(oracle, mode, seed, (q + qoff) & MASK, hole[q].tolist(), board[q, :3].tolist(),
                                            players, T_LONG, trial_offset=toff, opp_mask=mask, fast=not passes,
                                            known=[known[q, 0].tolist()] if n_known else ())
                got = (int(out["wins"][q]), int(out["ties"][q]), [int(x) for x in out["win_types"][q]])
                assert got == (m["wins"], m["ties"], m["win_types"]), (mode, passes, n_known, q)
                if passes:
                    assert int(out["passes"][q]) == m["passes"], (mode, n_known, q)
