"""Vectorised HoldemTable: N independent tables advanced in lock step on the GPU (include/npk_holdem.h).

Mirror of the reference's gym_env/env.py::HoldemTable for the part a self-play loop needs -- the betting state machine
(gym_env/cycle.py), card dealing (env.py:667-688), showdown (env.py:573-605), legal moves (:629-658), rewards (:280-306)
-- with the same attribute names, as tensors with a leading table dimension:

    tables = HoldemTables(65536, n_players=6, initial_stacks=100, small_blind=1, big_blind=2)
    tables.step(actions)                    # env.step(action) for every table (int8 CUDA tensor / array of Action values)
    tables.selfplay_step(agents)            # get_equity for every current player + agent decision + step, all on the GPU
    s = tables.state()                      # host copy: numpy structured array, one record per table

`Action` and `Stage` carry the reference's values (gym_env/enums.py).
"""
import ctypes
from enum import IntEnum

import numpy as np

from . import _lib

MAX_SEATS = 10


class Action(IntEnum):
    FOLD = 0
    CHECK = 1
    CALL = 2
    RAISE_3BB = 3
    RAISE_HALF_POT = 4
    RAISE_POT = 5
    RAISE_2POT = 6
    ALL_IN = 7
    SMALL_BLIND = 8
    BIG_BLIND = 9


class Stage(IntEnum):
    PREFLOP = 0
    FLOP = 1
    TURN = 2
    RIVER = 3
    END_HIDDEN = 4
    SHOWDOWN = 5


AGENT_EQUITY, AGENT_RANDOM = 0, 1

_S = MAX_SEATS
TABLE_DTYPE = np.dtype([
    ("stack", "f8", (_S,)), ("player_pots", "f8", (_S,)), ("player_max_win", "f8", (_S,)), ("funds_prev", "f8", (_S,)),
    ("funds_last", "f8", (_S,)), ("community_pot", "f8"), ("current_round_pot", "f8"), ("min_call", "f8"),
    ("last_player_pot", "f8"), ("reward", "f8"), ("small_blind", "f8"), ("big_blind", "f8"), ("initial_stacks", "f8"),
    ("rng_counter", "u8"), ("stage_data", "u8"), ("deck_mask", "u8"),
    ("idx", "i4"), ("dealer_idx", "i4"), ("step_counter", "i4"), ("cycle_round_number", "i4"), ("max_steps_total", "i4"),
    ("last_raiser_step", "i4"), ("max_steps_after_raiser", "i4"), ("max_steps_after_big_blind", "i4"), ("last_raiser", "i4"),
    ("checkers", "i4"), ("max_remaining_steps_without_raising", "i4"),
    ("stage", "i4"), ("current_player", "i4"), ("winner_ix", "i4"), ("dealer_pos", "i4"), ("done", "i4"), ("funds_rows", "i4"),
    ("n_players", "i4"), ("max_raises", "i4"), ("n_table_cards", "i4"), ("n_deck", "i4"), ("acting_agent", "i4"),
    ("hands_played", "i4"), ("error", "i4"), ("legal_moves", "u4"),
    ("can_still", "u1", (_S,)), ("out_of_cash", "u1", (_S,)), ("folder", "u1", (_S,)), ("alive", "u1", (_S,)),
    ("first_action", "u1", (_S,)), ("autoplay", "u1", (_S,)), ("num_raises", "u1", (_S, 4)), ("cards", "u1", (_S, 2)),
    ("table_cards", "u1", (5,)), ("reserved", "u1", (1,)),
], align=True)


def _bind(L):
    if getattr(L, "_holdem_bound", False):
        return L
    vp, i64, i32, f64, u64 = ctypes.c_void_p, ctypes.c_int64, ctypes.c_int, ctypes.c_double, ctypes.c_uint64
    L.npk_holdem_table_bytes.restype = i64
    L.npk_holdem_init.argtypes = [vp, i64, i32, f64, f64, f64, i32, vp, u64, i64, vp]
    L.npk_holdem_reset_done.argtypes = [vp, i64, u64, i64, vp]
    L.npk_holdem_step.argtypes = [vp, i64, vp, vp, u64, i64, i32, vp]
    L.npk_holdem_queries.argtypes = [vp, i64, vp, vp, vp, vp, vp]
    L.npk_holdem_decide.argtypes = [vp, i64, vp, vp, i64, vp, vp, vp, vp, u64, i64, i64, vp, vp]
    L.npk_holdem_attach_stage_data.argtypes = [vp, i64, vp, vp]
    L.npk_holdem_observation_size.argtypes = [i32]
    L.npk_holdem_observation_size.restype = i64
    L.npk_holdem_observe.argtypes = [vp, i64, vp, vp, vp]
    if L.npk_holdem_table_bytes() != TABLE_DTYPE.itemsize:
        raise RuntimeError("NpkHoldemTable is %d bytes in libnpk.so but %d in holdem.TABLE_DTYPE"
                           % (L.npk_holdem_table_bytes(), TABLE_DTYPE.itemsize))
    L._holdem_bound = True
    return L


class EquityAgents(object):
    """Per-seat agents of a self-play table: agent_consider_equity players (min_call_equity, min_bet_equity;
    agents/agent_consider_equity.py:12-19) and random players (agents/agent_random.py)."""

    def __init__(self, n_players):
        self.kind = np.zeros(MAX_SEATS, dtype=np.uint8)
        self.min_call_equity = np.zeros(MAX_SEATS, dtype=np.float64)
        self.min_bet_equity = np.zeros(MAX_SEATS, dtype=np.float64)
        self.n_players = n_players

    def equity(self, seat, min_call_equity, min_bet_equity):
        self.kind[seat] = AGENT_EQUITY
        self.min_call_equity[seat] = min_call_equity
        self.min_bet_equity[seat] = min_bet_equity
        return self

    def random(self, seat):
        self.kind[seat] = AGENT_RANDOM
        return self

    @staticmethod
    def equity_vs_random():
        """main.py:136-150: four equity players and two random ones."""
        a = EquityAgents(6)
        a.equity(0, .5, -.5).equity(1, .8, -.8).equity(2, .7, -.7).equity(3, .2, -.3).random(4).random(5)
        return a


class HoldemTables(object):
    """N tables of the reference's HoldemTable (same constructor arguments, env.py:67-69), created, dealt and reset on
    the current CUDA device.  `autoplay` marks seats that are autoplay agents (it only decides the sign of the final
    reward, env.py:294-296)."""

    def __init__(self, n_tables, n_players=6, initial_stacks=100, small_blind=1, big_blind=2,
                 max_raises_per_player_round=2, autoplay=None, seed=0, table_offset=0, device=None):
        import torch
        self.torch = torch
        from .equity import _resolve_device
        self.device = _resolve_device(device)
        self.L = _bind(_lib.ensure_init(self.device.index))
        self.n_tables, self.n_players = int(n_tables), int(n_players)
        self.seed, self.table_offset = int(seed), int(table_offset)
        self.params = (float(initial_stacks), float(small_blind), float(big_blind), int(max_raises_per_player_round))
        self.autoplay = np.zeros(MAX_SEATS, dtype=np.uint8)
        if autoplay is not None:
            self.autoplay[:len(autoplay)] = np.asarray(autoplay, dtype=np.uint8)
        nbytes = TABLE_DTYPE.itemsize * self.n_tables
        self.buf = torch.zeros(nbytes, dtype=torch.uint8, device=self.device)
        self.rewards = torch.zeros(self.n_tables, dtype=torch.float64, device=self.device)
        self.decisions = 0
        self._q = None
        self.stage_data = None
        self.reset()

    # ---- plumbing ----
    def _stream(self):
        return self.torch.cuda.current_stream(self.device).cuda_stream

    def _u64(self, v):
        return ctypes.c_uint64(int(v) & (2**64 - 1))

    def reset(self):
        """HoldemTable.reset() for every table (env.py:138-168): fresh stacks, first hand dealt, blinds posted."""
        st, sb, bb, mr = self.params
        with self.torch.cuda.device(self.device):
            _lib.check(self.L.npk_holdem_init(self.buf.data_ptr(), self.n_tables, self.n_players, st, sb, bb, mr,
                                              self.autoplay.ctypes.data_as(ctypes.c_void_p), self._u64(self.seed),
                                              self.table_offset, self._stream()))
        return self

    def reset_done(self):
        """Start a new game on every finished table."""
        with self.torch.cuda.device(self.device):
            _lib.check(self.L.npk_holdem_reset_done(self.buf.data_ptr(), self.n_tables, self._u64(self.seed),
                                                    self.table_offset, self._stream()))

    def step(self, actions, restart_finished=False):
        """env.step(action) on every table.  `actions`: int8 CUDA tensor, or anything array-like of Action values;
        negative = leave that table alone.  restart_finished: reset a table as soon as its game is over.
        Returns the rewards tensor [N] (float64, CUDA)."""
        torch = self.torch
        if not isinstance(actions, torch.Tensor):
            actions = torch.as_tensor(np.asarray(actions, dtype=np.int8))
        actions = actions.to(self.device, dtype=torch.int8).contiguous()
        assert actions.numel() == self.n_tables
        with torch.cuda.device(self.device):
            _lib.check(self.L.npk_holdem_step(self.buf.data_ptr(), self.n_tables, actions.data_ptr(), self.rewards.data_ptr(),
                                              self._u64(self.seed), self.table_offset, 1 if restart_finished else 0,
                                              self._stream()))
        return self.rewards

    def queries(self):
        """The get_equity arguments of _get_environment (env.py:249-264) for every table, as CUDA uint8 tensors
        (hole [N,2], board [N,5], n_players [N], active [N])."""
        torch = self.torch
        if self._q is None:
            n = self.n_tables
            self._q = (torch.empty((n, 2), dtype=torch.uint8, device=self.device),
                       torch.empty((n, 5), dtype=torch.uint8, device=self.device),
                       torch.empty(n, dtype=torch.uint8, device=self.device),
                       torch.empty(n, dtype=torch.uint8, device=self.device))
        hole, board, npl, active = self._q
        with torch.cuda.device(self.device):
            _lib.check(self.L.npk_holdem_queries(self.buf.data_ptr(), self.n_tables, hole.data_ptr(), board.data_ptr(),
                                                 npl.data_ptr(), active.data_ptr(), self._stream()))
        return hole, board, npl, active

    def decide(self, agents, equity=None, wins=None, ties=None, runs=0):
        """Agent decisions for every table from an equity tensor [N] (float64) or from Monte-Carlo counters."""
        torch = self.torch
        actions = torch.empty(self.n_tables, dtype=torch.int8, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(self.L.npk_holdem_decide(
                self.buf.data_ptr(), self.n_tables, wins.data_ptr() if wins is not None else None,
                ties.data_ptr() if ties is not None else None, int(runs), equity.data_ptr() if equity is not None else None,
                agents.kind.ctypes.data_as(ctypes.c_void_p), agents.min_call_equity.ctypes.data_as(ctypes.c_void_p),
                agents.min_bet_equity.ctypes.data_as(ctypes.c_void_p), self._u64(self.seed), self.decisions,
                self.table_offset, actions.data_ptr(), self._stream()))
        self.decisions += 1
        return actions

    # kernels of libnpk per self-play step: holdem_queries, classify_count, classify_fill, equity_mixed, holdem_decide,
    # holdem_step (+ one memset of the workspace header and one torch zero_ of the [2,N] counters)
    launches_per_step = 6

    def selfplay_step(self, agents, runs=1000, deal_mode="reference", restart_finished=True, sync_free=True, stderr=None):
        """One action on every table, entirely on the device: the equity query of every current player
        (env.py:262-264: 1,000 runs, all players alive), the Monte-Carlo kernel, the agents' decisions
        (agent_consider_equity / random) and the state machine.  Returns the actions taken (int8 CUDA tensor).
        The queries of a step mix player counts and streets: they are sorted by shape on the device and ONE persistent
        kernel handles all shapes (csrc/npk_mixed.cu); nothing is read back, so the step can be captured in a CUDA graph.
        stderr: None runs `runs` trials for every query.  A number asks every equity to that standard error instead
        (get_equity_batch_adaptive with max_trials = runs): a query stops at the first checkpoint that reaches it, and the
        agents decide on equity = (wins + ties) / trials.
        (`sync_free` is accepted for compatibility: every mixed batch is free of host round trips now.)"""
        from .equity import get_equity_batch, get_equity_batch_adaptive
        hole, board, npl, _ = self.queries()
        if stderr is not None:
            out = get_equity_batch_adaptive(hole, board, npl, runs, stderr, min_trials=min(256, runs),
                                            seed_value=(self.seed << 20) + self.decisions, deal_mode=deal_mode,
                                            query_offset=self.table_offset, validate=False, device=self.device)
            actions = self.decide(agents, equity=self.adaptive_equity(out))
            self.step(actions, restart_finished=restart_finished)
            return actions
        out = getattr(self, "_mc_out", None)
        if out is None:
            both = self.torch.zeros((2, self.n_tables), dtype=self.torch.int64, device=self.device)
            out = {"wins": both[0], "ties": both[1], "_both": both}
            self._mc_out = out
        out["_both"].zero_()
        get_equity_batch(hole, board, npl, runs, seed_value=(self.seed << 20) + self.decisions, deal_mode=deal_mode,
                         query_offset=self.table_offset, validate=False, out=out, device=self.device)
        actions = self.decide(agents, wins=out["wins"], ties=out["ties"], runs=runs)
        self.step(actions, restart_finished=restart_finished)
        return actions

    @staticmethod
    def adaptive_equity(out):
        """(wins + ties) / trials of get_equity_batch_adaptive's counters, float64; 0 for a query that ran no trial."""
        return (out["wins"] + out["ties"]).double() / out["trials"].clamp(min=1).double()

    # ---- observations ----
    def enable_observations(self):
        """Attach StageData bookkeeping (env.py:40-50, 383-391) so that observe() can build the reference's observation
        vector.  Call right after construction / reset()."""
        torch = self.torch
        self.stage_data = torch.zeros((self.n_tables, 4, 6, MAX_SEATS), dtype=torch.float64, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(self.L.npk_holdem_attach_stage_data(self.buf.data_ptr(), self.n_tables, self.stage_data.data_ptr(),
                                                           self._stream()))
        return self

    def observe(self, equity=None):
        """`array_everything` of _get_environment (env.py:266-270) for every table: float64 CUDA tensor
        [N, 22 + 51 * n_players].  equity: [N] float64 CUDA tensor for equity_to_river_alive, or None (nan)."""
        torch = self.torch
        if getattr(self, "stage_data", None) is None:
            raise RuntimeError("call enable_observations() first")
        width = int(self.L.npk_holdem_observation_size(self.n_players))
        obs = torch.empty((self.n_tables, width), dtype=torch.float64, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(self.L.npk_holdem_observe(self.buf.data_ptr(), self.n_tables,
                                                 equity.data_ptr() if equity is not None else None, obs.data_ptr(),
                                                 self._stream()))
        return obs

    # ---- host views ----
    def state(self):
        """Host copy of every table as a numpy structured array (dtype TABLE_DTYPE = struct NpkHoldemTable)."""
        return self.buf.cpu().numpy().view(TABLE_DTYPE)

    @staticmethod
    def legal_moves_list(mask):
        return [Action(a) for a in range(10) if int(mask) >> a & 1]


# ---- one table with the reference's own front end ---------------------------------------------------------------------------
class _Seat(object):
    """What the reference calls PlayerShell (env.py:753-777), read from the device state."""

    def __init__(self, agent, seat):
        self.agent_obj, self.seat, self.name = agent, seat, getattr(agent, "name", "player")
        self.stack, self.cards, self.equity_alive = None, [], float("nan")


class HoldemTable(object):
    """gym_env/env.py::HoldemTable for ONE table, state machine on the GPU: same constructor arguments, add_player(),
    reset(), step(action) with the reference's return values (observation, reward, done, truncated, info), and the same
    agent protocol -- an agent with an `autoplay` attribute is asked `agent.action(legal_moves, observation, info,
    funds_history)` (agents/agent_consider_equity.py, agent_random.py plug in unchanged), any other seat is driven by
    the `action` passed to step().  `get_equity` is the equity calculator of the plugin point (env.py:75-81); the default
    is this package's get_equity.  funds_history is a list of stack rows instead of a pandas frame."""

    def __init__(self, initial_stacks=100, small_blind=1, big_blind=2, render=False, funds_plot=True,
                 max_raises_per_player_round=2, use_cpp_montecarlo=False, raise_illegal_moves=False, calculate_equity=False,
                 get_equity=None, seed=0):
        from .equity import get_equity as _gpu_equity, montecarlo as _gpu_montecarlo
        self.get_equity = get_equity or (_gpu_montecarlo if use_cpp_montecarlo else _gpu_equity)
        self.initial_stacks, self.small_blind, self.big_blind = initial_stacks, small_blind, big_blind
        self.max_raises_per_player_round = max_raises_per_player_round
        self.raise_illegal_moves = raise_illegal_moves
        self.players, self.num_of_players = [], 0
        self.tables, self.seed = None, seed
        self.done, self.reward, self.info, self.observation, self.array_everything = False, None, None, None, None
        self.funds_history, self.legal_moves, self.illegal_move_reward = [], [], -1

    def add_player(self, agent):
        """env.py:526-535"""
        self.players.append(_Seat(agent, len(self.players)))
        self.num_of_players += 1

    # -- state mirrored from the device after every call --
    def _pull(self):
        from .cards import card_str
        s = self.tables.state()[0]
        self._s = s
        n = self.num_of_players
        for i, p in enumerate(self.players):
            p.stack = float(s["stack"][i])
            p.cards = [card_str(c) for c in s["cards"][i] if c < 52]
        self.stage = Stage(int(s["stage"]))
        self.done = bool(s["done"])
        self.winner_ix = int(s["winner_ix"]) if s["winner_ix"] >= 0 else None
        self.dealer_pos = int(s["dealer_pos"])
        self.community_pot, self.current_round_pot = float(s["community_pot"]), float(s["current_round_pot"])
        self.min_call = float(s["min_call"])
        self.player_pots = [float(x) for x in s["player_pots"][:n]]
        self.table_cards = [card_str(c) for c in s["table_cards"] if c < 52]
        self.legal_moves = HoldemTables.legal_moves_list(s["legal_moves"])
        cp = int(s["current_player"])
        self.current_player = self.players[cp] if cp >= 0 else None
        if int(s["funds_rows"]) > len(self.funds_history):
            self.funds_history.append([float(x) for x in s["funds_last"][:n]])

    def _get_environment(self):
        """env.py:232-278: equity of the current player, observation vector, info dictionary."""
        import torch
        s, cp = self._s, self.current_player
        alive = int(s["alive"][:self.num_of_players].sum())
        eq = float("nan")
        if cp is not None and len(cp.cards) == 2:
            eq = self.get_equity(set(cp.cards), set(self.table_cards), alive, 1000)
            cp.equity_alive = eq
        obs = self.tables.observe(torch.tensor([eq], dtype=torch.float64, device=self.tables.device))[0].cpu().numpy()
        self.array_everything = self.observation = obs
        unit = self.big_blind * 100
        self.info = {"player_data": {"position": cp.seat if cp else None, "equity_to_river_alive": eq,
                                     "equity_to_river_2plr": float("nan"), "equity_to_river_3plr": float("nan"),
                                     "stack": [p.stack / unit for p in self.players]},
                     "community_data": {"stage": [i == min(self.stage.value, 3) for i in range(4)],
                                        "community_pot": self.community_pot / unit,
                                        "current_round_pot": self.current_round_pot / unit,
                                        "big_blind": self.big_blind, "small_blind": self.small_blind,
                                        "legal_moves": [a in self.legal_moves for a in Action]},
                     "stage_data": self.tables.stage_data[0].cpu().numpy(), "legal_moves": self.legal_moves}

    def _autoplay(self):
        return self.current_player is not None and hasattr(self.current_player.agent_obj, "autoplay")

    def reset(self, seed=None, options=None):
        """env.py:138-168"""
        if seed is not None:
            self.seed = seed
        if not self.players:
            return self.array_everything, self.info
        self.tables = HoldemTables(1, n_players=self.num_of_players, initial_stacks=self.initial_stacks,
                                   small_blind=self.small_blind, big_blind=self.big_blind,
                                   max_raises_per_player_round=self.max_raises_per_player_round,
                                   autoplay=[int(hasattr(p.agent_obj, "autoplay")) for p in self.players], seed=self.seed)
        self.tables.enable_observations()
        self.funds_history = []
        self._pull()
        self._get_environment()
        if self._autoplay() and not self.done:
            self.step("initial_player_autoplay")
        return self.array_everything, self.info

    def _apply(self, action):
        action = Action(int(getattr(action, "value", action)))
        if action not in self.legal_moves:
            if self.raise_illegal_moves:
                raise ValueError("%s is an Illegal move, try again. Currently allowed: %s" % (action, self.legal_moves))
        self.reward = float(self.tables.step([int(action)])[0].item())
        self._pull()
        self._get_environment()

    def step(self, action):
        """env.py:170-200: autoplay agents act until a seat driven from outside is to move (or the game is over).
        The reward of an autoplay sequence follows the reference to the letter (:178-188): `acting_agent` is the seat that was
        to move when step() was entered, and after EVERY legal autoplay action `_calculate_reward` (:282-306) runs for that seat
        -- the final reward when the game is over, else the difference of its last two funds-history rows once there are two,
        else whatever the reward was before (the device step only rewards externally driven seats, :194-197)."""
        self.reward = 0
        if self._autoplay():
            acting = self.current_player.seat
            while self._autoplay() and not self.done and self.legal_moves:
                a = self.current_player.agent_obj.action(self.legal_moves, self.observation, self.info, self.funds_history)
                before = self.reward
                legal = Action(int(getattr(a, "value", a))) in self.legal_moves
                self._apply(a)
                if not legal:
                    continue                                   # _illegal_move sets its own reward (kept from the device step)
                s = self._s
                if self.done:
                    won = -1 if hasattr(self.players[self.winner_ix].agent_obj, "autoplay") else 1
                    self.reward = self.initial_stacks * len(self.players) * won
                elif int(s["funds_rows"]) > 1:
                    self.reward = float(s["funds_last"][acting]) - float(s["funds_prev"][acting])
                else:
                    self.reward = before
        else:
            self._apply(action)
        return self.array_everything, self.reward, self.done, False, self.info
