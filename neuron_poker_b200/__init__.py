"""neuron_poker_b200 -- B200-native (sm_100a) replacement for neuron_poker's Monte-Carlo equity hot path.

Public surface = the reference's own plugin interface for this path:
    get_equity(player_cards, table_cards, players, runs)            tools/montecarlo_python.py:401
    montecarlo(my_cards, cards_on_table, players, iterations)       tools/montecarlo_cpp/pymontecarlo.cpp:22
    MonteCarlo().run_montecarlo(...)                                tools/montecarlo_python.py:191
    numpy_montecarlo(my_cards, table, iterations, players)          tools/montecarlo_numpy2.py:333 (per cent)
    get_winner(player_hands, table_cards), eval_best_hand(hands)    tools/hand_evaluator.py:9, :20
plus batched entry points on CUDA tensors (get_equity_batch, get_equity_batch_adaptive -- each query to a target standard
error --, get_equity_ranges_batch, get_equity_ranges_batch_adaptive, rank7, showdown, enumerate_equity,
showdown_equity_batch), the exact equity of known hands (showdown_equity)
and the vectorised environment (holdem.HoldemTables: gym_env/env.py::HoldemTable for N tables on the GPU).
All compute runs in libnpk.so's CUDA kernels; importing this package does not import torch.
"""
from .cards import CARD_RANKS_ORIGINAL, SUITS_ORIGINAL, HAND_TYPES, card_id, card_str  # noqa: F401
from .equity import (DEAL_REFERENCE, DEAL_UNIFORM, MonteCarlo, equity_counts, equity_counts_batch,  # noqa: F401
                     equity_counts_ranges, get_equity, get_equity_batch, get_equity_batch_adaptive,
                     get_equity_ranges_batch, get_equity_ranges_batch_adaptive, montecarlo,
                     numpy_montecarlo, resident, seed)
from . import dist, holdem, ranges  # noqa: F401
from .evaluator import (enumerate_equity, eval_best_hand, get_winner, host_rank7, host_tables, rank7, rank7_colex,  # noqa: F401
                        showdown, showdown_equity, showdown_equity_batch)

__version__ = "0.1.0"
