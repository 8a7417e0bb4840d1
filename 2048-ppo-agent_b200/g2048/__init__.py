"""g2048 -- B200-native rollout engine for 2048 (env step + action selection + rollout records + GAE).

The compute lives in libg2048.so (hand-written sm_100a CUDA behind a C ABI, include/g2048.h);
this package is the thin Python host side that mirrors the reference's own API
(src/env_definitions.py, src/actions, src/runs, src/stats, src/ppo rollout pieces).
"""
from . import _native  # noqa: F401  loads libg2048.so; raises ImportError if it is missing
from . import engine, keys  # noqa: F401
from .actions import act_drul, act_randomly
from .env_definitions import ACTION_DIM, BOARD_DIM, BOARD_FLAT_DIM, OBS_DIM
from .expectimax import ExpectimaxPolicy, ExpectimaxValues, default_row_values, expectimax_values
from .playouts import MonteCarloPolicy, PlayoutValues, playout_values
from .ppo import DevicePPOBatches, PPODataset, PPOIterationLoop, RolloutBuffer, TorchActionFunction, compute_gae, create_ppo_dataloader
from .runs import BatchRunner, FixedHorizonRunner, FixedRollout, FlatRollout, PackedRollout, run_actions_batch, run_actions_max_tile
from .state import State
from .stats import RunningStatsVec
from .ntuple import NTupleNetwork
from .td import NTupleTCLearner, NTupleTDLearner, TDLearner

__all__ = [
    "ACTION_DIM", "BOARD_DIM", "BOARD_FLAT_DIM", "OBS_DIM", "BatchRunner", "DevicePPOBatches", "ExpectimaxPolicy", "ExpectimaxValues", "FixedHorizonRunner", "FixedRollout", "FlatRollout",
    "MonteCarloPolicy", "NTupleNetwork", "NTupleTCLearner", "NTupleTDLearner", "PPODataset", "PPOIterationLoop", "PackedRollout", "PlayoutValues",
    "RolloutBuffer", "RunningStatsVec", "State", "TDLearner", "TorchActionFunction", "act_drul", "act_randomly", "compute_gae",
    "create_ppo_dataloader", "default_row_values", "engine", "expectimax_values", "keys", "playout_values", "run_actions_batch", "run_actions_max_tile",
]
