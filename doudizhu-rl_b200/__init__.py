"""doudizhu-rl_b200 -- B200-native batched Doudizhu environment (drop-in for the rollout path of
charleschen003/doudizhu-rl: envi.py + its absent native modules `env` and `r`).

The directory name carries a hyphen, so import it as `ddz_b200` (the alias module at the repo root) or with
importlib.import_module("doudizhu-rl_b200").
"""
from . import _native as native  # raises ImportError when libddz_b200.so has not been built
from . import sharding
from .agent import BatchedGreedyPolicy, FusedQScorer
from .trainer import ReplayBuffer, PackedReplayBuffer, TransitionCollector, gather_states, decode_rows, td_step
from .game import BatchedGame, BatchedDQN
from .ingest import env_from_payloads, env_from_arrays, payload_arrays, evaluate_moves, mcts, mcts_batch, pimc_batch
from .search import UctSearch, uct_search, pimc_search
from .policy import policy_sample, policy_log_prob, legal_lists_of_states, LinearPolicyHead, HeadedPolicy
from .env import (Trajectory, GraphedRollout, GroupedEnv, HostRollout, HostRolloutGroups, GroupStepResults, StepResults, BatchedEnv, BatchedEnvComplicated, BatchedEnvCooperation, BatchedEnvCooperationSimplify,
                  Env, EnvComplicated, EnvCooperation, EnvCooperationSimplify,
                  MoveGenerator, get_moves, kth_moves, mcts_moves, move_ids, moves_of_ids, action_space, ActionSpace, pack_counts, unpack_counts, default_deals, random_deals, adversarial_pairs, ADVERSARIAL_POOL,
                  VARIANT_CHANNELS, DEFAULT_REWARDS)

__all__ = ["native", "sharding", "BatchedGreedyPolicy", "FusedQScorer", "ReplayBuffer", "PackedReplayBuffer", "TransitionCollector", "gather_states", "decode_rows", "td_step", "BatchedGame", "BatchedDQN", "env_from_payloads", "env_from_arrays", "payload_arrays", "evaluate_moves", "mcts", "mcts_batch", "pimc_batch", "UctSearch", "uct_search", "pimc_search", "policy_sample", "policy_log_prob", "legal_lists_of_states", "LinearPolicyHead", "HeadedPolicy", "Trajectory", "GraphedRollout", "GroupedEnv", "HostRollout", "HostRolloutGroups", "GroupStepResults", "StepResults", "BatchedEnv", "BatchedEnvComplicated", "BatchedEnvCooperation", "BatchedEnvCooperationSimplify",
           "Env", "EnvComplicated", "EnvCooperation", "EnvCooperationSimplify", "MoveGenerator", "get_moves", "kth_moves", "mcts_moves", "move_ids", "moves_of_ids", "action_space", "ActionSpace", "pack_counts",
           "unpack_counts", "default_deals", "random_deals", "adversarial_pairs", "ADVERSARIAL_POOL", "VARIANT_CHANNELS", "DEFAULT_REWARDS"]
