"""pbn_rl_b200 -- B200-native batched Probabilistic Boolean Network environment.

Drop-in for the gym-PBN env that jakub-zarzycki2022/pbn-rl's train_*.py / model_tester.py
drive: ISPL network loading, attractor pickles, gym reset()/step(), all served by
hand-written sm_100a CUDA kernels behind the C-ABI of include/pbn_b200.h.
"""
from .attractors import (AttractorSet, find_attractors_stg, load_attractor_pickle, save_attractor_pickle,
                         sorted_id_permutation)
from .ispl import BoolFunction, IsplError, compile_expression, logic_functions_from_ispl, parse_ispl, render_ispl
from .network import PBNNetwork, pack_states, unpack_states

__all__ = [
    "AttractorSet", "find_attractors_stg", "load_attractor_pickle", "save_attractor_pickle",
    "sorted_id_permutation", "BoolFunction", "IsplError", "compile_expression", "logic_functions_from_ispl",
    "parse_ispl", "render_ispl", "PBNNetwork", "pack_states", "unpack_states", "VecPBNEnv",
    "solve_control", "ControlSolution", "TabularPolicy", "policy_values", "tabulate_policy", "expected_all_pairs",
    "StateDistribution", "propagate", "stationary_distribution",
]

_CONTROL = ("solve_control", "ControlSolution", "TabularPolicy", "policy_values", "tabulate_policy", "expected_all_pairs")
_STEADY_STATE = ("StateDistribution", "propagate", "stationary_distribution")


def __getattr__(name):
    # torch-dependent parts load lazily so the pure-host loaders import without torch
    if name == "VecPBNEnv":
        from .vec_env import VecPBNEnv
        return VecPBNEnv
    if name in ("PBNEnv", "ControlPBNEnv", "make", "register_gym_ids"):
        from . import gym_env
        return getattr(gym_env, name)
    if name in _CONTROL:
        from . import control
        return getattr(control, name)
    if name in _STEADY_STATE:
        from . import steady_state
        return getattr(steady_state, name)
    raise AttributeError(name)
