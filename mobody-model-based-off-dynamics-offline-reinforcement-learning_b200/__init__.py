"""mobody_b200 — B200-native (sm_100a) hot path of MOBODY: fused model rollout and Q-weighted BC update.

Public names mirror the reference modules they replace:
  algo.dynamics.mobody_module     -> MOBODYModule, EnsembleLinear, Swish
  algo.dynamics.mobody_dynamics   -> MOBODYEnsembleDynamics, StandardScaler
  algo.mb_utils.terminal_funs     -> get_termination_fn
  algo.utils                      -> ReplayBuffer
  algo.offline_offline.mobody     -> MOBODY, Policy, DoubleQFunc, MLPNetwork, ValueFunc
  dataset.call_dataset            -> call_tar_dataset (+ transitions_from_raw, read_raw, load_buffers)
  train_mobody (evaluators)       -> eval_policy, eval_policy_batch (+ eval_policy_in_model: no simulator)
"""
from . import _ffi, parallel                                          # noqa: F401
from .module import MOBODYModule, EnsembleLinear, Swish, soft_clamp   # noqa: F401
from .dynamics import MOBODYEnsembleDynamics, StandardScaler          # noqa: F401
from .terminal_funs import get_termination_fn, TERM_KINDS             # noqa: F401
from .buffer import ReplayBuffer                                      # noqa: F401
from .dataset import call_tar_dataset, transitions_from_raw, read_raw, load_buffers   # noqa: F401
from .evaluate import eval_policy, eval_policy_batch, eval_policy_in_model   # noqa: F401
from .mobody import MOBODY, Policy, DoubleQFunc, MLPNetwork, ValueFunc, Classifier  # noqa: F401

__all__ = ["MOBODYModule", "EnsembleLinear", "Swish", "MOBODYEnsembleDynamics", "StandardScaler",
           "get_termination_fn", "ReplayBuffer", "MOBODY", "Policy", "DoubleQFunc", "MLPNetwork", "ValueFunc", "Classifier"]
