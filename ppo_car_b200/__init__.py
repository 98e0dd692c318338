"""ppo_car_b200 — B200-native batched CarEnv step + GAE (the hot path of ProfessorNova/PPO-Car).

Public surface (mirrors what the reference's train.py uses):
  VecCarEnv   batched, auto-resetting CarEnv           (gym.vector.AsyncVectorEnv of CarEnv-v0)
  Buffer      rollout buffer with the GAE kernel        (lib.buffer.Buffer)
  gae_reverse_scan, load_track, builtin_track, build
  evaluate_policy   whole episodes of a policy in one launch: returns, laps, crashes
  evaluate_population   the same for many stacked actors (a population's members) in one launch
  Population, train_population   many independent policies (seed / hyperparameter sweeps) trained in one process
"""
from ._lib import CarEnvError, build
from .buffer import Buffer, gae_reverse_scan
from .track import Track, builtin_track, load_track, validate_track
from .vec_env import MultiTrackVecEnv, VecCarEnv
from .policy import fused_rollout, fused_rollout_warp, pack_policy_weights, pack_policy_weights_tc
from .ppo_update import FusedPPOUpdate
from .evaluate import EvalResult, evaluate_policy, evaluate_population
from .population import Population, train_population

__all__ = ["VecCarEnv", "MultiTrackVecEnv", "validate_track", "Buffer", "gae_reverse_scan", "load_track", "builtin_track", "Track", "build", "CarEnvError",
           "fused_rollout", "fused_rollout_warp", "pack_policy_weights", "pack_policy_weights_tc", "FusedPPOUpdate",
           "evaluate_policy", "evaluate_population", "EvalResult", "Population", "train_population"]
