#!/usr/bin/env python
"""Fused rollout kernels versus shard size: the CUDA-core kernel (k_policy_rollout, column prefix cuda_core) and the
tensor-core kernel (k_policy_rollout_tc3, column prefix tc_shared_weight_loads).  One JSON line per size."""
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import ppo_car_b200  # noqa: E402
from ppo_car_b200.train_ppo import ActorCritic  # noqa: E402

dev = torch.device("cuda")
track = ppo_car_b200.builtin_track("big_track")
torch.manual_seed(0)
net = ActorCritic(18, 9).to(dev)
packed_cc = ppo_car_b200.pack_policy_weights(net.actor, net.critic)
packed_tc = ppo_car_b200.pack_policy_weights_tc(net.actor, net.critic)
SIZES = ((4096, 256), (8192, 256), (16384, 128), (32768, 128), (65536, 64), (131072, 64), (262144, 32), (1048576, 16))
if len(sys.argv) > 1:                                       # python benchmarks/fused_tiles.py 32768 1048576
    SIZES = tuple((n, T) for n, T in SIZES if str(n) in sys.argv[1:])
for n, T in SIZES:
    env = ppo_car_b200.VecCarEnv(n, track, reward_scaling=0.1, float_flags=True, with_info=False)
    buf = ppo_car_b200.Buffer((18,), T, n, dev)
    obs = env.reset()[0].clone()
    term, trunc, lv = torch.zeros(n, device=dev), torch.zeros(n, device=dev), torch.empty(n, device=dev)
    res = {"n_envs": n, "steps_per_launch": T}
    for tag, packed in (("cuda_core", packed_cc), ("tc_shared_weight_loads", packed_tc)):
        for i in range(2):
            ppo_car_b200.fused_rollout(env, packed, buf, obs, term, trunc, seed=1, step0=i * T, last_val=lv)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 5
        e0.record()
        for i in range(reps):
            ppo_car_b200.fused_rollout(env, packed, buf, obs, term, trunc, seed=1, step0=(i + 2) * T, last_val=lv)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / reps
        res[tag + "_us_per_step"] = round(ms / T * 1e3, 2)
        res[tag + "_env_steps_per_s"] = n * T / ms * 1e3
    print(json.dumps(res), flush=True)
    del buf, env
