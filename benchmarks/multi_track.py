#!/usr/bin/env python
"""Several tracks in one launch: the multi-track fused rollout (k_policy_rollout_tc3<0>, carenv_policy_rollout_tc_multi)
and the multi-track evaluation (k_policy_eval<0>, carenv_policy_eval_multi) against their single-track kernels.

Fused rollout, us per step (CUDA-event time of whole launches / steps per launch, after two warm-up launches) at
4,096, 32,768, 262,144 and 1,048,576 environments:
  tc3_single_big_track     k_policy_rollout_tc3<4, true> on big_track (what --fused-rollout runs today)
  tc3_multi_big_track      the multi-track kernel with every environment on big_track: the cost of the generic
                           segment loop with the track read through pointers
  tc3_multi_3_blocks       big_track, track and a 30-segment ring in contiguous blocks (train_ppo's assignment)
  tc3_multi_3_random       the same three tracks assigned at random per environment (mixed warps)
  eager_multi              MultiTrackVecEnv.step + the torch actor / critic per step (24 and 32,768 environments)
Evaluation, env-steps/s (sum of episode lengths over CUDA-event time) at 65,536 and 1,048,576 sampled episodes of a
freshly initialised actor: single-track big_track, multi-track with every episode on big_track, and the three tracks
by the default assignment (episode g on track g % 3).

One JSON line per measurement to --out, each with the GPU's name and power limit read in the same run."""
import argparse
import json
import math
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import ppo_car_b200  # noqa: E402
from ppo_car_b200.evaluate import evaluate_policy  # noqa: E402
from ppo_car_b200.train_ppo import ActorCritic  # noqa: E402
from tests.synth_tracks import ring_track  # noqa: E402

ROLLOUT_SIZES = (4096, 32768, 262144, 1048576)
EAGER_SIZES = (24, 32768)
EVAL_SIZES = (65536, 1048576)


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                              "-i", "0"], capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.TimeoutExpired):
        out = ""
    return {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": out}


def steps_for(n):
    return 1024 if n <= 32768 else (256 if n <= 262144 else 64)   # [T, n, 18] observation rows: 4.8 GB at 1 M envs


def time_fused(env, net, n, T):
    dev = env.device
    packed = ppo_car_b200.pack_policy_weights_tc(net.actor, net.critic)
    buf = ppo_car_b200.Buffer((18,), T, n, dev)
    obs = env.reset()[0].clone()
    term, trunc, lv = torch.zeros(n, device=dev), torch.zeros(n, device=dev), torch.empty(n, device=dev)

    def run(i):
        ppo_car_b200.fused_rollout(env, packed, buf, obs, term, trunc, seed=1, step0=i * T, last_val=lv)

    for i in range(2):
        run(i)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    run(2)
    e1.record()
    torch.cuda.synchronize()
    reps = max(1, min(10, math.ceil(0.5 / max(e0.elapsed_time(e1) / 1e3, 1e-6))))
    e0.record()
    for i in range(reps):
        run(3 + i)
    e1.record()
    torch.cuda.synchronize()
    s = e0.elapsed_time(e1) / 1e3
    return {"steps_per_launch": T, "launches": reps, "us_per_step": s / (reps * T) * 1e6,
            "env_steps_per_s": n * T * reps / s}


def time_eager(env, net, n, T):
    """The loop a user writes around MultiTrackVecEnv.step: actor and critic in torch, one env launch per step."""
    dev = env.device
    buf = ppo_car_b200.Buffer((18,), T, n, dev)

    def run():
        obs = env.reset()[0].clone()
        buf.ptr = 0
        with torch.no_grad():
            for _ in range(T):
                act, logp, _, val = net.act(obs)
                buf.store(obs, act, 0.0, val.view(-1), 0.0, 0.0, logp)
                o, rew, te, tr, _ = env.step(act)
                buf.rew_buf[buf.ptr - 1].copy_(rew)
                obs.copy_(o)

    run()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    run()
    torch.cuda.synchronize()
    s = time.perf_counter() - t0
    return {"steps_per_launch": T, "us_per_step": s / T * 1e6, "env_steps_per_s": n * T / s}


def time_eval(env, actor, n):
    evaluate_policy(env, actor, n, seed=1)                         # warm-up
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 3
    steps = 0
    e0.record()
    results = [evaluate_policy(env, actor, n, seed=2 + r) for r in range(reps)]
    e1.record()
    torch.cuda.synchronize()
    s = e0.elapsed_time(e1) / 1e3
    steps = sum(r.length.sum().item() for r in results)
    return {"reps": reps, "kernel_s_per_call": s / reps, "env_steps_per_s": steps / s, "mean_length": steps / (n * reps)}


def main():
    p = argparse.ArgumentParser()
    p.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_multi_track.jsonl"))
    p.add_argument("--rollout-sizes", default=",".join(map(str, ROLLOUT_SIZES)))
    p.add_argument("--eval-sizes", default=",".join(map(str, EVAL_SIZES)))
    args = p.parse_args()
    info = gpu_info()
    dev = torch.device("cuda", 0)
    torch.manual_seed(0)
    net = ActorCritic(18, 9).to(dev)
    big = ppo_car_b200.builtin_track("big_track")
    with tempfile.TemporaryDirectory() as d:
        three = [big, ppo_car_b200.builtin_track("track"), ring_track(os.path.join(d, "ring18_12.json"), 18, 12)]
        three_names = ["big_track", "track", "ring18_12"]
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            def emit(rec):
                rec.update(info)
                print(json.dumps(rec), flush=True)
                fh.write(json.dumps(rec) + "\n")

            for n in [int(x) for x in args.rollout_sizes.split(",")]:
                T = steps_for(n)
                rng = np.random.default_rng(n)
                variants = [
                    ("tc3_single_big_track", ["big_track"], lambda: ppo_car_b200.VecCarEnv(
                        n, big, reward_scaling=0.1, float_flags=True, with_info=False)),
                    ("tc3_multi_big_track", ["big_track"], lambda: ppo_car_b200.MultiTrackVecEnv(
                        track_paths=[big], track_ids=np.zeros(n, np.int32), reward_scaling=0.1, float_flags=True)),
                    ("tc3_multi_3_blocks", three_names, lambda: ppo_car_b200.MultiTrackVecEnv(
                        track_paths=three, track_ids=(np.arange(n) * 3 // n).astype(np.int32), reward_scaling=0.1,
                        float_flags=True)),
                    ("tc3_multi_3_random", three_names, lambda: ppo_car_b200.MultiTrackVecEnv(
                        track_paths=three, track_ids=rng.integers(0, 3, n).astype(np.int32), reward_scaling=0.1,
                        float_flags=True)),
                ]
                for name, tracks, make in variants:
                    env = make()
                    emit({"what": "fused_rollout", "variant": name, "tracks": tracks, "n_envs": n,
                          **time_fused(env, net, n, T)})
                    env.close()
                    torch.cuda.empty_cache()
            for n in EAGER_SIZES:
                T = 256 if n <= 1024 else 64
                env = ppo_car_b200.MultiTrackVecEnv(track_paths=three, track_ids=(np.arange(n) * 3 // n).astype(np.int32),
                                                    reward_scaling=0.1, float_flags=True)
                emit({"what": "fused_rollout", "variant": "eager_multi", "tracks": three_names, "n_envs": n,
                      **time_eager(env, net, n, T)})
                env.close()
            for n in [int(x) for x in args.eval_sizes.split(",")]:
                single = ppo_car_b200.VecCarEnv(1, big)
                emit({"what": "policy_eval", "variant": "single_big_track", "tracks": ["big_track"], "n_episodes": n,
                      **time_eval(single, net.actor, n)})
                single.close()
                for name, paths, names in (("multi_big_track", [big], ["big_track"]),
                                           ("multi_3_default", three, three_names)):
                    env = ppo_car_b200.MultiTrackVecEnv(track_paths=paths, track_ids=[0])
                    emit({"what": "policy_eval", "variant": name, "tracks": names, "n_episodes": n,
                          **time_eval(env, net.actor, n)})
                    env.close()


if __name__ == "__main__":
    main()
