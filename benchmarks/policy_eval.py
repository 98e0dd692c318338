#!/usr/bin/env python
"""Policy evaluation throughput: k_policy_eval (ppo_car_b200.evaluate_policy, one launch per call) at
n_episodes in {1, 24, 1,024, 16,384, 262,144, 1,048,576}, greedy and sampled, for a freshly initialised actor
(it crashes: about 270 steps per sampled episode, 106 greedy) and one trained in-script by the README run (24 envs
x 1024 steps x 200 epochs on big_track, fused rollout and update: about 840 steps and 2.5 laps per sampled
episode).  Beside it, at the small sizes, the eager loop a user would otherwise write: torch actor, VecCarEnv.step
on CUDA actions, bookkeeping until every episode has ended.

episodes/s and env-steps/s (sum of the episode lengths) over CUDA-event time of the kernel calls, after one
warm-up call per shape.  One JSON line per (actor, mode, size) to --out, with the GPU's name and power limit."""
import argparse
import json
import math
import os
import subprocess
import sys
import tempfile
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import ppo_car_b200  # noqa: E402
from ppo_car_b200.evaluate import evaluate_policy, load_checkpoint  # noqa: E402
from ppo_car_b200.train_ppo import ActorCritic, parse_args as train_args, train  # noqa: E402

SIZES = (1, 24, 1024, 16384, 262144, 1048576)
EAGER_SIZES = (1, 24, 1024)


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                              "-i", "0"], capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.TimeoutExpired):
        out = ""
    return {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": out}


def time_kernel(env, actor, n, greedy):
    evaluate_policy(env, actor, n, greedy=greedy, seed=1)          # warm-up (module load, attribute set-up)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    res = evaluate_policy(env, actor, n, greedy=greedy, seed=2)
    e1.record()
    torch.cuda.synchronize()
    one = e0.elapsed_time(e1) / 1e3
    reps = max(1, min(20, math.ceil(0.3 / max(one, 1e-6))))       # at least ~0.3 s of kernel time per number
    steps = res.length.sum().item()
    e0.record()
    for r in range(reps):
        res = evaluate_policy(env, actor, n, greedy=greedy, seed=3 + r)
    e1.record()
    torch.cuda.synchronize()
    s = e0.elapsed_time(e1) / 1e3
    if greedy:
        steps = res.length.sum().item() * reps                    # every call plays the same episodes
    else:                                                         # the seeds differ: count the timed calls' steps
        steps = sum(evaluate_policy(env, actor, n, greedy=False, seed=3 + r).length.sum().item() for r in range(reps))
    return {"reps": reps, "kernel_s_per_call": s / reps, "episodes_per_s": n * reps / s, "env_steps_per_s": steps / s,
            "mean_length": steps / (n * reps), "summary": res.summary()}


def eager_loop(track, actor, n, greedy):
    """What a user writes without the kernel: n environments, one episode each, torch actor between steps."""
    env = ppo_car_b200.VecCarEnv(n, track, reward_scaling=1.0)
    dev = env.device

    def run():
        obs = env.reset()[0].clone()
        done = torch.zeros(n, dtype=torch.bool, device=dev)
        ret = torch.zeros(n, dtype=torch.float64, device=dev)
        length = torch.zeros(n, dtype=torch.int64, device=dev)
        with torch.no_grad():
            while True:
                logits = actor(obs)
                a = logits.argmax(-1) if greedy else torch.multinomial(torch.softmax(logits, -1), 1).squeeze(-1)
                o, r, te, tr, _ = env.step(a)
                live = ~done
                ret += torch.where(live, r.double(), 0.0)
                length += live.long()
                done |= te.bool() | tr.bool()
                obs.copy_(o)
                if bool(done.all()):
                    return length.sum().item()

    run()                                                         # warm-up
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    steps = run()
    torch.cuda.synchronize()
    s = time.perf_counter() - t0
    env.close()
    return {"eager_s": s, "eager_episodes_per_s": n / s, "eager_env_steps_per_s": steps / s}


def main():
    p = argparse.ArgumentParser()
    p.add_argument("--out", default=os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))),
                                                 "profiles", "r3_policy_eval.jsonl"))
    p.add_argument("--sizes", default=",".join(map(str, SIZES)))
    args = p.parse_args()
    sizes = [int(x) for x in args.sizes.split(",")]
    info = gpu_info()
    track = ppo_car_b200.builtin_track("big_track")
    dev = torch.device("cuda", 0)
    torch.manual_seed(0)
    actors = {"fresh": ActorCritic(18, 9).actor.to(dev)}
    with tempfile.TemporaryDirectory() as d:
        t0 = time.perf_counter()
        hist = train(train_args(["--track", "big_track", "--n-envs", "24", "--fused-rollout", "--fused-update",
                                 "--checkpoint-dir", d, "--run-name", "readme"]))
        train_s = time.perf_counter() - t0
        actors["trained_readme"] = load_checkpoint(os.path.join(d, "readme", "model.dat")).actor.to(dev)
    env = ppo_car_b200.VecCarEnv(1, track)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        for name, actor in actors.items():
            for greedy in (False, True):
                for n in sizes:
                    rec = {"actor": name, "greedy": greedy, "n_episodes": n, "track": "big_track", **info}
                    if name == "trained_readme":
                        rec["train_final_avg_reward"] = hist[-1]["avg_reward"]
                        rec["train_wall_s"] = train_s
                    rec.update(time_kernel(env, actor, n, greedy))
                    if n in EAGER_SIZES:
                        rec.update(eager_loop(track, actor, n, greedy))
                        rec["speedup_vs_eager"] = rec["env_steps_per_s"] / rec["eager_env_steps_per_s"]
                    print(json.dumps(rec), flush=True)
                    fh.write(json.dumps(rec) + "\n")
    env.close()


if __name__ == "__main__":
    main()
