#!/usr/bin/env python
"""Scoring a population: one member-batched evaluation launch (``evaluate_population``, k_policy_eval<U, true>)
against the per-member loop ``train_population --eval-every`` ran before it (``evaluate_policy(env,
pop.member_actor(p), ...)`` and ``summary()`` for every member).

P in {1, 8, 32, 128} members x 1,024 episodes each on big_track, sampled and greedy, for three populations:
  fresh     the initial actors of seeds 0 .. P-1 (they crash: about 270 steps per sampled episode)
  trained   the README-trained actor (24 envs x 1024 steps x 200 epochs, fused rollout and update, trained in-script)
            stacked P times: about 840 steps per sampled episode
  mixed     half fresh, half trained (P >= 8): every member has CTAs of its own (8, or one wave / P when fewer),
            so the members with short episodes leave their slots idle while the long ones finish
Timed per case:
  batched   one evaluate_population call, CUDA events over repeated calls after a warm-up call
  batched+summaries   what train_population does per evaluation epoch: the call, every member's sums in one copy,
            the summaries; host clock ending in a synchronise, the median of three after a warm-up pass
  loop      the old loop, host clock ending in a synchronise, the median of three after a warm-up pass
env-steps/s count the episode lengths.  Every case also checks that the batched summaries equal the loop's.  At P = 1
the batched launch is timed against evaluate_policy alone, alternating the two.  One JSON line per case to --out,
with the GPU's name and power limit."""
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
from ppo_car_b200.evaluate import evaluate_policy, evaluate_population, load_checkpoint  # noqa: E402
from ppo_car_b200.population import Population  # noqa: E402
from ppo_car_b200.train_ppo import parse_args as train_args, train  # noqa: E402

SIZES = (1, 8, 32, 128)
EPISODES = 1024


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                              "-i", "0"], capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.TimeoutExpired):
        out = ""
    return {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": out}


def make_population(kind, P, trained, dev):
    pop = Population(list(range(P)), 1, device=dev)
    with torch.no_grad():
        for p in range(P):
            if kind == "trained" or (kind == "mixed" and p % 2 == 1):
                for dst, src in zip(pop.params[:4], trained):
                    dst[p].copy_(src)
    return pop


def events_per_call(fn, min_s=0.3):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    fn()                                                        # warm-up
    torch.cuda.synchronize()
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    reps = max(1, min(50, math.ceil(min_s / max(e0.elapsed_time(e1) / 1e3, 1e-6))))
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / 1e3 / reps, reps


def batched_with_summaries(env, pop, greedy):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    res = evaluate_population(env, pop.params[:4], EPISODES, greedy=greedy, seeds=pop.seeds)
    sums = torch.stack([r.sums() for r in res]).cpu()
    out = [r.summary(s) for r, s in zip(res, sums)]
    torch.cuda.synchronize()
    return time.perf_counter() - t0, out


def loop(env, pop, greedy):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = []
    for p in range(pop.P):
        res = evaluate_policy(env, pop.member_actor(p), EPISODES, greedy=greedy, seed=pop.seeds[p])
        out.append(res.summary())
    torch.cuda.synchronize()
    return time.perf_counter() - t0, out


def main():
    p = argparse.ArgumentParser()
    p.add_argument("--out", default=os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))),
                                                 "profiles", "r3_population_eval.jsonl"))
    p.add_argument("--sizes", default=",".join(map(str, SIZES)))
    args = p.parse_args()
    sizes = [int(x) for x in args.sizes.split(",")]
    info = gpu_info()
    dev = torch.device("cuda", 0)
    with tempfile.TemporaryDirectory() as d:
        train(train_args(["--track", "big_track", "--n-envs", "24", "--fused-rollout", "--fused-update",
                          "--checkpoint-dir", d, "--run-name", "readme"]))
        actor = load_checkpoint(os.path.join(d, "readme", "model.dat")).actor
    trained = [actor[0].weight.detach().to(dev), actor[0].bias.detach().to(dev), actor[2].weight.detach().to(dev),
               actor[2].bias.detach().to(dev)]
    env = ppo_car_b200.VecCarEnv(1, ppo_car_b200.builtin_track("big_track"), device=dev)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        for kind in ("fresh", "trained", "mixed"):
            for greedy in (False, True):
                for P in sizes:
                    if kind == "mixed" and P < 8:
                        continue
                    pop = make_population(kind, P, trained, dev)
                    call = lambda: evaluate_population(env, pop.params[:4], EPISODES, greedy=greedy, seeds=pop.seeds)
                    kernel_s, reps = events_per_call(call)
                    steps = sum(r.length.sum().item() for r in call())
                    batched_with_summaries(env, pop, greedy)                    # warm-up
                    bs = [batched_with_summaries(env, pop, greedy) for _ in range(3)]
                    loop(env, pop, greedy)                                      # warm-up
                    lp = [loop(env, pop, greedy) for _ in range(3)]
                    bs_s, b_sum = sorted(bs, key=lambda x: x[0])[1]             # the median of three
                    loop_s, l_sum = sorted(lp, key=lambda x: x[0])[1]
                    rec = {"population": kind, "greedy": greedy, "P": P, "episodes_per_member": EPISODES,
                           "track": "big_track", **info, "env_steps": steps, "mean_length": steps / (P * EPISODES),
                           "batched_reps": reps, "batched_s": kernel_s, "batched_env_steps_per_s": steps / kernel_s,
                           "batched_with_summaries_s": bs_s, "loop_s": loop_s, "loop_env_steps_per_s": steps / loop_s,
                           "speedup_batched_vs_loop": loop_s / kernel_s, "speedup_eval_epoch": loop_s / bs_s,
                           "summaries_identical": b_sum == l_sum}
                    if P == 1:                                                  # the batched launch at P = 1
                        actor1 = pop.member_actor(0)
                        single = lambda: evaluate_policy(env, actor1, EPISODES, greedy=greedy, seed=pop.seeds[0])
                        pairs = [(events_per_call(single, 0.15)[0], events_per_call(call, 0.15)[0]) for _ in range(3)]
                        rec["p1_single_s"] = [a for a, _ in pairs]
                        rec["p1_batched_s"] = [b for _, b in pairs]
                    print(json.dumps(rec), flush=True)
                    fh.write(json.dumps(rec) + "\n")
    env.close()


if __name__ == "__main__":
    main()
