#!/usr/bin/env python
"""Time-limit bootstrapping (--bootstrap-truncated): what the final-observation slots cost in the fused rollouts, what
the critic pass plus the bootstrapping scan cost against the plain GAE scan, and what the flag does to learning.

  rollout    k_policy_rollout_tc3 at 32,768 environments x 1,024 steps and 1,048,576 x 128 steps, and
             k_policy_rollout_warp at 24 x 1,024 (big_track, an untrained policy, start time steps spread over 0..999
             so that truncations happen at the steady-state rate), with and without slots, alternating in one process,
             CUDA events per launch; `spread` is (max - min) / median of the launches without slots: the run-to-run noise
             the slots are compared against
  gae        carenv_final_values + gae_reverse_scan_boot against gae_reverse_scan at [1024, 65536] and [1024, 262144]
             (two slots per column, one used), CUDA events, median of 20 after a warm-up
  learning   population --track big_track --n-envs 24 --seeds 0-7, 200 epochs, with and without the flag; every
             member's final actor scored on 1,024 greedy and 1,024 sampled episodes (evaluate_policy): mean return,
             truncation rate, laps.  Reported, not asserted.

One JSON line per measurement to --out (and stdout), each with the GPU's name and power limit read in the same run."""
import argparse
import json
import os
import statistics
import sys
import tempfile

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "benchmarks"))
import ppo_car_b200  # noqa: E402
from population import gpu_info, timed  # noqa: E402  (benchmarks/population.py)
from ppo_car_b200.train_ppo import ActorCritic  # noqa: E402


def rollout_case(kernel, n, T, reps):
    dev = torch.device("cuda")
    path = ppo_car_b200.builtin_track("big_track")
    env = ppo_car_b200.VecCarEnv(n, path, reward_scaling=0.1, float_flags=True)
    torch.manual_seed(0)
    net = ActorCritic(18, 9).to(dev)
    obs0 = env.reset()[0].clone()
    g = torch.Generator(device="cuda").manual_seed(1)
    env.ints[:, 1] = torch.randint(0, 1000, (n,), generator=g, device="cuda", dtype=torch.int32)
    snap = [t.clone() for t in (env.pos, env.vel, env.ints)]
    bufs = {s: ppo_car_b200.Buffer((18,), T, n, dev, bootstrap_truncated=s) for s in (False, True)}
    packed = ppo_car_b200.pack_policy_weights_tc(net.actor, net.critic)
    last_val = torch.empty(n, device=dev)
    times = {False: [], True: []}
    used = 0
    for r in range(reps + 1):
        for slots in (False, True):
            for dst, src in zip((env.pos, env.vel, env.ints), snap):
                dst.copy_(src)
            state = [obs0.clone(), torch.zeros(n, device=dev), torch.zeros(n, device=dev)]
            buf = bufs[slots]
            if kernel == "warp":
                fn = lambda: ppo_car_b200.fused_rollout_warp(env, net.actor, net.critic, buf, *state, seed=0, step0=0,
                                                             last_val=last_val)
            else:
                fn = lambda: ppo_car_b200.fused_rollout(env, packed, buf, *state, seed=0, step0=0, last_val=last_val)
            ms = timed(fn)
            if r > 0:                                        # launch 0 of each warms up
                times[slots].append(ms)
            if slots:
                used = int((buf.final_row_buf >= 0).sum())
    env.close()
    med = {s: statistics.median(v) for s, v in times.items()}
    return {"what": "rollout", "kernel": kernel, "envs": n, "steps": T, "reps": reps,
            "ms_plain": med[False], "ms_slots": med[True], "slots_over_plain": med[True] / med[False] - 1.0,
            "spread": (max(times[False]) - min(times[False])) / med[False], "ms_plain_all": times[False],
            "ms_slots_all": times[True], "truncations": used}


def gae_case(T, N):
    from ppo_car_b200.buffer import final_values

    dev = torch.device("cuda")
    g = torch.Generator(device="cuda").manual_seed(T + N)
    u = lambda *s: torch.rand(s, generator=g, device=dev)
    rew, val = u(T, N), torch.randn((T, N), generator=g, device=dev)
    term, trunc = (u(T, N) < 0.002).float(), (u(T, N) < 0.002).float()
    lv, lt, lu = torch.randn(N, generator=g, device=dev), torch.zeros(N, device=dev), torch.zeros(N, device=dev)
    S = 2
    fo = torch.rand((S, N, 18), generator=g, device=dev)
    fr = torch.full((S, N), -1, dtype=torch.int32, device=dev)
    fr[0] = torch.randint(0, T, (N,), generator=g, device=dev, dtype=torch.int32)
    boot = torch.empty((T, N), device=dev)
    adv, ret = torch.empty_like(rew), torch.empty_like(rew)
    torch.manual_seed(0)
    critic = ActorCritic(18, 9).to(dev).critic
    plain = lambda: ppo_car_b200.gae_reverse_scan(rew, val, term, trunc, lv, lt, lu, adv_out=adv, ret_out=ret)
    crit = lambda: final_values(critic, fo, fr, boot)
    scan = lambda: ppo_car_b200.gae_reverse_scan(rew, val, term, trunc, lv, lt, lu, adv_out=adv, ret_out=ret,
                                                 boot=boot)
    both = lambda: (crit(), scan())
    out = {}
    for name, fn in (("plain", plain), ("critic", crit), ("boot_scan", scan), ("critic_plus_boot_scan", both)):
        fn()
        out[name] = statistics.median(timed(fn) for _ in range(20))
    return {"what": "gae", "T": T, "N": N, "slots": S, **{f"ms_{k}": v for k, v in out.items()},
            "overhead": out["critic_plus_boot_scan"] / out["plain"] - 1.0}


def learning_case(flag, epochs):
    from ppo_car_b200.evaluate import evaluate_policy, load_checkpoint
    from ppo_car_b200.population import parse_args, train_population

    with tempfile.TemporaryDirectory() as d:
        argv = ["--track", "big_track", "--n-envs", "24", "--seeds", "0-7", "--n-epochs", str(epochs),
                "--checkpoint-dir", d, "--run-name", "bt"] + (["--bootstrap-truncated"] if flag else [])
        out = train_population(parse_args(argv))
        env = ppo_car_b200.VecCarEnv(1, ppo_car_b200.builtin_track("big_track"), device="cuda")
        members = []
        for p in range(8):
            actor = load_checkpoint(os.path.join(d, "bt", f"member_{p}", "model.dat")).cuda().actor
            rec = {"member": p, "final_avg_reward": out["final"][p]["avg_reward"]}
            for greedy in (True, False):
                s = evaluate_policy(env, actor, 1024, greedy=greedy, seed=p).summary()
                rec["greedy" if greedy else "sampled"] = {k: s[k] for k in ("mean_return", "truncation_rate",
                                                                            "crash_rate", "mean_laps")}
            members.append(rec)
        env.close()
    mean = lambda mode, k: statistics.mean(m[mode][k] for m in members)
    return {"what": "learning", "bootstrap_truncated": flag, "epochs": epochs, "members": members,
            **{f"{mode}_{k}_mean": mean(mode, k) for mode in ("greedy", "sampled")
               for k in ("mean_return", "truncation_rate", "mean_laps")}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_bootstrap_truncated.jsonl"))
    ap.add_argument("--reps", type=int, default=6)
    ap.add_argument("--epochs", type=int, default=200)
    ap.add_argument("--skip-learning", action="store_true")
    a = ap.parse_args()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    info = gpu_info()

    def emit(rec):
        rec.update(info)
        line = json.dumps(rec)
        print(line, flush=True)
        with open(a.out, "a") as fh:
            fh.write(line + "\n")

    for kernel, n, T in (("tc3", 32768, 1024), ("tc3", 1048576, 128), ("warp", 24, 1024)):
        emit(rollout_case(kernel, n, T, a.reps))
        torch.cuda.empty_cache()
    for T, N in ((1024, 65536), (1024, 262144)):
        emit(gae_case(T, N))
    if not a.skip_learning:
        for flag in (False, True):
            emit(learning_case(flag, a.epochs))


if __name__ == "__main__":
    main()
