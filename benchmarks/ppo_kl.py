#!/usr/bin/env python
"""Cost of the PPO divergence statistics in the one-launch epoch kernels: k_ppo_epoch<8> against
k_ppo_epoch<8, true> (carenv_ppo_epoch vs carenv_ppo_epoch_kl at target +inf, so both apply all 80 updates), and
k_ppo_epoch_pop<false> against k_ppo_epoch_pop<true> at P = 8, 32, 128.

Each timing is CUDA-event time of one 80-update epoch of 512-sample minibatches (the README schedule: train_iters 40
x 2 minibatches) on 24 x 1,024 = 24,576 samples per member, reported per update; the two variants alternate, 3 warm-up
and 20 timed epochs each, median kept.  The working set (a few MB) stays in L2, as in training.  One JSON line per
measurement to --out (and stdout) with the GPU's name and power limit read in the same run.

    python benchmarks/ppo_kl.py --out profiles/r3_ppo_kl.jsonl
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from ppo_car_b200 import population as popmod  # noqa: E402
from ppo_car_b200.ppo_update import FusedPPOUpdate  # noqa: E402
from ppo_car_b200.train_ppo import ActorCritic  # noqa: E402

N_SAMPLES, B, UPDATES = 24 * 1024, 512, 80


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                              "-i", "0"], capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.TimeoutExpired):
        out = ""
    return {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": out}


def timed(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b)


def data(M, dev, seed=0):
    g = torch.Generator(device=dev).manual_seed(seed)
    obs = torch.rand((M, 18), device=dev, generator=g)
    act = torch.randint(0, 9, (M,), device=dev, generator=g).float()
    old = torch.full((M,), -2.2, device=dev) + torch.randn(M, device=dev, generator=g) * 0.1
    adv, ret = torch.randn(M, device=dev, generator=g), torch.randn(M, device=dev, generator=g)
    return obs, act, old, adv, ret


def alternate(run_a, run_b, warm=3, reps=20):
    for _ in range(warm):
        run_a(); run_b()
    ta, tb = [], []
    for _ in range(reps):
        ta.append(timed(run_a))
        tb.append(timed(run_b))
    return statistics.median(ta), statistics.median(tb), ta, tb


def single(dev):
    torch.manual_seed(0)
    obs, act, old, adv, ret = data(N_SAMPLES, dev)
    nets = [ActorCritic(18, 9).to(dev) for _ in range(2)]
    nets[1].load_state_dict(nets[0].state_dict())
    # a tiny learning rate keeps the policy near its start over the many timed epochs
    ups = [FusedPPOUpdate(n.actor, n.critic, B, lr=1e-6) for n in nets]
    idx = torch.randint(0, N_SAMPLES, (UPDATES, B), device=dev)
    ma, mb, ta, tb = alternate(lambda: ups[0].run_epoch(obs, idx, act, old, adv, ret),
                               lambda: ups[1].run_epoch(obs, idx, act, old, adv, ret, target_kl=float("inf")))
    ups[0].check_epoch(); ups[1].check_epoch()
    same = all(torch.equal(p, q) for p, q in zip(ups[0].params, ups[1].params))
    return {"what": "k_ppo_epoch", "gpus": 1, "B": B, "updates": UPDATES, "us_per_update_plain": 1e3 * ma / UPDATES,
            "us_per_update_kl": 1e3 * mb / UPDATES, "kl_over_plain": mb / ma,
            "spread_plain_ms": [min(ta), max(ta)], "spread_kl_ms": [min(tb), max(tb)], "same_bits": same}


def population(P, dev):
    pops = [popmod.Population(list(range(P)), 24, {"learning_rate": 1e-6}, dev) for _ in range(2)]
    ups = [popmod.PopulationPPOUpdate(p, B) for p in pops]
    obs, act, old, adv, ret = data(N_SAMPLES * P, dev, seed=1)
    idx = torch.randint(0, N_SAMPLES * P, (P, UPDATES, B), device=dev)
    ma, mb, ta, tb = alternate(lambda: ups[0].launch(obs, idx, act, old, adv, ret),
                               lambda: ups[1].launch(obs, idx, act, old, adv, ret, target_kl=float("inf")),
                               warm=2, reps=8 if P >= 128 else 12)
    same = all(torch.equal(p, q) for p, q in zip(pops[0].params, pops[1].params))
    return {"what": "k_ppo_epoch_pop", "P": P, "B": B, "updates": UPDATES,
            "us_per_update_plain": 1e3 * ma / UPDATES, "us_per_update_kl": 1e3 * mb / UPDATES, "kl_over_plain": mb / ma,
            "spread_plain_ms": [min(ta), max(ta)], "spread_kl_ms": [min(tb), max(tb)], "same_bits": same}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--pop", default="8,32,128")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    dev = torch.device("cuda", 0)
    info = gpu_info()
    rows = [single(dev)] + [population(int(P), dev) for P in args.pop.split(",") if P]
    for r in rows:
        line = json.dumps({**r, **info})
        print(line, flush=True)
        if args.out:
            os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
            with open(args.out, "a") as fh:
                fh.write(line + "\n")


if __name__ == "__main__":
    main()
