#!/usr/bin/env python
"""Populations of independent PPO members (ppo_car_b200.population) at the README shape: 24 environments per member,
1,024 steps, 80 minibatch updates of 512 (train_iters 40 x 2), big_track.

Per population size P in 1, 8, 32, 128, CUDA-event time per epoch (mean of 3 epochs after one warm-up epoch) of
  rollout_ms   carenv_policy_rollout_warp_pop (one launch for all members)
  gae_ms       Buffer.calculate_advantages over the [1024, 24 P] buffer
  update_ms    carenv_ppo_epoch_pop (one cluster launch for all members), and us_per_update = update_ms / 80
and member-epochs per second = P / (rollout + GAE + update).  Also:
  k_ppo_epoch at P = 1   FusedPPOUpdate.run_epoch (the single-policy cooperative kernel) on the same data
  sequential             8 x train_ppo --fused-rollout --fused-update, epoch 2 of each run (wall clock, including its
                         host work), against epoch 2 of train_population with the same 8 seeds
  tensor cores           P = 4 members x 32,768 environments: carenv_policy_rollout_tc_pop against one member's
                         fused_rollout at 32,768 environments
  resident clusters      cudaOccupancyMaxActiveClusters of the update kernel

One JSON line per measurement to --out (and stdout), each with the GPU's name and power limit read in the same run."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import ppo_car_b200  # noqa: E402
from ppo_car_b200 import _lib  # noqa: E402
from ppo_car_b200 import population as popmod  # noqa: E402
from ppo_car_b200.ppo_update import FusedPPOUpdate  # noqa: E402
from ppo_car_b200.train_ppo import ActorCritic  # noqa: E402

N_ENVS, T, B, UPDATES = 24, 1024, 512, 80


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


def population_epochs(P, n, dev, epochs=3):
    track = ppo_car_b200.builtin_track("big_track")
    pop = popmod.Population(list(range(P)), n, None, dev)
    N = pop.num_envs
    env = ppo_car_b200.VecCarEnv(N, track, device=dev, reward_scaling=0.1, float_flags=True, with_info=False)
    buf = ppo_car_b200.Buffer((18,), T, N, dev)
    upd = popmod.PopulationPPOUpdate(pop, B)
    cur = env.reset()[0].clone()
    z1, z2, lv = torch.zeros(N, device=dev), torch.zeros(N, device=dev), torch.empty(N, device=dev)
    res = {"rollout_ms": [], "gae_ms": [], "update_ms": []}
    data = {}
    for e in range(epochs + 1):
        r = timed(lambda: popmod.population_rollout(env, pop, buf, cur, z1, z2, step0=e * T, last_val=lv))
        g = timed(lambda: data.update(zip(("adv", "ret"), buf.calculate_advantages(lv.view(1, -1), z1.view(1, -1),
                                                                                    z2.view(1, -1)))))
        obs, act, _, logp = buf.get()
        idx = upd.draw_indices(T, UPDATES)
        u = timed(lambda: upd.launch(obs.view(-1, 18), idx, act.view(-1), logp.view(-1), data["adv"].view(-1),
                                     data["ret"].view(-1)))
        if e > 0:
            res["rollout_ms"].append(r); res["gae_ms"].append(g); res["update_ms"].append(u)
    out = {k: sum(v) / len(v) for k, v in res.items()}
    out["epoch_ms"] = out["rollout_ms"] + out["gae_ms"] + out["update_ms"]
    out["us_per_update"] = out["update_ms"] * 1000.0 / UPDATES
    out["member_epochs_per_s"] = P / out["epoch_ms"] * 1000.0
    return out, (buf, data, pop)


def single_epoch_kernel(dev, buf, data, pop):
    torch.manual_seed(0)
    net = ActorCritic(18, 9).to(dev)
    upd = FusedPPOUpdate(net.actor, net.critic, B, 3e-4)
    obs, act, logp = buf.obs_buf.view(-1, 18), buf.act_buf.view(-1), buf.logprob_buf.view(-1)
    idx = torch.randint(0, T * N_ENVS, (UPDATES, B), device=dev)
    ts = [timed(lambda: upd.run_epoch(obs, idx, act, logp, data["adv"].view(-1), data["ret"].view(-1)))
          for _ in range(4)][1:]
    return sum(ts) / len(ts) * 1000.0 / UPDATES


def sequential_vs_population(dev):
    from ppo_car_b200.train_ppo import parse_args, train

    base = ["--track", "big_track", "--n-envs", str(N_ENVS), "--n-epochs", "2"]
    seq = 0.0
    for s in range(8):
        h = train(parse_args(base + ["--seed", str(s), "--fused-rollout", "--fused-update"]))
        seq += h[1]["wall_s"] - h[0]["wall_s"]
    out = popmod.train_population(popmod.parse_args(base + ["--seeds", "0-7"]))
    walls = sorted({r["wall_s"] for r in out["history"]})
    return {"sequential_8_train_ppo_epoch_s": seq, "population_8_epoch_s": walls[1] - walls[0]}


def tensor_core_case(dev, P=4, n=32768, Tt=1024):
    track = ppo_car_b200.builtin_track("big_track")
    pop = popmod.Population(list(range(P)), n, None, dev)
    N = pop.num_envs
    env = ppo_car_b200.VecCarEnv(N, track, device=dev, reward_scaling=0.1, float_flags=True, with_info=False)
    buf = ppo_car_b200.Buffer((18,), Tt, N, dev)
    cur = env.reset()[0].clone()
    z1, z2, lv = torch.zeros(N, device=dev), torch.zeros(N, device=dev), torch.empty(N, device=dev)
    packed = torch.empty((P, _lib.lib().carenv_policy_weights_floats_tc()), device=dev)
    ts = [timed(lambda: popmod.population_rollout(env, pop, buf, cur, z1, z2, step0=e * Tt, last_val=lv,
                                                  packed=packed)) for e in range(3)][1:]
    env1 = ppo_car_b200.VecCarEnv(n, track, device=dev, reward_scaling=0.1, float_flags=True, with_info=False)
    buf1 = ppo_car_b200.Buffer((18,), Tt, n, dev)
    cur1 = env1.reset()[0].clone()
    y1, y2, lv1 = torch.zeros(n, device=dev), torch.zeros(n, device=dev), torch.empty(n, device=dev)
    net = ActorCritic(18, 9).to(dev)
    w = ppo_car_b200.pack_policy_weights_tc(net.actor, net.critic)
    t1 = [timed(lambda: ppo_car_b200.fused_rollout(env1, w, buf1, cur1, y1, y2, seed=0, step0=e * Tt, last_val=lv1))
          for e in range(3)][1:]
    return {"members": P, "envs_per_member": n, "steps": Tt, "population_rollout_ms": sum(ts) / len(ts),
            "single_member_rollout_ms": sum(t1) / len(t1)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--sizes", default="1,8,32,128")
    ap.add_argument("--epochs-only", action="store_true",
                    help="only the per-size epoch timings (for comparing builds with another -DCARENV_POP_CLUSTER)")
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    info = gpu_info()
    L = _lib.lib()
    lines = []

    def emit(rec):
        rec = {**rec, **info}
        lines.append(rec)
        print(json.dumps(rec), flush=True)

    nc = C.c_int(0)
    _lib.check(L.carenv_ppo_epoch_pop_resident_clusters(C.byref(nc)), "resident clusters")
    emit({"what": "resident_clusters", "cluster_size": L.carenv_ppo_epoch_pop_cluster_size(), "clusters": nc.value})
    for P in [int(x) for x in args.sizes.split(",")]:
        res, keep = population_epochs(P, N_ENVS, dev)
        emit({"what": "population_epoch", "members": P, "envs_per_member": N_ENVS, "steps": T, "updates": UPDATES,
              "batch": B, **res})
        if P == 1 and not args.epochs_only:
            emit({"what": "k_ppo_epoch_single", "members": 1, "us_per_update": single_epoch_kernel(dev, *keep)})
        del keep
        torch.cuda.empty_cache()
    if not args.epochs_only:
        emit({"what": "sequential_vs_population", "members": 8, **sequential_vs_population(dev)})
        emit({"what": "tensor_core_rollout", **tensor_core_case(dev)})
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.writelines(json.dumps(r) + "\n" for r in lines)


if __name__ == "__main__":
    main()
