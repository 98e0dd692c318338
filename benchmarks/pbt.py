#!/usr/bin/env python
"""Population-based training (ppo_car_b200.pbt): what a round costs and what it does to the outcome.

Round cost, P in 8, 32, 128 members at the README shape (24 envs per member, 1,024 steps, 80 updates of 512,
big_track), against one population epoch (CUDA events per stage, mean of 3 epochs after a warm-up epoch, as
benchmarks/population.py).  For two sets of weights — the population after those 4 epochs ("early": episodes end in
crashes after a few hundred steps) and the README-trained actor in every member ("trained": about 840 steps):
  eval_ms      the round's evaluate_population call (1,024 sampled episodes per member), CUDA events
  fitness_ms   the call plus every member's sums and summaries, host clock ending in a synchronise
  pack_ms      Population.state_rows of every member: the local part of the torchrun exchange; the all-gather
               itself needs two GPUs and is not measured here
  copy_ms      copy_members of the round's floor(P / 4) pairs, CUDA events
  round_ms     pbt.pbt_round as train_population calls it (one rank), host clock ending in a synchronise
Each is the median of 5 after a warm-up; round_ms / (10 x epoch_ms) is the cost of --pbt-every 10.

Outcome (reported, not asserted; one run each): P = 32 members, learning rates 1e-4, 3e-4, 1e-3, 3e-3 x seeds 0-7,
200 epochs, without PBT and with --pbt-every 10 (default fraction and explore); the best and the median final greedy
evaluation return (1,024 episodes per member, --eval-every 200 --eval-greedy) and the wall time.

One JSON line per measurement to --out (and stdout), each with the GPU's name and power limit read in the same run."""
import argparse
import contextlib
import json
import os
import statistics
import sys
import tempfile
import time
from types import SimpleNamespace

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "benchmarks"))
import ppo_car_b200  # noqa: E402
import population as popbench  # noqa: E402  (benchmarks/population.py)
from ppo_car_b200 import pbt  # noqa: E402
from ppo_car_b200 import population as popmod  # noqa: E402
from ppo_car_b200.evaluate import evaluate_population, load_checkpoint  # noqa: E402
from ppo_car_b200.train_ppo import parse_args as train_args, train  # noqa: E402

EPISODES = 1024


def median_host(fn, reps=5):
    fn()
    ts = []
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        ts.append((time.perf_counter() - t0) * 1e3)
    return statistics.median(ts)


def median_events(fn, reps=5):
    fn()
    return statistics.median(popbench.timed(fn) for _ in range(reps))


def round_costs(pop, env):
    args = SimpleNamespace(eval_episodes=EPISODES, eval_greedy=False, pbt_seed=0, pbt_fraction=0.25)
    explore = ["learning_rate", "ent_coef"]
    call = lambda: evaluate_population(env, pop.params[:4], EPISODES, seeds=0)

    def fitness():
        res = call()
        sums = torch.stack([r.sums() for r in res]).cpu()
        return [r.summary(s)["mean_return"] for r, s in zip(res, sums)]

    dec = pbt.pbt_decisions(fitness(), 0.25, explore, torch.Generator().manual_seed(0))
    dst, src, fac = [d for d, _, _ in dec], [s for _, s, _ in dec], [f for _, _, f in dec]
    saved = [t.clone() for t in pop._state_tensors()]        # copy_members overwrites; keep the timed state fixed

    def copy():
        pop.copy_members(dst, src, fac)

    def restore():
        for t, s in zip(pop._state_tensors(), saved):
            t.copy_(s)

    gen = torch.Generator().manual_seed(0)
    out = {"eval_ms": median_events(call), "fitness_ms": median_host(fitness),
           "pack_ms": median_events(lambda: pop.state_rows(range(pop.P))), "copy_ms": median_events(copy),
           "round_ms": median_host(lambda: (restore(), pbt.pbt_round(pop, env, args, 0, 10, 0, [pop.P], gen, explore))),
           "replaced": len(dec),
           "mean_episode_length": sum(r.length.double().mean().item() for r in call()) / pop.P}
    restore()
    return out


def outcome(pbt_every):
    argv = ["--track", "big_track", "--n-envs", "24", "--seeds", "0-7", "--learning-rate", "1e-4,3e-4,1e-3,3e-3",
            "--n-epochs", "200", "--eval-every", "200", "--eval-greedy", "--eval-episodes", str(EPISODES),
            "--pbt-every", str(pbt_every)]
    t0 = time.perf_counter()
    with open(os.devnull, "w") as null, contextlib.redirect_stdout(null):
        out = popmod.train_population(popmod.parse_args(argv))
    wall = time.perf_counter() - t0
    rets = sorted(r["eval_return"] for r in out["final"])
    rec = {"what": "outcome", "members": 32, "pbt_every": pbt_every, "epochs": 200, "runs": 1,
           "best_greedy_return": rets[-1], "median_greedy_return": statistics.median(rets), "wall_s": wall}
    if pbt_every:
        rec["rounds"] = max(l["pbt_round"] for l in out["lineage"]) + 1
        rec["best_member_current_hparams"] = out["pbt_best"]["current_hparams"]
        best = max(out["final"], key=lambda r: r["eval_return"])
        rec["best_by_final_eval"] = {"member": best["member"], "initial_lr": best["hparams"]["learning_rate"],
                                     "ancestry": best["ancestry"]}
    else:
        best = max(out["final"], key=lambda r: r["eval_return"])
        rec["best_by_final_eval"] = {"member": best["member"], "initial_lr": best["hparams"]["learning_rate"]}
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--sizes", default="8,32,128")
    ap.add_argument("--skip-outcome", action="store_true")
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    info = popbench.gpu_info()
    lines = []

    def emit(rec):
        rec = {**rec, **info}
        lines.append(rec)
        print(json.dumps(rec), flush=True)

    with tempfile.TemporaryDirectory() as d, open(os.devnull, "w") as null, contextlib.redirect_stdout(null):
        train(train_args(["--track", "big_track", "--n-envs", "24", "--fused-rollout", "--fused-update",
                          "--checkpoint-dir", d, "--run-name", "readme"]))
        actor = load_checkpoint(os.path.join(d, "readme", "model.dat")).actor
    trained = [actor[0].weight, actor[0].bias, actor[2].weight, actor[2].bias]
    for P in [int(x) for x in args.sizes.split(",")]:
        epoch, (_, _, pop) = popbench.population_epochs(P, popbench.N_ENVS, dev)
        env = ppo_car_b200.VecCarEnv(1, ppo_car_b200.builtin_track("big_track"), device=dev)
        for weights in ("early", "trained"):
            if weights == "trained":
                with torch.no_grad():
                    for t, w in zip(pop.params[:4], trained):
                        t.copy_(w.detach().to(dev).expand_as(t))
            costs = round_costs(pop, env)
            emit({"what": "round_cost", "members": P, "weights": weights, "envs_per_member": popbench.N_ENVS,
                  "steps": popbench.T, "episodes_per_member": EPISODES, "epoch_ms": epoch["epoch_ms"], **costs,
                  "allgather_ms": "not measured (one GPU)",
                  "round_share_at_pbt_every_10": costs["round_ms"] / (costs["round_ms"] + 10 * epoch["epoch_ms"])})
        env.close()
        del pop
        torch.cuda.empty_cache()
    if not args.skip_outcome:
        for k in (0, 10):
            emit(outcome(k))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.writelines(json.dumps(r) + "\n" for r in lines)


if __name__ == "__main__":
    main()
