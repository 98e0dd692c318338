"""How many segment pairs the culled table kernels evaluate per warp-step: the mechanism behind their speed-up.

Runs a bench-size launch (1,048,576 environments x 256 steps of uniform random actions from reset, as bench.py does),
then replays its final states through the candidate table on the host (tests/host_cull/cull.cpp, compiled into a
temporary directory) with the kernel's OR over each warp of 32 consecutive environments.  ``--spread`` starts from
states spread uniformly over the track's bounding box instead (warps then see most of the track).

    python benchmarks/cull_stats.py [--envs 1048576] [--steps 256] [--track big_track] [--spread] [--out x.jsonl]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import ppo_car_b200  # noqa: E402
from ppo_car_b200.track import load_track  # noqa: E402


def harness():
    d = tempfile.mkdtemp(prefix="cull_stats_")
    so = os.path.join(d, "libcull.so")
    subprocess.check_call(["g++", "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-Wno-unknown-pragmas", "-x", "c++",
                           "-o", so, os.path.join(ROOT, "tests", "host_cull", "cull.cpp"), "-lm", "-pthread"])
    return C.CDLL(so)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=1_048_576)
    ap.add_argument("--steps", type=int, default=256)
    ap.add_argument("--track", default="big_track")
    ap.add_argument("--spread", action="store_true")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    path = ppo_car_b200.builtin_track(args.track)
    tr = load_track(path)
    env = ppo_car_b200.VecCarEnv(args.envs, path)
    env.reset()
    if args.spread:
        w = np.asarray(tr.walls)
        rng = np.random.default_rng(0)
        xs, ys = np.concatenate([w[:, 0], w[:, 2]]), np.concatenate([w[:, 1], w[:, 3]])
        env.pos[:, 0] = torch.from_numpy(rng.uniform(xs.min(), xs.max(), args.envs))
        env.pos[:, 1] = torch.from_numpy(rng.uniform(ys.min(), ys.max(), args.envs))
        env.ints[:, 0] = torch.from_numpy(rng.integers(0, 72, args.envs).astype(np.int32))
    g = torch.Generator(device="cuda").manual_seed(1)
    acts = torch.randint(0, 9, (args.steps, args.envs), generator=g, device="cuda", dtype=torch.uint8)
    env.rollout(acts, store_obs=False)
    torch.cuda.synchronize()
    pos = env.pos.cpu().numpy()
    px, py = np.ascontiguousarray(pos[:, 0]), np.ascontiguousarray(pos[:, 1])
    k = np.ascontiguousarray(env.ints[:, 0].cpu().numpy())
    L = harness()
    walls, gates = np.ascontiguousarray(tr.walls), np.ascontiguousarray(tr.gates)
    kept = np.zeros((args.envs + 31) // 32, np.int32)
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    rc = L.cull_warp_pairs(p(walls), len(walls), p(gates), len(gates), C.c_double(tr.start[0]), C.c_double(tr.start[1]),
                           C.c_double(tr.angle), C.c_longlong(args.envs), p(px), p(py), p(k), p(kept))
    assert rc == 0, rc
    n_pairs = len(walls) // 2
    rec = {"what": "cull_stats", "track": args.track, "envs": args.envs, "steps": args.steps, "spread": args.spread,
           "pairs": n_pairs, "kept_per_warp_step_mean": float(kept.mean()),
           "kept_percentiles_10_50_90": [float(x) for x in np.percentile(kept, [10, 50, 90])],
           "skipped_per_warp_step_mean": float(n_pairs - kept.mean())}
    print(json.dumps(rec))
    if args.out:
        with open(args.out, "a") as fh:
            fh.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
