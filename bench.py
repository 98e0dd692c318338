#!/usr/bin/env python
"""bench.py — CarEnv env-steps/sec (BASELINE.json metric) on N B200s of one node.

    python bench.py [--gpus N] [--steps K] [--warmup W]            # this repository's CUDA path
    python bench.py --impl reference [--gpus N] [--steps K] ...    # the reference's own CPU implementation
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload (config.workload): BASELINE.json configs[3] — tracks/big_track.json, 1,048,576
environments in total, i.i.d. uniform random actions, sharded over the N ranks by contiguous env
ranges with no data-path collective (strong scaling: the total is fixed).  One timed "step" is
`launches` back-to-back `carenv_rollout` launches per rank, each advancing every local environment
by `chunk` CarEnv steps and writing the observation, reward and both flags of every one of them to
HBM (default 1 x 256 env steps per environment per bench step, so that K = 20 steps keep the GPU busy
for about half a second and the clock samples are taken under load; a launch has a start-up transient
of about 25 us per wave of resident blocks — all warps begin in the same phase of the step and
compete for the FP64/XU pipes until they drift apart, benchmarks/sweep_launch.py — so short launches
such as 8 x 32 measure 2-18 % less, depending on the shard size).

  value     env-steps/s with actions already resident in HBM (device timed, CUDA events, max over ranks)
  e2e       env-steps/s through the reference-facing API VecCarEnv.step(numpy int64 actions) -> numpy
            results in the reference's dtypes (float32 obs, float64 rewards, bool flags, int info):
            host->device copy of the actions and device->host copy of observation + one 16-byte
            record per env from/to pinned memory inside the timed region, every step; `bound_gbs` is
            the pinned device->host rate all ranks reach copying at the same time, measured in the
            same run (the PCIe ceiling of this path)
  roofline  the step kernel against the FP32 pipe (SURVEY §8d: 5,286 algorithmic flop per env-step on
            big_track; nominal peak 148 SM x 128 lanes x 2 x sm_max_mhz, and an FFMA probe measured in
            the same run) plus its algorithmic HBM bytes against MEASURED_PEAKS.json
  cpu_baseline  the UNMODIFIED reference CarEnv (oracle/_ref: lib/car_env.py copied byte for byte by
            oracle/make_ref.py, imported through two inert stubs for gymnasium / pygame) on the host
            cores, one process per core, on a bounded sample; kind "reference".  The oracle port's rate
            is reported beside it (`port_value`).  Without oracle/_ref: the port, kind "port".
  configs   BASELINE.json's other configurations, measured after the timed region on rank 0:
            config 2 (24 envs x 1024 steps), config 3 (65,536 envs x 1024 steps rollout + GAE), the README
            training run and the fused policy + env rollout at 1 M envs (the callers of the hot path) and, at
            --gpus 8, config 5 (PPO loop, 262,144 envs: fused rollout, GAE kernel, all minibatch updates of an
            epoch in one launch with the gradient all-reduce over NVLink peer memory inside the kernel)

    python bench.py ... --dump-outputs DIR

writes, after the timed steps, the output buffers of the last launch of the last timed step (obs, reward, terminated,
truncated: what VecCarEnv.rollout hands its caller) as DIR/<name>.npy in float32, [steps per launch, DUMP_ENVS(, 18)],
for the global environment ids np.sort(np.random.default_rng(0).choice(envs, DUMP_ENVS, replace=False)) (and a
seeded sample of the rows when the launch is too long for DUMP_BYTES).  Actions and resets are seeded, so two builds
run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import contextlib
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

TOTAL_ENVS = 1_048_576
TRACK = "big_track"
N_SEG = 24
FLOP_PER_ENV_STEP = 18 * (12 * N_SEG + 4) + 30          # SURVEY §8(d): 5,286
# algorithmic bytes per env-step of the rollout launch (state stays in registers between steps):
# action u8 1 + obs 72 + reward 4 + term 1 + trunc 1; the 48 B state is read and written once per launch
BYTES_PER_ENV_STEP = 1 + 72 + 4 + 1 + 1
STATE_BYTES = 48
METRIC = "CarEnv env-steps/sec"
DUMP_ENVS = 2048                                         # --dump-outputs: sampled environments (all rows of a 256-step
DUMP_BYTES = 64 << 20                                    # launch: 44 MB) and the cap on all files together


# ----------------------------------------------------------------------------- CPU baseline
# Workers run either the UNMODIFIED reference CarEnv (oracle/_ref, kind "reference") or the oracle port (kind "port").
_W_ENV = None
_W_KIND = None


def _w_init(track_path, kind):
    global _W_ENV, _W_KIND
    sys.path.insert(0, ROOT)
    _W_KIND = kind
    if kind == "reference":
        from oracle.ref_import import import_reference

        CarEnv, _ = import_reference()
        _W_ENV = CarEnv(track_path=track_path)
        _W_ENV.reset(options={"track_path": track_path})
    else:
        from oracle.carenv_port import PortCarEnv

        _W_ENV = PortCarEnv(track_path)
        _W_ENV.reset()


def _w_run(args):
    seed, n_steps = args
    import numpy as np

    rng = np.random.default_rng(seed)
    acts = rng.integers(0, 9, size=n_steps)
    env = _W_ENV
    for a in acts:
        _, _, te, tr, _ = env.step(int(a))
        if te or tr:
            env.reset()                       # same-step autoreset (gymnasium AsyncVectorEnv worker)
    return n_steps


def reference_kind_and_track():
    """("reference", path inside oracle/_ref) when the unmodified reference files travelled with the repo, else
    ("port", the package's copy of the track)."""
    import ppo_car_b200.track as trk
    from oracle import ref_import

    root = ref_import.reference_root(prefer_copy=True)
    if root is not None:
        return "reference", os.path.join(root, "tracks", TRACK + ".json")
    return "port", trk.builtin_track(TRACK)


class CpuPool:
    """The reference's CPU path, one process per host core (what AsyncVectorEnv does, minus the pipes)."""

    def __init__(self, track_path, kind, cores=None):
        import multiprocessing as mp

        self.kind = kind
        self.cores = cores or min(os.cpu_count() or 1, 128)
        self.pool = mp.get_context("fork").Pool(self.cores, initializer=_w_init, initargs=(track_path, kind))
        self.seed = 0

    def run(self, steps_per_env):
        t0 = time.perf_counter()
        tasks = [(self.seed + i, steps_per_env) for i in range(self.cores)]
        self.seed += self.cores
        done = sum(self.pool.map(_w_run, tasks, chunksize=1))
        return done, time.perf_counter() - t0

    def close(self):
        self.pool.close()
        self.pool.join()


def _timed_sample(kind, path, target_seconds):
    pool = CpuPool(path, kind)
    try:
        pool.run(8)                                            # warm-up / calibration
        n, dt = pool.run(24)
        per_env = max(24, int(24 * target_seconds / max(dt, 1e-3)))
        n, dt = pool.run(per_env)
    finally:
        pool.close()
    return n / dt, pool.cores, per_env, dt


def cpu_baseline(target_seconds=12.0):
    import ppo_car_b200.track as trk

    kind, path = reference_kind_and_track()
    val, cores, per_env, dt = _timed_sample(kind, path, target_seconds)
    what = ("the UNMODIFIED reference lib/car_env.py (oracle/_ref, stub gymnasium / pygame), CarEnv.step + reset on done"
            if kind == "reference" else "oracle/carenv_port.py (Python restatement of lib/car_env.py)")
    out = {"value": val, "unit": "env-steps/s", "cores": cores, "kind": kind,
           "sample": f"{cores} envs x {per_env} steps, big_track.json, uniform random actions, {what}, "
                     f"one process per core, {dt:.1f} s"}
    if kind == "reference":                                    # the port beside it (a faster restatement)
        pval, _, pper, pdt = _timed_sample("port", trk.builtin_track(TRACK), 4.0)
        out["port_value"] = pval
        out["port_sample"] = f"{cores} envs x {pper} steps, oracle/carenv_port.py, {pdt:.1f} s"
    return out


# ----------------------------------------------------------------------------- clocks
class ClockSampler(threading.Thread):
    def __init__(self, index, period=0.01):
        super().__init__(daemon=True)
        self.index, self.period, self.samples, self.reasons, self.max_mhz = index, period, [], set(), None
        self._stop_evt = threading.Event()
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
                 nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap",
                 nv.nvmlClocksThrottleReasonHwPowerBrakeSlowdown: "hw_power_brake"}
        while not self._stop_evt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop_evt.wait(self.period)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=2)
        s = sorted(self.samples)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


# ----------------------------------------------------------------------------- reference arm
def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    kind, path = reference_kind_and_track()
    pool = CpuPool(path, kind)
    per_env = 32 if kind == "reference" else 96              # env-steps per worker per timed "step" (~0.15 s)
    try:
        for _ in range(max(args.warmup, 1)):
            pool.run(per_env)
        n_tot, t_tot = 0, 0.0
        for _ in range(args.steps):
            n, dt = pool.run(per_env)
            n_tot += n
            t_tot += dt
    finally:
        pool.close()
    val = n_tot / t_tot
    what = ("the UNMODIFIED reference lib/car_env.py from oracle/_ref (byte-for-byte copy made by oracle/make_ref.py, "
            "imported through inert gymnasium / pygame stubs): CarEnv.step, CarEnv.reset on done"
            if kind == "reference" else
            "oracle/carenv_port.py (Python restatement of lib/car_env.py; oracle/_ref is absent on this box)")
    sample = (f"{pool.cores} envs x {per_env} env-steps per step, big_track.json, uniform random actions, {what}, "
              "one process per host core")
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "env-steps/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t_tot / args.steps,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"tracks/{TRACK}.json, uniform random actions, same-step autoreset; "
                                   f"bounded sample of the {TOTAL_ENVS}-env workload: {sample}"},
            "cpu_baseline": {"value": val, "unit": "env-steps/s", "cores": pool.cores, "kind": kind, "sample": sample},
            "e2e": {"value": val, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)
    return 0


# ----------------------------------------------------------------------------- our arm
def kernel_source_hash():
    import hashlib

    hsh = hashlib.sha256()
    d = os.path.join(ROOT, "ppo_car_b200", "csrc")
    # the files the step kernels are compiled from (the policy / PPO kernels live in policy_*.cuh, ppo_update.cuh,
    # tc_mlp.cuh and do not enter k_rollout* machine code)
    for f in ("carenv_core.cuh", "carenv_tables.h", "carenv_kernels.cu"):
        hsh.update(open(os.path.join(d, f), "rb").read())
    return hsh.hexdigest()


def other_configs(dev, world):
    """BASELINE.json configs 2 and 3 on this rank's GPU (rank 0, after the timed region), CUDA-event timed."""
    import torch

    import ppo_car_b200

    track = ppo_car_b200.builtin_track(TRACK)
    out = {}

    def timed(fn, reps):
        fn()
        torch.cuda.synchronize()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(reps + 1)]
        ev[0].record()
        for i in range(reps):
            fn()
            ev[i + 1].record()
        torch.cuda.synchronize()
        ms = sorted(ev[i].elapsed_time(ev[i + 1]) for i in range(reps))
        return ms[len(ms) // 2]

    # config 2: 24 envs x 1024 steps (README training shape): warp-per-environment kernel, one launch
    g = torch.Generator(device=dev).manual_seed(2)
    env = ppo_car_b200.VecCarEnv(24, track, device=dev)
    env.reset()
    a = torch.randint(0, 9, (1024, 24), generator=g, device=dev, dtype=torch.uint8)
    ms = timed(lambda: env.rollout(a), 10)
    out["config2"] = {"workload": "big_track.json, 24 envs x 1024 steps, one launch (k_rollout_warp)", "ms": ms,
                      "env_steps_per_s": 24 * 1024 / (ms * 1e-3), "us_per_step": ms * 1e3 / 1024}
    del env
    # config 3: 65,536 envs x 1024 steps rollout (obs 4.8 GB written) + GAE over the [1024, 65536] buffer
    n, T = 65536, 1024
    env = ppo_car_b200.VecCarEnv(n, track, device=dev, float_flags=True)
    env.reset()
    a = torch.randint(0, 9, (T, n), generator=g, device=dev, dtype=torch.uint8)
    obs = torch.empty((T, n, 18), device=dev)
    rew, te, tr = (torch.empty((T, n), device=dev) for _ in range(3))
    val = torch.randn((T, n), generator=g, device=dev)
    adv, ret = torch.empty_like(val), torch.empty_like(val)
    lv, z = torch.randn(n, generator=g, device=dev), torch.zeros(n, device=dev)
    ms_r = timed(lambda: env.rollout(a, obs_out=obs, reward_out=rew, term_out=te, trunc_out=tr), 3)
    ms_g = timed(lambda: ppo_car_b200.gae_reverse_scan(rew, val, te, tr, lv, z, z, adv_out=adv, ret_out=ret), 10)
    out["config3"] = {"workload": "big_track.json, 65,536 envs x 1024 steps: rollout (obs/reward/flags f32 to HBM) + GAE",
                      "rollout_ms": ms_r, "rollout_env_steps_per_s": n * T / (ms_r * 1e-3), "gae_ms": ms_g,
                      "gae_gbs": n * T * 24 / (ms_g * 1e-3) / 1e9,
                      "env_steps_per_s": n * T / ((ms_r + ms_g) * 1e-3)}
    del env, obs, rew, te, tr, val, adv, ret, a
    # the callers of the hot path (SURVEY §8 f-1 / f-2), reported, never fatal: the reference's README training run
    # (24 envs x 1024 steps x 200 epochs, "about 35 minutes") and the fused policy + env rollout at the bench size
    try:
        import time

        from ppo_car_b200 import train_ppo

        targs = train_ppo.parse_args(["--track", TRACK, "--n-envs", "24", "--n-epochs", "200", "--fused-rollout",
                                      "--fused-update"])
        t0 = time.perf_counter()
        with contextlib.redirect_stdout(sys.stderr):         # the contract: ONE JSON line on stdout
            hist = train_ppo.train(targs)
        out["readme_training"] = {"workload": "PPO loop with the README hyper-parameters: big_track.json, 24 envs x 1024 "
                                              "steps x 200 epochs (fused warp-per-environment rollout, one update "
                                              "launch per epoch)", "wall_s": hist[-1]["wall_s"],   # the loop's own clock, as train.py logs it
                                  "wall_with_setup_s": time.perf_counter() - t0,
                                  "final_avg_reward": sum(h["avg_reward"] for h in hist[-10:]) / 10}
        from ppo_car_b200.train_ppo import ActorCritic

        torch.manual_seed(0)
        n, T = 1_048_576, 16
        net = ActorCritic(18, 9).to(dev)
        packed = ppo_car_b200.pack_policy_weights_tc(net.actor, net.critic)
        env = ppo_car_b200.VecCarEnv(n, track, device=dev, reward_scaling=0.1, float_flags=True, with_info=False)
        buf = ppo_car_b200.Buffer((18,), T, n, dev)
        cur = env.reset()[0].clone()
        z1, z2, lv = torch.zeros(n, device=dev), torch.zeros(n, device=dev), torch.empty(n, device=dev)
        step = [0]

        def fused():
            ppo_car_b200.fused_rollout(env, packed, buf, cur, z1, z2, seed=1, step0=step[0], last_val=lv)
            step[0] += T

        ms_f = timed(fused, 3)
        out["fused_rollout"] = {"workload": "policy forward (18-256-9 / 18-256-1, tcgen05) + sampling + env step + Buffer "
                                            "rows in one launch, 1,048,576 envs x 16 steps (k_policy_rollout_tc3)",
                                "ms": ms_f, "env_steps_per_s": n * T / (ms_f * 1e-3)}
    except Exception as exc:
        out["callers_error"] = repr(exc)[:300]
    return out


def config5(args):
    """BASELINE config 5 on 8 GPUs: the PPO loop of ppo_car_b200.train_ppo (README hyper-parameters, 262,144 envs in
    total, fused rollout + GAE kernel + all 80 minibatch updates of an epoch in one persistent launch whose gradient
    all-reduce runs over NVLink peer memory inside the kernel), 6 epochs, the first (lazy initialisation, IPC
    rendezvous) excluded.  Every rank takes part; rank 0 reports."""
    from ppo_car_b200 import train_ppo

    targs = train_ppo.parse_args(["--track", TRACK, "--n-envs", "262144", "--n-epochs", "6", "--fused-rollout",
                                  "--fused-update"])
    with contextlib.redirect_stdout(sys.stderr):             # the contract: ONE JSON line on stdout
        hist = train_ppo.train(targs)
    per_epoch = [hist[i]["wall_s"] - hist[i - 1]["wall_s"] for i in range(1, len(hist))]
    ms = 1e3 * sorted(per_epoch)[len(per_epoch) // 2]
    return {"workload": "PPO loop, README hyper-parameters, 262,144 envs over 8 GPUs x 1024 steps per epoch: fused "
                        "policy+env rollout, GAE, 80 minibatch updates in one persistent launch with the gradient "
                        "all-reduce over NVLink peer memory inside the kernel (carenv_ppo_epoch)",
            "epoch_ms": ms, "env_steps_per_s": 262144 * 1024 / (ms * 1e-3), "epochs_timed": len(per_epoch),
            "avg_reward_last": hist[-1]["avg_reward"]}


def dump_outputs(path, outs, total, lo, world, rank):
    """Save a seeded sample of this rank's output buffers `outs` (name -> [steps, envs on this rank, ...] CUDA tensor)
    as path/<name>.npy in float32 on rank 0: the same global environment ids and rows whatever the number of ranks."""
    import numpy as np
    import torch
    import torch.distributed as dist

    rng = np.random.default_rng(0)
    ids = np.sort(rng.choice(total, size=min(total, DUMP_ENVS), replace=False))
    first = next(iter(outs.values()))
    steps, n, dev = first.shape[0], first.shape[1], first.device
    row_bytes = len(ids) * 4 * sum(t[0, 0].numel() for t in outs.values())
    rows = None
    if steps * row_bytes > DUMP_BYTES:
        rows = np.sort(rng.choice(steps, size=max(1, DUMP_BYTES // row_bytes), replace=False))
    cols = torch.from_numpy(ids[(ids >= lo) & (ids < lo + n)] - lo).to(dev)
    part = {}
    for name, t in outs.items():
        s = t.index_select(1, cols)
        if rows is not None:
            s = s.index_select(0, torch.from_numpy(rows).to(dev))
        part[name] = s.float().cpu().numpy()
    parts = [part]
    if world > 1:                                       # shards are contiguous env ranges in rank order
        parts = [None] * world if rank == 0 else None
        dist.gather_object(part, parts, dst=0)
    if rank == 0:
        os.makedirs(path, exist_ok=True)
        for name in outs:
            np.save(os.path.join(path, name + ".npy"), np.concatenate([p[name] for p in parts], axis=1))


def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    import ppo_car_b200
    from ppo_car_b200 import _lib

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU path for --impl ours)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    from ppo_car_b200.shard import shard_range

    total = args.envs
    lo, hi = shard_range(total, world, rank)
    n = hi - lo
    chunk = args.chunk
    track = ppo_car_b200.builtin_track(TRACK)
    env = ppo_car_b200.VecCarEnv(n, track, device=dev, with_info=True)
    env.reset()
    # actions: shard-count-invariant stream (global env id decides the column), two alternating chunks
    gen = torch.Generator(device=dev).manual_seed(1234)
    n_act_bufs = 2
    acts = [torch.randint(0, 9, (chunk, total), generator=gen, device=dev, dtype=torch.uint8)[:, lo:hi].contiguous()
            for _ in range(n_act_bufs)]
    obs = torch.empty((chunk, n, 18), dtype=torch.float32, device=dev)
    rew = torch.empty((chunk, n), dtype=torch.float32, device=dev)
    term = torch.empty((chunk, n), dtype=torch.uint8, device=dev)
    trunc = torch.empty((chunk, n), dtype=torch.uint8, device=dev)

    launches = args.launches

    def one_step(i):
        for j in range(launches):
            env.rollout(acts[(i * launches + j) % n_act_bufs], obs_out=obs, reward_out=rew, term_out=term,
                        trunc_out=trunc)

    for i in range(args.warmup):
        one_step(i)
    barrier()
    sampler = ClockSampler(local, period=args.clock_period)
    sampler.start()
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    barrier()
    t_wall0 = time.perf_counter()
    evs[0].record()
    for i in range(args.steps):
        one_step(i)
        evs[i + 1].record()
    barrier()
    t_wall = time.perf_counter() - t_wall0
    clocks = sampler.stop()
    dev_ms = evs[0].elapsed_time(evs[-1])
    per_launch_ms = [evs[i].elapsed_time(evs[i + 1]) for i in range(args.steps)]
    t = torch.tensor([dev_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms_max = float(t.item())
    value = args.steps * launches * chunk * total / (dev_ms_max * 1e-3)
    slow = env.slow_path_counts()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"obs": obs, "reward": rew, "terminated": term, "truncated": trunc}, total, lo,
                     world, rank)

    # ---- e2e: reference-facing API with HOST buffers (numpy in, numpy out, the reference's dtypes), one env step per call
    e_steps = args.e2e_steps
    rng = np.random.default_rng(99 + rank)
    host_actions = [rng.integers(0, 9, size=n).astype(np.int64) for _ in range(4)]   # int64: what train.py:185 passes
    e2e_env = ppo_car_b200.VecCarEnv(n, track, device=dev)    # info = gates_passed / time_passed, as the reference
    e2e_env.reset()
    for i in range(3):
        e2e_env.step(host_actions[i % 4])
    barrier()
    t0 = time.perf_counter()
    sink = 0.0
    for i in range(e_steps):
        o, r, te, tr, info = e2e_env.step(host_actions[i % 4])
        sink += float(r[0])                       # the result is on the host (pinned buffer) when step() returns
    barrier()
    t_e2e = time.perf_counter() - t0
    assert r.dtype == np.float64 and te.dtype == np.bool_ and o.dtype == np.float32
    te2e = torch.tensor([t_e2e], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(te2e, op=dist.ReduceOp.MAX)
    e2e_value = e_steps * total / float(te2e.item())
    h2d = total * 1                               # uint8 actions (narrowed on the host before the copy)
    d2h = total * (72 + 16)                       # observation + one 16-byte record (reward, flags, info) per env
    del e2e_env
    # the ceiling of that path: pinned device->host copies of one step's results, ALL ranks copying at the same time
    pb = n * 88
    d_src = torch.empty(pb, dtype=torch.uint8, device=dev)
    h_dst = [torch.empty(pb, dtype=torch.uint8, pin_memory=True) for _ in range(2)]
    for i in range(2):
        h_dst[i].copy_(d_src, non_blocking=True)
    barrier()
    t0 = time.perf_counter()
    p_reps = 12
    for i in range(p_reps):
        h_dst[i % 2].copy_(d_src, non_blocking=True)
    torch.cuda.synchronize()
    t_probe = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
    barrier()
    if world > 1:
        dist.all_reduce(t_probe, op=dist.ReduceOp.MAX)
    bound_gbs = world * p_reps * pb / float(t_probe.item()) / 1e9
    del d_src, h_dst

    line = None
    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        hbm_src = "MEASURED_PEAKS.json hbm_gbs (measured copy)" if "hbm_gbs" in peaks else "fallback 6650 GB/s"
        sm_max = float(clocks.get("sm_max_mhz") or peaks.get("sm_max_mhz", 1965.0))
        fp32_nominal = 148 * 128 * 2 * sm_max * 1e6 / 1e12
        # FFMA probe, timed alone on this GPU
        L = _lib.lib()
        import ctypes as C

        scratch = torch.zeros(4, device=dev)
        st = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        blocks, iters = 148 * 8, 20000
        L.carenv_bench_ffma(blocks, 1000, C.c_void_p(scratch.data_ptr()), st)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        L.carenv_bench_ffma(blocks, iters, C.c_void_p(scratch.data_ptr()), st)
        e1.record()
        torch.cuda.synchronize()
        ffma_tflops = blocks * 256 * iters * 64 * 2 / (e0.elapsed_time(e1) * 1e-3) / 1e12

        launch_ms = sum(per_launch_ms) / len(per_launch_ms) / launches   # rank 0's average launch duration
        steps_per_launch = chunk * n
        achieved_tflops = steps_per_launch * FLOP_PER_ENV_STEP / (launch_ms * 1e-3) / 1e12
        bytes_per_launch = steps_per_launch * BYTES_PER_ENV_STEP + n * 2 * STATE_BYTES
        achieved_gbs = bytes_per_launch / (launch_ms * 1e-3) / 1e9
        # secondary kernel: GAE reverse scan at BASELINE config 3 size [1024, 65536] (HBM-bound, 24 B/element)
        Tg, Ng = 1024, 65536
        gg = torch.Generator(device=dev).manual_seed(7)
        g_rew = torch.rand((Tg, Ng), generator=gg, device=dev) * 1.4 - 0.3
        g_val = torch.randn((Tg, Ng), generator=gg, device=dev)
        g_term = (torch.rand((Tg, Ng), generator=gg, device=dev) < 0.004).float()
        g_trunc = (torch.rand((Tg, Ng), generator=gg, device=dev) < 0.001).float()
        g_lv, g_z = torch.randn(Ng, generator=gg, device=dev), torch.zeros(Ng, device=dev)
        g_adv, g_ret = torch.empty_like(g_rew), torch.empty_like(g_rew)
        for _ in range(3):
            ppo_car_b200.gae_reverse_scan(g_rew, g_val, g_term, g_trunc, g_lv, g_z, g_z, adv_out=g_adv, ret_out=g_ret)
        torch.cuda.synchronize()
        ge = [torch.cuda.Event(enable_timing=True) for _ in range(11)]
        ge[0].record()
        for i in range(10):
            ppo_car_b200.gae_reverse_scan(g_rew, g_val, g_term, g_trunc, g_lv, g_z, g_z, adv_out=g_adv, ret_out=g_ret)
            ge[i + 1].record()
        torch.cuda.synchronize()
        gae_ms = ge[0].elapsed_time(ge[-1]) / 10
        gae_gbs = Tg * Ng * 24 / (gae_ms * 1e-3) / 1e9
        del g_rew, g_val, g_term, g_trunc, g_adv, g_ret
        # measured DRAM bytes per env-step of the same kernel from the committed ncu capture — refused (null) when the
        # capture was taken from other kernel sources than the ones this library was built from
        traffic, traffic_note = None, "no ncu capture of the current kernel sources under profiles/"
        try:
            tr = json.load(open(os.path.join(ROOT, "profiles", "r2_traffic.json")))
            if tr.get("source_sha256") == kernel_source_hash():
                traffic = tr["dram_bytes_per_env_step"] * steps_per_launch
                traffic_note = (f"DRAM bytes per launch = ncu dram__bytes_read+write per env-step "
                                f"({tr['dram_bytes_per_env_step']:.2f}, profiles/r2_traffic.json, same kernel sources) x "
                                "env-steps per launch")
            else:
                traffic_note = "profiles/r2_traffic.json was captured from other kernel sources: refused"
        except Exception:
            pass
        # single-GPU side measurements: at N = 1 only (rank 0 would keep the other ranks waiting)
        configs = other_configs(dev, world) if (world == 1 and not args.no_configs) else None
        cpu = cpu_baseline() if (world == 1 and not args.no_cpu) else None
        line = {
            "metric": METRIC, "value": value, "unit": "env-steps/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dev_ms_max / args.steps, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32 ray casting, f64 state", "data": "synthetic",
            "config": {"workload": f"tracks/{TRACK}.json, {total} envs total ({n} per GPU), uniform random actions "
                                   f"resident in HBM, same-step autoreset, {launches} launches x {chunk} env steps per "
                                   "bench step; every env step writes obs[18] f32 + reward f32 + terminated/truncated "
                                   "u8 per env",
                       "envs_total": total, "envs_per_gpu": n, "steps_per_launch": chunk,
                       "launches_per_step": launches, "sharding": f"env{world}",
                       "cache": f"outputs per launch {obs.numel() * 4 / 1e6:.0f} MB > 126 MB L2 (no flush needed)"},
            "wall_s": t_wall,
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": "env-steps/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "api": "VecCarEnv.step(numpy int64 actions) -> numpy obs f32 / reward f64 / terminated, truncated "
                           "bool / info {gates_passed, time_passed} (the reference's dtypes)",
                    "steps": e_steps, "bound_gbs": bound_gbs, "achieved_gbs": e2e_value * 88 / 1e9,
                    "frac_of_bound": e2e_value * 88 / 1e9 / bound_gbs,
                    "bound_note": f"pinned D2H of {pb / 1e6:.1f} MB per rank x {world} ranks copying concurrently, "
                                  "measured in this run"},
            "gpu_launches": args.steps * launches,
            "roofline": {"bound": "fp32", "achieved": achieved_tflops, "peak": fp32_nominal, "unit": "TFLOP/s",
                         "frac": achieved_tflops / fp32_nominal, "traffic": traffic,
                         "traffic_note": traffic_note + f"; algorithmic bytes per launch = {bytes_per_launch}",
                         "kernel": ("k_rollout_tab_sliced<uint8,uint8,6>"      # the library's choice (launch_rollout_tab)
                                    if ((n + 31) // 32) // 148 >= 16 and chunk >= 4
                                    else "k_rollout_tab<uint8,uint8,6>"), "launch_ms": launch_ms,
                         "launch_ms_min": min(per_launch_ms) / launches, "launch_ms_max": max(per_launch_ms) / launches,
                         "flop_per_env_step": FLOP_PER_ENV_STEP,
                         "peak_source": f"nominal 148 SM x 128 lanes x 2 x {sm_max:.0f} MHz (MEASURED_PEAKS.json has no "
                                        "FP32 entry)",
                         "ffma_probe_tflops": ffma_tflops, "frac_of_ffma_probe": achieved_tflops / ffma_tflops},
            "roofline_hbm": {"bound": "hbm", "achieved": achieved_gbs, "peak": hbm_peak, "unit": "GB/s",
                             "frac": achieved_gbs / hbm_peak, "traffic": traffic, "bytes_per_env_step": BYTES_PER_ENV_STEP,
                             "peak_source": hbm_src},
            "gae": {"kernel": "k_gae", "shape": [Tg, Ng], "ms": gae_ms, "bound": "hbm", "achieved": gae_gbs,
                    "peak": hbm_peak, "unit": "GB/s", "frac": gae_gbs / hbm_peak, "bytes_per_element": 24,
                    "note": "inputs + outputs 1.6 GB > L2; 10 back-to-back launches, CUDA events"},
            "slow_path": {k: v for k, v in slow.items()},
            "configs": configs,
            "cpu_baseline": cpu,
        }
    if world == 8 and not args.no_configs:                     # BASELINE config 5 needs every rank
        try:
            c5 = config5(args)
        except Exception as exc:                               # reported, not fatal: the headline line stands
            c5 = {"error": repr(exc)[:300]}
        if rank == 0 and line is not None:
            line.setdefault("configs", {})
            line["configs"] = dict(line["configs"] or {}, config5=c5)
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--envs", type=int, default=TOTAL_ENVS, help="total environments over all GPUs")
    ap.add_argument("--chunk", type=int, default=256, help="env steps per rollout launch")
    ap.add_argument("--launches", type=int, default=1, help="rollout launches per timed bench step")
    ap.add_argument("--e2e-steps", type=int, default=20)
    ap.add_argument("--clock-period", type=float, default=0.01, help="seconds between NVML clock samples")
    ap.add_argument("--no-configs", action="store_true", help="skip BASELINE configs 2 / 3 / 5")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write a seeded sample of the outputs of the last launch of the last timed step to "
                         "DIR/<name>.npy (--impl ours)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours: the reference arm keeps no output buffers")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
