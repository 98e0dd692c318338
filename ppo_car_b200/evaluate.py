"""Policy evaluation on the GPU: whole episodes of one actor in one kernel launch (C ABI ``carenv_policy_eval``).

The reference scores a policy only by watching it (the video logger of train.py:23-50, greedy play every 10
epochs); ``avg_reward`` of training is a per-step mean over exploring rollouts.  Here every episode of a batch is
played to its end by ``k_policy_eval`` (csrc/policy_eval.cuh) — greedily or by sampling — and leaves one record:
its return, length, gates, laps, the step of its first lap and whether it crashed or ran into the 1000-step limit.

    python -m ppo_car_b200.evaluate --checkpoint model.dat --track big_track --episodes 65536 [--greedy]
    python -m torch.distributed.run --nproc-per-node 8 -m ppo_car_b200.evaluate --checkpoint model.dat ...

Episode ``episode0 + i`` of a call is a fixed function of (weights, seed, id, greedy): a batch can be split over
calls or ranks at any boundary and gives the same records.

Several tracks (``--track big_track,track``, or a ``MultiTrackVecEnv``): episode ``g`` plays on track ``g % n_tracks``
by default (``carenv_policy_eval_multi``, still one launch), and the summary gains ``"by_track"``.

Several actors (:func:`evaluate_population`, ``--checkpoint a.dat,b.dat,...``): the same episode ids of every actor in
one launch (``carenv_policy_eval_pop``); each actor's records are those ``evaluate_policy`` gives it alone.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import math
import os

import torch

from . import _lib
from .policy import ACTIONS, HIDDEN, OBS

TIME_LIMIT = 1000                   # steps per episode at most (lib/car_env.py:491)
RECORD_INT32 = 8                    # carenv_eval_record: double ret; int32 length, gates, laps, first_lap, outcome, pad
CRASH, TRUNCATED = 1, 2
SUM_FIELDS = ("count", "ret", "ret_sq", "length", "crashes", "truncations", "lapped", "laps", "first_lap", "gates")


def _p(t):
    return None if t is None else C.c_void_p(t.data_ptr())


class EvalResult:
    """Per-episode records of one evaluation call.  ``records`` is the int32 [n, 8] image of the C records;
    ``ret`` (float64), ``length``, ``gates``, ``laps``, ``first_lap`` (-1 without a lap) and ``outcome``
    (1 = crash, 2 = time limit) are views of it.  ``trace_actions`` [n_trace, 1000] uint8 (255 past an
    episode's end) and ``trace_u`` [n_trace, 1000] float32 (sampled calls only) are None without a trace."""

    def __init__(self, records: torch.Tensor, trace_actions: torch.Tensor | None = None,
                 trace_u: torch.Tensor | None = None, track: torch.Tensor | None = None, n_tracks: int | None = None):
        """``track`` [n] (int, on the records' device) and ``n_tracks``: the track of every episode of a
        multi-track call (None for single-track calls)."""
        if records.dtype != torch.int32 or records.dim() != 2 or records.shape[1] != RECORD_INT32:
            raise ValueError("records must be an int32 tensor of shape (n, 8)")
        if (track is None) != (n_tracks is None):
            raise ValueError("pass both track and n_tracks, or neither")
        if track is not None and (tuple(track.shape) != (records.shape[0],) or track.device != records.device):
            raise ValueError("track must hold one id per record, on the records' device")
        self.track, self.n_tracks = track, (None if n_tracks is None else int(n_tracks))
        self.records = records
        self.ret = records.view(torch.float64)[:, 0]
        self.length, self.gates, self.laps = records[:, 2], records[:, 3], records[:, 4]
        self.first_lap, self.outcome = records[:, 5], records[:, 6]
        self.trace_actions, self.trace_u = trace_actions, trace_u

    def __len__(self) -> int:
        return self.records.shape[0]

    def sums(self) -> torch.Tensor:
        """float64 [10] on the records' device, in the order of SUM_FIELDS: count, sum of returns, sum of squared
        returns, sum of lengths, crashes, truncations, episodes with a lap, sum of laps, sum of first-lap steps
        over the lapped episodes, sum of gates.  Sums of shards add up to the sums of their concatenation."""
        d = torch.float64
        lapped = self.laps > 0
        ret = self.ret
        return torch.stack([
            torch.tensor(float(len(self)), dtype=d, device=ret.device), ret.sum(), (ret * ret).sum(),
            self.length.to(d).sum(), (self.outcome == CRASH).to(d).sum(), (self.outcome == TRUNCATED).to(d).sum(),
            lapped.to(d).sum(), self.laps.to(d).sum(), torch.where(lapped, self.first_lap, 0).to(d).sum(),
            self.gates.to(d).sum()])

    def sums_by_track(self) -> torch.Tensor:
        """float64 [n_tracks, 10]: :meth:`sums` of the episodes of each track (multi-track calls only).  Rows of
        shards add up like :meth:`sums`."""
        if self.track is None:
            raise ValueError("sums_by_track needs the track column of a multi-track evaluation")
        d = torch.float64
        lapped = self.laps > 0
        ret = self.ret
        cols = torch.stack([
            torch.ones_like(ret), ret, ret * ret, self.length.to(d), (self.outcome == CRASH).to(d),
            (self.outcome == TRUNCATED).to(d), lapped.to(d), self.laps.to(d),
            torch.where(lapped, self.first_lap, 0).to(d), self.gates.to(d)], dim=1)
        out = torch.zeros((self.n_tracks, len(SUM_FIELDS)), dtype=d, device=ret.device)
        return out.index_add_(0, self.track.to(device=ret.device, dtype=torch.int64), cols)

    def summary_by_track(self, sums_by_track: torch.Tensor | None = None) -> list[dict]:
        """One :meth:`summary` per track from ``sums_by_track`` (e.g. all-reduced; default: this call's)."""
        rows = self.sums_by_track() if sums_by_track is None else sums_by_track
        return [self.summary(r) for r in rows]

    def summary(self, sums: torch.Tensor | None = None) -> dict:
        """Means and rates from ``sums`` (e.g. all-reduced over ranks; default: this call's).  ``avg_reward`` is
        the sum of returns over the sum of lengths: training's metric (times its reward scaling) without the
        exploration noise and over whole episodes.  Rates are fractions of the episodes; ``std_return`` is the
        population standard deviation; ``mean_first_lap_steps`` is over the episodes with a lap (None if none)."""
        s = dict(zip(SUM_FIELDS, (self.sums() if sums is None else sums).tolist()))
        n = s["count"]
        if n <= 0:
            return {"episodes": 0}
        mean = s["ret"] / n
        return {"episodes": int(n), "mean_return": mean,
                "std_return": math.sqrt(max(s["ret_sq"] / n - mean * mean, 0.0)),
                "avg_reward": s["ret"] / s["length"], "mean_length": s["length"] / n,
                "crash_rate": s["crashes"] / n, "truncation_rate": s["truncations"] / n,
                "lap_rate": s["lapped"] / n, "mean_laps": s["laps"] / n,
                "mean_first_lap_steps": s["first_lap"] / s["lapped"] if s["lapped"] > 0 else None,
                "mean_gates": s["gates"] / n}


def _actor_params(actor, device):
    params = [actor[0].weight, actor[0].bias, actor[2].weight, actor[2].bias]
    if [tuple(p.shape) for p in params] != [(HIDDEN, OBS), (HIDDEN,), (ACTIONS, HIDDEN), (ACTIONS,)]:
        raise ValueError("policy evaluation supports the reference actor only: 18-256-9")
    if any(p.dtype != torch.float32 or not p.is_contiguous() or p.device != device for p in params):
        raise ValueError(f"actor parameters must be contiguous float32 tensors on {device}")
    return [p.detach() for p in params]


def default_episode_tracks(n_episodes: int, n_tracks: int, episode0: int = 0, device=None) -> torch.Tensor:
    """Track of global episode id ``g``: ``g % n_tracks`` (int32 [n_episodes]); a batch split over calls or ranks
    gets the same assignment."""
    return ((int(episode0) % n_tracks + torch.arange(n_episodes, dtype=torch.int64, device=device)) % n_tracks
            ).to(torch.int32)


def evaluate_policy(env, actor, n_episodes: int, greedy: bool = False, seed: int = 0, episode0: int = 0,
                    trace: int = 0, episode_tracks=None) -> EvalResult:
    """Play episodes ``episode0 .. episode0 + n_episodes - 1`` of ``actor`` (``nn.Sequential(Linear(18, 256), ReLU,
    Linear(256, 9))`` on ``env.device``) on ``env``'s track, each from the start pose to its end, in one launch on
    the current stream.  ``greedy``: argmax actions; else sampled with the Philox stream keyed by ``seed``.  The
    first ``trace`` episodes also record their actions (and uniforms when sampled).  ``env``'s state is not
    touched; only its track handle and device are used.

    With a :class:`MultiTrackVecEnv`, episode ``i`` of the call plays on track ``episode_tracks[i]`` (default: the
    global id modulo the number of tracks, :func:`default_episode_tracks`) and its record equals the single-track
    record of the same id on that track; the result has a ``track`` column and per-track sums."""
    from .vec_env import MultiTrackVecEnv

    n_episodes, trace = int(n_episodes), int(trace)
    if n_episodes < 0 or trace < 0:
        raise ValueError("n_episodes and trace must be >= 0")
    if not 0 <= int(episode0) < 2 ** 64:
        raise ValueError("episode0 must fit in 64 bits")
    dev = env.device
    multi = isinstance(env, MultiTrackVecEnv)
    if episode_tracks is not None and not multi:
        raise ValueError("episode_tracks needs a MultiTrackVecEnv")
    if multi:
        n_tracks = len(env.track_paths)
        if episode_tracks is None:
            tracks = default_episode_tracks(n_episodes, n_tracks, episode0, dev)
        else:
            tracks = torch.as_tensor(episode_tracks).reshape(-1)
            if tracks.numel() != n_episodes:
                raise ValueError(f"expected {n_episodes} episode tracks, got {tracks.numel()}")
            if tracks.dtype.is_floating_point or tracks.dtype == torch.bool:
                raise ValueError("episode_tracks must be integers")
            if n_episodes and (int(tracks.min()) < 0 or int(tracks.max()) >= n_tracks):
                raise ValueError(f"episode tracks must be in 0..{n_tracks - 1}")
            tracks = tracks.to(device=dev, dtype=torch.int32).contiguous()
    params = _actor_params(actor, dev)
    records = torch.empty((n_episodes, RECORD_INT32), dtype=torch.int32, device=dev)
    n_trace = min(trace, n_episodes)
    trace_actions = trace_u = None
    if trace:
        trace_actions = torch.full((n_trace, TIME_LIMIT), 255, dtype=torch.uint8, device=dev)
        if not greedy:
            trace_u = torch.full((n_trace, TIME_LIMIT), float("nan"), dtype=torch.float32, device=dev)
    L = _lib.lib()
    if multi:
        with torch.cuda.device(dev):
            rc = L.carenv_policy_eval_multi(env._multi, _p(tracks), *[_p(p) for p in params], n_episodes, int(episode0),
                                            int(bool(greedy)), int(seed) & (2 ** 64 - 1), _p(records), n_trace,
                                            _p(trace_actions), _p(trace_u), env._stream())
        _lib.check(rc, "carenv_policy_eval_multi")
        return EvalResult(records, trace_actions, trace_u, track=tracks, n_tracks=n_tracks)
    with torch.cuda.device(dev):
        rc = L.carenv_policy_eval(env._handle, *[_p(p) for p in params], n_episodes, int(episode0), int(bool(greedy)),
                                  int(seed) & (2 ** 64 - 1), _p(records), n_trace, _p(trace_actions), _p(trace_u),
                                  env._stream())
    _lib.check(rc, "carenv_policy_eval")
    return EvalResult(records, trace_actions, trace_u)


def evaluate_population(env, actor_params, n_episodes: int, greedy: bool = False, seeds=0, episode0: int = 0,
                        trace: int = 0) -> list[EvalResult]:
    """:func:`evaluate_policy` of P actors in one launch (``carenv_policy_eval_pop``): episodes ``episode0 ..
    episode0 + n_episodes - 1`` of every member on ``env``'s track.  ``actor_params`` are the four stacked actor
    tensors ``w1 [P, 256, 18], b1 [P, 256], w2 [P, 9, 256], b2 [P, 9]`` (``Population.params[:4]``), contiguous float32
    on ``env.device``; ``seeds`` is one seed for every member or a list of P.  Returns one :class:`EvalResult` per
    member whose records (views of one ``[P, n, 8]`` tensor) and traces equal ``evaluate_policy`` of that member's
    actor with its seed.  Populations play on one track: a :class:`MultiTrackVecEnv` is refused."""
    from .vec_env import MultiTrackVecEnv

    if isinstance(env, MultiTrackVecEnv):
        raise ValueError("evaluate_population plays on one track; a MultiTrackVecEnv is not supported")
    n_episodes, trace = int(n_episodes), int(trace)
    if n_episodes < 0 or trace < 0:
        raise ValueError("n_episodes and trace must be >= 0")
    if not 0 <= int(episode0) < 2 ** 64:
        raise ValueError("episode0 must fit in 64 bits")
    dev = env.device
    params = list(actor_params)
    P = params[0].shape[0] if len(params) == 4 and params[0].dim() == 3 else 0
    if [tuple(p.shape) for p in params] != [(P, HIDDEN, OBS), (P, HIDDEN), (P, ACTIONS, HIDDEN), (P, ACTIONS)]:
        raise ValueError("actor_params must be the stacked reference actor tensors [P, 256, 18], [P, 256], "
                         "[P, 9, 256], [P, 9]")
    if not 1 <= P <= 65535:
        raise ValueError("a population has 1 .. 65535 members")
    if any(p.dtype != torch.float32 or not p.is_contiguous() or p.device != dev for p in params):
        raise ValueError(f"actor parameters must be contiguous float32 tensors on {dev}")
    seeds = [int(seeds)] * P if isinstance(seeds, int) else [int(s) for s in seeds]
    if len(seeds) != P:
        raise ValueError(f"expected one seed or {P} seeds, got {len(seeds)}")
    seeds = [s & (2 ** 64 - 1) for s in seeds]                 # as evaluate_policy
    records = torch.empty((P, n_episodes, RECORD_INT32), dtype=torch.int32, device=dev)
    n_trace = min(trace, n_episodes)
    trace_actions = trace_u = None
    if trace:
        trace_actions = torch.full((P, n_trace, TIME_LIMIT), 255, dtype=torch.uint8, device=dev)
        if not greedy:
            trace_u = torch.full((P, n_trace, TIME_LIMIT), float("nan"), dtype=torch.float32, device=dev)
    results = [EvalResult(records[p], None if trace_actions is None else trace_actions[p],
                          None if trace_u is None else trace_u[p]) for p in range(P)]
    if n_episodes == 0:
        return results
    # a pinned, stream-ordered copy: a pageable one would wait for the work already queued on the device
    seeds_dev = torch.tensor([s - 2 ** 64 if s >= 2 ** 63 else s for s in seeds], dtype=torch.int64).pin_memory()
    with torch.cuda.device(dev):
        seeds_dev = seeds_dev.to(dev, non_blocking=True)
        rc = _lib.lib().carenv_policy_eval_pop(env._handle, P, *[_p(p.detach()) for p in params], n_episodes,
                                               int(episode0), int(bool(greedy)), _p(seeds_dev), _p(records), n_trace,
                                               _p(trace_actions), _p(trace_u), env._stream())
    _lib.check(rc, "carenv_policy_eval_pop")
    return results


def load_checkpoint(path: str):
    """The state dict ``train_ppo`` saves (model.dat / checkpoint_{epoch}.dat, the reference Agent's keys
    actor.0.weight ... critic.2.bias), loaded strictly into a CPU ActorCritic."""
    from .train_ppo import ActorCritic

    net = ActorCritic(OBS, ACTIONS, HIDDEN)
    net.load_state_dict(torch.load(path, map_location="cpu", weights_only=True), strict=True)
    return net


def checkpoint_list(spec: str) -> list[str]:
    """``--checkpoint``: one path (kept whole when it names a file, commas included) or a comma-separated list."""
    if os.path.exists(spec):
        return [spec]
    paths = [c.strip() for c in spec.split(",")]
    if not all(paths):
        raise SystemExit(f"empty entry in --checkpoint {spec!r}")
    return paths


def parse_args(argv=None):
    p = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    p.add_argument("--checkpoint", required=True,
                   help="model.dat / checkpoint_{epoch}.dat written by train_ppo; a comma-separated list (e.g. every "
                        "member_*/model.dat of a population) scores all of them in one launch with the same --seed and "
                        "prints one summary per checkpoint under \"checkpoints\"")
    p.add_argument("--track", default="big_track",
                   help="track name shipped with the package or a JSON path; a comma-separated list plays episode g on "
                        "track g %% n_tracks and adds per-track summaries under \"by_track\"")
    p.add_argument("--episodes", type=int, default=65536, help="episodes in total over all ranks")
    p.add_argument("--greedy", action="store_true", help="argmax actions instead of sampled ones")
    p.add_argument("--seed", type=int, default=0, help="seed of the sampling stream")
    p.add_argument("--json", default=None, help="write the summary to this file")
    return p.parse_args(argv)


def main(argv=None) -> dict:
    import torch.distributed as dist

    from . import MultiTrackVecEnv, VecCarEnv, builtin_track
    from .shard import shard_range

    args = parse_args(argv)
    names = args.track.split(",")
    ckpts = checkpoint_list(args.checkpoint)
    if len(ckpts) > 1 and len(names) > 1:
        raise SystemExit("several checkpoints are scored on one track; pass several checkpoints or several tracks, "
                         "not both")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1 and not dist.is_initialized():
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    paths = [t if os.path.exists(t) else builtin_track(t) for t in names]
    if len(paths) == 1:
        env = VecCarEnv(1, paths[0], device=dev)
    else:
        env = MultiTrackVecEnv(track_paths=paths, track_ids=[0], device=dev)
    lo, hi = shard_range(args.episodes, world, rank)            # every rank plays its contiguous share of the ids
    if len(ckpts) > 1:
        actors = [load_checkpoint(c).actor for c in ckpts]
        stacked = [torch.stack([getattr(a[i], k).detach() for a in actors]).to(dev).contiguous()
                   for i, k in ((0, "weight"), (0, "bias"), (2, "weight"), (2, "bias"))]
        results = evaluate_population(env, stacked, hi - lo, greedy=args.greedy, seeds=args.seed, episode0=lo)
        sums = torch.stack([r.sums() for r in results])         # [P, 10]
        if world > 1:
            dist.all_reduce(sums, op=dist.ReduceOp.SUM)
        out = {"checkpoints": [{"checkpoint": c, "track": args.track, "greedy": bool(args.greedy), "seed": args.seed,
                                **r.summary(s)} for c, r, s in zip(ckpts, results, sums)]}
    else:
        actor = load_checkpoint(args.checkpoint).actor.to(dev)
        res = evaluate_policy(env, actor, hi - lo, greedy=args.greedy, seed=args.seed, episode0=lo)
        sums = res.sums()
        by_track = res.sums_by_track() if len(paths) > 1 else None
        if world > 1:
            dist.all_reduce(sums, op=dist.ReduceOp.SUM)
            if by_track is not None:
                dist.all_reduce(by_track, op=dist.ReduceOp.SUM)
        out = {"checkpoint": args.checkpoint, "track": args.track, "greedy": bool(args.greedy), "seed": args.seed,
               **res.summary(sums)}
        if by_track is not None:
            out["by_track"] = [{"track": name, **summ} for name, summ in zip(names, res.summary_by_track(by_track))]
    if rank == 0:
        print(json.dumps(out), flush=True)
        if args.json:
            with open(args.json, "w") as fh:
                json.dump(out, fh)
    env.close()
    if dist.is_initialized():
        dist.destroy_process_group()
    return out


if __name__ == "__main__":
    main()
