"""PPO loop harness on the GPU environment (SURVEY §8 f-1, BASELINE config 5).

The caller of the hot path, restated from the reference's ``train.py:114-301`` so that the batched
environment and the GAE kernel can be exercised exactly the way the reference uses them:

  * same flags (``--n-envs --n-epochs --n-steps --batch-size --train-iters --gamma --gae-lambda
    --clip-ratio --ent-coef --vf-coef --learning-rate --learning-rate-decay --max-grad-norm
    --reward-scaling``, train.py:72-92) plus ``--track`` (the reference asks with a tkinter dialog);
  * same network (actor 18-256-9, critic 18-256-1, orthogonal init with gains sqrt(2) / 0.01 / 1.0,
    lib/model.py:6-26), Adam(lr, eps=1e-5) + StepLR(gamma = decay) (train.py:146-147);
  * same update math: clipped surrogate, 0.5 * value MSE, entropy bonus, per-minibatch advantage
    normalisation with max(std, 1e-5), grad-norm clip (train.py:233-261);
  * same minibatch schedule: per train iteration only ``n_steps / batch_size`` minibatches are drawn
    from the ``n_steps * n_envs`` samples (train.py:228 iterates over n_steps).  The reference shuffles
    all indices on the host (O(T*N) per iteration); here the indices of the minibatches are sampled on
    the device (uniform without the full permutation — at these sizes duplicates are negligible).

What differs by design: nothing leaves the device during the rollout (the reference round-trips
actions, observations, rewards and flags through the host every step, train.py:185-192), GAE is one
kernel launch, and with more than one process (torchrun) every rank owns an env shard and gradients
are averaged with one NCCL all-reduce per minibatch step (12,298 floats).

    python -m ppo_car_b200.train_ppo --track big_track --n-envs 24 --n-epochs 200

Several tracks: ``--track big_track,track,my_track.json`` trains ONE policy on all of them.  Global env g of N runs on
track g * K // N (contiguous blocks), every rank steps its shard as a MultiTrackVecEnv, and every epoch record gains
``"by_track"`` (avg_reward and episodes per track, over all ranks).
"""
from __future__ import annotations

import argparse
import math
import os
import time

import torch
import torch.distributed as dist
import torch.nn as nn

from . import Buffer, MultiTrackVecEnv, VecCarEnv, builtin_track
from .shard import allreduce_rollout_stats, shard_range, track_blocks


def _ortho(layer: nn.Linear, gain: float) -> nn.Linear:
    nn.init.orthogonal_(layer.weight, gain)
    nn.init.zeros_(layer.bias)
    return layer


class ActorCritic(nn.Module):
    """Two independent 2-layer MLPs (lib/model.py:10-26)."""

    def __init__(self, obs_dim: int, n_actions: int, hidden: int = 256):
        super().__init__()
        g = math.sqrt(2.0)
        self.actor = nn.Sequential(_ortho(nn.Linear(obs_dim, hidden), g), nn.ReLU(),
                                   _ortho(nn.Linear(hidden, n_actions), 0.01))
        self.critic = nn.Sequential(_ortho(nn.Linear(obs_dim, hidden), g), nn.ReLU(),
                                    _ortho(nn.Linear(hidden, 1), 1.0))

    def value(self, obs):
        return self.critic(obs)

    def act(self, obs, action=None):
        logp_all = torch.log_softmax(self.actor(obs), dim=-1)
        if action is None:
            action = torch.multinomial(logp_all.exp(), 1).squeeze(-1)
        logp = logp_all.gather(-1, action.long().unsqueeze(-1)).squeeze(-1)
        entropy = -(logp_all.exp() * logp_all).sum(-1)
        return action, logp, entropy, self.critic(obs)


def parse_args(argv=None):
    p = argparse.ArgumentParser()
    p.add_argument("--run-name", default="b200")
    p.add_argument("--checkpoint-dir", default=None,
                   help="directory for checkpoint_{epoch}.dat (every 10 epochs) and model.dat (at exit), the "
                        "reference's files (train.py:280-283, 301); a sub-directory named after --run-name is created. "
                        "Default: no checkpoints")
    p.add_argument("--track", default="big_track",
                   help="track name shipped with the package or a JSON path, or a comma-separated list of them: one "
                        "policy trained on every track, env g of N on track g * K // N")
    p.add_argument("--n-envs", type=int, default=16, help="total environments over all ranks")
    p.add_argument("--n-epochs", type=int, default=200)
    p.add_argument("--n-steps", type=int, default=1024)
    p.add_argument("--batch-size", type=int, default=512)
    p.add_argument("--train-iters", type=int, default=40)
    p.add_argument("--gamma", type=float, default=0.99)
    p.add_argument("--gae-lambda", type=float, default=0.95)
    p.add_argument("--clip-ratio", type=float, default=0.2)
    p.add_argument("--ent-coef", type=float, default=0.001)
    p.add_argument("--vf-coef", type=float, default=0.5)
    p.add_argument("--learning-rate", type=float, default=3e-4)
    p.add_argument("--learning-rate-decay", type=float, default=0.99)
    p.add_argument("--max-grad-norm", type=float, default=1.0)
    p.add_argument("--reward-scaling", type=float, default=0.1)
    p.add_argument("--seed", type=int, default=0)
    p.add_argument("--log-json", default=None, help="append one JSON line per epoch to this file")
    p.add_argument("--fused-rollout", action="store_true",
                   help="run the whole rollout (policy forward, sampling, env step, buffer rows) in ONE kernel launch "
                        "per epoch (carenv_policy_rollout); needs the reference network shape")
    p.add_argument("--fused-cuda-cores", action="store_true",
                   help="with --fused-rollout: use the CUDA-core kernel instead of the tensor-core one")
    p.add_argument("--fused-update", action="store_true",
                   help="one minibatch update = three kernel launches (carenv_ppo_grad / carenv_ppo_adam: forward, "
                        "loss, backward, clip, Adam for the reference network) instead of a PyTorch autograd graph")
    p.add_argument("--per-minibatch-update", action="store_true",
                   help="with --fused-update: three launches (+ one NCCL all-reduce) per minibatch instead of ONE "
                        "persistent launch per epoch with the gradient all-reduce over NVLink peer memory inside it")
    p.add_argument("--compact-obs", action="store_true",
                   help="with --fused-rollout: store 32-byte pose records instead of observations and recompute the "
                        "minibatch observations in the update (VecCarEnv.observe)")
    p.add_argument("--graph-update", action="store_true",
                   help="capture one minibatch update (sampling, forward, backward, clip, Adam) in a CUDA graph and "
                        "replay it train_iters x minibatches times per epoch (the NCCL gradient all-reduce is captured too)")
    p.add_argument("--cuda-graph", action="store_true",
                   help="capture the whole n_steps rollout (policy forward, sampling, env step, buffer rows) in one "
                        "CUDA graph and replay it every epoch: removes the per-step launch overhead at small n_envs")
    p.add_argument("--eval-every", type=int, default=0,
                   help="every K epochs play --eval-episodes whole episodes of the current actor on the training track "
                        "(ppo_car_b200.evaluate, one kernel launch, shared out over the ranks) and add the summary to "
                        "the epoch's record under \"eval\".  Default 0: no evaluation")
    p.add_argument("--eval-episodes", type=int, default=1024, help="episodes per evaluation, over all ranks")
    p.add_argument("--eval-greedy", action="store_true", help="evaluate with argmax actions instead of sampled ones")
    p.add_argument("--target-kl", type=float, default=None,
                   help="stop an epoch's updates at the first minibatch whose approx KL, mean((ratio - 1) - log ratio) "
                        "at the parameters before its step, exceeds this (compared against the target itself, not "
                        "Stable-Baselines3's 1.5 x target).  Epoch records gain approx_kl, clip_fraction, updates and "
                        "explained_variance")
    p.add_argument("--kl-stats", action="store_true",
                   help="the epoch-record statistics of --target-kl without stopping (a target of +inf)")
    p.add_argument("--bootstrap-truncated", action="store_true",
                   help="time-limit bootstrapping: the last step of an episode cut by the 1000-step limit is "
                        "bootstrapped from the critic's value of the observation the episode ended in instead of the "
                        "next episode's reset observation (the reference's GAE).  Changes the targets only; the rollout "
                        "rows are the same bits")
    return p.parse_args(argv)


def kl_target(args) -> float | None:
    """The target KL of --target-kl / --kl-stats (+inf: statistics only), None without either.  Refuses, before any
    device work, a target that is NaN or <= 0 and the update paths that cannot report or stop."""
    if args.target_kl is None and not args.kl_stats:
        return None
    tau = float("inf") if args.target_kl is None else float(args.target_kl)
    if not tau > 0.0:
        raise SystemExit(f"--target-kl must be positive, got {args.target_kl}")
    if args.graph_update:
        raise SystemExit("--target-kl / --kl-stats do not work with --graph-update: a captured update cannot stop")
    if args.fused_update and (args.per_minibatch_update or args.compact_obs):
        raise SystemExit("--target-kl / --kl-stats with --fused-update need the one-launch epoch kernel: the "
                         "per-minibatch kernels (--per-minibatch-update, --compact-obs) have no KL output")
    return tau


def explained_variance(ret, val, world: int = 1) -> float:
    """1 - Var(ret - val) / Var(ret) over every sample of the rollout (of every rank: float64 sums all-reduced)."""
    r, d = ret.reshape(-1).double(), (ret - val).reshape(-1).double()
    z = torch.stack([torch.tensor(float(r.numel()), dtype=torch.float64, device=r.device), r.sum(), (r * r).sum(),
                     d.sum(), (d * d).sum()])
    if world > 1:
        dist.all_reduce(z, op=dist.ReduceOp.SUM)
    n, sr, srr, sd, sdd = z.tolist()
    var_r, var_d = srr / n - (sr / n) ** 2, sdd / n - (sd / n) ** 2
    return 1.0 - var_d / var_r if var_r > 0.0 else float("nan")


def kl_record(kl_rows, n_done: int) -> dict:
    """approx_kl and clip_fraction: means over the evaluated updates (the stopping one included); updates: applied."""
    n_eval = min(n_done + 1, len(kl_rows))
    rows = kl_rows[:n_eval]
    mean = lambda k: sum(r[k] for r in rows) / len(rows) if rows else float("nan")
    return {"approx_kl": mean(0), "clip_fraction": mean(1), "updates": int(n_done)}


def track_list(args) -> tuple[list[str], list[str]]:
    """(names, paths) of ``--track``: one entry, or several from a comma-separated list.  With several tracks the
    options that have no multi-track path are refused here, before any device work."""
    names = [args.track] if os.path.exists(args.track) else args.track.split(",")
    paths = [t if os.path.exists(t) else builtin_track(t) for t in names]
    if len(paths) > 1:
        for flag, on, why in (("--compact-obs", args.compact_obs, "pose records do not carry a track"),
                              ("--fused-cuda-cores", args.fused_cuda_cores,
                               "the multi-track fused rollout runs on the tensor cores"),
                              ("--cuda-graph", args.cuda_graph,
                               "the eager rollout is not captured; --fused-rollout is one launch per epoch"),
                              ("--bootstrap-truncated without --fused-rollout",
                               args.bootstrap_truncated and not args.fused_rollout,
                               "the eager multi-track step has no final observation; use --fused-rollout")):
            if on:
                raise SystemExit(f"{flag} does not work with several tracks: {why}")
        if args.n_envs < len(paths):
            raise SystemExit(f"--n-envs {args.n_envs} is smaller than the number of tracks ({len(paths)}): "
                             "every track needs at least one environment")
    return names, paths


def train(args) -> list[dict]:
    names, paths = track_list(args)
    tau = kl_target(args)
    multi = len(paths) > 1
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1 and not dist.is_initialized():
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    torch.manual_seed(args.seed)                       # same initial weights on every rank
    lo, hi = shard_range(args.n_envs, world, rank)
    n = hi - lo
    T = args.n_steps

    boot_trunc = bool(args.bootstrap_truncated)
    eager_boot = boot_trunc and not args.fused_rollout          # the eager loop stores critic(final observation)
    if multi:
        envs = MultiTrackVecEnv(track_paths=paths, track_ids=track_blocks(args.n_envs, len(paths), lo, hi), device=dev,
                                reward_scaling=args.reward_scaling, float_flags=True)
    else:
        envs = VecCarEnv(n, paths[0], device=dev, reward_scaling=args.reward_scaling, float_flags=True,
                         with_info=False, final_observation=eager_boot)
    obs_dim = envs.single_observation_space.shape
    agent = ActorCritic(obs_dim[0], envs.single_action_space.n).to(dev)
    graph_update = bool(args.graph_update)                 # with world > 1 the NCCL all-reduce is captured too
    fused_upd = None
    if args.fused_update:
        from .ppo_update import FusedPPOUpdate

        fused_upd = FusedPPOUpdate(agent.actor, agent.critic, args.batch_size, args.learning_rate, args.clip_ratio,
                                   args.vf_coef, args.ent_coef, args.max_grad_norm)
    # all minibatch updates of an epoch in one persistent launch (csrc/ppo_epoch.cuh); it reads observation rows, so
    # pose-record storage keeps the per-minibatch kernels
    epoch_kernel = fused_upd is not None and not args.per_minibatch_update and not args.compact_obs
    if epoch_kernel and world > 1:
        fused_upd.connect()                                 # IPC-mapped gradient exchange buffers of the peers
    if graph_update:                                        # capturable Adam with the learning rate in a tensor
        opt = torch.optim.Adam(agent.parameters(), lr=torch.tensor(args.learning_rate, device=dev), eps=1e-5,
                               capturable=True)
        sched = None
    else:
        opt = torch.optim.Adam(agent.parameters(), lr=args.learning_rate, eps=1e-5)
        sched = torch.optim.lr_scheduler.StepLR(opt, step_size=1, gamma=args.learning_rate_decay)
    params = [p for p in agent.parameters()]
    if args.compact_obs and not args.fused_rollout:
        raise SystemExit("--compact-obs needs --fused-rollout")
    buf = Buffer(obs_dim, T, n, dev, args.gamma, args.gae_lambda, compact_obs=args.compact_obs,
                 bootstrap_truncated=boot_trunc)
    torch.manual_seed(args.seed * 1000 + rank + 1)     # different sampling noise per shard

    # the rollout state lives in three static tensors so that the loop below can be captured in a graph
    next_obs = envs.reset()[0].clone()
    next_term = torch.zeros(n, device=dev)
    next_trunc = torch.zeros(n, device=dev)
    history, global_step, t_start = [], 0, time.time()
    n_mb = -(-T // args.batch_size)                        # range(0, n_steps, batch_size): ceil (train.py:228)
    ckpt_dir = None
    if args.checkpoint_dir and rank == 0:                  # train.py:125-126: checkpoints/<run>/
        ckpt_dir = os.path.join(args.checkpoint_dir, args.run_name)
        os.makedirs(ckpt_dir, exist_ok=True)

    def save_checkpoint(name):
        """The keys are the reference Agent's (actor.0.weight ... critic.2.bias): loads into lib/model.py:Agent."""
        if ckpt_dir is not None:
            torch.save({k: v.detach().cpu() for k, v in agent.state_dict().items()}, os.path.join(ckpt_dir, name))

    def rollout():
        """train.py:173-195 with everything on the device: row t of the buffer gets (obs_t, a_t, r_t, V(obs_t),
        term_t, trunc_t, logp_t); the env's outputs become the next step's inputs."""
        buf.ptr = 0
        for _ in range(T):
            act, logp, _, val = agent.act(next_obs)
            buf.store(next_obs, act, 0.0, val.view(-1), next_term, next_trunc, logp)
            o, rew, te, tr, info = envs.step(act)
            buf.rew_buf[buf.ptr - 1].copy_(rew)
            if eager_boot:                                  # read by the GAE only where the step truncated
                buf.boot_buf[buf.ptr - 1].copy_(agent.value(info["final_observation"]).view(-1))
            next_obs.copy_(o)
            next_term.copy_(te)
            next_trunc.copy_(tr)

    packed = last_val = None
    warp_rollout = False
    if args.fused_rollout:
        from .policy import (WARP_ROLLOUT_MAX_ENVS, fused_rollout, fused_rollout_warp, pack_policy_weights,
                             pack_policy_weights_tc)

        # small shards (the reference's 24 environments): one warp per environment, parameters read in place
        warp_rollout = (not multi and not args.fused_cuda_cores and n <= WARP_ROLLOUT_MAX_ENVS
                        and len(envs.track.walls) <= 32)

        # otherwise the tensor-core kernel (k_policy_rollout_tc3, 256-environment CTAs), or the CUDA-core kernel with
        # --fused-cuda-cores
        pack_policy = pack_policy_weights_tc if not args.fused_cuda_cores else pack_policy_weights
        packed = pack_policy(agent.actor, agent.critic)
        last_val = torch.empty(n, device=dev)

    def evaluate_epoch():
        """--eval-every: every rank plays its share of the episode ids 0 .. eval_episodes - 1 with the same seed, so
        every evaluation of a run scores the actor on the same episodes; the sums are all-reduced."""
        from .evaluate import evaluate_policy

        e_lo, e_hi = shard_range(args.eval_episodes, world, rank)
        with torch.no_grad():
            res = evaluate_policy(envs, agent.actor, e_hi - e_lo, greedy=args.eval_greedy, seed=args.seed,
                                  episode0=e_lo)
            sums = res.sums()
            by_track = res.sums_by_track() if multi else None
        if world > 1:
            dist.all_reduce(sums, op=dist.ReduceOp.SUM)
            if by_track is not None:
                dist.all_reduce(by_track, op=dist.ReduceOp.SUM)
        out = res.summary(sums)
        if by_track is not None:
            out["by_track"] = [{"track": name, **summ} for name, summ in zip(names, res.summary_by_track(by_track))]
        return out

    def rollout_by_track():
        """avg_reward and episodes of this epoch's rollout per track, summed over the ranks."""
        tid = envs.track_ids.to(torch.int64)
        z = torch.zeros((3, len(paths)), dtype=torch.float64, device=dev)
        z[0].index_add_(0, tid, buf.rew_buf.sum(0).double())
        z[1].index_add_(0, tid, torch.full((n,), float(T), dtype=torch.float64, device=dev))
        z[2].index_add_(0, tid, (buf.term_buf.sum(0) + buf.trunc_buf.sum(0)).double())
        if world > 1:
            dist.all_reduce(z, op=dist.ReduceOp.SUM)
        r, st, ep = z.tolist()
        return [{"track": name, "avg_reward": r[k] / st[k] / args.reward_scaling, "episodes": ep[k]}
                for k, name in enumerate(names)]

    graph = None
    if args.cuda_graph and not args.fused_rollout:
        with torch.no_grad():
            side = torch.cuda.Stream(device=dev)
            side.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(side):                  # warm-up outside capture (lazy inits, autotuning)
                rollout()
            torch.cuda.current_stream(dev).wait_stream(side)
            torch.cuda.synchronize(dev)
            next_obs.copy_(envs.reset()[0])                # discard the warm-up rollout
            next_term.zero_()
            next_trunc.zero_()
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                rollout()

    try:
        for epoch in range(1, args.n_epochs + 1):
            # ---- rollout
            with torch.no_grad():
                if warp_rollout:
                    fused_rollout_warp(envs, agent.actor, agent.critic, buf, next_obs, next_term, next_trunc,
                                       seed=args.seed, step0=(epoch - 1) * T, env_offset=lo, last_val=last_val)
                    if boot_trunc:
                        buf.final_values(agent.critic)
                    boot = last_val.reshape(1, -1)
                elif packed is not None:
                    pack_policy(agent.actor, agent.critic, out=packed)
                    fused_rollout(envs, packed, buf, next_obs, next_term, next_trunc, seed=args.seed,
                                  step0=(epoch - 1) * T, env_offset=lo, last_val=last_val)
                    if boot_trunc:
                        buf.final_values(agent.critic)
                    boot = last_val.reshape(1, -1)
                else:
                    if graph is not None:
                        graph.replay()
                        buf.ptr = T
                    else:
                        rollout()
                    boot = agent.value(next_obs).reshape(1, -1)
                global_step += T * args.n_envs
                adv, ret = buf.calculate_advantages(boot, next_term.reshape(1, -1), next_trunc.reshape(1, -1))
            rew_sum, steps, episodes = allreduce_rollout_stats(buf.rew_buf.sum(), torch.tensor(float(T * n), device=dev),
                                                               buf.term_buf.sum() + buf.trunc_buf.sum())
            by_track = rollout_by_track() if multi else None
            obs_b, act_b, val_b, logp_b = buf.get()
            obs_f = obs_b if args.compact_obs else obs_b.view(-1, *obs_dim)      # pose records / observations
            act_f, logp_f = act_b.view(-1), logp_b.view(-1)
            adv_f, ret_f = adv.view(-1), ret.view(-1)

            # ---- update (train.py:223-261)
            if epoch == 1:
                sums = torch.zeros(4, device=dev)
                idx_static = torch.zeros(args.batch_size, dtype=torch.int64, device=dev)

                def update_step():
                    """One minibatch: draw indices, clipped-surrogate loss, backward, (all-reduce), clip, Adam.  With
                    --target-kl / --kl-stats: returns True, without a step, when the approx KL exceeds the target."""
                    torch.randint(0, T * n, (args.batch_size,), device=dev, out=idx_static)
                    idx = idx_static
                    if fused_upd is not None:
                        obs_in = envs.observe(obs_f, idx) if args.compact_obs else obs_f
                        fused_upd.grad(obs_in, idx, act_f, logp_f, adv_f, ret_f, obs_is_gathered=args.compact_obs)
                        fused_upd.apply(world)
                        return
                    obs_mb = envs.observe(obs_f, idx) if args.compact_obs else obs_f[idx]
                    _, new_logp, ent, new_val = agent.act(obs_mb, act_f[idx])
                    ratio = torch.exp(new_logp - logp_f[idx])
                    if tau is not None:
                        with torch.no_grad():
                            st = torch.stack([((ratio - 1.0) - (new_logp - logp_f[idx])).mean(),
                                              ((ratio - 1.0).abs() > args.clip_ratio).float().mean()])
                            if world > 1:                           # every rank's minibatch: one small all-reduce
                                dist.all_reduce(st, op=dist.ReduceOp.SUM)
                                st /= world
                        kl_rows.append(st)
                        if tau != float("inf") and float(st[0]) > tau:
                            return True
                    a = adv_f[idx]
                    a = (a - a.mean()) / torch.clamp(a.std(), min=1e-5)
                    pol = torch.max(-a * ratio, -a * torch.clamp(ratio, 1 - args.clip_ratio, 1 + args.clip_ratio)).mean()
                    vl = 0.5 * ((new_val.view(-1) - ret_f[idx]) ** 2).mean()
                    e = ent.mean()
                    loss = pol + args.vf_coef * vl - args.ent_coef * e
                    opt.zero_grad(set_to_none=True)
                    loss.backward()
                    if world > 1:                                   # average the 12,298 gradients over the shards
                        flat = torch.cat([p.grad.reshape(-1) for p in params])
                        dist.all_reduce(flat, op=dist.ReduceOp.SUM)
                        flat /= world
                        off = 0
                        for p in params:
                            p.grad.copy_(flat[off:off + p.numel()].view_as(p))
                            off += p.numel()
                    nn.utils.clip_grad_norm_(params, args.max_grad_norm)
                    opt.step()
                    sums.add_(torch.stack([pol.detach(), vl.detach(), e.detach(), loss.detach()]))
                    return False

                update_graph = None
                if graph_update and not epoch_kernel:           # obs_f, act_f, ... are views of the static buffer tensors
                    side = torch.cuda.Stream(device=dev)
                    side.wait_stream(torch.cuda.current_stream(dev))
                    with torch.cuda.stream(side):
                        for _ in range(3):                      # warm-up (also creates Adam's state) counts as 3 real steps
                            update_step()
                    torch.cuda.current_stream(dev).wait_stream(side)
                    update_graph = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(update_graph):
                        update_step()
                    sums.zero_()
            sums.zero_()
            if fused_upd is not None:
                fused_upd.sums.zero_()
            kl_rows, n_done, stopped = [], 0, False
            if epoch_kernel:
                idx_all = torch.randint(0, T * n, (args.train_iters * n_mb, args.batch_size), device=dev)
                fused_upd.run_epoch(obs_f, idx_all, act_f, logp_f, adv_f, ret_f, world=world, target_kl=tau)
            for _ in range(0 if epoch_kernel else args.train_iters * n_mb):
                if update_graph is not None:
                    update_graph.replay()
                elif stopped:                                    # the stopped epoch still draws its indices
                    torch.randint(0, T * n, (args.batch_size,), device=dev, out=idx_static)
                else:
                    stopped = update_step()
                    n_done += not stopped
            if fused_upd is not None:
                fused_upd.lr.mul_(args.learning_rate_decay)
                sums.copy_(fused_upd.sums)
            elif sched is not None:
                sched.step()
            else:
                opt.param_groups[0]["lr"].mul_(args.learning_rate_decay)

            s = (sums / args.train_iters).tolist()
            rec = {"epoch": epoch, "global_step": global_step, "avg_reward": rew_sum / steps / args.reward_scaling,
                   "episodes": episodes, "policy_loss": s[0], "value_loss": s[1], "entropy": s[2], "total_loss": s[3],
                   "lr": float(fused_upd.lr if fused_upd is not None else opt.param_groups[0]["lr"]), "sps": global_step / (time.time() - t_start),
                   "wall_s": time.time() - t_start}
            if tau is not None:
                if epoch_kernel:
                    kl_rows, n_done = fused_upd.kl.tolist(), int(fused_upd.n_done.item())
                else:
                    kl_rows = torch.stack(kl_rows).tolist() if kl_rows else []
                rec.update(kl_record(kl_rows, n_done))
                rec["explained_variance"] = explained_variance(ret_f, val_b.reshape(-1), world)
            if by_track is not None:
                rec["by_track"] = by_track
            if args.eval_every > 0 and epoch % args.eval_every == 0:
                rec["eval"] = evaluate_epoch()
            history.append(rec)
            if rank == 0:
                print(f"Epoch {epoch} done in {rec['wall_s']:.2f}s. Avg reward: {rec['avg_reward']:.4f}. "
                      f"SPS {rec['sps']:.0f}  entropy {rec['entropy']:.3f}", flush=True)
                if by_track is not None:
                    print("  by track: " + ", ".join(f"{b['track']} {b['avg_reward']:.4f}" for b in by_track), flush=True)
                if "eval" in rec:
                    ev = rec["eval"]
                    print(f"  eval ({ev['episodes']} {'greedy' if args.eval_greedy else 'sampled'} episodes): return "
                          f"{ev['mean_return']:.3f} +- {ev['std_return']:.3f}, avg reward {ev['avg_reward']:.4f}, "
                          f"crashes {ev['crash_rate']:.1%}, laps/episode {ev['mean_laps']:.3f}", flush=True)
                if args.log_json:
                    import json

                    with open(args.log_json, "a") as fh:
                        fh.write(json.dumps(rec) + "\n")
            if epoch % 10 == 0:
                save_checkpoint(f"checkpoint_{epoch}.dat")
    finally:                                               # train.py:294-301
        save_checkpoint("model.dat")
    if fused_upd is not None:
        fused_upd.check_epoch()
        fused_upd.close()
    envs.close()
    return history


def main(argv=None):
    args = parse_args(argv)
    train(args)
    if dist.is_initialized():
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
