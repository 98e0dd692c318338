"""Populations: many independent PPO training runs in one process (seed and hyperparameter sweeps).

A *member* is one training run of ``train_ppo --fused-rollout --fused-update``: its own ActorCritic (the reference
shape, 18-256-9 actor and 18-256-1 critic), Adam moments and step count, learning rate and schedule, clip ratio,
loss coefficients, seed and ``n`` environments.  Members never exchange data.  Environment ``e`` of member ``p`` is
global column ``p * n + e`` of every ``[N]`` and ``[T, N]`` array (``N = P * n``), so one ``VecCarEnv(P * n)``, one
``Buffer`` and the GAE kernel serve the whole population, and each epoch is one rollout launch
(``carenv_policy_rollout_warp_pop`` / ``_tc_pop``), one GAE launch and one update launch (``carenv_ppo_epoch_pop``,
one thread-block cluster per member) for all members.

Member ``p`` is initialised, rolled out and given minibatches exactly as ``train_ppo --seed seeds[p]`` would be, so
its first epoch's rollout is bit-identical to that run's; its updates differ from ``k_ppo_epoch``'s only in the
summation order of the gradient.

``--pbt-every K`` turns on population-based training (:mod:`ppo_car_b200.pbt`): every K epochs the weakest members
take perturbed copies of the best members' training state.

    python -m ppo_car_b200.population --track big_track --n-envs 24 --n-epochs 200 --seeds 0-31 \\
        --learning-rate 3e-4,1e-3
"""
from __future__ import annotations

import argparse
import ctypes as C
import itertools
import json
import math
import os
import time

import torch
import torch.distributed as dist

from . import _lib
from .policy import ACTIONS, OBS, WARP_ROLLOUT_MAX_ENVS

HPARAMS = ("learning_rate", "learning_rate_decay", "clip_ratio", "ent_coef", "vf_coef", "max_grad_norm")
DEFAULTS = {"learning_rate": 3e-4, "learning_rate_decay": 0.99, "clip_ratio": 0.2, "ent_coef": 0.001, "vf_coef": 0.5,
            "max_grad_norm": 1.0}
# the [P] float32 device tensor of Population that holds each hyperparameter (lr: the current, decayed rate)
HPARAM_ATTRS = {"learning_rate": "lr", "learning_rate_decay": "lr_decay", "clip_ratio": "clip_ratio",
                "ent_coef": "ent_coef", "vf_coef": "vf_coef", "max_grad_norm": "max_grad_norm"}
CAPPED_AT_ONE = ("learning_rate_decay", "clip_ratio")         # a perturbed value is clamped to at most 1.0
STATE_KEYS = ("actor.0.weight", "actor.0.bias", "actor.2.weight", "actor.2.bias",
              "critic.0.weight", "critic.0.bias", "critic.2.weight", "critic.2.bias")
# the largest seed s whose minibatch generator seed s * 1000 + 1 (PopulationPPOUpdate, as train_ppo seeds rank 0) fits
# in the 64 bits a torch.Generator takes
MAX_SEED = (2 ** 64 - 2) // 1000                    # 18446744073709551
SEED_RANGE = f"seeds must be in 0 .. {MAX_SEED} (the minibatch generator of seed s is seeded s * 1000 + 1 < 2^64)"


def _p(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def parse_seeds(spec: str) -> list[int]:
    """``"0-31"`` -> 0..31, ``"0,5,9"`` -> [0, 5, 9]; ranges and single seeds may be mixed (``"0-3,7"``)."""
    seeds = []
    for part in str(spec).split(","):
        part = part.strip()
        if not part:
            raise ValueError(f"empty entry in --seeds {spec!r}")
        if "-" in part[1:]:
            a, b = part.split("-", 1) if not part.startswith("-") else (None, None)
            if a is None or int(b) < int(a):
                raise ValueError(f"bad seed range {part!r}")
            seeds.extend(range(int(a), int(b) + 1))
        else:
            seeds.append(int(part))
    if any(s < 0 or s > MAX_SEED for s in seeds):
        raise ValueError(SEED_RANGE)
    if len(set(seeds)) != len(seeds):
        raise ValueError(f"--seeds {spec!r} repeats a seed")
    return seeds


def parse_list(spec) -> list[float]:
    """One float or a comma-separated list of them."""
    vals = [float(v) for v in str(spec).split(",") if v.strip()]
    if not vals:
        raise ValueError(f"empty list {spec!r}")
    return vals


def expand_grid(seeds: list[int], lists: dict[str, list[float]]) -> tuple[list[dict], list[tuple[int, dict]]]:
    """(settings, members): the cross product of the hyperparameter lists (in HPARAMS order, the first list varying
    slowest) and, for each setting, one member per seed.  Member m has setting m // len(seeds), seed
    seeds[m % len(seeds)]."""
    names = [k for k in HPARAMS]
    settings = [dict(zip(names, combo)) for combo in itertools.product(*[lists.get(k, [DEFAULTS[k]]) for k in names])]
    members = [(s, h) for h in settings for s in seeds]
    return settings, members


class Population:
    """Stacked parameters ``[P, ...]`` and optimiser state of P members on one device.

    ``hparams`` is one dict for every member or a list of P dicts with the keys of :data:`HPARAMS` (missing keys take
    ``train_ppo``'s defaults).  Member p's weights are those of ``train_ppo --seed seeds[p]``: ``torch.manual_seed(s)``,
    then ``ActorCritic(18, 9)`` on the CPU, then moved to the device."""

    def __init__(self, seeds, n_envs_per_member: int, hparams=None, device="cuda"):
        from .train_ppo import ActorCritic

        seeds = [int(s) for s in seeds]
        if not seeds:
            raise ValueError("a population needs at least one member")
        if int(n_envs_per_member) < 1:
            raise ValueError("n_envs_per_member must be at least 1")
        if any(s < 0 or s > MAX_SEED for s in seeds):
            raise ValueError(SEED_RANGE)
        hp = hparams if isinstance(hparams, (list, tuple)) else [hparams or {}] * len(seeds)
        if len(hp) != len(seeds):
            raise ValueError("hparams must be one dict or one dict per member")
        unknown = {k for h in hp for k in h} - set(HPARAMS)
        if unknown:
            raise ValueError(f"unknown hyperparameters {sorted(unknown)}")
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise _lib.CarEnvError("a Population lives on a CUDA device (there is no CPU implementation)")
        self.L = _lib.lib()
        self.seeds, self.n_envs, self.P = seeds, int(n_envs_per_member), len(seeds)
        self.hparams = [{**DEFAULTS, **h} for h in hp]
        nets = []
        for s in seeds:
            torch.manual_seed(s)
            nets.append(ActorCritic(OBS, ACTIONS))
        with torch.no_grad():
            self.params = [torch.stack([dict(n.state_dict())[k] for n in nets]).float().contiguous().to(self.device)
                           for k in STATE_KEYS]
        n_par = self.L.carenv_ppo_num_params()
        f = lambda k: torch.tensor([h[k] for h in self.hparams], dtype=torch.float32, device=self.device)
        self.lr, self.clip_ratio, self.vf_coef = f("learning_rate"), f("clip_ratio"), f("vf_coef")
        self.ent_coef, self.max_grad_norm = f("ent_coef"), f("max_grad_norm")
        self.lr_decay = f("learning_rate_decay")
        self.exp_avg = torch.zeros((self.P, n_par), device=self.device)
        self.exp_avg_sq = torch.zeros((self.P, n_par), device=self.device)
        self.step_count = torch.zeros(self.P, dtype=torch.int32, device=self.device)
        self.sums = torch.zeros((self.P, 4), device=self.device)      # policy loss, value loss, entropy, total loss
        self.seeds_dev = torch.tensor([s if s < 2 ** 63 else s - 2 ** 64 for s in seeds], dtype=torch.int64,
                                      device=self.device)

    @property
    def num_envs(self) -> int:
        return self.P * self.n_envs

    def member_state_dict(self, p: int) -> dict:
        """Member p's weights under the reference Agent's keys (actor.0.weight ... critic.2.bias), on the CPU: what
        ``train_ppo`` saves and ``evaluate.load_checkpoint`` loads."""
        if not 0 <= p < self.P:
            raise IndexError(f"member {p} of {self.P}")
        return {k: t[p].detach().cpu().clone() for k, t in zip(STATE_KEYS, self.params)}

    def member_actor(self, p: int):
        """An ``nn.Sequential`` actor on the device with member p's weights (for :func:`evaluate_policy`)."""
        from .train_ppo import ActorCritic

        net = ActorCritic(OBS, ACTIONS).to(self.device)
        net.load_state_dict(self.member_state_dict(p))
        return net.actor

    def pack(self, tensor_cores: bool = True, out: torch.Tensor | None = None) -> torch.Tensor:
        """Every member's packed weights ``[P, floats]`` in one launch (``carenv_pack_policy_pop``); row p equals
        ``pack_policy_weights_tc`` (``pack_policy_weights`` without tensor cores) of member p."""
        n = self.L.carenv_policy_weights_floats_tc() if tensor_cores else self.L.carenv_policy_weights_floats()
        if out is None:
            out = torch.empty((self.P, n), device=self.device)
        elif tuple(out.shape) != (self.P, n) or out.dtype != torch.float32 or not out.is_contiguous() \
                or out.device != self.device:
            raise ValueError(f"out must be a contiguous float32 [{self.P}, {n}] tensor on {self.device}")
        with torch.cuda.device(self.device):
            rc = self.L.carenv_pack_policy_pop(int(tensor_cores), self.P, *[_p(t) for t in self.params], _p(out),
                                               _stream(self.device))
        _lib.check(rc, "carenv_pack_policy_pop")
        return out

    def decay_lr(self):
        """StepLR(gamma = learning_rate_decay) of every member, as ``train_ppo`` applies after each epoch."""
        self.lr.mul_(self.lr_decay)

    def current_hparams(self) -> list[dict]:
        """Every member's hyperparameters as the kernels use them now (``learning_rate``: the current, decayed rate),
        one dict per member with the keys of :data:`HPARAMS`, as Python floats of the float32 values."""
        cols = torch.stack([getattr(self, HPARAM_ATTRS[k]) for k in HPARAMS], 1).tolist()
        return [dict(zip(HPARAMS, row)) for row in cols]

    def _state_tensors(self):
        return list(self.params) + [self.exp_avg, self.exp_avg_sq]

    def state_rows(self, idx) -> tuple[torch.Tensor, torch.Tensor]:
        """The full training state of members ``idx`` as new tensors: float32 ``[k, S]`` (the eight parameter tensors,
        ``exp_avg``, ``exp_avg_sq``, then the hyperparameters in HPARAMS order) and their int32 step counts ``[k]``."""
        i = torch.as_tensor(list(idx), dtype=torch.int64).to(self.device)
        parts = [t[i].reshape(len(i), -1) for t in self._state_tensors()]
        parts.append(torch.stack([getattr(self, HPARAM_ATTRS[k])[i] for k in HPARAMS], 1))
        return torch.cat(parts, 1), self.step_count[i]

    def set_rows(self, dst, rows: torch.Tensor, steps: torch.Tensor, factors=None) -> None:
        """Write :meth:`state_rows` images into members ``dst``, then scale hyperparameter ``name`` of ``dst[j]`` by
        ``factors[j][name]`` (a float32 product on the device; a scaled ``clip_ratio`` or ``learning_rate_decay`` is
        clamped to at most 1.0).  Names missing from a member's dict keep the copied value bit for bit."""
        dst = list(dst)
        if not dst:
            return
        factors = list(factors) if factors is not None else [{}] * len(dst)
        if len(factors) != len(dst) or rows.shape[0] != len(dst) or steps.shape[0] != len(dst):
            raise ValueError("one state row, step count and factor dict per destination")
        if len(set(dst)) != len(dst) or not all(0 <= d < self.P for d in dst):
            raise ValueError(f"destinations must be distinct members of 0 .. {self.P - 1}")
        unknown = {k for f in factors for k in f} - set(HPARAMS)
        if unknown:
            raise ValueError(f"unknown hyperparameters {sorted(unknown)}")
        d = torch.as_tensor(dst, dtype=torch.int64).to(self.device)
        with torch.no_grad():
            off = 0
            for t in self._state_tensors():
                w = t[0].numel()
                t[d] = rows[:, off:off + w].reshape(len(dst), *t.shape[1:])
                off += w
            self.step_count[d] = steps.to(torch.int32)
            for k, name in enumerate(HPARAMS):
                v = rows[:, off + k]
                if any(name in f for f in factors):
                    v = v * torch.tensor([f.get(name, 1.0) for f in factors], dtype=torch.float32, device=self.device)
                    if name in CAPPED_AT_ONE:
                        cap = [1.0 if name in f else float("inf") for f in factors]
                        v = torch.minimum(v, torch.tensor(cap, dtype=torch.float32, device=self.device))
                getattr(self, HPARAM_ATTRS[name])[d] = v

    def copy_members(self, dst, src, factors=None) -> None:
        """PBT's exploit and explore: member ``src[j]``'s weights, Adam moments, step count and hyperparameters (the
        current learning rate included) into member ``dst[j]``, then :meth:`set_rows`'s scaling by ``factors[j]``.
        Every source is read before any destination is written.  Seeds, environments and minibatch generators stay
        with their slots."""
        dst, src = list(dst), list(src)
        if not all(0 <= s < self.P for s in src):
            raise ValueError(f"sources must be members of 0 .. {self.P - 1}")
        if len(src) != len(dst):
            raise ValueError("one source per destination")
        if src:
            self.set_rows(dst, *self.state_rows(src), factors)


def _stream(dev):
    return C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)


def use_warp_kernel(env, n_envs_per_member: int) -> bool:
    """``train_ppo``'s rule, applied to one member's environments: one warp per environment for up to
    WARP_ROLLOUT_MAX_ENVS environments on tracks of at most 32 wall segments, the tensor-core kernel otherwise."""
    return n_envs_per_member <= WARP_ROLLOUT_MAX_ENVS and len(env.track.walls) <= 32


def population_rollout(env, pop: Population, buf, cur_obs: torch.Tensor, cur_term: torch.Tensor,
                       cur_trunc: torch.Tensor, step0: int, last_val: torch.Tensor | None = None,
                       u_dbg: torch.Tensor | None = None, packed: torch.Tensor | None = None) -> None:
    """Fill every row of ``buf`` (``Buffer(.., T, P * n, ..)``) for all members with one launch.  Member p's columns
    are bit-identical to ``fused_rollout_warp`` / ``fused_rollout`` of member p alone with ``seed = seeds[p]``,
    ``env_offset = 0`` and n environments.  ``packed`` is an optional ``[P, floats]`` buffer the tensor-core path packs
    into (allocated per call otherwise).  A ``Buffer(bootstrap_truncated=True)`` runs the ``*_final`` twin, which also
    fills its final-observation slots."""
    from .policy import final_slot_args
    from .vec_env import MultiTrackVecEnv

    if isinstance(env, MultiTrackVecEnv):
        raise ValueError("a population trains on one track")
    n, T, N = pop.n_envs, buf.capacity, pop.num_envs
    if env.num_envs != N:
        raise ValueError(f"the environment has {env.num_envs} environments; the population needs {N}")
    if env.device != pop.device:
        raise ValueError("the environment and the population live on different devices")
    for name, t, shape in (("cur_obs", cur_obs, (N, OBS)), ("cur_term", cur_term, (N,)), ("cur_trunc", cur_trunc, (N,)),
                           ("last_val", last_val, (N,)), ("u_dbg", u_dbg, (T, N))):
        if t is not None and (tuple(t.shape) != shape or t.dtype != torch.float32 or not t.is_contiguous()
                              or t.device != env.device):
            raise ValueError(f"{name} must be a contiguous float32 tensor of shape {shape} on {env.device}")
    if getattr(buf, "compact_obs", False) or tuple(buf.obs_buf.shape) != (T, N, OBS):
        raise ValueError("a population needs a Buffer of full observation rows of shape (T, P * n, 18)")
    env.set_option("pose_rows", 0)
    common = (_p(env.pos), _p(env.vel), _p(env.ints), _p(cur_obs), _p(cur_term), _p(cur_trunc),
              float(env.reward_scaling), _p(buf.obs_buf), _p(buf.act_buf), _p(buf.rew_buf), _p(buf.val_buf),
              _p(buf.term_buf), _p(buf.trunc_buf), _p(buf.logprob_buf), _p(last_val), _p(u_dbg), env._stream())
    L = pop.L
    slots = final_slot_args(buf)
    sfx = "_final" if slots else ""
    with torch.cuda.device(env.device):
        if use_warp_kernel(env, n):
            what = "carenv_policy_rollout_warp_pop" + sfx
            rc = getattr(L, what)(env._handle, pop.P, *[_p(t) for t in pop.params], n, T, _p(pop.seeds_dev),
                                  int(step0), *common, *slots)
        else:
            packed = pop.pack(True, out=packed)
            what = "carenv_policy_rollout_tc_pop" + sfx
            rc = getattr(L, what)(env._handle, pop.P, _p(packed), n, T, _p(pop.seeds_dev), int(step0), *common,
                                  *slots)
    _lib.check(rc, what)
    buf.ptr = T


class PopulationPPOUpdate:
    """All minibatch updates of an epoch for every member in one launch (``carenv_ppo_epoch_pop``).

    Member p draws its minibatches with its own ``torch.Generator`` seeded ``seeds[p] * 1000 + 1`` — the seed
    ``train_ppo --seed seeds[p]`` gives the default generator on rank 0 — with ``train_ppo``'s call
    ``randint(0, T * n, (n_updates, batch))``, and sample k of its ``[T, n]`` block is global row
    ``(k // n) * N + p * n + k % n``.  So member p gets the minibatches of the single run."""

    def __init__(self, pop: Population, batch_size: int, betas=(0.9, 0.999), eps: float = 1e-5):
        if not 2 <= int(batch_size) <= 1024:
            raise ValueError("batch_size must be in 2..1024")
        self.pop, self.batch, self.betas, self.eps = pop, int(batch_size), betas, eps
        self.generators = [torch.Generator(device=pop.device).manual_seed(s * 1000 + 1) for s in pop.seeds]
        self.kl = None                   # launch(target_kl=...): [P, n_updates, 2] approx KL, clip fraction
        self.n_done = None               # launch(target_kl=...): [P] int32 updates that applied a step

    def draw_indices(self, T: int, n_updates: int) -> torch.Tensor:
        """int64 ``[P, n_updates, batch]`` global rows of the ``[T * N]`` flat arrays."""
        pop = self.pop
        n, N = pop.n_envs, pop.num_envs
        k = torch.stack([torch.randint(0, T * n, (n_updates, self.batch), device=pop.device, generator=g)
                         for g in self.generators])
        base = (torch.arange(pop.P, device=pop.device, dtype=torch.int64) * n).view(-1, 1, 1)
        return ((k // n) * N + base + k % n).contiguous()

    def run_epoch(self, obs, act, old_logp, adv, ret, T: int, n_updates: int,
                  target_kl: float | None = None) -> torch.Tensor:
        """Draw every member's indices and run the epoch; returns the indices."""
        idx = self.draw_indices(T, n_updates)
        if target_kl is None:
            self.launch(obs, idx, act, old_logp, adv, ret)
        else:
            self.launch(obs, idx, act, old_logp, adv, ret, target_kl=target_kl)
        return idx

    def launch(self, obs, idx, act, old_logp, adv, ret, target_kl: float | None = None) -> None:
        """One launch for the updates ``idx[:, u]`` of every member (``idx`` int64 ``[P, n_updates, batch]``).
        Asynchronous.

        ``target_kl`` (positive, ``inf`` for statistics only) launches ``carenv_ppo_epoch_pop_kl``: ``self.kl``
        [P, n_updates, 2] gets every member's per-update approx KL and clip fraction (NaN after its stopping update),
        ``self.n_done`` [P] int32 its applied updates; each member stops at its first update whose approx KL exceeds
        ``target_kl``.  ``None`` launches exactly what it launched before."""
        pop = self.pop
        if idx.dtype != torch.int64 or idx.dim() != 3 or idx.shape[0] != pop.P or idx.shape[2] != self.batch \
                or not idx.is_contiguous() or idx.device != pop.device:
            raise ValueError(f"idx must be a contiguous int64 [{pop.P}, n_updates, {self.batch}] tensor on {pop.device}")
        for name, t in (("obs", obs), ("act", act), ("old_logp", old_logp), ("adv", adv), ("ret", ret)):
            if t.dtype != torch.float32 or not t.is_contiguous() or t.device != pop.device:
                raise ValueError(f"{name} must be a contiguous float32 tensor on {pop.device}")
        if obs.shape[-1] != OBS:
            raise ValueError("obs must have 18 columns")
        if target_kl is not None:
            if not float(target_kl) > 0.0:
                raise ValueError("target_kl must be positive (inf: statistics without stopping)")
            shape = (pop.P, int(idx.shape[1]), 2)
            if self.kl is None or tuple(self.kl.shape) != shape:
                self.kl = torch.empty(shape, device=pop.device)
            if self.n_done is None or self.n_done.shape[0] != pop.P:
                self.n_done = torch.zeros(pop.P, dtype=torch.int32, device=pop.device)
        if idx.shape[1] == 0:
            if target_kl is not None:
                self.n_done.zero_()
            return
        args = (pop.P, *[_p(t) for t in pop.params], _p(obs), _p(idx), _p(act), _p(old_logp), _p(adv), _p(ret),
                self.batch, int(idx.shape[1]), _p(pop.lr), _p(pop.clip_ratio), _p(pop.vf_coef), _p(pop.ent_coef),
                _p(pop.max_grad_norm), self.betas[0], self.betas[1], self.eps, _p(pop.exp_avg), _p(pop.exp_avg_sq),
                _p(pop.step_count), _p(pop.sums), _stream(pop.device))
        with torch.cuda.device(pop.device):
            if target_kl is None:
                rc, what = pop.L.carenv_ppo_epoch_pop(*args), "carenv_ppo_epoch_pop"
            else:
                rc = pop.L.carenv_ppo_epoch_pop_kl(*args, float(target_kl), _p(self.kl), _p(self.n_done))
                what = "carenv_ppo_epoch_pop_kl"
        _lib.check(rc, what)


# ---- command line --------------------------------------------------------------------------------------------------
def parse_args(argv=None):
    from .train_ppo import parse_args as train_args

    p = argparse.ArgumentParser(description="train a population of independent PPO policies in one process",
                                add_help=False)
    p.add_argument("--seeds", default="0", help="seeds of the members: a range 0-31, a list 0,5,9, or a mix")
    p.add_argument("--pbt-every", type=int, default=0,
                   help="population-based training: every K epochs score every member (--eval-episodes, "
                        "--eval-greedy) and replace the bottom --pbt-fraction with perturbed copies of the top.  "
                        "Default 0: off (the other --pbt-* flags then do nothing)")
    p.add_argument("--pbt-fraction", type=float, default=0.25,
                   help="fraction f in (0, 0.5] of the members replaced per round, and of those they copy from")
    p.add_argument("--pbt-explore", default="learning_rate,ent_coef",
                   help="comma-separated hyperparameters scaled by 0.8 or 1.2 after a copy (names of --learning-rate "
                        "etc. with underscores; empty: copy only)")
    p.add_argument("--pbt-seed", type=int, default=0,
                   help="seed of the PBT decisions and of the sampled fitness evaluation (the same on every rank)")
    mine, rest = p.parse_known_args(argv)
    # lists are kept here (check_args parses them); train_ppo's parser sees one value of each
    first = lambda k, v: v.split(",")[0].strip() or str(DEFAULTS[k])
    for k in HPARAMS:
        flag = "--" + k.replace("_", "-")
        for i, a in enumerate(rest):
            if a == flag and i + 1 < len(rest):
                setattr(mine, k, rest[i + 1])
                rest[i + 1] = first(k, rest[i + 1])
            elif a.startswith(flag + "="):
                setattr(mine, k, a.split("=", 1)[1])
                rest[i] = flag + "=" + first(k, a.split("=", 1)[1])
    args = train_args(rest)
    args.seeds = mine.seeds
    args.pbt_every, args.pbt_fraction = mine.pbt_every, mine.pbt_fraction
    args.pbt_explore, args.pbt_seed = mine.pbt_explore, mine.pbt_seed
    for k in HPARAMS:
        setattr(args, k + "_list", getattr(mine, k, None) or str(getattr(args, k)))
    return args


def check_args(args) -> tuple[list[dict], list[tuple[int, dict]]]:
    """Refuse what the population path does not do, before any device work; returns expand_grid's result."""
    for flag, on in (("--compact-obs", args.compact_obs), ("--cuda-graph", args.cuda_graph),
                     ("--graph-update", args.graph_update), ("--per-minibatch-update", args.per_minibatch_update),
                     ("--fused-cuda-cores", args.fused_cuda_cores)):
        if on:
            raise SystemExit(f"{flag} does not work with a population: it always runs the fused rollout and the "
                             "one-launch epoch update")
    if not os.path.exists(args.track) and "," in args.track:
        raise SystemExit("a population trains on one track; several tracks are not supported")
    if args.n_envs < 1:
        raise SystemExit("--n-envs (environments per member) must be at least 1")
    try:
        seeds = parse_seeds(args.seeds)
        lists = {k: parse_list(getattr(args, k + "_list")) for k in HPARAMS}
    except ValueError as e:
        raise SystemExit(str(e))
    if not seeds:
        raise SystemExit("the population is empty")
    if not 2 <= args.batch_size <= 1024:
        raise SystemExit("--batch-size must be in 2..1024")
    from .train_ppo import kl_target

    kl_target(args)
    settings, members = expand_grid(seeds, lists)
    if args.pbt_every < 0:
        raise SystemExit("--pbt-every must be >= 0 (0: no population-based training)")
    if args.pbt_every > 0:
        from .pbt import parse_explore

        if not 0.0 < args.pbt_fraction <= 0.5:
            raise SystemExit("--pbt-fraction must be in (0, 0.5]")
        if int(len(members) * args.pbt_fraction) == 0:
            raise SystemExit(f"--pbt-fraction {args.pbt_fraction:g} of {len(members)} members replaces none: "
                             "floor(P * f) must be at least 1")
        try:
            parse_explore(args.pbt_explore)
        except ValueError as e:
            raise SystemExit(str(e))
        if not 0 <= args.pbt_seed < 2 ** 64:
            raise SystemExit("--pbt-seed must be in 0 .. 2^64 - 1")
        if args.eval_episodes < 1:
            raise SystemExit("--eval-episodes must be at least 1 with --pbt-every: it scores the members")
    return settings, members


def summarize(results: list[dict], settings: list[dict]) -> list[dict]:
    """One row per hyperparameter setting: mean and standard deviation over its seeds of the final avg_reward (and of
    the last evaluation's mean return when there was one)."""
    rows = []
    for h in settings:
        rs = [r for r in results if r["hparams"] == h]
        row = {"hparams": h, "members": len(rs)}
        for key, vals in (("avg_reward", [r["avg_reward"] for r in rs]),
                          ("eval_return", [r["eval_return"] for r in rs if r.get("eval_return") is not None])):
            if vals:
                m = sum(vals) / len(vals)
                row[key + "_mean"] = m
                row[key + "_std"] = math.sqrt(sum((v - m) ** 2 for v in vals) / len(vals))
        rows.append(row)
    return rows


def train_population(args) -> dict:
    """Train every member of the grid for ``args.n_epochs`` epochs; returns {"history": [per-epoch member records of
    this rank], "final": [one record per member, all ranks], "summary": rows of :func:`summarize`}.

    With ``args.pbt_every = K > 0`` a population-based-training round (:func:`pbt.pbt_round`) follows every K-th epoch
    but the last; epoch records then gain ``"current_hparams"``, final records ``"current_hparams"`` and
    ``"ancestry"`` (``[epoch, parent]`` per copy), and the result ``"lineage"`` (this rank's lineage records) and
    ``"pbt_best"`` (the best member by the last round's fitness, when there was a round)."""
    from . import Buffer, VecCarEnv, builtin_track
    from . import pbt
    from .shard import shard_range
    from .train_ppo import explained_variance, kl_record, kl_target

    settings, members = check_args(args)
    tau = kl_target(args)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    pbt_on = args.pbt_every > 0
    if pbt_on and world > len(members):
        raise SystemExit(f"--pbt-every needs at least one member per rank ({len(members)} members, {world} ranks)")
    track = args.track if os.path.exists(args.track) else builtin_track(args.track)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1 and not dist.is_initialized():
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    lo, hi = shard_range(len(members), world, rank)
    mine = members[lo:hi]
    n, T = args.n_envs, args.n_steps
    history, final = [], []
    lineage, fitness = [], None
    if mine:
        pop = Population([s for s, _ in mine], n, [h for _, h in mine], dev)
        N = pop.num_envs
        env = VecCarEnv(N, track, device=dev, reward_scaling=args.reward_scaling, float_flags=True, with_info=False)
        buf = Buffer((OBS,), T, N, dev, args.gamma, args.gae_lambda, bootstrap_truncated=args.bootstrap_truncated)
        upd = PopulationPPOUpdate(pop, args.batch_size)
        next_obs = env.reset()[0].clone()
        next_term, next_trunc = torch.zeros(N, device=dev), torch.zeros(N, device=dev)
        last_val = torch.empty(N, device=dev)
        packed = None if use_warp_kernel(env, n) else torch.empty((pop.P, pop.L.carenv_policy_weights_floats_tc()),
                                                                    device=dev)
        n_mb = -(-T // args.batch_size)
        ckpt_root = os.path.join(args.checkpoint_dir, args.run_name) if args.checkpoint_dir else None

        def save(p_local, name):
            if ckpt_root is not None:
                d = os.path.join(ckpt_root, f"member_{lo + p_local}")
                os.makedirs(d, exist_ok=True)
                torch.save(pop.member_state_dict(p_local), os.path.join(d, name))

        def emit(rec):
            print(json.dumps(rec), flush=True)
            if args.log_json:
                with open(args.log_json + (f".rank{rank}" if world > 1 else ""), "a") as fh:
                    fh.write(json.dumps(rec) + "\n")

        if pbt_on:
            counts = [b - a for a, b in (shard_range(len(members), world, r) for r in range(world))]
            explore = pbt.parse_explore(args.pbt_explore)
            gen = torch.Generator().manual_seed(args.pbt_seed)
            ancestry = [[] for _ in range(pop.P)]
        eval_ret = [None] * pop.P
        t_start = time.time()
        try:
            for epoch in range(1, args.n_epochs + 1):
                with torch.no_grad():
                    population_rollout(env, pop, buf, next_obs, next_term, next_trunc, step0=(epoch - 1) * T,
                                       last_val=last_val, packed=packed)
                    if args.bootstrap_truncated:
                        buf.final_values(pop)
                    adv, ret = buf.calculate_advantages(last_val.reshape(1, -1), next_term.reshape(1, -1),
                                                        next_trunc.reshape(1, -1))
                # per member as train_ppo sums its own contiguous [T, n] block: the same reduction, the same bits
                cols = lambda t, p: t.view(T, pop.P, n)[:, p].contiguous()
                stats = torch.stack([torch.stack([cols(buf.rew_buf, p).sum(),
                                                  cols(buf.term_buf, p).sum() + cols(buf.trunc_buf, p).sum()])
                                     for p in range(pop.P)]).double().tolist()
                obs_b, act_b, _, logp_b = buf.get()
                pop.sums.zero_()
                upd.run_epoch(obs_b.view(-1, OBS), act_b.view(-1), logp_b.view(-1), adv.view(-1), ret.view(-1), T,
                              args.train_iters * n_mb, target_kl=tau)
                kl_recs = None
                if tau is not None:                              # per member, over its own [T, n] block
                    val_b = buf.val_buf
                    kl_all, done = upd.kl.tolist(), upd.n_done.tolist()
                    kl_recs = [{**kl_record(kl_all[p], done[p]),
                                "explained_variance": explained_variance(cols(ret, p), cols(val_b, p))}
                               for p in range(pop.P)]
                pop.decay_lr()
                lr_now = pop.lr.tolist()                         # train_ppo records the decayed rate
                sums = (pop.sums / args.train_iters).tolist()
                evals = None
                if args.eval_every > 0 and epoch % args.eval_every == 0:
                    from .evaluate import evaluate_population

                    with torch.no_grad():                    # every member in one launch, with its own seed
                        res = evaluate_population(env, pop.params[:4], args.eval_episodes, greedy=args.eval_greedy,
                                                  seeds=pop.seeds)
                        eval_sums = torch.stack([r.sums() for r in res]).cpu()
                    evals = [r.summary(s) for r, s in zip(res, eval_sums)]
                current = pop.current_hparams() if pbt_on else None
                wall = time.time() - t_start
                for p in range(pop.P):
                    seed, h = mine[p]
                    rec = {"epoch": epoch, "member": lo + p, "seed": seed, "hparams": h,
                           "avg_reward": stats[p][0] / float(T * n) / args.reward_scaling, "episodes": stats[p][1],
                           "policy_loss": sums[p][0], "value_loss": sums[p][1], "entropy": sums[p][2],
                           "total_loss": sums[p][3], "lr": lr_now[p], "wall_s": wall}
                    if evals is not None:
                        rec["eval"] = evals[p]
                        eval_ret[p] = rec["eval"]["mean_return"]
                    if kl_recs is not None:
                        rec.update(kl_recs[p])
                    if pbt_on:
                        rec["current_hparams"] = current[p]
                    history.append(rec)
                    emit(rec)
                # a round after the last epoch would only overwrite final weights that nothing trains further
                if pbt_on and epoch % args.pbt_every == 0 and epoch < args.n_epochs:
                    fitness, lines = pbt.pbt_round(pop, env, args, epoch // args.pbt_every - 1, epoch, lo, counts,
                                                   gen, explore)
                    for line in lines:
                        ancestry[line["member"] - lo].append([epoch, line["parent"]])
                        lineage.append(line)
                        emit(line)
                if epoch % 10 == 0:
                    for p in range(pop.P):
                        save(p, f"checkpoint_{epoch}.dat")
        finally:
            for p in range(pop.P):
                save(p, "model.dat")
        env.close()
        last = history[-pop.P:] if history else []
        final = [{"member": r["member"], "seed": r["seed"], "hparams": r["hparams"], "avg_reward": r["avg_reward"],
                  "eval_return": eval_ret[i]} for i, r in enumerate(last)]
        if pbt_on:
            current = pop.current_hparams()
            for i, r in enumerate(final):
                r["current_hparams"], r["ancestry"] = current[i], ancestry[i]
    if world > 1:
        gathered = [None] * world
        dist.all_gather_object(gathered, final)
        final = [r for part in gathered for r in part]
    summary = summarize(final, settings)
    if rank == 0:
        for row in summary:
            h = ", ".join(f"{k}={v:g}" for k, v in row["hparams"].items())
            line = f"[{h}] {row['members']} seeds: final avg_reward {row.get('avg_reward_mean', float('nan')):.4f} " \
                   f"+- {row.get('avg_reward_std', float('nan')):.4f}"
            if "eval_return_mean" in row:
                line += f", eval return {row['eval_return_mean']:.3f} +- {row['eval_return_std']:.3f}"
            print(line, flush=True)
    out = {"history": history, "final": final, "summary": summary}
    if pbt_on:
        out["lineage"] = lineage
        if fitness is not None:                      # every rank holds every member's fitness of the last round
            best = min(range(len(fitness)), key=lambda g: (-fitness[g], g))
            out["pbt_best"] = {"member": best, "fitness": fitness[best],
                               "current_hparams": next(r for r in final if r["member"] == best)["current_hparams"]}
            if rank == 0:
                h = ", ".join(f"{k}={v:g}" for k, v in out["pbt_best"]["current_hparams"].items())
                print(f"best member by last PBT fitness: {best} (mean return {fitness[best]:.3f}) now [{h}]",
                      flush=True)
    return out


def main(argv=None):
    train_population(parse_args(argv))
    if dist.is_initialized():
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
