"""Fused PPO minibatch update (C ABI carenv_ppo_grad / carenv_ppo_adam, csrc/ppo_update.cuh).

Restates train.py:223-261 for the reference network (lib/model.py:10-26): clipped surrogate, value loss,
entropy bonus, per-minibatch advantage normalisation, clip_grad_norm_, Adam — three kernel launches per
minibatch (plus one NCCL all-reduce of the 12,298 gradients when there are several ranks) instead of an
autograd graph of about sixty — or, with :meth:`FusedPPOUpdate.run_epoch`, ALL minibatch updates of an epoch in one
persistent cooperative launch whose gradient all-reduce runs inside the kernel over NVLink peer memory
(C ABI carenv_ppo_epoch, csrc/ppo_epoch.cuh).  The parameters stay ordinary ``nn.Parameter`` tensors and are
updated in place.
"""
from __future__ import annotations

import ctypes as C

import torch
import torch.distributed as dist

from . import _lib


IPC_HANDLE_BYTES = 64


def _p(t):
    return C.c_void_p(t.data_ptr())


def exchange_ipc_handles(handle: bytes, group=None) -> bytes:
    """All ranks' 64-byte CUDA IPC handles concatenated in rank order (plumbing: torch.distributed object gather)."""
    if len(handle) != IPC_HANDLE_BYTES:
        raise ValueError("an IPC handle has 64 bytes")
    world = dist.get_world_size(group)
    out = [None] * world
    dist.all_gather_object(out, bytes(handle), group=group)
    if any(not isinstance(h, (bytes, bytearray)) or len(h) != IPC_HANDLE_BYTES for h in out):
        raise _lib.CarEnvError("a rank sent a malformed IPC handle")
    return b"".join(bytes(h) for h in out)


class FusedPPOUpdate:
    def __init__(self, actor, critic, batch_size: int, lr: float, clip_ratio: float = 0.2, vf_coef: float = 0.5,
                 ent_coef: float = 0.001, max_grad_norm: float = 1.0, betas=(0.9, 0.999), eps: float = 1e-5):
        self.L = _lib.lib()
        self.params = [actor[0].weight, actor[0].bias, actor[2].weight, actor[2].bias,
                       critic[0].weight, critic[0].bias, critic[2].weight, critic[2].bias]
        shapes = [tuple(p.shape) for p in self.params]
        if shapes != [(256, 18), (256,), (9, 256), (9,), (256, 18), (256,), (1, 256), (1,)]:
            raise ValueError("the fused update supports the reference network only: 18-256-9 actor, 18-256-1 critic")
        dev = self.params[0].device
        if dev.type != "cuda" or any(p.dtype != torch.float32 or not p.is_contiguous() for p in self.params):
            raise _lib.CarEnvError("parameters must be contiguous float32 CUDA tensors")
        n = self.L.carenv_ppo_num_params()
        scratch = self.L.carenv_ppo_scratch_floats(int(batch_size))
        if scratch < 0:
            raise ValueError("batch_size must be in 2..1024")
        self.device, self.batch = dev, int(batch_size)
        self.grads = torch.zeros(n, device=dev)
        self.exp_avg, self.exp_avg_sq = torch.zeros(n, device=dev), torch.zeros(n, device=dev)
        self.scratch = torch.zeros(scratch, device=dev)
        self.lr = torch.tensor([lr], dtype=torch.float32, device=dev)
        self.step_count = torch.zeros(1, dtype=torch.int32, device=dev)
        self.sums = torch.zeros(4, device=dev)                  # policy loss, value loss, entropy, total loss
        self.clip_ratio, self.vf_coef, self.ent_coef, self.max_grad_norm = clip_ratio, vf_coef, ent_coef, max_grad_norm
        self.betas, self.eps = betas, eps
        self._epoch_ws = None            # workspace of run_epoch, allocated on first use
        self._sync = None
        self._comm = None
        self._comm_world = 1
        self.kl = None                   # run_epoch(target_kl=...): [n_updates, 2] approx KL, clip fraction
        self.n_done = None               # run_epoch(target_kl=...): [1] int32 updates that applied a step

    # ---- one launch per epoch ---------------------------------------------------------------------------------
    def connect(self, group=None):
        """Several GPUs: allocate this rank's gradient exchange buffer, swap IPC handles with the peers (all ranks of
        ONE node) and map theirs.  Collective: every rank calls it once before the first run_epoch(world > 1)."""
        world, rank = dist.get_world_size(group), dist.get_rank(group)
        if world == 1 or self._comm is not None:
            return
        comm, handle = C.c_void_p(), C.create_string_buffer(IPC_HANDLE_BYTES)
        with torch.cuda.device(self.device):
            _lib.check(self.L.carenv_ppo_comm_create(world, rank, C.byref(comm), handle), "carenv_ppo_comm_create")
            everyone = exchange_ipc_handles(handle.raw, group)
            _lib.check(self.L.carenv_ppo_comm_connect(comm, everyone), "carenv_ppo_comm_connect")
        self._comm, self._comm_world = comm, world
        dist.barrier(group)              # every peer has mapped every buffer before anyone launches

    def close(self, group=None):
        """Collective when connected: a peer may still be reading this rank's exchange buffer (a rank's last update
        completes when the peers' flags have arrived, not when they have finished reading), so every rank drains its
        device and meets the others before anything is unmapped or freed."""
        if self._comm is not None:
            torch.cuda.synchronize(self.device)
            if dist.is_initialized():
                dist.barrier(group)
            self.L.carenv_ppo_comm_destroy(self._comm)
            self._comm = None

    def __del__(self):                   # not collective: a communicator that was never closed is left to process exit
        self._comm = None

    def run_epoch(self, obs, idx, act, old_logp, adv, ret, world: int = 1, n_ctas: int = 0, prof=None,
                  target_kl: float | None = None):
        """All ``idx.shape[0]`` minibatch updates (rows of ``idx`` [n_updates, batch] int64) in ONE launch: forward,
        loss, backward, gradient all-reduce over NVLink peer memory (``world`` > 1, after :meth:`connect`), clip,
        Adam, statistics into ``self.sums``.  Asynchronous; :meth:`check_epoch` reads the kernel's error word.

        ``target_kl`` (a positive float, ``inf`` for statistics only) launches ``carenv_ppo_epoch_kl``: ``self.kl``
        [n_updates, 2] gets each update's approx KL and clip fraction (NaN after the stopping update), ``self.n_done``
        [1] int32 the updates that applied a step; the epoch stops at the first update whose approx KL exceeds
        ``target_kl``.  ``None`` launches exactly what it launched before."""
        if idx.dtype != torch.int64 or idx.dim() != 2 or idx.shape[1] != self.batch or not idx.is_contiguous() \
                or idx.device != self.device:
            raise ValueError(f"idx must be a contiguous int64 [n_updates, {self.batch}] tensor on {self.device}")
        for name, t in (("obs", obs), ("act", act), ("old_logp", old_logp), ("adv", adv), ("ret", ret)):
            if t.dtype != torch.float32 or not t.is_contiguous() or t.device != self.device:
                raise ValueError(f"{name} must be a contiguous float32 tensor on {self.device}")
        if obs.shape[-1] != 18:
            raise ValueError("obs must have 18 columns")
        if prof is not None and (prof.dtype != torch.int64 or prof.numel() < 4 * idx.shape[0] or prof.device != self.device):
            raise ValueError("prof must be an int64 device tensor of n_updates x 4 elements")
        if world > 1 and (self._comm is None or self._comm_world != world):
            raise _lib.CarEnvError("run_epoch(world > 1) needs connect() on every rank first")
        if target_kl is not None and not float(target_kl) > 0.0:
            raise ValueError("target_kl must be positive (inf: statistics without stopping)")
        if target_kl is not None:
            n_upd = int(idx.shape[0])
            if self.kl is None or self.kl.shape[0] != n_upd:
                self.kl = torch.empty((n_upd, 2), device=self.device)
            if self.n_done is None:
                self.n_done = torch.zeros(1, dtype=torch.int32, device=self.device)
        if idx.shape[0] == 0:            # no updates; an empty idx has no storage (data_ptr 0), which the C ABI refuses
            if target_kl is not None:
                self.n_done.zero_()
            return
        if self._epoch_ws is None:
            self._epoch_ws = torch.zeros(self.L.carenv_ppo_epoch_workspace_floats(), device=self.device)
            self._sync = torch.zeros(2, dtype=torch.int32, device=self.device)
        args = (*[_p(p) for p in self.params], _p(obs), _p(idx), _p(act), _p(old_logp), _p(adv), _p(ret), self.batch,
                int(idx.shape[0]), self.clip_ratio, self.vf_coef, self.ent_coef, _p(self.exp_avg), _p(self.exp_avg_sq),
                _p(self.lr), _p(self.step_count), self.betas[0], self.betas[1], self.eps, self.max_grad_norm,
                _p(self.sums), _p(self._epoch_ws), _p(self._sync), self._comm if world > 1 else None, int(n_ctas),
                _p(prof) if prof is not None else None, self._stream())
        with torch.cuda.device(self.device):
            if target_kl is None:
                rc, what = self.L.carenv_ppo_epoch(*args), "carenv_ppo_epoch"
            else:
                rc = self.L.carenv_ppo_epoch_kl(*args, float(target_kl), _p(self.kl), _p(self.n_done))
                what = "carenv_ppo_epoch_kl"
        _lib.check(rc, what)

    def check_epoch(self):
        """Synchronises and raises if a wait inside run_epoch's kernel timed out (a peer rank that never launched)."""
        if self._sync is not None and int(self._sync[1].item()) != 0:
            raise _lib.CarEnvError("carenv_ppo_epoch: a grid or peer wait timed out; parameters are not updated consistently")

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def grad(self, obs, idx, act, old_logp, adv, ret, obs_is_gathered: bool = False):
        """Gradients of one minibatch into ``self.grads``.  ``idx`` [batch] int64 indexes the flat arrays."""
        if idx.dtype != torch.int64 or idx.numel() != self.batch or not idx.is_contiguous() or idx.device != self.device:
            raise ValueError(f"idx must be a contiguous int64 tensor of {self.batch} elements on {self.device}")
        for name, t in (("obs", obs), ("act", act), ("old_logp", old_logp), ("adv", adv), ("ret", ret)):
            if t.dtype != torch.float32 or not t.is_contiguous() or t.device != self.device:
                raise ValueError(f"{name} must be a contiguous float32 tensor on {self.device}")
        if obs.shape[-1] != 18 or (obs_is_gathered and obs.numel() != self.batch * 18):
            raise ValueError("obs must have 18 columns (and `batch` rows when it is already gathered)")
        with torch.cuda.device(self.device):
            rc = self.L.carenv_ppo_grad(*[_p(p) for p in self.params], _p(obs), int(obs_is_gathered), _p(idx), _p(act),
                                        _p(old_logp), _p(adv), _p(ret), self.batch, self.clip_ratio, self.vf_coef,
                                        self.ent_coef, _p(self.scratch), _p(self.grads), self._stream())
        _lib.check(rc, "carenv_ppo_grad")
        return self.grads

    def apply(self, world: int = 1):
        """(All-reduce,) clip, Adam step, statistics."""
        if world > 1:
            dist.all_reduce(self.grads, op=dist.ReduceOp.SUM)
        with torch.cuda.device(self.device):
            rc = self.L.carenv_ppo_adam(*[_p(p) for p in self.params], _p(self.grads), 1.0 / world, _p(self.exp_avg),
                                        _p(self.exp_avg_sq), _p(self.lr), _p(self.step_count), self.betas[0],
                                        self.betas[1], self.eps, self.max_grad_norm, _p(self.scratch), self.batch,
                                        self.vf_coef, self.ent_coef, _p(self.sums), self._stream())
        _lib.check(rc, "carenv_ppo_adam")
