"""Rollout buffer with the GAE reverse-scan kernel.

Same constructor, attributes and methods as the reference's ``lib.buffer.Buffer``
(/root/reference/lib/buffer.py:4-73): seven ``[size, num_envs(, obs_dim)]`` float32 tensors,
``store``, ``calculate_advantages`` (asserts the buffer is full, lib/buffer.py:46) and ``get``
(asserts and rewinds ``ptr``, lib/buffer.py:71-72).  ``calculate_advantages`` runs one
sm_100a kernel (``gae_reverse_scan``) that reproduces the reference's float32 operation order
bit for bit instead of ~12 tiny torch kernels per timestep.  CUDA only — no CPU fallback.

``Buffer(..., bootstrap_truncated=True)`` (no counterpart in the reference) adds time-limit bootstrapping (Pardo et
al. 2018): the last step of an episode cut by the 1000-step limit is bootstrapped from the critic's value of the
observation the episode ended in (``boot_buf``) instead of the value of the next episode's reset observation.
"""
from __future__ import annotations

import ctypes as C
import math

import torch

from . import _lib


def _ptr(t):
    return C.c_void_p(t.data_ptr())


TIME_LIMIT = 1000                     # CARENV_TIME_LIMIT: an episode is truncated at its 1000th step


def final_slots(n_steps: int) -> int:
    """S = ceil(n_steps / 1000): the most truncations one environment can have in n_steps steps, whatever its starting
    time step (the first after at most 1000 steps, then one every 1000 at the soonest)."""
    return math.ceil(n_steps / TIME_LIMIT)


def gae_reverse_scan(rew, val, term, trunc, last_val, last_term, last_trunc, gamma=0.99, gae_lambda=0.95,
                     adv_out=None, ret_out=None, boot=None):
    """adv, ret = GAE(lambda) over [T, N] float32 CUDA tensors (lib/buffer.py:51-63).

    ``boot`` [T, N] (C ABI gae_reverse_scan_boot): a row whose successor has trunc == 1 and term == 0 (for row T - 1:
    last_trunc / last_term) takes ``boot[t]`` as its next value instead of ``val[t + 1]`` / ``last_val``; no other
    entry of ``boot`` is read.  Without truncation flags the result is the same bits as without ``boot``."""
    L = _lib.lib()
    if not rew.is_cuda:
        raise _lib.CarEnvError("gae_reverse_scan only runs on CUDA tensors (there is no CPU implementation)")
    T, N = rew.shape
    for name, out in (("adv_out", adv_out), ("ret_out", ret_out)):      # the kernel writes T * N floats through them
        if out is not None and (not isinstance(out, torch.Tensor) or out.dtype != torch.float32
                                or tuple(out.shape) != (T, N) or not out.is_contiguous() or out.device != rew.device):
            raise ValueError(f"{name} must be a contiguous float32 ({T}, {N}) tensor on {rew.device}")
    f32 = lambda t, shape: t.to(device=rew.device, dtype=torch.float32).reshape(shape).contiguous()
    rew, val, term, trunc = (f32(t, (T, N)) for t in (rew, val, term, trunc))
    last_val, last_term, last_trunc = (f32(t, (N,)) for t in (last_val, last_term, last_trunc))
    adv = adv_out if adv_out is not None else torch.empty_like(rew)
    ret = ret_out if ret_out is not None else torch.empty_like(rew)
    with torch.cuda.device(rew.device):
        stream = C.c_void_p(torch.cuda.current_stream(rew.device).cuda_stream)
        if boot is None:
            rc = L.gae_reverse_scan(_ptr(rew), _ptr(val), _ptr(term), _ptr(trunc), _ptr(last_val), _ptr(last_term),
                                    _ptr(last_trunc), _ptr(adv), _ptr(ret), T, N, float(gamma), float(gae_lambda),
                                    stream)
        else:
            boot = f32(boot, (T, N))
            rc = L.gae_reverse_scan_boot(_ptr(rew), _ptr(val), _ptr(term), _ptr(trunc), _ptr(last_val),
                                         _ptr(last_term), _ptr(last_trunc), _ptr(boot), _ptr(adv), _ptr(ret), T, N,
                                         float(gamma), float(gae_lambda), stream)
    _lib.check(rc, "gae_reverse_scan" if boot is None else "gae_reverse_scan_boot")
    return adv, ret


def final_values(critic, final_obs, final_row, boot, n_envs_per_member=None):
    """``boot[final_row[k, c], c] = critic(final_obs[k, c])`` for every used slot (row >= 0) in one launch (C ABI
    carenv_final_values, float32 CUDA cores); other entries of ``boot`` [T, N] are not written.  ``critic`` is an
    ``nn.Sequential(Linear(18, 256), ReLU, Linear(256, 1))`` or a ``Population``, whose member p owns columns
    p * n .. p * n + n - 1 (n = ``n_envs_per_member``, the population's own by default)."""
    L = _lib.lib()
    S, N = final_row.shape
    if hasattr(critic, "params"):                       # Population: stacked critic tensors [P, ...]
        params, P = critic.params[4:8], critic.P
        n = int(n_envs_per_member or critic.n_envs)
    else:
        params, P, n = [critic[0].weight, critic[0].bias, critic[2].weight, critic[2].bias], 1, N
    if tuple(params[0].shape[-2:]) != (256, 18) or tuple(params[2].shape[-2:]) != (1, 256):
        raise ValueError("final_values supports the reference critic only: 18-256-1")
    if P * n != N or tuple(final_obs.shape) != (S, N, 18) or boot.dim() != 2 or boot.shape[1] != N:
        raise ValueError(f"final_obs must be [{S}, {N}, 18], boot [T, {N}], and members x n_envs = {N}")
    for t, dt in ((final_obs, torch.float32), (final_row, torch.int32), (boot, torch.float32)):
        if t.dtype != dt or not t.is_contiguous() or t.device != boot.device:
            raise ValueError("final_obs float32, final_row int32 and boot float32 must be contiguous on one device")
    params = [p.detach().float().contiguous() for p in params]
    with torch.cuda.device(boot.device):
        rc = L.carenv_final_values(P, *[_ptr(p) for p in params], _ptr(final_obs), _ptr(final_row), S, n,
                                   boot.shape[0], _ptr(boot), C.c_void_p(torch.cuda.current_stream(boot.device).cuda_stream))
    _lib.check(rc, "carenv_final_values")


class Buffer:
    """Buffer for storing trajectories (drop-in for lib.buffer.Buffer)."""

    def __init__(self, obs_dim, size, num_envs, device, gamma=0.99, gae_lambda=0.95, compact_obs=False,
                 bootstrap_truncated=False):
        """``compact_obs=True`` (no counterpart in the reference; SURVEY §8 f-3): no [size, num_envs, 18] observation
        tensor; ``pose_buf`` [size, num_envs, 4] float64 holds one 32-byte pose record per row instead, written by
        ``fused_rollout`` and turned back into observations by ``VecCarEnv.observe(pose_buf, index)``.

        ``bootstrap_truncated=True``: ``boot_buf`` [size, num_envs] holds, at row t of a step that truncated an
        episode, the critic's value of the observation the episode ended in, and ``calculate_advantages`` bootstraps
        that step from it (``gae_reverse_scan(boot=...)``).  The fused rollouts fill the final-observation slots
        ``final_obs_buf`` [S, num_envs, 18] and ``final_row_buf`` [S, num_envs] int32 (S = ceil(size / 1000)), and
        :meth:`final_values` turns them into ``boot_buf``; an eager loop writes ``boot_buf`` itself."""
        device = torch.device(device)
        if device.type != "cuda":
            raise _lib.CarEnvError("ppo_car_b200.Buffer lives on a CUDA device (there is no CPU implementation)")
        _lib.lib()
        self.capacity = size
        z = lambda *shape: torch.zeros(shape, dtype=torch.float32, device=device)
        self.compact_obs = bool(compact_obs)
        self.obs_buf = None if compact_obs else z(size, num_envs, *obs_dim)
        self.pose_buf = torch.zeros((size, num_envs, 4), dtype=torch.float64, device=device) if compact_obs else None
        self.act_buf = z(size, num_envs)
        self.rew_buf = z(size, num_envs)
        self.val_buf = z(size, num_envs)
        self.term_buf = z(size, num_envs)
        self.trunc_buf = z(size, num_envs)
        self.logprob_buf = z(size, num_envs)
        self.gamma, self.gae_lambda = gamma, gae_lambda
        self.bootstrap_truncated = bool(bootstrap_truncated)
        self.boot_buf = self.final_obs_buf = self.final_row_buf = None
        if bootstrap_truncated:
            S = final_slots(size)
            self.boot_buf = z(size, num_envs)
            self.final_obs_buf = z(S, num_envs, *obs_dim)
            self.final_row_buf = torch.full((S, num_envs), -1, dtype=torch.int32, device=device)
        self.ptr = 0
        self._adv = self._ret = None          # allocated on first use and reused (static addresses: CUDA graphs)

    def store(self, obs, act, rew, val, term, trunc, logprob):
        """Store one step; first dimension is the step, second the environment (lib/buffer.py:22-34)."""
        if self.compact_obs:
            raise _lib.CarEnvError("a compact_obs Buffer is filled by fused_rollout (pose records), not by store()")
        p = self.ptr
        self.obs_buf[p] = obs
        self.act_buf[p] = act
        self.rew_buf[p] = rew
        self.val_buf[p] = val
        self.term_buf[p] = term
        self.trunc_buf[p] = trunc
        self.logprob_buf[p] = logprob
        self.ptr += 1

    def calculate_advantages(self, last_vals, last_terminateds, last_truncateds):
        """GAE over the full buffer; returns (adv_buf, ret_buf) (lib/buffer.py:36-64)."""
        assert self.ptr == self.capacity, "Buffer not full"
        if self._adv is None:
            self._adv, self._ret = torch.empty_like(self.rew_buf), torch.empty_like(self.rew_buf)
        with torch.no_grad():
            return gae_reverse_scan(self.rew_buf, self.val_buf, self.term_buf, self.trunc_buf, last_vals,
                                    last_terminateds, last_truncateds, self.gamma, self.gae_lambda,
                                    adv_out=self._adv, ret_out=self._ret, boot=self.boot_buf)

    def final_values(self, critic) -> None:
        """``boot_buf`` from the final-observation slots the last fused rollout wrote (:func:`final_values`; ``critic``
        is the policy's critic or a ``Population``)."""
        final_values(critic, self.final_obs_buf, self.final_row_buf, self.boot_buf)

    def get(self):
        """obs_buf (pose_buf if compact_obs), act_buf, val_buf, logprob_buf; rewinds the write pointer
        (lib/buffer.py:66-73)."""
        assert self.ptr == self.capacity
        self.ptr = 0
        return (self.pose_buf if self.compact_obs else self.obs_buf), self.act_buf, self.val_buf, self.logprob_buf
