"""Rollout buffer with the GAE reverse-scan kernel.

Same constructor, attributes and methods as the reference's ``lib.buffer.Buffer``
(/root/reference/lib/buffer.py:4-73): seven ``[size, num_envs(, obs_dim)]`` float32 tensors,
``store``, ``calculate_advantages`` (asserts the buffer is full, lib/buffer.py:46) and ``get``
(asserts and rewinds ``ptr``, lib/buffer.py:71-72).  ``calculate_advantages`` runs one
sm_100a kernel (``gae_reverse_scan``) that reproduces the reference's float32 operation order
bit for bit instead of ~12 tiny torch kernels per timestep.  CUDA only — no CPU fallback.
"""
from __future__ import annotations

import ctypes as C

import torch

from . import _lib


def _ptr(t):
    return C.c_void_p(t.data_ptr())


def gae_reverse_scan(rew, val, term, trunc, last_val, last_term, last_trunc, gamma=0.99, gae_lambda=0.95,
                     adv_out=None, ret_out=None):
    """adv, ret = GAE(lambda) over [T, N] float32 CUDA tensors (lib/buffer.py:51-63)."""
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
        rc = L.gae_reverse_scan(_ptr(rew), _ptr(val), _ptr(term), _ptr(trunc), _ptr(last_val), _ptr(last_term),
                                _ptr(last_trunc), _ptr(adv), _ptr(ret), T, N, float(gamma), float(gae_lambda), stream)
    _lib.check(rc, "gae_reverse_scan")
    return adv, ret


class Buffer:
    """Buffer for storing trajectories (drop-in for lib.buffer.Buffer)."""

    def __init__(self, obs_dim, size, num_envs, device, gamma=0.99, gae_lambda=0.95, compact_obs=False):
        """``compact_obs=True`` (no counterpart in the reference; SURVEY §8 f-3): no [size, num_envs, 18] observation
        tensor; ``pose_buf`` [size, num_envs, 4] float64 holds one 32-byte pose record per row instead, written by
        ``fused_rollout`` and turned back into observations by ``VecCarEnv.observe(pose_buf, index)``."""
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
                                    adv_out=self._adv, ret_out=self._ret)

    def get(self):
        """obs_buf (pose_buf if compact_obs), act_buf, val_buf, logprob_buf; rewinds the write pointer
        (lib/buffer.py:66-73)."""
        assert self.ptr == self.capacity
        self.ptr = 0
        return (self.pose_buf if self.compact_obs else self.obs_buf), self.act_buf, self.val_buf, self.logprob_buf
