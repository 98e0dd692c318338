"""Fused rollout: policy forward + sampling + CarEnv.step + Buffer rows in one kernel launch.

Host side of ``carenv_policy_rollout`` (include/carenv_b200.h).  The network is the reference's
(lib/model.py:10-26): actor 18-256-9 and critic 18-256-1, two ``nn.Sequential(Linear, ReLU, Linear)``.
"""
from __future__ import annotations

import ctypes as C

import torch

from . import _lib

HIDDEN, OBS, ACTIONS = 256, 18, 9


def _pack_on_device(tensor_cores: bool, actor, critic, out):
    """One launch of k_pack_policy (C ABI carenv_pack_policy) for parameters that live on a CUDA device."""
    L = _lib.lib()
    params = [actor[0].weight, actor[0].bias, actor[2].weight, actor[2].bias,
              critic[0].weight, critic[0].bias, critic[2].weight, critic[2].bias]
    params = [p.detach().float().contiguous() for p in params]
    n = L.carenv_policy_weights_floats_tc() if tensor_cores else L.carenv_policy_weights_floats()
    dev = params[0].device
    if out is None:
        out = torch.empty(n, dtype=torch.float32, device=dev)
    elif out.numel() != n or out.dtype != torch.float32 or out.device != dev or not out.is_contiguous():
        raise ValueError(f"out must be a contiguous float32 tensor of {n} elements on {dev}")
    with torch.cuda.device(dev):
        rc = L.carenv_pack_policy(int(tensor_cores), *[C.c_void_p(p.data_ptr()) for p in params],
                                  C.c_void_p(out.data_ptr()), C.c_void_p(torch.cuda.current_stream(dev).cuda_stream))
    _lib.check(rc, "carenv_pack_policy")
    return out


def pack_policy_weights(actor, critic, out: torch.Tensor | None = None) -> torch.Tensor:
    """Lay the four Linear layers out the way policy_core.cuh reads them: per pair of hidden units
    (j, j+1) an actor block [18 x (W1[j,k], W1[j+1,k]) | b1 pair, pad | 5 x (W2[2q,j], W2[2q+1,j],
    W2[2q,j+1], W2[2q+1,j+1])] of 60 floats and a critic block [18 pairs | b1 pair, pad | (W2c[j],
    W2c[j+1]), pad] of 44 floats, then b2[0..9] (b2[9] = 0), b2c, pad.  Cheap enough to redo after
    every optimiser step (12,298 parameters)."""
    w1a, b1a, w2a, b2a = actor[0].weight, actor[0].bias, actor[2].weight, actor[2].bias
    w1c, b1c, w2c, b2c = critic[0].weight, critic[0].bias, critic[2].weight, critic[2].bias
    if tuple(w1a.shape) != (HIDDEN, OBS) or tuple(w2a.shape) != (ACTIONS, HIDDEN) or tuple(w2c.shape) != (1, HIDDEN):
        raise ValueError("fused rollout supports the reference network only: 18-256-9 actor, 18-256-1 critic")
    if w1a.is_cuda:                                         # one kernel launch; the code below documents the layout
        return _pack_on_device(False, actor, critic, out)
    dev, P = w1a.device, HIDDEN // 2
    with torch.no_grad():
        z2 = torch.zeros((P, 2), device=dev)
        w2pad = torch.cat([w2a, torch.zeros((1, HIDDEN), device=dev)])                 # [10, 256]
        blk_a = torch.cat([w1a.view(P, 2, OBS).permute(0, 2, 1).reshape(P, 36), b1a.view(P, 2), z2,
                           w2pad.view(5, 2, P, 2).permute(2, 0, 3, 1).reshape(P, 20)], dim=1)          # [128, 60]
        blk_c = torch.cat([w1c.view(P, 2, OBS).permute(0, 2, 1).reshape(P, 36), b1c.view(P, 2), z2,
                           w2c.view(P, 2), z2], dim=1)                                                  # [128, 44]
        tail = torch.cat([b2a, torch.zeros(1, device=dev), b2c, torch.zeros(1, device=dev)])            # 12
        packed = torch.cat([torch.cat([blk_a, blk_c], dim=1).reshape(-1), tail]).float().contiguous()
    if packed.numel() != _lib.lib().carenv_policy_weights_floats():
        raise _lib.CarEnvError("packed policy size does not match the library")
    if out is not None:
        out.copy_(packed)
        return out
    return packed


def _tf32(x: torch.Tensor) -> torch.Tensor:
    """Round float32 to TF32 (10 explicit mantissa bits), to nearest with ties away from zero (cvt.rna)."""
    i = x.contiguous().view(torch.int32)
    return ((i + 0x1000) & ~0x1FFF).view(torch.float32)


def pack_policy_weights_tc(actor, critic, out: torch.Tensor | None = None) -> torch.Tensor:
    """Weights for the tensor-core kernel: per net the first layer [256 x 24] (18 inputs, the bias in column
    18, zero padding) as TF32 hi and lo parts in the K-major no-swizzle UMMA shared-memory layout
    (csrc/tc_mlp.cuh: float index (j/8)*192 + (k/4)*32 + (j%8)*4 + k%4), then the actor's second layer as
    [j][5] pairs (W2[2q][j], W2[2q+1][j]), the critic's second layer w2c[j], b2[0..9] (b2[9] = 0), b2c."""
    w1a, b1a, w2a, b2a = actor[0].weight, actor[0].bias, actor[2].weight, actor[2].bias
    w1c, b1c, w2c, b2c = critic[0].weight, critic[0].bias, critic[2].weight, critic[2].bias
    if tuple(w1a.shape) != (HIDDEN, OBS) or tuple(w2a.shape) != (ACTIONS, HIDDEN) or tuple(w2c.shape) != (1, HIDDEN):
        raise ValueError("fused rollout supports the reference network only: 18-256-9 actor, 18-256-1 critic")
    if w1a.is_cuda:                                         # one kernel launch; the code below documents the layout
        return _pack_on_device(True, actor, critic, out)
    dev = w1a.device
    with torch.no_grad():
        j = torch.arange(HIDDEN, device=dev).view(-1, 1)
        k = torch.arange(24, device=dev).view(1, -1)
        index = ((j // 8) * 192 + (k // 4) * 32 + (j % 8) * 4 + (k % 4)).reshape(-1)

        def operand(w1, b1):
            ext = torch.zeros((HIDDEN, 24), device=dev)
            ext[:, :OBS] = w1
            ext[:, OBS] = b1
            hi = _tf32(ext)
            lo = _tf32(ext - hi)
            o_hi, o_lo = torch.empty(HIDDEN * 24, device=dev), torch.empty(HIDDEN * 24, device=dev)
            o_hi[index] = hi.reshape(-1)
            o_lo[index] = lo.reshape(-1)
            return o_hi, o_lo

        w2pad = torch.cat([w2a, torch.zeros((1, HIDDEN), device=dev)])                 # [10, 256]
        packed = torch.cat([*operand(w1a, b1a), *operand(w1c, b1c), w2pad.t().reshape(-1), w2c.reshape(-1), b2a,
                            torch.zeros(1, device=dev), b2c, torch.zeros(1, device=dev)]).float().contiguous()
    if packed.numel() != _lib.lib().carenv_policy_weights_floats_tc():
        raise _lib.CarEnvError("packed policy size does not match the library")
    if out is not None:
        out.copy_(packed)
        return out
    return packed


def _p(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def fused_rollout(env, packed: torch.Tensor, buf, cur_obs: torch.Tensor, cur_term: torch.Tensor,
                  cur_trunc: torch.Tensor, seed: int, step0: int, env_offset: int = 0,
                  last_val: torch.Tensor | None = None, u_dbg: torch.Tensor | None = None,
                  tensor_cores: bool | None = None) -> None:
    """Fill every row of ``buf`` (ppo_car_b200.Buffer) with one launch and leave the rollout state in
    ``cur_obs / cur_term / cur_trunc`` (in place).  ``step0`` is the global step index of row 0 (it
    selects the random stream together with ``seed`` and ``env_offset + env``).

    ``env`` may be a :class:`MultiTrackVecEnv` (C ABI carenv_policy_rollout_tc_multi): every environment runs on its
    track (``env.track_ids``) and its rows are bit-identical to a single-track run on that track.  That needs the
    tensor-core packing and full observation rows (no ``Buffer(compact_obs=True)``)."""
    from .vec_env import MultiTrackVecEnv

    multi = isinstance(env, MultiTrackVecEnv)
    n, T = env.num_envs, buf.capacity
    for name, t, shape in (("cur_obs", cur_obs, (n, OBS)), ("cur_term", cur_term, (n,)), ("cur_trunc", cur_trunc, (n,)),
                           ("last_val", last_val, (n,)), ("u_dbg", u_dbg, (T, n))):
        if t is not None and (tuple(t.shape) != shape or t.dtype != torch.float32 or not t.is_contiguous()
                              or t.device != env.device):
            raise ValueError(f"{name} must be a contiguous float32 tensor of shape {shape} on {env.device}")
    compact = bool(getattr(buf, "compact_obs", False))
    rows = buf.pose_buf if compact else buf.obs_buf
    if tuple(rows.shape) != ((T, n, 4) if compact else (T, n, OBS)):
        raise ValueError("buffer shape does not match the environment")
    L = _lib.lib()
    if tensor_cores is None:                                # the two packings have different sizes
        tensor_cores = packed.numel() == L.carenv_policy_weights_floats_tc()
    if multi:
        if compact:
            raise ValueError("several tracks need full observation rows: pose records do not carry a track "
                             "(use Buffer(compact_obs=False))")
        if not tensor_cores:
            raise ValueError("several tracks run on the tensor-core kernel only: pack the weights with "
                             "pack_policy_weights_tc")
        with torch.cuda.device(env.device):
            rc = L.carenv_policy_rollout_tc_multi(
                env._multi, _p(env.track_ids), _p(packed), n, T, int(env_offset), int(seed) & (2 ** 64 - 1),
                int(step0), _p(env.pos), _p(env.vel), _p(env.ints), _p(cur_obs), _p(cur_term), _p(cur_trunc),
                float(env.reward_scaling), _p(rows), _p(buf.act_buf), _p(buf.rew_buf), _p(buf.val_buf),
                _p(buf.term_buf), _p(buf.trunc_buf), _p(buf.logprob_buf), _p(last_val), _p(u_dbg), env._stream())
        _lib.check(rc, "carenv_policy_rollout_tc_multi")
        buf.ptr = T
        return
    env.set_option("pose_rows", int(compact))               # obs_buf argument = 32-byte pose records
    fn = L.carenv_policy_rollout_tc if tensor_cores else L.carenv_policy_rollout
    with torch.cuda.device(env.device):
        rc = fn(env._handle, _p(packed), n, T, int(env_offset), int(seed) & (2 ** 64 - 1), int(step0), _p(env.pos),
                _p(env.vel), _p(env.ints), _p(cur_obs), _p(cur_term), _p(cur_trunc), float(env.reward_scaling),
                _p(rows), _p(buf.act_buf), _p(buf.rew_buf), _p(buf.val_buf), _p(buf.term_buf),
                _p(buf.trunc_buf), _p(buf.logprob_buf), _p(last_val), _p(u_dbg), env._stream())
    _lib.check(rc, "carenv_policy_rollout_tc" if tensor_cores else "carenv_policy_rollout")
    buf.ptr = T


WARP_ROLLOUT_MAX_ENVS = 4096        # crossover against the tensor-core kernel (benchmarks/fused_small.py)


def fused_rollout_warp(env, actor, critic, buf, cur_obs: torch.Tensor, cur_term: torch.Tensor, cur_trunc: torch.Tensor,
                       seed: int, step0: int, env_offset: int = 0, last_val: torch.Tensor | None = None,
                       u_dbg: torch.Tensor | None = None) -> None:
    """:func:`fused_rollout` for small batches (C ABI carenv_policy_rollout_warp): one warp per environment, the
    network's parameters read in place (no packing).  Tracks with at most 32 wall segments."""
    n, T = env.num_envs, buf.capacity
    params = [actor[0].weight, actor[0].bias, actor[2].weight, actor[2].bias,
              critic[0].weight, critic[0].bias, critic[2].weight, critic[2].bias]
    if [tuple(p.shape) for p in params] != [(HIDDEN, OBS), (HIDDEN,), (ACTIONS, HIDDEN), (ACTIONS,), (HIDDEN, OBS),
                                            (HIDDEN,), (1, HIDDEN), (1,)]:
        raise ValueError("fused rollout supports the reference network only: 18-256-9 actor, 18-256-1 critic")
    if any(p.dtype != torch.float32 or not p.is_contiguous() or p.device != env.device for p in params):
        raise ValueError(f"parameters must be contiguous float32 tensors on {env.device}")
    for name, t, shape in (("cur_obs", cur_obs, (n, OBS)), ("cur_term", cur_term, (n,)), ("cur_trunc", cur_trunc, (n,)),
                           ("last_val", last_val, (n,)), ("u_dbg", u_dbg, (T, n))):
        if t is not None and (tuple(t.shape) != shape or t.dtype != torch.float32 or not t.is_contiguous()
                              or t.device != env.device):
            raise ValueError(f"{name} must be a contiguous float32 tensor of shape {shape} on {env.device}")
    compact = bool(getattr(buf, "compact_obs", False))
    rows = buf.pose_buf if compact else buf.obs_buf
    if tuple(rows.shape) != ((T, n, 4) if compact else (T, n, OBS)):
        raise ValueError("buffer shape does not match the environment")
    env.set_option("pose_rows", int(compact))
    L = _lib.lib()
    with torch.cuda.device(env.device):
        rc = L.carenv_policy_rollout_warp(env._handle, *[_p(p) for p in params], n, T, int(env_offset),
                                          int(seed) & (2 ** 64 - 1), int(step0), _p(env.pos), _p(env.vel), _p(env.ints),
                                          _p(cur_obs), _p(cur_term), _p(cur_trunc), float(env.reward_scaling), _p(rows),
                                          _p(buf.act_buf), _p(buf.rew_buf), _p(buf.val_buf), _p(buf.term_buf),
                                          _p(buf.trunc_buf), _p(buf.logprob_buf), _p(last_val), _p(u_dbg), env._stream())
    _lib.check(rc, "carenv_policy_rollout_warp")
    buf.ptr = T
