"""Fused rollout kernel (SURVEY §8 f-2) against a plain PyTorch float32 evaluation of the same network and
against the non-fused environment kernel."""
import math
import os

import numpy as np
import pytest
import torch

import ppo_car_b200
from ppo_car_b200.train_ppo import ActorCritic, parse_args, train


def test_pack_layout_matches_header_constants():
    torch.manual_seed(0)
    net = ActorCritic(18, 9)
    if not os.path.exists(ppo_car_b200._lib.LIB_PATH):
        pytest.skip("library not built")
    packed = ppo_car_b200.pack_policy_weights(net.actor, net.critic)
    assert packed.numel() == 128 * 104 + 12
    blk = packed[:128 * 104].view(128, 104)
    j = 7
    assert blk[j, 0] == net.actor[0].weight[2 * j, 0] and blk[j, 1] == net.actor[0].weight[2 * j + 1, 0]
    assert blk[j, 36] == net.actor[0].bias[2 * j] and blk[j, 40] == net.actor[2].weight[0, 2 * j]
    assert blk[j, 41] == net.actor[2].weight[1, 2 * j] and blk[j, 42] == net.actor[2].weight[0, 2 * j + 1]
    assert blk[j, 60 + 36] == net.critic[0].bias[2 * j] and blk[j, 60 + 40] == net.critic[2].weight[0, 2 * j]
    assert packed[128 * 104 + 10] == net.critic[2].bias[0]


@pytest.mark.gpu
@pytest.mark.parametrize("n,tensor_cores", [(24, False), (1000, False), (24, 5), (1000, 5), (1300, 5), (2049, 5)])
def test_fused_rollout_matches_torch_policy_and_env_kernel(tracks_dir, n, tensor_cores):
    """tensor_cores: False = CUDA-core kernel (k_policy_rollout), 5 = tensor-core kernel (k_policy_rollout_tc3, option
    tc_tiles 5).  2049 envs leave one environment in the last 256-env CTA."""
    dev = torch.device("cuda")
    path = os.path.join(tracks_dir, "big_track.json")
    T = 300
    torch.manual_seed(3)
    net = ActorCritic(18, 9).to(dev)
    with torch.no_grad():                                   # make the policy non-uniform so sampling matters
        net.actor[2].weight.mul_(40.0)
        net.actor[2].bias.copy_(torch.linspace(-1, 1, 9))
    env = ppo_car_b200.VecCarEnv(n, path, reward_scaling=0.1, float_flags=True)
    buf = ppo_car_b200.Buffer((18,), T, n, dev)
    cur_obs = env.reset()[0].clone()
    cur_term, cur_trunc = torch.zeros(n, device=dev), torch.zeros(n, device=dev)
    last_val, u = torch.empty(n, device=dev), torch.empty((T, n), device=dev)
    pack = ppo_car_b200.pack_policy_weights_tc if tensor_cores else ppo_car_b200.pack_policy_weights
    packed = pack(net.actor, net.critic)
    if tensor_cores:
        env.set_option("tc_tiles", int(tensor_cores))
    ppo_car_b200.fused_rollout(env, packed, buf, cur_obs, cur_term, cur_trunc, seed=11, step0=5, last_val=last_val, u_dbg=u)
    torch.cuda.synchronize()
    assert buf.ptr == T

    # (1) network outputs: float32 torch evaluation of the same weights on the stored observations
    with torch.no_grad():
        logits = net.actor(buf.obs_buf.view(-1, 18)).view(T, n, 9)
        val = net.critic(buf.obs_buf.view(-1, 18)).view(T, n)
        logp_all = torch.log_softmax(logits, -1)
    act = buf.act_buf.long()
    assert torch.allclose(buf.val_buf, val, rtol=1e-5, atol=1e-5)
    assert torch.allclose(buf.logprob_buf, logp_all.gather(-1, act.unsqueeze(-1)).squeeze(-1), rtol=1e-5, atol=1e-5)
    with torch.no_grad():
        assert torch.allclose(last_val, net.critic(cur_obs).view(-1), rtol=1e-5, atol=1e-5)
    # (2) sampling: the action is the inverse CDF of the recorded uniform (ties within 1e-5 of a boundary excused)
    cdf = torch.softmax(logits, -1).cumsum(-1)
    expect = (u.unsqueeze(-1) >= cdf).sum(-1).clamp(max=8)
    near = ((cdf - u.unsqueeze(-1)).abs() < 1e-5).any(-1)
    assert ((expect == act) | near).all() and near.float().mean() < 1e-3
    assert 0.0 <= float(u.min()) and float(u.max()) < 1.0 and abs(float(u.mean()) - 0.5) < 0.01
    assert len(torch.unique(act)) == 9
    # (3) environment: replaying the sampled actions through the plain rollout kernel gives the same rows
    env2 = ppo_car_b200.VecCarEnv(n, path, reward_scaling=0.1, float_flags=True)
    obs0 = env2.reset()[0].clone()
    out = env2.rollout(act.to(torch.uint8))
    assert torch.equal(buf.obs_buf[0], obs0) and torch.equal(buf.obs_buf[1:], out["obs"][:-1])
    assert torch.equal(buf.rew_buf, out["reward"])
    assert torch.equal(buf.term_buf[1:], out["terminated"][:-1]) and torch.equal(buf.trunc_buf[1:], out["truncated"][:-1])
    assert torch.equal(cur_obs, out["obs"][-1]) and torch.equal(cur_term, out["terminated"][-1])
    assert torch.equal(env.pos, env2.pos) and torch.equal(env.ints, env2.ints)
    # (4) the random stream depends on (seed, global env id, global step) only: shard invariance
    half = n // 2
    env3 = ppo_car_b200.VecCarEnv(n - half, path, reward_scaling=0.1, float_flags=True)
    buf3 = ppo_car_b200.Buffer((18,), T, n - half, dev)
    o3 = env3.reset()[0].clone()
    if tensor_cores:
        env3.set_option("tc_tiles", int(tensor_cores))     # same kernel variant: same logit bits
    z = torch.zeros(n - half, device=dev)
    ppo_car_b200.fused_rollout(env3, packed, buf3, o3, z.clone(), z.clone(), seed=11, step0=5, env_offset=half)
    assert torch.equal(buf3.act_buf, buf.act_buf[:, half:]) and torch.equal(buf3.rew_buf, buf.rew_buf[:, half:])


@pytest.mark.gpu
@pytest.mark.parametrize("n,track_name", [(24, "big_track.json"), (257, "big_track.json"), (50, "track.json")])
def test_warp_per_environment_fused_rollout(tracks_dir, n, track_name):
    """k_policy_rollout_warp (small batches: lane = wall segment in the env step, lane = 16 hidden units in the
    policy) against torch float32, the inverse CDF of the recorded uniform, a replay through the plain rollout kernel
    and a sharded run."""
    dev = torch.device("cuda")
    path = os.path.join(tracks_dir, track_name)
    T = 300
    torch.manual_seed(3)
    net = ActorCritic(18, 9).to(dev)
    with torch.no_grad():
        net.actor[2].weight.mul_(40.0)
        net.actor[2].bias.copy_(torch.linspace(-1, 1, 9))
        net.critic[2].bias.fill_(0.3)
    env = ppo_car_b200.VecCarEnv(n, path, reward_scaling=0.1, float_flags=True)
    buf = ppo_car_b200.Buffer((18,), T, n, dev)
    cur_obs = env.reset()[0].clone()
    cur_term, cur_trunc = torch.zeros(n, device=dev), torch.zeros(n, device=dev)
    last_val, u = torch.empty(n, device=dev), torch.empty((T, n), device=dev)
    ppo_car_b200.fused_rollout_warp(env, net.actor, net.critic, buf, cur_obs, cur_term, cur_trunc, seed=11, step0=5,
                                    last_val=last_val, u_dbg=u)
    torch.cuda.synchronize()
    assert buf.ptr == T
    with torch.no_grad():
        logits = net.actor(buf.obs_buf.view(-1, 18)).view(T, n, 9)
        val = net.critic(buf.obs_buf.view(-1, 18)).view(T, n)
        logp_all = torch.log_softmax(logits, -1)
        assert torch.allclose(last_val, net.critic(cur_obs).view(-1), rtol=1e-5, atol=1e-5)
    act = buf.act_buf.long()
    assert torch.allclose(buf.val_buf, val, rtol=1e-5, atol=1e-5)
    assert torch.allclose(buf.logprob_buf, logp_all.gather(-1, act.unsqueeze(-1)).squeeze(-1), rtol=1e-5, atol=1e-5)
    cdf = torch.softmax(logits, -1).cumsum(-1)
    expect = (u.unsqueeze(-1) >= cdf).sum(-1).clamp(max=8)
    near = ((cdf - u.unsqueeze(-1)).abs() < 1e-5).any(-1)
    assert ((expect == act) | near).all() and near.float().mean() < 1e-3
    assert len(torch.unique(act)) == 9
    env2 = ppo_car_b200.VecCarEnv(n, path, reward_scaling=0.1, float_flags=True)
    obs0 = env2.reset()[0].clone()
    out = env2.rollout(act.to(torch.uint8))
    assert torch.equal(buf.obs_buf[0], obs0) and torch.equal(buf.obs_buf[1:], out["obs"][:-1])
    assert torch.equal(buf.rew_buf, out["reward"])
    assert torch.equal(buf.term_buf[1:], out["terminated"][:-1]) and torch.equal(buf.trunc_buf[1:], out["truncated"][:-1])
    assert torch.equal(cur_obs, out["obs"][-1]) and torch.equal(env.pos, env2.pos) and torch.equal(env.ints, env2.ints)
    half = n // 2
    env3 = ppo_car_b200.VecCarEnv(n - half, path, reward_scaling=0.1, float_flags=True)
    buf3 = ppo_car_b200.Buffer((18,), T, n - half, dev)
    o3 = env3.reset()[0].clone()
    z = torch.zeros(n - half, device=dev)
    ppo_car_b200.fused_rollout_warp(env3, net.actor, net.critic, buf3, o3, z.clone(), z.clone(), seed=11, step0=5,
                                    env_offset=half)
    assert torch.equal(buf3.act_buf, buf.act_buf[:, half:]) and torch.equal(buf3.logprob_buf, buf.logprob_buf[:, half:])
    # the same random stream as the tensor-core kernels: identical uniforms
    env4 = ppo_car_b200.VecCarEnv(n, path, reward_scaling=0.1, float_flags=True)
    buf4 = ppo_car_b200.Buffer((18,), T, n, dev)
    o4, u4 = env4.reset()[0].clone(), torch.empty((T, n), device=dev)
    ppo_car_b200.fused_rollout(env4, ppo_car_b200.pack_policy_weights_tc(net.actor, net.critic), buf4, o4,
                               torch.zeros(n, device=dev), torch.zeros(n, device=dev), seed=11, step0=5, u_dbg=u4)
    assert torch.equal(u, u4)


@pytest.mark.gpu
def test_tensor_core_rollout_reproduces_pinned_bits(golden_dir):
    """k_policy_rollout_tc3 against tests/golden/fused_tc3.npz (one full 256-env CTA and a ragged one, 64 steps,
    bootstrap values): actions, log-probabilities, values, rewards, last values and final observations bit for bit.
    Option tc_tiles 0 and 5 select this kernel; 2, 3 and 4 named kernels that have been removed and are refused."""
    from tests.golden.make_golden import fused_tc3_rollout

    ref = np.load(os.path.join(golden_dir, "fused_tc3.npz"))
    for tiles in (0, 5):
        got = fused_tc3_rollout(tiles)
        for k, v in got.items():
            assert v.dtype == ref[k].dtype and np.array_equal(v, ref[k]), (tiles, k)
    for tiles in (2, 3, 4):
        with pytest.raises(ppo_car_b200.CarEnvError, match="removed"):
            fused_tc3_rollout(tiles)


@pytest.mark.gpu
@pytest.mark.parametrize("extra", [[], ["--fused-cuda-cores"]])
def test_training_with_fused_rollout_improves_reward(extra):
    args = parse_args(["--track", "big_track", "--n-envs", "64", "--n-epochs", "12", "--n-steps", "256",
                       "--fused-rollout"] + extra)
    hist = train(args)
    assert all(math.isfinite(h["total_loss"]) for h in hist)
    assert hist[-1]["avg_reward"] > hist[0]["avg_reward"] + 0.03


@pytest.mark.gpu
def test_tcgen05_gemm_building_block():
    """csrc/tc_mlp.cuh bring-up: D[128,256] = A[128,24] B[256,24]^T through tcgen05.mma kind::tf32 with the
    accumulator in tensor memory and tcgen05.ld read-back, against float64 on TF32-exact inputs."""
    import ctypes as C

    from ppo_car_b200 import _lib
    from ppo_car_b200.policy import _tf32

    L = _lib.lib()
    torch.manual_seed(0)
    A = _tf32(torch.randn(128, 24, device="cuda"))
    B = _tf32(torch.randn(256, 24, device="cuda"))
    D = torch.full((128, 256), float("nan"), device="cuda")
    p = lambda t: C.c_void_p(t.data_ptr())
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    _lib.check(L.carenv_tc_gemm_test(p(A), p(B), p(D), st), "carenv_tc_gemm_test")
    torch.cuda.synchronize()
    ref = A.double() @ B.double().T
    assert (D.double() - ref).abs().max().item() < 2e-5       # float32 accumulation of 24 exact products
    # structured probe: catches a wrong operand layout (row/column permutations) exactly
    A2, B2 = torch.zeros(128, 24, device="cuda"), torch.zeros(256, 24, device="cuda")
    A2[:, 0] = torch.arange(128, device="cuda").float()
    B2[:, 0] = 1.0
    A2[:, 21] = 1.0
    B2[:, 21] = torch.arange(256, device="cuda").float() * 1024
    _lib.check(L.carenv_tc_gemm_test(p(A2), p(B2), p(D), st), "carenv_tc_gemm_test")
    torch.cuda.synchronize()
    assert torch.equal(D, A2 @ B2.T)


@pytest.mark.gpu
@pytest.mark.parametrize("tensor_cores", [False, True])
def test_fused_rollout_pose_rows_reproduce_the_observation_rows(tracks_dir, tensor_cores):
    """Buffer(compact_obs=True): the fused kernels write 32-byte pose records instead of observations; observe()
    gives back exactly the observation rows of an ordinary run with the same seed (SURVEY §8 f-3)."""
    dev = torch.device("cuda")
    path = os.path.join(tracks_dir, "big_track.json")
    n, T = 777, 260
    torch.manual_seed(5)
    net = ActorCritic(18, 9).to(dev)
    pack = ppo_car_b200.pack_policy_weights_tc if tensor_cores else ppo_car_b200.pack_policy_weights
    packed = pack(net.actor, net.critic)
    bufs, envs = [], []
    for compact in (False, True):
        env = ppo_car_b200.VecCarEnv(n, path, reward_scaling=0.1, float_flags=True)
        buf = ppo_car_b200.Buffer((18,), T, n, dev, compact_obs=compact)
        cur_obs = env.reset()[0].clone()
        cur_term, cur_trunc = torch.zeros(n, device=dev), torch.zeros(n, device=dev)
        for part in range(2):                               # the second launch starts from a mid-episode state
            ppo_car_b200.fused_rollout(env, packed, buf, cur_obs, cur_term, cur_trunc, seed=3, step0=part * T)
            if part == 0:
                first = (buf.pose_buf if compact else buf.obs_buf).clone()
        bufs.append((first, buf))
        envs.append(env)
    (obs_first, full), (pose_first, comp) = bufs
    assert comp.obs_buf is None and comp.pose_buf.shape == (T, n, 4)
    assert (full.term_buf.sum() + full.trunc_buf.sum()) > n // 4           # episode ends are covered
    assert torch.equal(envs[1].observe(pose_first).view(T, n, 18), obs_first)
    assert torch.equal(envs[1].observe(comp.pose_buf).view(T, n, 18), full.obs_buf)
    for a, b in ((full.act_buf, comp.act_buf), (full.rew_buf, comp.rew_buf), (full.logprob_buf, comp.logprob_buf),
                 (full.val_buf, comp.val_buf), (full.term_buf, comp.term_buf)):
        assert torch.equal(a, b)
    with pytest.raises(ppo_car_b200.CarEnvError):
        comp.ptr = 0
        comp.store(None, None, None, None, None, None, None)


@pytest.mark.gpu
def test_training_with_pose_rows_and_graph_update():
    args = parse_args(["--track", "big_track", "--n-envs", "64", "--n-epochs", "12", "--n-steps", "256",
                       "--fused-rollout", "--compact-obs", "--graph-update"])
    hist = train(args)
    assert all(math.isfinite(h["total_loss"]) for h in hist)
    assert hist[-1]["avg_reward"] > hist[0]["avg_reward"] + 0.03


@pytest.mark.gpu
@pytest.mark.parametrize("tensor_cores", [False, True])
def test_device_packing_kernel_equals_the_torch_layout_code(tensor_cores):
    """carenv_pack_policy (one launch) against the PyTorch statement of the same layout evaluated on the CPU."""
    torch.manual_seed(13)
    net = ActorCritic(18, 9)
    with torch.no_grad():
        for p in net.parameters():
            p.add_(torch.randn_like(p) * 0.3)                # biases are zero after the reference's init
    pack = ppo_car_b200.pack_policy_weights_tc if tensor_cores else ppo_car_b200.pack_policy_weights
    ref = pack(net.actor, net.critic)                        # CPU tensors: the torch code path
    net_gpu = ActorCritic(18, 9).cuda()
    net_gpu.load_state_dict(net.state_dict())
    got = pack(net_gpu.actor, net_gpu.critic)
    assert got.is_cuda and torch.equal(got.cpu(), ref)
    out = torch.empty_like(got)
    assert pack(net_gpu.actor, net_gpu.critic, out=out) is out and torch.equal(out, got)
