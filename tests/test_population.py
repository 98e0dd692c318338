"""Populations of independent policies (ppo_car_b200.population, csrc/population.cuh).

GPU:
  * the member-batched rollouts (k_policy_rollout_warp<true>, k_policy_rollout_tc3<U, TAB, true>) against
    single-member fused_rollout_warp / fused_rollout runs, bit for bit, including u_dbg, last_val, the final state and
    two launches against one; the batched packing against the single packing;
  * the cluster-per-member epoch update (k_ppo_epoch_pop) against the float64 reference of tests/ppo_reference.py
    with hyperparameters that differ per member, a 60-update free run, and its independence and determinism;
  * end to end: rewards rise, epoch 1 equals train_ppo's, checkpoints load into evaluate.
CPU: seed and grid parsing, member sharding, refusals, C ABI error codes.
"""
import ctypes as C
import os
import subprocess
import sys
from types import SimpleNamespace

import numpy as np
import pytest
import torch

import ppo_car_b200
from ppo_car_b200 import _lib
from ppo_car_b200 import population as popmod
from ppo_car_b200.population import Population, PopulationPPOUpdate, population_rollout
from ppo_car_b200.shard import shard_range
from tests.ppo_reference import (N_PARAMS, as_float32_values, clip_adam_f64, dyadic_problem, flatten, hparams,
                                 loss_and_grads_f64, new_logp_f64, old_logp_with_margin, unflatten)

gpu = pytest.mark.gpu
SEEDS = [3, 2 ** 32 + 5, 11, 2 ** 40 + 7, 0, 19, 2 ** 33 + 1]          # distinct, some with a non-zero high word


# ---- CPU ---------------------------------------------------------------------------------------------------------
def test_parse_seeds():
    assert popmod.parse_seeds("0-3") == [0, 1, 2, 3]
    assert popmod.parse_seeds("0,5,9") == [0, 5, 9]
    assert popmod.parse_seeds("0-2,7") == [0, 1, 2, 7]
    assert popmod.parse_seeds("4") == [4]
    assert popmod.parse_seeds("18446744073709551") == [popmod.MAX_SEED]       # the largest s with s * 1000 + 1 < 2^64
    for bad in ("", "3-1", "1,1", "a", "0,,1", "-1", "18446744073709552"):
        with pytest.raises(ValueError):
            popmod.parse_seeds(bad)


def test_grid_is_the_cross_product_of_lists_and_seeds():
    settings, members = popmod.expand_grid([0, 1, 2], {"learning_rate": [3e-4, 1e-3], "clip_ratio": [0.1, 0.2]})
    assert len(settings) == 4 and len(members) == 12
    assert settings[0] == dict(popmod.DEFAULTS, learning_rate=3e-4, clip_ratio=0.1)
    assert settings[1] == dict(popmod.DEFAULTS, learning_rate=3e-4, clip_ratio=0.2)
    for m, (seed, h) in enumerate(members):
        assert seed == [0, 1, 2][m % 3] and h == settings[m // 3]
    args = popmod.parse_args(["--seeds", "0-1", "--learning-rate", "1e-3,3e-4", "--ent-coef=0.01,0", "--n-envs", "4"])
    settings, members = popmod.check_args(args)
    assert args.learning_rate == 1e-3 and args.ent_coef == 0.01 and args.n_envs == 4
    assert [h["learning_rate"] for h in settings] == [1e-3, 1e-3, 3e-4, 3e-4]
    assert [h["ent_coef"] for h in settings] == [0.01, 0.0, 0.01, 0.0] and len(members) == 8


def test_members_are_sharded_over_ranks():
    for P in (1, 5, 32, 33):
        for world in (1, 2, 3, 8):
            parts = [shard_range(P, world, r) for r in range(world)]
            assert parts[0][0] == 0 and parts[-1][1] == P
            assert all(a[1] == b[0] for a, b in zip(parts, parts[1:]))
            assert max(h - l for l, h in parts) - min(h - l for l, h in parts) <= 1


@pytest.mark.parametrize("argv, words", [
    (["--track", "big_track,track"], "one track"),
    (["--compact-obs"], "--compact-obs"),
    (["--cuda-graph"], "--cuda-graph"),
    (["--graph-update"], "--graph-update"),
    (["--per-minibatch-update"], "--per-minibatch-update"),
    (["--fused-cuda-cores"], "--fused-cuda-cores"),
    (["--n-envs", "0"], "--n-envs"),
    (["--seeds", "3-1"], "seed range"),
    (["--learning-rate", ","], "empty"),
    (["--batch-size", "2000"], "--batch-size"),
    (["--seeds", "18446744073709552"], "0 .. 18446744073709551"),     # s * 1000 + 1 overflows 64 bits
])
def test_refusals_come_before_any_device_work(argv, words, monkeypatch):
    monkeypatch.setattr(torch.cuda, "set_device", lambda *a: pytest.fail("device work before the refusal"))
    with pytest.raises(SystemExit, match=words):
        popmod.train_population(popmod.parse_args(argv))


def test_population_refuses_bad_arguments():
    with pytest.raises(ValueError):
        Population([], 4)
    with pytest.raises(ValueError):
        Population([0], 0)
    with pytest.raises(ValueError):
        Population([0, 1], 4, [{}])
    with pytest.raises(ValueError):
        Population([0], 4, {"gamma": 0.9})
    with pytest.raises(ValueError, match="18446744073709551"):
        Population([popmod.MAX_SEED + 1], 4)
    with pytest.raises(ValueError):
        PopulationPPOUpdate(SimpleNamespace(), 1)


def test_population_abi_error_codes():
    L = _lib.lib()
    assert L.carenv_ppo_epoch_pop_cluster_size() in (2, 4, 8, 16)
    assert L.carenv_ppo_epoch_pop_resident_clusters(None) == -1
    nul = [None] * 8
    assert L.carenv_pack_policy_pop(1, 0, *nul, None, None) == -1
    assert L.carenv_pack_policy_pop(1, 2, *nul, None, None) == -1 and b"null" in L.carenv_last_error()
    roll = lambda P, n, T: L.carenv_policy_rollout_warp_pop(None, P, *nul, n, T, None, 0, *([None] * 6), 1.0,
                                                            *([None] * 10))
    assert roll(2, 4, 4) == -1 and b"handle" in L.carenv_last_error()
    roll_tc = lambda P, n, T: L.carenv_policy_rollout_tc_pop(None, P, None, n, T, None, 0, *([None] * 6), 1.0,
                                                             *([None] * 10))
    assert roll_tc(2, 4, 4) == -1
    epoch = lambda P, B, U, p=None: L.carenv_ppo_epoch_pop(P, *([p] * 8), *([p] * 6), B, U, *([p] * 5), 0.9, 0.999,
                                                           1e-5, *([p] * 5))
    assert epoch(0, 512, 4) == -1 and b"n_members" in L.carenv_last_error()
    assert epoch(-3, 512, 4) == -1
    assert epoch(2, 1, 4) == -1 and b"batch" in L.carenv_last_error()
    assert epoch(2, 1025, 4) == -1 and b"batch" in L.carenv_last_error()
    assert epoch(2, 512, -1) == -1 and b"n_updates" in L.carenv_last_error()
    assert epoch(2, 512, 4) == -1 and b"null" in L.carenv_last_error()


# ---- GPU: rollouts ---------------------------------------------------------------------------------------------------
def _state(env):
    return [t.clone() for t in (env.pos, env.vel, env.ints)]


def _member_net(pop, p, dev):
    from ppo_car_b200.train_ppo import ActorCritic

    net = ActorCritic(18, 9).to(dev)
    net.load_state_dict(pop.member_state_dict(p))
    return net


def _single(pop, p, track, T, step0_list, last_val, tensor_cores, dev):
    """Member p alone: fused_rollout_warp / fused_rollout with its seed, env_offset 0, one launch per entry of
    step0_list (T steps each).  Returns the buffers' rows concatenated over the launches and the final state."""
    n = pop.n_envs
    net = _member_net(pop, p, dev)
    env = ppo_car_b200.VecCarEnv(n, track, device=dev, reward_scaling=0.1, float_flags=True, with_info=False)
    cur = env.reset()[0].clone()
    z1, z2 = torch.zeros(n, device=dev), torch.zeros(n, device=dev)
    lv = torch.empty(n, device=dev) if last_val else None
    rows = []
    for step0 in step0_list:
        buf = ppo_car_b200.Buffer((18,), T, n, dev)
        u = torch.empty((T, n), device=dev)
        if tensor_cores:
            ppo_car_b200.fused_rollout(env, ppo_car_b200.pack_policy_weights_tc(net.actor, net.critic), buf, cur, z1, z2,
                                       seed=pop.seeds[p], step0=step0, last_val=lv, u_dbg=u)
        else:
            ppo_car_b200.fused_rollout_warp(env, net.actor, net.critic, buf, cur, z1, z2, seed=pop.seeds[p], step0=step0,
                                            last_val=lv, u_dbg=u)
        rows.append([buf.obs_buf.clone(), buf.act_buf.clone(), buf.rew_buf.clone(), buf.val_buf.clone(),
                     buf.term_buf.clone(), buf.trunc_buf.clone(), buf.logprob_buf.clone(), u])
    rows = [torch.cat(c) for c in zip(*rows)]
    return rows, [cur, z1, z2] + _state(env), lv


def _population(pop, track, T, step0_list, last_val, dev):
    N = pop.num_envs
    env = ppo_car_b200.VecCarEnv(N, track, device=dev, reward_scaling=0.1, float_flags=True, with_info=False)
    cur = env.reset()[0].clone()
    z1, z2 = torch.zeros(N, device=dev), torch.zeros(N, device=dev)
    lv = torch.empty(N, device=dev) if last_val else None
    rows = []
    for step0 in step0_list:
        buf = ppo_car_b200.Buffer((18,), T, N, dev)
        u = torch.empty((T, N), device=dev)
        population_rollout(env, pop, buf, cur, z1, z2, step0=step0, last_val=lv, u_dbg=u)
        rows.append([buf.obs_buf.clone(), buf.act_buf.clone(), buf.rew_buf.clone(), buf.val_buf.clone(),
                     buf.term_buf.clone(), buf.trunc_buf.clone(), buf.logprob_buf.clone(), u])
    rows = [torch.cat(c) for c in zip(*rows)]
    return rows, [cur, z1, z2] + _state(env), lv


ROLLOUT_CASES = [   # P, n, T, last_val, launches, track
    (1, 24, 64, True, 1, "big_track"),
    (3, 1, 7, False, 1, "big_track"),
    (3, 3, 1, True, 1, "big_track"),
    (7, 24, 7, True, 1, "big_track"),
    (3, 257, 64, False, 1, "big_track"),
    (7, 3, 64, True, 2, "big_track"),
    (3, 24, 7, True, 2, "track"),
    (2, 4097, 7, True, 1, "big_track"),          # more than WARP_ROLLOUT_MAX_ENVS: the tensor-core kernel
    (3, 4097, 1, False, 2, "big_track"),
]


@gpu
@pytest.mark.parametrize("P, n, T, last_val, launches, track", ROLLOUT_CASES)
def test_population_rollout_equals_single_members(P, n, T, last_val, launches, track):
    dev = torch.device("cuda", 0)
    path = ppo_car_b200.builtin_track(track)
    pop = Population(SEEDS[:P], n, None, dev)
    env_probe = ppo_car_b200.VecCarEnv(1, path, device=dev)
    tensor_cores = not popmod.use_warp_kernel(env_probe, n)
    assert tensor_cores == (n > 4096)
    step0_list = [T * k + 5 for k in range(launches)] if launches > 1 else [2 ** 32 + 3]
    rows, state, lv = _population(pop, path, T, step0_list, last_val, dev)
    names = ["obs", "act", "rew", "val", "term", "trunc", "logp", "u_dbg"]
    for p in range(P):
        c = slice(p * n, (p + 1) * n)
        rows1, state1, lv1 = _single(pop, p, path, T, step0_list, last_val, tensor_cores, dev)
        for name, a, b in zip(names, rows, rows1):
            assert torch.equal(a[:, c], b), (p, name)
        for k, (a, b) in enumerate(zip(state, state1)):
            assert torch.equal(a[c], b), (p, "state", k)
        if last_val:
            assert torch.equal(lv[c], lv1), (p, "last_val")
    if launches > 1:                                  # two launches against one of 2T steps
        pop_one, _, _ = _population(pop, path, T * launches, [step0_list[0]], last_val, dev)
        for a, b in zip(rows, pop_one):
            assert torch.equal(a, b)


@gpu
def test_population_rollout_refuses_bad_shapes_and_pose_rows():
    dev = torch.device("cuda", 0)
    pop = Population([0, 1], 4, None, dev)
    env = ppo_car_b200.VecCarEnv(8, ppo_car_b200.builtin_track("big_track"), device=dev, float_flags=True)
    cur = env.reset()[0].clone()
    z1, z2 = torch.zeros(8, device=dev), torch.zeros(8, device=dev)
    buf = ppo_car_b200.Buffer((18,), 4, 8, dev)
    with pytest.raises(ValueError, match="environments"):
        population_rollout(ppo_car_b200.VecCarEnv(6, ppo_car_b200.builtin_track("big_track"), device=dev), pop, buf,
                           cur, z1, z2, step0=0)
    with pytest.raises(ValueError, match="full observation"):
        population_rollout(env, pop, ppo_car_b200.Buffer((18,), 4, 8, dev, compact_obs=True), cur, z1, z2, step0=0)
    L = _lib.lib()
    env.set_option("pose_rows", 1)
    p = lambda t: C.c_void_p(t.data_ptr())
    rc = L.carenv_policy_rollout_warp_pop(env._handle, 2, *[p(t) for t in pop.params], 4, 4, p(pop.seeds_dev), 0,
                                          p(env.pos), p(env.vel), p(env.ints), p(cur), p(z1), p(z2), 0.1,
                                          p(buf.obs_buf), p(buf.act_buf), p(buf.rew_buf), p(buf.val_buf),
                                          p(buf.term_buf), p(buf.trunc_buf), p(buf.logprob_buf), None, None,
                                          env._stream())
    assert rc == -1 and b"pose_rows" in L.carenv_last_error()


@gpu
@pytest.mark.parametrize("tensor_cores", [True, False])
def test_batched_packing_equals_single_packing(tensor_cores):
    dev = torch.device("cuda", 0)
    pop = Population(SEEDS[:5], 4, None, dev)
    packed = pop.pack(tensor_cores)
    torch.cuda.synchronize()
    pack1 = ppo_car_b200.pack_policy_weights_tc if tensor_cores else ppo_car_b200.pack_policy_weights
    for p in range(pop.P):
        net = _member_net(pop, p, dev)
        assert torch.equal(packed[p], pack1(net.actor, net.critic)), p


# ---- GPU: the population update against float64 -------------------------------------------------------------------
MEMBER_CASES = {   # name: B, dyadic options, inside fraction, hyperparameters
    "B2": dict(B=2, hp=dict(clip_ratio=0.2, vf_coef=0.5, ent_coef=0.001)),
    "B3": dict(B=3, hp=dict(clip_ratio=0.15, vf_coef=1.0, ent_coef=0.01)),
    "B512_mixed": dict(B=512, inside=0.5, hp=dict(clip_ratio=0.1, vf_coef=0.25, ent_coef=0.0)),
    "B512_inside": dict(B=512, inside=1.0, hp=dict(clip_ratio=0.3, vf_coef=0.5, ent_coef=0.005)),
    "B512_outside": dict(B=512, inside=0.0, hp=dict(clip_ratio=0.2, vf_coef=2.0, ent_coef=0.001)),
    "B512_const_adv": dict(B=512, adv_const=0.5, hp=dict(clip_ratio=0.2, vf_coef=0.5, ent_coef=0.02)),
    "B1024": dict(B=1024, hp=dict(clip_ratio=0.25, vf_coef=0.75, ent_coef=0.002)),
}


def _member_problem(name, seed):
    c = MEMBER_CASES[name]
    B = c["B"]
    rows = max(2 * B, 64)
    hp = as_float32_values(hparams(**c["hp"]))
    state, obs, act, adv, ret = dyadic_problem(rows, seed=seed, adv_const=c.get("adv_const"))
    old = old_logp_with_margin(new_logp_f64(state, obs, act), c.get("inside", 0.5), hp["clip_ratio"], seed=seed)
    idx = np.random.default_rng(50 + seed).choice(rows, B, replace=False)
    return SimpleNamespace(B=B, hp=hp, state=state, obs=obs, act=act, adv=adv, ret=ret, old=old, idx=idx, rows=rows)


def _stage(problems, B, dev, lr, max_grad_norm, eps=None):
    """A Population whose member p holds problems[p]'s network and hyperparameters; every member's samples are
    concatenated into one set of flat arrays (member p's at an offset, idx pointing at its own rows)."""
    P = len(problems)
    pop = Population(list(range(P)), 1, [{k: pb.hp[k] for k in ("clip_ratio", "vf_coef", "ent_coef")} for pb in problems],
                     dev)
    with torch.no_grad():
        for p, pb in enumerate(problems):
            for t, a in zip(pop.params, pb.state):
                t[p].copy_(torch.as_tensor(a).reshape(t[p].shape))
        pop.lr.copy_(torch.as_tensor(lr, dtype=torch.float32))
        pop.max_grad_norm.copy_(torch.as_tensor(max_grad_norm, dtype=torch.float32))
    cat = lambda key: torch.as_tensor(np.concatenate([getattr(pb, key) for pb in problems])).float().contiguous().to(dev)
    data = [cat(k) for k in ("obs", "act", "old", "adv", "ret")]
    offs = np.cumsum([0] + [pb.rows for pb in problems])[:-1]
    return pop, data, offs


def _flat(pop, p):
    return flatten([t[p] for t in pop.params])


@gpu
def test_population_update_gradients_match_float64_per_member():
    """Every member's gradient, read through one linear-Adam update (m = v = 0, t = 1, lr = 1e9, eps = 1e6: the step is
    -lr * g / (|g| + eps) = -1000 g to 1e-6 relative), against loss_and_grads_f64 with that member's hyperparameters;
    the bound of test_ppo_update_reference.py plus the probe's own rounding."""
    dev = torch.device("cuda", 0)
    for B in (2, 3, 512, 1024):
        names = [k for k, c in MEMBER_CASES.items() if c["B"] == B]
        problems = [_member_problem(nm, seed=10 + i) for i, nm in enumerate(names)]
        pop, data, offs = _stage(problems, B, dev, lr=[1e9] * len(problems), max_grad_norm=[1e30] * len(problems))
        upd = PopulationPPOUpdate(pop, B, eps=1e6)
        idx = torch.as_tensor(np.stack([pb.idx + o for pb, o in zip(problems, offs)])[:, None, :]).to(dev).contiguous()
        p0 = [_flat(pop, p) for p in range(pop.P)]
        upd.launch(data[0], idx, *data[1:])
        torch.cuda.synchronize()
        for p, (nm, pb) in enumerate(zip(names, problems)):
            ref = loss_and_grads_f64(pb.state, pb.obs[pb.idx], pb.act[pb.idx], pb.old[pb.idx], pb.adv[pb.idx],
                                     pb.ret[pb.idx], pb.hp)
            g64 = ref["grad"]
            g = -(_flat(pop, p) - p0[p]) / 1000.0
            tol = 2e-4 * np.abs(g64) + 2e-6 * np.abs(g64).max() + 2e-6 * np.abs(g64) + 1e-7 * (1 + np.abs(p0[p]))
            worst = float(np.max(np.abs(g - g64) / tol))
            print(f"\n[worst] population gradient {nm}: {worst:.3g} of the tolerance")
            assert worst <= 1.0, nm
            sums = pop.sums[p].cpu().numpy().astype(np.float64)
            assert np.allclose(sums, ref["stats"], rtol=2e-4, atol=2e-5 * (1 + np.abs(ref["stats"]).max())), nm
            assert int(pop.step_count[p]) == 1


@gpu
def test_population_update_free_run_tracks_float64():
    """Three members with different data, learning rates, clip norms and loss coefficients, 60 updates each in two
    launches, against 60 float64 updates each: every parameter within 1e-4 (about one learning rate: the float32 and
    float64 Adam trajectories part by up to a step where a moment is near zero)."""
    dev = torch.device("cuda", 0)
    names = ["B512_mixed", "B512_inside", "B512_outside"]
    problems = [_member_problem(nm, seed=30 + i) for i, nm in enumerate(names)]
    lrs, mgn = [1e-4, 5e-5, 3e-5], [1.0, 0.5, 2.0]
    pop, data, offs = _stage(problems, 512, dev, lr=lrs, max_grad_norm=mgn)
    upd = PopulationPPOUpdate(pop, 512)
    rng = np.random.default_rng(7)
    U = 60
    idx = np.stack([np.stack([rng.choice(pb.rows, 512, replace=False) for _ in range(U)]) + o
                    for pb, o in zip(problems, offs)])
    idx_t = torch.as_tensor(idx).to(dev)
    upd.launch(data[0], idx_t[:, :25].contiguous(), *data[1:])
    upd.launch(data[0], idx_t[:, 25:].contiguous(), *data[1:])
    torch.cuda.synchronize()
    for p, pb in enumerate(problems):
        hp = dict(pb.hp, max_grad_norm=float(np.float32(mgn[p])))
        lr = float(np.float32(lrs[p]))
        state = [a.astype(np.float64) for a in pb.state]
        q, m, v = flatten(state), np.zeros(N_PARAMS), np.zeros(N_PARAMS)
        for t in range(U):
            rows = idx[p, t] - offs[p]
            g = loss_and_grads_f64(unflatten(q), pb.obs[rows], pb.act[rows], pb.old[rows], pb.adv[rows], pb.ret[rows],
                                   hp)["grad"]
            q, m, v = clip_adam_f64(q, g, m, v, t + 1, lr, hp)
        err = float(np.max(np.abs(_flat(pop, p) - q)))
        print(f"\n[worst] population free run member {p}: {err:.3g} (bound 1e-4)")
        assert err <= 1e-4
        assert int(pop.step_count[p]) == U


def _snap(pop, p):
    return [t[p].clone() for t in pop.params] + [pop.exp_avg[p].clone(), pop.exp_avg_sq[p].clone(),
                                                  pop.sums[p].clone(), pop.step_count[p].clone()]


@gpu
def test_population_update_members_are_independent_and_deterministic():
    dev = torch.device("cuda", 0)
    names = ["B512_mixed", "B512_inside", "B512_outside", "B512_const_adv", "B512_mixed"]
    problems = [_member_problem(nm, seed=60 + i) for i, nm in enumerate(names)]
    lrs, mgn = [3e-4, 1e-3, 1e-4, 2e-4, 3e-4], [1.0, 0.3, 5.0, 1.0, 1.0]
    U = 12

    def run(members, splits):
        probs = [problems[i] for i in members]
        pop, data, offs = _stage(probs, 512, dev, lr=[lrs[i] for i in members], max_grad_norm=[mgn[i] for i in members])
        idx = torch.as_tensor(np.stack([np.stack([np.random.default_rng(100 + i * 1000 + t).choice(problems[i].rows, 512)
                                                  for t in range(U)]) + o for i, o in zip(members, offs)])).to(dev)
        upd = PopulationPPOUpdate(pop, 512)
        lo = 0
        for s in splits:
            upd.launch(data[0], idx[:, lo:lo + s].contiguous(), *data[1:])
            lo += s
        torch.cuda.synchronize()
        return pop

    alone = run([0], [U])
    inside = run([0, 1, 2, 3, 4], [U])
    split = run([0, 1, 2, 3, 4], [5, 7])
    split3 = run([2, 0], [1, 0, 11])
    ref = _snap(alone, 0)
    for pop, p in ((inside, 0), (split, 0), (split3, 1)):
        for a, b in zip(_snap(pop, p), ref):
            assert torch.equal(a, b)
    twin = run([4, 4], [U])                          # two members with identical inputs end bit-identical
    for a, b in zip(_snap(twin, 0), _snap(twin, 1)):
        assert torch.equal(a, b)
    assert not torch.equal(_snap(inside, 1)[0], ref[0])


@gpu
def test_resident_clusters_are_reported():
    L = _lib.lib()
    n = C.c_int(0)
    _lib.check(L.carenv_ppo_epoch_pop_resident_clusters(C.byref(n)), "carenv_ppo_epoch_pop_resident_clusters")
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    assert 1 <= n.value <= sms // L.carenv_ppo_epoch_pop_cluster_size()


# ---- GPU: end to end --------------------------------------------------------------------------------------------------
def _pop_args(argv):
    return popmod.parse_args(["--track", "big_track", "--n-envs", "24"] + argv)


@gpu
def test_epoch_one_equals_train_ppo_and_rewards_rise(capsys):
    from ppo_car_b200.train_ppo import parse_args, train

    out = popmod.train_population(_pop_args(["--seeds", "0-7", "--n-epochs", "30"]))
    hist = out["history"]
    assert len(hist) == 30 * 8 and len(out["final"]) == 8 and len(out["summary"]) == 1
    for m in range(8):
        rs = [r["avg_reward"] for r in hist if r["member"] == m]
        print(f"\nmember {m}: avg_reward epoch 1 {rs[0]:.4f}, last 5 {np.mean(rs[-5:]):.4f}")
        assert np.mean(rs[-5:]) > rs[0] + 0.02, m
    for seed in (0, 5):
        single = train(parse_args(["--track", "big_track", "--n-envs", "24", "--n-epochs", "1", "--seed", str(seed),
                                   "--fused-rollout", "--fused-update"]))[0]
        mine = next(r for r in hist if r["epoch"] == 1 and r["seed"] == seed)
        assert mine["avg_reward"] == single["avg_reward"] and mine["episodes"] == single["episodes"], seed
        assert mine["lr"] == single["lr"]


@gpu
def test_member_checkpoints_load_into_evaluate(tmp_path):
    from ppo_car_b200 import evaluate

    out = popmod.train_population(_pop_args(["--seeds", "4,9", "--n-epochs", "2", "--n-steps", "64",
                                             "--batch-size", "64", "--checkpoint-dir", str(tmp_path),
                                             "--run-name", "sweep", "--learning-rate", "3e-4,1e-3",
                                             "--eval-every", "2", "--eval-episodes", "64"]))
    assert len(out["final"]) == 4 and all(r["eval_return"] is not None for r in out["final"])
    assert {"eval_return_mean", "avg_reward_std"} <= set(out["summary"][0])
    dev = torch.device("cuda", 0)
    for m in range(4):
        path = tmp_path / "sweep" / f"member_{m}" / "model.dat"
        assert path.exists()
        net = evaluate.load_checkpoint(str(path))
        res = evaluate.main(["--checkpoint", str(path), "--episodes", "64", "--seed", "7"])
        env = ppo_car_b200.VecCarEnv(1, ppo_car_b200.builtin_track("big_track"), device=dev)
        direct = ppo_car_b200.evaluate_policy(env, net.actor.to(dev), 64, seed=7).summary()
        assert res["mean_return"] == direct["mean_return"] and res["episodes"] == direct["episodes"]


@pytest.mark.gpu
@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_two_ranks_split_the_members(tmp_path):
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    argv = ["--track", "big_track", "--n-envs", "8", "--n-epochs", "2", "--n-steps", "64", "--batch-size", "64",
            "--seeds", "0-2"]
    subprocess.check_call([sys.executable, "-m", "torch.distributed.run", "--nproc-per-node", "2", "-m",
                           "ppo_car_b200.population", *argv, "--log-json", str(tmp_path / "two.jsonl")], cwd=root)
    one = popmod.train_population(popmod.parse_args(argv))["history"]
    import json

    two = [json.loads(l) for r in (0, 1) for l in open(tmp_path / f"two.jsonl.rank{r}")]
    key = lambda r: (r["epoch"], r["member"])
    assert sorted((key(r), r["avg_reward"], r["policy_loss"]) for r in two) == \
        sorted((key(r), r["avg_reward"], r["policy_loss"]) for r in one)
