"""PPO divergence statistics and the early stop of the one-launch epoch kernels (carenv_ppo_epoch_kl,
carenv_ppo_epoch_pop_kl) and of train_ppo / population (--target-kl, --kl-stats).

  * CPU: the option refusals come before any device work; the C ABI refuses null outputs and bad targets.
  * k_ppo_epoch<8, true> with target +inf equals k_ppo_epoch<8> bit for bit over batch sizes and grid sizes; its
    approx KL tracks float64 at the kernel's own parameters, its clip fraction is exact; the stop rule stops where the
    kernel's own statistics say and leaves exactly the state of a shorter epoch; two ranks agree bit for bit.
  * k_ppo_epoch_pop<true>: target +inf equals k_ppo_epoch_pop; members stop on their own, each as it would alone.
  * train_ppo / population end to end.
"""
import ctypes as C
import math
import os

import numpy as np
import pytest
import torch

from tests.ppo_reference import (as_float32_values, dyadic_problem, hparams, new_logp_f64, old_logp_with_margin)

U32 = 2.0 ** -24                      # float32 unit roundoff


# ---- CPU --------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("argv,words", [
    (["--kl-stats", "--graph-update", "--fused-rollout"], "--graph-update"),
    (["--target-kl", "0.01", "--graph-update"], "--graph-update"),
    (["--target-kl", "0.01", "--fused-update", "--per-minibatch-update"], "per-minibatch"),
    (["--kl-stats", "--fused-update", "--fused-rollout", "--compact-obs"], "per-minibatch"),
    (["--target-kl", "0"], "positive"),
    (["--target-kl", "-0.01"], "positive"),
    (["--target-kl", "nan"], "positive"),
])
def test_train_ppo_refusals_come_before_any_device_work(argv, words, monkeypatch):
    from ppo_car_b200.train_ppo import parse_args, train

    monkeypatch.setattr(torch.cuda, "set_device", lambda *a: pytest.fail("device work before the refusal"))
    with pytest.raises(SystemExit, match=words):
        train(parse_args(["--track", "track"] + argv))


@pytest.mark.parametrize("argv", [["--target-kl", "nan"], ["--target-kl", "0"], ["--kl-stats", "--target-kl", "-1"]])
def test_population_refuses_a_bad_target_before_any_device_work(argv, monkeypatch):
    import ppo_car_b200.population as popmod

    monkeypatch.setattr(torch.cuda, "set_device", lambda *a: pytest.fail("device work before the refusal"))
    with pytest.raises(SystemExit, match="positive"):
        popmod.train_population(popmod.parse_args(["--seeds", "0-1"] + argv))


def test_kl_records_count_the_stopping_update():
    from ppo_car_b200.train_ppo import kl_record

    rows = [[0.1, 0.5], [0.3, 0.25], [float("nan")] * 2]
    assert kl_record(rows, 1) == {"approx_kl": 0.2, "clip_fraction": 0.375, "updates": 1}
    assert kl_record(rows[:2], 2)["updates"] == 2 and kl_record(rows[:2], 2)["approx_kl"] == 0.2


def test_abi_refuses_null_outputs_and_bad_targets():
    from ppo_car_b200 import _lib

    L = _lib.lib()
    dummy = C.c_void_p(64)                # never dereferenced: the checks come first
    single = [dummy] * 14 + [512, 4, 0.2, 0.5, 0.001] + [dummy] * 4 + [0.9, 0.999, 1e-5, 1.0] + [dummy] * 4 + [0, None,
                                                                                                             None]
    pop = [1] + [dummy] * 14 + [512, 4] + [dummy] * 5 + [0.9, 0.999, 1e-5] + [dummy] * 4 + [None]
    for fn, base in ((L.carenv_ppo_epoch_kl, single), (L.carenv_ppo_epoch_pop_kl, pop)):
        assert fn(*base, 0.01, None, dummy) == -1                                 # CARENV_E_INVAL: kl_out
        assert fn(*base, 0.01, dummy, None) == -1                                 # n_done
        for bad in (0.0, -1.0, float("nan"), -float("inf")):
            assert fn(*base, bad, dummy, dummy) == -1, bad
        assert b"target_kl" in L.carenv_last_error()


# ---- GPU: single policy ----------------------------------------------------------------------------------------------
def _problem(B, seed=1, inside=0.5):
    hp = as_float32_values(hparams())
    rows = max(2 * B, 64)
    state, obs, act, adv, ret = dyadic_problem(rows, seed=seed)
    old = old_logp_with_margin(new_logp_f64(state, obs, act), inside, hp["clip_ratio"], seed=seed)
    return hp, state, (obs, act, old, adv, ret)


def _updater(state, hp, B, dev, lr=3e-4):
    from ppo_car_b200.ppo_update import FusedPPOUpdate
    from ppo_car_b200.train_ppo import ActorCritic

    net = ActorCritic(18, 9).to(dev)
    with torch.no_grad():
        for p, s in zip([net.actor[0].weight, net.actor[0].bias, net.actor[2].weight, net.actor[2].bias,
                         net.critic[0].weight, net.critic[0].bias, net.critic[2].weight, net.critic[2].bias], state):
            p.copy_(torch.as_tensor(np.asarray(s, np.float32)).reshape(p.shape))
    return FusedPPOUpdate(net.actor, net.critic, B, lr=lr, clip_ratio=hp["clip_ratio"], vf_coef=hp["vf_coef"],
                          ent_coef=hp["ent_coef"], max_grad_norm=hp["max_grad_norm"], betas=hp["betas"], eps=hp["eps"])


def _dev_data(data, dev):
    return [torch.as_tensor(a).to(dev).contiguous() for a in data]


def _snap(upd):
    return [p.detach().clone() for p in upd.params] + [upd.exp_avg.clone(), upd.exp_avg_sq.clone(),
                                                        upd.step_count.clone()]


def _same(a, b):
    return all(torch.equal(x, y) for x, y in zip(a, b))


def _idx(rows, n, B, dev, seed=5):
    g = torch.Generator(device=dev).manual_seed(seed)
    return torch.randint(0, rows, (n, B), device=dev, generator=g)


@pytest.mark.gpu
@pytest.mark.parametrize("n_ctas", [49, 64, 86, 148])
@pytest.mark.parametrize("B", [2, 3, 512, 1024])
def test_kl_inf_equals_the_plain_epoch_kernel(B, n_ctas):
    """k_ppo_epoch<8, true> at target +inf: parameters, moments, step and loss sums equal k_ppo_epoch<8>'s bit for
    bit; every update is applied and reported.  At 86 CTAs the parameter slices fill 12,298 exactly, so the two
    statistic sums are reduced by threads outside every slice."""
    dev = torch.device("cuda")
    if n_ctas > torch.cuda.get_device_properties(dev).multi_processor_count:
        pytest.skip("more CTAs than SMs")
    hp, state, data = _problem(B)
    obs, act, old, adv, ret = _dev_data(data, dev)
    n = 7
    idx = _idx(obs.shape[0], n, B, dev)
    a, b = _updater(state, hp, B, dev), _updater(state, hp, B, dev)
    a.run_epoch(obs, idx, act, old, adv, ret, n_ctas=n_ctas)
    b.run_epoch(obs, idx, act, old, adv, ret, n_ctas=n_ctas, target_kl=float("inf"))
    a.check_epoch(); b.check_epoch()
    assert _same(_snap(a), _snap(b)) and torch.equal(a.sums, b.sums)
    assert int(b.n_done) == n and int(b.step_count) == n
    assert torch.isfinite(b.kl).all() and (b.kl[:, 1] >= 0).all() and (b.kl[:, 1] <= 1).all()


def _kl_f64(state, obs, act, old, idx, clip_ratio):
    """float64 approx KL, clip count and the ratios' least distance to the clip edges of one minibatch."""
    lr = new_logp_f64(state, obs[idx], act[idx]) - old[idx].astype(np.float64)
    r = np.exp(lr)
    terms = (r - 1.0) - lr
    edge = np.min(np.abs(np.abs(r - 1.0) - clip_ratio))
    return terms, int(np.sum(np.abs(r - 1.0) > clip_ratio)), edge, r


@pytest.mark.gpu
@pytest.mark.parametrize("B", [3, 512])
def test_kl_tracks_float64_and_clip_fraction_is_exact(B):
    """kl[u] of one 6-update launch against float64 at the parameters before update u, which one-update launches of
    the plain kernel reproduce bit for bit.  Bound: the float32 log ratio carries at most (256 + 16) u times the
    absolute logit sum S of the sample (dot product of 256 terms, bias, max, log-sum-exp), which moves the term
    (ratio - 1) - log ratio by |ratio - 1| times that; expf, the two subtractions and the term itself add 4 u ratio +
    u |term|; the fixed-order sum of B terms adds B u mean|term|.  Ratios stay clear of the clip edges, so the clip
    fraction equals the float64 count exactly."""
    dev = torch.device("cuda")
    hp, state, data = _problem(B, seed=2)
    obs_n, act_n, old_n, *_ = data
    obs, act, old, adv, ret = _dev_data(data, dev)
    n = 6
    idx = _idx(obs.shape[0], n, B, dev, seed=9)
    k = _updater(state, hp, B, dev, lr=1e-5)
    k.run_epoch(obs, idx, act, old, adv, ret, target_kl=float("inf"))
    kl = k.kl.double().cpu().numpy()
    one = _updater(state, hp, B, dev, lr=1e-5)
    idx_n = idx.cpu().numpy()
    worst = 0.0
    for u in range(n):
        st = [p.detach().double().cpu().numpy() for p in one.params]
        terms, count, edge, r = _kl_f64(st, obs_n, act_n, old_n, idx_n[u], hp["clip_ratio"])
        w2a, b2a = st[2], st[3]
        x = obs_n[idx_n[u]].astype(np.float64)
        h = np.maximum(x @ st[0].T + st[1], 0.0)
        S = (np.abs(h) @ np.abs(w2a).T + np.abs(b2a)).max(axis=1)
        per = (256 + 16) * U32 * S * np.abs(r - 1.0) + 4 * U32 * r + U32 * np.abs(terms)
        tol = per.max() + B * U32 * np.abs(terms).mean()
        err = abs(kl[u, 0] - terms.mean())
        worst = max(worst, err / tol)
        assert err <= tol, (u, err, tol)
        # 10x the log-ratio error bound: the float32 comparisons see the float64 sides
        assert edge > 10 * (256 + 16) * U32 * S.max() * (1 + hp["clip_ratio"]), "ratios drifted to a clip edge"
        assert np.float32(kl[u, 1]) == np.float32(np.float32(count) * np.float32(1.0 / np.float32(B))), u
        one.run_epoch(obs, idx[u:u + 1], act, old, adv, ret)
    assert _same(_snap(one), _snap(k))
    print(f"\n[worst] approx KL: {worst:.3g} of the tolerance")


@pytest.mark.gpu
def test_stop_rule_stops_where_the_kernel_says():
    """Targets placed between the kernel's own values: stop at update 0, in the middle, never.  n_done is the first u
    with kl[u] > target; the state equals a plain launch of exactly n_done updates; rows after the stop are NaN; a
    following launch continues as it would from that state."""
    dev = torch.device("cuda")
    B, n = 512, 12
    hp, state, data = _problem(B, seed=3)
    obs, act, old, adv, ret = _dev_data(data, dev)
    idx = _idx(obs.shape[0], n, B, dev, seed=11)
    idx2 = _idx(obs.shape[0], 5, B, dev, seed=12)
    ref = _updater(state, hp, B, dev, lr=1e-3)
    ref.run_epoch(obs, idx, act, old, adv, ret, target_kl=float("inf"))
    kl = ref.kl[:, 0].double().cpu().numpy()
    assert kl[0] > 0
    mid = next(s for s in range(n // 3, n) if kl[s] > kl[:s].max())
    for stop, tau in ((0, kl[0] / 2), (mid, float(kl[:mid].max())), (n, float(kl.max()) * 2)):
        k = _updater(state, hp, B, dev, lr=1e-3)
        k.run_epoch(obs, idx, act, old, adv, ret, target_kl=tau)
        plain = _updater(state, hp, B, dev, lr=1e-3)
        plain.run_epoch(obs, idx[:stop], act, old, adv, ret)
        assert int(k.n_done) == stop == next((u for u in range(n) if kl[u] > tau), n)
        assert _same(_snap(k), _snap(plain)) and int(k.step_count) == stop
        n_eval = min(stop + 1, n)
        assert torch.equal(k.kl[:n_eval], ref.kl[:n_eval]) and torch.isnan(k.kl[n_eval:]).all()
        k.run_epoch(obs, idx2, act, old, adv, ret, target_kl=float("inf"))
        plain.run_epoch(obs, idx2, act, old, adv, ret)
        assert _same(_snap(k), _snap(plain))


def _peer_worker(rank, world, port, q):
    import torch.distributed as dist

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", device_id=dev)
    try:
        B = 512
        hp, state, _ = _problem(B, seed=3)
        _, _, data = _problem(B, seed=20 + rank)                    # a different shard per rank
        obs, act, old, adv, ret = _dev_data(data, dev)
        upd = _updater(state, hp, B, dev, lr=1e-3)
        upd.connect()
        # exchanged updates per epoch: 1, 4, 1, 5, 1, 2 (odd and even), then a plain launch after the KL launches
        plan = [(4, 1e-30), (4, 1e30), (3, 1e-30), (5, 1e30), (4, 1e-30), (2, 1e30)]
        kls, dones = [], []
        for e, (n, tau) in enumerate(plan):
            torch.manual_seed(100 * e + rank)
            idx = torch.randint(0, obs.shape[0], (n, B), device=dev)
            upd.run_epoch(obs, idx, act, old, adv, ret, world=world, target_kl=tau)
            upd.check_epoch()
            kls.append(upd.kl.clone())
            dones.append(int(upd.n_done))
        upd.run_epoch(obs, torch.randint(0, obs.shape[0], (3, B), device=dev), act, old, adv, ret, world=world)
        upd.check_epoch()
        flat = torch.cat([p.detach().reshape(-1) for p in upd.params] + [torch.cat([k.reshape(-1) for k in kls])])
        gathered = [torch.empty_like(flat) for _ in range(world)]
        dist.all_gather(gathered, flat)
        same = all(torch.equal(torch.nan_to_num(gathered[0], nan=7.0), torch.nan_to_num(g, nan=7.0)) for g in gathered)
        upd.close()
        q.put((rank, same, dones, int(upd.step_count)))
    finally:
        dist.destroy_process_group()


@pytest.mark.gpu
@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_two_ranks_agree_and_keep_the_exchange_parity():
    import torch.multiprocessing as mp

    world = 2
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_peer_worker, args=(r, world, 29771, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = [q.get(timeout=300) for _ in range(world)]
    for p in procs:
        p.join(60)
    for rank, same, dones, steps in res:
        assert same and dones == [0, 4, 0, 5, 0, 2] and steps == 11 + 3, (rank, same, dones, steps)


# ---- GPU: population -------------------------------------------------------------------------------------------------
def _pop_problem(seeds, lrs, dev, M=4000, B=256, n=10):
    from ppo_car_b200.population import Population, PopulationPPOUpdate

    pop = Population(seeds, 4, [{"learning_rate": lr} for lr in lrs], dev)
    g = torch.Generator(device=dev).manual_seed(0)
    obs = torch.rand((M, 18), device=dev, generator=g)
    act = torch.randint(0, 9, (M,), device=dev, generator=g).float()
    old = torch.full((M,), -math.log(9.0), device=dev) + torch.randn(M, device=dev, generator=g) * 0.1
    adv, ret = torch.randn(M, device=dev, generator=g) * 2 + 0.5, torch.randn(M, device=dev, generator=g)
    upd = PopulationPPOUpdate(pop, B)
    return pop, upd, (obs, act, old, adv, ret)


def _pop_idx(seeds, M, n, B, dev):
    rows = []
    for s in seeds:                                           # a member's minibatches depend on its seed only
        g = torch.Generator(device=dev).manual_seed(1000 + s)
        rows.append(torch.randint(0, M, (n, B), device=dev, generator=g))
    return torch.stack(rows).contiguous()


def _pop_state(pop, p):
    return [t[p].clone() for t in pop.params] + [pop.exp_avg[p].clone(), pop.exp_avg_sq[p].clone(),
                                                  pop.step_count[p].clone()]


@pytest.mark.gpu
def test_population_kl_inf_equals_the_plain_population_kernel():
    dev = torch.device("cuda", 0)
    seeds, lrs = [0, 1, 2], [3e-4, 1e-3, 3e-3]
    a, ua, data = _pop_problem(seeds, lrs, dev)
    b, ub, _ = _pop_problem(seeds, lrs, dev)
    idx = _pop_idx(seeds, data[0].shape[0], 10, 256, dev)
    ua.launch(data[0], idx, *data[1:])
    ub.launch(data[0], idx, *data[1:], target_kl=float("inf"))
    for p in range(3):
        assert _same(_pop_state(a, p), _pop_state(b, p))
    assert torch.equal(a.sums, b.sums) and ub.n_done.tolist() == [10] * 3 and torch.isfinite(ub.kl).all()


@pytest.mark.gpu
def test_population_members_stop_on_their_own():
    """One target for members of different learning rates: they stop at different updates, each bit-identical (state,
    statistics, n_done) to the member run alone (P = 1) and to the same member in another order among others."""
    dev = torch.device("cuda", 0)
    seeds, lrs = [0, 1, 2, 3], [1e-4, 1e-3, 3e-3, 1e-2]
    n = 10
    pop, upd, data = _pop_problem(seeds, lrs, dev, n=n)
    idx = _pop_idx(seeds, data[0].shape[0], n, 256, dev)
    probe, uprobe, _ = _pop_problem(seeds, lrs, dev, n=n)
    uprobe.launch(data[0], idx, *data[1:], target_kl=float("inf"))
    tau = float(uprobe.kl[:, :, 0].median())
    upd.launch(data[0], idx, *data[1:], target_kl=tau)
    done = upd.n_done.tolist()
    kl_inf = uprobe.kl[:, :, 0].double().cpu().numpy()
    assert done == [next((u for u in range(n) if kl_inf[p, u] > tau), n) for p in range(4)]
    assert len(set(done)) >= 2 and min(done) < n
    for p in range(4):
        alone, ualone, _ = _pop_problem([seeds[p]], [lrs[p]], dev, n=n)
        ualone.launch(data[0], idx[p:p + 1].contiguous(), *data[1:], target_kl=tau)
        assert _same(_pop_state(pop, p), _pop_state(alone, 0))
        assert int(ualone.n_done[0]) == done[p]
        assert torch.equal(torch.nan_to_num(ualone.kl[0], nan=7.0), torch.nan_to_num(upd.kl[p], nan=7.0))
    order = [2, 0, 3, 1]
    perm, uperm, _ = _pop_problem([seeds[q] for q in order], [lrs[q] for q in order], dev, n=n)
    uperm.launch(data[0], idx[order].contiguous(), *data[1:], target_kl=tau)
    for i, q in enumerate(order):
        assert _same(_pop_state(perm, i), _pop_state(pop, q)) and int(uperm.n_done[i]) == done[q]


# ---- GPU: end to end -------------------------------------------------------------------------------------------------
SMALL = ["--track", "track", "--n-envs", "64", "--n-epochs", "3", "--n-steps", "256", "--batch-size", "128",
         "--train-iters", "2"]
KEYS = {"approx_kl", "clip_fraction", "updates", "explained_variance"}


def _final(tmp_path, name, extra):
    from ppo_car_b200.train_ppo import parse_args, train

    hist = train(parse_args(SMALL + extra + ["--checkpoint-dir", str(tmp_path), "--run-name", name]))
    return hist, torch.load(os.path.join(tmp_path, name, "model.dat"))


@pytest.mark.gpu
def test_train_ppo_kl_stats_keeps_the_weights(tmp_path):
    fused = ["--fused-rollout", "--fused-update"]
    h0, w0 = _final(tmp_path, "plain", fused)
    h1, w1 = _final(tmp_path, "stats", fused + ["--kl-stats"])
    assert all(torch.equal(w0[k], w1[k]) for k in w0)
    assert all(not (KEYS & set(r)) for r in h0) and all(KEYS <= set(r) for r in h1)
    assert all(r["updates"] == 2 * 2 and math.isfinite(r["approx_kl"]) and 0 <= r["clip_fraction"] <= 1 for r in h1)
    assert all(r[k] == s[k] for r, s in zip(h0, h1) for k in ("policy_loss", "value_loss", "entropy", "avg_reward"))
    h2, _ = _final(tmp_path, "stop", fused + ["--target-kl", "1e-7"])
    assert any(r["updates"] < 4 for r in h2)


@pytest.mark.gpu
def test_train_ppo_eager_path_stops_on_its_approx_kl(tmp_path):
    h0, w0 = _final(tmp_path, "plain", [])
    h1, w1 = _final(tmp_path, "stats", ["--kl-stats"])
    assert all(torch.equal(w0[k], w1[k]) for k in w0) and all(r["updates"] == 4 for r in h1)
    # the first update of an epoch sees the rollout's own policy: its approx KL is ~0, so the second one decides
    tau = min(r["approx_kl"] for r in h1[1:]) / 4
    h2, _ = _final(tmp_path, "stop", ["--target-kl", str(tau)])
    assert any(r["updates"] < 4 for r in h2)
    for r in h2:                               # the stopping update's KL is in the mean and exceeds the target
        if r["updates"] < 4:
            assert r["approx_kl"] * (r["updates"] + 1) > tau


@pytest.mark.gpu
def test_population_target_kl_with_pbt_runs_and_checkpoints_load(tmp_path):
    from ppo_car_b200 import evaluate
    import ppo_car_b200.population as popmod

    args = popmod.parse_args(["--seeds", "0-3", "--track", "track", "--n-envs", "8", "--n-epochs", "4", "--n-steps",
                              "128", "--batch-size", "64", "--train-iters", "2", "--target-kl", "0.001",
                              "--pbt-every", "2", "--pbt-fraction", "0.25", "--eval-episodes", "16",
                              "--checkpoint-dir", str(tmp_path), "--run-name", "p"])
    out = popmod.train_population(args)
    recs = [r for r in out["history"] if "approx_kl" in r]
    assert len(recs) == 4 * 4 and all(KEYS <= set(r) for r in recs)
    assert all(0 <= r["updates"] <= 2 * 2 for r in recs)
    path = os.path.join(tmp_path, "p", "member_0", "model.dat")
    res = evaluate.main(["--checkpoint", path, "--episodes", "16", "--seed", "1"])
    assert res is not None
