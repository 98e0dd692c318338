"""The fused PPO update kernels against the float64 restatement in tests/ppo_reference.py.

Both launch paths are covered: the per-minibatch kernels (FusedPPOUpdate.grad + apply: k_ppo_forward /
k_ppo_backward / k_ppo_adam) and the one-launch epoch kernel (FusedPPOUpdate.run_epoch: k_ppo_epoch, what train_ppo
runs by default).  run_epoch does not expose gradients, so its gradient is read through a "linear Adam" probe: one update
from m = v = 0 with eps = 1e6 and lr = 1e9 moves every parameter by -lr * g / (|g| + eps) = -1000 g to 1e-6 relative.

The minibatches come from tests/ppo_reference.dyadic_problem, whose first layer is exact in float32, so kernel and
reference take the same ReLU decisions, and from old_logp_with_margin, whose ratios stay clear of the clip boundaries.
Tolerance-based tests print the worst error they saw as a fraction of the tolerance (run pytest with -s to see it).
"""
import functools
import math
from types import SimpleNamespace

import numpy as np
import pytest
import torch
import torch.nn as nn

from tests.ppo_reference import (N_PARAMS, as_float32_values, clip_adam_f64, clip_coef_f64, dyadic_problem, flatten,
                                 hparams, loss_and_grads_f64, net_f64, new_logp_f64, old_logp_with_margin,
                                 unflatten)

U32 = 2.0 ** -24                      # float32 unit roundoff

# ---- the edge matrix ------------------------------------------------------------------------------------------------
CASES = {
    "B2": dict(B=2),                                   # two different advantages: the unbiased std divides by B - 1 = 1
    "B37": dict(B=37),
    "B512": dict(B=512),                               # ratios mixed: half inside the clip range, half outside
    "B1000": dict(B=1000),
    "B1024": dict(B=1024),
    "const_adv": dict(B=1000, adv_const=0.5),          # normalised advantages exactly 0: the std clamp at 1e-5
    "const_adv_B2": dict(B=2, adv_const=0.5),
    "idx_one_row": dict(B=64, dup="one"),
    "idx_half_repeated": dict(B=512, dup="half"),
    "zero_pre": dict(B=256, zero_pre=True),            # b1 = 0 and zero observation rows: pre-activations exactly 0
    "ratios_inside": dict(B=512, inside=1.0),
    "ratios_outside": dict(B=512, inside=0.0),         # alternately below and above the clip range
    # most probabilities underflow to 0.  Float32 logits of magnitude ~900 carry absolute errors ~1e-4, and the
    # softmax gradient's cancellation in d loss / d h = sum_q dz_q W2[q] amplifies them: float32 torch autograd of the
    # same loss misses the default gradient tolerance by up to 21x here, hence a 50x wider one
    "logits_x1000": dict(B=512, logit_scale=1000.0, tol_scale=50.0),
    "hparams": dict(B=512, hp=dict(clip_ratio=0.1, vf_coef=1.0, ent_coef=0.01, max_grad_norm=0.5, betas=(0.8, 0.99),
                                   eps=1e-7)),
}


@functools.lru_cache(maxsize=None)
def problem(name):
    """The case's data (float32 numpy, ``rows`` samples), minibatch indices and float64 reference of one update."""
    c = CASES[name]
    B = c["B"]
    rows = max(2 * B, 64)
    seed = sorted(CASES).index(name) + 1
    hp = as_float32_values(hparams(**c.get("hp", {})))          # the kernels take every scalar as float32
    state, obs, act, adv, ret = dyadic_problem(rows, seed=seed, zero_pre=c.get("zero_pre", False),
                                               logit_scale=c.get("logit_scale", 1.0), adv_const=c.get("adv_const"))
    old = old_logp_with_margin(new_logp_f64(state, obs, act), c.get("inside", 0.5), hp["clip_ratio"], seed=seed)
    rng = np.random.default_rng(100 + seed)
    if c.get("dup") == "one":
        idx = np.full(B, 5, np.int64)
    elif c.get("dup") == "half":
        first = rng.choice(rows, B // 2, replace=False)
        idx = rng.permutation(np.concatenate([first, first[:B - B // 2]]))
    else:
        idx = rng.choice(rows, B, replace=False)
    ref = loss_and_grads_f64(state, obs[idx], act[idx], old[idx], adv[idx], ret[idx], hp)
    return SimpleNamespace(name=name, B=B, hp=hp, tol_scale=c.get("tol_scale", 1.0), state=state, obs=obs, act=act, old=old, adv=adv, ret=ret, idx=idx,
                           ref=ref, p0=flatten(state))


def grad_tol(g64, scale=1.0):
    """Per-element tolerance of a float32 gradient: 2e-4 relative plus 2e-6 of the largest gradient element (times
    the case's ``tol_scale``)."""
    g64 = np.asarray(g64, np.float64)
    return scale * (2e-4 * np.abs(g64) + 2e-6 * np.abs(g64).max())


def ulp32(x):
    """Spacing of float32 numbers at |x|."""
    return np.spacing(np.abs(np.asarray(x, np.float64)).astype(np.float32)).astype(np.float64)


def _worst(err, tol, what):
    r = float(np.max(np.abs(err) / tol))
    print(f"\n[worst] {what}: {r:.3g} of the tolerance")
    return r


# ---- CPU: the reference itself ---------------------------------------------------------------------------------------
def test_clip_adam_f64_matches_torch_clip_and_adam():
    """clip_adam_f64 = nn.utils.clip_grad_norm_ + torch.optim.Adam(eps=...) in float64 over 10 steps, with the learning
    rate changed mid-way (train_ppo decays it between epochs), in both the clipped and the unclipped regime."""
    rng = np.random.default_rng(0)
    hp = hparams(max_grad_norm=0.5, betas=(0.85, 0.995), eps=1e-6)
    p0 = rng.standard_normal(N_PARAMS) * 0.1
    params = [nn.Parameter(torch.as_tensor(a.copy())) for a in unflatten(p0)]
    opt = torch.optim.Adam(params, lr=3e-4, betas=hp["betas"], eps=hp["eps"])
    p, m, v = p0, np.zeros(N_PARAMS), np.zeros(N_PARAMS)
    clipped = []
    for t in range(1, 11):
        lr = 3e-4 if t <= 5 else 3e-4 * 0.99 ** 150
        opt.param_groups[0]["lr"] = lr
        g = rng.standard_normal(N_PARAMS) * (0.02 if t % 2 else 0.001)      # norm ~2.2 / ~0.11 against max 0.5
        clipped.append(clip_coef_f64(g, hp["max_grad_norm"]) < 1.0)
        for q, gq in zip(params, unflatten(g)):
            q.grad = torch.as_tensor(gq.copy())
        nn.utils.clip_grad_norm_(params, hp["max_grad_norm"])
        opt.step()
        p, m, v = clip_adam_f64(p, g, m, v, t, lr, hp)
        np.testing.assert_allclose(flatten(params), p, rtol=1e-12, atol=1e-15)
        np.testing.assert_allclose(flatten([opt.state[q]["exp_avg"] for q in params]), m, rtol=1e-12, atol=1e-18)
        np.testing.assert_allclose(flatten([opt.state[q]["exp_avg_sq"] for q in params]), v, rtol=1e-12, atol=1e-20)
    assert any(clipped) and not all(clipped)


@pytest.mark.parametrize("zero_pre", [False, True])
def test_dyadic_problem_first_layer_is_exact_in_float32(zero_pre):
    """The float32 first layer equals the float64 one bit for bit (so every kernel takes the reference's ReLU
    decisions); without zero_pre no pre-activation is 0, with it the zero rows' pre-activations are exactly 0."""
    state, obs, *_ = dyadic_problem(1024, seed=3, zero_pre=zero_pre)
    for w, b in ((state[0], state[1]), (state[4], state[5])):
        pre32 = (torch.from_numpy(obs) @ torch.from_numpy(w).T + torch.from_numpy(b)).numpy()
        rev32 = np.zeros_like(pre32)                                         # another summation order
        for k in reversed(range(obs.shape[1])):
            rev32 = rev32 + obs[:, k:k + 1] * w[:, k][None, :]
        rev32 = rev32 + b
        pre64 = obs.astype(np.float64) @ w.astype(np.float64).T + b.astype(np.float64)
        assert np.array_equal(pre32.astype(np.float64), pre64) and np.array_equal(rev32.astype(np.float64), pre64)
        if zero_pre:
            assert np.all(pre64[::4] == 0.0) and np.all(b == 0.0)
        else:
            assert np.abs(pre64).min() >= 2.0 ** -15


def test_old_logp_margins_and_edge_cases_hold():
    """Every case of the edge matrix has the properties its name promises (checked in float64, no GPU needed)."""
    for name, c in CASES.items():
        pb = problem(name)
        lo, hi = 1.0 - pb.hp["clip_ratio"], 1.0 + pb.hp["clip_ratio"]
        r = pb.ref["ratio"]
        assert np.all(np.minimum(np.abs(r - lo), np.abs(r - hi)) >= 1e-3), name
        inside = float(np.mean((r > lo) & (r < hi)))
        if "inside" in c:
            assert inside == c["inside"], name
        if c.get("zero_pre"):
            assert np.any(pb.ref["pre_a"] == 0.0) and np.any(pb.ref["pre_c"] == 0.0)
        else:
            assert np.abs(pb.ref["pre_a"]).min() > 0 and np.abs(pb.ref["pre_c"]).min() > 0, name
        assert np.all(np.isfinite(pb.ref["grad"])) and np.abs(pb.ref["grad"]).max() > 0, name
    adv = problem("const_adv").adv
    B = problem("const_adv").B                          # the epoch kernel forms the mean as sum * (1 / B) in float32
    assert np.float32(np.float32(adv[0] * B) * np.float32(1.0 / B)) == adv[0]
    r = problem("ratios_outside").ref["ratio"]
    assert np.any(r < 0.8) and np.any(r > 1.2)                               # outside on both sides
    p = problem("logits_x1000")
    with torch.no_grad():
        lp = torch.log_softmax(net_f64(p.state).actor(torch.as_tensor(p.obs, dtype=torch.float64)), -1).numpy()
    assert np.mean(lp < -104.0) > 0.3                  # exp(lp) is 0 in float32 for a good share of the probabilities


# ---- GPU -------------------------------------------------------------------------------------------------------------
def _net(state, dev):
    from ppo_car_b200.train_ppo import ActorCritic

    net = ActorCritic(18, 9).to(dev)
    with torch.no_grad():
        for p, s in zip([net.actor[0].weight, net.actor[0].bias, net.actor[2].weight, net.actor[2].bias,
                         net.critic[0].weight, net.critic[0].bias, net.critic[2].weight, net.critic[2].bias], state):
            p.copy_(torch.as_tensor(np.asarray(s, np.float32)).reshape(p.shape))
    return net


def _updater(pb, dev, lr=3e-4, **overrides):
    from ppo_car_b200.ppo_update import FusedPPOUpdate

    net = _net(pb.state, dev)
    hp = dict(pb.hp)
    hp.update(overrides)
    upd = FusedPPOUpdate(net.actor, net.critic, pb.B, lr=lr, clip_ratio=hp["clip_ratio"], vf_coef=hp["vf_coef"],
                         ent_coef=hp["ent_coef"], max_grad_norm=hp["max_grad_norm"], betas=hp["betas"], eps=hp["eps"])
    return upd


def _data(pb, dev):
    t = lambda a: torch.as_tensor(a).to(dev).contiguous()
    return t(pb.obs), t(pb.act), t(pb.old), t(pb.adv), t(pb.ret)


def _flat_params(upd):
    return np.concatenate([p.detach().double().cpu().numpy().reshape(-1) for p in upd.params])


def _n_ctas(which, dev):
    if which == "max":                                  # the launcher accepts up to 160, and no more than the SMs
        return min(160, torch.cuda.get_device_properties(dev).multi_processor_count)
    return which


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(CASES))
def test_per_minibatch_gradients_match_float64(case):
    """(a) FusedPPOUpdate.grad (k_ppo_forward + k_ppo_backward) against the float64 gradient."""
    dev = torch.device("cuda")
    pb = problem(case)
    upd = _updater(pb, dev)
    obs, act, old, adv, ret = _data(pb, dev)
    g = upd.grad(obs, torch.as_tensor(pb.idx).to(dev), act, old, adv, ret).double().cpu().numpy()
    g64 = pb.ref["grad"]
    tol = grad_tol(g64, pb.tol_scale)
    assert _worst(g - g64, tol, f"per-minibatch gradient [{case}]") <= 1.0


@pytest.mark.gpu
@pytest.mark.parametrize("n_ctas", [0, 49, "max"])
@pytest.mark.parametrize("case", list(CASES))
def test_epoch_kernel_gradients_through_linear_adam_probe(case, n_ctas):
    """(b) k_ppo_epoch's gradient, read through one update with m = v = 0, t = 1, eps = 1e6, lr = 1e9: the step is
    -lr * c * g / (c |g| + eps) with c the clip coefficient, about -1000 c g.  Once without clipping (max_grad_norm
    1e30: c = 1 exactly, the cap of clip_grad_norm_) and once with max_grad_norm = 0.25 * |g|, which checks the
    kernel's global norm and clip coefficient."""
    dev = torch.device("cuda")
    pb = problem(case)
    g64 = pb.ref["grad"]
    norm64 = float(np.linalg.norm(g64))
    obs, act, old, adv, ret = _data(pb, dev)
    idx = torch.as_tensor(pb.idx).to(dev).reshape(1, -1).contiguous()
    lr, eps = 1e9, 1e6
    for max_norm in (1e30, float(np.float32(0.25 * norm64))):
        upd = _updater(pb, dev, lr=lr, max_grad_norm=max_norm, eps=eps)
        upd.run_epoch(obs, idx, act, old, adv, ret, n_ctas=_n_ctas(n_ctas, dev))
        upd.check_epoch()
        dp = _flat_params(upd) - pb.p0
        coef = clip_coef_f64(g64, max_norm)
        assert (coef < 0.3) if max_norm < 1e29 else (coef == 1.0)          # clipping active / inactive as intended
        want = -lr * coef * g64 / (coef * np.abs(g64) + eps)
        tol = lr / eps * coef * grad_tol(g64, pb.tol_scale) + ulp32(pb.p0 + dp)         # + rounding of the stored parameter
        assert _worst(dp - want, tol, f"epoch gradient probe [{case}, n_ctas={n_ctas}, clip={coef:.3g}]") <= 1.0
        assert int(upd.step_count) == 1


def adam_error_bound(pb, g64, m0, v0, m64, v64, dp64, coef, t, lr):
    """What a float32 clip + Adam step may differ from clip_adam_f64 by, per element, when the kernel's gradient is
    within grad_tol of the float64 one: the gradient error propagated through the moment updates and the step
    (step_size (1 - beta1) |dg| / (sqrt(v_hat) + eps) plus the v-term), plus float32 rounding of each operation, the
    <= 4 ulp of powf in the bias corrections and the approximate square root / divide of the epoch kernel."""
    hp = pb.hp
    b1, b2 = hp["betas"]
    eps = hp["eps"]
    tg = grad_tol(g64, pb.tol_scale)
    a = coef * np.abs(g64)
    dcoef = coef * float(np.linalg.norm(tg) / np.linalg.norm(g64)) if coef < 1.0 else 0.0
    dgc = coef * tg + dcoef * np.abs(g64) + 2 * U32 * a
    dm = (1 - b1) * dgc + 4 * U32 * (b1 * np.abs(m0) + (1 - b1) * a) + ulp32(m64)
    dv = (1 - b2) * (2 * a * dgc + dgc * dgc) + 4 * U32 * (b2 * v0 + (1 - b2) * a * a) + ulp32(v64)
    bc1, bc2 = 1 - b1 ** t, 1 - b2 ** t
    isb2 = 1.0 / math.sqrt(bc2)
    sv = np.sqrt(v64)
    D = sv * isb2 + eps
    dsv = np.minimum(dv / np.maximum(2 * sv, 1e-300), np.sqrt(dv))
    step = lr / bc1
    ddp = step * dm / D + step * np.abs(m64) * isb2 * dsv / (D * D)
    ddp += np.abs(dp64) * (4 * U32 * b1 ** t / bc1 + 2 * U32 * b2 ** t / bc2 + 12 * U32)
    return ddp, dm, dv


@pytest.mark.gpu
@pytest.mark.parametrize("lr", [3e-4, 3e-4 * 0.99 ** 150])
@pytest.mark.parametrize("t", [1, 2, 10, 1000, 100000])
@pytest.mark.parametrize("case", list(CASES))
def test_clip_adam_with_teacher_forced_state(case, t, lr):
    """(c) One full update (clip + Adam step t from given m, v) through grad + apply and through run_epoch, against
    clip_adam_f64 on the float64 gradient; the bound is twice adam_error_bound.  Also step_count == t afterwards and
    the loss statistics in ``sums`` against the float64 ones."""
    dev = torch.device("cuda")
    pb = problem(case)
    hp = pb.hp
    lr = float(np.float32(lr))
    g64 = pb.ref["grad"]
    rng = np.random.default_rng(t)
    scale = float(np.sqrt(np.mean(g64 * g64)))
    m0 = (rng.standard_normal(N_PARAMS) * scale).astype(np.float32)
    v0 = (m0.astype(np.float64) ** 2 * rng.uniform(0.5, 2.0, N_PARAMS) + 1e-3 * scale * scale).astype(np.float32)
    m0, v0 = m0.astype(np.float64), v0.astype(np.float64)
    p64, m64, v64 = clip_adam_f64(pb.p0, g64, m0, v0, t, lr, hp)
    dp64 = p64 - pb.p0
    coef = clip_coef_f64(g64, hp["max_grad_norm"])
    bp, bm, bv = adam_error_bound(pb, g64, m0, v0, m64, v64, dp64, coef, t, lr)
    obs, act, old, adv, ret = _data(pb, dev)
    idx = torch.as_tensor(pb.idx).to(dev)
    for path in ("per_minibatch", "epoch"):
        upd = _updater(pb, dev, lr=lr)
        upd.exp_avg.copy_(torch.as_tensor(m0, dtype=torch.float32))
        upd.exp_avg_sq.copy_(torch.as_tensor(v0, dtype=torch.float32))
        upd.step_count.fill_(t - 1)
        if path == "per_minibatch":
            upd.grad(obs, idx, act, old, adv, ret)
            upd.apply()
        else:
            upd.run_epoch(obs, idx.reshape(1, -1).contiguous(), act, old, adv, ret)
            upd.check_epoch()
        what = f"[{case}, t={t}, lr={lr:.3g}, {path}]"
        dp = _flat_params(upd) - pb.p0
        bound = 2 * (bp + ulp32(pb.p0 + dp))
        assert _worst(dp - dp64, bound, "Adam step " + what) <= 1.0
        assert _worst(upd.exp_avg.double().cpu().numpy() - m64, 2 * bm, "exp_avg " + what) <= 1.0
        assert _worst(upd.exp_avg_sq.double().cpu().numpy() - v64, 2 * bv, "exp_avg_sq " + what) <= 1.0
        assert int(upd.step_count) == t
        s, want = upd.sums.tolist(), pb.ref["stats"]
        for k in range(4):
            assert math.isclose(s[k], want[k], rel_tol=1e-4, abs_tol=1e-6), (what, k, s, want.tolist())


def _snapshot(upd):
    return [p.detach().clone() for p in upd.params] + [upd.exp_avg.clone(), upd.exp_avg_sq.clone(),
                                                       upd.step_count.clone(), upd.sums.clone()]


@pytest.mark.gpu
@pytest.mark.parametrize("n_ctas", [0, 49])
def test_epoch_state_carries_across_launches_bit_exact(n_ctas):
    """(d) 12 updates in one run_epoch, 12 launches of one update, and splits 5 + 7 and 1 + 0 + 11 (an empty launch is
    a no-op) give identical parameters, moments, step counter and statistics; so do splits with the learning rate
    decayed between launches, against single-update launches that change it at the same point."""
    dev = torch.device("cuda")
    pb = problem("B512")
    obs, act, old, adv, ret = _data(pb, dev)
    g = torch.Generator(device=dev).manual_seed(5)
    idx = torch.randint(0, pb.obs.shape[0], (12, pb.B), device=dev, generator=g)

    def run(splits, decay_after=()):
        upd = _updater(pb, dev)
        lo = 0
        for k, n in enumerate(splits):
            upd.run_epoch(obs, idx[lo:lo + n], act, old, adv, ret, n_ctas=n_ctas)
            lo += n
            if k in decay_after:
                upd.lr.mul_(0.99)
        upd.check_epoch()
        assert lo == 12
        return _snapshot(upd)

    def same(a, b):
        return all(torch.equal(x, y) for x, y in zip(a, b))

    one = run([12])
    assert int(one[10]) == 12
    assert same(one, run([1] * 12))
    assert same(one, run([5, 7]))
    assert same(one, run([1, 0, 11]))
    assert not same(one, run([5, 7], decay_after={0}))                  # the decay is visible...
    assert same(run([5, 7], decay_after={0}), run([1] * 12, decay_after={4}))
    assert same(run([1, 0, 11], decay_after={1}), run([1] * 12, decay_after={0}))


@pytest.mark.gpu
def test_epoch_kernel_free_running_tracks_float64():
    """(e) 3 launches x 20 updates from the dyadic start with the learning rate decayed between launches as train_ppo
    does, against 60 steps of loss_and_grads_f64 + clip_adam_f64: the float32 trajectory stays within one learning-rate
    step (3e-4) of the float64 one.  Measured on a B200: 1.2e-4."""
    dev = torch.device("cuda")
    pb = problem("B512")
    hp = pb.hp
    obs, act, old, adv, ret = _data(pb, dev)
    rng = np.random.default_rng(9)
    idx = rng.integers(0, pb.obs.shape[0], size=(3, 20, pb.B))
    upd = _updater(pb, dev)
    p, m, v = pb.p0, np.zeros(N_PARAMS), np.zeros(N_PARAMS)
    t = 0
    for launch in range(3):
        lr = float(upd.lr)
        upd.run_epoch(obs, torch.as_tensor(idx[launch]).to(dev), act, old, adv, ret)
        for u in range(20):
            t += 1
            i = idx[launch, u]
            g = loss_and_grads_f64(p, pb.obs[i], pb.act[i], pb.old[i], pb.adv[i], pb.ret[i], hp)["grad"]
            p, m, v = clip_adam_f64(p, g, m, v, t, lr, hp)
        upd.lr.mul_(0.99)
    upd.check_epoch()
    assert int(upd.step_count) == 60
    assert _worst(_flat_params(upd) - p, np.full(N_PARAMS, 3e-4), "free-running parameters after 60 updates") <= 1.0
    assert np.abs(p - pb.p0).max() > 3e-3                                # the parameters did move
