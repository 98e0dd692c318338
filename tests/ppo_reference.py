"""Float64 restatement of one fused PPO minibatch update, for tests of csrc/ppo_update.cuh and csrc/ppo_epoch.cuh.

``loss_and_grads_f64`` evaluates train_ppo.update_step's loss (ratio, per-minibatch advantage normalisation with the
unbiased std clamped at 1e-5, torch.max / clamp surrogate, 0.5 * MSE, entropy bonus) on a float64 copy of the network
and backpropagates it; ``clip_adam_f64`` is clip_grad_norm_ followed by one torch.optim.Adam step, written out.

A float64 reference can only be compared tightly with a float32 kernel when both take the same discrete decisions.
``dyadic_problem`` builds networks and observations whose first layer is exact in float32 in any summation order (so
every ReLU mask is the same everywhere), and ``old_logp_with_margin`` stale log-probabilities whose ratios stay clear
of the clip boundaries.
"""
from __future__ import annotations

import numpy as np
import torch

from ppo_car_b200.train_ppo import ActorCritic

N_IN, N_HIDDEN, N_ACT = 18, 256, 9
# the kernels' flat parameter layout: W1a, b1a, W2a, b2a, W1c, b1c, W2c, b2c
SHAPES = [(N_HIDDEN, N_IN), (N_HIDDEN,), (N_ACT, N_HIDDEN), (N_ACT,), (N_HIDDEN, N_IN), (N_HIDDEN,), (1, N_HIDDEN), (1,)]
N_PARAMS = sum(int(np.prod(s)) for s in SHAPES)                 # 12,298
HP = dict(clip_ratio=0.2, vf_coef=0.5, ent_coef=0.001, max_grad_norm=1.0, betas=(0.9, 0.999), eps=1e-5)


def hparams(**changes) -> dict:
    """train_ppo's defaults with ``changes`` applied."""
    hp = dict(HP)
    hp.update(changes)
    return hp


def as_float32_values(hp: dict) -> dict:
    """The hyperparameters as the kernels see them (each rounded to float32 once), as Python floats."""
    f = lambda x: float(np.float32(x))
    return {k: (tuple(f(b) for b in v) if isinstance(v, tuple) else f(v)) for k, v in hp.items()}


def _net_params(net):
    return [net.actor[0].weight, net.actor[0].bias, net.actor[2].weight, net.actor[2].bias,
            net.critic[0].weight, net.critic[0].bias, net.critic[2].weight, net.critic[2].bias]


def flatten(tensors) -> np.ndarray:
    """8 parameter-shaped arrays -> one float64 vector in the kernels' layout."""
    return np.concatenate([np.asarray(torch.as_tensor(t).detach().cpu(), np.float64).reshape(-1) for t in tensors])


def unflatten(flat) -> list:
    """Inverse of :func:`flatten`: float64 numpy arrays of the 8 parameter shapes."""
    flat = np.asarray(flat, np.float64)
    assert flat.shape == (N_PARAMS,)
    out, off = [], 0
    for s in SHAPES:
        n = int(np.prod(s))
        out.append(flat[off:off + n].reshape(s))
        off += n
    return out


def net_f64(state) -> ActorCritic:
    """A float64 CPU ActorCritic(18, 9) holding ``state`` (8 arrays in the kernels' order, or the flat vector)."""
    if not isinstance(state, (list, tuple)):
        state = unflatten(state)
    net = ActorCritic(N_IN, N_ACT).double()
    with torch.no_grad():
        for p, s in zip(_net_params(net), state):
            p.copy_(torch.as_tensor(np.asarray(torch.as_tensor(s).detach().cpu(), np.float64)).reshape(p.shape))
    return net


def new_logp_f64(state, obs, act) -> np.ndarray:
    """float64 log pi(act | obs) for every row."""
    net = net_f64(state)
    with torch.no_grad():
        _, logp, _, _ = net.act(torch.as_tensor(np.asarray(obs, np.float64)), torch.as_tensor(np.asarray(act)).long())
    return logp.numpy()


def loss_and_grads_f64(state, obs, act, old_logp, adv, ret, hp: dict) -> dict:
    """train_ppo.update_step's loss on ONE minibatch (rows already gathered: obs [B, 18], the rest [B]) in float64.

    Returns ``grad`` (the 12,298 gradients in the kernels' layout), ``stats`` (policy loss, value loss, entropy, total:
    what the kernels add to ``sums``), ``ratio`` [B] and the first-layer pre-activations ``pre_a`` / ``pre_c`` [B, 256].
    """
    net = net_f64(state)
    obs = torch.as_tensor(np.asarray(obs, np.float64))
    act = torch.as_tensor(np.asarray(act)).long()
    old_logp, adv, ret = (torch.as_tensor(np.asarray(a, np.float64)) for a in (old_logp, adv, ret))
    _, new_logp, ent, new_val = net.act(obs, act)
    ratio = torch.exp(new_logp - old_logp)
    a = (adv - adv.mean()) / torch.clamp(adv.std(), min=1e-5)
    clip = hp["clip_ratio"]
    pol = torch.max(-a * ratio, -a * torch.clamp(ratio, 1 - clip, 1 + clip)).mean()
    vl = 0.5 * ((new_val.view(-1) - ret) ** 2).mean()
    e = ent.mean()
    loss = pol + hp["vf_coef"] * vl - hp["ent_coef"] * e
    net.zero_grad()
    loss.backward()
    with torch.no_grad():
        pre_a = obs @ net.actor[0].weight.T + net.actor[0].bias
        pre_c = obs @ net.critic[0].weight.T + net.critic[0].bias
    return dict(grad=flatten([p.grad for p in _net_params(net)]),
                stats=np.array([float(x.detach()) for x in (pol, vl, e, loss)]),
                ratio=ratio.detach().numpy(), pre_a=pre_a.numpy(), pre_c=pre_c.numpy())


def clip_coef_f64(grads, max_grad_norm: float) -> float:
    """torch.nn.utils.clip_grad_norm_'s factor: max_norm / (norm + 1e-6), capped at 1."""
    norm = float(np.sqrt(np.sum(np.square(np.asarray(grads, np.float64)))))
    return min(max_grad_norm / (norm + 1e-6), 1.0)


def clip_adam_f64(params, grads, m, v, t: int, lr: float, hp: dict):
    """clip_grad_norm_(max_grad_norm) then Adam step number ``t`` (bias corrections 1 - beta^t, eps added to
    sqrt(v_hat)), everything flat float64.  Returns (new params, new m, new v)."""
    p, g, m, v = (np.asarray(x, np.float64) for x in (params, grads, m, v))
    b1, b2 = hp["betas"]
    g = g * clip_coef_f64(g, hp["max_grad_norm"])
    m = b1 * m + (1.0 - b1) * g
    v = b2 * v + (1.0 - b2) * g * g
    bc1, bc2 = 1.0 - b1 ** t, 1.0 - b2 ** t
    p = p - (lr / bc1) * m / (np.sqrt(v) / np.sqrt(bc2) + hp["eps"])
    return p, m, v


# ---- data whose float32 first layer is exact ------------------------------------------------------------------------
def dyadic_problem(rows: int, seed: int = 0, zero_pre: bool = False, logit_scale: float = 1.0, adv_const=None):
    """A network state and ``rows`` samples for the update kernels, all float32 numpy arrays.

    Observations are k/64 (k in 0..64), first-layer weights m/256 (|m| <= 64) and first-layer biases odd multiples of
    2^-15 (|b| < 1/4).  Every partial sum of a pre-activation is then an integer multiple of 2^-15 below 5, exact in
    float32 whatever the summation order, and the total is an odd multiple of 2^-15: never 0.  ``zero_pre`` sets both
    first-layer biases to 0 and every fourth observation row to zeros, so those pre-activations are exactly 0 (where
    torch's ReLU has subgradient 0).  The output layers are ordinary normal draws; ``logit_scale`` multiplies the
    actor's (W2a and b2a).  Advantages are multiples of 2^-8 below 16 in magnitude, so their minibatch sums are exact in
    float32 and a minibatch of one repeated row has normalised advantages of exactly 0, as in float64.  Returns (state [8 arrays, kernel order], obs, act, adv, ret).
    """
    rng = np.random.default_rng(seed)
    f32 = np.float32

    def w1():
        return (rng.integers(-64, 65, size=(N_HIDDEN, N_IN)) / 256.0).astype(f32)

    def b1():
        if zero_pre:
            return np.zeros(N_HIDDEN, f32)
        return ((2 * rng.integers(-4096, 4096, size=N_HIDDEN) + 1) / 32768.0).astype(f32)

    w1a, b1a, w1c, b1c = w1(), b1(), w1(), b1()
    w2a = (rng.standard_normal((N_ACT, N_HIDDEN)) * 0.05 * logit_scale).astype(f32)
    b2a = (rng.standard_normal(N_ACT) * 0.1 * logit_scale).astype(f32)
    w2c = (rng.standard_normal((1, N_HIDDEN)) * 0.05).astype(f32)
    b2c = (rng.standard_normal(1) * 0.1).astype(f32)
    obs = (rng.integers(0, 65, size=(rows, N_IN)) / 64.0).astype(f32)
    if zero_pre:
        obs[::4] = 0.0
    act = rng.integers(0, N_ACT, size=rows).astype(f32)
    adv = np.round((rng.standard_normal(rows) * 2.0 + 0.5) * 256.0) / 256.0 if adv_const is None else np.full(rows, adv_const)
    adv = adv.astype(f32)
    ret = rng.standard_normal(rows).astype(f32)
    return [w1a, b1a, w2a, b2a, w1c, b1c, w2c, b2c], obs, act, adv, ret


def old_logp_with_margin(new_logp64, inside_frac: float, clip_ratio: float = 0.2, margin: float = 2e-3, seed: int = 0):
    """float32 stale log-probabilities for which every float64 ratio exp(new - old) lies at least ``margin`` (>= 1e-3)
    away from 1 - clip_ratio and 1 + clip_ratio: a fraction ``inside_frac`` inside the clip range, the rest outside,
    alternately below and above it."""
    assert margin >= 1e-3
    new = np.asarray(new_logp64, np.float64)
    n = new.shape[0]
    rng = np.random.default_rng(seed)
    lo, hi = 1.0 - clip_ratio, 1.0 + clip_ratio
    inside = rng.permutation(n) < int(round(inside_frac * n))
    below = (np.arange(n) % 2) == 0
    r = np.where(inside, rng.uniform(lo + 2 * margin, hi - 2 * margin, n),
                 np.where(below, rng.uniform(0.5 * lo, lo - 2 * margin, n), rng.uniform(hi + 2 * margin, 1.5 * hi, n)))
    old = (new - np.log(r)).astype(np.float32)
    got = np.exp(new - old.astype(np.float64))                  # the ratios after rounding old to float32
    assert np.all(np.minimum(np.abs(got - lo), np.abs(got - hi)) >= margin)
    assert np.array_equal((got > lo) & (got < hi), inside)
    return old
