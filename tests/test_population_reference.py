"""The population kernels against float64 and Philox references, on the edges the single-policy kernels are tested at.

``k_ppo_epoch_pop`` (one 8-CTA cluster per member, gradient reduced through distributed shared memory) keeps its own
copy of ``k_ppo_epoch``'s loss, clip and Adam arithmetic, and the member-batched rollouts ``k_policy_rollout_warp<true>``
and ``k_policy_rollout_tc3<U, TAB, true>`` are separate instantiations of the single-policy kernels.  The references
and bounds are the ones of tests/test_ppo_update_reference.py and tests/test_fused_rollout_reference.py, unchanged:

1. Every case of the update edge matrix (``CASES``) and three batches that exercise the per-CTA sample split, as members
   of shared launches (one per B), each member with its own case's loss coefficients.  The gradient is read through the
   linear-Adam probe (lr = 1e9, eps = 1e6, m = v = 0, t = 1: the step is -lr c g / (c |g| + eps)), once unclipped
   (c = 1) and once with max_grad_norm = 0.25 |g| in the same launch, which checks the cluster's global norm.
2. Clip + Adam from teacher-forced moments with the members at different steps t and learning rates, within twice
   ``adam_error_bound``: the only check that every member reads its own step counter.
3. More members than clusters fit on the GPU at once (the launch runs in waves): the probe for every member, and a
   12-update epoch whose every member is bit-identical to the same member launched alone.
4. State carried across launches, with the learning rate decayed between them by ``Population.decay_lr``.
5. The member-batched rollouts on every instantiation: bit for bit against single-member runs, the uniforms against
   Philox, values / log-probabilities / actions against float64, and every row against a replay of the actions.
6. The minibatch schedule: member p gets exactly the minibatch rows of ``train_ppo --seed seeds[p]``.

Tests print the worst error they saw as a fraction of its bound (pytest -s), and the worst per part when the module
ends.
"""
import collections
import ctypes as C
import functools
import math
import re
from types import SimpleNamespace

import numpy as np
import pytest
import torch

import ppo_car_b200
from ppo_car_b200 import _lib
from ppo_car_b200 import population as popmod
from ppo_car_b200.policy import WARP_ROLLOUT_MAX_ENVS
from ppo_car_b200.population import Population, PopulationPPOUpdate, population_rollout
from ppo_car_b200.track import load_track
from tests import test_fused_rollout_reference as rollout_ref
from tests.ppo_reference import (N_PARAMS, _net_params, as_float32_values, clip_adam_f64, clip_coef_f64, dyadic_problem,
                                 flatten, hparams, loss_and_grads_f64, new_logp_f64, old_logp_with_margin)
from tests.test_fused_rollout_reference import (STEP0, check_network, check_replay, fused, instantiation, make_env,
                                                make_policy, rollout_uniforms, start_state, track_layout, track_path)
from tests.test_population import SEEDS, _flat, _snap
from tests.test_ppo_update_reference import CASES, _worst, adam_error_bound, grad_tol, problem, ulp32

gpu = pytest.mark.gpu
PART_WORST = collections.defaultdict(float)            # part -> worst error / bound over the module


def _note(part, frac):
    PART_WORST[part] = max(PART_WORST[part], frac)
    return frac


@pytest.fixture(scope="module", autouse=True)
def report_worst_per_part():
    yield
    for part, frac in sorted(PART_WORST.items()):
        print(f"worst {part}: {frac:.3g} of its bound")


@pytest.fixture(scope="module")
def tracks(tmp_path_factory):
    d = str(tmp_path_factory.mktemp("tracks"))
    return functools.lru_cache(maxsize=None)(lambda name: track_path(name, d))


# ---- the update's launches -----------------------------------------------------------------------------------------
SPLIT_B = (9, 65, 1023)          # batches chosen for the per-CTA sample split (test_cluster_split_of_the_split_batches)
DEFAULT_BETAS = (0.9, 0.999)


@functools.lru_cache(maxsize=None)
def split_problem(B):
    """A default-options dyadic problem at batch B, in the form of test_ppo_update_reference.problem."""
    rows, seed = max(2 * B, 64), 1000 + B
    hp = as_float32_values(hparams())
    state, obs, act, adv, ret = dyadic_problem(rows, seed=seed)
    old = old_logp_with_margin(new_logp_f64(state, obs, act), 0.5, hp["clip_ratio"], seed=seed)
    idx = np.random.default_rng(seed).choice(rows, B, replace=False)
    ref = loss_and_grads_f64(state, obs[idx], act[idx], old[idx], adv[idx], ret[idx], hp)
    return SimpleNamespace(name=f"split_B{B}", B=B, hp=hp, tol_scale=1.0, state=state, obs=obs, act=act, old=old,
                           adv=adv, ret=ret, idx=idx, ref=ref, p0=flatten(state))


def get_problem(name):
    return problem(name) if name in CASES else split_problem(int(name[len("split_B"):]))


def update_launches():
    """(label, case names, betas) of part 1: the CASES grouped by B with one launch per B, the hparams case in a launch
    of its own with its betas, and one launch per split batch."""
    by_b = {}
    for name, c in CASES.items():
        if name != "hparams":
            by_b.setdefault(c["B"], []).append(name)
    out = [(f"B{B}", names, DEFAULT_BETAS) for B, names in sorted(by_b.items())]
    out.append(("hparams", ["hparams"], problem("hparams").hp["betas"]))
    return out + [(f"split_B{B}", [f"split_B{B}"], DEFAULT_BETAS) for B in SPLIT_B]


UPDATE_LAUNCHES = update_launches()


def epoch_samples():
    """kEpochSamples of csrc/ppo_epoch.cuh: the chunk of samples a CTA stages at a time."""
    with open(_lib.SOURCES[0].replace("carenv_kernels.cu", "ppo_epoch.cuh")) as f:
        return int(re.search(r"constexpr int kEpochSamples = (\d+);", f.read()).group(1))


def cluster_split(B, cluster, chunk):
    """k_ppo_epoch_pop's split of a minibatch over the cluster: S = ceil(B / cluster) samples per CTA, CTA r takes
    samples [r S, r S + S) clipped to B, in max(1, ceil(count / chunk)) chunks.  Returns (S, counts, chunks)."""
    S = -(-B // cluster)
    counts = [max(0, min(S, B - r * S)) for r in range(cluster)]
    return S, counts, [max(1, -(-k // chunk)) for k in counts]


def test_cluster_split_of_the_split_batches():
    """The split batches reach the cluster paths they are there for; the update launches cover every CASES entry once."""
    cluster, chunk = _lib.lib().carenv_ppo_epoch_pop_cluster_size(), epoch_samples()
    assert (cluster, chunk) == (8, 8)
    S, counts, chunks = cluster_split(9, cluster, chunk)        # rank 4 has one sample, ranks 5-7 none
    assert S == 2 and counts == [2, 2, 2, 2, 1, 0, 0, 0]
    S, counts, chunks = cluster_split(65, cluster, chunk)       # a second chunk of one sample, a ragged last rank
    assert S == 9 and counts == [9] * 7 + [2] and chunks == [2] * 7 + [1]
    S, counts, chunks = cluster_split(1023, cluster, chunk)     # 16 full chunks, and 15 + one of 7 on rank 7
    assert S == 128 and counts == [128] * 7 + [127] and chunks == [16] * 8
    names = [n for _, names, _ in UPDATE_LAUNCHES for n in names]
    assert sorted(n for n in names if n in CASES) == sorted(CASES) and len(names) == len(set(names))
    for label, names, _ in UPDATE_LAUNCHES:
        assert len({get_problem(n).B for n in names}) == 1, label


def stage(problems, dev, lr, max_grad_norm, extra=None):
    """A Population whose member p holds problems[p]'s network, its loss coefficients, lr[p], max_grad_norm[p] and
    the hyperparameters extra[p]; member p's samples sit at offset offs[p] of one set of flat arrays.
    Returns (pop, [obs, act, old_logp, adv, ret], offs)."""
    hp = [dict(clip_ratio=pb.hp["clip_ratio"], vf_coef=pb.hp["vf_coef"], ent_coef=pb.hp["ent_coef"], learning_rate=l,
               max_grad_norm=m, **(extra[p] if extra else {}))
          for p, (pb, l, m) in enumerate(zip(problems, lr, max_grad_norm))]
    pop = Population(list(range(len(problems))), 1, hp, dev)
    with torch.no_grad():
        for p, pb in enumerate(problems):
            for t, a in zip(pop.params, pb.state):
                t[p].copy_(torch.as_tensor(a).reshape(t[p].shape))
    cat = lambda key: torch.as_tensor(np.concatenate([getattr(pb, key) for pb in problems])).float().contiguous().to(dev)
    offs = np.cumsum([0] + [pb.obs.shape[0] for pb in problems])[:-1]
    return pop, [cat(k) for k in ("obs", "act", "old", "adv", "ret")], offs


def one_update_idx(problems, offs, dev):
    """int64 [P, 1, B]: each problem's own minibatch, at its offset."""
    return torch.as_tensor(np.stack([pb.idx + o for pb, o in zip(problems, offs)])[:, None, :]).to(dev).contiguous()


PROBE_LR, PROBE_EPS = 1e9, 1e6


def probe_max_norm(pb, clipped):
    return float(np.float32(0.25 * np.linalg.norm(pb.ref["grad"]))) if clipped else 1e30


def check_probe(pop, p, pb, max_norm, part, what):
    """Member p after one probe update: its gradient against float64 through test_epoch_kernel_gradients_through_linear_
    adam_probe's expected step and bound, its loss statistics and its step counter."""
    g64 = pb.ref["grad"]
    coef = clip_coef_f64(g64, max_norm)
    assert (coef < 0.3) if max_norm < 1e29 else (coef == 1.0)          # clipping active / inactive as intended
    dp = _flat(pop, p) - pb.p0
    want = -PROBE_LR * coef * g64 / (coef * np.abs(g64) + PROBE_EPS)
    tol = PROBE_LR / PROBE_EPS * coef * grad_tol(g64, pb.tol_scale) + ulp32(pb.p0 + dp)
    assert _note(part, _worst(dp - want, tol, f"population gradient probe [{what}, clip={coef:.3g}]")) <= 1.0, what
    s, ref = pop.sums[p].tolist(), pb.ref["stats"]
    for k in range(4):
        assert math.isclose(s[k], ref[k], rel_tol=1e-4, abs_tol=1e-6), (what, k, s, ref.tolist())
    assert int(pop.step_count[p]) == 1, what


# ---- 1. the edge matrix, per member, in shared launches ------------------------------------------------------------
@gpu
@pytest.mark.parametrize("label, names, betas", UPDATE_LAUNCHES, ids=[u[0] for u in UPDATE_LAUNCHES])
def test_update_edge_matrix_per_member(label, names, betas):
    """One launch per batch size; every problem is staged twice, unclipped and clipped, so a launch has 2 to 12
    members with different loss coefficients and clip norms."""
    dev = torch.device("cuda", 0)
    members = [(get_problem(n), clipped) for n in names for clipped in (False, True)]
    problems = [pb for pb, _ in members]
    mgn = [probe_max_norm(pb, clipped) for pb, clipped in members]
    pop, data, offs = stage(problems, dev, [PROBE_LR] * len(members), mgn)
    upd = PopulationPPOUpdate(pop, problems[0].B, betas=betas, eps=PROBE_EPS)
    upd.launch(data[0], one_update_idx(problems, offs, dev), *data[1:])
    torch.cuda.synchronize()
    for p, (pb, clipped) in enumerate(members):
        check_probe(pop, p, pb, mgn[p], "1 update edge matrix", f"{label}: {pb.name}, member {p}")


# ---- 2. Adam from teacher-forced state, members at different steps --------------------------------------------------
ADAM_MEMBERS = [(t, lr) for t in (1, 2, 10, 1000, 100000) for lr in (3e-4, 3e-4 * 0.99 ** 150)]


def teacher_forced_moments(g64, t):
    """exp_avg and exp_avg_sq as test_clip_adam_with_teacher_forced_state builds them (float32 values, as float64)."""
    rng = np.random.default_rng(t)
    scale = float(np.sqrt(np.mean(g64 * g64)))
    m0 = (rng.standard_normal(N_PARAMS) * scale).astype(np.float32)
    v0 = (m0.astype(np.float64) ** 2 * rng.uniform(0.5, 2.0, N_PARAMS) + 1e-3 * scale * scale).astype(np.float32)
    return m0.astype(np.float64), v0.astype(np.float64)


@gpu
@pytest.mark.parametrize("case", ["B512", "hparams"])
def test_adam_with_teacher_forced_state_members_at_different_steps(case):
    """One launch of 10 members at t in {1, 2, 10, 1000, 100000} x two learning rates, each from its own moments and
    step counter, against clip_adam_f64 within twice adam_error_bound; also step_count == t and the sums."""
    dev = torch.device("cuda", 0)
    pb = problem(case)
    hp = pb.hp
    g64 = pb.ref["grad"]
    coef = clip_coef_f64(g64, hp["max_grad_norm"])
    lrs = [float(np.float32(lr)) for _, lr in ADAM_MEMBERS]
    pop, data, offs = stage([pb] * len(ADAM_MEMBERS), dev, lrs, [hp["max_grad_norm"]] * len(ADAM_MEMBERS))
    refs = []
    for p, (t, _) in enumerate(ADAM_MEMBERS):
        m0, v0 = teacher_forced_moments(g64, t)
        pop.exp_avg[p].copy_(torch.as_tensor(m0, dtype=torch.float32))
        pop.exp_avg_sq[p].copy_(torch.as_tensor(v0, dtype=torch.float32))
        pop.step_count[p] = t - 1
        refs.append((m0, v0))
    upd = PopulationPPOUpdate(pop, pb.B, betas=hp["betas"], eps=hp["eps"])
    upd.launch(data[0], one_update_idx([pb] * len(ADAM_MEMBERS), offs, dev), *data[1:])
    torch.cuda.synchronize()
    part = "2 teacher-forced Adam"
    for p, ((t, _), lr, (m0, v0)) in enumerate(zip(ADAM_MEMBERS, lrs, refs)):
        p64, m64, v64 = clip_adam_f64(pb.p0, g64, m0, v0, t, lr, hp)
        bp, bm, bv = adam_error_bound(pb, g64, m0, v0, m64, v64, p64 - pb.p0, coef, t, lr)
        what = f"[{case}, member {p}, t={t}, lr={lr:.3g}]"
        dp = _flat(pop, p) - pb.p0
        assert _note(part, _worst(dp - (p64 - pb.p0), 2 * (bp + ulp32(pb.p0 + dp)), "Adam step " + what)) <= 1.0
        m, v = pop.exp_avg[p].double().cpu().numpy(), pop.exp_avg_sq[p].double().cpu().numpy()
        assert _note(part, _worst(m - m64, 2 * bm, "exp_avg " + what)) <= 1.0
        assert _note(part, _worst(v - v64, 2 * bv, "exp_avg_sq " + what)) <= 1.0
        assert int(pop.step_count[p]) == t, what
        s, want = pop.sums[p].tolist(), pb.ref["stats"]
        for k in range(4):
            assert math.isclose(s[k], want[k], rel_tol=1e-4, abs_tol=1e-6), (what, k, s, want.tolist())


# ---- 3. more members than resident clusters -------------------------------------------------------------------------
B512_CASES = [name for name, c in CASES.items() if c["B"] == 512]


def resident_clusters():
    n = C.c_int(0)
    _lib.check(_lib.lib().carenv_ppo_epoch_pop_resident_clusters(C.byref(n)), "carenv_ppo_epoch_pop_resident_clusters")
    return n.value


@gpu
def test_more_members_than_resident_clusters():
    """P = 2R + 3 members (R clusters fit on the GPU at once, so the launch runs in at least three waves) cycling over
    the B = 512 cases: the probe of part 1 for every member, then a 12-update epoch in which every member (its own
    learning rate, clip norm, clip ratio and loss coefficients) ends bit-identical to the same member launched alone."""
    dev = torch.device("cuda", 0)
    R = resident_clusters()
    P = 2 * R + 3
    print(f"\n{R} resident clusters: {P} members")
    problems = [problem(B512_CASES[k % len(B512_CASES)]) for k in range(P)]
    clipped = [(k // len(B512_CASES)) % 2 == 1 for k in range(P)]
    mgn = [probe_max_norm(pb, c) for pb, c in zip(problems, clipped)]
    pop, data, offs = stage(problems, dev, [PROBE_LR] * P, mgn)
    PopulationPPOUpdate(pop, 512, eps=PROBE_EPS).launch(data[0], one_update_idx(problems, offs, dev), *data[1:])
    torch.cuda.synchronize()
    for p, pb in enumerate(problems):
        check_probe(pop, p, pb, mgn[p], "3 waves probe", f"{pb.name}, member {p} of {P}")

    U = 12
    lrs = [1e-4 * (1 + k % 7) for k in range(P)]
    norms = [(1.0, 0.3, 2.0, 0.5, 5.0)[k % 5] for k in range(P)]
    idx = [np.random.default_rng(500 + k).integers(0, pb.obs.shape[0], (U, 512)) for k, pb in enumerate(problems)]

    def run(members):
        probs = [problems[k] for k in members]
        pop, data, offs = stage(probs, dev, [lrs[k] for k in members], [norms[k] for k in members])
        ix = torch.as_tensor(np.stack([idx[k] + o for k, o in zip(members, offs)])).to(dev).contiguous()
        PopulationPPOUpdate(pop, 512).launch(data[0], ix, *data[1:])
        torch.cuda.synchronize()
        return pop

    together = run(list(range(P)))
    for k in range(P):
        alone = run([k])
        for a, b in zip(_snap(together, k), _snap(alone, 0)):
            assert torch.equal(a, b), k
        assert int(together.step_count[k]) == U


# ---- 4. state across launches with the learning rate decayed between them ---------------------------------------------
@gpu
def test_state_carries_across_launches_with_decay_bit_exact():
    """Three members with learning_rate_decay 0.99, 0.9 and 1.0: 12 updates in one launch, 12 launches of one update,
    5 + 7 and 1 + 0 + 11 (an empty launch is a no-op) give identical parameters, moments, steps and sums; decay_lr()
    between launches changes the members it decays (not the one at 1.0), and equals single-update launches that decay
    at the same update."""
    dev = torch.device("cuda", 0)
    problems = [problem(n) for n in ("B512", "ratios_inside", "ratios_outside")]
    decays = [0.99, 0.9, 1.0]
    gen = torch.Generator(device=dev).manual_seed(5)
    U = 12
    idx_rows = torch.randint(0, problems[0].obs.shape[0], (len(problems), U, 512), device=dev, generator=gen)

    def run(splits, decay_after=()):
        pop, data, offs = stage(problems, dev, [3e-4] * 3, [pb.hp["max_grad_norm"] for pb in problems],
                                [{"learning_rate_decay": d} for d in decays])
        idx = (idx_rows + torch.as_tensor(offs, device=dev).view(-1, 1, 1)).contiguous()
        upd = PopulationPPOUpdate(pop, 512)
        lo = 0
        for k, n in enumerate(splits):
            upd.launch(data[0], idx[:, lo:lo + n].contiguous(), *data[1:])
            lo += n
            if k in decay_after:
                pop.decay_lr()
        torch.cuda.synchronize()
        assert lo == U
        return [_snap(pop, p) for p in range(3)]

    def same(a, b, members=range(3)):
        return all(torch.equal(x, y) for p in members for x, y in zip(a[p], b[p]))

    one = run([U])
    assert all(int(s[-1]) == U for s in one)
    assert same(one, run([1] * U))
    assert same(one, run([5, 7]))
    assert same(one, run([1, 0, 11]))
    decayed = run([5, 7], decay_after={0})
    assert not same(one, decayed, [0]) and not same(one, decayed, [1])   # the decay is visible...
    assert same(one, decayed, [2])                                        # ... except at learning_rate_decay 1.0
    assert same(decayed, run([1] * U, decay_after={4}))
    assert same(run([1, 0, 11], decay_after={1}), run([1] * U, decay_after={0}))


# ---- 5. member-batched rollouts on every instantiation ------------------------------------------------------------------
POP_MATRIX = [   # track, env options, environments per member
    ("ring42_42", {}, 24),                       # tc3 <2, false>: 84 segments take the tensor cores at any n
    ("ring64_64", {}, 300),                      # tc3 <4, false>
    ("big_track", {}, 4097),                     # tc3 <4, true>
    ("big_track", {"tab": -1}, 4097),            # tc3 <4, false>
    ("big_track", {"max_unroll": 2}, 4097),      # tc3 <2, true>
    ("big_track", {"force_generic": 1}, 4097),   # tc3 <1, false>
    ("ring10_6", {}, 4097),                      # tc3 <2, true> (another pair count)
    ("ring16_16", {}, 257),                      # warp, 32 segments
    ("near_wall", {}, 24),                       # warp, every step terminates
    ("ring7_5", {}, 24),                         # warp, no unroll
]
POP_IDS = ["-".join([t] + [f"{k}{v}" for k, v in o.items()] + [f"n{n}"]) for t, o, n in POP_MATRIX]
POP_REQUIRED = {("tc3", 4, True), ("tc3", 4, False), ("tc3", 2, True), ("tc3", 2, False), ("tc3", 1, False), ("warp",)}
ROLL_T = 40


def pop_kernel(path, n):
    """The kernel population_rollout launches for a track and n environments per member, by its own rule."""
    warp = popmod.use_warp_kernel(SimpleNamespace(track=load_track(path)), n)
    assert warp == (n <= WARP_ROLLOUT_MAX_ENVS and track_layout(path).n_seg <= 32)
    return "warp" if warp else "tc3"


def test_pop_matrix_reaches_every_member_instantiation(tracks):
    reached = {}
    for (t, opts, n), name in zip(POP_MATRIX, POP_IDS):
        inst = instantiation(pop_kernel(tracks(t), n), track_layout(tracks(t)), opts)
        reached.setdefault(inst, []).append(name)
    assert set(reached) == POP_REQUIRED, POP_REQUIRED ^ set(reached)
    assert instantiation(pop_kernel(tracks("ring42_42"), 24), track_layout(tracks("ring42_42")), {}) == ("tc3", 2, False)
    assert pop_kernel(tracks("ring16_16"), 257) == "warp" and pop_kernel(tracks("big_track"), 4097) == "tc3"


def pop_rollout(path, opts, nets, seeds, n, T, step0):
    """One population_rollout of len(seeds) members (member p with nets[p]'s weights) from reset, with uniforms and
    bootstrap values.  Returns (env, [cur_obs, cur_term, cur_trunc], rows)."""
    dev = torch.device("cuda", 0)
    P = len(seeds)
    pop = Population(seeds, n, None, dev)
    with torch.no_grad():
        for p, net in enumerate(nets):
            for t, w in zip(pop.params, _net_params(net)):
                t[p].copy_(w.reshape(t[p].shape))
    env = make_env(path, P * n, opts)
    state = start_state(env)
    buf = ppo_car_b200.Buffer((18,), T, P * n, dev)
    lv = torch.full((P * n,), float("nan"), device=dev)
    u = torch.full((T, P * n), float("nan"), device=dev)
    population_rollout(env, pop, buf, *state, step0=step0, last_val=lv, u_dbg=u)
    torch.cuda.synchronize()
    return env, state, SimpleNamespace(obs=buf.obs_buf, act=buf.act_buf, rew=buf.rew_buf, val=buf.val_buf,
                                       term=buf.term_buf, trunc=buf.trunc_buf, logp=buf.logprob_buf, u=u, last_val=lv)


def member_rows(r, c):
    return SimpleNamespace(**{k: v[c] if k == "last_val" else v[:, c] for k, v in vars(r).items()})


def check_member_references(kernel, r, state, nets, seeds, n, T, step0, tag, monkeypatch):
    """Every member's uniforms against Philox (its seed, env_offset 0) and its rows against float64 with its weights."""
    monkeypatch.setattr(rollout_ref, "WORST", collections.defaultdict(float))    # check_network's records, this test
    for p, seed in enumerate(seeds):
        c = slice(p * n, (p + 1) * n)
        got = np.ascontiguousarray(r.u[:, c].cpu().numpy())
        want = rollout_uniforms(seed, 0, n, step0, T)
        assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), (p, int((got != want).sum()))
        check_network(kernel, nets[p], member_rows(r, c), state[0][c], tag=f"{tag} member {p}")
    for (k, what), frac in rollout_ref.WORST.items():
        _note(f"5 rollout {k} {what}", frac)


@gpu
@pytest.mark.parametrize("track, opts, n", POP_MATRIX, ids=POP_IDS)
def test_member_rollouts_on_every_instantiation(tracks, track, opts, n, monkeypatch):
    """Three members (seeds with non-zero high words), 40 steps from a step0 that crosses 2^32, with last_val: every
    member's columns, bootstrap values and final state bit for bit against the member alone through fused_rollout /
    fused_rollout_warp with the same env options; Philox, float64 and the replay of all P n environments."""
    path = tracks(track)
    kernel = pop_kernel(path, n)
    seeds = SEEDS[1:4]
    nets = [make_policy(seed=20 + p) for p in range(len(seeds))]
    env, state, r = pop_rollout(path, opts, nets, seeds, n, ROLL_T, STEP0)
    for p, seed in enumerate(seeds):
        c = slice(p * n, (p + 1) * n)
        env1 = make_env(path, n, opts)
        s1 = start_state(env1)
        r1 = fused(kernel, env1, nets[p], ROLL_T, STEP0, s1, last_val=True, env_offset=0, seed=seed)
        for k in ("obs", "act", "rew", "val", "term", "trunc", "logp", "u"):
            assert torch.equal(getattr(r, k)[:, c], getattr(r1, k)), (p, k)
        assert torch.equal(r.last_val[c], r1.last_val), (p, "last_val")
        for k, (a, b) in enumerate(zip(state, s1)):
            assert torch.equal(a[c], b), (p, "state", k)
        for k in ("pos", "vel", "ints"):
            assert torch.equal(getattr(env, k)[c], getattr(env1, k)), (p, k)
    check_member_references(kernel, r, state, nets, seeds, n, ROLL_T, STEP0, f"{track} {opts} n={n} {kernel}",
                            monkeypatch)
    check_replay(path, env, [r], state)
    if track == "near_wall":                                         # the start pose is inside the wall
        assert r.term[1:].all()
    else:
        assert len(torch.unique(r.act)) == 9


@gpu
@pytest.mark.parametrize("track, P, n", [("big_track", 300, 1), ("ring42_42", 17, 24)],
                         ids=["warp-P300-n1", "tc3-P17-n24"])
def test_many_members_in_one_rollout_launch(tracks, track, P, n, monkeypatch):
    """300 one-environment members on the warp path and 17 members of 24 on the tensor-core path: every member's
    uniforms against Philox and rows against float64 with its own weights, and the replay of the whole population."""
    path = tracks(track)
    kernel = pop_kernel(path, n)
    assert kernel == ("warp" if n == 1 else "tc3")
    seeds = [(p + 1) * 2 ** 32 + 7 * p + 3 for p in range(P)]
    nets = [make_policy(seed=100 + p) for p in range(P)]
    env, state, r = pop_rollout(path, {}, nets, seeds, n, ROLL_T, STEP0)
    check_member_references(kernel, r, state, nets, seeds, n, ROLL_T, STEP0, f"{track} P={P} n={n} {kernel}",
                            monkeypatch)
    check_replay(path, env, [r], state)


# ---- 6. the minibatch schedule is train_ppo's --------------------------------------------------------------------------
@gpu
def test_minibatch_schedule_is_train_ppos(monkeypatch):
    """train_ppo --fused-rollout --fused-update for seeds 0, 5 and 2^40 + 7, and one population of the same seeds, for
    3 epochs: in every epoch member p's minibatch rows, mapped back to its [T, n] block, are that seed's idx_all, and in
    epoch 1 (before the first update makes the runs differ) the gathered obs, act, logp, adv and ret are equal bit for
    bit."""
    from ppo_car_b200.ppo_update import FusedPPOUpdate
    from ppo_car_b200.train_ppo import parse_args, train

    seeds, n, T, epochs = [0, 5, 2 ** 40 + 7], 24, 64, 3
    argv = ["--track", "big_track", "--n-envs", str(n), "--n-steps", str(T), "--batch-size", "64",
            "--n-epochs", str(epochs)]
    log = []
    run_epoch, launch = FusedPPOUpdate.run_epoch, PopulationPPOUpdate.launch

    def record_run_epoch(self, obs, idx, act, old_logp, adv, ret, *args, **kwargs):
        log.append([t.clone() for t in (idx, obs, act, old_logp, adv, ret)])
        return run_epoch(self, obs, idx, act, old_logp, adv, ret, *args, **kwargs)

    def record_launch(self, obs, idx, act, old_logp, adv, ret):
        log.append([t.clone() for t in (idx, obs, act, old_logp, adv, ret)])
        return launch(self, obs, idx, act, old_logp, adv, ret)

    monkeypatch.setattr(FusedPPOUpdate, "run_epoch", record_run_epoch)
    monkeypatch.setattr(PopulationPPOUpdate, "launch", record_launch)
    single = {}
    for s in seeds:
        log.clear()
        train(parse_args(argv + ["--seed", str(s), "--fused-rollout", "--fused-update"]))
        single[s] = list(log)
    log.clear()
    popmod.train_population(popmod.parse_args(argv + ["--seeds", ",".join(map(str, seeds))]))
    assert len(log) == epochs and all(len(v) == epochs for v in single.values())
    N = len(seeds) * n
    for e in range(epochs):
        idx = log[e][0]
        for p, s in enumerate(seeds):
            rows = idx[p]
            assert torch.equal(rows % N // n, torch.full_like(rows, p)), (e, s)      # member p's own columns
            k = (rows // N) * n + rows % N - p * n
            assert torch.equal(k, single[s][e][0]), (e, s)
            if e == 0:
                for name, a, b in zip(("obs", "act", "logp", "adv", "ret"), log[e][1:], single[s][e][1:]):
                    assert torch.equal(a[rows], b[single[s][e][0]]), (s, name)
