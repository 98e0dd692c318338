"""Time-limit bootstrapping (--bootstrap-truncated): the final-observation slots of every fused rollout kernel, the
critic pass over them (carenv_final_values), the bootstrapping GAE scan (gae_reverse_scan_boot) and the training
paths that use them.

  CPU   the slot bound ceil(T / 1000) by brute force, a float32 numpy port of the bootstrapping scan, flag parsing
  GPU   the scan bit for bit against the port on the three launch paths of gae_reverse_scan; every *_final twin against
        its plain entry point (same bits) and against a replay through VecCarEnv(final_observation=True); the critic
        pass against float64; one epoch of train_ppo / population with the flag on every rollout path
"""
import math
import os

import numpy as np
import pytest
import torch

import ppo_car_b200
from oracle.carenv_port import gae_port
from ppo_car_b200.buffer import TIME_LIMIT, final_slots

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
START_TIMES = [0, 1, 998, 999]              # time_step of the environments at launch: 0..3 truncations in 2001 steps


@pytest.fixture(scope="module")
def track_path():
    return lambda name: ppo_car_b200.builtin_track(name)


@pytest.fixture(scope="module")
def synth_path(tmp_path_factory):
    from tests.synth_tracks import near_wall_track, ring_track

    d = tmp_path_factory.mktemp("bt_tracks")

    def make(name):
        path = str(d / f"{name}.json")
        if not os.path.exists(path):
            if name == "near_wall":
                near_wall_track(path)
            else:                                            # 40 segments: over the warp kernel's 32
                ring_track(path, 24, 16)
        return path
    return make


# ---- CPU -----------------------------------------------------------------------------------------------------------
def test_slot_bound_by_brute_force():
    """An environment that never crashes truncates most often; whatever its starting time step 0..999, in T steps it
    truncates at most ceil(T / 1000) times, and the bound is reached."""
    for T in (1, 999, 1000, 1001, 2000, 2001):
        most = 0
        for t0 in range(TIME_LIMIT):
            t, n = t0, 0
            for _ in range(T):
                t += 1
                if t >= TIME_LIMIT:
                    n, t = n + 1, 0
            most = max(most, n)
        assert most == final_slots(T) == math.ceil(T / TIME_LIMIT), T


def gae_boot_port(rew, val, term, trunc, last_val, last_term, last_trunc, boot, gamma=0.99, gae_lambda=0.95):
    """gae_port's float32 operation order with one substitution: a row whose successor has trunc == 1 and term == 0
    takes nv = boot[t]."""
    f = np.float32
    rew, val, term, trunc, boot = (np.asarray(a, f) for a in (rew, val, term, trunc, boot))
    T = rew.shape[0]
    g, gl, one = f(gamma), f(gamma * gae_lambda), f(1.0)
    adv = np.zeros_like(rew)
    last = np.zeros(rew.shape[1:], f)
    lv, lt, lu = (np.asarray(a, f).reshape(-1) for a in (last_val, last_term, last_trunc))
    for t in range(T - 1, -1, -1):
        nv = lv if t == T - 1 else val[t + 1]
        te = lt if t == T - 1 else term[t + 1]
        tr = lu if t == T - 1 else trunc[t + 1]
        nv = np.where((tr == 1) & (te == 0), boot[t], nv)
        tm, um = one - te, one - tr
        delta = (rew[t] + (g * nv) * tm) - val[t]
        last = delta + ((gl * tm) * um) * last
        adv[t] = last
    return adv, adv + val


def _gae_inputs_np(T, N, seed, trunc_p=0.05):
    r = np.random.default_rng(seed)
    rew = (r.random((T, N)) * 1.4 - 0.3).astype(np.float32)
    val = r.standard_normal((T, N)).astype(np.float32)
    term = (r.random((T, N)) < 0.05).astype(np.float32)
    trunc = (r.random((T, N)) < trunc_p).astype(np.float32)
    both = r.random((T, N)) < 0.01
    term[both] = trunc[both] = 1.0
    lv = r.standard_normal(N).astype(np.float32)
    lt, lu = (r.random(N) < 0.1).astype(np.float32), (r.random(N) < 0.2).astype(np.float32)
    return rew, val, term, trunc, lv, lt, lu


def _boot_for(term, trunc, lt, lu, seed):
    """boot [T, N]: random where the scan must read it, NaN everywhere else."""
    T, N = term.shape
    nxt_te = np.concatenate([term[1:], lt[None]], 0)
    nxt_tr = np.concatenate([trunc[1:], lu[None]], 0)
    need = (nxt_tr == 1) & (nxt_te == 0)
    boot = np.full((T, N), np.nan, np.float32)
    boot[need] = np.random.default_rng(seed).standard_normal(int(need.sum())).astype(np.float32)
    return boot, need


def test_boot_port_equals_gae_port_without_truncation():
    rew, val, term, trunc, lv, lt, lu = _gae_inputs_np(37, 11, 1, trunc_p=0.0)
    lu[:] = 0.0
    boot = np.full_like(rew, np.nan)
    for gamma, lam in ((0.99, 0.95), (0.9, 0.8)):
        a, r = gae_boot_port(rew, val, term, trunc, lv, lt, lu, boot, gamma, lam)
        b, s = gae_port(rew, val, term, trunc, lv, lt, lu, gamma, lam)
        assert np.array_equal(a, b) and np.array_equal(r, s)


def test_boot_port_changes_only_truncated_episodes():
    """Only rows whose successor is a truncation, and the rows before them in the same episode, change."""
    rew, val, term, trunc, lv, lt, lu = _gae_inputs_np(40, 7, 2)
    boot, need = _boot_for(term, trunc, lt, lu, 3)
    a, _ = gae_boot_port(rew, val, term, trunc, lv, lt, lu, boot)
    b, _ = gae_port(rew, val, term, trunc, lv, lt, lu)
    assert np.isfinite(a).all()
    changed = a != b
    assert changed[need].all()
    for e in range(7):                                       # the first changed row of an episode is a `need` row
        for t in range(40):
            if changed[t, e] and not need[t, e]:
                assert changed[t + 1, e] and trunc[t + 1, e] == 0 and term[t + 1, e] == 0


def test_flag_parsing_and_refusals(track_path):
    from ppo_car_b200.population import check_args, parse_args as pop_args
    from ppo_car_b200.train_ppo import parse_args, track_list

    assert parse_args([]).bootstrap_truncated is False
    assert parse_args(["--bootstrap-truncated"]).bootstrap_truncated is True
    a = pop_args(["--seeds", "0-3", "--bootstrap-truncated", "--pbt-every", "2"])
    assert a.bootstrap_truncated is True and a.seeds == "0-3"
    check_args(a)                                            # accepted with and without PBT
    check_args(pop_args(["--seeds", "0-3", "--bootstrap-truncated"]))
    with pytest.raises(SystemExit, match="--bootstrap-truncated"):
        track_list(parse_args(["--track", "big_track,track", "--bootstrap-truncated"]))
    track_list(parse_args(["--track", "big_track,track", "--bootstrap-truncated", "--fused-rollout"]))
    track_list(parse_args(["--track", "big_track", "--bootstrap-truncated"]))


def test_header_declares_the_twins_and_the_time_limit():
    text = open(os.path.join(ROOT, "include", "carenv_b200.h")).read()
    assert "#define CARENV_TIME_LIMIT 1000" in text
    for name in ("carenv_policy_rollout", "carenv_policy_rollout_tc", "carenv_policy_rollout_warp",
                 "carenv_policy_rollout_tc_multi", "carenv_policy_rollout_warp_pop", "carenv_policy_rollout_tc_pop"):
        assert f"int {name}_final(" in text
    assert "int carenv_final_values(" in text and "int gae_reverse_scan_boot(" in text


def test_twins_bind_the_plain_arguments_plus_three():
    L = ppo_car_b200._lib.lib()
    for name in ("carenv_policy_rollout", "carenv_policy_rollout_tc", "carenv_policy_rollout_warp",
                 "carenv_policy_rollout_tc_multi", "carenv_policy_rollout_warp_pop", "carenv_policy_rollout_tc_pop"):
        assert len(getattr(L, name + "_final").argtypes) == len(getattr(L, name).argtypes) + 3


def test_twins_refuse_null_slots_and_too_few_slots():
    """CARENV_E_INVAL before any device work (a null handle would be refused later: the slot check comes first)."""
    L = ppo_car_b200._lib.lib()
    dummy = 1 << 20                                          # never dereferenced: the calls fail on their arguments
    common_tc = [None, None, 4, 1001, 0, 0, 0] + [None] * 6 + [0.1] + [None] * 10
    for obs, row, slots in ((None, dummy, 2), (dummy, None, 2), (dummy, dummy, 1)):
        rc = L.carenv_policy_rollout_tc_final(*common_tc, obs, row, slots)
        assert rc == -1, (obs, row, slots)
    assert L.gae_reverse_scan_boot(*([dummy] * 7), None, dummy, dummy, 4, 4, 0.99, 0.95, None) == -1


# ---- GPU: the bootstrapping scan ------------------------------------------------------------------------------------
GAMMA_LAMBDA = [(0.99, 0.95), (0.9, 0.8), (1.0, 1.0), (0.99, 0.0)]
GAE_SHAPES = [(1, 1), (7, 63), (9, 65), (63, 4099), (511, 65), (512, 97), (1031, 4099), (519, 310_001),
              (1, 100_000), (17, 100_003), (511, 100_000)]


@pytest.mark.gpu
@pytest.mark.parametrize("T,N", GAE_SHAPES)
def test_boot_scan_matches_port_on_every_launch_path(T, N):
    """k_gae<8, true> one column per thread (T < 512, N < 100,000, or a wave that holds every column), k_gae<8, true>
    grid-stride (T >= 512, N = 310,001), k_gae<16, true> (T < 512, N >= 100,000).  boot is NaN wherever it must not
    be read, so reading it anywhere else would show."""
    host = list(_gae_inputs_np(T, N, T * 7 + N))
    boot, need = _boot_for(host[2], host[3], host[5], host[6], T + N)
    dev = [torch.from_numpy(a).cuda() for a in host]
    bd = torch.from_numpy(boot).cuda()
    pairs = GAMMA_LAMBDA if N < 300_000 else GAMMA_LAMBDA[:2]
    for gamma, lam in pairs:
        adv, ret = ppo_car_b200.gae_reverse_scan(*dev, gamma=gamma, gae_lambda=lam, boot=bd)
        ra, rr = gae_boot_port(*host, boot, gamma, lam)
        a, r = adv.cpu().numpy(), ret.cpu().numpy()
        assert np.isfinite(a).all() and np.isfinite(r).all()
        assert np.array_equal(a, ra) and np.array_equal(r, rr), (gamma, lam)
    # no truncation flags: the same bits as the plain scan
    dev[3].zero_()
    dev[6].zero_()
    for gamma, lam in pairs[:2]:
        a0, r0 = ppo_car_b200.gae_reverse_scan(*dev, gamma=gamma, gae_lambda=lam)
        a1, r1 = ppo_car_b200.gae_reverse_scan(*dev, gamma=gamma, gae_lambda=lam, boot=torch.full_like(bd, np.nan))
        assert torch.equal(a0, a1) and torch.equal(r0, r1)


# ---- GPU: final-observation slots of the fused rollouts -------------------------------------------------------------
def _policy(seed=7, still=5.0):
    """An actor that mostly picks action 8 (no thrust, no turn): episodes mostly run into the time limit, some crash."""
    from ppo_car_b200.train_ppo import ActorCritic

    torch.manual_seed(seed)
    net = ActorCritic(18, 9).cuda()
    with torch.no_grad():
        net.actor[2].weight.mul_(10.0)
        net.actor[2].bias.copy_(torch.tensor([0.0] * 8 + [still]))
    return net


def _start(env, n):
    """reset, then the start time steps 0, 1, 998, 999 in turn; returns the rollout state (obs, term, trunc)."""
    obs = env.reset()[0].clone()
    env.ints[:, 1] = torch.tensor(START_TIMES, dtype=torch.int32, device="cuda").repeat(n // 4 + 1)[:n]
    return obs, torch.zeros(n, device="cuda"), torch.zeros(n, device="cuda")


def _snapshot(env, state):
    return [t.clone() for t in (env.pos, env.vel, env.ints, *state)]


def _restore(env, snap):
    for dst, src in zip((env.pos, env.vel, env.ints), snap[:3]):
        dst.copy_(src)
    return [t.clone() for t in snap[3:]]


def _run(launch, env, snap, T, N, slots):
    """One launch from the snapshot; returns every output (buffer rows, state, last_val, u_dbg, slots)."""
    state = _restore(env, snap)
    buf = ppo_car_b200.Buffer((18,), T, N, "cuda", bootstrap_truncated=slots)
    if slots:
        buf.final_obs_buf.fill_(np.nan)
        buf.final_row_buf.fill_(-7)
    last_val, u = torch.empty(N, device="cuda"), torch.empty((T, N), device="cuda")
    launch(buf, *state, last_val, u)
    torch.cuda.synchronize()
    out = {k: getattr(buf, k).clone() for k in ("obs_buf", "act_buf", "rew_buf", "val_buf", "term_buf", "trunc_buf",
                                                "logprob_buf")}
    out.update(cur_obs=state[0], cur_term=state[1], cur_trunc=state[2], last_val=last_val, u=u, pos=env.pos.clone(),
               vel=env.vel.clone(), ints=env.ints.clone())
    if slots:
        out.update(final_obs=buf.final_obs_buf.clone(), final_row=buf.final_row_buf.clone())
    return out


def _replay_slots(path, snap, act, cols):
    """The actions of columns `cols` replayed through VecCarEnv(final_observation=True).step: per column the rows t
    whose step truncated and info["final_observation"] of those steps."""
    T, n = act.shape[0], len(cols)
    env = ppo_car_b200.VecCarEnv(n, path, reward_scaling=0.1, float_flags=True, final_observation=True)
    env.reset()
    c = torch.as_tensor(cols, device="cuda")
    env.pos.copy_(snap[0][c]); env.vel.copy_(snap[1][c]); env.ints.copy_(snap[2][c])
    rows, fobs = [[] for _ in range(n)], [[] for _ in range(n)]
    for t in range(T):
        _, _, _, tr, info = env.step(act[t, c].to(torch.int64))
        for e in torch.nonzero(tr != 0).view(-1).tolist():
            rows[e].append(t)
            fobs[e].append(info["final_observation"][e].clone())
    env.close()
    return rows, fobs


def _check_slots(path, snap, out, cols=None, expect_some=True):
    act = out["act_buf"]
    cols = list(range(act.shape[1])) if cols is None else list(cols)
    rows, fobs = _replay_slots(path, snap, act, cols)
    fr, fo = out["final_row"].cpu(), out["final_obs"]
    S = fr.shape[0]
    assert S == final_slots(act.shape[0])
    n_used = 0
    for j, c in enumerate(cols):
        k = len(rows[j])
        assert k <= S
        assert fr[:k, c].tolist() == rows[j], (c, fr[:, c].tolist(), rows[j])
        assert (fr[k:, c] == -1).all(), c
        for s in range(k):
            assert torch.equal(fo[s, c], fobs[j][s]), (c, s)
        n_used += k
    if expect_some:
        assert n_used > 0


def _same(a, b, skip=()):
    for k in a:
        if k in skip or k in ("final_obs", "final_row"):
            continue
        assert torch.equal(a[k], b[k]) or (a[k].dtype.is_floating_point and
                                           torch.equal(torch.nan_to_num(a[k], 123.0), torch.nan_to_num(b[k], 123.0))), k


TC_VARIANTS = [("tc3 U4 TAB", {}), ("tc3 U4", {"tab": -1}), ("tc3 U2 TAB", {"max_unroll": 2}),
               ("tc3 U2", {"max_unroll": 2, "tab": -1}), ("tc3 U1", {"force_generic": 1}), ("cuda U4", {}),
               ("cuda U1", {"force_generic": 1}), ("warp", {})]


@pytest.mark.gpu
@pytest.mark.parametrize("T", [1, 1000, 1001, 2001])
@pytest.mark.parametrize("name,opts", TC_VARIANTS, ids=[v[0] for v in TC_VARIANTS])
def test_single_policy_twins(track_path, name, opts, T):
    from ppo_car_b200 import fused_rollout, fused_rollout_warp, pack_policy_weights, pack_policy_weights_tc

    path = track_path("big_track")
    n = 24 if name == "warp" else 300
    env = ppo_car_b200.VecCarEnv(n, path, reward_scaling=0.1, float_flags=True)
    for k, v in opts.items():
        env.set_option(k, v)
    net = _policy()
    snap = _snapshot(env, _start(env, n))
    if name == "warp":
        def launch(buf, o, te, tr, lv, u):
            fused_rollout_warp(env, net.actor, net.critic, buf, o, te, tr, seed=5, step0=3, env_offset=2, last_val=lv,
                               u_dbg=u)
    else:
        packed = (pack_policy_weights_tc if name.startswith("tc3") else pack_policy_weights)(net.actor, net.critic)

        def launch(buf, o, te, tr, lv, u):
            fused_rollout(env, packed, buf, o, te, tr, seed=5, step0=3, env_offset=2, last_val=lv, u_dbg=u)
    plain = _run(launch, env, snap, T, n, False)
    final = _run(launch, env, snap, T, n, True)
    _same(plain, final)
    _check_slots(path, snap, final, expect_some=T >= 1000)


@pytest.mark.gpu
@pytest.mark.parametrize("T", [1, 1001, 2001])
def test_multi_track_twin(track_path, T):
    from ppo_car_b200 import MultiTrackVecEnv, fused_rollout, pack_policy_weights_tc

    paths = [track_path("big_track"), track_path("track")]
    n = 300
    ids = [i % 2 for i in range(n)]
    env = MultiTrackVecEnv(track_paths=paths, track_ids=ids, device="cuda", reward_scaling=0.1, float_flags=True)
    net = _policy(9)
    packed = pack_policy_weights_tc(net.actor, net.critic)
    snap = _snapshot(env, _start(env, n))

    def launch(buf, o, te, tr, lv, u):
        fused_rollout(env, packed, buf, o, te, tr, seed=5, step0=3, last_val=lv, u_dbg=u)
    plain = _run(launch, env, snap, T, n, False)
    final = _run(launch, env, snap, T, n, True)
    _same(plain, final)
    for k, path in enumerate(paths):                         # per track, against a single-track replay
        _check_slots(path, snap, final, cols=[c for c in range(n) if ids[c] == k], expect_some=T >= 1000)


@pytest.mark.gpu
@pytest.mark.parametrize("T", [1, 1001, 2001])
@pytest.mark.parametrize("kernel", ["warp", "tc3"])
def test_population_twins(track_path, synth_path, kernel, T):
    """Member-batched twins: warp (big_track, 32 segments or fewer) and tc3 (a 40-segment ring track)."""
    from ppo_car_b200.population import Population, population_rollout

    path = track_path("big_track") if kernel == "warp" else synth_path("ring40")
    n, P = 20, 3
    pop = Population([3, 4, 5], n, device="cuda:0")
    with torch.no_grad():
        pop.params[2].mul_(10.0)
        pop.params[3][:, 8] = 3.0
    env = ppo_car_b200.VecCarEnv(n * P, path, reward_scaling=0.1, float_flags=True)
    assert ppo_car_b200.population.use_warp_kernel(env, n) == (kernel == "warp")
    snap = _snapshot(env, _start(env, n * P))

    def launch(buf, o, te, tr, lv, u):
        population_rollout(env, pop, buf, o, te, tr, step0=3, last_val=lv, u_dbg=u)
    plain = _run(launch, env, snap, T, n * P, False)
    final = _run(launch, env, snap, T, n * P, True)
    _same(plain, final)
    _check_slots(path, snap, final, expect_some=T >= 1000)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["tc3", "cuda", "warp"])
def test_start_inside_the_wall_never_truncates(synth_path, name):
    """Every step terminates on this track: every slot stays unused (row -1)."""
    from ppo_car_b200 import fused_rollout, fused_rollout_warp, pack_policy_weights, pack_policy_weights_tc

    path = synth_path("near_wall")
    n, T = 64, 1001
    env = ppo_car_b200.VecCarEnv(n, path, reward_scaling=0.1, float_flags=True)
    net = _policy()
    snap = _snapshot(env, _start(env, n))
    if name == "warp":
        def launch(buf, o, te, tr, lv, u):
            fused_rollout_warp(env, net.actor, net.critic, buf, o, te, tr, seed=5, step0=3, last_val=lv, u_dbg=u)
    else:
        packed = (pack_policy_weights_tc if name == "tc3" else pack_policy_weights)(net.actor, net.critic)

        def launch(buf, o, te, tr, lv, u):
            fused_rollout(env, packed, buf, o, te, tr, seed=5, step0=3, last_val=lv, u_dbg=u)
    plain = _run(launch, env, snap, T, n, False)
    final = _run(launch, env, snap, T, n, True)
    _same(plain, final)
    assert (final["final_row"] == -1).all()
    _check_slots(path, snap, final, expect_some=False)


# ---- GPU: the critic pass -------------------------------------------------------------------------------------------
def _critic64(w1, b1, w2, b2, x):
    """float64 critic and the float64 magnitude bound of its float32 evaluation."""
    w1, b1, w2, b2, x = (t.double() for t in (w1, b1, w2, b2, x))
    h = x @ w1.T + b1
    v = torch.relu(h) @ w2.reshape(-1) + b2.reshape(())
    mag = (x.abs() @ w1.abs().T + b1.abs()) @ w2.abs().reshape(-1) + b2.abs().reshape(())
    return v, mag


@pytest.mark.gpu
def test_critic_pass_against_float64_and_member_independence():
    from ppo_car_b200.buffer import final_values
    from ppo_car_b200.population import Population

    torch.manual_seed(0)
    S, n, P, T = 3, 50, 3, 2500
    N = n * P
    pop = Population([11, 12, 13], n, device="cuda")
    fo = torch.rand((S, N, 18), device="cuda") * 2 - 1
    # increasing rows per column as the rollouts write them; unused slots (-1) at the end and in column 0..4
    fr = (torch.randint(0, 800, (S, N), device="cuda") + 800 * torch.arange(S, device="cuda")[:, None]).int()
    fr[2, ::3] = -1
    fr[:, :5] = -1
    boot = torch.full((T, N), float("nan"), device="cuda")
    final_values(pop, fo, fr, boot)
    used = fr >= 0
    for p in range(P):
        cols = slice(p * n, (p + 1) * n)
        w1, b1, w2, b2 = (t[p] for t in pop.params[4:8])
        v64, mag = _critic64(w1, b1, w2, b2, fo[:, cols])
        rows, c = fr[:, cols].long(), torch.arange(n, device="cuda").expand(S, n)
        got = boot[:, cols][rows.clamp(min=0), c].double()
        u = used[:, cols]
        assert ((got - v64).abs()[u] <= 64 * 2.0 ** -24 * mag[u] + 1e-30).all(), p
        # the single-policy call on member p alone gives the same bits
        one = torch.full((T, n), float("nan"), device="cuda")
        net = torch.nn.Sequential(torch.nn.Linear(18, 256), torch.nn.ReLU(), torch.nn.Linear(256, 1)).cuda()
        with torch.no_grad():
            for layer, (w, b) in ((net[0], (w1, b1)), (net[2], (w2, b2))):
                layer.weight.copy_(w)
                layer.bias.copy_(b)
        final_values(net, fo[:, cols].contiguous(), fr[:, cols].contiguous(), one)
        assert torch.equal(torch.nan_to_num(one, 7.0), torch.nan_to_num(boot[:, cols], 7.0)), p
    # unused entries are untouched; another member's parameters do not change member 0's values
    written = torch.zeros((T, N), dtype=torch.bool, device="cuda")
    for s in range(S):
        ok = used[s]
        written[fr[s][ok].long(), torch.arange(N, device="cuda")[ok]] = True
    assert boot[~written].isnan().all() and boot[written].isfinite().all()
    before = boot[:, :n].clone()
    with torch.no_grad():
        pop.params[4][1:].mul_(-3.0)
    boot.fill_(float("nan"))
    final_values(pop, fo, fr, boot)
    assert torch.equal(torch.nan_to_num(before, 7.0), torch.nan_to_num(boot[:, :n], 7.0))


# ---- GPU: one epoch of training with the flag -----------------------------------------------------------------------
class _Capture:
    """Records, per calculate_advantages call, the buffer rows, the bootstrap inputs and the result; and the critic and
    final-observation slots each Buffer.final_values call sees."""

    def __init__(self, monkeypatch, start_times=True):
        from ppo_car_b200.buffer import Buffer
        from ppo_car_b200.vec_env import MultiTrackVecEnv, VecCarEnv

        self.gae, self.finals, self.fobs = [], [], []
        orig_gae, orig_fv = Buffer.calculate_advantages, Buffer.final_values
        cap = self

        def gae(buf, lv, lt, lu):
            adv, ret = orig_gae(buf, lv, lt, lu)
            rows = {k: getattr(buf, k).clone() for k in ("act_buf", "rew_buf", "val_buf", "term_buf", "trunc_buf",
                                                         "logprob_buf")}
            rows["obs"] = (buf.pose_buf if buf.compact_obs else buf.obs_buf).clone()
            cap.gae.append(dict(rows=rows, last=(lv.clone(), lt.clone(), lu.clone()), adv=adv.clone(),
                                ret=ret.clone(), boot=None if buf.boot_buf is None else buf.boot_buf.clone()))
            return adv, ret

        def fv(buf, critic):
            orig_fv(buf, critic)
            cap.finals.append(dict(critic=[t.detach().clone() for t in (critic.params[4:8] if hasattr(critic, "params")
                                                                        else (critic[0].weight, critic[0].bias,
                                                                              critic[2].weight, critic[2].bias))],
                                   obs=buf.final_obs_buf.clone(), row=buf.final_row_buf.clone()))
        monkeypatch.setattr(Buffer, "calculate_advantages", gae)
        monkeypatch.setattr(Buffer, "final_values", fv)
        if start_times:                                      # episodes that reach the time limit within one epoch
            for cls in (VecCarEnv, MultiTrackVecEnv):
                orig_reset = cls.reset

                def reset(self, *a, _orig=orig_reset, **k):
                    out = _orig(self, *a, **k)
                    n = self.num_envs
                    # the same pattern in every block of 24 columns: a population member sees train_ppo's
                    self.ints[:, 1] = (990 + torch.arange(n, device=self.device, dtype=torch.int32) % 24) % 1000
                    return out
                monkeypatch.setattr(cls, "reset", reset)


def _gae64(rows, last, boot64, gamma=0.99, lam=0.95):
    """float64 GAE with time-limit bootstrapping (boot64: float64 next values where the successor truncated)."""
    rew, val, term, trunc = (rows[k].double() for k in ("rew_buf", "val_buf", "term_buf", "trunc_buf"))
    lv, lt, lu = (t.double().reshape(-1) for t in last)
    T = rew.shape[0]
    adv = torch.zeros_like(rew)
    a = torch.zeros_like(lv)
    for t in range(T - 1, -1, -1):
        nv, te, tr = (lv, lt, lu) if t == T - 1 else (val[t + 1], term[t + 1], trunc[t + 1])
        nv = torch.where((tr == 1) & (te == 0), boot64[t], nv)
        a = rew[t] + gamma * nv * (1 - te) - val[t] + gamma * lam * (1 - te) * (1 - tr) * a
        adv[t] = a
    return adv


def _truncated_episode_rows(rows, last):
    """[T, N] mask of the rows of episodes that end by truncation inside the rollout (the rows the flag may change)."""
    term, trunc = rows["term_buf"], rows["trunc_buf"]
    T, N = term.shape
    lt, lu = (t.reshape(-1) for t in last[1:])
    mask = torch.zeros((T, N), dtype=torch.bool, device=term.device)
    live = (lu.reshape(-1) == 1) & (lt.reshape(-1) == 0)
    for t in range(T - 1, -1, -1):
        mask[t] = live
        live = (trunc[t] == 1) & (term[t] == 0) | (live & (term[t] == 0) & (trunc[t] == 0))
    return mask


def _boot64_from_slots(fin, T, N, n_per_member):
    boot = torch.zeros((T, N), dtype=torch.float64, device="cuda")
    w = fin["critic"]
    P = N // n_per_member
    for s in range(fin["row"].shape[0]):
        for p in range(P):
            cols = torch.arange(p * n_per_member, (p + 1) * n_per_member, device="cuda")
            par = [t[p] for t in w] if w[0].dim() == 3 else w          # stacked [P, ...] or one critic
            v, _ = _critic64(*par, fin["obs"][s, cols])
            r = fin["row"][s, cols]
            ok = r >= 0
            boot[r[ok].long(), cols[ok]] = v[ok]
    return boot


def _check_epoch(off, on, boot64, tol=2e-4):
    for k in off["rows"]:
        assert torch.equal(off["rows"][k], on["rows"][k]), k
    mask = _truncated_episode_rows(on["rows"], on["last"])
    assert mask.any()
    assert torch.equal(off["adv"][~mask], on["adv"][~mask]) and torch.equal(off["ret"][~mask], on["ret"][~mask])
    ref = _gae64(on["rows"], on["last"], boot64)
    err = (on["adv"].double() - ref).abs()[mask]
    assert (err <= tol * (1 + ref.abs()[mask])).all(), float(err.max())


E2E = [("warp", ["--fused-rollout", "--fused-update"]),
       ("tc3", ["--fused-rollout", "--fused-update", "--n-envs", "4100"]),
       ("cuda", ["--fused-rollout", "--fused-cuda-cores"]),
       ("compact", ["--fused-rollout", "--compact-obs", "--fused-update"]),
       ("multi", ["--fused-rollout", "--track", "big_track,track", "--n-envs", "48"]),
       ("eager", []),
       ("eager-graph", ["--cuda-graph"])]


@pytest.mark.gpu
@pytest.mark.parametrize("name,extra", E2E, ids=[e[0] for e in E2E])
def test_one_epoch_of_train_ppo(monkeypatch, name, extra):
    from ppo_car_b200.train_ppo import parse_args, train

    base = ["--track", "big_track", "--n-envs", "24", "--n-epochs", "1", "--n-steps", "256", "--seed", "3"]
    runs = {}
    for flag in (False, True):
        cap = _Capture(monkeypatch)
        train(parse_args(base + extra + (["--bootstrap-truncated"] if flag else [])))
        runs[flag] = cap
    off, on = runs[False].gae[0], runs[True].gae[0]
    T, N = on["adv"].shape
    if name.startswith("eager"):
        boot64 = on["boot"].double()                          # critic(final observation) as the loop stored it
        _check_epoch(off, on, boot64, tol=1e-3)
    else:
        _check_epoch(off, on, _boot64_from_slots(runs[True].finals[0], T, N, N))


@pytest.mark.gpu
def test_one_epoch_of_population_equals_train_ppo(monkeypatch):
    """Member p of `population --bootstrap-truncated` equals `train_ppo --seed s --bootstrap-truncated` (the fused
    rollout and the one-launch update) on epoch 1: rollout rows, advantages and returns."""
    from ppo_car_b200.population import parse_args as pop_args, train_population
    from ppo_car_b200.train_ppo import parse_args, train

    common = ["--track", "big_track", "--n-envs", "24", "--n-epochs", "1", "--n-steps", "256",
              "--bootstrap-truncated"]
    cap = _Capture(monkeypatch)
    train_population(pop_args(common + ["--seeds", "0-2"]))
    pop_run = cap.gae[0]
    for p, seed in enumerate([0, 1, 2]):
        c1 = _Capture(monkeypatch)
        train(parse_args(common + ["--seed", str(seed), "--fused-rollout", "--fused-update"]))
        one = c1.gae[0]
        cols = slice(p * 24, (p + 1) * 24)
        for k in one["rows"]:
            assert torch.equal(one["rows"][k], pop_run["rows"][k][:, cols]), (p, k)
        assert torch.equal(one["adv"], pop_run["adv"][:, cols]) and torch.equal(one["ret"], pop_run["ret"][:, cols])


@pytest.mark.gpu
def test_one_epoch_of_population_bootstraps(monkeypatch):
    from ppo_car_b200.population import parse_args as pop_args, train_population

    base = ["--track", "big_track", "--n-envs", "24", "--n-epochs", "1", "--n-steps", "256", "--seeds", "0-2"]
    runs = {}
    for flag in (False, True):
        cap = _Capture(monkeypatch)
        train_population(pop_args(base + (["--bootstrap-truncated"] if flag else [])))
        runs[flag] = cap
    off, on = runs[False].gae[0], runs[True].gae[0]
    T, N = on["adv"].shape
    _check_epoch(off, on, _boot64_from_slots(runs[True].finals[0], T, N, 24))
