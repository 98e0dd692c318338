"""Several tracks in the fused rollout and in policy evaluation (C ABI carenv_policy_rollout_tc_multi /
carenv_policy_eval_multi, k_policy_rollout_tc3<0> / k_policy_eval<0>), train_ppo and the evaluation CLI.

The single-track kernels are the oracle: every environment of a multi-track rollout must produce, bit for bit, the rows
the single-track tensor-core rollout produces for the same environment on its track alone (the random stream is keyed
by the global env id, not by the track), and every multi-track evaluation record must equal the single-track record of
the same episode id on its track.

CPU: track assignment per shard, per-track sums and summaries of EvalResult, argument checks, train_ppo refusals.
GPU (-m gpu): bit-identity against the single-track kernels with tracks mixed inside warps, replay through
MultiTrackVecEnv.step, split launches, evaluation, refusals and short training runs."""
import ctypes as C
import functools
import math
import os
from types import SimpleNamespace

import numpy as np
import pytest
import torch

import ppo_car_b200
from ppo_car_b200 import _lib
from ppo_car_b200.evaluate import SUM_FIELDS, EvalResult, default_episode_tracks
from ppo_car_b200.shard import shard_range, track_blocks
from ppo_car_b200.track import builtin_track
from ppo_car_b200.train_ppo import ActorCritic, parse_args, track_list, train
from tests.synth_tracks import near_wall_track, ring_track

SEED = (0x5EED << 32) | 11             # a non-zero high key word
ENV_OFFSET = 70001
STEP0 = 2 ** 32 - 17
TRACKS = ("track", "big_track", "ring7_5", "ring64_64", "near_wall")   # 24 .. 128 segments, odd count, start in a wall


def make_records(ret, length, gates, laps, first_lap, outcome) -> torch.Tensor:
    n = len(ret)
    rec = torch.zeros((n, 8), dtype=torch.int32)
    rec.view(torch.float64)[:, 0] = torch.tensor(ret, dtype=torch.float64)
    for col, v in zip(range(2, 7), (length, gates, laps, first_lap, outcome)):
        rec[:, col] = torch.tensor(v, dtype=torch.int32)
    return rec


# ---------------------------------------------------------------------------------------------------- CPU
def test_track_blocks_are_contiguous_balanced_and_shard_independent():
    for n_total, k in ((64, 2), (1000, 3), (7, 7), (1_048_576, 3), (5, 1)):
        whole = track_blocks(n_total, k, 0, n_total)
        assert whole.dtype == np.int32 and whole.shape == (n_total,)
        assert (np.diff(whole) >= 0).all() and whole[0] == 0 and whole[-1] == k - 1
        sizes = np.bincount(whole, minlength=k)
        assert sizes.max() - sizes.min() <= 1                              # balanced blocks
        assert np.array_equal(whole, np.arange(n_total) * k // n_total)
        for world in (1, 2, 3, 8):
            parts = [track_blocks(n_total, k, *shard_range(n_total, world, r)) for r in range(world)]
            assert np.array_equal(np.concatenate(parts), whole)
    with pytest.raises(ValueError):
        track_blocks(2, 3, 0, 2)                                           # fewer envs than tracks
    with pytest.raises(ValueError):
        track_blocks(8, 2, 4, 9)


def test_default_episode_tracks_do_not_depend_on_the_split():
    whole = default_episode_tracks(1000, 3)
    assert whole.dtype == torch.int32 and torch.equal(whole, (torch.arange(1000) % 3).to(torch.int32))
    assert torch.equal(torch.cat([default_episode_tracks(400, 3), default_episode_tracks(600, 3, episode0=400)]), whole)
    big = 2 ** 64 - 5                                                      # ids near the top of the 64-bit range
    assert default_episode_tracks(5, 3, episode0=big).tolist() == [(big + i) % 3 for i in range(5)]


def test_sums_and_summaries_by_track_of_hand_made_records():
    rec = make_records(ret=[10.5, -2.0, 40.0, 1.5, 7.0], length=[1000, 20, 700, 1000, 300], gates=[12, 1, 30, 3, 5],
                       laps=[0, 0, 2, 0, 1], first_lap=[-1, -1, 350, -1, 250], outcome=[2, 1, 1, 2, 1])
    track = torch.tensor([0, 2, 0, 2, 0], dtype=torch.int32)
    res = EvalResult(rec, track=track, n_tracks=3)
    by = res.sums_by_track()
    assert by.shape == (3, len(SUM_FIELDS)) and by.dtype == torch.float64
    for k in range(3):
        sel = track == k
        assert by[k].tolist() == EvalResult(rec[sel]).sums().tolist()       # same fields, same arithmetic
    assert by[1].tolist() == [0.0] * len(SUM_FIELDS)
    assert torch.allclose(by.sum(0), res.sums())
    summ = res.summary_by_track()
    assert [s["episodes"] for s in summ] == [3, 0, 2]
    assert summ[1] == {"episodes": 0}
    assert summ[0]["mean_return"] == (10.5 + 40.0 + 7.0) / 3 and summ[0]["lap_rate"] == 2 / 3
    assert summ[2]["avg_reward"] == (-2.0 + 1.5) / 1020 and summ[2]["crash_rate"] == 0.5
    # shards add up
    a = EvalResult(rec[:2], track=track[:2], n_tracks=3).sums_by_track()
    b = EvalResult(rec[2:], track=track[2:], n_tracks=3).sums_by_track()
    assert torch.equal(a + b, by)
    assert res.summary_by_track(a + b) == summ
    with pytest.raises(ValueError):
        EvalResult(rec).sums_by_track()                                    # single-track result: no track column
    with pytest.raises(ValueError):
        EvalResult(rec, track=track[:3], n_tracks=3)
    with pytest.raises(ValueError):
        EvalResult(rec, track=track)


def test_null_multi_handles_are_errors():
    L = _lib.lib()
    assert L.carenv_policy_rollout_tc_multi(None, None, None, 4, 4, 0, 0, 0, *([None] * 6), 1.0, *([None] * 10)) == -1
    assert b"handle" in L.carenv_last_error()
    rec = torch.zeros((4, 8), dtype=torch.int32)
    w = torch.zeros(256 * 18)
    p = [C.c_void_p(w.data_ptr())] * 4
    assert L.carenv_policy_eval_multi(None, None, *p, 4, 0, 0, 0, C.c_void_p(rec.data_ptr()), 0, None, None,
                                      None) == -1


@pytest.mark.parametrize("extra,message", [
    (["--compact-obs", "--fused-rollout"], "--compact-obs"),
    (["--fused-rollout", "--fused-cuda-cores"], "--fused-cuda-cores"),
    (["--cuda-graph"], "--cuda-graph"),
    (["--n-envs", "2"], "smaller than the number of tracks"),
])
def test_train_ppo_refuses_what_has_no_multi_track_path(extra, message):
    args = parse_args(["--track", "big_track,track,big_track", "--n-envs", "64"] + extra)
    with pytest.raises(SystemExit) as e:
        train(args)
    assert message in str(e.value)


def test_track_flag_parsing():
    names, paths = track_list(parse_args(["--track", "big_track,track"]))
    assert names == ["big_track", "track"] and paths == [builtin_track("big_track"), builtin_track("track")]
    path = builtin_track("track")
    assert track_list(parse_args(["--track", path])) == ([path], [path])
    assert track_list(parse_args(["--track", "track", "--compact-obs", "--n-envs", "1"]))[1] == [path]   # one track: as before


# ---------------------------------------------------------------------------------------------------- GPU
RINGS = {"ring7_5": (7, 5), "ring64_64": (64, 64), "ring65_64": (65, 64)}


def track_path(name, directory):
    if name in ("big_track", "track"):
        return builtin_track(name)
    if name == "near_wall":
        return near_wall_track(os.path.join(directory, "near_wall.json"))
    n_outer, n_inner = RINGS[name]
    return ring_track(os.path.join(directory, name + ".json"), n_outer, n_inner,
                      wobble=0.03 if n_outer + n_inner > 64 else 0.08)


@pytest.fixture(scope="module")
def tracks(tmp_path_factory):
    d = str(tmp_path_factory.mktemp("tracks"))
    return functools.lru_cache(maxsize=None)(lambda name: track_path(name, d))


def make_policy(seed=3, actor_scale=4.0):
    """ActorCritic with a non-uniform actor on the GPU (so that all nine actions are taken)."""
    torch.manual_seed(seed)
    net = ActorCritic(18, 9).cuda()
    with torch.no_grad():
        net.actor[2].weight.mul_(actor_scale)
        net.actor[2].bias.copy_(torch.linspace(-1, 1, 9))
        net.critic[2].bias.fill_(0.3)
    return net


def random_ids(n, k, seed=0):
    return torch.from_numpy(np.random.default_rng(seed).integers(0, k, n).astype(np.int32))


def rollout(env, net, T, state, last_val=True, env_offset=ENV_OFFSET, step0=STEP0):
    """One fused tensor-core launch from ``state`` = [cur_obs, cur_term, cur_trunc] (updated in place)."""
    n = env.num_envs
    buf = ppo_car_b200.Buffer((18,), T, n, torch.device("cuda"))
    lv = torch.full((n,), float("nan"), device="cuda") if last_val else None
    u = torch.full((T, n), float("nan"), device="cuda")
    ppo_car_b200.fused_rollout(env, ppo_car_b200.pack_policy_weights_tc(net.actor, net.critic), buf, *state, seed=SEED,
                               step0=step0, env_offset=env_offset, last_val=lv, u_dbg=u)
    torch.cuda.synchronize()
    return SimpleNamespace(obs=buf.obs_buf, act=buf.act_buf, rew=buf.rew_buf, val=buf.val_buf, term=buf.term_buf,
                           trunc=buf.trunc_buf, logp=buf.logprob_buf, u=u, last_val=lv)


def start_state(env):
    n = env.num_envs
    return [env.reset()[0].clone(), torch.zeros(n, device="cuda"), torch.zeros(n, device="cuda")]


def multi_env(paths, ids):
    return ppo_car_b200.MultiTrackVecEnv(track_paths=paths, track_ids=ids, reward_scaling=0.1, float_flags=True)


ROWS = ("obs", "act", "rew", "val", "logp", "term", "trunc", "u")


def check_against_single_track(paths, ids, net, T, r, state, env, last_val):
    n = len(ids)
    for k, path in enumerate(paths):
        sel = (ids == k).cuda()
        if not sel.any():
            continue
        single = ppo_car_b200.VecCarEnv(n, path, reward_scaling=0.1, float_flags=True)
        s_state = start_state(single)
        s = rollout(single, net, T, s_state, last_val=last_val)
        for name in ROWS:
            assert torch.equal(getattr(r, name)[:, sel], getattr(s, name)[:, sel]), (path, name)
        if last_val:
            assert torch.equal(r.last_val[sel], s.last_val[sel]), (path, "last_val")
        for a, b, name in zip(state, s_state, ("cur_obs", "cur_term", "cur_trunc")):
            assert torch.equal(a[sel], b[sel]), (path, name)
        for name in ("pos", "vel", "ints"):
            assert torch.equal(getattr(env, name)[sel], getattr(single, name)[sel]), (path, name)
        single.close()


SHAPES = [(1, 1, True), (1, 300, False), (257, 7, True), (257, 300, True), (2049, 1, False), (2049, 7, True),
          (40003, 7, False), (40003, 300, True)]


@pytest.mark.gpu
@pytest.mark.parametrize("n,T,last_val", SHAPES, ids=[f"n{n}-T{T}-{'lv' if lv else 'nolv'}" for n, T, lv in SHAPES])
def test_rollout_equals_single_track_runs(tracks, n, T, last_val):
    paths = [tracks(t) for t in TRACKS]
    ids = random_ids(n, len(paths), seed=n + T)                            # tracks mixed inside every warp
    net = make_policy()
    env = multi_env(paths, ids)
    state = start_state(env)
    r = rollout(env, net, T, state, last_val=last_val)
    assert not torch.isnan(r.u).any() and (r.act < 9).all()
    if n >= 2049:
        assert len(torch.unique(ids)) == len(paths)
    check_against_single_track(paths, ids, net, T, r, state, env, last_val)
    env.close()


@pytest.mark.gpu
def test_rows_replay_through_the_multi_track_step(tracks):
    paths = [tracks(t) for t in TRACKS]
    n, T = 513, 300
    ids = random_ids(n, len(paths), seed=1)
    env = multi_env(paths, ids)
    state = start_state(env)
    r = rollout(env, make_policy(), T, state)
    rep = multi_env(paths, ids)
    obs = rep.reset()[0].clone()
    assert torch.equal(r.obs[0], obs) and not r.term[0].any() and not r.trunc[0].any()
    for t in range(T):
        o, rew, te, tr, _ = rep.step(r.act[t].to(torch.uint8))
        assert torch.equal(rew, r.rew[t]), t
        # the step's outputs are the next row's inputs; after the last step, the rollout state
        nxt = (r.obs[t + 1], r.term[t + 1], r.trunc[t + 1]) if t + 1 < T else state
        assert all(torch.equal(a, b) for a, b in zip((o, te, tr), nxt)), t
    for name in ("pos", "vel", "ints"):
        assert torch.equal(getattr(env, name), getattr(rep, name)), name
    assert (r.term.sum() + r.trunc.sum()) > 0                             # episodes end inside the window


@pytest.mark.gpu
def test_two_launches_and_two_halves_equal_one_launch(tracks):
    paths = [tracks(t) for t in TRACKS]
    n, T1, T2 = 2049, 40, 60
    ids = random_ids(n, len(paths), seed=2)
    net = make_policy()
    env = multi_env(paths, ids)
    state = start_state(env)
    one = rollout(env, net, T1 + T2, state)
    env2 = multi_env(paths, ids)
    state2 = start_state(env2)
    a = rollout(env2, net, T1, state2, last_val=False)
    b = rollout(env2, net, T2, state2, step0=STEP0 + T1)
    for name in ROWS:
        assert torch.equal(torch.cat([getattr(a, name), getattr(b, name)]), getattr(one, name)), name
    assert torch.equal(b.last_val, one.last_val)
    assert all(torch.equal(x, y) for x, y in zip(state, state2))
    h = 1000                                                               # two shards with env_offset
    halves = []
    for lo, hi in ((0, h), (h, n)):
        e = multi_env(paths, ids[lo:hi])
        st = start_state(e)
        halves.append((rollout(e, net, T1 + T2, st, env_offset=ENV_OFFSET + lo), st, e))
    for name in ROWS + ("last_val",):
        dim = 0 if name == "last_val" else 1
        assert torch.equal(torch.cat([getattr(x[0], name) for x in halves], dim=dim), getattr(one, name)), name
    for i in range(3):
        assert torch.equal(torch.cat([x[1][i] for x in halves]), state[i])
    for name in ("pos", "vel", "ints"):
        assert torch.equal(torch.cat([getattr(x[2], name) for x in halves]), getattr(env, name))


def _single_eval(path, actor, n, **kw):
    env = ppo_car_b200.VecCarEnv(1, path, device="cuda:0")
    res = ppo_car_b200.evaluate_policy(env, actor, n, **kw)
    torch.cuda.synchronize()
    env.close()
    return res


@pytest.mark.gpu
@pytest.mark.parametrize("greedy", [False, True])
def test_evaluation_equals_single_track_records(tracks, monkeypatch, greedy):
    from ppo_car_b200 import evaluate_policy

    paths = [tracks(t) for t in TRACKS]
    actor = make_policy(seed=5).actor
    N, n_tr = 3000, 200
    ep_tracks = random_ids(N, len(paths), seed=7)
    env = multi_env(paths, [0])
    res = evaluate_policy(env, actor, N, greedy=greedy, seed=SEED, episode0=ENV_OFFSET, trace=n_tr,
                          episode_tracks=ep_tracks)
    torch.cuda.synchronize()
    assert torch.equal(res.track.cpu(), ep_tracks)
    for k, path in enumerate(paths):
        sel = ep_tracks == k
        single = _single_eval(path, actor, N, greedy=greedy, seed=SEED, episode0=ENV_OFFSET, trace=n_tr)
        assert torch.equal(res.records.cpu()[sel], single.records.cpu()[sel]), path
        st = sel[:n_tr]
        assert torch.equal(res.trace_actions.cpu()[st], single.trace_actions.cpu()[st]), path
        if not greedy:
            bits = lambda t: t.cpu()[st].view(torch.int32)              # NaN past an episode's end
            assert torch.equal(bits(res.trace_u), bits(single.trace_u)), path
    assert (res.outcome[ep_tracks.cuda() == TRACKS.index("near_wall")] == 1).all()
    assert torch.allclose(res.sums_by_track().sum(0), res.sums())
    # splitting the batch and capping the grid change nothing
    k = 1234
    a = evaluate_policy(env, actor, k, greedy=greedy, seed=SEED, episode0=ENV_OFFSET, episode_tracks=ep_tracks[:k])
    b = evaluate_policy(env, actor, N - k, greedy=greedy, seed=SEED, episode0=ENV_OFFSET + k,
                        episode_tracks=ep_tracks[k:])
    monkeypatch.setenv("CARENV_EVAL_CTAS", "1")                            # 128 slots play 1,000 episodes
    capped = evaluate_policy(env, actor, 1000, greedy=greedy, seed=SEED, episode0=ENV_OFFSET,
                             episode_tracks=ep_tracks[:1000])
    monkeypatch.delenv("CARENV_EVAL_CTAS")
    torch.cuda.synchronize()
    assert torch.equal(torch.cat([a.records, b.records]), res.records)
    assert torch.equal(capped.records, res.records[:1000])
    # the default assignment: global id modulo the number of tracks
    d = evaluate_policy(env, actor, 500, greedy=greedy, seed=SEED, episode0=ENV_OFFSET)
    torch.cuda.synchronize()
    expect = default_episode_tracks(500, len(paths), ENV_OFFSET)
    assert torch.equal(d.track.cpu(), expect)
    e = evaluate_policy(env, actor, 500, greedy=greedy, seed=SEED, episode0=ENV_OFFSET, episode_tracks=expect)
    assert torch.equal(d.records, e.records)
    env.close()


@pytest.mark.gpu
def test_refusals(tracks):
    from ppo_car_b200 import evaluate_policy

    net = make_policy()
    paths = [tracks("track"), tracks("ring65_64")]                         # 129 segments
    env = multi_env(paths, [0, 1, 0, 1])
    state = start_state(env)
    with pytest.raises(ppo_car_b200.CarEnvError, match="128"):
        rollout(env, net, 4, state)
    with pytest.raises(ppo_car_b200.CarEnvError, match="128"):
        evaluate_policy(env, net.actor, 8)
    env.close()
    paths = [tracks("track"), tracks("big_track")]
    env = multi_env(paths, [0, 1, 0, 1])
    state = start_state(env)
    compact = ppo_car_b200.Buffer((18,), 4, 4, torch.device("cuda"), compact_obs=True)
    with pytest.raises(ValueError, match="pose records"):
        ppo_car_b200.fused_rollout(env, ppo_car_b200.pack_policy_weights_tc(net.actor, net.critic), compact, *state,
                                   seed=0, step0=0)
    buf = ppo_car_b200.Buffer((18,), 4, 4, torch.device("cuda"))
    with pytest.raises(ValueError, match="tensor-core"):
        ppo_car_b200.fused_rollout(env, ppo_car_b200.pack_policy_weights(net.actor, net.critic), buf, *state,
                                   seed=0, step0=0)
    with pytest.raises(ValueError):
        multi_env(paths, [0, 2, 1, 0])                                     # track id out of range
    with pytest.raises(ValueError):
        evaluate_policy(env, net.actor, 4, episode_tracks=[0, 1, 2, 0])
    with pytest.raises(ValueError):
        evaluate_policy(env, net.actor, 4, episode_tracks=[0, 1, 0])
    with pytest.raises(ValueError):
        evaluate_policy(env, net.actor, 2, episode_tracks=[-1, 0])
    single = ppo_car_b200.VecCarEnv(1, paths[0])
    with pytest.raises(ValueError):
        evaluate_policy(single, net.actor, 2, episode_tracks=[0, 0])
    L = _lib.lib()
    p = lambda t: C.c_void_p(t.data_ptr())
    ids = torch.zeros(4, dtype=torch.int32, device="cuda")
    w = torch.zeros(27404, device="cuda")
    f = torch.zeros(4 * 18, device="cuda")
    assert L.carenv_policy_rollout_tc_multi(env._multi, None, p(w), 4, 4, 0, 0, 0, *([p(f)] * 6), 1.0,
                                            *([p(f)] * 7), None, None, None) == -1
    assert L.carenv_policy_rollout_tc_multi(env._multi, p(ids), p(w), -1, 4, 0, 0, 0, *([p(f)] * 6), 1.0,
                                            *([p(f)] * 7), None, None, None) == -1
    rec = torch.zeros((4, 8), dtype=torch.int32, device="cuda")
    wa = [p(w)] * 4
    assert L.carenv_policy_eval_multi(env._multi, None, *wa, 4, 0, 0, 0, p(rec), 0, None, None, None) == -1
    assert L.carenv_policy_eval_multi(env._multi, p(ids), *wa, -1, 0, 0, 0, p(rec), 0, None, None, None) == -1
    assert L.carenv_policy_eval_multi(env._multi, p(ids), *wa, 4, 0, 0, 0, p(rec), 2, None, None, None) == -1
    assert L.carenv_policy_eval_multi(env._multi, p(ids), *wa, 0, 0, 0, 0, p(rec), 0, None, None, None) == 0
    env.close()


def _check_training(hist, names):
    assert len(hist) == 12 and all(math.isfinite(h["total_loss"]) for h in hist)
    for h in hist:
        assert [b["track"] for b in h["by_track"]] == names
        assert math.isclose(sum(b["episodes"] for b in h["by_track"]), h["episodes"])
    for k, name in enumerate(names):
        first, last = hist[0]["by_track"][k]["avg_reward"], hist[-1]["by_track"][k]["avg_reward"]
        assert last > first + 0.02, (name, first, last)


@pytest.mark.gpu
def test_fused_training_on_two_tracks():
    args = parse_args(["--track", "big_track,track", "--n-envs", "64", "--n-epochs", "12", "--n-steps", "256",
                       "--fused-rollout", "--fused-update", "--eval-every", "6"])
    hist = train(args)
    _check_training(hist, ["big_track", "track"])
    assert ["eval" in h for h in hist] == [False] * 5 + [True] + [False] * 5 + [True]
    ev = hist[-1]["eval"]
    assert [b["track"] for b in ev["by_track"]] == ["big_track", "track"]
    assert sum(b["episodes"] for b in ev["by_track"]) == ev["episodes"] == 1024


@pytest.mark.gpu
def test_eager_training_on_two_tracks():
    args = parse_args(["--track", "big_track,track", "--n-envs", "64", "--n-epochs", "12", "--n-steps", "256",
                       "--fused-update", "--per-minibatch-update"])
    _check_training(train(args), ["big_track", "track"])


@pytest.mark.gpu
def test_evaluate_cli_by_track(tmp_path):
    from ppo_car_b200.evaluate import main

    ckpt = str(tmp_path / "model.dat")
    torch.manual_seed(4)
    torch.save(ActorCritic(18, 9).state_dict(), ckpt)
    out = main(["--checkpoint", ckpt, "--track", "big_track,track", "--episodes", "3001", "--seed", "2"])
    assert [b["track"] for b in out["by_track"]] == ["big_track", "track"]
    assert [b["episodes"] for b in out["by_track"]] == [1501, 1500]
    one = main(["--checkpoint", ckpt, "--track", "track", "--episodes", "3001", "--seed", "2"])
    assert "by_track" not in one
