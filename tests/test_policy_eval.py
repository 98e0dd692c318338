"""Policy evaluation (ppo_car_b200.evaluate, C ABI carenv_policy_eval, csrc/policy_eval.cuh).

CPU: argument checks, checkpoint loading, the summary arithmetic.  GPU (-m gpu): every record and traced action is
checked against a replay of the traced actions through VecCarEnv.step (the path that is bit-exact against the
oracle) and against the torch actor on the replayed observations; results do not depend on how a batch is split or
scheduled; the start-inside-the-wall track; the train_ppo hook; the torchrun CLI."""
import ctypes as C
import json
import math
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from ppo_car_b200 import _lib
from ppo_car_b200.evaluate import SUM_FIELDS, TIME_LIMIT, EvalResult, load_checkpoint, parse_args
from ppo_car_b200.train_ppo import ActorCritic

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
THRUST_ACTIONS = (0, 4, 5)              # decode_action: thrust > 0 earns the 0.01 bonus (lib/car_env.py:698-722)


def make_records(ret, length, gates, laps, first_lap, outcome) -> torch.Tensor:
    n = len(ret)
    rec = torch.zeros((n, 8), dtype=torch.int32)
    rec.view(torch.float64)[:, 0] = torch.tensor(ret, dtype=torch.float64)
    for col, v in zip(range(2, 7), (length, gates, laps, first_lap, outcome)):
        rec[:, col] = torch.tensor(v, dtype=torch.int32)
    return rec


# ---------------------------------------------------------------------------------------------------- CPU
def test_null_handle_is_an_error():
    L = _lib.lib()
    rec = torch.zeros((4, 8), dtype=torch.int32)
    w = torch.zeros(256 * 18)
    p = [C.c_void_p(w.data_ptr())] * 4
    assert L.carenv_policy_eval(None, *p, 4, 0, 0, 0, C.c_void_p(rec.data_ptr()), 0, None, None, None) == -1
    assert b"handle" in L.carenv_last_error()


def test_load_checkpoint_reproduces_the_stored_outputs(golden_dir, tmp_path):
    g = np.load(os.path.join(golden_dir, "agent_checkpoint.npz"))
    path = str(tmp_path / "model.dat")
    torch.save({k[2:]: torch.from_numpy(g[k]) for k in g.files if k.startswith("w_")}, path)
    net = load_checkpoint(path)
    assert isinstance(net, ActorCritic)
    with torch.no_grad():
        _, logp, _, val = net.act(torch.from_numpy(g["obs"]), torch.from_numpy(g["act"]))
    assert torch.allclose(logp, torch.from_numpy(g["logp"]), atol=1e-6)
    assert torch.allclose(val, torch.from_numpy(g["value"]), atol=1e-6)
    bad = {k[2:]: torch.from_numpy(g[k]) for k in g.files if k.startswith("w_actor")}
    torch.save(bad, path)
    with pytest.raises(RuntimeError):                       # strict: the critic is missing
        load_checkpoint(path)


def test_summary_of_hand_made_records():
    res = EvalResult(make_records(ret=[10.5, -2.0, 40.0, 1.5], length=[1000, 20, 700, 1000], gates=[12, 1, 30, 3],
                                  laps=[0, 0, 2, 0], first_lap=[-1, -1, 350, -1], outcome=[2, 1, 1, 2]))
    s = res.sums()
    assert s.dtype == torch.float64
    assert s.tolist() == [4.0, 50.0, 10.5 ** 2 + 4.0 + 1600.0 + 2.25, 2720.0, 2.0, 2.0, 1.0, 2.0, 350.0, 46.0]
    m = res.summary()
    assert m["episodes"] == 4 and m["mean_return"] == 12.5
    assert math.isclose(m["std_return"], math.sqrt((10.5 ** 2 + 4.0 + 1600.0 + 2.25) / 4 - 12.5 ** 2))
    assert m["avg_reward"] == 50.0 / 2720.0 and m["mean_length"] == 680.0
    assert (m["crash_rate"], m["truncation_rate"], m["lap_rate"], m["mean_laps"]) == (0.5, 0.5, 0.25, 0.5)
    assert (m["mean_first_lap_steps"], m["mean_gates"]) == (350.0, 11.5)
    none = EvalResult(make_records([1.0], [5], [0], [0], [-1], [1])).summary()
    assert none["mean_first_lap_steps"] is None and none["lap_rate"] == 0.0
    assert EvalResult(torch.zeros((0, 8), dtype=torch.int32)).summary() == {"episodes": 0}
    with pytest.raises(ValueError):
        EvalResult(torch.zeros((3, 4), dtype=torch.int32))


def test_sums_of_shards_add_up():
    rng = np.random.default_rng(5)
    n = 57
    laps = rng.integers(0, 3, n)
    cols = dict(ret=rng.integers(-300, 300, n) / 8.0, length=rng.integers(1, 1001, n), gates=rng.integers(0, 60, n),
                laps=laps, first_lap=np.where(laps > 0, rng.integers(100, 1000, n), -1), outcome=rng.integers(1, 3, n))
    whole = make_records(**{k: v.tolist() for k, v in cols.items()})
    a, b = EvalResult(whole[:20]), EvalResult(whole[20:])
    assert torch.equal(a.sums() + b.sums(), EvalResult(whole).sums())      # dyadic returns: exact in any order
    assert set(EvalResult(whole).summary()) >= {"mean_return", "crash_rate", "lap_rate", "mean_gates"}
    assert len(SUM_FIELDS) == 10


def test_cli_and_train_flags():
    a = parse_args(["--checkpoint", "m.dat"])
    assert (a.track, a.episodes, a.greedy, a.seed, a.json) == ("big_track", 65536, False, 0, None)
    from ppo_car_b200.train_ppo import parse_args as train_args

    t = train_args([])
    assert (t.eval_every, t.eval_episodes, t.eval_greedy) == (0, 1024, False)


# ---------------------------------------------------------------------------------------------------- GPU
def _fresh_actor(seed=0):
    torch.manual_seed(seed)
    return ActorCritic(18, 9).actor.cuda()


@pytest.fixture(scope="module")
def trained_actor(tmp_path_factory):
    """The README run's shape (24 envs x 1024 steps x 200 epochs on big_track, fused rollout and update),
    read back from its model.dat."""
    from ppo_car_b200.train_ppo import parse_args as train_args, train

    d = tmp_path_factory.mktemp("ckpt")
    train(train_args(["--track", "big_track", "--n-envs", "24", "--fused-rollout", "--fused-update",
                      "--checkpoint-dir", str(d), "--run-name", "readme"]))
    return load_checkpoint(str(d / "readme" / "model.dat")).actor.cuda()


def _env(track, n=1):
    from ppo_car_b200 import VecCarEnv, builtin_track

    return VecCarEnv(n, track if os.path.exists(track) else builtin_track(track), device="cuda:0")


def replay(track, res: EvalResult, n: int):
    """Play the first n traced episodes again through VecCarEnv.step(numpy) (float64 rewards, debug info).
    Returns the replayed records and the (observation, action, uniform) of every live step."""
    from ppo_car_b200 import VecCarEnv, builtin_track

    env = VecCarEnv(n, track if os.path.exists(track) else builtin_track(track), device="cuda:0", reward_scaling=1.0,
                    debug_info=True, copy_outputs=True)
    obs = env.reset()[0].cpu().numpy().copy()
    acts = res.trace_actions[:n].cpu().numpy()
    us = None if res.trace_u is None else res.trace_u[:n].cpu().numpy()
    done = np.zeros(n, bool)
    ret = np.zeros(n)
    length, gates, laps, first, outcome = (np.zeros(n, np.int64), np.zeros(n, np.int64), np.zeros(n, np.int64),
                                           np.full(n, -1, np.int64), np.zeros(n, np.int64))
    rows_obs, rows_act, rows_u = [], [], []
    for t in range(TIME_LIMIT):
        live = ~done
        if not live.any():
            break
        a = acts[:, t].astype(np.int64)
        assert (a[live] < 9).all(), "a live episode has no traced action"
        a[~live] = 8
        rows_obs.append(obs[live]); rows_act.append(a[live])
        if us is not None:
            rows_u.append(us[live, t])
        o, r, te, tr, info = env.step(a)
        ret[live] = ret[live] + r[live]
        lap = live & ((info["events"] & 2) != 0)
        laps += lap
        first = np.where(lap & (first < 0), info["time_passed"], first)
        ended = live & (te | tr)
        length[ended] = info["time_passed"][ended]
        gates[ended] = info["gates_passed"][ended]
        outcome[ended] = np.where(te[ended], 1, 2)
        done |= ended
        obs = o
    assert done.all()
    for j in range(n):                                        # nothing written past an episode's end
        assert (acts[j, length[j]:] == 255).all()
        if us is not None:
            assert np.isnan(us[j, length[j]:]).all() and not np.isnan(us[j, :length[j]]).any()
    rep = dict(ret=ret, length=length, gates=gates, laps=laps, first_lap=first, outcome=outcome)
    return rep, np.concatenate(rows_obs), np.concatenate(rows_act), (np.concatenate(rows_u) if rows_u else None)


def check_records(res: EvalResult, rep: dict, n: int):
    assert np.array_equal(res.ret[:n].cpu().numpy(), rep["ret"])          # bit for bit: in-order float64 sums
    for k in ("length", "gates", "laps", "first_lap", "outcome"):
        assert np.array_equal(getattr(res, k)[:n].cpu().numpy(), rep[k]), k


def torch_probs(actor, obs):
    with torch.no_grad():
        logits = actor.cpu()(torch.from_numpy(obs))
    actor.cuda()
    return logits, torch.softmax(logits, dim=-1)


@pytest.mark.gpu
@pytest.mark.parametrize("which", ["fresh", "trained"])
@pytest.mark.parametrize("track", ["track", "big_track"])
def test_sampled_episodes_replay_bit_for_bit(request, which, track):
    from ppo_car_b200 import evaluate_policy

    actor = _fresh_actor(1) if which == "fresh" else request.getfixturevalue("trained_actor")
    n_tr = 64
    res = evaluate_policy(_env(track), actor, 4096, greedy=False, seed=11, trace=n_tr)
    torch.cuda.synchronize()
    out = res.outcome.cpu().numpy()
    length = res.length.cpu().numpy()
    assert set(np.unique(out)) <= {1, 2} and length.min() >= 1 and length.max() <= TIME_LIMIT
    assert (length[out == 2] == TIME_LIMIT).all()                      # a crash on step 1000 is still a crash
    rep, obs, act, u = replay(track, res, n_tr)
    check_records(res, rep, n_tr)
    # every action lies in the interval of the torch float32 softmax CDF that its uniform falls into
    _, p = torch_probs(actor, obs)
    cdf = torch.cumsum(p, dim=-1)[:, :-1].numpy()
    a_torch = np.minimum((cdf <= u[:, None]).sum(1), 8)
    near = np.abs(cdf - u[:, None]).min(1) < 1e-5
    assert ((a_torch == act) | near).all()
    assert near.sum() <= max(2, 0.002 * len(act)), (near.sum(), len(act))
    if which == "trained" and track == "big_track":
        assert res.laps.sum().item() > 0 and rep["laps"].sum() > 0        # laps and first_lap are exercised


@pytest.mark.gpu
def test_greedy_episodes_are_identical_and_argmax(trained_actor):
    from ppo_car_b200 import evaluate_policy

    env = _env("big_track")
    many = evaluate_policy(env, trained_actor, 2000, greedy=True, seed=3, trace=4)
    one = evaluate_policy(env, trained_actor, 1, greedy=True, seed=99, episode0=12345)
    torch.cuda.synchronize()
    assert many.trace_u is None
    assert torch.equal(many.records, one.records.expand(2000, 8))
    assert (many.trace_actions == many.trace_actions[0]).all()
    rep, obs, act, _ = replay("big_track", many, 4)
    check_records(many, rep, 4)
    logits, _ = torch_probs(trained_actor, obs)
    top2 = torch.topk(logits, 2, dim=-1).values
    clear = (top2[:, 0] - top2[:, 1] > 1e-5).numpy()
    assert clear.mean() > 0.99
    assert np.array_equal(logits.argmax(-1).numpy()[clear], act[clear])


@pytest.mark.gpu
@pytest.mark.parametrize("greedy", [False, True])
def test_records_do_not_depend_on_the_split_or_the_grid(monkeypatch, greedy):
    from ppo_car_b200 import evaluate_policy

    env, actor = _env("big_track"), _fresh_actor(2)
    N, k = 3000, 1234
    whole = evaluate_policy(env, actor, N, greedy=greedy, seed=5)
    a = evaluate_policy(env, actor, k, greedy=greedy, seed=5)
    b = evaluate_policy(env, actor, N - k, greedy=greedy, seed=5, episode0=k)
    monkeypatch.setenv("CARENV_EVAL_CTAS", "1")             # 128 slots play 1,000 episodes: the refill path
    capped = evaluate_policy(env, actor, 1000, greedy=greedy, seed=5)
    monkeypatch.delenv("CARENV_EVAL_CTAS")
    torch.cuda.synchronize()
    assert torch.equal(torch.cat([a.records, b.records]), whole.records)
    assert torch.equal(capped.records, whole.records[:1000])
    if not greedy:
        other = evaluate_policy(env, actor, 1000, greedy=False, seed=6)
        assert not torch.equal(other.records, whole.records[:1000])


@pytest.mark.gpu
def test_start_inside_the_wall(tmp_path):
    from tests.synth_tracks import near_wall_track

    from ppo_car_b200 import evaluate_policy

    path = near_wall_track(str(tmp_path / "near_wall.json"))
    n = 500
    res = evaluate_policy(_env(path), _fresh_actor(3), n, seed=1, trace=n)
    torch.cuda.synchronize()
    assert (res.length == 1).all() and (res.outcome == 1).all() and (res.laps == 0).all()
    a0 = res.trace_actions[:, 0].cpu().numpy()
    expect = np.where(np.isin(a0, THRUST_ACTIONS), 0.01, 0.0) - 3.0
    assert np.array_equal(res.ret.cpu().numpy(), expect)
    assert (res.trace_actions[:, 1:] == 255).all()


@pytest.mark.gpu
def test_bad_arguments_with_a_live_handle():
    L = _lib.lib()
    env = _env("track")
    w = torch.zeros(256 * 18, device="cuda")
    rec = torch.zeros((4, 8), dtype=torch.int32, device="cuda")
    p = [C.c_void_p(w.data_ptr())] * 4
    r = C.c_void_p(rec.data_ptr())
    assert L.carenv_policy_eval(env._handle, None, *p[1:], 4, 0, 0, 0, r, 0, None, None, None) == -1
    assert L.carenv_policy_eval(env._handle, *p, -1, 0, 0, 0, r, 0, None, None, None) == -1
    assert L.carenv_policy_eval(env._handle, *p, 4, 0, 0, 0, None, 0, None, None, None) == -1
    assert L.carenv_policy_eval(env._handle, *p, 4, 0, 0, 0, r, 2, None, None, None) == -1
    assert b"trace" in L.carenv_last_error()
    assert L.carenv_policy_eval(env._handle, *p, 0, 0, 0, 0, r, 0, None, None, None) == 0
    from ppo_car_b200 import evaluate_policy

    with pytest.raises(ValueError):
        evaluate_policy(env, ActorCritic(18, 9).actor, 4)                  # parameters on the CPU
    with pytest.raises(ValueError):
        evaluate_policy(env, torch.nn.Sequential(torch.nn.Linear(18, 64), torch.nn.ReLU(),
                                                 torch.nn.Linear(64, 9)).cuda(), 4)


@pytest.mark.gpu
def test_train_ppo_eval_every():
    from ppo_car_b200.train_ppo import parse_args as train_args, train

    base = ["--track", "track", "--n-envs", "32", "--n-epochs", "4", "--n-steps", "64", "--fused-rollout"]
    hist = train(train_args(base + ["--eval-every", "2", "--eval-episodes", "256"]))
    assert ["eval" in h for h in hist] == [False, True, False, True]
    ev = hist[1]["eval"]
    assert ev["episodes"] == 256 and 0.0 <= ev["crash_rate"] <= 1.0
    assert math.isclose(ev["crash_rate"] + ev["truncation_rate"], 1.0)
    json.dumps(hist)
    assert not any("eval" in h for h in train(train_args(base)))


@pytest.mark.gpu
@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_torchrun_cli_equals_one_rank(tmp_path):
    from ppo_car_b200.evaluate import main

    ckpt = str(tmp_path / "model.dat")
    torch.manual_seed(4)
    torch.save(ActorCritic(18, 9).state_dict(), ckpt)
    args = ["--checkpoint", ckpt, "--track", "track", "--episodes", "5000", "--seed", "2"]
    one = main(args)
    out = str(tmp_path / "two.json")
    subprocess.check_call([sys.executable, "-m", "torch.distributed.run", "--nproc-per-node", "2", "-m",
                           "ppo_car_b200.evaluate", *args, "--json", out], cwd=ROOT)
    two = json.load(open(out))
    assert one.keys() == two.keys()
    for key, v in one.items():
        if isinstance(v, float):
            assert math.isclose(v, two[key], rel_tol=1e-12, abs_tol=1e-12), key
        else:
            assert v == two[key], key
