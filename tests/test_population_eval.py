"""Member-batched policy evaluation (ppo_car_b200.evaluate.evaluate_population, C ABI carenv_policy_eval_pop,
k_policy_eval<U, true> in csrc/policy_eval.cuh).

GPU:
  * every member's records and traces against evaluate_policy of that member alone with its seed, bit for bit, on
    tracks that launch each population instantiation (U = 4, 2, 1) and on the start-inside-the-wall track;
  * a member's records do not depend on the other members, their order, P, the split of the ids over calls, the grid
    (CARENV_EVAL_CTAS) or on P exceeding one wave of CTAs;
  * train_population --eval-every against evaluate_policy of each member's weights; the multi-checkpoint CLI against
    the single-checkpoint CLI, and under torchrun against one rank.
CPU: the C ABI's null-handle refusal, the Python argument checks, the CLI's parsing and refusals.
"""
import ctypes as C
import json
import math
import os
import subprocess
import sys
from types import SimpleNamespace

import pytest
import torch

import ppo_car_b200
from ppo_car_b200 import _lib
from ppo_car_b200 import evaluate as evalmod
from ppo_car_b200 import population as popmod
from ppo_car_b200.evaluate import evaluate_policy, evaluate_population
from ppo_car_b200.train_ppo import ActorCritic
from tests.test_fused_rollout_reference import track_layout, track_path

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SEEDS = [3, 2 ** 32 + 5, 11, 2 ** 40 + 7, 0, 19, 2 ** 33 + 1]          # distinct, some with a non-zero high word


def eval_unroll(layout, opts):
    """The instantiation carenv_policy_eval / _pop launch (eval_unroll in policy_eval.cuh): U = 4, 2 or 1."""
    U = 1 if opts.get("force_generic") else layout.unroll4
    cap = opts.get("max_unroll", 0)
    if cap > 0 and U > cap:
        U = cap if U % cap == 0 else 1
    return U


# track, options, P, episodes per member, greedy, traced episodes, episode0
CASES = [
    ("big_track", {}, 7, 4097, False, 40, 0),
    ("big_track", {}, 3, 1000, True, 8, 2 ** 32 - 300),                 # ids cross 2^32
    ("big_track", {"force_generic": 1}, 1, 1000, False, 16, 0),
    ("track", {"max_unroll": 2}, 7, 33, True, 33, 5),
    ("ring10_6", {}, 3, 33, False, 33, 0),
    ("ring10_6", {}, 1, 4097, True, 4, 0),
    ("ring7_5", {}, 7, 1, False, 1, 0),
    ("ring7_5", {}, 3, 1000, False, 1000, 77),
    ("near_wall", {}, 3, 1000, False, 50, 0),
]
CASE_IDS = [f"{t}-{'-'.join(f'{k}{v}' for k, v in o.items()) or 'default'}-P{P}-n{n}-{'greedy' if g else 'sampled'}"
            for t, o, P, n, g, _, _ in CASES]


@pytest.fixture(scope="module")
def tracks(tmp_path_factory):
    d = str(tmp_path_factory.mktemp("tracks"))
    cache = {}
    return lambda name: cache.setdefault(name, track_path(name, d))


# ---- CPU ---------------------------------------------------------------------------------------------------------
def test_cases_reach_every_population_instantiation(tracks):
    reached = {eval_unroll(track_layout(tracks(t)), o) for t, o, *_ in CASES}
    assert reached == {4, 2, 1}
    assert {P for _, _, P, *_ in CASES} == {1, 3, 7} and {n for _, _, _, n, *_ in CASES} == {1, 33, 1000, 4097}
    assert {g for *_, g, _, _ in CASES} == {False, True}


def test_null_handle_is_an_error():
    L = _lib.lib()
    rec = torch.zeros((2, 4, 8), dtype=torch.int32)
    w = torch.zeros(2 * 256 * 18)
    s = torch.zeros(2, dtype=torch.int64)
    p = [C.c_void_p(w.data_ptr())] * 4
    assert L.carenv_policy_eval_pop(None, 2, *p, 4, 0, 0, C.c_void_p(s.data_ptr()), C.c_void_p(rec.data_ptr()), 0,
                                    None, None, None) == -1
    assert b"handle" in L.carenv_last_error()


def _stacked(P, device="cpu"):
    return [torch.zeros((P, 256, 18), device=device), torch.zeros((P, 256), device=device),
            torch.zeros((P, 9, 256), device=device), torch.zeros((P, 9), device=device)]


def test_python_argument_checks():
    env = SimpleNamespace(device=torch.device("cpu"))           # every check below comes before the library call
    good = _stacked(3)
    bad_shapes = [good[:3], [good[0][0]] + good[1:], good[:1] + [torch.zeros(2, 256)] + good[2:],
                  good[:2] + [torch.zeros((3, 8, 256))] + good[3:], _stacked(0)]
    for params in bad_shapes:
        with pytest.raises(ValueError, match="stacked|members"):
            evaluate_population(env, params, 4)
    with pytest.raises(ValueError, match="float32"):
        evaluate_population(env, [good[0].double()] + good[1:], 4)
    with pytest.raises(ValueError, match="float32"):
        evaluate_population(env, [torch.zeros((3, 18, 256)).transpose(1, 2)] + good[1:], 4)
    with pytest.raises(ValueError, match="float32"):
        evaluate_population(SimpleNamespace(device=torch.device("cuda", 0)), good, 4)
    with pytest.raises(ValueError, match="3 seeds"):
        evaluate_population(env, good, 4, seeds=[1, 2])
    with pytest.raises(ValueError, match=">= 0"):
        evaluate_population(env, good, -1)
    with pytest.raises(ValueError, match=">= 0"):
        evaluate_population(env, good, 4, trace=-1)
    with pytest.raises(ValueError, match="64 bits"):
        evaluate_population(env, good, 4, episode0=2 ** 64)
    multi = ppo_car_b200.MultiTrackVecEnv.__new__(ppo_car_b200.MultiTrackVecEnv)
    with pytest.raises(ValueError, match="one track"):
        evaluate_population(multi, good, 4)


def test_checkpoint_list_and_cli_refusals(tmp_path, monkeypatch):
    assert evalmod.checkpoint_list("a.dat") == ["a.dat"]
    assert evalmod.checkpoint_list("a.dat,b/c.dat, d.dat") == ["a.dat", "b/c.dat", "d.dat"]
    odd = tmp_path / "x,y.dat"
    odd.write_bytes(b"")
    assert evalmod.checkpoint_list(str(odd)) == [str(odd)]          # an existing file keeps its comma
    with pytest.raises(SystemExit, match="empty entry"):
        evalmod.checkpoint_list("a.dat,,b.dat")
    assert evalmod.parse_args(["--checkpoint", "a.dat,b.dat"]).checkpoint == "a.dat,b.dat"
    monkeypatch.setattr(torch.cuda, "set_device", lambda *a: pytest.fail("device work before the refusal"))
    with pytest.raises(SystemExit, match="one track"):
        evalmod.main(["--checkpoint", "a.dat,b.dat", "--track", "big_track,track"])


# ---- GPU ---------------------------------------------------------------------------------------------------------
def _actors(P, seed0=0):
    """P distinct actors on the GPU; every third one nearly always stands still (action 8), so its sampled episodes
    run into the 1000-step limit while the others crash early."""
    out = []
    for p in range(P):
        torch.manual_seed(seed0 + p)
        a = ActorCritic(18, 9).actor.cuda()
        with torch.no_grad():
            if p % 3 == 2:
                a[2].weight.mul_(0.1)
                a[2].bias.copy_(torch.tensor([0.0] * 8 + [20.0]))
            else:
                a[2].weight.mul_(4.0)
                a[2].bias.copy_(torch.linspace(-1, 1, 9))
        out.append(a)
    return out


def _stack(actors):
    return [torch.stack([getattr(a[i], k).detach() for a in actors]).contiguous()
            for i, k in ((0, "weight"), (0, "bias"), (2, "weight"), (2, "bias"))]


def _env(path, opts=None):
    env = ppo_car_b200.VecCarEnv(1, path, device="cuda:0")
    for k, v in (opts or {}).items():
        env.set_option(k, v)
    return env


def _bits_equal(a, b):
    if a is None or b is None:
        return a is None and b is None
    if a.dtype == torch.float32:
        a, b = a.view(torch.int32), b.view(torch.int32)             # the untouched entries are NaN
    return a.shape == b.shape and torch.equal(a, b)


@pytest.mark.gpu
@pytest.mark.parametrize("track, opts, P, n, greedy, trace, episode0", CASES, ids=CASE_IDS)
def test_members_equal_single_evaluations(tracks, track, opts, P, n, greedy, trace, episode0):
    env = _env(tracks(track), opts)
    actors = _actors(P, seed0=10 * P)
    seeds = SEEDS[:P]
    pop = evaluate_population(env, _stack(actors), n, greedy=greedy, seeds=seeds, episode0=episode0, trace=trace)
    single = [evaluate_policy(env, a, n, greedy=greedy, seed=s, episode0=episode0, trace=trace)
              for a, s in zip(actors, seeds)]
    torch.cuda.synchronize()
    assert len(pop) == P
    base = pop[0].records
    for p in range(P):
        assert pop[p].records.data_ptr() == base.data_ptr() + p * n * 32       # views of one [P, n, 8] tensor
        assert torch.equal(pop[p].records, single[p].records), p
        assert _bits_equal(pop[p].trace_actions, single[p].trace_actions), p
        assert _bits_equal(pop[p].trace_u, single[p].trace_u), p
        assert pop[p].summary() == single[p].summary(), p
    out = torch.cat([r.outcome for r in pop])
    assert set(out.unique().tolist()) <= {1, 2}
    if track == "near_wall":
        assert all((r.length == 1).all() for r in pop)
    if track == "big_track" and n >= 1000 and not greedy and P >= 3:
        assert (pop[2].outcome == 2).float().mean() > 0.5 and (pop[0].outcome == 1).any()   # long and short episodes
    env.close()


@pytest.mark.gpu
@pytest.mark.parametrize("greedy", [False, True])
def test_members_are_independent(tracks, monkeypatch, greedy):
    env = _env(tracks("big_track"))
    actors = _actors(5, seed0=40)
    seeds = [7, 2 ** 35 + 1, 9, 0, 2 ** 63 + 3]
    n, k = 3000, 1234
    whole = evaluate_population(env, _stack(actors), n, greedy=greedy, seeds=seeds)
    rev = evaluate_population(env, _stack(actors[::-1]), n, greedy=greedy, seeds=seeds[::-1])
    alone = evaluate_population(env, _stack(actors[1:2]), n, greedy=greedy, seeds=seeds[1:2])
    a = evaluate_population(env, _stack(actors), k, greedy=greedy, seeds=seeds)
    b = evaluate_population(env, _stack(actors), n - k, greedy=greedy, seeds=seeds, episode0=k)
    twins = evaluate_population(env, _stack([actors[3], actors[0], actors[3]]), n, greedy=greedy,
                                seeds=[seeds[3], 5, seeds[3]])
    monkeypatch.setenv("CARENV_EVAL_CTAS", "1")                 # 128 slots per member play 1,000 episodes each
    capped = evaluate_population(env, _stack(actors), 1000, greedy=greedy, seeds=seeds)
    monkeypatch.delenv("CARENV_EVAL_CTAS")
    torch.cuda.synchronize()
    for p in range(5):
        assert torch.equal(rev[4 - p].records, whole[p].records), p
        assert torch.equal(torch.cat([a[p].records, b[p].records]), whole[p].records), p
        assert torch.equal(capped[p].records, whole[p].records[:1000]), p
    assert torch.equal(alone[0].records, whole[1].records)
    assert torch.equal(twins[0].records, whole[3].records) and torch.equal(twins[2].records, whole[3].records)
    if not greedy:                                               # the seed matters: same weights, another seed
        other = evaluate_population(env, _stack(actors[:1]), n, greedy=False, seeds=[seeds[0] + 1])
        assert not torch.equal(other[0].records, whole[0].records)
    env.close()


@pytest.mark.gpu
def test_more_members_than_one_wave(tracks):
    """700 members x 2 episodes: 700 CTAs of one member each, more than the 592 resident at 4 per SM on 148 SMs."""
    env = _env(tracks("big_track"))
    distinct = _actors(7, seed0=70)
    P = 700
    actors = [distinct[p % 7] for p in range(P)]
    seeds = [1000 + p for p in range(P)]
    pop = evaluate_population(env, _stack(actors), 2, seeds=seeds, trace=2)
    for p in list(range(0, P, 41)) + [P - 1]:
        single = evaluate_policy(env, actors[p], 2, seed=seeds[p], trace=2)
        assert torch.equal(pop[p].records, single.records), p
        assert _bits_equal(pop[p].trace_u, single.trace_u), p
    out, length = torch.stack([r.outcome for r in pop]), torch.stack([r.length for r in pop])
    assert set(out.unique().tolist()) <= {1, 2} and 1 <= int(length.min()) and int(length.max()) <= 1000
    env.close()


@pytest.mark.gpu
def test_bad_arguments_with_a_live_handle(tracks, tmp_path):
    from tests.synth_tracks import ring_track

    L = _lib.lib()
    env = _env(tracks("track"))
    p = lambda t: C.c_void_p(t.data_ptr())
    w = [p(t) for t in _stacked(2, "cuda")]
    s = torch.zeros(2, dtype=torch.int64, device="cuda")
    rec = torch.zeros((2, 4, 8), dtype=torch.int32, device="cuda")
    call = lambda P, n, seeds, records, n_trace=0: L.carenv_policy_eval_pop(env._handle, P, *w, n, 0, 0, seeds,
                                                                            records, n_trace, None, None, None)
    assert call(0, 4, p(s), p(rec)) == -1 and b"n_members" in L.carenv_last_error()
    assert call(65536, 4, p(s), p(rec)) == -1 and b"n_members" in L.carenv_last_error()
    assert call(2, -1, p(s), p(rec)) == -1
    assert call(2, 4, None, p(rec)) == -1 and b"null" in L.carenv_last_error()
    assert call(2, 4, p(s), None) == -1 and b"null" in L.carenv_last_error()
    assert L.carenv_policy_eval_pop(env._handle, 2, None, *w[1:], 4, 0, 0, p(s), p(rec), 0, None, None, None) == -1
    assert call(2, 4, p(s), p(rec), n_trace=-1) == -1
    assert call(2, 4, p(s), p(rec), n_trace=2) == -1 and b"trace" in L.carenv_last_error()
    assert call(2, 0, p(s), p(rec)) == 0
    big = _env(ring_track(str(tmp_path / "ring_140.json"), 100, 40, wobble=0.03))
    assert L.carenv_policy_eval_pop(big._handle, 2, *w, 4, 0, 0, p(s), p(rec), 0, None, None, None) == -2
    assert b"128 wall segments" in L.carenv_last_error()
    with pytest.raises(ppo_car_b200.CarEnvError, match=r"\(code -2\)"):
        evaluate_population(big, _stacked(2, "cuda"), 4)
    empty = evaluate_population(env, _stacked(2, "cuda"), 0, trace=3)
    assert [tuple(r.records.shape) for r in empty] == [(0, 8), (0, 8)] and empty[0].summary() == {"episodes": 0}
    big.close()
    env.close()


@pytest.mark.gpu
def test_train_population_eval_equals_single_evaluations(tmp_path):
    args = popmod.parse_args(["--track", "big_track", "--n-envs", "8", "--n-epochs", "2", "--n-steps", "64",
                              "--batch-size", "64", "--seeds", "4,2-3", "--learning-rate", "3e-4,1e-3",
                              "--eval-every", "2", "--eval-episodes", "300", "--checkpoint-dir", str(tmp_path),
                              "--run-name", "sweep"])
    out = popmod.train_population(args)
    hist, final = out["history"], out["final"]
    assert [("eval" in r) for r in hist] == [False] * 6 + [True] * 6
    env = ppo_car_b200.VecCarEnv(1, ppo_car_b200.builtin_track("big_track"), device="cuda:0")
    for r in hist[6:]:
        # epoch 2 is the last one, so the member's model.dat holds the weights its evaluation saw
        net = evalmod.load_checkpoint(str(tmp_path / "sweep" / f"member_{r['member']}" / "model.dat"))
        want = evaluate_policy(env, net.actor.cuda(), 300, seed=r["seed"]).summary()
        assert r["eval"] == want, r["member"]
        assert final[r["member"]]["eval_return"] == want["mean_return"]
    assert len({r["eval"]["mean_return"] for r in hist[6:]}) == 6     # six different members
    env.close()


def _save_actors(tmp_path, n):
    paths = []
    for i in range(n):
        torch.manual_seed(20 + i)
        path = str(tmp_path / f"m{i}.dat")
        torch.save(ActorCritic(18, 9).state_dict(), path)
        paths.append(path)
    return paths


@pytest.mark.gpu
@pytest.mark.parametrize("greedy", [False, True])
def test_cli_several_checkpoints_equal_single_runs(tmp_path, greedy):
    paths = _save_actors(tmp_path, 3)
    common = ["--track", "track", "--episodes", "700", "--seed", "2"] + (["--greedy"] if greedy else [])
    both = evalmod.main(["--checkpoint", ",".join(paths), *common, "--json", str(tmp_path / "all.json")])
    assert list(both) == ["checkpoints"] and json.load(open(tmp_path / "all.json")) == both
    for entry, path in zip(both["checkpoints"], paths):
        assert entry == evalmod.main(["--checkpoint", path, *common])


@pytest.mark.gpu
@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_cli_several_checkpoints_torchrun_equals_one_rank(tmp_path):
    paths = _save_actors(tmp_path, 3)
    args = ["--checkpoint", ",".join(paths), "--track", "track", "--episodes", "5000", "--seed", "2"]
    one = evalmod.main(args)
    out = str(tmp_path / "two.json")
    subprocess.check_call([sys.executable, "-m", "torch.distributed.run", "--nproc-per-node", "2", "-m",
                           "ppo_car_b200.evaluate", *args, "--json", out], cwd=ROOT)
    two = json.load(open(out))
    assert len(one["checkpoints"]) == len(two["checkpoints"]) == 3
    for a, b in zip(one["checkpoints"], two["checkpoints"]):
        assert a.keys() == b.keys()
        for key, v in a.items():
            if isinstance(v, float):
                assert math.isclose(v, b[key], rel_tol=1e-12, abs_tol=1e-12), key
            else:
                assert v == b[key], key
