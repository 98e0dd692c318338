"""Population-based training of a population (ppo_car_b200.pbt, Population.copy_members, train_population --pbt-*).

CPU: pbt_decisions (how many members are replaced, from where, tie order, seeding, factors), the --pbt-* refusals
before any device work, and the unchanged parse without --pbt-* flags.
GPU:
  * copy_members: every destination row of every parameter, moment, step-count and hyperparameter tensor equals its
    source row bit for bit, explored values are the float32 product with the clamps, other members are untouched;
  * a README-shape run with --pbt-every 2: members never replaced keep the records and checkpoints of the same run
    without PBT; two identical runs give identical records, lineage and checkpoints; parents come from the top
    fraction of the round's fitness; checkpoints load into evaluate;
  * under torchrun on two GPUs the run equals the one-rank run bit for bit.
"""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from ppo_car_b200 import pbt
from ppo_car_b200 import population as popmod
from ppo_car_b200.pbt import parse_explore, pbt_decisions
from ppo_car_b200.population import HPARAM_ATTRS, HPARAMS, Population

gpu = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ---- CPU: decisions ----------------------------------------------------------------------------------------------
def _rank(fitness):
    return sorted(range(len(fitness)), key=lambda i: (-fitness[i], i))


@pytest.mark.parametrize("P, fraction", [(4, 0.25), (8, 0.25), (9, 0.5), (10, 0.3), (32, 0.25), (33, 0.5), (2, 0.5)])
def test_decisions_replace_the_bottom_m_from_the_top_m(P, fraction):
    fitness = torch.randn(P, generator=torch.Generator().manual_seed(P)).tolist()
    out = pbt_decisions(fitness, fraction, ["learning_rate", "ent_coef"], torch.Generator().manual_seed(0))
    m = int(P * fraction)
    order = _rank(fitness)
    assert len(out) == m
    assert [d for d, _, _ in out] == sorted(order[P - m:])          # destinations ascending, the bottom m
    assert all(s in order[:m] for _, s, _ in out)
    assert not {d for d, _, _ in out} & {s for _, s, _ in out}


def test_ties_go_to_the_lower_index():
    out = pbt_decisions([1.0] * 8, 0.25, [], torch.Generator().manual_seed(3))
    assert [d for d, _, _ in out] == [6, 7] and all(s in (0, 1) for _, s, _ in out)
    out = pbt_decisions([0.0, 5.0, 5.0, 0.0, 1.0, 0.0], 0.5, [], torch.Generator().manual_seed(3))
    # ranked 1, 2, 4, 0, 3, 5: the zeros at 0, 3, 5 tie and 0 ranks first, so the bottom three are 0, 3, 5
    assert [d for d, _, _ in out] == [0, 3, 5] and all(s in (1, 2, 4) for _, s, _ in out)


def test_decisions_follow_the_seed():
    fitness = torch.randn(64, generator=torch.Generator().manual_seed(1)).tolist()
    run = lambda seed: pbt_decisions(fitness, 0.5, HPARAMS, torch.Generator().manual_seed(seed))
    assert run(7) == run(7)
    assert run(7) != run(8)
    g = torch.Generator().manual_seed(7)                      # a second round continues the stream
    first, second = pbt_decisions(fitness, 0.5, HPARAMS, g), pbt_decisions(fitness, 0.5, HPARAMS, g)
    assert first == run(7) and second != first


def test_draw_order_is_destination_source_then_factors_in_hparams_order():
    fitness = list(range(8, 0, -1))                           # member i ranks i: top 0, 1; bottom 6, 7
    g = torch.Generator().manual_seed(11)
    out = pbt_decisions(fitness, 0.25, ["ent_coef", "learning_rate"], g)
    g = torch.Generator().manual_seed(11)
    draw = lambda n: int(torch.randint(0, n, (1,), generator=g))
    expect = []
    for d in (6, 7):
        s = (0, 1)[draw(2)]
        expect.append((d, s, {"learning_rate": pbt.FACTORS[draw(2)], "ent_coef": pbt.FACTORS[draw(2)]}))
    assert out == expect and [list(f) for _, _, f in out] == [["learning_rate", "ent_coef"]] * 2


def test_factors_are_only_for_explored_names_and_only_08_or_12():
    fitness = torch.randn(128, generator=torch.Generator().manual_seed(2)).tolist()
    for explore in ([], ["clip_ratio"], ["learning_rate", "ent_coef"], list(HPARAMS)):
        out = pbt_decisions(fitness, 0.5, explore, torch.Generator().manual_seed(5))
        assert all(set(f) == set(explore) for _, _, f in out)
        vals = [v for _, _, f in out for v in f.values()]
        assert set(vals) <= {0.8, 1.2}
        if explore:
            assert set(vals) == {0.8, 1.2}


def test_parse_explore():
    assert parse_explore("ent_coef,learning_rate") == ["learning_rate", "ent_coef"]
    assert parse_explore("") == []
    with pytest.raises(ValueError, match="gamma"):
        parse_explore("learning_rate,gamma")


# ---- CPU: command line -------------------------------------------------------------------------------------------
@pytest.mark.parametrize("argv, words", [
    (["--seeds", "0-7", "--pbt-every", "-1"], "--pbt-every"),
    (["--seeds", "0-7", "--pbt-every", "2", "--pbt-fraction", "0"], "--pbt-fraction"),
    (["--seeds", "0-7", "--pbt-every", "2", "--pbt-fraction", "0.6"], "--pbt-fraction"),
    (["--seeds", "0-2", "--pbt-every", "2"], "replaces none"),                  # floor(3 * 0.25) = 0
    (["--seeds", "0-7", "--pbt-every", "2", "--pbt-fraction", "0.1"], "replaces none"),
    (["--seeds", "0-7", "--pbt-every", "2", "--pbt-explore", "learning_rate,gamma"], "gamma"),
    (["--seeds", "0-7", "--pbt-every", "2", "--pbt-seed", "-1"], "--pbt-seed"),
    (["--seeds", "0-7", "--pbt-every", "2", "--eval-episodes", "0"], "--eval-episodes"),
])
def test_pbt_refusals_come_before_any_device_work(argv, words, monkeypatch):
    monkeypatch.setattr(torch.cuda, "set_device", lambda *a: pytest.fail("device work before the refusal"))
    with pytest.raises(SystemExit, match=words):
        popmod.train_population(popmod.parse_args(argv))


def test_pbt_needs_a_member_per_rank(monkeypatch):
    monkeypatch.setattr(torch.cuda, "set_device", lambda *a: pytest.fail("device work before the refusal"))
    monkeypatch.setenv("WORLD_SIZE", "8")
    with pytest.raises(SystemExit, match="one member per rank"):
        popmod.train_population(popmod.parse_args(["--seeds", "0-3", "--pbt-every", "2", "--pbt-fraction", "0.5"]))


def test_without_pbt_flags_the_arguments_are_unchanged():
    from ppo_car_b200.train_ppo import parse_args as train_args

    argv = ["--seeds", "0-3", "--learning-rate", "1e-3,3e-4", "--n-envs", "4", "--eval-every", "5"]
    args = popmod.parse_args(argv)
    assert (args.pbt_every, args.pbt_fraction, args.pbt_explore, args.pbt_seed) == (0, 0.25, "learning_rate,ent_coef", 0)
    ref = vars(train_args(["--learning-rate", "1e-3", "--n-envs", "4", "--eval-every", "5"]))
    mine = {k: v for k, v in vars(args).items() if not k.startswith("pbt_")}
    assert mine == {**ref, "seeds": "0-3", **{k + "_list": str(ref[k]) for k in HPARAMS},
                    "learning_rate_list": "1e-3,3e-4"}
    assert popmod.check_args(args) == popmod.expand_grid([0, 1, 2, 3], {"learning_rate": [1e-3, 3e-4]})
    one = popmod.parse_args(["--seeds", "0", "--pbt-fraction", "0.9", "--pbt-explore", "nope"])
    assert len(popmod.check_args(one)[1]) == 1             # the --pbt-* flags are not read while --pbt-every is 0


# ---- GPU: copy_members -------------------------------------------------------------------------------------------
def _snapshot(pop):
    return {"params": [t.clone() for t in pop.params], "exp_avg": pop.exp_avg.clone(),
            "exp_avg_sq": pop.exp_avg_sq.clone(), "step_count": pop.step_count.clone(),
            **{k: getattr(pop, HPARAM_ATTRS[k]).clone() for k in HPARAMS}}


def _rows(snap, p):
    return [t[p] for t in snap["params"]] + [snap["exp_avg"][p], snap["exp_avg_sq"][p], snap["step_count"][p]]


@gpu
def test_copy_members_is_exact():
    dev = torch.device("cuda", 0)
    P = 7
    hp = [dict(learning_rate=1e-4 * (p + 1), learning_rate_decay=0.99 - 0.01 * p, clip_ratio=0.15 + 0.12 * p,
               ent_coef=0.001 * (p + 2), vf_coef=0.5 + 0.1 * p, max_grad_norm=0.7 + p) for p in range(P)]
    pop = Population(list(range(P)), 3, hp, dev)
    g = torch.Generator(device=dev).manual_seed(0)
    with torch.no_grad():                          # a state where every tensor differs per member
        pop.exp_avg.copy_(torch.randn(pop.exp_avg.shape, generator=g, device=dev))
        pop.exp_avg_sq.copy_(torch.rand(pop.exp_avg_sq.shape, generator=g, device=dev))
        pop.step_count.copy_(torch.arange(P, dtype=torch.int32, device=dev) * 37 + 5)
        pop.decay_lr()
    before = _snapshot(pop)
    # member 5 is a source and a destination: member 1 must get its state from before the copy
    dst, src = [5, 1, 3], [0, 5, 6]
    factors = [{"learning_rate": 1.2, "clip_ratio": 1.2, "learning_rate_decay": 0.8},
               {},
               {"learning_rate_decay": 1.2, "ent_coef": 0.8, "vf_coef": 1.2, "max_grad_norm": 0.8,
                "clip_ratio": 1.2}]
    pop.copy_members(dst, src, factors)
    torch.cuda.synchronize()
    after = _snapshot(pop)
    for d, s, f in zip(dst, src, factors):
        for a, b in zip(_rows(after, d), _rows(before, s)):
            assert a.dtype == b.dtype and torch.equal(a, b), (d, s)
        for k in HPARAMS:
            v = np.float32(before[k][s].item())
            if k in f:
                v = np.float32(v * np.float32(f[k]))
                if k in popmod.CAPPED_AT_ONE:
                    v = min(v, np.float32(1.0))
            assert after[k][d].item() == float(v), (d, k)
    # the clamps were exercised: member 6's decay 0.93 and clip 0.87, scaled by 1.2, are cut to 1.0
    assert after["learning_rate_decay"][3].item() == 1.0 and after["clip_ratio"][3].item() == 1.0
    for p in (0, 2, 4, 6):
        for a, b in zip(_rows(after, p), _rows(before, p)):
            assert torch.equal(a, b), p
        for k in HPARAMS:
            assert torch.equal(after[k][p], before[k][p]), (p, k)
    # state_rows / set_rows (the torchrun path) are the same copy
    other = Population(list(range(P)), 3, hp, dev)
    other.set_rows(dst, *_from_snapshot(other, before).state_rows(src), factors)
    theirs = _snapshot(other)
    assert all(torch.equal(a, b) for a, b in zip(theirs.pop("params"), after["params"]))
    assert all(torch.equal(t, after[k]) for k, t in theirs.items())


def _from_snapshot(pop, snap):
    with torch.no_grad():
        for t, s in zip(pop.params, snap["params"]):
            t.copy_(s)
        pop.exp_avg.copy_(snap["exp_avg"])
        pop.exp_avg_sq.copy_(snap["exp_avg_sq"])
        pop.step_count.copy_(snap["step_count"])
        for k in HPARAMS:
            getattr(pop, HPARAM_ATTRS[k]).copy_(snap[k])
    return pop


@gpu
def test_copy_members_refuses_bad_arguments():
    pop = Population([0, 1, 2], 1, None, torch.device("cuda", 0))
    with pytest.raises(ValueError):
        pop.copy_members([0, 0], [1, 2])
    with pytest.raises(ValueError):
        pop.copy_members([0], [3])
    with pytest.raises(ValueError):
        pop.copy_members([0], [1, 2])
    with pytest.raises(ValueError):
        pop.copy_members([0], [1], [{"gamma": 1.2}])


# ---- GPU: training runs ------------------------------------------------------------------------------------------
BASE = ["--track", "big_track", "--n-envs", "24", "--seeds", "0-7", "--n-epochs", "6", "--n-steps", "64",
        "--batch-size", "64", "--eval-every", "2", "--eval-episodes", "64"]
PBT = ["--pbt-every", "2", "--pbt-seed", "5"]


def _strip(rec):
    return {k: v for k, v in rec.items() if k not in ("wall_s", "current_hparams")}


def _model(root, name, m):
    return torch.load(os.path.join(root, name, f"member_{m}", "model.dat"), weights_only=True)


@pytest.fixture(scope="module")
def runs(tmp_path_factory):
    """The same README-shape population without PBT and twice with it; the fitness every round ranked."""
    if not torch.cuda.is_available():
        pytest.skip("needs a GPU")
    root = str(tmp_path_factory.mktemp("pbt"))
    seen = []
    decide = pbt.pbt_decisions

    def spy(fitness, *a):
        seen.append(list(fitness))
        return decide(fitness, *a)

    pbt.pbt_decisions = spy
    try:
        out = {name: popmod.train_population(popmod.parse_args(
            BASE + extra + ["--checkpoint-dir", root, "--run-name", name,
                            "--log-json", os.path.join(root, name + ".jsonl")]))
            for name, extra in (("plain", []), ("pbt_a", PBT), ("pbt_b", PBT))}
    finally:
        pbt.pbt_decisions = decide
    return root, out, seen


@gpu
def test_members_never_replaced_train_as_without_pbt(runs):
    root, out, _ = runs
    replaced = {line["member"] for line in out["pbt_a"]["lineage"]}
    assert replaced and len(replaced) < 8
    plain, pbt_run = out["plain"]["history"], out["pbt_a"]["history"]
    assert len(plain) == len(pbt_run) == 6 * 8
    for a, b in zip(plain, pbt_run):
        assert a["member"] == b["member"] and "current_hparams" in b and "current_hparams" not in a
        assert b["current_hparams"]["learning_rate"] == b["lr"]
        if b["member"] not in replaced:
            assert _strip(a) == _strip(b), (b["epoch"], b["member"])
    for m in range(8):
        same = all(torch.equal(x, y) for x, y in zip(_model(root, "plain", m).values(),
                                                      _model(root, "pbt_a", m).values()))
        assert same == (m not in replaced), m
    # after its first replacement a member trains with a perturbed learning rate
    first = {}
    for line in out["pbt_a"]["lineage"]:
        first.setdefault(line["member"], line)
    for m, line in first.items():
        at = lambda h: next(r for r in h if r["member"] == m and r["epoch"] == line["epoch"] + 1)
        assert at(pbt_run)["lr"] != at(plain)["lr"]


@gpu
def test_pbt_runs_are_deterministic(runs):
    root, out, _ = runs
    a, b = out["pbt_a"], out["pbt_b"]
    assert [{k: v for k, v in r.items() if k != "wall_s"} for r in a["history"]] == \
        [{k: v for k, v in r.items() if k != "wall_s"} for r in b["history"]]
    assert a["lineage"] == b["lineage"] and a["final"] == b["final"] and a["pbt_best"] == b["pbt_best"]
    for m in range(8):
        for x, y in zip(_model(root, "pbt_a", m).values(), _model(root, "pbt_b", m).values()):
            assert torch.equal(x, y), m


@gpu
def test_pbt_end_to_end(runs):
    from ppo_car_b200 import evaluate

    root, out, seen = runs
    run = out["pbt_a"]
    assert len(seen) == 4                                    # rounds after epochs 2 and 4 of each PBT run
    lineage = run["lineage"]
    assert [(l["pbt_round"], l["epoch"]) for l in lineage] == [(0, 2), (0, 2), (1, 4), (1, 4)]
    for r in (0, 1):
        fitness = seen[r]
        order = _rank(fitness)
        lines = [l for l in lineage if l["pbt_round"] == r]
        assert sorted(l["member"] for l in lines) == sorted(order[-2:])
        for l in lines:
            assert l["parent"] in order[:2]
            assert l["fitness"] == {"member": fitness[l["member"]], "parent": fitness[l["parent"]]}
            before, after = l["hparams_before"], l["hparams_after"]
            assert set(before) == set(after) == set(HPARAMS)
            for k in ("clip_ratio", "vf_coef", "max_grad_norm", "learning_rate_decay"):   # copied, not explored
                parent_rec = next(x for x in run["history"] if x["member"] == l["parent"] and x["epoch"] == l["epoch"])
                assert after[k] == parent_rec["current_hparams"][k]
    logged = [json.loads(x) for x in open(os.path.join(root, "pbt_a.jsonl"))]
    assert [x for x in logged if "pbt_round" in x] == lineage
    ancestry = {r["member"]: r["ancestry"] for r in run["final"]}
    for l in lineage:
        assert [l["epoch"], l["parent"]] in ancestry[l["member"]]
    assert run["pbt_best"]["member"] == _rank(seen[1])[0]
    assert all("current_hparams" in r for r in run["final"])
    # "eval" records keep their format
    plain_eval = next(r for r in out["plain"]["history"] if "eval" in r)["eval"]
    for r in run["history"]:
        assert ("eval" in r) == (r["epoch"] % 2 == 0)
        if "eval" in r:
            assert set(r["eval"]) == set(plain_eval)
    assert "lineage" not in out["plain"] and "current_hparams" not in out["plain"]["final"][0]
    m = lineage[0]["member"]
    path = os.path.join(root, "pbt_a", f"member_{m}", "model.dat")
    res = evaluate.main(["--checkpoint", path, "--episodes", "64", "--seed", "7"])
    assert res["episodes"] == 64


@pytest.mark.gpu
@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_two_ranks_equal_one_rank(tmp_path):
    argv = ["--track", "big_track", "--n-envs", "8", "--n-epochs", "5", "--n-steps", "64", "--batch-size", "64",
            "--seeds", "0-4", "--pbt-every", "2", "--pbt-fraction", "0.4", "--eval-episodes", "32",
            "--pbt-explore", "learning_rate,clip_ratio"]
    subprocess.check_call([sys.executable, "-m", "torch.distributed.run", "--nproc-per-node", "2", "-m",
                           "ppo_car_b200.population", *argv, "--log-json", str(tmp_path / "two.jsonl")], cwd=ROOT)
    one = popmod.train_population(popmod.parse_args(argv + ["--log-json", str(tmp_path / "one.jsonl")]))
    two = [json.loads(x) for r in (0, 1) for x in open(tmp_path / f"two.jsonl.rank{r}")]
    ones = [json.loads(x) for x in open(tmp_path / "one.jsonl")]
    assert any("pbt_round" in x for x in ones)
    key = lambda r: (r.get("pbt_round", -1), r["epoch"], r["member"])
    strip = lambda rs: sorted(({k: v for k, v in r.items() if k != "wall_s"} for r in rs), key=key)
    assert strip(two) == strip(ones)
    assert len(ones) == len(one["history"]) + len(one["lineage"])
