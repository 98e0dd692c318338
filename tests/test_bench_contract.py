"""bench.py contract: the reference arm prints one JSON line with the documented keys, the product arm refuses to run
without a GPU (there is no CPU fallback), and on a GPU --dump-outputs writes a reproducible sample of its outputs."""
import json
import os
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line():
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "1"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert res.returncode == 0, res.stderr[-2000:]
    lines = [l for l in res.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "CarEnv env-steps/sec" and d["unit"] == "env-steps/s"
    assert d["higher_is_better"] is True and d["steps"] == 1 and d["warmup"] == 1 and d["value"] > 0
    assert d["vs_baseline"] is None and d["data"] == "synthetic" and "workload" in d["config"]
    from oracle.ref_import import reference_root

    want = "reference" if reference_root(prefer_copy=True) is not None else "port"   # oracle/_ref travels with the repo
    assert d["cpu_baseline"]["kind"] == want and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["gpu_launches"] == 0


@pytest.mark.gpu
def test_dump_outputs_is_a_reproducible_sample_of_the_last_step(tmp_path):
    """--dump-outputs writes the last timed step's obs / reward / flags for the sampled environments as float32 .npy
    files; two runs with the same arguments write the same bytes, and they equal the sampled columns of a replay of
    the bench's seeded action stream through VecCarEnv.rollout."""
    import numpy as np

    import ppo_car_b200

    total, chunk, warmup, steps = 4096, 32, 3, 2
    dumps = []
    for run in ("a", "b"):
        res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--envs", str(total), "--chunk", str(chunk),
                              "--steps", str(steps), "--warmup", str(warmup), "--no-configs", "--no-cpu", "--e2e-steps",
                              "1", "--dump-outputs", str(tmp_path / run)], capture_output=True, text=True, timeout=600,
                             cwd=ROOT)
        assert res.returncode == 0, res.stderr[-2000:]
        assert json.loads(res.stdout.strip().splitlines()[-1])["steps"] == steps
        dumps.append({k: np.load(tmp_path / run / f"{k}.npy") for k in ("obs", "reward", "terminated", "truncated")})
    a, b = dumps
    assert a["obs"].shape == (chunk, 2048, 18) and all(a[k].shape == (chunk, 2048) for k in ("reward", "terminated", "truncated"))
    assert all(v.dtype == np.float32 and np.array_equal(v, b[k]) for k, v in a.items())

    # replay: two seeded action chunks, alternating from 0 in the warm-up and again in the timed steps
    dev = torch.device("cuda", 0)
    gen = torch.Generator(device=dev).manual_seed(1234)
    acts = [torch.randint(0, 9, (chunk, total), generator=gen, device=dev, dtype=torch.uint8) for _ in range(2)]
    env = ppo_car_b200.VecCarEnv(total, ppo_car_b200.builtin_track("big_track"), device=dev)
    env.reset()
    for i in list(range(warmup)) + list(range(steps)):
        out = env.rollout(acts[i % 2])
    ids = torch.from_numpy(np.sort(np.random.default_rng(0).choice(total, size=2048, replace=False))).to(dev)
    for k in a:
        assert np.array_equal(a[k], out[k].index_select(1, ids).float().cpu().numpy()), k
    assert a["terminated"].sum() > 0


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU behaviour")
def test_product_arm_needs_a_gpu():
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1"], capture_output=True,
                         text=True, timeout=600, cwd=ROOT)
    assert res.returncode != 0 and "no CPU path" in (res.stdout + res.stderr)
