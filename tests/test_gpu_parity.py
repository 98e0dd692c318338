"""GPU parity tests proper: everything goes through the C ABI (ppo_car_b200.VecCarEnv / Buffer ->
libcarenv_b200.so) and is compared with (1) the golden trajectories recorded from the unmodified
reference, (2) the float64 C oracle on the same seeded inputs, (3) size-independent properties at
the full BASELINE sizes.  Integer outputs bit-exact, float outputs 1e-5 relative (tests/parity.py)."""
import os

import numpy as np
import pytest
import torch

import ppo_car_b200
from oracle.c_oracle import COracleVecEnv
from oracle.carenv_port import gae_port
from tests.parity import RTOL_SYNTHETIC, assert_floats_close, assert_trajectory_matches

pytestmark = pytest.mark.gpu
GROUPS = ["const", "lap", "random", "fwd"]


def _gpu_traj(out):
    info = out["info"]
    return dict(obs=out["obs"].cpu().numpy(), rew=out["reward"].cpu().numpy(), term=out["terminated"].cpu().numpy(),
                trunc=out["truncated"].cpu().numpy(), gates_passed=info["gates_passed"].cpu().numpy(),
                time_passed=info["time_passed"].cpu().numpy(), next_gate_index=info["next_gate_index"].cpu().numpy())


def _golden_group(g, group, T=None, n=None):
    """One trajectory group of a tests/golden file, its first T steps of the first n envs, as the autoresetting vector
    env returns it (the reset observation where an episode ended)."""
    def cut(a):
        return a[:T, :n]

    done = cut(g[f"{group}_term"] | g[f"{group}_trunc"]).astype(bool)
    rec = {k: cut(g[f"{group}_{k}"]) for k in ("actions", "rew", "term", "trunc", "gates_passed", "time_passed",
                                              "next_gate_index")}
    rec["obs"] = np.where(done[..., None], g["reset_obs"], cut(g[f"{group}_final_obs"]))
    return rec


@pytest.mark.parametrize("name", ["track", "big_track"])
def test_golden_trajectories_from_the_reference(golden_dir, tracks_dir, name):
    g = np.load(os.path.join(golden_dir, f"carenv_{name}.npz"))
    path = os.path.join(tracks_dir, name + ".json")
    for group in GROUPS:
        ref = _golden_group(g, group)
        acts = ref["actions"]
        env = ppo_car_b200.VecCarEnv(acts.shape[1], path)
        obs0, _ = env.reset()
        assert_floats_close(obs0.cpu().numpy(), np.broadcast_to(g["reset_obs"], obs0.shape), "reset obs")
        out = env.rollout(torch.from_numpy(acts).cuda(), store_info=True)
        assert_trajectory_matches(_gpu_traj(out), ref, what=f"{name}/{group}")
        if group == "lap":
            assert int(((out["info"]["events"] >> 1) & 1).sum()) == 1
        env.close()


@pytest.mark.parametrize("name,n_envs,biased", [("big_track", 4096, False), ("track", 4096, True), ("big_track", 24, False)])
def test_random_rollout_matches_float64_oracle(tracks_dir, name, n_envs, biased):
    """BASELINE configs 1/2 shape (24 x 1024) and a 4096-env case: same action tensor into both."""
    T = 1024
    rng = np.random.default_rng(11)
    p = [.3, .02, .1, .1, .2, .2, .02, .02, .04] if biased else None
    acts = rng.choice(9, size=(T, n_envs), p=p).astype(np.uint8)
    path = os.path.join(tracks_dir, name + ".json")
    ora = COracleVecEnv(n_envs, path, scan_all_gates=False)
    ora.reset()
    ref = ora.rollout(acts, want=("obs", "rew", "term", "trunc", "gates_passed", "time_passed", "next_gate_index"))
    env = ppo_car_b200.VecCarEnv(n_envs, path)
    env.reset()
    out = env.rollout(torch.from_numpy(acts).cuda(), store_info=True)
    assert_trajectory_matches(_gpu_traj(out), ref, what=name)
    counts = env.slow_path_counts()
    assert sum(counts.values()) < 2e-3 * acts.size, counts


def test_step_api_device_and_numpy_paths_agree_with_rollout(tracks_dir):
    """step() with CUDA int64 actions (Categorical.sample dtype), with numpy actions, and the
    multi-step rollout launch give identical results; reward_scaling and float flags work."""
    path = os.path.join(tracks_dir, "big_track.json")
    n, T = 257, 200                                  # ragged: not a multiple of the block size
    rng = np.random.default_rng(5)
    acts = rng.choice(9, size=(T, n), p=[.3, .02, .1, .1, .2, .2, .02, .02, .04])
    env_a = ppo_car_b200.VecCarEnv(n, path, reward_scaling=0.1)
    env_b = ppo_car_b200.VecCarEnv(n, path, reward_scaling=0.1)
    env_c = ppo_car_b200.VecCarEnv(n, path, reward_scaling=0.1, float_flags=True)
    oa, _ = env_a.reset()
    env_b.reset(options={"track_path": path})
    env_c.reset()
    assert env_a.single_observation_space.shape == (18,) and env_a.single_action_space.n == 9
    ref = env_c.rollout(torch.from_numpy(acts.astype(np.int32)).cuda(), store_info=True)
    for t in range(T):
        o1, r1, te1, tr1, i1 = env_a.step(torch.from_numpy(acts[t]).cuda())          # int64 on device
        o2, r2, te2, tr2, i2 = env_b.step(acts[t])                                    # numpy in, numpy out
        assert o1.dtype == torch.float32 and te1.dtype == torch.bool and r1.dtype == torch.float32
        assert isinstance(o2, np.ndarray) and te2.dtype == np.bool_ and tr2.dtype == np.bool_
        assert r2.dtype == np.float64 and o2.dtype == np.float32          # the reference's dtypes (lib/car_env.py:760)
        assert np.array_equal(o1.cpu().numpy(), o2) and np.array_equal(r1.cpu().numpy(), r2.astype(np.float32))
        assert np.array_equal(te1.cpu().numpy(), te2) and np.array_equal(tr1.cpu().numpy(), tr2)
        assert np.array_equal(o2, ref["obs"][t].cpu().numpy())
        assert np.array_equal(r2.astype(np.float32), ref["reward"][t].cpu().numpy())
        assert np.array_equal(te2.astype(np.float32), ref["terminated"][t].cpu().numpy())
        assert np.array_equal(i2["gates_passed"], ref["info"]["gates_passed"][t].cpu().numpy())
        assert np.array_equal(i2["time_passed"], ref["info"]["time_passed"][t].cpu().numpy())
        assert set(i2) == {"gates_passed", "time_passed"}                 # the reference's info dict, nothing else
    assert ref["terminated"].sum() > 0
    # state arrays agree after T single steps and after one T-step launch
    assert torch.equal(env_a.pos, env_c.pos) and torch.equal(env_a.ints, env_c.ints)


def test_full_size_properties_65536_envs(tracks_dir):
    """BASELINE config 3 size (65,536 envs): properties that need no oracle.
    Shard invariance (env i does not depend on how many envs share the launch), time counter
    consistency, reward value set, reset observation on every done step, bounded observations."""
    path = os.path.join(tracks_dir, "big_track.json")
    n, T = 65536, 256
    g = torch.Generator(device="cuda").manual_seed(0)
    acts = torch.randint(0, 9, (T, n), generator=g, device="cuda", dtype=torch.uint8)
    env = ppo_car_b200.VecCarEnv(n, path)
    env.reset()
    out = env.rollout(acts, store_info=True)
    done = (out["terminated"] | out["truncated"]).bool()
    assert not (out["terminated"] & out["truncated"]).any()
    robs = torch.from_numpy(env.reset_observation).cuda()
    assert torch.equal(out["obs"][done], robs.expand(int(done.sum()), 18))
    tp = out["info"]["time_passed"]
    prev = torch.cat([torch.zeros_like(tp[:1]), torch.where(done[:-1], torch.zeros_like(tp[:-1]), tp[:-1])])
    assert torch.equal(tp, prev + 1)
    vals = torch.unique(out["reward"]).cpu().numpy().astype(np.float64)
    allowed = np.array([r for r in (0.0, 0.01, 1.0, 0.01 + 1.0, -3.0, 0.01 - 3.0, 1.0 - 3.0, (0.01 + 1.0) - 3.0)],
                       np.float64).astype(np.float32)
    assert set(vals.astype(np.float32)) <= set(allowed)
    o = out["obs"]
    assert (o[..., 6:] > 0).all() and (o[..., 6:] <= 1.0).all() and (o[..., 2:6].abs() <= 1.0).all()
    # shard invariance: the first 1000 and the last 4097 envs replayed alone give the same traces
    for lo, hi in ((0, 1000), (n - 4097, n)):
        sub = ppo_car_b200.VecCarEnv(hi - lo, path)
        sub.reset()
        so = sub.rollout(acts[:, lo:hi].contiguous(), store_info=True)
        assert torch.equal(so["obs"], out["obs"][:, lo:hi]) and torch.equal(so["reward"], out["reward"][:, lo:hi])
        assert torch.equal(so["terminated"], out["terminated"][:, lo:hi])
        assert torch.equal(so["info"]["gates_passed"], out["info"]["gates_passed"][:, lo:hi])
    # and a 4096-env slice of it agrees with the float64 oracle
    ora = COracleVecEnv(4096, path, scan_all_gates=False)
    ora.reset()
    ref = ora.rollout(acts[:, :4096].cpu().numpy(), want=("term", "trunc", "gates_passed"))
    assert np.array_equal(out["terminated"][:, :4096].cpu().numpy(), ref["term"])
    assert np.array_equal(out["info"]["gates_passed"][:, :4096].cpu().numpy(), ref["gates_passed"])


@pytest.mark.parametrize("tag", ["small", "train", "wide"])
def test_gae_golden_bit_exact(golden_dir, tag):
    g = np.load(os.path.join(golden_dir, "gae.npz"))
    c = lambda k: torch.from_numpy(g[f"{tag}_{k}"]).cuda()
    adv, ret = ppo_car_b200.gae_reverse_scan(c("rew"), c("val"), c("term"), c("trunc"), c("last_val"), c("last_term"),
                                             c("last_trunc"))
    assert np.array_equal(adv.cpu().numpy(), g[f"{tag}_adv"]) and np.array_equal(ret.cpu().numpy(), g[f"{tag}_ret"])


def test_gae_buffer_api_and_full_size_bit_exact():
    """Buffer drop-in at BASELINE config 3 size [1024, 65536] against the float32 port of lib/buffer.py."""
    T, N = 1024, 65536
    g = torch.Generator(device="cuda").manual_seed(1)
    buf = ppo_car_b200.Buffer((18,), T, N, "cuda", gamma=0.99, gae_lambda=0.95)
    with pytest.raises(AssertionError):
        buf.calculate_advantages(torch.zeros(1, N).cuda(), torch.zeros(1, N).cuda(), torch.zeros(1, N).cuda())
    buf.rew_buf.copy_(torch.rand((T, N), generator=g, device="cuda") * 1.4 - 0.3)
    buf.val_buf.copy_(torch.randn((T, N), generator=g, device="cuda"))
    buf.term_buf.copy_((torch.rand((T, N), generator=g, device="cuda") < 0.004).float())
    buf.trunc_buf.copy_((torch.rand((T, N), generator=g, device="cuda") < 0.001).float())
    buf.ptr = T
    lv = torch.randn((1, N), generator=g, device="cuda")
    lt = (torch.rand((1, N), generator=g, device="cuda") < 0.01).float()
    lu = (torch.rand((1, N), generator=g, device="cuda") < 0.01).float()
    adv, ret = buf.calculate_advantages(lv, lt, lu)
    ra, rr = gae_port(buf.rew_buf.cpu().numpy(), buf.val_buf.cpu().numpy(), buf.term_buf.cpu().numpy(),
                      buf.trunc_buf.cpu().numpy(), lv.cpu().numpy(), lt.cpu().numpy(), lu.cpu().numpy())
    assert np.array_equal(adv.cpu().numpy(), ra) and np.array_equal(ret.cpu().numpy(), rr)
    obs, act, val, logp = buf.get()
    assert buf.ptr == 0 and obs.shape == (T, N, 18)


def test_buffer_store_rows_from_env_step(tracks_dir):
    """The train.py:173-195 loop shape: step -> store -> GAE, all on device."""
    path = os.path.join(tracks_dir, "track.json")
    n, T = 24, 64
    env = ppo_car_b200.VecCarEnv(n, path, reward_scaling=0.1, float_flags=True)
    buf = ppo_car_b200.Buffer((18,), T, n, "cuda")
    obs, _ = env.reset()
    term = trunc = torch.zeros(n, device="cuda")
    g = torch.Generator(device="cuda").manual_seed(2)
    for _ in range(T):
        a = torch.randint(0, 9, (n,), generator=g, device="cuda")
        o = obs.clone()
        obs, rew, nterm, ntrunc, _ = env.step(a)
        buf.store(o, a, rew, torch.zeros(n, device="cuda"), term, trunc, torch.zeros(n, device="cuda"))
        term, trunc = nterm.clone(), ntrunc.clone()
    adv, ret = buf.calculate_advantages(torch.zeros(1, n).cuda(), term.reshape(1, -1), trunc.reshape(1, -1))
    ra, rr = gae_port(buf.rew_buf.cpu().numpy(), buf.val_buf.cpu().numpy(), buf.term_buf.cpu().numpy(),
                      buf.trunc_buf.cpu().numpy(), np.zeros(n, np.float32), term.cpu().numpy(), trunc.cpu().numpy())
    assert np.array_equal(adv.cpu().numpy(), ra) and np.array_equal(ret.cpu().numpy(), rr)


def test_host_step_pipeline_large_batch(tracks_dir):
    """The numpy-in / numpy-out path cuts large batches into sub-ranges on side streams; results must equal
    the single-launch device path, also when device-side and host-side calls are interleaved."""
    path = os.path.join(tracks_dir, "big_track.json")
    n = 200_003                                        # >= 131072 -> 4 ranges, ragged sizes
    env_h, env_d = ppo_car_b200.VecCarEnv(n, path), ppo_car_b200.VecCarEnv(n, path)
    env_h.reset()
    env_d.reset()
    rng = np.random.default_rng(8)
    for t in range(40):
        a = rng.integers(0, 9, size=n)
        od, rd, ted, trd, idd = env_d.step(torch.from_numpy(a).cuda())
        if t % 5 == 4:                                 # interleave a device-side call on the default stream
            oh, rh, teh, trh, ih = env_h.step(torch.from_numpy(a).cuda())
            oh, rh, teh, trh = oh.cpu().numpy(), rh.cpu().numpy(), teh.cpu().numpy(), trh.cpu().numpy()
            ih = {k: v.cpu().numpy() for k, v in ih.items()}
        else:
            oh, rh, teh, trh, ih = env_h.step(a)
        assert np.array_equal(oh, od.cpu().numpy()) and np.array_equal(np.asarray(rh, np.float32), rd.cpu().numpy())
        assert np.array_equal(teh, ted.cpu().numpy()) and np.array_equal(trh, trd.cpu().numpy())
        assert np.array_equal(ih["gates_passed"], idd["gates_passed"].cpu().numpy())
    assert torch.equal(env_h.pos, env_d.pos) and torch.equal(env_h.ints, env_d.ints)


@pytest.mark.parametrize("n_outer,n_inner", [(7, 5), (10, 6), (16, 12)])
def test_other_segment_counts_on_gpu(tmp_path, n_outer, n_inner):
    """Synthetic tracks: odd polyline sizes run the generic loop, even ones the 2-/4-segment unrolled kernels;
    forcing the generic kernel must give identical bits."""
    from tests.synth_tracks import ring_track

    path = ring_track(str(tmp_path / "ring.json"), n_outer, n_inner)
    rng = np.random.default_rng(n_outer)
    acts = rng.choice(9, size=(400, 1024), p=[.3, .02, .1, .1, .2, .2, .02, .02, .04]).astype(np.uint8)
    ora = COracleVecEnv(1024, path, scan_all_gates=True)
    ora.reset()
    ref = ora.rollout(acts, want=("obs", "rew", "term", "trunc", "gates_passed", "time_passed", "next_gate_index"))
    env = ppo_car_b200.VecCarEnv(1024, path)
    env.reset()
    out = env.rollout(torch.from_numpy(acts).cuda(), store_info=True)
    assert_trajectory_matches(_gpu_traj(out), ref, what=f"ring {n_outer}+{n_inner}", rtol=RTOL_SYNTHETIC)
    gen = ppo_car_b200.VecCarEnv(1024, path)
    gen.set_option("force_generic", 1)
    gen.reset()
    out2 = gen.rollout(torch.from_numpy(acts).cuda(), store_info=True)
    assert torch.equal(out["obs"], out2["obs"]) and torch.equal(out["reward"], out2["reward"])
    assert torch.equal(out["terminated"], out2["terminated"]) and torch.equal(env.pos, gen.pos)


def test_config3_size_integer_traces_bit_exact(tracks_dir):
    """BASELINE config 3 width (65,536 envs) x 512 steps = 33.5 M env-steps (about 125 k episodes) against the
    float64 oracle: every terminated / truncated / gates_passed / time_passed / next_gate_index element equal."""
    path = os.path.join(tracks_dir, "big_track.json")
    n, T = 65536, 512
    g = torch.Generator(device="cuda").manual_seed(42)
    acts = torch.randint(0, 9, (T, n), generator=g, device="cuda", dtype=torch.uint8)
    env = ppo_car_b200.VecCarEnv(n, path)
    env.reset()
    out = env.rollout(acts, store_obs=False, store_info=True)
    ora = COracleVecEnv(n, path, scan_all_gates=False)
    ora.reset()
    ref = ora.rollout(acts.cpu().numpy(), want=("rew", "term", "trunc", "gates_passed", "time_passed", "next_gate_index"))
    assert np.array_equal(out["terminated"].cpu().numpy(), ref["term"])
    assert np.array_equal(out["truncated"].cpu().numpy(), ref["trunc"])
    for k in ("gates_passed", "time_passed", "next_gate_index"):
        assert np.array_equal(out["info"][k].cpu().numpy(), ref[k]), k
    assert np.array_equal(out["reward"].cpu().numpy(), ref["rew"].astype(np.float32))
    assert ref["term"].sum() > 100_000


def test_limits_many_gates_and_max_segments(tmp_path):
    """128 wall segments (the limit of the constant-bank kernels) with 1,500 gates (gate table > 48 KB of shared
    memory: opt-in dynamic shared memory attribute); 129 and 400 segments run the shared-memory-geometry kernel;
    more than 2,048 segments are rejected with an error."""
    from tests.synth_tracks import ring_track

    path = ring_track(str(tmp_path / "big_ring.json"), 64, 64, n_gates=1500, wobble=0.03)
    rng = np.random.default_rng(1)
    acts = rng.choice(9, size=(300, 512), p=[.3, .02, .1, .1, .2, .2, .02, .02, .04]).astype(np.uint8)
    ora = COracleVecEnv(512, path, scan_all_gates=False)
    ora.reset()
    ref = ora.rollout(acts, want=("obs", "rew", "term", "trunc", "gates_passed", "time_passed", "next_gate_index"))
    env = ppo_car_b200.VecCarEnv(512, path)
    env.reset()
    out = env.rollout(torch.from_numpy(acts).cuda(), store_info=True)
    assert_trajectory_matches(_gpu_traj(out), ref, what="64+64 segments, 1500 gates", rtol=RTOL_SYNTHETIC)
    assert ref["gates_passed"].max() > 20
    for n_outer, n_inner in ((65, 64), (230, 170)):
        big = ring_track(str(tmp_path / f"ring_{n_outer}.json"), n_outer, n_inner, n_gates=40, wobble=0.03)
        ora = COracleVecEnv(256, big, scan_all_gates=False)
        ora.reset()
        ref = ora.rollout(acts[:, :256], want=("obs", "rew", "term", "trunc", "gates_passed", "time_passed", "next_gate_index"))
        env = ppo_car_b200.VecCarEnv(256, big)
        env.reset()
        out = env.rollout(torch.from_numpy(acts[:, :256].copy()).cuda(), store_info=True)
        assert_trajectory_matches(_gpu_traj(out), ref, what=f"{n_outer}+{n_inner} segments (shared-memory geometry)", rtol=RTOL_SYNTHETIC)
        assert ref["term"].sum() > 20
    too_big = ring_track(str(tmp_path / "too_big.json"), 1500, 549)
    with pytest.raises(ppo_car_b200.CarEnvError, match="segments"):
        ppo_car_b200.VecCarEnv(8, too_big)


def test_api_errors_and_out_of_range_actions(tracks_dir):
    path = os.path.join(tracks_dir, "track.json")
    env = ppo_car_b200.VecCarEnv(16, path)
    with pytest.raises(ppo_car_b200.CarEnvError):
        env.step(np.zeros(16, np.int64))                      # step before reset
    env.reset()
    with pytest.raises(ValueError):
        env.step(np.zeros(15, np.int64))
    with pytest.raises(FileNotFoundError):
        env.reset(options={"track_path": os.path.join(tracks_dir, "missing.json")})
    # an action outside 0..8 falls through the reference's if/elif chain: same as "do nothing" (8)
    a = ppo_car_b200.VecCarEnv(16, path)
    b = ppo_car_b200.VecCarEnv(16, path)
    a.reset()
    b.reset()
    for _ in range(30):
        oa, ra, *_ = a.step(torch.full((16,), 8, device="cuda"))
        ob, rb, *_ = b.step(torch.full((16,), 11, device="cuda"))
        assert torch.equal(oa, ob) and torch.equal(ra, rb)
    env.close()
    env.close()                                               # idempotent


def test_full_size_properties_1M_envs(tracks_dir):
    """BASELINE config 4 width (1,048,576 envs): shard invariance against 8-way sharded replays of slices,
    counter consistency, reset observation on done steps, and a 2,048-env slice against the float64 oracle."""
    path = os.path.join(tracks_dir, "big_track.json")
    n, T = 1_048_576, 64
    g = torch.Generator(device="cuda").manual_seed(4)
    acts = torch.randint(0, 9, (T, n), generator=g, device="cuda", dtype=torch.uint8)
    env = ppo_car_b200.VecCarEnv(n, path)
    env.reset()
    out = env.rollout(acts, store_info=True)
    done = (out["terminated"] | out["truncated"]).bool()
    assert int(done.sum()) > 1_000
    robs = torch.from_numpy(env.reset_observation).cuda()
    assert torch.equal(out["obs"][done], robs.expand(int(done.sum()), 18))
    tp = out["info"]["time_passed"]
    prev = torch.cat([torch.zeros_like(tp[:1]), torch.where(done[:-1], torch.zeros_like(tp[:-1]), tp[:-1])])
    assert torch.equal(tp, prev + 1)
    from ppo_car_b200.shard import shard_range
    for rank in (0, 3, 7):                                   # what ranks 0, 3 and 7 of an 8-GPU run would compute
        lo, hi = shard_range(n, 8, rank)
        sub = ppo_car_b200.VecCarEnv(hi - lo, path)
        sub.reset()
        so = sub.rollout(acts[:, lo:hi].contiguous(), store_info=True)
        assert torch.equal(so["obs"], out["obs"][:, lo:hi]) and torch.equal(so["reward"], out["reward"][:, lo:hi])
        assert torch.equal(so["terminated"], out["terminated"][:, lo:hi])
        del sub, so
    lo = n - 2048
    ora = COracleVecEnv(2048, path, scan_all_gates=False)
    ora.reset()
    ref = ora.rollout(acts[:, lo:].cpu().numpy(), want=("obs", "rew", "term", "trunc", "gates_passed", "time_passed", "next_gate_index"))
    got = dict(obs=out["obs"][:, lo:].cpu().numpy(), rew=out["reward"][:, lo:].cpu().numpy(),
               term=out["terminated"][:, lo:].cpu().numpy(), trunc=out["truncated"][:, lo:].cpu().numpy(),
               gates_passed=out["info"]["gates_passed"][:, lo:].cpu().numpy(),
               time_passed=out["info"]["time_passed"][:, lo:].cpu().numpy(),
               next_gate_index=out["info"]["next_gate_index"][:, lo:].cpu().numpy())
    assert_trajectory_matches(got, ref, what="1M-env slice")


def test_adversarial_poses_on_gpu(tracks_dir):
    """Rays within 1e-8..1e-4 px of vertices and cardinal hits at 10 px +- 1e-9..1e-4 (tests/adversarial.py):
    states are written straight into the SoA tensors, one no-op step, flags and distances follow the oracle."""
    from tests.adversarial import make_poses, oracle_at_poses

    path = os.path.join(tracks_dir, "big_track.json")
    poses, tr = make_poses(path, seed=9, per_item=120)
    n = len(poses)
    term_ref, fobs_ref = oracle_at_poses(path, poses, tr)
    env = ppo_car_b200.VecCarEnv(n, path)
    env.reset()
    env.pos.copy_(torch.from_numpy(poses[:, :2].copy()))
    env.ints[:, 0] = torch.from_numpy(poses[:, 2].astype(np.int32))
    obs, rew, term, trunc, info = env.step(torch.full((n,), 8, device="cuda"))
    term = term.cpu().numpy()
    assert np.array_equal(term.astype(np.uint8), term_ref)
    alive = term_ref == 0
    assert_floats_close(obs.cpu().numpy()[alive][:, 6:], fobs_ref[alive][:, 6:], "ray distances at adversarial poses")
    counts = env.slow_path_counts()
    assert counts["line"] + counts["band"] > 500 and 0 < alive.sum() < n


def test_multi_track_vector_env(tracks_dir, tmp_path):
    """Three tracks in one vector env, ONE launch per step (carenv_multi_rollout): contiguous groups and a random
    per-env assignment — every env's rows equal a single-track VecCarEnv stepped with the same actions, bit for bit;
    reset(options=...) re-assigns environments and swaps the track list."""
    from tests.synth_tracks import ring_track

    pa, pb = os.path.join(tracks_dir, "track.json"), os.path.join(tracks_dir, "big_track.json")
    pc = ring_track(str(tmp_path / "ring.json"), 10, 6)
    multi = ppo_car_b200.MultiTrackVecEnv([(pa, 300), (pb, 500)], reward_scaling=0.1)
    ea, eb = ppo_car_b200.VecCarEnv(300, pa, reward_scaling=0.1), ppo_car_b200.VecCarEnv(500, pb, reward_scaling=0.1)
    obs, _ = multi.reset()
    oa, _ = ea.reset()
    ob, _ = eb.reset()
    assert torch.equal(obs[:300], oa) and torch.equal(obs[300:], ob) and not torch.equal(obs[0], obs[-1])
    g = torch.Generator(device="cuda").manual_seed(6)
    for _ in range(120):
        a = torch.randint(0, 9, (800,), generator=g, device="cuda")
        o, r, te, tr, info = multi.step(a)
        o1, r1, te1, tr1, i1 = ea.step(a[:300])
        o2, r2, te2, tr2, i2 = eb.step(a[300:])
        assert torch.equal(o[:300], o1) and torch.equal(o[300:], o2)
        assert torch.equal(r[:300], r1) and torch.equal(r[300:], r2)
        assert torch.equal(te[:300], te1) and torch.equal(te[300:], te2)
        assert torch.equal(info["gates_passed"][300:], i2["gates_passed"])
    assert torch.equal(multi.pos[:300], ea.pos) and torch.equal(multi.ints[300:], eb.ints)
    with pytest.raises(ValueError):
        multi.reset(options={"track_path": pa})                 # unknown option: refused, not ignored
    # arbitrary per-env assignment over three tracks (environments of different tracks share warps)
    n = 1500
    ids = np.random.default_rng(2).integers(0, 3, size=n).astype(np.int32)
    multi.close()
    multi = ppo_car_b200.MultiTrackVecEnv(track_paths=[pa, pb, pc], track_ids=ids)
    singles = [ppo_car_b200.VecCarEnv(int((ids == k).sum()), p) for k, p in enumerate((pa, pb, pc))]
    obs, _ = multi.reset()
    for k, e in enumerate(singles):
        o0, _ = e.reset()
        assert torch.equal(obs[torch.from_numpy(ids == k).cuda()], o0)
    for _ in range(150):
        a = torch.randint(0, 9, (n,), generator=g, device="cuda")
        o, r, te, tr, info = multi.step(a)
        for k, e in enumerate(singles):
            m = torch.from_numpy(ids == k).cuda()
            ok, rk, tek, trk, ik = e.step(a[m])
            assert torch.equal(o[m], ok) and torch.equal(r[m], rk) and torch.equal(te[m], tek) and torch.equal(tr[m], trk)
            assert torch.equal(info["time_passed"][m], ik["time_passed"])
    assert int(te.sum()) >= 0 and int(multi.ints[:, 3].max()) > 0
    # reset(options): new assignment, then a new track list
    ids2 = (ids + 1) % 3
    obs, _ = multi.reset(options={"track_ids": ids2})
    assert torch.equal(obs[torch.from_numpy(ids2 == 0).cuda()][0], singles[0].reset()[0][0])
    obs, _ = multi.reset(options={"track_paths": [pb, pa], "track_ids": np.zeros(n, np.int32)})
    assert torch.equal(obs[0], singles[1].reset()[0][0])
    multi.close()


def test_final_observation_output(tracks_dir):
    """gymnasium's info["final_observation"]: the observation each step ended in BEFORE the autoreset.  Equal to obs
    where the episode goes on; where it ended it must equal the oracle's pre-reset observation."""
    path = os.path.join(tracks_dir, "big_track.json")
    for n in (48, 5000):                                          # warp-per-env kernel and thread-per-env kernel
        T = 120
        acts = np.random.default_rng(n).choice(9, size=(T, n), p=[.5, .02, .05, .05, .15, .15, .02, .02, .04]).astype(np.uint8)
        ora = COracleVecEnv(n, path, scan_all_gates=False)
        ora.reset()
        ref = ora.rollout(acts, want=("obs", "fobs", "term", "trunc"))
        env = ppo_car_b200.VecCarEnv(n, path, final_observation=True)
        plain = ppo_car_b200.VecCarEnv(n, path)
        env.reset()
        plain.reset()
        n_done = 0
        for t in range(T):
            a = torch.from_numpy(acts[t]).cuda()
            o, r, te, tr, info = env.step(a)
            o2, r2, te2, tr2, _ = plain.step(a)
            assert torch.equal(o, o2) and torch.equal(r, r2) and torch.equal(te, te2)
            done = (te | tr)
            assert torch.equal(info["_final_observation"], done)
            f = info["final_observation"]
            assert torch.equal(f[~done], o[~done])
            assert_floats_close(f.cpu().numpy(), ref["fobs"][t], f"final observation, step {t}")
            n_done += int(done.sum())
        assert n_done > n // 4


def test_render_rgb_array_frames(tracks_dir):
    """Headless rgb_array frames (lib/car_env.py:762-812): shape / dtype and the colours at known places."""
    path = os.path.join(tracks_dir, "big_track.json")
    env = ppo_car_b200.VecCarEnv(16, path)
    env.reset()
    for _ in range(10):
        env.step(torch.zeros(16, dtype=torch.int64, device="cuda"))
    frames = env.render(env_indices=[0, 5])
    assert frames.shape == (2, 720, 1280, 3) and frames.dtype == torch.uint8
    f = frames[0].cpu().numpy()
    assert torch.equal(frames[0], frames[1])                       # same actions, same state
    assert tuple(f[2, 2]) == (11, 102, 35)                         # outside the outer polygon: background
    tr = env.track
    cx, cy = (int(round(v)) for v in env.pos[0].cpu().numpy())
    assert tuple(f[cy, cx]) in ((200, 30, 30), (250, 220, 60))     # the car
    wx, wy = (tr.walls[0, :2] + tr.walls[0, 2:]) / 2               # middle of the first wall segment: black
    assert tuple(f[int(wy), int(wx)]) == (0, 0, 0)
    nxt = int(env.ints[0, 2])
    gx, gy = (tr.gates[nxt, :2] * 0.5 + tr.gates[nxt, 2:] * 0.5)
    assert tuple(f[int(gy), int(gx)]) in ((255, 255, 0), (255, 255, 255), (200, 30, 30), (250, 220, 60))   # next gate: yellow
    later = min(nxt + 5, len(tr.gates) - 1)
    gx, gy = (tr.gates[later, :2] * 0.5 + tr.gates[later, 2:] * 0.5)
    assert tuple(f[int(gy), int(gx)]) in ((0, 255, 0), (255, 255, 255))                                     # later gates: green
    start = tr.start
    assert (f == np.array([190, 190, 190], np.uint8)).all(-1).sum() > 20_000                                # the corridor
    with pytest.raises(ValueError):
        env.render(env_indices=[99])


@pytest.mark.parametrize("name,n_envs", [("big_track", 4099), ("track", 1500), ("ring 90+80", 700), ("ring 7+5", 300)])
def test_pose_records_reproduce_observations_bit_for_bit(tracks_dir, tmp_path, name, n_envs):
    """SURVEY §8 f-3: a rollout that stores 32-byte pose records instead of 72-byte observations, and
    carenv_observe turning records (all, or a gathered minibatch) back into the very same observations."""
    if name.startswith("ring"):                              # 170 segments: geometry from shared memory; 12: generic loop
        from tests.synth_tracks import ring_track

        n_outer, n_inner = (int(v) for v in name.split()[1].split("+"))
        path = ring_track(str(tmp_path / "ring.json"), n_outer, n_inner)
    else:
        path = os.path.join(tracks_dir, name + ".json")
    T = 400
    g = torch.Generator(device="cuda").manual_seed(21)
    acts = torch.randint(0, 9, (T, n_envs), generator=g, device="cuda", dtype=torch.uint8)
    acts[:, : n_envs // 8] = 0                                # full throttle: collisions within ~30 steps
    acts[:, n_envs // 8: n_envs // 4] = 8                     # idle: truncation at 1000 is not reached, no resets
    ref = ppo_car_b200.VecCarEnv(n_envs, path, reward_scaling=0.1)
    ref.reset()
    full = ref.rollout(acts)
    env = ppo_car_b200.VecCarEnv(n_envs, path, reward_scaling=0.1)
    env.reset()
    out = env.rollout(acts, store_poses=True)
    assert out["obs"] is None and out["poses"].shape == (T, n_envs, 4) and out["poses"].dtype == torch.float64
    for k in ("reward", "terminated", "truncated"):
        assert torch.equal(out[k], full[k])
    done = (full["terminated"] | full["truncated"]).bool()
    assert int(done.sum()) > n_envs // 8
    obs = env.observe(out["poses"])
    assert torch.equal(obs.view(T, n_envs, 18), full["obs"])
    idx = torch.randint(0, T * n_envs, (512,), generator=g, device="cuda")
    assert torch.equal(env.observe(out["poses"], idx), full["obs"].view(-1, 18)[idx])
    buf = torch.empty((512, 18), device="cuda")
    assert env.observe(out["poses"], idx, out=buf) is buf
    with pytest.raises(ValueError):
        env.observe(out["poses"].float())
    with pytest.raises(ValueError):
        env.rollout(acts, obs_out=full["obs"], store_poses=True)
    # the slow path (rays through vertices, collision band) takes the same decisions in both kernels
    assert torch.equal(env.pos, ref.pos) and torch.equal(env.ints, ref.ints)


def test_reset_with_track_path_switches_the_track_mid_run(golden_dir, tracks_dir):
    """CarEnv.reset(options={"track_path": ...}) (lib/car_env.py:621-628, train.py:159): an env that has been
    stepping on one track is reset onto the other one and then follows that track's golden trajectories."""
    g = np.load(os.path.join(golden_dir, "carenv_big_track.npz"))
    acts = g["lap_actions"]
    env = ppo_car_b200.VecCarEnv(acts.shape[1], os.path.join(tracks_dir, "track.json"))
    env.reset()
    env.rollout(torch.randint(0, 9, (50, acts.shape[1]), device="cuda", dtype=torch.uint8))
    with pytest.raises(ppo_car_b200.CarEnvError):
        env._set_track(os.path.join(tracks_dir, "big_track.json")) or env.step(acts[0])   # new track: reset first
    obs0, _ = env.reset(options={"track_path": os.path.join(tracks_dir, "big_track.json")})
    assert_floats_close(obs0.cpu().numpy(), np.broadcast_to(g["reset_obs"], obs0.shape), "reset obs")
    out = env.rollout(torch.from_numpy(acts).cuda(), store_info=True)
    done = (g["lap_term"] | g["lap_trunc"]).astype(bool)
    ref = dict(obs=np.where(done[..., None], g["reset_obs"], g["lap_final_obs"]), rew=g["lap_rew"], term=g["lap_term"],
               trunc=g["lap_trunc"], gates_passed=g["lap_gates_passed"], time_passed=g["lap_time_passed"],
               next_gate_index=g["lap_next_gate_index"])
    assert_trajectory_matches(_gpu_traj(out), ref, what="big_track/lap after a track switch")


@pytest.mark.parametrize("name", ["track", "big_track"])
def test_warp_per_env_kernel_is_bit_identical_to_thread_per_env(golden_dir, tracks_dir, name):
    """Small batches run k_rollout_warp (one warp per environment, lane = wall segment, REDUX extrema); forcing
    either kernel gives the same bits — random rollouts, the lap trajectory of the golden file, pose records."""
    path = os.path.join(tracks_dir, name + ".json")
    n, T = 301, 700
    rng = np.random.default_rng(8)
    acts = torch.from_numpy(rng.choice(9, size=(T, n), p=[.3, .02, .1, .1, .2, .2, .02, .02, .04]).astype(np.uint8)).cuda()
    lap = torch.from_numpy(np.load(os.path.join(golden_dir, f"carenv_{name}.npz"))["lap_actions"]).cuda()
    outs = {}
    for mode in (1, -1):
        env = ppo_car_b200.VecCarEnv(n, path, reward_scaling=0.1)
        env.set_option("warp_per_env", mode)
        env.reset()
        out = env.rollout(acts, store_info=True)
        poses = env.rollout(acts[:50], store_poses=True)["poses"]
        env2 = ppo_car_b200.VecCarEnv(lap.shape[1], path)
        env2.set_option("warp_per_env", mode)
        env2.reset()
        out_lap = env2.rollout(lap, store_info=True)
        outs[mode] = (out, poses, env.pos.clone(), env.ints.clone(), out_lap, env.slow_path_counts())
    a, b = outs[1], outs[-1]
    for k in ("obs", "reward", "terminated", "truncated"):
        assert torch.equal(a[0][k], b[0][k]) and torch.equal(a[4][k], b[4][k]), k
    for k in ("gates_passed", "time_passed", "next_gate_index", "events"):
        assert torch.equal(a[0]["info"][k], b[0]["info"][k]) and torch.equal(a[4]["info"][k], b[4]["info"][k]), k
    assert torch.equal(a[1], b[1]) and torch.equal(a[2], b[2]) and torch.equal(a[3], b[3])
    assert a[5] == b[5]                                       # the float64 fallback ran equally often
    assert int(a[0]["terminated"].sum()) > n and int(((a[4]["info"]["events"] >> 1) & 1).sum()) == 1


def test_start_pose_inside_the_collision_distance_on_gpu(tmp_path):
    """`start_destroyed` (lib/car_env.py:682-686, 745-748): start pose 6 px from a wall — every step terminates with
    -3 (+0.01 when thrusting forward), time_passed is always 1, every observation is the reset observation."""
    from tests.synth_tracks import near_wall_track

    path = near_wall_track(str(tmp_path / "near_wall.json"))
    T, n = 40, 300
    acts = np.random.default_rng(12).integers(0, 9, size=(T, n)).astype(np.uint8)
    ora = COracleVecEnv(n, path, scan_all_gates=True)
    obs0_ref = ora.reset()
    ref = ora.rollout(acts, want=("obs", "rew", "term", "trunc", "gates_passed", "time_passed", "next_gate_index"))
    assert ref["term"].all()
    for mode in (-1, 1):                                         # thread-per-env and warp-per-env kernels
        env = ppo_car_b200.VecCarEnv(n, path)
        env.set_option("warp_per_env", mode)
        obs0, _ = env.reset()
        assert_floats_close(obs0.cpu().numpy(), obs0_ref, "reset obs", rtol=RTOL_SYNTHETIC)
        out = env.rollout(torch.from_numpy(acts).cuda(), store_info=True)
        assert_trajectory_matches(_gpu_traj(out), ref, what="near-wall ring start", rtol=RTOL_SYNTHETIC)
        assert bool(out["terminated"].all()) and int(out["info"]["time_passed"].max()) == 1
        # step() path too
        o, r, te, tr, info = env.step(torch.from_numpy(acts[0].astype(np.int64)).cuda())
        assert bool(te.all()) and torch.equal(o, obs0.expand_as(o))


def test_scale_config_full_integer_traces_on_all_eight_shards(tracks_dir):
    """BASELINE config 4 (1,048,576 envs, the bench workload, bench.py's action stream): for EACH of the eight
    shard_range shards a 16,384-env slice x 256 steps is compared with the float64 oracle — every terminated /
    truncated / gates_passed / time_passed / next_gate_index element and every reward (33.5 M env-steps in all),
    observations on a 1,024-env sub-slice of every shard.  Each shard runs as its own VecCarEnv of 131,072 envs,
    i.e. exactly what rank r of an 8-GPU run computes (k_rollout_tab with 2 x 148 balanced blocks)."""
    from ppo_car_b200.shard import shard_range

    path = os.path.join(tracks_dir, "big_track.json")
    total, T, S, SO = 1_048_576, 256, 16_384, 1_024
    gen = torch.Generator(device="cuda").manual_seed(1234)
    acts = torch.randint(0, 9, (T, total), generator=gen, device="cuda", dtype=torch.uint8)
    n_term = 0
    for rank in range(8):
        lo, hi = shard_range(total, 8, rank)
        a = acts[:, lo:hi].contiguous()
        env = ppo_car_b200.VecCarEnv(hi - lo, path)
        env.reset()
        out = env.rollout(a, store_info=True)
        off = (rank * 14_321) % (hi - lo - S)                   # a different place in every shard
        sl = slice(off, off + S)
        ora = COracleVecEnv(S, path, scan_all_gates=False)
        ora.reset()
        ref = ora.rollout(a[:, sl].cpu().numpy(), want=("rew", "term", "trunc", "gates_passed", "time_passed", "next_gate_index"))
        assert np.array_equal(out["terminated"][:, sl].cpu().numpy(), ref["term"]), rank
        assert np.array_equal(out["truncated"][:, sl].cpu().numpy(), ref["trunc"]), rank
        for k in ("gates_passed", "time_passed", "next_gate_index"):
            assert np.array_equal(out["info"][k][:, sl].cpu().numpy(), ref[k]), (rank, k)
        assert np.array_equal(out["reward"][:, sl].cpu().numpy(), ref["rew"].astype(np.float32)), rank
        ora = COracleVecEnv(SO, path, scan_all_gates=False)
        ora.reset()
        ref_o = ora.rollout(a[:, off:off + SO].cpu().numpy(), want=("obs",))
        assert_floats_close(out["obs"][:, off:off + SO].cpu().numpy(), ref_o["obs"], f"obs, shard {rank}")
        n_term += int(ref["term"].sum())
        del env, out
    assert n_term > 50_000


def test_config1_shape_track_json_24_envs_1024_uniform_steps_on_gpu(tracks_dir):
    """BASELINE configs[0] exactly (tracks/track.json, 24 envs x 1024 steps, i.i.d. uniform actions), oracle in its
    literal full-gate-scan mode; runs the warp-per-environment kernel (the one 24 envs get) and k_rollout."""
    path = os.path.join(tracks_dir, "track.json")
    acts = np.random.default_rng(101).integers(0, 9, size=(1024, 24)).astype(np.uint8)
    ora = COracleVecEnv(24, path, scan_all_gates=True)
    ora.reset()
    ref = ora.rollout(acts, want=("obs", "rew", "term", "trunc", "gates_passed", "time_passed", "next_gate_index"))
    for mode in (0, -1):
        env = ppo_car_b200.VecCarEnv(24, path)
        env.set_option("warp_per_env", mode)
        env.reset()
        out = env.rollout(torch.from_numpy(acts).cuda(), store_info=True)
        assert_trajectory_matches(_gpu_traj(out), ref, what=f"config 1 (warp_per_env={mode})")


@pytest.mark.parametrize("name", ["track", "big_track"])
def test_full_ordered_gate_scan_oracle_4096_envs(tracks_dir, name):
    """The reference scans every active gate in index order (lib/car_env.py:394-408); the kernel tests gate
    next_gate_index only.  4,096 envs x 768 forward-biased steps against the oracle in literal full-scan mode."""
    path = os.path.join(tracks_dir, name + ".json")
    n, T = 4096, 768
    acts = np.random.default_rng(78).choice(9, size=(T, n), p=[.3, .02, .1, .1, .2, .2, .02, .02, .04]).astype(np.uint8)
    ora = COracleVecEnv(n, path, scan_all_gates=True)
    ora.reset()
    ref = ora.rollout(acts, want=("obs", "rew", "term", "trunc", "gates_passed", "time_passed", "next_gate_index"))
    env = ppo_car_b200.VecCarEnv(n, path)
    env.reset()
    out = env.rollout(torch.from_numpy(acts).cuda(), store_info=True)
    assert_trajectory_matches(_gpu_traj(out), ref, what=f"{name}, full gate scan")
    assert int((out["info"]["events"] & 1).sum()) > 10_000


@pytest.mark.parametrize("name", ["track", "big_track"])
def test_table_kernel_is_bit_identical_to_the_arithmetic_kernel(tracks_dir, name):
    """k_rollout_tab (denominators from the shared-memory table, 512-thread CTAs walking balanced env blocks) and
    k_rollout (denominators recomputed) give the same bits: ragged env counts, several blocks per CTA, pose rows."""
    path = os.path.join(tracks_dir, name + ".json")
    T = 96
    for n in (40_003, 131_072, 200_003):
        g = torch.Generator(device="cuda").manual_seed(n)
        acts = torch.randint(0, 9, (T, n), generator=g, device="cuda", dtype=torch.uint8)
        outs = {}
        for mode in (1, -1):
            env = ppo_car_b200.VecCarEnv(n, path, reward_scaling=0.1)
            env.set_option("tab", mode)
            env.reset()
            out = env.rollout(acts, store_info=True)
            poses = env.rollout(acts[:8], store_poses=True)["poses"]
            outs[mode] = (out, poses, env.pos.clone(), env.vel.clone(), env.ints.clone(), env.slow_path_counts())
        a, b = outs[1], outs[-1]
        for k in ("obs", "reward", "terminated", "truncated"):
            assert torch.equal(a[0][k], b[0][k]), (n, k)
        for k in ("gates_passed", "time_passed", "next_gate_index", "events"):
            assert torch.equal(a[0]["info"][k], b[0]["info"][k]), (n, k)
        assert torch.equal(a[1], b[1]) and torch.equal(a[2], b[2]) and torch.equal(a[3], b[3]) and torch.equal(a[4], b[4])
        assert a[5] == b[5]


def test_cuda_path_against_the_unmodified_reference(golden_dir, tracks_dir, tmp_path):
    """The CUDA path against the reference's OWN code (lib/car_env.py, unmodified) with gymnasium's same-step autoreset
    emulated: both shipped tracks and the start_destroyed track.  Always against the stored trajectories
    (tests/golden: the forward-biased groups of carenv_*.npz, and near_wall.npz, whose `source` names what recorded
    it); where the reference itself is present ($PPO_CAR_REFERENCE, or the verified oracle/_ref copy), also against
    fresh trajectories of it.  Integers bit-exact, rewards
    float32(float64 reward), observations 1e-5 relative."""
    from oracle.ref_import import RefVecEnv, reference_available, track_path
    from tests.synth_tracks import near_wall_track

    cases = []                                                  # name, track, reset obs, trajectory with its actions
    for name in ("track", "big_track"):
        g = np.load(os.path.join(golden_dir, f"carenv_{name}.npz"))
        cases.append((name, os.path.join(tracks_dir, name + ".json"), g["reset_obs"], _golden_group(g, "fwd", 240, 6)))
    g = np.load(os.path.join(golden_dir, "near_wall.npz"))
    cases.append(("near_wall", os.path.join(golden_dir, "near_wall_track.json"), g["reset_obs"],
                  _golden_group(g, "destroyed")))
    if reference_available():
        rng = np.random.default_rng(31)
        nw = near_wall_track(str(tmp_path / "near_wall.json"))
        n = 6
        for name, ref_path, our_path, T in [("track", track_path("track.json"), os.path.join(tracks_dir, "track.json"), 240),
                                            ("big_track", track_path("big_track.json"),
                                             os.path.join(tracks_dir, "big_track.json"), 240),
                                            ("near_wall", nw, nw, 12)]:
            acts = rng.choice(9, size=(T, n), p=[.3, .02, .1, .1, .2, .2, .02, .02, .04]).astype(np.uint8)
            acts[:, 0] = 0                                      # one env at full throttle: gates, then a crash
            ref = RefVecEnv(n, ref_path)
            obs0 = ref.reset()
            rec = {k: [] for k in ("obs", "rew", "term", "trunc", "gates_passed", "time_passed", "next_gate_index")}
            for t in range(T):
                o, r, te, tr, info = ref.step(acts[t])
                for k, v in (("obs", o), ("rew", r), ("term", te), ("trunc", tr), ("gates_passed", info["gates_passed"]),
                             ("time_passed", info["time_passed"]), ("next_gate_index", info["next_gate_index"])):
                    rec[k].append(np.array(v))
            rec = {k: np.stack(v) for k, v in rec.items()}
            rec["actions"] = acts
            cases.append((name + " (live reference)", our_path, obs0, rec))
    for name, our_path, obs0, rec in cases:
        acts = rec["actions"]
        n, T = acts.shape[1], acts.shape[0]
        env = ppo_car_b200.VecCarEnv(n, our_path)
        g0, _ = env.reset()
        tol = RTOL_SYNTHETIC if name.startswith("near_wall") else 1e-5
        assert_floats_close(g0.cpu().numpy(), np.broadcast_to(obs0, g0.shape), f"{name}: reset obs vs reference", rtol=tol)
        out = env.rollout(torch.from_numpy(acts).cuda(), store_info=True)
        assert_trajectory_matches(_gpu_traj(out), rec, what=f"{name} vs unmodified reference", rtol=tol)
        assert rec["term"].sum() > 0
        # the numpy boundary: float64 rewards equal to TransformReward's r * 0.1 (train.py:65, 68) bit for bit
        env2 = ppo_car_b200.VecCarEnv(n, our_path, reward_scaling=0.1)
        env2.reset()
        for t in range(min(T, 40)):
            o, r, te, tr, info = env2.step(acts[t].astype(np.int64))
            assert r.dtype == np.float64 and np.array_equal(r, rec["rew"][t] * 0.1), (name, t)
            assert np.array_equal(te, rec["term"][t]) and np.array_equal(info["time_passed"], rec["time_passed"][t])


def test_numpy_step_records_debug_info_copy_outputs_and_device_records(tracks_dir):
    """The numpy step ships one 16-byte record per env (carenv_step_host_records): debug_info=True adds
    next_gate_index / events, copy_outputs=True returns arrays that survive the next step, and the device-buffer
    variant carenv_step_records writes the same records."""
    import ctypes as C
    from ppo_car_b200 import _lib

    path = os.path.join(tracks_dir, "big_track.json")
    n = 70_001                                                    # 4 sub-ranges, ragged
    rng = np.random.default_rng(3)
    env_v = ppo_car_b200.VecCarEnv(n, path, debug_info=True)
    env_c = ppo_car_b200.VecCarEnv(n, path, copy_outputs=True)
    env_d = ppo_car_b200.VecCarEnv(n, path)
    for e in (env_v, env_c, env_d):
        e.reset()
    rec_dev = torch.empty((n, 16), dtype=torch.uint8, device="cuda")
    obs_dev = torch.empty((n, 18), dtype=torch.float32, device="cuda")
    kept = None
    for t in range(60):
        a = rng.choice(9, size=n, p=[.3, .02, .1, .1, .2, .2, .02, .02, .04])
        ov, rv, tev, trv, iv = env_v.step(a)
        oc, rc_, tec, trc, ic = env_c.step(a)
        od, rd, ted, trd, idd = env_d.step(torch.from_numpy(a).cuda())
        assert np.array_equal(ov, oc) and np.array_equal(rv, rc_) and np.array_equal(tev, tec) and np.array_equal(trv, trc)
        assert np.array_equal(ov, od.cpu().numpy()) and np.array_equal(rv.astype(np.float32), rd.cpu().numpy())
        assert np.array_equal(iv["next_gate_index"], idd["next_gate_index"].cpu().numpy())
        assert np.array_equal(iv["events"], idd["events"].cpu().numpy())
        assert np.array_equal(iv["gates_passed"], ic["gates_passed"])
        if kept is not None:                                      # copies of step t-1 were not overwritten by step t
            assert np.array_equal(kept[0], kept[1]) and not np.array_equal(kept[0], oc)
        kept = (oc, oc.copy())
    # device records: same bytes as the host records of an identical env
    env_r = ppo_car_b200.VecCarEnv(n, path)
    env_r.reset()
    env_h = ppo_car_b200.VecCarEnv(n, path)
    env_h.reset()
    a = rng.integers(0, 9, size=n)
    L = _lib.lib()
    ad = torch.from_numpy(a).cuda()
    p = lambda t: C.c_void_p(t.data_ptr())
    rc = L.carenv_step_records(env_r._handle, n, p(env_r.pos), p(env_r.vel), p(env_r.ints), p(ad), _lib.ACT_I64, 1.0,
                               p(obs_dev), p(rec_dev), None, C.c_void_p(torch.cuda.current_stream().cuda_stream))
    assert rc == 0
    oh, rh, teh, trh, ih = env_h.step(a)
    rec = rec_dev.cpu().numpy().view(ppo_car_b200.VecCarEnv._REC_DTYPE).reshape(n)
    assert np.array_equal(rec["reward"], rh) and rec["reward"].dtype == np.float64 and np.array_equal(rec["terminated"], teh)
    assert np.array_equal(rec["time_passed"], ih["time_passed"]) and np.array_equal(obs_dev.cpu().numpy(), oh)


@pytest.mark.gpu
@pytest.mark.parametrize("n,T", [(75_776, 37), (100_003, 64), (200_003, 5), (131_072, 256)])
def test_time_sliced_table_kernel_is_bit_identical(tracks_dir, n, T):
    """k_rollout_tab_sliced (an SM's env-steps cut into 16 equal per-warp intervals, jobs that straddle two warps
    split in time with a state hand-over through memory) against the block-round table kernel: identical outputs and
    final state, at sizes with ragged last jobs and step counts that put the cuts in the middle of jobs; a second
    launch continues from the handed-over state."""
    path = os.path.join(tracks_dir, "big_track.json")
    g = torch.Generator(device="cuda").manual_seed(n + T)
    acts = torch.randint(0, 9, (2, T, n), generator=g, device="cuda", dtype=torch.uint8)
    outs = []
    for opt in (-1, 0):
        env = ppo_car_b200.VecCarEnv(n, path, reward_scaling=0.1)
        env.set_option("tab_slice", opt)
        env.reset()
        res = [env.rollout(acts[i], store_info=True) for i in range(2)]
        outs.append(([{k: (v.clone() if torch.is_tensor(v) else {kk: vv.clone() for kk, vv in v.items()})
                       for k, v in r.items()} for r in res], env.pos.clone(), env.vel.clone(), env.ints.clone()))
    (ra, pa, va, ia), (rb, pb, vb, ib) = outs
    assert torch.equal(pa, pb) and torch.equal(va, vb) and torch.equal(ia, ib)
    for a, b in zip(ra, rb):
        for k in ("obs", "reward", "terminated", "truncated"):
            assert torch.equal(a[k], b[k]), k
        for k in a["info"]:
            assert torch.equal(a["info"][k], b["info"][k]), k
