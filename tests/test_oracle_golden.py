"""Pin the oracle: the Python port and the C oracle must reproduce the trajectories
recorded from the UNMODIFIED reference (tests/golden/make_golden.py).  CPU only."""
import os

import numpy as np
import pytest

from oracle.carenv_port import PortVecEnv, PortCarEnv, gae_port, load_track
from oracle.c_oracle import COracleVecEnv

TRACK_NAMES = ["track", "big_track"]
GROUPS = ["const", "lap", "random", "fwd"]
INT_KEYS = ["term", "trunc", "gates_passed", "time_passed", "next_gate_index"]


def _gold(golden_dir, name):
    return np.load(os.path.join(golden_dir, f"carenv_{name}.npz"))


@pytest.mark.parametrize("name", TRACK_NAMES)
def test_track_loader_shapes(tracks_dir, name):
    tr = load_track(os.path.join(tracks_dir, name + ".json"))
    assert len(tr["walls"]) == {"track": 16, "big_track": 24}[name]
    assert len(tr["gates"]) == {"track": 45, "big_track": 55}[name]


@pytest.mark.parametrize("name", TRACK_NAMES)
def test_port_reset_obs_bit_exact(golden_dir, tracks_dir, name):
    g = _gold(golden_dir, name)
    env = PortCarEnv(os.path.join(tracks_dir, name + ".json"))
    obs, info = env.reset()
    assert obs.dtype == np.float32 and obs.shape == (18,)
    assert np.array_equal(obs, g["reset_obs"])
    assert info == {"gates_passed": 0, "time_passed": 0}


# the port replays a slice of every group bit-exactly (kept short: the port is as slow as the reference)
@pytest.mark.parametrize("name", TRACK_NAMES)
@pytest.mark.parametrize("group,steps", [("const", 64), ("lap", 1024), ("random", 320), ("fwd", 128)])
def test_port_matches_reference_bit_exact(golden_dir, tracks_dir, name, group, steps):
    g = _gold(golden_dir, name)
    acts = g[f"{group}_actions"][:steps]
    env = PortVecEnv(acts.shape[1], os.path.join(tracks_dir, name + ".json"))
    env.reset()
    for t in range(steps):
        obs, rew, term, trunc, info = env.step(acts[t])
        assert np.array_equal(info["final_obs"], g[f"{group}_final_obs"][t]), (group, t)
        assert np.array_equal(rew, g[f"{group}_rew"][t]), (group, t)          # float64, exact
        assert np.array_equal(term, g[f"{group}_term"][t]) and np.array_equal(trunc, g[f"{group}_trunc"][t])
        for k in ("gates_passed", "time_passed", "next_gate_index"):
            assert np.array_equal(info[k], g[f"{group}_{k}"][t]), (group, k, t)
        done = term | trunc
        assert np.array_equal(obs[done], np.broadcast_to(g["reset_obs"], obs.shape)[done])


@pytest.mark.parametrize("name", TRACK_NAMES)
@pytest.mark.parametrize("scan", [True, False])
def test_c_oracle_matches_reference(golden_dir, tracks_dir, name, scan):
    """Full 1024-step replay of all four groups.  Integers bit-exact; float32 obs within 1 ulp
    (libm vs numpy cos/sin may differ in the last bit of a double); rewards exact."""
    g = _gold(golden_dir, name)
    path = os.path.join(tracks_dir, name + ".json")
    for group in GROUPS:
        acts = g[f"{group}_actions"]
        env = COracleVecEnv(acts.shape[1], path, scan_all_gates=scan)
        obs0, dist0 = env.reset(return_dist=True)
        np.testing.assert_array_max_ulp(obs0, np.broadcast_to(g["reset_obs"], obs0.shape), maxulp=1)
        np.testing.assert_allclose(dist0[0], g["reset_dist"], rtol=1e-13)
        r = env.rollout(acts)
        for k in INT_KEYS:
            assert np.array_equal(r[k].astype(np.int64), g[f"{group}_{k}"].astype(np.int64)), (group, k)
        assert np.array_equal(r["rew"], g[f"{group}_rew"]), group
        np.testing.assert_array_max_ulp(r["fobs"], g[f"{group}_final_obs"], maxulp=1)
        done = (r["term"] | r["trunc"]).astype(bool)
        ref_obs = np.where(done[..., None], g["reset_obs"], g[f"{group}_final_obs"])
        np.testing.assert_array_max_ulp(r["obs"], ref_obs, maxulp=1)


def test_golden_covers_every_branch(golden_dir):
    """The fixtures exercise collision, truncation, gate, lap (+10) and every distinct reward value family."""
    for name in TRACK_NAMES:
        g = _gold(golden_dir, name)
        assert g["const_trunc"].sum() == 3 and g["const_term"].sum() > 100
        assert (g["lap_rew"] > 10.5).sum() == 1 and g["lap_trunc"].sum() == 1
        assert g["lap_gates_passed"].max() > {"track": 45, "big_track": 55}[name]
        vals = set(np.round(np.concatenate([g[f"{k}_rew"].ravel() for k in GROUPS]), 2))
        assert {0.0, 0.01, 1.0, 1.01, -3.0, -2.99}.issubset(vals)


@pytest.mark.parametrize("tag", ["small", "train", "wide"])
def test_gae_port_bit_exact(golden_dir, tag):
    g = np.load(os.path.join(golden_dir, "gae.npz"))
    adv, ret = gae_port(g[f"{tag}_rew"], g[f"{tag}_val"], g[f"{tag}_term"], g[f"{tag}_trunc"],
                        g[f"{tag}_last_val"], g[f"{tag}_last_term"], g[f"{tag}_last_trunc"])
    assert np.array_equal(adv, g[f"{tag}_adv"])
    assert np.array_equal(ret, g[f"{tag}_ret"])


def test_port_against_live_reference_when_available(tracks_dir):
    """Replay fresh random actions through the UNMODIFIED reference (the /root/reference mount in the build
    container, the verified oracle/_ref copy on the GPU box) and through the port: bit-exact."""
    from oracle.ref_import import RefVecEnv, reference_available, track_path

    if not reference_available():
        pytest.skip("neither /root/reference nor oracle/_ref (python oracle/make_ref.py) is present")
    rng = np.random.default_rng(2024)
    for name in TRACK_NAMES:
        acts = rng.choice(9, size=(150, 3), p=[.3, .02, .1, .1, .2, .2, .02, .02, .04])
        ref, port = RefVecEnv(3, track_path(name + ".json")), PortVecEnv(3, os.path.join(tracks_dir, name + ".json"))
        assert np.array_equal(ref.reset(), port.reset())
        for t in range(acts.shape[0]):
            o1, r1, te1, tr1, i1 = ref.step(acts[t])
            o2, r2, te2, tr2, i2 = port.step(acts[t])
            assert np.array_equal(o1, o2) and np.array_equal(r1, r2), (name, t)
            assert np.array_equal(te1, te2) and np.array_equal(tr1, tr2)
            assert np.array_equal(i1["gates_passed"], i2["gates_passed"])
            assert np.array_equal(i1["next_gate_index"], i2["next_gate_index"])


def test_port_against_live_reference_start_destroyed(golden_dir, tmp_path):
    """The branch the shipped tracks never take: a start pose inside the collision distance
    (lib/car_env.py:682-686).  Port vs the stored trajectory (tests/golden/near_wall.npz, its `source` names what
    recorded it) and, where the unmodified reference is present, vs the reference itself; bit-exact."""
    from oracle.ref_import import RefVecEnv, reference_available
    from tests.synth_tracks import near_wall_track

    g = np.load(os.path.join(golden_dir, "near_wall.npz"))
    acts = g["destroyed_actions"]
    port = PortVecEnv(acts.shape[1], os.path.join(golden_dir, "near_wall_track.json"))
    assert np.array_equal(port.reset(), np.broadcast_to(g["reset_obs"], (acts.shape[1], 18)))
    for t in range(acts.shape[0]):
        obs, rew, term, trunc, info = port.step(acts[t])
        assert term.all() and np.array_equal(term, g["destroyed_term"][t]), t
        assert np.array_equal(trunc, g["destroyed_trunc"][t]) and np.array_equal(rew, g["destroyed_rew"][t]), t
        assert np.array_equal(info["final_obs"], g["destroyed_final_obs"][t]), t
        assert np.array_equal(obs, np.broadcast_to(g["reset_obs"], obs.shape)), t
        for k in ("gates_passed", "time_passed", "next_gate_index"):
            assert np.array_equal(info[k], g[f"destroyed_{k}"][t]), (k, t)

    if not reference_available():
        return
    path = near_wall_track(str(tmp_path / "near_wall.json"))
    acts = np.random.default_rng(5).integers(0, 9, size=(12, 3))
    ref, port = RefVecEnv(3, path), PortVecEnv(3, path)
    assert np.array_equal(ref.reset(), port.reset())
    for t in range(acts.shape[0]):
        o1, r1, te1, tr1, i1 = ref.step(acts[t])
        o2, r2, te2, tr2, i2 = port.step(acts[t])
        assert te1.all() and np.array_equal(te1, te2) and np.array_equal(r1, r2) and np.array_equal(o1, o2)
        assert np.array_equal(i1["final_obs"], i2["final_obs"]) and np.array_equal(i1["time_passed"], i2["time_passed"])


def test_reference_copy_recipe_is_byte_identical(tmp_path, monkeypatch):
    """oracle/make_ref.py copies the hot-path files unmodified: when both the mount and the copy exist they are
    byte-identical, and the MANIFEST hashes verify.  The recipe is also run on a stand-in source tree, so that it is
    checked without a reference checkout: byte-identical copy, verified MANIFEST, and a changed copy is refused."""
    from oracle import make_ref, ref_import

    copy = ref_import.reference_root(prefer_copy=True)
    if copy is not None and copy.endswith("_ref"):
        assert ref_import._copy_is_intact()
        if os.path.isfile(os.path.join(ref_import._MOUNT, "lib", "car_env.py")):
            for rel in ("lib/car_env.py", "lib/buffer.py", "tracks/track.json", "tracks/big_track.json"):
                assert open(os.path.join(copy, rel), "rb").read() == open(os.path.join(ref_import._MOUNT, rel), "rb").read()

    src, dst = tmp_path / "src", tmp_path / "_ref"
    for i, rel in enumerate(make_ref.FILES):
        (src / rel).parent.mkdir(parents=True, exist_ok=True)
        (src / rel).write_bytes(b"stand-in %d\n" % i + bytes(range(256)))
    monkeypatch.setattr(make_ref, "SRC", str(src))
    monkeypatch.setattr(make_ref, "DST", str(dst))
    monkeypatch.setattr(ref_import, "_MOUNT", str(tmp_path / "no_mount"))
    monkeypatch.setattr(ref_import, "_COPY", str(dst))
    assert make_ref.make(verbose=False) == str(dst)
    for rel in make_ref.FILES:
        assert (dst / rel).read_bytes() == (src / rel).read_bytes()
    assert ref_import._copy_is_intact() and ref_import.reference_root(prefer_copy=True) == str(dst)
    (dst / "lib" / "car_env.py").write_bytes(b"changed")
    assert not ref_import._copy_is_intact() and ref_import.reference_root(prefer_copy=True) is None
