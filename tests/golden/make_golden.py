"""Generate the golden fixtures under tests/golden/ from the UNMODIFIED reference.

Run in the build container only (needs /root/reference):

    python tests/golden/make_golden.py

Everything written here comes out of the reference's own code
(/root/reference/lib/car_env.py and lib/buffer.py imported through
oracle/ref_import.py); nothing is computed by this repository's oracle or
kernels.  The fixtures pin the oracle (tests/test_oracle_golden.py) and the CUDA
path (tests/test_gpu_parity.py) on the GPU box, where /root/reference does not
exist.  The one exception is `--from-port`, for the two recordings that were added
when no reference checkout was at hand: they are then taken from
oracle/carenv_port.py and from ppo_car_b200.train_ppo.ActorCritic, which were
unchanged since they last matched the reference in the live tests (the port bit
for bit on the near-wall track, the network's checkpoint loading strictly into
lib/model.py:Agent with outputs within 1e-6).  Each file names its source.

Files written:
  carenv_<track>.npz   reset observation + four trajectory groups, each with the
                       action tensor that was played and every per-step output
  gae.npz              Buffer.calculate_advantages on seeded inputs
  near_wall.npz, near_wall_track.json
                       the start_destroyed branch (lib/car_env.py:682-686): a
                       synthetic track whose start pose is 6 px from a wall and
                       one trajectory group ("destroyed") in the layout above
  agent_checkpoint.npz a state dict of lib/model.py:Agent (seeded init) and its
                       log-probability, entropy and value on fixed inputs
  fused_tc3.npz        NOT from the reference: `python tests/golden/make_golden.py
                       fused_tc3` on a GPU records a fused rollout of this
                       repository's tensor-core kernel (k_policy_rollout_tc3)
                       with the agent_checkpoint.npz weights, so that
                       tests/test_fused_rollout.py can require the same bits
                       from every later build
  ../../ppo_car_b200/tracks/<track>.json   the two track files (input data in the
                       reference's schema; BASELINE.json names them as workloads)
"""
from __future__ import annotations

import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from oracle.carenv_port import PortVecEnv  # noqa: E402
from oracle.ref_import import RefVecEnv, import_reference, reference_root, track_path  # noqa: E402
from tests.synth_tracks import near_wall_track  # noqa: E402

T = 1024


def follower_action(obs: np.ndarray) -> int:
    """Closed-loop ray follower (SURVEY §4): steers towards the side with more room."""
    d = obs[6:18]
    speed = 10.0 * float(np.hypot(obs[2], obs[3]))
    left = d[11] + 0.5 * d[10]
    right = d[1] + 0.5 * d[2]
    turn = 0 if abs(left - right) < 0.005 else (1 if right > left else -1)
    if speed < 3:
        return {0: 0, 1: 5, -1: 4}[turn]
    return {0: 8, 1: 3, -1: 2}[turn]


def rollout(track: str, n_envs: int, policy, vec_env=RefVecEnv) -> dict:
    env = vec_env(n_envs, track)
    obs = env.reset()
    rec = {k: [] for k in ("actions", "final_obs", "rew", "term", "trunc", "gates_passed", "time_passed", "next_gate_index")}
    for t in range(T):
        a = np.asarray(policy(t, obs), dtype=np.uint8)
        obs, rew, term, trunc, info = env.step(a)
        rec["actions"].append(a)
        rec["final_obs"].append(info["final_obs"])
        rec["rew"].append(rew)
        rec["term"].append(term)
        rec["trunc"].append(trunc)
        for k in ("gates_passed", "time_passed", "next_gate_index"):
            rec[k].append(info[k])
    return {k: np.stack(v) for k, v in rec.items()}


def make_track(name: str) -> None:
    path = track_path(name + ".json")
    CarEnv, _ = import_reference()
    env = CarEnv(track_path=path)
    reset_obs, _ = env.reset(options={"track_path": path})
    car = env._CarEnv__car
    reset_dist = np.array(car.get_distances(env._CarEnv__boundaries), np.float64)
    out = dict(reset_obs=reset_obs, reset_dist=reset_dist)

    rng = np.random.default_rng(20240)
    groups = {
        # env i plays constant action i: collisions (0,1,4-7) and the 1000-step truncation (2,3,8)
        "const": (9, lambda t, obs: np.arange(9)),
        # closed-loop controller: completes laps (+10 branch) and reaches truncation
        "lap": (1, lambda t, obs: [follower_action(obs[0])]),
        # i.i.d. uniform actions (the benchmark's action distribution)
        "random": (8, lambda t, obs: rng.integers(0, 9, size=8)),
        # forward-biased random actions: many more gate hits per episode
        "fwd": (8, lambda t, obs: rng.choice(9, size=8, p=[.3, .02, .1, .1, .2, .2, .02, .02, .04])),
    }
    for gname, (n, pol) in groups.items():
        rec = rollout(path, n, pol)
        for k, v in rec.items():
            out[f"{gname}_{k}"] = v
        print(name, gname, "episodes ended:", int(rec["term"].sum()), "term,", int(rec["trunc"].sum()),
              "trunc; gate hits:", int((np.diff(rec["gates_passed"], axis=0) > 0).sum()),
              "lap rewards:", int((rec["rew"] > 10).sum()), flush=True)
    np.savez_compressed(os.path.join(HERE, f"carenv_{name}.npz"), **out)

    # re-serialise the track (input data, reference schema) next to the package
    with open(path) as fh:
        data = json.load(fh)
    dst = os.path.join(ROOT, "ppo_car_b200", "tracks", name + ".json")
    with open(dst, "w") as fh:
        json.dump(data, fh)


def make_gae() -> None:
    import torch

    _, Buffer = import_reference()
    out = {}
    for tag, (T_, N_, seed) in {"small": (37, 5, 1), "train": (1024, 24, 2), "wide": (64, 1000, 3)}.items():
        g = torch.Generator().manual_seed(seed)
        buf = Buffer((18,), T_, N_, "cpu", gamma=0.99, gae_lambda=0.95)
        buf.rew_buf = torch.rand((T_, N_), generator=g) * 1.4 - 0.3
        buf.val_buf = torch.randn((T_, N_), generator=g)
        buf.term_buf = (torch.rand((T_, N_), generator=g) < 0.05).float()
        buf.trunc_buf = (torch.rand((T_, N_), generator=g) < 0.02).float()
        buf.ptr = T_
        lv = torch.randn((1, N_), generator=g)
        lt = (torch.rand((1, N_), generator=g) < 0.1).float()
        lu = (torch.rand((1, N_), generator=g) < 0.1).float()
        adv, ret = buf.calculate_advantages(lv, lt, lu)
        for k, v in dict(rew=buf.rew_buf, val=buf.val_buf, term=buf.term_buf, trunc=buf.trunc_buf,
                         last_val=lv, last_term=lt, last_trunc=lu, adv=adv, ret=ret).items():
            out[f"{tag}_{k}"] = v.numpy()
    np.savez_compressed(os.path.join(HERE, "gae.npz"), **out)


def make_near_wall(from_port: bool) -> None:
    path = near_wall_track(os.path.join(HERE, "near_wall_track.json"))
    vec_env = PortVecEnv if from_port else RefVecEnv
    rng = np.random.default_rng(682)

    def policy(t, obs):
        a = rng.choice(9, size=6, p=[.3, .02, .1, .1, .2, .2, .02, .02, .04])
        a[0] = 0                                              # one env at full throttle
        return a

    reset_obs = vec_env(1, path).reset()[0]
    rec = rollout(path, 6, policy, vec_env)
    out = {f"destroyed_{k}": v for k, v in rec.items()}
    source = "oracle/carenv_port.py" if from_port else "lib/car_env.py"
    np.savez_compressed(os.path.join(HERE, "near_wall.npz"), reset_obs=reset_obs, source=np.array(source), **out)


def make_agent(from_port: bool) -> None:
    import importlib

    import torch

    if from_port:
        from ppo_car_b200.train_ppo import ActorCritic as Agent

        source = "ppo_car_b200/train_ppo.py:ActorCritic"
    else:
        root = reference_root()
        if root not in sys.path:
            sys.path.insert(0, root)
        Agent, source = importlib.import_module("lib.model").Agent, "lib/model.py:Agent"
    torch.manual_seed(3)
    net = Agent(18, 9)
    obs = torch.randn(32, 18)
    act = torch.randint(0, 9, (32,))
    with torch.no_grad():
        if from_port:
            _, logp, ent, val = net.act(obs, act)
        else:
            _, logp, ent, val = net.get_action_and_value(obs, act)
    out = {"w_" + k: v.numpy() for k, v in net.state_dict().items()}
    np.savez_compressed(os.path.join(HERE, "agent_checkpoint.npz"), obs=obs.numpy(), act=act.numpy(),
                        logp=logp.numpy(), entropy=ent.numpy(), value=val.numpy(), source=np.array(source), **out)


FUSED_TC3 = dict(n_envs=300, n_steps=64, seed=21, step0=7)   # one full 256-env CTA and a ragged one


def fused_tc3_rollout(tc_tiles: int = 0) -> dict:
    """The rollout pinned by fused_tc3.npz: the agent_checkpoint.npz network on big_track through
    ppo_car_b200.fused_rollout (tensor-core packing), with the handle option tc_tiles set to `tc_tiles`."""
    import torch

    import ppo_car_b200
    from ppo_car_b200.train_ppo import ActorCritic

    dev = torch.device("cuda")
    ck = np.load(os.path.join(HERE, "agent_checkpoint.npz"))
    net = ActorCritic(18, 9).to(dev)
    net.load_state_dict({k[2:]: torch.from_numpy(ck[k]) for k in ck.files if k.startswith("w_")})
    n, T = FUSED_TC3["n_envs"], FUSED_TC3["n_steps"]
    env = ppo_car_b200.VecCarEnv(n, ppo_car_b200.builtin_track("big_track"), reward_scaling=0.1, float_flags=True)
    env.set_option("tc_tiles", tc_tiles)
    buf = ppo_car_b200.Buffer((18,), T, n, dev)
    cur_obs = env.reset()[0].clone()
    cur_term, cur_trunc, last_val = (torch.zeros(n, device=dev), torch.zeros(n, device=dev),
                                     torch.empty(n, device=dev))
    packed = ppo_car_b200.pack_policy_weights_tc(net.actor, net.critic)
    ppo_car_b200.fused_rollout(env, packed, buf, cur_obs, cur_term, cur_trunc, seed=FUSED_TC3["seed"],
                               step0=FUSED_TC3["step0"], last_val=last_val)
    torch.cuda.synchronize()
    return dict(act_buf=buf.act_buf.to(torch.uint8).cpu().numpy(), logprob_buf=buf.logprob_buf.cpu().numpy(),
                val_buf=buf.val_buf.cpu().numpy(), rew_buf=buf.rew_buf.cpu().numpy(),
                last_val=last_val.cpu().numpy(), cur_obs=cur_obs.cpu().numpy())


def make_fused_tc3() -> None:
    out = fused_tc3_rollout()
    np.savez_compressed(os.path.join(HERE, "fused_tc3.npz"),
                        source=np.array("ppo_car_b200.fused_rollout: k_policy_rollout_tc3"), **out)


if __name__ == "__main__":
    from_port = "--from-port" in sys.argv
    which = [w for w in sys.argv[1:] if w != "--from-port"] or ["track", "big_track", "gae", "near_wall", "agent"]
    for w in which:
        if w == "gae":
            make_gae()
        elif w == "near_wall":
            make_near_wall(from_port)
        elif w == "agent":
            make_agent(from_port)
        elif w == "fused_tc3":
            make_fused_tc3()
        else:
            make_track(w)
    print("done")
