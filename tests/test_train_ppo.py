"""PPO loop harness (SURVEY §8 f-1): network/update math on CPU, a short real run on the GPU."""
import math

import pytest
import torch

from ppo_car_b200.train_ppo import ActorCritic, parse_args, train


def test_actor_critic_matches_reference_model_semantics():
    torch.manual_seed(0)
    net = ActorCritic(18, 9)
    assert sum(p.numel() for p in net.parameters()) == 12298          # SURVEY §2 row 6
    # orthogonal init with the reference's gains (lib/model.py:13-24): rows of the last layers are scaled
    w = net.actor[2].weight
    assert torch.allclose(w @ w.T, 0.01 ** 2 * torch.eye(9), atol=1e-6)
    w = net.critic[2].weight
    assert torch.allclose(w @ w.T, torch.eye(1), atol=1e-6)
    obs = torch.randn(64, 18)
    act, logp, ent, val = net.act(obs)
    dist = torch.distributions.Categorical(logits=net.actor(obs))       # what lib/model.py:34-40 uses
    assert torch.allclose(logp, dist.log_prob(act), atol=1e-6) and torch.allclose(ent, dist.entropy(), atol=1e-6)
    assert val.shape == (64, 1) and act.dtype == torch.int64
    a2, logp2, _, _ = net.act(obs, act.float())                         # actions come back from a float32 buffer
    assert torch.equal(a2, act.float()) and torch.allclose(logp2, logp)


def test_flag_defaults_match_reference_train_py():
    a = parse_args([])
    assert (a.n_envs, a.n_epochs, a.n_steps, a.batch_size, a.train_iters) == (16, 200, 1024, 512, 40)
    assert (a.gamma, a.gae_lambda, a.clip_ratio, a.ent_coef, a.vf_coef) == (0.99, 0.95, 0.2, 0.001, 0.5)
    assert (a.learning_rate, a.learning_rate_decay, a.max_grad_norm, a.reward_scaling) == (3e-4, 0.99, 1.0, 0.1)


@pytest.mark.gpu
def test_short_training_run_improves_reward():
    args = parse_args(["--track", "big_track", "--n-envs", "64", "--n-epochs", "12", "--n-steps", "256"])
    hist = train(args)
    assert len(hist) == 12 and all(math.isfinite(h["total_loss"]) for h in hist)
    assert hist[-1]["avg_reward"] > hist[0]["avg_reward"] + 0.03       # random policy is about 0.0


@pytest.mark.gpu
def test_cuda_graph_rollout_trains():
    args = parse_args(["--track", "track", "--n-envs", "32", "--n-epochs", "10", "--n-steps", "256", "--cuda-graph"])
    hist = train(args)
    assert all(math.isfinite(h["total_loss"]) for h in hist)
    assert hist[-1]["avg_reward"] > hist[0]["avg_reward"] + 0.02
    assert hist[0]["episodes"] > 0


@pytest.mark.gpu
def test_graph_update_trains():
    args = parse_args(["--track", "big_track", "--n-envs", "64", "--n-epochs", "12", "--n-steps", "256",
                       "--fused-rollout", "--graph-update"])
    hist = train(args)
    assert all(math.isfinite(h["total_loss"]) for h in hist)
    assert hist[-1]["avg_reward"] > hist[0]["avg_reward"] + 0.03
    assert abs(hist[-1]["lr"] - 3e-4 * 0.99 ** 12) < 1e-9


def test_state_dict_loads_into_the_reference_agent(golden_dir):
    """The checkpoints train_ppo writes (train.py:280-283, 301) carry the reference Agent's keys: the stored Agent
    checkpoint (tests/golden/agent_checkpoint.npz, its `source` names what recorded it) loads strictly into this
    harness's network, which then computes the stored outputs; where the UNMODIFIED lib/model.py is present, a state
    dict of this network also loads strictly into its Agent and both compute the same outputs."""
    import importlib
    import os
    import sys

    import numpy as np

    from oracle.ref_import import reference_root

    g = np.load(os.path.join(golden_dir, "agent_checkpoint.npz"))
    net = ActorCritic(18, 9)
    net.load_state_dict({k[2:]: torch.from_numpy(g[k]) for k in g.files if k.startswith("w_")}, strict=True)
    with torch.no_grad():
        _, logp, ent, val = net.act(torch.from_numpy(g["obs"]), torch.from_numpy(g["act"]))
    assert torch.allclose(logp, torch.from_numpy(g["logp"]), atol=1e-6)
    assert torch.allclose(ent, torch.from_numpy(g["entropy"]), atol=1e-6)
    assert val.shape == g["value"].shape and torch.allclose(val, torch.from_numpy(g["value"]), atol=1e-6)

    root = reference_root()
    if root is None:
        return
    if not os.path.isfile(os.path.join(root, "lib", "model.py")):
        pytest.skip("lib/model.py not in the reference copy (re-run oracle/make_ref.py)")
    if root not in sys.path:
        sys.path.insert(0, root)
    Agent = importlib.import_module("lib.model").Agent
    torch.manual_seed(3)
    ours, ref = ActorCritic(18, 9), Agent(18, 9)
    ref.load_state_dict(ours.state_dict(), strict=True)
    obs = torch.randn(32, 18)
    act, logp, ent, val = ours.act(obs)
    a2, logp2, ent2, val2 = ref.get_action_and_value(obs, act)
    assert torch.equal(a2, act) and torch.allclose(logp, logp2, atol=1e-6) and torch.allclose(ent, ent2, atol=1e-6)
    assert torch.allclose(val, val2, atol=1e-6)
