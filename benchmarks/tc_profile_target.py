"""Target for `ncu --set full -k regex:k_policy_rollout_tc3`: three fused tensor-core rollouts of 8 steps.
    python benchmarks/tc_profile_target.py [n_envs]     (default 262,144; 32,768 = one 256-env CTA per SM on 128 SMs,
                                                          the shard size of BASELINE config 5 on 8 GPUs)"""
import torch, sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import ppo_car_b200
from ppo_car_b200.train_ppo import ActorCritic
dev = torch.device("cuda"); torch.manual_seed(0)
net = ActorCritic(18, 9).to(dev)
packed = ppo_car_b200.pack_policy_weights_tc(net.actor, net.critic)
n, T = int(sys.argv[1]) if len(sys.argv) > 1 else 262144, 8
env = ppo_car_b200.VecCarEnv(n, ppo_car_b200.builtin_track("big_track"), reward_scaling=0.1, float_flags=True, with_info=False)
buf = ppo_car_b200.Buffer((18,), T, n, dev)
obs = env.reset()[0].clone(); term = torch.zeros(n, device=dev); trunc = torch.zeros(n, device=dev); lv = torch.empty(n, device=dev)
for i in range(3):
    ppo_car_b200.fused_rollout(env, packed, buf, obs, term, trunc, seed=1, step0=i*T, last_val=lv)
torch.cuda.synchronize()
print("ok")
