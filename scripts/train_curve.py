"""Training curves of the device-resident learner on the restated simulator, and the greedy controller's score on the
same episodes (reference utils.py:296-305: mean over the 720 control steps of the global reward, averaged over replicas).

  python scripts/train_curve.py --replicas 512 --episodes 300 --agent ma2c|ia2c|iqll|iqld [--scenario grid|real] [--policy lstm|fc]
                                [--fp32] [--reward-norm X] [--lr X] [--tag NAME] [--greedy]

--fp32         plain fp32 learner kernels (no tensor cores, no bf16 activation store): the A/B partner of the default path
--reward-norm  override MODEL_CONFIG.reward_norm (reference: 2000 for MA2C on the grid, config/config_ma2c_large.ini)
--agent iqll|iqld   batched IQL-LR / IQL-DQN (BatchedIQL + BatchedIQLTrainer); --lr sets lr_init (reference: 1e-4),
               --total-step the length of the epsilon / lr schedules (default: 720 x --episodes)
--greedy       no learning: the reference's greedy controller (envs/large_grid_env.py:56-60) on the same seeds
Writes gpurun_out/train_curve_<tag>.json.
"""
import argparse
import json
import sys
import time

import numpy as np
import torch

sys.path.insert(0, ".")
from deeprl_signal_control_b200.agents.layout import PolicyLayout
from deeprl_signal_control_b200.agents.learner import BatchedA2C
from deeprl_signal_control_b200.agents.trainer import BatchedTrainer
from deeprl_signal_control_b200.dist import episode_seeds
from deeprl_signal_control_b200.net.large_grid import build_large_grid
from deeprl_signal_control_b200.net.tables import EnvParams
from deeprl_signal_control_b200.sim import BatchedSim

p = argparse.ArgumentParser()
p.add_argument("--replicas", type=int, default=512)
p.add_argument("--episodes", type=int, default=24)
p.add_argument("--agent", default="ma2c")
p.add_argument("--scenario", default="grid", choices=["grid", "real"])
p.add_argument("--policy", default="lstm", choices=["lstm", "fc"])
p.add_argument("--fp32", action="store_true")
p.add_argument("--reward-norm", type=float, default=None)
p.add_argument("--lr", type=float, default=5e-4)
p.add_argument("--seed", type=int, default=1)
p.add_argument("--tag", default=None)
p.add_argument("--greedy", action="store_true")
p.add_argument("--total-step", type=float, default=None)
a = p.parse_args()
R, agent = a.replicas, a.agent
tag = a.tag or "%s_%s_%s%s" % (agent, a.scenario, a.policy, "_fp32" if a.fp32 else "")

if a.scenario == "real":
    from deeprl_signal_control_b200.net.real_net import real_net_tables
    net = real_net_tables("greedy" if a.greedy else agent)
    par = EnvParams(agent="greedy" if a.greedy else agent, objective="queue", norm_wave=5.0, norm_wait=30.0, clip_wave=2.0,
                    clip_wait=2.0, coef_wait=0.0, coop_gamma=0.9, teleport_sec=300, real_net_norm=True, use_wait=False,
                    det_len=-1.0, halt_speed=0.1, queue_cap=10)
    n_step, reward_norm = 40, 1.0
else:
    net = build_large_grid(agent="greedy" if a.greedy else agent)
    par = EnvParams(agent="greedy" if a.greedy else agent)
    n_step, reward_norm = 120, 2000.0 if agent == "ma2c" else 3000.0
if a.reward_norm is not None:
    reward_norm = a.reward_norm
sim = BatchedSim(net, par, R)
t0 = time.time()

if a.greedy:
    assert a.scenario == "grid", "greedy baseline: grid only"
    sim.set_train_mode(True)
    off = torch.tensor(net.node_obs_off[:net.n_nodes], device="cuda")
    idx = (off[:, None] + torch.arange(6, device="cuda")[None, :]).reshape(-1)
    curve = []
    for ep in range(a.episodes):
        sim.reset(episode_seeds(12, ep, 0, R, R))
        obs = sim.observe()
        acc = torch.zeros(R, device="cuda")
        for t in range(720):
            o = obs[:, idx].reshape(R, net.n_nodes, 6)
            flows = torch.stack([o[..., 0] + o[..., 3], o[..., 2] + o[..., 5], o[..., 1] + o[..., 4],
                                 o[..., 1] + o[..., 2], o[..., 4] + o[..., 5]], -1)
            act = flows.argmax(-1).to(torch.int32).contiguous()
            obs, _, g, _ = sim.step(act)
            acc += g
        curve.append(float((acc / 720).mean()))
        print("greedy episode %3d  mean step reward %9.2f" % (ep + 1, curve[-1]), flush=True)
    json.dump({"agent": "greedy", "scenario": a.scenario, "replicas": R, "episodes": len(curve), "mean_episode_reward": curve,
               "wall_s": time.time() - t0}, open("gpurun_out/train_curve_%s.json" % tag, "w"))
    sys.exit(0)

if agent in ("iqll", "iqld"):
    # IQL-LR / IQL-DQN (config/config_iql{l,d}_large.ini of the reference); the epsilon schedule decays over half of
    # --total-step control steps (default: the run's own length), lr = --lr
    import configparser
    from deeprl_signal_control_b200.agents.learner_iql import BatchedIQL
    from deeprl_signal_control_b200.agents.trainer import BatchedIQLTrainer
    cp = configparser.ConfigParser()
    cp.read_string("[MODEL_CONFIG]\nmax_grad_norm = 40\ngamma = 0.99\nlr_init = %g\nlr_decay = constant\n"
                   "epsilon_init = 1.0\nepsilon_min = 0.01\nepsilon_decay = linear\nepsilon_ratio = 0.5\nnum_fc = 128\n"
                   "num_h = 64\nbatch_size = 20\nbuffer_size = 1000\nreward_norm = %g\nreward_clip = 2.0\n"
                   % (a.lr, reward_norm))
    total_step = a.total_step or 720 * a.episodes
    model = BatchedIQL(net.n_s_ls, net.n_a_ls, net.n_w_ls, net.node_obs_off, net.n_obs, R, total_step, cp["MODEL_CONFIG"],
                       seed=a.seed, model_type="dqn" if agent == "iqld" else "lr")
    tr = BatchedIQLTrainer(sim, model, seed0=12)
    extra = {"total_step": total_step}
else:
    lay = PolicyLayout(net.n_s_ls, net.n_a_ls, net.n_w_ls, net.n_f_ls, net.node_obs_off, net.n_obs, fw=128, ft=32,
                       ff=64 if agent == "ma2c" else 0, h=64, max_na=net.max_na, recurrent=a.policy != "fc")
    kw = dict(use_tc=False, allow_tf32=False) if a.fp32 else {}
    if a.policy == "fc":
        from deeprl_signal_control_b200.agents.learner_fc import BatchedFcA2C as Learner
        kw = {}
    else:
        Learner = BatchedA2C
    model = Learner(lay, R, n_step=n_step, gamma=0.99, v_coef=0.5, max_grad_norm=40.0, alpha=0.99, eps=1e-5,
                    reward_norm=reward_norm, reward_clip=2.0, seed=a.seed, chunk=min(R, 1024), **kw)
    tr = BatchedTrainer(sim, model, agent, lr=a.lr, beta=0.01, seed0=12)
    extra = {"policy": a.policy, "fp32": bool(a.fp32)}
curve = []
while len(tr.episode_rewards) < a.episodes:
    tr.run(720)
    torch.cuda.synchronize()
    curve = list(tr.episode_rewards)
    if len(curve) % 10 == 0 or len(curve) == a.episodes:
        print("episode %3d  mean step reward %9.2f   grad-norm[0] %.3f   %.1fs" %
              (len(curve), curve[-1], float(model.norms[0]), time.time() - t0), flush=True)
json.dump({"agent": agent, "scenario": a.scenario, "replicas": R, "episodes": len(curve), "reward_norm": reward_norm,
           "lr": a.lr, "mean_episode_reward": curve, "wall_s": time.time() - t0, "env_steps": tr.n_env_steps, **extra},
          open("gpurun_out/train_curve_%s.json" % tag, "w"))
