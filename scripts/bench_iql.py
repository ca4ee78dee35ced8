"""Device-resident IQL training (BatchedIQL + BatchedIQLTrainer on csrc/tsc_iql.cu) on one GPU: one JSON line per
(model, scenario).

  python scripts/bench_iql.py [--models lr,dqn] [--scenarios grid,real] [--grid-replicas 8192] [--real-replicas 2048]
                              [--steps 40] [--td-reps 10] [--out-dir DIR]

Per line: agent-env-steps/s of the whole loop (forward, simulator, reward hand-over, the update every batch_size steps),
ms per control step split into simulator / Q forward / update (an update's time divided by batch_size), and the TD
kernel (tscl_iql_td_grad: TD kernel + fixed-order partial reduction) timed on its own over --td-reps calls, with the
FLOP and bytes it needs computed from the shapes below, the achieved rates, the share of the fp32 CUDA-core peak
(SM count x 128 lanes x 2 x max SM clock, read in the same run) and of 7.7 TB/s HBM bandwidth, and the bound: the peak
reached to at least one half, else neither.  GPU name and power limit are read in the same run.  Every shape is warmed before timing (the window
starts after at least two updates); times come from CUDA events.  There is no CPU path: without a GPU the script fails.
"""
import argparse
import configparser
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from deeprl_signal_control_b200.agents.learner_iql import BatchedIQL, N_ITER            # noqa: E402
from deeprl_signal_control_b200.agents.trainer import BatchedIQLTrainer                 # noqa: E402
from deeprl_signal_control_b200.net.tables import EnvParams                             # noqa: E402
from deeprl_signal_control_b200.sim import BatchedSim                                   # noqa: E402

HBM_BPS = 7.7e12
# config/config_iql{l,d}_{large,real}.ini of the reference
INI = """
[MODEL_CONFIG]
max_grad_norm = 40
gamma = 0.99
lr_init = 1e-4
lr_decay = constant
epsilon_init = 1.0
epsilon_min = 0.01
epsilon_decay = linear
epsilon_ratio = 0.5
num_fc = 128
num_h = 64
batch_size = 20
buffer_size = 1000
reward_norm = 3000.0
reward_clip = 2.0
"""


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits",
                        "-i", str(torch.cuda.current_device())], capture_output=True, text=True, check=True).stdout
    name, power, clk = [x.strip() for x in q.strip().split(",")]
    return dict(gpu=name, power_limit_w=float(power), max_sm_clock_mhz=float(clk),
                sm_count=torch.cuda.get_device_properties(0).multi_processor_count)


def scenario(name, agent):
    if name == "real":
        from deeprl_signal_control_b200.net.real_net import real_net_tables
        par = EnvParams(agent=agent, objective="queue", norm_wave=5.0, norm_wait=30.0, clip_wave=2.0, clip_wait=2.0,
                        coef_wait=0.0, coop_gamma=0.9, teleport_sec=300, real_net_norm=True, use_wait=False, det_len=-1.0,
                        halt_speed=0.1, queue_cap=10)
        return real_net_tables(agent), par, 1.0
    from deeprl_signal_control_b200.net.large_grid import build_large_grid
    return build_large_grid(agent=agent), EnvParams(agent=agent), 3000.0


def td_counts(m, B):
    """FLOP and bytes of one tscl_iql_td_grad call, from the shapes.  Per row: forward on s' and on s, weight gradients
    of every layer (the forward's MACs again) and, for dqn, the back-propagation into the first hidden layer.  Bytes:
    the gathered rows (s and s', action, reward, index, done) plus the per-CTA gradient partials (written by the TD
    kernel, read by the reduction) and the weights every CTA stages."""
    A, R = m.n_agent, m.R
    nf, nh = (m._cd.num_fc, m._cd.num_h)
    flop = byt = 0.0
    n_cta = max(1, min((296 if m.model_type == "dqn" else 1184) // A, (R * B + 63) // 64))   # csrc/tsc_iql.cu IQ_CTAS*
    for n_s, n_a, n_w in zip(m.n_s_ls, m.n_a_ls, m.n_w_ls):
        if m.model_type == "dqn":
            nt4 = nf // 4 if n_w > 0 else 0
            width = nf + nt4
            fwd = (n_s - n_w) * nf + n_w * nt4 + width * nh + nh * n_a
            mac = 3 * fwd + width * nh
        else:
            mac = 3 * n_s * n_a
        flop += 2.0 * mac * R * B
        byt += R * B * (2 * n_s + 4) * 4.0
    P = float(m.P.numel())
    byt += n_cta * P * 4.0 * 3            # staged weights, partials written, partials read
    return flop, byt


def run(model, scen, R, steps, td_reps, info):
    agent = "iqld" if model == "dqn" else "iqll"
    net, par, reward_norm = scenario(scen, agent)
    cp = configparser.ConfigParser(); cp.read_string(INI)
    cp["MODEL_CONFIG"]["reward_norm"] = str(reward_norm)
    sim = BatchedSim(net, par, R)
    m = BatchedIQL(net.n_s_ls, net.n_a_ls, net.n_w_ls, net.node_obs_off, net.n_obs, R, 1e6, cp["MODEL_CONFIG"], seed=1,
                   model_type=model)
    tr = BatchedIQLTrainer(sim, m, seed0=12)
    B = m.n_step
    tr.run(2 * B)                                         # two updates: every shape and buffer is warm
    torch.cuda.synchronize()
    assert tr.n_updates == 2
    tr.fwd_events, tr.sim_events, tr.update_events = [], [], []
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n_upd0 = tr.n_updates
    e0.record()
    tr.run(steps)
    e1.record()
    torch.cuda.synchronize()
    total_ms = e0.elapsed_time(e1)
    span = lambda ev: sum(a.elapsed_time(b) for a, b in ev)
    A = net.n_nodes
    # the TD kernel alone, on the ring the run filled
    idx = m.sample(10 ** 6, 0)
    m.td_grad(idx)
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(td_reps):
        m.td_grad(idx)
    t1.record()
    torch.cuda.synchronize()
    td_ms = t0.elapsed_time(t1) / td_reps
    flop, byt = td_counts(m, B)
    peak_flops = info["sm_count"] * 128 * 2 * info["max_sm_clock_mhz"] * 1e6
    f_share, b_share = flop / (td_ms * 1e-3) / peak_flops, byt / (td_ms * 1e-3) / HBM_BPS
    return dict(
        bench="iql_train", model=model, scenario=scen, agent=agent, replicas=R, agents=A, steps=steps,
        updates_in_window=tr.n_updates - n_upd0, batch_size=B, iterations_per_update=N_ITER, buffer_size=m.C,
        agent_env_steps_per_s=R * A * steps / (total_ms * 1e-3),
        ms_per_control_step=dict(total=total_ms / steps, simulator=span(tr.sim_events) / steps,
                                 q_forward=span(tr.fwd_events) / steps, update=span(tr.update_events) / steps,
                                 one_update=span(tr.update_events) / max(1, len(tr.update_events))),
        td_grad=dict(ms_per_call=td_ms, calls_per_update=N_ITER, flop=flop, bytes=byt,
                     tflop_per_s=flop / (td_ms * 1e-3) / 1e12, gb_per_s=byt / (td_ms * 1e-3) / 1e9,
                     share_of_fp32_cuda_core_peak=f_share, share_of_hbm_bandwidth=b_share,
                     fp32_cuda_core_peak_tflop_per_s=peak_flops / 1e12,
                     bound=("fp32 compute" if f_share >= 0.5 else "memory bandwidth" if b_share >= 0.5 else
                            "neither peak (under half of both): on-chip traffic / latency")),
        ring_gb=(m.obs_ring.numel() + m.act_ring.numel() + m.rew_ring.numel()) * 4 / 1e9,
        mean_loss=float(m.stats[:, 0].mean()), **info)


def main():
    p = argparse.ArgumentParser()
    p.add_argument("--models", default="lr,dqn")
    p.add_argument("--scenarios", default="grid,real")
    p.add_argument("--grid-replicas", type=int, default=8192)
    p.add_argument("--real-replicas", type=int, default=2048)
    p.add_argument("--steps", type=int, default=40)
    p.add_argument("--td-reps", type=int, default=10)
    p.add_argument("--out-dir", default=None)
    a = p.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_iql.py needs a CUDA device (there is no CPU path)")
    info = gpu_info()
    for scen in a.scenarios.split(","):
        for model in a.models.split(","):
            R = a.grid_replicas if scen == "grid" else a.real_replicas
            line = json.dumps(run(model, scen, R, a.steps, a.td_reps, info))
            print(line, flush=True)
            if a.out_dir:
                os.makedirs(a.out_dir, exist_ok=True)
                with open(os.path.join(a.out_dir, "bench_iql_%s_%s.json" % (model, scen)), "w") as f:
                    f.write(line + "\n")
            torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
