#!/usr/bin/env python
"""bench.py — agent-env-steps/sec of the 5x5 large_grid MA2C hot path on N B200s (one node).

Contract: `python bench.py --gpus N --steps K --warmup W` (N>1: launched by torchrun, one rank
per GPU).  Prints ONE JSON line on rank 0.

Workload (BASELINE.json configs[2]): 5x5 large_grid, MA2C observation layout (n_s in {32,42,52},
fingerprints), `--replicas` (default 8192) lock-stepped env replicas PER GPU ("weak" scaling),
synthetic demand of the named grid (large_grid/data/build_file.py flows 1100/925), replica r of
rank k seeded with seed0 + k*R + r.

A "step" is one control step (5 simulated seconds) of all local replicas:
   --mode sim   (default until the learner kernels land): uniform-random actions + fingerprints
                resident on the device -> tsc_step (one launch of tsc_step_kernel)
   --mode train: MA2C policy forward + sampling + tsc_step + transition store, and one n-step
                A2C update every n_step control steps (see deeprl_signal_control_b200.agents)
Before timing, every replica is advanced `--burnin` control steps (default 240 = 1200 simulated
seconds, the demand peak) so that the timed steps see a loaded network; burn-in is state
preparation, the W warm-up steps are on top of it.

value = (replicas over all ranks) * agents (25 grid / 28 Monaco) * K / max-over-ranks(device time of K steps).
e2e   = same metric through the host-buffer entry point tsc_step_host (actions/fingerprints in
        pinned host memory -> H2D, kernel, obs/reward/done -> D2H, every step).
roofline = tsc_step_kernel: algorithmic bytes (BASELINE.md §3 formula with the measured mean
        live vehicles) / mean launch duration (CUDA events around every launch) vs measured HBM peak.
cpu_baseline / --impl reference = the CPU port of the SAME work (SUMO + TF1 are absent): oracle/tsc_sim_ref.c on all
        usable host threads (cgroup cpu.max respected) for the control step and, in train mode, oracle/learner_cpu.py
        (torch CPU fp32, all threads) for the policy forward of every step and one n-step A2C update per n_step —
        a bounded sample of replicas, named in `sample`.  --impl reference times exactly --steps control steps after
        the burn-in, which must both fit in one episode (past its end the network drains: a different workload); the
        cpu_baseline of our arm times the same --steps, cut at the episode end, and reports its count in `steps`.
--scenario real_net = BASELINE configs[3] (Monaco, 28 agents, MA2C, 2048 replicas, n_step 40,
        config/config_ma2c_real.ini); the default large_grid = configs[2].
value_steady = the same metric with the update amortised over n_step control steps (the driver's short --steps
        window is forced to contain one whole update, which over-weights it; both numbers are printed).
--dump-outputs DIR = after the timed steps, what the timed path computed in its last step is written as DIR/<name>.npy
        (float32, see last_step_outputs); inputs are seeded, so two builds run with the same arguments can be compared
        output for output.  Our arm only: --impl reference times the CPU oracle on its own replica sample and
        inputs, with the learner's share timed apart from the simulator, so it has no last step to compare.
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_STEP = {"large_grid": 120, "real_net": 40}     # batch_size of config/config_ma2c_{large,real}.ini


def usable_cpus():
    """Host threads this process can really use: sched affinity capped by the cgroup CPU quota (cpu.max)."""
    n = len(os.sched_getaffinity(0))
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    n = min(n, max(1, int(float(txt[0]) / float(txt[1]))))
            else:
                q = int(txt[0])
                per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
                if q > 0:
                    n = min(n, max(1, q // per))
        except Exception:
            pass
    return n


def parse():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=120)
    p.add_argument("--warmup", type=int, default=5)
    p.add_argument("--impl", default="ours", choices=["ours", "reference"])
    p.add_argument("--scenario", default="large_grid", choices=["large_grid", "real_net"],
                   help="large_grid = BASELINE configs[2] (headline); real_net = configs[3] (Monaco MA2C, 2048 replicas)")
    p.add_argument("--replicas", type=int, default=None, help="env replicas per GPU (default 8192 grid / 2048 Monaco)")
    p.add_argument("--burnin", type=int, default=240)
    p.add_argument("--mode", default=None, choices=[None, "sim", "train"])
    p.add_argument("--chunk", type=int, default=4096,
                   help="replicas per update chunk (4096: 1600 BPTT work items = 10.8 waves of 148 CTAs; 1024: 2.7 waves)")
    p.add_argument("--fp32-gemm", action="store_true", help="plain fp32 (no TF32 tensor cores) in the learner GEMMs")
    p.add_argument("--seed", type=int, default=12)
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--profile-run", action="store_true", help="launch lists under ncu: one e2e window instead of seven")
    p.add_argument("--cpu-budget", type=float, default=20.0, help="seconds of CPU work of the oracle sample (both arms)")
    p.add_argument("--agent", default="ma2c", choices=["ma2c", "ia2c"],
                   help="ma2c = BASELINE configs[2] (the headline workload); ia2c with --policy fc = configs[1]")
    p.add_argument("--policy", default="lstm", choices=["lstm", "fc"], help="fc = FcACPolicy (agents/policies.py:214-256)")
    p.add_argument("--e2e-parts", type=int, default=4,
                   help="replica ranges of the host-buffer (e2e) loop, one stream each (1: single blocking tsc_step_host)")
    p.add_argument("--dump-outputs", metavar="DIR", default=None,
                   help="write what the timed path computed in its last timed step as DIR/<name>.npy")
    args = p.parse_args()
    if args.steps < 1:
        p.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        p.error("--dump-outputs writes the outputs of the device path (--impl ours)")
    return p, args


def workload_name(R, mode, agent="ma2c", policy="lstm", scenario="large_grid"):
    tag = "MA2C (configs[2])" if agent == "ma2c" else ("IA2C, FC policy (configs[1])" if policy == "fc" else "IA2C, LSTM policy")
    if scenario == "real_net":
        tag = "MA2C (configs[3])"
    return ("%s %s, %d env replicas per GPU, %s" %
            ("Monaco real_net 28-intersection" if scenario == "real_net" else "5x5 large_grid", tag, R,
             "policy+sim+update" if mode == "train" else "sim control step, uniform-random actions"))


def build_scenario(args):
    """(net tables, env params, n_step, reward_norm, wave block) of the benchmarked configuration."""
    from deeprl_signal_control_b200.net.tables import EnvParams
    if args.scenario == "real_net":
        from deeprl_signal_control_b200.net.real_net import real_net_tables
        net = real_net_tables(args.agent)
        # config/config_ma2c_real.ini [ENV_CONFIG]: queue objective, wave-only state, norm_wave 5, clip 2
        par = EnvParams(agent=args.agent, objective="queue", norm_wave=5.0, norm_wait=100.0, clip_wave=2.0, clip_wait=2.0,
                        coef_wait=0.0, coop_gamma=0.9, teleport_sec=300, real_net_norm=True, use_wait=False,
                        det_len=-1.0, halt_speed=0.1, queue_cap=10)
        return net, par, N_STEP["real_net"], 1.0
    from deeprl_signal_control_b200.net.large_grid import build_large_grid
    net, par = build_large_grid(agent=args.agent), EnvParams(agent=args.agent)
    return net, par, N_STEP["large_grid"], (2000.0 if args.agent == "ma2c" else 3000.0)


def algorithmic_bytes(net, v_live):
    """BASELINE.md §3: B_step = 2*V*16 + 2*L*8 + 2*A*4 + 4*A + 4*sum(N_s) + 4*A + 4 + 1."""
    L, A = net.n_lanes, net.n_nodes
    return 2 * v_live * 16 + 2 * L * 8 + 2 * A * 4 + 4 * A + 4 * net.n_obs + 4 * A + 4 + 1


# ------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons of one GPU every 100 ms while running."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag = index, [], set(), False
        self.max_mhz = None

    def run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            names = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown",
                     0x4: "sw_power_cap", 0x80: "hw_power_brake"}
            while not self.stop_flag:
                self.samples.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
                time.sleep(0.1)
        except Exception as e:  # pragma: no cover
            self.reasons.add("sampler_error:%s" % type(e).__name__)

    def summary(self):
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons)}


# ------------------------------------------------------------------------------------------------
def make_layout(net, args):
    from deeprl_signal_control_b200.agents.layout import PolicyLayout
    # config/config_ma2c_{large,real}.ini [MODEL_CONFIG]: num_fw 128, num_ft 32, num_fp 64, num_lstm 64
    return PolicyLayout(net.n_s_ls, net.n_a_ls, net.n_w_ls, net.n_f_ls, net.node_obs_off, net.n_obs, fw=128, ft=32,
                        ff=64 if args.agent == "ma2c" else 0, h=64, max_na=net.max_na, recurrent=args.policy != "fc")


DUMP_REPLICAS = 1024          # per-replica outputs are dumped for a fixed sample of this many replicas
DUMP_MAX_BYTES = 64 << 20


def last_step_outputs(sim, trainer):
    """What the timed path handed its caller in its last step, as host float32 arrays.
    train: the weights after the step's A2C update (the timed region always ends on one), the per-agent gradient norms
           of that update, and the step's transition: next observation, normalised / clipped reward, sampled actions,
           value estimates.
    sim:   what tsc_step returned: observation, per-agent reward, global reward, done.
    Per-replica arrays keep the replicas of a fixed, seeded sample (at most DUMP_REPLICAS, in ascending order), listed
    in `replicas`."""
    import torch
    rows = np.sort(np.random.default_rng(0).choice(sim.R, min(sim.R, DUMP_REPLICAS), replace=False))
    idx = torch.from_numpy(rows).to(sim.device)
    host = lambda x: x.index_select(0, idx).float().cpu().numpy()
    if trainer is not None:
        m = trainer.model
        assert m.t == 0, "the timed region must end on an update"
        out = {"params": m.P.cpu().numpy(), "grad_norms": m.norms.cpu().numpy(), "obs": host(m.obs_hist[m.T]),
               "reward": host(m.rew_hist[m.T - 1]), "action": host(m.act_hist[m.T - 1]),
               "value": host(m.val_hist[m.T - 1])}
    else:
        out = {"obs": host(sim.obs), "reward": host(sim.reward), "global_reward": host(sim.greward),
               "done": host(sim.done)}
    out["replicas"] = rows.astype(np.float32)
    assert sum(a.nbytes for a in out.values()) <= DUMP_MAX_BYTES
    return out


def episode_steps(par):
    return par.episode_length_sec // par.control_interval_sec


def sim_mode_inputs(net, R, dev, rank, n_act_sets=16):
    """Seeded device inputs of --mode sim: `n_act_sets` sets of uniform-random actions (step i of each phase plays set
    i % n_act_sets) and one set of fingerprints."""
    import torch
    gen = torch.Generator(device=dev)
    gen.manual_seed(1234 + rank)
    n_a_dev = torch.tensor(net.n_a_ls, device=dev, dtype=torch.int64)
    acts = [(torch.randint(0, 1 << 30, (R, net.n_nodes), device=dev, generator=gen) % n_a_dev).to(torch.int32)
            for _ in range(n_act_sets)]
    fp = torch.rand(R, net.n_nodes, net.max_na, device=dev, generator=gen)
    return acts, fp


def cpu_reference(net, par, args, threads, n_step, mode, n_t, budget_s=12.0):
    """Time the CPU port on `threads` host threads over a bounded sample of the workload: R_cpu replicas, burn-in to the
    same simulated time, then n_t timed control steps of the simulator (oracle/tsc_sim_ref.c, pthreads over replicas); in
    train mode the learner's share of the same steps is timed too (oracle/learner_cpu.py: policy forward of every step,
    one n-step update per n_step steps) and added — the reference runs env and learner serially (utils.py:142-193)."""
    from oracle.sim_ref import RefSim
    rng = np.random.default_rng(0)
    na = int(max(net.n_a_ls))
    acts_of = lambda *shape: (rng.integers(0, 1 << 30, shape + (net.n_nodes,)) % np.asarray(net.n_a_ls)).astype(np.int32)
    # pilot: cost of one replica control step on one thread, at a lightly loaded network
    pilot = RefSim(net, par, threads)
    pilot.reset(np.arange(threads, dtype=np.uint64))
    for _ in range(40):
        pilot.step(acts_of(threads), None, threads=threads)
    t0 = time.perf_counter()
    for _ in range(40):
        pilot.step(acts_of(threads), None, threads=threads)
    c_step = (time.perf_counter() - t0) / 40            # seconds per (threads replicas) step
    R_cpu = int(np.clip(budget_s / ((args.burnin + n_t) * c_step * 3.0) * threads, threads, 4096))
    R_cpu = max(threads, R_cpu // threads * threads)
    sim = RefSim(net, par, R_cpu)
    sim.reset(np.arange(R_cpu, dtype=np.uint64) + np.uint64(args.seed))
    fp = rng.random((R_cpu, net.n_nodes, net.max_na), dtype=np.float32)
    acts = acts_of(8, R_cpu)
    # one call per phase: every thread walks its replicas through all the steps (ref_run_mt), threads are created once
    sim.run(acts, args.burnin, fp, threads=threads)
    n, t0 = n_t, time.perf_counter()
    sim.run(acts, n_t, fp, threads=threads)
    el_sim = time.perf_counter() - t0
    live = float(np.mean([sim.misc(r)["live"] for r in range(R_cpu)]))
    el, learner_note = el_sim, "sim control step only (--mode sim)"
    if mode == "train":
        from oracle.learner_cpu import time_learner
        # measured on the 16-core lease: the update costs 60 ms / replica at 128 replicas and 161 ms / replica at 784 (cache
        # footprint of the autograd unroll), so the CPU arm is timed at its more efficient batch and scaled linearly
        R_upd = min(R_cpu, 128)
        t_fwd, t_upd = time_learner(make_layout(net, args), R_cpu, 3, R_upd, n_step, threads)
        el_fwd = t_fwd * n_t                               # one policy forward per control step
        el_upd = t_upd * (R_cpu / R_upd) * (n_t / n_step)  # one n-step update per n_step control steps
        el = el_sim + el_fwd + el_upd
        learner_note = ("+ policy forward of %d replicas x %d steps (%.2f s) + n-step A2C update amortised %.2f/%d steps "
                        "(measured on %d replicas: %.2f s, scaled x%.1f) on torch CPU fp32, %d threads"
                        % (R_cpu, n_t, el_fwd, n_t, n_step, R_upd, t_upd, R_cpu / R_upd, threads))
    return {"value": R_cpu * net.n_nodes * n / el, "unit": "agent-env-steps/s", "cores": threads,
            "kind": "port", "steps": n,
            "sample": "%d replicas x %d control steps after %d burn-in steps (mean live %.0f veh/replica): "
                      "oracle/tsc_sim_ref.c on %d pthreads (%.2f s) %s; SUMO + TF1 are absent from the image, so this is "
                      "the CPU port of the same work, not SUMO / TensorFlow"
                      % (R_cpu, n, args.burnin, live, threads, el_sim, learner_note),
            "sim_only_value": R_cpu * net.n_nodes * n / el_sim}, n, el, R_cpu


def main():
    parser, args = parse()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    mode = args.mode or "train"
    if args.scenario == "real_net":
        args.agent = "ma2c"
    if args.replicas is None:
        args.replicas = 2048 if args.scenario == "real_net" else 8192
    net, par, n_step, reward_norm = build_scenario(args)
    cores = usable_cpus()
    wl = workload_name(args.replicas, mode, args.agent, args.policy, args.scenario)

    # ---------------- reference arm: the CPU implementation of the path ----------------------
    if args.impl == "reference":
        if args.burnin + args.steps > episode_steps(par):
            parser.error("--burnin + --steps = %d control steps: the episode has %d"
                         % (args.burnin + args.steps, episode_steps(par)))
        if rank != 0:
            return
        cb, n, el, R_cpu = cpu_reference(net, par, args, cores, n_step, mode, args.steps, budget_s=args.cpu_budget)
        line = {"impl": "reference", "metric": "agent-env-steps/sec", "value": cb["value"],
                "unit": "agent-env-steps/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": 1e3 * el / n, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic",
                "config": {"workload": wl,
                           "note": "each reference step is a bounded sample: %d replicas instead of %d; see "
                                   "cpu_baseline.sample for what was timed" % (R_cpu, args.replicas)},
                "cpu_baseline": cb,
                "e2e": {"value": cb["value"], "unit": "agent-env-steps/s", "h2d_bytes_per_step": 0,
                        "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line))
        return

    # ---------------- our arm -----------------------------------------------------------------
    from deeprl_signal_control_b200.dist import bind_to_gpu_numa
    numa_cpus = bind_to_gpu_numa(local_rank)      # before torch allocates anything page-locked
    import torch
    import torch.distributed as dist
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank)
    from deeprl_signal_control_b200.sim import BatchedSim
    R = args.replicas
    sim = BatchedSim(net, par, R, device=local_rank)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    launches = 0
    trainer = None
    align_steps = 0
    if mode == "train":
        from deeprl_signal_control_b200.agents.layout import PolicyLayout
        from deeprl_signal_control_b200.agents.learner import BatchedA2C
        from deeprl_signal_control_b200.agents.trainer import BatchedTrainer
        # config/config_ma2c_large.ini [MODEL_CONFIG]
        lay = make_layout(net, args)
        if args.policy == "fc":
            from deeprl_signal_control_b200.agents.learner_fc import BatchedFcA2C as Learner
        else:
            Learner = BatchedA2C
        model = Learner(lay, R, n_step=n_step, gamma=0.99, v_coef=0.5, max_grad_norm=40.0, alpha=0.99, eps=1e-5,
                        reward_norm=reward_norm, reward_clip=2.0, seed=args.seed,
                        device=local_rank, chunk=args.chunk, replica0=rank * R, total_replicas=world * R,
                        process_group=dist.group.WORLD if world > 1 else None, allow_tf32=not args.fp32_gemm)
        trainer = BatchedTrainer(sim, model, args.agent, lr=5e-4, beta=0.01, seed0=args.seed, replica0=rank * R)

        def one_step(i):
            trainer.control_step()
    else:
        from deeprl_signal_control_b200.dist import shard_replicas
        _, _, seeds = shard_replicas(rank, world, R, args.seed)
        sim.reset(seeds)
        acts, fp = sim_mode_inputs(net, R, dev, rank)
        sim_events = []

        def one_step(i):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            sim.step(acts[i % len(acts)], fp)
            e1.record()
            sim_events.append((e0, e1))

    for i in range(args.burnin):
        one_step(i)
    for i in range(max(args.warmup, 3)):
        one_step(i)
    align_steps = 0
    if trainer is not None:
        # the timed region must never skip the learner update: align it so that it ENDS on an update boundary
        # (ceil(K / n_step) updates inside; for K < n_step this over-counts update work — conservative)
        while (trainer.model.t + args.steps) % n_step != 0:
            one_step(0)
            align_steps += 1
    live0 = sim.mean_live()
    sampler = ClockSampler(local_rank)
    sampler.start()
    if trainer is not None:
        trainer.sim_events = []
        trainer.update_events = []
        l0 = trainer.model.kernel_launches
        upd0 = trainer.n_updates
    else:
        sim_events.clear()
    barrier()
    t_start = torch.cuda.Event(enable_timing=True); t_end = torch.cuda.Event(enable_timing=True)
    t_start.record()
    for i in range(args.steps):
        one_step(i)
    t_end.record()
    barrier()
    # before the e2e loop below steps the same simulator / learner further
    dumped = last_step_outputs(sim, trainer) if args.dump_outputs and rank == 0 else None
    total_ms = t_start.elapsed_time(t_end)
    evs = trainer.sim_events if trainer is not None else sim_events
    kern_ms = float(np.mean([a.elapsed_time(b) for a, b in evs]))
    update_ms = None
    if trainer is not None:
        timed_launches = args.steps + (trainer.model.kernel_launches - l0)
        n_updates_timed = trainer.n_updates - upd0
        trainer.sim_events = None
        if trainer.update_events:
            update_ms = float(np.mean([a.elapsed_time(b) for a, b in trainer.update_events]))
        trainer.update_events = None
    else:
        timed_launches = args.steps
        n_updates_timed = 0
    sampler.stop_flag = True
    sampler.join(timeout=2)
    live1 = sim.mean_live()
    v_live = 0.5 * (live0 + live1)
    t = torch.tensor([total_ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms_max = float(t.item())
    value = world * R * net.n_nodes * args.steps / (total_ms_max * 1e-3)
    value_steady = None
    if update_ms is not None and n_updates_timed > 0:
        # the same measured quantities, re-weighted: K rollout steps + K/n_step updates (instead of n_updates_timed)
        t = torch.tensor([update_ms], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        upd = float(t.item())
        roll_ms = (total_ms_max - n_updates_timed * upd) / args.steps
        value_steady = {"value": world * R * net.n_nodes / ((roll_ms + upd / n_step) * 1e-3), "unit": "agent-env-steps/s",
                        "rollout_ms_per_step": roll_ms, "update_ms": upd, "n_step": n_step,
                        "how": "(timed ms - updates_in_timed_region x update_ms) / steps + update_ms / n_step, all "
                               "measured with CUDA events in this run"}

    # ---------------- e2e: the environment driven through the host-buffer C-ABI call ------------
    if trainer is not None:
        e2e_steps = n_step                     # one full rollout + one update
        if args.policy == "fc":
            args.e2e_parts = 1                 # the replica-range forward exists for the fused LSTM kernel only
        if args.e2e_parts > 1:
            host_step = lambda: trainer.control_step_host_pipelined(n_parts=args.e2e_parts)
        else:
            host_step = trainer.control_step_host
        for i in range(3):
            host_step()
        barrier()
        wait_s = [0.0]
        if os.environ.get("TSC_E2E_PROFILE"):          # how much of the host loop is spent blocked on the device
            for cls in (torch.cuda.Event, torch.cuda.Stream):
                def timed(self, _o=cls.synchronize):
                    t_ = time.perf_counter(); _o(self); wait_s[0] += time.perf_counter() - t_
                cls.synchronize = timed
        # seven back-to-back windows of one rollout + one update each; the MEDIAN window is reported (the host side of this
        # loop is sensitive to whatever else the lease's cores are doing: single windows were seen to take 2-5x as long on a
        # shared host; all seven are listed in the JSON line)
        e2e_windows = []
        import gc
        gc.collect(); gc.disable()             # no collector pauses inside the host-timed windows
        for w in range(1 if args.profile_run else 7):
            barrier()
            t0 = time.perf_counter()
            for i in range(e2e_steps):
                host_step()
            barrier()
            e2e_windows.append((time.perf_counter() - t0) * 1e3)
        gc.enable()
        e2e_ms = sorted(e2e_windows)[len(e2e_windows) // 2]
        if os.environ.get("TSC_E2E_PROFILE"):
            print("e2e host loop: %.3f ms/step, %.3f ms/step blocked in Event/Stream.synchronize" %
                  (e2e_ms / e2e_steps, wait_s[0] * 1e3 / (7 * e2e_steps)), file=sys.stderr)
        h2d = R * net.n_nodes * 4 + R * net.n_nodes * net.max_na * 4 + R * net.n_obs * 4 + R * net.n_nodes * 4 + R * 4
        d2h = R * net.n_nodes * 4 + R * net.n_nodes * net.max_na * 4 + R * net.n_obs * 4 + R * net.n_nodes * 4 + R * 4 + R
        e2e_api = ("BatchedTrainer.control_step_host: policy forward on device, actions+fingerprints D2H, "
                   "tsc_step_host (H2D, kernel, D2H), obs+reward H2D, update every %d steps" % n_step)
        if args.e2e_parts > 1:
            e2e_api = ("BatchedTrainer.control_step_host_pipelined: %d replica ranges, one stream each; per range: policy "
                       "forward (tscl_policy_step_v2r), actions+fingerprints D2H to pinned host buffers, "
                       "tsc_step_host_range (H2D, kernel, D2H, host sync), obs+reward H2D into the learner (tscl_host_transition); "
                       "median of seven windows; update "
                       "every %d steps" % (args.e2e_parts, n_step))
    else:
        e2e_steps = max(3, min(args.steps, 20))
        h_act = [(torch.randint(0, 1 << 30, (R, net.n_nodes)) % torch.tensor(net.n_a_ls)).to(torch.int32).pin_memory().numpy()
                 for _ in range(4)]
        h_fp = torch.rand(R, net.n_nodes, net.max_na).pin_memory().numpy()
        sim._h_out = tuple(torch.from_numpy(a).pin_memory().numpy() for a in (
            np.zeros((R, net.n_obs), np.float32), np.zeros((R, net.n_nodes), np.float32),
            np.zeros(R, np.float32), np.zeros(R, np.uint8)))
        for i in range(3):
            sim.step_host(h_act[i % 4], h_fp)
        barrier()
        t0 = time.perf_counter()
        for i in range(e2e_steps):
            sim.step_host(h_act[i % 4], h_fp)
        barrier()
        e2e_ms = (time.perf_counter() - t0) * 1e3
        h2d = R * net.n_nodes * 4 + R * net.n_nodes * net.max_na * 4
        d2h = R * net.n_obs * 4 + R * net.n_nodes * 4 + R * 4 + R
        e2e_api = "tsc_step_host (pinned host buffers)"
    t = torch.tensor([e2e_ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_windows_all = [round(x, 3) for x in e2e_windows] if trainer is not None else None
    e2e_value = world * R * net.n_nodes * e2e_steps / (float(t.item()) * 1e-3)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    # ---------------- roofline of the dominant kernel ----------------------------------------
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    else:
        peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
    alg_bytes = algorithmic_bytes(net, v_live) * R
    achieved = alg_bytes / (kern_ms * 1e-3) / 1e9
    traffic, issue = None, None
    prof = None
    for name in ("r02_sim_kernel_traffic.json", "r01_sim_kernel_traffic.json"):      # newest ncu capture of the kernel
        tr_path = os.path.join(ROOT, "profiles", name)
        if os.path.exists(tr_path):
            prof = json.load(open(tr_path))
            break
    if prof is not None and args.scenario == "large_grid" and prof.get("grid") == R:
        traffic = prof.get("dram_bytes_per_launch")
        if prof.get("warp_inst_per_launch"):
            # second roofline of the same kernel: instruction issue (what actually bounds it).  Warp instructions per
            # launch come from the committed ncu capture (smsp__inst_executed.sum); the rate uses the launch duration
            # measured live here; peak = 148 SMs x 4 warp schedulers x 1 instruction / cycle x the sampled SM clock.
            clk = (sampler.summary().get("sm_mhz") or 1965) * 1e6
            issue_peak = 148 * 4 * clk
            issue_rate = float(prof["warp_inst_per_launch"]) / (kern_ms * 1e-3)
            issue = {"bound": "issue", "achieved": issue_rate / 1e9, "peak": issue_peak / 1e9, "unit": "G warp-inst/s",
                     "frac": issue_rate / issue_peak, "warp_inst_per_launch": prof["warp_inst_per_launch"],
                     "source": prof.get("source")}
    roofline = {"bound": "hbm", "kernel": "tsc_step_kernel", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": alg_bytes, "mean_live_vehicles_per_replica": v_live,
                "kernel_ms_per_launch": kern_ms, "share_of_step": kern_ms * args.steps / total_ms,
                "issue": issue,
                "note": "SURVEY 8(d) names HBM as the bound, so `frac` is against the measured copy bandwidth; the kernel is "
                        "in fact instruction-issue-bound (five fused simulated seconds of Krauss updates per 24-32 B of "
                        "state per vehicle) - see `issue` and DESIGN.md section 5"}
    cb = None
    if not args.no_cpu_baseline:
        n_cpu = max(1, min(args.steps, episode_steps(par) - args.burnin))
        cb, _, _, _ = cpu_reference(net, par, args, cores, n_step, mode, n_cpu, budget_s=args.cpu_budget)
    line = {"metric": "agent-env-steps/sec", "value": value, "unit": "agent-env-steps/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": total_ms_max / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32" if mode == "sim" else "f32 (sim, LSTM cell, loss, optimizer) + bf16 tensor-core operands with f32 accumulation (learner GEMMs)",
            "data": "synthetic",
            "config": {"workload": wl, "scenario": args.scenario, "replicas_per_gpu": R, "agents": net.n_nodes,
                       "burnin_control_steps": args.burnin, "mode": mode, "n_step": n_step,
                       "updates_in_timed_region": n_updates_timed, "update_chunk_replicas": args.chunk, "untimed_alignment_steps": align_steps,
                       "learner_gemm_library": "none: own tcgen05 kernels for the forward, BPTT, dX and all weight gradients; "
                                               "own SIMT kernels for loss / heads / optimizer"
                       if mode == "train" else None,
                       "l2": "inputs larger than L2: %.0f MB of replica state per GPU is streamed every step"
                             % (R * sim.info()["state_bytes_per_replica"] / 1e6),
                       "parallelism": "replica-dp%d" % world,
                       "host_binding": ("rank bound to the %d host cores of its GPU's NUMA node" % len(numa_cpus))
                       if numa_cpus else "none (NVML affinity unavailable)"},
            "clocks": sampler.summary(),
            "value_steady": value_steady,
            "e2e": {"value": e2e_value, "unit": "agent-env-steps/s", "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "steps": e2e_steps, "api": e2e_api,
                    "windows_ms": e2e_windows_all},
            "gpu_launches": timed_launches,
            "roofline": roofline, "cpu_baseline": cb}
    if dumped is not None:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in dumped.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
