"""Device-resident training loop: the batched counterpart of reference utils.py:Trainer.explore/run.

Per control step (utils.py:146-165): policy/value forward -> fingerprint update (MA2C) -> action
sampling -> env.step -> add_transition; per n_step: bootstrap value, backward (utils.py:186-190,
288-291); per episode: env.reset(), model.reset(), pre-decision done = True (utils.py:277-281).
Everything stays on the GPU: the simulator writes the next observation straight into the
learner's rollout slot and reads actions / fingerprints from the learner's buffers.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

import numpy as np
import torch

from .. import _lib
from .. import dist as _dist
from ..sim import BatchedSim
from .learner import BatchedA2C


class BatchedTrainer:
    def __init__(self, sim: BatchedSim, model: BatchedA2C, agent: str, lr, beta,
                 seed0: int = 12, replica0: int = 0):
        """lr / beta: floats (the 'constant' schedules of every shipped A2C config) or objects with the reference's
        `Scheduler.get(n_step)` (agents/utils.py:268-281, agents/models.py:175-176); a schedule advances by n_step per
        update exactly as in the reference (its unit is control steps of ONE environment)."""
        self.sim, self.model, self.agent = sim, model, agent
        self.lr, self.beta = lr, beta
        self.seed0, self.replica0 = int(seed0), int(replica0)
        self.total_replicas = int(getattr(model, "total_replicas", sim.R))
        self.episode = 0
        self.T_episode = int(np.ceil(sim.params.episode_length_sec / sim.params.control_interval_sec))
        assert self.T_episode % model.T == 0                      # utils.py:121
        self.step_in_episode = 0
        self.done = True
        self.episode_rewards = []
        self._rew_acc = torch.zeros(sim.R, device=sim.device)
        self.n_updates = 0
        self.n_env_steps = 0
        self._uniform_fp = None
        self.sim_events = None        # list of (start, end) CUDA events around tsc_step when timing is on
        self.update_events = None     # same around update() (bootstrap forward + backward)
        self.start_episode()

    def start_episode(self):
        sim, m = self.sim, self.model
        # envs/env.py:560 (seed += 1 per episode and environment): disjoint over all (rank, episode) pairs
        seeds = _dist.episode_seeds(self.seed0, self.episode, self.replica0, sim.R, max(self.total_replicas, sim.R))
        self.episode += 1
        sim.reset(seeds)
        sim.set_train_mode(True)
        m.reset()
        fp = None
        if self.agent == 'ma2c':
            if self._uniform_fp is None:
                n = sim.net
                u = torch.zeros(sim.R, n.n_nodes, n.max_na, device=sim.device)
                for i, na in enumerate(n.n_a_ls):
                    u[:, i, :na] = 1.0 / na                       # envs/env.py:263-269
                self._uniform_fp = u
            fp = self._uniform_fp
        assert m.t == 0
        sim.observe(fp, obs_out=m.obs_slot(0))
        self.step_in_episode = 0
        self.done = True
        self._rew_acc.zero_()

    def control_step(self):
        """One control step of all replicas (utils.py:146-165)."""
        sim, m = self.sim, self.model
        t = m.t
        fused = bool(getattr(m, 'tc_v2', False))      # fused tensor-core forward: one-launch transition hand-over
        pi, val, act = m.forward(m.obs_slot(t), self.done, to_hist=True) if fused else m.forward(m.obs_slot(t), self.done)
        fp = pi if self.agent == 'ma2c' else None                 # env.update_fingerprint(policy)
        if self.sim_events is not None:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
        _, reward, greward, _ = sim.step(act, fp, obs_out=m.obs_hist[t + 1])
        if self.sim_events is not None:
            e1.record()
            self.sim_events.append((e0, e1))
        self.step_in_episode += 1
        new_done = self.step_in_episode >= self.T_episode         # lock-step: envs/env.py:577-579
        if fused:
            m.add_transition_device(reward, greward, self._rew_acc, self.done, new_done)
        else:
            m.add_transition(reward, self.done, new_done)
            self._rew_acc.add_(greward)
        self.done = new_done
        self.n_env_steps += 1
        if m.t == m.T:
            self.update()

    def control_step_host(self):
        """Same step with the environment driven through the HOST-buffer C-ABI call (tsc_step_host),
        i.e. the way a reference-style caller holds numpy arrays: actions / fingerprints D2H, env step
        (H2D + kernel + D2H inside), observation / reward H2D into the learner."""
        sim, m = self.sim, self.model
        t = m.t
        pi, val, act = m.forward(m.obs_slot(t), self.done)
        if not hasattr(self, '_pin_act'):       # page-locked staging for the D2H of actions / fingerprints
            self._pin_act = torch.zeros_like(act, device='cpu').pin_memory()
            self._pin_pi = torch.zeros_like(pi, device='cpu').pin_memory()
        self._pin_act.copy_(act, non_blocking=True)
        if self.agent == 'ma2c':
            self._pin_pi.copy_(pi, non_blocking=True)
        torch.cuda.current_stream(sim.device).synchronize()
        act_h = self._pin_act.numpy()
        fp_h = self._pin_pi.numpy() if self.agent == 'ma2c' else None
        obs_h, rew_h, grew_h, _ = sim.step_host(act_h, fp_h)
        m.obs_hist[t + 1].copy_(torch.from_numpy(obs_h), non_blocking=True)
        reward = torch.from_numpy(rew_h).to(sim.device, non_blocking=True)
        self.step_in_episode += 1
        new_done = self.step_in_episode >= self.T_episode
        m.add_transition(reward, self.done, new_done)
        self._rew_acc.add_(torch.from_numpy(grew_h).to(sim.device, non_blocking=True))
        self.done = new_done
        self.n_env_steps += 1
        if m.t == m.T:
            self.update()

    def control_step_host_pipelined(self, n_parts: int = 2):
        """control_step_host() with the replicas split into `n_parts` ranges, one CUDA stream each: while range k sits on
        the PCIe link (tsc_step_host_range: actions H2D, kernel, observations D2H; then observations H2D into the
        learner), the other ranges run their policy forward / simulator kernels.  Same results as control_step_host():
        ranges are independent and the sampling RNG is keyed by the absolute replica.  The host still receives every
        range's observations / rewards in page-locked numpy buffers before the learner consumes them."""
        sim, m = self.sim, self.model
        R, A, L = sim.R, m.lay.A, m.lay
        lib = _lib.lib()
        ma2c = self.agent == 'ma2c'
        if not hasattr(self, '_pp'):
            n_parts = max(1, min(n_parts, R))
            bounds = [R * k // n_parts for k in range(n_parts + 1)]
            pin = lambda *shape, dtype=torch.float32: torch.zeros(*shape, dtype=dtype).pin_memory()
            pp = dict(primed=False, act=pin(R, A, dtype=torch.int32), pi=pin(R, A, L.max_na), obs=pin(R, sim.net.n_obs),
                      rew=pin(R, A), grew=pin(R), done=pin(R, dtype=torch.uint8),
                      rew_stage=torch.zeros(R, A, device=m.dev), grew_stage=torch.zeros(R, device=m.dev), parts=[])
            at = lambda x, r0, per_row: C.c_void_p(x.data_ptr() + r0 * per_row * x.element_size())
            for k in range(n_parts):        # raw pointers of every range's slices: the per-step loop is host-issue-bound
                r0, n = bounds[k], bounds[k + 1] - bounds[k]
                st = torch.cuda.Stream(device=sim.device)
                pp['parts'].append(dict(
                    r0=r0, n=n, stream=st, sth=C.c_void_p(st.cuda_stream), ev=torch.cuda.Event(),
                    act_h=at(pp['act'], r0, A), pi_h=at(pp['pi'], r0, A * L.max_na) if ma2c else None,
                    obs_h=at(pp['obs'], r0, sim.net.n_obs), rew_h=at(pp['rew'], r0, A), grew_h=at(pp['grew'], r0, 1),
                    done_h=at(pp['done'], r0, 1), rew_stage=at(pp['rew_stage'], r0, A),
                    grew_stage=at(pp['grew_stage'], r0, 1), rew_acc=at(self._rew_acc, r0, 1)))
            self._pp = pp
        pp = self._pp

        def issue_forward(p, t, nf, done):
            pi, val, act = m.forward_range(p['r0'], p['n'], done, t, nf, stream=p['sth'], to_hist=True)
            _lib.check(lib.tscl_memcpy_async(m._h, p['act_h'], C.c_void_p(act.data_ptr()), C.c_int64(p['n'] * A * 4),
                                             C.c_int32(2), p['sth']))
            if ma2c:
                _lib.check(lib.tscl_memcpy_async(m._h, p['pi_h'], C.c_void_p(pi.data_ptr()),
                                                 C.c_int64(p['n'] * A * L.max_na * 4), C.c_int32(2), p['sth']))
            p['ev'].record(p['stream'])

        if not pp['primed']:
            cur = torch.cuda.current_stream(sim.device)
            for p in pp['parts']:
                p['stream'].wait_stream(cur)
                issue_forward(p, m.t, m.n_forward, self.done)
            m.end_forward_ranges()
            pp['primed'] = True
        t = m.t
        self.step_in_episode += 1
        new_done = self.step_in_episode >= self.T_episode
        boundary = (t + 1 == m.T)                       # an update (and possibly an episode end) follows this step
        n_obs = sim.net.n_obs
        for p in pp['parts']:                           # every range's env step is enqueued as soon as its actions are here
            p['ev'].synchronize()                       # the host holds this range's actions / fingerprints
            _lib.check(lib.tsc_step_host_range_async(sim._h, C.c_int32(p['r0']), C.c_int32(p['n']), p['act_h'], p['pi_h'],
                                                     p['obs_h'], p['rew_h'], p['grew_h'], p['done_h'], p['sth']))
        obs_next, rew_t = m.obs_hist[t + 1], m.rew_hist[t]
        for p in pp['parts']:
            r0, n = p['r0'], p['n']
            p['stream'].synchronize()                   # the host holds this range's observations / rewards ...
            # ... and hands them to the learner: obs -> rollout slot t+1, reward -> normalised / clipped slot t, episode sum
            _lib.check(lib.tscl_host_transition(
                m._h, p['obs_h'], C.c_void_p(obs_next.data_ptr() + r0 * n_obs * 4), C.c_int64(n * n_obs), p['rew_h'],
                p['rew_stage'], C.c_void_p(rew_t.data_ptr() + r0 * A * 4), C.c_int64(n * A),
                C.c_float(m.reward_norm or 0.0), C.c_float(m.reward_clip or 0.0), p['grew_h'], p['grew_stage'],
                p['rew_acc'], C.c_int64(n), p['sth']))
            if not boundary:
                issue_forward(p, t + 1, m.n_forward, False)
        m.end_transition_ranges(self.done, new_done)
        self.done = new_done
        self.n_env_steps += 1
        if not boundary:
            m.end_forward_ranges()
        else:
            cur = torch.cuda.current_stream(sim.device)
            for p in pp['parts']:
                cur.wait_stream(p['stream'])
            pp['primed'] = False
            self.update()

    def update(self):
        m = self.model
        if self.update_events is not None:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
        self._update()
        if self.update_events is not None:
            e1.record()
            self.update_events.append((e0, e1))

    def _update(self):
        m = self.model
        boot = None
        if not self.done:
            _, boot, _ = m.forward(m.obs_slot(m.T), False, out_type='v')    # utils.py:190
        lr = self.lr.get(m.T) if hasattr(self.lr, "get") else self.lr
        beta = self.beta.get(m.T) if hasattr(self.beta, "get") else self.beta
        m.backward(boot, lr, beta)
        self.n_updates += 1
        if self.done:
            self.episode_rewards.append(float((self._rew_acc / self.T_episode).mean()))   # utils.py:296-305
            self.start_episode()

    def run(self, n_control_steps: int):
        for _ in range(n_control_steps):
            self.control_step()


class BatchedIQLTrainer:
    """The episode protocol of `BatchedTrainer` for `BatchedIQL` (reference utils.py:Trainer.explore/run with an IQL
    model): per control step epsilon-greedy forward -> env.step -> add_transition; backward() every batch_size steps and
    at an episode end; per episode env.reset() with fresh seeds.  The simulator reads its actions from the ring's action
    slot and writes the next observation straight into the ring's observation slot.

    At an episode end the reset observation overwrites the terminal next observation of the last transition (both
    live in the same ring slot).  That is harmless: the transition is stored with done = True, whose TD target is r."""

    def __init__(self, sim: BatchedSim, model, seed0: int = 12):
        import torch.distributed as tdist
        assert not (tdist.is_available() and tdist.is_initialized() and tdist.get_world_size() > 1), \
            "BatchedIQLTrainer runs on one rank (no gradient all-reduce yet)"
        assert model.R == sim.R and model.C > 0
        self.sim, self.model = sim, model
        self.seed0 = int(seed0)
        self.episode = 0
        self.T_episode = int(np.ceil(sim.params.episode_length_sec / sim.params.control_interval_sec))
        self.step_in_episode = 0
        self.episode_rewards = []
        self._rew_acc = torch.zeros(sim.R, device=sim.device)
        self.n_env_steps = 0
        self.n_updates = 0
        self.fwd_events = None        # lists of (start, end) CUDA events around forward / tsc_step / backward
        self.sim_events = None
        self.update_events = None
        self.start_episode()

    def start_episode(self):
        sim, m = self.sim, self.model
        seeds = _dist.episode_seeds(self.seed0, self.episode, m.replica0, sim.R, sim.R)
        self.episode += 1
        sim.reset(seeds)
        sim.set_train_mode(True)
        m.reset()
        sim.observe(None, obs_out=m.obs_slot())
        self.step_in_episode = 0
        self._rew_acc.zero_()

    @staticmethod
    def _timed(events, fn):
        if events is None:
            return fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = fn()
        e1.record()
        events.append((e0, e1))
        return out

    def control_step(self):
        sim, m = self.sim, self.model
        act = self._timed(self.fwd_events, lambda: m.forward())
        _, reward, greward, _ = self._timed(self.sim_events,
                                            lambda: sim.step(act, None, obs_out=m.obs_slot(m.n_total + 1)))
        self.step_in_episode += 1
        done = self.step_in_episode >= self.T_episode                # lock-step: envs/env.py:577-579
        m.add_transition(reward, greward, self._rew_acc, done)
        self.n_env_steps += 1
        if done or self.step_in_episode % m.n_step == 0:             # utils.py:Trainer.explore returns -> backward
            if self._timed(self.update_events, lambda: m.backward()):
                self.n_updates += 1
        if done:
            self.episode_rewards.append(float((self._rew_acc / self.T_episode).mean()))   # utils.py:296-305
            self.start_episode()

    def run(self, n_control_steps: int):
        for _ in range(n_control_steps):
            self.control_step()
