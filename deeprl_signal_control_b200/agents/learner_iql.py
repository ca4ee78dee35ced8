"""`BatchedIQL`: independent Q-learning (IQL-LR / IQL-DQN) for all A agents and R lock-stepped replicas on one GPU.

Device-side counterpart of reference agents/models.py:IQL (+ agents/policies.py LRQPolicy / DeepQPolicy and
agents/utils.py ReplayBuffer), on the hand-written kernels of csrc/tsc_iql.cu.  A batched run behaves like R
independent copies of the reference's `IQL` + `Trainer.run` whose agents share one Q network per agent: the
gradient of every update step is the mean over the rows of all replicas (the convention of `BatchedA2C`).

* Networks, names and initial values are those of `models.IQL` (same seed and dims -> equal `named_weights()`);
  `save()` / `load()` read and write the same `checkpoint-<step>.npz`, so checkpoints move between the two classes.
* Acting (agents/models.py:347-362): `forward()` advances the epsilon schedule by one control step (all replicas move in
  lock-step); per (replica, agent) a uniform draw < eps picks a uniform action in [0, n_a), otherwise the argmax of the
  agent's q values (ties to the lowest index, as np.argmax).  Draws are keyed (seed, step, global replica, agent), so
  results do not depend on how replicas are split into ranges.  `forward(0.0)` is the evaluation ("act") mode.
* Replay (agents/utils.py:231-263): one ring of `buffer_size` transitions per replica, shared by all agents (the
  reference's per-agent buffers hold the same time steps; only the sampled indices differ per agent).  Rewards are
  stored divided by `reward_norm` and clipped.  Observations are kept once per step: transition n reads s from obs slot
  n % (C+1) and s' from slot (n+1) % (C+1), so the slot the simulator writes next is never the s' of a live transition.
* Update (agents/models.py:320-345): every `batch_size` control steps `lr = lr_scheduler.get(batch_size)`; when the ring
  holds >= batch_size transitions, 10 iterations, each over all agents: batch_size distinct live indices per
  (agent, replica) (random.sample), TD loss mean((q(s)[a] - stop_grad(done ? r : r + gamma max q(s')))^2) over all
  batch_size x R rows (no target network), per-agent clip_by_global_norm, TF1 Adam.  With R = 1 this is the reference.

One process, one GPU: a multi-rank run would need one gradient all-reduce per iteration and is not supported yet.
"""
from __future__ import annotations

import ctypes as C
import logging
import os
from typing import Optional

import numpy as np
import torch

from .. import _lib
from .layout import ortho_init
from .utils import Scheduler

N_ITER = 10          # minibatches per agent and backward() (agents/models.py:337-345)


def _p(t):
    return None if t is None else C.c_void_p(t.data_ptr())


class _IqlDims(C.Structure):
    _fields_ = [("n_agents", C.c_int32), ("n_obs", C.c_int32), ("max_na", C.c_int32), ("model", C.c_int32),
                ("num_fc", C.c_int32), ("num_h", C.c_int32), ("obs_off", C.POINTER(C.c_int32)),
                ("n_s", C.POINTER(C.c_int32)), ("n_w", C.POINTER(C.c_int32)), ("n_a", C.POINTER(C.c_int32)),
                ("par_off", C.POINTER(C.c_int64))]


def q_layers(model_type, n_s, n_a, n_w, num_fc, num_h):
    """(name, shape) of one agent's tensors in models.IQL order = the flat layout of csrc/tsc_iql.cu."""
    if model_type != 'dqn':
        return [('q/w', (n_s, n_a)), ('q/b', (n_a,))]
    out = [('q_fcw/w', (n_s - n_w, num_fc)), ('q_fcw/b', (num_fc,))]
    width = num_fc
    if n_w > 0:
        out += [('q_fct/w', (n_w, num_fc // 4)), ('q_fct/b', (num_fc // 4,))]
        width += num_fc // 4
    return out + [('q_fc_0/w', (width, num_h)), ('q_fc_0/b', (num_h,)), ('q/w', (num_h, n_a)), ('q/b', (n_a,))]


class BatchedIQL:
    name = 'iql'

    def __init__(self, n_s_ls, n_a_ls, n_w_ls, obs_off, n_obs, n_replicas, total_step, model_config, seed=0,
                 model_type='dqn', device=0, replica0=0):
        """Constructor arguments of models.IQL plus the observation layout (obs_off [A], n_obs: agent i reads
        obs[:, obs_off[i]:obs_off[i] + n_s[i]]), the replica count and `replica0`, the global id of replica 0 (keys of
        the random draws)."""
        if not torch.cuda.is_available():
            raise RuntimeError("BatchedIQL needs a CUDA device (no CPU fallback exists)")
        assert model_type in ('lr', 'dqn')
        self.model_type = model_type
        self.n_agent = A = len(n_s_ls)
        self.n_s_ls, self.n_a_ls, self.n_w_ls = [int(x) for x in n_s_ls], [int(x) for x in n_a_ls], [int(x) for x in n_w_ls]
        self.R, self.replica0 = int(n_replicas), int(replica0)
        self.n_obs = int(n_obs)
        self.max_na = max(self.n_a_ls)
        self.seed = int(seed)
        self.dev = torch.device("cuda", device)
        mc = model_config
        self.reward_clip = mc.getfloat('reward_clip')
        self.reward_norm = mc.getfloat('reward_norm')
        self.gamma = mc.getfloat('gamma')
        self.max_grad_norm = mc.getfloat('max_grad_norm')
        self.n_step = mc.getint('batch_size')
        self.total_step = total_step
        num_fc = mc.getint('num_fc') if model_type == 'dqn' else 0
        num_h = mc.getint('num_h') if model_type == 'dqn' else 0
        # flat layout + initial values of models.IQL (same RandomState draws, same order)
        rng = np.random.RandomState(seed)
        self.specs, flat, off = [], [], 0
        self.par_off = [0]
        for n_s, n_a, n_w in zip(self.n_s_ls, self.n_a_ls, self.n_w_ls):
            sp = []
            for k, shp in q_layers(model_type, n_s, n_a, n_w, num_fc, num_h):
                v = ortho_init(rng, shp) if k.endswith('/w') else np.zeros(shp, np.float32)
                sp.append((k, shp, off))
                flat.append(v.ravel())
                off += v.size
            self.specs.append(sp)
            self.par_off.append(off)
        self.P = torch.from_numpy(np.concatenate(flat)).to(self.dev)
        self.G = torch.zeros_like(self.P)
        self.M = torch.zeros_like(self.P)           # TF1 Adam moments and step count
        self.V = torch.zeros_like(self.P)
        self.adam_t = 0
        obs_off = [int(x) for x in obs_off][:A]
        self._arr = dict(obs_off=np.asarray(obs_off, np.int32), n_s=np.asarray(self.n_s_ls, np.int32),
                         n_w=np.asarray(self.n_w_ls, np.int32), n_a=np.asarray(self.n_a_ls, np.int32),
                         par_off=np.asarray(self.par_off, np.int64))
        a = self._arr
        self._cd = _IqlDims(A, self.n_obs, self.max_na, 1 if model_type == 'dqn' else 0, num_fc, num_h,
                            a['obs_off'].ctypes.data_as(C.POINTER(C.c_int32)), a['n_s'].ctypes.data_as(C.POINTER(C.c_int32)),
                            a['n_w'].ctypes.data_as(C.POINTER(C.c_int32)), a['n_a'].ctypes.data_as(C.POINTER(C.c_int32)),
                            a['par_off'].ctypes.data_as(C.POINTER(C.c_int64)))
        h = C.c_void_p()
        _lib.check(_lib.lib().tscl_iql_create(C.byref(self._cd), C.c_int32(device), C.byref(h)))
        self._h = h
        f32 = dict(dtype=torch.float32, device=self.dev)
        if total_step:
            lr_init, lr_decay = mc.getfloat('lr_init'), mc.get('lr_decay')
            self.lr_scheduler = Scheduler(lr_init, decay=lr_decay) if lr_decay == 'constant' else \
                Scheduler(lr_init, mc.getfloat('lr_min'), total_step, decay=lr_decay)
            eps_init, eps_decay = mc.getfloat('epsilon_init'), mc.get('epsilon_decay')
            self.eps_scheduler = Scheduler(eps_init, decay=eps_decay) if eps_decay == 'constant' else \
                Scheduler(eps_init, mc.getfloat('epsilon_min'), total_step * mc.getfloat('epsilon_ratio'), decay=eps_decay)
            Cap = self.C = int(mc.getfloat('buffer_size'))
            R = self.R
            self.obs_ring = torch.zeros(Cap + 1, R, self.n_obs, **f32)
            self.act_ring = torch.zeros(Cap, R, A, dtype=torch.int32, device=self.dev)
            self.rew_ring = torch.zeros(Cap, R, A, **f32)
            self.done_ring = torch.zeros(Cap, **f32)
            self._done_h = np.zeros(Cap, np.float32)       # lock-step: one done flag per transition, uploaded per update
            self.idx = torch.zeros(A, R, self.n_step, dtype=torch.int32, device=self.dev)
        else:                                              # evaluation only: one observation slot, one action slot
            self.C = 0
            self.obs_ring = torch.zeros(1, self.R, self.n_obs, **f32)
            self.act_ring = torch.zeros(1, self.R, A, dtype=torch.int32, device=self.dev)
        self.n_total = 0           # transitions stored so far
        self.n_forward = 0         # decisions taken (key of the exploration draws)
        self.n_backward = 0        # backward() calls (key of the replay draws)
        self.n_updates = 0         # backward() calls that updated the weights
        self.stats = torch.zeros(A, 2, **f32)      # loss, mean q of the last iteration
        self.norms = torch.zeros(A, **f32)
        self.q = torch.zeros(self.R, A, self.max_na, **f32)

    def close(self):
        if getattr(self, "_h", None) is not None:
            _lib.lib().tscl_iql_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _st(self):
        return C.c_void_p(torch.cuda.current_stream(self.dev).cuda_stream)

    # ---- ring ---------------------------------------------------------------------------------------------
    @property
    def size(self):
        return min(self.n_total, self.C)

    def obs_slot(self, n: Optional[int] = None) -> torch.Tensor:
        """[R, n_obs] observation of transition n (default: the next one to be stored); the simulator writes here."""
        n = self.n_total if n is None else n
        return self.obs_ring[n % (self.C + 1)]

    def act_slot(self, n: Optional[int] = None) -> torch.Tensor:
        """[R, A] int32 actions of transition n (default: the next one); forward() writes here, the simulator reads."""
        n = self.n_total if n is None else n
        return self.act_ring[n % max(self.C, 1)]

    def reset(self):
        return

    # ---- acting -------------------------------------------------------------------------------------------
    def forward(self, eps: Optional[float] = None, obs: Optional[torch.Tensor] = None, want_q: bool = False):
        """epsilon-greedy decision for all replicas / agents from obs (default: obs_slot()) into act_slot().
        eps None: the exploration schedule advances by one control step and gives eps (models.IQL 'explore');
        eps = 0: greedy ('act').  Returns act [R, A] int32 (and q [R, A, max_na] when want_q)."""
        if eps is None:
            eps = self.eps_scheduler.get(1)
        obs = self.obs_slot() if obs is None else obs
        assert obs.is_contiguous() and obs.numel() == self.R * self.n_obs
        act = self.act_slot()
        _lib.check(_lib.lib().tscl_iql_forward(self._h, _p(self.P), _p(obs), C.c_int64(self.R), C.c_float(eps),
                                               C.c_uint64(self.seed), C.c_int64(self.n_forward),
                                               C.c_int64(self.replica0), _p(act), _p(self.q) if want_q else None,
                                               self._st()))
        self.n_forward += 1
        return (act, self.q) if want_q else act

    def add_transition(self, reward: torch.Tensor, greward: torch.Tensor, rew_acc: torch.Tensor, done: bool):
        """Store transition n_total: s was obs_slot(), a is act_slot(), s' is already in obs_slot(n_total + 1);
        reward [R, A] -> clip(reward / reward_norm); rew_acc [R] += greward (episode sums)."""
        k = self.n_total % self.C
        _lib.check(_lib.lib().tscl_iql_transition(
            self._h, _p(reward), _p(self.rew_ring[k]), C.c_int64(reward.numel()), C.c_float(self.reward_norm or 0.0),
            C.c_float(self.reward_clip or 0.0), _p(greward), _p(rew_acc), C.c_int64(greward.numel()), self._st()))
        self._done_h[k] = 1.0 if done else 0.0
        self.n_total += 1

    # ---- update -------------------------------------------------------------------------------------------
    def sample(self, update: int, it: int) -> torch.Tensor:
        """idx [A, R, B]: batch_size distinct live ring slots per (agent, replica)."""
        _lib.check(_lib.lib().tscl_iql_sample(self._h, C.c_int64(self.R), C.c_int32(self.n_step), C.c_int64(self.size),
                                              C.c_uint64(self.seed), C.c_int64(update), C.c_int32(it),
                                              C.c_int64(self.replica0), _p(self.idx), self._st()))
        return self.idx

    def td_grad(self, idx: torch.Tensor):
        """G = gradient of the TD loss of the rows idx [A, R, B] selects (mean over B x R rows); stats [A, 2] =
        (loss, mean q(s)[a]) per agent."""
        assert idx.dtype == torch.int32 and idx.is_contiguous() and idx.shape == (self.n_agent, self.R, self.n_step)
        scale = 1.0 / (self.n_step * self.R)
        _lib.check(_lib.lib().tscl_iql_td_grad(
            self._h, _p(self.P), _p(self.obs_ring), _p(self.act_ring), _p(self.rew_ring), _p(self.done_ring),
            C.c_int64(self.C), C.c_int64(self.n_total), C.c_int64(self.R), C.c_int32(self.n_step), _p(idx),
            C.c_float(self.gamma), C.c_float(scale), _p(self.G), _p(self.stats), self._st()))
        return self.stats

    def clip_adam(self, lr: float):
        """per-agent clip_by_global_norm + one TF1 Adam step from G; norms [A] = pre-clip gradient norms."""
        self.adam_t += 1
        lr_t = lr * np.sqrt(1.0 - 0.999 ** self.adam_t) / (1.0 - 0.9 ** self.adam_t)
        _lib.check(_lib.lib().tscl_iql_clip_adam(self._h, _p(self.P), _p(self.G), _p(self.M), _p(self.V),
                                                 C.c_float(self.max_grad_norm), C.c_float(lr_t), _p(self.norms),
                                                 self._st()))
        return self.norms

    def backward(self, summary_writer=None, global_step=None) -> bool:
        """models.IQL.backward: lr schedule step, then (once the ring holds batch_size transitions) 10 minibatch
        updates of every agent.  Returns whether the weights changed."""
        lr = self.lr_scheduler.get(self.n_step)
        update = self.n_backward
        self.n_backward += 1
        if self.size < self.n_step:
            return False
        self.done_ring.copy_(torch.from_numpy(self._done_h))
        for it in range(N_ITER):
            self.td_grad(self.sample(update, it))
            self.clip_adam(lr)
        self.n_updates += 1
        return True

    # ---- names / checkpoints (models.IQL) ------------------------------------------------------------------
    def _prefix(self, i):
        return '%s_%da_q/' % ('dqn' if self.model_type == 'dqn' else 'lr', i)      # agents/policies.py:343,346,383,386

    def named_weights(self):
        flat = self.P.cpu().numpy()
        return {self._prefix(i) + k: flat[o:o + int(np.prod(shp))].reshape(shp).copy()
                for i, sp in enumerate(self.specs) for k, shp, o in sp}

    def load_named(self, named):
        flat = self.P.cpu().numpy().copy()
        for i, sp in enumerate(self.specs):
            for k, shp, o in sp:
                arr = np.asarray(named[self._prefix(i) + k], np.float32)
                if tuple(arr.shape) != tuple(shp):
                    raise ValueError('tensor %r has shape %s, expected %s' % (self._prefix(i) + k, arr.shape, tuple(shp)))
                flat[o:o + arr.size] = arr.ravel()
        self.P.copy_(torch.from_numpy(flat))

    def save(self, model_dir, global_step):
        """`checkpoint-<step>.npz` keyed by the reference's variable names (readable by models.IQL.load); the Adam state
        travels under `__b200__/` so that a batched run can resume."""
        from . import checkpoint as ck
        ck.save_npz(os.path.join(model_dir, 'checkpoint-%d.npz' % int(global_step)), self.named_weights(),
                    {'step': np.int64(global_step), 'adam_m': self.M.cpu().numpy(), 'adam_v': self.V.cpu().numpy(),
                     'adam_t': np.int64(self.adam_t)})

    def load(self, model_dir, checkpoint=None):
        from . import checkpoint as ck
        files = [f for f in os.listdir(model_dir)] if os.path.exists(model_dir) else []
        steps = [int(f.split('.')[0].split('-')[1]) for f in files
                 if f.startswith('checkpoint-') and len(f.split('.')[0].split('-')) == 2]
        if checkpoint is None and not steps:
            logging.error('Can not find old checkpoint for %s' % model_dir)
            return False
        step = int(checkpoint) if checkpoint is not None else max(steps)
        path = os.path.join(model_dir, 'checkpoint-%d.npz' % step)
        if not os.path.exists(path):
            logging.error('Can not find old checkpoint for %s' % model_dir)
            return False
        named, extra = ck.load_npz(path)
        self.load_named(named)
        if 'adam_m' in extra and extra['adam_m'].shape == tuple(self.M.shape):
            self.M.copy_(torch.from_numpy(extra['adam_m']))
            self.V.copy_(torch.from_numpy(extra['adam_v']))
            self.adam_t = int(extra['adam_t'])
        return True
