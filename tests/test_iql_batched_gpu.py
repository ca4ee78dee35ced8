"""GPU: the batched IQL learner (agents/learner_iql.py on csrc/tsc_iql.cu) against the reference's LRQPolicy /
DeepQPolicy graphs (tests/golden/learner_iql{,_wait}.npz), float64 autograd, models.IQL and a host ReplayBuffer."""
import configparser
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

GOLD = os.path.join(os.path.dirname(__file__), "golden")
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
buffer_size = 1000
batch_size = 20
reward_norm = 3.0
reward_clip = 2.0
num_fc = 128
num_h = 64
"""


def _cfg(**over):
    cp = configparser.ConfigParser(); cp.read_string(INI)
    for k, v in over.items():
        cp["MODEL_CONFIG"][k] = str(v)
    return cp["MODEL_CONFIG"]


def _model(n_s, n_a, n_w, kind, R, total_step=1000, seed=0, replica0=0, **over):
    from deeprl_signal_control_b200.agents.learner_iql import BatchedIQL
    off = np.concatenate([[0], np.cumsum(n_s)]).astype(np.int32)
    return BatchedIQL(n_s, n_a, n_w, off[:-1], int(off[-1]), R, total_step, _cfg(**over), seed=seed, model_type=kind,
                      replica0=replica0)


def _named(z, prefix):
    return {k[len(prefix) + 1:]: z[k] for k in z.files if k.startswith(prefix + "/")}


FIXTURES = {"lr": ("learner_iql.npz", "lr", [24, 36], [0, 0]), "dqn": ("learner_iql.npz", "dqn", [24, 36], [0, 0]),
            "dqn_wait": ("learner_iql_wait.npz", "dqn", [30, 36], [6, 6])}


def _q64(kind, named, prefix, S, n_w):
    """float64 restatement of models.IQL._q on named weights (torch tensors)."""
    p = {k[len(prefix):]: v for k, v in named.items() if k.startswith(prefix)}
    if kind == "lr":
        return S @ p["q/w"] + p["q/b"]
    if n_w == 0:
        h = torch.relu(S @ p["q_fcw/w"] + p["q_fcw/b"])
    else:
        ns = S.shape[1] - n_w
        h = torch.cat([torch.relu(S[:, :ns] @ p["q_fcw/w"] + p["q_fcw/b"]),
                       torch.relu(S[:, ns:] @ p["q_fct/w"] + p["q_fct/b"])], 1)
    h = torch.relu(h @ p["q_fc_0/w"] + p["q_fc_0/b"])
    return h @ p["q/w"] + p["q/b"]


def _td_grad64(kind, named, prefix, S, A, S1, Rw, D, n_w, gamma=0.99):
    w = {k: torch.tensor(v, dtype=torch.float64, requires_grad=True) for k, v in named.items() if k.startswith(prefix)}
    S, S1 = torch.as_tensor(S, dtype=torch.float64), torch.as_tensor(S1, dtype=torch.float64)
    q0 = _q64(kind, w, prefix, S, n_w).gather(1, torch.as_tensor(A, dtype=torch.int64)[:, None])[:, 0]
    with torch.no_grad():
        tq = torch.where(torch.as_tensor(D, dtype=torch.bool), torch.as_tensor(Rw, dtype=torch.float64),
                         torch.as_tensor(Rw, dtype=torch.float64) + gamma * _q64(kind, w, prefix, S1, n_w).max(1)[0])
    loss = ((q0 - tq) ** 2).mean()
    keys = list(w)
    return float(loss), dict(zip(keys, (g.numpy() for g in torch.autograd.grad(loss, [w[k] for k in keys]))))


def _grads_close(m, G, ref, tol=5e-4):
    flat = G.cpu().numpy()
    for i, sp in enumerate(m.specs):
        for k, shp, o in sp:
            r = ref[m._prefix(i) + k]
            got = flat[o:o + r.size].reshape(shp)
            scale = max(float(np.abs(r).max()), 1e-12)
            assert float(np.abs(got - r).max()) / scale < tol, (m._prefix(i) + k, float(np.abs(got - r).max()) / scale)


@pytest.mark.parametrize("case", ["lr", "dqn", "dqn_wait"])
def test_reference_pin_through_the_production_kernels(case):
    """The reference's fixed minibatches fed through tscl_iql_td_grad (given indices) and tscl_iql_clip_adam at R = 1:
    loss and norm to 5e-5, gradients to 5e-4 of each tensor's maximum, weights after three Adam steps to 3e-6.
    Agent i's B transitions are the ring's transitions 2B*i + 2b, so that s and s' of a row sit in two ring slots."""
    fname, kind, n_s, n_w = FIXTURES[case]
    z = np.load(os.path.join(GOLD, fname))
    n_a, B = [5, 4], 20
    m = _model(n_s, n_a, n_w, kind, 1, buffer_size=4 * B)
    w0 = _named(z, "%s/w0" % kind)
    assert sorted(m.named_weights()) == sorted(str(n) for n in z["%s/var_names" % kind])
    m.load_named(w0)
    off = [0, n_s[0]]
    idx = torch.zeros(2, 1, B, dtype=torch.int32)
    for i in range(2):
        idx[i, 0] = torch.arange(B, dtype=torch.int32) * 2 + 2 * B * i
    idx = idx.cuda()
    m.n_total = 4 * B
    for k in range(3):
        grads = {}
        for i in range(2):
            pre = "%s/k%d/a%d" % (kind, k, i)
            n = torch.arange(B) * 2 + 2 * B * i
            m.obs_ring[n, 0, off[i]:off[i] + n_s[i]] = torch.tensor(z[pre + "/obs"], dtype=torch.float32).cuda()
            m.obs_ring[n + 1, 0, off[i]:off[i] + n_s[i]] = torch.tensor(z[pre + "/next_obs"], dtype=torch.float32).cuda()
            m.act_ring[n, 0, i] = torch.tensor(z[pre + "/acts"], dtype=torch.int32).cuda()
            m.rew_ring[n, 0, i] = torch.tensor(z[pre + "/rs"], dtype=torch.float32).cuda()
            m.done_ring[n] = torch.tensor(z[pre + "/dones"], dtype=torch.float32).cuda()
            grads.update({k_: z[k_] for k_ in z.files if k_.startswith(pre + "/g/")})
        stats = m.td_grad(idx).cpu().numpy()
        for i in range(2):
            pre = "%s/k%d/a%d" % (kind, k, i)
            np.testing.assert_allclose(stats[i, 0], float(z[pre + "/loss"]), rtol=5e-5)
        _grads_close(m, m.G, {name.split("/g/", 1)[1]: v for name, v in grads.items()})
        norms = m.clip_adam(1e-4).cpu().numpy()
        for i in range(2):
            np.testing.assert_allclose(norms[i], float(z["%s/k%d/a%d/grad_norm" % (kind, k, i)]), rtol=5e-5)
    got = m.named_weights()
    for name, ref in _named(z, "%s/w3" % kind).items():
        np.testing.assert_allclose(got[name], ref, rtol=0, atol=3e-6, err_msg=name)
        assert float(np.abs(ref - w0[name]).max()) > 5e-5


def _random_ring(m, rng, n_total):
    C = m.C
    m.obs_ring.copy_(torch.from_numpy(rng.random(tuple(m.obs_ring.shape), dtype=np.float32) * 2))
    m.act_ring.copy_(torch.from_numpy(np.stack([rng.integers(0, na, (C, m.R)) for na in m.n_a_ls], -1).astype(np.int32)))
    m.rew_ring.copy_(torch.from_numpy(rng.normal(0, 1, tuple(m.rew_ring.shape)).astype(np.float32)))
    m.done_ring.copy_(torch.from_numpy((rng.random(C) < 0.3).astype(np.float32)))
    m.n_total = n_total


def _rows(m, r, i, idx_row):
    """s, a, r, done, s' of replica r, agent i at ring slots idx_row (the ring layout of learner_iql's docstring)."""
    C, nt = m.C, m.n_total
    off, ns = int(m._arr["obs_off"][i]), m.n_s_ls[i]
    k = np.asarray(idx_row, np.int64)
    n = k if nt <= C else (nt - C) + np.mod(k - (nt - C), C)
    obs = m.obs_ring.cpu().numpy()
    return (obs[n % (C + 1), r, off:off + ns], m.act_ring.cpu().numpy()[k, r, i], m.rew_ring.cpu().numpy()[k, r, i],
            m.done_ring.cpu().numpy()[k], obs[(n + 1) % (C + 1), r, off:off + ns])


def test_replica_average_and_replica_copies():
    """R = 8 replicas with different data: the gradient is the mean of the per-replica float64 autograd gradients;
    R = 8 copies of one replica's data give the R = 1 gradient.  Wrapped ring (n_total > C)."""
    z = np.load(os.path.join(GOLD, "learner_iql_wait.npz"))
    w0 = _named(z, "dqn/w0")
    n_s, n_a, n_w = [30, 36], [5, 4], [6, 6]
    rng = np.random.default_rng(3)
    m = _model(n_s, n_a, n_w, "dqn", 8, buffer_size=40)
    m.load_named(w0)
    _random_ring(m, rng, 137)
    idx = m.sample(0, 0)
    m.td_grad(idx)
    ix = idx.cpu().numpy()
    ref = {}
    for i in range(2):
        for r in range(8):
            S, A, Rw, D, S1 = _rows(m, r, i, ix[i, r])
            _, g = _td_grad64("dqn", w0, m._prefix(i), S, A, S1, Rw, D, n_w[i])
            for k, v in g.items():
                ref[k] = ref.get(k, 0) + v / 8
    _grads_close(m, m.G, ref)
    # R copies of replica 0
    m1 = _model(n_s, n_a, n_w, "dqn", 1, buffer_size=40)
    m8 = _model(n_s, n_a, n_w, "dqn", 8, buffer_size=40)
    for mm in (m1, m8):
        mm.load_named(w0)
        mm.obs_ring.copy_(m.obs_ring[:, :1].expand(-1, mm.R, -1))
        mm.act_ring.copy_(m.act_ring[:, :1].expand(-1, mm.R, -1))
        mm.rew_ring.copy_(m.rew_ring[:, :1].expand(-1, mm.R, -1))
        mm.done_ring.copy_(m.done_ring)
        mm.n_total = m.n_total
        mm.td_grad(idx[:, :1].expand(-1, mm.R, -1).contiguous())
    g1, g8 = m1.G.cpu().numpy(), m8.G.cpu().numpy()
    assert np.abs(g8 - g1).max() <= 1e-5 * np.abs(g1).max()


def test_forward_q_values_greedy_actions_and_exploration():
    from deeprl_signal_control_b200.agents.models import IQL
    for case in ("lr", "dqn_wait"):
        fname, kind, n_s, n_w = FIXTURES[case]
        z = np.load(os.path.join(GOLD, fname))
        w0 = _named(z, "%s/w0" % kind)
        R = 512
        m = _model(n_s, [5, 4], n_w, kind, R)
        m.load_named(w0)
        ref = IQL(n_s, [5, 4], n_w, 0, _cfg(), model_type=kind, device="cpu")
        ref.load_named(w0)
        obs = torch.rand(R, sum(n_s), generator=torch.Generator().manual_seed(1)) * 2
        act, q = m.forward(0.0, obs=obs.cuda().contiguous(), want_q=True)
        act, q = act.cpu().numpy(), q.cpu().numpy()
        off = [0, n_s[0]]
        for i in range(2):
            qr = ref._q(i, obs[:, off[i]:off[i] + n_s[i]]).detach().numpy()
            np.testing.assert_allclose(q[:, i, :[5, 4][i]], qr, rtol=1e-5, atol=1e-5 * np.abs(qr).max())
            assert np.all(q[:, i, [5, 4][i]:] == 0)
            srt = np.sort(qr, 1)
            clear = srt[:, -1] - srt[:, -2] > 1e-4
            greedy = np.array([ref.forward([o[:n_s[0]].numpy(), o[n_s[0]:].numpy()], mode="act")[0][i] for o in obs])
            assert clear.mean() > 0.9 and np.array_equal(act[clear, i], greedy[clear])
    # eps = 1 on Monaco's ragged action sets: every action in [0, n_a), none outside; eps = 0.3: explore fraction
    from deeprl_signal_control_b200.agents.learner_iql import BatchedIQL
    from deeprl_signal_control_b200.net.real_net import real_net_tables
    net = real_net_tables("iqld")
    R = 4096
    m = BatchedIQL(net.n_s_ls, net.n_a_ls, net.n_w_ls, net.node_obs_off, net.n_obs, R, 1000, _cfg(), seed=4)
    obs = (torch.rand(R, net.n_obs, device="cuda") * 2).contiguous()
    act = m.forward(1.0, obs=obs).cpu().numpy()
    for i, na in enumerate(net.n_a_ls):
        assert set(np.unique(act[:, i]).tolist()) == set(range(na)), (i, na)
    greedy = m.forward(0.0, obs=obs).cpu().numpy().copy()
    eps = 0.3
    act = m.forward(eps, obs=obs).cpu().numpy()
    p = np.array([eps * (na - 1) / na for na in net.n_a_ls])          # a uniform pick may equal the greedy action
    n_diff = float((act != greedy).sum())
    mean, var = float(R * p.sum()), float(R * (p * (1 - p)).sum())
    assert abs(n_diff - mean) < 5 * np.sqrt(var), (n_diff, mean)
    assert (act < np.array(net.n_a_ls)[None]).all() and (act >= 0).all()


def test_sampler_distinct_live_and_independent_of_the_replica_split():
    n_s, n_a, n_w = [24, 36], [5, 4], [0, 0]
    for size in (20, 37, 1000):
        m16 = _model(n_s, n_a, n_w, "lr", 16, seed=9)
        m16.n_total = size
        ix16 = m16.sample(5, 3).cpu().numpy().copy()
        assert ix16.min() >= 0 and ix16.max() < size
        for row in ix16.reshape(-1, 20):
            assert len(set(row.tolist())) == 20
        for r0 in (0, 4, 12):
            m4 = _model(n_s, n_a, n_w, "lr", 4, seed=9, replica0=r0)
            m4.n_total = size
            assert np.array_equal(m4.sample(5, 3).cpu().numpy(), ix16[:, r0:r0 + 4])
    assert not np.array_equal(m16.sample(5, 4).cpu().numpy(), ix16)        # another iteration draws other rows


def test_ring_equals_a_host_replay_buffer_across_wrap_and_episode_end():
    """Over more than buffer_size steps with an episode end: s, a, r (normalised, clipped) and s' gathered from the ring
    equal a host ReplayBuffer fed the same transitions; at the episode end the reset observation overwrites the terminal
    s' in the ring, which leaves the TD gradient unchanged because the transition is done (target = r)."""
    from deeprl_signal_control_b200.agents.utils import ReplayBuffer
    n_s, n_a, n_w = [30, 36], [5, 4], [6, 6]
    R, Cap, steps, T_ep = 3, 30, 47, 25
    m = _model(n_s, n_a, n_w, "dqn", R, buffer_size=Cap)
    host = [[ReplayBuffer(Cap, 20) for _ in range(2)] for _ in range(R)]
    rng = np.random.default_rng(5)
    acc = torch.zeros(R, device="cuda")
    off = [0, 30]
    ob = rng.random((R, 66), dtype=np.float32) * 2
    m.obs_slot().copy_(torch.from_numpy(ob))
    for t in range(steps):
        act = m.forward(1.0).cpu().numpy().copy()
        nxt = rng.random((R, 66), dtype=np.float32) * 2
        m.obs_slot(m.n_total + 1).copy_(torch.from_numpy(nxt))
        rew = rng.normal(0, 6, (R, 2)).astype(np.float32)
        done = (t + 1) % T_ep == 0
        m.add_transition(torch.from_numpy(rew).cuda(), torch.ones(R, device="cuda"), acc, done)
        r_h = np.clip(rew * np.float32(1 / 3.0), -2, 2)
        for r in range(R):
            for i in range(2):
                host[r][i].add_transition(ob[r, off[i]:off[i] + n_s[i]], int(act[r, i]), r_h[r, i],
                                          nxt[r, off[i]:off[i] + n_s[i]], done)
        ob = nxt
        if done:                       # env.reset(): the reset observation lands in the slot of the terminal s'
            ob = rng.random((R, 66), dtype=np.float32) * 2
            m.obs_slot().copy_(torch.from_numpy(ob))
    assert m.n_total == steps and m.size == Cap and float(acc[0]) == steps
    m.done_ring.copy_(torch.from_numpy(m._done_h))
    overwritten = 0
    for r in range(R):
        for i in range(2):
            S, A, Rw, D, S1 = _rows(m, r, i, np.arange(Cap))
            hs = host[r][i]._slots
            assert np.array_equal(S, np.stack([h[0] for h in hs])) and np.array_equal(A, [h[1] for h in hs])
            np.testing.assert_allclose(Rw, [h[2] for h in hs], rtol=1e-6)
            assert np.array_equal(D.astype(bool), [h[4] for h in hs])
            live = ~D.astype(bool)
            assert np.array_equal(S1[live], np.stack([h[3] for h in hs])[live])
            overwritten += int((S1[~live] != np.stack([h[3] for h in hs])[~live]).any())
    assert overwritten > 0                                      # the terminal s' really is gone from the ring ...
    m.load_named(_named(np.load(os.path.join(GOLD, "learner_iql_wait.npz")), "dqn/w0"))
    idx = m.sample(1, 0)
    m.td_grad(idx)
    ix = idx.cpu().numpy()
    ref = {}
    w0 = m.named_weights()
    for i in range(2):
        for r in range(R):
            hs = host[r][i]._slots
            rows = [hs[k] for k in ix[i, r]]
            _, g = _td_grad64("dqn", w0, m._prefix(i), np.stack([h[0] for h in rows]), [h[1] for h in rows],
                              np.stack([h[3] for h in rows]), [h[2] for h in rows], [h[4] for h in rows], n_w[i])
            for k, v in g.items():
                ref[k] = ref.get(k, 0) + v / R
    _grads_close(m, m.G, ref)                                  # ... and the gradient is the host buffer's


def _grid_trainer(kind, R, seed):
    from deeprl_signal_control_b200.agents.learner_iql import BatchedIQL
    from deeprl_signal_control_b200.agents.trainer import BatchedIQLTrainer
    from deeprl_signal_control_b200.net.large_grid import build_large_grid
    from deeprl_signal_control_b200.net.tables import EnvParams
    from deeprl_signal_control_b200.sim import BatchedSim
    agent = "iqld" if kind == "dqn" else "iqll"
    net, par = build_large_grid(agent=agent), EnvParams(agent=agent)
    sim = BatchedSim(net, par, R)
    m = BatchedIQL(net.n_s_ls, net.n_a_ls, net.n_w_ls, net.node_obs_off, net.n_obs, R, 1e6, _cfg(reward_norm=3000.0),
                   seed=seed, model_type=kind)
    return BatchedIQLTrainer(sim, m, seed0=12), m


@pytest.mark.parametrize("kind", ["lr", "dqn"])
def test_trainer_runs_a_grid_episode_reproducibly_and_checkpoints_with_models_iql(kind, tmp_path):
    from deeprl_signal_control_b200.agents.models import IQL
    from deeprl_signal_control_b200.agents.utils import Scheduler
    tr, m = _grid_trainer(kind, 16, seed=3)
    p0 = m.P.clone()
    assert m.backward() is False and torch.equal(m.P, p0)       # size 0 < batch_size: schedule steps, no update
    tr.run(19)
    assert torch.equal(m.P, p0) and tr.n_updates == 0
    tr.run(720 - 19)
    torch.cuda.synchronize()
    assert tr.n_updates == 36 and len(tr.episode_rewards) == 1 and np.isfinite(tr.episode_rewards[0])
    assert m.n_total == 720 and m.size == 720 and tr.episode == 2 and tr.step_in_episode == 0
    ref = Scheduler(1.0, 0.01, 1e6 * 0.5)
    for _ in range(720):
        e = ref.get(1)
    assert m.eps_scheduler.n == 720 and m.eps_scheduler.get(0) == ref.get(0) and e == ref.get(0)
    assert bool(torch.isfinite(m.P).all()) and not torch.equal(m.P, p0) and float(m.norms.min()) > 0
    # same seed -> the same bits
    tr2, m2 = _grid_trainer(kind, 16, seed=3)
    m2.backward()
    tr2.run(720)
    assert torch.equal(m.P, m2.P) and tr.episode_rewards == tr2.episode_rewards
    # checkpoints move between BatchedIQL and models.IQL in both directions
    net = tr.sim.net
    d = str(tmp_path) + "/"
    m.save(d, 720)
    host = IQL(net.n_s_ls, net.n_a_ls, net.n_w_ls, 0, _cfg(), seed=3, model_type=kind, device="cpu")
    fresh = host.named_weights()
    _, m0 = _grid_trainer(kind, 2, seed=3)
    for k, v in m0.named_weights().items():                     # same seed and dims -> the same initial weights
        assert np.array_equal(v, fresh[k]), k
    assert host.load(d) is True
    for k, v in m.named_weights().items():
        assert np.array_equal(host.named_weights()[k], v), k
    for p in host.nets:
        for v in p.values():
            v.data.mul_(0.5)
    host.save(d, 1440)
    assert m0.load(d) is True
    for k, v in host.named_weights().items():
        assert np.array_equal(m0.named_weights()[k], v), k
    assert m0.load(d, checkpoint=720) is True and torch.equal(m0.M, m.M) and m0.adam_t == m.adam_t == 360


def test_device_bandit_learns_the_best_actions():
    """test_iql_cpu's bandit at R = 32 on the device: done = True (target = r), +1 for the best action, -1 otherwise."""
    from deeprl_signal_control_b200.agents.learner_iql import BatchedIQL
    cfg = _cfg(lr_init=1e-2, reward_norm=1.0, num_fc=16, num_h=8)
    n_s, n_a = [4, 6], [3, 2]
    R = 32
    m = BatchedIQL(n_s, n_a, [0, 0], [0, 4], 10, R, 400, cfg, seed=0, model_type="lr")
    best = torch.tensor([2, 0], device="cuda", dtype=torch.int32)
    acc = torch.zeros(R, device="cuda")
    g = torch.Generator(device="cuda").manual_seed(0)
    m.obs_slot().copy_(torch.rand(R, 10, device="cuda", generator=g))
    for step in range(400):
        act = m.forward()
        m.obs_slot(m.n_total + 1).copy_(torch.rand(R, 10, device="cuda", generator=g))
        rew = torch.where(act == best[None], 1.0, -1.0).contiguous()
        m.add_transition(rew, torch.zeros(R, device="cuda"), acc, True)
        if step % 20 == 19:
            m.backward()
    assert abs(m.eps_scheduler.get(0) - 0.01) < 1e-9 and m.n_updates == 20
    obs = torch.rand(R, 10, device="cuda", generator=g)
    act = m.forward(0.0, obs=obs).cpu().numpy()
    assert (act == np.array([2, 0])[None]).all()
