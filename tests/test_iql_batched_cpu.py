"""CPU: what the batched IQL learner builds on without a GPU — the wait-branch reference pin of models.IQL
(tests/golden/learner_iql_wait.npz, made by tests/golden/gen_iql_wait_golden.py from the reference's DeepQPolicy), the
flat parameter layout shared by agents/learner_iql.py and csrc/tsc_iql.cu, and the Monaco tables of the iql agents."""
import configparser
import lzma
import os

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")

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


def _named(z, prefix):
    return {k[len(prefix) + 1:]: z[k] for k in z.files if k.startswith(prefix + "/")}


def test_iql_wait_branch_matches_reference_deepqpolicy():
    """DeepQPolicy with n_w = 6 (the grid's q_fct branch): q values, TD loss, gradient norm and the weights after each
    of three Adam steps of models.IQL equal the reference graph's."""
    from deeprl_signal_control_b200.agents.models import IQL
    z = np.load(os.path.join(GOLD, "learner_iql_wait.npz"))
    cp = configparser.ConfigParser(); cp.read_string(INI)
    n_s, n_w, n_a = [int(x) for x in z["n_s"]], [int(x) for x in z["n_w"]], [int(x) for x in z["n_a"]]
    m = IQL(n_s, n_a, n_w, 1000, cp["MODEL_CONFIG"], seed=0, model_type="dqn", device="cpu")
    w0 = _named(z, "dqn/w0")
    assert sorted(m.named_weights().keys()) == sorted(str(n) for n in z["dqn/var_names"])
    assert "dqn_0a_q/q_fct/w" in w0 and w0["dqn_0a_q/q_fct/w"].shape == (6, 32)
    m.load_named(w0)
    for k in range(3):
        for i in range(2):
            pre = "dqn/k%d/a%d" % (k, i)
            q = m._q(i, torch.from_numpy(z[pre + "/obs"].astype(np.float32))).detach().numpy()
            np.testing.assert_allclose(q, z[pre + "/q"], rtol=2e-5, atol=2e-6)
            loss, norm = m.td_update(i, z[pre + "/obs"], z[pre + "/acts"], z[pre + "/next_obs"], z[pre + "/dones"],
                                     z[pre + "/rs"], 1e-4)
            np.testing.assert_allclose(loss, float(z[pre + "/loss"]), rtol=2e-5)
            np.testing.assert_allclose(norm, float(z[pre + "/grad_norm"]), rtol=2e-5)
        got = m.named_weights()
        for name, ref in _named(z, "dqn/w%d" % (k + 1)).items():
            np.testing.assert_allclose(got[name], ref, rtol=0, atol=2e-6, err_msg=name)
            assert float(np.abs(ref - w0[name]).max()) > 5e-5


def test_flat_layout_follows_models_iql():
    """learner_iql.q_layers (the flat order the kernels read) lists models.IQL's tensors in its order and shapes, for
    both models, with and without the wait branch."""
    from deeprl_signal_control_b200.agents.learner_iql import q_layers
    from deeprl_signal_control_b200.agents.models import IQL
    cp = configparser.ConfigParser(); cp.read_string(INI)
    for kind in ("lr", "dqn"):
        m = IQL([30, 24, 12], [5, 4, 2], [6, 0, 6], 0, cp["MODEL_CONFIG"], seed=0, model_type=kind, device="cpu")
        for i, (n_s, n_a, n_w) in enumerate(zip(m.n_s_ls, m.n_a_ls, m.n_w_ls)):
            got = q_layers(kind, n_s, n_a, n_w, 128, 64)
            assert [(k, tuple(v.shape)) for k, v in m.nets[i].items()] == [(k, tuple(s)) for k, s in got]


def test_monaco_iql_tables_equal_the_tables_built_from_the_net_file(tmp_path):
    """real_net_tables('iqll' | 'iqld') without a net file serve the ia2c cache; that is what build_real_net makes
    from most.net.xml for those agents (iql observes and is rewarded like ia2c)."""
    from deeprl_signal_control_b200.net import real_net as rn
    from deeprl_signal_control_b200.net.tables import NetTables
    net_file = str(tmp_path / "most.net.xml")
    with lzma.open(os.path.join(GOLD, "monaco_most.net.xml.xz"), "rb") as src, open(net_file, "wb") as dst:
        dst.write(src.read())
    built = rn.build_real_net(net_file, agent="iqld")
    for agent in ("iqll", "iqld"):
        t = rn.real_net_tables(agent)
        for k in NetTables._ARRAYS:
            assert np.array_equal(np.asarray(getattr(t, k)), np.asarray(getattr(built, k))), (agent, k)
        assert t.node_names == built.node_names and t.n_s_ls == built.n_s_ls and t.n_w_ls == built.n_w_ls
        assert t.n_a_ls == built.n_a_ls and t.node_obs_off.tolist() == built.node_obs_off.tolist()
        assert t.n_obs == built.n_obs and max(t.n_a_ls) == 6 and set(t.n_w_ls) == {0}
