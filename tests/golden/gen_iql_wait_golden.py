"""Golden vectors of IQL-DQN WITH the wait branch (`q_fct`, agents/policies.py:352-360: n_w > 0, layer width
num_fc / 4), the case every agent of the large grid runs and learner_iql.npz (n_w = 0) does not cover.  Produced by
executing the reference's own DeepQPolicy graph (through agents/models.py:IQL) on tests/golden/tf1_shim.py, with the
protocol and key scheme of gen_learner_golden.run_iql: three consecutive policy.backward() calls per agent on fixed
minibatches; per minibatch the inputs, q values, loss, pre-clip gradient norm and gradients; weights after every Adam
step.

Output (committed): tests/golden/learner_iql_wait.npz
Run:  python tests/golden/gen_iql_wait_golden.py        (needs the reference checkout; NOT needed at test time)
"""
import os
import random

import numpy as np

import gen_learner_golden as g       # installs the TF1 shim and imports the reference's agents package

N_S, N_W, N_A = [30, 36], [6, 6], [5, 4]


def run_iql_wait():
    out = dict(n_s=np.array(N_S), n_w=np.array(N_W), n_a=np.array(N_A))
    np.random.seed(23); random.seed(23)
    model = g.ref_models.IQL(N_S, N_A, N_W, 1000, g.cfg(batch_size=20, lr_init=1e-4), seed=0, model_type="dqn")
    rng = np.random.default_rng(6)
    g.perturb_biases(rng)
    out["dqn/var_names"] = np.array(list(g.weights().keys()))
    g.put(out, "dqn/w0", g.f32(g.weights()))
    B = model.n_step
    for k in range(3):
        for i, p in enumerate(model.policy_ls):
            obs = rng.random((B, N_S[i])) * 2
            nxt = rng.random((B, N_S[i])) * 2
            acts = rng.integers(0, N_A[i], B)
            rs = rng.normal(0, 1, B)
            dones = rng.random(B) < 0.2
            wts = g.tf.trainable_variables(scope=p.name)
            feed = {p.S: obs, p.A: acts, p.S1: nxt, p.DONE: dones, p.R: rs}
            vals = model.sess.run([p.loss, p.grad_norm, p.qvalues] + g.tf.gradients(p.loss, wts), feed)
            pre = "dqn/k%d/a%d" % (k, i)
            out[pre + "/obs"], out[pre + "/next_obs"], out[pre + "/acts"] = obs, nxt, acts
            out[pre + "/rs"], out[pre + "/dones"] = rs, dones
            out[pre + "/loss"], out[pre + "/grad_norm"], out[pre + "/q"] = vals[0], vals[1], vals[2]
            for w, gr in zip(wts, vals[3:]):
                out[pre + "/g/" + w.name] = gr.astype(np.float32)
            p.backward(model.sess, obs, acts, nxt, dones, rs, 1e-4)
        g.put(out, "dqn/w%d" % (k + 1), g.f32(g.weights()))
    return out


def main():
    o = run_iql_wait()
    np.savez_compressed(os.path.join(g.HERE, "learner_iql_wait.npz"), **o)
    print("iql wait: loss", o["dqn/k0/a0/loss"], o["dqn/k0/a1/loss"], "grad_norm", o["dqn/k0/a0/grad_norm"])
    print("variables", list(o["dqn/var_names"]))


if __name__ == "__main__":
    main()
