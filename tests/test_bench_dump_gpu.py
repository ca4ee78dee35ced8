"""GPU: `bench.py --dump-outputs DIR` writes what the timed path computed in its last step, from seeded inputs, so that
two runs with the same arguments give the same arrays and `--steps` decides which step that is."""
import json
import os
import subprocess
import sys
import types

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
R = 256
SMALL = ["--replicas", str(R), "--warmup", "3", "--no-cpu-baseline"]


def _bench(out_dir, *args):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + SMALL + list(args) +
                         ["--dump-outputs", str(out_dir)], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    return json.loads(lines[0]), {f[:-4]: np.load(os.path.join(out_dir, f)) for f in sorted(os.listdir(out_dir))}


def _check_layout(d, names):
    assert sorted(d) == sorted(names)
    assert all(a.dtype == np.float32 for a in d.values())
    assert sum(a.nbytes for a in d.values()) <= 64 << 20
    assert np.array_equal(d["replicas"], np.arange(R))            # fewer replicas than the sample: all of them
    assert all(d[k].shape[0] == R for k in names if k not in ("params", "grad_norms"))


def _oracle_sim_mode(burnin, warmup, steps):
    """The CPU oracle (bit-exact with tsc_step) driven with bench.py's --mode sim inputs and step schedule."""
    import torch
    import bench
    from deeprl_signal_control_b200.dist import shard_replicas
    from deeprl_signal_control_b200.net.large_grid import build_large_grid
    from deeprl_signal_control_b200.net.tables import EnvParams
    from oracle.sim_ref import RefSim
    net, par = build_large_grid(agent="ma2c"), EnvParams(agent="ma2c")
    acts, fp = bench.sim_mode_inputs(net, R, torch.device("cuda", 0), 0)
    acts, fp = [a.cpu().numpy() for a in acts], fp.cpu().numpy()
    ref = RefSim(net, par, R)
    ref.reset(shard_replicas(0, 1, R, 12)[2])
    for n in (burnin, max(warmup, 3), steps):
        for i in range(n):
            out = ref.step(acts[i % len(acts)], fp)
    return dict(zip(("obs", "reward", "global_reward", "done"), out))


@pytest.mark.gpu
def test_sim_mode_dump_is_the_last_timed_step(tmp_path):
    line, a = _bench(tmp_path / "a", "--mode", "sim", "--burnin", "4", "--steps", "2")
    assert line["steps"] == 2
    _check_layout(a, ["obs", "reward", "global_reward", "done", "replicas"])
    want = _oracle_sim_mode(4, 3, 2)
    for k, v in want.items():
        assert np.array_equal(a[k], v.astype(np.float32)), k
    _, b = _bench(tmp_path / "b", "--mode", "sim", "--burnin", "4", "--steps", "2")
    for k in a:
        assert np.array_equal(a[k], b[k]), k
    _, c = _bench(tmp_path / "c", "--mode", "sim", "--burnin", "4", "--steps", "3")
    assert np.array_equal(c["obs"], _oracle_sim_mode(4, 3, 3)["obs"]) and not np.array_equal(a["obs"], c["obs"])


@pytest.mark.gpu
def test_train_mode_dump_is_reproducible(tmp_path):
    line, a = _bench(tmp_path / "a", "--burnin", "0", "--steps", "2")
    assert line["steps"] == 2 and line["config"]["updates_in_timed_region"] == 1
    _check_layout(a, ["params", "grad_norms", "obs", "reward", "action", "value", "replicas"])
    assert np.isfinite(a["params"]).all() and (a["grad_norms"] > 0).all()
    _, b = _bench(tmp_path / "b", "--burnin", "0", "--steps", "2")
    for k in ("obs", "reward", "action", "value", "replicas"):
        assert np.array_equal(a[k], b[k]), k
    for k in ("params", "grad_norms"):                  # gradient sums may be accumulated in any order
        np.testing.assert_allclose(a[k], b[k], rtol=1e-5, atol=1e-7, err_msg=k)


@pytest.mark.gpu
def test_train_mode_dump_holds_what_the_last_step_handed_out():
    """bench.last_step_outputs after a rollout that ends on an update equals what that last step's policy forward and
    simulator step returned (captured as they were returned) and the weights / norms after the update."""
    import bench
    from deeprl_signal_control_b200.agents.learner import BatchedA2C
    from deeprl_signal_control_b200.agents.trainer import BatchedTrainer
    from deeprl_signal_control_b200.net.large_grid import build_large_grid
    from deeprl_signal_control_b200.net.tables import EnvParams
    from deeprl_signal_control_b200.sim import BatchedSim
    net, par = build_large_grid(agent="ma2c"), EnvParams(agent="ma2c")
    Rt, n_step, norm, clip = 128, 4, 2000.0, 2.0
    sim = BatchedSim(net, par, Rt, device=0)
    lay = bench.make_layout(net, types.SimpleNamespace(agent="ma2c", policy="lstm"))
    model = BatchedA2C(lay, Rt, n_step=n_step, gamma=0.99, v_coef=0.5, max_grad_norm=40.0,
                       alpha=0.99, eps=1e-5, reward_norm=norm, reward_clip=clip, seed=1, chunk=Rt)
    tr = BatchedTrainer(sim, model, "ma2c", lr=5e-4, beta=0.01, seed0=12)
    seen = {}
    step0, forward0 = sim.step, model.forward

    def step(*a, **k):
        out = step0(*a, **k)
        seen["obs"], seen["reward"] = out[0].clone(), out[1].clone()
        return out

    def forward(*a, **k):
        out = forward0(*a, **k)
        if out[2] is not None:                          # a decision (not the bootstrap value of the update)
            seen["value"], seen["action"] = out[1].clone(), out[2].clone()
        return out

    sim.step, model.forward = step, forward
    tr.run(2 * n_step)
    assert tr.n_updates == 2
    d = bench.last_step_outputs(sim, tr)
    assert np.array_equal(d["replicas"], np.arange(Rt))
    got = {k: v.cpu().numpy() for k, v in seen.items()}
    assert np.array_equal(d["obs"], got["obs"]) and np.array_equal(d["value"], got["value"])
    assert np.array_equal(d["action"], got["action"].astype(np.float32))
    assert np.array_equal(d["reward"], np.clip(got["reward"] * np.float32(1.0 / norm), -clip, clip))
    assert np.array_equal(d["params"], model.P.cpu().numpy()) and np.array_equal(d["grad_norms"], model.norms.cpu().numpy())
