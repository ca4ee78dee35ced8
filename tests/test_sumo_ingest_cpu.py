"""CPU: general SUMO ingest (net/sumo_ingest.py, SURVEY 8f.2): signal programs, neighbour map and demand are read from
scenario FILES.  (1) a synthetic two-junction scenario written by tests/fixtures/make_mini_sumo.py loads, routes, and
runs in the oracle with vehicle conservation; (2) the Monaco scenario ingested from the reference's most.net.xml + a
route file written by the reference's own generator equals the hand-wired Monaco tables."""
import lzma
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests", "fixtures"))


def _mini(tmp_path):
    import make_mini_sumo
    return make_mini_sumo.write(str(tmp_path))


def test_mini_scenario_is_read_from_files(tmp_path):
    from deeprl_signal_control_b200.net import sumo_ingest as ing
    net_file, rou_file = _mini(tmp_path)
    phases = ing.read_tls_programs(net_file)
    assert phases == {"A": ["GGgrrrGGgrrr", "rrrGGgrrrGGg"], "B": ["GGgrrrGGgrrr", "rrrGGgrrrGGg"]}   # no yellow, no all-red
    assert ing.derive_neighbor_map(net_file, phases.keys()) == {"A": ["B"], "B": ["A"]}
    defs, flows = ing.read_flows(rou_file, 3600)
    assert defs[0] == ("W_A", "B_E", "A_B") and defs[3] == ("NB_B", "B_SB", "")
    assert flows[2] == (2, 100, 500, 450.0) and flows[3] == (3, 0, 300, 600.0)        # period 8 s; 50 vehicles / 300 s
    net = ing.load_sumo_scenario(net_file, rou_file, agent="ma2c", use_wait=True)
    assert net.node_names == ["A", "B"] and net.n_a_ls == [2, 2] and net.n_routes == 5
    for name in net.node_names:                       # controlled lanes in link-index order, 12 links, 4 detector lanes
        assert len(net.lanes_in[name]) == 12 and len(net.ilds_in[name]) == 4
    assert net.lanes_in["A"][:3] == ["NA_A_0"] * 3 and net.lanes_in["A"][9:] == ["W_A_0"] * 3
    # the route W_A -> A_B -> B_E crosses both signals: links carry (node, link index) of the straight movements
    r0 = [int(k) for k in net.route_link[0, :int(net.route_len[0])]]
    assert [int(net.link_node[k]) for k in r0[:2]] == [0, 1] and [int(net.link_tlidx[k]) for k in r0[:2]] == [10, 10]
    # the left turn NA_A -> A_B (link 2) yields to the opposing straight / right (junction response matrix -> foe mask)
    left = [k for k in range(net.n_links) if net.link_node[k] == 0 and net.link_tlidx[k] == 2]
    assert left and int(net.link_cross[left[0]]) == (1 << 7) | (1 << 6)
    # internal lane length is carried by the feeding lane; lane ends sit on the 1/64 m position grid
    assert np.allclose(net.lane_len[net.route_lane[0, 0]], 129.0) and np.all(net.lane_len * 64 == np.round(net.lane_len * 64))
    # demand: 600 veh/h for 600 s + 450 for 600 s + one per 8 s for 400 s + 50 + 240 veh/h for 600 s
    assert int(net.src_due.sum()) == 100 + 75 + 50 + 50 + 40
    # MA2C observation: own waves + neighbour waves + own waits + neighbour fingerprints
    assert net.n_s_ls == [4 + 4 + 4 + 1, 4 + 4 + 4 + 1] and net.n_f_ls == [1, 1] and net.n_w_ls == [4, 4]   # fingerprint = pi[:-1]


def test_mini_scenario_runs_in_the_oracle(tmp_path):
    from deeprl_signal_control_b200.net import sumo_ingest as ing
    from deeprl_signal_control_b200.net.tables import EnvParams
    from oracle.sim_ref import RefSim
    net = ing.load_sumo_scenario(*_mini(tmp_path), agent="greedy", use_wait=True)
    par = EnvParams(agent="greedy", episode_length_sec=900)
    sim = RefSim(net, par, 2)
    sim.reset(np.array([3, 4], np.uint64)); sim.set_train_mode(False)
    obs = sim.observe()
    for t in range(180):
        act = np.stack([[(t // 4) % 2, (t // 4 + 1) % 2]] * 2).astype(np.int32)      # alternate the two phases every 20 s
        obs, rew, g, d = sim.step(act)
        assert np.isfinite(obs).all() and (rew <= 0).all()
    m = sim.misc(0)
    assert m["departed"] + m["backlog"] == 315 and m["departed"] - m["arrived"] == m["live"]
    assert m["arrived"] > 250 and bool(d[0])


def test_monaco_from_files_equals_the_hand_wired_scenario(tmp_path):
    """most.net.xml + the route file the reference's generator writes (real_net/data/build_file.py:output_flows) +
    the reference's phase sets and neighbour lists -> the same tables as net/real_net.py's Monaco definition; the
    tlLogic programs of the net file themselves yield an action set for each of the 28 agents as well.
    Both files are stored under tests/golden: monaco_most.net.xml.xz is the reference's real_net/data/in/most.net.xml
    (xz-compressed, byte-identical once unpacked) and monaco_most_325.rou.xml is output_flows(325, seed=None)."""
    from deeprl_signal_control_b200.net import real_net as rn, sumo_ingest as ing
    gold = os.path.join(ROOT, "tests", "golden")
    rou = os.path.join(gold, "monaco_most_325.rou.xml")
    net_file = str(tmp_path / "most.net.xml")
    with lzma.open(os.path.join(gold, "monaco_most.net.xml.xz"), "rb") as src, open(net_file, "wb") as dst:
        dst.write(src.read())
    a = ing.load_sumo_scenario(net_file, rou, tls_phases={n: rn.PHASES[v[0]] for n, v in rn.NODES.items()},
                               neighbor_map={k: list(v[1]) for k, v in rn.NODES.items()}, agent="ma2c")
    b = rn.real_net_tables("ma2c")
    # routes (hence lane / link numbering) come in file order there and in FLOWS order here: compare by NAME
    assert a.node_names == b.node_names and a.n_s_ls == b.n_s_ls and a.n_a_ls == b.n_a_ls
    assert int(a.src_due.sum()) == int(b.src_due.sum()) == 2464
    assert sorted(a.lane_names) == sorted(b.lane_names) and a.n_links == b.n_links and a.n_routes == b.n_routes
    la, lb = dict(zip(a.lane_names, zip(a.lane_len, a.lane_vmax, a.lane_cap))), dict(zip(b.lane_names, zip(b.lane_len, b.lane_vmax, b.lane_cap)))
    assert la == lb
    assert a.lanes_in == b.lanes_in and a.ilds_in == b.ilds_in and a.neighbor_map == b.neighbor_map and a.phases == b.phases
    assert np.array_equal(a.node_green, b.node_green) and np.array_equal(a.node_major, b.node_major)
    ra = sorted(tuple(a.lane_names[l] for l in a.route_lane[r, :int(a.route_len[r])]) for r in range(a.n_routes))
    rb = sorted(tuple(b.lane_names[l] for l in b.route_lane[r, :int(b.route_len[r])]) for r in range(b.n_routes))
    assert ra == rb
    # per-second demand per route (by the route's lane-name tuple)
    da = {tuple(a.lane_names[l] for l in a.route_lane[r, :int(a.route_len[r])]): a.src_due[:, q].astype(int).tolist()
          for q, r in enumerate(a.src_route)}
    db = {tuple(b.lane_names[l] for l in b.route_lane[r, :int(b.route_len[r])]): b.src_due[:, q].astype(int).tolist()
          for q, r in enumerate(b.src_route)}
    assert da == db
    derived = ing.read_tls_programs(net_file)
    assert set(rn.NODES) <= set(derived)
    for n, v in rn.NODES.items():
        assert len(derived[n][0]) == len(rn.PHASES[v[0]][0]) and 1 <= len(derived[n]) <= 8
    nbr = ing.derive_neighbor_map(net_file, rn.NODES.keys())
    hits = sum(len(set(nbr[n]) & set(v[1])) for n, v in rn.NODES.items())
    total = sum(len(v[1]) for v in rn.NODES.values())
    assert hits >= 0.6 * total            # the hand-written lists are mostly the topological neighbours
