"""Monaco `real_net` scenario: SUMO net-file ingest -> NetTables.

Inputs (reference files, read-only): `real_net/data/in/most.net.xml` (netconvert output: edges, lanes,
connections with tl/linkIndex, junction right-of-way matrices) and the scenario definition of
`envs/real_net_env.py:20-68` (NODES, PHASES) + demand of `real_net/data/build_file.py:15-105`.

What is built (same conventions as net/large_grid.py, DESIGN.md §3):
  * lanes   = lanes used by the 16 demand routes + every lane a signalised node controls
              (agents observe all of them, envs/env.py:219-230), passenger lanes only for routing;
  * links   = the `<connection>`s along the routes; signalised ones carry (tl, linkIndex);
              foes = the junction's `response` row (who this link yields to) mapped to tl link indices;
  * routes  = fastest path (length / speed) from -> via... -> to on the passenger edge graph
              (SUMO's `<flow from to via>` semantics, build_file.py:76);
  * junction interiors have zero length in the model; the internal-lane length of the connection a
    route uses is added to the length of the lane that feeds it, so trip lengths are preserved.
Uncontrolled (priority) junctions on the way are treated as always open.
"""
from __future__ import annotations

import heapq
import os
import xml.etree.ElementTree as ET
from typing import Dict, List, Tuple

import numpy as np

from .tables import NetTables, build_obs_program, flow_due_table, phase_masks

# envs/real_net_env.py:20-47 — node: (phase key, neighbor list)
NODES = {'10026': ('6.0', ['9431', '9561', 'cluster_9563_9597', '9531']),
         '8794': ('4.0', ['cluster_8985_9609', '9837', '9058', 'cluster_9563_9597']),
         '8940': ('2.1', ['9007', '9429']),
         '8996': ('2.2', ['cluster_9389_9689', '9713']),
         '9007': ('2.3', ['9309', '8940']),
         '9058': ('4.0', ['cluster_8985_9609', '8794', 'joinedS_0']),
         '9153': ('2.0', ['9643']),
         '9309': ('4.0', ['9466', '9007', 'cluster_9043_9052']),
         '9413': ('2.3', ['9721', '9837']),
         '9429': ('5.0', ['cluster_9043_9052', 'joinedS_1', '8940']),
         '9431': ('2.4', ['9721', '9884', '9561', '10026']),
         '9433': ('2.5', ['joinedS_1']),
         '9466': ('4.0', ['9309', 'joinedS_0', 'cluster_9043_9052']),
         '9480': ('2.3', ['8996', '9713']),
         '9531': ('2.6', ['joinedS_1', '10026']),
         '9561': ('4.0', ['cluster_9389_9689', '10026', '9431', '9884']),
         '9643': ('2.3', ['9153']),
         '9713': ('3.0', ['9721', '9884', '8996']),
         '9721': ('6.0', ['9431', '9713', '9413']),
         '9837': ('3.1', ['9413', '8794', 'cluster_8985_9609']),
         '9884': ('2.7', ['9713', '9431', 'cluster_9389_9689', '9561']),
         'cluster_8751_9630': ('4.0', ['cluster_9389_9689']),
         'cluster_8985_9609': ('4.0', ['9837', '8794', '9058']),
         'cluster_9043_9052': ('4.1', ['cluster_9563_9597', '9466', '9309', '10026', 'joinedS_1']),
         'cluster_9389_9689': ('4.0', ['9884', '9561', 'cluster_8751_9630', '8996']),
         'cluster_9563_9597': ('4.2', ['10026', '8794', 'joinedS_0', 'cluster_9043_9052']),
         'joinedS_0': ('6.1', ['9058', 'cluster_9563_9597', '9466']),
         'joinedS_1': ('3.2', ['9531', '9429'])}

# envs/real_net_env.py:49-68
PHASES = {'4.0': ['GGgrrrGGgrrr', 'rrrGGgrrrGGg', 'rrGrrrrrGrrr', 'rrrrrGrrrrrG'],
          '4.1': ['GGgrrGGGrrr', 'rrGrrrrrrrr', 'rrrGgrrrGGg', 'rrrrGrrrrrG'],
          '4.2': ['GGGGrrrrrrrr', 'GGggrrGGggrr', 'rrrGGGGrrrrr', 'grrGGggrrGGg'],
          '2.0': ['GGrrr', 'ggGGG'],
          '2.1': ['GGGrrr', 'rrGGGg'],
          '2.2': ['Grr', 'gGG'],
          '2.3': ['GGGgrr', 'GrrrGG'],
          '2.4': ['GGGGrr', 'rrrrGG'],
          '2.5': ['Gg', 'rG'],
          '2.6': ['GGGg', 'rrrG'],
          '2.7': ['GGg', 'rrG'],
          '3.0': ['GGgrrrGGg', 'rrGrrrrrG', 'rrrGGGGrr'],
          '3.1': ['GgrrGG', 'rGrrrr', 'rrGGGr'],
          '3.2': ['GGGGrrrGG', 'rrrrGGGGr', 'GGGGrrGGr'],
          '5.0': ['GGGGgrrrrGGGggrrrr', 'grrrGrrrrgrrGGrrrr', 'GGGGGrrrrrrrrrrrrr',
                  'rrrrrrrrrGGGGGrrrr', 'rrrrrGGggrrrrrggGg'],
          '6.0': ['GGGgrrrGGGgrrr', 'rrrGrrrrrrGrrr', 'GGGGrrrrrrrrrr', 'rrrrrrrrrrGGGG',
                  'rrrrGGgrrrrGGg', 'rrrrrrGrrrrrrG'],
          '6.1': ['GGgrrGGGrrrGGGgrrrGGGg', 'rrGrrrrrrrrrrrGrrrrrrG', 'GGGrrrrrGGgrrrrGGgrrrr',
                  'GGGrrrrrrrGrrrrrrGrrrr', 'rrrGGGrrrrrrrrrrrrGGGG', 'rrrGGGrrrrrGGGgrrrGGGg']}

# real_net/data/build_file.py:27-67 — (from, to, via) per group
FLOWS = [
    [('-10114#1', '-10079', '10115#2 -10109'), ('-10114#1', '-10079', '-10114#0 10108#0 gneE5'),
     ('-10114#1', '-10079', '-10114#0 10108#0 10102'), ('-10114#1', '10076', '-10114#0 10107 10102')],
    [('10096#1', '10063', '10089#3'), ('-10185#1', '-10071#3', 'gneE20'),
     ('10096#1', '10063', '10109'), ('-10185#1', '-10061#5', 'gneE19')],
    [('10052#1', '10104', '10181#1 -10089#3'), ('-10064#9', '10104', '-10068 10102'),
     ('-10051#2', '10043', '10181#1 gneE4'), ('-10064#9', '-10110', '-10064#4 -10064#3')],
    [('10061#4', '-10085', '10065#2 10102'), ('10071#3', '10085', '10065#2 -10064#3'),
     ('-10070#1', '-10086', 'gneE9'), ('-10063', '10085', 'gneE8')],
]
VOLS_A = [1, 2, 4, 4, 4, 4, 2, 1, 0, 0, 0]     # build_file.py:72-74
VOLS_B = [0, 0, 0, 1, 2, 4, 4, 4, 4, 2, 1]


def _passenger(lane) -> bool:
    allow, dis = lane.get('allow'), lane.get('disallow')
    if allow is not None:
        return 'passenger' in allow.split()
    if dis is not None:
        return 'passenger' not in dis.split()
    return True


def parse_net(net_file: str):
    root = ET.parse(net_file).getroot()
    edges, internal_len = {}, {}
    for e in root.findall('edge'):
        lanes = e.findall('lane')
        if e.get('function') == 'internal':
            for l in lanes:
                internal_len[l.get('id')] = float(l.get('length'))
            continue
        edges[e.get('id')] = dict(
            lanes=[dict(id=l.get('id'), length=float(l.get('length')), speed=float(l.get('speed')),
                        passenger=_passenger(l)) for l in lanes])
    cons = [dict(c.attrib) for c in root.findall('connection') if not c.get('from').startswith(':')]
    junctions = {}
    for j in root.findall('junction'):
        if j.get('type') == 'internal':
            continue
        junctions[j.get('id')] = dict(int_lanes=(j.get('intLanes') or '').split(),
                                      response=[r.get('response') for r in j.findall('request')])
    return edges, cons, junctions, internal_len


def _fastest_path(adj, cost, src, dst):
    dist, prev, pq = {src: 0.0}, {}, [(0.0, src)]
    while pq:
        dcur, u = heapq.heappop(pq)
        if u == dst:
            break
        if dcur > dist.get(u, 1e30):
            continue
        for v in adj.get(u, ()):
            nd = dcur + cost[v]
            if nd < dist.get(v, 1e30) - 1e-12:
                dist[v], prev[v] = nd, u
                heapq.heappush(pq, (nd, v))
    if dst not in dist:
        raise ValueError('no route %s -> %s' % (src, dst))
    path = [dst]
    while path[-1] != src:
        path.append(prev[path[-1]])
    return path[::-1]


def monaco_flow_list(flow_rate: int = 325):
    """(route index, begin, end, vehsPerHour) of real_net/data/build_file.py:72-105."""
    times = np.arange(0, 3301, 300)
    flow_list = []
    for i in range(len(times) - 1):
        tb, te = int(times[i]), int(times[i + 1])
        for j in (0, 1):
            for ind in range(VOLS_A[i]):
                flow_list.append((j * 4 + ind, tb, te, int(flow_rate)))
        for j in (2, 3):
            for ind in range(VOLS_B[i]):
                flow_list.append((j * 4 + ind, tb, te, int(flow_rate)))
    return flow_list


def build_real_net(net_file: str, flow_rate: int = 325, agent: str = 'ma2c', coop_gamma: float = 0.9,
                   episode_length_sec: int = 3600, veh_len: float = 5.0, min_gap: float = 2.5) -> NetTables:
    """The Monaco scenario of the reference: its hand-written NODES / PHASES / flows on most.net.xml."""
    return build_from_sumo(net_file, tls_phases={n: PHASES[v[0]] for n, v in NODES.items()},
                           neighbor_map={k: list(v[1]) for k, v in NODES.items()},
                           flow_defs=[fl for grp in FLOWS for fl in grp], flow_list=monaco_flow_list(flow_rate),
                           agent=agent, coop_gamma=coop_gamma, episode_length_sec=episode_length_sec,
                           veh_len=veh_len, min_gap=min_gap, use_wait=False)     # STATE_NAMES = ['wave'] (:18)


def build_from_sumo(net_file: str, tls_phases: Dict[str, List[str]], neighbor_map: Dict[str, List[str]],
                    flow_defs: List[Tuple[str, str, str]], flow_list: List[Tuple[int, int, int, float]],
                    agent: str = 'ma2c', coop_gamma: float = 0.9, episode_length_sec: int = 3600,
                    veh_len: float = 5.0, min_gap: float = 2.5, use_wait: bool = False) -> NetTables:
    """Any SUMO scenario -> NetTables (SURVEY 8f.2).
      tls_phases    signalised node -> its phase strings = the agent's action set (envs/real_net_env.py:49-68 for
                    Monaco; net/sumo_ingest.py derives them from the <tlLogic> programs of a net file)
      neighbor_map  node -> neighbour nodes in observation order (envs/real_net_env.py:20-47)
      flow_defs     routes as (from edge, to edge, 'via edges'), routed as SUMO routes <flow from to via>
      flow_list     (route index, begin s, end s, vehsPerHour)"""
    edges, cons, junctions, internal_len = parse_net(net_file)
    NODES_ = {n: (n, list(neighbor_map.get(n, []))) for n in tls_phases}
    PHASES_ = dict(tls_phases)
    node_names = sorted(NODES_.keys())
    node_idx = {n: i for i, n in enumerate(node_names)}

    # ---- signalised links: lanes_in[node][linkIndex] (== traci getControlledLanes) -------------------
    lanes_in: Dict[str, List[str]] = {}
    tl_con = {}
    for c in cons:
        if c.get('tl'):
            tl_con.setdefault(c['tl'], {})[int(c['linkIndex'])] = c
    for name in node_names:
        links = tl_con[name]
        n_link = len(PHASES_[name][0])
        assert sorted(links) == list(range(n_link)), (name, sorted(links), n_link)
        lanes_in[name] = ['%s_%s' % (links[i]['from'], links[i]['fromLane']) for i in range(n_link)]
    ilds_in = {n: list(dict.fromkeys(lanes_in[n])) for n in node_names}

    # ---- routes on the passenger edge graph -------------------------------------------------------------
    usable = {eid for eid, e in edges.items() if any(l['passenger'] for l in e['lanes'])}
    adj: Dict[str, set] = {}
    con_of: Dict[Tuple[str, str], List[dict]] = {}
    for c in cons:
        f, t = c['from'], c['to']
        if f in usable and t in usable and edges[f]['lanes'][int(c['fromLane'])]['passenger'] \
                and edges[t]['lanes'][int(c['toLane'])]['passenger']:
            adj.setdefault(f, set()).add(t)
            con_of.setdefault((f, t), []).append(c)
    cost = {eid: edges[eid]['lanes'][0]['length'] / max(l['speed'] for l in edges[eid]['lanes'])
            for eid in usable}
    route_edges = []
    for (src, dst, via) in flow_defs:
        stops = [src] + via.split() + [dst]
        path = [src]
        for a, b in zip(stops[:-1], stops[1:]):
            path += _fastest_path(adj, cost, a, b)[1:]
        route_edges.append(path)

    # ---- lane set ------------------------------------------------------------------------------------------
    lane_names: List[str] = []
    lane_id: Dict[str, int] = {}

    def add_lane(name):
        if name not in lane_id:
            lane_id[name] = len(lane_names)
            lane_names.append(name)
        return lane_id[name]

    # per route hop: the connection used and the lane it leaves from (rightmost lane that connects)
    hop_con: List[List[dict]] = []
    for path in route_edges:
        cs = []
        for a, b in zip(path[:-1], path[1:]):
            cand = sorted(con_of[(a, b)], key=lambda c: (int(c['fromLane']), int(c['toLane'])))
            cs.append(cand[0])
        hop_con.append(cs)
    for path, cs in zip(route_edges, hop_con):
        for k, e in enumerate(path):
            if k < len(cs):
                add_lane('%s_%s' % (e, cs[k]['fromLane']))
            else:
                first = next(i for i, l in enumerate(edges[e]['lanes']) if l['passenger'])
                add_lane('%s_%d' % (e, first))
    for name in node_names:
        for ln in ilds_in[name]:
            add_lane(ln)

    def lane_attr(name):
        eid, li = name.rsplit('_', 1)
        return edges[eid]['lanes'][int(li)]

    lane_len = np.array([lane_attr(n)['length'] for n in lane_names], np.float64)
    lane_vmax = np.array([lane_attr(n)['speed'] for n in lane_names], np.float32)

    # ---- links ------------------------------------------------------------------------------------------------
    link_key: Dict[Tuple[int, str], int] = {}
    link_from, link_to, link_node, link_tlidx, link_vmax, link_cross = [], [], [], [], [], []
    link_to_edge: List[str] = []
    via_of: List[str] = []

    def add_link(c):
        f = lane_id['%s_%s' % (c['from'], c['fromLane'])]
        key = (f, c['to'])
        if key in link_key:
            return link_key[key]
        to_name = '%s_%s' % (c['to'], c['toLane'])
        lid = len(link_from)
        link_key[key] = lid
        link_from.append(f)
        link_to.append(lane_id.get(to_name, -1))
        tl = c.get('tl')
        link_node.append(node_idx[tl] if tl in node_idx else -1)
        link_tlidx.append(int(c['linkIndex']) if tl in node_idx else 0)
        link_vmax.append(1.0e9)
        link_cross.append(0)
        link_to_edge.append(c['to'])
        via_of.append(c.get('via', ''))
        return lid

    routes_lane, routes_link = [], []
    for path, cs in zip(route_edges, hop_con):
        ls, ks = [], []
        for k, e in enumerate(path):
            if k < len(cs):
                ls.append(lane_id['%s_%s' % (e, cs[k]['fromLane'])])
                ks.append(add_link(cs[k]))
            else:
                first = next(i for i, l in enumerate(edges[e]['lanes']) if l['passenger'])
                ls.append(lane_id['%s_%d' % (e, first)])
                ks.append(-1)
        routes_lane.append(ls); routes_link.append(ks)
    n_links = len(link_from)
    # junction interiors: add the used connection's internal length to the feeding lane
    extra = np.zeros(len(lane_names))
    for l in range(n_links):
        v = via_of[l]
        if v:
            extra[link_from[l]] = max(extra[link_from[l]], internal_len.get(v, 0.0))
    lane_len = (lane_len + extra).astype(np.float32)
    # foes from the junction right-of-way matrix (`response`: bit j set = yield to request j)
    int_to_tl: Dict[str, Tuple[int, int]] = {}
    for c in cons:
        if c.get('tl') in node_idx and c.get('via'):
            int_to_tl[c['via']] = (node_idx[c['tl']], int(c['linkIndex']))
    for l in range(n_links):
        v = via_of[l]
        if link_node[l] < 0 or not v:
            continue
        jid = v[1:].rsplit('_', 2)[0]
        j = junctions.get(jid)
        if j is None or v not in j['int_lanes']:
            continue
        resp = j['response'][j['int_lanes'].index(v)]
        mask = 0
        for jj, il in enumerate(j['int_lanes']):
            if resp[len(resp) - 1 - jj] == '1' and il in int_to_tl and int_to_tl[il][0] == link_node[l]:
                mask |= 1 << int_to_tl[il][1]
        link_cross[l] = mask
    # links entering each lane (by destination EDGE: lane choice at entry), straight-ish order = link id
    n_lanes = len(lane_names)
    inl = [[] for _ in range(n_lanes)]
    lane_edge = [n.rsplit('_', 1)[0] for n in lane_names]
    for l in range(n_links):
        for ln in range(n_lanes):
            if lane_edge[ln] == link_to_edge[l]:
                inl[ln].append(l)
    lane_inl_off = np.concatenate([[0], np.cumsum([len(x) for x in inl])]).astype(np.int32)
    lane_inl = np.array([l for x in inl for l in x], np.int32)
    lane_cap = np.array([int(np.ceil(L / (veh_len + min_gap))) + 1 for L in lane_len], np.int32)
    lane_slot0 = np.concatenate([[0], np.cumsum(lane_cap)[:-1]]).astype(np.int32)

    # ---- per-node tables ---------------------------------------------------------------------------------------
    n_nodes = len(node_names)
    max_phases = max(len(PHASES_[n]) for n in node_names)
    node_green = np.zeros((n_nodes, max_phases), np.uint32)
    node_major = np.zeros((n_nodes, max_phases), np.uint32)
    node_n_phases = np.zeros(n_nodes, np.int32)
    for i, name in enumerate(node_names):
        ph = PHASES_[name]
        g, m = phase_masks(ph)
        node_green[i, :len(ph)] = g; node_major[i, :len(ph)] = m
        node_n_phases[i] = len(ph)
    det_lane, node_det_off = [], [0]
    for name in node_names:
        det_lane += [lane_id[s] for s in ilds_in[name]]
        node_det_off.append(len(det_lane))
    neighbor_map = {k: [n for n in v[1] if n in node_idx] for k, v in NODES_.items()}
    node_nbr, node_nbr_off = [], [0]
    for name in node_names:
        node_nbr += [node_idx[n] for n in neighbor_map[name]]
        node_nbr_off.append(len(node_nbr))

    # ---- demand: build_file.py:72-105 --------------------------------------------------------------------------------
    max_hops = max(len(r) for r in routes_lane)
    route_lane = np.full((len(routes_lane), max_hops), -1, np.int16)
    route_link = np.full((len(routes_lane), max_hops), -1, np.int16)
    for r, (ls, ks) in enumerate(zip(routes_lane, routes_link)):
        route_lane[r, :len(ls)] = ls; route_link[r, :len(ks)] = ks
    src_lane = [r[0] for r in routes_lane]
    src_route = list(range(len(routes_lane)))
    flow_list = [(int(r), int(tb), int(te), rate) for r, tb, te, rate in flow_list]
    src_due = flow_due_table(flow_list, episode_length_sec, len(src_lane))

    net = NetTables(
        node_names=node_names, lane_names=lane_names, neighbor_map=neighbor_map,
        phases={n: list(PHASES_[n]) for n in node_names}, lanes_in=lanes_in, ilds_in=ilds_in,
        max_hops=max_hops, horizon=episode_length_sec, max_phases=max_phases, max_na=max_phases,
        lane_len=lane_len, lane_vmax=lane_vmax, lane_cap=lane_cap, lane_slot0=lane_slot0,
        lane_inl_off=lane_inl_off, lane_inl=lane_inl,
        link_from=np.array(link_from, np.int32), link_to=np.array(link_to, np.int32),
        link_node=np.array(link_node, np.int32), link_tlidx=np.array(link_tlidx, np.int32),
        link_vmax=np.array(link_vmax, np.float32), link_cross=np.array(link_cross, np.uint32),
        link_merge=np.zeros(n_links, np.uint32),
        route_len=np.array([len(r) for r in routes_lane], np.int32), route_lane=route_lane, route_link=route_link,
        node_n_phases=node_n_phases, node_green=node_green, node_major=node_major,
        node_det_off=np.array(node_det_off, np.int32), det_lane=np.array(det_lane, np.int32),
        node_nbr_off=np.array(node_nbr_off, np.int32), node_nbr=np.array(node_nbr, np.int32),
        src_lane=np.array(src_lane, np.int32), src_route=np.array(src_route, np.int32), src_due=src_due,
        route_names=['%s->%s via %s' % f for f in flow_defs],
    )
    net.flow_list = flow_list
    net.route_edges = route_edges
    build_obs_program(net, agent, coop_gamma, use_wait=use_wait)
    return net.finalize()


# --------------------------------------------------------------------------------------------------------------------
_CACHE = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'data', 'real_net_tables_%s.npz')
_LIST_FIELDS = ('node_names', 'lane_names', 'route_names', 'n_s_ls', 'n_a_ls', 'n_w_ls', 'n_f_ls')


def save_tables(net: NetTables, path: str):
    import json
    arrays = {k: getattr(net, k) for k in NetTables._ARRAYS}
    meta = dict(max_hops=net.max_hops, horizon=net.horizon, max_phases=net.max_phases, max_na=net.max_na,
                neighbor_map=net.neighbor_map, phases=net.phases, lanes_in=net.lanes_in, ilds_in=net.ilds_in,
                **{k: list(getattr(net, k)) for k in _LIST_FIELDS})
    os.makedirs(os.path.dirname(path), exist_ok=True)
    np.savez_compressed(path, meta=json.dumps(meta), **arrays)


def load_tables(path: str) -> NetTables:
    import json
    z = np.load(path, allow_pickle=False)
    meta = json.loads(str(z['meta']))
    net = NetTables(node_names=meta['node_names'], lane_names=meta['lane_names'], neighbor_map=meta['neighbor_map'],
                    phases=meta['phases'], lanes_in=meta['lanes_in'], ilds_in=meta['ilds_in'],
                    max_hops=meta['max_hops'], horizon=meta['horizon'], max_phases=meta['max_phases'],
                    max_na=meta['max_na'])
    for k in NetTables._ARRAYS:
        if k in z.files:                     # caches written before a table was added keep their defaults
            setattr(net, k, z[k])
    for k in _LIST_FIELDS:
        setattr(net, k, [x for x in meta[k]])
    return net.finalize()


def real_net_tables(agent: str = 'ma2c', net_file: str | None = None, flow_rate: int = 325,
                    coop_gamma: float = 0.9) -> NetTables:
    """Tables for the Monaco scenario: parsed from `net_file` when given (a reference checkout),
    else from the derived table cache shipped with the package (generated by the same code)."""
    if net_file is not None and os.path.exists(net_file):
        return build_real_net(net_file, flow_rate=flow_rate, agent=agent, coop_gamma=coop_gamma)
    # iqll / iqld observe and are rewarded like ia2c (AGENT_MODES, build_obs_program): they share its cache
    path = _CACHE % ('ia2c' if agent in ('iqll', 'iqld') else agent)
    if not os.path.exists(path):
        raise FileNotFoundError('no Monaco net file given and no derived table cache at %s' % path)
    return load_tables(path)
