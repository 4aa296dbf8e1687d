"""
TEST INFRASTRUCTURE -- golden-vector generator.

Runs the UNMODIFIED reference Python (/root/reference/graph_ltpl, commit 18763ef9) in THIS container and stores its
inputs/outputs as small fixtures under tests/golden/.  The reference cannot be imported as is (SURVEY.md section 0):
  * `igraph` and `trajectory_planning_helpers` are absent  -> oracle/shims/{igraph,trajectory_planning_helpers} (restated)
  * `zmq` absent (objectlist_dummy.py:2)                    -> oracle/shims/zmq (empty)
  * NumPy-2 removals `np.object` (main_offline_callback.py:160) and `np.Inf` (MOPG:96) -> aliased below
Everything else (Graph_LTPL, OnlineTrajectoryHandler, main_online_path_gen, gen_local_node_template, GraphBase,
ObjectListInterface, VpForwardBackward, calc_vel_profile_follow, the whole offline pipeline ...) is the reference's own
code, executed verbatim.  /root/reference does not travel to the GPU box, hence the committed fixtures.

Usage (from the repo root):   python -m oracle.gen_golden [--quick]
"""

import argparse
import configparser
import os
import sys
import time

os.environ.setdefault('OPENBLAS_NUM_THREADS', '1')

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = '/root/reference'
GOLDEN = os.path.join(REPO, 'tests', 'golden')
ACTIONS = ("straight", "follow", "left", "right")


def load_reference(use_shims=True):
    """import the reference package on top of the shims (use_shims=False: on REAL python-igraph /
    trajectory_planning_helpers installs, to compare the reference on them with the stored fixtures); returns the
    `graph_ltpl` module."""
    if not os.path.isdir(REF):
        raise RuntimeError("/root/reference is not available on this box")
    for p in ((REPO, os.path.join(REPO, 'oracle', 'shims'), REF) if use_shims else (REPO, REF)):
        if p not in sys.path:
            sys.path.insert(0, p)
    if not hasattr(np, 'object'):
        np.object = object
    if not hasattr(np, 'Inf'):
        np.Inf = np.inf
    # The reference addresses graph vertices by str((layer, node)) (GB:163, 742); with its pinned NumPy 1.x a NumPy
    # integer prints as '41', with NumPy 2 as 'np.int64(41)' -- which silently disables remove_nodes_filter once GLNT:74
    # has turned the zone lists into NumPy integers.  Restore the NumPy 1.x scalar repr the reference was written for.
    np.set_printoptions(legacy="1.25")
    import graph_ltpl  # noqa
    import graph_ltpl.Graph_LTPL as gl
    gl.FORCE_RECALC = False
    return graph_ltpl


def write_offline_ini(path, overrides):
    cfg = configparser.ConfigParser()
    cfg.read(os.path.join(REF, 'params', 'ltpl_config_offline.ini'))
    for key, val in (overrides or {}).items():
        for sec in cfg.sections():
            if key in cfg[sec]:
                cfg[sec][key] = str(val)
    with open(path, 'w') as fh:
        cfg.write(fh)


OPEN_ROWS = 560   # data rows of the Monteblanco file kept for the open-track fixture (~1.67 km, 88 layers)


def write_open_track_csv(dst):
    """an OPEN track: the first OPEN_ROWS points of the reference's Monteblanco trajectory file (header kept); the
    reference detects it as unclosed (main_offline_callback.py:90-99)."""
    lines = open(REF + "/inputs/traj_ltpl_cl/traj_ltpl_cl_monteblanco.csv").read().splitlines()
    hdr = [ln for ln in lines if ln.startswith('#')]
    rows = [ln for ln in lines if not ln.startswith('#')]
    open(dst, 'w').write("\n".join(hdr + rows[:OPEN_ROWS]) + "\n")


def make_ltpl(graph_ltpl, tag, overrides=None, controller_type=None, veh=None, csv=None):
    ini = '/tmp/golden_offline_%s.ini' % tag
    write_offline_ini(ini, overrides)
    online = REF + "/params/ltpl_config_online.ini"
    if controller_type is not None:                       # same file, other follow-mode controller (ini line 35)
        txt = open(online).read()
        assert txt.count("controller_type=PD\n") == 1
        online = '/tmp/golden_online_%s_%s.ini' % (tag, controller_type)
        open(online, 'w').write(txt.replace("controller_type=PD\n", "controller_type=%s\n" % controller_type))
    path_dict = {'globtraj_input_path': csv or (REF + "/inputs/traj_ltpl_cl/traj_ltpl_cl_monteblanco.csv"),
                 'graph_store_path': "/tmp/golden_graph_%s.pckl" % tag,
                 'ltpl_offline_param_path': ini,
                 'ltpl_online_param_path': online}
    ltpl = graph_ltpl.Graph_LTPL.Graph_LTPL(path_dict=path_dict, visual_mode=False, log_to_file=False)
    t0 = time.time()
    ltpl.graph_init(**(veh or {}))
    print("[%s] reference graph_init: %.1f s" % (tag, time.time() - t0))
    return ltpl, path_dict


def ax_max_machines_table():
    tab = np.loadtxt(REF + "/inputs/veh_dyn_info/ax_max_machines.csv", comments='#', delimiter=',')
    return np.vstack((tab, [100.0, tab[-1, 1]]))


def run_tick(ltpl, pos, heading, vel, object_list, vel_kwargs, full=False, blocked_zones=None, vel_est=None, gg_fn=None):
    """one stateless planning tick through the reference's public API (main_min_example.py:69-104 flow).
    gg_fn: location dependent friction -- local_gg = {action: [gg_fn(path[:, 0:2])]} (OTH:649-666)."""
    name = '_Graph_LTPL__nmbr_export_points'
    keep = getattr(ltpl, name)
    if full:
        setattr(ltpl, name, 10 ** 6)
    try:
        out_of_track = ltpl.set_startpos(pos_est=np.array(pos), heading_est=float(heading), vel_est=float(vel))
        rec = {'out_of_track': bool(out_of_track)}
        if out_of_track:
            return rec
        oth = ltpl._Graph_LTPL__oth
        # zone objects persist inside the reference instance: every tick here is a FIRST tick, so start without zones
        ltpl._Graph_LTPL__obj_zone = []
        ltpl._Graph_LTPL__obj_list_handler._ObjectListInterface__object_zones = []
        path_dict = ltpl.calc_paths(prev_action_id="straight", object_list=object_list, blocked_zones=blocked_zones)
        rec['paths'] = {k: [np.array(a) for a in v] for k, v in path_dict.items()}
        rec['nodes'] = {k: [list(map(list, n)) for n in v]
                        for k, v in oth._OnlineTrajectoryHandler__last_action_set_nodes.items()}
        rec['node_idx'] = {k: [np.array(n) for n in v]
                           for k, v in oth._OnlineTrajectoryHandler__last_action_set_node_idx.items()}
        rec['coeff'] = {k: [np.array(n) for n in v]
                        for k, v in oth._OnlineTrajectoryHandler__last_action_set_coeff.items()}
        rec['red_len'] = {k: list(v) for k, v in oth._OnlineTrajectoryHandler__last_action_set_red_len.items()}
        rec['closest_obj_index'] = oth._OnlineTrajectoryHandler__closest_obj_index
        rec['start_node'] = list(oth._OnlineTrajectoryHandler__start_node)
        if gg_fn is not None:
            vel_kwargs = dict(vel_kwargs, local_gg={k: [gg_fn(v[0][:, 0:2])] for k, v in path_dict.items()})
        traj, ids, _ = ltpl.calc_vel_profile(pos_est=np.array(pos), vel_est=float(vel if vel_est is None else vel_est),
                                             **vel_kwargs)
        rec['traj'] = {k: [np.array(a) for a in v] for k, v in traj.items()}
        rec['ids'] = dict(ids)
        return rec
    finally:
        setattr(ltpl, name, keep)


def pack_ticks(recs, pmax=None):
    """ragged per-scenario records -> padded arrays."""
    n = len(recs)
    hmax = 1
    for r in recs:
        for k in r.get('paths', {}):
            pmax = max(pmax or 0, r['paths'][k][0].shape[0])
            hmax = max(hmax, len(r['nodes'][k][0]))
    out = dict(
        out_of_track=np.array([r['out_of_track'] for r in recs]),
        path=np.zeros((n, 4, pmax, 5)), path_len=np.zeros((n, 4), dtype=np.int32),
        nodes=np.full((n, 4, hmax, 2), -1, dtype=np.int32), nodes_len=np.zeros((n, 4), dtype=np.int32),
        node_idx=np.full((n, 4, hmax), -1, dtype=np.int32),
        coeff=np.zeros((n, 4, hmax, 8)), coeff_len=np.zeros((n, 4), dtype=np.int32),
        red_len=np.zeros((n, 4), dtype=np.int8),
        traj=np.zeros((n, 4, pmax, 7)), traj_len=np.zeros((n, 4), dtype=np.int32),
        traj_id=np.full((n, 4), -1, dtype=np.int32),
        closest_obj_index=np.full(n, -1, dtype=np.int32), start_node=np.full((n, 2), -1, dtype=np.int32))
    for i, r in enumerate(recs):
        if r['out_of_track']:
            continue
        out['closest_obj_index'][i] = -1 if r['closest_obj_index'] is None else r['closest_obj_index']
        out['start_node'][i] = r['start_node']
        for a, act in enumerate(ACTIONS):
            if act in r['paths'] and len(r['paths'][act]) and np.size(r['paths'][act][0]):
                p = r['paths'][act][0]
                out['path'][i, a, :p.shape[0]] = p
                out['path_len'][i, a] = p.shape[0]
                nd = [[-1 if v is None else int(v) for v in pair] for pair in r['nodes'][act][0]]
                out['nodes'][i, a, :len(nd)] = nd
                out['nodes_len'][i, a] = len(nd)
                ni = r['node_idx'][act][0]
                out['node_idx'][i, a, :len(ni)] = ni
                c = r['coeff'][act][0]
                out['coeff'][i, a, :c.shape[0]] = c
                out['coeff_len'][i, a] = c.shape[0]
                out['red_len'][i, a] = int(bool(r['red_len'][act][0]))
            if act in r['traj'] and len(r['traj'][act]):
                t = r['traj'][act][0]
                out['traj'][i, a, :t.shape[0]] = t
                out['traj_len'][i, a] = t.shape[0]
                out['traj_id'][i, a] = r['ids'][act]
    return out


def make_zone(lat, rng, pos):
    """random blocked zone ('nodes' type: [layer ids, node ids, left bound, right bound], LTPL:311-312) ahead of /
    around the ego position: 3-12 layers, the left or the right part of every layer (10 %: one fully blocked layer)."""
    near = int(np.argmin(np.sum(np.power(lat.refline - np.asarray(pos), 2), axis=1)))
    first = (near + int(rng.integers(0, 11))) % lat.num_layers
    length = int(rng.integers(3, 13))
    full_width = rng.random() < 0.1
    left = rng.random() < 0.5
    layers, nodes = [], []
    for k in range(1 if full_width else length):
        l = (first + k) % lat.num_layers
        n_l = lat.nodes_in_layer(l)
        m = int(rng.integers(1, n_l))
        ids = range(n_l) if full_width else (range(0, m) if left else range(m, n_l))
        for j in ids:
            layers.append(l)
            nodes.append(j)
    return [layers, nodes, np.zeros((2, 2)), np.zeros((2, 2))]


def ext_fixture(ltpl, lat, track, n, vel_kwargs):
    """zones (GLNT:43-99) + emergency trajectory (OTH:1027-1034): stateless first ticks through the reference."""
    from graphbasedlocaltrajectoryplanner_b200.scenarios import make_scenarios
    sc = make_scenarios(track, n, seed=777, n_obj_min=0, n_obj_max=3)
    rng = np.random.default_rng(778)
    vk = dict(vel_kwargs, incl_emerg_traj=True)
    recs, zones = [], []
    for b in range(sc.size):
        zone = make_zone(lat, rng, sc.pos[b]) if b % 4 != 3 else None
        zones.append(zone)
        bz = None if zone is None else {'zone_%d' % b: zone}
        recs.append(run_tick(ltpl, sc.pos[b], sc.heading[b], sc.vel[b], sc.object_list(b), vk, full=True,
                             blocked_zones=bz))
    pk = pack_ticks(recs)
    pmax = pk['path'].shape[2]
    zmax = max([len(z[0]) for z in zones if z is not None] + [1])
    em = np.zeros((n, pmax, 7))
    em_len = np.zeros(n, dtype=np.int32)
    em_id = np.full(n, -1, dtype=np.int32)
    z_layers = np.full((n, zmax), -1, dtype=np.int32)
    z_nodes = np.full((n, zmax), -1, dtype=np.int32)
    for i, r in enumerate(recs):
        if zones[i] is not None:
            z_layers[i, :len(zones[i][0])] = zones[i][0]
            z_nodes[i, :len(zones[i][1])] = zones[i][1]
        if 'traj' in r and 'emergency' in r['traj']:
            t = r['traj']['emergency'][0]
            em[i, :t.shape[0]] = t
            em_len[i] = t.shape[0]
            em_id[i] = r['ids']['emergency']
    pk.update(em_traj=em, em_len=em_len, em_id=em_id, zone_layers=z_layers, zone_nodes=z_nodes, sc_pos=sc.pos,
              sc_heading=sc.heading, sc_vel=sc.vel, sc_n_obj=sc.n_obj, sc_obj=sc.obj,
              ax_max_machines=vel_kwargs['ax_max_machines'])
    acts = {a: int((pk['path_len'][:, i] > 0).sum()) for i, a in enumerate(ACTIONS)}
    print("[ext] zones: %d of %d scenarios; action paths %s; emergency trajectories %d; reduced %d; out of track %d" %
          (sum(z is not None for z in zones), n, acts, int((em_len > 0).sum()), int(pk['red_len'].sum()),
           int(pk['out_of_track'].sum())))
    return pk


def pred_fixture(ltpl, track, n, vel_kwargs):
    """objects that carry an explicit 'prediction' array (OLI:117-119; GLNT:180-189 blocks the edges under every
    prediction point, the LAST one decides the object's layer -- quirk q14): 0-4 points per object, some objects without
    the key in the same list."""
    from graphbasedlocaltrajectoryplanner_b200.scenarios import make_scenarios
    sc = make_scenarios(track, n, seed=5150, n_obj_min=1, n_obj_max=3)
    rng = np.random.default_rng(5151)
    kp = 4
    sc.pred = np.zeros((n, sc.obj.shape[1], kp, 2))
    sc.n_pred = np.full((n, sc.obj.shape[1]), -1, dtype=np.int32)
    for b in range(n):
        for k in range(int(sc.n_obj[b])):
            if rng.random() < 0.25:
                continue                                   # no 'prediction' key -> built-in 0.2 s point
            m = int(rng.integers(0, kp + 1))
            x, y, th, v, _ = sc.obj[b, k]
            drift = rng.uniform(-0.4, 0.4)
            for j in range(m):
                t = 0.3 * (j + 1)
                sc.pred[b, k, j] = [x - np.sin(th) * v * t + np.cos(th) * drift * t * 3.0,
                                    y + np.cos(th) * v * t + np.sin(th) * drift * t * 3.0]
            sc.n_pred[b, k] = m
    recs = [run_tick(ltpl, sc.pos[b], sc.heading[b], sc.vel[b], sc.object_list(b), vel_kwargs, full=True)
            for b in range(n)]
    pk = pack_ticks(recs)
    pk.update(sc_pos=sc.pos, sc_heading=sc.heading, sc_vel=sc.vel, sc_n_obj=sc.n_obj, sc_obj=sc.obj, sc_pred=sc.pred,
              sc_n_pred=sc.n_pred, ax_max_machines=vel_kwargs['ax_max_machines'])
    print("[pred] %d objects with explicit predictions (%d points); action paths %s" % (
        int((sc.n_pred >= 0).sum()), int(np.maximum(sc.n_pred, 0).sum()),
        {a: int((pk['path_len'][:, i] > 0).sum()) for i, a in enumerate(ACTIONS)}))
    return pk


class ScriptedClock(object):
    """stands in for the `time` module inside OnlineTrajectoryHandler (OTH:353-354, 395, 672): the calculation time the
    reference measures with the wall clock becomes an input of the fixture."""

    def __init__(self):
        self.t = 1000.0

    def time(self):
        return self.t


def advance_on_traj(traj, dt):
    """vehicle dummy: position / velocity after dt on a trajectory (s, x, y, psi, kappa, vx, ax), constant-acceleration
    step with the first row's values (cf. testing_tools/src/vdc_dummy.py)."""
    ds = max(traj[0, 5] * dt + 0.5 * traj[0, 6] * dt * dt, 0.0)
    s = traj[0, 0] + ds
    return (np.array([np.interp(s, traj[:, 0], traj[:, 1]), np.interp(s, traj[:, 0], traj[:, 2])]),
            float(np.interp(s, traj[:, 0], traj[:, 5])))


def multitick_fixture(graph_ltpl, ltpl, track, n_seq, n_ticks, vel_kwargs, lat=None, seed=31337, gg_drop=None,
                      em_select=None, bad_select=None, n_obj=(0, 2), zone_swap=None, s_max=None, hmax=40, s_min=0.0,
                      gg_fn=None):
    """closed-loop sequences through the unmodified reference with a scripted clock: per tick the inputs (clock step,
    selected action, object list, position / velocity estimate) and the outputs (node sequences, trajectories, ids).
    em_select=(k0, k1): the odd sequences execute the 'emergency' trajectory of ticks k0 .. k1 (OTH:307-309; code 4).
    bad_select=(k, ...): after those ticks the odd sequences name an action the tick did NOT return (OTH:393-407: no valid
    last solution; the vehicle dummy keeps driving on the first returned trajectory).
    zone_swap=k: from tick k on the sequences with a zone pass ANOTHER zone under a new id (the old one is flagged removed
    by ObjectListInterface.update_zone and emptied at once, BLOCK_N_LAYERS_WHEN_REMOVING_ZONE = 0; GLNT:43-99)."""
    import graph_ltpl.online_graph.src.OnlineTrajectoryHandler as oth_mod
    from graphbasedlocaltrajectoryplanner_b200.scenarios import make_scenarios
    clock = ScriptedClock()
    real_time = oth_mod.time
    oth_mod.time = clock
    try:
        sc = make_scenarios(track, n_seq, seed=seed, n_obj_min=n_obj[0], n_obj_max=n_obj[1], s_max=s_max, s_min=s_min)
        rng = np.random.default_rng(seed + 1)
        emerg = bool(vel_kwargs.get('incl_emerg_traj'))
        zones = [(make_zone(lat, rng, sc.pos[q]) if (lat is not None and q % 2 == 0) else None) for q in range(n_seq)]
        zmax = max([len(z[0]) for z in zones if z is not None] + [1])
        prefer = (("right", "left", "straight", "follow"), ("follow", "straight", "left", "right"),
                  ("left", "straight", "follow", "right"))
        pmax = 115
        out = dict(dt=np.zeros((n_seq, n_ticks)), sel=np.full((n_seq, n_ticks), -1, dtype=np.int32),
                   pos_est=np.zeros((n_seq, n_ticks, 2)), vel_est=np.zeros((n_seq, n_ticks)),
                   obj=np.zeros((n_seq, n_ticks, sc.obj.shape[1], 5)),
                   traj=np.zeros((n_seq, n_ticks, 4, pmax, 7)), traj_len=np.zeros((n_seq, n_ticks, 4), dtype=np.int32),
                   traj_id=np.full((n_seq, n_ticks, 4), -1, dtype=np.int32),
                   nodes=np.full((n_seq, n_ticks, 4, hmax, 2), -1, dtype=np.int32),
                   nodes_len=np.zeros((n_seq, n_ticks, 4), dtype=np.int32),
                   path_len=np.zeros((n_seq, n_ticks, 4), dtype=np.int32), n_done=np.zeros(n_seq, dtype=np.int32),
                   em_traj=np.zeros((n_seq, n_ticks, pmax, 7)), em_len=np.zeros((n_seq, n_ticks), dtype=np.int32),
                   zone_layers=np.full((n_seq, zmax), -1, dtype=np.int32),
                   zone_nodes=np.full((n_seq, zmax), -1, dtype=np.int32), gg_scale=np.ones((n_seq, n_ticks)))
        for q in range(n_seq):
            if zones[q] is not None:
                out['zone_layers'][q, :len(zones[q][0])] = zones[q][0]
                out['zone_nodes'][q, :len(zones[q][1])] = zones[q][1]
        if zone_swap is not None:
            out.update(zone_swap_tick=np.int32(zone_swap), zone2_layers=np.full((n_seq, 400), -1, dtype=np.int32),
                       zone2_nodes=np.full((n_seq, 400), -1, dtype=np.int32))
        for q in range(n_seq):
            if ltpl.set_startpos(pos_est=np.array(sc.pos[q]), heading_est=float(sc.heading[q]), vel_est=float(sc.vel[q])):
                continue
            oth = ltpl._Graph_LTPL__oth
            ltpl._Graph_LTPL__obj_zone = []
            ltpl._Graph_LTPL__obj_list_handler._ObjectListInterface__object_zones = []
            objs = sc.obj[q, :int(sc.n_obj[q])].copy()
            pos_est, vel_est, sel, traj_set = np.array(sc.pos[q]), float(sc.vel[q]), "straight", None
            drive = sel
            order = prefer[q % len(prefer)]
            for k in range(n_ticks):
                dt = float(rng.uniform(0.04, 0.16))
                clock.t += dt
                for j in range(objs.shape[0]):            # opponents keep heading and speed
                    objs[j, 0] -= np.sin(objs[j, 2]) * objs[j, 3] * dt
                    objs[j, 1] += np.cos(objs[j, 2]) * objs[j, 3] * dt
                ol = [{'id': j + 1, 'type': 'physical', 'X': float(o[0]), 'Y': float(o[1]), 'theta': float(o[2]),
                       'v': float(o[3]), 'length': float(o[4]), 'width': 2.5} for j, o in enumerate(objs)]
                if traj_set is not None:
                    pos_est, vel_est = advance_on_traj(traj_set[drive][0], dt)
                out['dt'][q, k], out['sel'][q, k] = dt, (4 if sel == 'emergency' else ACTIONS.index(sel))
                out['pos_est'][q, k], out['vel_est'][q, k] = pos_est, vel_est
                out['obj'][q, k, :objs.shape[0]] = objs
                bz = None if zones[q] is None else {'zone_%d' % q: zones[q]}
                if zone_swap is not None and zones[q] is not None and k >= zone_swap:
                    if k == zone_swap:
                        z2 = make_zone(lat, rng, pos_est)
                        out['zone2_layers'][q, :len(z2[0])] = z2[0]
                        out['zone2_nodes'][q, :len(z2[1])] = z2[1]
                    n2 = int((out['zone2_layers'][q] >= 0).sum())
                    bz = {'zone_%d_b' % q: [out['zone2_layers'][q, :n2].tolist(), out['zone2_nodes'][q, :n2].tolist(),
                                            np.zeros((2, 2)), np.zeros((2, 2))]}
                paths = ltpl.calc_paths(prev_action_id=sel, object_list=ol, blocked_zones=bz)
                nodes = oth._OnlineTrajectoryHandler__last_action_set_nodes
                for a, act in enumerate(ACTIONS):
                    if act in paths and len(paths[act]) and np.size(paths[act][0]):
                        out['path_len'][q, k, a] = paths[act][0].shape[0]
                        nd = [[-1 if v is None else int(v) for v in pair] for pair in nodes[act][0]]
                        out['nodes'][q, k, a, :len(nd)] = nd
                        out['nodes_len'][q, k, a] = len(nd)
                vk = dict(vel_kwargs)
                if gg_drop is not None and q % 2 == 1 and k >= gg_drop[0]:
                    vk['gg_scale'] = gg_drop[1]       # grip drops: profiles can no longer start at the planned velocity
                out['gg_scale'][q, k] = vk.get('gg_scale', 1.0)
                if gg_fn is not None:                 # location dependent friction along this tick's paths (OTH:649-666)
                    vk['local_gg'] = {a: [gg_fn(p[0][:, 0:2])] for a, p in paths.items()}
                traj_set, ids, _ = ltpl.calc_vel_profile(pos_est=pos_est, vel_est=vel_est, **vk)
                for a, act in enumerate(ACTIONS):
                    if act in traj_set and len(traj_set[act]):
                        t = traj_set[act][0]
                        out['traj'][q, k, a, :t.shape[0]] = t
                        out['traj_len'][q, k, a] = t.shape[0]
                        out['traj_id'][q, k, a] = ids[act]
                if emerg and 'emergency' in traj_set:
                    t = traj_set['emergency'][0]
                    out['em_traj'][q, k, :t.shape[0]] = t
                    out['em_len'][q, k] = t.shape[0]
                out['n_done'][q] = k + 1
                cand = [a for a in order if a in traj_set and len(traj_set[a])]
                if not cand:
                    break
                sel = cand[0]
                if (em_select is not None and q % 2 == 1 and em_select[0] <= k <= em_select[1]
                        and 'emergency' in traj_set):
                    sel = 'emergency'
                drive = sel
                if bad_select is not None and q % 2 == 1 and k in bad_select:
                    missing = [a for a in ("left", "right", "follow", "straight") if a not in traj_set]
                    if missing:
                        sel, drive = missing[0], cand[0]
        out.update(sc_pos=sc.pos, sc_heading=sc.heading, sc_vel=sc.vel, sc_n_obj=sc.n_obj,
                   ax_max_machines=vel_kwargs['ax_max_machines'])
        print("[multitick] %d sequences, %d ticks; selected actions %s" % (
            n_seq, int(out['n_done'].sum()), {a: int((out['sel'] == i).sum()) for i, a in enumerate(ACTIONS + ('emergency',))}))
        return out
    finally:
        oth_mod.time = real_time


VARIANTS = (
    # follow-mode controller with tan activation (CVPF:65-71), friction-ellipse exponent != 1 (tph.calc_ax_poss), other
    # vehicle mass / drag (LTPL:189-192), reduced gg scale, asymmetric gg, lower v_max, ego estimate != planned velocity
    dict(name="pdtan_exp15", controller_type="PDtan", veh=dict(veh_param_dyn_model_exp=1.5, veh_param_dragcoeff=0.9,
                                                               veh_param_mass=1200.0),
         vel=dict(vel_max=85.0, gg_scale=0.9, local_gg=(4.5, 5.5), safety_d=20.0), vel_est_offset=-2.0),
    dict(name="pd_exp20", controller_type=None, veh=dict(veh_param_dyn_model_exp=2.0, veh_param_dragcoeff=0.7,
                                                         veh_param_mass=900.0),
         vel=dict(vel_max=90.0, gg_scale=1.0, local_gg=(6.0, 4.0), safety_d=40.0), vel_est_offset=3.0),
)


def variants_fixture(graph_ltpl, track, n):
    """parameter variants of the velocity planner / follow controller, default lattice, first ticks."""
    from graphbasedlocaltrajectoryplanner_b200.scenarios import make_scenarios
    out = {}
    for vi, var in enumerate(VARIANTS):
        ltpl, _ = make_ltpl(graph_ltpl, "default", {}, controller_type=var["controller_type"], veh=var["veh"])
        sc = make_scenarios(track, n, seed=9000 + vi, n_obj_min=1, n_obj_max=3)
        vk = dict(var["vel"], ax_max_machines=ax_max_machines_table(), incl_emerg_traj=False)
        recs = [run_tick(ltpl, sc.pos[b], sc.heading[b], sc.vel[b], sc.object_list(b), vk, full=True,
                         vel_est=sc.vel[b] + var["vel_est_offset"]) for b in range(sc.size)]
        pk = pack_ticks(recs)
        pk.update(sc_pos=sc.pos, sc_heading=sc.heading, sc_vel=sc.vel, sc_n_obj=sc.n_obj, sc_obj=sc.obj)
        for k, v in pk.items():
            out["%s__%s" % (var["name"], k)] = v
        acts = {a: int((pk['traj_len'][:, i] > 0).sum()) for i, a in enumerate(ACTIONS)}
        print("[variant %s] trajectories %s" % (var["name"], acts))
    out["ax_max_machines"] = ax_max_machines_table()
    return out


SEED86420 = (("default", {}, 48, 0, 3), ("l216", {"lat_resolution": 1.0, "lon_straight_step": 12.0}, 24, 1, 3))
SEED86420_STRIDE = 4


def seed86420_fixture(graph_ltpl, track, tag, overrides, n, omin, omax, vel_kwargs):
    """first ticks of the seed-86420 scenarios of tests/test_against_reference.py: the arrays H.compare_record reads
    (no spline coefficients) and the scenario inputs.  To keep the file small, paths and trajectories keep every
    SEED86420_STRIDE-th point (point_stride) in float32 (relative rounding 6e-8, the comparison tolerance is 1e-4)."""
    from graphbasedlocaltrajectoryplanner_b200.scenarios import make_scenarios
    ltpl, _ = make_ltpl(graph_ltpl, tag, overrides)
    sc = make_scenarios(track, n, seed=86420, n_obj_min=omin, n_obj_max=omax)
    recs = [run_tick(ltpl, sc.pos[b], sc.heading[b], sc.vel[b], sc.object_list(b), vel_kwargs, full=True)
            for b in range(sc.size)]
    pk = pack_ticks(recs)
    del pk['coeff'], pk['coeff_len']
    for k in ('path', 'traj'):
        pk[k] = pk[k][:, :, ::SEED86420_STRIDE].astype(np.float32)
    payload = {('full_' + k): v for k, v in pk.items()}
    payload['point_stride'] = np.int32(SEED86420_STRIDE)
    payload.update(sc_pos=sc.pos, sc_heading=sc.heading, sc_vel=sc.vel, sc_n_obj=sc.n_obj, sc_obj=sc.obj,
                   ax_max_machines=vel_kwargs['ax_max_machines'], overrides=np.array(repr(sorted(overrides.items()))))
    return payload


def lattice_fixture(graph_ltpl, ltpl, n_edge_samples=300, seed=7):
    """compact description of the reference-built GraphBase (validates the product's lattice builder)."""
    from graphbasedlocaltrajectoryplanner_b200.lattice import Lattice
    gb = ltpl._Graph_LTPL__graph_base
    lat = Lattice.from_graph_base(gb)
    rng = np.random.default_rng(seed)
    pick = np.sort(rng.choice(lat.num_edges, size=min(n_edge_samples, lat.num_edges), replace=False))
    samp = []
    for e in pick:
        a0, a1 = lat.samp_off[e], lat.samp_off[e + 1]
        samp.append(np.column_stack((lat.samp_x[a0:a1], lat.samp_y[a0:a1], lat.samp_psi[a0:a1],
                                     lat.samp_kappa[a0:a1], lat.samp_el[a0:a1])))
    fx = dict(num_layers=lat.num_layers, closed=lat.closed, node_off=lat.node_off, raceline_index=lat.raceline_index,
              s_raceline=lat.s_raceline, vel_raceline=lat.vel_raceline,
              node_xy_psi=np.column_stack((lat.node_x, lat.node_y, lat.node_psi)),
              edge_layer_off=lat.edge_layer_off, edge_src=lat.edge_src.astype(np.int16),
              edge_dst=lat.edge_dst.astype(np.int16), edge_cost=lat.edge_cost, edge_len=lat.edge_len,
              samp_off=lat.samp_off, pick=pick.astype(np.int32), pick_samples=np.concatenate(samp, axis=0),
              checksums=np.array([lat.samp_x.sum(), lat.samp_y.sum(), lat.samp_psi.sum(), lat.samp_kappa.sum(),
                                  lat.samp_el.sum(), np.abs(lat.samp_kappa).sum()]))
    return fx, lat


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--quick', action='store_true', help='default lattice only')
    ap.add_argument('--n-default', type=int, default=96)
    ap.add_argument('--n-other', type=int, default=32)
    ap.add_argument('--ext-only', action='store_true', help='only the zone / emergency fixture (default lattice)')
    ap.add_argument('--n-ext', type=int, default=64)
    ap.add_argument('--multitick-only', action='store_true', help='only the closed-loop (stateful) fixture')
    ap.add_argument('--emsel-only', action='store_true', help="only the closed-loop fixture executing 'emergency'")
    ap.add_argument('--mt-l216-only', action='store_true', help='only the closed-loop fixture on the ~200 x 11 lattice')
    ap.add_argument('--mt-l430-only', action='store_true', help='only the closed-loop fixture on the 400 x 21 lattice')
    ap.add_argument('--mt-variant-only', action='store_true', help='only the closed-loop fixture with the PDtan variant')
    ap.add_argument('--mt-open-only', action='store_true', help='only the closed-loop fixture on the open track')
    ap.add_argument('--zswap-only', action='store_true', help='only the closed-loop fixture with a zone replaced')
    ap.add_argument('--invalid-only', action='store_true', help='only the closed-loop fixture naming actions not returned')
    ap.add_argument('--pred-only', action='store_true', help="only the explicit-'prediction' fixture (default lattice)")
    ap.add_argument('--only', default=None, help='only this lattice configuration of the main loop (e.g. layers14)')
    ap.add_argument('--open-only', action='store_true', help='only the open-track fixture')
    ap.add_argument('--n-open', type=int, default=64)
    ap.add_argument('--variants-only', action='store_true', help='only the parameter-variant fixture')
    ap.add_argument('--n-variant', type=int, default=24)
    ap.add_argument('--ggpp-only', action='store_true', help='only the location dependent local_gg fixtures')
    ap.add_argument('--seed86420-only', action='store_true', help='only the fixtures of tests/test_against_reference.py')
    args = ap.parse_args()

    graph_ltpl = load_reference()
    from graphbasedlocaltrajectoryplanner_b200.scenarios import Track, make_scenarios, DEFAULT_SEED
    os.makedirs(GOLDEN, exist_ok=True)
    track = Track(REF + "/inputs/traj_ltpl_cl/traj_ltpl_cl_monteblanco.csv")
    vel_kwargs = dict(vel_max=100.0, gg_scale=1.0, local_gg=(5.0, 5.0), ax_max_machines=ax_max_machines_table(),
                      safety_d=30.0, incl_emerg_traj=False)

    if args.seed86420_only:
        for tag, overrides, n, omin, omax in SEED86420:
            np.savez_compressed(os.path.join(GOLDEN, 'ticks_seed86420_%s.npz' % tag),
                                **seed86420_fixture(graph_ltpl, track, tag, overrides, n, omin, omax, vel_kwargs))
        return
    if args.ggpp_only:
        # location dependent friction: local_gg = {action: [ndarray(P, 2)]} (OTH:649-666, VPFB:194-227), emergency
        # trajectory on (its brake profile takes the raw local_gg of the base trajectory, OTH:1030); closed loop with a grip
        # drop on the odd sequences (the brake on the backup plan takes the LAST tick's local_gg, OTH:970-975)
        sys.path.insert(0, REPO)
        from tests.helpers import local_gg_field
        ltpl, _ = make_ltpl(graph_ltpl, "default", {})
        vk = dict(vel_kwargs, incl_emerg_traj=True)
        sc = make_scenarios(track, 32, seed=2468, n_obj_min=0, n_obj_max=3)
        recs = [run_tick(ltpl, sc.pos[b], sc.heading[b], sc.vel[b], sc.object_list(b), vk, full=True, gg_fn=local_gg_field)
                for b in range(sc.size)]
        pk = pack_ticks(recs)
        n, pmax = sc.size, pk['path'].shape[2]
        em, em_len, em_id = np.zeros((n, pmax, 7)), np.zeros(n, dtype=np.int32), np.full(n, -1, dtype=np.int32)
        for i, r in enumerate(recs):
            if 'traj' in r and 'emergency' in r['traj']:
                t = r['traj']['emergency'][0]
                em[i, :t.shape[0]] = t
                em_len[i] = t.shape[0]
                em_id[i] = r['ids']['emergency']
        payload = {('full_' + k): v for k, v in pk.items()}
        payload.update(em_traj=em, em_len=em_len, em_id=em_id, sc_pos=sc.pos, sc_heading=sc.heading, sc_vel=sc.vel, sc_n_obj=sc.n_obj,
                       sc_obj=sc.obj, ax_max_machines=vel_kwargs['ax_max_machines'], overrides=np.array(repr([])))
        np.savez_compressed(os.path.join(GOLDEN, 'ticks_ggpp_default.npz'), **payload)
        print("[ggpp] action paths %s; emergency %d" % (
            {a: int((pk['path_len'][:, i] > 0).sum()) for i, a in enumerate(ACTIONS)}, int((em_len > 0).sum())))
        np.savez_compressed(os.path.join(GOLDEN, 'ticks_multitick_ggpp_default.npz'),
                            **multitick_fixture(graph_ltpl, ltpl, track, 12, 8, vk, seed=1357, gg_drop=(3, 0.45),
                                                n_obj=(0, 3), gg_fn=local_gg_field))
        return
    if args.open_only or args.mt_open_only or not (args.quick or args.variants_only or args.ext_only or args.only or args.pred_only
                              or args.multitick_only or args.emsel_only or args.invalid_only or args.mt_l216_only
                              or args.zswap_only or args.mt_l430_only or args.mt_variant_only):
        # open (unclosed) track: planning range clamp at the last layer, reduced horizons, v_end = 0 (GLNT:112-124, quirk
        # q7; MOPG:203-243; OTH:846-859)
        open_csv = os.path.join(REPO, "inputs", "traj_ltpl_cl", "traj_ltpl_cl_monteblanco_open.csv")
        write_open_track_csv(open_csv)
        ltpl, _ = make_ltpl(graph_ltpl, "open", {}, csv=open_csv)
        fx, lat = lattice_fixture(graph_ltpl, ltpl)
        np.savez_compressed(os.path.join(GOLDEN, 'lattice_open.npz'), **fx)
        print("[open] lattice: %s" % lat.summary())
        tr_open = Track(open_csv)
        # closed loop on the open track: the vehicle runs towards the end of the race line (reduced horizons, v_end = 0)
        np.savez_compressed(os.path.join(GOLDEN, 'ticks_multitick_open.npz'),
                            **multitick_fixture(graph_ltpl, ltpl, tr_open, 16, 8, vel_kwargs, seed=1212,
                                                s_max=tr_open.length - 8.0))
        # ... and starting on the last 150 m: trajectories shrink tick by tick until nothing is left to plan
        np.savez_compressed(os.path.join(GOLDEN, 'ticks_multitick_openend.npz'),
                            **multitick_fixture(graph_ltpl, ltpl, tr_open, 12, 10, vel_kwargs, seed=1313,
                                                s_max=tr_open.length - 15.0, s_min=tr_open.length - 150.0))
        if args.mt_open_only:
            return
        sc = make_scenarios(tr_open, args.n_open, seed=DEFAULT_SEED + 99, n_obj_min=0, n_obj_max=3,
                            s_max=tr_open.length - 8.0)
        recs = [run_tick(ltpl, sc.pos[b], sc.heading[b], sc.vel[b], sc.object_list(b), vel_kwargs, full=True)
                for b in range(sc.size)]
        pk = pack_ticks(recs)
        payload = {('full_' + k): v for k, v in pk.items()}
        payload.update(sc_pos=sc.pos, sc_heading=sc.heading, sc_vel=sc.vel, sc_n_obj=sc.n_obj, sc_obj=sc.obj,
                       ax_max_machines=vel_kwargs['ax_max_machines'], overrides=np.array(repr([])))
        np.savez_compressed(os.path.join(GOLDEN, 'ticks_open.npz'), **payload)
        print("[open] action paths %s; reduced %d; out of track %d" % (
            {a: int((pk['path_len'][:, i] > 0).sum()) for i, a in enumerate(ACTIONS)}, int(pk['red_len'].sum()),
            int(pk['out_of_track'].sum())))
        if args.open_only:
            return
    if args.mt_variant_only or not (args.quick or args.variants_only or args.ext_only or args.only or args.pred_only
                                    or args.multitick_only or args.emsel_only or args.invalid_only
                                    or args.mt_l216_only or args.zswap_only or args.mt_l430_only or args.open_only):
        # closed loop with the first parameter variant (PDtan follow controller, friction-ellipse exponent 1.5, other
        # mass / drag, gg scale 0.9, asymmetric gg, v_max 85)
        var = VARIANTS[0]
        ltpl_v, _ = make_ltpl(graph_ltpl, "default", {}, controller_type=var["controller_type"], veh=var["veh"])
        np.savez_compressed(os.path.join(GOLDEN, 'ticks_multitick_pdtan_default.npz'),
                            **multitick_fixture(graph_ltpl, ltpl_v, track, 12, 8,
                                                dict(var["vel"], ax_max_machines=ax_max_machines_table(),
                                                     incl_emerg_traj=False), seed=3131, n_obj=(1, 3)))
        if args.mt_variant_only:
            return
    if args.variants_only:
        np.savez_compressed(os.path.join(GOLDEN, 'ticks_variants_default.npz'),
                            **variants_fixture(graph_ltpl, track, args.n_variant))
        return
    configs = [("default", {}, args.n_default, 0, 3)]
    if not args.quick:
        configs.append(("l216", {"lat_resolution": 1.0, "lon_straight_step": 12.0}, args.n_other, 1, 3))
        configs.append(("l430", {"lon_curve_step": 6.0, "lon_straight_step": 6.0, "lat_resolution": 0.5},
                        args.n_other, 5, 5))
        # planning horizon as a fixed number of layers (GLNT:126-136)
        configs.append(("layers14", {"plan_horizon_mode": "layers", "min_plan_horizon": 14}, args.n_other, 0, 3))
    if args.mt_l216_only:
        args.only = "l216"
    if args.mt_l430_only:
        args.only = "l430"
    if args.only:
        configs = [c for c in configs if c[0] == args.only]

    for tag, overrides, n, omin, omax in configs:
        ltpl, path_dict = make_ltpl(graph_ltpl, tag, overrides)
        fx, lat = lattice_fixture(graph_ltpl, ltpl)
        if tag == "l216":
            # BASELINE's ~200 x 11 lattice: node lists of more than 32 entries, 1-3 objects, emergency trajectory on
            np.savez_compressed(os.path.join(GOLDEN, 'ticks_multitick_l216.npz'),
                                **multitick_fixture(graph_ltpl, ltpl, track, 12, 8,
                                                    dict(vel_kwargs, incl_emerg_traj=True), seed=8181, n_obj=(1, 3)))
            if args.mt_l216_only:
                return
        if tag == "l430":
            # config 4: 430 layers x 13-25 nodes, 5 objects per scenario
            np.savez_compressed(os.path.join(GOLDEN, 'ticks_multitick_l430.npz'),
                                **multitick_fixture(graph_ltpl, ltpl, track, 8, 6, vel_kwargs, seed=4343, n_obj=(5, 5),
                                                    hmax=80))
            if args.mt_l430_only:
                return
        if tag == "default" and (args.zswap_only or args.multitick_only or not (args.pred_only or args.ext_only)):
            # the even sequences replace their zone by another one at tick 4
            np.savez_compressed(os.path.join(GOLDEN, 'ticks_multitick_zswap_default.npz'),
                                **multitick_fixture(graph_ltpl, ltpl, track, 12, 8, vel_kwargs, lat=lat, seed=9191,
                                                    zone_swap=4))
            if args.zswap_only:
                return
        if tag == "default" and (args.invalid_only or args.multitick_only or not (args.pred_only or args.ext_only)):
            # the odd sequences name an action that was not returned after ticks 2 and 5 (OTH:393-407)
            np.savez_compressed(os.path.join(GOLDEN, 'ticks_multitick_invalid_default.npz'),
                                **multitick_fixture(graph_ltpl, ltpl, track, 12, 8, vel_kwargs, seed=7171,
                                                    bad_select=(2, 5)))
            if args.invalid_only:
                return
        if tag == "default" and (args.emsel_only or args.multitick_only or not (args.pred_only or args.ext_only)):
            # the odd sequences execute the emergency trajectory of ticks 2 .. 4 (OTH:307-309, get_ref_idx on it)
            np.savez_compressed(os.path.join(GOLDEN, 'ticks_multitick_emsel_default.npz'),
                                **multitick_fixture(graph_ltpl, ltpl, track, 12, 8,
                                                    dict(vel_kwargs, incl_emerg_traj=True), seed=6161, em_select=(2, 4)))
            if args.emsel_only:
                return
            np.savez_compressed(os.path.join(GOLDEN, 'ticks_multitick_default.npz'),
                                **multitick_fixture(graph_ltpl, ltpl, track, 16, 10, vel_kwargs))
            # the same with a blocked zone on every second sequence and the emergency trajectory switched on
            np.savez_compressed(os.path.join(GOLDEN, 'ticks_multitick_ext_default.npz'),
                                **multitick_fixture(graph_ltpl, ltpl, track, 12, 8,
                                                    dict(vel_kwargs, incl_emerg_traj=True), lat=lat, seed=4141))
            # grip drop on every second sequence from tick 3 on: recursive infeasibility -> brake on the backup plan
            # (OTH:950-1006)
            np.savez_compressed(os.path.join(GOLDEN, 'ticks_multitick_backup_default.npz'),
                                **multitick_fixture(graph_ltpl, ltpl, track, 12, 7, vel_kwargs, seed=5151,
                                                    gg_drop=(3, 0.45)))
            if args.multitick_only:
                return
        if tag == "default":
            np.savez_compressed(os.path.join(GOLDEN, 'ticks_pred_default.npz'),
                                **pred_fixture(ltpl, track, args.n_other, vel_kwargs))
            if args.pred_only:
                return
            np.savez_compressed(os.path.join(GOLDEN, 'ticks_ext_default.npz'),
                                **ext_fixture(ltpl, lat, track, args.n_ext, vel_kwargs))
            if args.ext_only:
                return
        np.savez_compressed(os.path.join(GOLDEN, 'lattice_%s.npz' % tag), **fx)
        print("[%s] lattice: %s" % (tag, lat.summary()))

        sc = make_scenarios(track, n, seed=DEFAULT_SEED + len(tag), n_obj_min=omin, n_obj_max=omax)
        recs, recs_full = [], []
        t0 = time.time()
        for b in range(sc.size):
            ol = sc.object_list(b)
            recs.append(run_tick(ltpl, sc.pos[b], sc.heading[b], sc.vel[b], ol, vel_kwargs, full=False))
            recs_full.append(run_tick(ltpl, sc.pos[b], sc.heading[b], sc.vel[b], ol, vel_kwargs, full=True))
        print("[%s] %d reference ticks (x2) in %.1f s" % (tag, sc.size, time.time() - t0))
        full = pack_ticks(recs_full)
        cut = pack_ticks(recs, pmax=full['path'].shape[2])
        assert np.array_equal(cut['traj_len'], np.minimum(full['traj_len'], 115))
        payload = {('full_' + k): v for k, v in full.items()}
        payload['cut_traj_len'] = cut['traj_len']
        payload.update(sc_pos=sc.pos, sc_heading=sc.heading, sc_vel=sc.vel, sc_n_obj=sc.n_obj, sc_obj=sc.obj,
                       ax_max_machines=vel_kwargs['ax_max_machines'],
                       overrides=np.array(repr(sorted(overrides.items()))))
        np.savez_compressed(os.path.join(GOLDEN, 'ticks_%s.npz' % tag), **payload)
        acts = {a: int((full['path_len'][:, i] > 0).sum()) for i, a in enumerate(ACTIONS)}
        print("[%s] action paths: %s; trajectories: %s; reduced: %d" %
              (tag, acts, {a: int((full['traj_len'][:, i] > 0).sum()) for i, a in enumerate(ACTIONS)},
               int(full['red_len'].sum())))

        if tag == "default":
            # SURVEY 8(d) config 1: main_min_example.py start pose + the static dummy object of objectlist_dummy.py:175
            refline = graph_ltpl.imp_global_traj.src.import_globtraj_csv.import_globtraj_csv(
                import_path=path_dict['globtraj_input_path'])[0]
            pos = refline[0, :]
            heading = float(np.arctan2(np.diff(refline[0:2, 1]), np.diff(refline[0:2, 0]))[0] - np.pi / 2)
            obj = {'id': 1, 'type': 'physical', 'X': 127, 'Y': 82, 'theta': 0.0, 'length': 5.0, 'width': 2.5,
                   'v': 0.0}
            api_default = dict()  # calc_vel_profile API defaults (LTPL:344-352)
            r1 = [run_tick(ltpl, pos, heading, 0.0, [obj], api_default, full=True)]
            # variant: ego ~180 m before the static object so that follow / left / right are exercised
            p2, h2, _ = track.raceline_pose(np.array([1300.0]))
            r2 = [run_tick(ltpl, p2[0], h2[0], 20.0, [obj], api_default, full=True)]
            pk = pack_ticks(r1 + r2)
            pk.update(sc_pos=np.vstack((pos, p2[0])), sc_heading=np.array([heading, h2[0]]),
                      sc_vel=np.array([0.0, 20.0]), obj=np.array([127.0, 82.0, 0.0, 0.0, 5.0]))
            np.savez_compressed(os.path.join(GOLDEN, 'config1_min_example.npz'), **pk)
            print("[config1] actions:", {a: pk['path_len'][:, i].tolist() for i, a in enumerate(ACTIONS)})
    if not args.quick and not args.only:
        np.savez_compressed(os.path.join(GOLDEN, 'ticks_variants_default.npz'),
                            **variants_fixture(graph_ltpl, track, args.n_variant))


if __name__ == "__main__":
    main()
