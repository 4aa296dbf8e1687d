"""The drop-in facade driven like the reference's own example loops (main_min_example.py:56-107, main_std_example.py:99-135):
`import graph_ltpl` swapped for the B200 package, nothing else -- incl. visual_mode=True, the per-tick visual() / log()
calls, a growing object list inside one session and an action the last tick did not return."""
import numpy as np
import pytest

from tests import helpers as H

pytestmark = pytest.mark.gpu


class _Clock(object):
    def __init__(self):
        self.t = 100.0

    def __call__(self):
        return self.t


def _path_dict(tmp_path):
    # main_min_example.py:42-46 passes exactly these four entries (log_to_file=False needs no log paths, LTPL:62-68)
    return {'globtraj_input_path': H.TRACK_CSV, 'graph_store_path': str(tmp_path / "lattice_default.npz"),
            'ltpl_offline_param_path': H.OFFLINE_INI, 'ltpl_online_param_path': H.ONLINE_INI}


def test_min_example_loop_runs_unchanged(tmp_path):
    """body of main_min_example.py:52-107 with the import swapped: graph_init, set_startpos at the first reference-line
    point, then the online loop (brute-force action choice, calc_paths, vehicle dummy, calc_vel_profile, visual)."""
    from graphbasedlocaltrajectoryplanner_b200.Graph_LTPL import Graph_LTPL
    from graphbasedlocaltrajectoryplanner_b200.lattice import import_globtraj_csv
    from oracle.gen_golden import advance_on_traj   # stands in for testing_tools/src/vdc_dummy.py (test infrastructure)
    ltpl_obj = Graph_LTPL(path_dict=_path_dict(tmp_path), visual_mode=True, log_to_file=False)
    ltpl_obj.graph_init()
    refline = import_globtraj_csv(H.TRACK_CSV)["refline"]
    pos_est = refline[0, :]
    heading_est = np.arctan2(np.diff(refline[0:2, 1]), np.diff(refline[0:2, 0])) - np.pi / 2   # an array, as there
    vel_est = 0.0
    assert ltpl_obj.set_startpos(pos_est=pos_est, heading_est=heading_est) is False
    clk = _Clock()
    ltpl_obj.clock = clk
    traj_set = {'straight': None}
    s_driven = 0.0
    for it in range(25):
        for sel_action in ["right", "left", "straight", "follow"]:
            if sel_action in traj_set.keys():
                break
        ltpl_obj.calc_paths(prev_action_id=sel_action, object_list=[])
        clk.t += 0.08
        if traj_set[sel_action] is not None:
            new_pos, vel_est = advance_on_traj(traj_set[sel_action][0], 0.08)
            s_driven += float(np.hypot(*(new_pos - pos_est)))
            pos_est = new_pos
        traj_set = ltpl_obj.calc_vel_profile(pos_est=pos_est, vel_est=vel_est)[0]
        ltpl_obj.visual()
        ltpl_obj.log()
        assert traj_set and "straight" in traj_set, "tick %d returned %s" % (it, sorted(traj_set))
        t = traj_set["straight"][0]
        assert t.shape[1] == 7 and 2 < t.shape[0] <= 115 and np.all(np.isfinite(t)) and np.all(np.diff(t[:, 0]) > 0)
    assert s_driven > 0.0 and t[-1, 5] > t[0, 5] + 5.0   # the dummy moved; the plans accelerate away from standstill


def test_session_with_growing_object_list_and_unknown_action(tmp_path):
    """one stateful session through the facade against the session oracle (pinned on the reference): the object list
    grows from 0 to 3 entries between ticks (the scenario input buffers are re-created, the device memory must
    survive), and one tick names an action the last tick did not return (OTH:393-407)."""
    from graphbasedlocaltrajectoryplanner_b200.Graph_LTPL import Graph_LTPL
    from graphbasedlocaltrajectoryplanner_b200.scenarios import Track, make_scenarios
    from oracle.gen_golden import advance_on_traj
    from oracle.ltpl_oracle import OracleLTPL
    from oracle.ltpl_session import OracleSession
    g = H.golden("ticks_multitick_default.npz")
    vel = dict(vel_max=100.0, gg_scale=1.0, local_gg=(5.0, 5.0), ax_max_machines=g["ax_max_machines"], safety_d=30.0)
    ltpl = Graph_LTPL(path_dict=_path_dict(tmp_path), visual_mode=False, log_to_file=False, device="cuda:0")
    ltpl.graph_init()
    lat = H.lattice_for("default")
    sc = make_scenarios(Track(H.TRACK_CSV), 6, seed=4711, n_obj_min=3, n_obj_max=3)
    compared = 0
    for q in range(sc.size):
        clk_a, clk_b = _Clock(), _Clock()
        ltpl.clock = clk_a
        ses = OracleSession(OracleLTPL(lat), clock=clk_b)
        if ltpl.set_startpos(pos_est=sc.pos[q], heading_est=sc.heading[q], vel_est=sc.vel[q]):
            continue
        assert ses.set_startpos(sc.pos[q], sc.heading[q], sc.vel[q]) is False
        objs = sc.obj[q].copy()
        pos_est, vel_est, sel = sc.pos[q].copy(), float(sc.vel[q]), "straight"
        last = None
        for k in range(7):
            dt = 0.06 + 0.01 * k
            clk_a.t += dt
            clk_b.t += dt
            objs[:, 0] -= np.sin(objs[:, 2]) * objs[:, 3] * dt
            objs[:, 1] += np.cos(objs[:, 2]) * objs[:, 3] * dt
            n_obj = min(k, 3)                                   # 0, 1, 2, 3, 3, ... objects
            ol = [{'id': j + 1, 'type': 'physical', 'X': float(o[0]), 'Y': float(o[1]), 'theta': float(o[2]),
                   'v': float(o[3]), 'length': float(o[4]), 'width': 2.5} for j, o in enumerate(objs[:n_obj])]
            if last is not None:
                pos_est, vel_est = advance_on_traj(last, dt)
            name = sel
            if k == 4:                                          # an action tick 3 did not return (if there is one)
                missing = [a for a in ("left", "right", "follow", "straight") if a not in have]
                name = missing[0] if missing else sel
            ctx = "sequence %d tick %d (%d objects, action %s)" % (q, k, n_obj, name)
            paths = ltpl.calc_paths(prev_action_id=name, object_list=ol)
            want_paths = ses.calc_paths(name, ol)
            assert sorted(paths) == sorted(want_paths), ctx + ": paths %s vs %s" % (sorted(paths), sorted(want_paths))
            traj, ids, _ = ltpl.calc_vel_profile(pos_est=pos_est, vel_est=vel_est, **vel)
            want, _ = ses.calc_vel_profile(pos_est, vel_est, **vel)
            assert sorted(traj) == sorted(want), ctx + ": trajectories %s vs %s" % (sorted(traj), sorted(want))
            for act in want:
                if ses.tie.get(act):
                    continue
                H.assert_close("traj[%s]" % act, traj[act][0], want[act][0][:115],
                               ("s", "x", "y", "psi", "kappa", "vx", "ax"), ctx)
                compared += 1
            have = sorted(traj)
            if not have:
                break
            sel = [a for a in ("follow", "straight", "left", "right") if a in traj][0]
            last = traj[sel][0].astype(np.float64)
    assert compared > 25
