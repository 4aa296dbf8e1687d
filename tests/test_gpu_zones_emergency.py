"""blocked zones (GLNT:43-99) and the emergency trajectory (OTH:1027-1034) through the C-ABI, against the golden vectors
produced by the unmodified reference (tests/golden/ticks_ext_default.npz) and against the oracle on seeded scenarios."""
import numpy as np
import pytest

from tests import helpers as H

pytestmark = pytest.mark.gpu


def _planner(g):
    from graphbasedlocaltrajectoryplanner_b200.planner import BatchPlanner
    pl = BatchPlanner(H.lattice_for("default"), device="cuda:0")
    pl.set_subbatches(3)   # zones, emergency rows and prediction arrays across three scenario windows
    pl.set_vel_params(vel_max=100.0, gg_scale=1.0, local_gg=(5.0, 5.0), ax_max_machines=g["ax_max_machines"],
                      safety_d=30.0, incl_emerg_traj=True)
    return pl


def _golden_record(rec, g, b):
    H.compare_record(rec, g, b, prefix="", ctx="ext gpu")
    n = int(g["em_len"][b])
    has = "emergency" in rec.get("traj", {})
    assert has == (n > 0), "scenario %d: emergency present=%s, golden rows %d" % (b, has, n)
    if has:
        ne = min(n, 115)
        assert rec["traj"]["emergency"][0].shape == (ne, 7)
        assert int(rec["ids"]["emergency"]) % 10 == int(g["em_id"][b]) % 10
        H.assert_close("traj[emergency]", rec["traj"]["emergency"][0], g["em_traj"][b, :ne],
                       ("s", "x", "y", "psi", "kappa", "vx", "ax"), "ext gpu scenario %d" % b, w_rel=H.W_REL_BRAKE)


def test_zones_and_emergency_match_reference_golden():
    from graphbasedlocaltrajectoryplanner_b200.scenarios import ScenarioBatch
    g = H.golden("ticks_ext_default.npz")
    n = g["sc_pos"].shape[0]
    ols = [H.object_list(g, b) for b in range(n)]
    sc = ScenarioBatch.from_object_lists(g["sc_pos"], g["sc_heading"], g["sc_vel"], ols, k_max=3,
                                         blocked_zones=[H.zone_of(g, b) for b in range(n)])
    assert sc.zones is not None and int((sc.zone_sel >= 0).sum()) == int((g["zone_layers"][:, 0] >= 0).sum())
    pl = _planner(g)
    pl.stage_scenarios(sc)
    pl.upload()
    pl.set_startpos()
    pl.tick()
    recs = pl.records()
    for b in range(n):
        _golden_record(recs[b], g, b)


def test_zones_and_emergency_match_oracle_seeded():
    """larger seeded batch incl. scenarios that share a zone; zone-free scenarios in the same batch use the follow table."""
    from oracle.ltpl_oracle import OracleLTPL
    from oracle.gen_golden import make_zone
    from graphbasedlocaltrajectoryplanner_b200.scenarios import Track, make_scenarios
    g = H.golden("ticks_ext_default.npz")
    lat = H.lattice_for("default")
    sc = make_scenarios(Track(H.TRACK_CSV), 192, seed=4711, n_obj_min=0, n_obj_max=3)
    rng = np.random.default_rng(4712)
    zones = []
    for b in range(sc.size):
        if b % 3 == 2:
            zones.append(None)
        elif b % 3 == 1 and zones[b - 1] is not None:
            zones.append(zones[b - 1])              # same zone object as the previous scenario
        else:
            zones.append({"z%d" % b: make_zone(lat, rng, sc.pos[b])})
    sc.set_zones(zones)
    assert len(sc.zones) < int((sc.zone_sel >= 0).sum())
    pl = _planner(g)
    pl.stage_scenarios(sc)
    pl.upload()
    pl.set_startpos()
    pl.tick()
    recs = pl.records()
    orc = OracleLTPL(lat)
    vk = dict(vel_max=100.0, gg_scale=1.0, local_gg=(5.0, 5.0), ax_max_machines=g["ax_max_machines"], safety_d=30.0,
              incl_emerg_traj=True)
    n_em = 0
    for b in range(sc.size):
        want = orc.tick(sc.pos[b], sc.heading[b], sc.vel[b], sc.object_list(b), vk, blocked_zones=zones[b])
        got = recs[b]
        em_g = got.get("traj", {}).pop("emergency", None) if not got["out_of_track"] else None
        id_g = got.get("ids", {}).pop("emergency", None) if not got["out_of_track"] else None
        em_w = want.get("traj", {}).pop("emergency", None) if not want["out_of_track"] else None
        if not want["out_of_track"]:
            want["traj_full"].pop("emergency", None)
            id_w = want["ids"].pop("emergency", None)
        H.compare_records(got, want, ctx="zones seeded %d" % b)
        assert (em_g is None) == (em_w is None), "scenario %d emergency presence" % b
        if em_w is not None:
            n_em += 1
            assert id_g % 10 == id_w % 10
            H.assert_close("traj[emergency]", em_g[0], em_w[0], ("s", "x", "y", "psi", "kappa", "vx", "ax"),
                           "zones seeded %d" % b, w_rel=H.W_REL_BRAKE)
    assert n_em > sc.size // 2


def test_facade_blocked_zones_and_emergency(tmp_path):
    from graphbasedlocaltrajectoryplanner_b200.Graph_LTPL import Graph_LTPL
    g = H.golden("ticks_ext_default.npz")
    pd = {'globtraj_input_path': H.TRACK_CSV, 'graph_store_path': str(tmp_path / "lattice_default.npz"),
          'ltpl_offline_param_path': H.OFFLINE_INI, 'ltpl_online_param_path': H.ONLINE_INI}
    ltpl = Graph_LTPL(path_dict=pd, visual_mode=False, log_to_file=False, device="cuda:0")
    ltpl.graph_init()
    done = 0
    for b in range(g["sc_pos"].shape[0]):
        if H.zone_of(g, b) is None or int(g["em_len"][b]) == 0:
            continue
        ltpl.set_startpos(pos_est=g["sc_pos"][b], heading_est=g["sc_heading"][b], vel_est=g["sc_vel"][b])
        paths = ltpl.calc_paths(prev_action_id="straight", object_list=H.object_list(g, b),
                                blocked_zones=H.zone_of(g, b))
        traj, ids, _ = ltpl.calc_vel_profile(pos_est=g["sc_pos"][b], vel_est=float(g["sc_vel"][b]), vel_max=100.0,
                                             gg_scale=1.0, local_gg=(5.0, 5.0), ax_max_machines=g["ax_max_machines"],
                                             safety_d=30.0, incl_emerg_traj=True)
        for a, act in enumerate(H.ACTIONS):
            assert (act in paths) == (int(g["path_len"][b, a]) > 0)
        assert "emergency" in traj and list(traj.keys())[-1] == "emergency"
        ne = min(int(g["em_len"][b]), 115)
        H.assert_close("traj[emergency]", traj["emergency"][0], g["em_traj"][b, :ne],
                       ("s", "x", "y", "psi", "kappa", "vx", "ax"), "facade %d" % b, w_rel=H.W_REL_BRAKE)
        done += 1
        if done == 4:
            break
    assert done == 4


def test_unpack_batch_matches_records():
    """Graph_LTPL.unpack_batch (views of the pinned host result) against BatchPlanner.records() incl. 'emergency'."""
    from graphbasedlocaltrajectoryplanner_b200.Graph_LTPL import Graph_LTPL
    from graphbasedlocaltrajectoryplanner_b200.scenarios import Track, make_scenarios
    import torch
    g = H.golden("ticks_ext_default.npz")
    pl = _planner(g)
    sc = make_scenarios(Track(H.TRACK_CSV), 96, seed=31, n_obj_min=0, n_obj_max=3)
    pl.stage_scenarios(sc)
    pl.upload()
    pl.set_startpos()
    pl.tick()
    out = pl.download()
    torch.cuda.synchronize()
    recs = pl.records()
    views = Graph_LTPL.unpack_batch(out)
    assert len(views) == sc.size
    n_em = 0
    for b in range(sc.size):
        traj, ids = views[b]
        want = recs[b].get("traj", {})
        assert sorted(traj) == sorted(want), "scenario %d: %s vs %s" % (b, sorted(traj), sorted(want))
        for name in want:
            assert np.array_equal(traj[name][0].astype(np.float64), want[name][0])
            assert ids[name] == recs[b]["ids"][name]
        n_em += int("emergency" in traj)
    assert n_em > sc.size // 2


def test_explicit_predictions_match_reference_golden_and_oracle():
    """objects with an explicit 'prediction' array (OLI:117-119): up to 4 points per object, mixed with objects that use
    the built-in 0.2 s point; golden vectors of the reference + a seeded batch against the oracle."""
    from oracle.ltpl_oracle import OracleLTPL
    from graphbasedlocaltrajectoryplanner_b200.planner import BatchPlanner
    from graphbasedlocaltrajectoryplanner_b200.scenarios import ScenarioBatch, Track, make_scenarios
    g = H.golden("ticks_pred_default.npz")
    n = g["sc_pos"].shape[0]
    ols = [H.object_list(g, b) for b in range(n)]
    sc = ScenarioBatch.from_object_lists(g["sc_pos"], g["sc_heading"], g["sc_vel"], ols, k_max=3)
    assert sc.pred is not None and np.array_equal(sc.n_pred, g["sc_n_pred"])
    vel = dict(vel_max=100.0, gg_scale=1.0, local_gg=(5.0, 5.0), ax_max_machines=g["ax_max_machines"], safety_d=30.0)
    pl = BatchPlanner(H.lattice_for("default"), device="cuda:0")
    pl.set_vel_params(**vel)
    pl.stage_scenarios(sc)
    pl.upload()
    pl.set_startpos()
    pl.tick()
    recs = pl.records()
    for b in range(n):
        H.compare_record(recs[b], g, b, prefix="", ctx="pred gpu")
    # seeded: many prediction points (up to 6) so that several scenarios hold > 10 discs
    sc2 = make_scenarios(Track(H.TRACK_CSV), 128, seed=606, n_obj_min=1, n_obj_max=4)
    rng = np.random.default_rng(607)
    kp = 6
    sc2.pred = np.zeros((sc2.size, sc2.obj.shape[1], kp, 2))
    sc2.n_pred = np.full((sc2.size, sc2.obj.shape[1]), -1, dtype=np.int32)
    for b in range(sc2.size):
        for k in range(int(sc2.n_obj[b])):
            if rng.random() < 0.2:
                continue
            m = int(rng.integers(0, kp + 1))
            x, y, th, v, _ = sc2.obj[b, k]
            for j in range(m):
                t = 0.25 * (j + 1)
                sc2.pred[b, k, j] = [x - np.sin(th) * v * t, y + np.cos(th) * v * t]
            sc2.n_pred[b, k] = m
    pl.stage_scenarios(sc2)
    pl.upload()
    pl.set_startpos()
    pl.tick()
    recs2 = pl.records()
    orc = OracleLTPL(H.lattice_for("default"))
    for b in range(sc2.size):
        want = orc.tick(sc2.pos[b], sc2.heading[b], sc2.vel[b], sc2.object_list(b), vel)
        H.compare_records(recs2[b], want, ctx="pred seeded %d" % b)
    # a later batch WITHOUT predictions on the same planner goes back to the built-in rule
    sc3 = make_scenarios(Track(H.TRACK_CSV), 128, seed=608, n_obj_min=1, n_obj_max=4)
    pl.stage_scenarios(sc3)
    pl.upload()
    pl.set_startpos()
    pl.tick()
    recs3 = pl.records()
    for b in range(0, sc3.size, 4):
        want = orc.tick(sc3.pos[b], sc3.heading[b], sc3.vel[b], sc3.object_list(b), vel)
        H.compare_records(recs3[b], want, ctx="no-pred after pred %d" % b)


def test_location_dependent_local_gg_matches_reference_golden(tmp_path):
    """calc_vel_profile(local_gg={action: [ndarray(P, 2)]}) (OTH:649-666, VPFB:194-227) against the reference: friction
    as a function of the position along every path (buffers.gg planes, k_vel_res<.., GG>), emergency trajectory on
    (raw local_gg of its base trajectory, OTH:1030); batch API and the facade's dict form."""
    from graphbasedlocaltrajectoryplanner_b200.Graph_LTPL import Graph_LTPL
    from graphbasedlocaltrajectoryplanner_b200.planner import BatchPlanner
    from graphbasedlocaltrajectoryplanner_b200.scenarios import ScenarioBatch
    g = H.golden("ticks_ggpp_default.npz")
    sc = ScenarioBatch(g["sc_pos"], g["sc_heading"], g["sc_vel"], g["sc_n_obj"], g["sc_obj"])
    pl = BatchPlanner(H.lattice_for("default"), device="cuda:0")
    pl.set_vel_params(vel_max=100.0, gg_scale=1.0, local_gg=None, ax_max_machines=g["ax_max_machines"], safety_d=30.0,
                      incl_emerg_traj=True)
    pl.stage_scenarios(sc)
    pl.upload()
    pl.set_startpos()
    pl.calc_paths()
    pl.set_local_gg_planes(*H.local_gg_planes(pl))
    pl.calc_vel_profile()
    recs = pl.records()
    n_em = 0
    for b in range(sc.size):
        H.compare_record(recs[b], g, b, ctx="ggpp")
        n = min(int(g["em_len"][b]), 115)
        assert ("emergency" in recs[b].get("traj", {})) == (n > 0), "scenario %d emergency presence" % b
        if n:
            H.assert_close("traj[emergency]", recs[b]["traj"]["emergency"][0], g["em_traj"][b, :n],
                           ("s", "x", "y", "psi", "kappa", "vx", "ax"), "ggpp scenario %d" % b, w_rel=H.W_REL_BRAKE)
            n_em += 1
    assert n_em >= sc.size // 2
    # the facade takes the reference's dict form
    pd = {'globtraj_input_path': H.TRACK_CSV, 'graph_store_path': str(tmp_path / "lattice_default.npz"),
          'ltpl_offline_param_path': H.OFFLINE_INI, 'ltpl_online_param_path': H.ONLINE_INI}
    ltpl = Graph_LTPL(path_dict=pd, visual_mode=False, log_to_file=False, device="cuda:0")
    ltpl.graph_init()
    done = 0
    for b in range(sc.size):
        if bool(g["full_out_of_track"][b]) or done >= 6:
            continue
        assert ltpl.set_startpos(pos_est=sc.pos[b], heading_est=sc.heading[b], vel_est=sc.vel[b]) is False
        paths = ltpl.calc_paths(prev_action_id="straight", object_list=sc.object_list(b))
        gg = {a: [H.local_gg_field(p[0][:, 0:2])] for a, p in paths.items()}
        traj, ids, _ = ltpl.calc_vel_profile(pos_est=sc.pos[b], vel_est=float(sc.vel[b]), local_gg=gg,
                                             ax_max_machines=g["ax_max_machines"])
        for a, act in enumerate(H.ACTIONS):
            t_want = int(g["full_traj_len"][b, a])
            assert (act in traj) == (t_want > 0), "facade scenario %d %s" % (b, act)
            if t_want:
                H.assert_close("traj[%s]" % act, traj[act][0], g["full_traj"][b, a, :min(t_want, 115)],
                               ("s", "x", "y", "psi", "kappa", "vx", "ax"), "facade ggpp scenario %d" % b)
        with pytest.raises(ValueError):   # an array that does not match its path
            bad = {a: [v[0][:-1]] for a, v in gg.items()}
            ltpl.set_startpos(pos_est=sc.pos[b], heading_est=sc.heading[b], vel_est=sc.vel[b])
            ltpl.calc_paths(prev_action_id="straight", object_list=sc.object_list(b))
            ltpl.calc_vel_profile(pos_est=sc.pos[b], vel_est=float(sc.vel[b]), local_gg=bad)
        done += 1
    assert done >= 4
