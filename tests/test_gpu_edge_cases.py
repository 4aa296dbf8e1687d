"""edge cases of the batched path (GPU): empty / ragged inputs, flagged scenarios, single-scenario facade calls."""
import numpy as np
import pytest

from tests import helpers as H

pytestmark = pytest.mark.gpu
VEL = dict(vel_max=100.0, gg_scale=1.0, local_gg=(5.0, 5.0), safety_d=30.0)


def _oracle(tag):
    from oracle.ltpl_oracle import OracleLTPL
    return OracleLTPL(H.lattice_for(tag))


def _planner(tag):
    from graphbasedlocaltrajectoryplanner_b200.planner import BatchPlanner
    return BatchPlanner(H.lattice_for(tag), device="cuda:0")


@pytest.mark.parametrize("batch", [1, 7, 33, 257])
def test_ragged_batch_sizes_and_object_counts(batch):
    """batch sizes that do not fill a CTA / warp group; scenarios with 0..K objects mixed in one batch."""
    from graphbasedlocaltrajectoryplanner_b200.scenarios import Track, make_scenarios
    g = H.golden("ticks_default.npz")
    sc = make_scenarios(Track(H.TRACK_CSV), batch, seed=900 + batch, n_obj_min=0, n_obj_max=5, k_max=5)
    pl = _planner("default")
    pl.set_vel_params(ax_max_machines=g["ax_max_machines"], **VEL)
    pl.stage_scenarios(sc)
    pl.upload()
    pl.set_startpos()
    pl.tick()
    recs = pl.records()
    orc = _oracle("default")
    vk = dict(ax_max_machines=g["ax_max_machines"], **VEL)
    for b in range(batch):
        want = orc.tick(sc.pos[b], sc.heading[b], sc.vel[b], sc.object_list(b), vk)
        H.compare_records(recs[b], want, ctx="batch %d scenario %d" % (batch, b))


def test_out_of_track_heading_mismatch_and_offtrack_objects():
    """flag semantics of set_startpos (OTH:214-241) and the on-track filter of the object list (OLI:104-112)."""
    from graphbasedlocaltrajectoryplanner_b200 import capi
    from graphbasedlocaltrajectoryplanner_b200.scenarios import ScenarioBatch, Track
    tr = Track(H.TRACK_CSV)
    p, h, v = tr.raceline_pose(np.array([100.0, 100.0, 100.0, 600.0]))
    pos = p.copy()
    heading = h.copy()
    pos[0] = p[0] + np.array([500.0, 500.0])         # far off the track
    heading[1] = h[1] + np.pi                         # driving the wrong way
    far = {'id': 1, 'type': 'physical', 'X': 1e4, 'Y': 1e4, 'theta': 0.0, 'v': 3.0, 'length': 5.0, 'width': 2.5}
    po, _, _ = tr.raceline_pose(np.array([700.0]))
    near = {'id': 2, 'type': 'physical', 'X': float(po[0, 0]), 'Y': float(po[0, 1]), 'theta': 0.0, 'v': 3.0,
            'length': 5.0, 'width': 2.5}
    ols = [[], [], [far], [far, near]]
    sc = ScenarioBatch.from_object_lists(pos, heading, [20.0] * 4, ols, k_max=2)
    pl = _planner("default")
    pl.set_vel_params(**VEL)
    pl.stage_scenarios(sc)
    pl.upload()
    pl.set_startpos()
    pl.tick()
    recs = pl.records()
    orc = _oracle("default")
    assert recs[0]["flags"] & capi.SC_OUT_OF_TRACK and recs[0]["out_of_track"]
    assert recs[1]["flags"] & capi.SC_HEADING_MISMATCH and recs[1]["out_of_track"]
    for b in range(4):
        want = orc.tick(sc.pos[b], sc.heading[b], sc.vel[b], ols[b], dict(VEL))
        H.compare_records(recs[b], want, ctx="scenario %d" % b)
    assert list(recs[2]["paths"]) == ["straight"]            # the only object is off the track -> ignored
    assert recs[3]["closest_obj_index"] == 0                  # index into the ON-TRACK object list (OLI:143)


def test_vel_max_below_planned_velocity_is_reported():
    """vel_plan > vel_max + 0.1: the reference's brake-prefix branch cannot produce a trajectory (DESIGN.md section 7)."""
    from graphbasedlocaltrajectoryplanner_b200 import capi
    from graphbasedlocaltrajectoryplanner_b200.scenarios import Track, make_scenarios
    sc = make_scenarios(Track(H.TRACK_CSV), 16, seed=5, n_obj_min=1, n_obj_max=2)
    sc.vel[:] = 30.0
    pl = _planner("l216")
    pl.set_vel_params(vel_max=20.0, gg_scale=1.0, local_gg=(5.0, 5.0), ax_max_machines=np.atleast_2d([100.0, 5.0]),
                      safety_d=30.0)
    pl.stage_scenarios(sc)
    pl.upload()
    pl.set_startpos()
    pl.tick()
    f = pl.fetch("sc_flags", "traj_len")
    ok = f["sc_flags"] & (capi.SC_OUT_OF_TRACK | capi.SC_HEADING_MISMATCH) == 0
    assert np.all((f["sc_flags"][ok] & capi.SC_BRAKE_PREFIX) != 0) and int(f["traj_len"].sum()) == 0


def test_single_scenario_facade_matches_config1_and_errors(tmp_path):
    """Graph_LTPL facade with the reference's call sequence (main_min_example.py:69-104) + error behaviour."""
    from graphbasedlocaltrajectoryplanner_b200.Graph_LTPL import Graph_LTPL
    g = H.golden("config1_min_example.npz")
    pd = {'globtraj_input_path': H.TRACK_CSV, 'graph_store_path': str(tmp_path / "lattice_default.npz"),
          'ltpl_offline_param_path': H.OFFLINE_INI, 'ltpl_online_param_path': H.ONLINE_INI}
    ltpl = Graph_LTPL(path_dict=pd, visual_mode=False, log_to_file=False, device="cuda:0")
    ltpl.graph_init()
    x, y, th, v, ln = (float(a) for a in g["obj"])
    obj = [{'id': 1, 'type': 'physical', 'X': x, 'Y': y, 'theta': th, 'length': ln, 'width': 2.5, 'v': v}]
    for b in range(2):
        assert ltpl.set_startpos(pos_est=g["sc_pos"][b], heading_est=g["sc_heading"][b], vel_est=g["sc_vel"][b]) is False
        paths = ltpl.calc_paths(prev_action_id="straight", object_list=obj)
        traj, ids, t = ltpl.calc_vel_profile(pos_est=g["sc_pos"][b], vel_est=float(g["sc_vel"][b]))
        for a, act in enumerate(H.ACTIONS):
            n = int(g["path_len"][b, a])
            assert (act in paths) == (n > 0)
            if n:
                H.assert_close("path", paths[act][0], g["path"][b, a, :n], ("x", "y", "psi", "kappa", "el"), act)
            tl = min(int(g["traj_len"][b, a]), 115)
            assert (act in traj) == (tl > 0)
            if tl:
                assert traj[act][0].shape == (tl, 7) and ids[act] % 10 == int(g["traj_id"][b, a]) % 10
                H.assert_close("traj", traj[act][0], g["traj"][b, a, :tl], ("s", "x", "y", "psi", "kappa", "vx", "ax"),
                               act)
    with pytest.raises(ValueError):      # OTH:651-653
        ltpl.set_startpos(pos_est=g["sc_pos"][0], heading_est=g["sc_heading"][0])
        ltpl.calc_paths(prev_action_id="straight", object_list=[])
        ltpl.calc_vel_profile(pos_est=g["sc_pos"][0], vel_est=0.0, local_gg=[5.0, 5.0])
    with pytest.raises(RuntimeError):    # tph.calc_vel_profile: ax_max_machines must cover v_max
        ltpl.set_startpos(pos_est=g["sc_pos"][0], heading_est=g["sc_heading"][0])
        ltpl.calc_paths(prev_action_id="straight", object_list=[])
        ltpl.calc_vel_profile(pos_est=g["sc_pos"][0], vel_est=0.0, vel_max=120.0)
    assert ltpl.set_startpos(pos_est=np.array([1e4, 1e4]), heading_est=0.0) is True      # out of track


def test_c_abi_error_convention():
    """entry points return < 0 and ltpl_last_error() names the problem (INTEGRATION.md section 2); nothing is launched."""
    import ctypes as C
    from graphbasedlocaltrajectoryplanner_b200 import capi
    from graphbasedlocaltrajectoryplanner_b200.scenarios import Track, make_scenarios
    pl = _planner("l216")
    pl.set_vel_params(**VEL)
    pl.stage_scenarios(make_scenarios(Track(H.TRACK_CSV), 8, seed=1))
    pl.upload()
    pl.set_startpos()
    n0 = pl.launch_count()
    keep = pl.dims.batch
    pl.dims.batch = 0
    with pytest.raises(RuntimeError, match="batch"):
        pl.tick()
    pl.dims.batch = keep
    keep_ptr = pl.buf.path
    pl.buf.path = None
    with pytest.raises(RuntimeError, match="NULL"):
        pl.tick()
    pl.buf.path = keep_ptr
    pl.dims.n_zones = 1                                   # zones announced without bitmasks
    keep_z = pl.buf.zone_bits
    pl.buf.zone_bits = None
    with pytest.raises(RuntimeError, match="zone"):
        pl.calc_paths()
    pl.buf.zone_bits = keep_z
    pl.dims.n_zones = 0
    assert pl.launch_count() == n0
    rc = pl.lib.ltpl_tick_batch(None, C.byref(pl.params), C.byref(pl.dims), C.byref(pl.buf), pl.stream)
    assert rc < 0 and b"null" in pl.lib.ltpl_last_error()
    pl.tick()                                             # still usable afterwards
    assert pl.launch_count() > n0


def test_tick_under_cuda_graph_capture_replays_identically():
    """a tick (three scenario windows = fork / join over the library's internal streams) captured into a CUDA graph
    and replayed gives the bytes of the eager tick (rows of the compact export compared through traj_row)."""
    import torch
    from graphbasedlocaltrajectoryplanner_b200.scenarios import Track, make_scenarios
    g = H.golden("ticks_default.npz")
    sc = make_scenarios(Track(H.TRACK_CSV), 300, seed=77, n_obj_min=0, n_obj_max=3)
    pl = _planner("default")
    pl.set_subbatches(3)
    pl.set_vel_params(ax_max_machines=g["ax_max_machines"], incl_emerg_traj=True, **VEL)
    pl.stage_scenarios(sc)
    pl.upload()
    pl.set_startpos()
    names = ("action_id", "status", "n_nodes", "nodes", "path_len", "traj_len", "traj_row", "traj", "em_info", "sc_flags")

    def snapshot():
        torch.cuda.synchronize()
        f = pl.fetch(*names)
        ok = f["traj_row"] >= 0
        rows = np.zeros(f["traj_row"].shape + f["traj"].shape[1:], dtype=np.float32)
        rows[ok] = f["traj"][f["traj_row"][ok]]
        rows[np.arange(rows.shape[2])[None, None, :] >= f["traj_len"][..., None]] = 0.0
        nodes = f["nodes"].copy()
        nodes[np.arange(nodes.shape[2])[None, None, :] >= f["n_nodes"][..., None]] = -1
        em = f["em_info"].copy()
        em_rows = f["traj"][np.maximum(em[:, 0], 0)] * (em[:, 0] >= 0)[:, None, None]
        return dict(action_id=f["action_id"], status=f["status"], nodes=nodes, path_len=f["path_len"],
                    traj_len=f["traj_len"], rows=rows, em_len=em[:, 1], em_rows=em_rows, flags=f["sc_flags"])

    pl.tick()                                   # eager (also the warm-up that sets the kernels' attributes)
    want = snapshot()
    assert (want["traj_len"] > 0).sum() > 300
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=side):
        pl.tick()                               # launches on the capturing stream (torch's current stream)
    torch.cuda.current_stream().wait_stream(side)
    for name in ("traj", "traj_row", "traj_len", "action_id", "status"):   # the replay has to produce everything again
        pl.t[name].zero_()
    graph.replay()
    got = snapshot()
    for k in want:
        assert np.array_equal(got[k], want[k]), k
