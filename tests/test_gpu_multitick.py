"""Stateful tick on the device (csrc/ltpl_state.cuh, BatchPlanner.next_tick) against the closed-loop
sequences of the unmodified reference (tests/golden/ticks_multitick_default.npz, scripted clock): the 16 sequences run
as ONE batch, tick 0 = set_startpos + first tick, ticks 1.. = next_tick with the recorded inputs."""
import numpy as np
import pytest

from tests import helpers as H

pytestmark = pytest.mark.gpu


def _t_const(dts):
    """OTH:353-375: moving average (5) of the calculation times * calc_time_safety (2.0), capped at 0.5 s."""
    buf, out = [], []
    for dt in dts:
        if len(buf) >= 5:
            buf.pop(0)
        buf.append(float(dt))
        out.append(min(float(np.sum(buf) / len(buf)) * 2.0, 0.5))
    return out


class _Rows(object):
    """the sequences `idx` of a multi-tick fixture (gg_scale is a per-batch parameter: grip-drop sequences run apart)."""

    def __init__(self, g, idx):
        self.g, self.idx, self.files = g, np.asarray(idx), g.files

    def __getitem__(self, k):
        a = self.g[k]
        return a if k == "ax_max_machines" else a[self.idx]


@pytest.mark.parametrize("fixture,emerg,group,tag", [("ticks_multitick_default.npz", False, None, "default"),
                                                     ("ticks_multitick_ext_default.npz", True, None, "default"),
                                                     ("ticks_multitick_backup_default.npz", False, 0, "default"),
                                                     ("ticks_multitick_backup_default.npz", False, 1, "default"),
                                                     ("ticks_multitick_emsel_default.npz", True, None, "default"),
                                                     ("ticks_multitick_l216.npz", True, None, "l216"),
                                                     ("ticks_multitick_l430.npz", False, None, "l430"),
                                                     ("ticks_multitick_open.npz", False, None, "open"),
                                                     ("ticks_multitick_zswap_default.npz", False, None, "default"),
                                                     ("ticks_multitick_invalid_default.npz", False, None, "default"),
                                                     ("ticks_multitick_openend.npz", False, None, "open"),
                                                     ("ticks_multitick_pdtan_default.npz", False, None,
                                                      "default:pdtan_exp15"),
                                                     ("ticks_multitick_ggpp_default.npz", True, 0, "default:ggpp"),
                                                     ("ticks_multitick_ggpp_default.npz", True, 1, "default:ggpp")])
def test_next_tick_matches_reference_sequences(fixture, emerg, group, tag):
    """second fixture: a blocked zone on every second sequence + the emergency trajectory in every tick; third fixture:
    the grip (gg_scale) drops on the odd sequences from tick 3 on -> brake on the backup plan (OTH:950-1006); fourth
    fixture: the odd sequences execute the 'emergency' trajectory of ticks 2 .. 4 (sel_action 4; OTH:307-309, 518-601)."""
    from graphbasedlocaltrajectoryplanner_b200 import capi
    from graphbasedlocaltrajectoryplanner_b200.planner import BatchPlanner
    from graphbasedlocaltrajectoryplanner_b200.scenarios import ScenarioBatch
    g = H.golden(fixture)
    if group is not None:
        g = _Rows(g, np.arange(group, g["dt"].shape[0], 2))
    n_seq, n_ticks = g["dt"].shape
    n_done = g["n_done"]                                   # open track: sequences end when no trajectory is left
    tag, _, variant = tag.partition(":")
    pl_kw, vel = {}, dict(vel_max=100.0, gg_scale=1.0, local_gg=(5.0, 5.0), safety_d=30.0)
    ggpp = variant == "ggpp"   # location dependent local_gg = H.local_gg_field along every path (OTH:649-666), grip drop
    if ggpp:
        variant = ""
    if variant:                                            # other controller / vehicle / velocity parameters (H.VARIANTS)
        online, veh, vel_v, _ = H.VARIANTS[variant]
        pl_kw = dict(online=online, **veh)
        vel.update(vel_v)
    pl = BatchPlanner(H.lattice_for(tag), device="cuda:0", stateful=True, **pl_kw)
    pl.set_subbatches(1 + n_seq % 4)                       # 1 .. 4 scenario windows inside the library
    pl.set_vel_params(ax_max_machines=g["ax_max_machines"], incl_emerg_traj=emerg, **vel)
    tc = np.array([_t_const(g["dt"][q, 1:]) for q in range(n_seq)])       # t_const of ticks 1 ..
    fails, compared = [], 0
    alive = np.ones(n_seq, dtype=bool)
    for k in range(n_ticks):
        sc = ScenarioBatch(g["pos_est"][:, k].copy(), g["sc_heading"].copy(), g["sc_vel"].copy(), g["sc_n_obj"].copy(),
                           g["obj"][:, k].copy())
        zones = [H.zone_of(g, q, k) for q in range(n_seq)]
        if any(z is not None for z in zones):
            sc.set_zones(zones)
        assert len(set(g["gg_scale"][:, k].tolist())) == 1
        pl.set_vel_params(ax_max_machines=g["ax_max_machines"], incl_emerg_traj=emerg,
                          **dict(vel, gg_scale=float(g["gg_scale"][0, k])))
        if k == 0:
            pl.stage_scenarios(sc, vel_est=g["vel_est"][:, k])
            pl.upload()
            pl.set_startpos()
            if ggpp:
                pl.calc_paths()
                pl.set_local_gg_planes(*H.local_gg_planes(pl))
                pl.calc_vel_profile()
            else:
                pl.tick()
        elif ggpp:
            pl.next_calc_paths(sc, sel_action=g["sel"][:, k], t_const=tc[:, k - 1])
            pl.set_local_gg_planes(*H.local_gg_planes(pl))
            pl.next_calc_vel_profile(vel_est=g["vel_est"][:, k])
        else:
            pl.next_tick(sc, sel_action=g["sel"][:, k], t_const=tc[:, k - 1], vel_est=g["vel_est"][:, k])
        recs = pl.records()
        for q in range(n_seq):
            if not alive[q] or k >= int(n_done[q]):
                continue
            ctx = "sequence %d tick %d" % (q, k)
            rec = recs[q]
            try:
                assert not (rec["flags"] & capi.SC_STATE_FALLBACK), ctx + " fell back (flags %d)" % rec["flags"]
                assert not rec["out_of_track"] and "error" not in rec, ctx + " flags %d" % rec["flags"]
                for a, act in enumerate(H.ACTIONS):
                    n_want = int(g["path_len"][q, k, a])
                    has = act in rec["paths"]
                    assert has == (n_want > 0), "%s: path %s present=%s, golden %d" % (ctx, act, has, n_want)
                    if has and not rec["tie"].get(act):
                        nd = [[-1 if v is None else int(v) for v in p] for p in rec["nodes"][act][0]]
                        want = g["nodes"][q, k, a, :int(g["nodes_len"][q, k, a])].tolist()
                        assert nd == want, "%s: nodes of %s\\n got  %s\\n want %s" % (ctx, act, nd, want)
                        assert rec["paths"][act][0].shape[0] == n_want, "%s: path length %s %d vs %d" % (
                            ctx, act, rec["paths"][act][0].shape[0], n_want)
                    t_want = int(g["traj_len"][q, k, a])
                    t_has = act in rec["traj"]
                    assert t_has == (t_want > 0), "%s: trajectory %s present=%s, golden %d" % (ctx, act, t_has, t_want)
                    if t_has:
                        assert rec["traj"][act][0].shape[0] == t_want, "%s: rows of %s %d vs %d" % (
                            ctx, act, rec["traj"][act][0].shape[0], t_want)
                        H.assert_close("traj[%s]" % act, rec["traj"][act][0], g["traj"][q, k, a, :t_want],
                                       ("s", "x", "y", "psi", "kappa", "vx", "ax"), ctx)
                        compared += 1
                if emerg:
                    n_em = min(int(g["em_len"][q, k]), 115)
                    assert ("emergency" in rec["traj"]) == (n_em > 0), ctx + " emergency presence"
                    if n_em:
                        H.assert_close("traj[emergency]", rec["traj"]["emergency"][0], g["em_traj"][q, k, :n_em],
                                       ("s", "x", "y", "psi", "kappa", "vx", "ax"), ctx, w_rel=H.W_REL_BRAKE)
            except AssertionError as e:
                fails.append(str(e).split("\\n")[0][:400] if "nodes of" not in str(e) else str(e)[:700])
                alive[q] = False            # later ticks of this sequence depend on this one
    assert not fails, "%d sequences diverged (of %d; %d trajectories matched before):\\n%s" % (
        len(fails), n_seq, compared, "\\n".join(fails[:8]))
    assert compared > (30 if (group is not None or n_seq < 12) else (80 if (emerg or n_seq < 16) else 150))


@pytest.mark.parametrize("tag,n_seq,omin,omax", [("default", 96, 0, 2), ("l216", 64, 1, 3), ("open", 48, 0, 2)])
def test_closed_loop_matches_session_oracle(tag, n_seq, omin, omax):
    """larger closed loop driven by the DEVICE results (vehicle dummy on the selected trajectory, moving opponents,
    changing action preference); the stateful oracle (oracle/ltpl_session.py, pinned against the reference) replays the
    same inputs tick by tick.  Sequences the device flags (memory not usable, capacity) leave the loop -- at most 5 %.
    Second case: BASELINE's ~200 x 11 lattice, whose node lists exceed 32 entries.  Third case: the OPEN track, seeded
    over its whole length -- the vehicles near the end plan reduced horizons, shrinking trajectories and stop."""
    from graphbasedlocaltrajectoryplanner_b200 import capi
    from graphbasedlocaltrajectoryplanner_b200.planner import BatchPlanner
    from graphbasedlocaltrajectoryplanner_b200.scenarios import ScenarioBatch, Track, make_scenarios
    from oracle.gen_golden import advance_on_traj
    from oracle.ltpl_oracle import OracleLTPL
    from oracle.ltpl_session import OracleSession
    g = H.golden("ticks_multitick_default.npz")
    lat = H.lattice_for(tag)
    n_ticks = 8
    vel = dict(vel_max=100.0, gg_scale=1.0, local_gg=(5.0, 5.0), ax_max_machines=g["ax_max_machines"], safety_d=30.0)
    trk = Track(H.track_csv_for(tag))
    sc0 = make_scenarios(trk, n_seq, seed=2718, n_obj_min=omin, n_obj_max=omax,
                         s_max=(trk.length - 10.0) if tag == "open" else None)
    rng = np.random.default_rng(2719)
    prefer = (("right", "left", "straight", "follow"), ("follow", "straight", "left", "right"),
              ("left", "right", "follow", "straight"), ("straight", "follow", "right", "left"))
    pl = BatchPlanner(lat, device="cuda:0", stateful=True)
    pl.set_subbatches(5)                                   # five scenario windows inside the library (uneven split)
    pl.set_vel_params(**vel)

    class Clk(object):
        def __init__(self):
            self.t = 50.0

        def __call__(self):
            return self.t
    clks = [Clk() for _ in range(n_seq)]
    ses = [OracleSession(OracleLTPL(lat), clock=clks[q]) for q in range(n_seq)]
    objs = sc0.obj.copy()
    pos_est, vel_est = sc0.pos.copy(), sc0.vel.copy()
    sel = ["straight"] * n_seq
    cbuf = [[] for _ in range(n_seq)]
    alive = np.ones(n_seq, dtype=bool)
    fails, compared, fell_back, ticks_ok, flagged = [], 0, 0, 0, 0
    last_traj = [None] * n_seq
    for k in range(n_ticks):
        dts = rng.uniform(0.04, 0.16, size=n_seq)
        tcs = np.zeros(n_seq)
        for q in range(n_seq):
            dt = float(dts[q])
            clks[q].t += dt
            for j in range(int(sc0.n_obj[q])):
                objs[q, j, 0] -= np.sin(objs[q, j, 2]) * objs[q, j, 3] * dt
                objs[q, j, 1] += np.cos(objs[q, j, 2]) * objs[q, j, 3] * dt
            if k > 0:
                if last_traj[q] is not None:
                    pos_est[q], vel_est[q] = advance_on_traj(last_traj[q], dt)
                if len(cbuf[q]) >= 5:
                    cbuf[q].pop(0)
                cbuf[q].append(dt)
                tcs[q] = min(float(np.sum(cbuf[q]) / len(cbuf[q])) * 2.0, 0.5)
        sc = ScenarioBatch(pos_est.copy(), sc0.heading.copy(), sc0.vel.copy(), sc0.n_obj.copy(), objs.copy())
        if k == 0:
            pl.stage_scenarios(sc, vel_est=vel_est)
            pl.upload()
            pl.set_startpos()
            pl.tick()
        else:
            pl.next_tick(sc, sel_action=[H.ACTIONS.index(a) for a in sel], t_const=tcs, vel_est=vel_est)
        recs = pl.records()
        for q in range(n_seq):
            if not alive[q]:
                continue
            ctx = "sequence %d tick %d (sel %s)" % (q, k, sel[q])
            rec = recs[q]
            if rec["out_of_track"] or (rec["flags"] & (capi.SC_STATE_FALLBACK | capi.SC_CAPACITY | capi.SC_BRAKE_PREFIX)):
                alive[q] = False
                fell_back += int(bool(rec["flags"] & capi.SC_STATE_FALLBACK))
                flagged += int(not rec["out_of_track"])
                continue
            try:
                if k == 0:
                    assert ses[q].set_startpos(sc.pos[q], sc.heading[q], sc.vel[q]) is False
                paths = ses[q].calc_paths(sel[q], sc.object_list(q))
                traj, ids = ses[q].calc_vel_profile(sc.pos[q], float(vel_est[q]), **vel)
            except Exception as e:   # noqa: BLE001  (e.g. the reference's own brake-prefix failure)
                alive[q] = False
                continue
            try:
                assert sorted(rec["paths"]) == sorted(paths), "%s: paths %s vs %s" % (ctx, sorted(rec["paths"]),
                                                                                   sorted(paths))
                for act in paths:
                    if ses[q].tie.get(act) or rec["tie"].get(act):
                        continue
                    nd = [[-1 if v is None else int(v) for v in p] for p in rec["nodes"][act][0]]
                    want = [[-1 if v is None else int(v) for v in p] for p in ses[q].m_nodes[act][0]] \
                        if act in ses[q].m_nodes else None
                    assert want is None or nd == want, "%s: nodes of %s\n got  %s\n want %s" % (ctx, act, nd, want)
                    assert rec["paths"][act][0].shape[0] == paths[act][0].shape[0], ctx + " path length " + act
                assert sorted(rec["traj"]) == sorted(traj), "%s: trajectories %s vs %s" % (ctx, sorted(rec["traj"]),
                                                                                        sorted(traj))
                for act in traj:
                    assert rec["traj"][act][0].shape == traj[act][0].shape, ctx + " rows " + act
                    H.assert_close("traj[%s]" % act, rec["traj"][act][0], traj[act][0],
                                   ("s", "x", "y", "psi", "kappa", "vx", "ax"), ctx)
                    compared += 1
                ticks_ok += 1
            except AssertionError as e:
                fails.append(str(e).split("\\n")[0][:400])
                alive[q] = False
                continue
            cand = [a for a in prefer[(q + k) % len(prefer)] if a in rec["traj"]]
            if not cand:
                alive[q] = False
                continue
            sel[q] = cand[0]
            last_traj[q] = rec["traj"][sel[q]][0]
    assert not fails, "%d sequences diverged (%d ticks matched, %d fell back):\\n%s" % (
        len(fails), ticks_ok, fell_back, "\\n".join(fails[:8]))
    print("closed loop: %d of %d ticks compared, %d trajectories, %d sequences fell back, %d alive at the end" % (
        ticks_ok, n_seq * n_ticks, compared, fell_back, int(alive.sum())))
    assert ticks_ok > n_seq * n_ticks // 2 and compared > n_seq * n_ticks // 2, (ticks_ok, compared, fell_back)
    assert flagged <= n_seq // 20, "%d of %d sequences were flagged by the device (%d state fallbacks)" % (
        flagged, n_seq, fell_back)


@pytest.mark.parametrize("fixture,seqs,emerg", [("ticks_multitick_default.npz", (0, 5, 11), False),
                                                ("ticks_multitick_emsel_default.npz", (1, 3), True)])
def test_facade_runs_closed_loop_like_the_reference(fixture, seqs, emerg, tmp_path):
    """Graph_LTPL facade with the reference's call sequence over several ticks (main_std_example.py:99-126): an injected
    clock takes the place of time.time(); recorded sequences of the reference are replayed (second case: the caller
    executes the 'emergency' trajectory for three ticks, prev_action_id='emergency')."""
    from graphbasedlocaltrajectoryplanner_b200.Graph_LTPL import Graph_LTPL
    g = H.golden(fixture)
    pd = {'globtraj_input_path': H.TRACK_CSV, 'graph_store_path': str(tmp_path / "lattice_default.npz"),
          'ltpl_offline_param_path': H.OFFLINE_INI, 'ltpl_online_param_path': H.ONLINE_INI}
    ltpl = Graph_LTPL(path_dict=pd, visual_mode=False, log_to_file=False, device="cuda:0")
    ltpl.graph_init()

    class Clk(object):
        t = 10.0

        def __call__(self):
            return self.t
    clk = Clk()
    ltpl.clock = clk
    vel = dict(vel_max=100.0, gg_scale=1.0, local_gg=(5.0, 5.0), ax_max_machines=g["ax_max_machines"], safety_d=30.0,
               incl_emerg_traj=emerg)
    n_ticks = g["dt"].shape[1]
    compared = 0
    for q in seqs:
        assert ltpl.set_startpos(pos_est=g["sc_pos"][q], heading_est=g["sc_heading"][q], vel_est=g["sc_vel"][q]) is False
        n_obj = int(g["sc_n_obj"][q])
        for k in range(n_ticks):
            clk.t += float(g["dt"][q, k])
            ol = [{'id': j + 1, 'type': 'physical', 'X': float(o[0]), 'Y': float(o[1]), 'theta': float(o[2]),
                   'v': float(o[3]), 'length': float(o[4]), 'width': 2.5} for j, o in enumerate(g["obj"][q, k, :n_obj])]
            paths = ltpl.calc_paths(prev_action_id=(H.ACTIONS + ("emergency",))[int(g["sel"][q, k])], object_list=ol)
            traj, ids, _ = ltpl.calc_vel_profile(pos_est=g["pos_est"][q, k], vel_est=float(g["vel_est"][q, k]), **vel)
            ctx = "facade sequence %d tick %d" % (q, k)
            for a, act in enumerate(H.ACTIONS):
                assert (act in paths) == (int(g["path_len"][q, k, a]) > 0), ctx + " paths " + act
                t_want = int(g["traj_len"][q, k, a])
                assert (act in traj) == (t_want > 0), ctx + " trajectories " + act
                if t_want:
                    H.assert_close("traj[%s]" % act, traj[act][0], g["traj"][q, k, a, :t_want],
                                   ("s", "x", "y", "psi", "kappa", "vx", "ax"), ctx)
                    compared += 1
            if emerg and int(g["em_len"][q, k]):
                H.assert_close("traj[emergency]", traj["emergency"][0], g["em_traj"][q, k, :int(g["em_len"][q, k])],
                               ("s", "x", "y", "psi", "kappa", "vx", "ax"), ctx, w_rel=H.W_REL_BRAKE)
    assert compared > (20 if emerg else 40)
