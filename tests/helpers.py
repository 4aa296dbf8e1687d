"""Shared helpers of the parity tests: lattice construction per golden tag, golden loading, record comparison."""
import ast
import functools
import os

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(REPO, "tests", "golden")
TRACK_CSV = os.path.join(REPO, "inputs", "traj_ltpl_cl", "traj_ltpl_cl_monteblanco.csv")
OPEN_TRACK_CSV = os.path.join(REPO, "inputs", "traj_ltpl_cl", "traj_ltpl_cl_monteblanco_open.csv")   # first 560 points
OFFLINE_INI = os.path.join(REPO, "params", "ltpl_config_offline.ini")
ONLINE_INI = os.path.join(REPO, "params", "ltpl_config_online.ini")
ACTIONS = ("straight", "follow", "left", "right")

# tolerances of BASELINE.json north_star: node sequences bit-exact; coordinates / velocity 1e-4 relative
# (absolute floors for quantities that pass through zero: heading [rad], curvature [1/m], acceleration [m/s^2]).
RTOL = 1e-4
ATOL = dict(s=1e-3, x=1e-3, y=1e-3, psi=1e-4, kappa=2e-6, el=1e-4, vx=2e-3, ax=5e-3)


def golden(name):
    return np.load(os.path.join(GOLDEN, name), allow_pickle=False)


@functools.lru_cache(maxsize=None)
def lattice_for(tag):
    from graphbasedlocaltrajectoryplanner_b200.lattice import build_lattice
    ov = dict(ast.literal_eval(str(golden("ticks_%s.npz" % tag)["overrides"])))
    return build_lattice(track_csv_for(tag), OFFLINE_INI, overrides=ov)


def track_csv_for(tag):
    return OPEN_TRACK_CSV if tag == "open" else TRACK_CSV


def object_list(g, b):
    out = []
    for k in range(int(g["sc_n_obj"][b])):
        x, y, th, v, ln = (float(a) for a in g["sc_obj"][b, k])
        out.append({'id': k + 1, 'type': 'physical', 'X': x, 'Y': y, 'theta': th, 'v': v, 'length': ln, 'width': 2.5})
        if "sc_n_pred" in g.files and int(g["sc_n_pred"][b, k]) >= 0:
            out[-1]['prediction'] = g["sc_pred"][b, k, :int(g["sc_n_pred"][b, k])].copy()
    return out


W_REL_BRAKE = 2e-5   # see assert_close(w_rel=...)


def assert_close(name, got, want, cols, ctx="", w_rel=None):
    """w_rel: a brake-to-standstill profile (the 'emergency' trajectory) is integrated in w = v^2 from its start
    velocity v0; a relative difference eps in v0 (1e-6 from the fp32 velocity recurrences, against a tolerance of 1e-4)
    becomes eps v0^2 / v in v just before standstill.  Such profiles are therefore ALSO accepted where
    |v_got^2 - v_want^2| <= w_rel * v0^2 (the same tolerance, stated in the quantity the profile is integrated in)."""
    got = np.asarray(got, dtype=np.float64)
    want = np.asarray(want, dtype=np.float64)
    assert got.shape == want.shape, "%s %s: shape %s vs %s" % (ctx, name, got.shape, want.shape)
    for c, key in enumerate(cols):
        d = np.abs(got[:, c] - want[:, c])
        if key == "psi":   # headings are compared modulo 2 pi
            d = np.abs(np.mod(got[:, c] - want[:, c] + np.pi, 2 * np.pi) - np.pi)
        lim = ATOL[key] + RTOL * np.abs(want[:, c])
        if w_rel is not None and key == "vx":
            lim = np.where(np.abs(got[:, c] ** 2 - want[:, c] ** 2) <= w_rel * want[0, c] ** 2, np.inf, lim)
        if w_rel is not None and key == "ax":   # ax = d(v^2) / (2 ds): the same band, ds >= 0.5 m
            w0 = want[0, cols.index("vx")] ** 2
            lim = np.maximum(lim, 2.0 * w_rel * w0)
        bad = np.nonzero(d > lim)[0]
        assert bad.size == 0, "%s %s col %s: %d/%d rows off, worst |d|=%.3e at row %d (want %.6e got %.6e)" % (
            ctx, name, key, bad.size, d.size, d.max(), int(np.argmax(d)), want[int(np.argmax(d)), c],
            got[int(np.argmax(d)), c])


def compare_record(rec, g, b, prefix="full_", ctx=""):
    """compare one tick record (dict of dicts like oracle.tick()) against row b of a golden ticks file.  A file with
    `point_stride` s stores every s-th point of the paths and trajectories; path_len / traj_len stay the full lengths
    and are compared exactly."""
    ctx = "%s scenario %d" % (ctx, b)
    s = int(g["point_stride"]) if "point_stride" in g.files else 1
    assert bool(rec["out_of_track"]) == bool(g[prefix + "out_of_track"][b]), ctx
    if rec["out_of_track"]:
        return
    assert list(rec["start_node"]) == g[prefix + "start_node"][b].tolist(), ctx + " start node"
    coi = -1 if rec["closest_obj_index"] is None else int(rec["closest_obj_index"])
    assert coi == int(g[prefix + "closest_obj_index"][b]), ctx + " closest_obj_index"
    for a, act in enumerate(ACTIONS):
        n_want = int(g[prefix + "path_len"][b, a])
        has = act in rec["paths"] and len(rec["paths"][act]) > 0
        assert has == (n_want > 0), "%s: action %s present=%s, golden len %d" % (ctx, act, has, n_want)
        if has:
            nodes = [[-1 if v is None else int(v) for v in pair] for pair in rec["nodes"][act][0]]
            want_nodes = g[prefix + "nodes"][b, a, :int(g[prefix + "nodes_len"][b, a])].tolist()
            assert nodes == want_nodes, "%s: node sequence of %s differs\n got  %s\n want %s" % (ctx, act, nodes,
                                                                                                 want_nodes)
            ni = np.asarray(rec["node_idx"][act][0]).tolist()
            assert ni == g[prefix + "node_idx"][b, a, :len(ni)].tolist(), ctx + " node_idx " + act
            assert bool(rec["red_len"][act][0]) == bool(g[prefix + "red_len"][b, a]), ctx + " red_len " + act
            assert len(rec["paths"][act][0]) == n_want, "%s: path %s has %d points, golden %d" % (
                ctx, act, len(rec["paths"][act][0]), n_want)
            assert_close("path[%s]" % act, rec["paths"][act][0][::s], g[prefix + "path"][b, a, :(n_want + s - 1) // s],
                         ("x", "y", "psi", "kappa", "el"), ctx)
        t_want = int(g[prefix + "traj_len"][b, a])
        t_has = act in rec["traj_full"] and len(rec["traj_full"][act]) > 0
        assert t_has == (t_want > 0), "%s: trajectory %s present=%s, golden len %d" % (ctx, act, t_has, t_want)
        if t_has:
            # the id base (+10 per calc_vel_profile call, OTH:669) is instance state; the action code is id % 10
            assert int(rec["ids"][act]) % 10 == int(g[prefix + "traj_id"][b, a]) % 10, ctx + " traj id " + act
            assert len(rec["traj_full"][act][0]) == t_want, "%s: trajectory %s has %d points, golden %d" % (
                ctx, act, len(rec["traj_full"][act][0]), t_want)
            assert_close("traj[%s]" % act, rec["traj_full"][act][0][::s], g[prefix + "traj"][b, a, :(t_want + s - 1) // s],
                         ("s", "x", "y", "psi", "kappa", "vx", "ax"), ctx)
            assert rec["traj"][act][0].shape[0] == int(g["cut_traj_len"][b, a]) if "cut_traj_len" in g.files else True


def compare_records(got, want, ctx=""):
    """compare two tick records (e.g. CUDA path vs oracle) with the same rules as compare_record."""
    assert bool(got["out_of_track"]) == bool(want["out_of_track"]), ctx + " out_of_track"
    if want["out_of_track"]:
        return
    assert "error" not in got, ctx + " error flags %s" % got.get("error")
    assert list(got["start_node"]) == list(want["start_node"]), ctx + " start node"
    assert got["closest_obj_index"] == want["closest_obj_index"], ctx + " closest_obj_index %s vs %s" % (
        got["closest_obj_index"], want["closest_obj_index"])
    assert sorted(got["paths"].keys()) == sorted(want["paths"].keys()), ctx + " action sets %s vs %s" % (
        sorted(got["paths"]), sorted(want["paths"]))
    for act in want["paths"]:
        gn = [[-1 if v is None else int(v) for v in p] for p in got["nodes"][act][0]]
        wn = [[-1 if v is None else int(v) for v in p] for p in want["nodes"][act][0]]
        if want.get("tie", {}).get(act) or got.get("tie", {}).get(act):
            continue   # exact cost tie: igraph's choice is heap-order dependent (flagged, not compared)
        assert gn == wn, "%s: node sequence of %s differs\n got  %s\n want %s" % (ctx, act, gn, wn)
        assert np.asarray(got["node_idx"][act][0]).tolist() == np.asarray(want["node_idx"][act][0]).tolist(), \
            ctx + " node_idx " + act
        assert bool(got["red_len"][act][0]) == bool(want["red_len"][act][0]), ctx + " red_len " + act
        assert_close("path[%s]" % act, got["paths"][act][0], want["paths"][act][0], ("x", "y", "psi", "kappa", "el"),
                     ctx)
        c_g, c_w = np.asarray(got["coeff"][act][0]), np.asarray(want["coeff"][act][0])
        assert c_g.shape == c_w.shape, ctx + " coeff shape " + act
        assert np.all(np.abs(c_g - c_w) <= 1e-6 + 1e-6 * np.abs(c_w)), ctx + " spline coefficients " + act
    assert sorted(got["traj_full"].keys()) == sorted(want["traj_full"].keys()), ctx + " trajectory sets %s vs %s" % (
        sorted(got["traj_full"]), sorted(want["traj_full"]))
    for act in want["traj_full"]:
        assert int(got["ids"][act]) % 10 == int(want["ids"][act]) % 10, ctx + " traj id " + act
        assert_close("traj[%s]" % act, got["traj_full"][act][0], want["traj_full"][act][0],
                     ("s", "x", "y", "psi", "kappa", "vx", "ax"), ctx)
        n_cut = want["traj"][act][0].shape[0]
        assert got["traj"][act][0].shape[0] == n_cut, ctx + " exported rows " + act
        assert_close("export[%s]" % act, got["traj"][act][0], want["traj"][act][0][:n_cut],
                     ("s", "x", "y", "psi", "kappa", "vx", "ax"), ctx)


def local_gg_field(xy):
    """location dependent friction of the per-point local_gg fixtures: (ax_max, ay_max) as a smooth function of the
    position, one row per path point -- calc_vel_profile(local_gg={action: [local_gg_field(path[:, 0:2])]}) (OTH:649-666)."""
    xy = np.asarray(xy, dtype=np.float64)
    return np.column_stack((4.2 + 1.1 * np.sin(0.011 * xy[:, 0] + 0.5), 4.6 + 0.9 * np.cos(0.013 * xy[:, 1] - 0.3)))


def local_gg_planes(pl):
    """[NSLOT][B][p_max] planes (ax, ay) of local_gg_field along the paths a BatchPlanner just planned (calc_paths)."""
    f = pl.fetch("path")
    path = f["path"]                                   # [5][NSLOT * B][p_max]
    gg = local_gg_field(np.column_stack((path[0].ravel(), path[1].ravel())))
    shape = (path.shape[1] // pl.dims.batch, pl.dims.batch, path.shape[2])
    return gg[:, 0].reshape(shape), gg[:, 1].reshape(shape)


def zone_of(g, b, tick=0):
    """blocked_zones dict of scenario b of the zone / emergency fixture (None: no zone); fixtures with a zone swap pass
    another zone under a new id from tick `zone_swap_tick` on."""
    n = int((g["zone_layers"][b] >= 0).sum())
    if n == 0:
        return None
    if "zone_swap_tick" in g.files and tick >= int(g["zone_swap_tick"]):
        n2 = int((g["zone2_layers"][b] >= 0).sum())
        return {"zone_%d_b" % b: [g["zone2_layers"][b, :n2].tolist(), g["zone2_nodes"][b, :n2].tolist(), np.zeros((2, 2)),
                                  np.zeros((2, 2))]}
    return {"zone_%d" % b: [g["zone_layers"][b, :n].tolist(), g["zone_nodes"][b, :n].tolist(), np.zeros((2, 2)),
                            np.zeros((2, 2))]}


def compare_emergency(rec, g, b, ctx=""):
    """'emergency' entry (OTH:1027-1034) of a tick record against the zone / emergency fixture."""
    n = int(g["em_len"][b])
    has = "emergency" in rec.get("traj_full", {})
    assert has == (n > 0), "%s scenario %d: emergency present=%s, golden len %d" % (ctx, b, has, n)
    if has:
        assert int(rec["ids"]["emergency"]) % 10 == int(g["em_id"][b]) % 10, "%s scenario %d emergency id" % (ctx, b)
        assert_close("traj[emergency]", rec["traj_full"]["emergency"][0], g["em_traj"][b, :n],
                     ("s", "x", "y", "psi", "kappa", "vx", "ax"), "%s scenario %d" % (ctx, b), w_rel=W_REL_BRAKE)


VARIANTS = {   # oracle/gen_golden.py VARIANTS: online overrides, vehicle parameters, velocity arguments, vel_est offset
    "pdtan_exp15": (dict(controller_type="PDtan", control_params={"c_p": 1.15, "k_d": 0.025, "k_p": 0.2, "tan_w": 15.0}),
                    dict(veh_param_dyn_model_exp=1.5, veh_param_dragcoeff=0.9, veh_param_mass=1200.0),
                    dict(vel_max=85.0, gg_scale=0.9, local_gg=(4.5, 5.5), safety_d=20.0), -2.0),
    "pd_exp20": (dict(), dict(veh_param_dyn_model_exp=2.0, veh_param_dragcoeff=0.7, veh_param_mass=900.0),
                 dict(vel_max=90.0, gg_scale=1.0, local_gg=(6.0, 4.0), safety_d=40.0), 3.0),
}


class _Sub(object):
    """view of the arrays of one variant inside ticks_variants_default.npz (keys '<variant>__<name>')."""

    def __init__(self, g, name):
        self.g, self.p = g, name + "__"
        self.files = [k[len(self.p):] for k in g.files if k.startswith(self.p)]

    def __getitem__(self, k):
        return self.g[self.p + k]
