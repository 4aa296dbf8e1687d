"""Exact ties in the graph search and in the nearest-vertex argmins.

Real lattices carry arbitrary float64 edge costs, so an exact tie between two in-edges of a node (or two goal-layer
nodes of the virtual goal) practically never occurs and the tie rules of the search would go untested.  The lattices
here round every edge cost to a multiple of a power of two q (and one lattice costs 1.0 per edge), with a virtual
goal cost of q per lateral step: every partial sum is then an exact float64, the float64 DP *is* the exact DP, and
ties are frequent.  Only the search reads the costs, so everything downstream stays comparable with the oracle.

Checked here:
  * every search of the oracle against a plain exact DP (integers in units of q / 4): minimum cost, the pick of the
    documented rule (smaller own distance first, then CSC order / goal-layer index order), and the tie flag
    LTPL_ST_TIE_AMBIGUOUS = some node, or the virtual goal, has its final (cost, own distance) minimum attained by two
    or more candidates (ties that a later candidate beats do not count);
  * (GPU) the device against the oracle on every action, flagged ones included: the flag, the node sequence and the
    node indices must be identical; the follow table (k_follow_table) row by row; stateful closed loops;
  * (GPU) positions exactly equidistant from two vertices: the device picks np.argmin's first minimum.
"""
import dataclasses
import functools
from fractions import Fraction

import numpy as np
import pytest

from tests import helpers as H

# coarse q: many ties.  The sparse lattices (l216: 72 % of the nodes have at most one in-edge, l430: 95 % have none)
# only tie often with a coarser grid (l430 at q = 1024: 94 % of the costs round to 0).
Q_COARSE = {"default": 64.0, "layers14": 64.0, "open": 64.0, "l216": 256.0, "l430": 1024.0}
Q_FINE = 1.0      # few ties (none at all on the sparse lattices: there it checks the exact minimum and the pick)
UNIT = None       # every edge costs 1.0: all paths of equal length tie
TIE_LATTICES = [(tag, q) for tag in ("default", "l216", "l430", "layers14", "open") for q in (Q_COARSE[tag], Q_FINE)] \
    + [("default", UNIT)]
N_CPU = {"default": 40, "layers14": 40, "open": 40, "l216": 150, "l430": 150}   # first ticks of the CPU check
TIE_IDS = ["%s-%s" % (t, "unit" if q is None else "q%g" % q) for t, q in TIE_LATTICES]
GOAL_STEP = 1     # virtual goal cost of one lateral step off the race line, in units of q
W_EXACT = [0.0, 0.5, 0.75]   # cost factors along the last solution that keep every factored cost a multiple of q / 4
VEL = dict(vel_max=100.0, gg_scale=1.0, local_gg=(5.0, 5.0), safety_d=30.0)


@functools.lru_cache(maxsize=None)
def tie_lattice(tag, q):
    """(lattice with quantised costs, q).  q = None: every edge costs 1.0 (q = 1)."""
    lat = H.lattice_for(tag)
    if q is None:
        q = 1.0
        cost = np.ones_like(lat.edge_cost)
    else:
        cost = np.round(lat.edge_cost / q) * q
    return dataclasses.replace(lat, edge_cost=cost, virt_goal_node_cost=GOAL_STEP * q / lat.lat_resolution), q


def _axm():
    return H.golden("ticks_default.npz")["ax_max_machines"]


def tie_scenarios(tag, n, seed):
    """seeded first-tick scenarios with 0-5 objects; every third one carries a blocked zone."""
    from graphbasedlocaltrajectoryplanner_b200.scenarios import Track, make_scenarios
    from oracle.gen_golden import make_zone
    lat = H.lattice_for(tag)
    trk = Track(H.track_csv_for(tag))
    sc = make_scenarios(trk, n, seed=seed, n_obj_min=0, n_obj_max=5, ahead=(20.0, 160.0),
                        s_max=(trk.length - 8.0) if tag == "open" else None)
    rng = np.random.default_rng(seed + 1)
    zones = [({"z%d" % b: make_zone(lat, rng, sc.pos[b])} if b % 3 == 2 else None) for b in range(n)]
    sc.set_zones(zones)
    return sc, zones


# ----------------------------------------------------------------------------------------------------------------------
# plain exact reference of one search
# ----------------------------------------------------------------------------------------------------------------------
class ExactSearch(object):
    """The layered search of OracleLTPL.search restated on integers (units of q / 4), keeping for every node the SET of
    in-edges that attain its minimum."""

    def __init__(self, lat, q):
        self.lat = lat
        self.unit = q / 4.0
        cu = lat.edge_cost / self.unit
        assert np.array_equal(cu, np.round(cu)), "edge costs are not multiples of q"
        self.cu = [int(c) for c in cu]
        self.goal = []
        for dn in range(lat.max_nodes_per_layer + 1):
            t = dn * lat.lat_resolution * lat.virt_goal_node_cost   # the oracle's / the kernel's operation order
            assert t == dn * GOAL_STEP * q and t / q == np.round(t / q), "goal term %r is not a multiple of q" % t
            self.goal.append(int(t / self.unit))

    def cost(self, e, cost_factor):
        c = self.cu[e]
        if cost_factor is not None and e in cost_factor:
            f = Fraction(cost_factor[e]) * c
            assert f.denominator == 1, "factored cost of edge %d is not a multiple of q / 4" % e
            c = int(f)
        return c

    @staticmethod
    def _pick(cands):
        """cands [(alt, own distance, id)] in scan order -> (min alt, picked id, ambiguous, decided)."""
        m = min(c[0] for c in cands)
        att = [c for c in cands if c[0] == m]
        dmin = min(c[1] for c in att)
        win = [c for c in att if c[1] == dmin]
        return m, win[0][2], len(win) > 1, len(win) < len(att)

    def search(self, start_node, goal_layer, range_layers, blocked, removed_layer=None, removed_lo=0, removed_hi=0,
               cost_factor=None, zone=None):
        """None, or dict(nodes, cost, ambiguous, n_amb, n_dec): n_amb nodes (incl. the goal) whose minimum is attained by
        two candidates with the same own distance, n_dec nodes where the smaller own distance decided an equal cost."""
        lt = self.lat
        sl, sn = start_node

        def absent(layer, j):
            return ((removed_layer is not None and layer == removed_layer and removed_lo <= j < removed_hi)
                    or bool(zone and (layer, j) in zone))
        if absent(sl, sn):
            return None
        layers = [sl]
        while layers[-1] != goal_layer:
            nxt = (layers[-1] + 1) % lt.num_layers
            if nxt not in range_layers:
                return None
            layers.append(nxt)
        dist = {sn: 0}
        parents = []
        n_amb = n_dec = 0
        for b in layers[1:]:
            nd, par = {}, {}
            for j in range(lt.nodes_in_layer(b)):
                if absent(b, j):
                    continue
                e0, cnt = lt.in_off[lt.node_off[b] + j]
                cands = []
                for e in range(e0, e0 + cnt):   # CSC order
                    i = int(lt.edge_src[e])
                    if i in dist and not (blocked is not None and e in blocked):
                        cands.append((dist[i] + self.cost(e, cost_factor), dist[i], i))
                if cands:
                    nd[j], par[j], amb, dec = self._pick(cands)
                    n_amb += amb
                    n_dec += dec
            if not nd:
                return None
            dist = nd
            parents.append(par)
        rl = int(lt.raceline_index[goal_layer])
        cost, gj, amb, dec = self._pick([(dist[j] + self.goal[abs(rl - j)], dist[j], j) for j in sorted(dist)])
        n_amb += amb
        n_dec += dec
        seq = [gj]
        for par in reversed(parents):
            seq.append(par[seq[-1]])
        seq.reverse()
        return dict(nodes=[[layers[k], seq[k]] for k in range(len(layers))], cost=cost, ambiguous=n_amb > 0,
                    n_amb=n_amb, n_dec=n_dec)

    def path_cost(self, nodes, cost_factor):
        lt = self.lat
        c = 0
        for k in range(1, len(nodes)):
            c += self.cost(lt.edge_id(nodes[k - 1][0], nodes[k - 1][1], nodes[k][1]), cost_factor)
        return c + self.goal[abs(int(lt.raceline_index[nodes[-1][0]]) - nodes[-1][1])]


def record_searches(orc):
    """wraps orc.search: every call with copies of its inputs and its result."""
    calls = []
    inner = orc.search

    def search(start_node, goal_layer, range_layers, blocked, **kw):
        out = inner(start_node, goal_layer, range_layers, blocked, **kw)
        kw = dict(kw)
        if kw.get("zone") is not None:
            kw["zone"] = frozenset(kw["zone"])
        if kw.get("cost_factor") is not None:
            kw["cost_factor"] = dict(kw["cost_factor"])
        calls.append(((list(start_node), goal_layer, frozenset(range_layers),
                       None if blocked is None else frozenset(blocked)), kw, out))
        return out
    orc.search = search
    return calls


def check_searches(ex, calls, ctx):
    """every recorded oracle search against the exact reference; returns the counts met."""
    n = dict(searches=0, found=0, flagged=0, ambiguities=0, decided=0)
    for args, kw, (nodes, tie) in calls:
        want = ex.search(*args, **kw)
        c = "%s: search from %s to layer %d (%s)" % (ctx, args[0], args[1],
                                                     ", ".join("%s=%s" % (k, v) for k, v in kw.items()
                                                               if k in ("removed_layer", "removed_lo", "removed_hi")))
        n["searches"] += 1
        assert (nodes is None) == (want is None), c + ": found %s, exact %s" % (nodes is not None, want is not None)
        if want is None:
            continue
        n["found"] += 1
        n["flagged"] += int(bool(tie))
        n["ambiguities"] += want["n_amb"]
        n["decided"] += want["n_dec"]
        got_cost = ex.path_cost(nodes, kw.get("cost_factor"))
        assert got_cost == want["cost"], c + ": path cost %d, exact minimum %d (units of q/4)" % (got_cost, want["cost"])
        assert nodes == want["nodes"], c + ": not the rule's pick\n got  %s\n want %s" % (nodes, want["nodes"])
        assert bool(tie) == want["ambiguous"], c + ": tie flag %s, exact rule %s (%d ambiguous nodes)" % (
            bool(tie), want["ambiguous"], want["n_amb"])
    return n


def assert_counts(n, tag, q, ctx):
    """non-vacuity: a coarse quantisation that produces no ties must fail.  On the unit-cost lattice every reached node
    of a layer has the same distance, so no tie there can be decided by the own distance.  q = 1 leaves few ties on the
    dense lattices and none on the sparse ones."""
    if q == Q_FINE:
        assert tag in ("l216", "l430") or n["decided"] >= 20, "%s: only %d decided ties met %s" % (ctx, n["decided"], n)
        return
    assert n["ambiguities"] >= 20, "%s: only %d ambiguous nodes met %s" % (ctx, n["ambiguities"], n)
    if q is not UNIT:
        assert n["decided"] >= 20, "%s: only %d decided ties met %s" % (ctx, n["decided"], n)
    assert n["flagged"] >= 1 and (q is UNIT or n["found"] > n["flagged"]), "%s: %s" % (ctx, n)


def _oracle(lat, online=None):
    from oracle.ltpl_oracle import OracleLTPL
    return OracleLTPL(lat, online=online)


# ----------------------------------------------------------------------------------------------------------------------
# CPU: the tie lattices and the oracle against the exact reference
# ----------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("tag,q", TIE_LATTICES, ids=TIE_IDS)
def test_tie_lattice_sums_are_exact(tag, q):
    from oracle.ltpl_oracle import OracleLTPL
    lat, qq = tie_lattice(tag, q)
    ex = ExactSearch(lat, qq)                                   # asserts costs and goal terms are multiples of q
    orc = OracleLTPL(lat)
    horizon = max(orc.end_layer_of(s)[1] for s in range(lat.num_layers))
    largest = horizon * float(lat.edge_cost.max()) + ex.goal[-1] * ex.unit
    assert largest < 2.0 ** 52 * qq
    if q is UNIT:
        assert np.all(lat.edge_cost == 1.0)
    else:
        assert np.all(np.abs(lat.edge_cost - H.lattice_for(tag).edge_cost) <= qq / 2)


@pytest.mark.parametrize("tag,q", TIE_LATTICES, ids=TIE_IDS)
def test_oracle_search_matches_exact_reference(tag, q):
    lat, qq = tie_lattice(tag, q)
    ex = ExactSearch(lat, qq)
    orc = _oracle(lat)
    calls = record_searches(orc)
    sc, zones = tie_scenarios(tag, N_CPU[tag], seed=515)
    for b in range(sc.size):                   # set_startpos + calc_paths: the searches of a first tick
        st = orc.set_startpos(np.asarray(sc.pos[b]), float(sc.heading[b]), float(sc.vel[b]))
        if st['in_track'] and st['cor_heading']:
            orc.calc_paths(st, orc.process_object_list(sc.object_list(b)), zones[b])
    n = check_searches(ex, calls, "%s q=%s" % (tag, q))
    print("%s q=%s: %s" % (tag, q, n))
    assert_counts(n, tag, q, "%s q=%s" % (tag, q))


def _crafted(lat, costs):
    """the lattice with every edge costing 100 + its id (no two alternatives tie) except `costs` {edge id: cost}, one
    unit of virtual goal cost per lateral step"""
    cost = 100.0 + np.arange(lat.num_edges, dtype=np.float64)
    for e, c in costs.items():
        cost[e] = c
    return dataclasses.replace(lat, edge_cost=cost, virt_goal_node_cost=1.0 / lat.lat_resolution)


def _out_edges(lat, layer, node):
    return {int(lat.edge_dst[e]): e for e in range(lat.edge_layer_off[layer], lat.edge_layer_off[layer + 1])
            if int(lat.edge_src[e]) == node}


def test_tie_flag_ignores_a_beaten_goal_tie():
    """goal scan: j = rl - 1 and rl + 1 with equal (cost, distance), then rl + 2 beats both -> no tie; without rl + 2
    the tie is at the final minimum -> flagged."""
    from oracle.ltpl_oracle import OracleLTPL
    lat0 = H.lattice_for("default")
    for sl in range(lat0.num_layers - 2):
        gl, rl = sl + 1, int(lat0.raceline_index[sl + 1])
        for sn in range(lat0.nodes_in_layer(sl)):
            out = _out_edges(lat0, sl, sn)
            if all(j in out for j in (rl - 1, rl + 1, rl + 2)):
                lat = _crafted(lat0, {out[rl - 1]: 10.0, out[rl + 1]: 10.0, out[rl + 2]: 0.0})
                ex = ExactSearch(lat, 1.0)
                orc = OracleLTPL(lat)
                for kw, pick, tie in ((dict(), rl + 2, False),
                                      (dict(removed_layer=gl, removed_lo=rl + 2, removed_hi=rl + 3), rl - 1, True)):
                    nodes, flag = orc.search([sl, sn], gl, {sl, gl}, None, **kw)
                    want = ex.search([sl, sn], gl, {sl, gl}, None, **kw)
                    assert nodes == want["nodes"] == [[sl, sn], [gl, pick]]
                    assert flag is tie and want["ambiguous"] is tie
                return
    pytest.fail("no node with successors rl - 1, rl + 1, rl + 2")


def test_tie_flag_ignores_a_beaten_relax_tie():
    """relax: the first two in-edges of a node (CSC order) tie in (cost, own distance), the third beats both -> no tie;
    with the third one blocked the tie is at the final minimum -> flagged."""
    from oracle.ltpl_oracle import OracleLTPL
    lat0 = H.lattice_for("default")
    for sl in range(lat0.num_layers - 3):
        for t in range(lat0.nodes_in_layer(sl + 2)):
            e0, cnt = lat0.in_off[lat0.node_off[sl + 2] + t]
            if cnt < 3:
                continue
            src = [int(lat0.edge_src[e]) for e in range(e0, e0 + 3)]
            for sn in range(lat0.nodes_in_layer(sl)):
                out = _out_edges(lat0, sl, sn)
                if not all(p in out for p in src):
                    continue
                # dist 5, 5, 0 at the sources; edge costs 5, 5, 0 into t: alt 10, 10 (tie), then 0
                lat = _crafted(lat0, {out[src[0]]: 5.0, out[src[1]]: 5.0, out[src[2]]: 0.0, e0: 5.0, e0 + 1: 5.0,
                                      e0 + 2: 0.0})
                ex = ExactSearch(lat, 1.0)
                orc = OracleLTPL(lat)
                gl = sl + 2
                for blocked, pick, tie in ((None, src[2], False), ({e0 + 2}, src[0], True)):
                    nodes, flag = orc.search([sl, sn], gl, {sl, sl + 1, gl}, blocked)
                    want = ex.search([sl, sn], gl, {sl, sl + 1, gl}, blocked)
                    assert nodes == want["nodes"] and nodes[1] == [sl + 1, pick] and nodes[2] == [gl, t], nodes
                    assert flag is tie and want["ambiguous"] is tie
                return
    pytest.fail("no node with three in-edges from successors of one node")


# ----------------------------------------------------------------------------------------------------------------------
# GPU: the device against the oracle on the tie lattices, flagged actions included
# ----------------------------------------------------------------------------------------------------------------------
def compare_strict(got, want, ctx):
    """tie flag, node sequence and node indices identical on EVERY action (flagged ones included), then the rules of
    H.compare_records."""
    assert bool(got["out_of_track"]) == bool(want["out_of_track"]), ctx + " out_of_track"
    if not want["out_of_track"]:
        assert sorted(got["paths"]) == sorted(want["paths"]), ctx + " action sets %s vs %s" % (sorted(got["paths"]),
                                                                                             sorted(want["paths"]))
        for act in want["paths"]:
            tg, tw = bool(got["tie"].get(act)), bool(want.get("tie", {}).get(act))
            assert tg == tw, "%s: tie flag of %s: device %s, oracle %s" % (ctx, act, tg, tw)
            gn = [[-1 if v is None else int(v) for v in p] for p in got["nodes"][act][0]]
            wn = [[-1 if v is None else int(v) for v in p] for p in want["nodes"][act][0]]
            assert gn == wn, "%s: node sequence of %s (tie %s) differs\n got  %s\n want %s" % (ctx, act, tw, gn, wn)
            assert np.asarray(got["node_idx"][act][0]).tolist() == np.asarray(want["node_idx"][act][0]).tolist(), \
                ctx + " node_idx " + act
    H.compare_records(got, want, ctx)


def _first_tick(pl, sc, vk):
    pl.set_vel_params(**vk)
    pl.stage_scenarios(sc)
    pl.upload()
    pl.set_startpos()
    pl.tick()
    return pl.records()


@pytest.mark.gpu
@pytest.mark.parametrize("tag,q", TIE_LATTICES, ids=TIE_IDS)
def test_device_matches_oracle_on_ties(tag, q):
    """first ticks: 0-5 objects (the overtake pair: snapshot resume on the default lattice, dp_run_pair on l216's
    <= 16 nodes per layer; the DENSE relax on the default lattice), zones on a third of the scenarios, 1-5 windows."""
    from graphbasedlocaltrajectoryplanner_b200.planner import BatchPlanner
    lat, qq = tie_lattice(tag, q)
    sc, zones = tie_scenarios(tag, 256, seed=8080 + TIE_LATTICES.index((tag, q)))
    pl = BatchPlanner(lat, device="cuda:0")
    pl.set_subbatches(1 + TIE_LATTICES.index((tag, q)) % 5)
    vk = dict(VEL, ax_max_machines=_axm())
    recs = _first_tick(pl, sc, vk)
    orc = _oracle(lat)
    calls = record_searches(orc)
    fails, acts, flagged = [], 0, 0
    for b in range(sc.size):
        want = orc.tick(sc.pos[b], sc.heading[b], sc.vel[b], sc.object_list(b), vk, blocked_zones=zones[b])
        try:
            compare_strict(recs[b], want, "%s q=%s scenario %d" % (tag, q, b))
        except AssertionError as e:
            fails.append(str(e)[:600])
        if not want["out_of_track"]:
            acts += len(want["paths"])
            flagged += sum(bool(want["tie"].get(a)) for a in want["paths"])
    overtake = sum(1 for _, kw, _ in calls if kw.get("removed_layer") is not None)
    n = check_searches(ExactSearch(lat, qq), calls, "%s q=%s" % (tag, q))
    print("%s q=%s: %d actions compared, %d tie-flagged, %d overtake searches; searches %s" % (
        tag, q, acts, flagged, overtake, n))
    assert not fails, "%d/%d scenarios differ:\n%s" % (len(fails), sc.size, "\n".join(fails[:6]))
    assert_counts(n, tag, q, "%s q=%s" % (tag, q))
    assert overtake >= 20 and acts > sc.size


@pytest.mark.gpu
@pytest.mark.parametrize("tag,q", TIE_LATTICES, ids=TIE_IDS)
def test_follow_table_matches_oracle(tag, q):
    """k_follow_table (built once per lattice): every row against the oracle's unblocked planning-range search from
    that node -- steps, tie bit (bit 8 of tab_reach), nodes and edge ids."""
    from graphbasedlocaltrajectoryplanner_b200.planner import BatchPlanner
    lat, _ = tie_lattice(tag, q)
    pl = BatchPlanner(lat, device="cuda:0")
    blob = pl.blob.cpu().numpy()
    h = pl.header
    nn, stride = lat.num_nodes, int(h.tab_stride)

    def arr(off, dtype, count):
        return blob[int(off): int(off) + np.dtype(dtype).itemsize * count].view(dtype)
    reach = arr(h.off_tab_reach, np.int32, nn)
    tnode = arr(h.off_tab_node, np.uint8, nn * stride).reshape(nn, stride)
    tedge = arr(h.off_tab_edge, np.int32, nn * stride).reshape(nn, stride)
    orc = _oracle(lat)
    node_layer = np.repeat(np.arange(lat.num_layers), np.diff(lat.node_off))
    fails, flagged, rows = [], 0, 0
    for g in range(nn):
        sl, sn = int(node_layer[g]), g - int(lat.node_off[node_layer[g]])
        end_layer, planning_dist = orc.end_layer_of(sl)
        assert planning_dist < 256, "%s: %d steps do not fit below the tie bit" % (tag, planning_dist)
        assert 0 <= reach[g] < 512, "%s row %d: tab_reach %#x" % (tag, g, reach[g])
        if planning_dist < 1 or planning_dist + 2 > stride:
            continue                             # k_plan flags such scenarios itself
        rng_l = set(orc.layers_in_range(sl, end_layer))
        steps, nodes, tie = planning_dist, None, False
        while steps >= 1:                        # the follow action's goal moves towards the vehicle (MOPG:203-220)
            nodes, tie = orc.search([sl, sn], (sl + steps) % lat.num_layers, rng_l, None)
            if nodes is not None:
                break
            steps -= 1
        want_steps = steps if nodes is not None else 0
        rows += 1
        try:
            assert reach[g] & 0xff == want_steps, "row %d (%d, %d): steps %d, oracle %d" % (g, sl, sn, reach[g] & 0xff,
                                                                                         want_steps)
            if want_steps:
                flagged += int(tie)
                assert bool(reach[g] >> 8) == bool(tie), "row %d (%d, %d): tie bit %d, oracle %s" % (
                    g, sl, sn, reach[g] >> 8, tie)
                assert tnode[g, :want_steps].tolist() == [p[1] for p in nodes[1:]], "row %d nodes" % g
                eids = [lat.edge_id(nodes[k][0], nodes[k][1], nodes[k + 1][1]) for k in range(want_steps)]
                assert tedge[g, :want_steps].tolist() == eids, "row %d edge ids" % g
        except AssertionError as e:
            fails.append(str(e))
    print("%s q=%s: %d follow-table rows compared, %d tie-flagged" % (tag, q, rows, flagged))
    assert not fails, "%s q=%s: %d/%d rows differ:\n%s" % (tag, q, len(fails), rows, "\n".join(fails[:8]))
    assert rows > nn // 2


@pytest.mark.gpu
@pytest.mark.parametrize("tag,w", [("default", W_EXACT), ("l216", W_EXACT), ("default", None), ("l216", None)],
                         ids=["default-exact-w", "l216-exact-w", "default-shipped-w", "l216-shipped-w"])
def test_closed_loop_on_ties_matches_session_oracle(tag, w):
    """8 stateful ticks on the coarse tie lattice against the session oracle without skipping flagged actions.  With
    w_last_edges = W_EXACT the factored costs stay exact, so the oracle's searches are also checked against the exact
    reference; with the shipped factors both sides make the same float64 roundings."""
    from graphbasedlocaltrajectoryplanner_b200 import capi
    from graphbasedlocaltrajectoryplanner_b200.planner import BatchPlanner
    from graphbasedlocaltrajectoryplanner_b200.scenarios import ScenarioBatch, Track, make_scenarios
    from oracle.gen_golden import advance_on_traj
    from oracle.ltpl_session import OracleSession
    lat, qq = tie_lattice(tag, Q_COARSE[tag])
    online = None if w is None else dict(w_last_edges=list(w))
    n_seq, n_ticks = 64, 8
    vel = dict(VEL, ax_max_machines=_axm())
    trk = Track(H.track_csv_for(tag))
    sc0 = make_scenarios(trk, n_seq, seed=3141, n_obj_min=0, n_obj_max=3)
    rng = np.random.default_rng(3142)
    prefer = (("right", "left", "straight", "follow"), ("follow", "straight", "left", "right"),
              ("left", "right", "follow", "straight"), ("straight", "follow", "right", "left"))
    pl = BatchPlanner(lat, online=online, device="cuda:0", stateful=True)
    pl.set_subbatches(3)
    pl.set_vel_params(**vel)

    class Clk(object):
        def __init__(self):
            self.t = 50.0

        def __call__(self):
            return self.t
    clks = [Clk() for _ in range(n_seq)]
    orcs = [_oracle(lat, online) for _ in range(n_seq)]
    calls = [record_searches(o) for o in orcs]
    ses = [OracleSession(orcs[q], clock=clks[q]) for q in range(n_seq)]
    objs = sc0.obj.copy()
    pos_est, vel_est = sc0.pos.copy(), sc0.vel.copy()
    sel = ["straight"] * n_seq
    cbuf = [[] for _ in range(n_seq)]
    alive = np.ones(n_seq, dtype=bool)
    fails, ticks_ok, acts, flagged, flagged_seq = [], 0, 0, 0, 0
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
                flagged_seq += int(not rec["out_of_track"])
                continue
            try:
                if k == 0:
                    assert ses[q].set_startpos(sc.pos[q], sc.heading[q], sc.vel[q]) is False
                paths = ses[q].calc_paths(sel[q], sc.object_list(q))
                traj, _ = ses[q].calc_vel_profile(sc.pos[q], float(vel_est[q]), **vel)
            except Exception:   # noqa: BLE001  (e.g. the reference's own brake-prefix failure)
                alive[q] = False
                continue
            try:
                assert sorted(rec["paths"]) == sorted(paths), "%s: paths %s vs %s" % (ctx, sorted(rec["paths"]),
                                                                                   sorted(paths))
                for act in paths:
                    tg, tw = bool(rec["tie"].get(act)), bool(ses[q].tie.get(act))
                    assert tg == tw, "%s: tie flag of %s: device %s, oracle %s" % (ctx, act, tg, tw)
                    acts += 1
                    flagged += int(tw)
                    nd = [[-1 if v is None else int(v) for v in p] for p in rec["nodes"][act][0]]
                    want = [[-1 if v is None else int(v) for v in p] for p in ses[q].m_nodes[act][0]] \
                        if act in ses[q].m_nodes else None
                    assert want is None or nd == want, "%s: nodes of %s (tie %s)\n got  %s\n want %s" % (
                        ctx, act, tw, nd, want)
                    assert rec["paths"][act][0].shape[0] == paths[act][0].shape[0], ctx + " path length " + act
                assert sorted(rec["traj"]) == sorted(traj), "%s: trajectories %s vs %s" % (ctx, sorted(rec["traj"]),
                                                                                        sorted(traj))
                for act in traj:
                    assert rec["traj"][act][0].shape == traj[act][0].shape, ctx + " rows " + act
                    H.assert_close("traj[%s]" % act, rec["traj"][act][0], traj[act][0],
                                   ("s", "x", "y", "psi", "kappa", "vx", "ax"), ctx)
                ticks_ok += 1
            except AssertionError as e:
                fails.append(str(e)[:600])
                alive[q] = False
                continue
            cand = [a for a in prefer[(q + k) % len(prefer)] if a in rec["traj"]]
            if not cand:
                alive[q] = False
                continue
            sel[q] = cand[0]
            last_traj[q] = rec["traj"][sel[q]][0]
    n = None
    if w is not None:
        ex = ExactSearch(lat, qq)
        n = dict(searches=0, found=0, flagged=0, ambiguities=0, decided=0)
        for q in range(n_seq):
            for key, v in check_searches(ex, calls[q], "%s sequence %d" % (tag, q)).items():
                n[key] += v
    print("%s w=%s: %d of %d ticks compared, %d actions, %d tie-flagged; exact searches %s" % (
        tag, w, ticks_ok, n_seq * n_ticks, acts, flagged, n))
    assert not fails, "%d sequences diverged (%d ticks matched):\n%s" % (len(fails), ticks_ok, "\n".join(fails[:6]))
    assert ticks_ok > n_seq * n_ticks // 2 and flagged >= 5, (ticks_ok, acts, flagged)
    assert flagged_seq <= n_seq // 20
    if n is not None:
        assert n["decided"] >= 20 and n["ambiguities"] >= 20, n


# ----------------------------------------------------------------------------------------------------------------------
# GPU: nearest-vertex argmins on exact ties
# ----------------------------------------------------------------------------------------------------------------------
def _d2(pts, p):
    """squared distances in the oracle's operation order (closest_path_index, GB:341, GIE:41)."""
    return np.power(pts[:, 0] - p[0], 2) + np.power(pts[:, 1] - p[1], 2)


def exact_midpoints(pts, pairs):
    """midpoints of the vertex pairs (a, b) whose nearest vertices are exactly a and b, tied in float64: [(pos, a, b)]"""
    out = []
    for a, b in pairs:
        p = (pts[a] + pts[b]) / 2.0
        d = _d2(pts, p)
        if d[a] == d[b] and np.count_nonzero(d == d.min()) == 2 and d[a] == d.min():
            out.append((p, a, b))
    return out


def tie_positions(lat):
    """exactly equidistant positions: start poses between two lattice nodes of consecutive layers, objects between two
    consecutive centre-line / reference-line vertices (incl. the seam of the closed track: last vertex vs vertex 0)."""
    L = lat.num_layers
    node_xy = np.column_stack((lat.node_x, lat.node_y))
    rl = lat.raceline_index
    pairs = []
    for l in range(L):                 # race line node of layer l against the nodes of layer l + 1 (and l + 1 -> l)
        a = int(lat.node_off[l] + rl[l])
        nxt = (l + 1) % L
        for j in range(lat.nodes_in_layer(nxt)):
            pairs.append((a, int(lat.node_off[nxt] + j)))
    starts = exact_midpoints(node_xy, pairs)
    bound1 = lat.refline + lat.normvec * np.expand_dims(lat.w_right, 1)
    bound2 = lat.refline - lat.normvec * np.expand_dims(lat.w_left, 1)
    center = (bound1 + bound2) / 2
    cl = exact_midpoints(center, [(i, (i + 1) % L) for i in range(L)])
    ref = exact_midpoints(lat.refline, [(i, (i + 1) % L) for i in range(L)])
    return starts, cl, ref, center


@pytest.mark.gpu
def test_nearest_vertex_ties_pick_the_first_minimum():
    from graphbasedlocaltrajectoryplanner_b200.planner import BatchPlanner
    from graphbasedlocaltrajectoryplanner_b200.scenarios import ScenarioBatch, Track
    from oracle.ltpl_oracle import OracleLTPL
    lat = H.lattice_for("default")
    L = lat.num_layers
    starts, cl, ref, center = tie_positions(lat)
    assert len(starts) >= 10 and len(cl) >= 10 and len(ref) >= 10, (len(starts), len(cl), len(ref))
    assert any(b == 0 for _, _, b in cl) or any(b == 0 for _, _, b in ref), "no tie at the seam of the closed track"
    assert not any(b < a for _, a, b in starts if b != 0)
    trk = Track(H.TRACK_CSV)
    pos, heading, vel, objs = [], [], [], []

    def ego_behind(i, gap):
        xy, psi, v = trk.raceline_pose(np.array([lat.s_raceline[i] - gap]))
        return xy[0], float(psi[0]), max(float(v[0]) * 0.5, 5.0)
    for p, a, b in starts:             # start pose between two nodes: the closest layer comes from the first minimum
        g = a if a < b else b
        layer = int(np.searchsorted(lat.node_off, g, side="right") - 1)
        gl = (layer + 2) % (L - 1)
        pos.append(p)
        heading.append(float(lat.node_psi[lat.node_off[gl] + lat.raceline_index[gl]]))
        vel.append(10.0)
        objs.append([])
    for p, a, b in cl + ref:           # a standing object between two vertices, 40 m in front of the ego
        i = min(a, b) if abs(a - b) == 1 else max(a, b)
        xy, psi, v = ego_behind(i, 40.0)
        pos.append(xy)
        heading.append(psi)
        vel.append(v)
        objs.append([{'id': 1, 'type': 'physical', 'X': float(p[0]), 'Y': float(p[1]), 'theta': psi, 'v': 0.0,
                      'length': 5.0, 'width': 2.5}])
    far = center[0] + np.array([3000.0, 3000.0])     # far from the track: the scans without a grid bound
    xy, psi, v = ego_behind(5, 40.0)
    pos += [far, xy]
    heading += [0.0, psi]
    vel += [10.0, v]
    objs += [[], [{'id': 1, 'type': 'physical', 'X': float(far[0]), 'Y': float(far[1]), 'theta': 0.0, 'v': 0.0,
                   'length': 5.0, 'width': 2.5}]]
    sc = ScenarioBatch.from_object_lists(np.array(pos), np.array(heading), np.array(vel), objs, k_max=1)
    vk = dict(VEL, ax_max_machines=_axm())
    pl = BatchPlanner(lat, device="cuda:0")
    pl.set_subbatches(2)
    recs = _first_tick(pl, sc, vk)
    orc = OracleLTPL(lat)
    fails, in_track = [], 0
    for b in range(sc.size):
        want = orc.tick(sc.pos[b], sc.heading[b], sc.vel[b], sc.object_list(b), vk)
        in_track += int(not want["out_of_track"])
        try:
            compare_strict(recs[b], want, "tie position %d" % b)
        except AssertionError as e:
            fails.append(str(e)[:600])
    print("nearest-vertex ties: %d start poses, %d centre-line, %d reference-line objects, %d in track" % (
        len(starts), len(cl), len(ref), in_track))
    assert not fails, "%d/%d scenarios differ:\n%s" % (len(fails), sc.size, "\n".join(fails[:6]))
    assert in_track >= sc.size // 2
