"""
TEST INFRASTRUCTURE -- NOT PRODUCT CODE.

CPU restatement (NumPy float64, scenario-at-a-time) of the reference's online per-tick planning path on the flat
lattice arrays of ``graphbasedlocaltrajectoryplanner_b200.lattice.Lattice``:

    set_startpos  ->  calc_paths  ->  calc_vel_profile            (first tick after set_startpos, i.e. stateless)

Every function cites the reference file:line it follows (paths relative to /root/reference; abbreviations as in
SURVEY.md: LTPL, OTH, MOPG, GLNT, GIE, GB, OLI, VPFB, CVPF).  The tph / igraph arithmetic comes from oracle/tph_port.py
(restated third-party semantics).  PINNING: tests/test_oracle_golden.py checks this file against tests/golden/*.npz,
which oracle/gen_golden.py produced by executing the reference's own Python files verbatim in the build container.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may import this module; the
product (graphbasedlocaltrajectoryplanner_b200/) never does.
"""

import bisect
import math

import numpy as np

from oracle import tph_port as tph

ACTIONS = ("straight", "follow", "left", "right")
ACTION_ID_MAP = {"straight": 0, "follow": 1, "left": 2, "right": 3}   # OTH:14-17


# ----------------------------------------------------------------------------------------------------------------------
# helper_funcs
# ----------------------------------------------------------------------------------------------------------------------
def closest_path_index(path, pos):
    """closest_path_index.py:24-30 (n_closest=1).  argpartition's tie order is undefined (q10) -> first minimum."""
    d2 = np.power(path[:, 0] - pos[0], 2) + np.power(path[:, 1] - pos[1], 2)
    return int(np.argmin(d2)), d2


def angle3pt(a, b, c):
    """get_s_coord.py:102-121"""
    ang = math.atan2(c[1] - b[1], c[0] - b[0]) - math.atan2(a[1] - b[1], a[0] - b[0])
    if ang > math.pi:
        ang -= 2 * math.pi
    elif ang <= -math.pi:
        ang += 2 * math.pi
    return ang


def get_s_coord(ref_line, pos, s_array=None, only_index=False, closed=False):
    """get_s_coord.py:8-99"""
    idx_nb = closest_path_index(ref_line, pos)[0]
    n = ref_line.shape[0]
    if closed:
        idx1 = idx_nb - 1
        idx2 = idx_nb + 1
        if idx2 > n - 1:
            idx2 = 0
    else:
        idx1 = max(idx_nb - 1, 0)
        idx2 = min(idx_nb + 1, n - 1)

    ang1 = abs(angle3pt(ref_line[idx_nb, :], pos, ref_line[idx1, :]))
    ang2 = abs(angle3pt(ref_line[idx_nb, :], pos, ref_line[idx2, :]))

    if not only_index:
        if ang1 > ang2:
            a_pos = ref_line[idx1, :]
            b_pos = ref_line[idx_nb, :]
        else:
            a_pos = ref_line[idx_nb, :]
            b_pos = ref_line[idx2, :]

        if s_array is None:
            s_array = np.cumsum(np.sqrt(np.sum(np.power(np.diff(ref_line, axis=0), 2), axis=1)))
        if s_array[0] > 0.05:
            s_array = np.insert(s_array, 0, 0.0)

        t = ((pos[0] - a_pos[0]) * (b_pos[0] - a_pos[0]) + (pos[1] - a_pos[1]) * (b_pos[1] - a_pos[1])) / \
            (np.power(b_pos[0] - a_pos[0], 2) + np.power(b_pos[1] - a_pos[1], 2))
        s_pos = [a_pos[0] + t * (b_pos[0] - a_pos[0]), a_pos[1] + t * (b_pos[1] - a_pos[1])]
        ds = np.sqrt(np.power(a_pos[0] - s_pos[0], 2) + np.power(a_pos[1] - s_pos[1], 2))

        if ang1 > ang2:
            s = s_array[idx1] + ds
        else:
            s = s_array[idx_nb] + ds
    else:
        s = None

    if ang1 >= ang2:
        closest_indexes = [idx1, idx_nb]
    else:
        closest_indexes = [idx_nb, idx2]
    return s, closest_indexes


def check_inside_bounds(bound1, bound2, pos):
    """check_inside_bounds.py:26-59"""
    centerline = (bound1 + bound2) / 2
    b_idx = get_s_coord(centerline, tuple(pos), only_index=True, closed=True)[1]
    b1 = np.column_stack((np.linspace(bound1[b_idx[0], 0], bound1[b_idx[1], 0]),
                          np.linspace(bound1[b_idx[0], 1], bound1[b_idx[1], 1])))
    b2 = np.column_stack((np.linspace(bound2[b_idx[0], 0], bound2[b_idx[1], 0]),
                          np.linspace(bound2[b_idx[0], 1], bound2[b_idx[1], 1])))
    cl = np.column_stack((np.linspace(centerline[b_idx[0], 0], centerline[b_idx[1], 0]),
                          np.linspace(centerline[b_idx[0], 1], centerline[b_idx[1], 1])))
    i = closest_path_index(cl, tuple(pos))[0]
    d_track_2 = np.power(b1[i, 0] - b2[i, 0], 2) + np.power(b1[i, 1] - b2[i, 1], 2)
    d_b1_2 = np.power(b1[i, 0] - pos[0], 2) + np.power(b1[i, 1] - pos[1], 2)
    d_b2_2 = np.power(b2[i, 0] - pos[0], 2) + np.power(b2[i, 1] - pos[1], 2)
    return not (d_b1_2 > d_track_2 or d_b2_2 > d_track_2)


# ----------------------------------------------------------------------------------------------------------------------
# online parameters (ltpl_config_online.ini as read at OTH:99-122, LTPL:168-173)
# ----------------------------------------------------------------------------------------------------------------------
DEFAULT_ONLINE = dict(max_heading_offset=0.8, v_max_offset=0.1, filt_window_width=1, w_last_edges=[0.0, 0.5, 0.8],
                      controller_type="PD", control_params={"c_p": 1.25, "k_d": 0.025, "k_p": 0.2}, delaycomp=0.1,
                      nmbr_export_points=115)


class VehObject(object):
    """OLI:240-295 (radius = length / 2, OLI:133; one constant-velocity prediction point at 0.2 s, OLI:121-127)."""

    def __init__(self, obj):
        self.pos = [obj['X'], obj['Y']]
        self.radius = obj['length'] / 2.0
        self.vel = obj['v']
        if 'prediction' in obj:
            self.prediction = np.asarray(obj['prediction'])
        else:
            dt = 0.2
            pred = np.zeros((1, 2))
            pred[0, 0] = obj['X'] - np.sin(obj['theta']) * obj['v'] * dt
            pred[0, 1] = obj['Y'] + np.cos(obj['theta']) * obj['v'] * dt
            self.prediction = pred


class OracleLTPL(object):
    """float64 restatement of one stateless planning tick of Graph_LTPL (LTPL:262-408)."""

    def __init__(self, lattice, online=None, veh_param_dyn_model_exp=1.0, veh_param_dragcoeff=0.85,
                 veh_param_mass=1000.0):
        self.lat = lattice
        self.p = dict(DEFAULT_ONLINE)
        if online:
            self.p.update(online)
        self.dyn_model_exp = veh_param_dyn_model_exp      # LTPL:189-192
        self.drag_coeff = veh_param_dragcoeff
        self.m_veh = veh_param_mass
        lt = lattice
        # OLI:70-72 / OTH:208-211
        self.bound1 = lt.refline + lt.normvec * np.expand_dims(lt.w_right, 1)
        self.bound2 = lt.refline - lt.normvec * np.expand_dims(lt.w_left, 1)
        self.node_xy = np.column_stack((lt.node_x, lt.node_y))
        self.node_layer = np.repeat(np.arange(lt.num_layers), np.diff(lt.node_off))
        self.edge_sl = lt.edge_start_layer()
        self.samp_xy = np.column_stack((lt.samp_x, lt.samp_y))
        self.samp_param = np.column_stack((lt.samp_x, lt.samp_y, lt.samp_psi, lt.samp_kappa, lt.samp_el))
        self.old_gg_scale = None     # VPFB:60,80-81

    # -- geometry helpers ---------------------------------------------------------------------------------------------------
    def node_pos(self, layer, node):
        g = self.lat.node_off[layer] + node
        return self.node_xy[g], self.lat.node_psi[g]

    # ----------------------------------------------------------------------------------------------------------------------
    # set_startpos  (LTPL:262-296 -> OTH.set_initial_pose OTH:181-270)
    # ----------------------------------------------------------------------------------------------------------------------
    def set_startpos(self, pos, heading, vel):
        lt = self.lat
        st = dict(v_start=vel, in_track=True, cor_heading=True)
        if not check_inside_bounds(self.bound1, self.bound2, pos):                # OTH:214-219
            st['in_track'] = False
            return st
        d2 = np.power(self.node_xy[:, 0] - pos[0], 2) + np.power(self.node_xy[:, 1] - pos[1], 2)   # GB:341
        closest_layer = int(self.node_layer[int(np.argmin(d2))])                 # GB:345 (argpartition, limit=1)
        goal_layer = (closest_layer + 2) % (lt.num_layers - 1)                     # OTH:226 (quirk q5)
        goal_node = int(lt.raceline_index[goal_layer])
        st['start_node'] = [goal_layer, goal_node]
        end_pos, end_heading = self.node_pos(goal_layer, goal_node)
        heading_diff = abs(heading - end_heading)                                 # OTH:234-240
        if heading_diff > np.pi:
            heading_diff = abs(2 * np.pi - heading_diff)
        if heading_diff > self.p['max_heading_offset']:
            st['cor_heading'] = False
            return st
        x_coeff, y_coeff, _, _ = tph.calc_splines(path=np.vstack((pos, end_pos)), psi_s=heading, psi_e=end_heading)
        path, inds, t_values, _ = tph.interp_splines(coeffs_x=x_coeff, coeffs_y=y_coeff,
                                                     stepsize_approx=lt.sampled_resolution, incl_last_point=True)
        psi, kappa = tph.calc_head_curv_an(coeffs_x=x_coeff, coeffs_y=y_coeff, ind_spls=inds, t_spls=t_values)
        el_lengths = np.sqrt(np.sum(np.power(np.diff(path, axis=0), 2), axis=1))   # OTH:259
        st['coeff'] = np.hstack((x_coeff, y_coeff))                                # OTH:265-268
        st['path_param'] = np.column_stack((path, psi, kappa, np.append(el_lengths, 0)))
        st['nodes'] = [[None, None], st['start_node']]
        st['node_idx'] = [0, path.shape[0] - 1]
        return st

    # ----------------------------------------------------------------------------------------------------------------------
    # object list  (OLI:75-153)
    # ----------------------------------------------------------------------------------------------------------------------
    def process_object_list(self, object_list):
        out = []
        for o in (object_list or []):
            if o.get('type', 'physical') != 'physical':
                continue
            if check_inside_bounds(self.bound1, self.bound2, [o['X'], o['Y']]):     # OLI:104-112
                out.append(VehObject(o))
        return out

    # ----------------------------------------------------------------------------------------------------------------------
    # planning range / layer helpers
    # ----------------------------------------------------------------------------------------------------------------------
    def end_layer_of(self, start_layer):
        """GLNT:104-142 ('distance' mode and 'layers' mode)."""
        lt = self.lat
        if lt.plan_horizon_mode == 'distance':
            des_dist = lt.s_raceline[start_layer] + lt.min_plan_horizon
            if des_dist > lt.s_raceline[-1]:
                if lt.closed:
                    des_dist -= lt.s_raceline[-1]
                else:
                    des_dist = lt.s_raceline[-1]
            end_layer = bisect.bisect_left(lt.s_raceline, des_dist)
        elif lt.plan_horizon_mode == 'layers':
            if lt.closed:
                end_layer = (start_layer + int(lt.min_plan_horizon)) % lt.num_layers
            else:
                end_layer = max((start_layer + int(lt.min_plan_horizon)), lt.num_layers - 1)   # quirk q7
        else:
            raise ValueError('Unsupported planning horizon mode "' + lt.plan_horizon_mode + '"!')
        planning_dist = end_layer - start_layer
        if planning_dist < 0:
            planning_dist = lt.num_layers - start_layer + end_layer
        return int(end_layer), int(planning_dist)

    def layers_in_range(self, start_layer, end_layer):
        """GB:704-709 layer set of the 'planning_range' filter (wrap when start >= end)."""
        if start_layer < end_layer:
            return list(range(start_layer, end_layer + 1))
        return list(range(start_layer, self.lat.num_layers)) + list(range(0, end_layer + 1))

    # ----------------------------------------------------------------------------------------------------------------------
    # obstacle -> blocked edges  (GIE:36-63, GB:567-646)
    # ----------------------------------------------------------------------------------------------------------------------
    def intersec_edges(self, obj_pos, obj_radius, plan_start, plan_end, range_layers):
        lt = self.lat
        lo = 1
        d2 = np.power(lt.refline[:, 0] - obj_pos[0], 2) + np.power(lt.refline[:, 1] - obj_pos[1], 2)
        obj_layer = int(np.argmin(d2))                       # GIE:42: min((val, idx)) == first minimum
        if not (plan_start - lo <= obj_layer <= plan_end + lo
                or (plan_start > plan_end and (plan_start - lo <= obj_layer or obj_layer <= plan_end + lo))):
            return [], None
        s_l = obj_layer - lo
        e_l = obj_layer + lo
        if s_l < 0:                                          # GB:597-600 (quirk q4: '>' instead of '>=')
            s_l += lt.num_layers
        if e_l > lt.num_layers:
            e_l -= lt.num_layers
        if s_l < e_l:
            lset = set(l for l in range(s_l, e_l + 1) if l < lt.num_layers)
        else:
            lset = set(list(range(s_l, lt.num_layers)) + list(range(0, e_l + 1)))
        lset &= range_layers                                  # active filter = planning_range (GLNT:177 remove_filters=False)
        ref = np.power(obj_radius + lt.veh_width / 2, 2) + np.power(lt.sampled_resolution, 2) / 4   # GB:626-629
        edges = []
        for a in sorted(lset):
            b = (a + 1) % lt.num_layers
            if b not in lset or (b == 0 and not lt.closed):
                continue
            for e in range(lt.edge_layer_off[a], lt.edge_layer_off[a + 1]):
                s0, s1 = lt.samp_off[e], lt.samp_off[e + 1]
                x = self.samp_xy[s0:s1, 0] - obj_pos[0]
                y = self.samp_xy[s0:s1, 1] - obj_pos[1]
                if np.any(x * x + y * y <= ref):             # GB:640-643
                    edges.append(e)
        return edges, obj_layer

    # ----------------------------------------------------------------------------------------------------------------------
    # gen_local_node_template  (GLNT:13-222)
    # ----------------------------------------------------------------------------------------------------------------------
    def zone_removed_nodes(self, start_node, blocked_zones):
        """GLNT:43-99 for the first tick after set_startpos: every zone is new (not processed, not disabled, not fixed).
        Returns the set {(layer, node)} removed by the 'overtaking_zones' filter.

        Graph_LTPL.calc_paths (LTPL:324-329) calls update_zone once per dict key, and update_zone (OLI:155-237) flags
        every zone that is not the one passed in as removed -- with more than one key the reference then fails in
        GLNT:69-83 (boolean index of the wrong length), so only a single zone per scenario is a defined input."""
        lt = self.lat
        if not blocked_zones:
            return set()
        if len(blocked_zones) != 1:
            raise NotImplementedError("more than one blocked zone per tick is not a defined input of the reference")
        zone = list(blocked_zones.values())[0]
        layer_ids = np.array(zone[0], dtype=np.int64)
        node_ids = np.array(zone[1], dtype=np.int64)
        n = 4                                                 # UNBLOCK_N_LAYERS_WHEN_IN_ZONE (GLNT:9)
        s0 = start_node[0]
        if (s0 + n) <= lt.num_layers:                         # GLNT:58-66 (quirk q6 in the wrap branch)
            u_l = np.logical_and(layer_ids >= s0, layer_ids < (s0 + n))
        else:
            u_l = np.logical_or(np.logical_and(layer_ids >= s0, layer_ids < lt.num_layers),
                                np.logical_and(layer_ids >= 0, layer_ids < ((s0 + n) % (lt.num_layers - 1) - 1)))
        if np.any(u_l):                                       # vehicle within the zone -> unblock (GLNT:70-77)
            layer_ids = layer_ids[~u_l]
            node_ids = node_ids[~u_l]
        return set(zip(layer_ids.tolist(), node_ids.tolist()))

    def gen_local_node_template(self, start_node, obj_veh):
        lt = self.lat
        start_layer = start_node[0]
        end_layer, planning_dist = self.end_layer_of(start_layer)
        range_layers = set(self.layers_in_range(start_layer, end_layer))
        blocked = set()
        closest_obj_layer_dist = None
        closest_obj_index = None
        closest_obj_node = None
        for idx, veh in enumerate(obj_veh):
            e, obj_layer = self.intersec_edges(veh.pos, veh.radius, start_layer, end_layer, range_layers)
            blocked.update(e)
            for pos_pred in veh.prediction:                  # GLNT:180-189: obj_layer overwritten (quirk q14)
                e, obj_layer = self.intersec_edges(pos_pred, veh.radius, start_layer, end_layer, range_layers)
                blocked.update(e)
            if obj_layer is not None:
                layer_dist = obj_layer - start_layer
                if layer_dist < 0:
                    layer_dist = lt.num_layers - start_layer + obj_layer
                if layer_dist <= planning_dist and (closest_obj_layer_dist is None
                                                    or layer_dist < closest_obj_layer_dist):
                    closest_obj_layer_dist = layer_dist
                    closest_obj_index = idx
                    closest_obj_node = [obj_layer, None]
        if closest_obj_layer_dist is not None:               # GLNT:206-213
            l = closest_obj_node[0]
            pos = self.node_xy[lt.node_off[l]:lt.node_off[l + 1]]
            op = obj_veh[closest_obj_index].pos
            d2 = np.power(pos[:, 0] - op[0], 2) + np.power(pos[:, 1] - op[1], 2)
            closest_obj_node[1] = int(np.argmin(d2))
        return end_layer, closest_obj_index, closest_obj_node, blocked, range_layers

    # ----------------------------------------------------------------------------------------------------------------------
    # graph search  (GB:854-929 search_graph_layer with virtual goal node; igraph Dijkstra semantics as a layered DP)
    # ----------------------------------------------------------------------------------------------------------------------
    def search(self, start_node, goal_layer, range_layers, blocked, removed_layer=None, removed_lo=0, removed_hi=0,
               cost_factor=None, zone=None):
        """returns (node list [[layer, node], ...] or None, tie_flag).

        nodes [removed_lo, removed_hi) of `removed_layer` are absent (MOPG:148-159); `blocked` = edge ids removed from
        the active filter (None for the un-blocked 'planning_range' graph); cost_factor = {edge id: factor} (GB:478-512).
        tie_flag: some node of the search, or its virtual goal, has its final (cost, own distance) minimum attained by
        two or more candidates (in-edges of a node, goal-layer nodes of the goal); ties a later candidate beats do not
        count.
        """
        lt = self.lat
        sl, sn = start_node
        if removed_layer is not None and sl == removed_layer and removed_lo <= sn < removed_hi:
            return None, False                               # GB:882-885 start node filtered
        if zone and (sl, sn) in zone:
            return None, False
        layers = [sl]
        l = sl
        while l != goal_layer:
            l = (l + 1) % lt.num_layers
            if l not in range_layers:
                return None, False
            layers.append(l)
        inf = math.inf
        dist = {sn: 0.0}
        parents = []
        tie = False
        for li in range(1, len(layers)):
            a, b = layers[li - 1], layers[li]
            nd = {}
            par = {}
            for j in range(lt.nodes_in_layer(b)):
                if removed_layer is not None and b == removed_layer and removed_lo <= j < removed_hi:
                    continue
                if zone and (b, j) in zone:                   # 'overtaking_zones' is the base of every other filter
                    continue
                g = lt.node_off[b] + j
                e0, cnt = lt.in_off[g]
                best = inf
                best_ds = inf
                best_i = -1
                tie_here = False
                for e in range(e0, e0 + cnt):
                    i = int(lt.edge_src[e])
                    ds = dist.get(i)
                    if ds is None or (blocked is not None and e in blocked):
                        continue
                    c = lt.edge_cost[e]
                    if cost_factor is not None and e in cost_factor:
                        c = c * cost_factor[e]
                    alt = ds + c
                    if alt < best or (alt == best and ds < best_ds):
                        best, best_ds, best_i = alt, ds, i
                        tie_here = False
                    elif alt == best and ds == best_ds:
                        tie_here = True
                tie = tie or tie_here
                if best_i >= 0:
                    nd[j] = best
                    par[j] = best_i
            if not nd:
                return None, tie
            dist = nd
            parents.append(par)
        # virtual goal node of the goal layer (GB:188: |raceline_index - n| * lat_resolution * w_virt_goal)
        rl = int(lt.raceline_index[goal_layer])
        best = inf
        best_ds = inf
        best_j = -1
        tie_here = False
        for j in sorted(dist):
            alt = dist[j] + abs(rl - j) * lt.lat_resolution * lt.virt_goal_node_cost
            if alt < best or (alt == best and dist[j] < best_ds):
                best, best_ds, best_j = alt, dist[j], j
                tie_here = False
            elif alt == best and dist[j] == best_ds:
                tie_here = True
        tie = tie or tie_here
        seq = [best_j]
        for par in reversed(parents):
            seq.append(par[seq[-1]])
        seq.reverse()
        return [[layers[k], int(seq[k])] for k in range(len(layers))], tie

    # ----------------------------------------------------------------------------------------------------------------------
    # main_online_path_gen  (MOPG:11-334)
    # ----------------------------------------------------------------------------------------------------------------------
    def main_online_path_gen(self, start_node, obj_veh, last_action_id, const_path_seg, pos_est, zone=None,
                             cost_factor=None):
        lt = self.lat
        end_layer, closest_obj_index, closest_obj_node, blocked, range_layers = \
            self.gen_local_node_template(start_node, obj_veh)

        obj_in_const_path = False
        object_besides_const_path = False
        if const_path_seg is not None and np.size(const_path_seg, axis=0) >= 2:      # MOPG:78-122
            pos_start = pos_est if pos_est is not None else const_path_seg[0, 0:2]
            s_start, _ = get_s_coord(lt.raceline, pos_start, lt.s_raceline, closed=True)
            s_end, _ = get_s_coord(lt.raceline, const_path_seg[-1, 0:2], lt.s_raceline, closed=True)
            smallest_obj_dist = np.inf
            for obj_idx, veh in enumerate(obj_veh):
                s_obj, _ = get_s_coord(lt.raceline, veh.pos, lt.s_raceline, closed=True)
                if s_start <= s_obj <= s_end or (s_start > s_end and (s_obj > s_start or s_obj < s_end)):
                    object_besides_const_path = True
                    if s_obj < s_start:
                        obj_dist = s_obj + lt.s_raceline[-1] - s_start
                    else:
                        obj_dist = s_obj - s_start
                    if closest_obj_index is None or obj_dist < smallest_obj_dist:      # quirk q15
                        closest_obj_index = obj_idx
                        smallest_obj_dist = obj_dist
                    obstacle_ref = np.power(veh.radius + lt.veh_width / 2, 2)
                    d2 = np.power(const_path_seg[:, 0] - veh.pos[0], 2) + np.power(const_path_seg[:, 1] - veh.pos[1], 2)
                    if any(d2 <= obstacle_ref):
                        obj_in_const_path = True

        # action sets (MOPG:124-174); filter tags: 'range' (un-blocked), 'default' (blocked edges removed),
        # 'left' / 'right' (default + node removal in the object's layer)
        if obj_in_const_path or object_besides_const_path:
            filters = ["range"]
            names = ["follow"]
            if not obj_in_const_path and (last_action_id == "left" or last_action_id == "right"):
                filters.append("default")
                names.append(last_action_id)
            elif not obj_in_const_path:
                filters.extend(["default", "default"])
                names.extend(["left", "right"])
        elif closest_obj_index is not None and closest_obj_node is not None:
            filters = ["range", "left", "right"]
            names = ["follow", "left", "right"]
        else:
            filters = ["default"]
            names = ["straight"]

        out = dict(nodes={}, node_idx={}, coeff={}, path_param={}, red_len={}, tie={})
        goal_layer = end_layer
        mod_goal = goal_layer
        for flt, name in zip(filters, names):
            kw = {}
            if flt == "range":
                blk = None
            else:
                blk = blocked
                if flt == "left":                             # MOPG:148-152: remove nodes [n_obj, n_l)
                    kw = dict(removed_layer=closest_obj_node[0], removed_lo=closest_obj_node[1],
                              removed_hi=lt.nodes_in_layer(closest_obj_node[0]))
                elif flt == "right":                          # MOPG:155-159: remove nodes [0, n_obj)
                    kw = dict(removed_layer=closest_obj_node[0], removed_lo=0, removed_hi=closest_obj_node[1])
            nodes = None
            tie = False
            while True:                                       # MOPG:203-220
                if mod_goal == start_node[0]:
                    break
                nodes, tie = self.search(start_node, mod_goal, range_layers, blk, zone=zone, cost_factor=cost_factor,
                                         **kw)
                if nodes is not None or not (name == "follow" or name == "straight"):
                    break
                mod_goal -= 1
                if mod_goal < 0:
                    mod_goal = lt.num_layers - 1

            reduced = (mod_goal != goal_layer or (not lt.closed and goal_layer == lt.num_layers - 1))   # MOPG:223-243
            if reduced:
                in_mod = (closest_obj_node is not None
                          and ((start_node[0] <= closest_obj_node[0] <= mod_goal)
                               or (start_node[0] > mod_goal
                                   and (closest_obj_node[0] >= start_node[0] or closest_obj_node[0] <= mod_goal))))
                if not obj_in_const_path and closest_obj_node is not None and not in_mod:
                    if name == "follow" or name == "straight":
                        name = "straight"
                    else:
                        nodes = None
            if nodes is None:
                continue

            # path assembly (MOPG:259-297)
            node_idx = [0]
            fuse = []
            dists = []
            eids = []
            for k in range(1, len(nodes)):
                e = lt.edge_id(nodes[k - 1][0], nodes[k - 1][1], nodes[k][1])
                eids.append(e)
                sp = self.samp_param[lt.samp_off[e]:lt.samp_off[e + 1]]
                lastseg = (k == len(nodes) - 1)
                fuse.append(sp if lastseg else sp[:-1])
                dists.append(lt.edge_len[e])
                tot = sum(f.shape[0] for f in fuse)
                node_idx.append(tot - 1 * lastseg)
            fuse = np.concatenate(fuse, axis=0).copy()
            dists = np.array(dists)

            psi_s = const_path_seg[-1, 2] if const_path_seg is not None else fuse[0, 2]      # MOPG:300-303
            cmat = np.column_stack(tph.calc_splines(path=fuse[node_idx, 0:2], psi_s=psi_s, psi_e=fuse[-1, 2],
                                                    el_lengths=dists)[0:2])
            fuse[:, 0:2], inds, tvals, _ = tph.interp_splines(coeffs_x=cmat[:, :4], coeffs_y=cmat[:, 4:],
                                                              incl_last_point=True,
                                                              stepnum_fixed=(np.diff(node_idx) + 1).tolist())
            fuse[:, 2], fuse[:, 3] = tph.calc_head_curv_an(coeffs_x=cmat[:, :4], coeffs_y=cmat[:, 4:],
                                                           ind_spls=inds, t_spls=tvals)
            out['nodes'][name] = [nodes]
            out['node_idx'][name] = [node_idx]
            out['coeff'][name] = [cmat]
            out['path_param'][name] = [fuse]
            out['red_len'][name] = [reduced]
            out['tie'][name] = tie
        return out, closest_obj_index

    # ----------------------------------------------------------------------------------------------------------------------
    # OTH.calc_paths, first tick after set_initial_pose  (OTH:289-516)
    # ----------------------------------------------------------------------------------------------------------------------
    def calc_paths(self, st, obj_veh, blocked_zones=None):
        action_id_sel = "straight"                            # forced action id (OTH:262-263, 313-315)
        last_pp = st['path_param']
        start_node = st['start_node']
        start_node_pos = self.node_pos(start_node[0], start_node[1])[0]             # OTH:398-404
        loc = closest_path_index(last_pp[:, 0:2], start_node_pos)[0]
        start_node_idx = st['nodes'].index(start_node)
        const_path_seg = last_pp[:loc + 1, :]

        zone = self.zone_removed_nodes(start_node, blocked_zones)
        res, closest_obj_index = self.main_online_path_gen(start_node, obj_veh, action_id_sel, const_path_seg, None,
                                                           zone=zone)

        for name in list(res['nodes'].keys()):                # OTH:433-472
            pp = res['path_param'][name][0]
            if loc > 0:
                pp = np.concatenate((last_pp[:loc, :], pp))
                if np.size(last_pp, axis=0) == loc:
                    j = loc - 1
                    pp[j, 4] = np.sqrt(np.power(np.diff(pp[j:j + 2, 0]), 2) + np.power(np.diff(pp[j:j + 2, 1]), 2))
                res['path_param'][name][0] = pp
            res['node_idx'][name][0] = np.concatenate((np.array(st['node_idx'][:start_node_idx]),
                                                       np.array(res['node_idx'][name][0]) + loc))
            if start_node_idx > 0:
                res['nodes'][name][0] = st['nodes'][:start_node_idx] + res['nodes'][name][0]
                res['coeff'][name][0] = np.concatenate((st['coeff'][:start_node_idx], res['coeff'][name][0]))

        if not res['nodes']:                                  # OTH:475-506 "track blocked"
            if const_path_seg.shape[0] > 2:
                loc += 1
                start_node_idx += 1
                res['path_param'][action_id_sel] = [last_pp[:loc, :]]
                res['node_idx'][action_id_sel] = [np.array(st['node_idx'][:start_node_idx])]
                res['nodes'][action_id_sel] = [st['nodes'][:start_node_idx]]
                res['coeff'][action_id_sel] = [st['coeff'][:start_node_idx]]
                res['red_len'][action_id_sel] = [True]
        res['closest_obj_index'] = closest_obj_index
        res['const_path_seg'] = const_path_seg
        return res

    # ----------------------------------------------------------------------------------------------------------------------
    # velocity planner wrappers (VPFB)
    # ----------------------------------------------------------------------------------------------------------------------
    def vp_calc_vel_profile(self, kappa, el_lengths, loc_gg, v_start, v_end, vk):
        """VPFB:194-227"""
        return tph.calc_vel_profile(loc_gg=loc_gg * vk['gg_scale'], ax_max_machines=vk['ax_max_machines'],
                                    v_max=vk['vel_max'], kappa=kappa, el_lengths=el_lengths, v_start=v_start,
                                    v_end=v_end, dyn_model_exp=self.dyn_model_exp, drag_coeff=self.drag_coeff,
                                    m_veh=self.m_veh, closed=False)

    def vp_check_brake_prefix(self, vel_plan, vel_course, kappa, el_lengths, loc_gg, vk):
        """VPFB:86-139"""
        if self.old_gg_scale is None:                         # VPFB:80-81 (update_dyn_parameters)
            self.old_gg_scale = vk['gg_scale']
        if vel_plan > (vk['vel_max'] + 0.1):
            gg_brake = loc_gg * self.old_gg_scale
            vx_decel = tph.calc_vel_profile_brake(loc_gg=gg_brake, kappa=kappa, el_lengths=el_lengths,
                                                  v_start=vel_plan, dyn_model_exp=self.dyn_model_exp,
                                                  drag_coeff=self.drag_coeff, m_veh=self.m_veh)
            idx = np.argmax(vx_decel <= vk['vel_max'])
            if idx == 0:
                idx = len(vx_decel) - 1
            vx_prefix = np.concatenate((vel_course, vx_decel[:idx]))
            return vx_prefix, int(idx), vx_decel[idx]
        self.old_gg_scale = vk['gg_scale']
        return vel_course, 0, vel_plan

    def calc_vel_profile_follow(self, kappa, el_lengths, loc_gg, v_start, v_ego, v_obj, safety_d, obj_dist, obj_pos,
                                vk):
        """CVPF:78-313 (called through VPFB:141-192 with loc_gg * gg_scale)."""
        lt = self.lat
        cp = self.p['control_params']
        loc_gg = loc_gg * vk['gg_scale']
        ax_max_machines = vk['ax_max_machines']
        v_max = vk['vel_max']
        ggv = np.atleast_2d([100.0, 14.0, 14.0])              # CVPF:134 (quirk q12)
        vel_bound_fulfilled = True
        control_d = cp['c_p'] * safety_d + lt.veh_length
        safety_d = safety_d + lt.veh_length
        too_close = (obj_dist - safety_d) < 0

        v_ego_brake = tph.calc_vel_profile_brake(loc_gg=loc_gg, kappa=kappa, el_lengths=el_lengths[:kappa.shape[0] - 1],
                                                 v_start=v_start, dyn_model_exp=self.dyn_model_exp,
                                                 drag_coeff=self.drag_coeff, m_veh=self.m_veh)
        id_brake = 0
        while id_brake < len(kappa) and v_ego_brake[id_brake] > 0.1:
            id_brake += 1
        ego_stop_dist = np.sum(el_lengths[0:id_brake])

        glob_rl = np.column_stack((lt.glob_rl[:-1], np.diff(lt.glob_rl[:, 0])))                    # CVPF:166
        s_opp, idxs_tmp = get_s_coord(glob_rl[:, 1:3], tuple(obj_pos), glob_rl[:, 0], closed=True)
        idx_s_opp = idxs_tmp[0]
        rolled = np.roll(glob_rl, glob_rl.shape[0] - idx_s_opp, axis=0)
        vel_start = min(v_obj, rolled[0, 4])
        v_opp_brake = tph.calc_vel_profile_brake(ggv=ggv, kappa=rolled[:, 3], el_lengths=rolled[:-1, 5],
                                                 v_start=vel_start, dyn_model_exp=self.dyn_model_exp,
                                                 drag_coeff=self.drag_coeff, m_veh=self.m_veh)
        id_brake = 0
        while id_brake < len(v_opp_brake) and v_opp_brake[id_brake] > 0.1:
            id_brake += 1
        opp_stop_dist = np.sum(rolled[0:id_brake, 5])

        s = np.concatenate(([0], np.cumsum(el_lengths[:-1])))
        stop_idx = 0
        s_stop = obj_dist - safety_d + opp_stop_dist
        while stop_idx < len(s) - 1 and s[stop_idx] < s_stop:
            stop_idx += 1
        v_end = 0.0
        if s_stop > s[-1]:
            s_loctraj_ends = opp_stop_dist - (s_stop - s[-1])
            idx = 0
            s_summed = 0.0
            while s_summed < s_loctraj_ends and idx < rolled.shape[0]:
                s_summed += rolled[idx, 5]
                idx += 1
            v_end = rolled[idx, 4]

        if self.p['controller_type'] == 'PD':                 # CVPF:65-67
            v_control = v_obj - cp['k_p'] * (control_d - obj_dist) + cp['k_d'] * (v_obj - v_ego)
        elif self.p['controller_type'] == 'PDtan':
            arg = min(max((control_d - obj_dist) * math.pi / 2 * 1 / cp['tan_w'], -math.pi / 2 + 1e-5),
                      math.pi / 2 - 1e-5)
            v_control = v_obj - math.tan(arg) * cp['k_p'] + cp['k_d'] * (v_obj - v_ego)
        else:
            raise ValueError('Unsupported control type')
        v_control = min(max(v_control, 0.0), v_max)

        if ego_stop_dist < s_stop:
            if v_start > v_control and stop_idx >= 2:
                vx_decel = v_ego_brake
                idx_c = min(int(np.argmax(vx_decel <= v_control)), stop_idx)
                if idx_c == 0:
                    idx_c = stop_idx
                vx_decel = vx_decel[:(idx_c + 1)]
                vx_control_start = vx_decel[-1]
            else:
                if not stop_idx >= 2:
                    vel_bound_fulfilled = False
                idx_c = 0
                vx_decel = []
                vx_control_start = v_start
            if (stop_idx - idx_c) > 0:
                vx_control = tph.calc_vel_profile(loc_gg=loc_gg[idx_c:(stop_idx + 1)], ax_max_machines=ax_max_machines,
                                                  v_max=v_control, kappa=kappa[idx_c:(stop_idx + 1)],
                                                  el_lengths=el_lengths[idx_c:stop_idx], v_start=vx_control_start,
                                                  v_end=v_end, dyn_model_exp=self.dyn_model_exp,
                                                  drag_coeff=self.drag_coeff, m_veh=self.m_veh, closed=False)
                if np.abs(vx_control[0] - vx_control_start) > 1.0:
                    vel_bound_fulfilled = False
            elif (stop_idx - idx_c) == 0:
                vx_control = [vx_control_start]
            else:
                vx_control = []
            vx_profile = np.concatenate((vx_decel[:-1], vx_control, [0.0] * (len(kappa) - stop_idx - 1)))
            if np.abs(vx_profile[0] - v_start) > 1.0:
                vel_bound_fulfilled = False
        else:
            vx_profile = v_ego_brake

        vx_compl = tph.calc_vel_profile(loc_gg=loc_gg, ax_max_machines=ax_max_machines, v_max=v_max, kappa=kappa,
                                        el_lengths=el_lengths[:-1], v_start=v_start, dyn_model_exp=self.dyn_model_exp,
                                        drag_coeff=self.drag_coeff, m_veh=self.m_veh, closed=False)
        return np.minimum(vx_profile, vx_compl), too_close, vel_bound_fulfilled

    def vel_one(self, action_id, pp, gg, end_node_in, red_len, vel_plan, vel_course, vel_est, closest_obj_index, obj_veh,
                pos_est, safety_d, vk):
        """velocity profile of ONE action's path `pp` (already cut at the ego position), OTH:733-941; returns
        (bp_out (P, 7) or [], vel_bound)."""
        lt = self.lat
        bp_out = []
        vel_bound = True
        if np.size(pp, axis=0) > 0:
            vel_idx = vel_course.shape[0]
            s = np.concatenate(([0], np.cumsum(pp[:-1, 4])))                      # OTH:743
            vx_prefix, pref_idx_add, vel_start = self.vp_check_brake_prefix(
                vel_plan, vel_course, pp[vel_idx:, 3], pp[vel_idx:-1, 4], gg[vel_idx:, :], vk)
            pref_idx = vel_idx + pref_idx_add

            if action_id == "follow":                     # OTH:763-830
                if closest_obj_index is None:
                    obj_dist = 0.0
                    c_obj_vel = 0.0
                    c_obj_pos = None
                else:
                    c_obj_pos = obj_veh[closest_obj_index].pos
                    c_obj_vel = obj_veh[closest_obj_index].vel
                    s_obj, _ = get_s_coord(pp[:, 0:2], c_obj_pos, np.cumsum(pp[:, 4]))
                    s_start, _ = get_s_coord(pp[:, 0:2], pos_est, np.cumsum(pp[:, 4]))
                    obj_dist = s_obj - s_start
                vx, too_close, vel_bound = self.calc_vel_profile_follow(
                    kappa=pp[pref_idx:, 3], el_lengths=pp[pref_idx:, 4], loc_gg=gg[pref_idx:, :],
                    v_start=vel_start, v_ego=vel_est, v_obj=c_obj_vel, safety_d=safety_d, obj_dist=obj_dist,
                    obj_pos=c_obj_pos, vk=vk)
                vx = np.concatenate((vel_course, vx))
                if vx.shape[0] > s.shape[0]:
                    vx = vx[0:len(s)]
                bp_out = np.column_stack((s, pp[:, 0:4], vx))

            if action_id != "follow" or (action_id == "follow" and red_len):   # OTH:834-923
                end_node = end_node_in
                num_el = len(pp[:, 4])
                raceline_index = lt.raceline_index[end_node[0]]
                raceline_offset = abs(end_node[1] - raceline_index) * lt.lat_offset      # quirk q3
                if red_len:
                    v_end = 0.0
                    spl_len = np.sum(pp[:-1, 4])
                    v_idx = np.argmin(np.cumsum(pp[:-1, 4]) < (spl_len - 5.0)) + 1
                    if v_idx == 1 and num_el > 1:
                        v_idx = num_el
                else:
                    v_end = lt.vel_raceline[end_node[0]]
                    v_end -= min(v_end * lt.vel_decrease_lat * raceline_offset, v_end)
                    v_idx = num_el
                if v_idx - pref_idx > 1:
                    vx = self.vp_calc_vel_profile(kappa=pp[pref_idx:v_idx, 3], el_lengths=pp[pref_idx:v_idx - 1, 4],
                                                  loc_gg=gg[pref_idx:v_idx, :], v_start=vel_start, v_end=v_end,
                                                  vk=vk)
                else:
                    vx = [0.0]
                if v_idx != num_el or v_idx <= 2:
                    vx = np.append(vx, [0.0] * (num_el - v_idx))
                vel_bound = True
                if not abs(vx[0] - vel_plan) < self.p['v_max_offset']:
                    vel_bound = False
                vx = np.concatenate((vel_course, vx))[:num_el]
                if action_id != "follow":
                    bp_out = np.column_stack((s, pp[:, 0:4], vx))
                else:
                    bp_out2 = np.column_stack((s, pp[:, 0:4], vx))
                    bp_out = np.where(bp_out[5, :] < bp_out2[5, :], bp_out, bp_out2)     # quirk q1

            vx_f = tph.conv_filt(signal=bp_out[:, 5], filt_window=self.p['filt_window_width'], closed=False)
            ax_f = tph.calc_ax_profile(vx_profile=vx_f, el_lengths=np.diff(bp_out[:, 0]))
            ax_f[np.logical_and(np.isclose(vx_f[:-1], 0.0), np.isclose(ax_f, 0.0))] = -5.0      # OTH:939
            bp_out = np.column_stack((bp_out[:, :-1], vx_f, np.append(ax_f, [0.0])))

        return bp_out, vel_bound

    # ----------------------------------------------------------------------------------------------------------------------
    # OTH.get_ref_idx + OTH.calc_vel_profile, first tick  (OTH:518-601, 603-1040)
    # ----------------------------------------------------------------------------------------------------------------------
    def calc_vel_profile(self, st, res, obj_veh, pos_est, vel_est, vel_max=100.0, gg_scale=1.0, local_gg=(5.0, 5.0),
                         ax_max_machines=np.atleast_2d([100.0, 5.0]), safety_d=30.0, incl_emerg_traj=False):
        lt = self.lat
        vk = dict(vel_max=vel_max, gg_scale=gg_scale, ax_max_machines=np.asarray(ax_max_machines, dtype=np.float64))
        # get_ref_idx, never planned before (OTH:590-599)
        vel_plan = st['v_start']
        vel_course = np.array([])
        if type(local_gg) is not dict and (type(local_gg) is not tuple or len(local_gg) != 2):   # OTH:649-653
            raise ValueError("Provided local_gg does not satisfy requested format! Read parameter documentation.")
        traj_base_id = 10                                      # OTH:669
        closest_obj_index = res['closest_obj_index']

        out_traj = {}
        out_ids = {}
        vel_bound_flags = {}
        gg_used = {}
        for action_id in list(res['path_param'].keys()):
            pp = res['path_param'][action_id][0]
            if type(local_gg) is dict:                         # location dependent friction, aligned with the path
                gg = np.asarray(local_gg[action_id][0], dtype=np.float64)
            else:
                gg = np.ones((pp.shape[0], 2)) * tuple(local_gg)  # OTH:665-666
            gg_used[action_id] = gg
            out_ids[action_id] = traj_base_id + ACTION_ID_MAP.get(action_id, 9)
            red_len = res['red_len'][action_id][0]
            bp_out, vel_bound = self.vel_one(action_id, pp, gg, res['nodes'][action_id][0][-1], red_len, vel_plan,
                                             vel_course, vel_est, closest_obj_index, obj_veh, pos_est, safety_d, vk)
            vel_bound_flags[action_id] = vel_bound
            # first tick: no backup plan exists (OTH:339-344) -> OTH:945-948 / 1007-1015
            if vel_bound or action_id in ["follow", "straight"]:
                out_traj[action_id] = [bp_out]
            # else: action set removed (vel constraints broken)

        if incl_emerg_traj and out_traj:                       # OTH:1027-1034 + calc_brake_emergency.py:9-47
            em_base = list(out_traj.keys())[0]
            traj = out_traj[em_base][0]
            el = np.diff(traj[:, 0])
            v_brake = tph.calc_vel_profile_brake(kappa=traj[:, 4], el_lengths=el, v_start=traj[0, 5], drag_coeff=0.854,
                                                 m_veh=1160.0, loc_gg=gg_used[em_base][:traj.shape[0]])   # OTH:1030
            idx_em = len(v_brake)
            a_brake = tph.calc_ax_profile(vx_profile=v_brake, el_lengths=el[:idx_em], eq_length_output=True)
            out_traj['emergency'] = [np.column_stack((traj[:idx_em, 0:5], v_brake, a_brake))]
            out_ids['emergency'] = out_ids[em_base]

        n_exp = self.p['nmbr_export_points']
        cut = {k: [v[0][:n_exp, :]] for k, v in out_traj.items()}       # LTPL:401-406
        return dict(traj_full=out_traj, traj=cut, ids={k: out_ids[k] for k in out_traj}, vel_bound=vel_bound_flags)

    # ----------------------------------------------------------------------------------------------------------------------
    # one stateless tick = set_startpos -> calc_paths -> calc_vel_profile  (main_min_example.py:69-104)
    # ----------------------------------------------------------------------------------------------------------------------
    def tick(self, pos, heading, vel, object_list, vel_kwargs=None, blocked_zones=None, vel_est=None, gg_fn=None):
        """gg_fn: location dependent friction, local_gg = {action: [gg_fn(path[:, 0:2])]} (OTH:649-666)."""
        vel_kwargs = dict(vel_kwargs or {})
        self.old_gg_scale = None
        st = self.set_startpos(np.asarray(pos, dtype=np.float64), float(heading), float(vel))
        if not (st['in_track'] and st['cor_heading']):
            return dict(out_of_track=True)
        obj_veh = self.process_object_list(object_list)
        res = self.calc_paths(st, obj_veh, blocked_zones)
        if gg_fn is not None:
            vel_kwargs['local_gg'] = {k: [gg_fn(v[0][:, 0:2])] for k, v in res['path_param'].items()}
        vp = self.calc_vel_profile(st, res, obj_veh, np.asarray(pos, dtype=np.float64),
                                   float(vel if vel_est is None else vel_est), **vel_kwargs)
        return dict(out_of_track=False, start_node=st['start_node'], paths=res['path_param'], nodes=res['nodes'],
                    node_idx=res['node_idx'], coeff=res['coeff'], red_len=res['red_len'], tie=res.get('tie', {}),
                    closest_obj_index=res['closest_obj_index'], const_path_seg=res['const_path_seg'],
                    traj_full=vp['traj_full'], traj=vp['traj'], ids=vp['ids'], vel_bound=vp['vel_bound'])
