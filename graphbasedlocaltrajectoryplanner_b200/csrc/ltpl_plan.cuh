// ltpl_plan.cuh -- k_startpos (set_initial_pose) and k_plan (object handling, edge blocking, action sets, layered DP).
// One WARP per scenario; all decisions in float64 (see ltpl_common.cuh).
#pragma once
#include "ltpl_common.cuh"

#define LTPL_KMAX 16          // object slots per scenario held in shared memory
#define LTPL_DMAX 32          // obstacle discs per scenario (one warp ballot): on-track vehicles + their prediction points
#define LTPL_WARPS_PER_CTA 4

// ---------------------------------------------------------------------------------------------------------------------
// k_startpos: Graph_LTPL.set_startpos -> OnlineTrajectoryHandler.set_initial_pose (OTH:181-270)
// ---------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ double cubic_rn(double a0, double a1, double a2, double a3, double t) {
    // a0 + a1 * t + a2 * pow(t, 2) + a3 * pow(t, 3), evaluated left to right (tph.interp_splines)
    double t2 = __dmul_rn(t, t);
    double t3 = __dmul_rn(t2, t);
    return __dadd_rn(__dadd_rn(__dadd_rn(a0, __dmul_rn(a1, t)), __dmul_rn(a2, t2)), __dmul_rn(a3, t3));
}

__device__ __forceinline__ void head_curv(double ax1, double ax2, double ax3, double ay1, double ay2, double ay3,
                                          double t, double* psi, double* kappa) {
    // tph.calc_head_curv_an
    double t2 = t * t;
    double xd = ax1 + 2 * ax2 * t + 3 * ax3 * t2;
    double yd = ay1 + 2 * ay2 * t + 3 * ay3 * t2;
    double xdd = 2 * ax2 + 6 * ax3 * t;
    double ydd = 2 * ay2 + 6 * ay3 * t;
    // tph.normalize_psi(atan2(y', x') - pi/2): the argument lies in [-3 pi / 2, pi / 2], where the modulo of the
    // reference is the identity and only the "< -pi -> + 2 pi" branch can fire
    // (the heading stays a float64 atan2: it becomes the boundary condition of the next spline, whose coefficients are
    // compared at 1e-6; q^-1.5 comes from a Newton-refined reciprocal square root instead of a float64 sqrt and division)
    double h = atan2(yd, xd) - LTPL_PI / 2;
    if (h < -LTPL_PI) h += 2 * LTPL_PI;
    *psi = h;
    const double q = xd * xd + yd * yd;
    const double r = fast_rsqrt(q);
    *kappa = (xd * ydd - yd * xdd) * (r * r * r);
}

__global__ void __launch_bounds__(LTPL_WARPS_PER_CTA * 32)
k_startpos(const LatDev lt, const LtplParams prm, const LtplDims dm, const LtplBuffers bf) {
    const int lane = threadIdx.x & 31;
    const int b = blockIdx.x * LTPL_WARPS_PER_CTA + (threadIdx.x >> 5);
    if (b >= dm.batch) return;
    const double px = bf.pos[2 * b], py = bf.pos[2 * b + 1], heading = bf.heading[b];
    int flags = 0;
    if (lane == 0) {
        bf.start_node[2 * b] = -1;
        bf.start_node[2 * b + 1] = -1;
        bf.const_len[b] = 0;
    }
    if (!inside_bounds(lt, px, py, lane)) {  // OTH:214-219
        if (lane == 0) bf.sc_flags[b] = LTPL_SC_OUT_OF_TRACK;
        return;
    }
    ArgMinD m = warp_closest_point(lt.node_xy, lt.Nn, px, py, lane);  // GB:341-345
    const int closest_layer = lt.node_layer[m.i];
    const int goal_layer = (closest_layer + 2) % (lt.L - 1);  // OTH:226 (quirk q5)
    const int goal_node = lt.rl_idx[goal_layer];
    const int g = lt.node_off[goal_layer] + goal_node;
    const double2 pe = lt.node_xy[g];
    const double psi_e = lt.node_psi[g];
    if (lane == 0) {
        bf.start_node[2 * b] = goal_layer;
        bf.start_node[2 * b + 1] = goal_node;
    }
    double hd = fabs(heading - psi_e);  // OTH:234-240
    if (hd > LTPL_PI) hd = fabs(2 * LTPL_PI - hd);
    if (hd > prm.max_heading_offset) {
        if (lane == 0) bf.sc_flags[b] = LTPL_SC_HEADING_MISMATCH;
        return;
    }
    // single-segment spline pose -> start node (tph.calc_splines N = 1, el = |P1 - P0|)
    const double dx = pe.x - px, dy = pe.y - py;
    const double el = sqrt(__dadd_rn(sq_rn(dx), sq_rn(dy)));
    const double ax0 = px, ay0 = py;
    const double ax1 = cos(heading + LTPL_PI / 2) * el, ay1 = sin(heading + LTPL_PI / 2) * el;
    const double ex1 = cos(psi_e + LTPL_PI / 2) * el, ey1 = sin(psi_e + LTPL_PI / 2) * el;
    const double ax2 = 3 * dx - 2 * ax1 - ex1, ay2 = 3 * dy - 2 * ay1 - ey1;
    const double ax3 = -2 * dx + ax1 + ex1, ay3 = -2 * dy + ay1 + ey1;
    // tph.calc_spline_lengths: 15-point polyline, summed like np.sum over 14 values
    double seg = 0.0;
    if (lane < 14) {
        double t0 = (lane == 0) ? 0.0 : lane * (1.0 / 14.0);
        double t1 = (lane == 13) ? 1.0 : (lane + 1) * (1.0 / 14.0);
        double x0 = cubic_rn(ax0, ax1, ax2, ax3, t0), y0 = cubic_rn(ay0, ay1, ay2, ay3, t0);
        double x1 = cubic_rn(ax0, ax1, ax2, ax3, t1), y1 = cubic_rn(ay0, ay1, ay2, ay3, t1);
        seg = sqrt(__dadd_rn(sq_rn(x1 - x0), sq_rn(y1 - y0)));
    }
    double r[14];
#pragma unroll
    for (int k = 0; k < 14; ++k) r[k] = __shfl_sync(LTPL_FULL, seg, k);
    double len = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]));
#pragma unroll
    for (int k = 8; k < 14; ++k) len += r[k];
    const int p0 = (int)ceil(len / lt.step) + 1;  // tph.interp_splines(stepsize_approx)
    if (p0 > dm.p0_max || p0 < 2) {
        if (lane == 0) bf.sc_flags[b] = LTPL_SC_CAPACITY;
        return;
    }
    const double dstep = len / (double)(p0 - 1);
    const size_t plane = (size_t)dm.batch * dm.p0_max;
    double* cs = bf.const_seg + (size_t)b * dm.p0_max;
    #pragma unroll 1
    for (int k = lane; k < p0; k += 32) {
        double t, x, y, tn, xn, yn;
        if (k < p0 - 1) {
            t = (k * dstep) / len;
            x = cubic_rn(ax0, ax1, ax2, ax3, t);
            y = cubic_rn(ay0, ay1, ay2, ay3, t);
        } else {
            t = 1.0;
            x = ((ax0 + ax1) + ax2) + ax3;
            y = ((ay0 + ay1) + ay2) + ay3;
        }
        double elk = 0.0;
        if (k < p0 - 1) {
            if (k + 1 < p0 - 1) {
                tn = ((k + 1) * dstep) / len;
                xn = cubic_rn(ax0, ax1, ax2, ax3, tn);
                yn = cubic_rn(ay0, ay1, ay2, ay3, tn);
            } else {
                xn = ((ax0 + ax1) + ax2) + ax3;
                yn = ((ay0 + ay1) + ay2) + ay3;
            }
            elk = sqrt(__dadd_rn(sq_rn(xn - x), sq_rn(yn - y)));  // OTH:259
        }
        double psi, kap;
        head_curv(ax1, ax2, ax3, ay1, ay2, ay3, t, &psi, &kap);
        cs[0 * plane + k] = x;
        cs[1 * plane + k] = y;
        cs[2 * plane + k] = psi;
        cs[3 * plane + k] = kap;
        cs[4 * plane + k] = elk;
    }
    if (lane == 0) {
        bf.sc_flags[b] = flags;
        bf.const_len[b] = p0;
        double* cc = bf.const_coeff + (size_t)b * 8;
        cc[0] = ax0; cc[1] = ax1; cc[2] = ax2; cc[3] = ax3;
        cc[4] = ay0; cc[5] = ay1; cc[6] = ay2; cc[7] = ay3;
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// layered shortest-path DP (igraph Dijkstra semantics on the layered DAG: GB:818-821, 854-929)
// ---------------------------------------------------------------------------------------------------------------------
struct DpCtx {
    double* dist;        // [2][maxn]
    double* dsave;       // [maxn] dist after step snap_li: prefix shared by the overtake-left / -right searches
    unsigned char* pred; // [hl][maxn]  predecessor (node index in the layer before) of the node, 255 = unreachable
    const int4* meta;    // [hl] per layer step li: (first node of the next layer, #nodes, first edge of the pair, #edges)
    int maxn;
    int cur;             // which half of dist holds the last completed layer
    int layer;           // lattice layer of the last completed step
    int tie;             // some node's final (cost, own distance) minimum has two in-edges (igraph's pick then depends
                         // on heap order)
    int snap_li;         // step whose result dsave holds (0: no snapshot)
    int tie_save;        // tie flag at the snapshot
    int fe0, fe1, fe2;   // stateful tick: edges of the last solution whose cost is scaled (GLNT:155-162), -1: none
    double ff0, ff1, ff2;
};

// planning range (GLNT:104-142): layer the plan has to reach from start_layer
__device__ __forceinline__ int plan_end_layer(const LatDev& lt, int start_layer, int lane) {
    if (lt.plan_mode == 0) {
        double des = __dadd_rn(lt.s_rl[start_layer], lt.min_plan_horizon);
        const double s_last = lt.s_rl[lt.L - 1];
        if (des > s_last) {
            if (lt.closed)
                des = __dsub_rn(des, s_last);
            else
                des = s_last;
        }
        // bisect.bisect_left(s_raceline, des): first index with s >= des
        int cnt = 0;
        #pragma unroll 1
        for (int i = lane; i < lt.L; i += 32) cnt += (lt.s_rl[i] < des) ? 1 : 0;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(LTPL_FULL, cnt, o);
        return cnt;
    }
    const int hz = (int)lt.min_plan_horizon;
    if (lt.closed) return (start_layer + hz) % lt.L;
    return max(start_layer + hz, lt.L - 1);  // quirk q7
}

// per-step lattice offsets of the planning range (shared by all searches of a scenario)
__device__ __forceinline__ void dp_fill_meta(const LatDev& lt, int lane, int4* meta, int start_layer, int planning_dist) {
    #pragma unroll 1
    for (int li = 1 + lane; li <= planning_dist; li += 32) {
        int lay = start_layer + li - 1;
        if (lay >= lt.L) lay -= lt.L;
        const int nxt = (lay + 1 >= lt.L) ? 0 : lay + 1;
        const int nb = lt.node_off[nxt], e0 = lt.edge_layer_off[lay];
        meta[li] = make_int4(nb, lt.node_off[nxt + 1] - nb, e0, lt.edge_layer_off[lay + 1] - e0);
    }
    __syncwarp();
}

// blocked zones, first tick (GLNT:43-99): a new zone that overlaps the next UNBLOCK_N_LAYERS_WHEN_IN_ZONE = 4 layers from
// the start layer is unblocked on those layers (GLNT:58-77; the wrap branch keeps the reference's arithmetic, quirk q6)
__device__ __forceinline__ bool zone_unblocked(int l, int s0, int L) {
    const int n = 4;
    if (s0 + n <= L) return l >= s0 && l < s0 + n;
    return (l >= s0 && l < L) || (l >= 0 && l < ((s0 + n) % (L - 1) - 1));
}

// Runs the layer transitions li_begin .. n_steps; returns the number of completed steps (last layer with a reachable
// node).  li_begin == 1 starts at start_node; li_begin > 1 resumes from the snapshot in c.dsave (the pred rows below
// li_begin are those of the run that took the snapshot).  After step snap_at the state is saved to c.dsave.
// Each lane owns one node of the next layer and scans its in-edges IN CSC ORDER, which keeps igraph's relaxation order
// and tie rule (strict <, then smaller dist[src]) bit for bit.
// DENSE: lattices with several in-edges per node keep two edge records in flight (6 % on the shipped lattice); sparse ones
// (mostly 0 or 1 in-edge: the "216 x 11" / "430 x 21" parameter sets) run the plain loop, which is faster there
template <bool ZONE, bool COSTF = false, bool DENSE = false>
__device__ __forceinline__ int dp_run(const LatDev& lt, int lane, DpCtx& c, int start_layer, int start_node, int n_steps,
                                      const unsigned* mask, int e_base, int rem_layer, int rem_lo, int rem_hi,
                                      int li_begin, int snap_at, const unsigned* zone, int zone_s0 = -1) {
    const int maxn = c.maxn;
    int tie = 0;
    if (li_begin == 1) {
        #pragma unroll 1
        for (int j = lane; j < maxn; j += 32) c.dist[j] = (j == start_node) ? 0.0 : LTPL_INF;
    } else {
        #pragma unroll 1
        for (int j = lane; j < maxn; j += 32) c.dist[j] = c.dsave[j];
        tie = c.tie_save;
    }
    __syncwarp();
    int cur = 0, reach = li_begin - 1;
    int layer = start_layer + li_begin - 1;
    if (layer >= lt.L) layer -= lt.L;
    #pragma unroll 1
    for (int li = li_begin; li <= n_steps; ++li) {
        int nxt = layer + 1;
        if (nxt >= lt.L) nxt = 0;
        const int4 mt = c.meta[li];
        const int nbase = mt.x, nl = mt.y;
        const int moff = (mt.z >= e_base) ? -e_base : lt.E - e_base;  // edge id -> bit of the window mask
        // 'overtaking_zones' is the base of every other filter (GLNT:96-99, 144-147): zone nodes are absent everywhere
        const unsigned* zs = (ZONE && zone && !zone_unblocked(nxt, zone_s0, lt.L)) ? zone : nullptr;
        const double* dcur = c.dist + cur * maxn;
        double* dnxt = c.dist + (cur ^ 1) * maxn;
        int any = 0;
        #pragma unroll 1
        for (int j = lane; j < maxn; j += 32) {
            double best = LTPL_INF, best_ds = LTPL_INF;
            int best_k = 255;   // start-layer node index of the chosen in-edge (255: unreachable)
            int tie_here = 0;   // the current (best, best_ds) is attained by a second in-edge
            bool present = j < nl && !(nxt == rem_layer && j >= rem_lo && j < rem_hi);
            if (ZONE && present && zs) present = !((zs[(nbase + j) >> 5] >> ((nbase + j) & 31)) & 1u);
            if (present) {
                const int2 io = lt.in_off[nbase + j];
                auto relax = [&](const LtplEdgeRec& r, int e) {
                    const double ds = dcur[r.src];
                    if (!(ds < LTPL_INF)) return;
                    if (mask) {
                        const int idx = e + moff;
                        if ((mask[idx >> 5] >> (idx & 31)) & 1u) return;
                    }
                    double cost = r.cost;
                    if (COSTF) {   // offline_cost *= factor on this tick's copy of the planning range (GB:505-508)
                        if (e == c.fe0) cost = __dmul_rn(cost, c.ff0);
                        else if (e == c.fe1) cost = __dmul_rn(cost, c.ff1);
                        else if (e == c.fe2) cost = __dmul_rn(cost, c.ff2);
                    }
                    const double alt = __dadd_rn(ds, cost);
                    if (alt < best || (alt == best && ds < best_ds)) {
                        best = alt;
                        best_ds = ds;
                        best_k = r.src;
                        tie_here = 0;
                    } else if (alt == best && ds == best_ds) {
                        tie_here = 1;
                    }
                };
                // in-edges in CSC order (igraph's relaxation order); nodes with many in-edges keep two records in flight
                int k = 0;
                #pragma unroll 1
                for (; DENSE && k + 1 < io.y; k += 2) {
                    const LtplEdgeRec ra = lt.edge_rec[io.x + k], rb = lt.edge_rec[io.x + k + 1];
                    relax(ra, io.x + k);
                    relax(rb, io.x + k + 1);
                }
                #pragma unroll 1
                for (; k < io.y; ++k) relax(lt.edge_rec[io.x + k], io.x + k);
            }
            tie |= tie_here;
            dnxt[j] = best;
            c.pred[li * maxn + j] = (unsigned char)best_k;
            any |= (best_k != 255);
        }
        any = __any_sync(LTPL_FULL, any);
        __syncwarp();
        if (!any) break;
        cur ^= 1;
        reach = li;
        layer = nxt;
        if (li == snap_at) {
            #pragma unroll 1
            for (int j = lane; j < maxn; j += 32) c.dsave[j] = dnxt[j];
            c.tie_save = __any_sync(LTPL_FULL, tie) ? 1 : 0;
            c.snap_li = li;
        }
    }
    c.cur = cur;
    c.layer = layer;
    c.tie = __any_sync(LTPL_FULL, tie) ? 1 : 0;
    return reach;
}

// The 'overtake_left' / 'overtake_right' pair (MOPG:148-159) on lattices with <= 16 nodes per layer: the two searches only
// differ in which nodes of the object's layer are removed, and a layer leaves half of the warp idle -- lanes 0-15 carry
// the search without the nodes [split, n_l) (left), lanes 16-31 the one without [0, split) (right), in ONE loop over the
// layers.  Halves of the dist rows / pred rows at offset 16 hold the second search.  Returns the steps of the first
// search; *reach_b, *tie_b those of the second.
template <bool ZONE, bool COSTF>
__device__ __forceinline__ int dp_run_pair(const LatDev& lt, int lane, DpCtx& c, int start_layer, int start_node,
                                           int n_steps, const unsigned* mask, int e_base, int rem_layer, int split,
                                           const unsigned* zone, int zone_s0, int* reach_b, int* tie_b) {
    const int maxn = c.maxn;   // 32
    const int half = lane >> 4, j = lane & 15, hoff = half << 4;
    int tie = 0;
    c.dist[lane] = (j == start_node) ? 0.0 : LTPL_INF;
    __syncwarp();
    int cur = 0, reach_a = 0, reach_2 = 0;
    int layer = start_layer;
    #pragma unroll 1
    for (int li = 1; li <= n_steps; ++li) {
        int nxt = layer + 1;
        if (nxt >= lt.L) nxt = 0;
        const int4 mt = c.meta[li];
        const int nbase = mt.x, nl = mt.y;
        const int moff = (mt.z >= e_base) ? -e_base : lt.E - e_base;
        const unsigned* zs = (ZONE && zone && !zone_unblocked(nxt, zone_s0, lt.L)) ? zone : nullptr;
        const double* dcur = c.dist + cur * maxn + hoff;
        double* dnxt = c.dist + (cur ^ 1) * maxn + hoff;
        double best = LTPL_INF, best_ds = LTPL_INF;
        int best_k = 255, tie_here = 0;
        bool present = j < nl && !(nxt == rem_layer && (half ? (j < split) : (j >= split)));
        if (ZONE && present && zs) present = !((zs[(nbase + j) >> 5] >> ((nbase + j) & 31)) & 1u);
        if (present) {
            const int2 io = lt.in_off[nbase + j];
            #pragma unroll 1
            for (int k = 0; k < io.y; ++k) {
                const int e = io.x + k;
                const LtplEdgeRec r = lt.edge_rec[e];
                const double ds = dcur[r.src];
                if (!(ds < LTPL_INF)) continue;
                if (mask) {
                    const int idx = e + moff;
                    if ((mask[idx >> 5] >> (idx & 31)) & 1u) continue;
                }
                double cost = r.cost;
                if (COSTF) {
                    if (e == c.fe0) cost = __dmul_rn(cost, c.ff0);
                    else if (e == c.fe1) cost = __dmul_rn(cost, c.ff1);
                    else if (e == c.fe2) cost = __dmul_rn(cost, c.ff2);
                }
                const double alt = __dadd_rn(ds, cost);
                if (alt < best || (alt == best && ds < best_ds)) {
                    best = alt;
                    best_ds = ds;
                    best_k = r.src;
                    tie_here = 0;
                } else if (alt == best && ds == best_ds) {
                    tie_here = 1;
                }
            }
        }
        tie |= tie_here;
        dnxt[j] = best;
        c.pred[li * maxn + lane] = (unsigned char)best_k;
        const unsigned alive = __ballot_sync(LTPL_FULL, best_k != 255);
        __syncwarp();
        if (!alive) break;
        // a search without a reachable node in this layer has none in any later layer either (all its distances are inf)
        if ((alive & 0xffffu) && reach_a == li - 1) reach_a = li;
        if ((alive >> 16) && reach_2 == li - 1) reach_2 = li;
        cur ^= 1;
        layer = nxt;
    }
    c.cur = cur;
    c.layer = layer;
    const unsigned tb = __ballot_sync(LTPL_FULL, tie != 0);
    c.tie = (tb & 0xffffu) ? 1 : 0;
    *tie_b = (tb >> 16) ? 1 : 0;
    *reach_b = reach_2;
    return reach_a;
}

// the lattice edge (src node js of the layer before) -> (node jd of the layer whose first node is nbase); the lattice
// holds at most one edge per node pair
__device__ __forceinline__ int dp_edge_id(const LatDev& lt, int nbase, int jd, int js) {
    const int2 io = lt.in_off[nbase + jd];
    int e = io.x;
    #pragma unroll 1
    for (int k = 0; k < io.y; ++k)
        if (lt.edge_src[io.x + k] == js) e = io.x + k;
    return e;
}

// virtual goal node: argmin_j dist[j] + |raceline_index - j| * lat_resolution * w_virt_goal (GB:188)
__device__ __forceinline__ int dp_goal(const LatDev& lt, int lane, const DpCtx& c, int* tie_out, int off = 0) {
    const int layer = c.layer;
    const int nl = lt.node_off[layer + 1] - lt.node_off[layer];
    const int rl = lt.rl_idx[layer];
    const double* d = c.dist + c.cur * c.maxn + off;   // off = 16: the second search of dp_run_pair
    double best = LTPL_INF, best_ds = LTPL_INF;
    int best_j = 0x7fffffff, tie = 0;
    #pragma unroll 1
    for (int j = lane; j < nl; j += 32) {
        const double ds = d[j];
        if (!(ds < LTPL_INF)) continue;
        int dn = rl - j;
        if (dn < 0) dn = -dn;
        const double alt = __dadd_rn(ds, __dmul_rn(__dmul_rn((double)dn, lt.lat_res), lt.virt_cost));
        if (alt < best || (alt == best && ds < best_ds)) {
            best = alt;
            best_ds = ds;
            best_j = j;
            tie = 0;   // a tie with a candidate this lane has since beaten does not count
        } else if (alt == best && ds == best_ds) {
            tie = 1;
        }
    }
    // lexicographic minimum of (alt, dist, j) over the lanes; costs are >= 0, so their bit patterns order like the values
    // and every key is two 32-bit warp reductions
    const unsigned long long ua = (unsigned long long)__double_as_longlong(best);
    const unsigned long long ud = (unsigned long long)__double_as_longlong(best_ds);
    const unsigned ah = __reduce_min_sync(LTPL_FULL, (unsigned)(ua >> 32));
    bool in = ((unsigned)(ua >> 32) == ah);
    const unsigned al = __reduce_min_sync(LTPL_FULL, in ? (unsigned)ua : 0xffffffffu);
    in = in && ((unsigned)ua == al);
    const unsigned dh = __reduce_min_sync(LTPL_FULL, in ? (unsigned)(ud >> 32) : 0xffffffffu);
    in = in && ((unsigned)(ud >> 32) == dh);
    const unsigned dl = __reduce_min_sync(LTPL_FULL, in ? (unsigned)ud : 0xffffffffu);
    in = in && ((unsigned)ud == dl) && (best < LTPL_INF);
    const unsigned win = __ballot_sync(LTPL_FULL, in);
    const unsigned gj = __reduce_min_sync(LTPL_FULL, in ? (unsigned)best_j : 0x7fffffffu);
    // tie: the minimum is attained by several goal-layer nodes, across lanes or within a winning lane
    if (__popc(win) > 1 || __any_sync(LTPL_FULL, tie && in)) *tie_out = 1;
    return (int)gj;
}

// ---------------------------------------------------------------------------------------------------------------------
// k_plan: OLI.process_object_list + gen_local_node_template + main_online_path_gen (action sets + graph search)
// ---------------------------------------------------------------------------------------------------------------------
struct PlanSmem {  // per warp, followed by dist / mask / pred (sizes depend on the lattice)
    double vx[LTPL_KMAX], vy[LTPL_KMAX], vr[LTPL_KMAX], vv[LTPL_KMAX];
    // obstacle discs (GLNT:169-189): per on-track vehicle its current position followed by its prediction points
    double dx[LTPL_DMAX], dy[LTPL_DMAX], dref[LTPL_DMAX];
    int vd0[LTPL_KMAX], vdn[LTPL_KMAX];   // first disc of a vehicle, number of prediction discs behind it
    int n_veh;
    int pad[3];
};

// per warp: PlanSmem | dist f64[2 maxn] | dsave f64[maxn] | meta int4[hl] | mask u32[mask_words] | pred u8[hl maxn]
__host__ __device__ inline size_t plan_smem_bytes_per_warp(int maxn, int hl, int mask_words) {
    size_t s = sizeof(PlanSmem) + sizeof(double) * 3 * (size_t)maxn + sizeof(int4) * (size_t)hl +
               sizeof(unsigned) * mask_words + (size_t)hl * maxn;
    return (s + 15) & ~(size_t)15;
}

// mark edges of layer pair a -> a+1 that hold a sample inside one of the inflated obstacle discs in `discs` (bit d ->
// ps->dx/dy/dref[d]) (GB:626-644).  All discs that touch the pair share ONE sweep over its samples (the current and the
// 0.2 s predicted disc of a vehicle nearly always do); four samples per lane are in flight.
__device__ __forceinline__ void block_pair(const LatDev& lt, int lane, int a, unsigned discs, const PlanSmem* ps,
                                           unsigned* mask, int e_base) {
    const int e0 = lt.edge_layer_off[a], e1 = lt.edge_layer_off[a + 1];
    if (e1 <= e0) return;
    const int s0 = lt.samp_off[e0], s1 = lt.samp_off[e1];
    const int moff = (e0 >= e_base) ? -e_base : lt.E - e_base;
    #pragma unroll 1
    for (int sb = s0; sb < s1; sb += 128) {
        const int s = sb + lane;
        double2 p[4];
        int ed[4];   // owning edge of every sample, loaded together with it (a hit does not wait for a second round trip)
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int si = s + 32 * u;
            p[u] = lt.samp_xy[(si < s1) ? si : sb];
            ed[u] = lt.samp_edge[(si < s1) ? si : sb];
        }
        unsigned hit = 0;
        #pragma unroll 1
        for (unsigned mm = discs; mm; mm &= mm - 1) {
            const int d = __ffs(mm) - 1;
            const double ox = ps->dx[d], oy = ps->dy[d], ref = ps->dref[d];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const double x = __dsub_rn(p[u].x, ox), y = __dsub_rn(p[u].y, oy);
                if (__dadd_rn(__dmul_rn(x, x), __dmul_rn(y, y)) <= ref) hit |= 1u << u;
            }
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int si = s + 32 * u;
            if (((hit >> u) & 1u) && si < s1) {
                const int idx = ed[u] + moff;
                atomicOr(&mask[idx >> 5], 1u << (idx & 31));
            }
        }
    }
}

// get_intersec_edges (GIE:36-63) for one disc: layer of the disc's centre (or -1 when outside the planning range) and
// the (up to) two layer pairs pa -> pa+1, pb -> pb+1 whose edges the disc can block (-1: none)
// (o = nearest reference-line layer of the disc's centre; per lane)
__device__ __forceinline__ int disc_pairs(const LatDev& lt, int o, int p_start, int p_end, int* pa, int* pb) {
    *pa = -1;
    *pb = -1;
    const int lo = 1;
    const bool in_rng = (p_start - lo <= o && o <= p_end + lo) ||
                        (p_start > p_end && (p_start - lo <= o || o <= p_end + lo));
    if (!in_rng) return -1;
    // layer window {o-1, o, o+1} with the reference's wrap handling (GB:597-600: quirk q4 drops o+1 when o == L-1)
    int s_l = o - lo, e_l = o + lo;
    if (s_l < 0) s_l += lt.L;
    if (e_l > lt.L) e_l -= lt.L;
    const bool has_next = (e_l < lt.L);       // e_l == L  -> layer L does not exist
    const int prev = s_l;                     // o-1 (mod L) is always part of the window
    const int next = e_l;
    if (layer_in_range(prev, p_start, p_end) && layer_in_range(o, p_start, p_end) && ((prev + 1) % lt.L) == o)
        *pa = prev;
    if (has_next && layer_in_range(o, p_start, p_end) && layer_in_range(next, p_start, p_end) &&
        ((o + 1) % lt.L) == next)
        *pb = o;
    return o;
}

#ifndef LTPL_PLAN_MINB
#define LTPL_PLAN_MINB 10  // resident CTAs per SM the register allocation is held to (occupancy hides the L1/L2 latency)
#endif
// STATE: stateful tick (ltpl_state.cuh): start node / constant segment come from k_state, the constant segment lives in
// the previous tick's path planes, pos_est and the last action id enter the action-set logic, the first edges of the
// last solution are cheaper
template <bool ZONE, bool STATE = false, bool DENSE = false>
__global__ void __launch_bounds__(LTPL_WARPS_PER_CTA * 32, LTPL_PLAN_MINB)
k_plan(const LatDev lt, const LtplParams prm, const LtplDims dm, const LtplBuffers bf, const int maxn, const int hl,
       const int mask_words) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31;
    const int wib = threadIdx.x >> 5;
    const int b = sub_scenario(dm, LTPL_WARPS_PER_CTA);
    if (b < 0) return;
    unsigned char* base = smem_raw + plan_smem_bytes_per_warp(maxn, hl, mask_words) * wib;
    PlanSmem* ps = reinterpret_cast<PlanSmem*>(base);
    double* dist = reinterpret_cast<double*>(base + sizeof(PlanSmem));
    double* dsave = dist + 2 * maxn;
    int4* meta = reinterpret_cast<int4*>(dsave + maxn);
    unsigned* mask = reinterpret_cast<unsigned*>(meta + hl);
    unsigned char* pred = reinterpret_cast<unsigned char*>(mask + mask_words);
    const int B = dm.batch;

    // defaults
    if (lane < LTPL_NSLOT) {
        bf.action_id[lane * B + b] = LTPL_ACT_NONE;
        bf.status[lane * B + b] = 0;
        bf.n_nodes[lane * B + b] = 0;
        bf.path_len[lane * B + b] = 0;
        bf.traj_len[lane * B + b] = 0;
        bf.traj_id[lane * B + b] = -1;
        bf.traj_row[lane * B + b] = -1;
    }
    if (lane == 0) {
        bf.closest_obj[b] = -1;
        bf.cobj[4 * b + 3] = 0.0;
    }
    if (bf.sc_flags[b] != 0) return;
    LTPL_PH_INIT

    const int start_layer = bf.start_node[2 * b], start_node = bf.start_node[2 * b + 1];
    const int p0 = bf.const_len[b];
    size_t cplane = (size_t)B * dm.p0_max;
    const double* cs = bf.const_seg + (size_t)b * dm.p0_max;
    int cnd = 1;   // entries of the node / node-index / coefficient lists in front of the start node
    if (STATE) {
        const int* sinfo = bf.st_info + 8 * (size_t)b;
        cplane = (size_t)LTPL_NSLOT * B * dm.p_max;
        cs = bf.prev_path + (size_t)sinfo[0] * dm.p_max + sinfo[1];
        cnd = sinfo[3];
    }

    // ---- OLI.process_object_list (OLI:96-141): drop off-track objects, radius = length / 2, prediction points: the
    // caller's 'prediction' array (OLI:117-119) or one constant-velocity point at 0.2 s (OLI:121-127) ----
    int n_veh = 0, n_disc = 0;
    {
        int n_in = bf.n_obj[b];
        if (n_in > dm.k_obj) n_in = dm.k_obj;
        // lane k = object k (k_obj <= 16): on-track test, radius, discs -- all objects at once; the on-track objects keep
        // their order (vehicle index = number of on-track objects in front, disc index = their discs in front)
        const bool act = lane < n_in;
        const double* o = bf.obj + ((size_t)b * dm.k_obj + (act ? lane : 0)) * 5;
        const double ox = o[0], oy = o[1];
        const int nb = lanes_closest_point(lt, lt.grid_center, lt.center, lt.L, ox, oy, act, lane);
        const bool inside = act && inside_bounds_from_vertex(lt, nb, ox, oy);
        const unsigned in_mask = __ballot_sync(LTPL_FULL, inside);
        int np_k = -1;   // -1: built-in prediction
        if (inside && dm.k_pred > 0 && bf.n_pred) np_k = min(bf.n_pred[(size_t)b * dm.k_obj + lane], dm.k_pred);
        const int n_pd = (np_k < 0) ? 1 : np_k;
        const int mine = inside ? 1 + n_pd : 0;
        int incl = mine;   // inclusive prefix sum of the disc counts
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            const int up = __shfl_up_sync(LTPL_FULL, incl, off);
            if (lane >= off) incl += up;
        }
        n_disc = __shfl_sync(LTPL_FULL, incl, 31);
        n_veh = __popc(in_mask);
        if (n_disc > LTPL_DMAX) {   // (the reference has no limit; one warp ballot holds 32 discs)
            if (lane == 0) bf.sc_flags[b] = LTPL_SC_CAPACITY;
            return;
        }
        if (inside) {
            const int v_i = __popc(in_mask & ((1u << lane) - 1u)), d_i = incl - mine;
            const double th = o[2], v = o[3], r = o[4] / 2.0;
            ps->vx[v_i] = ox;
            ps->vy[v_i] = oy;
            ps->vr[v_i] = r;
            ps->vv[v_i] = v;
            ps->vd0[v_i] = d_i;
            ps->vdn[v_i] = n_pd;
            // obstacle_ref = (r + veh_width / 2)^2 + stepsize^2 / 4  (GB:626-629)
            const double ref = __dadd_rn(sq_rn(__dadd_rn(r, __ddiv_rn(lt.veh_width, 2.0))),
                                         __ddiv_rn(sq_rn(lt.step), 4.0));
            ps->dx[d_i] = ox;
            ps->dy[d_i] = oy;
            ps->dref[d_i] = ref;
            if (np_k < 0) {
                ps->dx[d_i + 1] = __dsub_rn(ox, __dmul_rn(__dmul_rn(sin(th), v), 0.2));
                ps->dy[d_i + 1] = __dadd_rn(oy, __dmul_rn(__dmul_rn(cos(th), v), 0.2));
                ps->dref[d_i + 1] = ref;
            } else {
                const double* pp = bf.obj_pred + (((size_t)b * dm.k_obj + lane) * dm.k_pred) * 2;
                for (int j = 0; j < np_k; ++j) {
                    ps->dx[d_i + 1 + j] = pp[2 * j];
                    ps->dy[d_i + 1 + j] = pp[2 * j + 1];
                    ps->dref[d_i + 1 + j] = ref;
                }
            }
        }
    }
    #pragma unroll 1
    for (int i = lane; i < mask_words; i += 32) mask[i] = 0u;
    __syncwarp();
    LTPL_PH(16)

    // ---- planning range (GLNT:104-142) ----
    const int end_layer = plan_end_layer(lt, start_layer, lane);
    int planning_dist = end_layer - start_layer;
    if (planning_dist < 0) planning_dist = lt.L - start_layer + end_layer;
    if (end_layer >= lt.L || planning_dist + 1 > hl || planning_dist + 1 + cnd > dm.h_max) {
        if (lane == 0) bf.sc_flags[b] = LTPL_SC_CAPACITY;
        return;
    }
    const int e_base = lt.edge_layer_off[start_layer];
    LTPL_PH(17)

    // ---- obstacles -> blocked edges, closest object (GLNT:165-213) ----
    int closest_dist = -1, closest_idx = -1, con_layer = -1, con_node = -1;
    int my_pa = -1, my_pb = -1;  // lane d: layer pairs disc d can block
    int my_layer = -1;           // lane d: nearest reference-line layer of disc d, -1 outside the planning range
    __syncwarp();
    {
        const bool act = lane < n_disc;
        const double ox = act ? ps->dx[lane] : 0.0, oy = act ? ps->dy[lane] : 0.0;
        const int o = lanes_closest_point(lt, lt.grid_refline, lt.refline, lt.L, ox, oy, act, lane);
        if (act) my_layer = disc_pairs(lt, o, start_layer, end_layer, &my_pa, &my_pb);
    }
    #pragma unroll 1
    for (int v = 0; v < n_veh; ++v) {
        // current position, then the prediction points: the LAST one sets obj_layer (q14)
        const int obj_layer = __shfl_sync(LTPL_FULL, my_layer, ps->vd0[v] + ps->vdn[v]);
        if (obj_layer >= 0) {
            int ld = obj_layer - start_layer;
            if (ld < 0) ld = lt.L - start_layer + obj_layer;
            if (ld <= planning_dist && (closest_dist < 0 || ld < closest_dist)) {
                closest_dist = ld;
                closest_idx = v;
                con_layer = obj_layer;
            }
        }
    }
    __syncwarp();
    #pragma unroll 1
    for (int d = 0; d < n_disc; ++d) {  // one sweep per distinct layer pair, shared by every disc that touches it
        #pragma unroll 1
        for (int slot = 0; slot < 2; ++slot) {
            const int a = __shfl_sync(LTPL_FULL, slot ? my_pb : my_pa, d);
            if (a < 0) continue;
            const unsigned discs = __ballot_sync(LTPL_FULL, my_pa == a || my_pb == a);
            if (discs & ((1u << d) - 1u)) continue;  // swept together with an earlier disc
            block_pair(lt, lane, a, discs, ps, mask, e_base);
        }
    }
    __syncwarp();
    if (closest_dist >= 0) {  // GLNT:206-213
        const int nb = lt.node_off[con_layer];
        const ArgMinD m = warp_closest_point(lt.node_xy + nb, lt.node_off[con_layer + 1] - nb, ps->vx[closest_idx],
                                             ps->vy[closest_idx], lane);
        con_node = m.i;
    }
    LTPL_PH(18)

    // ---- objects in / beside the constant path segment (MOPG:76-122) ----
    bool obj_in_const = false, obj_beside = false;
    if (p0 >= 2) {
        // MOPG:80-84: pos_est of the previous calc_vel_profile call; None on the first tick -> first point of the segment
        const double sx0 = STATE ? bf.pos_last[2 * b] : cs[0], sy0 = STATE ? bf.pos_last[2 * b + 1] : cs[cplane];
        const double sxe = cs[p0 - 1], sye = cs[cplane + p0 - 1];
        // s coordinates on the race line: lane 0 the start, lane 1 the end of the segment, lane 2 + v object v (n_veh <= 16)
        double qx = sx0, qy = sy0;
        if (lane == 1) {
            qx = sxe;
            qy = sye;
        } else if (lane >= 2 && lane - 2 < n_veh) {
            qx = ps->vx[lane - 2];
            qy = ps->vy[lane - 2];
        }
        const bool q_act = lane < 2 + n_veh;
        const int q_nb = lanes_closest_point(lt, lt.grid_raceline, lt.raceline, lt.L, qx, qy, q_act, lane);
        const double s_mine = q_act ? s_coord_from_vertex(lt.raceline, lt.s_rl, lt.L, q_nb, qx, qy) : 0.0;
        const double s_start = __shfl_sync(LTPL_FULL, s_mine, 0), s_end = __shfl_sync(LTPL_FULL, s_mine, 1);
        double smallest = LTPL_INF;
        #pragma unroll 1
        for (int v = 0; v < n_veh; ++v) {
            const double ox = ps->vx[v], oy = ps->vy[v];
            const double s_obj = __shfl_sync(LTPL_FULL, s_mine, 2 + v);
            if ((s_start <= s_obj && s_obj <= s_end) || (s_start > s_end && (s_obj > s_start || s_obj < s_end))) {
                obj_beside = true;
                double od;
                if (s_obj < s_start)
                    od = __dsub_rn(__dadd_rn(s_obj, lt.s_rl[lt.L - 1]), s_start);
                else
                    od = __dsub_rn(s_obj, s_start);
                if (closest_idx < 0 || od < smallest) {  // quirk q15
                    closest_idx = v;
                    smallest = od;
                }
                const double oref = sq_rn(__dadd_rn(ps->vr[v], __ddiv_rn(lt.veh_width, 2.0)));
                int hit = 0;
                #pragma unroll 1
                for (int k = lane; k < p0; k += 32) hit |= (dist2_rn(cs[k], cs[cplane + k], ox, oy) <= oref) ? 1 : 0;
                if (__any_sync(LTPL_FULL, hit)) obj_in_const = true;
            }
        }
    }
    LTPL_PH(19)
    // match the closest object to the (closed) global race line: get_s_coord(glob_rl[:, 1:3], obj_pos, closed=True)[1][0]
    // (CVPF:166-172) -- warp-parallel here instead of a serial 800-point scan per follow path in the velocity kernel
    if (closest_idx >= 0) {
        const int ng = lt.n_glob - 1;
        const double ox = ps->vx[closest_idx], oy = ps->vy[closest_idx];
        const ArgMinD m = warp_closest_point_grid(lt, lt.grid_glob, lt.glob_xy, ng, ox, oy, lane);
        const int nb = m.i;
        const int i1 = (nb - 1 < 0) ? ng - 1 : nb - 1;
        const int i2 = (nb + 1 > ng - 1) ? 0 : nb + 1;
        const double2 gn = lt.glob_xy[nb], g1 = lt.glob_xy[i1], g2 = lt.glob_xy[i2];
        if (lane == 0) bf.cobj_start[b] = angle_cmp(gn, ox, oy, g1, g2).ge ? i1 : nb;
    }
    LTPL_PH(20)
    if (lane == 0) {
        bf.closest_obj[b] = closest_idx;
        if (closest_idx >= 0) {
            bf.cobj[4 * b + 0] = ps->vx[closest_idx];
            bf.cobj[4 * b + 1] = ps->vy[closest_idx];
            bf.cobj[4 * b + 2] = ps->vv[closest_idx];
            bf.cobj[4 * b + 3] = 1.0;
        }
    }

    // ---- action sets (MOPG:124-174); filter: 0 planning_range, 1 default, 2 overtake_left, 3 overtake_right ----
    int n_act, names[3], filt[3];
    if (obj_in_const || obj_beside) {
        n_act = 1;
        names[0] = LTPL_ACT_FOLLOW;
        filt[0] = 0;
        // last_action_id (MOPG:130): the executed action, 'emergency' already translated by k_state (st_info[0] = its slot)
        const int last_act = STATE ? bf.prev_action_id[bf.st_info[8 * (size_t)b]] : LTPL_ACT_STRAIGHT;
        if (!obj_in_const && (last_act == LTPL_ACT_LEFT || last_act == LTPL_ACT_RIGHT)) {   // MOPG:130-133: keep overtaking
            names[1] = last_act;
            filt[1] = 1;
            n_act = 2;
        } else if (!obj_in_const) {  // last_action_id is the forced "straight" on the first tick -> offer left and right
            names[1] = LTPL_ACT_LEFT;  filt[1] = 1;
            names[2] = LTPL_ACT_RIGHT; filt[2] = 1;
            n_act = 3;
        }
    } else if (closest_idx >= 0 && con_node >= 0) {
        n_act = 3;
        names[0] = LTPL_ACT_FOLLOW; filt[0] = 0;
        names[1] = LTPL_ACT_LEFT;   filt[1] = 2;
        names[2] = LTPL_ACT_RIGHT;  filt[2] = 3;
    } else {
        n_act = 1;
        names[0] = LTPL_ACT_STRAIGHT;
        filt[0] = 1;
    }

    // ---- graph search per action (MOPG:188-257) ----
    // Three observations cut the number of DPs without touching any result:
    //  * a search on the unblocked lattice (filter 'planning_range', or 'default' with an empty mask) depends only on
    //    the start node -> read from the follow table built once per lattice (k_follow_table);
    //  * two consecutive actions with the same filter ('left' and 'right' on 'default') are the same search;
    //  * 'overtake_left' and 'overtake_right' differ only from the object's layer onwards -> the second one resumes
    //    from a snapshot of the first one's state one layer before it.
    const unsigned* zone = nullptr;   // k_plan<false> is launched when the batch carries no zones (dims.n_zones == 0)
    int zone_s0 = start_layer;        // start layer of the tick that processed the zone (GLNT:43-77)
    if (ZONE) {
        const int zsel = bf.zone_sel[b];
        if (zsel >= 0 && zsel < dm.n_zones) zone = bf.zone_bits + (size_t)zsel * dm.n_zone_words;
        if (bf.zone_s0) {
            if (STATE && zone && bf.zone_s0[b] >= 0) zone_s0 = bf.zone_s0[b];
            __syncwarp();
            if (lane == 0) bf.zone_s0[b] = zone ? zone_s0 : -1;
        }
    }
    unsigned mask_any = 0;
    #pragma unroll 1
    for (int i = lane; i < mask_words; i += 32) mask_any |= mask[i];
    mask_any = __any_sync(LTPL_FULL, mask_any != 0);
    dp_fill_meta(lt, lane, meta, start_layer, planning_dist);
    DpCtx c;
    c.dist = dist;
    c.dsave = dsave;
    c.pred = pred;
    c.meta = meta;
    c.maxn = maxn;
    c.snap_li = 0;
    c.tie_save = 0;
    c.fe0 = c.fe1 = c.fe2 = -1;
    c.ff0 = c.ff1 = c.ff2 = 1.0;
    int n_fe = 0;
    if (STATE) {
        const int* sinfo = bf.st_info + 8 * (size_t)b;
        n_fe = sinfo[4];
        c.fe0 = sinfo[5];
        c.fe1 = sinfo[6];
        c.fe2 = sinfo[7];
        c.ff0 = prm.w_last_edges[0];
        c.ff1 = prm.w_last_edges[1];
        c.ff2 = prm.w_last_edges[2];
    }
    const int goal_steps = planning_dist;
    const int tab_row = lt.node_off[start_layer] + start_node;
    int mod_steps = goal_steps;
    int prev_q = -1, prev_f = -1, prev_reach = 0;
    int pair_reach = -1, pair_tie = 0;   // second search of an 'overtake_left' / 'overtake_right' pair (dp_run_pair)
    #pragma unroll 1
    for (int a = 0; a < n_act; ++a) {
        int name = names[a];
        const int f = filt[a];
        int rem_layer = -1, rem_lo = 0, rem_hi = 0;
        if (f == 2) {  // remove nodes [n_obj, n_l) of the object's layer (MOPG:148-152)
            rem_layer = con_layer;
            rem_lo = con_node;
            rem_hi = lt.node_off[con_layer + 1] - lt.node_off[con_layer];
        } else if (f == 3) {  // remove nodes [0, n_obj) (MOPG:155-159)
            rem_layer = con_layer;
            rem_lo = 0;
            rem_hi = con_node;
        }
        // 0: follow table, 1: DP, 2: same search as the previous action
        int src = (f == 0 || (f == 1 && !mask_any)) ? 0 : ((f == 1 && prev_f == 1) ? 2 : 1);
        const int tr = lt.tab_reach[tab_row];
        if (src == 0 && (tr & 0xff) > mod_steps) src = 1;  // table rows end at their own goal layer (open track only)
        if (ZONE && src == 0 && zone) src = 1;              // the table holds searches on the zone-free lattice
        if (STATE && src == 0 && n_fe > 0) src = 1;         // ... with the offline costs
        int st = 0, tie = 0, found = 0, reach = 0, goal_off = 0;
        if (mod_steps > 0) {
            const bool start_removed = (rem_layer == start_layer && start_node >= rem_lo && start_node < rem_hi);
            if (start_removed) {
                st |= LTPL_ST_START_BLOCKED;  // GB:882-885
            } else if (src == 0) {
                reach = tr & 0xff;
                tie = (tr >> 8) & 1;
            } else if (src == 2) {
                reach = prev_reach;
            } else {
                const bool with_next = (f == 2 && a + 1 < n_act && filt[a + 1] == 3);
                if (f == 3 && pair_reach >= 0) {          // searched together with 'overtake_left' (dp_run_pair)
                    reach = pair_reach;
                    tie = pair_tie;
                    goal_off = 16;
                } else if (with_next && maxn == 32 && lt.max_nodes <= 16) {
                    reach = dp_run_pair<ZONE, STATE>(lt, lane, c, start_layer, start_node, mod_steps, mask, e_base, con_layer,
                                                     con_node, zone, zone_s0, &pair_reach, &pair_tie);
                    tie = c.tie;
                } else {
                    const int li_begin = (f == 3 && c.snap_li >= 1) ? c.snap_li + 1 : 1;
                    const int snap_at = with_next ? closest_dist - 1 : 0;
                    reach = dp_run<ZONE, STATE, DENSE>(lt, lane, c, start_layer, start_node, mod_steps, (f == 0) ? nullptr : mask,
                                                       e_base, rem_layer, rem_lo, rem_hi, li_begin, snap_at, zone, zone_s0);
                    tie = c.tie;
                }
            }
            LTPL_PH(21)
            if (name == LTPL_ACT_FOLLOW || name == LTPL_ACT_STRAIGHT) {
                if (reach < mod_steps) mod_steps = reach;  // goal layer moves towards the vehicle (MOPG:203-220)
                found = (reach >= 1);
            } else {
                found = (reach == mod_steps);
            }
        }
        const int mod_goal = (start_layer + mod_steps) % lt.L;
        const bool reduced = (mod_steps != goal_steps) || (!lt.closed && end_layer == lt.L - 1);
        if (reduced) {
            st |= LTPL_ST_REDUCED_HORIZON;
            const bool in_mod = (con_layer >= 0) &&
                                ((start_layer <= con_layer && con_layer <= mod_goal) ||
                                 (start_layer > mod_goal && (con_layer >= start_layer || con_layer <= mod_goal)));
            if (!obj_in_const && con_layer >= 0 && !in_mod) {
                if (name == LTPL_ACT_FOLLOW || name == LTPL_ACT_STRAIGHT) {
                    if (name == LTPL_ACT_FOLLOW) st |= LTPL_ST_RENAMED_STRAIGHT;
                    name = LTPL_ACT_STRAIGHT;
                } else {
                    found = 0;
                }
            }
        }
        const int slot = (name == LTPL_ACT_LEFT) ? 1 : ((name == LTPL_ACT_RIGHT) ? 2 : 0);
        const int q = slot * B + b;
        int* nd = bf.nodes + (size_t)q * dm.h_max * 2;
        int* es = bf.edge_seq + (size_t)q * dm.h_max;
        if (found && src == 0) {  // rows of the follow table: node / edge of every step
            const unsigned char* tn = lt.tab_node + (size_t)tab_row * lt.tab_stride;
            const int* te = lt.tab_edge + (size_t)tab_row * lt.tab_stride;
            #pragma unroll 1
            for (int li = 1 + lane; li <= reach; li += 32) {
                int layer = start_layer + li;
                if (layer >= lt.L) layer -= lt.L;
                nd[2 * (li + cnd)] = layer;
                nd[2 * (li + cnd) + 1] = tn[li - 1];
                es[li - 1] = te[li - 1];
            }
        } else if (found && src == 2) {  // copy of the previous action's plan
            const int* pn = bf.nodes + (size_t)prev_q * dm.h_max * 2;
            const int* pe = bf.edge_seq + (size_t)prev_q * dm.h_max;
            #pragma unroll 1
            for (int i = lane; i < 2 * (reach + 1 + cnd); i += 32) nd[i] = pn[i];
            #pragma unroll 1
            for (int i = lane; i < reach; i += 32) es[i] = pe[i];
            st |= bf.status[prev_q] & LTPL_ST_TIE_AMBIGUOUS;
        }
        if (found) {
            int gj = 0;
            if (src == 1) gj = dp_goal(lt, lane, c, &tie, goal_off);
            if (tie) st |= LTPL_ST_TIE_AMBIGUOUS;
            st |= LTPL_ST_FOUND;
            if (STATE && src != 2) {   // constant nodes in front of the start node: the memory of the last tick (OTH:462-466)
                const int* sinfo = bf.st_info + 8 * (size_t)b;
                const int* pn = bf.prev_nodes + ((size_t)sinfo[0] * dm.h_max + sinfo[2]) * 2;
                for (int i = lane; i < 2 * cnd; i += 32) nd[i] = pn[i];
            }
            if (lane == 0) {
                if (!STATE) {
                    nd[0] = -1;
                    nd[1] = -1;
                }
                nd[2 * cnd] = start_layer;
                nd[2 * cnd + 1] = start_node;
                if (src == 1) {   // node sequence: a chain through the predecessor table in shared memory
                    int j = gj, layer = c.layer;
                    #pragma unroll 1
                    for (int li = reach; li >= 1; --li) {
                        nd[2 * (li + cnd)] = layer;
                        nd[2 * (li + cnd) + 1] = j;
                        j = pred[li * maxn + goal_off + j];
                        layer = (layer == 0) ? lt.L - 1 : layer - 1;
                    }
                }
                bf.n_nodes[q] = reach + 1 + cnd;
                bf.action_id[q] = name;
                bf.status[q] = st;
            }
            if (src == 1) {   // edge ids of all steps at once (lane = step)
                __syncwarp();
                #pragma unroll 1
                for (int li = 1 + lane; li <= reach; li += 32)
                    es[li - 1] = dp_edge_id(lt, meta[li].x, __ldcg(&nd[2 * (li + cnd) + 1]), __ldcg(&nd[2 * (li - 1 + cnd) + 1]));
            }
        } else if (lane == 0 && bf.action_id[q] == LTPL_ACT_NONE) {
            bf.status[q] = st;
        }
        prev_q = q;
        prev_f = f;
        prev_reach = reach;
        __syncwarp();
        LTPL_PH(22)
    }

    // ---- "track blocked": no action at all -> constant segment only (OTH:475-506) ----
    if (lane == 0) {
        bool any = false;
        for (int s = 0; s < LTPL_NSLOT; ++s) any |= (bf.action_id[s * B + b] != LTPL_ACT_NONE);
        if (!any && p0 > 2) {
            const int q = b;
            int* nd = bf.nodes + (size_t)q * dm.h_max * 2;
            if (STATE) {
                const int* sinfo = bf.st_info + 8 * (size_t)b;
                const int* pn = bf.prev_nodes + ((size_t)sinfo[0] * dm.h_max + sinfo[2]) * 2;
                for (int i = 0; i < 2 * cnd; ++i) nd[i] = pn[i];
            } else {
                nd[0] = -1;
                nd[1] = -1;
            }
            nd[2 * cnd] = start_layer;
            nd[2 * cnd + 1] = start_node;
            bf.n_nodes[q] = cnd + 1;
            bf.action_id[q] = LTPL_ACT_STRAIGHT;
            bf.status[q] = LTPL_ST_FOUND | LTPL_ST_CONST_ONLY | LTPL_ST_REDUCED_HORIZON;
        }
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// k_follow_table: search on the UNBLOCKED lattice from every node over its planning range (same dp_run / dp_goal as the
// online kernel; runs once in ltpl_lattice_create).  Row n: tab_reach[n] = steps | tie << 8, then node index and edge id
// of every step.  k_plan reads these rows instead of repeating a search whose inputs are all lattice constants.
// ---------------------------------------------------------------------------------------------------------------------
__host__ __device__ inline size_t table_smem_bytes_per_warp(int maxn, int hl) {
    size_t s = sizeof(double) * 2 * (size_t)maxn + sizeof(int4) * (size_t)hl + (size_t)hl * maxn;
    return (s + 15) & ~(size_t)15;
}

__global__ void __launch_bounds__(LTPL_WARPS_PER_CTA * 32)
k_follow_table(const LatDev lt, const int maxn, int* tab_reach, unsigned char* tab_node, int* tab_edge) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31;
    const int wib = threadIdx.x >> 5;
    const int n = blockIdx.x * LTPL_WARPS_PER_CTA + wib;
    if (n >= lt.Nn) return;
    const int hl = lt.tab_stride;
    unsigned char* base = smem_raw + table_smem_bytes_per_warp(maxn, hl) * wib;
    double* dist = reinterpret_cast<double*>(base);
    int4* meta = reinterpret_cast<int4*>(dist + 2 * maxn);
    unsigned char* pred = reinterpret_cast<unsigned char*>(meta + hl);
    const int start_layer = lt.node_layer[n];
    const int start_node = n - lt.node_off[start_layer];
    const int end_layer = plan_end_layer(lt, start_layer, lane);
    int planning_dist = end_layer - start_layer;
    if (planning_dist < 0) planning_dist = lt.L - start_layer + end_layer;
    if (end_layer >= lt.L || planning_dist + 2 > hl || planning_dist < 1) {  // k_plan flags these scenarios itself
        if (lane == 0) tab_reach[n] = 0;
        return;
    }
    dp_fill_meta(lt, lane, meta, start_layer, planning_dist);
    DpCtx c;
    c.dist = dist;
    c.dsave = dist;
    c.pred = pred;
    c.meta = meta;
    c.maxn = maxn;
    c.snap_li = 0;
    c.tie_save = 0;
    const int reach = dp_run<false>(lt, lane, c, start_layer, start_node, planning_dist, nullptr, 0, -1, 0, 0, 1, 0, nullptr);
    int tie = c.tie;
    int gj = 0;
    if (reach >= 1) gj = dp_goal(lt, lane, c, &tie);
    if (lane == 0) {
        int j = gj;
        #pragma unroll 1
        for (int li = reach; li >= 1; --li) {
            tab_node[(size_t)n * hl + li - 1] = (unsigned char)j;
            j = pred[li * maxn + j];
        }
        tab_reach[n] = reach | (tie << 8);
    }
    __syncwarp();
    #pragma unroll 1
    for (int li = 1 + lane; li <= reach; li += 32) {
        const int js = (li == 1) ? start_node : (int)__ldcg(&tab_node[(size_t)n * hl + li - 2]);
        tab_edge[(size_t)n * hl + li - 1] = dp_edge_id(lt, meta[li].x, (int)__ldcg(&tab_node[(size_t)n * hl + li - 1]), js);
    }
}
