/*
 * ltpl_b200.h -- C-ABI of the B200-native batched online planning path of Graph_LTPL.
 *
 * The reference (TUMFTM/GraphBasedLocalTrajectoryPlanner @ 18763ef9) has no FFI / plugin seam; its boundary for this
 * path is the Python API  Graph_LTPL.set_startpos / calc_paths / calc_vel_profile  (graph_ltpl/Graph_LTPL.py:262-296,
 * 300-340, 344-408), one level down  OnlineTrajectoryHandler.set_initial_pose / calc_paths / calc_vel_profile
 * (graph_ltpl/online_graph/src/OnlineTrajectoryHandler.py:181-270, 289-516, 603-1040)  and  main_online_path_gen
 * (graph_ltpl/online_graph/src/main_online_path_gen.py:11-21).  Each entry point below names the reference interface
 * it replaces.  The binding a maintainer adds on the reference side is a ctypes stub (INTEGRATION.md).
 *
 * Conventions
 *   - plain C, no torch types: every buffer is a raw DEVICE pointer owned by the caller (PyTorch tensors are used only
 *     as allocators on the Python side); the library never allocates on the hot path.
 *   - every call is asynchronous on the given CUDA stream (cudaStream_t passed as void*).
 *   - return value: 0 = ok, < 0 = error (message via ltpl_last_error()).
 *   - per (scenario, action slot) results carry a status bit field (LTPL_ST_*); infeasible actions are flagged, never
 *     silently dropped, mirroring "omitted from the dict" in the reference (MOPG:246-248, OTH:1007-1025).
 *   - ltpl_tick_batch plans the stateless FIRST tick after set_startpos; ltpl_next_* plan every later tick with the
 *     iterative memory of the reference (OTH:64-87) held in caller-owned device buffers -- the wall clock the reference
 *     reads (OTH:353-378) is an input (t_const).
 */
#ifndef LTPL_B200_H
#define LTPL_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LTPL_ABI_VERSION 12

/* action ids (OTH:14-17 ACTION_ID_MAP) */
#define LTPL_ACT_NONE (-1)
#define LTPL_ACT_STRAIGHT 0
#define LTPL_ACT_FOLLOW 1
#define LTPL_ACT_LEFT 2
#define LTPL_ACT_RIGHT 3
#define LTPL_ACT_EMERGENCY 4 /* only as `sel_action`: the caller executed the 'emergency' trajectory (OTH:307-309) */

/* action slots per scenario: slot 0 = straight | follow (mutually exclusive, MOPG:124-174), 1 = left, 2 = right */
#define LTPL_NSLOT 3

/* status bits per (scenario, slot) */
#define LTPL_ST_FOUND            (1 << 0)  /* a path exists for this slot (MOPG:246-257)                               */
#define LTPL_ST_REDUCED_HORIZON  (1 << 1)  /* goal layer was moved towards the vehicle (MOPG:203-243)                  */
#define LTPL_ST_TIE_AMBIGUOUS    (1 << 2)  /* some node of the search, or its virtual goal, has its final (cost, own
                                              distance) minimum attained by >= 2 candidates (in-edges / goal-layer
                                              nodes); igraph's pick there is heap-order dependent. Ties that a later
                                              candidate beats do not count                                          */
#define LTPL_ST_START_BLOCKED    (1 << 3)  /* start node removed by the action's node filter (GB:882-885)              */
#define LTPL_ST_TRAJ_VALID       (1 << 4)  /* trajectory kept in the action set after calc_vel_profile (OTH:945-948)   */
#define LTPL_ST_VEL_BOUND_VIOL   (1 << 5)  /* |vx[0] - vel_plan| >= v_max_offset or follow-mode bound broken (OTH:907)  */
#define LTPL_ST_TOO_CLOSE        (1 << 6)  /* follow mode: inside the safety distance (OTH:821-822)                    */
#define LTPL_ST_CONST_ONLY       (1 << 7)  /* "track blocked": constant segment only (OTH:475-506)                     */
#define LTPL_ST_RENAMED_STRAIGHT (1 << 8)  /* follow renamed to straight after horizon reduction (MOPG:233-238)        */

/* per scenario flags */
#define LTPL_SC_OUT_OF_TRACK     (1 << 0)  /* OTH:214-219                                                             */
#define LTPL_SC_HEADING_MISMATCH (1 << 1)  /* OTH:234-240                                                             */
#define LTPL_SC_CAPACITY         (1 << 2)  /* a fixed-capacity buffer (P0_MAX / P_MAX / H_MAX) would overflow          */
#define LTPL_SC_STATE_FALLBACK   (1 << 4)  /* stateful tick: the last executed trajectory is not usable as memory       */
                                           /* (see the reason codes; re-anchor with ltpl_set_startpos_batch)                */
#define LTPL_SC_REASON_SHIFT 8             /* bits 8..10: why STATE_FALLBACK was raised (diagnostic detail):            */
                                           /* 1 the executed action is not in the memory and the last tick was not      */
                                           /*   planned either (an action the last tick merely did not return is        */
                                           /*   planned per OTH:393-407), 2 its trajectory has <= 2 rows, 3 fewer than  */
                                           /*   2 memory nodes, 4 the start node is the placeholder, 5 the constant     */
                                           /*   segment exceeds p_max, 6 follow / straight cannot start at the planned  */
                                           /*   velocity and no backup plan exists, 7 the position estimate lies at the */
                                           /*   last row of the last trajectory (np.argmin of an empty array, OTH:570)  */
#define LTPL_SC_BRAKE_PREFIX     (1 << 3)  /* vel_plan > vel_max + 0.1: the reference path raises here (OTH:747-754,   */
                                           /* 830/919 column_stack length mismatch); reported instead of planned       */

/* ------------------------------------------------------------------------------------------------------------------ */
/* lattice blob: ONE contiguous device buffer (so it can be NCCL-broadcast as bytes) + this host-side header.          */
/* All `off_*` are byte offsets into the blob, 256-byte aligned.  Layout documented in DESIGN.md "HBM layout".         */
/* Replaces the pickled GraphBase (GraphBase.py:93-135) as the input of the online path.                               */
/* ------------------------------------------------------------------------------------------------------------------ */
typedef struct LtplLatticeHeader {
    int32_t abi_version;
    int32_t num_layers, num_nodes, num_edges, num_samples, n_glob_rl;
    int32_t closed;              /* GB:116                                            */
    int32_t plan_horizon_mode;   /* 0 = 'distance', 1 = 'layers' (GLNT:104-136)       */
    int32_t max_nodes_per_layer; /* <= 64                                             */
    int32_t max_window_edges;    /* max #edges inside any planning window (+1 layer)  */
    int32_t max_pair_edges;      /* max #edges between two consecutive layers         */
    int32_t tab_stride;          /* row length of the follow table (>= max plan layers + 2) */
    int32_t grid_nx, grid_ny;    /* cells of the nearest-vertex grids (off_grid_*)                  */
    double lat_offset, lat_resolution, sampled_resolution, vel_decrease_lat, veh_width, veh_length;
    double virt_goal_node_cost, min_plan_horizon;
    double grid_x0, grid_y0, grid_inv_cell; /* cell of (x, y) = floor((x - grid_x0) * grid_inv_cell), same for y */
    /* per layer [L] */
    uint64_t off_node_off;       /* int32 [L+1]                                       */
    uint64_t off_raceline_index; /* int32 [L]                                         */
    uint64_t off_s_raceline;     /* f64 [L]                                           */
    uint64_t off_vel_raceline;   /* f64 [L]                                           */
    uint64_t off_refline;        /* f64x2 [L]                                         */
    uint64_t off_raceline;       /* f64x2 [L]                                         */
    uint64_t off_bound1;         /* f64x2 [L]  refline + normvec * w_right (OTH:208)  */
    uint64_t off_bound2;         /* f64x2 [L]  refline - normvec * w_left  (OTH:210)  */
    uint64_t off_centerline;     /* f64x2 [L]  (bound1 + bound2) / 2                  */
    /* per node [Nn] */
    uint64_t off_node_xy;        /* f64x2 [Nn]                                        */
    uint64_t off_node_psi;       /* f64 [Nn]                                          */
    uint64_t off_node_layer;     /* int32 [Nn]                                        */
    uint64_t off_in_off;         /* int32x2 [Nn] (first in-edge, #in-edges)           */
    /* per edge [E], CSC order (start_layer, dst, src) */
    uint64_t off_edge_layer_off; /* int32 [L+1]                                       */
    uint64_t off_edge_src;       /* int32 [E]                                         */
    uint64_t off_edge_dst;       /* int32 [E]                                         */
    uint64_t off_edge_cost;      /* f64 [E]                                           */
    uint64_t off_edge_len;       /* f64 [E]                                           */
    uint64_t off_edge_psi1;      /* f64 [E] heading of the last sample                */
    uint64_t off_edge_psi0;      /* f64 [E] heading of the first sample (MOPG:302-303)*/
    uint64_t off_samp_off;       /* int32 [E+1]                                       */
    /* per sample [S] */
    uint64_t off_samp_xy;        /* f64x2 [S]                                         */
    uint64_t off_samp_el;        /* f64 [S]                                           */
    uint64_t off_samp_edge;      /* int32 [S] owning edge                             */
    /* global race line, rows (s, x, y, kappa, vel, el) with el = diff(s) (CVPF:166)  */
    uint64_t off_glob_rl;        /* f64 [n_glob_rl - 1][6]                            */
    uint64_t off_glob_xy;        /* f64x2 [n_glob_rl - 1] x, y (coalesced matching)   */
    /* derived sections (search acceleration)                                         */
    uint64_t off_edge_rec;       /* LtplEdgeRec [E]                                   */
    uint64_t off_tab_reach;      /* int32 [Nn]             -- zero on input, filled   */
    uint64_t off_tab_node;       /* uint8 [Nn][tab_stride] -- by ltpl_lattice_create  */
    uint64_t off_tab_edge;       /* int32 [Nn][tab_stride] -- (k_follow_table)        */
    /* nearest-vertex grids, int32 [grid_ny][grid_nx] each: entry = first << 6 | count: for every position inside the  */
    /* cell the nearest vertex of the polyline (first minimum) is one of the count <= 32 vertices first, first + 1, ...  */
    /* (cyclic on closed tracks); count = 0: no such bound, scan the whole polyline (lattice_blob.nearest_grid)         */
    uint64_t off_grid_center, off_grid_refline, off_grid_raceline, off_grid_glob;
    uint64_t blob_bytes;
} LtplLatticeHeader;

/* one edge of the lattice as the DP reads it (16 bytes, one load) */
typedef struct LtplEdgeRec {
    double cost;  /* GB:818-821 offline edge cost */
    int32_t src;  /* node index within the start layer */
    int32_t dst;  /* node index within the end layer */
} LtplEdgeRec;

typedef struct LtplLattice LtplLattice; /* opaque handle: header copy + resolved device pointers */

/* ------------------------------------------------------------------------------------------------------------------ */
/* parameters: online ini (OTH:99-122, LTPL:168-173) + per-call arguments of calc_vel_profile (LTPL:344-352)           */
/* ------------------------------------------------------------------------------------------------------------------ */
#define LTPL_MAX_AXM 32
typedef struct LtplParams {
    double max_heading_offset;   /* GENERAL.max_heading_offset                        */
    double v_max_offset;         /* ACTIONSET.v_max_offset                            */
    double follow_c_p, follow_k_d, follow_k_p, follow_tan_w;
    int32_t follow_control_type; /* 0 = PD, 1 = PDtan (CVPF:65-71)                    */
    int32_t nmbr_export_points;  /* EXPORT.nmbr_export_points                         */
    double dyn_model_exp, drag_coeff, m_veh; /* graph_init arguments (LTPL:189-192)   */
    double vel_max, gg_scale, gg_ax, gg_ay, safety_d;
    int32_t n_axm;               /* rows of ax_max_machines (<= LTPL_MAX_AXM)         */
    int32_t traj_base_id;        /* OTH:669 (+10 per calc_vel_profile call)           */
    int32_t incl_emerg_traj;     /* calc_vel_profile(incl_emerg_traj=True): append the brake-to-stop profile on the   */
                                 /* first kept trajectory of every scenario (OTH:1027-1034, calc_brake_emergency.py)   */
    int32_t pad0;
    double delaycomp;            /* DELAY.delaycomp (OTH:117, 570)                    */
    double w_last_edges[4];      /* COST.w_last_edges, first three entries (GLNT:155-162); [3] unused */
    double axm_v[LTPL_MAX_AXM];
    double axm_a[LTPL_MAX_AXM];
    double axm_s[LTPL_MAX_AXM];  /* slopes (a[i+1] - a[i]) / (v[i+1] - v[i]) exactly as np.interp forms them  */
} LtplParams;

/* capacities chosen by the host from the lattice (see lattice_blob.py: capacities()) */
typedef struct LtplDims {
    int32_t batch;     /* B scenarios                                                  */
    int32_t k_obj;     /* K object slots per scenario                                  */
    int32_t p0_max;    /* points of the constant segment (pose -> start node)          */
    int32_t p_max;     /* points of a full path (constant segment + new plan), % 4 == 0 */
    int32_t h_max;     /* nodes of a node sequence incl. the leading [None, None] entry */
    int32_t n_export;  /* rows of an exported trajectory (nmbr_export_points)          */
    int32_t n_zone_words; /* 32-bit words of one zone bitmask = ceil(num_nodes / 32)   */
    int32_t n_zones;      /* zone bitmasks in LtplBuffers.zone_bits (0: no zones)      */
    int32_t k_pred;       /* prediction points per object slot in obj_pred (0: built-in 0.2 s prediction only) */
    /* sub-batch window of ONE launch, filled by the library itself (callers pass 0): a tick runs as n independent     */
    /* scenario windows [sub_off, sub_off + sub_cnt) on n internal streams, so that the kernels of different stages     */
    /* overlap (ltpl_set_subbatches)                                                                                     */
    int32_t sub_id, sub_off, sub_cnt;
} LtplDims;
#define LTPL_MAX_SUB 8

/* Caller-owned device buffers.  q = slot * B + b indexes a path ("action major").                                      */
typedef struct LtplBuffers {
    /* scenario inputs (Graph_LTPL.set_startpos / calc_paths arguments)                                                 */
    const double* pos;        /* [B][2]                                                                                  */
    const double* heading;    /* [B]                                                                                     */
    const double* vel;        /* [B]  start velocity of set_startpos (planned velocity of the first tick, OTH:595)       */
    const double* vel_est;    /* [B]  velocity estimate passed to calc_vel_profile (follow-mode controller, OTH:794)     */
    const int32_t* n_obj;     /* [B]                                                                                     */
    const double* obj;        /* [B][K][5] X, Y, theta, v, length (OLI:96-141)                                           */
    /* set_startpos results (OTH:262-268 iterative memory of the forced 'straight' action)                               */
    int32_t* sc_flags;        /* [B] LTPL_SC_*                                                                           */
    int32_t* start_node;      /* [B][2] (layer, node)                                                                    */
    int32_t* const_len;       /* [B] points of the constant segment                                                      */
    double* const_seg;        /* [5][B][p0_max] planes x, y, psi, kappa, el                                              */
    double* const_coeff;      /* [B][8] spline coefficients x(4) | y(4) (OTH:265)                                        */
    /* calc_paths results                                                                                                */
    int32_t* action_id;       /* [NSLOT][B] LTPL_ACT_*                                                                   */
    int32_t* status;          /* [NSLOT][B] LTPL_ST_*                                                                    */
    int32_t* n_nodes;         /* [NSLOT][B] nodes in the sequence incl. the leading (-1, -1)                             */
    int32_t* nodes;           /* [NSLOT][B][h_max][2]                                                                    */
    int32_t* node_idx;        /* [NSLOT][B][h_max] index of every node in the path arrays (MOPG:295)                     */
    int32_t* edge_seq;        /* [NSLOT][B][h_max] lattice edge ids of the new plan (scratch for path assembly)          */
    int32_t* closest_obj;     /* [B] closest_obj_index (into the on-track object list) or -1 (GLNT:191-203, MOPG:113)    */
    double* cobj;             /* [B][4] x, y, v, valid of that object (OTH:770-771)                                      */
    int32_t* cobj_start;      /* [B] index of that object on the global race line = closest_indexes[0] of CVPF:169-172    */
    int32_t* path_len;        /* [NSLOT][B]                                                                              */
    double* path;             /* [5][NSLOT*B][p_max] planes x, y, psi, kappa, el  (path_dict of calc_paths)              */
    double* coeff;            /* [NSLOT*B][h_max][8] (MOPG:305-309 spline_coeff_mat, stitched OTH:470-472)               */
    int32_t* queue;           /* [2][NSLOT*B] dense work queues of path ids q: class 0 follow, class 1 other (k_path->k_vel); */
                              /*     sub-batch window [o, o + n) owns the entries [6 o, 6 (o + n)) as its own [2][NSLOT n]   */
    int32_t* queue_cnt;       /* [4 + 4 LTPL_MAX_SUB]: total fill counts of the two queue classes ([0], [1]), number of    */
                              /*     exported trajectories ([2]); [4 + 4 s + c] = fill count of class c in sub-batch s;     */
                              /*     zeroed by the library before k_plan / k_path / k_vel                                 */
    int32_t* exp_q;           /* [NSLOT*B] path id q of every exported trajectory row (compact export list)               */
    int32_t* traj_row;        /* [NSLOT][B] row of path q in `traj`, or -1                                                 */
    /* calc_vel_profile results                                                                                          */
    double* s_vx_ax;          /* [3][NSLOT*B][p_max] planes s, vx, ax                                                    */
    float* traj;              /* [NSLOT*B][n_export][7] s, x, y, psi, kappa, vx, ax (OTH:941, LTPL:401-406); COMPACT: only  */
                              /* the first queue_cnt[2] rows are filled (one per kept trajectory, row -> path via exp_q)   */
    int32_t* traj_len;        /* [NSLOT][B]                                                                              */
    int32_t* traj_id;         /* [NSLOT][B] traj_base_id + action id (OTH:696-697)                                       */
    /* blocked zones (calc_paths(blocked_zones=...), LTPL:324-329; 'nodes' type, GLNT:43-99): bit (node_off[l] + n) of    */
    /* a mask = node n of layer l is blocked.  A scenario selects one mask or none; may be NULL when n_zones == 0.        */
    const uint32_t* zone_bits; /* [n_zones][n_zone_words]                                                                */
    const int32_t* zone_sel;  /* [B] index into zone_bits or -1                                                          */
    /* emergency trajectory (params.incl_emerg_traj): row in `traj` (or -1), rows, id -- key 'emergency' of the           */
    /* reference's trajectory dict (OTH:1030-1034); `traj` needs (NSLOT + 1) * B rows then                                */
    int32_t* em_info;         /* [B][3]                                                                                  */
    /* explicit prediction arrays of the objects (object dict key 'prediction', OLI:117-119); may be NULL when k_pred == 0 */
    const double* obj_pred;   /* [B][K][k_pred][2] x, y                                                                  */
    const int32_t* n_pred;    /* [B][K] number of prediction points of the object, -1: none given -> one constant-        */
                              /*        velocity point at 0.2 s (OLI:121-127).  At most 32 discs (on-track objects +     */
                              /*        their prediction points) per scenario, else LTPL_SC_CAPACITY                     */
    /* ---- stateful tick (ltpl_next_*_batch, see DESIGN.md section 11): the iterative memory of            */
    /* OnlineTrajectoryHandler (OTH:64-87) = the output buffers of the previous tick (a second buffer set, used            */
    /* ping-pong) + per-path trims instead of the slicing of OTH:705-731.  NULL for first ticks.                           */
    const double* prev_path;        /* previous tick's `path`                                                             */
    const int32_t* prev_path_len;   /* ... `path_len`                                                                     */
    const int32_t* prev_node_idx;   /* ... `node_idx`                                                                     */
    const int32_t* prev_nodes;      /* ... `nodes`                                                                        */
    const int32_t* prev_n_nodes;    /* ... `n_nodes`                                                                      */
    const double* prev_coeff;       /* ... `coeff`                                                                        */
    const double* prev_s_vx_ax;     /* ... `s_vx_ax` (rows 0 .. traj_len-1 = the exported trajectory = __last_bp_action_set) */
    const int32_t* prev_action_id;  /* ... `action_id`                                                                    */
    const int32_t* prev_traj_len;   /* ... `traj_len`                                                                     */
    const int32_t* prev_trim;       /* ... `trim`                                                                         */
    const int32_t* sel_action;      /* [B] LTPL_ACT_* the caller executed since the previous tick (prev_action_id)        */
    const double* pos_last;         /* [B][2] pos_est of the previous calc_vel_profile call (OTH:537, MOPG:80-84)         */
    const double* t_const;          /* [B] min(average calculation time * calc_time_safety, 0.5) (OTH:353-375): the host  */
                                    /*     keeps the moving average, so the wall clock is an input                         */
    int32_t* st_info;               /* [B][8] k_state: prev path id, prev m, prev L, constant nodes, #factored edges, e0..e2 */
    int32_t* trim;                  /* [NSLOT*B][4] m = first memory point, L = first memory node, c = first trajectory   */
                                    /*     point (path-plane indices of THIS tick, OTH:586-598, 705-731), pref = #points    */
                                    /*     of vel_course; zero on first ticks                                               */
    double* vel_plan;               /* [B] planned velocity at the cut (OTH:572); the kernels read it through `vel`        */
    double* course;                 /* [B][n_export] vel_course (OTH:574): at most the rows of an exported trajectory      */
    double* obj_dist;               /* [B] s_obj - s_start on the cut follow path (OTH:774-784)                            */
    int32_t* zone_s0;               /* [B] start layer of the tick in which the scenario's zone was processed (GLNT:43-77:  */
                                    /*     the unblock window is evaluated once), -1: not yet; needed for zones in stateful  */
                                    /*     ticks, optional (NULL) otherwise                                                   */
    /* executed 'emergency' trajectory (sel_action = LTPL_ACT_EMERGENCY): get_ref_idx (OTH:518-601) reads the velocity of  */
    /* THAT trajectory; optional (NULL: such scenarios are flagged LTPL_SC_STATE_FALLBACK)                                 */
    double* em_vx;                  /* [B][n_export] f64 velocity of this tick's emergency trajectory (k_emergency)        */
    const double* prev_em_vx;       /* [B][n_export] the previous tick's                                                   */
    const int32_t* prev_em_info;    /* [B][3] the previous tick's em_info (all -1 when it had no emergency trajectory)     */
    /* location dependent friction: calc_vel_profile(local_gg={action: [ndarray(P, 2)]}) (OTH:649-666, VPFB:194-227).     */
    /* NULL: the constant params.gg_ax / gg_ay of the tuple form.  Rows are aligned with the path planes.                 */
    const double* gg;               /* [2][NSLOT*B][p_max] planes ax_max, ay_max per path point (without gg_scale)         */
    const double* prev_gg;          /* the previous tick's `gg` (brake on the backup plan, OTH:970-975); NULL: constant     */
} LtplBuffers;

/* stand-alone forward/backward ggv velocity profile over dense path arrays (BASELINE.json config 5).                   */
/* Replaces VpForwardBackward.calc_vel_profile -> tph.calc_vel_profile(closed=False) (VpForwardBackward.py:194-227).    */
typedef struct LtplVelBatch {
    int32_t n_paths, n_points; /* every path has n_points curvature values and n_points - 1 used element lengths         */
    const double* kappa;       /* [n_paths][n_points]                                                                    */
    const double* el;          /* [n_paths][n_points] (last column ignored)                                              */
    const double* v_start;     /* [n_paths]                                                                              */
    const double* v_end;       /* [n_paths]                                                                              */
    double* vx;                /* [n_paths][n_points]                                                                    */
    double* ax;                /* [n_paths][n_points] (last column 0)                                                    */
} LtplVelBatch;

int ltpl_version(void);
const char* ltpl_last_error(void);
int ltpl_sizeof(int which); /* 0 header, 1 params, 2 dims, 3 buffers, 4 velbatch: ABI self check for the ctypes mirror */

/* lattice handle over a caller-owned device blob -- replaces unpickling GraphBase (main_offline_callback.py:60-66)      */
/* Fills the blob's follow table (search on the unblocked lattice from every node: one kernel on the legacy default  */
/* stream, synchronised before returning) -- the blob is read-only afterwards.                                         */
int ltpl_lattice_create(const LtplLatticeHeader* header, void* dev_blob, LtplLattice** out);
int ltpl_lattice_destroy(LtplLattice* lat);

/* Graph_LTPL.set_startpos (LTPL:262-296 -> OTH.set_initial_pose OTH:181-270), batched                                   */
int ltpl_set_startpos_batch(const LtplLattice* lat, const LtplParams* prm, const LtplDims* dims, const LtplBuffers* buf,
                            void* stream);
/* Graph_LTPL.calc_paths (LTPL:300-340 -> OLI:75-153, OTH:289-516, MOPG:11-334, GLNT:13-222, GIE:5-63, GB:567-646,       */
/* GB:854-929), batched, first tick after set_startpos                                                                   */
int ltpl_calc_paths_batch(const LtplLattice* lat, const LtplParams* prm, const LtplDims* dims, const LtplBuffers* buf,
                          void* stream);
/* Graph_LTPL.calc_vel_profile (LTPL:344-408 -> OTH:518-601, 603-1040, VPFB, CVPF), batched                              */
int ltpl_calc_vel_profile_batch(const LtplLattice* lat, const LtplParams* prm, const LtplDims* dims,
                                const LtplBuffers* buf, void* stream);
/* calc_paths + calc_vel_profile back to back (one planning tick)                                                        */
/* stateful tick: start node + constant segment from the previous tick (replaces ltpl_set_startpos_batch  */
/* from the second tick on), then calc_paths / calc_vel_profile with the iterative memory                               */
int ltpl_next_calc_paths_batch(const LtplLattice* lat, const LtplParams* params, const LtplDims* dims,
                               const LtplBuffers* buffers, void* stream);       /* OTH:289-516 with memory           */
int ltpl_next_calc_vel_profile_batch(const LtplLattice* lat, const LtplParams* params, const LtplDims* dims,
                                     const LtplBuffers* buffers, void* stream); /* OTH:518-601 + 603-1040            */
int ltpl_next_tick_batch(const LtplLattice* lat, const LtplParams* params, const LtplDims* dims,
                         const LtplBuffers* buffers, void* stream);             /* both                              */
int ltpl_tick_batch(const LtplLattice* lat, const LtplParams* prm, const LtplDims* dims, const LtplBuffers* buf,
                    void* stream);
/* number of scenario windows a tick is split into (1 .. LTPL_MAX_SUB; default 4, or the environment variable           */
/* LTPL_SUBBATCHES at ltpl_lattice_create): window s runs its kernels on an internal stream forked from / joined into    */
/* the caller's stream (events), so k_plan of one window overlaps k_path / k_vel of another.  Results do not depend on it */
/* (only the order of the compact export rows, which is unspecified anyway).                                             */
int ltpl_set_subbatches(LtplLattice* lat, int n);
/* one kernel of the tick on its own (profiling / per-kernel roofline timing in bench.py):                               */
/* stage 0 k_startpos, 1 k_plan, 2 k_path, 3 k_vel, 4 k_export                                                            */
int ltpl_launch_stage(int stage, const LtplLattice* lat, const LtplParams* prm, const LtplDims* dims,
                      const LtplBuffers* buf, void* stream);
/* tph.calc_vel_profile(closed=False, loc_gg mode) over dense arrays                                                     */
int ltpl_velprofile_batch(const LtplParams* prm, const LtplVelBatch* vb, void* stream);

/* number of kernel launches issued by this library since load (bench.py "gpu_launches")                                 */
uint64_t ltpl_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* LTPL_B200_H */
