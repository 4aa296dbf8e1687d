#!/usr/bin/env python
"""
bench.py -- planning ticks/s of the batched online planning path (BASELINE.json metric) on N B200 GPUs.

    python bench.py --gpus N --steps K --warmup W            (N > 1: launched by torchrun, one rank per GPU)
    python bench.py --impl reference ...                     (CPU arm: oracle port on all host cores)

A "step" = one planning tick (calc_paths + calc_vel_profile, 3 kernels) over one batch of 10 000 synthetic scenarios
(SURVEY 8(d) config 2: Monteblanco lattice with lat_resolution=1.0, lon_straight_step=12.0 -> 216 layers x 7..12 nodes;
random ego arc length + 1..3 dynamic obstacles, seed 20260924).  set_startpos is setup (BASELINE.md section 2).
  value : device-timed (CUDA events on the launching stream), inputs resident in HBM, L2 flushed between steps
  e2e   : same metric through the public API Graph_LTPL.plan_stream with HOST buffers: per step host staging + H2D of
          the scenario arrays, set_startpos + tick kernels, D2H of the per-path arrays and of the kept trajectory rows,
          all inside the timed region (the D2H of step i overlaps the kernels of step i + 1)
  roofline / cpu_baseline : see DESIGN.md "Measurement"
Multi-GPU (config 3, "strong" scaling): the SAME seeded 10 000-scenario batch is sharded i % world over the ranks; the
lattice blob is NCCL-broadcast from rank 0 at init; the timed region of `value` holds the tick of every shard AND the
gather of all action sets into rank 0's HBM (parallel.PeerGather: the export kernels store their rows straight into the
consumer's memory over NVLink; fallback: point-to-point sends of the live rows).  The weak-scaling variant (10 000
scenarios per GPU, replicas, no gather) is reported under extra.weak.
"""

import argparse
import atexit
import json
import os
import shutil
import subprocess
import sys
import tempfile
import threading
import time

REPO = os.path.dirname(os.path.abspath(__file__))
if REPO not in sys.path:
    sys.path.insert(0, REPO)
# stdout carries exactly ONE JSON line.  NCCL prints its version banner (and any NCCL_DEBUG output) to the process's
# stdout, so file descriptor 1 is pointed at stderr for the whole run and the JSON line goes to a duplicate of the
# original stdout.
os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
sys.stdout.flush()
_JSON_OUT = os.fdopen(os.dup(1), "w")
os.dup2(2, 1)


def emit(line: dict) -> None:
    _JSON_OUT.write(json.dumps(line) + "\n")
    _JSON_OUT.flush()


import numpy as np  # noqa: E402

TRACK_CSV = os.path.join(REPO, "inputs", "traj_ltpl_cl", "traj_ltpl_cl_monteblanco.csv")
OFFLINE_INI = os.path.join(REPO, "params", "ltpl_config_offline.ini")
ONLINE_INI = os.path.join(REPO, "params", "ltpl_config_online.ini")
AXM_CSV = os.path.join(REPO, "inputs", "veh_dyn_info", "ax_max_machines.csv")
LATTICES = {"l216": {"lat_resolution": 1.0, "lon_straight_step": 12.0}, "default": {},
            "l430": {"lon_curve_step": 6.0, "lon_straight_step": 6.0, "lat_resolution": 0.5}}
WORKLOADS = {"l216": "config2: 10k scenarios x (ego start + 1-3 dynamic obstacles), Monteblanco 216 layers x 7-12 nodes "
                     "(lat_resolution=1.0, lon_straight_step=12.0)",
             "default": "10k scenarios x (ego start + 1-3 dynamic obstacles), Monteblanco shipped ini 128 layers x 13-25",
             "l430": "config4: 10k scenarios x 5 dynamic obstacles, Monteblanco 430 layers x 13-25 nodes"}
METRIC = "planning ticks/s (10k-scenario batch, ~200x11 lattice)"
SEED = 20260924


def ax_max_machines():
    tab = np.loadtxt(AXM_CSV, comments='#', delimiter=',')
    return np.vstack((tab, [100.0, tab[-1, 1]]))


def vel_kwargs():
    return dict(vel_max=100.0, gg_scale=1.0, local_gg=(5.0, 5.0), ax_max_machines=ax_max_machines(), safety_d=30.0)


_CACHE_DIR = []


def lattice_cache_path(tag):
    """The CPU workers load the lattice from this file, so it must be written somewhere writable even when the tree is
    read-only.  It is written fresh in a directory of this run: the cache key covers the input files but not the code,
    so a file left by another build could be stale.  Every run therefore builds its lattices anew, outside the timed
    regions."""
    if not _CACHE_DIR:
        _CACHE_DIR.append(tempfile.mkdtemp(prefix="ltpl_bench_"))
        atexit.register(shutil.rmtree, _CACHE_DIR[0], True)
    return os.path.join(_CACHE_DIR[0], "lattice_%s.npz" % tag)


def get_lattice(tag):
    from graphbasedlocaltrajectoryplanner_b200.lattice import load_or_build_lattice
    lat, _ = load_or_build_lattice(TRACK_CSV, OFFLINE_INI, store_path=lattice_cache_path(tag), overrides=LATTICES[tag])
    return lat


def make_batch(tag, batch, seed=SEED):
    from graphbasedlocaltrajectoryplanner_b200.scenarios import Track, make_scenarios
    omin, omax = (5, 5) if tag == "l430" else (1, 3)
    return make_scenarios(Track(TRACK_CSV), batch, seed=seed, n_obj_min=omin, n_obj_max=omax)


# ----------------------------------------------------------------------------------------------------------------------
# CPU arm: the oracle port (oracle/ltpl_oracle.py) on the host cores; only this leg may execute oracle/
# ----------------------------------------------------------------------------------------------------------------------
_W = {}
_ONE_THREAD = ("OPENBLAS_NUM_THREADS", "OMP_NUM_THREADS", "MKL_NUM_THREADS", "NUMEXPR_NUM_THREADS")


def _cpu_init(lat_path):
    from graphbasedlocaltrajectoryplanner_b200.lattice import Lattice
    from oracle.ltpl_oracle import OracleLTPL
    _W['orc'] = OracleLTPL(Lattice.load(lat_path))
    _W['vk'] = vel_kwargs()


def _cpu_work(args):
    pos, heading, vel, objs = args
    orc, vk = _W['orc'], _W['vk']
    t0 = time.perf_counter()
    for i in range(pos.shape[0]):
        ol = [{'id': k + 1, 'type': 'physical', 'X': o[0], 'Y': o[1], 'theta': o[2], 'v': o[3], 'length': o[4],
               'width': 2.5} for k, o in enumerate(objs[i])]
        orc.tick(pos[i], heading[i], vel[i], ol, vk)
    return pos.shape[0], time.perf_counter() - t0


def usable_cores():
    """host cores this process may use: the scheduler affinity mask, capped by the cgroup CPU quota (a container often
    sees every core of the box in os.cpu_count() but may only run on a few of them)."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    n = min(n, max(1, int(float(txt[0]) / float(txt[1]) + 0.5)))
            else:
                quota = int(txt[0])
                period = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
                if quota > 0:
                    n = min(n, max(1, int(quota / period + 0.5)))
            break
        except (OSError, ValueError, IndexError):
            continue
    return max(1, n)


class CpuArm(object):
    """`cores` worker processes, one oracle each, one BLAS thread each (main_min_example.py:8; the variables are set in
    the parent BEFORE the workers are spawned -- a child imports NumPy before its initializer runs).  A run hands every
    worker ONE chunk of `per_worker` scenarios (static partition: no dispatch noise) and waits for all of them."""

    def __init__(self, tag, cores=None):
        import multiprocessing as mp
        get_lattice(tag)   # make sure the cache file exists
        self.tag = tag
        self.cores = cores or usable_cores()
        keep = {k: os.environ.get(k) for k in _ONE_THREAD}
        for k in _ONE_THREAD:
            os.environ[k] = "1"
        try:
            ctx = mp.get_context("spawn")
            self.pool = ctx.Pool(self.cores, initializer=_cpu_init, initargs=(lattice_cache_path(tag),))
            warm = make_batch(tag, self.cores * 2, seed=1)
            self.pool.map(_cpu_work, [self._chunk(warm, 2 * i, 2 * i + 2) for i in range(self.cores)], chunksize=1)
        finally:
            for k, v in keep.items():
                if v is None:
                    os.environ.pop(k, None)
                else:
                    os.environ[k] = v

    @staticmethod
    def _chunk(sc, a, b):
        return (sc.pos[a:b], sc.heading[a:b], sc.vel[a:b],
                [sc.obj[i, :sc.n_obj[i]].tolist() for i in range(a, b)])

    def run(self, sc, workers=None):
        """wall time of one pass over `sc` with `workers` processes (default: all), and the summed in-worker time"""
        w = workers or self.cores
        n = sc.size
        per = (n + w - 1) // w
        chunks = [self._chunk(sc, a, min(a + per, n)) for a in range(0, n, per)]
        t0 = time.perf_counter()
        res = self.pool.map(_cpu_work, chunks, chunksize=1)
        dt = time.perf_counter() - t0
        assert sum(r[0] for r in res) == n
        return dt, sum(r[1] for r in res)

    def measure(self, per_worker=160, runs=2):
        """single-core ticks/s (one worker, per_worker scenarios) and all-core ticks/s (median of `runs` passes over
        cores x per_worker scenarios of the seeded batch); BASELINE.md section 2 asks for both.  When the workers
        share fewer physical cores than reported (in-worker time far above the single-core time) that is said."""
        sc = make_batch(self.tag, self.cores * per_worker)
        sc1 = sc.subset(np.arange(per_worker))
        t_one = self.run(sc1, workers=1)[0]
        passes = sorted(self.run(sc) for _ in range(runs))
        t_all, busy = passes[(runs - 1) // 2]
        return dict(all=sc.size / t_all, one=sc1.size / t_one, sample=sc.size, seconds_all=t_all, seconds_one=t_one,
                    per_worker=per_worker, runs=runs, parallel_efficiency=(sc.size / t_all) / (self.cores * sc1.size / t_one),
                    in_worker_slowdown=(busy / sc.size) / (t_one / sc1.size))

    def close(self):
        self.pool.close()
        self.pool.join()


def cpu_baseline_dict(arm, m):
    return {"value": m["all"], "unit": "ticks/s", "cores": arm.cores, "kind": "port",
            "ticks_per_s_cpu_allcores": m["all"], "ticks_per_s_cpu_1core": m["one"],
            "os_cpu_count": os.cpu_count(), "parallel_efficiency": m.get("parallel_efficiency"),
            "in_worker_slowdown_vs_1core": m.get("in_worker_slowdown"),
            "sample": "%d scenarios of the seeded workload (%d per worker process, %d processes, 1 BLAS thread each), "
                      "median of %d passes, %.2f s per pass; single core: %d scenarios in %.2f s" % (
                          m["sample"], m["per_worker"], arm.cores, m["runs"], m["seconds_all"], m["per_worker"],
                          m["seconds_one"]),
            "note": "float64 NumPy restatement of the reference path (oracle/ltpl_oracle.py); the reference itself needs "
                    "igraph + tph, not installable offline (its single-core rate on shims, measured in the build "
                    "container: profiles/r2_cpu_reference_shims.json)"}


# ----------------------------------------------------------------------------------------------------------------------
def clocks_sampler(gpu_index, stop_evt, out, ready_evt=None):
    q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
    try:
        p = subprocess.Popen(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader,nounits", "-lms", "20", "-i",
                              str(gpu_index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
    except OSError:
        if ready_evt is not None:
            ready_evt.set()
        return
    lines = []

    def reader():
        for line in p.stdout:
            lines.append(line)
            if ready_evt is not None:
                ready_evt.set()
    th = threading.Thread(target=reader, daemon=True)
    th.start()
    stop_evt.wait()
    p.terminate()
    th.join(timeout=2)
    sm, mx, reasons = [], [], set()
    for line in lines:
        f = [x.strip() for x in line.split(",")]
        if len(f) < 6:
            continue
        try:
            sm.append(float(f[0]))
            mx.append(float(f[1]))
        except ValueError:
            continue
        for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[2:6]):
            if val.lower().startswith("active"):
                reasons.add(name)
    if sm:
        out.update(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(mx)), reasons=sorted(reasons), samples=len(sm))


def algorithmic_bytes(lat, stats):
    """ALGORITHMIC bytes per launch of each kernel: inputs + outputs of the kernel, every logical array element once, with
    the element sizes the kernels use (float64 / int32); scratch is not counted.  Formulas: DESIGN.md section 5.
    k_plan is counted for the work the kernel DOES (one sample sweep per touched layer pair, table rows instead of
    searches where it reads them); `k_plan_as_reference` is the reference's work (three searches per tick)."""
    n_pairs = max(1, lat.num_layers)
    e_l = lat.num_edges / n_pairs                     # edges per layer pair
    s_l = lat.num_samples / n_pairs                   # samples per layer pair
    n_l = lat.num_nodes / lat.num_layers
    discs = 2.0 * stats["n_obj_sum"]                  # object + 0.2 s prediction (OLI:121-127)
    ah = stats["seg_sum"]                             # sum over found actions of path segments (H)
    pts = stats["pts_sum"]                            # sum over found actions of path points (P)
    pts_follow = stats["pts_follow_sum"]
    acts = stats["n_actions"]
    B = stats["batch"]
    plan_io = B * (16 + 8 + 8 + 4) + stats["n_obj_sum"] * 40 + B * stats["p0_mean"] * 16 + stats["nodes_sum"] * (8 + 4)
    plan = plan_io + discs * s_l * (16 + 4) + ah * (1 + 4)          # one shared sweep per object, table row per step
    plan_ref = plan_io + discs * 2 * s_l * (16 + 4) + ah * e_l * (8 + 4 + 0.125) + ah * n_l * 1
    path = pts * (5 * 8 + 8) + ah * (8 * 8 + 16 + 8 + 8 + 4) + acts * stats["p0_mean"] * 5 * 8 * 2
    # kappa, el in; s, vx, ax out; x, y in (follow); exported rows (first ticks: fused): x, y, psi, kappa in, 7 fp32 out
    vel = pts * (2 * 8 + 3 * 8) + pts_follow * (2 * 8) + stats["export_rows"] * (4 * 8 + 7 * 4)
    vel_fp32 = pts * (2 * 4 + 3 * 4) + pts_follow * (2 * 4) + stats["export_rows"] * (4 * 4 + 7 * 4)   # SURVEY 8(d) sizes
    # SURVEY 8(d) B_tick (fp32 / int32 element sizes, lattice gathers included), with the batch's own H, K, A, P
    s_e = lat.num_samples / max(1, lat.num_edges)
    b_tick = discs * 2 * e_l * s_e * 8 + ah * e_l * (4 + 4 + 0.125) + ah * n_l * 4 + pts * 20 \
        + (pts * 28 + (ah + acts) * 8 + ah * 32) + discs * 12 + B * 64
    return dict(k_plan=plan, k_path=path, k_vel=vel, k_plan_as_reference=plan_ref,
                k_vel_fp32_sizes=vel_fp32, tick_survey_8d=b_tick)


DUMP_BYTES = 64 << 20
DUMP_SAMPLE = 1024


def dump_outputs(pl, out_dir, seed=SEED):
    """The result of the planner's last tick as out_dir/<name>.npy: the per-path arrays of every scenario ([slot, B] or
    [B, ...]) and, for a fixed seeded sample of scenarios (sample.npy), the paths, node sequences, f64 trajectories
    (s, vx, ax) and exported f32 trajectory rows, indexed [slot, sample, ...] and zeroed past their lengths.  Exported
    rows are looked up through traj_row: the kernels claim them in a run-dependent order.  Everything is float64 except
    the exported rows (float32), at most DUMP_BYTES in all."""
    from graphbasedlocaltrajectoryplanner_b200 import capi
    f = pl.fetch("sc_flags", "start_node", "closest_obj", "action_id", "status", "path_len", "n_nodes", "traj_len",
                 "traj_id", "nodes", "node_idx", "path", "s_vx_ax", "traj", "traj_row")
    out = {k: f[k].astype(np.float64) for k in ("sc_flags", "start_node", "closest_obj", "action_id", "status",
                                                "path_len", "n_nodes", "traj_len", "traj_id")}
    B = pl.dims.batch
    nslot, _, H, _ = f["nodes"].shape
    P, NE = f["path"].shape[2], f["traj"].shape[1]
    per_scenario = nslot * (8 * P * (5 + 3) + 8 * H * (2 + 1) + 4 * NE * 7) + 8
    n = min(B, DUMP_SAMPLE, (DUMP_BYTES - sum(v.nbytes for v in out.values())) // per_scenario)
    idx = np.sort(np.random.default_rng(seed).choice(B, n, replace=False))
    q = np.arange(nslot)[:, None] * B + idx[None, :]                      # [slot, sample] -> row of path / s_vx_ax
    planned = f["action_id"][:, idx] != capi.ACT_NONE
    valid = planned & ((f["status"][:, idx] & capi.ST_TRAJ_VALID) != 0) & (f["traj_row"][:, idx] >= 0)
    on_path = (planned[..., None] & (np.arange(P) < f["path_len"][:, idx][..., None]))[..., None]
    on_traj = (valid[..., None] & (np.arange(P) < f["path_len"][:, idx][..., None]))[..., None]
    on_nodes = planned[..., None] & (np.arange(H) < f["n_nodes"][:, idx][..., None])
    on_rows = (valid[..., None] & (np.arange(NE) < f["traj_len"][:, idx][..., None]))[..., None]
    out["sample"] = idx.astype(np.float64)
    out["path"] = np.where(on_path, f["path"][:, q].transpose(1, 2, 3, 0), 0.0)
    out["s_vx_ax"] = np.where(on_traj, f["s_vx_ax"][:, q].transpose(1, 2, 3, 0), 0.0)
    out["nodes"] = np.where(on_nodes[..., None], f["nodes"][:, idx], -1).astype(np.float64)
    out["node_idx"] = np.where(on_nodes, f["node_idx"][:, idx], -1).astype(np.float64)
    out["traj"] = np.where(on_rows, f["traj"][np.where(valid, f["traj_row"][:, idx], 0)], np.float32(0.0))
    assert sum(v.nbytes for v in out.values()) <= DUMP_BYTES
    os.makedirs(out_dir, exist_ok=True)
    for name, arr in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), arr)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=10000, help="scenarios of the job (sharded over the GPUs)")
    ap.add_argument("--lattice", default="l216", choices=sorted(LATTICES))
    ap.add_argument("--cpu-per-worker", type=int, default=160, help="scenarios per CPU worker process and pass")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the extra lines (other lattices, stateful tick, config 5, weak)")
    ap.add_argument("--no-peer", action="store_true", help="multi-GPU gather by point-to-point sends instead of peer stores")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the result of the last timed step as DIR/<name>.npy (--gpus 1)")
    args = ap.parse_args()
    if args.dump_outputs and (args.gpus > 1 or args.impl != "b200"):
        ap.error("--dump-outputs writes the result of the GPU tick of --gpus 1")
    if args.warmup < 3:
        args.warmup = 3

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.gpus > 1 and world == 1:   # convenience: re-exec under torchrun
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(args.gpus),
               "--master-addr", "127.0.0.1", "--master-port", "29533", os.path.abspath(__file__)] + sys.argv[1:]
        sys.exit(subprocess.call(cmd))

    tag = args.lattice
    config = {"workload": WORKLOADS[tag], "lattice": tag, "job_batch": args.batch, "seed": SEED,
              "stateless_first_tick": True, "velocity_planner": "fb"}

    # ------------------------------------------------------------------------------------------------------------------
    if args.impl == "reference":
        if rank != 0:
            return
        arm = CpuArm(tag)
        sc = make_batch(tag, arm.cores * args.cpu_per_worker)
        for _ in range(args.warmup):
            arm.run(sc.subset(np.arange(min(sc.size, arm.cores * 4))))
        t = [arm.run(sc)[0] for _ in range(args.steps)]
        t_one = arm.run(sc.subset(np.arange(args.cpu_per_worker)), workers=1)[0]
        arm.close()
        total = float(np.sum(t))
        value = sc.size * args.steps / total
        m = dict(all=value, one=args.cpu_per_worker / t_one, sample=sc.size, seconds_all=total / args.steps,
                 seconds_one=t_one, per_worker=args.cpu_per_worker, runs=args.steps)
        emit(({
            "impl": "reference", "metric": METRIC, "value": value, "unit": "ticks/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps,
            "higher_is_better": True, "scaling": "strong" if args.gpus > 1 else "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": dict(config, cpu_sample=sc.size, step="one pass of all host cores over the sample"),
            "cpu_baseline": cpu_baseline_dict(arm, m),
            "e2e": {"value": value, "unit": "ticks/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}))
        return

    # ------------------------------------------------------------------------------------------------------------------
    cpu = None
    if rank == 0 and not args.no_cpu_baseline:   # before CUDA is initialised in this process (spawned workers)
        arm = CpuArm(tag)
        cpu = cpu_baseline_dict(arm, arm.measure(per_worker=args.cpu_per_worker, runs=3))
        arm.close()

    import ctypes as C

    import torch
    import torch.distributed as dist
    from graphbasedlocaltrajectoryplanner_b200 import capi, parallel
    from graphbasedlocaltrajectoryplanner_b200.Graph_LTPL import Graph_LTPL
    from graphbasedlocaltrajectoryplanner_b200.planner import BatchPlanner, read_online_config

    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(device)

    def max_over_ranks(x):
        if world == 1:
            return float(x)
        t = torch.tensor([x], dtype=torch.float64, device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    online = read_online_config(ONLINE_INI)
    # lattice: built on rank 0, broadcast as one byte blob (NCCL), every rank creates its own handle
    lat = get_lattice(tag) if rank == 0 or world == 1 else None
    packed_blob = None
    if world > 1:
        header, cap, blob_t = parallel.broadcast_lattice(lat, device, src=0)
        packed_blob = ((header, cap), blob_t)
        pl = BatchPlanner(online=online, device=device, packed=(header, cap), blob_tensor=blob_t)
        if lat is None:
            lat = get_lattice(tag)   # host-side statistics only
    else:
        pl = BatchPlanner(lat, online=online, device=device)
    pl.set_vel_params(**vel_kwargs())

    # the job's batch; N > 1: scenario i is planned by rank i % world (SURVEY 8(e), config 3)
    sc_job = make_batch(tag, args.batch, seed=SEED)
    sc = sc_job.shard(rank, world) if world > 1 else sc_job
    pl.stage_scenarios(sc)
    pl.upload()
    pl.set_startpos()
    torch.cuda.synchronize(device)

    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=device)   # > 126 MB L2
    stream = torch.cuda.current_stream(device)

    def timed_loop(fn, steps):
        """sum of per-step device times (CUDA events on the launching stream), L2 flushed before every step."""
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        for e0, e1 in evs:
            flush.fill_(1)
            e0.record(stream)
            fn()
            e1.record(stream)
        torch.cuda.synchronize(device)
        return sum(e0.elapsed_time(e1) for e0, e1 in evs) * 1e-3

    # multi-GPU: gather of all action sets into rank 0's HBM inside the timed region
    gather, gather_kind, gather_out = None, None, [None]
    if world > 1:
        if not args.no_peer:
            try:
                gather = parallel.PeerGather(pl, dst=0)
                gather.attach()
                gather_kind = "peer stores: k_export writes the live rows into rank 0's HBM over NVLink (symmetric memory) " \
                              "+ one peer copy of the per-path arrays + device-side barrier per tick"
            except Exception as e:   # noqa: BLE001
                gather = None
                gather_kind = "point-to-point sends of the live rows (peer memory unavailable: %s)" % str(e)[:120]
        else:
            gather_kind = "point-to-point sends of the live rows (--no-peer)"

    def step():
        pl.tick()
        if world > 1:
            if gather is not None:
                gather.finish()
            else:   # row count to the host, then sends of exactly the live rows + the packed per-path arrays
                n = int(pl.t["queue_cnt"][2].item())
                gather_out[0], _ = parallel.gather_rows(pl.t["traj"], n, dst=0, out=gather_out[0])

    for _ in range(args.warmup):
        step()
    clocks = {}
    stop_evt = threading.Event()
    ready_evt = threading.Event()
    th = threading.Thread(target=clocks_sampler, args=(local_rank, stop_evt, clocks, ready_evt), daemon=True)
    if rank == 0:
        th.start()
        ready_evt.wait(timeout=10.0)   # first nvidia-smi sample has arrived: the sampler covers the timed region
    barrier()
    l0 = pl.launch_count()
    t_dev = timed_loop(step, args.steps)
    launches = pl.launch_count() - l0
    barrier()
    t_dev = max_over_ranks(t_dev)
    value = args.batch * args.steps / t_dev
    if args.dump_outputs:
        dump_outputs(pl, args.dump_outputs)
    gathered_rows = None
    if world > 1 and rank == 0 and gather is not None:   # the consumer sees every rank's rows: count them
        gathered_rows = 0
        for rows, meta in gather.regions():
            v = pl._packed(pl._meta_spec, lambda n, m=meta: m)[1] if hasattr(pl, "_meta_spec") else None
            gathered_rows += int(v["queue_cnt"][2].item()) if v is not None else 0
    if gather is not None:
        gather.detach()

    def batch_stats(plx, scx):
        f = plx.fetch("sc_flags", "status", "action_id", "n_nodes", "path_len", "traj_len", "const_len")
        found = (f["status"] & capi.ST_FOUND) != 0
        st = dict(batch=scx.size, n_obj_sum=float(scx.n_obj.sum()), n_actions=float(found.sum()),
                  seg_sum=float(np.maximum(f["n_nodes"] - 2, 0)[found].sum()), nodes_sum=float(f["n_nodes"][found].sum()),
                  pts_sum=float(f["path_len"][found].sum()),
                  pts_follow_sum=float(f["path_len"][found & (f["action_id"] == capi.ACT_FOLLOW)].sum()),
                  export_rows=float(f["traj_len"].sum()), p0_mean=float(f["const_len"].mean()))
        bad = {name: int(((f["sc_flags"] & bit) != 0).sum()) for name, bit in (
            ("out_of_track", capi.SC_OUT_OF_TRACK), ("heading_mismatch", capi.SC_HEADING_MISMATCH),
            ("capacity", capi.SC_CAPACITY), ("brake_prefix", capi.SC_BRAKE_PREFIX))}
        return st, bad

    stage_names = {1: "k_plan", 2: "k_path", 3: "k_vel"}   # first tick: the export is fused into k_vel (k_vel_res)

    def kernel_times(plx, steps):
        """per-kernel device time (each kernel launched alone through ltpl_launch_stage, same buffers, L2 flushed)"""
        kt = {}
        for stage, name in stage_names.items():
            def one(stage=stage, name=name):
                capi.check(plx.lib, plx.lib.ltpl_launch_stage(stage, plx.handle, C.byref(plx.params), C.byref(plx.dims),
                                                              C.byref(plx.buf), plx.stream), name)
            for _ in range(3):
                one()
            kt[name] = timed_loop(one, steps) / steps
        return kt

    peaks_path = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.isfile(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (measured copy)"
    else:
        peak, peak_src = 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"
    try:
        traffic_tab = json.load(open(os.path.join(REPO, "profiles", "traffic.json")))
    except Exception:   # noqa: BLE001
        traffic_tab = {}

    def roofline_of(latx, tagx, stats, ktime, ms_step, blob_mb):
        alg = algorithmic_bytes(latx, stats)
        dom = max(ktime, key=ktime.get)
        achieved = alg[dom] / ktime[dom] / 1e9
        step_s = ms_step * 1e-3
        return {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": traffic_tab.get(tagx, {}).get(dom), "peak_source": peak_src,
                "algorithmic_bytes_per_launch": alg[dom],
                "algorithmic_bytes_definition": "inputs + outputs of the kernel, float64 / int32 as computed, no scratch",
                "kernel_ms": {k: 1e3 * v for k, v in ktime.items()},
                "kernel_share_of_step": {k: v / step_s for k, v in ktime.items()},
                "per_kernel_gbs": {k: alg[k] / ktime[k] / 1e9 for k in ktime},
                "per_kernel_frac": {k: alg[k] / ktime[k] / 1e9 / peak for k in ktime},
                "k_vel_frac_fp32_element_sizes": alg["k_vel_fp32_sizes"] / ktime["k_vel"] / 1e9 / peak,
                "k_plan_gbs_counted_as_reference_work": alg["k_plan_as_reference"] / ktime["k_plan"] / 1e9,
                "whole_tick": {"bytes_per_tick_survey_8d": alg["tick_survey_8d"] / stats["batch"],
                               "achieved_gbs": alg["tick_survey_8d"] / step_s / 1e9,
                               "frac": alg["tick_survey_8d"] / step_s / 1e9 / peak,
                               "bound_ticks_per_s": peak * 1e9 / (alg["tick_survey_8d"] / stats["batch"])},
                "note": "latency / issue bound: the lattice (%.1f MB) is L2-resident, DRAM traffic ~ compulsory bytes "
                        "(DESIGN.md section 5)" % blob_mb}

    stats, n_bad = batch_stats(pl, sc)
    ktime = kernel_times(pl, args.steps)

    # ------------------------------------------------------------------------------------------------------------------
    # e2e: public API with host buffers (pinned): H2D scenario arrays + set_startpos + tick + D2H action sets per step
    ltpl = Graph_LTPL.__new__(Graph_LTPL)
    ltpl._Graph_LTPL__planner = pl           # reuse the planner (same lattice handle / buffers)

    def feed(scx, n):
        for _ in range(n):
            yield scx      # the same host-side ScenarioBatch is staged, uploaded and planned every step

    def e2e_run(scx, steps):
        for out in ltpl.plan_stream(feed(scx, 3)):
            pass
        barrier()
        t0 = time.perf_counter()
        rows = 0
        for out in ltpl.plan_stream(feed(scx, steps)):
            rows += int(out["n_rows"])
        torch.cuda.synchronize(device)
        barrier()
        return max_over_ranks(time.perf_counter() - t0), rows, out

    t_e2e, rows, out = e2e_run(sc, args.steps)
    e2e_value = args.batch * args.steps / t_e2e
    rows_per_step = rows / args.steps
    if rank == 0:
        stop_evt.set()
        th.join(timeout=3)

    # third timing of SURVEY 8(d): the per-scenario Python view of one result (reference-style dicts)
    t0 = time.perf_counter()
    unpacked = Graph_LTPL.unpack_batch(out)              # lazy per-scenario view (index arrays, no Python loop)
    first = unpacked[0]
    t_unpack = time.perf_counter() - t0
    t0 = time.perf_counter()
    n_dicts = sum(1 for _ in unpacked)                   # ... and every scenario's two dicts materialised
    t_unpack_all = time.perf_counter() - t0
    assert len(unpacked) == sc.size == n_dicts and isinstance(first, tuple)

    # ------------------------------------------------------------------------------------------------------------------
    # weak scaling (N > 1): every rank plans its own 10 000-scenario batch, replicas, no gather
    weak = None
    if world > 1 and not args.no_extra:
        pl_w = BatchPlanner(online=online, device=device, packed=packed_blob[0], blob_tensor=packed_blob[1])
        pl_w.set_vel_params(**vel_kwargs())
        sc_w = make_batch(tag, args.batch, seed=SEED + rank)
        pl_w.stage_scenarios(sc_w)
        pl_w.upload()
        pl_w.set_startpos()
        for _ in range(args.warmup):
            pl_w.tick()
        barrier()
        tw = max_over_ranks(timed_loop(pl_w.tick, args.steps))
        ltpl._Graph_LTPL__planner = pl_w
        tw_e2e, _, _ = e2e_run(sc_w, args.steps)
        ltpl._Graph_LTPL__planner = pl
        weak = {"scaling": "weak", "per_gpu_batch": args.batch, "value": world * args.batch * args.steps / tw,
                "ms_per_step": 1e3 * tw / args.steps, "e2e_value": world * args.batch * args.steps / tw_e2e,
                "e2e_ms_per_step": 1e3 * tw_e2e / args.steps,
                "mode": "replicas: every rank keeps its action sets (rank-local consumers), no gather"}
        del pl_w

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    ms_step = 1e3 * t_dev / args.steps
    blob_mb = pl.blob.numel() / 1e6
    # per-kernel times were taken on this rank's shard; the step of `value` additionally holds the gather (N > 1)
    roofline = roofline_of(lat, tag, stats, ktime, 1e3 * sum(ktime.values()) if world > 1 else ms_step, blob_mb)
    result = {
        "metric": METRIC, "value": value, "unit": "ticks/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True,
        "scaling": "strong" if world > 1 else "weak",
        "vs_baseline": None, "dtype": "f64 (decisions, splines, arc lengths) + f32 (velocity recurrences)",
        "data": "synthetic",
        "config": dict(config, l2="256 MiB buffer written before every timed step (L2 = 126 MB)",
                       scenarios_per_gpu=sc.size, actions_per_tick=stats["n_actions"] / sc.size,
                       path_points_per_action=stats["pts_sum"] / max(stats["n_actions"], 1),
                       scenarios_flagged=n_bad,
                       parallelism="%d GPU(s): the seeded batch sharded i %% world, lattice broadcast once" % world
                       + ("; timed region = tick of every shard + gather of all action sets into rank 0's HBM (%s)"
                          % gather_kind if world > 1 else "")),
        "e2e": {"value": e2e_value, "unit": "ticks/s", "h2d_bytes_per_step": pl.h2d_bytes(),
                "d2h_bytes_per_step": pl.d2h_bytes(int(rows_per_step)), "ms_per_step": 1e3 * t_e2e / args.steps,
                "kept_trajectories_per_step": rows_per_step, "facade_unpack_ms_per_batch": 1e3 * t_unpack,
                "facade_unpack_all_scenario_dicts_ms": 1e3 * t_unpack_all,
                "api": "Graph_LTPL.plan_stream: per step host staging + H2D + set_startpos + calc_paths + "
                       "calc_vel_profile + D2H of the compact action sets; D2H of step i overlaps the kernels of step "
                       "i+1 (copy stream, 3 buffer sets)" + ("; every rank stages / uploads its shard and downloads its "
                                                              "shard's action sets (bytes per rank)" if world > 1 else "")},
        "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline}
    if gathered_rows is not None:
        result["config"]["rows_in_rank0_hbm_after_gather"] = gathered_rows
    if cpu is not None:
        result["cpu_baseline"] = cpu
    extra = {}
    if weak is not None:
        extra["weak"] = weak

    if not args.no_extra and world == 1:
        def side_line(tagx, key):
            """another lattice as a first-class line: ticks/s, per-kernel split and roofline like the headline"""
            try:
                lat_x = get_lattice(tagx)
                pl_x = BatchPlanner(lat_x, online=online, device=device)
                pl_x.set_vel_params(**vel_kwargs())
                sc_x = make_batch(tagx, args.batch)
                pl_x.stage_scenarios(sc_x)
                pl_x.upload()
                pl_x.set_startpos()
                for _ in range(args.warmup):
                    pl_x.tick()
                tx = timed_loop(pl_x.tick, args.steps)
                st_x, bad_x = batch_stats(pl_x, sc_x)
                kt_x = kernel_times(pl_x, args.steps)
                extra[key] = {"workload": WORKLOADS[tagx], "ticks_per_s": args.batch * args.steps / tx,
                              "ms_per_step": 1e3 * tx / args.steps,
                              "actions_per_tick": st_x["n_actions"] / args.batch, "scenarios_flagged": bad_x,
                              "lattice": {"layers": lat_x.num_layers, "nodes": lat_x.num_nodes, "edges": lat_x.num_edges},
                              "roofline": roofline_of(lat_x, tagx, st_x, kt_x, 1e3 * tx / args.steps,
                                                      pl_x.blob.numel() / 1e6)}
                del pl_x
            except Exception as e:   # noqa: BLE001
                extra[key + "_error"] = str(e)[:300]
        side_line("default", "default_lattice")   # shipped ini: 128 layers x 13-25 nodes, 14 k edges (the DP workload)
        side_line("l430", "config4_l430")         # SURVEY 8(d) config 4: 430 layers, 5 objects

        try:   # stateful ticks (DESIGN.md section 11): closed loop of 8 ticks on the bench workload; a
            # vehicle dummy advances every scenario 0.1 s on its first kept trajectory; the loop is recorded once
            # (untimed host work between the ticks) and replayed with CUDA events around every next_tick
            from graphbasedlocaltrajectoryplanner_b200.scenarios import ScenarioBatch
            pl_s = BatchPlanner(lat, online=online, device=device, stateful=True)
            pl_s.set_vel_params(**vel_kwargs())
            n_loop, dt_loop = 8, 0.1

            def first_tick():
                pl_s.stage_scenarios(sc)
                pl_s.upload()
                pl_s.set_startpos()
                pl_s.tick()

            def advance(out):
                rows = out["traj_row"].numpy()
                lens = out["traj_len"].numpy()
                acts = out["action_id"].numpy()
                slot = np.argmax(rows >= 0, axis=0)                      # first kept trajectory of every scenario
                bidx = np.arange(rows.shape[1])
                ok = rows[slot, bidx] >= 0
                r = np.where(ok, rows[slot, bidx], 0)
                tr = out["traj"].numpy()[r].astype(np.float64)           # (B, 115, 7)
                n = np.maximum(lens[slot, bidx], 2)
                s_t = tr[:, 0, 0] + np.maximum(tr[:, 0, 5] * dt_loop + 0.5 * tr[:, 0, 6] * dt_loop ** 2, 0.0)
                valid = np.arange(tr.shape[1])[None, :] < n[:, None]
                i0 = np.clip((np.where(valid, tr[:, :, 0], np.inf) <= s_t[:, None]).sum(axis=1) - 1, 0, n - 2)
                s0, s1 = tr[bidx, i0, 0], tr[bidx, i0 + 1, 0]
                f = np.clip((s_t - s0) / np.maximum(s1 - s0, 1e-9), 0.0, 1.0)
                lerp = lambda c: tr[bidx, i0, c] * (1 - f) + tr[bidx, i0 + 1, c] * f   # noqa: E731
                return np.column_stack((lerp(1), lerp(2))), lerp(5), np.where(ok, acts[slot, bidx], 0), ok

            first_tick()
            rec_in = []
            pos_e, vel_e = sc.pos.copy(), sc.vel.copy()
            for _ in range(n_loop):
                out_s = pl_s.download()
                p_new, v_new, sel_a, ok = advance(out_s)
                pos_e, vel_e = np.where(ok[:, None], p_new, pos_e), np.where(ok, v_new, vel_e)
                rec_in.append((pos_e.copy(), vel_e.copy(), sel_a.astype(np.int32)))
                sc_k = ScenarioBatch(pos_e.copy(), sc.heading, sc.vel, sc.n_obj, sc.obj)
                pl_s.next_tick(sc_k, sel_a, 2.0 * dt_loop, vel_est=vel_e)
            torch.cuda.synchronize(device)
            flags = pl_s.fetch("sc_flags")["sc_flags"]
            first_tick()
            t_st, t_wall, t_dev = 0.0, 0.0, 0.0
            e_dev = [None]

            def mark_device_start():
                e_dev[0] = torch.cuda.Event(enable_timing=True)
                e_dev[0].record(stream)
            pl_s.on_device_start = mark_device_start
            for pos_k, vel_k, sel_k in rec_in:
                sc_k = ScenarioBatch(pos_k, sc.heading, sc.vel, sc.n_obj, sc.obj)
                flush.fill_(1)
                torch.cuda.synchronize(device)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                w0 = time.perf_counter()
                e0.record(stream)
                pl_s.next_tick(sc_k, sel_k, 2.0 * dt_loop, vel_est=vel_k)
                e1.record(stream)
                torch.cuda.synchronize(device)
                t_wall += time.perf_counter() - w0
                t_st += e0.elapsed_time(e1) * 1e-3
                t_dev += e_dev[0].elapsed_time(e1) * 1e-3
            pl_s.on_device_start = None
            extra["stateful_tick"] = {"ticks_per_s": args.batch * n_loop / t_st, "ms_per_tick": 1e3 * t_st / n_loop,
                                      "wall_ms_per_tick_incl_host_staging": 1e3 * t_wall / n_loop,
                                      "device_ms_per_tick_after_host_staging": 1e3 * t_dev / n_loop,
                                      "ticks": n_loop, "scenarios_still_planned_at_the_end": int((flags == 0).sum()),
                                      "flags_at_the_end": {name: int(((flags & bit) != 0).sum()) for name, bit in (
                                          ("out_of_track", capi.SC_OUT_OF_TRACK),
                                          ("heading_mismatch", capi.SC_HEADING_MISMATCH), ("capacity", capi.SC_CAPACITY),
                                          ("brake_prefix", capi.SC_BRAKE_PREFIX),
                                          ("state_fallback", capi.SC_STATE_FALLBACK))},
                                      "note": "closed loop, 0.1 s per tick; device time of one next_tick incl. its ONE "
                                              "packed input upload and the carry copy of the per-path arrays"}
            del pl_s
        except Exception as e:   # noqa: BLE001
            extra["stateful_tick_error"] = str(e)[:300]
        try:   # SURVEY 8(d) config 5: 100 k paths x 500 points forward/backward solver
            from graphbasedlocaltrajectoryplanner_b200.scenarios import make_velocity_microbench
            from graphbasedlocaltrajectoryplanner_b200.velprofile import velprofile_batch_device
            mb = make_velocity_microbench(100000, 500)
            d = {k: torch.from_numpy(np.ascontiguousarray(mb[k])).to(device) for k in ("kappa", "el", "v_start", "v_end")}
            vx = torch.empty_like(d["kappa"])
            ax = torch.empty_like(d["kappa"])
            pl.set_vel_params(vel_max=60.0, gg_scale=1.0, local_gg=(5.0, 5.0), ax_max_machines=ax_max_machines(),
                              safety_d=30.0)

            def vp():
                velprofile_batch_device(pl, d["kappa"], d["el"], d["v_start"], d["v_end"], vx, ax)
            for _ in range(3):
                vp()
            tv = timed_loop(vp, 10) / 10
            nbytes = 100000 * 500 * 4 * 8
            extra["velprofile_100k_x_500"] = {
                "ms": 1e3 * tv, "paths_per_s": 100000 / tv, "algorithmic_GBps": nbytes / tv / 1e9,
                "frac_of_peak": nbytes / tv / 1e9 / peak,
                "frac_of_peak_fp32_element_sizes": nbytes / 2 / tv / 1e9 / peak,
                "traffic": traffic_tab.get("velprofile", {}).get("k_velprofile"),
                "dtype": "kappa, el in; vx, ax out as float64 = 32 B / point (SURVEY 8(d): 16 B / point in fp32)"}
        except Exception as e:   # noqa: BLE001
            extra["velprofile_error"] = str(e)[:200]
    if extra:
        result["extra"] = extra

    emit(result)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
