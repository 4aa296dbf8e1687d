"""host-side logic that needs no GPU: C-ABI library loads and exports every declared symbol, struct mirrors match,
scenario generator, facade argument checks, product never imports the oracle, NCCL plumbing on gloo (world size 2)."""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from tests import helpers as H


def test_capi_library_exports_every_declared_symbol():
    from graphbasedlocaltrajectoryplanner_b200 import capi
    capi.build_library()
    lib = capi.load_library()
    header = open(os.path.join(H.REPO, "include", "ltpl_b200.h")).read()
    declared = set(re.findall(r"\b(ltpl_[a-z_0-9]+)\s*\(", header))
    assert declared == set(capi.EXPORTS), declared ^ set(capi.EXPORTS)
    for name in declared:
        assert hasattr(lib, name), name
    assert lib.ltpl_version() == capi.ABI_VERSION
    for which, st in enumerate((capi.LatticeHeader, capi.Params, capi.Dims, capi.Buffers, capi.VelBatch)):
        assert lib.ltpl_sizeof(which) == ctypes.sizeof(st)
    # error convention without touching a GPU: null arguments are rejected with a message
    assert lib.ltpl_lattice_create(None, None, None) != 0
    assert b"null" in lib.ltpl_last_error()


def test_product_does_not_import_oracle():
    pkg = os.path.join(H.REPO, "graphbasedlocaltrajectoryplanner_b200")
    for root, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh")):
                src = open(os.path.join(root, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle", src, flags=re.M), f
    for f in os.listdir(os.path.join(H.REPO, "tools")):   # GPU tuning / profiling helpers: no checker needed, none used
        if f.endswith(".py"):
            assert not re.search(r"^\s*(from|import)\s+oracle", open(os.path.join(H.REPO, "tools", f)).read(), flags=re.M), f


def test_missing_gpu_fails_loudly():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from graphbasedlocaltrajectoryplanner_b200.planner import BatchPlanner
    with pytest.raises(RuntimeError):
        BatchPlanner(H.lattice_for("l216"))


def test_scenarios_deterministic_and_in_track():
    from graphbasedlocaltrajectoryplanner_b200.scenarios import Track, make_scenarios, ScenarioBatch
    from oracle.ltpl_oracle import OracleLTPL, check_inside_bounds
    tr = Track(H.TRACK_CSV)
    a = make_scenarios(tr, 64, seed=5)
    b = make_scenarios(tr, 64, seed=5)
    assert np.array_equal(a.obj, b.obj) and np.array_equal(a.pos, b.pos)
    assert a.n_obj.min() >= 1 and a.n_obj.max() <= 3
    orc = OracleLTPL(H.lattice_for("l216"))
    inside = [check_inside_bounds(orc.bound1, orc.bound2, a.pos[i]) for i in range(a.size)]
    assert all(inside)
    sh = a.shard(1, 2)
    assert sh.size == 32 and np.array_equal(sh.pos[0], a.pos[1])
    ol = a.object_list(0)
    rt = ScenarioBatch.from_object_lists([a.pos[0]], [a.heading[0]], [a.vel[0]], [ol], k_max=3)
    assert np.allclose(rt.obj[0, :len(ol)], a.obj[0, :len(ol)])


def test_facade_argument_checks(tmp_path):
    from graphbasedlocaltrajectoryplanner_b200.Graph_LTPL import Graph_LTPL
    with pytest.raises(ValueError):   # LTPL:62-68 missing path entries
        Graph_LTPL(path_dict={'globtraj_input_path': H.TRACK_CSV}, log_to_file=False)
    pd = {'globtraj_input_path': H.TRACK_CSV, 'graph_store_path': str(tmp_path / "lattice_default.npz"),
          'ltpl_offline_param_path': H.OFFLINE_INI, 'ltpl_online_param_path': H.ONLINE_INI}
    obj = Graph_LTPL(path_dict=pd, log_to_file=False)
    with pytest.raises(ValueError):   # LTPL:277-280 graph not initialised
        obj.set_startpos(np.zeros(2), 0.0)


GLOO_SCRIPT = r'''
import os, sys
sys.path.insert(0, %(repo)r)
import numpy as np, torch, torch.distributed as dist
from tests import helpers as H
from graphbasedlocaltrajectoryplanner_b200 import parallel
dist.init_process_group("gloo")
rank, world = dist.get_rank(), dist.get_world_size()
lat = H.lattice_for("l216") if rank == 0 else None
header, cap, blob = parallel.broadcast_lattice(lat, torch.device("cpu"), src=0)
ref = H.lattice_for("l216")
from graphbasedlocaltrajectoryplanner_b200.lattice_blob import pack_lattice
h2, blob2, cap2 = pack_lattice(ref)
assert bytes(header) == bytes(h2) and cap == cap2 and np.array_equal(blob.numpy(), blob2)
# gather of the LIVE rows only: rank r holds 2 + 3 r live rows of a compact export buffer with 9 rows
rows = torch.full((9, 5, 7), float(rank), dtype=torch.float32)
n_live = 2 + 3 * rank
got, counts = parallel.gather_rows(rows, n_live, dst=0)
assert counts == [2 + 3 * r for r in range(world)]
if rank == 0:
    assert got.shape == (sum(counts), 5, 7)
    off = 0
    for r in range(world):
        assert float(got[off:off + counts[r]].min()) == r == float(got[off:off + counts[r]].max())
        off += counts[r]
else:
    assert got is None
# a rank without live rows takes part without sending
got, counts = parallel.gather_rows(rows, 0 if rank == 1 else 4, dst=0)
assert counts == [4, 0] and (rank != 0 or got.shape[0] == 4)
assert parallel.shard_indices(10, rank, world).tolist() == list(range(rank, 10, world))
# the shards of a seeded batch: scenario i on rank (i mod world), together exactly the batch
from graphbasedlocaltrajectoryplanner_b200.scenarios import Track, make_scenarios
sc = make_scenarios(Track(H.TRACK_CSV), 11, seed=5)
sh = sc.shard(rank, world)
assert sh.size == len(range(rank, 11, world)) and np.array_equal(sh.pos, sc.pos[rank::world])
dist.destroy_process_group()
print("rank", rank, "ok")
'''


def test_parallel_plumbing_gloo_world2(tmp_path):
    script = tmp_path / "gloo_w2.py"
    script.write_text(GLOO_SCRIPT % {"repo": H.REPO})
    res = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                          "--master-addr", "127.0.0.1", "--master-port", "29577", str(script)],
                         stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600)
    assert res.returncode == 0 and res.stdout.count("ok") == 2, res.stdout[-2000:]


def test_zone_ids_and_masks_of_a_scenario_batch():
    """set_zones: zones are de-duplicated by content, identified by the crc of their id (a stateful planner processes a zone
    anew when the id changes, OLI:155-237), and travel through subset() / shard()."""
    from graphbasedlocaltrajectoryplanner_b200.scenarios import ScenarioBatch
    z1 = [[3, 3, 4], [0, 1, 0], np.zeros((2, 2)), np.zeros((2, 2))]
    z2 = [[7], [2], np.zeros((2, 2)), np.zeros((2, 2))]
    sc = ScenarioBatch.from_object_lists(np.zeros((4, 2)), np.zeros(4), np.ones(4), [[], [], [], []],
                                         blocked_zones=[{"a": z1}, None, {"b": z1}, {"a": z2}])
    assert sc.zone_sel.tolist() == [0, -1, 0, 1] and len(sc.zones) == 2          # same content -> same mask
    assert sc.zone_key[1] == 0 and sc.zone_key[0] == sc.zone_key[3] != sc.zone_key[2] and sc.zone_key[0] > 0
    sub = sc.subset([3, 1])
    assert sub.zone_sel.tolist() == [1, -1] and sub.zone_key.tolist() == [int(sc.zone_key[3]), 0]
    assert sc.shard(1, 2).zone_key.tolist() == [0, int(sc.zone_key[3])]
    with pytest.raises(NotImplementedError):
        ScenarioBatch.from_object_lists(np.zeros((1, 2)), np.zeros(1), np.ones(1), [[]], blocked_zones=[{"a": z1, "b": z2}])
    plain = ScenarioBatch.from_object_lists(np.zeros((2, 2)), np.zeros(2), np.ones(2), [[], []])
    assert plain.zones is None and plain.zone_key is None


def test_nearest_vertex_grid_bounds_the_argmin():
    """lattice_blob.nearest_grid: for random positions around the track the candidates of the position's cell contain
    np.argmin's answer (first minimum) of the scan over the whole polyline -- closed and open track."""
    from graphbasedlocaltrajectoryplanner_b200 import lattice_blob as LB
    rng = np.random.default_rng(7)
    for tag in ("l216", "open"):
        lat = H.lattice_for(tag)
        LB.pack_lattice(lat)
        g = lat._nearest_grids
        polys = dict(refline=lat.refline, raceline=lat.raceline, glob=np.ascontiguousarray(lat.glob_rl[:-1, 1:3]))
        for name, pts in polys.items():
            n = pts.shape[0]
            q = pts[rng.integers(0, n, 4000)] + rng.normal(0.0, 10.0, (4000, 2))
            q[:200] = pts[rng.integers(0, n, 200)]                       # exactly on vertices
            ix = np.floor((q[:, 0] - g["x0"]) / LB.GRID_CELL).astype(int)
            iy = np.floor((q[:, 1] - g["y0"]) / LB.GRID_CELL).astype(int)
            ent = g[name][iy, ix]
            cnt, first = ent & 63, ent >> 6
            d2 = ((q[:, None, :] - pts[None]) ** 2).sum(-1)
            full = d2.argmin(axis=1)
            assert (cnt > 0).mean() > 0.95 and cnt.max() <= LB.GRID_MAX_COUNT
            for i in np.nonzero(cnt > 0)[0]:
                idx = first[i] + np.arange(cnt[i])
                idx = idx % n if lat.closed else idx
                assert idx.max() < n
                dd = d2[i, idx]
                assert idx[dd == dd.min()].min() == full[i], (tag, name, i)
