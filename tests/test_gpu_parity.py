"""GPU parity tests proper: the CUDA path (through the C-ABI) against
  (1) the committed golden vectors of the unmodified reference (tests/golden/*.npz), and
  (2) the float64 oracle on fresh seeded scenario batches.
Node sequences bit-exact; coordinates / velocities within 1e-4 relative (absolute floors in tests/helpers.py)."""
import numpy as np
import pytest

from tests import helpers as H

pytestmark = pytest.mark.gpu

VEL = dict(vel_max=100.0, gg_scale=1.0, local_gg=(5.0, 5.0), safety_d=30.0)


SUBBATCHES = {"default": 3, "l216": 4, "l430": 1, "open": 5, "layers14": 2}   # scenario windows inside the library


def _planner(tag):
    from graphbasedlocaltrajectoryplanner_b200.planner import BatchPlanner
    pl = BatchPlanner(H.lattice_for(tag), device="cuda:0")
    pl.set_subbatches(SUBBATCHES[tag])   # explicit: also for these small batches (uneven windows incl.)
    return pl


def _run_batch(pl, sc, axm):
    pl.set_vel_params(ax_max_machines=axm, **VEL)
    pl.stage_scenarios(sc)
    pl.upload()
    pl.set_startpos()
    pl.calc_paths()
    pl.calc_vel_profile()
    return pl.records()


def _collect(fn, n):
    fails = []
    for b in range(n):
        try:
            fn(b)
        except AssertionError as e:   # noqa: PERF203
            fails.append(str(e).split("\n")[0][:300])
    return fails


@pytest.mark.parametrize("tag", ["default", "l216", "l430", "open", "layers14"])
def test_cuda_matches_reference_golden(tag):
    from graphbasedlocaltrajectoryplanner_b200.scenarios import ScenarioBatch
    g = H.golden("ticks_%s.npz" % tag)
    sc = ScenarioBatch(g["sc_pos"], g["sc_heading"], g["sc_vel"], g["sc_n_obj"], g["sc_obj"])
    recs = _run_batch(_planner(tag), sc, g["ax_max_machines"])
    fails = _collect(lambda b: H.compare_record(recs[b], g, b, ctx=tag), sc.size)
    assert not fails, "%d/%d scenarios differ from the reference golden vectors:\n%s" % (
        len(fails), sc.size, "\n".join(fails[:10]))


def test_cuda_config1_min_example():
    from graphbasedlocaltrajectoryplanner_b200.scenarios import ScenarioBatch
    g = H.golden("config1_min_example.npz")
    obj = np.tile(g["obj"][None, None, :], (2, 1, 1))
    sc = ScenarioBatch(g["sc_pos"], g["sc_heading"], g["sc_vel"], np.ones(2, dtype=np.int32), obj)
    pl = _planner("default")
    pl.set_vel_params()     # API defaults of calc_vel_profile (LTPL:344-352)
    pl.stage_scenarios(sc)
    pl.upload()
    pl.set_startpos()
    pl.calc_paths()
    pl.calc_vel_profile()
    recs = pl.records()
    for b in range(2):
        H.compare_record(recs[b], g, b, prefix="", ctx="config1")


@pytest.mark.parametrize("tag,n,omin,omax", [("default", 384, 0, 3), ("l216", 256, 1, 3), ("l430", 128, 5, 5), ("open", 256, 0, 3), ("layers14", 128, 0, 3)])
def test_cuda_matches_oracle_seeded(tag, n, omin, omax):
    """fresh seeded batches (different seed than the golden files), oracle as the checker."""
    from graphbasedlocaltrajectoryplanner_b200.scenarios import Track, make_scenarios
    from oracle.ltpl_oracle import OracleLTPL
    g = H.golden("ticks_%s.npz" % tag)
    axm = g["ax_max_machines"]
    track = Track(H.track_csv_for(tag))
    sc = make_scenarios(track, n, seed=4242 + n, n_obj_min=omin, n_obj_max=omax,
                        s_max=(track.length - 8.0) if tag == "open" else None)
    recs = _run_batch(_planner(tag), sc, axm)
    orc = OracleLTPL(H.lattice_for(tag))
    vk = dict(ax_max_machines=axm, **VEL)

    def one(b):
        want = orc.tick(sc.pos[b], sc.heading[b], sc.vel[b], sc.object_list(b), vk)
        H.compare_records(recs[b], want, ctx="%s scenario %d" % (tag, b))
    fails = _collect(one, sc.size)
    assert not fails, "%d/%d scenarios differ from the oracle:\n%s" % (len(fails), sc.size, "\n".join(fails[:10]))


def test_plan_stream_pipelining_matches_plan_batch(tmp_path):
    """the pipelined end-to-end API (two export buffers, D2H overlapping the next step) returns, for every step, the
    same action sets as the synchronous plan_batch call."""
    from graphbasedlocaltrajectoryplanner_b200.Graph_LTPL import Graph_LTPL
    from graphbasedlocaltrajectoryplanner_b200.scenarios import Track, make_scenarios
    g = H.golden("ticks_default.npz")
    pd = {'globtraj_input_path': H.TRACK_CSV, 'graph_store_path': str(tmp_path / "lattice_default.npz"),
          'ltpl_offline_param_path': H.OFFLINE_INI, 'ltpl_online_param_path': H.ONLINE_INI}
    ltpl = Graph_LTPL(path_dict=pd, log_to_file=False, device="cuda:0")
    ltpl.graph_init()
    ltpl.planner.set_vel_params(ax_max_machines=g["ax_max_machines"], **VEL)
    tr = Track(H.TRACK_CSV)
    batches = [make_scenarios(tr, 512, seed=100 + i, n_obj_min=0, n_obj_max=3) for i in range(5)]

    def snapshot(out):
        n = int(out["n_rows"])
        order = np.argsort(out["exp_q"][:n].numpy())          # rows are appended in arbitrary (atomic) order
        return (n, out["exp_q"][:n].numpy()[order].copy(), out["traj"][:n].numpy()[order].copy(),
                out["traj_len"].numpy().copy(), out["action_id"].numpy().copy(), out["status"].numpy().copy())

    want = [snapshot(ltpl.plan_batch(sc)) for sc in batches]
    got = [snapshot(out) for out in ltpl.plan_stream(iter(batches))]
    assert len(got) == len(want) == 5
    for a, b in zip(got, want):
        assert a[0] == b[0] and a[0] > 0
        for x, y in zip(a[1:], b[1:]):
            assert np.array_equal(x, y)
    # rows <-> paths bookkeeping
    out = ltpl.plan_batch(batches[0])
    n = int(out["n_rows"])
    rows = out["traj_row"].numpy().reshape(-1)
    q = out["exp_q"][:n].numpy()
    assert np.array_equal(rows[q], np.arange(n)) and int((rows >= 0).sum()) == n
