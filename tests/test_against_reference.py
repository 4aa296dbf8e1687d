"""Differential test of the oracle against the unmodified reference on the scenarios of seed 86420.

The expected arrays are the reference's own output (graph_ltpl @ 18763ef9, one first tick per scenario through its
public API), produced by ``python -m oracle.gen_golden --seed86420-only`` and stored as
tests/golden/ticks_seed86420_<tag>.npz, so the comparison needs neither the reference checkout nor its dependencies.
python-igraph==0.8.2 and trajectory_planning_helpers==0.75 are not installable offline, so the reference ran on their
restatements under oracle/shims; what stays unpinned by that is the third-party arithmetic itself (tph functions,
igraph's heap order on exact ties)."""
import pytest

from tests import helpers as H


@pytest.mark.parametrize("tag,n,omin,omax", [("default", 48, 0, 3), ("l216", 24, 1, 3)])
def test_oracle_matches_stored_reference_ticks(tag, n, omin, omax):
    from oracle.ltpl_oracle import OracleLTPL
    g = H.golden("ticks_seed86420_%s.npz" % tag)
    assert g["sc_pos"].shape[0] == n and omin <= g["sc_n_obj"].min() and g["sc_n_obj"].max() <= omax
    vk = dict(vel_max=100.0, gg_scale=1.0, local_gg=(5.0, 5.0), ax_max_machines=g["ax_max_machines"], safety_d=30.0)
    orc = OracleLTPL(H.lattice_for(tag))
    compared = 0
    for b in range(n):
        rec = orc.tick(g["sc_pos"][b], g["sc_heading"][b], g["sc_vel"][b], H.object_list(g, b), vk)
        H.compare_record(rec, g, b, ctx="seed86420 " + tag)
        compared += int(not rec["out_of_track"])
    assert compared > n // 2
