"""GPU results against the REFERENCE'S OWN planner sources directly (oracle/_ref/libmplref.so, see oracle/ref_harness.cpp),
without the oracle in between.  The reference side replays tests/golden/reference_calls/test_gpu_vs_reference.npz (see
tests/ref_replay.py)."""
import numpy as np
import pytest

import oracle
import ref_replay as ref
from ref_replay import recorded_reference  # noqa: F401 (autouse fixture)
import mpl_ros_b200 as mp
from mpl_ros_b200 import maps
from helpers import load_config

pytestmark = pytest.mark.gpu

FIELDS = ("n_seg", "cost", "pops", "n_nodes", "n_open", "n_closed", "n_prims", "n_valid", "pop_hash", "closed_hash")


def _planners(m, dim, params, U):
    mu = mp.MapUtil(dim)
    mu.setMap(m.origin, m.dim, m.data, m.res)
    mu.freeUnknown()
    pl = mp.MapPlanner(dim, False)
    pl.setMapUtil(mu)
    rm = ref.RefMap(m.origin, m.dim, m.data, m.res)
    rm.free_unknown()
    rp = ref.RefPlanner(dim)
    rp.set_map(rm)
    setters = dict(v_max="setVmax", a_max="setAmax", j_max="setJmax", dt="setDt", w="setW", epsilon="setEpsilon",
                   max_num="setMaxNum")
    for k, v in params.items():
        rp.set_param(k, v)
        if k in setters:
            getattr(pl, setters[k])(v)
    pl.setTol(params.get("tol_pos", 0.5), params.get("tol_vel", -1), params.get("tol_acc", -1))
    pl.setU(U)
    rp.set_controls(U)
    pl._keep, rp._keep = mu, rm
    return pl, rp


def _wps(pos, control):
    a, b = mp.waypoints_array(len(np.atleast_2d(pos))), oracle.make_waypoints(len(np.atleast_2d(pos)))
    for w in (a, b):
        p = np.atleast_2d(np.asarray(pos, dtype=np.float64))
        w["pos"][:, :p.shape[1]] = p
        w["control"] = control
    return a, b


def _same(rg, rr, ctx):
    sg, sr = int(rg["status"]), int(rr["status"])
    assert sg == sr or (sr == -1 and sg in (2, 3, 4)), (ctx, sg, sr)
    for f in FIELDS:
        if f == "n_seg" and sg != 0:
            continue
        a, b = rg[f], rr[f]
        assert a == b or (f == "cost" and np.isinf(a) and np.isinf(b)), (ctx, f, a, b)


@pytest.mark.parametrize("name", ["corridor", "simple", "skir"])
def test_single_plans(name):
    m, dim, params, U, start, goal = load_config(name)
    pl, rp = _planners(m, dim, params, U)
    sg, sr = _wps(start, mp.ACC)
    gg, gr = _wps(goal, mp.ACC)
    pl.plan(sg, gg)
    rr = rp.plan(sr, gr)
    rg = pl.result()
    _same(rg, rr, name)
    if name == "corridor":
        assert rr["n_closed"] == 615 and rr["cost"] == 351.5  # MPL/README.md:200-202 out of the reference's own code
    gn = pl.getNodes()
    assert ref.same(gn["key"][pl.getPopLog()], rp.pop_keys(rr["pops"]))
    # trajectory: coefficient rows of every primitive (what toTrajectoryROSMsg would publish)
    coeffs = rp.traj_coeffs(rr["n_seg"])
    prs = pl.getTraj().getPrimitives()
    assert len(prs) == rr["n_seg"]
    for i, pr in enumerate(prs):
        assert np.array_equal(pr.coeffs, coeffs[i, :dim]), i


def test_bench_workload_sample():
    """96 queries of bench.py's workload (levine-256, |U| = 27): the GPU batch against the reference's sources."""
    m = maps.levine256()
    U = maps.make_U(1.0, 1, 3)
    pl, rp = _planners(m, 3, dict(v_max=2.0, a_max=1.0, dt=1.0, tol_pos=0.5), U)
    S, G = maps.sample_queries(m, 96, seed=0)
    sg, sr = _wps(S, mp.ACC)
    gg, gr = _wps(G, mp.ACC)
    rg, _, _ = pl.plan_batch(sg, gg, max_seg=64)
    rr = rp.plan_batch(sr, gr, nthreads=16)
    for i in range(96):
        _same(rg[i], rr[i], i)


def test_cost_shaping_flow():
    """test_distance_map_planner_2d.cpp flow: GPU vs the reference's setSearchRegion / updatePotentialMap / plan."""
    m, dim, params, U, start, goal = load_config("corridor")
    pl, rp = _planners(m, dim, dict(params, potential_weight=0.5, gradient_weight=0.3), U)
    pl.setPotentialWeight(0.5)
    pl.setGradientWeight(0.3)
    sg, sr = _wps(start, mp.ACC)
    gg, gr = _wps(goal, mp.ACC)
    assert pl.plan(sg, gg)
    path = np.zeros((pl.result()["n_seg"] + 1, 3))
    path[:, :2] = np.array([w.pos for w in pl.getTraj().getWaypoints()])
    pl.setSearchRadius([0.5, 0.5])
    rp.set_vec("search_radius", [0.5, 0.5, 0.0])
    pl.setSearchRegion(list(path[:, :2]))
    rp.set_search_region(path, dense=False)
    ncell = int(np.prod(m.dim))
    assert np.array_equal(pl.getSearchRegionMask(), rp.get_search_region(ncell))
    pl.setPotentialRadius([1.0, 1.0])
    rp.set_vec("potential_radius", [1.0, 1.0, 0.0])
    pl.updatePotentialMap(start)
    rp.update_potential_map(np.array([start[0], start[1], 0.0]))
    assert ref.same(pl._keep.getMap(), rp._keep.get_data())
    pl.plan(sg, gg)
    rr = rp.plan(sr, gr)
    _same(pl.result(), rr, "shaped")
    gn = pl.getNodes()
    assert ref.same(gn["key"][pl.getPopLog()], rp.pop_keys(rr["pops"]))
