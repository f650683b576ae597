"""Seeded random comparison of the oracle with the REFERENCE'S OWN planner sources (oracle/_ref, see
oracle/ref_harness.cpp): random 2D / 3D box maps, controls (VEL / ACC / JRK / SNP and the yaw variants), control sets,
bounds, dt, w, epsilon, tolerances, max_num, start velocities, unknown cells, potential maps with local ranges and
search regions along random paths.  Every counter and both key hashes must agree exactly.  (An offline run of the same
generators over 500 cases found no mismatch; the test keeps 64.)  The reference side replays
tests/golden/reference_calls/test_oracle_fuzz_vs_reference.npz (see tests/ref_replay.py)."""
import numpy as np
import pytest

import oracle
import ref_replay as ref
from ref_replay import recorded_reference  # noqa: F401 (autouse fixture)
from mpl_ros_b200 import maps

FIELDS=("cost","pops","n_nodes","n_open","n_closed","n_prims","n_valid","pop_hash","closed_hash")
def rand_case(rng, dim):
    nd = rng.integers(24, 56, size=dim)
    res = float(np.float32(rng.choice([0.1, 0.2, 0.25, 0.05])))
    origin = rng.uniform(-2, 2, size=dim).round(2)
    grid = np.zeros(tuple(nd[::-1]), dtype=np.int8)
    for _ in range(rng.integers(3, 12)):
        lo = [rng.integers(0, n) for n in nd]; sz=[rng.integers(1, max(2,n//4)) for n in nd]
        sl = tuple(slice(lo[k], lo[k]+sz[k]) for k in range(dim))[::-1]
        grid[sl] = 100
    if rng.random() < 0.3: grid[rng.random(grid.shape) < 0.02] = -1
    ctl = int(rng.choice([1,3,3,7,15]))
    u = float(rng.choice([0.5, 1.0])); nper = int(rng.choice([1,1,2]))
    U = maps.make_U(u*nper, nper, dim)
    if U.shape[0] > 60: U = U[rng.choice(U.shape[0], 40, replace=False)]
    prm = dict(v_max=float(rng.choice([1.0, 1.5, 2.0])), a_max=float(rng.choice([1.0, 2.0])), j_max=float(rng.choice([1.0, 3.0])),
               dt=float(rng.choice([0.5, 1.0])), w=float(rng.choice([1.0, 10.0, 3.5])), epsilon=float(rng.choice([1.0, 1.0, 2.0, 0.0])),
               tol_pos=float(rng.choice([0.5, 0.3, 1.0])), max_num=int(rng.choice([300, 800, 2000])))
    if rng.random() < 0.3: prm["tol_vel"] = float(rng.choice([0.0, 0.5, 1.0]))
    free = np.argwhere(grid == 0)
    a, b = free[rng.integers(len(free))][::-1], free[rng.integers(len(free))][::-1]
    start = (a + 0.5) * res + origin; goal = (b + 0.5) * res + origin
    vel = rng.choice([0.0, 0.5, -0.5], size=dim) if (ctl != 1 and rng.random() < 0.4) else np.zeros(dim)
    return nd, origin, res, grid.reshape(-1), ctl, U, prm, start, goal, vel
def run_plain(seed, dim):
    rng = np.random.default_rng(seed)
    nd, origin, res, data, ctl, U, prm, start, goal, vel = rand_case(rng, dim)
    if "tol_vel" in prm and ctl == 1: prm.pop("tol_vel")
    om = oracle.OracleMap(origin, nd, data, res); om.free_unknown()
    rm = ref.RefMap(origin, nd, data, res); rm.free_unknown()
    op, rp = oracle.OraclePlanner(dim), ref.RefPlanner(dim)
    op.set_map(om); rp.set_map(rm)
    for k,v in prm.items(): op.set_param(k,v); rp.set_param(k,v)
    op.set_controls(U); rp.set_controls(U)
    s, g = oracle.make_waypoints(1), oracle.make_waypoints(1)
    s["pos"][0,:dim]=start; g["pos"][0,:dim]=goal; s["vel"][0,:dim]=vel; s["control"]=g["control"]=ctl
    ro, rr = op.plan(s,g), rp.plan(s,g)
    ok = (ro["status"]==rr["status"]) or (rr["status"]==-1 and ro["status"] in (2,3,4))
    bad=[f for f in FIELDS if not (ro[f]==rr[f] or (f=="cost" and np.isinf(ro[f]) and np.isinf(rr[f])))]
    if ro["status"]==0 and ro["n_seg"]!=rr["n_seg"]: bad.append("n_seg")
    return ok and not bad, (seed, dim, ctl, prm, int(ro["status"]), int(rr["status"]), bad, int(ro["pops"]))


def run_shaped(seed, dim):
    rng = np.random.default_rng(1000+seed)
    nd = rng.integers(24, 48, size=dim)
    res = float(np.float32(rng.choice([0.1, 0.2, 0.25])))
    origin = rng.uniform(-2, 2, size=dim).round(2)
    grid = np.zeros(tuple(nd[::-1]), dtype=np.int8)
    for _ in range(rng.integers(3, 10)):
        lo = [rng.integers(0, n) for n in nd]; sz=[rng.integers(1, max(2,n//5)) for n in nd]
        grid[tuple(slice(lo[k], lo[k]+sz[k]) for k in range(dim))[::-1]] = 100
    data = grid.reshape(-1)
    yaw = rng.random() < 0.5
    base = int(rng.choice([1,3,7]))
    ctl = base | (16 if yaw else 0)
    if yaw:
        U = np.array([[dx,dy]+([0.0] if dim==3 else [])+[dyaw] for dx in (-1.0,0,1.0) for dy in (-1.0,0,1.0) for dyaw in (-0.5,0,0.5)])
    else:
        U = maps.make_U(1.0, 1, dim)
    prm = dict(v_max=float(rng.choice([1.0, 2.0])), a_max=float(rng.choice([1.0, 2.0])), dt=float(rng.choice([0.5, 1.0])),
               w=float(rng.choice([10.0, 3.5])), tol_pos=0.5, max_num=int(rng.choice([300, 1000])))
    if yaw:
        prm["yaw_max"] = float(rng.choice([-1.0, 0.7, 1.3])); prm["wyaw"] = float(rng.choice([0.0, 1.0, 2.5]))
    shaping = rng.random() < 0.7
    if shaping:
        prm["potential_weight"] = float(rng.choice([0.1, 0.5])); prm["gradient_weight"] = float(rng.choice([0.0, 0.3]))
    free = np.argwhere(grid == 0)
    a, b = free[rng.integers(len(free))][::-1], free[rng.integers(len(free))][::-1]
    start = (a + 0.5) * res + origin; goal = (b + 0.5) * res + origin
    om = oracle.OracleMap(origin, nd, data, res); om.free_unknown()
    rm = ref.RefMap(origin, nd, data, res); rm.free_unknown()
    op, rp = oracle.OraclePlanner(dim), ref.RefPlanner(dim)
    op.set_map(om); rp.set_map(rm)
    for k,v in prm.items(): op.set_param(k,v); rp.set_param(k,v)
    op.set_param("trig_mode", 0)
    op.set_controls(U); rp.set_controls(U)
    extra=[]
    if shaping:
        pr = np.zeros(3); pr[:dim] = rng.choice([0.3, 0.6, 1.0]); 
        if dim==3: pr[2] = rng.choice([0.2, 0.5])
        rngv = np.zeros(3)
        if rng.random() < 0.5: rngv[:dim] = rng.choice([1.0, 2.0, 3.0], size=dim)
        for p in (op, rp):
            p.set_vec("potential_radius", pr); p.set_vec("potential_map_range", rngv)
            p.update_potential_map(np.r_[start, np.zeros(3-dim)])
        ncell=int(np.prod(nd))
        if not ref.same(om.get_data(ncell), rm.get_data()): extra.append("potmap")
        if rng.random() < 0.6:
            npts = rng.integers(2, 6)
            path = np.zeros((npts,3)); path[0,:dim]=start; path[-1,:dim]=goal
            for i in range(1,npts-1): path[i,:dim] = origin + rng.random(dim)*nd*res
            sr = np.zeros(3); sr[:dim] = rng.choice([0.3, 0.8, 1.5])
            dense = bool(rng.random()<0.3)
            for p in (op, rp):
                p.set_vec("search_radius", sr); p.set_search_region(path, dense=dense)
            if not np.array_equal(op.get_search_region(ncell), rp.get_search_region(ncell)): extra.append("region")
    s, g = oracle.make_waypoints(1), oracle.make_waypoints(1)
    s["pos"][0,:dim]=start; g["pos"][0,:dim]=goal; s["control"]=g["control"]=ctl
    if yaw: s["yaw"] = float(rng.uniform(-3,3))
    ro, rr = op.plan(s,g), rp.plan(s,g)
    ok = (ro["status"]==rr["status"]) or (rr["status"]==-1 and ro["status"] in (2,3,4))
    bad=extra+[f for f in FIELDS if not (ro[f]==rr[f] or (f=="cost" and np.isinf(ro[f]) and np.isinf(rr[f])))]
    return ok and not bad, (seed, dim, ctl, prm, shaping, int(ro["status"]), int(rr["status"]), bad, int(ro["pops"]))


@pytest.mark.parametrize("dim", [2, 3])
def test_fuzz_plain(dim):
    bad = [info for ok, info in (run_plain(seed, dim) for seed in range(16)) if not ok]
    assert not bad, bad


@pytest.mark.parametrize("dim", [2, 3])
def test_fuzz_yaw_and_cost_shaping(dim):
    bad = [info for ok, info in (run_shaped(seed, dim) for seed in range(16)) if not ok]
    assert not bad, bad
