"""The oracle against the REFERENCE'S OWN planner sources (oracle/_ref/libmplref.so: graph_search.h, state_space.h,
env_base.h, env_map.h, primitive.h, waypoint.h, map_util.h and map_planner.cpp compiled from /root/reference against
the stand-in Eigen/Boost headers of oracle/shim/, driven by oracle/ref_harness.cpp).

This widens the oracle's pin from the single published known answer (MPL/README.md:200-202) to every configuration
the GPU parity tests use: 3D, |U| = 27, JRK, yaw controls, search region / potential map, iterativePlan.  Everything is
compared exactly: counters, the order-dependent hash of the popped lattice keys and the pop sequence itself, every
node of the hash map (stored state, g, h, flags), and the trajectory's coefficient rows.

The reference side replays tests/golden/reference_calls/test_oracle_vs_reference.npz (see tests/ref_replay.py).
"""
import math

import numpy as np
import pytest

import oracle
import ref_replay as ref
from ref_replay import recorded_reference  # noqa: F401 (autouse fixture)
from mpl_ros_b200 import maps
from helpers import load_config

EXACT_FIELDS = ("n_seg", "cost", "pops", "n_nodes", "n_open", "n_closed", "n_prims", "n_valid", "pop_hash", "closed_hash")


def _pair(m, dim, params, U):
    om = oracle.OracleMap(m.origin, m.dim, m.data, m.res)
    om.free_unknown()
    rm = ref.RefMap(m.origin, m.dim, m.data, m.res)
    rm.free_unknown()
    op, rp = oracle.OraclePlanner(dim), ref.RefPlanner(dim)
    op.set_map(om)
    rp.set_map(rm)
    for k, v in params.items():
        op.set_param(k, v)
        rp.set_param(k, v)
    op.set_controls(U)
    rp.set_controls(U)
    op._keep, rp._keep = om, rm
    return op, rp


def _wp(pos, control, yaw=0.0, vel=None):
    w = oracle.make_waypoints(1)
    w["pos"][0, :len(pos)] = pos
    if vel is not None:
        w["vel"][0, :len(vel)] = vel
    w["yaw"] = yaw
    w["control"] = control
    return w


def _same_status(so, sr):
    return (so == sr) or (sr == -1 and so in (2, 3, 4))  # the reference's bool does not say why a search failed


def _coeff_rows(dim, control, actions, seg_states, U, yaw_col):
    order = {1: 1, 3: 2, 7: 3, 15: 4}[control & 15]
    out = np.zeros((len(actions), 4, 6))
    for i, (a, st) in enumerate(zip(actions, seg_states)):
        for ax in range(dim):
            for d in range(order):
                out[i, ax, 5 - d] = st[d * 3 + ax]
            out[i, ax, 5 - order] = U[a][ax]
        if control & 16:
            out[i, 3, 4], out[i, 3, 5] = U[a][yaw_col], st[12]
    return out


def _compare(op, rp, s, g, dim, control, U, ctx, nodes=True):
    ro, rr = op.plan(s, g), rp.plan(s, g)
    assert _same_status(int(ro["status"]), int(rr["status"])), (ctx, ro["status"], rr["status"])
    for f in EXACT_FIELDS:
        a, b = ro[f], rr[f]
        if f == "n_seg" and ro["status"] != 0:
            continue
        assert a == b or (f == "cost" and np.isinf(a) and np.isinf(b)), (ctx, f, a, b)
    assert ref.same(op.pop_keys(ro["pops"]), rp.pop_keys(rr["pops"])), ctx
    if nodes:  # the same set of keys, and per key the same stored state, g, h and flags
        assert ref.same(op.nodes(ro["n_nodes"]), rp.nodes(rr["n_nodes"])), ctx
    if ro["status"] == 0:
        exp = _coeff_rows(dim, control, op.actions(ro["n_seg"]), op.seg_states(ro["n_seg"]), U, dim)
        assert np.array_equal(exp, rp.traj_coeffs(rr["n_seg"])), ctx
    return ro, rr


def test_published_known_answer_both():
    m, dim, params, U, start, goal = load_config("corridor")
    op, rp = _pair(m, dim, params, U)
    ro, rr = _compare(op, rp, _wp(start, 3), _wp(goal, 3), dim, 3, U, "corridor")
    assert rr["n_closed"] == 615 and rr["n_seg"] == 35 and rr["cost"] == 351.5  # MPL/README.md:200-202, from the reference's code


@pytest.mark.parametrize("name", ["simple", "skir"])
def test_3d_reference_configs(name):
    m, dim, params, U, start, goal = load_config(name)
    op, rp = _pair(m, dim, params, U)
    _compare(op, rp, _wp(start, 3), _wp(goal, 3), dim, 3, U, name)
    _compare(op, rp, _wp(goal, 3), _wp(start, 3), dim, 3, U, name + " reversed")


def test_levine_batch_sample():
    """BASELINE configs[1] shape: 3D, |U| = 27, random free-voxel pairs (unreachable ones included)."""
    m = maps.load_fixture("levine")
    U = maps.make_U(1.0, 1, 3)
    op, rp = _pair(m, 3, dict(v_max=2.0, a_max=1.0, dt=1.0, tol_pos=0.5), U)
    S, G = maps.sample_queries(m, 24, seed=0)
    kinds = set()
    for i in range(24):
        ro, _ = _compare(op, rp, _wp(S[i], 3), _wp(G[i], 3), 3, 3, U, ("levine", i), nodes=(i % 6 == 0))
        kinds.add(int(ro["status"]))
    assert 0 in kinds and 3 in kinds


def test_levine256_bench_sample_identity():
    """The bench workload (BASELINE configs[1] on the 256^3 map): 96 of the rank-0 queries, threads on both sides."""
    m = maps.levine256()
    U = maps.make_U(1.0, 1, 3)
    op, rp = _pair(m, 3, dict(v_max=2.0, a_max=1.0, dt=1.0, tol_pos=0.5), U)
    S, G = maps.sample_queries(m, 96, seed=0)
    s, g = oracle.make_waypoints(96), oracle.make_waypoints(96)
    s["pos"], g["pos"], s["control"], g["control"] = S, G, 3, 3
    ro, _ = op.plan_batch(s, g, nthreads=8)
    rr = rp.plan_batch(s, g, nthreads=8)
    for f in EXACT_FIELDS:
        assert np.array_equal(ro[f], rr[f]), f
    assert all(_same_status(int(a), int(b)) for a, b in zip(ro["status"], rr["status"]))
    # includes the search in which the textbook hash_combine merges six pairs of distinct states (see oracle/shim/boost)
    assert ro["n_nodes"].max() > 6000


def test_jrk_epsilon_startvel_maxnum():
    m, dim, params, U, start, goal = load_config("corridor")
    op, rp = _pair(m, dim, dict(v_max=1.0, a_max=1.0, j_max=2.0, dt=1.0, tol_pos=0.5, max_num=3000), U)
    _compare(op, rp, _wp(start, 7), _wp(goal, 7), dim, 7, U, "JRK 2D")
    op, rp = _pair(m, dim, dict(params, epsilon=2.0), U)
    ro, rr = op.plan(_wp(start, 3, vel=[0.5, 0.0]), _wp(goal, 3)), rp.plan(_wp(start, 3, vel=[0.5, 0.0]), _wp(goal, 3))
    # with epsilon > 1 the oracle pins status, cost and the expansion sequence (see DESIGN section 2)
    assert ro["status"] == rr["status"] == 0 and ro["cost"] == rr["cost"] and ro["pop_hash"] == rr["pop_hash"]
    op, rp = _pair(m, dim, dict(params, max_num=50), U)
    ro, rr = op.plan(_wp(start, 3), _wp(goal, 3)), rp.plan(_wp(start, 3), _wp(goal, 3))
    assert ro["status"] == 2 and rr["status"] == -1 and ro["pops"] == rr["pops"] == 50 and ro["pop_hash"] == rr["pop_hash"]
    # start inside an obstacle, start inside the goal region
    occ = np.argwhere(m.data.reshape(m.dim[1], m.dim[0]) == 100)[0]
    bad = np.array([(occ[1] + 0.5) * m.res + m.origin[0], (occ[0] + 0.5) * m.res + m.origin[1]])
    assert op.plan(_wp(bad, 3), _wp(goal, 3))["status"] == rp.plan(_wp(bad, 3), _wp(goal, 3))["status"] == 1
    assert op.plan(_wp(goal, 3), _wp(goal, 3))["status"] == rp.plan(_wp(goal, 3), _wp(goal, 3))["status"] == 5


def test_snp_2d_and_jrk_125_controls_3d():
    """Snap control (order 4) on the corridor, and BASELINE configs[4]'s shape at test size (3D jerk control, |U| = 125)."""
    m, dim, params, U, start, goal = load_config("corridor")
    op, rp = _pair(m, dim, dict(v_max=1.0, a_max=1.0, j_max=1.0, dt=1.0, tol_pos=0.5, max_num=1500), U)
    _compare(op, rp, _wp(start, 15), _wp(goal, 15), dim, 15, U, "SNP 2D")
    Uh = maps.make_U(1.0, 1, 2) * 0.5
    op, rp = _pair(m, dim, dict(v_max=1.5, a_max=1.0, j_max=2.0, dt=0.5, tol_pos=0.5, max_num=800), Uh)
    _compare(op, rp, _wp(start, 15, vel=[0.5, 0.0]), _wp(goal, 15), dim, 15, Uh, "SNP 2D dt 0.5")
    m = maps.load_fixture("skir")
    U5 = maps.make_U(2.0, 2, 3)
    assert U5.shape[0] == 125
    op, rp = _pair(m, 3, dict(v_max=3.0, a_max=2.0, dt=0.5, max_num=400, tol_pos=0.5), U5)
    _compare(op, rp, _wp([5.5, 5.5, 0.5], 7), _wp([1.5, 1.5, 5.5], 7), 3, 7, U5, "JRK 125", nodes=False)


def test_goal_tolerances_and_weights():
    """Goal region with velocity / acceleration tolerances (env_map.h:25-45), other w / epsilon / dt values."""
    m, dim, params, U, start, goal = load_config("corridor")
    for prm, ctl in ((dict(params, tol_vel=0.3), 3), (dict(params, tol_vel=0.0, max_num=4000), 3),
                     (dict(v_max=1.0, a_max=1.0, j_max=2.0, dt=1.0, tol_pos=0.5, tol_vel=0.5, tol_acc=0.5, max_num=2500), 7),
                     (dict(params, w=3.0), 3), (dict(params, w=25.0, epsilon=0.5), 3), (dict(params, dt=0.5, max_num=5000), 3),
                     (dict(params, epsilon=0.0, max_num=3000), 3)):
        op, rp = _pair(m, dim, prm, U)
        ro, rr = op.plan(_wp(start, ctl), _wp(goal, ctl)), rp.plan(_wp(start, ctl), _wp(goal, ctl))
        assert _same_status(int(ro["status"]), int(rr["status"])), prm
        for f in ("cost", "pops", "n_nodes", "n_open", "n_closed", "n_prims", "n_valid", "pop_hash", "closed_hash"):
            assert ro[f] == rr[f] or (f == "cost" and np.isinf(ro[f]) and np.isinf(rr[f])), (prm, f, ro[f], rr[f])


@pytest.mark.parametrize("yaw_max,wyaw", [(0.7, 1.0), (-1.0, 1.0), (1.2, 2.5)])
def test_yaw_controls_libm_definition(yaw_max, wyaw):
    """MPL/test/test_planner_2d_with_yaw.cpp; the oracle in trig_mode 0 calls the same libm as the reference code does."""
    m, dim, params, _, start, goal = load_config("corridor")
    U = np.array([[dx, dy, dyaw] for dx in (-0.5, 0, 0.5) for dy in (-0.5, 0, 0.5) for dyaw in (-0.5, 0, 0.5)])
    op, rp = _pair(m, dim, dict(params, yaw_max=yaw_max, wyaw=wyaw), U)
    op.set_param("trig_mode", 0)
    _compare(op, rp, _wp(start, 19, yaw=math.pi / 2), _wp(goal, 19), dim, 19, U, ("yaw", yaw_max, wyaw))
    Uv = np.array([[dx, dy, dyaw] for dx in (-1.0, 0, 1.0) for dy in (-1.0, 0, 1.0) for dyaw in (-0.4, 0, 0.4)])
    op, rp = _pair(m, dim, dict(dt=1.0, tol_pos=0.5, yaw_max=0.9, w=10.0, v_max=1.0), Uv)
    _compare(op, rp, _wp(start, 17, yaw=0.3), _wp(goal, 17), dim, 17, Uv, "VELxYAW")


@pytest.mark.parametrize("grad_w", [0.0, 0.3])
def test_distance_map_flow(grad_w):
    """MPL/test/test_distance_map_planner_2d.cpp:46-93 on both sides, then iterativePlan (map_planner.cpp:394-434)."""
    m, dim, params, U, start, goal = load_config("corridor")
    ncell = int(np.prod(m.dim))
    op, rp = _pair(m, dim, params, U)
    s, g = _wp(start, 3), _wp(goal, 3)
    ro, rr = _compare(op, rp, s, g, dim, 3, U, "plain")
    st, acts = op.seg_states(ro["n_seg"]), op.actions(ro["n_seg"])
    path = np.zeros((ro["n_seg"] + 1, 3))
    path[:-1, :2] = st[:, :2]
    last = st[-1]
    path[-1, :2] = last[:2] + last[3:5] * params["dt"] + 0.5 * U[acts[-1]] * params["dt"] ** 2  # exact here: dyadic values
    op2, rp2 = _pair(m, dim, dict(params, epsilon=1.0, potential_weight=0.5, gradient_weight=grad_w), U)
    op2.set_map(op._keep)
    rp2.set_map(rp._keep)
    for p in (op2, rp2):
        p.set_vec("search_radius", [0.5, 0.5, 0.0])
        p.set_search_region(path, dense=False)
        p.set_vec("potential_radius", [1.0, 1.0, 0.0])
        p.update_potential_map(np.array([start[0], start[1], 0.0]))
    assert np.array_equal(op2.get_search_region(ncell), rp2.get_search_region(ncell))
    assert ref.same(op._keep.get_data(ncell), rp._keep.get_data())  # the rewritten map (map_planner.cpp:387)
    ro2, rr2 = _compare(op2, rp2, s, g, dim, 3, U, "shaped")
    if grad_w == 0.0:
        assert rr2["n_seg"] == 36 and rr2["pops"] == 2732 and abs(rr2["cost"] - 647.1) < 1e-9  # now from the reference's code too
    # the first planners see the rewritten map
    _compare(op, rp, s, g, dim, 3, U, "plain on the rewritten map")
    # iterativePlan: the reference's loop against the same loop spelled out on the oracle
    rit = rp2.iterative_plan(s, g, rp2, 3)
    prev, traj_states, traj_acts = 0.0, op2.seg_states(ro2["n_seg"]), op2.actions(ro2["n_seg"])
    for _ in range(3):
        n = len(traj_acts)
        pth = np.zeros((n + 1, 3))
        pth[:-1, :2] = traj_states[:, :2]
        lt = traj_states[-1]
        pth[-1, :2] = lt[:2] + lt[3:5] * params["dt"] + 0.5 * U[traj_acts[-1]] * params["dt"] ** 2
        op2.set_search_region(pth, dense=False)
        roi = op2.plan(s, g)
        assert roi["status"] == 0
        traj_states, traj_acts = op2.seg_states(roi["n_seg"]), op2.actions(roi["n_seg"])
        if prev == roi["cost"]:
            break
        prev = roi["cost"]
    assert rit["status"] == 0 and rit["cost"] == roi["cost"] and rit["n_seg"] == roi["n_seg"] and rit["pop_hash"] == roi["pop_hash"]


def test_prior_trajectory_heuristic():
    """MPL/test/test_planner_2d_with_prior_traj.cpp:29-105: a VEL-control plan becomes the prior trajectory of a second
    planner whose heuristic then follows it (env_base.h:46-53,249-256).  Oracle-only groundwork: the CUDA path does not
    implement prior trajectories yet (DESIGN section 7)."""
    m, dim, params, _, start, goal = load_config("corridor")
    U1 = maps.make_U(1.0, 1, 2)
    op1, rp1 = _pair(m, dim, dict(v_max=1.0, a_max=1.0, dt=1.0), U1)
    ro1, rr1 = _compare(op1, rp1, _wp(start, 1), _wp(goal, 1), dim, 1, U1, "VEL prior")
    assert ro1["status"] == 0
    U2 = maps.make_U(1.0, 1, 2) * 0.5
    for ctl, prm in ((7, dict(epsilon=1.0, v_max=1.0, a_max=1.0, dt=1.0, w=10.0, tol_pos=0.5, max_num=20000)),
                     (3, dict(epsilon=1.0, v_max=1.0, a_max=1.0, dt=1.0, w=10.0, tol_pos=0.5))):
        op2, rp2 = _pair(m, dim, prm, U2)
        op2.set_prior_trajectory(op1)
        rp2.set_prior_trajectory(rp1)
        ro2, rr2 = op2.plan(_wp(start, ctl), _wp(goal, ctl)), rp2.plan(_wp(start, ctl), _wp(goal, ctl))
        assert _same_status(int(ro2["status"]), int(rr2["status"])), ctl
        for f in ("cost", "pops", "n_nodes", "n_open", "n_closed", "n_prims", "n_valid", "pop_hash", "closed_hash"):
            assert ro2[f] == rr2[f] or (f == "cost" and np.isinf(ro2[f]) and np.isinf(rr2[f])), (ctl, f, ro2[f], rr2[f])
        assert ref.same(op2.pop_keys(ro2["pops"]), rp2.pop_keys(rr2["pops"]))
        # the prior changes the search: a plain planner with the same parameters expands a different set
        op3, _ = _pair(m, dim, prm, U2)
        assert op3.plan(_wp(start, ctl), _wp(goal, ctl))["pop_hash"] != ro2["pop_hash"]


def test_potential_map_3d_local_range():
    m, dim, params, U, start, goal = load_config("skir")
    op, rp = _pair(m, dim, dict(params, potential_weight=0.2, gradient_weight=0.1), U)
    for p in (op, rp):
        p.set_vec("potential_radius", [0.4, 0.4, 0.2])
        p.set_vec("potential_map_range", [3.0, 2.5, 1.0])
        p.update_potential_map(np.asarray(start, dtype=np.float64))
    assert ref.same(op._keep.get_data(int(np.prod(m.dim))), rp._keep.get_data())
    _compare(op, rp, _wp(start, 3), _wp(goal, 3), dim, 3, U, "potential 3d")


def test_map_ops_against_reference_sources():
    """MapUtil::freeUnknown / dilate (map_util.h:221-276) of the reference's code against the numpy formulation that
    tests/test_gpu_parity.py::test_map_ops holds the GPU map kernels to."""
    m = maps.load_fixture("simple")
    data = m.data.copy()
    data[::7] = -1
    rm = ref.RefMap(m.origin, m.dim, data, m.res)
    assert ref.same(rm.get_data(), data)
    rm.free_unknown()
    want = np.where(data == -1, 0, data)
    assert ref.same(rm.get_data(), want)
    ns = np.array([[1, 0, 0], [-1, 0, 0], [0, 1, 0], [0, -1, 0]], dtype=np.int32)
    rm.dilate(ns)
    g = want.reshape(tuple(int(x) for x in m.dim[::-1]))
    out = g.copy()
    occ = g == 100
    out[:, :, 1:][occ[:, :, :-1]] = 100
    out[:, :, :-1][occ[:, :, 1:]] = 100
    out[:, 1:, :][occ[:, :-1, :]] = 100
    out[:, :-1, :][occ[:, 1:, :]] = 100
    assert ref.same(rm.get_data(), out.reshape(-1))
