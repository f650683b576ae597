"""The replanning flow of mpl_test_node/src/map_replanner_node.cpp:107-241 as a script over any planner object that has
the LpaMixin call shapes (oracle.OraclePlanner, oracle.ref.RefPlanner, and the CUDA path's adaptor in test_gpu_lpa.py):
plan with LPA*, link the graph to the map (visualizeGraph -> getLinkedNodes), drop an obstacle on the trajectory
(addCloudCallback: edit the map, updateBlockedNodes), replan, remove part of it again (clearCloudCallback:
updateClearedNodes), replan, move the root one step along the trajectory (subtreeCallback: getSubStateSpace(1), start =
the next waypoint), replan.  `snapshots` receives the full state (result record, node dump in hm_ order, heap array,
best_child_, linked points) after every step so that two implementations can be compared step by step."""
import numpy as np

import oracle
from helpers import fill_waypoints, load_config
from ref_replay import Digest, same


def build(cls_map, cls_planner, name, extra_params=None):
    m, dim, params, U, start, goal = load_config(name)
    mp_ = cls_map(m.origin, m.dim, m.data, m.res)
    mp_.free_unknown()
    pl = cls_planner(dim)
    pl.set_map(mp_)
    for k, v in dict(params, **(extra_params or {})).items():
        pl.set_param(k, v)
    pl.set_controls(U)
    return m, mp_, pl, dim, start, goal


def cells_on_path(m, dim, path_pts, half):
    """cells of a (2*half+1)^2 patch (x, y) around every path point — the 5 x 5 fill of addCloudCallback"""
    out, seen = [], set()
    for p in path_pts:
        pn = np.round((np.asarray(p[:dim]) - m.origin[:dim]) / m.res - 0.5).astype(int)
        for dx in range(-half, half + 1):
            for dy in range(-half, half + 1):
                c = pn.copy()
                c[0] += dx
                c[1] += dy
                if np.all(c >= 0) and np.all(c < m.dim[:dim]) and tuple(c) not in seen:
                    seen.add(tuple(c))
                    out.append(c)
    return np.array(out, dtype=np.int32)


def snapshot(pl, res, linked=None):
    return dict(res=res.copy() if res is not None else None, nodes=pl.lpa_nodes(), heap=pl.lpa_heap(), best=pl.lpa_best_child(),
                linked=None if linked is None else linked.copy())


def run(pl, mp_, m, dim, start, goal, control, path_of, n_rounds=3, block_at=(0.45, 0.7), half=2, free_of=None):
    """path_of(pl, res) -> list of trajectory waypoint positions of the last plan (implementation specific).
    Returns the list of snapshots."""
    snaps = []
    s, g = oracle.make_waypoints(1), oracle.make_waypoints(1)
    fill_waypoints(s, start, control)
    fill_waypoints(g, goal, control)
    res = pl.lpa_plan(s, g)
    snaps.append(snapshot(pl, res))
    grid = m.data.reshape(-1).copy()
    for rnd in range(n_rounds):
        if res["status"] != 0:
            break
        path = path_of(pl, res)
        linked = pl.lpa_get_linked_nodes()
        # --- addCloudCallback: new obstacle cells across the trajectory (only cells that are free, map_replanner_node.cpp:212-219)
        k = int(len(path) * block_at[rnd % len(block_at)])
        cand = cells_on_path(m, dim, path[k:k + 1], half)
        lin = cand[:, 0] + m.dim[0] * cand[:, 1] + (m.dim[0] * m.dim[1] * cand[:, 2] if dim == 3 else 0)
        new_obs = cand[(grid[lin] >= 0) & (grid[lin] < 100)]
        new_obs = np.concatenate([new_obs, new_obs[:3]])  # the node's list carries duplicates (overlapping 5 x 5 patches)
        lin = new_obs[:, 0] + m.dim[0] * new_obs[:, 1] + (m.dim[0] * m.dim[1] * new_obs[:, 2] if dim == 3 else 0)
        grid[lin] = 100
        mp_.set_cells(new_obs, 100)
        pl.lpa_update_blocked_nodes(new_obs)
        snaps.append(snapshot(pl, None, linked))
        res = pl.lpa_plan(s, g)
        snaps.append(snapshot(pl, res))
        if res["status"] != 0:
            break
        # --- clearCloudCallback: half of those cells become free again
        linked = pl.lpa_get_linked_nodes()
        cleared = new_obs[: max(1, len(new_obs) // 2)]
        lin = cleared[:, 0] + m.dim[0] * cleared[:, 1] + (m.dim[0] * m.dim[1] * cleared[:, 2] if dim == 3 else 0)
        grid[lin] = 0
        mp_.set_cells(cleared, 0)
        pl.lpa_update_cleared_nodes(cleared)
        snaps.append(snapshot(pl, None, linked))
        res = pl.lpa_plan(s, g)
        snaps.append(snapshot(pl, res))
        if res["status"] != 0:
            break
        # --- subtreeCallback: the root moves one step along the trajectory
        path = path_of(pl, res)
        if len(path) < 3:
            break
        nxt = start_of_step(pl, 1)
        pl.lpa_get_sub_state_space(1)
        snaps.append(snapshot(pl, None))
        s = nxt
        res = pl.lpa_plan(s, g)
        snaps.append(snapshot(pl, res))
    return snaps


def start_of_step(pl, k):
    """the waypoint the replanner node takes as its next start (traj.getWaypoints()[k]); implementation hook"""
    return pl.lpa_waypoint(k)


def assert_same(a, b, what=""):
    assert len(a) == len(b), (what, len(a), len(b))
    for i, (x, y) in enumerate(zip(a, b)):
        if x["res"] is not None:
            sx, sy = int(x["res"]["status"]), int(y["res"]["status"])
            if sx == -1 or sy == -1:  # the reference's plan() returns a bool: -1 = "failed", whatever the reason
                assert (sx in (-1, 2, 3, 4)) and (sy in (-1, 2, 3, 4)), (what, i, "status", sx, sy)
            else:
                assert sx == sy, (what, i, "status", sx, sy)
            if sx in (1, 5):  # start not free / start already in the goal region: nothing was searched, only the verdict counts
                assert x["res"]["cost"] == y["res"]["cost"] or sx == 1, (what, i, "cost")
                continue
            for f in ("n_seg", "cost", "n_nodes", "n_open", "n_closed", "n_prims", "n_valid", "pop_hash", "closed_hash"):
                assert x["res"][f] == y["res"][f], (what, i, f, x["res"][f], y["res"][f])
            if x["res"]["status"] == 0:
                assert x["res"]["pops"] == y["res"]["pops"], (what, i, "pops")
        assert len(x["nodes"]) == len(y["nodes"]), (what, i, "hm size", len(x["nodes"]), len(y["nodes"]))
        if isinstance(y["nodes"], Digest):  # the reference's recorded dumps (tests/ref_replay.py): all fields at once
            assert same(x["nodes"], y["nodes"]), (what, i, "nodes")
            assert same(x["heap"], y["heap"]), (what, i, "heap")  # its records are (fval, key_hash)
        else:
            for f in x["nodes"].dtype.names:
                assert np.array_equal(x["nodes"][f], y["nodes"][f]), (what, i, "node field", f,
                                                                       int(np.argmax(np.any(np.atleast_2d(x["nodes"][f] != y["nodes"][f]).reshape(len(x["nodes"]), -1), axis=1))))
            assert np.array_equal(x["heap"]["key_hash"], y["heap"]["key_hash"]) and np.array_equal(x["heap"]["fval"], y["heap"]["fval"]), (what, i, "heap")
        assert np.array_equal(x["best"], y["best"]), (what, i, "best_child")
        if x["linked"] is not None:
            assert same(x["linked"], y["linked"]), (what, i, "linked points")


VEL, ACC, JRK = 1, 3, 7
# name -> (fixture config, control, extra planner parameters, rounds)
FLOWS = {
    "corridor_acc": ("corridor", ACC, {}, 3),
    "skir_acc": ("skir", ACC, {}, 3),
    "simple_acc": ("simple", ACC, {}, 2),
    "corridor_eps2": ("corridor", ACC, {"epsilon": 2.0}, 3),
    "skir_jrk": ("skir", JRK, {"max_num": 30000}, 1),      # 76 657 nodes: outgrows the initial 65 536-node arrays on the GPU
    "corridor_jrk": ("corridor", JRK, {"max_num": 30000}, 2),
    "skir_maxnum": ("skir", ACC, {"max_num": 120}, 2),  # the first plans stop at MaxExpandStep and continue from the kept state
}


def path_of_best_child(pl, res):
    return pl.lpa_best_child_states()[:, :3]


def run_flow(name, cls_map, cls_planner, extra=None):
    cfg, control, params, rounds = FLOWS[name]
    m, mp_, pl, dim, start, goal = build(cls_map, cls_planner, cfg, dict(params, **(extra or {})))
    pl._lpa_control = control
    if name == "skir_maxnum":  # keep planning until the search gets through, like a node that re-triggers the replan
        return run_until_ok(pl, mp_, m, dim, start, goal, control)
    return run(pl, mp_, m, dim, start, goal, control, path_of_best_child, n_rounds=rounds), pl


def run_until_ok(pl, mp_, m, dim, start, goal, control):
    snaps = []
    s, g = oracle.make_waypoints(1), oracle.make_waypoints(1)
    fill_waypoints(s, start, control)
    fill_waypoints(g, goal, control)
    for _ in range(6):
        res = pl.lpa_plan(s, g)
        snaps.append(snapshot(pl, res))
        if res["status"] == 0:
            break
    linked = pl.lpa_get_linked_nodes()
    snaps.append(snapshot(pl, None, linked))
    return snaps, pl


def digest(snaps):
    """a compact, implementation-independent record of a flow for the committed fixture"""
    import hashlib
    rows = []
    for x in snaps:
        hsh = hashlib.blake2b(digest_size=8)
        for f in ("key", "g", "rhs", "h", "opened", "closed", "n_succ", "n_pred", "succ_hash", "pred_hash"):
            hsh.update(np.ascontiguousarray(x["nodes"][f]).tobytes())
        hsh.update(np.ascontiguousarray(x["heap"]["fval"]).tobytes())
        hsh.update(np.ascontiguousarray(x["heap"]["key_hash"]).tobytes())
        hsh.update(np.ascontiguousarray(x["best"]).tobytes())
        if x["linked"] is not None:
            hsh.update(np.ascontiguousarray(x["linked"]).tobytes())
        r = x["res"]
        ok = r is not None and int(r["status"]) == 0
        rows.append((int.from_bytes(hsh.digest(), "little"), len(x["nodes"]), len(x["heap"]), len(x["best"]),
                     -9 if r is None else (0 if ok else (5 if int(r["status"]) == 5 else 1 if int(r["status"]) == 1 else -1)),
                     float(r["cost"]) if ok else 0.0, int(r["pops"]) if ok else 0))
    return np.array(rows, dtype=[("digest", "u8"), ("n_nodes", "i8"), ("n_heap", "i8"), ("n_best", "i8"), ("status", "i8"), ("cost", "f8"), ("pops", "i8")])
