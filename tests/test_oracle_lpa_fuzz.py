"""Seeded random LPA* replanning sequences: random 2D / 3D box maps, controls (VEL / ACC / JRK / SNP), control sets, bounds,
epsilon, max_num; then rounds of { drop a random patch of obstacle cells near the trajectory | clear some of the cells dropped
earlier | re-root at the k-th node of the trajectory | plan again }.  After EVERY step the oracle, the reference's own LPA*
sources (oracle/_ref, replayed from tests/golden/reference_calls/, see tests/ref_replay.py) and the device core built for
the host (tests/cpp/lpa_emul.cpp) must agree on the whole state: result record, hm_ in iteration order (g, rhs, h, flags, list hashes), the priority-queue array, best_child_, the
linked points.  Two situations the reference leaves undefined end a sequence (the oracle detects them first so that the
reference's code is never driven into them): a plan that starts on an empty priority queue, and getSubStateSpace meeting a
stored successor that is no longer in the state space (state_space.h:160-163).  A third one was FOUND by this test (seed 21,
2D): after re-rooting, recoverTraj's best-predecessor walk can enter a cycle that does not contain the start, and the
reference's loop (graph_search.h:377-438) never returns; the oracle and the device core report a failed trace-back with an
empty best_child_ instead, and the reference's sources are not run on that step."""
import numpy as np
import pytest

import oracle
import ref_replay as ref
from ref_replay import recorded_reference  # noqa: F401 (autouse fixture)
import lpa_emul
import lpa_flow
from test_oracle_fuzz_vs_reference import rand_case


def run_sequence(seed, dim, impls, rounds=4):
    rng = np.random.default_rng(7000 + seed)
    nd, origin, res, data, ctl, U, prm, start, goal, vel = rand_case(rng, dim)
    prm = {k: v for k, v in prm.items() if k in ("v_max", "a_max", "j_max", "dt", "w", "epsilon", "tol_pos", "max_num")}
    if prm["epsilon"] == 0.0:
        prm["epsilon"] = 1.0
    prm["max_num"] = int(prm["max_num"]) * 2
    pls, maps_ = [], []
    for cm, cp, extra in impls:
        m = cm(origin, nd, data, res)
        m.free_unknown()
        p = cp(dim)
        p.set_map(m)
        for k, v in dict(prm, **extra).items():
            p.set_param(k, v)
        p.set_controls(U)
        p._lpa_control = ctl
        pls.append(p)
        maps_.append(m)
    s, g = oracle.make_waypoints(1), oracle.make_waypoints(1)
    s["pos"][0, :dim], g["pos"][0, :dim], s["vel"][0, :dim] = start, goal, vel
    s["control"] = g["control"] = ctl
    grid = np.where(data.reshape(-1) == -1, 0, data.reshape(-1)).astype(np.int8)
    dropped = []
    steps = 0

    def lin(c):
        return c[:, 0] + nd[0] * c[:, 1] + (nd[0] * nd[1] * c[:, 2] if dim == 3 else 0)

    def everyone(fn, check_res=True):
        nonlocal steps
        snaps = []
        cycle = False
        for p in pls:
            if cycle and isinstance(p, ref.RefPlanner):
                continue  # graph_search.h:377-438 would walk the predecessor cycle forever
            r = fn(p)
            if p is pls[0] and isinstance(r, str):
                return r
            if p is pls[0] and check_res and (p.lpa_last_fault() & 2):
                cycle = True
            snaps.append(lpa_flow.snapshot(p, r if check_res and not isinstance(r, (int, np.integer)) else None))
        for k in range(1, len(snaps)):
            lpa_flow.assert_same([snaps[0]], [snaps[k]], "seed %d dim %d step %d impl %d" % (seed, dim, steps, k))
        steps += 1
        return "cycle" if cycle else snaps[0]

    def plan(p):
        r = p.lpa_plan(s, g)
        if p is pls[0] and r["status"] == 3 and r["pops"] == 0:
            return "empty-queue"
        return r

    x = everyone(plan)
    for rnd in range(rounds):
        if isinstance(x, str) or x["res"] is None or x["res"]["status"] != 0:
            break
        path = pls[0].lpa_best_child_states()[:, :dim]
        linked = [p.lpa_get_linked_nodes() for p in pls]
        for k in range(1, len(pls)):
            assert ref.same(linked[0], linked[k]), (seed, dim, "linked", k)
        action = rng.choice(["block", "block", "clear", "subtree"])
        if action == "clear" and not dropped:
            action = "block"
        if action == "block":
            c = np.round((path[rng.integers(len(path))] - origin) / res - 0.5).astype(int)
            half = int(rng.integers(0, 3))
            cand = np.array([[c[0] + dx, c[1] + dy] + ([c[2]] if dim == 3 else []) for dx in range(-half, half + 1) for dy in range(-half, half + 1)])
            cand = cand[np.all((cand >= 0) & (cand < nd), axis=1)]
            cand = cand[(grid[lin(cand)] >= 0) & (grid[lin(cand)] < 100)] if len(cand) else cand
            sc = np.round((s["pos"][0, :dim] - origin) / res - 0.5).astype(int)
            cand = cand[np.any(cand != sc, axis=1)] if len(cand) else cand  # the robot's own cell stays free
            if len(cand) == 0:
                continue
            grid[lin(cand)] = 100
            dropped.extend(map(tuple, cand))
            for m, p in zip(maps_, pls):
                m.set_cells(cand, 100)
            x = everyone(lambda p: p.lpa_update_blocked_nodes(cand), check_res=False)
        elif action == "clear":
            take = rng.permutation(len(dropped))[: max(1, len(dropped) // 2)]
            cells = np.array([dropped[i] for i in take])
            dropped = [d for i, d in enumerate(dropped) if i not in set(take.tolist())]
            grid[lin(cells)] = 0
            for m in maps_:
                m.set_cells(cells, 0)
            x = everyone(lambda p: p.lpa_update_cleared_nodes(cells), check_res=False)
        else:
            if len(path) < 3:
                continue
            k = int(rng.integers(1, min(3, len(path) - 1)))
            nxt = pls[0].lpa_waypoint(k)
            first = pls[0].lpa_get_sub_state_space(k)
            if first < 0:
                return steps, "fault"
            for p in pls[1:]:
                p.lpa_get_sub_state_space(k)
            x = everyone(lambda p: 0, check_res=False)
            s = nxt
        x = everyone(plan)
    return steps, "ok"


@pytest.mark.parametrize("dim", [2, 3])
def test_lpa_fuzz(dim):
    impls = [(oracle.OracleMap, oracle.OraclePlanner, {}), (ref.RefMap, ref.RefPlanner, {}),
             (lpa_emul.EmuMap, lpa_emul.EmuPlanner, dict(init_cap=128, init_pred=512))]
    total = 0
    for seed in range(24):
        n, why = run_sequence(seed, dim, impls)
        total += n
    assert total > 60, total  # the sequences actually ran several steps each
