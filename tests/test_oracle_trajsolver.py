"""TrajSolver / PolySolver oracle (oracle/poly_oracle.cpp) pinned three ways (CPU only):
(1) against the reference's OWN traj_solver.h / poly_solver.cpp / poly_traj.cpp compiled here over the stand-in Eigen
    (oracle/_ref, replayed from tests/golden/reference_calls/, see tests/ref_replay.py) — bit for bit;
(2) against the committed fixture tests/golden/trajsolver.npz recorded from those sources (tools/make_golden_trajsolver.py);
(3) against the mathematics: the spline interpolates every fixed derivative, is C^(N/2-1) at interior waypoints, and no
    random perturbation of the free derivatives lowers the integral of the squared R-th derivative (the reference
    publishes no numbers for this component: MPL/test/test_traj_solver.cpp only draws)."""
import math
import os

import numpy as np
import pytest

import oracle
import ref_replay as ref
from ref_replay import recorded_reference  # noqa: F401 (autouse fixture)
from trajsolver_cases import ACC, JRK, SNP, VEL, cases, random_case

GOLD = os.path.join(os.path.dirname(__file__), "golden", "trajsolver.npz")


def poly_eval(row, t, der):
    """d^der/dt^der of the Primitive1D polynomial with coefficient row `row` (highest order first, c_k / k!)."""
    v = 0.0
    for k in range(der, 6):
        ck = row[5 - k]  # coefficient of t^k / k!
        v += ck * t ** (k - der) / math.factorial(k - der)
    return v


def test_oracle_equals_reference_sources():
    for name, dim, control, yaw_control, wps, dts in cases():
        a = oracle.traj_solve(dim, control, wps, dts, yaw_control)
        b = ref.traj_solve(dim, control, wps, dts, yaw_control)
        assert a.shape == b.shape == (len(wps) - 1, dim + 1, 6), name
        assert ref.same(a, b), name
    path = [(0, 0), (1, 0), (2, 1), (5, 1)]  # the reference's own setPath / setV(1) / allocate_time flow
    for c in (VEL, ACC, JRK):
        co, dts = ref.traj_solve_path(2, c, path, 1.0)
        assert np.array_equal(dts, oracle.traj_allocate_time(2, path, 1.0))
        assert np.array_equal(dts, [1.0, 1.0, 3.0]) and co.shape == (3, 3, 6)


def test_oracle_equals_golden_fixture():
    gold = np.load(GOLD)
    n = 0
    for name, dim, control, yaw_control, wps, dts in cases():
        assert np.array_equal(oracle.traj_solve(dim, control, wps, dts, yaw_control), gold[name]), name
        n += 1
    assert n == len(gold.files)


def test_uninitialised_solver_and_short_lists():
    rs = np.random.RandomState(3)
    w, d = random_case(rs, 3, 5, SNP)
    assert len(oracle.traj_solve(3, SNP, w, d)) == 0      # traj_solver.h:28-30: no solver for SNP -> empty Trajectory
    assert len(oracle.traj_solve(3, JRK, w, d, yaw_control=SNP)) == 0
    assert len(oracle.traj_solve(3, JRK, w[:1], d[:0])) == 0  # poly_solver.cpp:31


def test_spline_properties():
    for name, dim, control, yaw_control, wps, dts in cases():
        co = oracle.traj_solve(dim, control, wps, dts, yaw_control)
        H = {VEL: 1, ACC: 2, JRK: 3}[control]
        scale = 1.0 + np.abs(co).max()
        for s in range(len(dts)):
            for a in range(dim):
                for end, w in ((0.0, wps[s]), (dts[s], wps[s + 1])):
                    for k, fld in enumerate(("pos", "vel", "acc")[:H]):
                        if (w["control"] >> k) & 1:  # a fixed derivative is interpolated
                            assert abs(poly_eval(co[s, a], end, k) - w[fld][a]) < 1e-8 * scale, (name, s, a, k)
                if s + 1 < len(dts):  # continuity of the first H derivatives at the interior waypoint
                    for k in range(H):
                        assert abs(poly_eval(co[s, a], dts[s], k) - poly_eval(co[s + 1, a], 0.0, k)) < 1e-7 * scale, (name, s, a, k)
        Hy = {VEL: 1, ACC: 2, JRK: 3}[yaw_control]  # yaw: key frames interpolated, end derivatives zero where fixed
        for s in range(len(dts)):
            assert abs(poly_eval(co[s, dim], 0.0, 0) - wps["yaw"][s]) < 1e-8 * scale
            assert abs(poly_eval(co[s, dim], dts[s], 0) - wps["yaw"][s + 1]) < 1e-8 * scale
        for k in range(1, Hy):
            assert abs(poly_eval(co[0, dim], 0.0, k)) < 1e-7 * scale
            assert abs(poly_eval(co[-1, dim], dts[-1], k)) < 1e-7 * scale


def test_minimises_the_cost():
    """Moving any interior free derivative away from the solver's choice (re-solving with it pinned) cannot lower
    sum_axes int (d^R p / dt^R)^2 dt."""
    rs = np.random.RandomState(5)

    def cost(co, dts, dim, R):
        j = 0.0
        for s in range(len(dts)):
            ts = np.linspace(0, dts[s], 400)
            for a in range(dim):
                v = np.array([poly_eval(co[s, a], t, R) for t in ts])
                j += np.trapezoid(v * v, ts)
        return j

    for control, R in ((ACC, 2), (JRK, 3)):
        w, d = random_case(rs, 2, 5, control, (VEL,))
        base = oracle.traj_solve(2, control, w, d)
        j0 = cost(base, d, 2, R)
        for trial in range(6):
            w2 = w.copy()
            i = 1 + trial % 3
            w2["control"][i] = ACC  # pin the velocity of an interior waypoint somewhere else
            w2["vel"][i, :2] = [poly_eval(base[i, a], 0.0, 1) for a in range(2)] + rs.uniform(-0.5, 0.5, size=2)
            j1 = cost(oracle.traj_solve(2, control, w2, d), d, 2, R)
            assert j1 >= j0 * (1 - 1e-6), (control, trial, j0, j1)


def numpy_poly_solve(dim, N, R, wps, dts, ncol_get):
    """The same closed form with numpy's LAPACK-backed dense algebra (an implementation that shares no code with the oracle or
    the stand-in Eigen): assembles A, Q, M exactly as poly_solver.cpp:40-171 does and solves with np.linalg.solve."""
    W, S, H = len(wps), len(wps) - 1, N // 2
    A = np.zeros((S * N, S * N))
    Q = np.zeros((S * N, S * N))
    for i in range(S):
        T = dts[i]
        for n in range(N):
            if n < H:
                A[i * N + n, i * N + n] = math.factorial(n)
            for r in range(H):
                if r <= n:
                    A[i * N + H + r, i * N + n] = math.factorial(n) // math.factorial(n - r) * T ** (n - r)
            for r in range(N):
                if r >= R and n >= R:
                    val = 1
                    for m in range(R):
                        val *= (r - m) * (n - m)
                    Q[i * N + r, i * N + n] = val * T ** (r + n - 2 * R + 1) / (r + n - 2 * R + 1)
    use = lambda w, k: (int(w["control"]) >> k) & 1  # noqa: E731
    nfixed = sum(use(w, k) for w in wps for k in range(H))
    table, raw, fix, fre = [], 0, 0, 0
    for wid, w in enumerate(wps):
        interior = 0 < wid < W - 1
        for k in range(H):
            nid = fix if use(w, k) else nfixed + fre
            table.append((raw, nid, wid, k))
            if interior:
                table.append((raw + H, nid, wid, k))
            raw += 1
            if use(w, k):
                fix += 1
            else:
                fre += 1
        if interior:
            raw += H
    M = np.zeros((S * N, W * H))
    for r, nid, _, _ in table:
        M[r, nid] = 1
    X = np.linalg.solve(A, M)
    Rm = X.T @ Q @ X
    D = np.zeros((W * H, dim))
    for r, nid, wid, k in table:
        if nid < nfixed:
            D[nid] = ncol_get(wps[wid], k)
    nfree = W * H - nfixed
    if W > 2 and nfree > 0:
        D[nfixed:] = -np.linalg.solve(Rm[nfixed:, nfixed:], Rm[nfixed:, :nfixed] @ D[:nfixed])
    d = M @ D
    out = np.zeros((S, dim, 6))
    for i in range(S):
        p = np.linalg.solve(A[i * N:(i + 1) * N, i * N:(i + 1) * N], d[i * N:(i + 1) * N])
        for a in range(dim):
            c = np.zeros(6)
            for k in range(N):
                c[k] = p[k, a] * math.factorial(k)
            out[i, a] = c[::-1]
    return out


def test_against_numpy_lapack():
    """Independent of the LU restatement: numpy (LAPACK getrf/getrs, BLAS products) on the same matrices agrees with the oracle to
    rounding — the bound that also covers a real Eigen build, whose blocked LU differs from the unblocked one in the same way."""
    worst = 0.0
    for name, dim, control, yaw_control, wps, dts in cases():
        N, R = {VEL: (2, 1), ACC: (4, 2), JRK: (6, 3)}[control]
        want = numpy_poly_solve(dim, N, R, wps, dts, lambda w, k: (w["pos"], w["vel"], w["acc"])[k][:dim])
        got = oracle.traj_solve(dim, control, wps, dts, yaw_control)[:, :dim]
        err = np.abs(got - want).max() / (1.0 + np.abs(want).max())
        worst = max(worst, err)
        assert err < 1e-7, (name, err)
    assert worst > 0  # different arithmetic, not the same code path
