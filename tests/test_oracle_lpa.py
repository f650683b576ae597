"""LPA* (SURVEY 8f.3) on the CPU side of the parity chain:
(1) the oracle's literal restatement equals the reference's OWN LPA* sources (oracle/_ref, replayed from
    tests/golden/reference_calls/, see tests/ref_replay.py) step by step
    over the replanning flows of tests/lpa_flow.py — result records, the whole state space in hm_ order (key, g, rhs, h,
    flags, hashes of the stored successor / predecessor lists), the priority-queue ARRAY, best_child_, the linked points;
(2) the oracle reproduces the committed fixture recorded from those sources (tests/golden/lpa_flows.npz);
(3) the DEVICE core (mpl_ros_b200/csrc/mplb_lpa_core.h), compiled for the host by tests/cpp/lpa_emul.cpp with the kernels'
    lane loops unrolled, equals the oracle on the same flows — with tiny initial arrays so that the stop / grow / resume path
    runs many times.  That build is test infrastructure; the product has no CPU path.
Known answer inside: the first LPA* plan on corridor.yaml expands 615 states at cost 351.5 (MPL/README.md:199-202; LPA* and A*
coincide on a first plan with a consistent heuristic)."""
import os

import numpy as np
import pytest

import oracle
import ref_replay as ref
from ref_replay import recorded_reference  # noqa: F401 (autouse fixture)
import lpa_emul
import lpa_flow

GOLD = os.path.join(os.path.dirname(__file__), "golden", "lpa_flows.npz")
FAST = [n for n in lpa_flow.FLOWS if n != "skir_jrk"]


@pytest.mark.parametrize("name", FAST)
def test_oracle_equals_reference_sources(name):
    a, _ = lpa_flow.run_flow(name, ref.RefMap, ref.RefPlanner)
    b, _ = lpa_flow.run_flow(name, oracle.OracleMap, oracle.OraclePlanner)
    lpa_flow.assert_same(b, a, name)


@pytest.mark.parametrize("name", list(lpa_flow.FLOWS))
def test_oracle_and_device_core_equal_the_fixture(name):
    gold = np.load(GOLD)[name]
    a, _ = lpa_flow.run_flow(name, oracle.OracleMap, oracle.OraclePlanner)
    small = dict(init_cap=256, init_pred=2048)
    b, emu = lpa_flow.run_flow(name, lpa_emul.EmuMap, lpa_emul.EmuPlanner, small)
    lpa_flow.assert_same(a, b, name + " (device core, host build)")
    assert emu.grows() >= 1, emu.grows()  # the stop-before-overflow / grow / resume path ran
    for snaps in (a, b):
        d = lpa_flow.digest(snaps)
        assert len(d) == len(gold), name
        for f in gold.dtype.names:
            assert np.array_equal(d[f], gold[f]), (name, f)


@pytest.mark.parametrize("name", ["skir_acc", "corridor_jrk"])
def test_device_core_variants(name):
    """(a) the one-lane tail (pop_finish) and the warp-wide tail (pop_finish_warp) leave identical states; (b) the warp-wide tail
    does not depend on the order in which the lanes of a phase run (build with the lane loops reversed)."""
    a, _ = lpa_flow.run_flow(name, oracle.OracleMap, oracle.OraclePlanner)
    for cm, cp, extra in ((lpa_emul.EmuMap, lpa_emul.EmuPlanner, dict(serial_finish=1)),
                          (lpa_emul.EmuMapRev, lpa_emul.EmuPlannerRev, dict(init_cap=512, init_pred=4096))):
        b, _ = lpa_flow.run_flow(name, cm, cp, extra)
        lpa_flow.assert_same(a, b, name + " " + cp.__name__)


def test_known_answer_corridor():
    snaps, _ = lpa_flow.run_flow("corridor_acc", oracle.OracleMap, oracle.OraclePlanner)
    r = snaps[0]["res"]
    assert (int(r["status"]), int(r["pops"]), float(r["cost"])) == (0, 615, 351.5)
