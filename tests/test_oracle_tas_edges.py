"""The kb_tas_find edge fixtures (tests/tas_edges.py) on the CPU oracle: each one reaches the path it is built for, and
the overcommitted hand cases give the values the reference's code paths give."""
import pytest

import oracle
from tests import tas_edges


@pytest.mark.parametrize("name", list(tas_edges.BUILDERS))
def test_fixture_precondition(name):
    case = tas_edges.BUILDERS[name]()
    case.check(oracle.tas_find(case.topo, case.reqs, case.capacity))


def test_case_a_hand_values():
    """addNonTASUsage (tas_flavor_snapshot.go:250-255) leaves n00-n19 with 4000 - 5000 = -1000m cpu; CountIn
    (requests.go:181-203) gives int32(-1000 / 1000) = -1 pods there (pods: 50 / 1 is larger) and 40 on n20 / n21.  The
    rack holds 20 * -1 + 2 * 40 = 60 >= 1 slice, so it is the fit domain and gets 1 pod.  Below the slice level its hosts
    are sorted by state ascending (sortedDomains :1495-1515): n00-n19, n20, n21.  updateCountsToMinimumGeneric
    (:1361-1428) with remaining 1 takes each -1 host whole (remaining grows to 21), then n20 (40 >= 21; the best fit
    among n20 / n21 keeps the first of equal states) with 21.  buildTopologyAssignmentForLevels drops only zero counts."""
    case = tas_edges.case_a()
    want = oracle.tas_find(case.topo, case.reqs, case.capacity)
    assert want.status.tolist() == [0]
    assert want.assignment(0) == [(i, -1) for i in range(20)] + [(20, 21)]


def test_case_b_hand_values():
    """n0: 4000 - 7000 = -3000m, so -3 pods; n1, n2: 4 each; the rack: 5 >= 2.  Hosts in ascending state: n0 (-3) raises
    remaining from 2 to 5, n1 (4 < 5) leaves 1, n2 takes that 1."""
    case = tas_edges.case_b()
    want = oracle.tas_find(case.topo, case.reqs, case.capacity)
    assert want.status.tolist() == [0]
    assert want.assignment(0) == [(0, -3), (1, 4), (2, 1)]
