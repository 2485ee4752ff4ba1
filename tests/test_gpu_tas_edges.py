"""kb_tas_find on the device against the CPU oracle at the edges of its kernels (fixtures: tests/tas_edges.py):
overcommitted leaves with negative counts, long walks through the sorted cache and its reset between requests, 1-,
2- and 5-level topologies, the request fields and CountIn's quantities, the full cfg5 topology, repeated calls on one
handle and a too-small assignment buffer."""
import ctypes as C

import numpy as np
import pytest

import oracle
from kueue_b200 import abi, tas
from tests import tas_edges
from tests.test_gpu_tas import _same

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ev():
    from kueue_b200 import native
    e = native.Evaluator(0)
    yield e
    e.close()


_WANT = {}


def _case(name):
    """A fixture and the oracle's result, built once per module."""
    if name not in _WANT:
        case = tas_edges.BUILDERS[name]()
        want = oracle.tas_find(case.topo, case.reqs, case.capacity)
        case.check(want)
        _WANT[name] = (case, want)
    return _WANT[name]


@pytest.mark.parametrize("name", list(tas_edges.BUILDERS))
def test_matches_oracle(ev, name):
    case, want = _case(name)
    _same(ev.tas_find(case.topo, case.reqs, case.capacity), want)


def test_repeatable_after_larger_batch(ev):
    """The handle's device buffer only grows: a batch run twice, and again after a larger unrelated batch, gives the same
    output each time (nothing is read from an earlier call's leftovers)."""
    small = [_case(n) for n in ("case_a", "overcommit", "two_levels")]
    big, big_want = _case("cache_reset")
    first = [ev.tas_find(c.topo, c.reqs, c.capacity) for c, _ in small]
    again = [ev.tas_find(c.topo, c.reqs, c.capacity) for c, _ in small]
    _same(ev.tas_find(big.topo, big.reqs, big.capacity), big_want)
    after = [ev.tas_find(c.topo, c.reqs, c.capacity) for c, _ in small]
    for (c, want), a, b, d in zip(small, first, again, after):
        _same(a, want); _same(b, want); _same(d, want)


@pytest.mark.parametrize("name", ["overcommit", "two_levels"])
def test_small_capacity(ev, name):
    """An assignment buffer smaller than the result: KB_ERR_CAPACITY, n_assigned and every status and start as with
    room enough, and the first `capacity` entries written."""
    from kueue_b200 import native
    case, want = _case(name)
    n = int(want.asg_start[-1])
    cap = n // 2
    assert 0 < cap < n
    out = tas.TasOut(case.reqs, cap)
    rc = native.lib().kb_tas_find(ev._h, C.byref(case.topo.struct), C.byref(case.reqs.struct), C.byref(out.struct))
    assert rc == abi.KB_ERR_CAPACITY
    assert out.struct.n_assigned == n
    assert np.array_equal(out.status, want.status) and np.array_equal(out.asg_start, want.asg_start)
    assert np.array_equal(out.asg_leaf[:cap], want.asg_leaf[:cap]) and np.array_equal(out.asg_count[:cap], want.asg_count[:cap])
