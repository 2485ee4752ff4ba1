"""GPU parity of k_cycle_flat's flavor walk for single-podset heads (kb_flat.cuh: flat_walk) against the CPU oracle,
on flat-cohort shapes that the BASELINE synth leaves out: borrowing limits, fair weights, fungibility policies,
remembered flavors, several resource groups, a pods resource, the PodSetReducer and more flavors than lanes."""
import numpy as np
import pytest

import oracle
from kueue_b200 import abi, synth
from tests.helpers import assert_cycle_equal

pytestmark = pytest.mark.gpu

K_CYCLE_FLAT = abi.KERNEL_NAMES.index("k_cycle_flat")


@pytest.fixture(scope="module")
def ev():
    from kueue_b200 import native
    e = native.Evaluator(0)
    e.set_profile(True)
    yield e
    e.close()


def _snap(seed=3, **kw):
    kw.setdefault("W", 3000); kw.setdefault("Q", 300)
    return synth.make_snapshot(3, heads="one_per_cq", seed=seed, **kw)


def _classical(snap):
    snap.flags &= ~abi.F_FAIR_SHARING
    return snap


def _borrow_limits(snap, seed=1):
    """BorrowingLimit on about half the ClusterQueue cells: 0, a third of nominal or nominal."""
    rng = np.random.default_rng(seed)
    Q, FR = snap.n_cq, snap.n_fr
    nom = np.asarray(snap.arrays["nominal"]).reshape(-1, FR)
    bl = np.asarray(snap.arrays["borrow_limit"]).reshape(-1, FR).copy()
    pick = rng.random((Q, FR)) < 0.5
    choice = rng.integers(0, 3, (Q, FR))
    val = np.where(choice == 0, 0, np.where(choice == 1, nom[:Q] // 3, nom[:Q]))
    bl[:Q] = np.where(pick, val, bl[:Q])
    snap.set("borrow_limit", bl)
    return snap.finalize()


def _weights(snap, seed=2):
    """Fair weights 0 (zero-weight borrowers), 0.5, 1 and 3 side by side in every cohort."""
    rng = np.random.default_rng(seed)
    fw = np.asarray(snap.arrays["fair_weight"]).copy()
    fw[:snap.n_cq] = rng.choice([0.0, 0.5, 1.0, 3.0], snap.n_cq)
    snap.set("fair_weight", fw)
    return snap.finalize()


def _no_prioritize_non_borrowing(snap):
    snap.flags &= ~abi.F_FS_PRIORITIZE_NON_BORROWING
    return snap


def _last_tried(snap, seed=4, nfl=None):
    """Workloads remembered from a previous cycle: with a current generation the walk starts past ps_last_tried
    (an index into the resource group's nfl flavors)."""
    rng = np.random.default_rng(seed)
    Q, F, R = snap.n_cq, snap.n_flavor, snap.n_resource
    gen = rng.integers(0, 4, Q)
    snap.set("cq_generation", gen)
    W = len(snap.arrays["wl_cq"])
    lg = np.where(rng.random(W) < 0.7, gen[snap.arrays["wl_cq"]] + rng.integers(-1, 2, W), -1)
    snap.set("wl_last_gen", lg)
    P = len(snap.arrays["ps_count"])
    snap.set("ps_last_tried", rng.integers(-1, (nfl or F) - 1, (P, R)))
    return snap.finalize()


def _fungibility(snap, seed=5):
    """whenCanBorrow / whenCanPreempt = TryNextFlavor or MayStopSearch, and all three preference settings."""
    rng = np.random.default_rng(seed)
    Q = snap.n_cq
    snap.set("cq_when_can_borrow", rng.choice([abi.FUNG_MAY_STOP_SEARCH, abi.FUNG_TRY_NEXT_FLAVOR], Q))
    snap.set("cq_when_can_preempt", rng.choice([abi.FUNG_MAY_STOP_SEARCH, abi.FUNG_TRY_NEXT_FLAVOR], Q))
    snap.set("cq_preference", rng.choice([abi.PREF_UNSET, abi.PREF_BORROWING_OVER_PREEMPTION, abi.PREF_PREEMPTION_OVER_BORROWING], Q))
    return snap.finalize()


def _no_fungibility(snap):
    snap.flags &= ~abi.F_FLAVOR_FUNGIBILITY
    return snap


def _two_groups(snap, uncovered=False):
    """Two resource groups per ClusterQueue: resources [0, R/2) on the first half of the flavors, the rest on the
    second half.  uncovered: every third ClusterQueue leaves its last resource out of both groups."""
    Q, F, R = snap.n_cq, snap.n_flavor, snap.n_resource
    lo = (1 << (R // 2)) - 1
    hi = ((1 << R) - 1) & ~lo
    masks = np.tile(np.array([lo, hi], np.int64), (Q, 1))
    if uncovered:
        masks[::3, 1] &= ~(1 << (R - 1))
    snap.set("cq_rg_start", np.arange(Q + 1) * 2)
    snap.set("rg_res_mask", masks.reshape(-1))
    snap.set("rg_flavor_start", np.arange(2 * Q + 1) * (F // 2))
    snap.set("rg_flavors", np.tile(np.arange(F), Q))
    return snap.finalize()


def _pods(snap, seed=6):
    """Resource R-1 is the pods resource: its request is the podset's count.  Every fourth ClusterQueue's group
    leaves it out (covers_pods false there)."""
    R = snap.n_resource
    snap.pods_resource = R - 1
    cnt = np.asarray(snap.arrays["ps_count"]).astype(np.int64)
    req = np.asarray(snap.arrays["ps_req"]).reshape(-1, R).copy()
    req[:, R - 1] = cnt
    snap.set("ps_req", req)
    Q = snap.n_cq
    masks = np.full(Q, (1 << R) - 1, np.int64)
    masks[::4] &= ~(1 << (R - 1))
    snap.set("rg_res_mask", masks)
    nom = np.asarray(snap.arrays["nominal"]).reshape(-1, snap.n_fr).copy()
    use = np.asarray(snap.arrays["cq_usage"]).reshape(Q, snap.n_fr).copy()
    rng = np.random.default_rng(seed)
    for f in range(snap.n_flavor):  # pods quota of a few dozen per flavor, usage around it
        c = f * R + R - 1
        nom[:Q, c] = rng.integers(4, 40, Q)
        use[:, c] = (nom[:Q, c] * rng.uniform(0.6, 1.2, Q)).astype(np.int64)
    snap.set("nominal", nom); snap.set("cq_usage", use)
    return snap.finalize()


# A root's relocated copy must fit shared memory for the cycle to run k_cycle_flat: with FR = 48 or 64 the synth's
# single root stays at 60 or 50 ClusterQueues.
CASES = {
    # single- and multi-podset heads in the same warps: both branches of the nominate phase side by side
    "mixed_podsets": lambda: _snap(podsets_max=3),
    "mixed_podsets_classical": lambda: _classical(_snap(podsets_max=3, seed=7)),
    # single podsets with min_count: the PodSetReducer runs for some heads, the rest take the flat walk
    "min_count_single": lambda: _snap(partial=True),
    "min_count_mixed": lambda: _classical(_snap(partial=True, podsets_max=2, seed=8)),
    "borrow_limits": lambda: _borrow_limits(_snap()),
    "borrow_limits_classical": lambda: _classical(_borrow_limits(_snap(seed=9))),
    "fair_weights": lambda: _weights(_snap()),
    "fair_weights_no_prio_nb": lambda: _no_prioritize_non_borrowing(_weights(_borrow_limits(_snap(seed=10)))),
    "last_tried": lambda: _last_tried(_snap()),
    "last_tried_16": lambda: _last_tried(_snap(F=16, W=500, Q=50)),
    "fungibility": lambda: _fungibility(_snap()),
    "fungibility_limits": lambda: _fungibility(_borrow_limits(_last_tried(_snap(seed=11)))),
    "no_fungibility": lambda: _no_fungibility(_snap()),
    "two_groups": lambda: _two_groups(_snap()),
    "two_groups_uncovered": lambda: _two_groups(_snap(seed=12), uncovered=True),
    "two_groups_16": lambda: _last_tried(_two_groups(_snap(F=16, W=500, Q=50)), nfl=8),
    "pods": lambda: _pods(_snap()),
    "pods_classical_min_count": lambda: _classical(_pods(_snap(partial=True, seed=13))),
    "flavors_12": lambda: _fungibility(_snap(F=12, W=600, Q=60)),
    "flavors_16_R2": lambda: _borrow_limits(_snap(F=16, R=2, W=1200, Q=120)),
}


@pytest.mark.parametrize("name", list(CASES))
def test_flat_walk_matches_oracle(ev, name):
    snap = CASES[name]()
    got = ev.run_cycle(snap)
    assert ev.stats().kernel_ms[K_CYCLE_FLAT] > 0, "the cycle did not run k_cycle_flat"
    assert_cycle_equal(got, oracle.run_cycle(snap))


def test_cases_cover_both_branches():
    """The mixed cases hold single-podset heads and heads that keep the generic walk."""
    snap = CASES["mixed_podsets"]()
    n = np.diff(np.asarray(snap.arrays["wl_ps_start"]))[np.asarray(snap.arrays["heads"])]
    assert (n == 1).any() and (n > 1).any()
    snap = CASES["min_count_single"]()
    h = np.asarray(snap.arrays["wl_ps_start"])[np.asarray(snap.arrays["heads"])]
    mc, cnt = np.asarray(snap.arrays["ps_min_count"])[h], np.asarray(snap.arrays["ps_count"])[h]
    reducer = (mc >= 0) & (cnt > mc)
    assert reducer.any() and (~reducer).any()
