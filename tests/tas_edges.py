"""kb_tas_find fixtures at the edges of its kernels (kueue_b200/csrc/kb_tas.cuh), shared by test_oracle_tas_edges.py
(CPU: every precondition) and test_gpu_tas_edges.py (device == oracle).

Every builder returns a Case: the topology, the finalized requests, an assignment capacity large enough for the oracle's
result (negative counts can make an assignment longer than its podset's count), and `check(want)`, which asserts on
the oracle's output that the fixture reaches the kernel path its docstring names."""
from __future__ import annotations

from collections import namedtuple

import numpy as np

from kueue_b200 import tas

H = tas.HOSTNAME
CACHE_MIN = 2048        # KB_TAS_CACHE_MIN: larger level sets are walked through the sorted cache (TasSel::next_cached)
CACHE_KEYS = 128 * 4    # KB_TAS_THREADS * KB_TAS_LOCAL: keys one fill of that cache holds
SEL_GRID_MAX = 8 * 148  # k_tas_select's grid on a 148-SM B200: a round with more requests runs several on one CTA
LIST_SLACK = 8          # k_tas_select's lists hold max(count) + 8 entries before they grow

Case = namedtuple("Case", "topo reqs capacity check")


def asg(out, q):
    return out.assignment(q)


def n_req(reqs):
    return len(reqs.rows)


def _node(name, labels, alloc, taints=None):
    return dict(name=name, labels=labels, allocatable=alloc, taints=taints or [])


# ---------------------------------------------------------------------------------------------------------------------
# overcommitted leaves: free capacity below zero gives negative counts (requests.go CountIn), and a walk in ascending
# state order takes those leaves first, each one raising what the rest of the walk has to place
# ---------------------------------------------------------------------------------------------------------------------
def case_a():
    """[rack, hostname], one rack of 22 hosts: n00-n19 hold 4000m cpu with 5000m of non-TAS usage (count -1 each),
    n20 / n21 hold 40000m.  One pod sliced at the rack: the rack's pods are distributed over its hosts in ascending
    state order, so all 20 negative hosts are taken before n20 takes 21 pods: 21 entries for a count of 1, longer than
    the list of max(count) + 8 entries and than the output region of min(count, leaves) entries."""
    nodes = [_node(f"n{i:02d}", {"rack": "r0", H: f"n{i:02d}"}, {"cpu": 40000 if i >= 20 else 4000, "pods": 50}) for i in range(22)]
    topo = tas.TasTopology(["rack", H], nodes, non_tas_usage={f"n{i:02d}": {"cpu": 5000} for i in range(20)})
    reqs = tas.TasRequests(topo).add(1, {"cpu": 1000}, 1, {"required": "rack", "sliceRequiredTopology": "rack", "sliceSize": 1}).finalize()

    def check(want):
        assert want.status[0] == 0 and len(asg(want, 0)) > int(reqs.count.max()) + LIST_SLACK
    return Case(topo, reqs, 64, check)


def case_b():
    """Three hosts of 4000m cpu in one rack, n0 carries 7000m of non-TAS usage (count -3).  Two pods sliced at the rack:
    three entries for an output region of two."""
    nodes = [_node(f"n{i}", {"rack": "r0", H: f"n{i}"}, {"cpu": 4000, "pods": 10}) for i in range(3)]
    topo = tas.TasTopology(["rack", H], nodes, non_tas_usage={"n0": {"cpu": 7000}})
    reqs = tas.TasRequests(topo).add(1, {"cpu": 1000}, 2, {"required": "rack", "sliceRequiredTopology": "rack", "sliceSize": 1}).finalize()

    def check(want):
        assert want.status[0] == 0 and len(asg(want, 0)) > min(int(reqs.count[0]), topo.n_leaves)
    return Case(topo, reqs, 64, check)


def _overcommit(t, rng, frac):
    """Push usage over capacity on `frac` of the leaves, half of them through TAS usage, half through non-TAS usage
    (negative free capacity).  Edits the arrays in place: the topology's ctypes struct points at them."""
    NL = t.n_leaves
    over = rng.random(NL) < frac
    via_tas = over & (rng.random(NL) < 0.5)
    via_free = over & ~via_tas
    t.usage[via_tas, :3] = (t.free[via_tas, :3] * rng.uniform(1.0, 1.3, (int(via_tas.sum()), 3))).astype(np.int64)
    t.free[via_free, :3] -= (t.free[via_free, :3] * rng.uniform(1.0, 1.3, (int(via_free.sum()), 3))).astype(np.int64)
    return over


def overcommit(seed=3):
    """2 blocks x 8 racks x 40 hosts, 20 % of the hosts overcommitted, 240 podsets in chains of 1-4: slices at the rack
    and at the block (levels above the leaves), LeastFreeCapacity walks of more pods than any host holds,
    unconstrained BestFit, preferred / required racks and blocks, implied requests.  Negative assumed usage of an
    earlier podset raises the capacity the next podset of its chain sees."""
    t = tas.synth_topology(2, 8, 40, seed=seed)
    rng = np.random.default_rng(seed)
    _overcommit(t, rng, 0.2)
    B, R_ = t.levels[0], t.levels[1]
    modes = []
    reqs = tas.TasRequests(t)
    chain, left = 0, 0
    for i in range(240):
        if left == 0:
            chain += int(rng.integers(1, 4))
            left = int(rng.integers(1, 5))
        left -= 1
        m = i % 8
        count = int(rng.integers(1, 41))
        req = {"cpu": int(rng.integers(1, 33)) * 1000, "memory": int(rng.integers(1, 65)) << 30}
        if rng.random() < 0.3:
            req["gpu"] = int(rng.integers(1, 3))
        mixed = True
        tr = [{"required": B, "sliceRequiredTopology": R_, "sliceSize": int(rng.integers(1, 3))},
              {"preferred": R_, "sliceRequiredTopology": R_, "sliceSize": 2},
              {"unconstrained": True},
              {"unconstrained": True},
              None,
              {"required": R_},
              {"preferred": B},
              {"sliceRequiredTopology": B, "sliceSize": 3}][m]
        if m == 2:
            req["cpu"] = max(req["cpu"], 8000); count = int(rng.integers(20, 41))  # no single host holds the podset
        if m == 3:
            mixed = False
        modes.append(m)
        reqs.add(chain, req, count, tr, profile_mixed=mixed)
    reqs.finalize()
    NL = t.n_leaves

    def check(want):
        n = n_req(reqs)
        ok = [q for q in range(n) if want.status[q] == 0]
        neg = [q for q in ok if any(c < 0 for _, c in asg(want, q))]
        assert any(len(asg(want, q)) > min(int(reqs.count[q]), NL) for q in ok)
        assert any(len(asg(want, q)) > int(reqs.count.max()) + LIST_SLACK for q in ok)
        assert any(modes[q] in (0, 7) for q in neg), "slices above the leaves over negative counts"
        assert any(modes[q] == 2 and sum(c > 0 for _, c in asg(want, q)) > 1 for q in neg), "LeastFreeCapacity walk, no host fits"
        assert any(modes[q] in (0, 1, 5, 6) for q in neg), "BestFit over negative counts"
        assert any(modes[q] == 3 for q in ok), "unconstrained BestFit"
        assert any(q > 0 and reqs.chain[q] == reqs.chain[q - 1] and want.status[q - 1] == 0 and any(c < 0 for _, c in asg(want, q - 1))
                   for q in ok), "a chained podset placed after one with negative counts"
        assert (want.status != 0).any()
    return Case(t, reqs, n_req(reqs) * NL, check)


def overcommit_deep(seed=5):
    """Five levels (2 x 3 x 2 x 3 x 2 = 72 hosts), a third of the hosts overcommitted, a slice level at every level.
    Domains whose count is 0 over negative hosts still hand pods down to them, at every depth below the slice level."""
    topo = _deep_topology(seed, over=0.35)
    reqs = _deep_requests(topo, seed)

    # counts of the chains' first podsets ({cpu: 1000}, nothing assumed yet): leaves, then sums up the tree
    pods = topo.free[:, topo.pods_resource]
    cpu = topo.free[:, topo.resources.index("cpu")]
    state = np.zeros(int(topo.level_start[-1]), np.int64)
    state[topo.level_start[-2]:] = np.minimum(np.trunc(cpu / 1000), pods)
    for d in range(int(topo.level_start[-1]) - 1, int(topo.level_start[1]) - 1, -1):
        state[topo.parent[d]] += state[d]

    def check(want):
        ok = [q for q in range(n_req(reqs)) if want.status[q] == 0]
        assert any(any(c < 0 for _, c in asg(want, q)) for q in ok)
        assert any(len(asg(want, q)) > min(int(reqs.count[q]), topo.n_leaves) for q in ok)
        for s in range(5):
            assert any(reqs.slice_level[q] == s for q in ok), s
        first = [q for q in ok if q == 0 or reqs.chain[q] != reqs.chain[q - 1]]

        def zero_ancestor(lf):
            d = int(topo.parent[topo.level_start[-2] + lf])
            while d >= 0 and state[d] != 0:
                d = int(topo.parent[d])
            return d >= 0
        assert any(c != 0 and zero_ancestor(lf) for q in first for lf, c in asg(want, q)), "pods below a domain of count 0"
    return Case(topo, reqs, n_req(reqs) * topo.n_leaves, check)


# ---------------------------------------------------------------------------------------------------------------------
# long walks through the sorted cache (level sets larger than CACHE_MIN), and its reset between requests of one CTA
# ---------------------------------------------------------------------------------------------------------------------
def _pods_per_host(t, rng, lo, hi):
    t.free[:, t.pods_resource] = rng.integers(lo, hi + 1, t.n_leaves)
    t.usage[:, t.pods_resource] = 0


def long_cached_hosts(seed=11):
    """1 block x 2 racks x 3000 hosts of 1-2 pods: podsets of 3000 pods walk past the cache's first fill (more than
    CACHE_KEYS leaves) at the 6000-host level, under LeastFreeCapacity, under BestFit and as an implied request."""
    t = tas.synth_topology(1, 2, 3000, seed=seed)
    _pods_per_host(t, np.random.default_rng(seed), 1, 2)
    reqs = tas.TasRequests(t)
    reqs.add(1, {"cpu": 1000}, 3000, {"unconstrained": True})
    reqs.add(2, {"cpu": 1000}, 3000, {"unconstrained": True}, profile_mixed=False)
    reqs.add(3, {"cpu": 2000}, 3000, None)
    reqs.finalize()

    def check(want):
        assert t.n_leaves > CACHE_MIN
        for q in range(3):
            assert want.status[q] == 0 and len(asg(want, q)) > CACHE_KEYS, q
    return Case(t, reqs, int(reqs.count.sum()) + 16, check)


def long_cached_racks(seed=13):
    """[rack, hostname] with 2100 racks of two hosts holding 0-1 pods: the level-0 walk (a preferred rack no rack
    holds, a slice-only request) goes through the cache past its first fill."""
    rng = np.random.default_rng(seed)
    nodes = [_node(f"h{i:05d}", {"rack": f"r{i // 2:05d}", H: f"h{i:05d}"}, {"cpu": 16000, "pods": int(rng.integers(0, 2)) if i % 7 else 1})
             for i in range(4200)]
    topo = tas.TasTopology(["rack", H], nodes)
    reqs = tas.TasRequests(topo)
    reqs.add(1, {"cpu": 1000}, 1500, {"preferred": "rack"})                                      # BestFit walk at level 0
    reqs.add(2, {"cpu": 1000}, 1200, {"sliceRequiredTopology": "rack", "sliceSize": 1})          # LeastFreeCapacity walk at level 0
    reqs.add(3, {"cpu": 1000}, 1300, {"preferred": "rack"}, profile_mixed=False)
    reqs.finalize()

    def check(want):
        assert topo.level_start[1] - topo.level_start[0] > CACHE_MIN
        for q in range(3):
            a = asg(want, q)
            assert want.status[q] == 0 and len({topo.parent[topo.level_start[1] + lf] for lf, _ in a}) > CACHE_KEYS, q
    return Case(topo, reqs, int(reqs.count.sum()) + 16, check)


def cache_reset(seed=17, n=1300):
    """More single-podset requests than SEL_GRID_MAX in one round over a level of 2200 hosts, cycling through three
    shapes (LeastFreeCapacity, BestFit, simulate-empty implied): a CTA's next request walks the same level with the
    same filter, so it would read a stale cache if the cache were not reset per request."""
    t = tas.synth_topology(1, 2, 1100, seed=seed)
    rng = np.random.default_rng(seed)
    _pods_per_host(t, rng, 1, 2)
    reqs = tas.TasRequests(t)
    for i in range(n):
        m = i % 3
        count = int(rng.integers(100, 900)) if m != 1 else int(rng.integers(1100, 1600))  # BestFit takes 2-pod hosts first
        if m == 0:
            reqs.add(i, {"cpu": 4000}, count, {"unconstrained": True})
        elif m == 1:
            reqs.add(i, {"cpu": 6000, "memory": 8 << 30}, count, {"unconstrained": True}, profile_mixed=False)
        else:
            reqs.add(i, {"cpu": 2000}, count, None, simulate_empty=True)
    reqs.finalize()

    def check(want):
        assert n > SEL_GRID_MAX and len(set(reqs.chain.tolist())) == n and t.n_leaves > CACHE_MIN
        assert SEL_GRID_MAX % 3 != 0  # request q and q + SEL_GRID_MAX (same CTA) have different shapes
        long = [q for q in range(n) if want.status[q] == 0 and len(asg(want, q)) > CACHE_KEYS]
        assert any(q >= SEL_GRID_MAX for q in long) and len({q % 3 for q in long}) == 3
    return Case(t, reqs, int(reqs.count.sum()) + 16, check)


# ---------------------------------------------------------------------------------------------------------------------
# topology shapes and request fields
# ---------------------------------------------------------------------------------------------------------------------
MEM_TRUNC_POS = (1 << 32) + 9   # (int32_t)(cap / 1) = 9
MEM_TRUNC_NEG = (1 << 32) - 5   # -5
MEM_TRUNC_MIN = 3 << 31         # INT32_MIN


def hostname_only():
    """L = 1 (the hostname level only: no reduce launch), 45 hosts (the last leaf_ok word is partial), tainted hosts
    and node selectors, and the CountIn edges: int64 capacities whose quotient does not fit int32 (memory in bytes
    with a 1-byte request truncates to 9, -5 and INT32_MIN), a zero request for a resource (INT32_MAX), a requested
    resource the host does not have (0) and a host without pods capacity (0)."""
    nodes = []
    for i in range(45):
        alloc = {"cpu": 8000 + 1000 * (i % 5), "memory": 1 << 30, "pods": 16 if i == 3 else 4 + i % 3}
        if i % 4 != 1:
            alloc["gpu"] = 2
        if i == 9:
            del alloc["pods"]
            alloc["cpu"] = 1 << 20
        alloc["memory"] = {3: MEM_TRUNC_POS, 5: MEM_TRUNC_NEG, 40: MEM_TRUNC_MIN}.get(i, alloc["memory"])
        taints = [{"key": "dedicated", "value": "x", "effect": "NoSchedule"}] if i % 6 == 2 else []
        nodes.append(_node(f"n{i:02d}", {H: f"n{i:02d}", "zone": "a" if i % 3 else "b"}, alloc, taints))
    topo = tas.TasTopology([H], nodes)
    tol = [{"key": "dedicated", "operator": "Exists", "effect": "NoSchedule"}]
    reqs = tas.TasRequests(topo)
    # n03 holds 16 pods and 2^32 + 9 bytes: 9 pods of one byte after the int32 truncation, 16 without it
    reqs.add(1, {"memory": 1}, 9, {"required": H})                                      # 0: fits n03 only
    reqs.add(2, {"memory": 1}, 10, {"required": H})                                     # 1: fits nowhere
    reqs.add(3, {"cpu": 1000}, 3, {"required": H}, tolerations=tol)                     # 2
    reqs.add(4, {"cpu": 1000}, 3, {"required": H})                                      # 3
    reqs.add(5, {"cpu": 1000, "gpu": 0}, 3, {"required": H})                            # 4: == 3
    reqs.add(6, {"cpu": 1000, "gpu": 1}, 40, {"unconstrained": True})                   # 5: hosts without gpu hold 0
    reqs.add(7, {"cpu": 4000}, 30, {"unconstrained": True}, node_selector={"zone": "a"})  # 6
    reqs.add(8, {"cpu": 4000}, 30, {"unconstrained": True}, profile_mixed=False, tolerations=tol)  # 7
    reqs.add(9, {"cpu": 1000}, 0, {"required": H})                                      # 8: count 0
    reqs.add(10, {"cpu": 1000}, 60, None, node_selector={"zone": "a"}, tolerations=tol)  # 9
    reqs.add(11, {"cpu": 1000}, 2000, {"preferred": H})                                 # 10: no fit
    reqs.finalize()
    leaf = {v[0]: i for i, v in enumerate(topo.leaf_values)}

    def check(want):
        assert topo.n_leaves % 32 != 0 and topo.level_start.tolist() == [0, topo.n_leaves]
        assert (np.int64(MEM_TRUNC_POS).astype(np.int32), np.int64(MEM_TRUNC_NEG).astype(np.int32)) == (9, -5)
        assert np.int64(MEM_TRUNC_MIN).astype(np.int32) == np.iinfo(np.int32).min
        assert want.status[0] == 0 and asg(want, 0) == [(leaf["n03"], 9)]
        assert want.status[1] == 1
        assert want.status[3] == 0 and asg(want, 3) == asg(want, 4)
        assert want.status[5] == 0 and all(lf % 4 != 1 for lf, _ in asg(want, 5))
        assert want.status[6] == 0 and all(lf % 3 for lf, _ in asg(want, 6))
        assert any(lf % 6 == 2 for q in (2, 7, 9) for lf, _ in asg(want, q)), "a tolerated taint"
        assert not any(lf % 6 == 2 for q in (3, 4, 5, 6) for lf, _ in asg(want, q))
        assert not any(lf == leaf["n09"] for q in range(n_req(reqs)) for lf, _ in asg(want, q)), "no pods capacity"
        assert any(lf >= 32 for q in (6, 7, 9) for lf, _ in asg(want, q)), "the last leaf_ok word"
        assert want.status[8] == 0 and asg(want, 8) == []
        assert want.status[10] == 1
    return Case(topo, reqs, 4096, check)


def two_levels():
    """L = 2: 5 racks x 7 hosts with TAS usage on some hosts; required / preferred at both levels, slices of 2 and 3
    at the rack with counts of 0, below the slice size and not divisible by it; simulate-empty next to an otherwise
    identical plain request (they must not share a shape's counts); chains of 5 and 6 podsets in which podset k
    fails or is a bad request (level below the slice level, slice size 0), so the rest report -1; chain ids that jump
    and many chains of one round-0 shape."""
    nodes, tas_usage = [], {}
    for r in range(5):
        for h in range(7):
            name = f"r{r}h{h}"
            nodes.append(_node(name, {"rack": f"r{r}", H: name}, {"cpu": 6000 + 1000 * h, "pods": 8}))
            if (r + h) % 3 == 0:
                tas_usage[name] = {"cpu": 3000, "pods": 2}
    topo = tas.TasTopology(["rack", H], nodes, tas_usage=tas_usage)
    reqs = tas.TasRequests(topo)
    s2 = {"required": "rack", "sliceRequiredTopology": "rack", "sliceSize": 2}
    s3 = {"preferred": "rack", "sliceRequiredTopology": "rack", "sliceSize": 3}
    reqs.add(1, {"cpu": 1000}, 20, {"preferred": "rack"})
    reqs.add(2, {"cpu": 1000}, 20, {"preferred": "rack"}, simulate_empty=True)
    reqs.add(3, {"cpu": 1000}, 7, {"required": "rack"})
    reqs.add(4, {"cpu": 1000}, 4, {"required": H})
    reqs.add(5, {"cpu": 1000}, 4, {"preferred": H})
    reqs.add(6, {"cpu": 1000}, 9, s2)       # not divisible: 4 slices of 2
    reqs.add(7, {"cpu": 1000}, 1, s2)       # below the slice size: no slice, nothing placed
    reqs.add(8, {"cpu": 1000}, 0, s3)
    reqs.add(9, {"cpu": 1000}, 13, s3)
    reqs.add(10, {"cpu": 1000}, 40, {"unconstrained": True}, profile_mixed=False)
    # chains: podset k fails (or is a bad request), the later ones report -1
    cid = 20
    for k, bad in ((2, None), (3, "level"), (1, "slice0"), (4, None)):
        cid += 7
        for i in range(6):
            if i == k and bad == "level":
                reqs.add(cid, {"cpu": 1000}, 2, {"required": H, "sliceRequiredTopology": "rack", "sliceSize": 1})
            elif i == k and bad == "slice0":
                reqs.add(cid, {"cpu": 1000}, 2, {"required": "rack", "sliceRequiredTopology": "rack"})
            elif i == k:
                reqs.add(cid, {"cpu": 1000}, 500, {"required": "rack"})
            else:
                reqs.add(cid, {"cpu": 2000}, 3, {"preferred": "rack"})
    for j in range(12):  # one round-0 shape shared by many chains
        cid += 1 + j
        reqs.add(cid, {"cpu": 1500}, 2 + j, {"preferred": "rack"})
        reqs.add(cid, {"cpu": 1500}, 2, {"required": H})
    reqs.finalize()

    def check(want):
        st = want.status.tolist()
        assert st[0] == 0 and st[1] == 0 and asg(want, 0) != asg(want, 1), "simulate-empty sees other counts"
        assert st[5] == 0 and sum(c for _, c in asg(want, 5)) == 8
        assert st[6] == 0 and asg(want, 6) == [] and st[7] == 0 and asg(want, 7) == []
        assert st[8] == 0 and sum(c for _, c in asg(want, 8)) == 12
        chains = {}
        for q in range(n_req(reqs)):
            chains.setdefault(int(reqs.chain[q]), []).append(st[q])
        failing = [c for c in chains.values() if len(c) >= 5]
        assert len(failing) == 4
        assert sorted(next(s for s in c if s > 0) for c in failing) == [1, 1, 2, 2]
        for c in failing:
            k = next(i for i, s in enumerate(c) if s != 0)
            assert all(s == 0 for s in c[:k]) and all(s == -1 for s in c[k + 1:]) and k + 1 < len(c)
    return Case(topo, reqs, 4096, check)


def _deep_topology(seed, over):
    rng = np.random.default_rng(seed)
    levels = ["l0", "l1", "l2", "l3", H]
    fan = [2, 3, 2, 3, 2]
    nodes, non_tas = [], {}
    for i in range(int(np.prod(fan))):
        digits, x = [], i
        for f in reversed(fan):
            digits.append(x % f); x //= f
        digits = digits[::-1]
        name = "h" + "".join(map(str, digits))
        labels = {lv: "".join(map(str, digits[:j + 1])) for j, lv in enumerate(levels[:-1])}
        labels[H] = name
        nodes.append(_node(name, labels, {"cpu": int(rng.integers(2, 9)) * 1000, "pods": 16}))
        if rng.random() < over:
            non_tas[name] = {"cpu": int(rng.integers(9, 13)) * 1000}
    return tas.TasTopology(levels, nodes, non_tas_usage=non_tas)


def _deep_requests(topo, seed):
    rng = np.random.default_rng(seed + 1)
    reqs = tas.TasRequests(topo)
    chain = 0
    for s in range(5):
        for lv in range(s + 1):
            for kind in ("required", "preferred"):
                for ss in (1, 2, 3):
                    chain += 1
                    count = int(rng.integers(0, 25)) if lv < 4 else int(rng.integers(0, 8))
                    tr = {kind: topo.levels[lv], "sliceRequiredTopology": topo.levels[s], "sliceSize": ss}
                    reqs.add(chain, {"cpu": 1000}, count, tr)
                    reqs.add(chain, {"cpu": 500}, max(1, count // 2), {"unconstrained": True}, profile_mixed=bool(ss % 2))
    return reqs.finalize()


def five_levels(seed=7):
    """L = 5 (2 x 3 x 2 x 3 x 2 hosts, no overcommit): the slice level at every level with slice sizes 1-3, required and
    preferred at every level at or above it, each followed in its chain by an unconstrained podset."""
    topo = _deep_topology(seed, over=0.0)
    reqs = _deep_requests(topo, seed)

    def check(want):
        ok = [q for q in range(n_req(reqs)) if want.status[q] == 0]
        for s in range(5):
            assert any(reqs.slice_level[q] == s and reqs.slice_size[q] > 1 and reqs.count[q] > 0 for q in ok), s
        for lv in range(5):
            for f in (1, 0):
                assert any(reqs.level[q] == lv and (reqs.flags[q] & 1) == f for q in ok), (lv, f)
        assert (want.status != 0).any()
    return Case(topo, reqs, n_req(reqs) * topo.n_leaves, check)


def odd_sizes(seed=19):
    """3 blocks x 100 racks x 3 hosts: 300 racks and 900 hosts, neither a multiple of 128 or 256, with 10 % of the
    hosts overcommitted; the synthetic request mix in chains."""
    t = tas.synth_topology(3, 100, 3, seed=seed)
    _overcommit(t, np.random.default_rng(seed), 0.1)
    reqs = tas.synth_requests(t, 300, seed=seed, chains=True, max_pods=48)

    def check(want):
        sizes = np.diff(t.level_start)
        assert all(s % 128 for s in sizes[1:])
        assert (want.status == 0).any() and (want.status != 0).any()
        assert any(any(c < 0 for _, c in asg(want, q)) for q in range(n_req(reqs)) if want.status[q] == 0)
    return Case(t, reqs, n_req(reqs) * t.n_leaves, check)


def cfg5(n=1000):
    """The benchmark's cfg5 topology (10 blocks x 100 racks x 100 hosts) and request mix (seed 7), cut to n requests."""
    t = tas.synth_topology(10, 100, 100)
    reqs = tas.synth_requests(t, n, seed=7, shapes=16)

    def check(want):
        assert t.n_leaves == 100_000 and (want.status == 0).any() and (want.status != 0).any()
    return Case(t, reqs, int(reqs.count.sum()) + 16, check)


BUILDERS = {f.__name__: f for f in (case_a, case_b, overcommit, overcommit_deep, long_cached_hosts, long_cached_racks, cache_reset,
                                    hostname_only, two_levels, five_levels, odd_sizes, cfg5)}
