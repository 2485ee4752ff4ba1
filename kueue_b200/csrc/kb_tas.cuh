// kb_tas.cuh — topology-aware placement of one TAS ResourceFlavor on the device (kb_tas_find, SURVEY.md §8 a19 / K7).
//
// Reference: pkg/cache/scheduler/tas_flavor_snapshot.go — FindTopologyAssignmentsForFlavor :485-560,
// findTopologyAssignment :765-970, findLevelWithFitDomains :1200-1282, updateCountsToMinimumGeneric :1361-1428,
// sortedDomains :1495-1515, fillInCounts / fillInCountsHelper :1517-1672, Requests.CountIn pkg/resources/requests.go:172-205.
//
// Phase 1 (fillInCounts) is the O(leaves) part and does not depend on the podset's count or level, only on its
// per-pod request "shape": it runs ONCE PER DISTINCT SHAPE of the batch (k_tas_leaf: one thread per leaf, coalesced
// [leaf][resource] rows; k_tas_reduce: one thread per parent, its children are contiguous because domains are
// numbered in lexicographic levelValues order).  Phase 2 (level choice, greedy minimisation level by level) is one
// CTA per podset on the read-only counts of its shape: the reference's "sort the domains, walk them in order" becomes
// "repeated block-wide arg-min over the candidate set" (no sort, no per-podset copy of the tree); the only values the
// reference mutates are the counts of the domains it selects, which live in the podset's own result list.
#pragma once

#include <climits>

#include "kb_device.cuh"

struct TasDev {
  int L, n_domains, n_leaves, leaf0, R, pods_res, n_req;
  const int32_t *level_start, *parent, *child_start;  // child_start[d]..child_start[d+1]: children (next level), contiguous
  const i64 *free_cap, *tas_usage; const uint32_t *cap_mask, *usage_mask;
  // requests
  const i64 *pod_request; const uint32_t *request_mask, *flags, *leaf_ok;
  const int32_t *count, *slice_size, *level, *slice_level, *slot, *chain_slot, *pred;
  int ok_words;
  // per shape slot: counts of every domain
  int32_t *state, *slice;   // [n_slots][n_domains]
  // per chain with more than one podset: assumed usage
  i64 *assumed; uint32_t *assumed_mask;  // [n_chain_slots][n_leaves][R] / [n_chain_slots][n_leaves]
  // results
  int32_t *status, *n_out, *tmp_start, *tmp_leaf, *tmp_count;
  // per-CTA lists of k_tas_select
  int32_t *lists; int list_cap;
  // grow[0]: longest list a request needed beyond list_cap; grow[1]: requests whose output region was too small;
  // grow[2 + q]: entries request q needed.  A request that overflows stores nothing and reports KB_TAS_GROW; the host
  // reruns the whole call with larger buffers.
  int32_t *grow;
  // per shape slot of the current round: some leaf has a negative count (overcommitted: free capacity below zero)
  int32_t *neg;
};
// internal status of a request that needs larger buffers (never returned: kb_tas_find reruns)
#define KB_TAS_GROW 3

// slot descriptors: which request defines the shape of slot s (its request row / mask / flags / eligibility / chain)
__global__ void k_tas_leaf(TasDev T, const int32_t *slot_req, int n_slots) {
  const int lf = blockIdx.x * blockDim.x + threadIdx.x;
  const int s = blockIdx.y;
  if (lf >= T.n_leaves || s >= n_slots) return;
  const int q = slot_req[s];
  const int R = T.R;
  int32_t st = 0;
  bool ok = !T.leaf_ok || ((T.leaf_ok[(size_t)q * T.ok_words + lf / 32] >> (lf % 32)) & 1);  // taints / selectors, host-evaluated (:1541-1571)
  if (ok) {
    const int cs = T.chain_slot[q];
    uint32_t mask = T.cap_mask[lf];
    const bool sim_empty = T.flags[q] & KB_TAS_SIMULATE_EMPTY;
    if (!sim_empty) mask |= T.usage_mask[lf];
    if (cs >= 0) mask |= T.assumed_mask[(size_t)cs * T.n_leaves + lf];
    const uint32_t keys = T.request_mask[q] | (1u << T.pods_res);
    bool have = false; int32_t result = 0;
    for (int k = 0; k < R; k++) {  // Requests.CountIn requests.go:172-205
      if (!((keys >> k) & 1)) continue;
      i64 v = k == T.pods_res ? 1 : T.pod_request[(size_t)q * R + k];
      if (!((mask >> k) & 1) && v != 0) { have = true; result = 0; break; }
      i64 cap = T.free_cap[(size_t)lf * R + k];
      if (!sim_empty) cap -= T.tas_usage[(size_t)lf * R + k];
      if (cs >= 0) cap -= T.assumed[((size_t)cs * T.n_leaves + lf) * R + k];
      int32_t c = v == 0 ? INT32_MAX : (int32_t)(cap / v);
      if (!have || c < result) { result = c; have = true; }
    }
    st = have ? result : 0;
    if (st < 0) T.neg[s] = 1;
  }
  const int L = T.L;
  T.state[(size_t)s * T.n_domains + T.leaf0 + lf] = st;
  T.slice[(size_t)s * T.n_domains + T.leaf0 + lf] = (L - 1 == T.slice_level[q]) ? st / T.slice_size[q] : 0;  // fillInCountsHelper leaf :1622-1629
}
// one level up: domain = sum of its (contiguous) children; sliceState re-derived at the slice level (:1630-1671)
__global__ void k_tas_reduce(TasDev T, const int32_t *slot_req, int n_slots, int level) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const int s = blockIdx.y;
  const int a = T.level_start[level], b = T.level_start[level + 1];
  if (a + i >= b || s >= n_slots) return;
  const int d = a + i;
  const int q = slot_req[s];
  const int32_t *st = T.state + (size_t)s * T.n_domains, *sl = T.slice + (size_t)s * T.n_domains;
  int32_t cap = 0, sc = 0;
  for (int c = T.child_start[d]; c < T.child_start[d + 1]; c++) { cap += st[c]; sc += sl[c]; }
  if (level == T.slice_level[q]) sc = cap / T.slice_size[q];
  T.state[(size_t)s * T.n_domains + d] = cap;
  T.slice[(size_t)s * T.n_domains + d] = sc;
}

// ---------------------------------------------------------------------------
// Phase 2: one CTA per podset request.
// ---------------------------------------------------------------------------
#define KB_TAS_THREADS 128
#define KB_TAS_LOCAL 4        // cached candidates per thread
#define KB_TAS_CACHE_MIN 2048 // level sets larger than this are walked through the sorted cache
struct TasKey { int v, k0, k1, d; };  // lexicographic; d < 0 = none
__device__ __forceinline__ bool tk_less(const TasKey &a, const TasKey &b) {
  if (b.d < 0) return a.d >= 0;
  if (a.d < 0) return false;
  if (a.v != b.v) return a.v < b.v;
  if (a.k0 != b.k0) return a.k0 < b.k0;
  if (a.k1 != b.k1) return a.k1 < b.k1;
  return a.d < b.d;
}
__device__ inline TasKey tk_block_min(TasKey k, TasKey *s_red) {
  for (int o = 16; o > 0; o >>= 1) {
    TasKey x;
    x.v = __shfl_xor_sync(0xffffffffu, k.v, o); x.k0 = __shfl_xor_sync(0xffffffffu, k.k0, o);
    x.k1 = __shfl_xor_sync(0xffffffffu, k.k1, o); x.d = __shfl_xor_sync(0xffffffffu, k.d, o);
    if (tk_less(x, k)) k = x;
  }
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  __syncthreads();
  if (lane == 0) s_red[w] = k;
  __syncthreads();
  TasKey r = s_red[0];
  for (int i = 1; i < (int)(blockDim.x >> 5); i++) if (tk_less(s_red[i], r)) r = s_red[i];
  return r;
}

// A candidate set: a contiguous range of domains, or the children of a list of parent domains.
struct TasSet { int a, b; const int32_t *parents; int np; };

struct TasSel {
  const TasDev &T;
  const int32_t *st, *sl;  // counts of the request's shape (read-only)
  bool lfc;                // LeastFreeCapacity order (:1291-1294)
  TasKey *s_red;
  TasKey *s_cache; int *s_cmeta;  // sorted candidate cache of a large level set + {a, b, filter, arg, n valid, complete}
  // sort key of sortedDomains :1495-1515: sliceState (desc, or asc under LeastFreeCapacity), state asc, levelValues asc.
  // ~x = -x - 1 reverses the order of every int32, INT32_MIN included (a truncated CountIn can produce it)
  __device__ __forceinline__ TasKey key(int d) const { TasKey k; k.v = 0; k.k0 = lfc ? sl[d] : ~sl[d]; k.k1 = st[d]; k.d = d; return k; }
  template <typename F> __device__ inline void for_each(const TasSet &S, F f) const {
    if (!S.parents) { for (int d = S.a + threadIdx.x; d < S.b; d += blockDim.x) f(d); return; }
    for (int i = 0; i < S.np; i++) {
      int p = S.parents[i];
      for (int d = T.child_start[p] + threadIdx.x; d < T.child_start[p + 1]; d += blockDim.x) f(d);
    }
  }
  // next domain of S in sorted order strictly after `after` (after.d < 0: the first).  filter 1: only domains whose
  // sliceState >= arg; filter 2 / 3: skip domains whose sliceState / state is 0 — the reference appends them with zero
  // pods (they sort first under LeastFreeCapacity), which changes nothing downstream while no count is negative: their
  // descendants get zero pods and buildTopologyAssignmentForLevels drops zero counts (:1443-1446).  A zero domain
  // over a negative leaf does hand pods to its descendants, so a shape with a negative leaf walks with filter 0.
  // Large level sets (tens of thousands of hosts) are walked through a sorted CACHE of their smallest keys: one pass
  // keeps every thread's KB_TAS_LOCAL best candidates, the block sorts their union in shared memory, and all keys up
  // to T = the smallest "worst kept key" among the threads that had to drop something are provably complete (every
  // dropped key is larger than its thread's worst kept key >= T).  Successive next() calls are served from the cache;
  // a new pass starts behind the last served key only when the walk runs past T.
  __device__ inline TasKey next(const TasSet &S, TasKey after, int filter, int arg) const {
    if (!S.parents && S.b - S.a > KB_TAS_CACHE_MIN) return next_cached(S, after, filter, arg);
    return next_pass(S, after, filter, arg);
  }
  __device__ inline TasKey next_cached(const TasSet &S, TasKey after, int filter, int arg) const {
    const TasKey none{0, 0, 0, -1};
    for (int attempt = 0; attempt < 2; attempt++) {
      __syncthreads();
      // the cache answers walks that are at or behind the key it was filled from
      const TasKey from = s_cache[KB_TAS_THREADS * KB_TAS_LOCAL];
      const bool valid = s_cmeta[0] == S.a && s_cmeta[1] == S.b && s_cmeta[2] == filter && s_cmeta[3] == arg && s_cmeta[4] >= 0 &&
                         (from.d < 0 || (after.d >= 0 && !tk_less(after, from)));
      if (valid) {
        const int n = s_cmeta[4];
        // first cached key after `after` (the cache is sorted ascending); lanes search disjoint strides, block-min picks the first
        TasKey best = none;
        for (int i = threadIdx.x; i < n; i += blockDim.x) { TasKey k = s_cache[i]; if (after.d < 0 || tk_less(after, k)) { best = k; break; } }
        best = tk_block_min(best, s_red);
        if (best.d >= 0) return best;
        if (s_cmeta[5]) return none;  // the cache held every qualifying domain
        // past the complete part: is `after` at or beyond the cache's first key?  then refill behind it, else (walk restarted
        // before the cached window) refill from `after` as well
      }
      // ---- fill: one pass, KB_TAS_LOCAL best per thread
      TasKey loc[KB_TAS_LOCAL];
#pragma unroll
      for (int j = 0; j < KB_TAS_LOCAL; j++) loc[j] = none;
      bool dropped = false;
      for (int d = S.a + threadIdx.x; d < S.b; d += blockDim.x) {
        TasKey k = key(d);
        if (after.d >= 0 && !tk_less(after, k)) continue;
        if (filter == 1 && sl[d] < arg) continue;
        if (filter == 2 && sl[d] == 0) continue;
        if (filter == 3 && st[d] == 0) continue;
        if (loc[KB_TAS_LOCAL - 1].d >= 0 && !tk_less(k, loc[KB_TAS_LOCAL - 1])) { dropped = true; continue; }
        if (loc[KB_TAS_LOCAL - 1].d >= 0) dropped = true;
        loc[KB_TAS_LOCAL - 1] = k;
#pragma unroll
        for (int j = KB_TAS_LOCAL - 1; j > 0; j--) if (tk_less(loc[j], loc[j - 1])) { TasKey t = loc[j]; loc[j] = loc[j - 1]; loc[j - 1] = t; }
      }
      __syncthreads();
#pragma unroll
      for (int j = 0; j < KB_TAS_LOCAL; j++) s_cache[threadIdx.x * KB_TAS_LOCAL + j] = loc[j];
      // T: smallest worst-kept key among the threads that dropped something
      TasKey tmin = dropped ? loc[KB_TAS_LOCAL - 1] : none;
      tmin = tk_block_min(tmin, s_red);
      // bitonic sort of the KB_TAS_THREADS * KB_TAS_LOCAL cached keys (`none` sorts last)
      const int NC = KB_TAS_THREADS * KB_TAS_LOCAL;
      for (int k2 = 2; k2 <= NC; k2 <<= 1)
        for (int j = k2 >> 1; j > 0; j >>= 1) {
          __syncthreads();
          for (int i = threadIdx.x; i < NC; i += blockDim.x) {
            int l = i ^ j;
            if (l > i) {
              TasKey a = s_cache[i], b = s_cache[l];
              bool up = (i & k2) == 0;
              if (up ? tk_less(b, a) : tk_less(a, b)) { s_cache[i] = b; s_cache[l] = a; }
            }
          }
        }
      __syncthreads();
      if (threadIdx.x == 0) {
        int n = 0;
        while (n < NC && s_cache[n].d >= 0 && (tmin.d < 0 || !tk_less(tmin, s_cache[n]))) n++;  // keys <= T are complete
        s_cmeta[0] = S.a; s_cmeta[1] = S.b; s_cmeta[2] = filter; s_cmeta[3] = arg; s_cmeta[4] = n; s_cmeta[5] = tmin.d < 0;
        s_cache[NC] = after;
      }
    }
    return next_pass(S, after, filter, arg);  // not reached in practice: a fresh cache always holds the successor when one exists
  }
  __device__ inline TasKey next_pass(const TasSet &S, TasKey after, int filter, int arg) const {
    TasKey best; best.d = -1; best.v = best.k0 = best.k1 = 0;
    for_each(S, [&](int d) {
      TasKey k = key(d);
      if (after.d >= 0 && !tk_less(after, k)) return;
      if (filter == 1 && sl[d] < arg) return;
      if (filter == 2 && sl[d] == 0) return;
      if (filter == 3 && st[d] == 0) return;
      if (tk_less(k, best)) best = k;
    });
    return tk_block_min(best, s_red);
  }
  // findBestFitDomainBy :1183-1198 over the part of S at or after `from` in sorted order: lowest value >= needed, first
  // occurrence in sorted order; `from` itself when nothing qualifies better
  __device__ inline TasKey best_fit(const TasSet &S, TasKey from, int needed, bool slices) const {
    TasKey best; best.d = -1; best.v = best.k0 = best.k1 = 0;
    for_each(S, [&](int d) {
      TasKey k = key(d);
      if (tk_less(k, from)) return;  // before `from` in sorted order
      int val = slices ? sl[d] : st[d];
      if (val < needed) return;
      k.v = val;
      if (tk_less(k, best)) best = k;
    });
    best = tk_block_min(best, s_red);
    int fv = slices ? sl[from.d] : st[from.d];
    if (best.d < 0 || !(best.v < fv)) return from;  // strictly lower value required to replace (:1190)
    best.v = 0;
    return best;
  }
};

// result lists of one CTA: [domain][assigned state][assigned sliceState], two buffers (current / next level)
__device__ inline void tas_select_one(const TasDev &T, const int q, TasKey *s_red, int &s_n, TasKey *s_cache, int *s_cmeta) {
  const int cap = T.list_cap;
  int32_t *base = T.lists + (size_t)blockIdx.x * 6 * cap;
  int32_t *c_d = base, *c_st = base + cap, *c_sl = base + 2 * cap, *n_d = base + 3 * cap, *n_st = base + 4 * cap, *n_sl = base + 5 * cap;
  const uint32_t flags = T.flags[q];
  const int32_t count = T.count[q], sliceSize = T.slice_size[q];
  const int levelIdx = T.level[q], sliceLevel = T.slice_level[q], L = T.L;
  const bool required = flags & KB_TAS_REQUIRED, unconstrained = flags & KB_TAS_UNCONSTRAINED;
  auto finish = [&](int status, int n) { if (threadIdx.x == 0) { T.status[q] = status; T.n_out[q] = n; } };
  // a list longer than list_cap: record its length and give up (kb_tas_find reruns with larger lists)
  auto grow_lists = [&](int n) { if (threadIdx.x == 0) atomicMax(&T.grow[0], n); finish(KB_TAS_GROW, 0); };
  if (T.pred[q] >= 0 && T.status[T.pred[q]] != KB_TAS_OK) { finish(-1, 0); return; }  // the chain stopped at an earlier podset (:551-553)
  if (levelIdx < 0 || levelIdx >= L || sliceLevel < 0 || sliceLevel >= L || levelIdx > sliceLevel || sliceSize < 1) { finish(KB_TAS_BAD_REQUEST, 0); return; }
  const int slot = T.slot[q];
  TasSel X{T, T.state + (size_t)slot * T.n_domains, T.slice + (size_t)slot * T.n_domains, unconstrained && (flags & KB_TAS_PROFILE_MIXED), s_red, s_cache, s_cmeta};
  if (threadIdx.x == 0) s_cmeta[4] = -1;  // the cache belongs to one request (its shape's counts)
  __syncthreads();
  const bool lfc = X.lfc;
  const bool skip0 = !T.neg[slot];
  const int f_slices = skip0 ? 2 : 0, f_pods = skip0 ? 3 : 0;
  const TasKey none{0, 0, 0, -1};
  // ---- findLevelWithFitDomains :1200-1282 (no leaders)
  int ncur = 0, fitLevel = levelIdx;
  const int32_t sliceCount = count / sliceSize;
  for (int lv = levelIdx;; lv--) {
    TasSet S{T.level_start[lv], T.level_start[lv + 1], nullptr, 0};
    if (S.a >= S.b) { finish(KB_TAS_NO_FIT, 0); return; }
    TasKey top = X.next(S, none, 0, 0);
    if (!lfc && X.sl[top.d] >= sliceCount) top = X.best_fit(S, top, sliceCount, true);
    if (lfc) {
      TasKey c = X.next(S, none, 1, sliceCount);
      if (c.d >= 0) { if (threadIdx.x == 0) { c_d[0] = c.d; } ncur = 1; fitLevel = lv; break; }
      if (required) { finish(KB_TAS_NO_FIT, 0); return; }
    }
    if (X.sl[top.d] < sliceCount) {
      if (required) { finish(KB_TAS_NO_FIT, 0); return; }
      if (lv > 0 && !unconstrained) continue;
      int32_t remaining = sliceCount;
      TasKey cur = none;
      ncur = 0;
      while (remaining > 0) {
        TasKey d = X.next(S, cur, f_slices, 0);
        if (d.d < 0) break;
        cur = d;
        if (!lfc && X.sl[d.d] >= remaining) d = X.best_fit(S, d, remaining, true);
        if (threadIdx.x == 0 && ncur < cap) c_d[ncur] = d.d;
        ncur++;
        remaining -= X.sl[d.d];
      }
      if (remaining > 0) { finish(KB_TAS_NO_FIT, 0); return; }
      if (ncur > cap) { grow_lists(ncur); return; }
      fitLevel = lv;
      break;
    }
    if (threadIdx.x == 0) c_d[0] = top.d;
    ncur = 1; fitLevel = lv;
    break;
  }
  __syncthreads();
  // ---- updateCountsToMinimumGeneric :1361-1428 on the explicit list (slices = true)
  {
    if (threadIdx.x == 0) {
      int32_t remaining = sliceCount;
      int n = 0; bool done = false;
      for (int i = 0; i < ncur && !done; i++) {
        int d = c_d[i];
        if (!lfc && X.sl[d] >= remaining) {  // best fit over the rest of the list
          int best = d; int32_t bs = X.sl[d];
          for (int j = i; j < ncur; j++) { int32_t s2 = X.sl[c_d[j]]; if (s2 >= remaining && s2 < bs) { best = c_d[j]; bs = s2; } }
          d = best;
        }
        if (X.sl[d] >= remaining) { n_d[n] = d; n_st[n] = remaining * sliceSize; n_sl[n] = remaining; n++; done = true; break; }
        n_d[n] = d; n_st[n] = X.sl[d] * sliceSize; n_sl[n] = X.sl[d]; n++;
        remaining -= X.sl[d];
      }
      s_n = done ? n : -1;
    }
    __syncthreads();
    if (s_n < 0) { finish(KB_TAS_NO_FIT, 0); return; }
    ncur = s_n;
    int32_t *t; t = c_d; c_d = n_d; n_d = t; t = c_st; c_st = n_st; n_st = t; t = c_sl; c_sl = n_sl; n_sl = t;
  }
  // ordered greedy over a SET (children of parents) walked in sorted order; appends to the next-level list.  Entries
  // past list_cap are counted, not stored: the walk itself reads only the current list.
  auto update_set = [&](const TasSet &S, int32_t cnt, int32_t ss, bool slices, int *nn) -> bool {
    int32_t remaining = slices ? cnt / ss : cnt;
    TasKey cur = none;
    while (true) {
      TasKey d = X.next(S, cur, remaining > 0 ? (slices ? f_slices : f_pods) : 0, 0);
      if (d.d < 0) return false;
      cur = d;
      int32_t v = slices ? X.sl[d.d] : X.st[d.d];
      if (!lfc && v >= remaining) { d = X.best_fit(S, d, remaining, slices); v = slices ? X.sl[d.d] : X.st[d.d]; }
      const bool store = threadIdx.x == 0 && *nn < cap;
      if (v >= remaining) {
        if (store) { n_d[*nn] = d.d; n_st[*nn] = slices ? remaining * ss : remaining; n_sl[*nn] = slices ? remaining : X.sl[d.d]; }
        (*nn)++;
        return true;
      }
      if (store) { n_d[*nn] = d.d; n_st[*nn] = slices ? v * ss : v; n_sl[*nn] = X.sl[d.d]; }
      (*nn)++;
      remaining -= v;
    }
  };
  int lv = fitLevel;
  for (; lv < min(L - 1, sliceLevel); lv++) {  // above the slice level: all children of the chosen domains together (:901-906)
    __syncthreads();
    TasSet S{0, 0, c_d, ncur};
    int nn = 0;
    if (!update_set(S, count, sliceSize, true, &nn)) { finish(KB_TAS_NO_FIT, 0); return; }
    if (nn > cap) { grow_lists(nn); return; }
    __syncthreads();
    ncur = nn;
    int32_t *t; t = c_d; c_d = n_d; n_d = t; t = c_st; c_st = n_st; n_st = t; t = c_sl; c_sl = n_sl; n_sl = t;
  }
  for (; lv < L - 1; lv++) {  // at / below the slice level: every parent distributes its own pods (:908-941)
    __syncthreads();
    int nn = 0;
    for (int i = 0; i < ncur; i++) {
      TasSet S{0, 0, c_d + i, 1};
      if (!update_set(S, c_st[i], 1, false, &nn)) { finish(KB_TAS_NO_FIT, 0); return; }
    }
    if (nn > cap) { grow_lists(nn); return; }
    __syncthreads();
    ncur = nn;
    int32_t *t; t = c_d; c_d = n_d; n_d = t; t = c_st; c_st = n_st; n_st = t; t = c_sl; c_sl = n_sl; n_sl = t;
  }
  __syncthreads();
  // ---- buildAssignment :1455-1466: leaves in lexicographic (= index) order, zero counts dropped.  Negative counts
  // (overcommitted leaves) can make the assignment longer than the podset's count, hence than its output region.
  if (threadIdx.x == 0) { int n = 0; for (int j = 0; j < ncur; j++) if (c_st[j] != 0) n++; s_n = n; }
  __syncthreads();
  const int nout = s_n;
  const int out0 = T.tmp_start[q];
  if (nout > T.tmp_start[q + 1] - out0) {
    if (threadIdx.x == 0) { T.grow[2 + q] = nout; atomicAdd(&T.grow[1], 1); }
    finish(KB_TAS_GROW, 0);
    return;
  }
  for (int i = threadIdx.x; i < ncur; i += blockDim.x) {
    if (c_st[i] == 0) continue;
    int rank = 0;
    for (int j = 0; j < ncur; j++) if (c_st[j] != 0 && c_d[j] < c_d[i]) rank++;
    T.tmp_leaf[out0 + rank] = c_d[i] - T.leaf0; T.tmp_count[out0 + rank] = c_st[i];
  }
  // ---- addAssumedUsage :619-627 for the next podset of the chain
  const int cs = T.chain_slot[q];
  if (cs >= 0) {
    const int R = T.R;
    for (int i = threadIdx.x; i < ncur; i += blockDim.x) {
      if (c_st[i] == 0) continue;
      int lf = c_d[i] - T.leaf0;
      for (int k = 0; k < R; k++)
        if ((T.request_mask[q] >> k) & 1) T.assumed[((size_t)cs * T.n_leaves + lf) * R + k] += T.pod_request[(size_t)q * R + k] * c_st[i];
      T.assumed_mask[(size_t)cs * T.n_leaves + lf] |= T.request_mask[q];
    }
  }
  finish(KB_TAS_OK, nout);
}

__global__ void __launch_bounds__(KB_TAS_THREADS) k_tas_select(TasDev T, const int32_t *round_req, int n_round) {
  __shared__ TasKey s_red[KB_TAS_THREADS / 32];
  __shared__ TasKey s_cache[KB_TAS_THREADS * KB_TAS_LOCAL + 1];  // + the key the cache was filled from
  __shared__ int s_cmeta[8];
  __shared__ int s_n;
  for (int i = blockIdx.x; i < n_round; i += gridDim.x) {
    __syncthreads();
    tas_select_one(T, round_req[i], s_red, s_n, s_cache, s_cmeta);
  }
}

// temporary per-request regions -> CSR
__global__ void k_tas_compact(TasDev T, const int32_t *asg_start, int32_t *asg_leaf, int32_t *asg_count, int capacity) {
  int q = blockIdx.x;
  int n = T.n_out[q], src = T.tmp_start[q], dst = asg_start[q];
  for (int i = threadIdx.x; i < n; i += blockDim.x)
    if (dst + i < capacity) { asg_leaf[dst + i] = T.tmp_leaf[src + i]; asg_count[dst + i] = T.tmp_count[src + i]; }
}
