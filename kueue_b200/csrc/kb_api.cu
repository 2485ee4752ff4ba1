// kb_api.cu — C-ABI of libkueue_b200 (include/kueue_b200.h): handle, snapshot upload
// (host -> HBM, plus the static topology tables the kernels need), cycle launch,
// result download.  One handle = one CUDA device + one stream; calls are blocking and
// not re-entrant per handle (SURVEY.md §8b threading row).
#include <algorithm>
#include <cstdio>
#include <cstring>
#include <string>
#include <chrono>
#include <vector>
#include <map>
#include <mutex>

#include "kb_kernels.cuh"

#define KB_VERSION 100

namespace {

struct Arena {  // grow-only device arena, 256 B aligned sub-allocations
  char *base = nullptr;
  size_t cap = 0, used = 0;
  void reset() { used = 0; }
  bool reserve(size_t bytes) {
    if (bytes <= cap) return true;
    if (base) cudaFree(base);
    base = nullptr; cap = 0;
    size_t want = bytes + bytes / 4 + (1 << 20);
    if (cudaMalloc(&base, want) != cudaSuccess) return false;
    cap = want;
    return true;
  }
  template <typename T> T *take(size_t n) {
    size_t b = (n * sizeof(T) + 255) & ~(size_t)255;
    if (b == 0) b = 256;
    T *p = (T *)(base + used);
    used += b;
    return p;
  }
};
inline size_t pad256(size_t b) { b = (b + 255) & ~(size_t)255; return b ? b : 256; }

}  // namespace

struct kb_handle {
  int device = 0;
  int sm_count = 0;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr, ev2 = nullptr, ev3 = nullptr, ev4 = nullptr, ev5 = nullptr;
  Arena arena;   // per-cycle scratch, outputs
  Arena iarena;  // per-cycle input tables (copied before the host-side checks finish)
  char *d_out_block = nullptr;  // result tables of the cycle in the canonical layout
  int32_t *d_tgt_start = nullptr, *d_tgt_adm = nullptr; uint8_t *d_tgt_reason = nullptr;  // preemption targets, CSR by entry
  bool tgt_csr = false;
  Arena sarena;  // static tables (quotas, policies, topology): kept while kb_snapshot.static_generation is unchanged
  int64_t static_gen = 0;
  int s_dims[6] = {-1, -1, -1, -1, -1, -1};
  DevSnap D{};
  bool uploaded = false;
  bool profile = false;
  cudaEvent_t kev[KB_N_KERNELS + 1] = {};
  int kev_id[KB_N_KERNELS + 1] = {};
  int kev_n = 0;
  std::string err;
  kb_stats stats{};
  uint32_t *host_words = nullptr;  // pinned scratch words; [32..63] = copy of the cycle header
  const uint32_t *hdr_host = nullptr;  // where the last cycle's header landed (host_words or the caller's result block)
  int last_launches = 0;
  int64_t last_d2h_bytes = 0;
  // tree_eval scratch
  i64 *d_drs_rounded = nullptr; int32_t *d_drs_res = nullptr; uint8_t *d_drs_borrowing = nullptr;
  // host-side derived topology
  std::vector<int32_t> root_slot, depth, height, tree_start, tree_nodes, tree_level, lone, cq_adm_start, cq_adm, local_idx, child_start, child_list, adm_sorted, root_adm_start, adm_rank, root_cq_start;
  std::vector<uint8_t> tree_flat;
  // host copies of the static tables build_dynamic consults every cycle (the caller's static pointers are not read
  // again while static_generation is unchanged)
  std::vector<int32_t> s_parent; std::vector<uint8_t> s_within_cq, s_reclaim_within;
  std::vector<uint32_t> seen; uint32_t seen_stamp = 0;  // one-head-per-ClusterQueue check without clearing a table per cycle
  bool s_any_lone_within = false, s_preempt_policy = false;  // static: some cohort-less CQ has WithinClusterQueue != Never / some CQ has a preemption policy
  std::vector<int32_t> sn_node, slot_base, nd_tin, nd_tout, cq_path, cq_plen; int path_stride = 1;
  int max_root_adm = 1;
  int max_frl_len = 1;      // longest (root, flavor-resource) candidate bucket of this cycle
  int max_head_podsets = 1; // most podsets of one entry (bounds the columns a GetTargets search tracks)
  // launch configuration of the warp-cooperative classical search (k_search_cells / k_nominate_walk)
  int sa_wpb = 1, sa_grid = 1, sa_col_elems = 0, sa_codes = 0; size_t sa_smem = 0;
  int sb_wpb = 1, sb_grid = 1, sb_col_elems = 0; size_t sb_smem = 0;
  int sa_list_cap = 32, sb_list_cap = 32;
  // kb_run_drain: capacity reserved beyond the snapshot's admitted tables, heads chosen on the device
  size_t drain_extra_adm = 0, drain_extra_au = 0; bool drain_mode = false; bool preempt_possible = true;
  char *drain_buf = nullptr; size_t drain_buf_cap = 0; cudaEvent_t ev_d = nullptr;
  char *tas_buf = nullptr; size_t tas_buf_cap = 0;
  bool fused_on = false; size_t fused_smem = 0; bool one_head_per_cq = false; int32_t *d_cq_entry = nullptr;
  // k_cycle_flat (kb_flat.cuh): static per-tree blocks in local numbering, head records per tree node
  std::vector<unsigned char> tree_blob; std::vector<int32_t> tree_blob_off; int max_blob_bytes = 16;
  // incremental usage (kb_snapshot.usage_delta_*): the ClusterQueue usage table kept between calls
  i64 *d_usage_res = nullptr; size_t usage_res_cells = 0; bool usage_res_valid = false; int64_t usage_res_gen = 0;
  std::vector<uint32_t> delta_seen; uint32_t delta_stamp = 0;
  bool flat_on = false, flat_attr_set = false, hdr_clean = false; size_t flat_static_smem = 0; unsigned rec_stamp = 0; const void *rec_seen = nullptr; size_t rec_seen_n = 0; size_t flat_smem = 0; int flat_rcap = 1; int4 *d_cq_rec = nullptr;
  bool sg_on = false; int sg_wpb = 1, sg_grid = 1, sg_ncap = 1; size_t sg_smem = 0;  // grouped form of k_search_cells
  // device ranking of the admitted workloads (kb_rank.cuh)
  u64 *rk_keys[2] = {nullptr, nullptr}; int32_t *rk_vals[2] = {nullptr, nullptr}; void *rk_temp = nullptr; size_t rk_temp_bytes = 0;
  int search_grid = 1;
  bool search_smem = true;
  size_t search_smem_bytes = 0;
  int max_tree_nodes = 1;
  int max_root_entries_hint = 0;
};

static thread_local std::string g_err;

static int32_t fail(kb_handle *h, int32_t code, const std::string &msg) {
  if (h) h->err = msg; else g_err = msg;
  return code;
}
#define CUDA_TRY(h, expr)                                                                           \
  do {                                                                                              \
    cudaError_t _e = (expr);                                                                        \
    if (_e != cudaSuccess) return fail(h, KB_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e)); \
  } while (0)

extern "C" {

int32_t kb_version(void) { return KB_VERSION; }

const char *kb_last_error(const kb_handle *h) { return h ? h->err.c_str() : g_err.c_str(); }

// blocks handed out by kb_alloc_pinned: a span upload only ever reads inside ONE of them
static std::mutex g_pin_mu;
static std::map<uintptr_t, size_t> g_pinned;
static bool inside_one_pinned_block(uintptr_t lo, uintptr_t hi) {
  std::lock_guard<std::mutex> lk(g_pin_mu);
  auto it = g_pinned.upper_bound(lo);
  if (it == g_pinned.begin()) return false;
  --it;
  return lo >= it->first && hi <= it->first + it->second;
}

// Canonical layout of the eight per-entry / per-podset output tables: the device block of every cycle and the host
// block of kb_alloc_cycle_out use the same offsets, so those results come back with ONE device-to-host DMA.
// The block ends with the 128-byte cycle header (status word, counters), so that it too needs no copy of its own.
struct OutLayout { size_t off[8]; size_t hdr; size_t prefix; };
static OutLayout out_layout(size_t H, size_t P, size_t R) {
  const size_t sz[8] = {H, H, 4 * H, 4 * H, P * R, P * R, P * R, 4 * P};  // decision mode borrow rank flavor res_mode tried count
  OutLayout L; size_t o = 0;
  for (int i = 0; i < 8; i++) { L.off[i] = o; o += pad256(sz[i]); }
  L.hdr = o; o += 256;
  L.prefix = o;
  return L;
}
struct OutBlock { size_t H, P, R; };
static std::map<uintptr_t, OutBlock> g_out_blocks;  // base of a kb_alloc_cycle_out block -> its dimensions

int32_t kb_alloc_cycle_out(int32_t n_heads, int32_t n_podset, int32_t n_resource, int32_t tgt_capacity, int64_t n_node_cells, kb_cycle_out *out) {
  if (!out || n_heads < 0 || n_podset < 0 || n_resource < 0 || tgt_capacity < 0 || n_node_cells < 0) return KB_ERR_INVALID;
  const size_t H = (size_t)n_heads, P = (size_t)n_podset, R = (size_t)n_resource, cap = (size_t)tgt_capacity;
  OutLayout L = out_layout(H, P, R);
  size_t o_ts = L.prefix, o_ta = o_ts + pad256(4 * (H + 1)), o_tr = o_ta + pad256(4 * cap), o_nu = o_tr + pad256(cap);
  size_t total = o_nu + pad256(8 * (size_t)n_node_cells);
  void *base = nullptr;
  int32_t rc = kb_alloc_pinned(&base, total);
  if (rc != KB_OK) return rc;
  memset(base, 0, total);
  char *b = (char *)base;
  out->decision = (uint8_t *)(b + L.off[0]); out->mode = (uint8_t *)(b + L.off[1]);
  out->borrow = (int32_t *)(b + L.off[2]); out->commit_rank = (int32_t *)(b + L.off[3]);
  out->ps_flavor = (int8_t *)(b + L.off[4]); out->ps_res_mode = (int8_t *)(b + L.off[5]); out->ps_tried_idx = (int8_t *)(b + L.off[6]);
  out->ps_count = (int32_t *)(b + L.off[7]);
  out->tgt_start = (int32_t *)(b + o_ts); out->tgt_adm = (int32_t *)(b + o_ta); out->tgt_reason = (uint8_t *)(b + o_tr);
  out->tgt_capacity = tgt_capacity; out->n_targets = 0;
  out->node_usage = n_node_cells ? (int64_t *)(b + o_nu) : nullptr;
  std::lock_guard<std::mutex> lk(g_pin_mu);
  g_out_blocks[(uintptr_t)base] = OutBlock{H, P, R};
  return KB_OK;
}

int32_t kb_alloc_pinned(void **ptr, uint64_t bytes) {
  if (!ptr) return KB_ERR_INVALID;
  cudaError_t e = cudaHostAlloc(ptr, bytes ? bytes : 1, cudaHostAllocDefault);
  if (e != cudaSuccess) { g_err = cudaGetErrorString(e); return KB_ERR_CUDA; }
  std::lock_guard<std::mutex> lk(g_pin_mu);
  g_pinned[(uintptr_t)*ptr] = bytes ? bytes : 1;
  return KB_OK;
}
int32_t kb_free_pinned(void *ptr) {
  if (!ptr) return KB_OK;
  { std::lock_guard<std::mutex> lk(g_pin_mu); g_pinned.erase((uintptr_t)ptr); g_out_blocks.erase((uintptr_t)ptr); }
  return cudaFreeHost(ptr) == cudaSuccess ? KB_OK : KB_ERR_CUDA;
}

int32_t kb_create(const kb_config *cfg, kb_handle **out) {
  if (!out) return KB_ERR_INVALID;
  *out = nullptr;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail(nullptr, KB_ERR_NO_DEVICE, "no CUDA device");
  int dev = cfg ? cfg->device : 0;
  if (dev < 0 || dev >= ndev) return fail(nullptr, KB_ERR_INVALID, "bad device ordinal");
  kb_handle *h = new kb_handle();
  h->device = dev;
  if (cudaSetDevice(dev) != cudaSuccess) { delete h; return fail(nullptr, KB_ERR_CUDA, "cudaSetDevice failed"); }
  cudaDeviceGetAttribute(&h->sm_count, cudaDevAttrMultiProcessorCount, dev);
  if (cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking) != cudaSuccess) { delete h; return fail(nullptr, KB_ERR_CUDA, "stream"); }
  cudaEventCreate(&h->ev0); cudaEventCreate(&h->ev1); cudaEventCreate(&h->ev2); cudaEventCreate(&h->ev3); cudaEventCreate(&h->ev4); cudaEventCreate(&h->ev5);
  for (int i = 0; i <= KB_N_KERNELS; i++) cudaEventCreate(&h->kev[i]);
  cudaHostAlloc((void **)&h->host_words, 256, cudaHostAllocDefault);
  h->stats.sm_count = h->sm_count;
  *out = h;
  return KB_OK;
}

void kb_destroy(kb_handle *h) {
  if (!h) return;
  cudaSetDevice(h->device);
  if (h->arena.base) cudaFree(h->arena.base);
  if (h->sarena.base) cudaFree(h->sarena.base);
  if (h->iarena.base) cudaFree(h->iarena.base);
  if (h->drain_buf) cudaFree(h->drain_buf);
  if (h->d_usage_res) cudaFree(h->d_usage_res);
  if (h->tas_buf) cudaFree(h->tas_buf);
  if (h->ev_d) cudaEventDestroy(h->ev_d);
  if (h->host_words) cudaFreeHost(h->host_words);
  if (h->stream) cudaStreamDestroy(h->stream);
  if (h->ev0) cudaEventDestroy(h->ev0);
  if (h->ev1) cudaEventDestroy(h->ev1);
  if (h->ev2) cudaEventDestroy(h->ev2);
  if (h->ev3) cudaEventDestroy(h->ev3);
  if (h->ev4) cudaEventDestroy(h->ev4);
  if (h->ev5) cudaEventDestroy(h->ev5);
  for (int i = 0; i <= KB_N_KERNELS; i++) if (h->kev[i]) cudaEventDestroy(h->kev[i]);
  delete h;
}

}  // extern "C"

// ---------------------------------------------------------------------------
// validation + static topology
// ---------------------------------------------------------------------------
// static part: validation of the node tables + everything derived from the cohort forest alone
static int32_t build_static(kb_handle *h, const kb_snapshot *s) {
  int Q = s->n_cq, C = s->n_cohort, N = Q + C;
  if (Q < 0 || C < 0 || s->n_flavor < 1 || s->n_flavor > KB_MAX_FLAVORS || s->n_resource < 1 ||
      s->n_resource > KB_MAX_RESOURCES || s->n_wl < 0 || s->n_podset < 0 || s->n_adm < 0 || s->n_heads < 0)
    return fail(h, KB_ERR_INVALID, "bad dimensions");
  if (s->n_flavor > 127) return fail(h, KB_ERR_INVALID, "flavor index must fit int8");
  if (s->n_rg < 0 || s->pods_resource < -1 || s->pods_resource >= s->n_resource) return fail(h, KB_ERR_INVALID, "bad n_rg / pods_resource");
  // resource-group CSR tables (resource.go:31-38): monotone, in range, flavor indexes < F
  if (Q > 0) {
    if (s->cq_rg_start[0] != 0 || s->cq_rg_start[Q] != s->n_rg) return fail(h, KB_ERR_INVALID, "cq_rg_start must run from 0 to n_rg");
    for (int q = 0; q < Q; q++) if (s->cq_rg_start[q + 1] < s->cq_rg_start[q]) return fail(h, KB_ERR_INVALID, "cq_rg_start not monotone");
  }
  if (s->n_rg > 0) {
    if (s->rg_flavor_start[0] != 0) return fail(h, KB_ERR_INVALID, "rg_flavor_start[0] != 0");
    for (int g = 0; g < s->n_rg; g++) if (s->rg_flavor_start[g + 1] < s->rg_flavor_start[g]) return fail(h, KB_ERR_INVALID, "rg_flavor_start not monotone");
    for (int k = 0; k < s->rg_flavor_start[s->n_rg]; k++)
      if (s->rg_flavors[k] < 0 || s->rg_flavors[k] >= s->n_flavor) return fail(h, KB_ERR_INVALID, "rg_flavors out of range");
  }
  for (int n = 0; n < N; n++) {
    int p = s->parent[n];
    if (p != -1 && (p < Q || p >= N)) return fail(h, KB_ERR_INVALID, "parent must be a cohort node or -1");
  }
  h->depth.assign(N, -1);
  h->root_slot.assign(N, -1);
  std::vector<int32_t> root(N, -1);
  for (int n = 0; n < N; n++) {  // depth + root with cycle detection (hierarchy/cycle.go:31-44)
    int steps = 0, t = n;
    while (s->parent[t] >= 0) {
      t = s->parent[t];
      if (++steps > KB_MAX_DEPTH) return fail(h, KB_ERR_INVALID, "cohort tree deeper than KB_MAX_DEPTH or cyclic");
    }
    h->depth[n] = steps;
    root[n] = t;
  }
  // roots: every parentless node; slots in ascending node order
  int nroots = 0;
  std::vector<int32_t> slot_of_root(N, -1);
  for (int n = 0; n < N; n++) if (s->parent[n] < 0) slot_of_root[n] = nroots++;
  for (int n = 0; n < N; n++) h->root_slot[n] = slot_of_root[root[n]];
  // children counts -> height (getNodeHeight hierarchical_preemption.go:202-208)
  std::vector<int32_t> nchild(N, 0);
  for (int n = 0; n < N; n++) if (s->parent[n] >= 0) nchild[s->parent[n]]++;
  h->height.assign(N, 0);
  for (int n = Q; n < N; n++) h->height[n] = std::min(nchild[n], 1);
  {  // process cohorts by depth descending so children are final before parents
    std::vector<int32_t> order;
    for (int n = Q; n < N; n++) order.push_back(n);
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return h->depth[a] > h->depth[b]; });
    for (int n : order) {
      int p = s->parent[n];
      if (p >= 0) h->height[p] = std::max(h->height[p], h->height[n] + 1);
    }
  }
  // cohort-rooted trees: nodes grouped by root, ordered by depth ascending
  std::vector<int32_t> tree_of_root(N, -1);
  int ntrees = 0;
  for (int n = Q; n < N; n++) if (s->parent[n] < 0) tree_of_root[n] = ntrees++;
  std::vector<int32_t> cnt(ntrees + 1, 0);
  h->lone.clear();
  for (int n = 0; n < N; n++) {
    int t = tree_of_root[root[n]];
    if (t >= 0) cnt[t + 1]++;
    else h->lone.push_back(n);  // parentless CQ
  }
  for (int t = 0; t < ntrees; t++) cnt[t + 1] += cnt[t];
  h->tree_start.assign(cnt.begin(), cnt.end());
  h->tree_nodes.assign(cnt[ntrees], 0);
  h->tree_level.assign((size_t)ntrees * KB_LEVELS, 0);
  {
    // counting sort by (tree, depth)
    std::vector<int32_t> lvlcnt((size_t)ntrees * KB_LEVELS, 0);
    for (int n = 0; n < N; n++) { int t = tree_of_root[root[n]]; if (t >= 0) lvlcnt[(size_t)t * KB_LEVELS + h->depth[n] + 1]++; }
    for (int t = 0; t < ntrees; t++)
      for (int l = 0; l + 1 < KB_LEVELS; l++) lvlcnt[(size_t)t * KB_LEVELS + l + 1] += lvlcnt[(size_t)t * KB_LEVELS + l];
    h->tree_level = lvlcnt;
    std::vector<int32_t> cur = lvlcnt;
    for (int n = 0; n < N; n++) {
      int t = tree_of_root[root[n]];
      if (t < 0) continue;
      int pos = cur[(size_t)t * KB_LEVELS + h->depth[n]]++;
      h->tree_nodes[h->tree_start[t] + pos] = n;
    }
  }
  // children CSR (cohort children first: their node ids are >= Q, so sort descending by class)
  h->child_start.assign(N + 1, 0);
  for (int n = 0; n < N; n++) if (s->parent[n] >= 0) h->child_start[s->parent[n] + 1]++;
  for (int n = 0; n < N; n++) h->child_start[n + 1] += h->child_start[n];
  h->child_list.assign(std::max(1, h->child_start[N]), 0);
  {
    std::vector<int32_t> cur(h->child_start.begin(), h->child_start.end() - 1);
    for (int n = Q; n < N; n++) if (s->parent[n] >= 0) h->child_list[cur[s->parent[n]]++] = n;  // cohorts ascending
    for (int n = 0; n < Q; n++) if (s->parent[n] >= 0) h->child_list[cur[s->parent[n]]++] = n;  // then CQs ascending
  }
  h->tree_flat.assign(std::max(1, ntrees), 1);
  for (int n = 0; n < Q; n++) { int t = tree_of_root[root[n]]; if (t >= 0 && h->depth[n] != 1) h->tree_flat[t] = 0; }
  h->local_idx.assign(N, 0);
  h->max_tree_nodes = 1;
  for (int t = 0; t < ntrees; t++) {
    int nn = h->tree_start[t + 1] - h->tree_start[t];
    h->max_tree_nodes = std::max(h->max_tree_nodes, nn);
    for (int i = 0; i < nn; i++) h->local_idx[h->tree_nodes[h->tree_start[t] + i]] = i;
  }
  h->root_cq_start.assign(nroots + 1, 0);
  for (int q = 0; q < Q; q++) h->root_cq_start[h->root_slot[q] + 1]++;
  for (int r = 0; r < nroots; r++) h->root_cq_start[r + 1] += h->root_cq_start[r];
  h->D.nTrees = ntrees;
  h->D.nLone = (int)h->lone.size();
  h->D.nRoots = nroots;
  {  // static ClusterQueue -> root paths (global-table admit loop)
    int maxd = 0;
    for (int q = 0; q < Q; q++) maxd = std::max(maxd, h->depth[q]);
    h->path_stride = maxd + 1;
    h->cq_path.assign((size_t)std::max(1, Q) * h->path_stride, -1); h->cq_plen.assign(std::max(1, Q), 1);
    for (int q = 0; q < Q; q++) { int k = 0; for (int t = q; t >= 0; t = s->parent[t]) h->cq_path[(size_t)q * h->path_stride + k++] = t; h->cq_plen[q] = k; }
  }
  h->s_parent.assign(s->parent, s->parent + N);
  h->s_within_cq.assign(s->cq_within_cq, s->cq_within_cq + Q);
  h->s_reclaim_within.assign(s->cq_reclaim_within, s->cq_reclaim_within + Q);
  h->s_any_lone_within = false; h->s_preempt_policy = false;
  for (int q = 0; q < Q; q++) {
    if (s->parent[q] < 0 && s->cq_within_cq[q] != KB_POLICY_NEVER) h->s_any_lone_within = true;
    if (s->cq_within_cq[q] != KB_POLICY_NEVER || (s->parent[q] >= 0 && s->cq_reclaim_within[q] != KB_POLICY_NEVER)) h->s_preempt_policy = true;
  }
  {  // slot-node numbering (cohort-less ClusterQueues, then the trees) and Euler-tour intervals inside every tree
    int nl = (int)h->lone.size();
    h->sn_node.assign(std::max(1, N), 0); h->nd_tin.assign(std::max(1, N), 0); h->nd_tout.assign(std::max(1, N), 1);
    h->slot_base.assign(nroots + 1, 0);
    for (int i = 0; i < nl; i++) { h->sn_node[i] = h->lone[i]; h->slot_base[i] = i; }
    for (int t = 0; t < ntrees; t++) h->slot_base[nl + t] = nl + h->tree_start[t];
    h->slot_base[nroots] = N;
    for (size_t i = 0; i < h->tree_nodes.size(); i++) h->sn_node[nl + i] = h->tree_nodes[i];
    std::vector<int32_t> stack, it;
    for (int t = 0; t < ntrees; t++) {
      int base = nl + h->tree_start[t];
      int rootn = h->tree_nodes[h->tree_start[t]];
      int clock = 0;
      stack.assign(1, rootn); it.assign(1, h->child_start[rootn]);
      h->nd_tin[base + h->local_idx[rootn]] = clock++;
      while (!stack.empty()) {
        int n = stack.back();
        if (it.back() < h->child_start[n + 1]) {
          int c = h->child_list[it.back()++];
          h->nd_tin[base + h->local_idx[c]] = clock++;
          stack.push_back(c); it.push_back(h->child_start[c]);
        } else {
          h->nd_tout[base + h->local_idx[n]] = clock;
          stack.pop_back(); it.pop_back();
        }
      }
    }
  }
  {  // static per-tree blocks in local numbering (TreeBlobHdr, kb_flat.cuh)
    h->tree_blob.clear(); h->tree_blob_off.assign(ntrees + 1, 0); h->max_blob_bytes = 16;
    for (int t = 0; t < ntrees; t++) {
      const int nn = h->tree_start[t + 1] - h->tree_start[t];
      const int32_t *nodes = h->tree_nodes.data() + h->tree_start[t];
      int nrg = 0, nfl = 0;
      for (int i = 0; i < nn; i++) if (nodes[i] < Q) for (int g = s->cq_rg_start[nodes[i]]; g < s->cq_rg_start[nodes[i] + 1]; g++) { nrg++; nfl += s->rg_flavor_start[g + 1] - s->rg_flavor_start[g]; }
      TreeBlobHdr H{};
      size_t o = sizeof(TreeBlobHdr);
      auto take = [&](size_t bytes) { o = (o + 15) & ~(size_t)15; size_t at = o; o += bytes; return (int32_t)at; };
      H.nn = nn; H.nrg = nrg; H.nfl = nfl;
      H.gid = take((size_t)nn * 4); H.par = take((size_t)nn * 4); H.hgt = take((size_t)nn * 4); H.rgs = take((size_t)(nn + 1) * 4);
      H.gen = take((size_t)nn * 8); H.wgt = take((size_t)nn * 8);
      H.within = take(nn); H.reclaim = take(nn); H.borrow_w = take(nn); H.wcb = take(nn); H.wcp = take(nn); H.pref = take(nn);
      H.rgmask = take((size_t)nrg * 4); H.rgfl = take((size_t)(nrg + 1) * 4); H.fl = take((size_t)nfl * 4);
      o = (o + 15) & ~(size_t)15;
      H.bytes = (int32_t)o;
      size_t base = h->tree_blob.size();
      if (base + o >= (size_t)INT32_MAX) return fail(h, KB_ERR_INVALID, "static tree tables exceed 2 GiB");
      h->tree_blob.resize(base + o, 0);
      unsigned char *b = h->tree_blob.data() + base;
      memcpy(b, &H, sizeof(H));
      int32_t *gid = (int32_t *)(b + H.gid), *par = (int32_t *)(b + H.par), *hgt = (int32_t *)(b + H.hgt), *rgs = (int32_t *)(b + H.rgs);
      i64 *gen = (i64 *)(b + H.gen); double *wgt = (double *)(b + H.wgt);
      uint32_t *rgmask = (uint32_t *)(b + H.rgmask); int32_t *rgfl = (int32_t *)(b + H.rgfl), *fl = (int32_t *)(b + H.fl);
      int lg = 0, lf = 0;
      for (int i = 0; i < nn; i++) {
        const int nd = nodes[i];
        gid[i] = nd; par[i] = s->parent[nd] < 0 ? -1 : h->local_idx[s->parent[nd]]; hgt[i] = h->height[nd]; rgs[i] = lg;
        wgt[i] = s->fair_weight[nd];
        if (nd >= Q) continue;
        gen[i] = s->cq_generation[nd];
        b[H.within + i] = s->cq_within_cq[nd]; b[H.reclaim + i] = s->cq_reclaim_within[nd]; b[H.borrow_w + i] = s->cq_borrow_within[nd];
        b[H.wcb + i] = s->cq_when_can_borrow[nd]; b[H.wcp + i] = s->cq_when_can_preempt[nd]; b[H.pref + i] = s->cq_preference[nd];
        for (int g = s->cq_rg_start[nd]; g < s->cq_rg_start[nd + 1]; g++) {
          rgmask[lg] = s->rg_res_mask[g]; rgfl[lg] = lf;
          for (int k = s->rg_flavor_start[g]; k < s->rg_flavor_start[g + 1]; k++) fl[lf++] = s->rg_flavors[k];
          lg++;
        }
      }
      rgs[nn] = lg; rgfl[lg] = lf;
      h->tree_blob_off[t + 1] = (int32_t)(base + o);
      h->max_blob_bytes = std::max(h->max_blob_bytes, (int)o);
    }
    if (h->tree_blob.empty()) h->tree_blob.resize(16, 0);
  }
  return KB_OK;
}

// per-cycle part: admitted workloads (grouping, candidate pre-order) and bounds checks of the entry tables
static int32_t build_dynamic(kb_handle *h, const kb_snapshot *s) {
  int Q = s->n_cq;
  int nroots = h->D.nRoots;
  if (s->n_wl < 0 || s->n_podset < 0 || s->n_adm < 0 || s->n_heads < 0) return fail(h, KB_ERR_INVALID, "bad dimensions");
  // admitted workloads grouped by CQ (ClusterQueueSnapshot.Workloads)
  h->cq_adm_start.assign(Q + 1, 0);
  for (int a = 0; a < s->n_adm; a++) {
    int c = s->adm_cq[a];
    if (c < 0 || c >= Q) return fail(h, KB_ERR_INVALID, "adm_cq out of range");
    h->cq_adm_start[c + 1]++;
  }
  for (int q = 0; q < Q; q++) h->cq_adm_start[q + 1] += h->cq_adm_start[q];
  // admitted workloads per root: only the counts are needed on the host (scratch sizing); the ranking by the
  // preemptor-independent part of CandidatesOrdering runs on the device every cycle (kb_rank.cuh)
  h->root_adm_start.assign(nroots + 1, 0);
  for (int a = 0; a < s->n_adm; a++) h->root_adm_start[h->root_slot[s->adm_cq[a]] + 1]++;
  h->max_root_adm = 1;
  for (int r = 0; r < nroots; r++) { h->max_root_adm = std::max(h->max_root_adm, h->root_adm_start[r + 1]); h->root_adm_start[r + 1] += h->root_adm_start[r]; }
  h->max_root_adm += (int)h->drain_extra_adm;  // a drain may admit everything into one root
  if (h->max_root_adm >= (1 << 28)) return fail(h, KB_ERR_INVALID, "more than 2^28 admitted workloads under one root");
  {  // longest (root, flavor-resource) bucket: sizes the per-warp candidate-code scratch of the single-cell searches
    int FRn = s->n_flavor * s->n_resource;
    std::vector<int32_t> cnt((size_t)nroots * FRn + 1, 0);
    for (int a = 0; a < s->n_adm; a++) {
      if (s->adm_use_start[a + 1] < s->adm_use_start[a]) return fail(h, KB_ERR_INVALID, "adm_use_start not monotone");
      size_t b = (size_t)h->root_slot[s->adm_cq[a]] * FRn;
      for (int k = s->adm_use_start[a]; k < s->adm_use_start[a + 1]; k++) {
        int fr = s->adm_use_fr[k];
        if (fr < 0 || fr >= FRn) return fail(h, KB_ERR_INVALID, "adm_use_fr out of range");
        cnt[b + fr]++;
      }
    }
    h->max_frl_len = 1;
    for (int32_t c : cnt) h->max_frl_len = std::max(h->max_frl_len, c);
    h->max_frl_len += (int)h->drain_extra_adm;
    h->max_head_podsets = 1;
    if (h->drain_mode) for (int w = 0; w < s->n_wl; w++) h->max_head_podsets = std::max(h->max_head_podsets, s->wl_ps_start[w + 1] - s->wl_ps_start[w]);
  }
  // light bounds checks on the hot tables
  for (int w = 0; w < s->n_wl; w++) {
    if (s->wl_cq[w] < 0 || s->wl_cq[w] >= Q) return fail(h, KB_ERR_INVALID, "wl_cq out of range");
    if (s->wl_ps_start[w + 1] < s->wl_ps_start[w]) return fail(h, KB_ERR_INVALID, "wl_ps_start not monotone");
  }
  if (s->n_wl && (s->wl_ps_start[0] != 0 || s->wl_ps_start[s->n_wl] != s->n_podset)) return fail(h, KB_ERR_INVALID, "wl_ps_start must run from 0 to n_podset");
  // heads: range, most podsets of one entry, one head per ClusterQueue? (fairSharingIterator keeps one entry per CQ,
  // fair_sharing_iterator.go:52-54) — one pass
  h->one_head_per_cq = true;
  if (!h->drain_mode) {
    h->seen_stamp++;
    if ((int)h->seen.size() < Q || h->seen_stamp == 0) { h->seen.assign((size_t)std::max(1, Q), 0); h->seen_stamp = 1; }
    const uint32_t stamp = h->seen_stamp;
    int maxps = 1; bool dup = false;
    for (int i = 0; i < s->n_heads; i++) {
      const int w = s->heads[i];
      if (w < 0 || w >= s->n_wl) return fail(h, KB_ERR_INVALID, "heads out of range");
      maxps = std::max(maxps, s->wl_ps_start[w + 1] - s->wl_ps_start[w]);
      const int c = s->wl_cq[w];
      if (h->seen[c] == stamp) dup = true;
      h->seen[c] = stamp;
    }
    h->max_head_podsets = std::max(h->max_head_podsets, maxps);
    if (dup) {
      if (s->flags & KB_F_FAIR_SHARING) return fail(h, KB_ERR_INVALID, "fair sharing: more than one head for a ClusterQueue");
      h->one_head_per_cq = false;
    }
  }
  if (s->n_adm_use < 0 || (s->n_adm && (s->adm_use_start[0] != 0 || s->adm_use_start[s->n_adm] != s->n_adm_use)))
    return fail(h, KB_ERR_INVALID, "adm_use_start must run from 0 to n_adm_use");
  {  // ps_last_tried >= -1 (int8): eight at a time — a byte below -1 has its top bit set and is not 0xff
    const size_t nb = (size_t)s->n_podset * s->n_resource;
    const int8_t *lt = s->ps_last_tried;
    size_t i = 0;
    bool bad = false;
    for (; i + 8 <= nb; i += 8) {
      uint64_t v; memcpy(&v, lt + i, 8);
      const uint64_t top = v & 0x8080808080808080ull;         // bytes that are negative
      if (top) { for (int k = 0; k < 8; k++) if (lt[i + k] < -1) bad = true; }
    }
    for (; i < nb; i++) if (lt[i] < -1) bad = true;
    if (bad) return fail(h, KB_ERR_INVALID, "ps_last_tried below -1");
  }
  if (s->ps_group)  // the podsets of one PodSetGroup are adjacent rows of their workload
    for (int w = 0; w < s->n_wl; w++)
      for (int a = s->wl_ps_start[w]; a < s->wl_ps_start[w + 1]; a++) {
        int g = s->ps_group[a];
        if (g < 0 || (a > s->wl_ps_start[w] && s->ps_group[a - 1] == g)) continue;
        int b = a + 1;
        while (b < s->wl_ps_start[w + 1] && s->ps_group[b] == g) b++;
        for (int c = b; c < s->wl_ps_start[w + 1]; c++)
          if (s->ps_group[c] == g) return fail(h, KB_ERR_INVALID, "ps_group: podsets of one group must be adjacent");
      }
  // warp-per-root admit for cohort-less CQs: only when none of them can ever get preemption targets
  {
    bool any = false;
    if (h->s_any_lone_within) {
      for (int q = 0; q < Q && !any; q++)
        if (h->s_parent[q] < 0 && h->s_within_cq[q] != KB_POLICY_NEVER && h->cq_adm_start[q + 1] > h->cq_adm_start[q]) any = true;
      if (h->drain_mode) any = true;  // admitted workloads appear during the drain
    }
    h->D.lone_fast = !any && s->n_flavor * s->n_resource <= 64;
    // can any ClusterQueue ever have preemption candidates?  (candidates_possible, kb_kernels.cuh)
    h->preempt_possible = h->s_preempt_policy;
  }
  return KB_OK;
}

// next stamp of the head records (kb_flat.cuh); the table is cleared when it moved, grew or the 16-bit stamp wrapped
static int32_t flat_rec_stamp(kb_handle *h) {
  const size_t n = h->tree_nodes.size() + 1;
  if (h->rec_seen != (const void *)h->d_cq_rec || h->rec_seen_n != n || h->rec_stamp >= 0xffffu) {
    CUDA_TRY(h, cudaMemsetAsync(h->d_cq_rec, 0, sizeof(int4) * n, h->stream));
    h->rec_seen = h->d_cq_rec; h->rec_seen_n = n; h->rec_stamp = 0;
  }
  h->D.rec_stamp = ++h->rec_stamp;
  return KB_OK;
}

// rows of the resident usage table replaced by the caller's deltas (kb_snapshot.usage_delta_*)
__global__ void k_usage_patch(i64 *usage, const int32_t *cq, const i64 *rows, int n, int FR) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n * FR) return;
  usage[(size_t)cq[i / FR] * FR + i % FR] = rows[i];
}

template <typename T>
static cudaError_t up(kb_handle *h, Arena &arena, const T *&dst, const T *src, size_t n, int64_t *bytes) {
  T *d = arena.take<T>(n);
  dst = d;
  if (n == 0) return cudaSuccess;
  *bytes += (int64_t)(n * sizeof(T));
  return cudaMemcpyAsync(d, src, n * sizeof(T), cudaMemcpyHostToDevice, h->stream);
}

static int32_t upload_impl(kb_handle *h, const kb_snapshot *s, bool sync) {
  if (!h || !s) return KB_ERR_INVALID;
  cudaSetDevice(h->device);
  h->uploaded = false;
  DevSnap &D = h->D;
  int Q = s->n_cq, C = s->n_cohort, N = Q + C, F = s->n_flavor, R = s->n_resource, FR = F * R;
  // A / AU are CAPACITIES (kb_run_drain grows the admitted tables on the device); A_in / AU_in what the caller passed
  const size_t A_in = (size_t)s->n_adm, AU_in = (size_t)s->n_adm_use;
  size_t NF = (size_t)N * FR, P = (size_t)s->n_podset, W = (size_t)s->n_wl, A = A_in + h->drain_extra_adm, H = (size_t)s->n_heads;
  const size_t AUc = AU_in + h->drain_extra_au;
  int n_rg_fl = (s->n_rg > 0 && s->rg_flavor_start) ? s->rg_flavor_start[s->n_rg] : 0;
  int dims[6] = {Q, C, F, R, s->n_rg, n_rg_fl};
  bool reuse = s->static_generation != 0 && s->static_generation == h->static_gen && memcmp(dims, h->s_dims, sizeof(dims)) == 0;
  int64_t bytes = 0;
  int32_t rc;
  if (!reuse) {
    h->static_gen = 0;
    rc = build_static(h, s);
    if (rc != KB_OK) return rc;
    size_t stot = 0;
    auto sneed = [&](size_t n, size_t sz) { stot += pad256(n * sz); };
    sneed(N, 4); sneed(N, 8); sneed(NF, 8); sneed(NF, 8); sneed(NF, 8);
    for (int k = 0; k < 4; k++) sneed(Q, 1);
    sneed(Q, 4); for (int k = 0; k < 4; k++) sneed(Q, 1); sneed(Q, 8);
    sneed(Q + 1, 4); sneed(s->n_rg, 4); sneed(s->n_rg + 1, 4); sneed(n_rg_fl, 4);
    sneed(N, 4); sneed(N, 4); sneed(N, 4); sneed(D.nTrees + 1, 4); sneed(h->tree_nodes.size(), 4); sneed(h->tree_level.size(), 4);
    sneed(h->lone.size(), 4); sneed(N, 4); sneed(h->tree_flat.size(), 1); sneed(N + 1, 4); sneed(h->child_list.size(), 4); sneed(h->root_cq_start.size(), 4);
    sneed(h->sn_node.size(), 4); sneed(h->slot_base.size(), 4); sneed(h->nd_tin.size(), 4); sneed(h->nd_tout.size(), 4);
    sneed(h->cq_path.size(), 4); sneed(h->cq_plen.size(), 4);
    sneed(h->tree_blob.size(), 1); sneed(h->tree_blob_off.size(), 4);
    const size_t tl_cells = h->tree_nodes.size() * (size_t)FR;
    sneed(tl_cells, 8); sneed(tl_cells, 8); sneed(tl_cells, 8);
    if (!h->sarena.reserve(stot + 4096)) return fail(h, KB_ERR_CUDA, "cudaMalloc failed");
    h->sarena.reset();
#define SUP(field, src, n) CUDA_TRY(h, up(h, h->sarena, D.field, src, (size_t)(n), &bytes))
    SUP(parent, s->parent, N); SUP(fair_weight, s->fair_weight, N);
    SUP(nominal, (const i64 *)s->nominal, NF); SUP(blimit, (const i64 *)s->borrow_limit, NF); SUP(llimit, (const i64 *)s->lend_limit, NF);
    SUP(cq_within_cq, s->cq_within_cq, Q); SUP(cq_reclaim_within, s->cq_reclaim_within, Q); SUP(cq_borrow_within, s->cq_borrow_within, Q);
    SUP(cq_has_bwc_threshold, s->cq_has_bwc_threshold, Q); SUP(cq_bwc_threshold, s->cq_bwc_threshold, Q);
    SUP(cq_when_can_borrow, s->cq_when_can_borrow, Q); SUP(cq_when_can_preempt, s->cq_when_can_preempt, Q);
    SUP(cq_preference, s->cq_preference, Q); SUP(cq_strategy, s->cq_strategy, Q); SUP(cq_generation, (const i64 *)s->cq_generation, Q);
    SUP(cq_rg_start, s->cq_rg_start, Q + 1); SUP(rg_res_mask, s->rg_res_mask, s->n_rg); SUP(rg_flavor_start, s->rg_flavor_start, s->n_rg + 1);
    SUP(rg_flavors, s->rg_flavors, n_rg_fl);
    SUP(root_slot, h->root_slot.data(), N); SUP(depth, h->depth.data(), N); SUP(height, h->height.data(), N);
    SUP(tree_start, h->tree_start.data(), D.nTrees + 1); SUP(tree_nodes, h->tree_nodes.data(), h->tree_nodes.size());
    SUP(tree_level, h->tree_level.data(), h->tree_level.size()); SUP(lone_cqs, h->lone.data(), h->lone.size());
    SUP(local_idx, h->local_idx.data(), N);
    SUP(tree_flat, h->tree_flat.data(), h->tree_flat.size());
    SUP(child_start, h->child_start.data(), N + 1); SUP(child_list, h->child_list.data(), h->child_list.size());
    SUP(root_cq_start, h->root_cq_start.data(), h->root_cq_start.size());
    SUP(sn_node, h->sn_node.data(), h->sn_node.size()); SUP(slot_base, h->slot_base.data(), h->slot_base.size());
    SUP(nd_tin, h->nd_tin.data(), h->nd_tin.size()); SUP(nd_tout, h->nd_tout.data(), h->nd_tout.size());
    SUP(cq_path, h->cq_path.data(), h->cq_path.size()); SUP(cq_plen, h->cq_plen.data(), h->cq_plen.size());
    SUP(tree_blob, h->tree_blob.data(), h->tree_blob.size()); SUP(tree_blob_off, h->tree_blob_off.data(), h->tree_blob_off.size());
    D.tl_nominal = D.tl_blimit = D.tl_llimit = nullptr; D.tl_usage = nullptr;
    if (tl_cells && tl_cells < (size_t)INT32_MAX) {  // quota tables in tree-local row order (k_cycle_flat's bulk staging)
      i64 *tn = h->sarena.take<i64>(tl_cells), *tb_ = h->sarena.take<i64>(tl_cells), *tl_ = h->sarena.take<i64>(tl_cells);
      D.FR = FR; D.Q = Q;
      k_tl_static<<<(unsigned)((tl_cells + 255) / 256), 256, 0, h->stream>>>(D, tn, tb_, tl_, (int)tl_cells);
      D.tl_nominal = tn; D.tl_blimit = tb_; D.tl_llimit = tl_;
    }
    D.path_stride = h->path_stride;
#undef SUP
    memcpy(h->s_dims, dims, sizeof(dims));
    h->static_gen = s->static_generation;
  }
  // Per-cycle input tables, enqueued FIRST: the DMA runs while the host validates the tables and sizes the scratch
  // arena below (build_dynamic).  The caller's tables (dynamic part of kb_snapshot) usually sit close together in
  // one pinned block (kb_alloc_pinned carved by the shim): when their host span is not much larger than their
  // total size the whole span goes to the device with ONE DMA and the device tables alias into it at the same
  // offsets; otherwise every table is copied on its own.
  struct Tab { const void *src; size_t bytes; const void **dst; size_t cap; };
  std::vector<Tab> tabs;
#define UPC(field, src, n, capn) tabs.push_back(Tab{(const void *)(src), (size_t)(n) * sizeof(*D.field), (const void **)&D.field, (size_t)(capn) * sizeof(*D.field)})
#define UP(field, src, n) UPC(field, src, n, n)
  // ClusterQueue usage: the full table with the other per-cycle tables | into the resident buffer (KB_F_USAGE_RESIDENT)
  // | the resident buffer patched with the caller's rows (usage_delta_*)
  const bool delta = s->usage_delta_cq != nullptr;
  const bool keep_usage = (s->flags & KB_F_USAGE_RESIDENT) != 0 && !h->drain_mode;
  const int32_t *d_delta_cq = nullptr; const i64 *d_delta_rows = nullptr;
  if (delta) {
    if (h->drain_mode) return fail(h, KB_ERR_INVALID, "usage deltas are not available for kb_run_drain");
    if (!reuse || !h->usage_res_valid || h->usage_res_gen != s->static_generation || h->usage_res_cells != (size_t)Q * FR)
      return fail(h, KB_ERR_INVALID, "usage_delta_*: no resident usage table of this static_generation (pass cq_usage with KB_F_USAGE_RESIDENT first)");
    if (s->n_usage_delta < 0 || (s->n_usage_delta > 0 && !s->usage_delta_rows)) return fail(h, KB_ERR_INVALID, "usage_delta_*: bad count / null rows");
    h->delta_stamp++;
    if ((int)h->delta_seen.size() < Q || h->delta_stamp == 0) { h->delta_seen.assign((size_t)std::max(1, Q), 0); h->delta_stamp = 1; }
    for (int i = 0; i < s->n_usage_delta; i++) {
      const int c = s->usage_delta_cq[i];
      if (c < 0 || c >= Q) return fail(h, KB_ERR_INVALID, "usage_delta_cq out of range");
      if (h->delta_seen[c] == h->delta_stamp) return fail(h, KB_ERR_INVALID, "usage_delta_cq lists a ClusterQueue twice");
      h->delta_seen[c] = h->delta_stamp;
    }
    tabs.push_back(Tab{(const void *)s->usage_delta_cq, (size_t)s->n_usage_delta * 4, (const void **)&d_delta_cq, (size_t)s->n_usage_delta * 4});
    tabs.push_back(Tab{(const void *)s->usage_delta_rows, (size_t)s->n_usage_delta * FR * 8, (const void **)&d_delta_rows, (size_t)s->n_usage_delta * FR * 8});
  } else if (keep_usage) {
    if (h->usage_res_cells != (size_t)Q * FR || !h->d_usage_res) {
      if (h->d_usage_res) cudaFree(h->d_usage_res);
      h->d_usage_res = nullptr; h->usage_res_cells = 0;
      if (cudaMalloc((void **)&h->d_usage_res, std::max<size_t>(8, (size_t)Q * FR * 8)) != cudaSuccess) { cudaStreamSynchronize(h->stream); return fail(h, KB_ERR_CUDA, "cudaMalloc failed"); }
      h->usage_res_cells = (size_t)Q * FR;
    }
  } else {
    UP(cq_usage, (const i64 *)s->cq_usage, (size_t)Q * FR);
  }
  if (!delta) h->usage_res_valid = false;  // a full table supersedes whatever was resident
  UP(wl_cq, s->wl_cq, W); UP(wl_priority, s->wl_priority, W); UP(wl_ts, (const i64 *)s->wl_ts, W); UP(wl_uid, (const i64 *)s->wl_uid, W);
  UP(wl_last_gen, (const i64 *)s->wl_last_gen, W); UP(wl_ps_start, s->wl_ps_start, W + 1);
  UP(ps_req, (const i64 *)s->ps_req, P * R); UP(ps_req_mask, s->ps_req_mask, P); UP(ps_count, s->ps_count, P);
  UP(ps_min_count, s->ps_min_count, P); UP(ps_flavor_ok, (const u64 *)s->ps_flavor_ok, P); UP(ps_last_tried, s->ps_last_tried, P * R);
  UPC(adm_cq, s->adm_cq, A_in, A); UPC(adm_priority, s->adm_priority, A_in, A); UPC(adm_ts, (const i64 *)s->adm_ts, A_in, A);
  UPC(adm_qr_ts, (const i64 *)s->adm_qr_ts, A_in, A); UPC(adm_uid, (const i64 *)s->adm_uid, A_in, A); UPC(adm_evicted, s->adm_evicted, A_in, A);
  UPC(adm_use_start, s->adm_use_start, A_in + 1, A + 1); UPC(adm_use_fr, s->adm_use_fr, AU_in, AUc); UPC(adm_use_qty, (const i64 *)s->adm_use_qty, AU_in, AUc);
  if (!h->drain_mode) UP(heads, s->heads, H);
  D.wl_has_qr = nullptr; D.wl_sched_hash = nullptr; D.ps_group = nullptr;
  if (s->ps_group) UP(ps_group, s->ps_group, P);
  if (s->wl_has_quota_reservation) UP(wl_has_qr, s->wl_has_quota_reservation, W);
  if (s->wl_sched_hash) UP(wl_sched_hash, (const i64 *)s->wl_sched_hash, W);
  size_t caller_tabs = tabs.size();
#undef UP
#undef UPC
  {
    uintptr_t lo = UINTPTR_MAX, hi = 0; size_t sum = 0;
    for (size_t i = 0; i < caller_tabs; i++) {
      if (!tabs[i].bytes) continue;
      if (!tabs[i].src) return fail(h, KB_ERR_INVALID, "null table with non-zero length");
      if (tabs[i].cap != tabs[i].bytes) continue;  // growable table: its own allocation
      lo = std::min(lo, (uintptr_t)tabs[i].src); hi = std::max(hi, (uintptr_t)tabs[i].src + tabs[i].bytes); sum += tabs[i].bytes;
    }
    uintptr_t lo_al = lo & ~(uintptr_t)255;
    bool span = sum > 0 && (hi - lo) <= sum + sum / 4 + (64u << 10) && inside_one_pinned_block(lo_al, hi);
    size_t itot = span ? pad256(hi - lo_al) : 0;
    for (size_t i = 0; i < tabs.size(); i++) {
      const Tab &t = tabs[i];
      if (!(span && i < caller_tabs && t.bytes && t.cap == t.bytes)) itot += pad256(std::max(t.bytes, t.cap));
    }
    if (!h->iarena.reserve(itot + 4096)) return fail(h, KB_ERR_CUDA, "cudaMalloc failed");
    h->iarena.reset();
    CUDA_TRY(h, cudaEventRecord(h->ev0, h->stream));
    char *dspan = span ? h->iarena.take<char>(hi - lo_al) : nullptr;
    if (span) {
      CUDA_TRY(h, cudaMemcpyAsync(dspan, (const void *)lo_al, hi - lo_al, cudaMemcpyHostToDevice, h->stream));
      bytes += (int64_t)(hi - lo_al);
    }
    for (size_t i = 0; i < tabs.size(); i++) {
      const Tab &t = tabs[i];
      if (span && i < caller_tabs && t.bytes && t.cap == t.bytes) { *t.dst = dspan + ((uintptr_t)t.src - lo_al); continue; }
      char *d = h->iarena.take<char>(std::max(t.bytes, t.cap));
      *t.dst = d;
      if (t.bytes) { CUDA_TRY(h, cudaMemcpyAsync(d, t.src, t.bytes, cudaMemcpyHostToDevice, h->stream)); bytes += (int64_t)t.bytes; }
    }
  }
  if (delta) {
    D.cq_usage = h->d_usage_res;
    const int nd = s->n_usage_delta;
    if (nd > 0) k_usage_patch<<<(unsigned)(((size_t)nd * FR + 255) / 256), 256, 0, h->stream>>>(h->d_usage_res, d_delta_cq, d_delta_rows, nd, FR);
  } else if (keep_usage) {
    if ((size_t)Q * FR) {
      if (!s->cq_usage) { cudaStreamSynchronize(h->stream); return fail(h, KB_ERR_INVALID, "null table with non-zero length"); }
      CUDA_TRY(h, cudaMemcpyAsync(h->d_usage_res, s->cq_usage, (size_t)Q * FR * 8, cudaMemcpyHostToDevice, h->stream));
      bytes += (int64_t)Q * FR * 8;
    }
    D.cq_usage = h->d_usage_res;
    h->usage_res_valid = s->static_generation != 0; h->usage_res_gen = s->static_generation;
  }
  CUDA_TRY(h, cudaEventRecord(h->ev1, h->stream));
  rc = build_dynamic(h, s);
  if (rc != KB_OK) { cudaStreamSynchronize(h->stream); return rc; }  // the copies read the caller's buffers
  D.tab_local = 0; D.gparent = D.parent; D.lq = nullptr; D.cq_entry = nullptr; D.ent_gid = nullptr; D.node_gid = nullptr; D.local_flat = 0; D.cq_rec = nullptr;
  D.Q = Q; D.C = C; D.N = N; D.F = F; D.R = R; D.FR = FR; D.W = s->n_wl; D.P = s->n_podset; D.A = s->n_adm;
  D.AU = s->n_adm_use; D.H = s->n_heads; D.NRG = s->n_rg; D.pods_res = s->pods_resource; D.flags = s->flags; D.now_ns = s->now_ns;
  int nroots = D.nRoots;
  // exact size of the per-cycle arena
  size_t tot = 0;
  auto need = [&](size_t n, size_t sz) { tot += pad256(n * sz); };
  need((size_t)Q * FR, 8);
  need(W, 4); need(W, 4); need(W, 8); need(W, 8); need(W, 8); need(W + 1, 4);
  need(P * R, 8); need(P, 4); need(P, 4); need(P, 4); need(P, 8); need(P * R, 1);
  need(A, 4); need(A, 4); need(A, 8); need(A, 8); need(A, 8); need(A, 1); need(A + 1, 4); need(AUc, 4); need(AUc, 8);
  need(H, 4); need(W, 1); need(W, 8); need(P, 4); need(Q, 4); need(h->tree_nodes.size() + 1, 16); need(256, 1); need(h->tree_nodes.size() * (size_t)FR, 8);
  need(Q + 1, 4); need(A, 4); need(A, 4); need(Q, 4); need(nroots, 4);
  need(nroots + 2, 4); need(Q + 2, 4); need(A, 8); need(A, 8); need(A, 4); need(A, 4);
  size_t rk_temp_bytes = 0;
  if (A) {
    size_t b1 = 0, b2 = 0;
    cub::DoubleBuffer<u64> dk(nullptr, nullptr); cub::DoubleBuffer<int32_t> dv(nullptr, nullptr);
    cub::DeviceRadixSort::SortPairs(nullptr, b1, dk, dv, (int)A, 0, 64, h->stream);
    cub::DeviceRadixSort::SortPairs(nullptr, b2, (const u64 *)nullptr, (u64 *)nullptr, (const int32_t *)nullptr, (int32_t *)nullptr, (int)A, 0, 32, h->stream);
    rk_temp_bytes = std::max(b1, b2) + 256;
  }
  need(rk_temp_bytes, 1);
  need(NF, 8); need(NF, 8); need(NF, 8); need(NF, 8);
  need(nroots, 4); need(nroots + 1, 4); need(nroots, 4); need(H, 4); need(H, 4); need(H, 4); need(H * 4, 8); need(H * 4, 8); need((size_t)Q * R, 8); need((size_t)N * R, 8);
  need(H, 1); need(H, 1); need(H, 4); need(H, 4); need(P * R, 1); need(P * R, 1); need(P * R, 1); need(P, 4);
  need(1, 4); need(N, 8); need(N, 4); need(N, 1);
  // fair-sharing preemption: search kernel configuration (single-warp CTAs on a private copy of the whole tree)
  bool fair = (s->flags & KB_F_FAIR_SHARING) != 0;
  h->search_grid = 1; h->search_smem = true; h->search_smem_bytes = 0;
  size_t fair_memo_items = 0;
  if (fair && A) {
    // private tree tables [nodes][FR] x 4, parent links, per-node search state (16 B: queue head, cached share, flags)
    size_t tb = (size_t)h->max_tree_nodes * FR * 32 + (size_t)h->max_tree_nodes * 4 + (size_t)h->max_tree_nodes * 16 + 128;
    h->search_smem = tb <= 190 * 1024;
    h->search_smem_bytes = h->search_smem ? tb : 0;
    // resident single-warp CTAs per SM as the occupancy calculator sees them (registers / shared memory)
    int per_sm = 1;
    if (h->search_smem) {
      cudaFuncSetAttribute(k_nominate_search_fair<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
      cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_nominate_search_fair<true, true>, 32, h->search_smem_bytes);
    } else {
      cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_nominate_search_fair<false, true>, 32, 0);
    }
    per_sm = std::max(1, std::min(per_sm, 16));
    // the oracle-cell pass has up to FR tasks per entry
    h->search_grid = (int)std::max<size_t>(1, std::min<size_t>((size_t)h->sm_count * per_sm, std::max<size_t>(1, H * (size_t)FR)));
    fair_memo_items = std::min<size_t>(H, (64u << 20) / ((size_t)FR * sizeof(SimMemo)));
  }
  // warp-cooperative classical search: shared memory per warp = context + private column(s) + candidate codes
  size_t ws_warps = 1, ws_col_stride = 0, memo_items = 0, ws_list_total = 32;
  if (A && !fair) {
    const size_t kSmemBudget = 200 * 1024;
    size_t ncap_s = (size_t)h->max_tree_nodes;
    // k_search_cells: one column, codes of the longest bucket
    size_t ctxA = (sizeof(WCtx<1>) + 15) & ~(size_t)15;
    size_t colA = ncap_s * 8 <= 48 * 1024 ? ncap_s : 0;
    size_t codesA = (size_t)h->max_frl_len <= 8192 ? (((size_t)h->max_frl_len + 31) & ~(size_t)31) : 0;
    size_t perA = ctxA + ((colA * 8 + 15) & ~(size_t)15) + ((codesA + 15) & ~(size_t)15);
    int wpbA = (int)std::max<size_t>(1, std::min<size_t>(16, kSmemBudget / perA));
    int bpsA = (int)std::max<size_t>(1, std::min<size_t>(32 / wpbA, (220 * 1024) / (perA * wpbA + 1024)));
    h->sa_wpb = wpbA; h->sa_col_elems = (int)colA; h->sa_codes = (int)codesA; h->sa_smem = perA * wpbA;
    h->sa_grid = std::max(1, std::min(h->sm_count * bpsA, (int)((H * (size_t)FR + 31) / 32)));
    // grouped form: one column's statics + base usage shared by the CTA, private column + codes per warp
    {
      size_t shared_b = ((ncap_s * (sizeof(ColStat) + 8)) + 15) & ~(size_t)15;
      size_t perG = ctxA + ((ncap_s * 8 + 15) & ~(size_t)15) + ((codesA + 15) & ~(size_t)15);
      size_t budget = 220 * 1024;
      int wpbG = shared_b + perG <= budget ? (int)std::min<size_t>(16, (budget - shared_b) / perG) : 0;
      h->sg_on = wpbG >= 4;
      h->sg_wpb = std::max(1, wpbG); h->sg_ncap = (int)ncap_s; h->sg_smem = shared_b + perG * h->sg_wpb;
      h->sg_grid = h->sm_count;
      if (h->sg_on) { wpbA = std::max(wpbA, wpbG); h->sa_grid = std::max(h->sa_grid, h->sg_grid); }
    }
    // k_nominate_walk: up to Kcap columns (cells of one workload's assignment)
    size_t kcap = std::min<size_t>(std::min<size_t>((size_t)FR, KB_MAX_CELLS), (size_t)h->max_head_podsets * R);
    size_t ctxB = (sizeof(WCtx<KB_MAX_CELLS>) + 15) & ~(size_t)15;
    // The walk is a chain of dependent loads per entry: occupancy (16 warps per SM at 128 registers) hides more
    // latency than shared-memory columns would save, so the private columns of its searches live in global scratch.
    size_t colB = 0;
    size_t perB = ctxB;
    int wpbB = 8;
    int bpsB = 2;
    h->sb_wpb = wpbB; h->sb_col_elems = (int)colB; h->sb_smem = perB * wpbB;
    h->sb_grid = std::max(1, std::min(h->sm_count * bpsB, (int)((H + wpbB - 1) / wpbB)));
    ws_warps = std::max((size_t)h->sa_grid * wpbA, (size_t)h->sb_grid * wpbB);
    // per-warp candidate-code / target scratch: a single-cell search sees one bucket, GetTargets at most the root's list
    h->sa_list_cap = (int)(((size_t)h->max_frl_len + 31) & ~(size_t)31);
    h->sb_list_cap = (int)(((size_t)h->max_root_adm + 31) & ~(size_t)31);
    ws_list_total = std::max((size_t)h->sa_grid * wpbA * h->sa_list_cap, (size_t)h->sb_grid * wpbB * h->sb_list_cap);
    if (colA == 0) ws_col_stride = ncap_s;
    if (kcap * ncap_s > colB) ws_col_stride = std::max(ws_col_stride, std::min<size_t>((size_t)FR, KB_MAX_CELLS) * ncap_s);
    memo_items = std::min<size_t>(H, (64u << 20) / ((size_t)FR * sizeof(SimMemo)));
  }
  if (fair && A) memo_items = fair_memo_items;
  size_t G = (fair && A) ? (size_t)h->search_grid : 1, acap = (fair && A) ? (size_t)h->max_root_adm : 1, ncap = (size_t)h->max_tree_nodes;
  size_t pool_cap = A * 4 + 1024;
  need(A, 4); need(nroots + 1, 4); need(H, 4); need(2, 4); need(H, 4); need(H, 4); need(pool_cap, 4); need(pool_cap, 1); need(1, 4);
  need(H + 1, 4); need(pool_cap, 4); need(pool_cap, 1);  // preemption targets in CSR order (download)
  need(A, 1); need(A, 4); need(nroots, 4); need(A ? NF : 1, 8);
  need(G * acap, 4); need(G * acap, 4); need(G * acap, 4); need(G * acap, 4); need(G * ncap, 4); need(G * acap, 1); need(G * acap, 1); need(G * ncap, 1); need(G * ncap, 1); need(G * ncap, 1); need(G * ncap, 8); need(G * ncap, 1);
  if (fair && A && !h->search_smem) need(G * ncap * FR, 8);
  // classical search tables + per-warp scratch
  const size_t nbuckets = (size_t)nroots * FR;
  const size_t sNF = A ? NF : 1, sAU = A ? AUc : 1;
  need(A, 4); need(sNF, 8); need(sNF, sizeof(ColStat)); need(sNF, 4); need(A ? nbuckets + 1 : 1, 4); need(A ? nbuckets + 2 : 1, 4); need(sAU, sizeof(FrRec)); need(A, sizeof(FrRec));
  need(memo_items * FR, sizeof(SimMemo)); need(1, 4); need(8, 8);
  need(A ? nbuckets + 2 : 1, 4); need(A ? nbuckets + 2 : 1, 4); need(A ? nbuckets + 2 : 1, 4); need(memo_items * FR, 4); need(memo_items * FR, 4);
  need(ws_warps * ws_col_stride, 8); need(ws_list_total, 1); need(ws_list_total, 4); need(ws_list_total, 1); need(ws_warps * (size_t)h->sa_list_cap, 8);
  if (fair) { need(H * FR, 8); need(H * (48 + 16 * KB_MAX_DEPTH), 1); need(N, 4); need(N, 4); }
  if (!h->arena.reserve(tot + (1u << 20))) { cudaStreamSynchronize(h->stream); return fail(h, KB_ERR_CUDA, "cudaMalloc failed"); }
  h->arena.reset();
  if (h->drain_mode) D.heads = h->arena.take<int32_t>(H);
  h->d_cq_entry = h->arena.take<int32_t>(Q); D.cq_entry = h->d_cq_entry;
  {  // fused per-root cycle (k_cycle_root): see the kernel's header for the conditions
    bool all_flat = true;
    for (uint8_t f : h->tree_flat) if (!f) all_flat = false;
    size_t nnm = (size_t)h->max_tree_nodes, tbm = nnm * FR;
    size_t sm = 6 * tbm * 8 + 2 * nnm * R * 8 + 4 * nnm * 4 + 7 * KB_TILE * 4 + (KB_MAX_DEPTH + 2 + 4) * 4 + 32 + nnm * 32;
    h->fused_smem = sm;
    h->fused_on = D.nLone == 0 && D.nTrees > 0 && h->one_head_per_cq && sm <= 220 * 1024 && (A_in == 0 || !h->preempt_possible) &&
                  (!(s->flags & KB_F_FAIR_SHARING) || all_flat) && getenv("KB_NO_FUSED") == nullptr;
    // k_cycle_flat: every tree flat, FR <= 64, the relocated copy of the largest root fits shared memory
    h->d_cq_rec = h->arena.take<int4>(h->tree_nodes.size() + 1); D.cq_rec = h->d_cq_rec;
    D.tl_usage = D.tl_nominal ? h->arena.take<i64>(h->tree_nodes.size() * (size_t)FR) : nullptr;
    h->flat_rcap = (int)std::min<size_t>((size_t)1 << 20, nnm * (size_t)std::max(1, h->max_head_podsets));
    h->flat_smem = flat_layout((int)nnm, FR, R, h->flat_rcap, h->max_blob_bytes).total;
    if (h->flat_static_smem == 0) { cudaFuncAttributes fa{}; cudaFuncGetAttributes(&fa, k_cycle_flat); h->flat_static_smem = std::max<size_t>(16, fa.sharedSizeBytes); }
    h->flat_on = h->fused_on && all_flat && FR <= 64 && h->flat_smem + h->flat_static_smem <= 227 * 1024 && getenv("KB_FUSED_V1") == nullptr;
    h->flat_on = h->flat_on && h->max_head_podsets < 65536;
    if (h->fused_on && !h->flat_on && !h->drain_mode) {
      CUDA_TRY(h, cudaMemsetAsync(h->d_cq_entry, 0xff, sizeof(int32_t) * (size_t)Q, h->stream));
      if (H) k_cq_entry<<<(unsigned)((H + 255) / 256), 256, 0, h->stream>>>(D, h->d_cq_entry);
    }
  }
  D.over_list = h->arena.take<int32_t>(Q); D.over_count = h->arena.take<int32_t>(nroots);
  D.root_adm_start = h->arena.take<int32_t>(nroots + 1); D.cq_adm_start = h->arena.take<int32_t>(Q + 1);
  D.cq_adm = h->arena.take<int32_t>(A); D.adm_rank = h->arena.take<int32_t>(A);
  D.root_adm_count = h->arena.take<int32_t>(nroots + 2); D.cq_adm_count = h->arena.take<int32_t>(Q + 2);
  h->rk_keys[0] = h->arena.take<u64>(A); h->rk_keys[1] = h->arena.take<u64>(A);
  h->rk_vals[0] = h->arena.take<int32_t>(A); h->rk_vals[1] = h->arena.take<int32_t>(A);
  h->rk_temp = h->arena.take<char>(rk_temp_bytes); h->rk_temp_bytes = rk_temp_bytes;
  D.adm_sorted = h->rk_vals[0];
  if (!A) {  // candidates_possible() reads the (empty) group tables
    CUDA_TRY(h, cudaMemsetAsync(D.root_adm_start, 0, sizeof(int32_t) * (size_t)(nroots + 1), h->stream));
    CUDA_TRY(h, cudaMemsetAsync(D.cq_adm_start, 0, sizeof(int32_t) * (size_t)(Q + 1), h->stream));
  }
  D.subtree = h->arena.take<i64>(NF); D.usage = h->arena.take<i64>(NF);
  D.avail = h->arena.take<i64>(NF); D.potential = h->arena.take<i64>(NF);
  D.root_count = h->arena.take<int32_t>(nroots); D.root_offset = h->arena.take<int32_t>(nroots + 1);
  D.root_cursor = h->arena.take<int32_t>(nroots); D.root_entries = h->arena.take<int32_t>(H);
  D.sorted = h->arena.take<int32_t>(H); D.pos_slot = h->arena.take<int32_t>(H); D.ekey = h->arena.take<u64>(H * 4); D.skey = h->arena.take<u64>(H * 4);
  D.fs_over = h->arena.take<i64>((size_t)Q * R); D.fs_lend = h->arena.take<i64>((size_t)N * R);
  {  // the result tables in the canonical layout (out_layout)
    OutLayout L = out_layout(H, P, (size_t)R);
    char *ob = h->arena.take<char>(L.prefix);
    h->d_out_block = ob;
    D.decision = (uint8_t *)(ob + L.off[0]); D.mode = (uint8_t *)(ob + L.off[1]);
    D.borrow = (int32_t *)(ob + L.off[2]); D.rank = (int32_t *)(ob + L.off[3]);
    D.ps_flavor = (int8_t *)(ob + L.off[4]); D.ps_res_mode = (int8_t *)(ob + L.off[5]); D.ps_tried = (int8_t *)(ob + L.off[6]);
    D.ps_count_out = (int32_t *)(ob + L.off[7]);
  }
  {  // cycle header block, cleared once per cycle: [0] status, [2..3] ps_n / ps_cursor, [4] target pool cursor, [8..23] search counters
    uint32_t *hdr = (uint32_t *)(h->d_out_block + out_layout(H, P, (size_t)R).hdr);
    D.status = hdr; D.ps_n = (int32_t *)(hdr + 2); D.ps_cursor = D.ps_n + 1; D.tgt_pool_used = (int32_t *)(hdr + 4); D.sstat = (u64 *)(hdr + 8);
  }
  D.ps_list = h->arena.take<int32_t>(H);
  D.tgt_off = h->arena.take<int32_t>(H); D.tgt_cnt = h->arena.take<int32_t>(H);
  D.tgt_pool_adm = h->arena.take<int32_t>(pool_cap); D.tgt_pool_reason = h->arena.take<uint8_t>(pool_cap);
  D.tgt_pool_cap = (int)pool_cap;
  h->d_tgt_start = h->arena.take<int32_t>(H + 1); h->d_tgt_adm = h->arena.take<int32_t>(pool_cap); h->d_tgt_reason = h->arena.take<uint8_t>(pool_cap);
  D.preempted = h->arena.take<uint8_t>(A);
  D.usage_shadow = h->arena.take<i64>(A ? NF : 1);
  D.sc_cand = h->arena.take<int32_t>(G * acap); D.sc_tgt = h->arena.take<int32_t>(G * acap); D.sc_cq_lca = h->arena.take<int32_t>(G * ncap);
  D.sc_aux1 = h->arena.take<int32_t>(G * acap); D.sc_aux2 = h->arena.take<int32_t>(G * acap);
  D.sc_variant = h->arena.take<uint8_t>(G * acap); D.sc_tgt_reason = h->arena.take<uint8_t>(G * acap);
  D.sc_cq_class = h->arena.take<int8_t>(G * ncap); D.sc_on_path = h->arena.take<int8_t>(G * ncap);
  D.sc_dirty = h->arena.take<uint8_t>(G * ncap); D.sc_drs_ratio = h->arena.take<double>(G * ncap); D.sc_drs_meta = h->arena.take<int8_t>(G * ncap);
  D.sc_usage = (fair && A && !h->search_smem) ? h->arena.take<i64>(G * ncap * FR) : nullptr;
  D.sc_adm_cap = (int)acap; D.sc_node_cap = (int)ncap;
  D.colU = h->arena.take<i64>(sNF); D.colS = h->arena.take<ColStat>(sNF); D.ovm = h->arena.take<uint32_t>(sNF);
  D.frl_count = h->arena.take<int32_t>(A ? nbuckets + 1 : 1); D.frl_start = h->arena.take<int32_t>(A ? nbuckets + 2 : 1);
  D.frl = h->arena.take<FrRec>(sAU); D.rrec = h->arena.take<FrRec>(A);
  D.memo = h->arena.take<SimMemo>(memo_items * FR); D.memo_items = (int)memo_items;
  D.cell_cursor = h->arena.take<int32_t>(1);
  D.cell_count = h->arena.take<int32_t>(A ? nbuckets + 2 : 1); D.cell_start = h->arena.take<int32_t>(A ? nbuckets + 2 : 1);
  D.cell_fill = h->arena.take<int32_t>(A ? nbuckets + 2 : 1);
  D.cell_list = h->arena.take<int32_t>(memo_items * FR); D.cell_bucket = h->arena.take<int32_t>(memo_items * FR);
  D.ws_col = h->arena.take<i64>(ws_warps * ws_col_stride); D.ws_col_stride = ws_col_stride;
  D.ws_codes = h->arena.take<uint8_t>(ws_list_total); D.ws_tgt = h->arena.take<int32_t>(ws_list_total);
  D.ws_tgt_reason = h->arena.take<uint8_t>(ws_list_total);
  D.ws_tgtq = h->arena.take<i64>(ws_warps * (size_t)h->sa_list_cap); D.ws_tgtq_cap = h->sa_list_cap;
  if (fair) {
    D.q_scratch = h->arena.take<i64>(H * FR); D.fs_state = h->arena.take<unsigned char>(H * (48 + 16 * KB_MAX_DEPTH));
    D.fs_cq_entry = h->arena.take<int32_t>(N); D.fs_winner = h->arena.take<int32_t>(N);
  }
  h->d_drs_rounded = h->arena.take<i64>(N); h->d_drs_res = h->arena.take<int32_t>(N); h->d_drs_borrowing = h->arena.take<uint8_t>(N);
  if (h->arena.used > h->arena.cap) { cudaStreamSynchronize(h->stream); return fail(h, KB_ERR_CUDA, "device arena accounting"); }
  h->hdr_clean = false;
  if (h->flat_on && !h->drain_mode) {  // head records + result-row fills + cleared header: one launch (k_flat_prep)
    int32_t rc2 = flat_rec_stamp(h);
    if (rc2 != KB_OK) return rc2;
    const size_t fill_words = 3 * pad256(P * R) / 4;
    const size_t tlc = D.tl_usage ? h->tree_nodes.size() * (size_t)FR : 0;
    const size_t nthr = std::max(std::max(std::max(H, fill_words), std::max(P, (size_t)32)), tlc);
    k_flat_prep<<<(unsigned)((nthr + 255) / 256), 256, 0, h->stream>>>(D, h->d_cq_rec, (int)fill_words, (int)P, (int)tlc);
    h->hdr_clean = true;
  } else {
    // rows of workloads that are not heads stay at -1
    CUDA_TRY(h, cudaMemsetAsync(D.ps_flavor, 0xff, 3 * pad256(P * R), h->stream));  // flavor, res_mode, tried are adjacent (out_layout)
    CUDA_TRY(h, cudaMemsetAsync(D.ps_count_out, 0, P * 4, h->stream));
  }
  h->stats.h2d_bytes = bytes;
  h->uploaded = true;
  if (sync) {  // caller buffers may be released after return
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    float ms = 0; cudaEventElapsedTime(&ms, h->ev0, h->ev1);
    h->stats.last_h2d_ms = ms;
  }
  return KB_OK;
}

extern "C" int32_t kb_upload(kb_handle *h, const kb_snapshot *s) { return upload_impl(h, s, true); }

// per-kernel timing: an event before each kernel (and one after the last) when profiling
static inline void kmark(kb_handle *h, int id) {
  if (!h->profile || h->kev_n > KB_N_KERNELS) return;
  h->kev_id[h->kev_n] = id;
  cudaEventRecord(h->kev[h->kev_n++], h->stream);
}
static int32_t launch_tree(kb_handle *h, int *launches) {
  DevSnap &D = h->D;
  if (D.nTrees) { kmark(h, KB_K_TREE); k_tree<<<D.nTrees, 1024, 0, h->stream>>>(D); (*launches)++; }
  if (D.nLone) { kmark(h, KB_K_LONE); int n = D.nLone * D.FR; k_lone<<<(n + 255) / 256, 256, 0, h->stream>>>(D); (*launches)++; }
  return KB_OK;
}

// admit kernel launches: lone-CQ roots (slots [0, nLone)) and cohort-tree roots
// (slots [nLone, nRoots)) separately so each class gets the shared memory it needs.
static size_t admit_smem(int nn_tables, int FR, int sort_cap, int nn_stage = 0) {
  size_t tb = (size_t)nn_tables * FR * 32;
  size_t mid = (size_t)KB_TILE * FR * 8; (void)sort_cap;
  // global-table mode: staging buffers of the commit pipeline (k_admit: cells, path table, target ids, scratch)
  size_t staging = nn_stage ? sizeof(TgCell) * 2 * KB_SUB * KB_ECAP + 4 * (size_t)nn_stage * KB_PF + 4 * 2 * KB_SUB * KB_TCAP +
                                  4 * KB_SUB * (KB_TCAP + 1) + 4 * KB_SUB * 32 + 2 * 2 * KB_SUB * 34 + (size_t)nn_stage + 2 * KB_SUB + 64
                            : 0;
  return tb + mid + 16 + (size_t)nn_tables * 4 + KB_TILE * 28 + (KB_MAX_DEPTH + 2) * 4 + 64 + staging;
}
static int32_t launch_admit(kb_handle *h, int *launches) {
  DevSnap &D = h->D;
  const size_t kMaxSmem = 200 * 1024;
  // sort capacity: entries per root are at most H; cap by what shared memory allows
  auto pick_cap = [&](int nn_tables) {
    int cap = 64;
    while (cap < KB_SORT_CAP && cap < D.H && admit_smem(nn_tables, D.FR, cap * 2) <= kMaxSmem) cap *= 2;
    return cap;
  };
  if (D.nLone && D.lone_fast) {
    size_t sm = (size_t)KB_LONE_WARPS * 32 * D.FR * 8;
    CUDA_TRY(h, cudaFuncSetAttribute(k_admit_lone, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxSmem));
    k_admit_lone<<<(D.nLone + KB_LONE_WARPS - 1) / KB_LONE_WARPS, KB_LONE_WARPS * 32, sm, h->stream>>>(D); (*launches)++;
  }
  if (D.nLone) {
    int cap = pick_cap(1);
    size_t sm = admit_smem(1, D.FR, cap);
    CUDA_TRY(h, cudaFuncSetAttribute(k_admit<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxSmem));
    k_admit<true><<<D.nLone, KB_ADMIT_THREADS, sm, h->stream>>>(D, 0, cap, 0); (*launches)++;
  }
  bool fair_trees = D.nTrees && (D.flags & KB_F_FAIR_SHARING);
  bool any_deep = false;
  for (uint8_t f : h->tree_flat) if (!f) any_deep = true;
  if (fair_trees && any_deep) {  // tournament kernel for the non-flat trees (flat ones exit at once)
    // shared memory: [quota tables][path][per-entry tournament state]; entries per tree <= its ClusterQueues
    size_t tables = (size_t)h->max_tree_nodes * D.FR * 32 + (size_t)h->max_tree_nodes * 4 + 16;
    size_t misc = (KB_MAX_DEPTH + 2) * 4 + ((size_t)h->max_tree_nodes * 4 + 1) * 4 + 128 * 4 + 64;
    size_t state = (size_t)h->max_tree_nodes * (48 + 16 * KB_MAX_DEPTH);
    CUDA_TRY(h, cudaFuncSetAttribute(k_admit_fair<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxSmem));
    CUDA_TRY(h, cudaFuncSetAttribute(k_admit_fair<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxSmem));
    if (tables + misc <= kMaxSmem) {
      int in_smem = tables + misc + state <= kMaxSmem;
      k_admit_fair<true><<<D.nTrees, 128, tables + misc + (in_smem ? state : 0), h->stream>>>(D, D.nLone, in_smem); (*launches)++;
    } else {
      int in_smem = misc + state <= kMaxSmem;
      k_admit_fair<false><<<D.nTrees, 128, misc + (in_smem ? state : 0), h->stream>>>(D, D.nLone, in_smem); (*launches)++;
    }
  }
  if (D.nTrees) {  // classical order, and fair sharing in flat cohorts (static key order)
    bool fits = admit_smem(h->max_tree_nodes, D.FR, 64) <= kMaxSmem;
    if (fits) {
      int cap = pick_cap(h->max_tree_nodes);
      size_t sm = admit_smem(h->max_tree_nodes, D.FR, cap);
      CUDA_TRY(h, cudaFuncSetAttribute(k_admit<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxSmem));
      k_admit<true><<<D.nTrees, KB_ADMIT_THREADS, sm, h->stream>>>(D, D.nLone, cap, 0); (*launches)++;
    } else {
      int cap = pick_cap(0);
      size_t sm = admit_smem(0, D.FR, cap, h->max_tree_nodes);
      int staged = sm <= kMaxSmem;
      if (!staged) sm = admit_smem(0, D.FR, cap);
      CUDA_TRY(h, cudaFuncSetAttribute(k_admit<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxSmem));
      k_admit<false><<<D.nTrees, KB_ADMIT_THREADS, sm, h->stream>>>(D, D.nLone, cap, staged); (*launches)++;
    }
  }
  return KB_OK;
}

static int32_t cycle_enqueue(kb_handle *h, bool hdr_copy = true) {
  if (!h || !h->uploaded) return fail(h, KB_ERR_INVALID, "kb_upload first");
  cudaSetDevice(h->device);
  DevSnap &D = h->D;
  int launches = 0;
  CUDA_TRY(h, cudaEventRecord(h->ev2, h->stream));
  // cycle header (status word, deferred-entry counters, target pool cursor, search counters): one contiguous block
  if (!h->hdr_clean) CUDA_TRY(h, cudaMemsetAsync(D.status, 0, 128, h->stream));  // (k_flat_prep cleared it with the upload)
  h->hdr_clean = false;
  if (!(h->fused_on && D.H)) CUDA_TRY(h, cudaMemsetAsync(D.root_count, 0, sizeof(int32_t) * (size_t)std::max(1, D.nRoots), h->stream));
  if (D.A) CUDA_TRY(h, cudaMemsetAsync(D.preempted, 0, (size_t)D.A, h->stream));
  h->kev_n = 0;
  int32_t rc_admit = KB_OK;
  if (D.A && !h->preempt_possible) { D.A = 0; D.AU = 0; }  // no ClusterQueue can ever preempt: the cycle never looks at the admitted tables
  if (D.A) {  // rank the admitted workloads (kb_rank.cuh): stable LSD passes UID -> reservation time -> (root | evicted | priority)
    kmark(h, KB_K_RANKADM);
    const int A = D.A, tb = 256, nb = (A + tb - 1) / tb;
    CUDA_TRY(h, cudaMemsetAsync(D.root_adm_count, 0, sizeof(int32_t) * (size_t)(D.nRoots + 2), h->stream));
    CUDA_TRY(h, cudaMemsetAsync(D.cq_adm_count, 0, sizeof(int32_t) * (size_t)(D.Q + 2), h->stream));
    cub::DoubleBuffer<u64> dk(h->rk_keys[0], h->rk_keys[1]);
    cub::DoubleBuffer<int32_t> dv(h->rk_vals[0], h->rk_vals[1]);
    size_t bytes = h->rk_temp_bytes;
    k_rank_keys_uid<<<nb, tb, 0, h->stream>>>(D, dk.Current(), dv.Current()); launches++;
    CUDA_TRY(h, cub::DeviceRadixSort::SortPairs(h->rk_temp, bytes, dk, dv, A, 0, 64, h->stream));
    k_rank_keys_qr<<<nb, tb, 0, h->stream>>>(D, dv.Current(), dk.Current()); launches++;
    CUDA_TRY(h, cub::DeviceRadixSort::SortPairs(h->rk_temp, bytes, dk, dv, A, 0, 64, h->stream));
    k_rank_keys_root<<<nb, tb, 0, h->stream>>>(D, dv.Current(), dk.Current()); launches++;
    int root_bits = 1; while ((1ll << root_bits) < (long long)D.nRoots) root_bits++;
    CUDA_TRY(h, cub::DeviceRadixSort::SortPairs(h->rk_temp, bytes, dk, dv, A, 0, 33 + root_bits, h->stream));
    D.adm_sorted = dv.Current();
    int32_t *other_vals = dv.Alternate();
    k_scan_i32<<<1, 1024, 0, h->stream>>>(D.root_adm_count, D.root_adm_start, D.nRoots); launches++;
    k_rank_positions<<<nb, tb, 0, h->stream>>>(D); launches++;
    // per-ClusterQueue lists in the same order: one more stable pass keyed by the ClusterQueue
    k_rank_keys_cq<<<nb, tb, 0, h->stream>>>(D, D.adm_sorted, dk.Current()); launches++;
    int cq_bits = 1; while ((1ll << cq_bits) < (long long)D.Q) cq_bits++;
    CUDA_TRY(h, cub::DeviceRadixSort::SortPairs(h->rk_temp, bytes, (const u64 *)dk.Current(), dk.Alternate(), (const int32_t *)D.adm_sorted, D.cq_adm, A, 0, cq_bits, h->stream));
    (void)other_vals;
    k_scan_i32<<<1, 1024, 0, h->stream>>>(D.cq_adm_count, D.cq_adm_start, D.Q); launches++;
    launches += 8;  // radix-sort passes (cub): histogram + onesweep kernels, counted coarsely
  }
  if (h->fused_on && D.H) {
    if (h->drain_mode) {
      if (h->flat_on) {
        int32_t rc2 = flat_rec_stamp(h);
        if (rc2 != KB_OK) return rc2;
        const size_t tlc = D.tl_usage ? h->tree_nodes.size() * (size_t)D.FR : 0;
        k_cq_rec<<<(unsigned)((std::max<size_t>((size_t)D.H, tlc) + 255) / 256), 256, 0, h->stream>>>(D, h->d_cq_rec, (int)tlc); launches++;
      } else {
        CUDA_TRY(h, cudaMemsetAsync(h->d_cq_entry, 0xff, sizeof(int32_t) * (size_t)D.Q, h->stream));
        k_cq_entry<<<(D.H + 255) / 256, 256, 0, h->stream>>>(D, h->d_cq_entry); launches++;
      }
    }
    kmark(h, KB_K_CYCLE_ROOT);
    if (h->flat_on) {
      if (!h->flat_attr_set) { CUDA_TRY(h, cudaFuncSetAttribute(k_cycle_flat, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(227 * 1024 - h->flat_static_smem))); h->flat_attr_set = true; }
      k_cycle_flat<<<D.nTrees, KB_FLAT_THREADS, h->flat_smem, h->stream>>>(D, flat_layout(h->max_tree_nodes, D.FR, D.R, h->flat_rcap, h->max_blob_bytes)); launches++;
    } else {
      CUDA_TRY(h, cudaFuncSetAttribute(k_cycle_root, cudaFuncAttributeMaxDynamicSharedMemorySize, 224 * 1024));
      k_cycle_root<<<D.nTrees, KB_ROOT_THREADS, h->fused_smem, h->stream>>>(D); launches++;
    }
  } else {
  launch_tree(h, &launches);
  if (D.H) {
    // per-(node, resource) sums the DominantResourceShare reads (fair target search, fair admit loop); only needs the tree pass
    if (D.flags & KB_F_FAIR_SHARING) { kmark(h, KB_K_FAIR_PREP); k_fair_prep<<<(D.N * D.R + 255) / 256, 256, 0, h->stream>>>(D); launches++; }
    kmark(h, KB_K_NOMINATE);
    // few entries: latency-bound -> KB_NG lanes per entry; many entries: throughput-bound -> one thread per entry
    if ((size_t)D.H * KB_NG <= (size_t)h->sm_count * 2048) k_nominate_coop<<<(int)(((size_t)D.H * KB_NG + 127) / 128), 128, 0, h->stream>>>(D);
    else k_nominate<<<(D.H + 127) / 128, 128, 0, h->stream>>>(D);
    launches++;
    if (D.A) {  // target search for the entries k_nominate deferred
      if (D.flags & KB_F_FAIR_SHARING) {
        kmark(h, KB_K_PREEMPT);
        CUDA_TRY(h, cudaMemsetAsync(D.over_count, 0, sizeof(int32_t) * (size_t)std::max(1, D.nRoots), h->stream));
        k_over<<<(D.Q + 255) / 256, 256, 0, h->stream>>>(D); launches++;
        CUDA_TRY(h, cudaMemsetAsync(D.cell_cursor, 0, 4, h->stream));
        if (h->search_smem) {
          CUDA_TRY(h, cudaFuncSetAttribute(k_nominate_search_fair<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
          CUDA_TRY(h, cudaFuncSetAttribute(k_nominate_search_fair<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
          if (D.memo_items) { k_nominate_search_fair<true, true><<<h->search_grid, 32, h->search_smem_bytes, h->stream>>>(D); launches++; }
          k_nominate_search_fair<true, false><<<h->search_grid, 32, h->search_smem_bytes, h->stream>>>(D);
        } else {
          if (D.memo_items) { k_nominate_search_fair<false, true><<<h->search_grid, 32, 0, h->stream>>>(D); launches++; }
          k_nominate_search_fair<false, false><<<h->search_grid, 32, 0, h->stream>>>(D);
        }
        launches++;
      } else {
        // per-cycle search tables: transposed columns + above-nominal masks, candidate buckets per (root, flavor-resource)
        kmark(h, KB_K_SEARCH_TABLES);
        size_t nf = (size_t)D.N * D.FR;
        int nb = D.nRoots * D.FR;
        k_columns<<<(unsigned)((nf + 255) / 256), 256, 0, h->stream>>>(D); launches++;
        CUDA_TRY(h, cudaMemsetAsync(D.frl_count, 0, sizeof(int32_t) * (size_t)(nb + 1), h->stream));
        CUDA_TRY(h, cudaMemsetAsync(D.cell_cursor, 0, 4, h->stream));
        if (D.AU) { k_frl_count<<<(D.AU + 255) / 256, 256, 0, h->stream>>>(D); launches++; }
        k_scan_i32<<<1, 1024, 0, h->stream>>>(D.frl_count, D.frl_start, nb); launches++;
        k_root_recs<<<(D.A + 255) / 256, 256, 0, h->stream>>>(D); launches++;
        if (D.AU) { k_frl_fill<<<(unsigned)(((size_t)nb * 32 + 127) / 128), 128, 0, h->stream>>>(D); launches++; }
        CUDA_TRY(h, cudaFuncSetAttribute(k_search_cells, cudaFuncAttributeMaxDynamicSharedMemorySize, 224 * 1024));
        CUDA_TRY(h, cudaFuncSetAttribute(k_nominate_walk, cudaFuncAttributeMaxDynamicSharedMemorySize, 224 * 1024));
        kmark(h, KB_K_SEARCH_CELLS);
        if (h->sg_on && D.memo_items) {
          long long ncell = (long long)D.memo_items * D.FR;
          CUDA_TRY(h, cudaMemsetAsync(D.cell_count, 0, sizeof(int32_t) * (size_t)(nb + 1), h->stream));
          CUDA_TRY(h, cudaMemsetAsync(D.cell_fill, 0, sizeof(int32_t) * (size_t)(nb + 1), h->stream));
          k_cells_mark<<<(unsigned)((ncell + 255) / 256), 256, 0, h->stream>>>(D); launches++;
          k_scan_i32<<<1, 1024, 0, h->stream>>>(D.cell_count, D.cell_start, nb); launches++;
          k_cells_scatter<<<(unsigned)((ncell + 255) / 256), 256, 0, h->stream>>>(D); launches++;
          CUDA_TRY(h, cudaFuncSetAttribute(k_search_cells_grouped, cudaFuncAttributeMaxDynamicSharedMemorySize, 224 * 1024));
          k_search_cells_grouped<<<h->sg_grid, h->sg_wpb * 32, h->sg_smem, h->stream>>>(D, h->sg_ncap, h->sa_codes, h->sa_list_cap); launches++;
        } else {
          k_search_cells<<<h->sa_grid, h->sa_wpb * 32, h->sa_smem, h->stream>>>(D, h->sa_col_elems, h->sa_codes, h->sa_list_cap); launches++;
        }
        kmark(h, KB_K_WALK);
        k_nominate_walk<<<h->sb_grid, h->sb_wpb * 32, h->sb_smem, h->stream>>>(D, h->sb_col_elems, h->sb_list_cap); launches++;
      }
    }
    kmark(h, KB_K_SCAN); k_scan_roots<<<1, 1024, 0, h->stream>>>(D); launches++;
    kmark(h, KB_K_SCATTER); k_scatter<<<(D.H + 255) / 256, 256, 0, h->stream>>>(D); launches++;
    kmark(h, KB_K_RANK); k_rank<<<(D.H + 255) / 256, 256, 0, h->stream>>>(D); launches++;
    kmark(h, KB_K_ADMIT);
    rc_admit = launch_admit(h, &launches);
  }
  }
  kmark(h, -1);
  CUDA_TRY(h, cudaEventRecord(h->ev3, h->stream));
  if (rc_admit != KB_OK) return rc_admit;
  CUDA_TRY(h, cudaGetLastError());
  h->last_launches = launches;
  // the cycle header (status word, counters, search / phase statistics: 128 contiguous bytes) comes back with one copy —
  // or, when the caller's result block has the canonical layout, inside the block's own copy (download_enqueue)
  h->hdr_host = &h->host_words[32];
  if (hdr_copy) CUDA_TRY(h, cudaMemcpyAsync(&h->host_words[32], D.status, 128, cudaMemcpyDeviceToHost, h->stream));
  return KB_OK;
}

// after the stream has been synchronized: timings + device status word
static int32_t cycle_finish(kb_handle *h) {
  float ms = 0; cudaEventElapsedTime(&ms, h->ev2, h->ev3);
  h->stats.last_cycle_gpu_ms = ms;
  h->stats.kernel_launches = h->last_launches;
  for (int i = 0; i < KB_N_KERNELS; i++) h->stats.kernel_ms[i] = 0.f;
  for (int i = 0; i + 1 < h->kev_n; i++) {
    float kms = 0; cudaEventElapsedTime(&kms, h->kev[i], h->kev[i + 1]);
    if (h->kev_id[i] >= 0) h->stats.kernel_ms[h->kev_id[i]] += kms;
  }
  memcpy(h->stats.search_stat, h->hdr_host + 8, 64);
  uint32_t st = h->hdr_host[0];
  if (st & KBS_UNSUPPORTED_PREEMPTION) return fail(h, KB_ERR_UNSUPPORTED, "unsupported preemption configuration");
  if (st & KBS_TARGET_OVERFLOW) return fail(h, KB_ERR_CAPACITY, "per-entry usage cell / target pool capacity exceeded");
  if (st & KBS_INTERNAL_LOOP) return fail(h, KB_ERR_CUDA, "internal: iteration guard tripped in the target search");
  return KB_OK;
}

extern "C" int32_t kb_cycle_resident(kb_handle *h) {
  int32_t rc = cycle_enqueue(h);
  if (rc != KB_OK) return rc;
  CUDA_TRY(h, cudaStreamSynchronize(h->stream));
  return cycle_finish(h);
}

// preemption targets of the cycle from the per-entry pool slices into CSR order (kb_cycle_out.tgt_start / tgt_adm / tgt_reason)
__global__ void k_tgt_compact(DevSnap D, const int32_t *start, int32_t *adm, uint8_t *reason) {
  int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= D.H) return;
  int n = D.tgt_cnt[e], o = D.tgt_off[e], s = start[e];
  for (int k = 0; k < n; k++) { adm[s + k] = D.tgt_pool_adm[o + k]; reason[s + k] = D.tgt_pool_reason[o + k]; }
}

// a kb_alloc_cycle_out block of this cycle's dimensions, pointers untouched: its tables have the device block's layout
static bool out_is_canonical_block(kb_handle *h, const kb_cycle_out *out) {
  const DevSnap &D = h->D;
  const size_t H = D.H;
  if (!out || !out->decision || !H) return false;
  OutLayout L = out_layout(H, (size_t)D.P, (size_t)D.R);
  const char *b = (const char *)out->decision;
  bool ok;
  {
    std::lock_guard<std::mutex> lk(g_pin_mu);
    auto it = g_out_blocks.find((uintptr_t)b);
    ok = it != g_out_blocks.end() && it->second.H == H && it->second.P == (size_t)D.P && it->second.R == (size_t)D.R;
  }
  return ok && (const char *)out->mode == b + L.off[1] && (const char *)out->borrow == b + L.off[2] && (const char *)out->commit_rank == b + L.off[3] &&
         (const char *)out->ps_flavor == b + L.off[4] && (const char *)out->ps_res_mode == b + L.off[5] && (const char *)out->ps_tried_idx == b + L.off[6] &&
         (const char *)out->ps_count == b + L.off[7];
}

static int32_t download_enqueue(kb_handle *h, kb_cycle_out *out) {
  if (!h || !h->uploaded || !out) return fail(h, KB_ERR_INVALID, "nothing to download");
  cudaSetDevice(h->device);
  DevSnap &D = h->D;
  size_t H = D.H, PR = (size_t)D.P * D.R;
  int64_t bytes = 0;
  CUDA_TRY(h, cudaEventRecord(h->ev4, h->stream));
#define DOWN(dst, src, n, T) if (out->dst && (n)) { CUDA_TRY(h, cudaMemcpyAsync(out->dst, D.src, (n) * sizeof(T), cudaMemcpyDeviceToHost, h->stream)); bytes += (n) * sizeof(T); }
  const bool one_dma = out_is_canonical_block(h, out);
  if (one_dma) {  // the eight result tables and the cycle header: one copy
    OutLayout L = out_layout(H, (size_t)D.P, (size_t)D.R);
    CUDA_TRY(h, cudaMemcpyAsync(out->decision, h->d_out_block, L.prefix, cudaMemcpyDeviceToHost, h->stream)); bytes += (int64_t)L.prefix;
    h->hdr_host = (const uint32_t *)((const char *)out->decision + L.hdr);
  }
  if (!one_dma) {
    DOWN(decision, decision, H, uint8_t); DOWN(mode, mode, H, uint8_t); DOWN(borrow, borrow, H, int32_t); DOWN(commit_rank, rank, H, int32_t);
    DOWN(ps_flavor, ps_flavor, PR, int8_t); DOWN(ps_res_mode, ps_res_mode, PR, int8_t); DOWN(ps_tried_idx, ps_tried, PR, int8_t);
    DOWN(ps_count, ps_count_out, (size_t)D.P, int32_t);
  }
  DOWN(node_usage, usage, (size_t)D.N * D.FR, i64);
#undef DOWN
  h->tgt_csr = false;
  if (out->tgt_start && D.A && H) {  // target lists -> CSR on the device: scan of the per-entry counts, one gather
    k_scan_i32<<<1, 1024, 0, h->stream>>>(D.tgt_cnt, h->d_tgt_start, (int)H);
    k_tgt_compact<<<(unsigned)((H + 127) / 128), 128, 0, h->stream>>>(D, h->d_tgt_start, h->d_tgt_adm, h->d_tgt_reason);
    CUDA_TRY(h, cudaMemcpyAsync(out->tgt_start, h->d_tgt_start, (H + 1) * 4, cudaMemcpyDeviceToHost, h->stream));
    bytes += (int64_t)(H + 1) * 4;
    h->tgt_csr = true;
  }
  CUDA_TRY(h, cudaEventRecord(h->ev5, h->stream));
  h->last_d2h_bytes = bytes;
  return KB_OK;
}

// after the stream has been synchronized (and cycle_finish filled host_words): preemption targets -> CSR
static int32_t download_finish(kb_handle *h, kb_cycle_out *out) {
  DevSnap &D = h->D;
  size_t H = D.H;
  int64_t bytes = h->last_d2h_bytes;
  out->n_targets = 0;
  if (out->tgt_start) {
    if (!h->tgt_csr) memset(out->tgt_start, 0, sizeof(int32_t) * (H + 1));
    else {
      int32_t nt = out->tgt_start[H];
      out->n_targets = nt;
      if (nt > out->tgt_capacity) return fail(h, KB_ERR_CAPACITY, "target buffer too small");
      if (nt > 0 && out->tgt_adm && out->tgt_reason) {
        CUDA_TRY(h, cudaMemcpyAsync(out->tgt_adm, h->d_tgt_adm, (size_t)nt * 4, cudaMemcpyDeviceToHost, h->stream));
        CUDA_TRY(h, cudaMemcpyAsync(out->tgt_reason, h->d_tgt_reason, (size_t)nt, cudaMemcpyDeviceToHost, h->stream));
        CUDA_TRY(h, cudaStreamSynchronize(h->stream));
        bytes += (int64_t)nt * 5;
      }
    }
  }
  float ms = 0; cudaEventElapsedTime(&ms, h->ev4, h->ev5);
  h->stats.last_d2h_ms = ms; h->stats.d2h_bytes = bytes;
  return KB_OK;
}

extern "C" int32_t kb_download(kb_handle *h, kb_cycle_out *out) {
  int32_t rc = download_enqueue(h, out);
  if (rc != KB_OK) return rc;
  // the target count of the last cycle is re-read here in case kb_cycle_resident ran several times
  CUDA_TRY(h, cudaStreamSynchronize(h->stream));
  return download_finish(h, out);
}

// One blocking call, one stream synchronisation: H2D copies, kernels and D2H copies are all enqueued first.
extern "C" int32_t kb_run_cycle(kb_handle *h, const kb_snapshot *s, kb_cycle_out *out) {
  static const bool trace = getenv("KB_TRACE") != nullptr;  // host-side phase times of the call on stderr
  auto now = [] { return std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
  double t0 = trace ? now() : 0, t1 = 0, t2 = 0, t3 = 0;
  int32_t rc = upload_impl(h, s, false);
  if (rc != KB_OK) return rc;
  if (trace) t1 = now();
  rc = cycle_enqueue(h, !out_is_canonical_block(h, out));
  if (rc != KB_OK) return rc;
  if (trace) t2 = now();
  rc = download_enqueue(h, out);
  if (rc != KB_OK) return rc;
  if (trace) t3 = now();
  CUDA_TRY(h, cudaStreamSynchronize(h->stream));
  if (trace) fprintf(stderr, "kb_run_cycle host us: upload %.1f enqueue %.1f download-enqueue %.1f wait %.1f\n", t1 - t0, t2 - t1, t3 - t2, now() - t3);
  { float ms = 0; cudaEventElapsedTime(&ms, h->ev0, h->ev1); h->stats.last_h2d_ms = ms; }
  rc = cycle_finish(h);
  if (rc != KB_OK) return rc;
  return download_finish(h, out);
}

// ---------------------------------------------------------------------------
// kb_run_drain: iterated cycles with the queue layer on the device (kb_drain.cuh)
// ---------------------------------------------------------------------------
static int32_t drain_impl(kb_handle *h, const kb_snapshot *s, kb_drain_out *out) {
  const int Q = s->n_cq, W = s->n_wl, R = s->n_resource, FR = s->n_flavor * s->n_resource;
  const int Hcap = std::min(Q, W);
  const int max_cycles = std::max(0, out->max_cycles);
  out->n_cycles = 0; out->n_decisions = 0; out->n_admitted = 0; out->gpu_ms = 0;
  if (Hcap == 0 || max_cycles == 0) return KB_OK;
  size_t extra = (size_t)std::min<long long>((long long)W, (long long)Hcap * max_cycles);
  h->drain_extra_adm = extra;
  h->drain_extra_au = std::min<size_t>((size_t)s->n_podset * R, extra * (size_t)FR);
  h->drain_mode = true;
  kb_snapshot s2 = *s;
  s2.n_heads = Hcap; s2.heads = nullptr;
  int32_t rc = upload_impl(h, &s2, false);
  if (rc != KB_OK) return rc;
  DevSnap &D = h->D;
  if (!h->ev_d) cudaEventCreate(&h->ev_d);
  // ---- drain-only device buffers
  const size_t Wz = (size_t)W, Hz = (size_t)Hcap;
  size_t sort_bytes = 0;
  {
    cub::DoubleBuffer<u64> dk(nullptr, nullptr); cub::DoubleBuffer<int32_t> dv(nullptr, nullptr);
    cub::DeviceRadixSort::SortPairs(nullptr, sort_bytes, dk, dv, W, 0, 64, h->stream);
    sort_bytes += 256;
  }
  const size_t trace_cap = out->trace_wl && out->trace_decision ? (size_t)std::max<int64_t>(0, out->trace_capacity) : 0;
  size_t tot = 0;
  auto need = [&](size_t n, size_t sz) { tot += pad256(n * sz); };
  need(Wz, 8); need(Wz, 8); need(Wz, 4); need(Wz, 4); need(sort_bytes, 1);
  need((size_t)Q + 2, 4); need((size_t)Q + 2, 4); need(Q, 4); need(Wz, 1); need((size_t)Q + 2, 4); need((size_t)Q + 2, 4);
  for (int k = 0; k < 4; k++) need(Hz + 2, 4);
  need(16, 4); need(Wz, 4); need(Wz, 4); need(Wz, 1); need(trace_cap, 4); need(trace_cap, 1);
  if (tot > h->drain_buf_cap) {
    if (h->drain_buf) cudaFree(h->drain_buf);
  if (h->tas_buf) cudaFree(h->tas_buf);
    h->drain_buf = nullptr; h->drain_buf_cap = 0;
    CUDA_TRY(h, cudaMalloc(&h->drain_buf, tot + (1 << 20)));
    h->drain_buf_cap = tot + (1 << 20);
  }
  size_t used = 0;
  auto take = [&](size_t n, size_t sz) { char *p = h->drain_buf + used; used += pad256(n * sz); return p; };
  u64 *keys[2] = {(u64 *)take(Wz, 8), (u64 *)take(Wz, 8)};
  int32_t *vals[2] = {(int32_t *)take(Wz, 4), (int32_t *)take(Wz, 4)};
  void *sort_tmp = take(sort_bytes, 1);
  DrainDev X{};
  int32_t *q_count = (int32_t *)take((size_t)Q + 2, 4);
  X.q_start = (int32_t *)take((size_t)Q + 2, 4); X.cursor = (int32_t *)take(Q, 4); X.gone = (uint8_t *)take(Wz, 1);
  X.flag = (int32_t *)take((size_t)Q + 2, 4); X.pos = (int32_t *)take((size_t)Q + 2, 4);
  X.e_assumed = (int32_t *)take(Hz + 2, 4); X.e_ncells = (int32_t *)take(Hz + 2, 4);
  X.e_adm_off = (int32_t *)take(Hz + 2, 4); X.e_cell_off = (int32_t *)take(Hz + 2, 4);
  X.counters = (int32_t *)take(16, 4);
  X.wl_admit_cycle = (int32_t *)take(Wz, 4); X.wl_evals = (int32_t *)take(Wz, 4); X.wl_last_decision = (uint8_t *)take(Wz, 1);
  X.trace_wl = trace_cap ? (int32_t *)take(trace_cap, 4) : nullptr; X.trace_dec = trace_cap ? (uint8_t *)take(trace_cap, 1) : nullptr;
  X.trace_cap = (long long)trace_cap;
  X.cq_usage = const_cast<i64 *>(D.cq_usage); X.wl_last_gen = const_cast<i64 *>(D.wl_last_gen); X.ps_last_tried = const_cast<int8_t *>(D.ps_last_tried);
  X.adm_cq = const_cast<int32_t *>(D.adm_cq); X.adm_priority = const_cast<int32_t *>(D.adm_priority);
  X.adm_ts = const_cast<i64 *>(D.adm_ts); X.adm_qr_ts = const_cast<i64 *>(D.adm_qr_ts); X.adm_uid = const_cast<i64 *>(D.adm_uid);
  X.adm_evicted = const_cast<uint8_t *>(D.adm_evicted); X.adm_use_start = const_cast<int32_t *>(D.adm_use_start);
  X.adm_use_fr = const_cast<int32_t *>(D.adm_use_fr); X.adm_use_qty = const_cast<i64 *>(D.adm_use_qty);
  // ---- per-ClusterQueue order (queueOrderingFunc): stable LSD passes uid -> timestamp -> (ClusterQueue | priority desc)
  const int tb = 256, nbW = (W + tb - 1) / tb, nbQ = (Q + tb - 1) / tb;
  CUDA_TRY(h, cudaMemsetAsync(q_count, 0, sizeof(int32_t) * ((size_t)Q + 2), h->stream));
  {
    cub::DoubleBuffer<u64> dk(keys[0], keys[1]); cub::DoubleBuffer<int32_t> dv(vals[0], vals[1]);
    size_t bytes = sort_bytes;
    k_drain_keys_uid<<<nbW, tb, 0, h->stream>>>(D, dk.Current(), dv.Current());
    CUDA_TRY(h, cub::DeviceRadixSort::SortPairs(sort_tmp, bytes, dk, dv, W, 0, 64, h->stream));
    k_drain_keys_ts<<<nbW, tb, 0, h->stream>>>(D, dv.Current(), dk.Current());
    CUDA_TRY(h, cub::DeviceRadixSort::SortPairs(sort_tmp, bytes, dk, dv, W, 0, 64, h->stream));
    k_drain_keys_cq<<<nbW, tb, 0, h->stream>>>(D, dv.Current(), dk.Current(), q_count);
    int cq_bits = 1; while ((1ll << cq_bits) < (long long)Q) cq_bits++;
    CUDA_TRY(h, cub::DeviceRadixSort::SortPairs(sort_tmp, bytes, dk, dv, W, 0, 32 + cq_bits, h->stream));
    X.q_order = dv.Current();
  }
  k_scan_i32<<<1, 1024, 0, h->stream>>>(q_count, X.q_start, Q);
  k_drain_init<<<std::max(nbW, nbQ), tb, 0, h->stream>>>(D, X);
  int32_t *d_heads = const_cast<int32_t *>(D.heads);
  auto enqueue_heads = [&]() {
    k_drain_flag<<<nbQ, tb, 0, h->stream>>>(D, X);
    k_scan_i32<<<1, 1024, 0, h->stream>>>(X.flag, X.pos, Q);
    k_drain_heads<<<nbQ, tb, 0, h->stream>>>(D, X, d_heads);
  };
  enqueue_heads();
  CUDA_TRY(h, cudaMemcpyAsync(&h->host_words[8], X.counters, 4, cudaMemcpyDeviceToHost, h->stream));
  CUDA_TRY(h, cudaStreamSynchronize(h->stream));
  int n_live = (int)h->host_words[8];
  int A_cur = s->n_adm, AU_cur = s->n_adm_use;
  const bool pre = h->preempt_possible;
  double gpu_ms = 0;
  for (int cyc = 0; cyc < max_cycles && n_live > 0; cyc++) {
    D.H = n_live; D.now_ns = s->now_ns + cyc;
    D.A = pre ? A_cur : 0; D.AU = pre ? AU_cur : 0;  // without preemption policies the cycle never looks at the admitted tables
    rc = cycle_enqueue(h);
    if (rc != KB_OK) return rc;
    X.A = A_cur; X.AU = AU_cur; X.cycle = cyc; X.trace_off = (long long)out->n_decisions;
    const int nbH = (n_live + tb - 1) / tb;
    k_drain_apply<<<nbH, tb, 0, h->stream>>>(D, X);
    k_scan_i32<<<1, 1024, 0, h->stream>>>(X.e_assumed, X.e_adm_off, n_live);
    k_scan_i32<<<1, 1024, 0, h->stream>>>(X.e_ncells, X.e_cell_off, n_live);
    k_drain_admit<<<nbH, tb, 0, h->stream>>>(D, X, s->now_ns + cyc);
    enqueue_heads();
    CUDA_TRY(h, cudaEventRecord(h->ev_d, h->stream));
    CUDA_TRY(h, cudaMemcpyAsync(&h->host_words[8], X.counters, 4, cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaMemcpyAsync(&h->host_words[9], X.e_adm_off + n_live, 4, cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaMemcpyAsync(&h->host_words[10], X.e_cell_off + n_live, 4, cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    rc = cycle_finish(h);
    if (rc != KB_OK) return rc;
    { float ms = 0; cudaEventElapsedTime(&ms, h->ev2, h->ev_d); gpu_ms += ms; }
    int n_new = (int)h->host_words[9], n_cells = (int)h->host_words[10];
    if (out->cycle_heads) out->cycle_heads[cyc] = n_live;
    if (out->cycle_admitted) out->cycle_admitted[cyc] = n_new;
    out->n_cycles = cyc + 1; out->n_decisions += n_live; out->n_admitted += n_new;
    A_cur += n_new; AU_cur += n_cells;
    n_live = (int)h->host_words[8];
    if (n_new == 0) break;  // nothing admitted: the next cycle would see the same snapshot
  }
  out->gpu_ms = gpu_ms;
  h->stats.last_cycle_gpu_ms = gpu_ms;
  // ---- results
  size_t PR = (size_t)D.P * D.R;
  if (out->wl_admit_cycle) CUDA_TRY(h, cudaMemcpyAsync(out->wl_admit_cycle, X.wl_admit_cycle, Wz * 4, cudaMemcpyDeviceToHost, h->stream));
  if (out->wl_last_decision) CUDA_TRY(h, cudaMemcpyAsync(out->wl_last_decision, X.wl_last_decision, Wz, cudaMemcpyDeviceToHost, h->stream));
  if (out->wl_evals) CUDA_TRY(h, cudaMemcpyAsync(out->wl_evals, X.wl_evals, Wz * 4, cudaMemcpyDeviceToHost, h->stream));
  if (out->ps_flavor && PR) CUDA_TRY(h, cudaMemcpyAsync(out->ps_flavor, D.ps_flavor, PR, cudaMemcpyDeviceToHost, h->stream));
  if (out->ps_count && D.P) CUDA_TRY(h, cudaMemcpyAsync(out->ps_count, D.ps_count_out, (size_t)D.P * 4, cudaMemcpyDeviceToHost, h->stream));
  if (out->cq_usage) CUDA_TRY(h, cudaMemcpyAsync(out->cq_usage, D.cq_usage, (size_t)Q * FR * 8, cudaMemcpyDeviceToHost, h->stream));
  size_t nt = std::min<size_t>(trace_cap, (size_t)out->n_decisions);
  if (nt) {
    CUDA_TRY(h, cudaMemcpyAsync(out->trace_wl, X.trace_wl, nt * 4, cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaMemcpyAsync(out->trace_decision, X.trace_dec, nt, cudaMemcpyDeviceToHost, h->stream));
  }
  CUDA_TRY(h, cudaStreamSynchronize(h->stream));
  return KB_OK;
}

extern "C" int32_t kb_run_drain(kb_handle *h, const kb_snapshot *s, kb_drain_out *out) {
  if (!h || !s || !out) return KB_ERR_INVALID;
  int32_t rc = drain_impl(h, s, out);
  h->drain_mode = false; h->drain_extra_adm = 0; h->drain_extra_au = 0;
  h->uploaded = false;  // the resident snapshot was consumed (queues advanced, admitted tables grown)
  return rc;
}

// ---------------------------------------------------------------------------
// kb_tas_find: topology-aware placement (kb_tas.cuh)
// ---------------------------------------------------------------------------
extern "C" int32_t kb_tas_find(kb_handle *h, const kb_tas_topology *t, const kb_tas_requests *r, kb_tas_out *out) {
  if (!h || !t || !r || !out) return KB_ERR_INVALID;
  cudaSetDevice(h->device);
  const int L = t->n_levels, ND = t->n_domains, R = t->n_resource, NQ = r->n_req;
  if (L < 1 || ND < 0 || R < 1 || R > 32 || t->pods_resource < 0 || t->pods_resource >= R || NQ < 0) return fail(h, KB_ERR_INVALID, "tas: bad dimensions");
  if (ND == 0) {  // no node of the flavor is schedulable: "no topology domains at level" (:1203-1205) for the first podset of every chain
    for (int q = 0; q < NQ; q++) {
      bool first = q == 0 || r->chain[q] != r->chain[q - 1];
      bool bad = r->level[q] < 0 || r->level[q] >= L || r->slice_level[q] < 0 || r->slice_level[q] >= L || r->level[q] > r->slice_level[q] || r->slice_size[q] < 1;
      out->status[q] = first ? (bad ? KB_TAS_BAD_REQUEST : KB_TAS_NO_FIT) : -1;
      out->asg_start[q] = 0;
    }
    out->asg_start[NQ] = 0; out->n_assigned = 0;
    return KB_OK;
  }
  if (t->level_start[0] != 0 || t->level_start[L] != ND) return fail(h, KB_ERR_INVALID, "tas: level_start must cover [0, n_domains)");
  const int leaf0 = t->level_start[L - 1], NL = ND - leaf0;
  // Children of a domain are contiguous in the next level (lexicographic numbering) and the child ranges of level l
  // tile level l+1 in order, so one [ND+1] table serves as child_start[d] .. child_start[d+1]: the end of the last
  // domain of level l is level_start[l+2], which is also where the children of the first domain of level l+1 start.
  std::vector<int32_t> cstart(ND + 1, ND);
  for (int l = 0; l < L; l++) {
    int a = t->level_start[l], b = t->level_start[l + 1];
    if (b < a) return fail(h, KB_ERR_INVALID, "tas: level_start not monotone");
    for (int d = a; d < b; d++) {
      int p = t->parent[d];
      if (l == 0) { if (p != -1) return fail(h, KB_ERR_INVALID, "tas: level-0 domains have no parent"); continue; }
      if (p < t->level_start[l - 1] || p >= a) return fail(h, KB_ERR_INVALID, "tas: parent must be a domain of the previous level");
      if (d > a && p < t->parent[d - 1]) return fail(h, KB_ERR_INVALID, "tas: domains of a level must be numbered in lexicographic levelValues order (children of one parent contiguous)");
    }
    if (l + 1 < L) {
      int c = t->level_start[l + 1], ce = t->level_start[l + 2];
      for (int d = a; d < b; d++) { cstart[d] = c; while (c < ce && t->parent[c] == d) c++; }
      if (c != ce) return fail(h, KB_ERR_INVALID, "tas: a domain of the next level has no parent in this level");
    }
  }
  // chains, rounds, shape slots
  std::vector<int32_t> pred(std::max(1, NQ), -1), chain_slot(std::max(1, NQ), -1), pos(std::max(1, NQ), 0), slot(std::max(1, NQ), 0);
  int n_chain_slots = 0, n_rounds = 0, max_count = 1;
  for (int q = 0; q < NQ;) {
    int e = q;
    while (e + 1 < NQ && r->chain[e + 1] == r->chain[q]) e++;
    if (e + 1 < NQ && r->chain[e + 1] < r->chain[q]) return fail(h, KB_ERR_INVALID, "tas: chain ids must be non-decreasing");
    int len = e - q + 1;
    int cs = len > 1 ? n_chain_slots++ : -1;
    for (int i = q; i <= e; i++) { pos[i] = i - q; pred[i] = i > q ? i - 1 : -1; chain_slot[i] = cs; }
    n_rounds = std::max(n_rounds, len);
    q = e + 1;
  }
  for (int q = 0; q < NQ; q++) max_count = std::max(max_count, r->count[q]);
  const int ok_words = (NL + 31) / 32;
  std::vector<std::vector<int32_t>> round_req(n_rounds), round_slot_req(n_rounds);
  {
    std::map<std::string, int> shapes;  // round 0: requests with the same shape share the counts
    for (int q = 0; q < NQ; q++) {
      int rd = pos[q];
      round_req[rd].push_back(q);
      if (rd == 0) {
        std::string key((const char *)(r->pod_request + (size_t)q * R), (size_t)R * 8);
        key.append((const char *)&r->request_mask[q], 4);
        uint32_t fl = r->flags[q] & KB_TAS_SIMULATE_EMPTY; key.append((const char *)&fl, 4);
        key.append((const char *)&r->slice_size[q], 4); key.append((const char *)&r->slice_level[q], 4);
        if (r->leaf_ok) key.append((const char *)(r->leaf_ok + (size_t)q * ok_words), (size_t)ok_words * 4);
        auto it = shapes.find(key);
        if (it == shapes.end()) { it = shapes.emplace(key, (int)round_slot_req[0].size()).first; round_slot_req[0].push_back(q); }
        slot[q] = it->second;
      } else { slot[q] = (int)round_slot_req[rd].size(); round_slot_req[rd].push_back(q); }
    }
  }
  size_t max_slots = 1, max_round = 1;
  for (int rd = 0; rd < n_rounds; rd++) { max_slots = std::max(max_slots, round_slot_req[rd].size()); max_round = std::max(max_round, round_req[rd].size()); }
  int max_level = 1;  // no list of a level is longer than the level
  for (int l = 0; l < L; l++) max_level = std::max(max_level, t->level_start[l + 1] - t->level_start[l]);
  // Lists and output regions are sized for assignments of at most `count` leaves.  Overcommitted leaves (negative free
  // capacity, so negative counts: requests.go CountIn) can make an assignment longer; such a request reports the size
  // it needed and the whole call runs again with larger buffers, which keeps the chains' order.
  std::vector<int32_t> region(std::max(1, NQ), 0);
  for (int q = 0; q < NQ; q++) region[q] = std::max(0, std::min(r->count[q], NL));
  int list_cap = std::min(max_count, max_level) + 8;
  const int sel_grid = (int)std::min<size_t>(max_round, (size_t)h->sm_count * 8);
  std::vector<int32_t> grow(NQ + 2, 0);
  for (;;) {
    std::vector<int32_t> tmp_start(NQ + 1, 0);
    for (int q = 0; q < NQ; q++) tmp_start[q + 1] = tmp_start[q] + region[q];
    // ---- device buffer (grow-only)
    size_t tot = 0;
    auto need = [&](size_t n, size_t sz) { tot += pad256(n * sz); };
    need(L + 1, 4); need(ND, 4); need(ND + 1, 4); need((size_t)NL * R, 8); need(NL, 4); need((size_t)NL * R, 8); need(NL, 4);
    need((size_t)NQ * R, 8); for (int k = 0; k < 10; k++) need(NQ, 4); need(r->leaf_ok ? (size_t)NQ * ok_words : 1, 4);
    need(max_slots * ND, 4); need(max_slots * ND, 4); need((size_t)n_chain_slots * NL * R, 8); need((size_t)n_chain_slots * NL, 4);
    need(NQ + 1, 4); need(NQ + 2, 4); need((size_t)n_rounds * max_slots, 4); need(NQ + 1, 4); need(NQ + 2, 4);
    need(tmp_start[NQ] + 1, 4); need(tmp_start[NQ] + 1, 4);
    need((size_t)sel_grid * 6 * list_cap, 4); need(max_round, 4); need(max_slots, 4); need(std::max(1, out->capacity), 4); need(std::max(1, out->capacity), 4);
    if (tot > h->tas_buf_cap) {
      if (h->tas_buf) cudaFree(h->tas_buf);
      h->tas_buf = nullptr; h->tas_buf_cap = 0;
      CUDA_TRY(h, cudaMalloc(&h->tas_buf, tot + (1 << 20)));
      h->tas_buf_cap = tot + (1 << 20);
    }
    size_t used = 0;
    auto take = [&](size_t n, size_t sz) { char *p = h->tas_buf + used; used += pad256(n * sz); return p; };
    auto upl = [&](const void *src, size_t n, size_t sz) -> char * { char *d = take(n, sz); if (n) cudaMemcpyAsync(d, src, n * sz, cudaMemcpyHostToDevice, h->stream); return d; };
    TasDev T{};
    T.L = L; T.n_domains = ND; T.n_leaves = NL; T.leaf0 = leaf0; T.R = R; T.pods_res = t->pods_resource; T.n_req = NQ;
    T.level_start = (const int32_t *)upl(t->level_start, L + 1, 4); T.parent = (const int32_t *)upl(t->parent, ND, 4);
    T.child_start = (const int32_t *)upl(cstart.data(), ND + 1, 4);
    T.free_cap = (const i64 *)upl(t->free_capacity, (size_t)NL * R, 8); T.cap_mask = (const uint32_t *)upl(t->cap_mask, NL, 4);
    T.tas_usage = (const i64 *)upl(t->tas_usage, (size_t)NL * R, 8); T.usage_mask = (const uint32_t *)upl(t->usage_mask, NL, 4);
    T.pod_request = (const i64 *)upl(r->pod_request, (size_t)NQ * R, 8); T.request_mask = (const uint32_t *)upl(r->request_mask, NQ, 4);
    T.flags = (const uint32_t *)upl(r->flags, NQ, 4); T.count = (const int32_t *)upl(r->count, NQ, 4);
    T.slice_size = (const int32_t *)upl(r->slice_size, NQ, 4); T.level = (const int32_t *)upl(r->level, NQ, 4);
    T.slice_level = (const int32_t *)upl(r->slice_level, NQ, 4);
    T.slot = (const int32_t *)upl(slot.data(), NQ, 4); T.chain_slot = (const int32_t *)upl(chain_slot.data(), NQ, 4); T.pred = (const int32_t *)upl(pred.data(), NQ, 4);
    T.leaf_ok = r->leaf_ok ? (const uint32_t *)upl(r->leaf_ok, (size_t)NQ * ok_words, 4) : nullptr; T.ok_words = ok_words;
    T.state = (int32_t *)take(max_slots * ND, 4); T.slice = (int32_t *)take(max_slots * ND, 4);
    T.assumed = (i64 *)take((size_t)n_chain_slots * NL * R, 8); T.assumed_mask = (uint32_t *)take((size_t)n_chain_slots * NL, 4);
    if (n_chain_slots) { cudaMemsetAsync(T.assumed, 0, (size_t)n_chain_slots * NL * R * 8, h->stream); cudaMemsetAsync(T.assumed_mask, 0, (size_t)n_chain_slots * NL * 4, h->stream); }
    // zeroed together: n_out, grow, the negative-leaf flags of every round's slots
    T.n_out = (int32_t *)take(NQ + 1, 4); T.grow = (int32_t *)take(NQ + 2, 4);
    int32_t *d_neg = (int32_t *)take((size_t)n_rounds * max_slots, 4);
    CUDA_TRY(h, cudaMemsetAsync(T.n_out, 0, (char *)h->tas_buf + used - (char *)T.n_out, h->stream));
    T.status = (int32_t *)take(NQ + 1, 4);
    int32_t *d_asg_start = (int32_t *)take(NQ + 2, 4);
    T.tmp_start = (int32_t *)upl(tmp_start.data(), NQ + 1, 4);
    T.tmp_leaf = (int32_t *)take(tmp_start[NQ] + 1, 4); T.tmp_count = (int32_t *)take(tmp_start[NQ] + 1, 4);
    T.lists = (int32_t *)take((size_t)sel_grid * 6 * list_cap, 4); T.list_cap = list_cap;
    int32_t *d_round = (int32_t *)take(max_round, 4), *d_slotreq = (int32_t *)take(max_slots, 4);
    int32_t *d_leaf = (int32_t *)take(std::max(1, out->capacity), 4), *d_cnt = (int32_t *)take(std::max(1, out->capacity), 4);
    CUDA_TRY(h, cudaEventRecord(h->ev2, h->stream));
    h->kev_n = 0;
    int launches = 0;
    for (int rd = 0; rd < n_rounds; rd++) {
      int ns = (int)round_slot_req[rd].size(), nr = (int)round_req[rd].size();
      CUDA_TRY(h, cudaMemcpyAsync(d_slotreq, round_slot_req[rd].data(), (size_t)ns * 4, cudaMemcpyHostToDevice, h->stream));
      CUDA_TRY(h, cudaMemcpyAsync(d_round, round_req[rd].data(), (size_t)nr * 4, cudaMemcpyHostToDevice, h->stream));
      T.neg = d_neg + (size_t)rd * max_slots;
      if (rd == 0) kmark(h, KB_K_TAS_LEAF);
      k_tas_leaf<<<dim3((NL + 255) / 256, ns), 256, 0, h->stream>>>(T, d_slotreq, ns); launches++;
      if (rd == 0) kmark(h, KB_K_TAS_REDUCE);
      for (int l = L - 2; l >= 0; l--) {
        int n = t->level_start[l + 1] - t->level_start[l];
        k_tas_reduce<<<dim3((n + 127) / 128, ns), 128, 0, h->stream>>>(T, d_slotreq, ns, l); launches++;
      }
      if (rd == 0) kmark(h, KB_K_TAS_SELECT);
      k_tas_select<<<std::min(nr, sel_grid), KB_TAS_THREADS, 0, h->stream>>>(T, d_round, nr); launches++;
      if (rd == 0) kmark(h, KB_K_TAS);
    }
    if (NQ) {
      k_scan_i32<<<1, 1024, 0, h->stream>>>(T.n_out, d_asg_start, NQ); launches++;
      k_tas_compact<<<NQ, 64, 0, h->stream>>>(T, d_asg_start, d_leaf, d_cnt, out->capacity); launches++;
    }
    kmark(h, -1);
    CUDA_TRY(h, cudaEventRecord(h->ev3, h->stream));
    CUDA_TRY(h, cudaGetLastError());
    if (NQ) {
      CUDA_TRY(h, cudaMemcpyAsync(out->status, T.status, (size_t)NQ * 4, cudaMemcpyDeviceToHost, h->stream));
      CUDA_TRY(h, cudaMemcpyAsync(out->asg_start, d_asg_start, (size_t)(NQ + 1) * 4, cudaMemcpyDeviceToHost, h->stream));
      CUDA_TRY(h, cudaMemcpyAsync(grow.data(), T.grow, 2 * 4, cudaMemcpyDeviceToHost, h->stream));
    } else out->asg_start[0] = 0;
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    if (grow[0] || grow[1]) {  // some request overflowed its list or its output region: enlarge them and run again
      bool larger = false;
      if (grow[0] > list_cap) {
        if (grow[0] > max_level) return fail(h, KB_ERR_INVALID, "tas: a list is longer than its level");
        list_cap = std::min(max_level, std::max(grow[0], 2 * list_cap));
        larger = true;
      }
      if (grow[1]) {
        CUDA_TRY(h, cudaMemcpy(grow.data() + 2, T.grow + 2, (size_t)NQ * 4, cudaMemcpyDeviceToHost));
        for (int q = 0; q < NQ; q++) if (grow[2 + q] > region[q]) { region[q] = grow[2 + q]; larger = true; }
      }
      if (!larger) return fail(h, KB_ERR_INVALID, "tas: overflow without a larger buffer to retry with");
      continue;
    }
    out->n_assigned = out->asg_start[NQ];
    int ncopy = std::min(out->n_assigned, out->capacity);
    if (ncopy > 0) {
      CUDA_TRY(h, cudaMemcpy(out->asg_leaf, d_leaf, (size_t)ncopy * 4, cudaMemcpyDeviceToHost));
      CUDA_TRY(h, cudaMemcpy(out->asg_count, d_cnt, (size_t)ncopy * 4, cudaMemcpyDeviceToHost));
    }
    { float ms = 0; cudaEventElapsedTime(&ms, h->ev2, h->ev3); h->stats.last_cycle_gpu_ms = ms; }
    h->stats.kernel_launches = launches;
    for (int i = 0; i < KB_N_KERNELS; i++) h->stats.kernel_ms[i] = 0.f;
    for (int i = 0; i + 1 < h->kev_n; i++) {
      float kms = 0; cudaEventElapsedTime(&kms, h->kev[i], h->kev[i + 1]);
      if (h->kev_id[i] >= 0) h->stats.kernel_ms[h->kev_id[i]] += kms;
    }
    if (out->n_assigned > out->capacity) return fail(h, KB_ERR_CAPACITY, "tas: assignment buffer too small");
    return KB_OK;
  }
}

extern "C" int32_t kb_tree_eval(kb_handle *h, const kb_snapshot *s, kb_tree_out *out) {
  int32_t rc = kb_upload(h, s);
  if (rc != KB_OK) return rc;
  DevSnap &D = h->D;
  int launches = 0;
  launch_tree(h, &launches);
  k_drs<<<(D.N + 127) / 128, 128, 0, h->stream>>>(D, h->d_drs_rounded, h->d_drs_res, h->d_drs_borrowing);
  CUDA_TRY(h, cudaGetLastError());
  size_t NF = (size_t)D.N * D.FR, QF = (size_t)D.Q * D.FR;
  if (out->subtree_quota) CUDA_TRY(h, cudaMemcpyAsync(out->subtree_quota, D.subtree, NF * 8, cudaMemcpyDeviceToHost, h->stream));
  if (out->usage) CUDA_TRY(h, cudaMemcpyAsync(out->usage, D.usage, NF * 8, cudaMemcpyDeviceToHost, h->stream));
  if (out->available) CUDA_TRY(h, cudaMemcpyAsync(out->available, D.avail, QF * 8, cudaMemcpyDeviceToHost, h->stream));
  if (out->potential_available) CUDA_TRY(h, cudaMemcpyAsync(out->potential_available, D.potential, QF * 8, cudaMemcpyDeviceToHost, h->stream));
  if (out->drs_rounded) CUDA_TRY(h, cudaMemcpyAsync(out->drs_rounded, h->d_drs_rounded, (size_t)D.N * 8, cudaMemcpyDeviceToHost, h->stream));
  if (out->drs_resource) CUDA_TRY(h, cudaMemcpyAsync(out->drs_resource, h->d_drs_res, (size_t)D.N * 4, cudaMemcpyDeviceToHost, h->stream));
  if (out->drs_borrowing) CUDA_TRY(h, cudaMemcpyAsync(out->drs_borrowing, h->d_drs_borrowing, (size_t)D.N, cudaMemcpyDeviceToHost, h->stream));
  CUDA_TRY(h, cudaStreamSynchronize(h->stream));
  if (out->available) for (size_t i = 0; i < QF; i++) if (out->available[i] < 0) out->available[i] = 0;  // Available() clamps at the CQ (clusterqueue_snapshot.go:154-156)
  return KB_OK;
}

extern "C" int32_t kb_set_profile(kb_handle *h, int32_t on) {
  if (!h) return KB_ERR_INVALID;
  h->profile = on != 0;
  return KB_OK;
}

extern "C" int32_t kb_get_stats(const kb_handle *h, kb_stats *out) {
  if (!h || !out) return KB_ERR_INVALID;
  *out = h->stats;
  return KB_OK;
}
