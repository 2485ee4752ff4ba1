// kb_flat.cuh — the scheduling cycle of one flat root cohort, start to finish in shared memory (k_cycle_flat).
//
// Same cycle as k_cycle_root's flat branch (kb_kernels.cuh: tree pass -> nominate -> iterator order -> threshold
// admit loop; scheduler.go:218-427 on a cohort whose ClusterQueues all hang directly off the root), rebuilt around
// one idea: the CTA first RELOCATES its root's slice of the snapshot into shared memory — quota tables, the static
// per-ClusterQueue policy / resource-group tables (one contiguous host-built block per tree, DevSnap::tree_blob) and
// the per-cycle head / podset records of its entries — renumbering every id (entry, workload, podset row,
// ClusterQueue, resource group) to be local to the root.  Heads with one podset and no PodSetReducer take a flavor
// walk, DRS term and request row specialised to the flat tree (flat_walk, flat_share_ratio).  For every other head the
// flavor assigner, the DRS term and the request expansion are the SAME device functions every other kernel uses
// (get_assignments_coop, entry_share_ratio, expand_entry): they run on a DevSnap whose table pointers all point into
// that relocated copy (tab_local == 2), so
// their chains of dependent loads (head -> workload -> podset rows -> resource group -> flavors -> quota cells) cost
// shared-memory latency instead of an L2 / HBM round trip per hop.  Global memory is touched in two bursts: the
// staging at the start (every load independent, at most three dependent hops: tree_start -> node / head record ->
// rows) and the publication of usage + decisions at the end.
//
// Used when k_cycle_root's conditions hold and, in addition, every tree is flat, FR <= 64 and the relocated copy fits
// shared memory (host: flat_layout).  Reference semantics are cited at the shared device functions.
#pragma once

struct FlatLay {  // byte offsets into the dynamic shared memory of k_cycle_flat (computed on the host, passed by value)
  uint32_t u, sub, lq, bl, av, pot, over, lend, blob, n_e, n_wl, n_ps0, n_psn, e_gid, e_cq, e_prio, e_ident, e_psn, e_wl, e_ps0, e_ts, e_lg, e_qr,
      e_flat, e_mode, e_borrow, e_rank, sorted, m_sorted, d_sorted, r_gid, r_count, r_min, r_mask, r_group, r_ok, r_req, r_last, o_fl, o_md, o_tr, o_cnt, key, misc, snap, rec, total;
};
__host__ __device__ inline FlatLay flat_layout(int ncap, int FR, int R, int rcap, int bcap) {
  FlatLay L;
  size_t o = 0;
  auto take = [&](size_t bytes) { size_t at = o; o += (bytes + 15) & ~(size_t)15; return (uint32_t)(at < 0xffffffffu ? at : 0xffffffffu); };
  const size_t T = (size_t)ncap * FR;
  L.u = take(T * 8); L.sub = take(T * 8); L.lq = take(T * 8); L.bl = take(T * 8); L.av = take(T * 8); L.pot = take(T * 8);
  L.over = take((size_t)ncap * R * 8); L.lend = take((size_t)ncap * R * 8);
  L.blob = take((size_t)bcap);
  L.n_e = take((size_t)ncap * 4); L.n_wl = take((size_t)ncap * 4); L.n_ps0 = take((size_t)ncap * 4); L.n_psn = take((size_t)ncap * 4);
  L.e_gid = take((size_t)ncap * 4); L.e_cq = take((size_t)ncap * 4); L.e_prio = take((size_t)ncap * 4); L.e_ident = take((size_t)ncap * 4);
  L.e_psn = take((size_t)(ncap + 1) * 4); L.e_wl = take((size_t)ncap * 4); L.e_ps0 = take((size_t)ncap * 4);
  L.e_ts = take((size_t)ncap * 8); L.e_lg = take((size_t)ncap * 8); L.e_qr = take((size_t)ncap); L.e_flat = take((size_t)ncap);
  L.e_mode = take((size_t)ncap * 4); L.e_borrow = take((size_t)ncap * 4); L.e_rank = take((size_t)ncap * 4);
  L.sorted = take((size_t)ncap * 4); L.m_sorted = take((size_t)ncap * 4); L.d_sorted = take(((size_t)ncap / 32 + 2) * 4);
  L.r_gid = take((size_t)rcap * 4); L.r_count = take((size_t)rcap * 4); L.r_min = take((size_t)rcap * 4); L.r_mask = take((size_t)rcap * 4);
  L.r_group = take((size_t)rcap * 4); L.r_ok = take((size_t)rcap * 8); L.r_req = take((size_t)rcap * R * 8); L.r_last = take((size_t)rcap * R);
  L.o_fl = take((size_t)rcap * R); L.o_md = take((size_t)rcap * R); L.o_tr = take((size_t)rcap * R); L.o_cnt = take((size_t)rcap * 4);
  L.key = take((size_t)ncap * 32);
  L.misc = take(64 + 256);
  L.snap = take(sizeof(DevSnap));
  L.rec = take((size_t)ncap * 16);
  L.total = (uint32_t)(o < 0xffffffffu ? o : 0xffffffffu);
  return L;
}

// Header of one tree's static block (DevSnap::tree_blob): counts + byte offsets (from the block start, 16 B aligned)
// of its arrays, all in the tree's local numbering (node handle = position in tree_nodes, resource groups and flavor
// lists renumbered in node order).
struct TreeBlobHdr {
  int32_t nn, nrg, nfl, bytes;
  int32_t gid, par, hgt, rgs;           // int32 [nn] global node id, local parent (-1 root), height, [nn+1] first local resource group
  int32_t gen, wgt;                     // i64 [nn] cq_generation, f64 [nn] fair_weight
  int32_t within, reclaim, borrow_w, wcb, wcp, pref;  // u8 [nn] each
  int32_t rgmask, rgfl, fl;             // u32 [nrg], int32 [nrg+1] first flavor slot, int32 [nfl] flavors
  int32_t pad;
};
static_assert(sizeof(TreeBlobHdr) == 80, "TreeBlobHdr layout");

// Head records: per tree node (tree-local order) {entry, workload, first podset row, podset count | stamp << 16} of the
// ClusterQueue's head.  A record is valid only when its stamp is the current one (DevSnap::rec_stamp), so the table
// is never cleared between cycles (the host clears it when it is (re)allocated or the 16-bit stamp wraps).
__device__ __forceinline__ void cq_rec_write(const DevSnap &D, int4 *rec, int e) {
  const int wl = D.heads[e];
  const int cq = D.wl_cq[wl];
  const int slot = D.root_slot[cq] - D.nLone;
  if (slot < 0) return;
  const int ps0 = D.wl_ps_start[wl];
  rec[D.tree_start[slot] + D.local_idx[cq]] = make_int4(e, wl, ps0, (D.wl_ps_start[wl + 1] - ps0) | (int)(D.rec_stamp << 16));
}
// usage rows into tree-local order (cohort rows zero): cell i of [tree nodes][FR]
__device__ __forceinline__ void tl_usage_write(const DevSnap &D, int i) {
  const int nd = D.tree_nodes[i / D.FR];
  D.tl_usage[i] = nd < D.Q ? D.cq_usage[(size_t)nd * D.FR + i % D.FR] : 0;
}
__global__ void k_cq_rec(DevSnap D, int4 *rec, int tl_cells) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < D.H) cq_rec_write(D, rec, i);
  if (i < tl_cells) tl_usage_write(D, i);
}
// static quota tables into tree-local row order (once per static upload)
__global__ void k_tl_static(DevSnap D, i64 *nominal, i64 *blimit, i64 *llimit, int tl_cells) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= tl_cells) return;
  const size_t g = (size_t)D.tree_nodes[i / D.FR] * D.FR + i % D.FR;
  nominal[i] = D.nominal[g]; blimit[i] = D.blimit[g]; llimit[i] = D.llimit[g];
}
// Everything the cycle needs prepared on the device, in one launch: head records, result rows of workloads that are
// not heads (-1 / 0), cleared cycle header.
__global__ void k_flat_prep(DevSnap D, int4 *rec, int fill_words, int P, int tl_cells) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < D.H) cq_rec_write(D, rec, i);
  if (i < tl_cells) tl_usage_write(D, i);
  if (i < fill_words) ((uint32_t *)D.ps_flavor)[i] = 0xffffffffu;  // flavor, res_mode, tried are adjacent (out_layout)
  if (i < P) D.ps_count_out[i] = 0;
  if (i < 32) D.status[i] = 0;
}

__device__ __forceinline__ void cp_async16(void *smem_dst, const void *gsrc) {
  unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d), "l"(gsrc) : "memory");
}
// 1-D bulk copies (the TMA engine, no tensor map) completing on an mbarrier
__device__ __forceinline__ void mbar_init(unsigned long long *bar, unsigned count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n\tfence.mbarrier_init.release.cluster;" ::"r"((unsigned)__cvta_generic_to_shared(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long *bar, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"((unsigned)__cvta_generic_to_shared(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void *smem_dst, const void *gsrc, unsigned bytes, unsigned long long *bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"((unsigned)__cvta_generic_to_shared(smem_dst)), "l"(gsrc), "r"(bytes), "r"((unsigned)__cvta_generic_to_shared(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(unsigned long long *bar, unsigned parity) {
  unsigned ok;
  asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.b32 %0, 1, 0, p;\n\t}"
               : "=r"(ok) : "r"((unsigned)__cvta_generic_to_shared(bar)), "r"(parity) : "memory");
  return ok != 0;
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.commit_group;\ncp.async.wait_group 0;" ::: "memory"); }

// ordered admit loop over the entries in iterator order (scheduler.go:269-401) on one threshold per (position, column):
//   Fit      : fits <=> usage_root[c] <= lim[pos][c] for every column   (INT64_MAX: no condition, INT64_MIN: never)
//              admitted: usage_root[c] += max(0, SubtreeQuota_root[c] - lim)
//   Preempt  : (no targets possible) reserves unconditionally (:303-318); lim holds SubtreeQuota_root - reserved amount,
//              so the amount added has the same form as for Fit
// One warp; lane = column (and column + 32 when kTwo).  Per entry the dependent chain is compare -> vote -> add; the
// thresholds of the next four positions are in flight while the current four are decided.  Results: one bit per
// position (the vote) in ok_bits; the decision follows from the bit and the entry's mode.
template <bool kTwo>
__device__ inline void flat_ordered_loop(int n, int FR, int lane, const i64 *s_lim, const int *m_sorted, uint32_t *ok_bits, i64 *s_u, const i64 *s_sub) {
  const int fr0 = lane, fr1 = lane + 32;
  const bool c0 = fr0 < FR, c1 = kTwo && fr1 < FR;
  i64 urt0 = c0 ? s_u[fr0] : 0, urt1 = c1 ? s_u[fr1] : 0;
  const i64 srt0 = c0 ? s_sub[fr0] : 0, srt1 = c1 ? s_sub[fr1] : 0;
  const i64 *col0 = s_lim + (c0 ? fr0 : 0), *col1 = s_lim + (c1 ? fr1 : 0);
  auto fetch = [&](i64 (&v0)[4], i64 (&v1)[4], int p0) {  // clamped: positions >= n are masked out by their mode bits
#pragma unroll
    for (int k = 0; k < 4; k++) {
      const size_t row = (size_t)min(p0 + k, n - 1) * FR;
      v0[k] = col0[row];
      if (kTwo) v1[k] = col1[row];
    }
  };
  i64 a0[4], a1[4], b0[4], b1[4];
  fetch(a0, a1, 0);
  for (int blk = 0; blk < n; blk += 32) {
    const int m = blk + lane < n ? m_sorted[blk + lane] : KB_MODE_NOFIT;
    const unsigned fitm = __ballot_sync(0xffffffffu, m == KB_MODE_FIT), anym = fitm | __ballot_sync(0xffffffffu, m == KB_MODE_PREEMPT);
    unsigned okb = 0;
    auto decide = [&](const i64 (&v0)[4], const i64 (&v1)[4], int p) {
#pragma unroll
      for (int k = 0; k < 4; k++) {
        const bool fit = (fitm >> (p + k)) & 1, any = (anym >> (p + k)) & 1;
        const i64 t0 = (fit && c0) ? v0[k] : INT64_MAX;
        const i64 d0r = (i64)((u64)srt0 - (u64)v0[k]);
        const i64 d0 = (any && c0 && d0r > 0) ? d0r : 0;
        i64 t1 = INT64_MAX, d1 = 0;
        if (kTwo) { t1 = (fit && c1) ? v1[k] : INT64_MAX; const i64 d1r = (i64)((u64)srt1 - (u64)v1[k]); d1 = (any && c1 && d1r > 0) ? d1r : 0; }
        const bool ok = __all_sync(0xffffffffu, urt0 <= t0 && (!kTwo || urt1 <= t1));  // the chain: compare -> vote -> add
        urt0 += ok ? d0 : 0;
        if (kTwo) urt1 += ok ? d1 : 0;
        okb |= (ok ? 1u : 0u) << (p + k);
      }
    };
    for (int p = 0; p < 32 && blk + p < n; p += 8) {
      fetch(b0, b1, blk + p + 4);
      decide(a0, a1, p);
      fetch(a0, a1, blk + p + 8);
      decide(b0, b1, p + 4);
    }
    if (lane == 0) ok_bits[blk >> 5] = okb;
  }
  if (c0) s_u[fr0] = urt0;
  if (c1) s_u[fr1] = urt1;
}
__device__ __forceinline__ int flat_decision(int mode, const uint32_t *ok_bits, int pos) {
  if (mode == KB_MODE_FIT) return (ok_bits[pos >> 5] >> (pos & 31)) & 1 ? KB_DEC_ASSUMED : KB_DEC_SKIPPED_NO_FIT;
  return mode == KB_MODE_PREEMPT ? KB_DEC_PREEMPT_NO_TARGETS : KB_DEC_NOFIT;
}

// e_flat bits of an entry, set when its records are gathered
enum {
  KB_FLAT_WALK = 1,  // one podset and no PodSetReducer (not: PartialAdmission, min_count >= 0, count > min_count)
  KB_FLAT_PODS = 2   // its ClusterQueue has a resource group with the pods resource (covers_pods)
};

// get_assignments_coop for an entry with KB_FLAT_WALK, on the relocated tables.  With one podset there is no usage
// assumed from earlier podsets, no PodSetGroup and no count scaling: request(r) = ps_req, or the pod count for the pods
// resource (ps_request).  On a flat tree every ClusterQueue's parent is the root, which has no parent, so find_height
// is closed form: over nominal (usage + val > nominal) -> height of the root and no reclaim, else 0 and may reclaim.
// No ClusterQueue of a relocated root has preemption candidates, so the oracle's answer is always PM_NOCAND.
// Tables are addressed from the layout (shared-memory offsets), not through the relocated DevSnap.  Same results
// (rows, mode, borrowing) as get_assignments_coop; lane 0 of the group writes them.
template <int NG>
__device__ __forceinline__ void flat_walk(const DevSnap &D, const FlatLay &Y, unsigned char *sm, int i, unsigned gmask, int gbase, int glane) {
  const int R = D.R, FR = D.FR;
  const unsigned char *blob = sm + Y.blob;
  const TreeBlobHdr &BH = *(const TreeBlobHdr *)blob;
  const i64 *s_u = (const i64 *)(sm + Y.u), *s_sub = (const i64 *)(sm + Y.sub), *s_av = (const i64 *)(sm + Y.av), *s_pot = (const i64 *)(sm + Y.pot);
  const int cq = ((const int *)(sm + Y.e_cq))[i], l = ((const int *)(sm + Y.e_psn))[i];
  const bool covers_pods = sm[Y.e_flat + i] & KB_FLAT_PODS;
  const int full = ((const int *)(sm + Y.r_count))[l];
  const uint32_t mask = ((const uint32_t *)(sm + Y.r_mask))[l] | (covers_pods ? 1u << D.pods_res : 0u);
  const u64 ok = ((const u64 *)(sm + Y.r_ok))[l];
  const i64 *req = (const i64 *)(sm + Y.r_req) + (size_t)l * R;
  const i64 lg = ((const i64 *)(sm + Y.e_lg))[i];
  const bool use_last = lg >= 0 && !(((const i64 *)(blob + BH.gen))[cq] > lg);
  const bool fung = D.flags & KB_F_FLAVOR_FUNGIBILITY;
  const int pref = blob[BH.pref + cq], wcb = blob[BH.wcb + cq], wcp = blob[BH.wcp + cq];
  const bool can_pwb = blob[BH.borrow_w + cq] != KB_POLICY_NEVER || ((D.flags & KB_F_FAIR_SHARING) && blob[BH.reclaim + cq] != KB_POLICY_NEVER);
  const int h_root = ((const int32_t *)(blob + BH.hgt))[0];
  const int32_t *rg_start = (const int32_t *)(blob + BH.rgs), *rg_fl = (const int32_t *)(blob + BH.rgfl), *fls = (const int32_t *)(blob + BH.fl);
  const uint32_t *rg_mask = (const uint32_t *)(blob + BH.rgmask);
  const int g0 = rg_start[cq], g1 = rg_start[cq + 1];
  int8_t *o_fl = (int8_t *)(sm + Y.o_fl) + (size_t)l * R, *o_md = (int8_t *)(sm + Y.o_md) + (size_t)l * R, *o_tr = (int8_t *)(sm + Y.o_tr) + (size_t)l * R;
  auto request = [&](int r) { return covers_pods && r == D.pods_res ? (i64)full : req[r]; };
  if (glane == 0) {
    for (int r = 0; r < R; r++) { o_fl[r] = -1; o_md[r] = -1; o_tr[r] = -1; }
    ((int *)(sm + Y.o_cnt))[l] = full;
  }
  bool has_reasons = false, failed = false;
  int ps_borrow = 0;
  uint32_t assigned = 0, ps_pmask = 0;
  for (int r0 = 0; r0 < R; r0++) {
    if (!(mask & (1u << r0)) || (assigned & (1u << r0))) continue;
    int g = -1;
    for (int k = g0; k < g1 && g < 0; k++) if (rg_mask[k] & (1u << r0)) g = k;
    if (g < 0) {
      if (request(r0) == 0) continue;
      failed = true; break;
    }
    const uint32_t rgm = rg_mask[g] & mask;
    const int fl0 = rg_fl[g], nfl = rg_fl[g + 1] - fl0;
    int best_f = -1, best_pm = PM_NOFIT, best_rb = INT32_MAX, best_maxb = 0;
    uint32_t best_pmask = 0;
    bool any_reason = false, done = false;
    int attempted = -1;
    const int idx0 = fung && use_last ? ((const int8_t *)(sm + Y.r_last))[(size_t)l * R + r0] + 1 : 0;
    for (int base = idx0; base < nfl && !done; base += NG) {
      // ---- one flavor per lane: every cell of the group is loaded before the first is decided ----
      const int idx = base + glane;
      u64 res = 0;  // packed as in assign_workload_coop
      int myf = -1;
      if (idx < nfl) {
        const int f = fls[fl0 + idx];
        myf = f;
        if ((ok >> f) & 1) {
          int rpm = PM_FIT, rb = 0, maxb = 0; uint32_t pmask = 0; bool reason = false;
          for (int rc = 0; rc < R && rpm != PM_NOFIT; rc += 4) {
            int pmv[4], bv[4];
#pragma unroll
            for (int j = 0; j < 4; j++) {  // cell_eval
              const int r = rc + j;
              pmv[j] = PM_FIT; bv[j] = 0;
              if (r < R && (rgm & (1u << r))) {
                const int c = cq * FR + f * R + r;
                const i64 val = request(r), pot = s_pot[c], nom = s_sub[c], u = s_u[c], av = s_av[c];
                const bool over = u + val > nom;
                if (val > pot) pmv[j] = PM_NOFIT;
                else {
                  bv[j] = over ? h_root : 0;
                  if (!(val <= imax(0, av))) pmv[j] = (val <= nom || !over || can_pwb) ? PM_NOCAND : PM_NOFIT;
                }
              }
            }
#pragma unroll
            for (int j = 0; j < 4; j++) {
              const int r = rc + j;
              if (r >= R || !(rgm & (1u << r))) continue;
              const int pm = pmv[j], b = bv[j];
              if (pm != PM_FIT) reason = true;
              if (gm_preferred(rpm, rb, pm, b, pref)) { rpm = pm; rb = b; }
              if (rpm == PM_NOFIT) break;
              if (fa_mode(pm) == KB_MODE_PREEMPT) pmask |= 1u << r;
              if (b > maxb) maxb = b;
            }
          }
          res = (u64)rpm | ((u64)(rb & 127) << 3) | ((u64)(maxb & 127) << 10) | ((u64)reason << 17) | (1ull << 19) | ((u64)pmask << 32);
        }
      }
      // ---- ordered scan over the flavors of this round (assign_workload_coop) ----
      for (int j = 0; j < NG && base + j < nfl; j++) {
        const u64 rj = __shfl_sync(gmask, res, gbase + j);
        const int fj = __shfl_sync(gmask, myf, gbase + j);
        attempted = base + j;
        if (!((rj >> 19) & 1)) { any_reason = true; continue; }
        const int rpm = (int)(rj & 7), rb = (int)((rj >> 3) & 127), maxb = (int)((rj >> 10) & 127);
        const uint32_t pmask = (uint32_t)(rj >> 32) & 0xffffu;
        if ((rj >> 17) & 1) any_reason = true;
        bool take = false;
        if (fung) {
          const bool try_next = rpm == PM_NOFIT || rpm == PM_NOCAND ||
                                ((rpm == PM_PREEMPT || rpm == PM_RECLAIM) && wcp == KB_FUNG_TRY_NEXT_FLAVOR) ||
                                (rb != 0 && wcb == KB_FUNG_TRY_NEXT_FLAVOR);
          if (!try_next) { take = true; done = true; }
          else if (gm_preferred(rpm, rb, best_pm, best_rb, pref)) take = true;
        } else if (rpm > best_pm) {
          take = true;
          done = rpm == PM_FIT;
        }
        if (take) { best_f = fj; best_pm = rpm; best_rb = rb; best_maxb = maxb; best_pmask = pmask; }
        if (done) break;
      }
    }
    if (best_f < 0) { failed = true; break; }
    const int tried = fung ? (attempted == nfl - 1 ? -1 : attempted) : 0;
    if (glane == 0)
      for (int r = 0; r < R; r++) {
        if (!(rgm & (1u << r))) continue;
        o_fl[r] = (int8_t)best_f; o_md[r] = (best_pmask >> r) & 1 ? KB_MODE_PREEMPT : KB_MODE_FIT; o_tr[r] = (int8_t)tried;
      }
    assigned |= rgm;
    ps_pmask |= best_pmask & rgm;
    if (best_maxb > ps_borrow) ps_borrow = best_maxb;
    if (best_pm != PM_FIT && any_reason) has_reasons = true;
  }
  int mode = KB_MODE_FIT, borrowing = ps_borrow;
  if (failed) {
    mode = KB_MODE_NOFIT; borrowing = 0;
    if (glane == 0) for (int r = 0; r < R; r++) { o_fl[r] = -1; o_md[r] = -1; o_tr[r] = -1; }
  } else if (has_reasons) {
    if ((assigned & mask) == 0) mode = KB_MODE_NOFIT;
    else if (ps_pmask & mask) mode = KB_MODE_PREEMPT;
  }
  if (glane == 0) { ((int *)(sm + Y.e_mode))[i] = mode; ((int *)(sm + Y.e_borrow))[i] = borrowing; }
}

// entry_share_ratio of a KB_FLAT_WALK entry: its one podset puts request(r) on a single cell (flavor o_fl[r]), counted
// at its full count, and the ClusterQueue's parent is the root (local handle 0)
__device__ __forceinline__ double flat_share_ratio(const DevSnap &D, const FlatLay &Y, const unsigned char *sm, int i, int r) {
  const int R = D.R;
  const int hq = ((const int *)(sm + Y.e_cq))[i], l = ((const int *)(sm + Y.e_psn))[i];
  i64 b = ((const i64 *)(sm + Y.over))[hq * R + r];
  const int f = ((const int8_t *)(sm + Y.o_fl))[(size_t)l * R + r];
  if (f >= 0) {
    const i64 q = (sm[Y.e_flat + i] & KB_FLAT_PODS) && r == D.pods_res ? (i64)((const int *)(sm + Y.o_cnt))[l] : ((const i64 *)(sm + Y.r_req))[(size_t)l * R + r];
    const int c = hq * D.FR + f * R + r;
    const i64 base = ((const i64 *)(sm + Y.u))[c] - ((const i64 *)(sm + Y.sub))[c];
    b += imax(0, base + (q > 0 ? q : 0)) - imax(0, base);
  }
  const i64 lend = ((const i64 *)(sm + Y.lend))[r];
  return (b > 0 && lend > 0) ? (double)b * 1000.0 / (double)lend : 0.0;
}
// entry_key_finish on the relocated records (local workload = local entry); the key reads no podset
__device__ __forceinline__ void flat_key_finish(const DevSnap &D, const FlatLay &Y, const unsigned char *sm, int i, bool fair, double best, u64 *k) {
  unsigned prio = 0;
  if (D.flags & KB_F_PRIORITY_SORTING_WITHIN_COHORT) prio = ~((unsigned)((const int *)(sm + Y.e_prio))[i] ^ 0x80000000u);
  const u64 ts = (u64)((const i64 *)(sm + Y.e_ts))[i] ^ 0x8000000000000000ull;
  const int borrow = ((const int *)(sm + Y.e_borrow))[i];
  if (!fair) {
    const u64 no_qr = (D.wl_has_qr && sm[Y.e_qr + i]) ? 0ull : 1ull;
    k[0] = (no_qr << 63) | ((u64)(unsigned)borrow << 32) | prio; k[1] = ts; k[2] = (u64)(unsigned)((const int *)(sm + Y.e_gid))[i]; k[3] = 0;
    return;
  }
  const unsigned char *blob = sm + Y.blob;
  const TreeBlobHdr &BH = *(const TreeBlobHdr *)blob;
  const int cq = ((const int *)(sm + Y.e_cq))[i];
  const double w = ((const double *)(blob + BH.wgt))[cq];
  const bool zwb = w == 0 && best != 0;
  const double value = zwb ? best : (best == 0 ? 0.0 : best / w);
  const u64 vb = (u64)__double_as_longlong(value);
  const u64 flags = ((D.flags & KB_F_FS_PRIORITIZE_NON_BORROWING) && borrow > 0 ? 2 : 0) | (zwb ? 1 : 0);
  k[0] = (flags << 32) | (vb >> 32); k[1] = (vb << 32) | prio; k[2] = ts; k[3] = (u64)(unsigned)((const int32_t *)(blob + BH.gid))[cq];
}

// get_assignments_coop for the entries without KB_FLAT_WALK, kept out of line: its inlined copies of
// assign_workload_coop (four, three of them for the PodSetReducer) would otherwise share the kernel's 64 registers
// with the rest of the cycle and push its long-lived values to the stack.
template <int NG>
__device__ __noinline__ void flat_generic_assign(const DevSnap &L, int i, unsigned gmask, int gbase, int glane, int *e_mode, int *e_borrow) {
  bool need_search = false;
  int borrowing;
  const int mode = get_assignments_coop<NG>(L, &need_search, i, &borrowing, gmask, gbase, glane);
  if (glane == 0) { e_mode[i] = mode; e_borrow[i] = borrowing; }
}

#define KB_FLAT_THREADS 1024
#ifndef KB_FLAT_NG
#define KB_FLAT_NG 8  // lanes per entry in the nominate phase
#endif
__global__ void __launch_bounds__(KB_FLAT_THREADS) k_cycle_flat(const __grid_constant__ DevSnap D, const __grid_constant__ FlatLay Y) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int FR = D.FR, R = D.R;
  const int t = blockIdx.x, tid = threadIdx.x, nthreads = blockDim.x;
  const int lane = tid & 31, warp = tid >> 5;
  const int fr_sh = 31 - __clz(FR); const bool fr_p2 = (1 << fr_sh) == FR;
  auto row_of = [&](int i) { return fr_p2 ? i >> fr_sh : i / FR; };
  auto col_of = [&](int i) { return fr_p2 ? i & (FR - 1) : i % FR; };
  long long tk0 = clock64();
#ifndef KB_FLAT_PROBE
#define KB_FLAT_PROBE 0
#endif
  // fine-grained probe points of thread 0 (instrumented builds only: -DKB_FLAT_PROBE=<set>): cycles since the previous point
#define KB_PP(set, k) do { if (KB_FLAT_PROBE == (set) && blockIdx.x == 0 && threadIdx.x == 0) { long long now_ = clock64(); D.sstat[k] = (u64)(now_ - tk0); tk0 = now_; } } while (0)
#define KB_FPHASE(k) do { if (KB_FLAT_PROBE) break; if (blockIdx.x == 0 && threadIdx.x == 0) { long long now_ = clock64(); D.sstat[k] = (u64)(now_ - tk0); tk0 = now_; } } while (0)
  i64 *s_u = (i64 *)(smem_raw + Y.u), *s_sub = (i64 *)(smem_raw + Y.sub), *s_lq = (i64 *)(smem_raw + Y.lq), *s_bl = (i64 *)(smem_raw + Y.bl);
  i64 *s_av = (i64 *)(smem_raw + Y.av), *s_pot = (i64 *)(smem_raw + Y.pot), *s_over = (i64 *)(smem_raw + Y.over), *s_lend = (i64 *)(smem_raw + Y.lend);
  unsigned char *s_blob = smem_raw + Y.blob;
  int *n_e = (int *)(smem_raw + Y.n_e), *n_wl = (int *)(smem_raw + Y.n_wl), *n_ps0 = (int *)(smem_raw + Y.n_ps0), *n_psn = (int *)(smem_raw + Y.n_psn);
  int *e_gid = (int *)(smem_raw + Y.e_gid), *e_cq = (int *)(smem_raw + Y.e_cq), *e_prio = (int *)(smem_raw + Y.e_prio), *e_ident = (int *)(smem_raw + Y.e_ident);
  int *e_psn = (int *)(smem_raw + Y.e_psn), *e_wl = (int *)(smem_raw + Y.e_wl), *e_ps0 = (int *)(smem_raw + Y.e_ps0);
  i64 *e_ts = (i64 *)(smem_raw + Y.e_ts), *e_lg = (i64 *)(smem_raw + Y.e_lg); uint8_t *e_qr = smem_raw + Y.e_qr, *e_flat = smem_raw + Y.e_flat;
  int *e_mode = (int *)(smem_raw + Y.e_mode), *e_borrow = (int *)(smem_raw + Y.e_borrow), *e_rank = (int *)(smem_raw + Y.e_rank);
  int *s_sorted = (int *)(smem_raw + Y.sorted), *m_sorted = (int *)(smem_raw + Y.m_sorted); uint32_t *ok_bits = (uint32_t *)(smem_raw + Y.d_sorted);
  int *r_gid = (int *)(smem_raw + Y.r_gid), *r_count = (int *)(smem_raw + Y.r_count), *r_min = (int *)(smem_raw + Y.r_min);
  uint32_t *r_mask = (uint32_t *)(smem_raw + Y.r_mask); int *r_group = (int *)(smem_raw + Y.r_group); u64 *r_ok = (u64 *)(smem_raw + Y.r_ok);
  i64 *r_req = (i64 *)(smem_raw + Y.r_req); int8_t *r_last = (int8_t *)(smem_raw + Y.r_last);
  int8_t *o_fl = (int8_t *)(smem_raw + Y.o_fl), *o_md = (int8_t *)(smem_raw + Y.o_md), *o_tr = (int8_t *)(smem_raw + Y.o_tr); int *o_cnt = (int *)(smem_raw + Y.o_cnt);
  u64 *s_key = (u64 *)(smem_raw + Y.key);
  int *s_misc = (int *)(smem_raw + Y.misc);  // [0] n entries, [1] total rows

  // ---- 0. staging.  Everything this CTA will read from global memory is requested here, all loads independent.
  const int ts0 = D.tree_start[t];
  const int nn = D.tree_start[t + 1] - ts0;
  const int32_t *nodes = D.tree_nodes + ts0;
  const int tb = nn * FR;
  int4 *s_rec = (int4 *)(smem_raw + Y.rec);
  __shared__ __align__(8) unsigned long long s_mbar;
  // Tree-local tables (DevSnap::tl_*): a root's rows are contiguous -> one bulk copy per table, issued by one thread,
  // completion counted in bytes on an mbarrier.  Otherwise (odd rows: 16 B alignment) per-thread cp.async gathers.
  const bool bulk = D.tl_nominal != nullptr && (FR & 1) == 0;
  if (bulk) {
    if (tid == 0) mbar_init(&s_mbar, 1);
    __syncthreads();
    if (tid == 0) {
      const int b0 = D.tree_blob_off[t], bn = D.tree_blob_off[t + 1] - b0;  // static block of the tree (multiple of 16 B)
      const unsigned tbytes = (unsigned)tb * 8u;
      mbar_expect_tx(&s_mbar, 4u * tbytes + (unsigned)bn + (unsigned)nn * 16u);
      const size_t r0 = (size_t)ts0 * FR;
      bulk_g2s(s_sub, D.tl_nominal + r0, tbytes, &s_mbar);  // SubtreeQuota = Nominal (updateCohortResourceNode resource_node.go:184-190)
      bulk_g2s(s_bl, D.tl_blimit + r0, tbytes, &s_mbar);
      bulk_g2s(s_lq, D.tl_llimit + r0, tbytes, &s_mbar);    // lending limit for now; localQuota once SubtreeQuota is final
      bulk_g2s(s_u, D.tl_usage + r0, tbytes, &s_mbar);      // ClusterQueue usage, zero rows for cohorts
      bulk_g2s(s_blob, D.tree_blob + b0, (unsigned)bn, &s_mbar);
      bulk_g2s(s_rec, D.cq_rec + ts0, (unsigned)nn * 16u, &s_mbar);
    }
    if (tid == nthreads - 1) *(DevSnap *)(smem_raw + Y.snap) = D;  // bulk of the relocated view (patched below), under the load latency
    {
      unsigned spins = 0;
      while (!mbar_try_wait(&s_mbar, 0)) if (++spins > (1u << 24)) __trap();  // a lost copy must not hang the device
    }
  } else {
  {
    const int b0 = D.tree_blob_off[t], bn = D.tree_blob_off[t + 1] - b0;  // static block of the tree (multiple of 16 B)
    for (int c = tid * 16; c < bn; c += nthreads * 16) cp_async16(s_blob + c, D.tree_blob + b0 + c);
  }
  if ((FR & 1) == 0) {  // rows are 16 B aligned: two cells per request, straight into shared memory
    const int half = tb >> 1;
    for (int c = tid; c < half; c += nthreads) {
      const int i = c << 1;
      const int nd = nodes[row_of(i)];
      const size_t g = (size_t)nd * FR + col_of(i);
      cp_async16(s_sub + i, D.nominal + g);
      cp_async16(s_bl + i, D.blimit + g);
      cp_async16(s_lq + i, D.llimit + g);
      if (nd < D.Q) cp_async16(s_u + i, D.cq_usage + g);
      else { s_u[i] = 0; s_u[i + 1] = 0; }
    }
  } else {
    for (int i = tid; i < tb; i += nthreads) {
      const int nd = nodes[row_of(i)];
      const size_t g = (size_t)nd * FR + col_of(i);
      s_sub[i] = D.nominal[g]; s_bl[i] = D.blimit[g]; s_lq[i] = D.llimit[g];
      s_u[i] = nd < D.Q ? D.cq_usage[g] : 0;
    }
  }
  for (int h = tid; h < nn; h += nthreads) s_rec[h] = D.cq_rec[ts0 + h];
  if (tid == nthreads - 1) *(DevSnap *)(smem_raw + Y.snap) = D;
  cp_async_wait_all();
  __syncthreads();
  }
  for (int h = tid; h < nn; h += nthreads) {  // the head of every ClusterQueue of the tree (record written by k_flat_prep / k_cq_rec)
    const int4 rc = s_rec[h];
    const bool live = ((unsigned)rc.w >> 16) == D.rec_stamp;  // written for this cycle
    n_e[h] = live ? rc.x : -1; n_wl[h] = rc.y; n_ps0[h] = rc.z; n_psn[h] = live ? (rc.w & 0xffff) : 0;
    if (live) {  // the entry's per-cycle records are gathered in phase 2: request their lines now
      auto touch = [](const void *p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); };
      const int wl = rc.y, row = rc.z;
      touch(D.wl_priority + wl); touch(D.wl_ts + wl); touch(D.wl_last_gen + wl);
      if (D.wl_has_qr) touch(D.wl_has_qr + wl);
      if ((rc.w & 0xffff) > 0) {
        touch(D.ps_count + row); touch(D.ps_min_count + row); touch(D.ps_req_mask + row); touch(D.ps_flavor_ok + row);
        touch(D.ps_req + (size_t)row * R); touch(D.ps_last_tried + (size_t)row * R);
        if (D.ps_group) touch(D.ps_group + row);
      }
    }
  }
  __syncthreads();
  KB_FPHASE(0);
  KB_PP(1, 0);
  const TreeBlobHdr *BH = (const TreeBlobHdr *)s_blob;
  const int32_t *b_gid = (const int32_t *)(s_blob + BH->gid), *b_par = (const int32_t *)(s_blob + BH->par), *b_hgt = (const int32_t *)(s_blob + BH->hgt);
  const uint8_t *b_reclaim = s_blob + BH->reclaim;

  // ---- 1. entries of the root in ClusterQueue (= local handle) order + local podset-row numbering (warp 0), and the
  // bottom-up pass of the flat tree for everyone: accumulateFromChild resource_node.go:210-217, children -> root
  // one warp per 32 nodes: ballot + warp scan, then the warps' totals are scanned (chunks of 32 warps, carried)
  {
    const int nw = nthreads >> 5;
    int *w_cnt = s_misc + 4, *w_rows = s_misc + 4 + 32;  // [32] each (misc is 64 + 256 B)
    int cnt_base = 0, rows_base = 0;
    for (int c0 = 0; c0 < nn; c0 += nthreads) {
      const int h = c0 + tid;
      const int e = h < nn ? n_e[h] : -1;
      const int pn = e >= 0 ? n_psn[h] : 0;
      const unsigned m = __ballot_sync(0xffffffffu, e >= 0);
      int incl = pn;  // inclusive scan of the row counts over the lanes
      for (int o = 1; o < 32; o <<= 1) { int v = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += v; }
      if (lane == 31) { w_cnt[warp] = __popc(m); w_rows[warp] = incl; }
      __syncthreads();
      int pc = 0, pr = 0, tc = 0, tr = 0;  // totals of the warps before mine / of all warps of this chunk
      {
        const int wc = lane < nw ? w_cnt[lane] : 0, wr = lane < nw ? w_rows[lane] : 0;
        int ic = wc, ir = wr;
        for (int o = 1; o < 32; o <<= 1) { int a = __shfl_up_sync(0xffffffffu, ic, o), b = __shfl_up_sync(0xffffffffu, ir, o); if (lane >= o) { ic += a; ir += b; } }
        pc = __shfl_sync(0xffffffffu, ic - wc, warp & 31); pr = __shfl_sync(0xffffffffu, ir - wr, warp & 31);
        tc = __shfl_sync(0xffffffffu, ic, 31); tr = __shfl_sync(0xffffffffu, ir, 31);
      }
      if (e >= 0) {
        const int i = cnt_base + pc + __popc(m & ((1u << lane) - 1));
        e_gid[i] = e; e_cq[i] = h; e_ident[i] = i; e_wl[i] = n_wl[h]; e_ps0[i] = n_ps0[h]; e_psn[i] = rows_base + pr + incl - pn;
      }
      cnt_base += tc; rows_base += tr;
      if (c0 + nthreads < nn) __syncthreads();  // w_cnt / w_rows are rewritten by the next chunk
    }
    if (tid == 0) { e_psn[cnt_base] = rows_base; s_misc[0] = cnt_base; s_misc[1] = rows_base; }
  }
  KB_PP(1, 1);
  // the relocated snapshot: every table the shared device functions read, in local numbering.  It lives in shared
  // memory itself (one thread fills it in): ~50 patched pointers would otherwise sit in every thread's stack.
  if (tid == nthreads - 1) {
  DevSnap &L = *(DevSnap *)(smem_raw + Y.snap);
  L.tab_local = 2; L.local_flat = 1; L.ent_gid = e_gid; L.node_gid = b_gid;
  L.parent = b_par; L.height = b_hgt; L.lq = s_lq;
  L.nominal = s_sub;  // only ever read for ClusterQueues: SubtreeQuota == Nominal there (resource_node.go:160-166)
  L.subtree = s_sub; L.usage = s_u; L.avail = s_av; L.potential = s_pot; L.blimit = s_bl; L.fs_over = s_over; L.fs_lend = s_lend;
  L.fair_weight = (const double *)(s_blob + BH->wgt); L.cq_generation = (const i64 *)(s_blob + BH->gen);
  L.cq_within_cq = s_blob + BH->within; L.cq_reclaim_within = b_reclaim; L.cq_borrow_within = s_blob + BH->borrow_w;
  L.cq_when_can_borrow = s_blob + BH->wcb; L.cq_when_can_preempt = s_blob + BH->wcp; L.cq_preference = s_blob + BH->pref;
  L.cq_rg_start = (const int32_t *)(s_blob + BH->rgs); L.rg_res_mask = (const uint32_t *)(s_blob + BH->rgmask);
  L.rg_flavor_start = (const int32_t *)(s_blob + BH->rgfl); L.rg_flavors = (const int32_t *)(s_blob + BH->fl);
  L.heads = e_ident; L.wl_cq = e_cq; L.wl_priority = e_prio; L.wl_ts = e_ts; L.wl_last_gen = e_lg; L.wl_ps_start = e_psn;
  L.wl_has_qr = D.wl_has_qr ? e_qr : nullptr;
  L.ps_req = r_req; L.ps_req_mask = r_mask; L.ps_count = r_count; L.ps_min_count = r_min; L.ps_flavor_ok = r_ok; L.ps_last_tried = r_last;
  L.ps_group = D.ps_group ? r_group : nullptr;
  L.ps_flavor = o_fl; L.ps_res_mode = o_md; L.ps_tried = o_tr; L.ps_count_out = o_cnt;
  L.borrow = e_borrow;
  }
  if (nthreads % FR == 0) {  // a thread stays in one column: private partial sums over its rows
    const int fr = tid % FR, g = tid / FR, G = nthreads / FR;
    i64 dsub = 0, dus = 0;
    for (int h = 1 + g; h < nn; h += G) {
      const int c = h * FR + fr;
      const i64 sub = s_sub[c];
      const i64 lq = local_quota(sub, s_lq[c]);
      dsub += sub - lq;
      dus += imax(0, s_u[c] - lq);
    }
    const int pitch = FR + 1;  // padded: the column-wise read below is conflict free
    if ((size_t)2 * tb >= (size_t)2 * G * pitch) {
      // partials -> scratch (avail / potential are not written yet), one warp per column sums them by shuffles
      i64 *p_sub = s_av, *p_u = s_av + (size_t)G * pitch;
      p_sub[g * pitch + fr] = dsub; p_u[g * pitch + fr] = dus;
      KB_PP(1, 2);
      __syncthreads();
      KB_PP(1, 3);
      for (int c = warp; c < FR; c += nthreads >> 5) {
        i64 a = 0, b = 0;
        for (int k = lane; k < G; k += 32) { a += p_sub[k * pitch + c]; b += p_u[k * pitch + c]; }
        for (int o = 16; o > 0; o >>= 1) { a += __shfl_xor_sync(0xffffffffu, a, o); b += __shfl_xor_sync(0xffffffffu, b, o); }
        if (lane == 0) { s_sub[c] += a; s_u[c] += b; }
      }
    } else {  // small tree: few rows per column, little contention
      if (dsub) atomicAdd((u64 *)&s_sub[fr], (u64)dsub);
      if (dus) atomicAdd((u64 *)&s_u[fr], (u64)dus);
    }
  } else {
    for (int c = FR + tid; c < tb; c += nthreads) {
      const int fr = col_of(c);
      const i64 sub = s_sub[c];
      const i64 lq = local_quota(sub, s_lq[c]);
      if (sub - lq) atomicAdd((u64 *)&s_sub[fr], (u64)(sub - lq));
      const i64 spill = imax(0, s_u[c] - lq);
      if (spill) atomicAdd((u64 *)&s_u[fr], (u64)spill);
    }
  }
  KB_PP(1, 4);
  __syncthreads();
  KB_FPHASE(1);
  KB_PP(1, 5);
  const int n = s_misc[0], nrows = s_misc[1];
  if (n == 0) {
    for (int i = tid; i < tb; i += nthreads) D.usage[(size_t)b_gid[row_of(i)] * FR + col_of(i)] = s_u[i];
    return;
  }
  // ---- 2. per-cycle records of the entries (one hop: the workload / row ids are known), then localQuota and
  // available / potentialAvailable (resource_node.go:104-133) for every cell in one sweep: the root's cells are final
  for (int i = tid; i < n; i += nthreads) {
    // all loads of a record are issued before its first store (read-only path: the compiler may hoist them freely)
    const int wl = e_wl[i];
    const int ps0 = e_ps0[i], l0 = e_psn[i], np = e_psn[i + 1] - l0;
    const int pr = __ldg(D.wl_priority + wl); const i64 ts = __ldg(D.wl_ts + wl), lg = __ldg(D.wl_last_gen + wl);
    const uint8_t qr = D.wl_has_qr ? __ldg(D.wl_has_qr + wl) : 0;
    bool single = np == 1;
    for (int k = 0; k < np; k++) {
      const int row = ps0 + k, l = l0 + k;
      const int cnt = __ldg(D.ps_count + row), mn = __ldg(D.ps_min_count + row); const uint32_t msk = __ldg(D.ps_req_mask + row);
      if ((D.flags & KB_F_PARTIAL_ADMISSION) && mn >= 0 && cnt > mn) single = false;  // the PodSetReducer may run
      const int grp = D.ps_group ? __ldg(D.ps_group + row) : -1; const u64 ok = __ldg(D.ps_flavor_ok + row);
      for (int r0 = 0; r0 < R; r0 += 4) {
        i64 q[4]; int8_t lt[4];
#pragma unroll
        for (int j = 0; j < 4; j++) if (r0 + j < R) { q[j] = __ldg(D.ps_req + (size_t)row * R + r0 + j); lt[j] = __ldg(D.ps_last_tried + (size_t)row * R + r0 + j); }
#pragma unroll
        for (int j = 0; j < 4; j++) if (r0 + j < R) { r_req[(size_t)l * R + r0 + j] = q[j]; r_last[(size_t)l * R + r0 + j] = lt[j]; }
      }
      r_gid[l] = row; r_count[l] = cnt; r_min[l] = mn; r_mask[l] = msk; r_group[l] = grp; r_ok[l] = ok;
    }
    e_prio[i] = pr; e_ts[i] = ts; e_lg[i] = lg; e_qr[i] = qr;
    bool covers_pods = false;  // the ClusterQueue has a resource group with the pods resource (assign_workload_coop)
    if (single && D.pods_res >= 0) {
      const int32_t *rgs = (const int32_t *)(s_blob + BH->rgs); const uint32_t *rgmask = (const uint32_t *)(s_blob + BH->rgmask);
      for (int g = rgs[e_cq[i]]; g < rgs[e_cq[i] + 1]; g++) if (rgmask[g] & (1u << D.pods_res)) covers_pods = true;
    }
    e_flat[i] = (single ? KB_FLAT_WALK : 0) | (covers_pods ? KB_FLAT_PODS : 0);
  }
  KB_PP(1, 6);
  for (int i = tid; i < tb; i += nthreads) {
    const int fr = col_of(i);
    const i64 sub = s_sub[i], u = s_u[i];
    const i64 lq = local_quota(sub, s_lq[i]);
    s_lq[i] = lq;
    if (i < FR) { s_av[i] = sub - u; s_pot[i] = sub; }
    else {
      const i64 bl = s_bl[i];
      i64 pa = s_sub[fr] - s_u[fr], pot = lq + s_sub[fr];
      if (bl != KB_NO_LIMIT) { pa = imin((sub - lq) - imax(0, u - lq) + bl, pa); pot = imin(sub + bl, pot); }
      s_av[i] = imax(0, lq - u) + pa;
      s_pot[i] = pot;
    }
  }
  KB_PP(1, 7);
  __syncthreads();
  KB_FPHASE(2);
  KB_PP(2, 0);
  const DevSnap &L = *(const DevSnap *)(smem_raw + Y.snap);
  // ---- 4. fair sharing inputs (k_fair_prep): over-usage per (ClusterQueue, resource), lendable per (node, resource)
  if (D.flags & KB_F_FAIR_SHARING) {
    const int Fn = D.F;
    const bool r_p2 = (R & (R - 1)) == 0;
    if (FR <= 32 && fr_p2 && r_p2) {  // a row is one aligned segment of a warp: sum over the flavors by shuffles
      const int tb32 = (tb + 31) & ~31;
      for (int i = tid; i < tb32; i += nthreads) {
        i64 lend = 0, over = 0;
        if (i < tb) { lend = s_pot[i]; const i64 o = s_u[i] - s_sub[i]; over = o > 0 ? o : 0; }
        for (int o = R; o < FR; o <<= 1) { lend += __shfl_xor_sync(0xffffffffu, lend, o); over += __shfl_xor_sync(0xffffffffu, over, o); }
        if (i < tb && col_of(i) < R) { const int h = row_of(i); s_lend[h * R + col_of(i)] = lend; s_over[h * R + col_of(i)] = over; }
      }
    } else {
      for (int i = tid; i < nn * R; i += nthreads) {
        const int h = i / R, r = i % R;
        i64 over = 0, lend = 0;
        for (int f = 0; f < Fn; f++) {
          const int c = h * FR + f * R + r;
          lend += s_pot[c];
          const i64 o = s_u[c] - s_sub[c];
          if (o > 0) over += o;
        }
        s_lend[i] = lend; s_over[i] = over;
      }
    }
  }
  KB_PP(2, 1);
  // ---- 5. nominate: KB_FLAT_NG lanes per entry (get_assignments_coop) on the relocated tables.  A round evaluates
  // KB_FLAT_NG flavors of a resource group at once; the walk usually stops in its first round, so fewer lanes per entry
  // mean fewer warps competing for the SM's issue slots at the same chain length.
  {
    const int glane = lane % KB_FLAT_NG, gbase = lane - glane;
    const unsigned gmask = (KB_FLAT_NG == 32 ? 0xffffffffu : ((1u << KB_FLAT_NG) - 1u)) << gbase;
    const int groups = nthreads / KB_FLAT_NG;
    for (int i0 = 0; i0 < n; i0 += groups) {
      const int i = i0 + tid / KB_FLAT_NG;
      if (i < n) {  // whole lane groups take the branch together
        if (e_flat[i] & KB_FLAT_WALK) flat_walk<KB_FLAT_NG>(D, Y, smem_raw, i, gmask, gbase, glane);
        else flat_generic_assign<KB_FLAT_NG>(L, i, gmask, gbase, glane, e_mode, e_borrow);
      }
    }
  }
  KB_PP(2, 2);
  __syncthreads();
  KB_FPHASE(3);
  KB_PP(2, 3);
  // ---- 6. iterator keys (threads of the lower half) | dense request rows (upper half); avail / potential are dead
  i64 *s_q = s_av;    // [n][FR] Assignment.Usage.Quota per entry, absent = -1
  i64 *s_lim = s_pot; // [n][FR] thresholds in iterator order
  const bool fair = (D.flags & KB_F_FAIR_SHARING) != 0;  // every tree is flat here: all entries take the fair flat key
  double *s_ratio = (double *)s_key;                     // [n][4] terms of the DominantResourceShare, in the entry's key slots
  const bool split = fair && R <= 4;
  for (int c = tid; c < n * FR; c += nthreads) s_q[c] = -1;  // row-major: a row per thread would hit one bank 32 ways
  __syncthreads();
  KB_PP(2, 4);
  {
    auto share = [&](int i, int r) { return e_flat[i] & KB_FLAT_WALK ? flat_share_ratio(D, Y, smem_raw, i, r) : entry_share_ratio(L, i, r); };
    const int half = nthreads / 2;
    if (tid < half) {
      if (split) { for (int c = tid; c < n * R; c += half) s_ratio[(size_t)(c / R) * 4 + c % R] = share(c / R, c % R); }  // one division per thread
      else
        for (int i = tid; i < n; i += half) {
          double best = 0.0;
          if (fair) for (int r = 0; r < R; r++) { const double ratio = share(i, r); if (ratio > best) best = ratio; }
          flat_key_finish(D, Y, smem_raw, i, fair, best, s_key + (size_t)i * 4);
        }
    } else {
      for (int i = tid - half; i < n; i += half) {
        if (e_flat[i] & KB_FLAT_WALK) {  // expand_entry: one podset, one cell per assigned resource
          const int l = e_psn[i];
          for (int r = 0; r < R; r++) {
            const int f = o_fl[(size_t)l * R + r];
            if (f >= 0) s_q[(size_t)i * FR + f * R + r] = (e_flat[i] & KB_FLAT_PODS) && r == D.pods_res ? (i64)o_cnt[l] : r_req[(size_t)l * R + r];
          }
        } else expand_entry(L, i, s_q + (size_t)i * FR);
      }
    }
  }
  KB_PP(2, 5);
  if (split) {
    __syncthreads();
    for (int i = tid; i < n; i += nthreads) {
      double best = 0.0;
      for (int r = 0; r < R; r++) { const double ratio = s_ratio[(size_t)i * 4 + r]; if (ratio > best) best = ratio; }
      flat_key_finish(D, Y, smem_raw, i, true, best, s_key + (size_t)i * 4);  // overwrites the entry's own four slots
    }
  }
  KB_PP(2, 6);
  __syncthreads();
  KB_FPHASE(4);
  KB_PP(2, 7); KB_PP(3, 0);
  // ---- 7. position in the iterator order: S lanes share the comparisons of one entry
  {
    int S = 32;
    while (S > 1 && n * S > nthreads) S >>= 1;
    const int per = nthreads / S, sub = tid % S;
    for (int base = 0; base < n; base += per) {
      const int i = base + tid / S;
      const bool act = i < n;
      int cnt = 0;
      if (act) {
        const u64 *mine = s_key + (size_t)i * 4;
        for (int j = sub; j < n; j += S) cnt += key4_less(s_key + (size_t)j * 4, mine) ? 1 : 0;
      }
      for (int o = S >> 1; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
      if (act && sub == 0) { s_sorted[cnt] = i; e_rank[i] = cnt; }
    }
  }
  KB_PP(3, 1);
  __syncthreads();
  // ---- 8. thresholds, stored in iterator order (see flat_ordered_loop)
  for (int c = tid; c < n * FR; c += nthreads) {
    const int pos = row_of(c), fr = col_of(c);
    const int i = s_sorted[pos];
    const i64 q = s_q[(size_t)i * FR + fr];
    const int hq = e_cq[i];
    const int r = hq * FR + fr;
    const i64 u = s_u[r], l = s_lq[r], bl = s_bl[r], sub = s_sub[r];
    const i64 A = imax(0, l - u);
    i64 v = INT64_MAX;  // Fit: threshold on the root usage; Preempt: SubtreeQuota_root - amount added to the root
    const int mode = e_mode[i];
    if (mode == KB_MODE_FIT) {
      if (q > 0) {
        const i64 x = q - A;
        const bool cap_ok = bl == KB_NO_LIMIT || (sub - l) - imax(0, u - l) + bl >= x;
        v = cap_ok ? s_sub[fr] - x : INT64_MIN;
      }
    } else if (mode == KB_MODE_PREEMPT) {
      i64 amt = 0;
      if (q >= 0 && b_reclaim[hq] != KB_POLICY_ANY) {  // quotaResourcesToReserve scheduler.go:530-548
        const i64 rsv = e_borrow[i] > 0 ? (bl == KB_NO_LIMIT ? q : imin(q, sub + bl - u)) : imax(0, imin(q, sub - u));
        amt = rsv > A ? rsv - A : 0;
      }
      v = s_sub[fr] - amt;
    }
    s_lim[c] = v;
    if (fr == 0) m_sorted[pos] = mode;
  }
  KB_PP(3, 2);
  __syncthreads();
  KB_FPHASE(5);
  // ---- 9. the ordered loop
  if (warp == 0) {
    if (FR > 32) flat_ordered_loop<true>(n, FR, lane, s_lim, m_sorted, ok_bits, s_u, s_sub);
    else flat_ordered_loop<false>(n, FR, lane, s_lim, m_sorted, ok_bits, s_u, s_sub);
  }
  __syncthreads();
  KB_FPHASE(6);
  KB_PP(3, 3);
  // ---- 10. ClusterQueue rows of the admitted / reserving entries (cq.AddUsage)
  for (int c = tid; c < n * FR; c += nthreads) {
    const int i = row_of(c), fr = col_of(c);
    const int dec = flat_decision(e_mode[i], ok_bits, e_rank[i]);
    const i64 q = s_q[c];
    const int hq = e_cq[i];
    const int r = hq * FR + fr;
    if (dec == KB_DEC_ASSUMED) { if (q > 0) s_u[r] += q; }
    else if (dec == KB_DEC_PREEMPT_NO_TARGETS && q >= 0 && b_reclaim[hq] != KB_POLICY_ANY) {
      const i64 u = s_u[r], bl = s_bl[r], sub = s_sub[r];
      s_u[r] = u + (e_borrow[i] > 0 ? (bl == KB_NO_LIMIT ? q : imin(q, sub + bl - u)) : imax(0, imin(q, sub - u)));
    }
  }
  KB_PP(3, 4);
  __syncthreads();
  // ---- 11. publish: usage table, decisions, flavor assignment rows
  KB_PP(3, 5);
  if ((FR & 1) == 0) {
    const int half = tb >> 1;
    for (int c = tid; c < half; c += nthreads) {
      const int i = c << 1;
      *(longlong2 *)(D.usage + (size_t)b_gid[row_of(i)] * FR + col_of(i)) = *(const longlong2 *)(s_u + i);
    }
  } else {
    for (int i = tid; i < tb; i += nthreads) D.usage[(size_t)b_gid[row_of(i)] * FR + col_of(i)] = s_u[i];
  }
  KB_PP(3, 6);
  for (int i = tid; i < n; i += nthreads) {
    const int e = e_gid[i];
    D.mode[e] = (uint8_t)e_mode[i]; D.borrow[e] = e_borrow[i]; D.decision[e] = (uint8_t)flat_decision(e_mode[i], ok_bits, e_rank[i]); D.rank[e] = e_rank[i];
    D.tgt_cnt[e] = 0; D.tgt_off[e] = 0;
  }
  if ((R & 3) == 0) {  // rows of R bytes are word aligned in both copies
    const int wpr = R >> 2;
    for (int c = tid; c < nrows * wpr; c += nthreads) {
      const int l = c / wpr, w = c % wpr;
      const size_t dst = (size_t)r_gid[l] * wpr + w, src = (size_t)l * wpr + w;
      ((uint32_t *)D.ps_flavor)[dst] = ((const uint32_t *)o_fl)[src];
      ((uint32_t *)D.ps_res_mode)[dst] = ((const uint32_t *)o_md)[src];
      ((uint32_t *)D.ps_tried)[dst] = ((const uint32_t *)o_tr)[src];
      if (w == 0) D.ps_count_out[r_gid[l]] = o_cnt[l];
    }
  } else {
    for (int l = tid; l < nrows; l += nthreads) {
      const int row = r_gid[l];
      D.ps_count_out[row] = o_cnt[l];
      for (int r = 0; r < R; r++) {
        D.ps_flavor[(size_t)row * R + r] = o_fl[(size_t)l * R + r];
        D.ps_res_mode[(size_t)row * R + r] = o_md[(size_t)l * R + r];
        D.ps_tried[(size_t)row * R + r] = o_tr[(size_t)l * R + r];
      }
    }
  }
  KB_PP(3, 7);
  KB_FPHASE(7);
#undef KB_FPHASE
}
