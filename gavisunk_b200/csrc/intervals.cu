// intervals.cu -- contig-wide connected components of validated SUNK groups -> validated intervals
// (workflow/scripts/process-by-contig_lowmem_AR.py:215-260), interval merge + gap sweep
// (workflow/scripts/get_gaps.py:17-123) and the gap-spanning probability table
// (workflow/scripts/covprob.py:56-100).  SURVEY.md A.6 step 7, A.7, A.8; quirks Q15, Q16.
//
// The reference expands every read into the clique of its validated IDs (:219) and labels
// components (:237); connectivity only needs a chain through the read's IDs, so each validated
// pair is unioned with its predecessor of the same read in a lock-free union-find over the dense
// group index (hook larger root under smaller: the root is the component's first group).
// Multi-GPU: every rank builds its forest; the gathered forests are merged in one pass by unioning g with
// each peer's parent[g].  Intervals come out in (contig, start) order whatever the order of the group table.
#include "common.cuh"
#include <algorithm>

__device__ __forceinline__ u32 guf_find(u32* par, u32 x) {
  u32 p = par[x];
  while (p != x) {
    u32 gp = par[p];
    if (gp != p) par[x] = gp;  // path halving (benign race: only ever points higher up the same tree)
    x = p;
    p = gp;
  }
  return x;
}
__device__ __forceinline__ void guf_union(u32* par, u32 a, u32 b) {
  for (;;) {
    a = guf_find(par, a);
    b = guf_find(par, b);
    if (a == b) return;
    u32 hi = a > b ? a : b, lo = a > b ? b : a;
    if (atomicCAS(&par[hi], hi, lo) == hi) return;
  }
}

__global__ void __launch_bounds__(256) k_iota(u32* p, u64 n) {
  u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = (u32)i;
}
// a read contributes edges only if it has >= 2 validated IDs (`combinations(g['ID'], 2)`, :219)
__global__ void __launch_bounds__(256) k_comp_pairs(const u32* __restrict__ read, const u32* __restrict__ gidx, u64 n, u32* par,
                                                    u8* present) {
  u64 j = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (j == 0 || j >= n) return;
  if (read[j] != read[j - 1]) return;
  u32 a = gidx[j - 1], b = gidx[j];
  present[a] = 1;
  present[b] = 1;
  if (a != b) guf_union(par, a, b);
}
// forest -> every entry points at its root (depth 1): what the peers receive, and what makes their merge cheap
__global__ void __launch_bounds__(256) k_comp_flatten(u32* par, u64 ng) {
  u64 g = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= ng) return;
  u32 r = guf_find(par, (u32)g);
  if (par[g] != r) par[g] = r;  // (only ever moves an entry higher up its own tree)
}
// all peers' forests in one pass: gathered[r * ng + g] = parent of g on rank r
__global__ void __launch_bounds__(256) k_comp_merge_all(const u32* __restrict__ gathered, u32 n_ranks, u32 own, u64 ng, u32* par,
                                                        u8* present) {
  u64 g = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= ng) return;
  for (u32 r = 0; r < n_ranks; r++) {
    if (r == own) continue;
    u32 p = __ldg(gathered + (u64)r * ng + g);
    if (p == (u32)g || p >= ng) continue;
    present[g] = 1;
    present[p] = 1;
    guf_union(par, (u32)g, p);
  }
}
// count / smallest / largest group start per component root.  Neighbouring groups almost always share their root
// (a component is a run of groups along a contig; at 30x a contig is a handful of components), so the lanes of a
// warp are combined per distinct root first: one atomic triple per root and warp instead of per group.
// BY_RANK (group index not in (contig, start) order): also the smallest (contig, start) rank of the members, which
// places the component's interval in the output
template <bool BY_RANK>
__global__ void __launch_bounds__(256) k_comp_stats(u32* par, const u8* __restrict__ present, u64 ng,
                                                    const u32* __restrict__ grp_start, u32* cnt, u32* mn, u32* mx,
                                                    const u32* __restrict__ rank_of, u32* rmn) {
  const u64 g = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  const int lane = threadIdx.x & 31;
  const bool act = g < ng && present[g];
  const u32 r = act ? guf_find(par, (u32)g) : 0xFFFFFFFFu;
  const u32 s = act ? grp_start[g] : 0u;
  u32 q = 0;
  if (BY_RANK) q = act ? rank_of[g] : 0xFFFFFFFFu;
  u32 todo = __ballot_sync(0xFFFFFFFFu, act);
  while (todo) {  // warp-uniform
    const int leader = __ffs(todo) - 1;
    const u32 rl = __shfl_sync(0xFFFFFFFFu, r, leader);
    const bool mine = act && r == rl;
    const u32 m = __ballot_sync(0xFFFFFFFFu, mine);
    const u32 lo = __reduce_min_sync(0xFFFFFFFFu, mine ? s : 0xFFFFFFFFu);
    const u32 hi = __reduce_max_sync(0xFFFFFFFFu, mine ? s : 0u);
    u32 qlo = 0;
    if (BY_RANK) qlo = __reduce_min_sync(0xFFFFFFFFu, mine ? q : 0xFFFFFFFFu);
    if (lane == leader) {
      atomicAdd(&cnt[rl], (u32)__popc(m));
      atomicMin(&mn[rl], lo);
      atomicMax(&mx[rl], hi);
      if (BY_RANK) atomicMin(&rmn[rl], qlo);
    }
    todo &= ~m;
  }
}
__global__ void __launch_bounds__(256) k_iv_write(const u32* __restrict__ excl, const u32* __restrict__ cnt, u64 ng,
                                                  const u32* __restrict__ grp_contig, const u32* __restrict__ mn,
                                                  const u32* __restrict__ mx, u32* iv_contig, u32* iv_start, u32* iv_end) {
  u64 g = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= ng || cnt[g] < 3) return;  // `if len(sunks) <= 2: continue` (:248)
  u32 o = excl[g];
  iv_contig[o] = grp_contig[g];
  iv_start[o] = mn[g];
  iv_end[o] = mx[g];  // end = largest group ID, not +k (Q15)
}
// unsorted group table: every kept component's root at its smallest member rank, so that a scan over rank space
// numbers the intervals in (contig, start) order
__global__ void __launch_bounds__(256) k_iv_slot(const u32* __restrict__ cnt, const u32* __restrict__ rmn, u64 ng, u32* slot) {
  u64 g = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= ng || cnt[g] < 3) return;
  slot[rmn[g]] = (u32)g;
}
__global__ void __launch_bounds__(256) k_iv_write_rank(const u32* __restrict__ excl, const u32* __restrict__ slot, u64 ng,
                                                       const u32* __restrict__ grp_contig, const u32* __restrict__ mn,
                                                       const u32* __restrict__ mx, u32* iv_contig, u32* iv_start, u32* iv_end) {
  u64 q = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= ng) return;
  const u32 g = slot[q];
  if (g == 0xFFFFFFFFu) return;
  u32 o = excl[q];
  iv_contig[o] = grp_contig[g];
  iv_start[o] = mn[g];
  iv_end[o] = mx[g];
}

// singleton forest over the group index, no group present
static int ensure_forest(gvs_ctx* ctx) {
  u64 ng = ctx->n_groups ? ctx->n_groups : 1;
  CKR(gvs_reserve(ctx, ctx->parent, ng * 4));
  CKR(gvs_reserve(ctx, ctx->present, ng));
  LAUNCH(k_iota, (unsigned)cdiv(ng, 256), 256, 0, ctx->parent.as<u32>(), ng);
  CK(cudaMemsetAsync(ctx->present.p, 0, ng, ctx->stream));
  return 0;
}

extern "C" int gvs_components_local(gvs_ctx* ctx, uint32_t** parent_dev) {
  if (!ctx) return GVS_E_ARG;
  if (!ctx->val_ready) return gvs_fail(ctx, GVS_E_STATE, "gvs_components_local before gvs_validate");
  if (!ctx->groups_ready) return gvs_fail(ctx, GVS_E_STATE, "gvs_components_local: no group index");
  CK(cudaSetDevice(ctx->device));
  StageTimer tm(ctx, GVS_ST_COMPONENTS);
  CKR(ensure_forest(ctx));
  u64 n = ctx->n_pairs;
  if (n > 1)
    LAUNCH(k_comp_pairs, (unsigned)cdiv(n, 256), 256, 0, ctx->pair_read.as<u32>(), ctx->pair_gidx.as<u32>(), n,
           ctx->parent.as<u32>(), ctx->present.as<u8>());
  // entries point straight at their roots: the array that crosses GPUs is a depth-1 forest
  if (n > 1) LAUNCH(k_comp_flatten, (unsigned)cdiv(ctx->n_groups ? ctx->n_groups : 1, 256), 256, 0, ctx->parent.as<u32>(), ctx->n_groups);
  ctx->comp_ready = true;
  ctx->iv_ready = false;
  if (parent_dev) *parent_dev = ctx->parent.as<u32>();
  return 0;
}

extern "C" int gvs_components_merge_all(gvs_ctx* ctx, const uint32_t* gathered_dev, uint32_t n_ranks, uint32_t own_rank) {
  if (!ctx || !gathered_dev) return GVS_E_ARG;
  if (!ctx->comp_ready) return gvs_fail(ctx, GVS_E_STATE, "gvs_components_merge_all before gvs_components_local");
  CK(cudaSetDevice(ctx->device));
  StageTimer tm(ctx, GVS_ST_MERGE);
  u64 ng = ctx->n_groups;
  if (ng && n_ranks > 1)
    LAUNCH(k_comp_merge_all, (unsigned)cdiv(ng, 256), 256, 0, gathered_dev, n_ranks, own_rank, ng, ctx->parent.as<u32>(), ctx->present.as<u8>());
  ctx->iv_ready = false;
  return 0;
}

extern "C" int gvs_intervals(gvs_ctx* ctx, uint64_t* n_intervals) {
  if (!ctx) return GVS_E_ARG;
  if (!ctx->comp_ready) return gvs_fail(ctx, GVS_E_STATE, "gvs_intervals before gvs_components_local");
  CK(cudaSetDevice(ctx->device));
  StageTimer tm(ctx, GVS_ST_INTERVALS);
  u64 ng = ctx->n_groups;
  ctx->n_iv = 0;
  if (n_intervals) *n_intervals = 0;
  CKR(gvs_reserve(ctx, ctx->comp_cnt, (ng ? ng : 1) * 4));
  CKR(gvs_reserve(ctx, ctx->comp_min, (ng ? ng : 1) * 4));
  CKR(gvs_reserve(ctx, ctx->comp_max, (ng ? ng : 1) * 4));
  CKR(gvs_reserve(ctx, ctx->flags_b, (ng ? ng : 1) * 4));
  if (ng == 0) {
    ctx->iv_ready = true;
    return 0;
  }
  // intervals come out in (contig, start) order, as the reference's bed rows and gvs_gaps want them.  The root of a
  // component is its smallest group index, which is its leftmost group when the group table is sorted (a built
  // database, a sorted kmer.loc): then the roots are written in index order.  Otherwise (groups from rows, an
  // unsorted kmer.loc) each component is placed by the smallest (contig, start) rank of its members.
  CKR(gvs_ensure_rank(ctx));
  const bool by_rank = !ctx->rank_identity;
  CK(cudaMemsetAsync(ctx->comp_cnt.p, 0, ng * 4, ctx->stream));
  CK(cudaMemsetAsync(ctx->comp_min.p, 0xFF, ng * 4, ctx->stream));
  CK(cudaMemsetAsync(ctx->comp_max.p, 0, ng * 4, ctx->stream));
  const u32* cnt = ctx->comp_cnt.as<u32>();
  u32* ex = ctx->flags_b.as<u32>();
  u32 ni = 0;
  if (!by_rank) {
    LAUNCH(k_comp_stats<false>, (unsigned)cdiv(ng, 256), 256, 0, ctx->parent.as<u32>(), ctx->present.as<u8>(), ng, ctx->grp_start.as<u32>(),
           ctx->comp_cnt.as<u32>(), ctx->comp_min.as<u32>(), ctx->comp_max.as<u32>(), nullptr, nullptr);
    auto f = [cnt] __device__(u64 g) -> u32 { return cnt[g] >= 3 ? 1u : 0u; };
    auto g2 = [ex] __device__(u64 g, u32 e, u32 v) { ex[g] = e; };
    CKR(scan_total(ctx, ng, f, g2, OpSum(), &ni));
  } else {
    CKR(gvs_reserve(ctx, ctx->comp_rank, ng * 2 * 4));
    u32 *rmn = ctx->comp_rank.as<u32>(), *slot = rmn + ng;
    CK(cudaMemsetAsync(rmn, 0xFF, ng * 2 * 4, ctx->stream));
    LAUNCH(k_comp_stats<true>, (unsigned)cdiv(ng, 256), 256, 0, ctx->parent.as<u32>(), ctx->present.as<u8>(), ng, ctx->grp_start.as<u32>(),
           ctx->comp_cnt.as<u32>(), ctx->comp_min.as<u32>(), ctx->comp_max.as<u32>(), ctx->rank_of.as<u32>(), rmn);
    LAUNCH(k_iv_slot, (unsigned)cdiv(ng, 256), 256, 0, cnt, rmn, ng, slot);
    auto f = [slot] __device__(u64 q) -> u32 { return slot[q] != 0xFFFFFFFFu ? 1u : 0u; };
    auto g2 = [ex] __device__(u64 q, u32 e, u32 v) { ex[q] = e; };
    CKR(scan_total(ctx, ng, f, g2, OpSum(), &ni));
  }
  CKR(gvs_reserve(ctx, ctx->iv_contig, (u64)ni * 4));
  CKR(gvs_reserve(ctx, ctx->iv_start, (u64)ni * 4));
  CKR(gvs_reserve(ctx, ctx->iv_end, (u64)ni * 4));
  if (ni && !by_rank)
    LAUNCH(k_iv_write, (unsigned)cdiv(ng, 256), 256, 0, ex, cnt, ng, ctx->grp_contig.as<u32>(), ctx->comp_min.as<u32>(),
           ctx->comp_max.as<u32>(), ctx->iv_contig.as<u32>(), ctx->iv_start.as<u32>(), ctx->iv_end.as<u32>());
  if (ni && by_rank)
    LAUNCH(k_iv_write_rank, (unsigned)cdiv(ng, 256), 256, 0, ex, ctx->comp_rank.as<u32>() + ng, ng, ctx->grp_contig.as<u32>(),
           ctx->comp_min.as<u32>(), ctx->comp_max.as<u32>(), ctx->iv_contig.as<u32>(), ctx->iv_start.as<u32>(), ctx->iv_end.as<u32>());
  ctx->n_iv = ni;
  ctx->iv_ready = true;
  ctx->gaps_ready = false;
  if (n_intervals) *n_intervals = ni;
  return 0;
}

extern "C" int gvs_intervals_get(gvs_ctx* ctx, uint32_t* contig, uint32_t* start, uint32_t* end) {
  if (!ctx) return GVS_E_ARG;
  if (!ctx->iv_ready) return gvs_fail(ctx, GVS_E_STATE, "gvs_intervals_get before gvs_intervals");
  CK(cudaSetDevice(ctx->device));
  u64 n = ctx->n_iv;
  if (n == 0) return 0;
  if (contig) CK(cudaMemcpyAsync(contig, ctx->iv_contig.p, n * 4, cudaMemcpyDeviceToHost, ctx->stream));
  if (start) CK(cudaMemcpyAsync(start, ctx->iv_start.p, n * 4, cudaMemcpyDeviceToHost, ctx->stream));
  if (end) CK(cudaMemcpyAsync(end, ctx->iv_end.p, n * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return 0;
}

// ---------------------------------------------------------------------------------------------
// gaps (get_gaps.py): intervals are sorted by (contig, start); a gap opens wherever an interval
// starts beyond the running max end of its contig: (contig, prev_end, start - 1) (:60-61)
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_contig_has_iv(const u32* __restrict__ iv_contig, u64 n, u8* has) {
  u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) has[iv_contig[i]] = 1;
}

extern "C" int gvs_gaps(gvs_ctx* ctx, const uint32_t* contig_len, uint64_t* n_gaps, uint64_t* n_nodata) {
  if (!ctx) return GVS_E_ARG;
  if (!ctx->iv_ready) return gvs_fail(ctx, GVS_E_STATE, "gvs_gaps before gvs_intervals");
  CK(cudaSetDevice(ctx->device));
  StageTimer tm(ctx, GVS_ST_INTERVALS);
  u64 n = ctx->n_iv;
  u32 nc = ctx->n_contigs;
  (void)contig_len;  // lengths are only needed by the caller for the nodata rows (contig, 0, len)
  CKR(gvs_reserve(ctx, ctx->gap_contig, (n ? n : 1) * 4));
  CKR(gvs_reserve(ctx, ctx->gap_start, (n ? n : 1) * 4));
  CKR(gvs_reserve(ctx, ctx->gap_end, (n ? n : 1) * 4));
  CKR(gvs_reserve(ctx, ctx->nodata_contig, (nc ? nc : 1) * 4));
  CKR(gvs_reserve(ctx, ctx->flags_a, (nc ? nc : 1) + n * 8 + 64));
  u8* has = ctx->flags_a.as<u8>();
  CK(cudaMemsetAsync(has, 0, nc ? nc : 1, ctx->stream));
  ctx->n_gaps = 0;
  ctx->n_nodata = 0;
  const u32 *ivc = ctx->iv_contig.as<u32>(), *ivs = ctx->iv_start.as<u32>(), *ive = ctx->iv_end.as<u32>();
  if (n) {
    LAUNCH(k_contig_has_iv, (unsigned)cdiv(n, 256), 256, 0, ivc, n, has);
    // running max end per contig (segmented prefix max through the packed key contig:end)
    u64* pm = (u64*)(ctx->flags_a.as<u8>() + (((nc ? nc : 1) + 63) & ~63ull));
    {
      auto f = [ivc, ive] __device__(u64 i) -> u64 { return ((u64)(ivc[i] + 1) << 32) | ive[i]; };
      auto g = [pm] __device__(u64 i, u64 ex, u64 v) { pm[i] = ex; };
      CKR((device_scan<u64>(ctx, n, f, g, OpMax(), (u64*)nullptr)));
    }
    u32 *gc = ctx->gap_contig.as<u32>(), *gs = ctx->gap_start.as<u32>(), *ge = ctx->gap_end.as<u32>();
    u32 ngap = 0;
    {
      // pyranges merge joins overlapping and book-ended intervals: a new run starts iff start > max end
      auto f = [ivc, ivs, pm] __device__(u64 i) -> u32 {
        u64 e = pm[i];
        return ((u32)(e >> 32) == ivc[i] + 1 && ivs[i] > (u32)e) ? 1u : 0u;
      };
      auto g = [ivc, ivs, pm, gc, gs, ge] __device__(u64 i, u32 ex, u32 v) {
        if (v) {
          gc[ex] = ivc[i];
          gs[ex] = (u32)pm[i];
          ge[ex] = ivs[i] - 1;
        }
      };
      CKR(scan_total(ctx, n, f, g, OpSum(), &ngap));
    }
    ctx->n_gaps = ngap;
  }
  {
    u32* nd = ctx->nodata_contig.as<u32>();
    auto f = [has] __device__(u64 c) -> u32 { return has[c] ? 0u : 1u; };
    auto g = [nd] __device__(u64 c, u32 ex, u32 v) { if (v) nd[ex] = (u32)c; };
    u32 nn = 0;
    CKR(scan_total(ctx, nc, f, g, OpSum(), &nn));
    ctx->n_nodata = nn;
  }
  ctx->gaps_ready = true;
  if (n_gaps) *n_gaps = ctx->n_gaps;
  if (n_nodata) *n_nodata = ctx->n_nodata;
  return 0;
}

extern "C" int gvs_gaps_get(gvs_ctx* ctx, uint32_t* contig, uint32_t* start, uint32_t* end, uint32_t* nodata_contig) {
  if (!ctx) return GVS_E_ARG;
  if (!ctx->gaps_ready) return gvs_fail(ctx, GVS_E_STATE, "gvs_gaps_get before gvs_gaps");
  CK(cudaSetDevice(ctx->device));
  u64 n = ctx->n_gaps;
  if (n && contig) CK(cudaMemcpyAsync(contig, ctx->gap_contig.p, n * 4, cudaMemcpyDeviceToHost, ctx->stream));
  if (n && start) CK(cudaMemcpyAsync(start, ctx->gap_start.p, n * 4, cudaMemcpyDeviceToHost, ctx->stream));
  if (n && end) CK(cudaMemcpyAsync(end, ctx->gap_end.p, n * 4, cudaMemcpyDeviceToHost, ctx->stream));
  if (ctx->n_nodata && nodata_contig)
    CK(cudaMemcpyAsync(nodata_contig, ctx->nodata_contig.p, ctx->n_nodata * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return 0;
}

// intervals read from bed_files/*.bed instead of computed here (input of get_gaps.py:30): sorted by
// (contig, start) on the way in, like pyranges does before merging
extern "C" int gvs_intervals_set(gvs_ctx* ctx, const uint32_t* contig, const uint32_t* start, const uint32_t* end, uint64_t n,
                                 uint32_t n_contigs) {
  if (!ctx || (n && (!contig || !start || !end))) return GVS_E_ARG;
  CK(cudaSetDevice(ctx->device));
  std::vector<u64> order(n);
  for (u64 i = 0; i < n; i++) {
    if (contig[i] >= n_contigs) return gvs_fail(ctx, GVS_E_ARG, "gvs_intervals_set: contig id %u out of range", contig[i]);
    order[i] = i;
  }
  std::stable_sort(order.begin(), order.end(), [&](u64 a, u64 b) {
    return contig[a] != contig[b] ? contig[a] < contig[b] : start[a] < start[b];
  });
  std::vector<u32> c(n), s(n), e(n);
  for (u64 i = 0; i < n; i++) { c[i] = contig[order[i]]; s[i] = start[order[i]]; e[i] = end[order[i]]; }
  ctx->n_contigs = n_contigs;
  CKR(to_dev(ctx, ctx->iv_contig, c.data(), n));
  CKR(to_dev(ctx, ctx->iv_start, s.data(), n));
  CKR(to_dev(ctx, ctx->iv_end, e.data(), n));
  CK(cudaStreamSynchronize(ctx->stream));
  ctx->n_iv = n;
  ctx->iv_ready = true;
  ctx->gaps_ready = false;
  return 0;
}

// ---------------------------------------------------------------------------------------------
// covprob table (covprob.py:56-60,86-100), float64
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) k_covprob(const i64* __restrict__ kbp, const i64* __restrict__ cnt, u32 n_bins, double G,
                                                 double pn, double* table) {
  u32 I = blockIdx.x * blockDim.x + threadIdx.x;
  if (I >= 3500) return;
  if (I == 0) { table[0] = 1.0; return; }  // covprobdict[0] = 1.0 (:100)
  double cum = 1.0;
  double pn2 = pn * pn;  // (pn**2)
  for (u32 b = 0; b < n_bins; b++) {
    double Lk = (double)kbp[b];
    double prob;
    if ((double)I > Lk) prob = 1.0;
    else prob = pow(1.0 - (((Lk - (double)I) / G) * pn2), (double)cnt[b]);  // (:56-60)
    cum = cum * prob;
  }
  table[I] = 1.0 - cum;
}

extern "C" int gvs_covprob_table(gvs_ctx* ctx, const int64_t* kbp, const int64_t* cnt, uint32_t n_bins, double genome_kbp,
                                 double pn, double* table3500) {
  if (!ctx || !table3500 || (n_bins && (!kbp || !cnt))) return GVS_E_ARG;
  CK(cudaSetDevice(ctx->device));
  DevBuf dk, dc, dt;
  int rc = to_dev(ctx, dk, kbp, n_bins);
  if (!rc) rc = to_dev(ctx, dc, cnt, n_bins);
  if (!rc) rc = gvs_reserve(ctx, dt, 3500 * 8);
  if (!rc) {
    k_covprob<<<(3500 + 127) / 128, 128, 0, ctx->stream>>>(dk.as<i64>(), dc.as<i64>(), n_bins, genome_kbp, pn, dt.as<double>());
    ctx->launches++;
    if (cudaGetLastError() != cudaSuccess) rc = gvs_fail(ctx, GVS_E_CUDA, "k_covprob launch failed");
  }
  if (!rc && cudaMemcpyAsync(table3500, dt.p, 3500 * 8, cudaMemcpyDeviceToHost, ctx->stream) != cudaSuccess)
    rc = gvs_fail(ctx, GVS_E_CUDA, "covprob D2H failed");
  cudaStreamSynchronize(ctx->stream);
  gvs_release(dk); gvs_release(dc); gvs_release(dt);
  return rc;
}

// ---------------------------------------------------------------------------------------------
// covprob per-gap lookup (covprob.py:35-40,109-131) and slop_gaps (tagONT.smk:249)
// ---------------------------------------------------------------------------------------------
// groups = first row of every (contig, group) of kmer.loc in FILE order, which is (contig, start) order
// (defineSUNKs.smk:101-126 sorts it).  dist[i] = max(id[i] - id[i-1], 0) with dist[0] = id[0]; the diff
// runs across contig boundaries exactly like pandas' Series.diff on the concatenated file (:39-40).
__global__ void __launch_bounds__(128) k_covprob_gaps(const u32* __restrict__ g_contig, const u32* __restrict__ g_id, u64 ng,
                                                      const u32* __restrict__ gap_contig, const i64* __restrict__ gap_start,
                                                      const i64* __restrict__ gap_end, u64 n_gaps,
                                                      const double* __restrict__ table, i64* max_gap, double* prob, u32* err) {
  u64 t = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_gaps) return;
  const u32 c = gap_contig[t];
  const i64 lo_id = gap_start[t] - 2, hi_id = gap_end[t] + 2;  // ID > xmin-2 and ID < xmax+2 (:115)
  // first group with (contig, id) > (c, lo_id)
  u64 lo = 0, hi = ng;
  while (lo < hi) {
    u64 mid = (lo + hi) >> 1;
    u32 mc = g_contig[mid];
    bool le = mc < c || (mc == c && (i64)g_id[mid] <= lo_id);
    if (le) lo = mid + 1; else hi = mid;
  }
  i64 best = -1;
  for (u64 i = lo; i < ng && g_contig[i] == c && (i64)g_id[i] < hi_id; i++) {
    i64 d = i == 0 ? (i64)g_id[0] : (i64)g_id[i] - (i64)g_id[i - 1];
    if (d < 0) d = 0;
    if (d > best) best = d;
  }
  max_gap[t] = best;
  if (best < 0) {  // no group in range: the reference dies on int(nan)
    atomicOr(err, 1u);
    prob[t] = 0.0;
    return;
  }
  i64 kb = best / 1000;  // int(x/1000) (:130)
  if (kb >= 3500) {      // KeyError in covprobsdict
    atomicOr(err, 2u);
    prob[t] = 0.0;
    return;
  }
  prob[t] = table[kb];
}

extern "C" int gvs_covprob_gaps(gvs_ctx* ctx, const uint32_t* grp_contig, const uint32_t* grp_id, uint64_t n_groups,
                                const uint32_t* gap_contig, const int64_t* gap_start, const int64_t* gap_end, uint64_t n_gaps,
                                const double* table3500, int64_t* max_gap, double* covprob) {
  if (!ctx || !table3500 || (n_groups && (!grp_contig || !grp_id)) || (n_gaps && (!gap_contig || !gap_start || !gap_end || !max_gap || !covprob)))
    return GVS_E_ARG;
  if (n_gaps == 0) return 0;
  CK(cudaSetDevice(ctx->device));
  DevBuf gc, gi, pc, ps, pe, tb, mg, pr;
  u32* err = counter(ctx, CNT_COVPROB_ERR);
  int rc = to_dev(ctx, gc, grp_contig, n_groups);
  if (!rc) rc = to_dev(ctx, gi, grp_id, n_groups);
  if (!rc) rc = to_dev(ctx, pc, gap_contig, n_gaps);
  if (!rc) rc = to_dev(ctx, ps, gap_start, n_gaps);
  if (!rc) rc = to_dev(ctx, pe, gap_end, n_gaps);
  if (!rc) rc = to_dev(ctx, tb, table3500, 3500);
  if (!rc) rc = gvs_reserve(ctx, mg, n_gaps * 8);
  if (!rc) rc = gvs_reserve(ctx, pr, n_gaps * 8);
  u32 herr = 0;
  if (!rc) {
    cudaMemsetAsync(err, 0, 4, ctx->stream);
    if (n_groups > 1) {
      k_groups_sorted<<<(unsigned)cdiv(n_groups, 256), 256, 0, ctx->stream>>>(gc.as<u32>(), gi.as<u32>(), n_groups, err);
      ctx->launches++;
    }
    k_covprob_gaps<<<(unsigned)cdiv(n_gaps, 128), 128, 0, ctx->stream>>>(gc.as<u32>(), gi.as<u32>(), n_groups, pc.as<u32>(), ps.as<i64>(),
                                                                         pe.as<i64>(), n_gaps, tb.as<double>(), mg.as<i64>(), pr.as<double>(), err);
    ctx->launches++;
    if (cudaGetLastError() != cudaSuccess) rc = gvs_fail(ctx, GVS_E_CUDA, "k_covprob_gaps launch failed");
  }
  if (!rc) rc = read_dev(ctx, err, &herr);
  if (!rc && cudaMemcpyAsync(max_gap, mg.p, n_gaps * 8, cudaMemcpyDeviceToHost, ctx->stream) != cudaSuccess) rc = gvs_fail(ctx, GVS_E_CUDA, "D2H failed");
  if (!rc && cudaMemcpyAsync(covprob, pr.p, n_gaps * 8, cudaMemcpyDeviceToHost, ctx->stream) != cudaSuccess) rc = gvs_fail(ctx, GVS_E_CUDA, "D2H failed");
  cudaStreamSynchronize(ctx->stream);
  gvs_release(gc); gvs_release(gi); gvs_release(pc); gvs_release(ps); gvs_release(pe); gvs_release(tb); gvs_release(mg); gvs_release(pr);
  if (rc) return rc;
  if (herr & 4u) return gvs_fail(ctx, GVS_E_ARG, "gvs_covprob_gaps: group rows are not in (contig, start) order (kmer.loc must be sorted)");
  if (herr & 1u) return gvs_fail(ctx, GVS_E_KEYERROR, "ValueError: a gap has no SUNK group within [start-2, end+2] (covprob.py:118)");
  if (herr & 2u) return gvs_fail(ctx, GVS_E_KEYERROR, "KeyError: max_gap >= 3500 kbp has no covprob entry (covprob.py:130)");
  return 0;
}

// bedtools slop -b B clipped to [0, contig length] (tagONT.smk:249)
__global__ void __launch_bounds__(256) k_slop(const u32* __restrict__ contig, const u32* __restrict__ contig_len, u64 n, i64 b, i64* start,
                                              i64* end) {
  u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  i64 L = contig_len[contig[i]];
  i64 s = start[i] - b, e = end[i] + b;
  start[i] = s < 0 ? 0 : (s > L ? L : s);
  end[i] = e > L ? L : (e < 0 ? 0 : e);
}
extern "C" int gvs_slop(gvs_ctx* ctx, const uint32_t* contig, int64_t* start, int64_t* end, uint64_t n, const uint32_t* contig_len,
                        uint32_t n_contigs, int64_t b) {
  if (!ctx || (n && (!contig || !start || !end || !contig_len))) return GVS_E_ARG;
  if (n == 0) return 0;
  CK(cudaSetDevice(ctx->device));
  for (u64 i = 0; i < n; i++)
    if (contig[i] >= n_contigs) return gvs_fail(ctx, GVS_E_ARG, "gvs_slop: contig id %u out of range", contig[i]);
  DevBuf dc, dl, ds, de;
  int rc = to_dev(ctx, dc, contig, n);
  if (!rc) rc = to_dev(ctx, dl, contig_len, (size_t)n_contigs);
  if (!rc) rc = to_dev(ctx, ds, start, n);
  if (!rc) rc = to_dev(ctx, de, end, n);
  if (!rc) {
    k_slop<<<(unsigned)cdiv(n, 256), 256, 0, ctx->stream>>>(dc.as<u32>(), dl.as<u32>(), n, b, ds.as<i64>(), de.as<i64>());
    ctx->launches++;
    if (cudaGetLastError() != cudaSuccess) rc = gvs_fail(ctx, GVS_E_CUDA, "k_slop launch failed");
  }
  if (!rc && cudaMemcpyAsync(start, ds.p, n * 8, cudaMemcpyDeviceToHost, ctx->stream) != cudaSuccess) rc = gvs_fail(ctx, GVS_E_CUDA, "D2H failed");
  if (!rc && cudaMemcpyAsync(end, de.p, n * 8, cudaMemcpyDeviceToHost, ctx->stream) != cudaSuccess) rc = gvs_fail(ctx, GVS_E_CUDA, "D2H failed");
  cudaStreamSynchronize(ctx->stream);
  gvs_release(dc); gvs_release(dl); gvs_release(ds); gvs_release(de);
  return rc;
}
