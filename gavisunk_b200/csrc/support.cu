// support.cu -- support tracks of the validated reads: one placement per read, the number of placements over
// every base (runs of equal depth) -- what a pile-up plot shows, as text a genome browser loads.  No reference
// counterpart: the reference only draws matplotlib plots (viz.py, viz_detailed.py).
//
// Everything works on the dense group index.  A placement spans [smallest, largest) validated ID of a read and
// every ID is a group start, so the depth is constant between consecutive group starts of a contig: a difference
// array over the groups in (contig, start) order -- their rank -- and one prefix sum give it, without sorting any
// coordinates.  The rank is the identity for a built database and for a sorted kmer.loc (checked on the device);
// otherwise (rows without a database: groups in first-appearance order; an unsorted .loc) it is computed once
// per group table by a bitonic sort of the (contig, start) keys and cached until the table changes.
#include "common.cuh"

// ---------------------------------------------------------------------------------------------
// group rank
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_rank_keys(const u32* __restrict__ gc, const u32* __restrict__ gs, u64 ng, u64 n2, u64* key,
                                                   u32* val) {
  u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n2) return;
  key[i] = i < ng ? (((u64)gc[i] << 32) | gs[i]) : ~0ull;  // (contig, start) of a group is unique
  val[i] = (u32)i;
}
__global__ void __launch_bounds__(256) k_bitonic(u64* key, u32* val, u64 n2, u64 j, u64 k) {
  u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n2) return;
  u64 l = i ^ j;
  if (l <= i) return;
  const u64 a = key[i], b = key[l];
  if ((i & k) == 0 ? a > b : a < b) {
    key[i] = b;
    key[l] = a;
    u32 t = val[i];
    val[i] = val[l];
    val[l] = t;
  }
}
__global__ void __launch_bounds__(256) k_rank_of(const u32* __restrict__ rank_grp, u64 ng, u32* rank_of) {
  u64 r = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (r < ng) rank_of[rank_grp[r]] = (u32)r;
}

static int rank_sort(gvs_ctx* ctx, DevBuf& key) {
  const u64 ng = ctx->n_groups, n2 = next_pow2(ng);
  CKR(gvs_reserve(ctx, key, n2 * 8));
  CKR(gvs_reserve(ctx, ctx->rank_grp, n2 * 4));
  CKR(gvs_reserve(ctx, ctx->rank_of, ng * 4));
  const unsigned grid = (unsigned)cdiv(n2, 256);
  LAUNCH(k_rank_keys, grid, 256, 0, ctx->grp_contig.as<u32>(), ctx->grp_start.as<u32>(), ng, n2, key.as<u64>(), ctx->rank_grp.as<u32>());
  for (u64 k = 2; k <= n2; k <<= 1)
    for (u64 j = k >> 1; j > 0; j >>= 1) LAUNCH(k_bitonic, grid, 256, 0, key.as<u64>(), ctx->rank_grp.as<u32>(), n2, j, k);
  LAUNCH(k_rank_of, (unsigned)cdiv(ng, 256), 256, 0, ctx->rank_grp.as<u32>(), ng, ctx->rank_of.as<u32>());
  CK(cudaStreamSynchronize(ctx->stream));
  return 0;
}

int gvs_check_group_order(gvs_ctx* ctx) {
  const u64 ng = ctx->n_groups;
  u32 h = 0;
  if (ng > 1) {
    u32* err = counter(ctx, CNT_ORDER_ERR);
    CK(cudaMemsetAsync(err, 0, 4, ctx->stream));
    LAUNCH(k_groups_sorted, (unsigned)cdiv(ng, 256), 256, 0, ctx->grp_contig.as<u32>(), ctx->grp_start.as<u32>(), ng, err);
    CKR(read_dev(ctx, err, &h));
  }
  ctx->rank_identity = (h & 4u) == 0;
  ctx->order_gen = ctx->grp_gen;
  return 0;
}

int gvs_ensure_rank(gvs_ctx* ctx) {
  if (ctx->rank_gen == ctx->grp_gen) return 0;
  if (ctx->order_gen != ctx->grp_gen) CKR(gvs_check_group_order(ctx));
  if (!ctx->rank_identity) {
    DevBuf key;
    int rc = rank_sort(ctx, key);
    cudaStreamSynchronize(ctx->stream);
    gvs_release(key);
    CKR(rc);
  }
  ctx->rank_gen = ctx->grp_gen;
  return 0;
}

// ---------------------------------------------------------------------------------------------
// placements: one warp per segment (read) of gvs_validate
// ---------------------------------------------------------------------------------------------
struct PlaceParams {
  const u32 *seg_cnt, *seg_off;                    // validated IDs per segment and their offset in the pairs
  const u32 *p_group, *p_gidx;                     // compacted pairs
  const u8* orient;
  u32 n_seg;
  const u32* rank_of;                              // null: rank = group index
  i32* diff;
  uint4* tmp;                                      // per placed segment: (start, end, n_ids, strand)
};

__global__ void __launch_bounds__(256) k_place(const PlaceParams P) {
  const u32 s = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (s >= P.n_seg) return;
  const u32 c = P.seg_cnt[s];
  if (c < 2) return;  // the validated IDs of a read are distinct vertices: c is their count
  const u32 o = P.seg_off[s];
  u64 mn = ~0ull, mx = 0;  // (ID << 32 | group index)
  for (u32 i = lane; i < c; i += 32) {
    const u64 kv = ((u64)P.p_group[o + i] << 32) | P.p_gidx[o + i];
    mn = kv < mn ? kv : mn;
    mx = kv > mx ? kv : mx;
  }
  for (int d = 16; d; d >>= 1) {
    const u64 a = __shfl_xor_sync(0xFFFFFFFFu, mn, d), b = __shfl_xor_sync(0xFFFFFFFFu, mx, d);
    mn = a < mn ? a : mn;
    mx = b > mx ? b : mx;
  }
  if (lane == 0) {
    const u32 g0 = (u32)mn, g1 = (u32)mx;
    atomicAdd(&P.diff[P.rank_of ? P.rank_of[g0] : g0], 1);
    atomicAdd(&P.diff[P.rank_of ? P.rank_of[g1] : g1], -1);
    P.tmp[s] = make_uint4((u32)(mn >> 32), (u32)(mx >> 32), c, P.orient[s]);
  }
}

extern "C" int gvs_placements(gvs_ctx* ctx, uint64_t* n, int32_t** diff_dev) {
  if (!ctx) return GVS_E_ARG;
  if (!ctx->val_ready) return gvs_fail(ctx, GVS_E_STATE, "gvs_placements before gvs_validate");
  if (!ctx->groups_ready) return gvs_fail(ctx, GVS_E_STATE, "gvs_placements: no group index");
  CK(cudaSetDevice(ctx->device));
  StageTimer tm(ctx, GVS_ST_SUPPORT);
  ctx->pl.ready = ctx->sup.ready = false;
  ctx->pl.n = 0;
  if (n) *n = 0;
  CKR(gvs_ensure_rank(ctx));
  const u64 ng = ctx->n_groups;
  CKR(gvs_reserve(ctx, ctx->sup_diff, (ng ? ng : 1) * 4));
  CK(cudaMemsetAsync(ctx->sup_diff.p, 0, (ng ? ng : 1) * 4, ctx->stream));
  const u64 n_seg = ctx->n_kseg;
  if (ctx->n_pairs) {
    const u32 *seg_cnt = ctx->val_seg_cnt, *seg_off = ctx->val_seg_off;
    CKR(gvs_reserve(ctx, ctx->pl_tmp, n_seg * 16));
    PlaceParams P;
    P.seg_cnt = seg_cnt; P.seg_off = seg_off;
    P.p_group = ctx->pair_group.as<u32>(); P.p_gidx = ctx->pair_gidx.as<u32>();
    P.orient = ctx->seg_orient.as<u8>();
    P.n_seg = (u32)n_seg;
    P.rank_of = ctx->rank_identity ? nullptr : ctx->rank_of.as<u32>();
    P.diff = ctx->sup_diff.as<i32>();
    P.tmp = ctx->pl_tmp.as<uint4>();
    LAUNCH(k_place, (unsigned)cdiv(n_seg * 32, 256), 256, 0, P);
    CKR(rec_reserve(ctx, ctx->pl, 5, n_seg));
    CKR(gvs_reserve(ctx, ctx->pl_strand, n_seg));
    const u32 *prd = ctx->pair_read.as<u32>(), *pct = ctx->pair_contig.as<u32>();
    const uint4* tmp = ctx->pl_tmp.as<uint4>();
    u32 *o_read = ctx->pl.col(0), *o_contig = ctx->pl.col(1), *o_start = ctx->pl.col(2), *o_end = ctx->pl.col(3), *o_nids = ctx->pl.col(4);
    u8* o_strand = ctx->pl_strand.as<u8>();
    auto f = [seg_cnt] __device__(u64 s) -> u32 { return seg_cnt[s] >= 2 ? 1u : 0u; };
    auto g = [=] __device__(u64 s, u32 ex, u32 v) {
      if (!v) return;
      const u32 o = seg_off[s];
      const uint4 t = tmp[s];
      o_read[ex] = prd[o];
      o_contig[ex] = pct[o];
      o_start[ex] = t.x;
      o_end[ex] = t.y;
      o_nids[ex] = t.z;
      o_strand[ex] = (u8)t.w;
    };
    u32 np = 0;
    CKR(scan_total(ctx, n_seg, f, g, OpSum(), &np));
    ctx->pl.n = np;
  }
  ctx->pl.ready = true;
  if (n) *n = ctx->pl.n;
  if (diff_dev) *diff_dev = ctx->sup_diff.as<i32>();
  return 0;
}

extern "C" int gvs_placements_get(gvs_ctx* ctx, uint32_t* read_idx, uint32_t* contig, uint32_t* start, uint32_t* end, uint32_t* n_ids,
                                  uint8_t* strand) {
  if (!ctx) return GVS_E_ARG;
  if (ctx->pl.ready && ctx->pl.n && strand) {  // (u8: queued before the u32 columns, whose getter waits for both)
    CK(cudaSetDevice(ctx->device));
    CK(cudaMemcpyAsync(strand, ctx->pl_strand.p, ctx->pl.n, cudaMemcpyDeviceToHost, ctx->stream));
  }
  return rec_get(ctx, ctx->pl, "gvs_placements_get before gvs_placements", {read_idx, contig, start, end, n_ids});
}

// ---------------------------------------------------------------------------------------------
// runs of equal per-group values: support depth (one value), discordance counts (three, discordance.cu).  Per contig:
// a head run from 0 (all values 0) unless the first group starts at 0, then one run per group whose values differ from
// the previous group's; a run ends where the next run of its contig starts, the last at the contig's length.
// Contigs without groups are one head run.
// ---------------------------------------------------------------------------------------------
struct RankView {
  const u32 *rg, *gc, *gs;  // rg null: rank = group index
  const i32* val;           // per rank, nv columns of ng
  u32 nv;
  u64 ng;
  __device__ __forceinline__ u32 grp(u64 r) const { return rg ? rg[r] : (u32)r; }
  __device__ __forceinline__ u32 contig(u64 r) const { return gc[grp(r)]; }
  __device__ __forceinline__ bool first(u64 r, u32 c) const { return r == 0 || contig(r - 1) != c; }
  __device__ __forceinline__ bool last(u64 r, u32 c) const { return r + 1 == ng || contig(r + 1) != c; }
  __device__ __forceinline__ u32 starts_run(u64 r) const {
    const u32 g = grp(r), c = gc[g];
    const bool head = first(r, c);
    bool differs = false;
    for (u32 t = 0; t < nv; t++) differs |= val[t * ng + r] != (head ? 0 : val[t * ng + r - 1]);
    return (head && gs[g] == 0) || differs;
  }
};

// per contig: [0] run starts among its groups before it (exclusive scan), [1] ... after its last group,
// [2] start of its first group (none: 0xFFFFFFFF), [3] index of its first run
__global__ void __launch_bounds__(256) k_runs_groups(const RankView V, const u32* __restrict__ gx, const u32* __restrict__ cst, u32 nc,
                                                     const u32* __restrict__ clen, u32* rc, u32* rs, u32* rv, u64 nr, u32* err) {
  const u64 r = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= V.ng) return;
  const u32 g = V.grp(r), c = V.gc[g], s = V.gs[g];
  if (s >= clen[c]) atomicOr(err, 1u);
  if (!V.starts_run(r)) return;
  const u32 head = cst[2 * nc + c] != 0;
  const u32 o = cst[3 * nc + c] + head + gx[r] - cst[c];
  rc[o] = c;
  rs[o] = s;
  for (u32 t = 0; t < V.nv; t++) rv[t * nr + o] = (u32)V.val[t * V.ng + r];
}
__global__ void __launch_bounds__(256) k_runs_heads(const u32* __restrict__ cst, u32 nc, u32* rc, u32* rs, u32* rv, u32 nv, u64 nr) {
  const u32 c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= nc || cst[2 * nc + c] == 0) return;
  const u32 o = cst[3 * nc + c];
  rc[o] = c;
  rs[o] = 0;
  for (u32 t = 0; t < nv; t++) rv[t * nr + o] = 0;
}
__global__ void __launch_bounds__(256) k_runs_end(const u32* __restrict__ rc, const u32* __restrict__ rs, u64 n, const u32* __restrict__ clen,
                                                  u32* re) {
  const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  re[i] = (i + 1 < n && rc[i + 1] == rc[i]) ? rs[i + 1] : clen[rc[i]];
}

int gvs_rank_runs(gvs_ctx* ctx, const i32* diff, u32 nv, const uint32_t* contig_len, RecTable& out, const char* who) {
  out.ready = false;
  out.n = 0;
  const u32 nc = ctx->n_contigs;
  if (nc && !contig_len) return gvs_fail(ctx, GVS_E_ARG, "%s: null contig_len", who);
  const u64 ng = ctx->n_groups;
  CKR(to_dev(ctx, ctx->contig_len, contig_len, nc));
  CKR(gvs_reserve(ctx, ctx->sup_depth, (ng ? ng : 1) * 4 * nv));
  CKR(gvs_reserve(ctx, ctx->sup_gx, (ng ? ng : 1) * 4));
  CKR(gvs_reserve(ctx, ctx->sup_cstat, ((u64)nc ? nc : 1) * 16));
  u32* cst = ctx->sup_cstat.as<u32>();
  CK(cudaMemsetAsync(cst, 0, (u64)nc * 8, ctx->stream));
  CK(cudaMemsetAsync(cst + 2 * (u64)nc, 0xFF, (u64)nc * 4, ctx->stream));
  RankView V;
  V.rg = ctx->rank_identity ? nullptr : ctx->rank_grp.as<u32>();
  V.gc = ctx->grp_contig.as<u32>();
  V.gs = ctx->grp_start.as<u32>();
  V.val = ctx->sup_depth.as<i32>();
  V.nv = nv;
  V.ng = ng;
  u32* err = counter(ctx, CNT_RUNS_ERR);
  CK(cudaMemsetAsync(err, 0, 4, ctx->stream));
  if (ng) {
    for (u32 t = 0; t < nv; t++) {
      const i32* d = diff + t * ng;
      i32* v = ctx->sup_depth.as<i32>() + t * ng;
      auto f = [d] __device__(u64 r) -> i32 { return d[r]; };
      auto g = [v] __device__(u64 r, i32 ex, i32 x) { v[r] = ex + x; };
      CKR((device_scan<i32>(ctx, ng, f, g, OpSum(), (i32*)nullptr)));
    }
    u32* gx = ctx->sup_gx.as<u32>();
    auto f = [V] __device__(u64 r) -> u32 { return V.starts_run(r); };
    auto g = [V, gx, cst, nc] __device__(u64 r, u32 ex, u32 v) {
      gx[r] = ex;
      const u32 grp = V.grp(r), c = V.gc[grp];
      if (V.first(r, c)) {
        cst[c] = ex;
        cst[2 * nc + c] = V.gs[grp];
      }
      if (V.last(r, c)) cst[nc + c] = ex + v;
    };
    CKR((device_scan<u32>(ctx, ng, f, g, OpSum(), (u32*)nullptr)));
  }
  u32 nr = 0;
  {
    auto f = [cst, nc] __device__(u64 c) -> u32 { return (cst[2 * nc + c] != 0 ? 1u : 0u) + cst[nc + c] - cst[c]; };
    auto g = [cst, nc] __device__(u64 c, u32 ex, u32 v) { cst[3 * nc + c] = ex; };
    CKR(scan_total(ctx, nc, f, g, OpSum(), &nr));
  }
  CKR(rec_reserve(ctx, out, 3 + nv, nr));
  const u32* clen = ctx->contig_len.as<u32>();
  u32 *rc = out.col(0), *rs = out.col(1), *rv = out.col(3);
  if (ng) LAUNCH(k_runs_groups, (unsigned)cdiv(ng, 256), 256, 0, V, ctx->sup_gx.as<u32>(), cst, nc, clen, rc, rs, rv, (u64)nr, err);
  if (nc) LAUNCH(k_runs_heads, (unsigned)cdiv(nc, 256), 256, 0, cst, nc, rc, rs, rv, nv, (u64)nr);
  if (nr) LAUNCH(k_runs_end, (unsigned)cdiv(nr, 256), 256, 0, rc, rs, nr, clen, out.col(2));
  u32 h = 0;
  CKR(read_dev(ctx, err, &h));
  if (h) return gvs_fail(ctx, GVS_E_ARG, "%s: a SUNK group starts at or beyond its contig's length", who);
  out.n = nr;
  out.ready = true;
  return 0;
}

extern "C" int gvs_support(gvs_ctx* ctx, const uint32_t* contig_len, uint64_t* n_runs) {
  if (!ctx) return GVS_E_ARG;
  if (!ctx->pl.ready) return gvs_fail(ctx, GVS_E_STATE, "gvs_support before gvs_placements");
  CK(cudaSetDevice(ctx->device));
  StageTimer tm(ctx, GVS_ST_SUPPORT);
  if (n_runs) *n_runs = 0;
  CKR(gvs_rank_runs(ctx, ctx->sup_diff.as<i32>(), 1, contig_len, ctx->sup, "gvs_support"));
  if (n_runs) *n_runs = ctx->sup.n;
  return 0;
}

extern "C" int gvs_support_get(gvs_ctx* ctx, uint32_t* contig, uint32_t* start, uint32_t* end, uint32_t* depth) {
  return ctx ? rec_get(ctx, ctx->sup, "gvs_support_get before gvs_support", {contig, start, end, depth}) : GVS_E_ARG;
}
