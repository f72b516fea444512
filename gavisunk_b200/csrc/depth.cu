// depth.cu -- SUNK hit depth: per group the match rows (hits) and the distinct reads among them (reads), and their runs
// with the bad-SUNK histogram (kept) in segment space.  No reference counterpart.  Definition: include/gavisunk_b200.h
// (gvs_sunk_depth, gvs_depth_runs).
//
// A collapse of c genomic copies into one assembled copy sends the reads of every copy to its SUNKs: about c times the
// hits of a single-copy region.  The bad-SUNK filter removes exactly those groups from validation, so no other stage
// shows them.  Here every match row counts, before the diag filter keeps one contig per read: reads from a collapsed copy
// elsewhere often have their best contig elsewhere.
//
// gvs_sunk_depth: one warp per read segment of the match rows, with no cap on rows.  One pass adds every row to hits and
// tests, with a shuffle carried across the 32-row chunks, whether the read's group indices are monotone (either
// direction).  A monotone sequence holds equal values contiguously, so its distinct groups are its value changes: exact.
// Most reads walk the assembly in one direction and leave there.  The others rank-sort their group indices into per-row
// scratch (warp_order): equal values land on one slot, so the written slots are the distinct groups.  One atomicAdd per
// distinct (read, group) either way.
// gvs_depth_runs: the rank-ordered differences of (hits, reads, kept), prefix-summed back by the run tiling of the
// support depth (gvs_rank_runs).
#include "common.cuh"

#define DP_NONE 0xFFFFFFFFu

// .loc rows per group (a k_hist of the group index of every .loc row)
__global__ void __launch_bounds__(256) k_dp_sunks(const u32* __restrict__ loc_gidx, u64 n, u32* sunks) {
  const u64 j = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (j < n) atomicAdd(&sunks[loc_gidx[j]], 1u);
}

// cnt[g] += rows of group g, cnt[ng + g] += reads with a row of group g; scr: per-row scratch at the segment's first row
__global__ void __launch_bounds__(256) k_dp_count(const u32* __restrict__ gidx, const u32* __restrict__ seg_start, u32 n_seg, u32* scr,
                                                  i32* cnt, u64 ng) {
  const u32 s = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (s >= n_seg) return;
  const u32 a = seg_start[s], b = seg_start[s + 1];
  bool up = true, down = true;
  u32 carry = 0;
  for (u32 c = a; c < b; c += 32) {
    const u32 i = c + lane;
    const bool q = i < b;
    const u32 v = q ? gidx[i] : 0u;
    if (q) atomicAdd(&cnt[v], 1);
    const u32 pv = __shfl_up_sync(0xFFFFFFFFu, v, 1);
    if (q && (lane || c > a)) {  // the previous row: the lane below, or the last row of the previous (full) chunk
      const u32 p = lane ? pv : carry;
      up &= p <= v;
      down &= p >= v;
    }
    carry = __shfl_sync(0xFFFFFFFFu, v, 31);
  }
  if (__all_sync(0xFFFFFFFFu, up) || __all_sync(0xFFFFFFFFu, down)) {
    for (u32 i = a + lane; i < b; i += 32)
      if (i == a || gidx[i] != gidx[i - 1]) atomicAdd(&cnt[ng + gidx[i]], 1);
    return;
  }
  const u32 n = b - a;
  u32* y = scr + a;
  for (u32 k = lane; k < n; k += 32) y[k] = DP_NONE;
  __syncwarp();
  warp_order(gidx + a, y, n, [](u32 g) -> u64 { return g; }, lane);
  for (u32 k = lane; k < n; k += 32)
    if (y[k] != DP_NONE) atomicAdd(&cnt[ng + y[k]], 1);
}

// diff[t][r] = v_t(r) - v_t(r - 1) over the ranks r in (contig, start) order, v = (hits, reads, kept)
__global__ void __launch_bounds__(256) k_dp_diff(const i32* __restrict__ cnt, const i32* __restrict__ kept, const u32* __restrict__ rank_grp,
                                                 u64 ng, i32* diff) {
  const u64 r = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= ng) return;
  const u32 g = rank_grp ? rank_grp[r] : (u32)r;
  const u32 p = r ? (rank_grp ? rank_grp[r - 1] : (u32)(r - 1)) : 0u;
  diff[r] = cnt[g] - (r ? cnt[p] : 0);
  diff[ng + r] = cnt[ng + g] - (r ? cnt[ng + p] : 0);
  diff[2 * ng + r] = kept[g] - (r ? kept[p] : 0);
}

extern "C" int gvs_sunk_depth(gvs_ctx* ctx, int accumulate, int32_t** depth_dev) {
  if (!ctx) return GVS_E_ARG;
  if (!ctx->groups_ready) return gvs_fail(ctx, GVS_E_STATE, "gvs_sunk_depth: no group index");
  CK(cudaSetDevice(ctx->device));
  StageTimer tm(ctx, GVS_ST_DEPTH);
  const u64 ng = ctx->n_groups, bytes = (ng ? 2 * ng : 1) * 4;
  const bool fresh = ctx->dp_cnt.cap < bytes;
  CKR(gvs_reserve(ctx, ctx->dp_cnt, bytes));
  if (!accumulate || fresh || !ctx->dp_ready || ctx->dp_gen != ctx->grp_gen) CK(cudaMemsetAsync(ctx->dp_cnt.p, 0, bytes, ctx->stream));
  if (ctx->dp_sunks_gen != ctx->grp_gen) {  // once per group table
    CKR(gvs_reserve(ctx, ctx->dp_sunks, (ng ? ng : 1) * 4));
    CK(cudaMemsetAsync(ctx->dp_sunks.p, 0, (ng ? ng : 1) * 4, ctx->stream));
    if (ctx->db_ready && ctx->n_loc)
      LAUNCH(k_dp_sunks, (unsigned)cdiv(ctx->n_loc, 256), 256, 0, ctx->loc_gidx.as<u32>(), ctx->n_loc, ctx->dp_sunks.as<u32>());
    ctx->dp_sunks_gen = ctx->grp_gen;
  }
  ctx->dp_gen = ctx->grp_gen;
  const u64 n = ctx->match_ready ? ctx->rows.n : 0;  // no current match rows (a rank without a batch): adds nothing
  if (n) {
    u64 n_seg = 0;
    CKR(gvs_build_segments(ctx, ctx->rows.read.as<u32>(), n, ctx->dp_seg_start, ctx->dp_row_seg, &n_seg));
    CKR(gvs_reserve(ctx, ctx->dp_scr, n * 4));
    LAUNCH(k_dp_count, (unsigned)cdiv(n_seg * 32, 256), 256, 0, ctx->rows.gidx.as<u32>(), ctx->dp_seg_start.as<u32>(), (u32)n_seg,
           ctx->dp_scr.as<u32>(), ctx->dp_cnt.as<i32>(), ng);
  }
  ctx->dp_ready = true;
  ctx->dp_runs.ready = false;
  if (depth_dev) *depth_dev = ctx->dp_cnt.as<i32>();
  return 0;
}

extern "C" int gvs_sunk_depth_get(gvs_ctx* ctx, int32_t* hits, int32_t* reads, uint32_t* sunks) {
  if (!ctx) return GVS_E_ARG;
  if (!ctx->dp_ready) return gvs_fail(ctx, GVS_E_STATE, "gvs_sunk_depth_get before gvs_sunk_depth");
  if (ctx->dp_gen != ctx->grp_gen) return gvs_fail(ctx, GVS_E_STATE, "gvs_sunk_depth_get: the group table changed since gvs_sunk_depth");
  CK(cudaSetDevice(ctx->device));
  const u64 ng = ctx->n_groups;
  if (ng == 0) return 0;
  if (hits) CK(cudaMemcpyAsync(hits, ctx->dp_cnt.p, ng * 4, cudaMemcpyDeviceToHost, ctx->stream));
  if (reads) CK(cudaMemcpyAsync(reads, ctx->dp_cnt.as<i32>() + ng, ng * 4, cudaMemcpyDeviceToHost, ctx->stream));
  if (sunks) CK(cudaMemcpyAsync(sunks, ctx->dp_sunks.p, ng * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return 0;
}

extern "C" int gvs_depth_runs(gvs_ctx* ctx, const uint32_t* contig_len, uint64_t* n_runs) {
  if (!ctx) return GVS_E_ARG;
  if (n_runs) *n_runs = 0;
  if (!ctx->hist_ready) return gvs_fail(ctx, GVS_E_STATE, "gvs_depth_runs before gvs_group_hist");
  if (!ctx->dp_ready) return gvs_fail(ctx, GVS_E_STATE, "gvs_depth_runs before gvs_sunk_depth");
  if (ctx->dp_gen != ctx->grp_gen) return gvs_fail(ctx, GVS_E_STATE, "gvs_depth_runs: the group table changed since gvs_sunk_depth");
  CK(cudaSetDevice(ctx->device));
  StageTimer tm(ctx, GVS_ST_DEPTH);
  CKR(gvs_ensure_rank(ctx));
  const u64 ng = ctx->n_groups;
  CKR(gvs_reserve(ctx, ctx->dp_diff, (ng ? 3 * ng : 1) * 4));
  if (ng)
    LAUNCH(k_dp_diff, (unsigned)cdiv(ng, 256), 256, 0, ctx->dp_cnt.as<i32>(), ctx->hist.as<i32>(),
           ctx->rank_identity ? nullptr : ctx->rank_grp.as<u32>(), ng, ctx->dp_diff.as<i32>());
  CKR(gvs_rank_runs(ctx, ctx->dp_diff.as<i32>(), 3, contig_len, ctx->dp_runs, "gvs_depth_runs"));
  if (n_runs) *n_runs = ctx->dp_runs.n;
  return 0;
}

extern "C" int gvs_depth_runs_get(gvs_ctx* ctx, uint32_t* contig, uint32_t* start, uint32_t* end, uint32_t* hits, uint32_t* reads,
                                  uint32_t* kept) {
  return ctx ? rec_get(ctx, ctx->dp_runs, "gvs_depth_runs_get before gvs_depth_runs", {contig, start, end, hits, reads, kept})
             : GVS_E_ARG;
}
