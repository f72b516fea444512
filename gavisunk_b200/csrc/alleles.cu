// alleles.cu -- allele support: per SUNK group the distinct reads of its own haplotype (own) and of the other haplotype
// (other) among every match row, and their runs in segment space.  No reference counterpart.  Definition:
// include/gavisunk_b200.h (gvs_allele_support, gvs_allele_runs), DESIGN.md section 5.5h.
//
// At a heterozygous site the two haplotypes' k-mers differ, so each haplotype has its own SUNK group there and only the
// reads of that haplotype should carry it.  A phase flip shows as a group carried by the other haplotype's reads only; a
// consensus error as a group no read carries.  The counts are taken before the diag filter (which keeps one contig per
// read) on the contigs of both haplotypes, exactly as gvs_sunk_depth counts its reads, split by the read's haplotype.
//
// gvs_allele_support:
//   k_al_hap / k_al_vote  the file haplotype of every read of the batch: its chunk's; for an unbinned chunk the one the
//                         haplotype-mode records of the batch's diag filter assign, and for a tie or no vote the parity
//                         of the read's run-wide index (as gvs_batch_stash will number it).
//   k_al_count            one warp per read segment of the match rows, with no cap on rows: a shuffle carried across
//                         the 32-row chunks tests whether the group indices are monotone; a monotone read counts its
//                         distinct groups as value changes (exact), the others rank-sort into scratch (warp_order) and
//                         count the written slots.  One atomicAdd per distinct (read, group) into own or other.
//   k_al_loc              once per group table: .loc rows per group, and the group's end (its last SUNK's start + k).
// gvs_allele_runs: the rank-ordered differences of (own, other), prefix-summed back by the run tiling of the support
// depth (gvs_rank_runs).
#include "common.cuh"

#define AL_NONE 0xFFFFFFFFu

// hap[r] = the chunk's haplotype of read r, or for an unbinned chunk the parity of its run-wide index base + r
__global__ void __launch_bounds__(256) k_al_hap(u64 n_reads, const u64* __restrict__ chunk_first, const u8* __restrict__ chunk_hap,
                                                u32 n_chunks, u32 base, u8* hap) {
  const u64 r = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n_reads) return;
  const u8 h = chunk_hap[chunk_of_read(chunk_first, n_chunks, (u32)r)];
  hap[r] = h < GVS_HAP_ANY ? h : (u8)((base + (u32)r) & 1u);
}

// the haplotype-mode records of the batch's diag filter: an unbinned read with a decisive vote takes its assignment
__global__ void __launch_bounds__(256) k_al_vote(u64 n_rec, const u32* __restrict__ rec_read, const u32* __restrict__ rec_hap,
                                                 const u64* __restrict__ chunk_first, const u8* __restrict__ chunk_hap, u32 n_chunks,
                                                 u8* hap) {
  const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_rec) return;
  const u32 r = rec_read[i], h = rec_hap[i];
  if (h <= 1 && chunk_hap[chunk_of_read(chunk_first, n_chunks, r)] == GVS_HAP_ANY) hap[r] = (u8)h;
}

// one distinct (read, group): own when the group's contig is of the read's haplotype, other when of the other one
__device__ __forceinline__ void al_add(i32* cnt, u64 ng, const u32* __restrict__ grp_contig, const u8* __restrict__ contig_hap,
                                       u32 g, u32 h) {
  const u32 gh = contig_hap[grp_contig[g]];
  if (gh <= 1) atomicAdd(&cnt[(gh == h ? 0 : ng) + g], 1);
}

// cnt[g] += reads of g's haplotype with a row of group g, cnt[ng + g] += those of the other; scr: per-row scratch at the
// segment's first row
__global__ void __launch_bounds__(256) k_al_count(const u32* __restrict__ gidx, const u32* __restrict__ read,
                                                  const u32* __restrict__ seg_start, u32 n_seg, const u8* __restrict__ hap,
                                                  const u32* __restrict__ grp_contig, const u8* __restrict__ contig_hap, u32* scr,
                                                  i32* cnt, u64 ng) {
  const u32 s = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (s >= n_seg) return;
  const u32 a = seg_start[s], b = seg_start[s + 1];
  const u32 h = hap[read[a]];
  bool up = true, down = true;
  u32 carry = 0;
  for (u32 c = a; c < b; c += 32) {
    const u32 i = c + lane;
    const bool q = i < b;
    const u32 v = q ? gidx[i] : 0u;
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
      if (i == a || gidx[i] != gidx[i - 1]) al_add(cnt, ng, grp_contig, contig_hap, gidx[i], h);
    return;
  }
  const u32 n = b - a;
  u32* y = scr + a;
  for (u32 k = lane; k < n; k += 32) y[k] = AL_NONE;
  __syncwarp();
  warp_order(gidx + a, y, n, [](u32 g) -> u64 { return g; }, lane);
  for (u32 k = lane; k < n; k += 32)
    if (y[k] != AL_NONE) al_add(cnt, ng, grp_contig, contig_hap, y[k], h);
}

// end[g] = the group's start + k before k_al_loc raises it to its last SUNK's start + k
__global__ void __launch_bounds__(256) k_al_end0(const u32* __restrict__ grp_start, u64 ng, u32 k, u32* end) {
  const u64 g = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (g < ng) end[g] = grp_start[g] + k;
}

// per .loc row: sunks[g] += 1, end[g] = max(end[g], start + k)
__global__ void __launch_bounds__(256) k_al_loc(const u32* __restrict__ loc_gidx, const u32* __restrict__ loc_start, u64 n, u32 k,
                                                u32* sunks, u32* end) {
  const u64 j = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n) return;
  const u32 g = loc_gidx[j];
  atomicAdd(&sunks[g], 1u);
  atomicMax(&end[g], loc_start[j] + k);
}

// diff[t][r] = v_t(r) - v_t(r - 1) over the ranks r in (contig, start) order, v = (own, other)
__global__ void __launch_bounds__(256) k_al_diff(const i32* __restrict__ cnt, const u32* __restrict__ rank_grp, u64 ng, i32* diff) {
  const u64 r = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= ng) return;
  const u32 g = rank_grp ? rank_grp[r] : (u32)r;
  const u32 p = r ? (rank_grp ? rank_grp[r - 1] : (u32)(r - 1)) : 0u;
  diff[r] = cnt[g] - (r ? cnt[p] : 0);
  diff[ng + r] = cnt[ng + g] - (r ? cnt[ng + p] : 0);
}

extern "C" int gvs_allele_support(gvs_ctx* ctx, int accumulate, int32_t** support_dev) {
  if (!ctx) return GVS_E_ARG;
  if (!ctx->groups_ready) return gvs_fail(ctx, GVS_E_STATE, "gvs_allele_support: no group index");
  if (ctx->contig_hap.cap == 0) return gvs_fail(ctx, GVS_E_STATE, "gvs_allele_support: contig haplotypes unknown (gvs_contigs_set)");
  const u64 n = ctx->match_ready ? ctx->rows.n : 0;  // no current match rows (a rank without a batch): adds nothing
  bool unbinned = false;
  for (u8 h : ctx->h_chunk_hap) unbinned |= h == GVS_HAP_ANY;
  if (n && unbinned && !(ctx->diag_ready && ctx->rh.ready))
    return gvs_fail(ctx, GVS_E_STATE, "gvs_allele_support: a batch with unbinned chunks needs its diag filter first");
  CK(cudaSetDevice(ctx->device));
  StageTimer tm(ctx, GVS_ST_ALLELES);
  const u64 ng = ctx->n_groups, bytes = (ng ? 2 * ng : 1) * 4;
  const bool fresh = ctx->al_cnt.cap < bytes;
  CKR(gvs_reserve(ctx, ctx->al_cnt, bytes));
  if (!accumulate || fresh || !ctx->al_ready || ctx->al_gen != ctx->grp_gen) CK(cudaMemsetAsync(ctx->al_cnt.p, 0, bytes, ctx->stream));
  if (ctx->al_loc_gen != ctx->grp_gen) {  // once per group table
    CKR(gvs_reserve(ctx, ctx->al_sunks, (ng ? ng : 1) * 4));
    CKR(gvs_reserve(ctx, ctx->al_end, (ng ? ng : 1) * 4));
    CK(cudaMemsetAsync(ctx->al_sunks.p, 0, (ng ? ng : 1) * 4, ctx->stream));
    if (ng) LAUNCH(k_al_end0, (unsigned)cdiv(ng, 256), 256, 0, ctx->grp_start.as<u32>(), ng, (u32)ctx->k, ctx->al_end.as<u32>());
    if (ctx->db_ready && ctx->n_loc)
      LAUNCH(k_al_loc, (unsigned)cdiv(ctx->n_loc, 256), 256, 0, ctx->loc_gidx.as<u32>(), ctx->loc_start.as<u32>(), ctx->n_loc,
             (u32)ctx->k, ctx->al_sunks.as<u32>(), ctx->al_end.as<u32>());
    ctx->al_loc_gen = ctx->grp_gen;
  }
  ctx->al_gen = ctx->grp_gen;
  if (n) {
    // read indices as gvs_batch_stash will number this batch's reads (the parity of an undecided unbinned read)
    const u64 base = ctx->jn_in_run ? ctx->stash_reads : 0, nr = ctx->n_reads;
    CKR(gvs_reserve(ctx, ctx->al_hap, nr ? nr : 1));
    if (nr)
      LAUNCH(k_al_hap, (unsigned)cdiv(nr, 256), 256, 0, nr, ctx->chunk_first.as<u64>(), ctx->chunk_hap.as<u8>(), ctx->n_chunks, (u32)base,
             ctx->al_hap.as<u8>());
    if (unbinned && ctx->rh.n)
      LAUNCH(k_al_vote, (unsigned)cdiv(ctx->rh.n, 256), 256, 0, ctx->rh.n, ctx->rh.col(0), ctx->rh.col(7), ctx->chunk_first.as<u64>(),
             ctx->chunk_hap.as<u8>(), ctx->n_chunks, ctx->al_hap.as<u8>());
    u64 n_seg = 0;
    CKR(gvs_build_segments(ctx, ctx->rows.read.as<u32>(), n, ctx->al_seg_start, ctx->al_row_seg, &n_seg));
    CKR(gvs_reserve(ctx, ctx->al_scr, n * 4));
    LAUNCH(k_al_count, (unsigned)cdiv(n_seg * 32, 256), 256, 0, ctx->rows.gidx.as<u32>(), ctx->rows.read.as<u32>(),
           ctx->al_seg_start.as<u32>(), (u32)n_seg, ctx->al_hap.as<u8>(), ctx->grp_contig.as<u32>(), ctx->contig_hap.as<u8>(),
           ctx->al_scr.as<u32>(), ctx->al_cnt.as<i32>(), ng);
  }
  ctx->al_ready = true;
  ctx->al_runs.ready = false;
  if (support_dev) *support_dev = ctx->al_cnt.as<i32>();
  return 0;
}

extern "C" int gvs_allele_support_get(gvs_ctx* ctx, int32_t* own, int32_t* other, uint32_t* sunks, uint32_t* end) {
  if (!ctx) return GVS_E_ARG;
  if (!ctx->al_ready) return gvs_fail(ctx, GVS_E_STATE, "gvs_allele_support_get before gvs_allele_support");
  if (ctx->al_gen != ctx->grp_gen)
    return gvs_fail(ctx, GVS_E_STATE, "gvs_allele_support_get: the group table changed since gvs_allele_support");
  CK(cudaSetDevice(ctx->device));
  const u64 ng = ctx->n_groups;
  if (ng == 0) return 0;
  if (own) CK(cudaMemcpyAsync(own, ctx->al_cnt.p, ng * 4, cudaMemcpyDeviceToHost, ctx->stream));
  if (other) CK(cudaMemcpyAsync(other, ctx->al_cnt.as<i32>() + ng, ng * 4, cudaMemcpyDeviceToHost, ctx->stream));
  if (sunks) CK(cudaMemcpyAsync(sunks, ctx->al_sunks.p, ng * 4, cudaMemcpyDeviceToHost, ctx->stream));
  if (end) CK(cudaMemcpyAsync(end, ctx->al_end.p, ng * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return 0;
}

extern "C" int gvs_allele_runs(gvs_ctx* ctx, const uint32_t* contig_len, uint64_t* n_runs) {
  if (!ctx) return GVS_E_ARG;
  if (n_runs) *n_runs = 0;
  if (!ctx->al_ready) return gvs_fail(ctx, GVS_E_STATE, "gvs_allele_runs before gvs_allele_support");
  if (ctx->al_gen != ctx->grp_gen) return gvs_fail(ctx, GVS_E_STATE, "gvs_allele_runs: the group table changed since gvs_allele_support");
  CK(cudaSetDevice(ctx->device));
  StageTimer tm(ctx, GVS_ST_ALLELES);
  CKR(gvs_ensure_rank(ctx));
  const u64 ng = ctx->n_groups;
  CKR(gvs_reserve(ctx, ctx->al_diff, (ng ? 2 * ng : 1) * 4));
  if (ng)
    LAUNCH(k_al_diff, (unsigned)cdiv(ng, 256), 256, 0, ctx->al_cnt.as<i32>(), ctx->rank_identity ? nullptr : ctx->rank_grp.as<u32>(), ng,
           ctx->al_diff.as<i32>());
  CKR(gvs_rank_runs(ctx, ctx->al_diff.as<i32>(), 2, contig_len, ctx->al_runs, "gvs_allele_runs"));
  if (n_runs) *n_runs = ctx->al_runs.n;
  return 0;
}

extern "C" int gvs_allele_runs_get(gvs_ctx* ctx, uint32_t* contig, uint32_t* start, uint32_t* end, uint32_t* own, uint32_t* other) {
  return ctx ? rec_get(ctx, ctx->al_runs, "gvs_allele_runs_get before gvs_allele_runs", {contig, start, end, own, other}) : GVS_E_ARG;
}
