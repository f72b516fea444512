// batches.cu -- several read batches of ONE run (two-phase engine).
//
// The reference scatters a sample's reads into chunk files, runs kmerpos_annot3 / diag_filter per chunk and
// gathers per haplotype before anything global happens (workflow/Snakefile:23-24 scattergather,
// workflow/rules/tagONT.smk:112-131 combine_ont): badsunks_AR.py:20-27 counts the rows of ALL chunks,
// process-by-contig_lowmem_AR.py sees every read of a contig.  A run whose reads do not fit one batch (93 Gbp
// for a 30x human sample) therefore has two phases:
//   phase 1, per batch:  gvs_reads_set* -> gvs_match -> gvs_diag_filter -> gvs_group_hist(accumulate = 1)
//                        -> gvs_batch_stash   (the kept rows, 24 B each, stay resident; the reads may go)
//   [multi-GPU: ONE all-reduce of the histogram]   gvs_hist_mode / gvs_bad_groups
//   phase 2, once:       gvs_batches_bind -> gvs_validate -> gvs_components_local
//   [multi-GPU: ONE all-gather of the forests + gvs_components_merge_all]   gvs_intervals -> gvs_gaps
// Read indices of the bound rows count through the batches in stash order (batch b's reads start at the
// *read_base gvs_batch_stash returned for it).
#include "common.cuh"

// grow a device buffer to `need` bytes keeping its first `keep` bytes
int grow_keep(gvs_ctx* ctx, DevBuf& b, size_t need, size_t keep) {
  if (b.cap >= need) return 0;
  size_t want = need + need / 2 + 256;
  void* p = nullptr;
  cudaError_t e = cudaMalloc(&p, want);
  if (e != cudaSuccess) return gvs_fail(ctx, GVS_E_NOMEM, "cudaMalloc(%zu bytes): %s", want, cudaGetErrorString(e));
  if (b.p) {
    if (keep) CK(cudaMemcpyAsync(p, b.p, keep, cudaMemcpyDeviceToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    CK(cudaFree(b.p));
  }
  b.p = p;
  b.cap = want;
  return 0;
}

__global__ void __launch_bounds__(256) k_stash_rows(u64 n, u32 base, const u32* __restrict__ s_read, const u32* __restrict__ s_pos,
                                                    const u32* __restrict__ s_contig, const u32* __restrict__ s_start,
                                                    const u32* __restrict__ s_group, const u32* __restrict__ s_gidx, u32* d_read,
                                                    u32* d_pos, u32* d_contig, u32* d_start, u32* d_group, u32* d_gidx) {
  u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  d_read[i] = s_read[i] + base;
  d_pos[i] = s_pos[i];
  d_contig[i] = s_contig[i];
  d_start[i] = s_start[i];
  d_group[i] = s_group[i];
  d_gidx[i] = s_gidx[i];
}
__global__ void __launch_bounds__(256) k_stash_len(u64 n, const ReadLens len, u32* dst) {
  u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  dst[i] = len((u32)i);
}

// the batch's read-haplotype records (8 columns, read first) appended to the run's at `have`, read indices made run-wide
__global__ void __launch_bounds__(256) k_stash_recs(u64 n, u32 base, const u32* __restrict__ src, u64 src_stride, u32* dst,
                                                    u64 dst_stride, u64 have) {
  u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  dst[have + i] = src[i] + base;
#pragma unroll
  for (u32 c = 1; c < 8; c++) dst[c * dst_stride + have + i] = src[c * src_stride + i];
}

// grow the run's record table to hold `need` records, keeping the `have` it holds (columns move to the new stride)
static int grow_recs(gvs_ctx* ctx, RecTable& t, u64 need, u64 have) {
  if (t.stride >= need) return 0;
  const u64 stride = need + need / 2 + 64;
  DevBuf nb;
  CKR(gvs_reserve(ctx, nb, stride * 8 * 4));
  for (u32 c = 0; c < 8 && have; c++)
    CK(cudaMemcpyAsync(nb.as<u32>() + c * stride, t.col(c), have * 4, cudaMemcpyDeviceToDevice, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  gvs_release(t.buf);
  t.buf = nb;
  t.stride = stride;
  return 0;
}

extern "C" int gvs_batches_begin(gvs_ctx* ctx) {
  if (!ctx) return GVS_E_ARG;
  CK(cudaSetDevice(ctx->device));
  ctx->stash.n = 0;
  ctx->stash_reads = 0;
  ctx->hist_ready = false;  // the next gvs_group_hist(accumulate = 1) starts from zero
  ctx->bad_ready = false;
  ctx->comp_ready = false;  // ... and gvs_intervals waits for the run's gvs_components_local
  ctx->val_ready = false;
  ctx->jn_stash.n = 0;  // the junction screens of the run append from here (junctions.cu)
  ctx->jn_reads = 0;
  ctx->jn_in_run = true;
  ctx->rh_run.n = 0;
  ctx->rh_run.ready = false;
  return 0;
}

extern "C" int gvs_batch_stash(gvs_ctx* ctx, uint64_t* read_base) {
  if (!ctx) return GVS_E_ARG;
  if (!ctx->diag_ready) return gvs_fail(ctx, GVS_E_STATE, "gvs_batch_stash before gvs_diag_filter / gvs_rows_set(1)");
  if (!ctx->read_off && !ctx->have_read_len) return gvs_fail(ctx, GVS_E_STATE, "gvs_batch_stash: read lengths unknown");
  CK(cudaSetDevice(ctx->device));
  const u64 base = ctx->stash_reads, n = ctx->kept.n, have = ctx->stash.n, nr = ctx->n_reads;
  if (base + nr >= 0xFFFFFFF0ull) return gvs_fail(ctx, GVS_E_OVERFLOW, "more than 2^32 reads in one run");
  if (have + n >= 0xFFFFFFF0ull) return gvs_fail(ctx, GVS_E_OVERFLOW, "more than 2^32 kept rows in one run");
  Rows& S = ctx->stash;
  DevBuf* dst[6] = {&S.read, &S.pos, &S.contig, &S.start, &S.group, &S.gidx};
  for (DevBuf* b : dst) CKR(grow_keep(ctx, *b, (have + n + 1) * 4, have * 4));
  CKR(grow_keep(ctx, ctx->stash_len, (base + nr + 1) * 4, base * 4));
  const Rows& K = ctx->kept;
  if (n)
    LAUNCH(k_stash_rows, (unsigned)cdiv(n, 256), 256, 0, n, (u32)base, K.read.as<u32>(), K.pos.as<u32>(), K.contig.as<u32>(),
           K.start.as<u32>(), K.group.as<u32>(), K.gidx.as<u32>(), S.read.as<u32>() + have, S.pos.as<u32>() + have,
           S.contig.as<u32>() + have, S.start.as<u32>() + have, S.group.as<u32>() + have, S.gidx.as<u32>() + have);
  if (nr)
    LAUNCH(k_stash_len, (unsigned)cdiv(nr, 256), 256, 0, nr, read_lens(ctx), ctx->stash_len.as<u32>() + base);
  if (ctx->rh.ready) {  // the batch's diag filter ran in haplotype mode
    RecTable &R = ctx->rh_run, &B = ctx->rh;
    CKR(grow_recs(ctx, R, R.n + B.n + 1, R.n));
    if (B.n) LAUNCH(k_stash_recs, (unsigned)cdiv(B.n, 256), 256, 0, B.n, (u32)base, B.col(0), B.stride, R.col(0), R.stride, R.n);
    R.n += B.n;
    R.ready = true;
  }
  S.n = have + n;
  ctx->stash_reads = base + nr;
  if (read_base) *read_base = base;
  return 0;
}

extern "C" int gvs_batches_bind(gvs_ctx* ctx, uint64_t* n_rows, uint64_t* n_reads) {
  if (!ctx) return GVS_E_ARG;
  CK(cudaSetDevice(ctx->device));
  CKR(gvs_pipe_join(ctx));
  // the stashed rows become "the rows kept by the diag filter", the stashed lengths the read table; the buffers
  // swap places, so that the next run stashes into this run's (already sized) memory
  std::swap(ctx->kept, ctx->stash);
  std::swap(ctx->read_len, ctx->stash_len);
  std::swap(ctx->rh, ctx->rh_run);  // the run's read-haplotype records (ready when a batch ran in haplotype mode)
  ctx->rh_run.n = 0;
  ctx->rh_run.ready = false;
  if (ctx->kept.read.cap == 0) CKR(gvs_reserve_rows(ctx, ctx->kept, 1));
  if (ctx->read_len.cap == 0) CKR(gvs_reserve(ctx, ctx->read_len, 16));
  ctx->stash.n = 0;
  ctx->have_read_len = true;
  ctx->read_off = nullptr;
  ctx->seq = nullptr;
  ctx->seg_tile_end.clear();
  ctx->seg_packed.clear();
  ctx->n_reads = ctx->stash_reads;
  ctx->total_bases = 0;
  ctx->stash_reads = 0;
  ctx->reads_ready = false;
  ctx->match_ready = false;
  ctx->diag_ready = true;
  ctx->val_ready = false;
  ctx->jn_in_run = false;
  if (n_rows) *n_rows = ctx->kept.n;
  if (n_reads) *n_reads = ctx->n_reads;
  return 0;
}
