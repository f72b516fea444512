// rowsio.cu -- rows / read tables supplied by the host instead of the previous GPU stage: what the
// per-rule CLI shims need (diag_filter_v3 <sunkpos> <fai>, badsunks_AR.py, process-by-contig...),
// where the reference exchanges .sunkpos / .rlen files between processes (SURVEY.md 8b).
#include "table.cuh"

int gvs_reserve_rows(gvs_ctx* ctx, Rows& r, u64 n) {
  CKR(gvs_reserve(ctx, r.read, n * 4));
  CKR(gvs_reserve(ctx, r.pos, n * 4));
  CKR(gvs_reserve(ctx, r.contig, n * 4));
  CKR(gvs_reserve(ctx, r.start, n * 4));
  CKR(gvs_reserve(ctx, r.group, n * 4));
  CKR(gvs_reserve(ctx, r.gidx, n * 4));
  return 0;
}

__global__ void k_gt_fill(u64* keys, u64 n) {
  for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) keys[i] = GVS_EMPTY_KEY;
}
__global__ void k_gt_insert(const u32* __restrict__ grp_contig, const u32* __restrict__ grp_start, u64 n_groups, u64* keys,
                            u32* val, u64 slots) {
  u64 g = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= n_groups) return;
  u64 key = ((u64)grp_contig[g] << 32) | grp_start[g];
  u64 s = tab_insert(keys, slots, key, gvs_mix(key));
  val[s] = (u32)g;
}
__global__ void k_gt_lookup(const u32* __restrict__ contig, const u32* __restrict__ group, u64 n, const u64* __restrict__ keys,
                            const u32* __restrict__ val, u64 slots, u32* gidx, u32* missing) {
  u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  u64 key = ((u64)contig[i] << 32) | group[i];
  u64 nb = slots >> 2, b = gvs_tab_bucket(gvs_mix(key), slots);
  for (u64 it = 0; it < nb; it++) {
    for (int j = 0; j < 4; j++) {
      u64 cur = keys[(b << 2) + j];
      if (cur == key) { gidx[i] = val[(b << 2) + j]; return; }
      if (cur == GVS_EMPTY_KEY) { gidx[i] = 0; atomicAdd(missing, 1u); return; }
    }
    b = (b + 1) & (nb - 1);
  }
  gidx[i] = 0;
  atomicAdd(missing, 1u);
}

static int ensure_group_table(gvs_ctx* ctx) {
  if (ctx->gt_slots) return 0;
  u64 ng = ctx->n_groups;
  u64 slots = next_pow2(ng * 2 < 1024 ? 1024 : ng * 2);
  CKR(gvs_reserve(ctx, ctx->gt_keys, slots * 8));
  CKR(gvs_reserve(ctx, ctx->gt_val, slots * 4));
  LAUNCH(k_gt_fill, (unsigned)(cdiv(slots, 256) > 4096 ? 4096 : cdiv(slots, 256)), 256, 0, ctx->gt_keys.as<u64>(), slots);
  if (ng)
    LAUNCH(k_gt_insert, (unsigned)cdiv(ng, 256), 256, 0, ctx->grp_contig.as<u32>(), ctx->grp_start.as<u32>(), ng,
           ctx->gt_keys.as<u64>(), ctx->gt_val.as<u32>(), slots);
  ctx->gt_slots = slots;
  return 0;
}

extern "C" int gvs_reads_meta(gvs_ctx* ctx, const uint32_t* read_len, uint64_t n_reads, const uint64_t* chunk_first,
                              const uint8_t* chunk_hap, uint32_t n_chunks) {
  if (!ctx) return GVS_E_ARG;
  CK(cudaSetDevice(ctx->device));
  if (!chunk_first || !chunk_hap || n_chunks == 0) return gvs_fail(ctx, GVS_E_ARG, "null chunk arrays");
  if (chunk_first[0] != 0 || chunk_first[n_chunks] != n_reads) return gvs_fail(ctx, GVS_E_ARG, "chunk_first must span [0, n_reads]");
  for (u32 c = 0; c < n_chunks; c++)
    if (chunk_hap[c] > GVS_HAP_ANY) return gvs_fail(ctx, GVS_E_ARG, "chunk haplotype %u (0, 1 or GVS_HAP_ANY)", chunk_hap[c]);
  CKR(gvs_pipe_join(ctx));
  ctx->seg_tile_end.clear();
  ctx->seg_packed.clear();
  ctx->reads_ready = false;
  ctx->match_ready = ctx->diag_ready = ctx->val_ready = false;
  ctx->seq = nullptr;
  ctx->read_off = nullptr;
  ctx->n_reads = n_reads;
  ctx->total_bases = 0;
  ctx->n_chunks = n_chunks;
  ctx->h_chunk_first.assign(chunk_first, chunk_first + n_chunks + 1);
  ctx->h_chunk_hap.assign(chunk_hap, chunk_hap + n_chunks);
  CKR(to_dev(ctx, ctx->chunk_first, chunk_first, (size_t)n_chunks + 1));
  CKR(to_dev(ctx, ctx->chunk_hap, chunk_hap, (size_t)n_chunks));
  ctx->have_read_len = read_len != nullptr;
  if (read_len) CKR(to_dev(ctx, ctx->read_len, read_len, n_reads));
  CK(cudaStreamSynchronize(ctx->stream));
  return 0;
}

extern "C" int gvs_rows_set(gvs_ctx* ctx, int which, const uint32_t* read_idx, const uint32_t* pos, const uint32_t* contig,
                            const uint32_t* start, const uint32_t* group, uint64_t n, uint32_t n_contigs) {
  if (!ctx) return GVS_E_ARG;
  if (which != 0 && which != 1) return gvs_fail(ctx, GVS_E_ARG, "which must be 0 or 1");
  if (n && (!read_idx || !pos || !contig || !start || !group)) return gvs_fail(ctx, GVS_E_ARG, "null row column");
  if (ctx->n_chunks == 0) return gvs_fail(ctx, GVS_E_STATE, "gvs_rows_set: call gvs_reads_set / gvs_reads_meta first");
  CK(cudaSetDevice(ctx->device));
  {
    // rows index the read table and the contig tables of later stages (read_len[read], contig_hap[contig]): a row
    // outside them would be an out-of-bounds device read there, so it is refused here
    const u64 nc = ctx->db_ready ? ctx->n_contigs : n_contigs;
    for (u64 i = 0; i < n; i++) {
      if (read_idx[i] >= ctx->n_reads)
        return gvs_fail(ctx, GVS_E_ARG, "row %llu: read index %u outside the read table (%llu reads)", (unsigned long long)i,
                        read_idx[i], (unsigned long long)ctx->n_reads);
      if (contig[i] >= nc)
        return gvs_fail(ctx, GVS_E_ARG, "row %llu: contig %u outside the contig list (%llu contigs)", (unsigned long long)i, contig[i],
                        (unsigned long long)nc);
    }
  }
  Rows& R = which == 0 ? ctx->rows : ctx->kept;
  CKR(gvs_reserve_rows(ctx, R, n));
  if (n) {
    CK(cudaMemcpyAsync(R.read.p, read_idx, n * 4, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(R.pos.p, pos, n * 4, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(R.contig.p, contig, n * 4, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(R.start.p, start, n * 4, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(R.group.p, group, n * 4, cudaMemcpyHostToDevice, ctx->stream));
  }
  if (ctx->db_ready) {
    CKR(ensure_group_table(ctx));
    u32* miss = counter(ctx, CNT_MISS);
    CK(cudaMemsetAsync(miss, 0, 4, ctx->stream));
    if (n)
      LAUNCH(k_gt_lookup, (unsigned)cdiv(n, 256), 256, 0, R.contig.as<u32>(), R.group.as<u32>(), n, ctx->gt_keys.as<u64>(),
             ctx->gt_val.as<u32>(), ctx->gt_slots, R.gidx.as<u32>(), miss);
    u32 m = 0;
    CKR(read_dev(ctx, miss, &m));
    if (m) return gvs_fail(ctx, GVS_E_ARG, "%u rows name a (contig, group) that is not in the database", m);
  } else {
    ctx->n_contigs = n_contigs;
    CKR(gvs_group_index_rows(ctx, R.contig.as<u32>(), R.group.as<u32>(), n, R.gidx.as<u32>()));
    ctx->groups_ready = true;
  }
  CK(cudaStreamSynchronize(ctx->stream));
  R.n = n;
  if (which == 0) {
    ctx->match_ready = true;
    ctx->diag_ready = ctx->val_ready = false;
  } else {
    ctx->diag_ready = true;
    ctx->val_ready = false;
  }
  return 0;
}
