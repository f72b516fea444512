// table.cu -- SUNK probe table + filter construction from .loc rows (kmerpos_annot3's table
// load, workflow/src/kmerpos_annot3.nim:20-26,57-69) and database export.
#include "table.cuh"
#include <stdlib.h>

// ---- kernels -------------------------------------------------------------------------------
__global__ void k_fill_u64(u64* p, u64 n, u64 v) {
  for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) p[i] = v;
}
__global__ void k_fill_u32(u32* p, u64 n, u32 v) {
  for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) p[i] = v;
}

// .loc rows: later rows of the same k-mer win (nim:68 `coords[...] = curcoord`): slot value =
// max(row index + 1)
__global__ void k_tab_insert_loc(const u64* __restrict__ kmer, u64 n, u64* keys, u32* rows, u64 slots) {
  for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
    u64 key = kmer[i];
    u64 s = tab_insert(keys, slots, key, gvs_mix(key));
    atomicMax(&rows[s], (u32)(i + 1));
  }
}
// db set membership (nim:20-26): bit 31 of the slot value
__global__ void k_tab_mark_db(const u64* __restrict__ kmer, u64 n, u64* keys, u32* rows, u64 slots) {
  for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
    u64 key = kmer[i];
    u64 s = tab_insert(keys, slots, key, gvs_mix(key));
    atomicOr(&rows[s], 0x80000000u);
  }
}
__global__ void k_tab_finalize(const u64* __restrict__ keys, u32* rows, u64 slots, u32* filt, u64 filt_blocks, int k,
                               u32* filt1, u32 filt1_words, int fp_layout) {
  const int J = GVS_FJ(k), L = k - J + 1;
  const u64 lmask = (L >= 32) ? ~0ull : ((1ull << (2 * L)) - 1);
  for (u64 s = (u64)blockIdx.x * blockDim.x + threadIdx.x; s < slots; s += (u64)gridDim.x * blockDim.x) {
    u64 key = keys[s];
    if (key == GVS_EMPTY_KEY) continue;
    u32 v = rows[s];
    u32 r = v & 0x7FFFFFFFu;
    if (!(v >> 31)) {
      rows[s] = GVS_ROW_NOTINDB;  // in .loc but not in the db set: `x in uniqueKmers` is false
      continue;
    }
    rows[s] = r ? r - 1 : GVS_ROW_MISSING;
    // one insertion per sub-mer offset: J consecutive read windows then share a single block
    u32 h = gvs_fhash(key);
    for (int j = 0; j < J; j++) {
      u64 sub = (key >> (2 * (J - 1 - j))) & lmask;
      u64 rc = gvs_revcomp(sub, L);
      u32 hb = gvs_bhash(sub < rc ? sub : rc);
      u64 blk = hb & (filt_blocks - 1);
      atomicOr(&filt1[gvs_p1_word(hb, filt1_words)], gvs_p1_bits(hb));
      atomicOr(&filt[4 * blk + 0], 1u << (h & 31));
      atomicOr(&filt[4 * blk + 1], 1u << ((h >> 5) & 31));
      atomicOr(&filt[4 * blk + 2], 1u << ((h >> 10) & 31));
      atomicOr(&filt[4 * blk + 3], 1u << (fp_layout ? gvs_fp_bit(hb) : ((h >> 15) & 31)));
    }
  }
}

// group identity (contig, group start) -> representative (first) row, through a scratch table
__global__ void k_grp_insert(const u32* __restrict__ contig, const u32* __restrict__ group, u64 n, u64* keys,
                             u32* minrow, u64 slots) {
  for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
    u64 key = ((u64)contig[i] << 32) | group[i];
    u64 s = tab_insert(keys, slots, key, gvs_mix(key));
    atomicMin(&minrow[s], (u32)i);
  }
}
__global__ void k_grp_rep(const u32* __restrict__ contig, const u32* __restrict__ group, u64 n, u64* keys,
                          const u32* __restrict__ minrow, u64 slots, u32* rep) {
  for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
    u64 key = ((u64)contig[i] << 32) | group[i];
    u64 s = tab_insert(keys, slots, key, gvs_mix(key));
    rep[i] = minrow[s];
  }
}
__global__ void k_grp_fill(const u32* __restrict__ rep, const u32* __restrict__ dense_of_row, u64 n, u32* gidx,
                           const u32* __restrict__ contig, const u32* __restrict__ group, u32* grp_contig,
                           u32* grp_start) {
  for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
    u32 r = rep[i];
    u32 g = dense_of_row[r];
    gidx[i] = g;
    if (r == i) {
      grp_contig[g] = contig[i];
      grp_start[g] = group[i];
    }
  }
}

static unsigned grid_for(gvs_ctx* ctx, u64 n, int block) {
  u64 g = cdiv(n, block);
  u64 cap = (u64)ctx->n_sm * 16;
  if (g > cap) g = cap;
  if (g == 0) g = 1;
  return (unsigned)g;
}

// Build tab_keys/tab_rows/filt from ctx->loc_kmer (device) and a device array of db k-mers
// (d_db_kmer == nullptr: the db set is exactly the .loc k-mers).
int gvs_tab_build_impl(gvs_ctx* ctx, const u64* d_db_kmer, u64 n_db) {
  u64 n_loc = ctx->n_loc;
  u64 nk = n_loc + (d_db_kmer ? n_db : 0);
  u64 slots = next_pow2(nk * 2 < 1024 ? 1024 : nk * 2);
  if (n_loc >= 0x7FFFFFF0ull) return gvs_fail(ctx, GVS_E_OVERFLOW, "more than 2^31 .loc rows");
  ctx->tab_slots = slots;
  CKR(gvs_reserve(ctx, ctx->tab_keys, slots * sizeof(u64)));
  CKR(gvs_reserve(ctx, ctx->tab_rows, slots * sizeof(u32)));
  // blocked filter: 16-byte blocks, J insertions per key, ~12 entries per block (FP ~1 %), power of
  // two; 32 MiB for 5.9 M SUNKs (L2-resident), capped at 2^27 blocks (2 GiB) for human-size databases
  u64 fw = next_pow2(cdiv((n_loc ? n_loc : 1) * (u64)GVS_FJ(ctx->k), 12));
  if (fw < (1ull << 10)) fw = 1ull << 10;
  if (fw > (1ull << 27)) fw = 1ull << 27;
  ctx->filt_words = fw;  // number of blocks
  // beyond L2 (or forced by gvs_set_probe_variant): the large-database probe variant and its block layout
  ctx->filt_fp = ctx->probe_variant == 2 || (ctx->probe_variant == 0 && fw * 16 > (32ull << 20));
  CKR(gvs_reserve(ctx, ctx->filt, fw * 16));
  // presence filter of the sub-mers in front of it: ~16 bits per distinct sub-mer, at most 64 MiB (L2)
  {
    u64 w1 = next_pow2((n_loc ? n_loc : 1) * 5 / 8);
    if (w1 < (1ull << 10)) w1 = 1ull << 10;
    if (w1 > (1ull << 24)) w1 = 1ull << 24;
    if (const char* e = getenv("GVS_EXP_FILT1_LOG2W")) {  // experiments: presence filter size (log2 of its 32-bit words)
      int l2 = atoi(e);
      if (l2 >= 10 && l2 <= 28) w1 = 1ull << l2;
    }
    if (const char* e = getenv("GVS_EXP_FILT1_MIB")) {  // experiments: presence filter size in MiB (any value)
      int mib = atoi(e);
      if (mib >= 1 && mib <= 1024) w1 = (u64)mib << 18;
    }
    ctx->filt1_words = w1;
    CKR(gvs_reserve(ctx, ctx->filt1, w1 * 4));
    LAUNCH(k_fill_u32, grid_for(ctx, w1, 256), 256, 0, ctx->filt1.as<u32>(), w1, 0u);
  }
  u64* keys = ctx->tab_keys.as<u64>();
  u32* rows = ctx->tab_rows.as<u32>();
  LAUNCH(k_fill_u64, grid_for(ctx, slots, 256), 256, 0, keys, slots, GVS_EMPTY_KEY);
  LAUNCH(k_fill_u32, grid_for(ctx, slots, 256), 256, 0, rows, slots, 0u);
  LAUNCH(k_fill_u32, grid_for(ctx, fw * 4, 256), 256, 0, ctx->filt.as<u32>(), fw * 4, 0u);
  if (n_loc) LAUNCH(k_tab_insert_loc, grid_for(ctx, n_loc, 256), 256, 0, ctx->loc_kmer.as<u64>(), n_loc, keys, rows, slots);
  if (d_db_kmer) {
    if (n_db) LAUNCH(k_tab_mark_db, grid_for(ctx, n_db, 256), 256, 0, d_db_kmer, n_db, keys, rows, slots);
  } else if (n_loc) {
    LAUNCH(k_tab_mark_db, grid_for(ctx, n_loc, 256), 256, 0, ctx->loc_kmer.as<u64>(), n_loc, keys, rows, slots);
  }
  LAUNCH(k_tab_finalize, grid_for(ctx, slots, 256), 256, 0, keys, rows, slots, ctx->filt.as<u32>(), fw, ctx->k,
         ctx->filt1.as<u32>(), (u32)ctx->filt1_words, ctx->filt_fp ? 1 : 0);
  return 0;
}

__global__ void k_loc_pack(const u32* __restrict__ contig, const u32* __restrict__ start, const u32* __restrict__ group, u64 n, uint4* out) {
  for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x)
    out[i] = make_uint4(contig[i], start[i], group[i], 0u);
}
__global__ void k_tab_kv(const u64* __restrict__ keys, const u32* __restrict__ rows, u64 slots, const u32* __restrict__ loc_gidx, u64 n_loc,
                         u64* kv) {
  for (u64 s = (u64)blockIdx.x * blockDim.x + threadIdx.x; s < slots; s += (u64)gridDim.x * blockDim.x) {
    const u32 r = rows[s];
    const u64 o = ((s >> 2) << 3) + (s & 3);  // bucket * 8 + slot: keys; + 4: values
    kv[o] = keys[s];
    kv[o + 4] = ((u64)(r < n_loc ? loc_gidx[r] : 0xFFFFFFFFu) << 32) | r;
  }
}
// the probe's table: every bucket's 4 keys and 4 (row, group index) words in one 64-byte unit, so that a lookup is a
// single access to HBM; the key and row arrays of the build are released
int gvs_tab_attach_gidx(gvs_ctx* ctx) {
  CKR(gvs_reserve(ctx, ctx->tab_kv, ctx->tab_slots * 2 * sizeof(u64)));
  LAUNCH(k_tab_kv, grid_for(ctx, ctx->tab_slots, 256), 256, 0, ctx->tab_keys.as<u64>(), ctx->tab_rows.as<u32>(), ctx->tab_slots,
         ctx->loc_gidx.as<u32>(), ctx->n_loc, ctx->tab_kv.as<u64>());
  // the emit pass turns a hit's .loc row into (contig, start, group): one 16-byte load instead of three scattered 4-byte ones
  CKR(gvs_reserve(ctx, ctx->loc_pack, (ctx->n_loc ? ctx->n_loc : 1) * sizeof(uint4)));
  if (ctx->n_loc)
    LAUNCH(k_loc_pack, grid_for(ctx, ctx->n_loc, 256), 256, 0, ctx->loc_contig.as<u32>(), ctx->loc_start.as<u32>(), ctx->loc_group.as<u32>(),
           ctx->n_loc, ctx->loc_pack.as<uint4>());
  CK(cudaStreamSynchronize(ctx->stream));
  gvs_release(ctx->tab_rows);
  gvs_release(ctx->tab_keys);
  return 0;
}

// dense group index by first appearance of (contig, group) in .loc row order
static int build_group_index_body(gvs_ctx* ctx, const u32* contig, const u32* group, u64 n, u32* gidx_out, DevBuf& gk,
                                  DevBuf& gm, DevBuf& rep, DevBuf& dense, u64 slots) {
  LAUNCH(k_fill_u64, grid_for(ctx, slots, 256), 256, 0, gk.as<u64>(), slots, GVS_EMPTY_KEY);
  LAUNCH(k_fill_u32, grid_for(ctx, slots, 256), 256, 0, gm.as<u32>(), slots, 0xFFFFFFFFu);
  LAUNCH(k_grp_insert, grid_for(ctx, n, 256), 256, 0, contig, group, n, gk.as<u64>(), gm.as<u32>(), slots);
  LAUNCH(k_grp_rep, grid_for(ctx, n, 256), 256, 0, contig, group, n, gk.as<u64>(), gm.as<u32>(), slots, rep.as<u32>());
  const u32* repp = rep.as<u32>();
  u32* densep = dense.as<u32>();
  auto f = [repp] __device__(u64 i) -> u32 { return repp[i] == (u32)i ? 1u : 0u; };
  auto g = [densep] __device__(u64 i, u32 ex, u32 v) { densep[i] = ex; };
  u32 ng = 0;
  CKR(scan_total(ctx, n, f, g, OpSum(), &ng));
  ctx->n_groups = ng;
  CKR(gvs_reserve(ctx, ctx->grp_contig, (u64)ng * sizeof(u32)));
  CKR(gvs_reserve(ctx, ctx->grp_start, (u64)ng * sizeof(u32)));
  LAUNCH(k_grp_fill, grid_for(ctx, n, 256), 256, 0, repp, densep, n, gidx_out, contig, group,
         ctx->grp_contig.as<u32>(), ctx->grp_start.as<u32>());
  CK(cudaStreamSynchronize(ctx->stream));
  return 0;
}

// dense index of the distinct (contig, group) pairs of n rows, in order of first appearance;
// fills gidx_out[n], ctx->n_groups, ctx->grp_contig / grp_start
int gvs_group_index_rows(gvs_ctx* ctx, const u32* contig, const u32* group, u64 n, u32* gidx_out) {
  CKR(gvs_reserve(ctx, ctx->counters, 64 * sizeof(u64)));
  ctx->grp_gen++;
  if (n == 0) {
    ctx->n_groups = 0;
    return gvs_check_group_order(ctx);
  }
  u64 slots = next_pow2(n * 2 < 1024 ? 1024 : n * 2);
  DevBuf gk, gm, rep, dense;
  int rc = gvs_reserve(ctx, gk, slots * sizeof(u64));
  if (!rc) rc = gvs_reserve(ctx, gm, slots * sizeof(u32));
  if (!rc) rc = gvs_reserve(ctx, rep, n * sizeof(u32));
  if (!rc) rc = gvs_reserve(ctx, dense, n * sizeof(u32));
  if (!rc) rc = build_group_index_body(ctx, contig, group, n, gidx_out, gk, gm, rep, dense, slots);
  if (!rc) rc = gvs_check_group_order(ctx);
  cudaStreamSynchronize(ctx->stream);
  gvs_release(gk); gvs_release(gm); gvs_release(rep); gvs_release(dense);
  return rc;
}

static int build_group_index(gvs_ctx* ctx) {
  CKR(gvs_reserve(ctx, ctx->loc_gidx, ctx->n_loc * sizeof(u32)));
  return gvs_group_index_rows(ctx, ctx->loc_contig.as<u32>(), ctx->loc_group.as<u32>(), ctx->n_loc, ctx->loc_gidx.as<u32>());
}

// ---- C ABI ---------------------------------------------------------------------------------
extern "C" int gvs_db_load_loc(gvs_ctx* ctx, const uint64_t* db_kmer, uint64_t n_db, const uint64_t* loc_kmer,
                               const uint32_t* loc_contig, const uint32_t* loc_start, const uint32_t* loc_group,
                               uint64_t n_loc, uint32_t n_contigs) {
  if (!ctx) return GVS_E_ARG;
  if (n_loc && (!loc_kmer || !loc_contig || !loc_start || !loc_group)) return gvs_fail(ctx, GVS_E_ARG, "null .loc column");
  CK(cudaSetDevice(ctx->device));
  ctx->db_ready = false;
  ctx->n_loc = n_loc;
  ctx->n_contigs = n_contigs;
  CKR(to_dev(ctx, ctx->loc_kmer, loc_kmer, n_loc));
  CKR(to_dev(ctx, ctx->loc_contig, loc_contig, n_loc));
  CKR(to_dev(ctx, ctx->loc_start, loc_start, n_loc));
  CKR(to_dev(ctx, ctx->loc_group, loc_group, n_loc));
  DevBuf dbk;
  int rc = 0;
  if (db_kmer || n_db == 0) {
    rc = to_dev(ctx, dbk, db_kmer, n_db);
    if (!rc) rc = gvs_tab_build_impl(ctx, dbk.as<u64>(), n_db);
  } else {
    rc = gvs_fail(ctx, GVS_E_ARG, "null db_kmer with n_db > 0");
  }
  if (!rc) rc = build_group_index(ctx);
  if (!rc) rc = gvs_tab_attach_gidx(ctx);
  cudaStreamSynchronize(ctx->stream);
  gvs_release(dbk);
  if (rc) return rc;
  ctx->db_ready = true;
  ctx->groups_ready = true;
  ctx->gt_slots = 0;
  return 0;
}

extern "C" int gvs_db_size(gvs_ctx* ctx, uint64_t* n_sunks, uint64_t* n_groups) {
  if (!ctx) return GVS_E_ARG;
  if (!ctx->db_ready) return gvs_fail(ctx, GVS_E_STATE, "no database");
  if (n_sunks) *n_sunks = ctx->n_loc;
  if (n_groups) *n_groups = ctx->n_groups;
  return 0;
}

extern "C" int gvs_db_export(gvs_ctx* ctx, uint64_t* kmer, uint32_t* contig, uint32_t* start, uint32_t* group,
                             uint32_t* group_index) {
  if (!ctx) return GVS_E_ARG;
  if (!ctx->db_ready) return gvs_fail(ctx, GVS_E_STATE, "no database");
  CK(cudaSetDevice(ctx->device));
  u64 n = ctx->n_loc;
  if (n == 0) return 0;
  if (kmer) CK(cudaMemcpyAsync(kmer, ctx->loc_kmer.p, n * 8, cudaMemcpyDeviceToHost, ctx->stream));
  if (contig) CK(cudaMemcpyAsync(contig, ctx->loc_contig.p, n * 4, cudaMemcpyDeviceToHost, ctx->stream));
  if (start) CK(cudaMemcpyAsync(start, ctx->loc_start.p, n * 4, cudaMemcpyDeviceToHost, ctx->stream));
  if (group) CK(cudaMemcpyAsync(group, ctx->loc_group.p, n * 4, cudaMemcpyDeviceToHost, ctx->stream));
  if (group_index) CK(cudaMemcpyAsync(group_index, ctx->loc_gidx.p, n * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return 0;
}
