// junctions.cu -- reads whose SUNKs jump from one contig to another: contig-end links, misjoins and phase switches.
// No reference counterpart: the diag filter keeps each read's rows on one best contig, and every later stage only sees
// those rows.  Definition: include/gavisunk_b200.h (gvs_junctions).
//
// Two phases, like the rest of a batches run:
//   gvs_junction_screen, per batch, on the match rows (every contig, before the diag filter drops any): one warp per
//     read segment.  Reads that are too short or whose rows all lie on one contig (nearly every read) leave after one
//     pass.  The others anchor their rows (pair tests), count distinct anchored IDs per contig without bad groups, and
//     when at least 2 contigs qualify, their anchored rows of qualifying contigs go to a run-long stash.
//   gvs_junctions, once the bad groups are known: one warp per stashed read drops bad rows, anchors again, and builds
//     qualifying contigs, runs, blocks, strands and records.
//
// The screen is exact.  Removing bad rows can only remove anchors: a row anchored without bad groups may lose its
// anchor, never the reverse, so the anchored rows and the qualifying contigs after the bad groups are subsets of the
// screen's.  A read with fewer than 2 qualifying contigs at the screen has fewer than 2 afterwards and no record.  And
// an anchored row's partner (same contig, other ID, ratio test) is itself anchored, on the same contig, so it is in the
// stash whenever the row is: anchoring the stashed rows again gives what anchoring all rows of the read would give.
#include "common.cuh"

#define JN_MIN_IDS 3  // distinct IDs for a qualifying contig and for a run (the >= 3-group rule of the intervals)

// per-row flag bits (jn_flags: byte 0 of a row)
#define JN_ANCH 1u  // not bad, anchored
#define JN_QUAL 2u  // anchored, on a qualifying contig
#define JN_SURV 4u  // QUAL, in a run of >= JN_MIN_IDS distinct IDs (a block row)

struct JnRows : SegRows {
  u8 *fa, *fb;  // per row: flag bits, scratch bit (first of its ID)
};

// ANCH and QUAL bits of the rows [a, b) of one read (one warp; fb is scratch)
__device__ void jn_qualify(const JnRows& R, u32 a, u32 b, int lane) {
  for (u32 i = a + lane; i < b; i += 32) {
    u8 f = 0;
    if (!R.is_bad(i)) {
      const u32 c = R.contig[i], id = R.group[i], p = R.pos[i], s = R.start[i];
      for (u32 j = a; j < b; j++) {
        if (R.contig[j] != c || R.group[j] == id || R.is_bad(j)) continue;
        if (gvs_ratio_ok(p, s, R.pos[j], R.start[j])) {
          f = JN_ANCH;
          break;
        }
      }
    }
    R.fa[i] = f;
  }
  __syncwarp();
  // the first anchored row of each (contig, ID)
  for (u32 i = a + lane; i < b; i += 32) {
    u8 first = 0;
    if (R.fa[i] & JN_ANCH) {
      const u32 c = R.contig[i], id = R.group[i];
      first = 1;
      for (u32 j = a; j < i; j++)
        if ((R.fa[j] & JN_ANCH) && R.contig[j] == c && R.group[j] == id) {
          first = 0;
          break;
        }
    }
    R.fb[i] = first;
  }
  __syncwarp();
  // qualifying contig: >= JN_MIN_IDS distinct anchored IDs (each lane writes only its own rows' fa)
  for (u32 i = a + lane; i < b; i += 32) {
    if (!(R.fa[i] & JN_ANCH)) continue;
    const u32 c = R.contig[i];
    u32 n = 0;
    for (u32 j = a; j < b && n < JN_MIN_IDS; j++) n += (R.fb[j] && R.contig[j] == c) ? 1u : 0u;
    if (n >= JN_MIN_IDS) R.fa[i] |= JN_QUAL;
  }
  __syncwarp();
}

// per segment of the match rows: the rows it stashes (0 unless >= 2 contigs qualify)
__global__ void __launch_bounds__(256) k_jn_screen(const JnRows R, const ReadLens len, u32 min_len, u32* seg_cnt) {
  const u32 s = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (s >= R.n_seg) return;
  const u32 a = R.seg_start[s], b = R.seg_start[s + 1];
  const u32 c0 = R.contig[a];
  bool other = false;
  if (len(R.read[a]) >= min_len)
    for (u32 j = a + lane; j < b; j += 32) other |= R.contig[j] != c0;
  if (!__any_sync(0xFFFFFFFFu, other)) {  // too short, or every row on one contig
    if (lane == 0) seg_cnt[s] = 0;
    return;
  }
  jn_qualify(R, a, b, lane);
  u32 first = 0xFFFFFFFFu, n = 0;
  for (u32 i = a + lane; i < b; i += 32)
    if (R.fa[i] & JN_QUAL) {
      first = min(first, i);
      n++;
    }
  first = __reduce_min_sync(0xFFFFFFFFu, first);
  n = __reduce_add_sync(0xFFFFFFFFu, n);
  bool two = false;
  if (first != 0xFFFFFFFFu) {
    const u32 cq = R.contig[first];
    for (u32 i = a + lane; i < b; i += 32) two |= (R.fa[i] & JN_QUAL) && R.contig[i] != cq;
  }
  two = __any_sync(0xFFFFFFFFu, two);
  if (lane == 0) seg_cnt[s] = two ? n : 0u;
}

// QUAL rows of the segments with a count, to the stash at dst + seg_off[s], read indices + base
__global__ void __launch_bounds__(256) k_jn_fill(const JnRows R, const u32* __restrict__ seg_cnt, const u32* __restrict__ seg_off,
                                                 u32 base, u32* d_read, u32* d_pos, u32* d_contig, u32* d_start, u32* d_group,
                                                 u32* d_gidx) {
  const u32 s = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (s >= R.n_seg || seg_cnt[s] == 0) return;
  const u32 a = R.seg_start[s], b = R.seg_start[s + 1];
  u32 o = seg_off[s];
  for (u32 c0 = a; c0 < b; c0 += 32) {
    const u32 i = c0 + lane;
    const bool q = i < b && (R.fa[i] & JN_QUAL);
    const u32 m = __ballot_sync(0xFFFFFFFFu, q);
    if (q) {
      const u32 k = o + __popc(m & ((1u << lane) - 1));
      d_read[k] = R.read[i] + base;
      d_pos[k] = R.pos[i];
      d_contig[k] = R.contig[i];
      d_start[k] = R.start[i];
      d_group[k] = R.group[i];
      d_gidx[k] = R.gidx[i];
    }
    o += __popc(m);
  }
}

// per-row u32 scratch of gvs_junctions, indexed by row (R) or by (segment's first row + run / block index)
struct JnScratch {
  u32* idx;   // per QUAL row: its run, then (SURV rows) its block
  u32* nids;  // per run: distinct IDs; then per block: distinct IDs
  u32 *first, *last, *up, *down;  // per block: first / last row, ratio-passing pairs rising / falling
};

// runs of the flagged rows (fa & flag) on one contig, in row order (warp_runs)
__device__ __forceinline__ u32 jn_runs(const JnRows& R, u32 a, u32 b, u8 flag, u32* idx, u32* first_row, u32* last_row, int lane) {
  return warp_runs(a, b, [&](u32 i) { return (R.fa[i] & flag) != 0; }, [&](u32 i) { return R.contig[i]; }, idx, first_row,
                   last_row, lane);
}

// first flagged row of its ID within its run / block (warp_first_in)
__device__ __forceinline__ bool jn_first_in(const JnRows& R, const u32* idx, u32 a, u32 i, u8 flag) {
  return warp_first_in(idx, a, i, [&](u32 j) { return (R.fa[j] & flag) != 0; }, [&](u32 j) { return R.group[j]; });
}

// per stashed read: blocks, and the number of records (consecutive block pairs)
__global__ void __launch_bounds__(256) k_jn_resolve(const JnRows R, const JnScratch X, u32* seg_cnt) {
  const u32 s = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (s >= R.n_seg) return;
  const u32 a = R.seg_start[s], b = R.seg_start[s + 1];
  jn_qualify(R, a, b, lane);
  // runs of QUAL rows, and their distinct IDs
  const u32 nrun = jn_runs(R, a, b, JN_QUAL, X.idx, nullptr, nullptr, lane);
  for (u32 r = lane; r < nrun; r += 32) X.nids[a + r] = 0;
  __syncwarp();
  for (u32 i = a + lane; i < b; i += 32)
    if ((R.fa[i] & JN_QUAL) && jn_first_in(R, X.idx, a, i, JN_QUAL)) atomicAdd(&X.nids[a + X.idx[i]], 1u);
  __syncwarp();
  // runs of >= JN_MIN_IDS distinct IDs survive; blocks = maximal runs of surviving rows on one contig, which merges
  // the runs that dropping the short ones left adjacent (one pass: no surviving run is dropped afterwards)
  for (u32 i = a + lane; i < b; i += 32)
    if ((R.fa[i] & JN_QUAL) && X.nids[a + X.idx[i]] >= JN_MIN_IDS) R.fa[i] |= JN_SURV;
  __syncwarp();
  const u32 nblk = jn_runs(R, a, b, JN_SURV, X.idx, X.first, X.last, lane);
  for (u32 k = lane; k < nblk; k += 32) X.nids[a + k] = X.up[a + k] = X.down[a + k] = 0;
  __syncwarp();
  if (nblk >= 2) {
    for (u32 i = a + lane; i < b; i += 32) {
      if (!(R.fa[i] & JN_SURV)) continue;
      const u32 k = X.idx[i], id = R.group[i], p = R.pos[i], st = R.start[i];
      if (jn_first_in(R, X.idx, a, i, JN_SURV)) atomicAdd(&X.nids[a + k], 1u);
      // strand: pairs of the block with different IDs that pass the ratio test, by the sign of dpos * dstart
      u32 up = 0, down = 0;
      for (u32 j = i + 1, e = X.last[a + k]; j <= e; j++) {
        if (!(R.fa[j] & JN_SURV) || R.group[j] == id || !gvs_ratio_ok(p, st, R.pos[j], R.start[j])) continue;
        if ((R.pos[j] > p) == (R.start[j] > st)) up++; else down++;
      }
      if (up) atomicAdd(&X.up[a + k], up);
      if (down) atomicAdd(&X.down[a + k], down);
    }
  }
  if (lane == 0) seg_cnt[s] = nblk >= 2 ? nblk - 1 : 0u;
}

extern "C" int gvs_junction_screen(gvs_ctx* ctx, uint32_t min_read_len, uint64_t* stash_rows, uint64_t* stash_reads) {
  if (!ctx) return GVS_E_ARG;
  if (!ctx->match_ready) return gvs_fail(ctx, GVS_E_STATE, "gvs_junction_screen before gvs_match / gvs_rows_set(0)");
  if (!ctx->read_off && !ctx->have_read_len) return gvs_fail(ctx, GVS_E_STATE, "gvs_junction_screen: read lengths unknown");
  CK(cudaSetDevice(ctx->device));
  StageTimer tm(ctx, GVS_ST_SCREEN);
  ctx->jn.ready = false;
  if (!ctx->jn_in_run) {  // outside a batches run a screen replaces the stash
    ctx->jn_stash.n = 0;
    ctx->jn_reads = 0;
  }
  // read indices as gvs_batch_stash will number this batch's reads
  const u64 base = ctx->jn_in_run ? ctx->stash_reads : 0, have = ctx->jn_stash.n;
  const Rows& M = ctx->rows;
  const u64 n = M.n;
  if (n) {
    if (base + ctx->n_reads >= 0xFFFFFFF0ull) return gvs_fail(ctx, GVS_E_OVERFLOW, "more than 2^32 reads in one run");
    u64 n_seg = 0;
    CKR(gvs_build_segments(ctx, M.read.as<u32>(), n, ctx->jn_seg_start, ctx->jn_row_seg, &n_seg));
    JnRows R;
    (SegRows&)R = seg_rows(ctx, M, ctx->jn_seg_start, n_seg);
    R.bad = nullptr;  // bad groups are not known before the run's histogram
    CKR(gvs_reserve(ctx, ctx->jn_flags, n * 2));
    R.fa = ctx->jn_flags.as<u8>();
    R.fb = R.fa + n;
    CKR(gvs_reserve(ctx, ctx->jn_seg_cnt, n_seg * 8));
    u32 *seg_cnt = ctx->jn_seg_cnt.as<u32>(), *seg_off = seg_cnt + n_seg;
    LAUNCH(k_jn_screen, (unsigned)cdiv(n_seg * 32, 256), 256, 0, R, read_lens(ctx), min_read_len, seg_cnt);
    u64 packed = 0;  // (reads << 32) + rows
    {
      auto f = [seg_cnt] __device__(u64 s) -> u64 { return seg_cnt[s] ? (1ull << 32) | seg_cnt[s] : 0ull; };
      auto g = [seg_off] __device__(u64 s, u64 ex, u64 v) { seg_off[s] = (u32)ex; };
      CKR(scan_total(ctx, n_seg, f, g, OpSum(), &packed));
    }
    const u64 add = packed & 0xFFFFFFFFull;
    if (add) {
      if (have + add >= 0xFFFFFFF0ull) return gvs_fail(ctx, GVS_E_OVERFLOW, "more than 2^32 junction rows in one run");
      Rows& S = ctx->jn_stash;
      DevBuf* dst[6] = {&S.read, &S.pos, &S.contig, &S.start, &S.group, &S.gidx};
      for (DevBuf* d : dst) CKR(grow_keep(ctx, *d, (have + add) * 4, have * 4));
      LAUNCH(k_jn_fill, (unsigned)cdiv(n_seg * 32, 256), 256, 0, R, seg_cnt, seg_off, (u32)base, S.read.as<u32>() + have,
             S.pos.as<u32>() + have, S.contig.as<u32>() + have, S.start.as<u32>() + have, S.group.as<u32>() + have,
             S.gidx.as<u32>() + have);
      S.n = have + add;
      ctx->jn_reads += packed >> 32;
    }
  }
  if (stash_rows) *stash_rows = ctx->jn_stash.n;
  if (stash_reads) *stash_reads = ctx->jn_reads;
  return 0;
}

extern "C" int gvs_junctions(gvs_ctx* ctx, uint64_t* n_records) {
  if (!ctx) return GVS_E_ARG;
  CK(cudaSetDevice(ctx->device));
  StageTimer tm(ctx, GVS_ST_JUNCTIONS);
  ctx->jn.ready = false;
  ctx->jn.n = 0;
  if (n_records) *n_records = 0;
  const Rows& S = ctx->jn_stash;
  const u64 n = S.n;
  if (n == 0) {
    ctx->jn.ready = true;
    return 0;
  }
  u64 n_seg = 0;
  CKR(gvs_build_segments(ctx, S.read.as<u32>(), n, ctx->jn_seg_start, ctx->jn_row_seg, &n_seg));
  JnRows R;
  (SegRows&)R = seg_rows(ctx, S, ctx->jn_seg_start, n_seg);
  CKR(gvs_reserve(ctx, ctx->jn_flags, n * 2));
  R.fa = ctx->jn_flags.as<u8>();
  R.fb = R.fa + n;
  CKR(gvs_reserve(ctx, ctx->jn_scr, n * 6 * 4));
  JnScratch X;
  X.idx = ctx->jn_scr.as<u32>();
  X.nids = X.idx + n; X.first = X.nids + n; X.last = X.first + n; X.up = X.last + n; X.down = X.up + n;
  CKR(gvs_reserve(ctx, ctx->jn_seg_cnt, n_seg * 8));
  u32* seg_cnt = ctx->jn_seg_cnt.as<u32>();
  LAUNCH(k_jn_resolve, (unsigned)cdiv(n_seg * 32, 256), 256, 0, R, X, seg_cnt);
  // a block holds >= 3 rows, so a read has fewer records than rows / 3
  const u64 stride = n / JN_MIN_IDS + 1;
  CKR(rec_reserve(ctx, ctx->jn, 13, stride));
  u32* rec = ctx->jn.col(0);
  u32 nr = 0;
  {
    const JnRows Rc = R;
    const JnScratch Xc = X;
    auto f = [seg_cnt] __device__(u64 s) -> u32 { return seg_cnt[s]; };
    auto g = [Rc, Xc, rec, stride] __device__(u64 s, u32 ex, u32 v) {
      const u32 a = Rc.seg_start[s];
      for (u32 t = 0; t < v; t++) {
        const u32 k = a + t, i = Xc.last[k], j = Xc.first[k + 1];
        u32* o = rec + ex + t;  // columns as in gvs_junctions_get; strand 0 = '+' (a tie counts as rising)
        o[0] = Rc.read[a];
        o[stride] = Rc.contig[i];
        o[2 * stride] = Xc.up[k] >= Xc.down[k] ? 0u : 1u;
        o[3 * stride] = Xc.nids[k];
        o[4 * stride] = Rc.group[i];
        o[5 * stride] = Rc.start[i];
        o[6 * stride] = Rc.pos[i];
        o[7 * stride] = Rc.contig[j];
        o[8 * stride] = Xc.up[k + 1] >= Xc.down[k + 1] ? 0u : 1u;
        o[9 * stride] = Xc.nids[k + 1];
        o[10 * stride] = Rc.group[j];
        o[11 * stride] = Rc.start[j];
        o[12 * stride] = Rc.pos[j];
      }
    };
    CKR(scan_total(ctx, n_seg, f, g, OpSum(), &nr));
  }
  ctx->jn.n = nr;
  ctx->jn.ready = true;
  if (n_records) *n_records = nr;
  return 0;
}

extern "C" int gvs_junctions_get(gvs_ctx* ctx, uint32_t* read, uint32_t* contig1, uint32_t* strand1, uint32_t* ids1, uint32_t* id1,
                                 uint32_t* start1, uint32_t* pos1, uint32_t* contig2, uint32_t* strand2, uint32_t* ids2,
                                 uint32_t* id2, uint32_t* start2, uint32_t* pos2) {
  return ctx ? rec_get(ctx, ctx->jn, "gvs_junctions_get before gvs_junctions",
                       {read, contig1, strand1, ids1, id1, start1, pos1, contig2, strand2, ids2, id2, start2, pos2})
             : GVS_E_ARG;
}
