// inversions.cu -- strand switches: reads whose SUNKs switch strand inside one contig (inversions, fold-back chimeras).
// No reference counterpart: the validation takes each read's orientation majority and drops the pairs of the other
// orientation, and an inversion keeps its length, so a read validates straight across it.  Definition:
// include/gavisunk_b200.h (gvs_strand_switches).
//
// One phase, after the bad groups, on the kept rows of the run (resident after gvs_batches_bind): k_sw_resolve runs one
// warp per read segment with no cap on rows.  Nearly every read leaves after one pass over its rows: a read whose usable
// rows (on its first row's contig, not bad) are in pos order and whose starts are monotone along them, in either
// direction, has no record.  That exit is exact: a ratio-passing pair has dpos != 0 and dstart != 0, so along monotone
// starts every such pair has the sign of the monotone direction, every oriented row takes that one strand, and one
// strand makes at most one block.  The other reads order their usable rows (a copy when pos is already non-decreasing in
// row order, else a rank sort), orient every row with O(m^2) pair tests, and cut blocks with the junction stage's run
// passes (warp_runs) keyed by strand.  A device scan places the records in (segment, block) order, and k_sw_emit
// writes them.
#include "common.cuh"

#define SW_MIN_IDS 3   // distinct IDs of a run that survives (the junction rule)
#define SW_MIN_ROWS 6  // usable rows a read needs for two blocks
#define SW_NONE 2u     // strand of an unoriented row
#define SW_SURV 4u     // flag: oriented row in a run of >= SW_MIN_IDS distinct IDs (a block row)

struct SwRows : SegRows {  // kept rows
  ReadLens len;
  u32 min_len;
};

// per-row scratch of gvs_strand_switches, indexed from the segment's first row a: by ordered position (a + k) or by run /
// block (a + r)
struct SwScratch {
  u32* ord;    // per ordered position: its row
  u32* idx;    // per ordered position: its run, then (SW_SURV) its block
  u32* nids;   // per run, then per block: distinct IDs
  u32 *first, *last;  // per block: first / last ordered position
  u32 *lo, *hi;       // per block: smallest / largest start
  u8* st;      // per ordered position: strand 0 / 1 or SW_NONE, | SW_SURV
};

// blocks of the read [a, b) with nu usable rows (sorted: their pos is non-decreasing in row order); returns their number
__device__ u32 sw_blocks(const SwRows& R, const SwScratch& X, u32 a, u32 b, u32 nu, bool sorted, int lane) {
  const u32 c0 = R.contig[a];
  auto usable = [&](u32 i) { return R.contig[i] == c0 && !R.is_bad(i); };
  // order: rows by (pos, row)
  if (sorted) {
    u32 o = a;
    for (u32 c = a; c < b; c += 32) {
      const u32 i = c + lane;
      const bool q = i < b && usable(i);
      const u32 m = __ballot_sync(0xFFFFFFFFu, q);
      if (q) X.ord[o + __popc(m & ((1u << lane) - 1))] = i;
      o += __popc(m);
    }
  } else {
    for (u32 i = a + lane; i < b; i += 32) {
      if (!usable(i)) continue;
      const u32 p = R.pos[i];
      u32 r = 0;
      for (u32 j = a; j < b; j++) r += usable(j) && (R.pos[j] < p || (R.pos[j] == p && j < i));
      X.ord[a + r] = i;
    }
  }
  __syncwarp();
  const u32 e = a + nu;
  // row strands
  for (u32 k = a + lane; k < e; k += 32) {
    const u32 i = X.ord[k], id = R.group[i], p = R.pos[i], s = R.start[i];
    u32 up = 0, down = 0;
    for (u32 t = a; t < e; t++) {
      const u32 j = X.ord[t];
      if (R.group[j] == id || !gvs_ratio_ok(p, s, R.pos[j], R.start[j])) continue;
      if ((R.pos[j] > p) == (R.start[j] > s)) up++; else down++;
    }
    X.st[k] = up > down ? 0u : (down > up ? 1u : SW_NONE);
  }
  __syncwarp();
  auto id = [&](u32 k) { return R.group[X.ord[k]]; };
  auto oriented = [&](u32 k) { return X.st[k] != SW_NONE; };
  auto strand = [&](u32 k) { return (u32)(X.st[k] & 1u); };
  // runs of one strand and their distinct IDs
  const u32 nrun = warp_runs(a, e, oriented, strand, X.idx, nullptr, nullptr, lane);
  for (u32 r = lane; r < nrun; r += 32) X.nids[a + r] = 0;
  __syncwarp();
  for (u32 k = a + lane; k < e; k += 32)
    if (oriented(k) && warp_first_in(X.idx, a, k, oriented, id)) atomicAdd(&X.nids[a + X.idx[k]], 1u);
  __syncwarp();
  // runs of >= SW_MIN_IDS distinct IDs survive; blocks = maximal runs of surviving rows of one strand, which merges the
  // runs that dropping the short ones left adjacent (one pass)
  for (u32 k = a + lane; k < e; k += 32)
    if (oriented(k) && X.nids[a + X.idx[k]] >= SW_MIN_IDS) X.st[k] |= SW_SURV;
  __syncwarp();
  auto surv = [&](u32 k) { return (X.st[k] & SW_SURV) != 0; };
  const u32 nblk = warp_runs(a, e, surv, strand, X.idx, X.first, X.last, lane);
  if (nblk < 2) return nblk;
  for (u32 r = lane; r < nblk; r += 32) {
    X.nids[a + r] = X.hi[a + r] = 0;
    X.lo[a + r] = 0xFFFFFFFFu;
  }
  __syncwarp();
  for (u32 k = a + lane; k < e; k += 32) {
    if (!surv(k)) continue;
    const u32 r = a + X.idx[k], s = R.start[X.ord[k]];
    if (warp_first_in(X.idx, a, k, surv, id)) atomicAdd(&X.nids[r], 1u);
    atomicMin(&X.lo[r], s);
    atomicMax(&X.hi[r], s);
  }
  return nblk;
}

// per segment: its records (blocks - 1, or 0)
__global__ void __launch_bounds__(256) k_sw_resolve(const SwRows R, const SwScratch X, u32* seg_cnt) {
  const u32 s = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (s >= R.n_seg) return;
  const u32 a = R.seg_start[s], b = R.seg_start[s + 1];
  u32 nblk = 0;
  if (R.len(R.read[a]) >= R.min_len) {
    // one pass: usable rows, and whether pos and start are monotone along them (previous usable row by shuffle, carried
    // across the 32-row chunks)
    const u32 c0 = R.contig[a], lt = (1u << lane) - 1;
    u32 nu = 0, cp = 0, cs = 0;
    bool have = false, sorted = true, up = true, down = true;
    for (u32 c = a; c < b; c += 32) {
      const u32 i = c + lane;
      const bool q = i < b && R.contig[i] == c0 && !R.is_bad(i);
      const u32 p = q ? R.pos[i] : 0u, st = q ? R.start[i] : 0u;
      const u32 m = __ballot_sync(0xFFFFFFFFu, q), pm = m & lt;
      const int src = pm ? 31 - __clz(pm) : lane;
      const u32 pp = __shfl_sync(0xFFFFFFFFu, p, src), ps = __shfl_sync(0xFFFFFFFFu, st, src);
      if (q && (pm || have)) {
        const u32 qp = pm ? pp : cp, qs = pm ? ps : cs;
        sorted &= qp <= p;
        up &= qs <= st;
        down &= qs >= st;
      }
      if (m) {
        const int hi = 31 - __clz(m);
        cp = __shfl_sync(0xFFFFFFFFu, p, hi);
        cs = __shfl_sync(0xFFFFFFFFu, st, hi);
        have = true;
      }
      nu += __popc(m);
    }
    sorted = __all_sync(0xFFFFFFFFu, sorted);
    const bool mono = __all_sync(0xFFFFFFFFu, up) || __all_sync(0xFFFFFFFFu, down);
    if (nu >= SW_MIN_ROWS && !(sorted && mono)) nblk = sw_blocks(R, X, a, b, nu, sorted, lane);
  }
  if (lane == 0) seg_cnt[s] = nblk >= 2 ? nblk - 1 : 0u;
}

// records of segment s at seg_off[s], in block order (one thread per segment)
__global__ void __launch_bounds__(256) k_sw_emit(const SwRows R, const SwScratch X, const u32* __restrict__ seg_cnt,
                                                 const u32* __restrict__ seg_off, u32* rec, u64 stride) {
  const u64 s = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= R.n_seg) return;
  const u32 a = R.seg_start[s], v = seg_cnt[s];
  for (u32 t = 0; t < v; t++) {
    const u32 k = a + t, p = X.last[k], q = X.first[k + 1], i = X.ord[p], j = X.ord[q];
    u32* o = rec + seg_off[s] + t;  // columns as in gvs_strand_switches_get
    o[0] = R.read[a];
    o[stride] = R.contig[a];
    o[2 * stride] = X.st[p] & 1u;
    o[3 * stride] = X.nids[k];
    o[4 * stride] = X.lo[k];
    o[5 * stride] = X.hi[k];
    o[6 * stride] = R.group[i];
    o[7 * stride] = R.start[i];
    o[8 * stride] = R.pos[i];
    o[9 * stride] = X.st[q] & 1u;
    o[10 * stride] = X.nids[k + 1];
    o[11 * stride] = X.lo[k + 1];
    o[12 * stride] = X.hi[k + 1];
    o[13 * stride] = R.group[j];
    o[14 * stride] = R.start[j];
    o[15 * stride] = R.pos[j];
  }
}

extern "C" int gvs_strand_switches(gvs_ctx* ctx, uint32_t min_read_len, uint64_t* n_records) {
  if (!ctx) return GVS_E_ARG;
  if (!ctx->diag_ready) return gvs_fail(ctx, GVS_E_STATE, "gvs_strand_switches: no kept rows (gvs_diag_filter / gvs_rows_set(1))");
  if (!ctx->read_off && !ctx->have_read_len) return gvs_fail(ctx, GVS_E_STATE, "gvs_strand_switches: read lengths unknown");
  CK(cudaSetDevice(ctx->device));
  StageTimer tm(ctx, GVS_ST_SWITCHES);
  ctx->sw.ready = false;
  ctx->sw.n = 0;
  if (n_records) *n_records = 0;
  const Rows& K = ctx->kept;
  const u64 n = K.n;
  if (n == 0) {
    ctx->sw.ready = true;
    return 0;
  }
  // segments of the kept rows: gvs_validate's while they are current, else built here
  const DevBuf* segs = &ctx->kseg_start;
  u64 n_seg = ctx->n_kseg;
  if (!ctx->val_ready) {
    CKR(gvs_build_segments(ctx, K.read.as<u32>(), n, ctx->sw_seg_start, ctx->flags_c, &n_seg));
    segs = &ctx->sw_seg_start;
  }
  SwRows R;
  (SegRows&)R = seg_rows(ctx, K, *segs, n_seg);
  R.len = read_lens(ctx);
  R.min_len = min_read_len;
  CKR(gvs_reserve(ctx, ctx->sw_scr, n * (7 * 4 + 1)));
  SwScratch X;
  X.ord = ctx->sw_scr.as<u32>();
  X.idx = X.ord + n; X.nids = X.idx + n; X.first = X.nids + n; X.last = X.first + n; X.lo = X.last + n; X.hi = X.lo + n;
  X.st = (u8*)(X.hi + n);
  CKR(gvs_reserve(ctx, ctx->sw_seg, n_seg * 8));
  u32 *seg_cnt = ctx->sw_seg.as<u32>(), *seg_off = seg_cnt + n_seg;
  LAUNCH(k_sw_resolve, (unsigned)cdiv(n_seg * 32, 256), 256, 0, R, X, seg_cnt);
  u32 nr = 0;
  {
    auto f = [seg_cnt] __device__(u64 s) -> u32 { return seg_cnt[s]; };
    auto g = [seg_off] __device__(u64 s, u32 ex, u32 v) { seg_off[s] = ex; };
    CKR(scan_total(ctx, n_seg, f, g, OpSum(), &nr));
  }
  if (nr) {
    CKR(rec_reserve(ctx, ctx->sw, 16, nr));
    LAUNCH(k_sw_emit, (unsigned)cdiv(n_seg, 256), 256, 0, R, X, seg_cnt, seg_off, ctx->sw.col(0), (u64)nr);
  }
  ctx->sw.n = nr;
  ctx->sw.ready = true;
  if (n_records) *n_records = nr;
  return 0;
}

extern "C" int gvs_strand_switches_get(gvs_ctx* ctx, uint32_t* read, uint32_t* contig, uint32_t* strand1, uint32_t* ids1,
                                       uint32_t* lo1, uint32_t* hi1, uint32_t* id1, uint32_t* start1, uint32_t* pos1,
                                       uint32_t* strand2, uint32_t* ids2, uint32_t* lo2, uint32_t* hi2, uint32_t* id2,
                                       uint32_t* start2, uint32_t* pos2) {
  return ctx ? rec_get(ctx, ctx->sw, "gvs_strand_switches_get before gvs_strand_switches",
                       {read, contig, strand1, ids1, lo1, hi1, id1, start1, pos1, strand2, ids2, lo2, hi2, id2, start2, pos2})
             : GVS_E_ARG;
}
