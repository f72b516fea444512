// gap_evidence.cu -- the reads that bridge each gap without validating it, and the size change their SUNK distances
// imply.  No reference counterpart: the reference only draws pile-up plots (viz.py, viz_detailed.py).
//
// Per gap (contig, gs, ge) and per read, on the read's kept rows of that contig minus the bad groups: a row is left
// when ID <= gs, right when ID >= ge + 1 (sides by ID, as intervals are built from IDs); it is anchored when another
// row of its side with a different ID passes the ratio test with it (9*|dstart| < 10*|dpos| < 11*|dstart|, Q12); a
// read bridges the gap when it has anchored rows on both sides.  Its flanks are the anchored left row with the
// largest (start, -pos) and the anchored right row with the smallest (start, pos) -- ties on both: smallest ID.
//
// Two kernels.  k_ge_cand: one warp per kept-row segment (a read); reads that are too short or whose contig has no
// gap leave after one row, the others reduce their smallest and largest non-bad ID, and a binary search over the
// contig's gaps gives the contiguous range the read could bridge (min ID <= gs and max ID > ge).  A device scan emits
// the (segment, gap) candidates.  k_ge_resolve: one warp per candidate decides anchoring with O(m^2) pair tests and
// picks the flanks with warp reductions; a second scan compacts the bridging candidates in candidate order.
#include "common.cuh"

// per contig [lo, hi) of its gaps (gaps are sorted by (contig, start)); contigs without gaps keep lo = hi = 0
__global__ void __launch_bounds__(256) k_ge_contig_gaps(const u32* __restrict__ gc, u64 n, u32* lo, u32* hi) {
  const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const u32 c = gc[i];
  if (i == 0 || gc[i - 1] != c) lo[c] = (u32)i;
  if (i + 1 == n || gc[i + 1] != c) hi[c] = (u32)i + 1;
}

struct GeRows : SegRows {  // kept rows
  ReadLens len;
  u32 min_len;
  const u32 *gap_contig, *gap_start, *gap_end;
  const u32 *cg_lo, *cg_hi;  // per contig: its gaps
  u32 n_contigs;
};

// per segment: (first gap it may bridge, number of such gaps)
__global__ void __launch_bounds__(256) k_ge_cand(const GeRows R, uint2* seg_cand) {
  const u32 s = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (s >= R.n_seg) return;
  const u32 a = R.seg_start[s], b = R.seg_start[s + 1];
  const u32 rd = R.read[a], c = R.contig[a];
  const u32 rlen = R.len(rd);
  const u32 glo = c < R.n_contigs ? R.cg_lo[c] : 0, ghi = c < R.n_contigs ? R.cg_hi[c] : 0;
  if (rlen < R.min_len || glo == ghi) {
    if (lane == 0) seg_cand[s] = make_uint2(0, 0);
    return;
  }
  u32 mn = 0xFFFFFFFFu, mx = 0;
  for (u32 j = a + lane; j < b; j += 32) {
    if (R.contig[j] != c || R.is_bad(j)) continue;
    const u32 id = R.group[j];
    mn = min(mn, id);
    mx = max(mx, id);
  }
  mn = __reduce_min_sync(0xFFFFFFFFu, mn);
  mx = __reduce_max_sync(0xFFFFFFFFu, mx);
  if (lane != 0) return;
  // gaps of a contig are disjoint and sorted: gs and ge both rise.  [i0, i1) = gaps with gs >= mn and ge < mx
  u32 l = glo, h = ghi;
  while (l < h) {
    const u32 m = (l + h) >> 1;
    if (R.gap_start[m] < mn) l = m + 1; else h = m;
  }
  const u32 i0 = l;
  h = ghi;
  while (l < h) {
    const u32 m = (l + h) >> 1;
    if (R.gap_end[m] < mx) l = m + 1; else h = m;
  }
  seg_cand[s] = make_uint2(i0, mn <= mx && l > i0 ? l - i0 : 0u);
}

// per candidate: [0] bridges, [1..3] left (ID, start, pos), [4..6] right (ID, start, pos)
__global__ void __launch_bounds__(256) k_ge_resolve(const GeRows R, const u32* __restrict__ cand_seg, const u32* __restrict__ cand_gap,
                                                    u32 n_cand, u32* res) {
  const u32 k = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (k >= n_cand) return;
  const u32 s = cand_seg[k], gi = cand_gap[k];
  const u32 a = R.seg_start[s], b = R.seg_start[s + 1];
  const u32 c = R.gap_contig[gi], gs = R.gap_start[gi], ge1 = R.gap_end[gi] + 1;
  // side of a row: 1 left, 2 right, 0 neither (other contig, bad group, inside the gap)
  auto side = [&](u32 j, u32& id) -> u32 {
    if (R.contig[j] != c || R.is_bad(j)) return 0;
    id = R.group[j];
    return id <= gs ? 1u : (id >= ge1 ? 2u : 0u);
  };
  // best flank keys of this lane: left max (start, ~pos), right min (start, pos); ID breaks ties (smallest)
  u64 lk = 0, rk = ~0ull;
  u32 lid = 0xFFFFFFFFu, rid = 0xFFFFFFFFu;
  bool lany = false, rany = false;
  for (u32 i = a + lane; i < b; i += 32) {
    u32 idi = 0;
    const u32 si = side(i, idi);
    if (!si) continue;
    const u32 pi = R.pos[i], sti = R.start[i];
    bool anchored = false;
    for (u32 j = a; j < b && !anchored; j++) {
      u32 idj = 0;
      if (side(j, idj) != si || idj == idi) continue;
      anchored = gvs_ratio_ok(pi, sti, R.pos[j], R.start[j]);
    }
    if (!anchored) continue;
    if (si == 1) {
      const u64 key = ((u64)sti << 32) | (u32)~pi;
      if (!lany || key > lk || (key == lk && idi < lid)) { lk = key; lid = idi; }
      lany = true;
    } else {
      const u64 key = ((u64)sti << 32) | pi;
      if (!rany || key < rk || (key == rk && idi < rid)) { rk = key; rid = idi; }
      rany = true;
    }
  }
  const bool has_l = __any_sync(0xFFFFFFFFu, lany);
  const bool has_r = __any_sync(0xFFFFFFFFu, rany);
  if (!has_l || !has_r) {
    if (lane == 0) res[(u64)k * 8] = 0;
    return;
  }
  u64 lbest = lany ? lk : 0, rbest = rany ? rk : ~0ull;
  for (int d = 16; d; d >>= 1) {
    const u64 x = __shfl_xor_sync(0xFFFFFFFFu, lbest, d), y = __shfl_xor_sync(0xFFFFFFFFu, rbest, d);
    lbest = x > lbest ? x : lbest;
    rbest = y < rbest ? y : rbest;
  }
  const u32 lmin = __reduce_min_sync(0xFFFFFFFFu, lany && lk == lbest ? lid : 0xFFFFFFFFu);
  const u32 rmin = __reduce_min_sync(0xFFFFFFFFu, rany && rk == rbest ? rid : 0xFFFFFFFFu);
  if (lane == 0) {
    u32* o = res + (u64)k * 8;
    o[0] = 1;
    o[1] = lmin; o[2] = (u32)(lbest >> 32); o[3] = ~(u32)lbest;
    o[4] = rmin; o[5] = (u32)(rbest >> 32); o[6] = (u32)rbest;
  }
}

extern "C" int gvs_gap_evidence(gvs_ctx* ctx, uint32_t min_read_len, uint64_t* n_records) {
  if (!ctx) return GVS_E_ARG;
  if (!ctx->gaps_ready) return gvs_fail(ctx, GVS_E_STATE, "gvs_gap_evidence before gvs_gaps");
  if (!ctx->diag_ready) return gvs_fail(ctx, GVS_E_STATE, "gvs_gap_evidence: no kept rows (gvs_diag_filter / gvs_rows_set(1))");
  if (!ctx->read_off && !ctx->have_read_len) return gvs_fail(ctx, GVS_E_STATE, "gvs_gap_evidence: read lengths unknown");
  CK(cudaSetDevice(ctx->device));
  StageTimer tm(ctx, GVS_ST_EVIDENCE);
  ctx->ge.ready = false;
  ctx->ge.n = 0;
  if (n_records) *n_records = 0;
  Rows& K = ctx->kept;
  const u64 n = K.n, ngap = ctx->n_gaps;
  const u32 nc = ctx->n_contigs;
  if (n == 0 || ngap == 0 || nc == 0) {
    ctx->ge.ready = true;
    return 0;
  }
  // segments of the kept rows: gvs_validate's while they are current, else built here
  const DevBuf* segs = &ctx->kseg_start;
  u64 n_seg = ctx->n_kseg;
  if (!ctx->val_ready) {
    CKR(gvs_build_segments(ctx, K.read.as<u32>(), n, ctx->ge_seg_start, ctx->flags_c, &n_seg));
    segs = &ctx->ge_seg_start;
  }
  const u32* seg_start = segs->as<u32>();
  CKR(gvs_reserve(ctx, ctx->ge_cgap, (u64)nc * 8));
  u32 *cg_lo = ctx->ge_cgap.as<u32>(), *cg_hi = cg_lo + nc;
  CK(cudaMemsetAsync(cg_lo, 0, (u64)nc * 8, ctx->stream));
  LAUNCH(k_ge_contig_gaps, (unsigned)cdiv(ngap, 256), 256, 0, ctx->gap_contig.as<u32>(), ngap, cg_lo, cg_hi);
  GeRows R;
  (SegRows&)R = seg_rows(ctx, K, *segs, n_seg);
  R.len = read_lens(ctx);
  R.min_len = min_read_len;
  R.gap_contig = ctx->gap_contig.as<u32>(); R.gap_start = ctx->gap_start.as<u32>(); R.gap_end = ctx->gap_end.as<u32>();
  R.cg_lo = cg_lo; R.cg_hi = cg_hi; R.n_contigs = nc;
  CKR(gvs_reserve(ctx, ctx->ge_seg, n_seg * 8));
  uint2* seg_cand = ctx->ge_seg.as<uint2>();
  LAUNCH(k_ge_cand, (unsigned)cdiv(n_seg * 32, 256), 256, 0, R, seg_cand);
  // candidates: count per segment, scan, fill
  u32 ncand = 0;
  {
    auto f = [seg_cand] __device__(u64 s) -> u32 { return seg_cand[s].y; };
    auto g = [] __device__(u64 s, u32 ex, u32 v) {};
    CKR(scan_total(ctx, n_seg, f, g, OpSum(), &ncand));
  }
  if (ncand == 0) {
    ctx->ge.ready = true;
    return 0;
  }
  CKR(gvs_reserve(ctx, ctx->ge_cand, (u64)ncand * 8));
  CKR(gvs_reserve(ctx, ctx->ge_res, (u64)ncand * 32));
  u32 *cseg = ctx->ge_cand.as<u32>(), *cgap = cseg + ncand;
  {
    auto f = [seg_cand] __device__(u64 s) -> u32 { return seg_cand[s].y; };
    auto g = [seg_cand, cseg, cgap] __device__(u64 s, u32 ex, u32 v) {
      const u32 g0 = seg_cand[s].x;
      for (u32 t = 0; t < v; t++) {
        cseg[ex + t] = (u32)s;
        cgap[ex + t] = g0 + t;
      }
    };
    CKR((device_scan<u32>(ctx, n_seg, f, g, OpSum(), (u32*)nullptr)));
  }
  u32* res = ctx->ge_res.as<u32>();
  LAUNCH(k_ge_resolve, (unsigned)cdiv((u64)ncand * 32, 256), 256, 0, R, cseg, cgap, ncand, res);
  // records in candidate order (segment, then gap): 8 columns of ncand entries
  CKR(rec_reserve(ctx, ctx->ge, 8, ncand));
  u32* rec = ctx->ge.col(0);
  const u32* rread = K.read.as<u32>();
  u32 nr = 0;
  {
    auto f = [res] __device__(u64 k) -> u32 { return res[k * 8]; };
    auto g = [res, rec, ncand, cseg, cgap, seg_start, rread] __device__(u64 k, u32 ex, u32 v) {
      if (!v) return;
      const u32* r = res + k * 8;
      rec[ex] = rread[seg_start[cseg[k]]];
      rec[(u64)ncand + ex] = cgap[k];
      for (int t = 1; t < 7; t++) rec[(u64)(t + 1) * ncand + ex] = r[t];
    };
    CKR(scan_total(ctx, ncand, f, g, OpSum(), &nr));
  }
  ctx->ge.n = nr;
  ctx->ge.ready = true;
  if (n_records) *n_records = nr;
  return 0;
}

extern "C" int gvs_gap_evidence_get(gvs_ctx* ctx, uint32_t* read, uint32_t* gap, uint32_t* left_id, uint32_t* left_start,
                                    uint32_t* left_pos, uint32_t* right_id, uint32_t* right_start, uint32_t* right_pos) {
  return ctx ? rec_get(ctx, ctx->ge, "gvs_gap_evidence_get before gvs_gap_evidence",
                       {read, gap, left_id, left_start, left_pos, right_id, right_start, right_pos})
             : GVS_E_ARG;
}
