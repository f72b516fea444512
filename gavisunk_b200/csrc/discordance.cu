// discordance.cu -- collapses and expansions inside validated intervals, from the SUNK spacing of the validated reads.
// No reference counterpart.  Definition: include/gavisunk_b200.h (gvs_spans, gvs_discordance).
//
// The validation's ratio test lets a read through an event smaller than about a tenth of its reach: its close SUNK pairs
// across the event fail, its far pairs pass, and the read joins both sides.  Here every consecutive pair of a read's
// usable rows (non-bad, validated ID, the only row with that ID) is a span; a span whose SUNK distance on the read
// differs from the assembly's by more than the bound is longer or shorter.  A span from group a to group b contains
// every segment [ID_r, ID_r+1) with rank(a) <= r < rank(b), so an event inside segment r changes exactly the spans
// that cover r: three difference arrays over the group ranks (all spans, longer, shorter) locate it in segment space.
//
// gvs_spans: one warp per validation segment (a read) marks its usable rows -- the validated IDs sorted in scratch,
// a count of the read's non-bad rows per validated ID -- orders them by (start, ID), forms and classifies the spans
// and adds them to the difference arrays; a device scan places the records, a second warp pass writes them.
// gvs_discordance: prefix sums and runs of equal (spans, longer, shorter) through the run tiling of the support depth.
#include "common.cuh"

#define DC_NONE 0xFFFFFFFFu

struct DcParams : SegRows {     // kept rows, gvs_validate's segments
  const u32 *val_cnt, *val_id;  // gvs_validate: validated IDs per segment, and the IDs from the segment's first row on
  const u32* rank_of;           // null: rank = group index
  u64 ng;
  i64 min_delta, rel_permille;
  u32 *vid, *cnt, *uidx, *sidx;  // per row scratch, at the segment's first row: sorted validated IDs, their row counts,
                                 // usable rows (then span classes), usable rows by start
  u32 *seg_u, *seg_n;            // per segment: usable rows, non-concordant spans
  i32* diff;                     // 3 x ng
};

// index of row i's ID among the c sorted validated IDs of its read, DC_NONE when the row is bad, on another contig than
// the read's first row, or not validated
__device__ __forceinline__ u32 dc_find(const DcParams& P, const u32* vid, u32 c, u32 i, u32 c0) {
  if (P.contig[i] != c0 || P.is_bad(i)) return DC_NONE;
  const u32 id = P.group[i];
  u32 l = 0, h = c;
  while (l < h) {
    const u32 m = (l + h) >> 1;
    if (vid[m] < id) l = m + 1; else h = m;
  }
  return l < c && vid[l] == id ? l : DC_NONE;
}

// Order the n distinct keys key(x[k]) ascending into y: a copy or a reversal when they are monotone (a one-strand read),
// else a rank sort.  One warp.
template <typename K>
__device__ __forceinline__ void dc_order(const u32* x, u32* y, u32 n, K key, int lane) {
  bool up = true, down = true;
  for (u32 k = lane; k + 1 < n; k += 32) {
    const u64 k0 = key(x[k]), k1 = key(x[k + 1]);
    up &= k0 < k1;
    down &= k0 > k1;
  }
  up = __all_sync(0xFFFFFFFFu, up);
  down = __all_sync(0xFFFFFFFFu, down);
  for (u32 k = lane; k < n; k += 32) {
    u32 r = up ? k : n - 1 - k;
    if (!up && !down) {
      const u64 kk = key(x[k]);
      r = 0;
      for (u32 j = 0; j < n; j++) r += key(x[j]) < kk;
    }
    y[r] = x[k];
  }
  __syncwarp();
}

__global__ void __launch_bounds__(256) k_dc_spans(const DcParams P) {
  const u32 s = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (s >= P.n_seg) return;
  const u32 a = P.seg_start[s], b = P.seg_start[s + 1];
  const u32 c = P.val_cnt[s];
  u32 nu = 0, nrec = 0;
  if (c >= 2) {
    u32 *vid = P.vid + a, *cnt = P.cnt + a;
    // validated IDs in ascending order (gvs_validate lists them in vertex order: usually row order, so monotone)
    dc_order(P.val_id + a, vid, c, [](u32 id) -> u64 { return id; }, lane);
    for (u32 j = lane; j < c; j += 32) cnt[j] = 0;
    __syncwarp();
    const u32 c0 = P.contig[a];
    for (u32 i = a + lane; i < b; i += 32) {
      const u32 j = dc_find(P, vid, c, i, c0);
      if (j != DC_NONE) atomicAdd(&cnt[j], 1u);
    }
    __syncwarp();
    // usable rows, in row order: a validated ID on exactly one non-bad row
    u32* u = P.uidx + a;
    for (u32 base = a; base < b; base += 32) {
      const u32 i = base + lane;
      bool q = false;
      if (i < b) {
        const u32 j = dc_find(P, vid, c, i, c0);
        q = j != DC_NONE && cnt[j] == 1;
      }
      const u32 m = __ballot_sync(0xFFFFFFFFu, q);
      if (q) u[nu + __popc(m & ((1u << lane) - 1))] = i;
      nu += __popc(m);
    }
    __syncwarp();
    if (nu >= 2) {
      u32* srt = P.sidx + a;
      const u32 *st = P.start, *gr = P.group;
      dc_order(u, srt, nu, [st, gr](u32 i) -> u64 { return ((u64)st[i] << 32) | gr[i]; }, lane);
      // spans (srt[k], srt[k+1]); their classes go to u[k] (the row-order copy is dead)
      for (u32 k = lane; k + 1 < nu; k += 32) {
        const u32 i = srt[k], j = srt[k + 1];
        const i64 ds = (i64)P.start[j] - (i64)P.start[i];
        const i64 dp = P.pos[j] > P.pos[i] ? (i64)(P.pos[j] - P.pos[i]) : (i64)(P.pos[i] - P.pos[j]);
        const i64 delta = dp - ds, bound = 1000 * P.min_delta + P.rel_permille * ds;
        const u32 kind = 1000 * delta >= bound ? 1u : (-1000 * delta >= bound ? 2u : 0u);
        const u32 gi = P.gidx[i], gj = P.gidx[j];
        const u32 ra = P.rank_of ? P.rank_of[gi] : gi, rb = P.rank_of ? P.rank_of[gj] : gj;
        atomicAdd(&P.diff[ra], 1);
        atomicAdd(&P.diff[rb], -1);
        if (kind) {
          atomicAdd(&P.diff[kind * P.ng + ra], 1);
          atomicAdd(&P.diff[kind * P.ng + rb], -1);
          nrec++;
        }
        u[k] = kind;
      }
      nrec = __reduce_add_sync(0xFFFFFFFFu, nrec);
    }
  }
  if (lane == 0) {
    P.seg_u[s] = nu;
    P.seg_n[s] = nrec;
  }
}

// non-concordant spans of segment s to the records at seg_off[s], in span order
__global__ void __launch_bounds__(256) k_dc_emit(const DcParams P, const u32* __restrict__ seg_off, u32* rec, u64 stride) {
  const u32 s = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (s >= P.n_seg || P.seg_n[s] == 0) return;
  const u32 a = P.seg_start[s], nsp = P.seg_u[s] - 1;
  const u32 *kind = P.uidx + a, *srt = P.sidx + a;
  u32 o = seg_off[s];
  for (u32 k0 = 0; k0 < nsp; k0 += 32) {
    const u32 k = k0 + lane;
    const bool q = k < nsp && kind[k] != 0;
    const u32 m = __ballot_sync(0xFFFFFFFFu, q);
    if (q) {
      const u32 i = srt[k], j = srt[k + 1];
      u32* r = rec + o + __popc(m & ((1u << lane) - 1));  // columns as in gvs_spans_get
      r[0] = P.read[a];
      r[stride] = P.contig[i];
      r[2 * stride] = P.group[i];
      r[3 * stride] = P.start[i];
      r[4 * stride] = P.pos[i];
      r[5 * stride] = P.group[j];
      r[6 * stride] = P.start[j];
      r[7 * stride] = P.pos[j];
    }
    o += __popc(m);
  }
}

extern "C" int gvs_spans(gvs_ctx* ctx, uint32_t min_delta, uint32_t rel_permille, uint64_t* n_records, int32_t** diff_dev) {
  if (!ctx) return GVS_E_ARG;
  if (!ctx->val_ready) return gvs_fail(ctx, GVS_E_STATE, "gvs_spans before gvs_validate");
  if (!ctx->groups_ready) return gvs_fail(ctx, GVS_E_STATE, "gvs_spans: no group index");
  if (rel_permille > 1000000u) return gvs_fail(ctx, GVS_E_ARG, "gvs_spans: rel_permille %u > 1000000", rel_permille);
  CK(cudaSetDevice(ctx->device));
  StageTimer tm(ctx, GVS_ST_DISCORDANCE);
  ctx->dc.ready = ctx->dc_runs.ready = false;
  ctx->dc.n = 0;
  if (n_records) *n_records = 0;
  CKR(gvs_ensure_rank(ctx));
  const u64 ng = ctx->n_groups;
  CKR(gvs_reserve(ctx, ctx->dc_diff, (ng ? 3 * ng : 1) * 4));
  CK(cudaMemsetAsync(ctx->dc_diff.p, 0, (ng ? 3 * ng : 1) * 4, ctx->stream));
  const u64 n = ctx->kept.n, n_seg = ctx->n_kseg;
  u32 nr = 0;
  if (n && ctx->n_pairs) {
    const Rows& K = ctx->kept;
    DcParams P;
    (SegRows&)P = seg_rows(ctx, K, ctx->kseg_start, n_seg);
    P.val_id = ctx->val_id;
    P.val_cnt = ctx->val_seg_cnt;
    P.rank_of = ctx->rank_identity ? nullptr : ctx->rank_of.as<u32>();
    P.ng = ng;
    P.min_delta = min_delta;
    P.rel_permille = rel_permille;
    CKR(gvs_reserve(ctx, ctx->dc_scr, n * 4 * 4));
    P.vid = ctx->dc_scr.as<u32>(); P.cnt = P.vid + n; P.uidx = P.cnt + n; P.sidx = P.uidx + n;
    CKR(gvs_reserve(ctx, ctx->dc_seg, n_seg * 3 * 4));
    P.seg_u = ctx->dc_seg.as<u32>(); P.seg_n = P.seg_u + n_seg;
    u32* seg_off = P.seg_n + n_seg;
    P.diff = ctx->dc_diff.as<i32>();
    LAUNCH(k_dc_spans, (unsigned)cdiv(n_seg * 32, 256), 256, 0, P);
    {
      const u32* seg_n = P.seg_n;
      auto f = [seg_n] __device__(u64 s) -> u32 { return seg_n[s]; };
      auto g = [seg_off] __device__(u64 s, u32 ex, u32 v) { seg_off[s] = ex; };
      CKR(scan_total(ctx, n_seg, f, g, OpSum(), &nr));
    }
    if (nr) {
      CKR(rec_reserve(ctx, ctx->dc, 8, nr));
      LAUNCH(k_dc_emit, (unsigned)cdiv(n_seg * 32, 256), 256, 0, P, seg_off, ctx->dc.col(0), (u64)nr);
    }
  }
  ctx->dc.n = nr;
  ctx->dc.ready = true;
  if (n_records) *n_records = nr;
  if (diff_dev) *diff_dev = ctx->dc_diff.as<i32>();
  return 0;
}

extern "C" int gvs_spans_get(gvs_ctx* ctx, uint32_t* read, uint32_t* contig, uint32_t* id1, uint32_t* start1, uint32_t* pos1,
                             uint32_t* id2, uint32_t* start2, uint32_t* pos2) {
  return ctx ? rec_get(ctx, ctx->dc, "gvs_spans_get before gvs_spans", {read, contig, id1, start1, pos1, id2, start2, pos2}) : GVS_E_ARG;
}

extern "C" int gvs_discordance(gvs_ctx* ctx, const uint32_t* contig_len, uint64_t* n_runs) {
  if (!ctx) return GVS_E_ARG;
  if (!ctx->dc.ready) return gvs_fail(ctx, GVS_E_STATE, "gvs_discordance before gvs_spans");
  CK(cudaSetDevice(ctx->device));
  StageTimer tm(ctx, GVS_ST_DISCORDANCE);
  if (n_runs) *n_runs = 0;
  CKR(gvs_rank_runs(ctx, ctx->dc_diff.as<i32>(), 3, contig_len, ctx->dc_runs, "gvs_discordance"));
  if (n_runs) *n_runs = ctx->dc_runs.n;
  return 0;
}

extern "C" int gvs_discordance_get(gvs_ctx* ctx, uint32_t* contig, uint32_t* start, uint32_t* end, uint32_t* spans, uint32_t* longer,
                                   uint32_t* shorter) {
  return ctx ? rec_get(ctx, ctx->dc_runs, "gvs_discordance_get before gvs_discordance", {contig, start, end, spans, longer, shorter})
             : GVS_E_ARG;
}
