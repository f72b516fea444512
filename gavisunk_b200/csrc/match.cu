// match.cu -- SUNK matching of reads: the GPU replacement of kmerpos_annot3's main loop
// (workflow/src/kmerpos_annot3.nim:81-97; SURVEY.md A.3, quirks Q1-Q6).
//
//   k_probe2       (probe.cu) ★ hot kernel: every k-mer window of every read through the presence filter,
//                  the blocked Bloom filter and the exact table; emits hit RECORDS (first hit of a run of
//                  consecutive hits on one SUNK group inside a read + number of followers) into one
//                  region per probe span, in position order
//   k_gather_hits  span regions copied into one dense array in global position order (scan of span counts)
//   k_emit_flags / scans / k_emit_rows
//                  consecutive-(contig,group) suppression across the whole chunk (prevLoc is
//                  never reset between reads, Q4) and the position drift it causes (Q3)
#include "table.cuh"

int gvs_probe_launch(gvs_ctx* ctx, u64* n_warps_out, u64* cap_w_out);  // probe.cu

#define FLAG_KEYERROR 1u
#define FLAG_OVERFLOW 2u

// per-span record regions -> dense arrays in global position order (span order = position order)
__global__ void __launch_bounds__(128) k_gather_hits(const u32* __restrict__ warp_cnt, const u64* __restrict__ warp_dst, u64 cap_w,
                                                     const u32* __restrict__ a0, const u32* __restrict__ a1,
                                                     const u32* __restrict__ a2, const u32* __restrict__ a3,
                                                     const u8* __restrict__ a4, u32* b0, u32* b1, u32* b2, u32* b3, u8* b4,
                                                     const u64* __restrict__ read_off) {
  const u64 w = blockIdx.x;
  const u32 c = warp_cnt[w];
  const u64 s = w * cap_w, d = warp_dst[w];
  for (u32 i = threadIdx.x; i < c; i += blockDim.x) {
    const u32 rd = a0[s + i];
    b0[d + i] = rd;
    // the probe leaves the low word of the hit's batch position: window = position - start of its read (mod 2^32)
    b1[d + i] = a1[s + i] - (u32)read_off[rd];
    b2[d + i] = a2[s + i];
    b3[d + i] = a3[s + i];
    b4[d + i] = a4[s + i];
  }
}

__device__ __forceinline__ u32 chunk_of(const u64* __restrict__ chunk_first, u32 n_chunks, u32 read) {
  u32 lo = 0, hi = n_chunks;  // last c with chunk_first[c] <= read
  while (hi - lo > 1) {
    u32 mid = (lo + hi) >> 1;
    if (chunk_first[mid] <= read) lo = mid; else hi = mid;
  }
  return lo;
}

// flags: bit0 = emitted (curLoc != prevLoc, nim:92), bit1 = first record of its read
__global__ void __launch_bounds__(256) k_emit_flags(const u32* __restrict__ hread, const u32* __restrict__ hgidx, u64 n,
                                                    const u64* __restrict__ chunk_first, u32 n_chunks, u8* flags) {
  u64 j = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n) return;
  u32 rd = hread[j];
  bool head = true, emit = true;
  if (j > 0) {
    u32 rp = hread[j - 1];
    head = rp != rd;
    bool same_chunk = !head || chunk_of(chunk_first, n_chunks, rp) == chunk_of(chunk_first, n_chunks, rd);
    if (same_chunk) emit = hgidx[j] != hgidx[j - 1];
  }
  flags[j] = (emit ? 1 : 0) | (head ? 2 : 0);
}

__global__ void __launch_bounds__(256) k_emit_rows(const u32* __restrict__ hread, const u32* __restrict__ hw,
                                                   const u32* __restrict__ hrow, const u32* __restrict__ hgidx,
                                                   const u8* __restrict__ flags,
                                                   const u64* __restrict__ packed_excl, const u32* __restrict__ seg_base,
                                                   u64 n, const uint4* __restrict__ loc_pack,
                                                   u32* r_read, u32* r_pos,
                                                   u32* r_contig, u32* r_start, u32* r_group, u32* r_gidx) {
  u64 j = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n) return;
  if (!(flags[j] & 1)) return;
  u64 pe = packed_excl[j];
  u32 out = (u32)(pe >> 32);        // emitted rows before j
  u32 supp = (u32)pe;               // suppressed hits before record j (whole batch)
  u32 base = seg_base[j] - 1;       // suppressed hits before the first hit of j's read
  u32 row = hrow[j];
  r_read[out] = hread[j];
  r_pos[out] = hw[j] - (supp - base);  // `continue` skips `inc i` (nim:92,96; Q3)
  const uint4 l = __ldg(loc_pack + row);  // (contig, start, group) of the .loc row
  r_contig[out] = l.x;
  r_start[out] = l.y;
  r_group[out] = l.z;
  r_gidx[out] = hgidx[j];
}


// ---- SUNK_len = 32 ------------------------------------------------------------------------------------
// The reference's k-mer iterator breaks at k = 32 (nim-kmer 0.2.6 `forward_add` masks with (1 shl 2k) - 1 = 0,
// SURVEY Q2) but kmerpos_annot3 still prints rows; tests/golden/kat_k32, kat_k32b and ksweep[k=32] pin what it
// yields through the executable: window 0 = min(fwd, rc | 3) (the forward value is exact, the reverse
// complement comes out with its last base read as T), window w >= 1 = min(code(seq[w+31]), rc) (the
// forward value keeps only the incoming base, the rolling reverse complement stays right).  Outside
// BASELINE.json's sweep and of no use to anybody, so no tiles and no filters: one thread per window, the hits
// go straight into the ordered hit arrays and the common emit pass takes over.
struct K32View {
  const u8* seq;
  int packed;
  const u64* read_off;
  u64 n_reads, total;
  TabView tab;
  u32* flags;
};
__device__ __forceinline__ u32 k32_code(const K32View& v, u64 g) {
  if (v.packed) return (((const u32*)v.seq)[g >> 4] >> (30 - 2 * (int)(g & 15))) & 3u;
  const u32 x = v.seq[g], l = x | 0x20u;
  if (l == 'c') return 1;
  if (l == 'g') return 2;
  if (l == 't' || l == 'u') return 3;
  return x <= 3 ? x : 0;  // A/a and everything else 0, bytes 1..3 themselves (kat_bytes)
}
// hit of the window that starts at base g: .loc row (or GVS_NOHIT); *rd / *w = read and window index
__device__ u32 k32_hit(const K32View& v, u64 g, u32* rd, u32* w, u32* gi) {
  u64 lo = 1, hi = v.n_reads;  // first boundary index j >= 1 with read_off[j] > g
  while (lo < hi) {
    u64 mid = (lo + hi) >> 1;
    if (v.read_off[mid] > g) hi = mid; else lo = mid + 1;
  }
  const u64 r = lo - 1, o0 = v.read_off[r], o1 = v.read_off[r + 1];
  if (g < o0 || g >= o1) return GVS_NOHIT;
  const u64 len = o1 - o0, win = g - o0;
  const u64 n_win = len >= 32 ? len - 31 : (len == 31 ? 1 : 0);  // a 31-long read: one window, NUL read as A (Q6)
  if (win >= n_win) return GVS_NOHIT;
  u64 f = 0, rc = 0;
  u32 last = 0;
  for (int j = 0; j < 32; j++) {
    last = (g + j < o1) ? k32_code(v, g + j) : 0u;
    f = (f << 2) | last;
    rc |= (u64)(3u - last) << (2 * j);
  }
  u64 val;
  if (win == 0) {
    rc |= 3ull;
    val = f < rc ? f : rc;
  } else {
    val = (u64)last < rc ? (u64)last : rc;
  }
  u32 row = tab_lookup(v.tab, val, gvs_mix(val), gi);
  if (row == GVS_ROW_MISSING) {
    atomicOr(v.flags, FLAG_KEYERROR);
    return GVS_NOHIT;
  }
  if (row >= GVS_NOHIT) return GVS_NOHIT;
  *rd = (u32)r;
  *w = (u32)win;
  return row;
}

static int match_k32(gvs_ctx* ctx, u64* n_hits) {
  StageTimer tm(ctx, GVS_ST_PROBE);
  u64* counters = counter<u64>(ctx, CNT_HITS);
  CK(cudaMemsetAsync(counters, 0, 4 * sizeof(u64), ctx->stream));
  if (!ctx->seg_packed.empty()) return gvs_fail(ctx, GVS_E_STATE, "k = 32: host batches are not packed on the way");
  K32View v;
  v.seq = ctx->seq;
  v.packed = ctx->seq_packed ? 1 : 0;
  v.read_off = ctx->read_off;
  v.n_reads = ctx->n_reads;
  v.total = ctx->total_bases;
  v.tab.kv = ctx->tab_kv.as<u64>();
  v.tab.slots = ctx->tab_slots;
  v.flags = counter(ctx, CNT_FLAGS);
  // the segments of a pipelined host batch must have landed (gvs_probe_launch waits per segment)
  for (size_t s = 0; s < ctx->seg_tile_end.size() && ctx->seq == ctx->own_seq.as<u8>(); s++)
    CK(cudaStreamWaitEvent(ctx->stream, ctx->seg_ev[s], 0));
  auto f = [v] __device__(u64 i) -> u64 {
    u32 rd, w, gi;
    return k32_hit(v, i, &rd, &w, &gi) != GVS_NOHIT ? 1ull : 0ull;
  };
  auto g0 = [] __device__(u64 i, u64 ex, u64 val) {};
  CKR((device_scan<u64>(ctx, v.total, f, g0, OpSum(), counters)));
  u64 h[2];  // hits, flags
  CKR(read_dev(ctx, counters, h, 2));
  if ((u32)h[1] & FLAG_KEYERROR)
    return gvs_fail(ctx, GVS_E_KEYERROR, "KeyError: a read matched a db k-mer that has no .loc row (kmerpos_annot3.nim:90)");
  const u64 nh = h[0];
  *n_hits = nh;
  if (nh == 0) return 0;
  if (nh >= 0xFFFFFFF0ull) return gvs_fail(ctx, GVS_E_OVERFLOW, "more than 2^32 hits in one batch");
  CKR(gvs_reserve(ctx, ctx->ohit_read, nh * 4));
  CKR(gvs_reserve(ctx, ctx->ohit_w, nh * 4));
  CKR(gvs_reserve(ctx, ctx->ohit_row, nh * 4));
  CKR(gvs_reserve(ctx, ctx->ohit_gidx, nh * 4));
  CKR(gvs_reserve(ctx, ctx->ohit_nf, nh));
  u32 *o_rd = ctx->ohit_read.as<u32>(), *o_w = ctx->ohit_w.as<u32>(), *o_row = ctx->ohit_row.as<u32>(),
      *o_gi = ctx->ohit_gidx.as<u32>();
  u8* o_nf = ctx->ohit_nf.as<u8>();
  auto g1 = [v, o_rd, o_w, o_row, o_gi, o_nf] __device__(u64 i, u64 ex, u64 val) {
    if (!val) return;
    u32 rd = 0, w = 0, gi = 0;
    u32 row = k32_hit(v, i, &rd, &w, &gi);
    o_rd[ex] = rd;
    o_w[ex] = w;
    o_row[ex] = row;
    o_gi[ex] = gi;
    o_nf[ex] = 0;
  };
  CKR((device_scan<u64>(ctx, v.total, f, g1, OpSum(), (u64*)nullptr)));
  return 0;
}

static int match_once(gvs_ctx* ctx, u64* n_warps, u64* cap_w, bool* overflow, u64* total_hits, u64* max_per_warp) {
  u64* counters = counter<u64>(ctx, CNT_HITS);
  CK(cudaMemsetAsync(counters, 0, 4 * sizeof(u64), ctx->stream));
  {
    StageTimer tm(ctx, GVS_ST_PROBE);
    CKR(gvs_probe_launch(ctx, n_warps, cap_w));
  }
  // totals of the per-warp counts (+ their exclusive scan = destination of every region)
  const u32* wc = ctx->tile_cnt.as<u32>();
  u64* wd = ctx->tile_dst.as<u64>();
  {
    auto f = [wc] __device__(u64 i) -> u64 { return (u64)wc[i]; };
    auto g = [wd] __device__(u64 i, u64 ex, u64 v) { wd[i] = ex; };
    CKR((device_scan<u64>(ctx, *n_warps, f, g, OpSum(), counters)));
    auto g2 = [] __device__(u64 i, u64 ex, u64 v) {};
    CKR((device_scan<u64>(ctx, *n_warps, f, g2, OpMax(), counter<u64>(ctx, CNT_HIT_MAX))));
  }
  u64 h[4];  // CNT_HITS .. CNT_HIT_MAX
  CKR(read_dev(ctx, counters, h, 4));
  *total_hits = h[CNT_HITS];
  *max_per_warp = h[CNT_HIT_MAX];
  u32 fl = (u32)h[CNT_FLAGS];
  if (fl & FLAG_KEYERROR)
    return gvs_fail(ctx, GVS_E_KEYERROR, "KeyError: a read matched a db k-mer that has no .loc row (kmerpos_annot3.nim:90)");
  *overflow = (fl & FLAG_OVERFLOW) != 0;
  return 0;
}

extern "C" int gvs_match(gvs_ctx* ctx, uint64_t* n_rows_out) {
  if (!ctx) return GVS_E_ARG;
  if (!ctx->db_ready) return gvs_fail(ctx, GVS_E_STATE, "gvs_match: no database");
  if (!ctx->reads_ready) return gvs_fail(ctx, GVS_E_STATE, "gvs_match: no reads");
  CK(cudaSetDevice(ctx->device));
  ctx->match_ready = ctx->diag_ready = ctx->val_ready = false;
  ctx->rows.n = 0;
  ctx->n_hits = 0;
  u64 total = ctx->total_bases;
  if (n_rows_out) *n_rows_out = 0;
  if (total == 0 || ctx->n_reads == 0) {
    ctx->match_ready = true;
    return 0;
  }
  if (((uintptr_t)ctx->seq & 15) != 0) return gvs_fail(ctx, GVS_E_ARG, "read buffer must be 16-byte aligned");
  u64 n_warps = 0, cap_w = 0;
  const bool k32 = ctx->k >= 32;  // Q2: the reference's broken-but-deterministic k = 32 (match_k32)
  if (k32) {
    CKR(match_k32(ctx, &ctx->n_hits));
  } else {
    // hit capacity: start at 1/32 of the windows (typical density is <1 %), retry once with the
    // exact need if a batch is denser
    if (ctx->hit_cap == 0) ctx->hit_cap = total / 32 + 4096;
    for (int attempt = 0;; attempt++) {
      CKR(gvs_reserve(ctx, ctx->hit_read, ctx->hit_cap * 4));
      CKR(gvs_reserve(ctx, ctx->hit_w, ctx->hit_cap * 4));
      CKR(gvs_reserve(ctx, ctx->hit_row, ctx->hit_cap * 4));
      CKR(gvs_reserve(ctx, ctx->hit_gidx, ctx->hit_cap * 4));
      CKR(gvs_reserve(ctx, ctx->hit_nf, ctx->hit_cap));
      bool overflow = false;
      u64 need = 0, max_w = 0;
      CKR(match_once(ctx, &n_warps, &cap_w, &overflow, &need, &max_w));
      if (!overflow) {
        ctx->n_hits = need;
        break;
      }
      if (attempt >= 1) return gvs_fail(ctx, GVS_E_OVERFLOW, "hit buffer overflow after resize");
      ctx->hit_cap = (max_w + max_w / 4 + 64) * n_warps;  // every warp region must hold the densest span
    }
  }
  u64 nh = ctx->n_hits;
  if (nh == 0) {
    ctx->match_ready = true;
    return 0;
  }
  if (nh >= 0xFFFFFFF0ull) return gvs_fail(ctx, GVS_E_OVERFLOW, "more than 2^32 hits in one batch");
  StageTimer tm(ctx, GVS_ST_EMIT);
  if (!k32) {
    // ---- order the hits ----
    CKR(gvs_reserve(ctx, ctx->ohit_read, nh * 4));
    CKR(gvs_reserve(ctx, ctx->ohit_w, nh * 4));
    CKR(gvs_reserve(ctx, ctx->ohit_row, nh * 4));
    CKR(gvs_reserve(ctx, ctx->ohit_gidx, nh * 4));
    CKR(gvs_reserve(ctx, ctx->ohit_nf, nh));
    LAUNCH(k_gather_hits, (unsigned)n_warps, 128, 0, ctx->tile_cnt.as<u32>(), ctx->tile_dst.as<u64>(), cap_w, ctx->hit_read.as<u32>(),
           ctx->hit_w.as<u32>(), ctx->hit_row.as<u32>(), ctx->hit_gidx.as<u32>(), ctx->hit_nf.as<u8>(), ctx->ohit_read.as<u32>(),
           ctx->ohit_w.as<u32>(), ctx->ohit_row.as<u32>(), ctx->ohit_gidx.as<u32>(), ctx->ohit_nf.as<u8>(),
           ctx->read_off);
  }
  // ---- suppression + position drift ----
  CKR(gvs_reserve(ctx, ctx->flags_a, nh));          // u8 flags
  CKR(gvs_reserve(ctx, ctx->flags_b, nh * 8));      // packed exclusive counts
  CKR(gvs_reserve(ctx, ctx->flags_c, nh * 4));      // per-hit base of its read
  u8* fl = ctx->flags_a.as<u8>();
  u64* pex = ctx->flags_b.as<u64>();
  u32* sb = ctx->flags_c.as<u32>();
  const u8* nf = ctx->ohit_nf.as<u8>();
  LAUNCH(k_emit_flags, (unsigned)cdiv(nh, 256), 256, 0, ctx->ohit_read.as<u32>(), ctx->ohit_gidx.as<u32>(), nh,
         ctx->chunk_first.as<u64>(), ctx->n_chunks, fl);
  u64* tot = counter<u64>(ctx, CNT_EMIT);
  {
    // high word: rows emitted; low word: suppressed hits = the record's followers (+ the record's own
    // first hit when it continues the previous record's group)
    auto f = [fl, nf] __device__(u64 i) -> u64 { return ((fl[i] & 1) ? (1ull << 32) : 1ull) + nf[i]; };
    auto g = [pex] __device__(u64 i, u64 ex, u64 v) { pex[i] = ex; };
    CKR((device_scan<u64>(ctx, nh, f, g, OpSum(), tot)));
  }
  {
    // base of the read = suppressed count before its first hit (+1 so that 0 is the identity);
    // the counts are non-decreasing, so an inclusive prefix max picks the latest head
    auto f = [fl, pex] __device__(u64 i) -> u32 { return (fl[i] & 2) ? (u32)pex[i] + 1u : 0u; };
    auto g = [sb] __device__(u64 i, u32 ex, u32 v) { sb[i] = ex > v ? ex : v; };
    CKR((device_scan<u32>(ctx, nh, f, g, OpMax(), (u32*)nullptr)));
  }
  u64 packed_total = 0;
  CKR(read_dev(ctx, tot, &packed_total));
  u64 n_rows = packed_total >> 32;
  CKR(gvs_reserve_rows(ctx, ctx->rows, n_rows));
  LAUNCH(k_emit_rows, (unsigned)cdiv(nh, 256), 256, 0, ctx->ohit_read.as<u32>(), ctx->ohit_w.as<u32>(),
         ctx->ohit_row.as<u32>(), ctx->ohit_gidx.as<u32>(), fl, pex, sb, nh, ctx->loc_pack.as<uint4>(), ctx->rows.read.as<u32>(),
         ctx->rows.pos.as<u32>(),
         ctx->rows.contig.as<u32>(), ctx->rows.start.as<u32>(), ctx->rows.group.as<u32>(), ctx->rows.gidx.as<u32>());
  ctx->rows.n = n_rows;
  ctx->match_ready = true;
  if (n_rows_out) *n_rows_out = n_rows;
  return 0;
}

extern "C" int gvs_rows_get(gvs_ctx* ctx, int which, uint32_t* read_idx, uint32_t* pos, uint32_t* contig,
                            uint32_t* start, uint32_t* group) {
  if (!ctx) return GVS_E_ARG;
  CK(cudaSetDevice(ctx->device));
  Rows* r;
  if (which == 0) {
    if (!ctx->match_ready) return gvs_fail(ctx, GVS_E_STATE, "gvs_rows_get(0) before gvs_match");
    r = &ctx->rows;
  } else if (which == 1) {
    if (!ctx->diag_ready) return gvs_fail(ctx, GVS_E_STATE, "gvs_rows_get(1) before gvs_diag_filter");
    r = &ctx->kept;
  } else {
    return gvs_fail(ctx, GVS_E_ARG, "which must be 0 or 1");
  }
  u64 n = r->n;
  if (n == 0) return 0;
  if (read_idx) CK(cudaMemcpyAsync(read_idx, r->read.p, n * 4, cudaMemcpyDeviceToHost, ctx->stream));
  if (pos) CK(cudaMemcpyAsync(pos, r->pos.p, n * 4, cudaMemcpyDeviceToHost, ctx->stream));
  if (contig) CK(cudaMemcpyAsync(contig, r->contig.p, n * 4, cudaMemcpyDeviceToHost, ctx->stream));
  if (start) CK(cudaMemcpyAsync(start, r->start.p, n * 4, cudaMemcpyDeviceToHost, ctx->stream));
  if (group) CK(cudaMemcpyAsync(group, r->group.p, n * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return 0;
}
