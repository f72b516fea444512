// dbbuild.cu -- SUNK database build on the GPU: the replacement of workflow/rules/defineSUNKs.smk
// (combine_asm_haps :1-19, jellyfish count -C -U 1 :22-40, define_SUNKs :43-61, mrsfast
// index/search -e 0 :64-103, bed_convert :106-127).  SURVEY.md A.1/A.2.
//
//   k_db_count     every valid window (only ACGT, inside one contig) -> canonical k-mer ->
//                  find-or-insert into an open-addressed HBM table; the first window registers its
//                  position, any later window of the same k-mer sets a DUP bit (count > 1)
//   k_db_mark      singleton slots set bit `position` of the SUNK bitmap (position order falls out
//                  of the bitmap: no sort, and mrsfast's "where is it" is the registered position)
//   k_db_rank      popcount per bitmap word -> scan -> .loc row of every SUNK
//   k_db_rows      per SUNK: contig, start, canonical k-mer, "starts a new merged run" flag
//                  (bedtools merge joins overlapping or book-ended [start,start+k): a new group
//                  starts iff no SUNK lies in [start-k, start-1] on the same contig)
//   scans          group start (max-scan of run heads) and dense group index
// The key space is processed in P passes (hash-partitioned) so that the count table fits HBM for
// a 6.2 Gbp diploid assembly.
#include "table.cuh"

#define DT 256
#define DWPT 16
#define DTILE (DT * DWPT)
#define DBW ((DTILE + 64) / 32 + 2)

#define VAL_EMPTY 0xFFFFFFFFFFFFFFFFull
#define VAL_DUP 0x8000000000000000ull

// assembly bases: only A/C/G/T (any case) are valid; returns codes and a per-byte invalid mask
__device__ __forceinline__ void asm_codes4(u32 x, u32& code, u32& inv) {
  u32 f = ((x >> 1) ^ (x >> 2)) & 0x03030303u;
  u32 l = x | 0x20202020u;
  u32 ok = __vcmpeq4(l, 0x61616161u) | __vcmpeq4(l, 0x63636363u) | __vcmpeq4(l, 0x67676767u) |
           __vcmpeq4(l, 0x74747474u);
  code = f & ok;
  inv = ~ok;
}
__device__ __forceinline__ u32 squeeze4b(u32 c) {
  c = (c | (c >> 6)) & 0x000F000Fu;
  c = (c | (c >> 12)) & 0xFFu;
  return c;
}
// invalid mask bytes (0xFF / 0x00) -> 4 bits
__device__ __forceinline__ u32 mask4(u32 m) {
  m &= 0x01010101u;
  return (m | (m >> 7) | (m >> 14) | (m >> 21)) & 0xFu;
}
__device__ __forceinline__ void asm_load16(const u8* __restrict__ seq, u64 g, u64 total, u32& packed, u32& inv16) {
  uint4 v = make_uint4(0x4E4E4E4Eu, 0x4E4E4E4Eu, 0x4E4E4E4Eu, 0x4E4E4E4Eu);  // 'N' beyond the end
  if (g + 16 <= total) {
    v = __ldg((const uint4*)(seq + g));
  } else if (g < total) {
    u32 w[4] = {0x4E4E4E4Eu, 0x4E4E4E4Eu, 0x4E4E4E4Eu, 0x4E4E4E4Eu};
    for (int i = 0; i < 16 && g + i < total; i++) {
      w[i >> 2] &= ~(0xFFu << (8 * (i & 3)));
      w[i >> 2] |= (u32)seq[g + i] << (8 * (i & 3));
    }
    v = make_uint4(w[0], w[1], w[2], w[3]);
  }
  u32 c0, c1, c2, c3, i0, i1, i2, i3;
  asm_codes4(v.x, c0, i0);
  asm_codes4(v.y, c1, i1);
  asm_codes4(v.z, c2, i2);
  asm_codes4(v.w, c3, i3);
  packed = squeeze4b(c0) | (squeeze4b(c1) << 8) | (squeeze4b(c2) << 16) | (squeeze4b(c3) << 24);
  inv16 = mask4(i0) | (mask4(i1) << 4) | (mask4(i2) << 8) | (mask4(i3) << 12);
}

__global__ void __launch_bounds__(256) k_db_tile_index(const u64* __restrict__ off, u64 n, u64 n_tiles, u32* tile_first) {
  u64 t = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_tiles) return;
  u64 ts = t * DTILE;
  u64 lo = 1, hi = n;
  while (lo < hi) {
    u64 mid = (lo + hi) >> 1;
    if (__ldg(off + mid) > ts) hi = mid; else lo = mid + 1;
  }
  tile_first[t] = (u32)lo;
}

// find-or-insert into the count table: buckets of 4 slots, ANY bucket count (multiply-shift range reduction
// instead of a mask, so that the table can be sized to the memory that is free rather than to a power of
// two -- half as many passes over a 6.2 Gbp assembly)
// Layout: a bucket is 64 bytes -- its 4 keys followed by their 4 value words -- so that the value update that follows
// every find-or-insert lands in the line the key access has just brought into L2: one random HBM line per window instead
// of two (the build is bound by exactly that: a line fill and a write-back per random atomic).
// Returns the index of the key's VALUE word in kv.
__device__ __forceinline__ u64 cnt_insert(u64* kv, u64 n_buckets, u64 key, u64 h) {
  u64 b = ((h >> 32) * n_buckets) >> 32;
  for (;;) {
#pragma unroll
    for (int j = 0; j < 4; j++) {
      u64 s = (b << 3) + j;
      u64 cur = kv[s];
      if (cur == key) return s + 4;
      if (cur == GVS_EMPTY_KEY) {
        u64 old = atomicCAS((unsigned long long*)&kv[s], (unsigned long long)GVS_EMPTY_KEY, (unsigned long long)key);
        if (old == GVS_EMPTY_KEY || old == key) return s + 4;
      }
    }
    b = b + 1 == n_buckets ? 0 : b + 1;
  }
}

struct DbCountParams {
  const u8* __restrict__ seq;
  u64 total;
  const u64* __restrict__ contig_off;
  u64 n_contigs;
  const u32* __restrict__ tile_first;
  u64 n_tiles;
  int k;
  u64* kv;  // count table: buckets of 4 keys + 4 values (cnt_insert)
  u64 slots;
  u32 n_parts, part;
};

#ifndef DB_BLOCKS
#define DB_BLOCKS 2  // resident blocks per SM of the count kernel (3 / 4 / 6 measured: 0.76 ... 3.7 s instead of 0.9 s -- CAS storms, erratic)
#endif
__global__ void __launch_bounds__(DT, DB_BLOCKS) k_db_count(const DbCountParams P) {
  __shared__ u32 s_bases[DT + 4];
  __shared__ u32 s_inv[(DT + 4) / 2 + 2];  // 16 invalid bits per packed word, two per u32
  __shared__ u32 s_bound[DBW];
  const int t = threadIdx.x;
  const int k = P.k;
  const u64 kmask = (k >= 32) ? ~0ull : ((1ull << (2 * k)) - 1);
  const int topsh = 2 * (k - 1);
  const u64 vmask = (k >= 2) ? ((1ull << (k - 1)) - 1) : 0ull;
  const u64 imask = (k >= 64) ? ~0ull : ((1ull << k) - 1);
  u16* s_inv16 = (u16*)s_inv;
  for (u64 tile = blockIdx.x; tile < P.n_tiles; tile += gridDim.x) {
    const u64 ts = tile * DTILE;
    {
      u32 pk, iv;
      asm_load16(P.seq, ts + 16ull * t, P.total, pk, iv);
      s_bases[t] = pk;
      s_inv16[t] = (u16)iv;
      if (t < 4) {
        asm_load16(P.seq, ts + DTILE + 16ull * t, P.total, pk, iv);
        s_bases[DT + t] = pk;
        s_inv16[DT + t] = (u16)iv;
      }
    }
    if (t < DBW) s_bound[t] = 0;
    __syncthreads();
    const u32 j0 = __ldg(P.tile_first + tile);
    const u64 limit = ts + DTILE + (u64)(k > 1 ? k - 1 : 1);
    for (u64 j = (u64)j0 + t; j <= P.n_contigs; j += DT) {
      u64 o = __ldg(P.contig_off + j);
      if (o >= limit) break;
      u32 rel = (u32)(o - ts);
      atomicOr(&s_bound[rel >> 5], 1u << (rel & 31));
    }
    __syncthreads();
    const u32 w0 = s_bases[t], w1 = s_bases[t + 1], w2 = s_bases[t + 2];
    const u64 lo = (u64)w0 | ((u64)w1 << 32);
    u64 B, I;
    {
      int idx = t >> 1, sh = (t & 1) * 16;
      u64 b01 = (u64)s_bound[idx] | ((u64)s_bound[idx + 1] << 32);
      B = b01 >> sh;
      if (sh) B |= (u64)s_bound[idx + 2] << 48;
      I = (u64)s_inv16[t] | ((u64)s_inv16[t + 1] << 16) | ((u64)s_inv16[t + 2] << 32);
    }
    u64 f = 0, r = 0;
#pragma unroll 1
    for (int i = 0; i < k - 1; i++) {
      u64 b = (lo >> (2 * i)) & 3;
      f = (f << 2) | b;
      r = (r >> 2) | ((3 - b) << topsh);
    }
    const u64 p0 = ts + 16ull * t;
#pragma unroll
    for (int i = 0; i < DWPT; i++) {
      int bi = k - 1 + i;
      u64 b = (bi < 32) ? ((lo >> (2 * bi)) & 3) : (u64)((w2 >> (2 * (bi - 32))) & 3);
      f = ((f << 2) | b) & kmask;
      r = (r >> 2) | ((3 - b) << topsh);
      bool ok = (p0 + i < P.total) && (((B >> (i + 1)) & vmask) == 0) && (((I >> i) & imask) == 0);
      if (ok) {
        u64 c = f < r ? f : r;
        u64 h = gvs_mix(c);
        if (P.n_parts == 1 || (u32)h % P.n_parts == P.part) {  // low hash bits pick the pass, high bits the bucket
          u64 s = cnt_insert(P.kv, P.slots >> 2, c, h);
          u64 old = atomicCAS((unsigned long long*)&P.kv[s], (unsigned long long)VAL_EMPTY, (unsigned long long)(p0 + i));
          if (old != VAL_EMPTY && !(old & VAL_DUP)) atomicOr((unsigned long long*)&P.kv[s], (unsigned long long)VAL_DUP);
        }
      }
    }
    __syncthreads();
  }
}

__global__ void __launch_bounds__(256) k_db_mark(const u64* __restrict__ kv, u64 slots, u32* bitmap) {
  for (u64 s = (u64)blockIdx.x * blockDim.x + threadIdx.x; s < slots; s += (u64)gridDim.x * blockDim.x) {
    const u64 o = ((s >> 2) << 3) + (s & 3);  // key of slot s; its value sits 4 words on
    if (kv[o] == GVS_EMPTY_KEY) continue;
    u64 v = kv[o + 4];
    if (v == VAL_EMPTY || (v & VAL_DUP)) continue;
    atomicOr(&bitmap[v >> 5], 1u << (v & 31));
  }
}

__global__ void __launch_bounds__(256) k_fill64(u64* p, u64 n, u64 v) {
  for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) p[i] = v;
}

// per SUNK (bit of the bitmap): the .loc row
__global__ void __launch_bounds__(256) k_db_rows(const u32* __restrict__ bitmap, const u32* __restrict__ word_rank,
                                                 u64 n_words, const u8* __restrict__ seq, u64 total,
                                                 const u64* __restrict__ contig_off, u32 n_contigs, int k, u64* loc_kmer,
                                                 u32* loc_contig, u32* loc_start, u8* head) {
  u64 w = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= n_words) return;
  u32 bits = bitmap[w];
  if (!bits) return;
  u32 row = word_rank[w];
  u32 prevw = w ? bitmap[w - 1] : 0u;
  u64 hist = ((u64)bits << 32) | prevw;  // bit (32 + b) = position 32w + b
  // contig of the first set bit; later bits of the same word may cross into the next contig
  u64 p_first = w * 32 + (__ffs(bits) - 1);
  u32 lo = 0, hi = n_contigs;  // last c with contig_off[c] <= p
  while (hi - lo > 1) {
    u32 mid = (lo + hi) >> 1;
    if (__ldg(contig_off + mid) <= p_first) lo = mid; else hi = mid;
  }
  u32 c = lo;
  u64 cstart = __ldg(contig_off + c), cend = __ldg(contig_off + c + 1);
  while (bits) {
    int b = __ffs(bits) - 1;
    bits &= bits - 1;
    u64 p = w * 32 + b;
    while (p >= cend) {
      c++;
      cstart = cend;
      cend = __ldg(contig_off + c + 1);
    }
    // canonical k-mer at p
    u64 f = 0, r = 0;
    for (int i = 0; i < k; i++) {
      u32 x = seq[p + i];
      u64 code = ((x >> 1) ^ (x >> 2)) & 3;
      f = (f << 2) | code;
      r = (r >> 2) | ((3 - code) << (2 * (k - 1)));
    }
    loc_kmer[row] = f < r ? f : r;
    loc_contig[row] = c;
    loc_start[row] = (u32)(p - cstart);
    // SUNKs in [max(p-k, cstart), p-1]?  (k <= 32 positions back: inside `hist`)
    u64 lowp = (p >= (u64)k && p - k > cstart) ? p - k : cstart;
    int span = (int)(p - lowp);  // 0..k
    u64 m = span ? (((1ull << span) - 1) << (32 + b - span)) : 0ull;
    head[row] = (hist & m) ? 0 : 1;
    row++;
  }
}

__global__ void __launch_bounds__(256) k_db_groups(const u32* __restrict__ headrow_incl, const u32* __restrict__ gidx_excl,
                                                   const u8* __restrict__ head, u64 n, const u32* __restrict__ loc_contig,
                                                   const u32* __restrict__ loc_start, u32* loc_group, u32* loc_gidx,
                                                   u32* grp_contig, u32* grp_start) {
  u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  u32 hr = headrow_incl[i] - 1;
  // gidx_excl counts heads strictly before i; a head row starts group number gidx_excl[i]
  u32 gi = head[i] ? gidx_excl[i] : gidx_excl[i] - 1;
  loc_group[i] = loc_start[hr];
  loc_gidx[i] = gi;
  if (head[i]) {
    grp_contig[gi] = loc_contig[i];
    grp_start[gi] = loc_start[i];
  }
}

static unsigned grid_cap(gvs_ctx* ctx, u64 n, int block, int per_sm) {
  u64 g = cdiv(n, block);
  u64 cap = (u64)ctx->n_sm * per_sm;
  if (g > cap) g = cap;
  if (g == 0) g = 1;
  return (unsigned)g;
}

static int db_build_device(gvs_ctx* ctx, const u8* seq, const u64* contig_off, u32 n_contigs, u64 total,
                           DevBuf& keys, DevBuf& vals, DevBuf& bitmap, DevBuf& wrank, DevBuf& head, DevBuf& hrow,
                           DevBuf& gex) {
  const int k = ctx->k;
  u64 n_tiles = cdiv(total, DTILE);  // 0 when every contig is empty: no window, an empty database
  CKR(gvs_reserve(ctx, ctx->tile_first, n_tiles * 4));
  if (n_tiles)
    LAUNCH(k_db_tile_index, (unsigned)cdiv(n_tiles, 256), 256, 0, contig_off, (u64)n_contigs, n_tiles, ctx->tile_first.as<u32>());
  // count-table sizing: <= `total` distinct k-mers; load <= 2/3; P passes so that it fits (or as gvs_set_db_passes says)
  size_t free_b = 0, tot_b = 0;
  CK(cudaMemGetInfo(&free_b, &tot_b));
  u64 n_words = cdiv(total, 32) + 2;
  u64 budget = (u64)(free_b * 0.70) - n_words * 4;
  u32 n_parts = ctx->db_passes ? (u32)ctx->db_passes : 1;
  u64 slots;
  for (;;) {
    slots = (((total / n_parts) * 3 / 2 + 1024) + 3) & ~3ull;  // load <= 2/3, whole buckets of 4
    if (ctx->db_passes || slots * 16 <= budget || n_parts >= 64) break;
    n_parts += 1;
  }
  if ((slots >> 2) >= (1ull << 32)) return gvs_fail(ctx, GVS_E_OVERFLOW, "SUNK count table has too many buckets");
  if (slots * 16 > budget) return gvs_fail(ctx, GVS_E_NOMEM, "SUNK count table does not fit (%llu slots)", (unsigned long long)slots);
  CKR(gvs_reserve(ctx, keys, slots * 16));  // keys and values, bucket by bucket (cnt_insert)
  (void)vals;
  CKR(gvs_reserve(ctx, bitmap, n_words * 4));
  CK(cudaMemsetAsync(bitmap.p, 0, n_words * 4, ctx->stream));
  for (u32 part = 0; part < n_parts; part++) {
    static_assert(GVS_EMPTY_KEY == VAL_EMPTY, "one fill value for keys and values");
    LAUNCH(k_fill64, grid_cap(ctx, slots * 2, 256, 16), 256, 0, keys.as<u64>(), slots * 2, GVS_EMPTY_KEY);
    DbCountParams P;
    P.seq = seq; P.total = total; P.contig_off = contig_off; P.n_contigs = n_contigs;
    P.tile_first = ctx->tile_first.as<u32>(); P.n_tiles = n_tiles; P.k = k;
    P.kv = keys.as<u64>(); P.slots = slots; P.n_parts = n_parts; P.part = part;
    u64 grid = (u64)ctx->n_sm * DB_BLOCKS;
    if (grid > n_tiles) grid = n_tiles;
    if (grid) LAUNCH(k_db_count, (unsigned)grid, DT, 0, P);
    LAUNCH(k_db_mark, grid_cap(ctx, slots, 256, 16), 256, 0, keys.as<u64>(), slots, bitmap.as<u32>());
  }
  // rank of every SUNK
  CKR(gvs_reserve(ctx, wrank, n_words * 4));
  const u32* bm = bitmap.as<u32>();
  u32* wr = wrank.as<u32>();
  u64 n_sunks = 0;
  {
    auto f = [bm] __device__(u64 i) -> u64 { return (u64)__popc(bm[i]); };
    auto g = [wr] __device__(u64 i, u64 ex, u64 v) { wr[i] = (u32)ex; };
    CKR(scan_total(ctx, n_words, f, g, OpSum(), &n_sunks));
  }
  if (n_sunks >= 0x7FFFFFF0ull) return gvs_fail(ctx, GVS_E_OVERFLOW, "more than 2^31 SUNKs");
  ctx->n_loc = n_sunks;
  ctx->n_contigs = n_contigs;
  CKR(gvs_reserve(ctx, ctx->loc_kmer, n_sunks * 8));
  CKR(gvs_reserve(ctx, ctx->loc_contig, n_sunks * 4));
  CKR(gvs_reserve(ctx, ctx->loc_start, n_sunks * 4));
  CKR(gvs_reserve(ctx, ctx->loc_group, n_sunks * 4));
  CKR(gvs_reserve(ctx, ctx->loc_gidx, n_sunks * 4));
  CKR(gvs_reserve(ctx, head, n_sunks));
  CKR(gvs_reserve(ctx, hrow, n_sunks * 4));
  CKR(gvs_reserve(ctx, gex, n_sunks * 4));
  ctx->n_groups = 0;
  ctx->grp_gen++;
  if (n_sunks) {
    LAUNCH(k_db_rows, (unsigned)cdiv(n_words, 256), 256, 0, bm, wr, n_words, seq, total, contig_off, n_contigs, k,
           ctx->loc_kmer.as<u64>(), ctx->loc_contig.as<u32>(), ctx->loc_start.as<u32>(), head.as<u8>());
    const u8* hd = head.as<u8>();
    u32* hr = hrow.as<u32>();
    u32* ge = gex.as<u32>();
    {
      auto f = [hd] __device__(u64 i) -> u32 { return hd[i] ? (u32)i + 1u : 0u; };
      auto g = [hr] __device__(u64 i, u32 ex, u32 v) { hr[i] = ex > v ? ex : v; };
      CKR((device_scan<u32>(ctx, n_sunks, f, g, OpMax(), (u32*)nullptr)));
    }
    u32 ng = 0;
    {
      auto f = [hd] __device__(u64 i) -> u32 { return hd[i] ? 1u : 0u; };
      auto g = [ge] __device__(u64 i, u32 ex, u32 v) { ge[i] = ex; };
      CKR(scan_total(ctx, n_sunks, f, g, OpSum(), &ng));
    }
    ctx->n_groups = ng;
    CKR(gvs_reserve(ctx, ctx->grp_contig, (u64)ng * 4));
    CKR(gvs_reserve(ctx, ctx->grp_start, (u64)ng * 4));
    LAUNCH(k_db_groups, (unsigned)cdiv(n_sunks, 256), 256, 0, hr, ge, hd, n_sunks, ctx->loc_contig.as<u32>(),
           ctx->loc_start.as<u32>(), ctx->loc_group.as<u32>(), ctx->loc_gidx.as<u32>(), ctx->grp_contig.as<u32>(),
           ctx->grp_start.as<u32>());
  } else {
    CKR(gvs_reserve(ctx, ctx->grp_contig, 4));
    CKR(gvs_reserve(ctx, ctx->grp_start, 4));
  }
  // free the big count table before allocating the probe table
  CK(cudaStreamSynchronize(ctx->stream));
  gvs_release(keys);
  gvs_release(vals);
  CKR(gvs_tab_build_impl(ctx, nullptr, 0));
  CKR(gvs_tab_attach_gidx(ctx));
  CK(cudaStreamSynchronize(ctx->stream));
  return 0;
}

extern "C" int gvs_db_build(gvs_ctx* ctx, const uint8_t* seq, const uint64_t* contig_off, uint32_t n_contigs,
                            int seq_on_device) {
  if (!ctx) return GVS_E_ARG;
  if (!seq || !contig_off || n_contigs == 0) return gvs_fail(ctx, GVS_E_ARG, "gvs_db_build: null input");
  CK(cudaSetDevice(ctx->device));
  StageTimer tm(ctx, GVS_ST_DBBUILD);
  ctx->db_ready = false;
  DevBuf dseq, doff, keys, vals, bitmap, wrank, head, hrow, gex;
  int rc = 0;
  u64 total = 0;
  const u8* s = seq;
  const u64* o = contig_off;
  if (!seq_on_device) {
    total = contig_off[n_contigs];
    rc = gvs_reserve(ctx, dseq, total + 64);
    if (!rc) rc = to_dev(ctx, doff, contig_off, (size_t)n_contigs + 1);
    if (!rc && total && cudaMemcpyAsync(dseq.p, seq, total, cudaMemcpyHostToDevice, ctx->stream) != cudaSuccess)
      rc = gvs_fail(ctx, GVS_E_CUDA, "H2D copy of the assembly failed");
    s = dseq.as<u8>();
    o = doff.as<u64>();
  } else {
    rc = read_dev(ctx, contig_off + n_contigs, &total);
    if (!rc && ((uintptr_t)seq & 15)) rc = gvs_fail(ctx, GVS_E_ARG, "assembly buffer must be 16-byte aligned");
  }
  if (!rc && total >= (1ull << 62)) rc = gvs_fail(ctx, GVS_E_ARG, "assembly too large");
  if (!rc) {
    // contigs must fit 32-bit starts
    rc = db_build_device(ctx, s, o, n_contigs, total, keys, vals, bitmap, wrank, head, hrow, gex);
  }
  if (!rc) rc = gvs_check_group_order(ctx);
  cudaStreamSynchronize(ctx->stream);
  DevBuf* tmp[] = {&dseq, &doff, &keys, &vals, &bitmap, &wrank, &head, &hrow, &gex};
  for (DevBuf* b : tmp) gvs_release(*b);
  if (rc) return rc;
  ctx->db_ready = true;
  ctx->groups_ready = true;
  ctx->gt_slots = 0;
  return 0;
}
