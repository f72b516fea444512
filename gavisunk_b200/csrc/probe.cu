// probe.cu -- ★ the hot kernel: every k-mer window of every read against the SUNK table
// (inner loop of workflow/src/kmerpos_annot3.nim:85-96; nim-kmer 0.2.6 encode/slide semantics,
// SURVEY.md Q1/Q2/Q6).
//
// Warp-synchronous design (no block barriers; a warp that takes the rare exact-probe path never
// stalls its neighbours):
//   * a warp walks a span of consecutive 512-window tiles with a private cursor into read_off (no
//     per-tile binary search)
//   * per tile ONE coalesced 16-byte cp.async per lane brings the ASCII bases into shared memory two
//     tiles ahead of the compute (the copy of tile T+2 is in flight while tile T is processed); the
//     bases are packed to 2 bits twice -- forward (big-endian) and reverse complement -- into a
//     two-tile ring, so the 32-base halo of a tile is simply the head of the next ring slot and both
//     strands of every window are constant-shift funnel extractions (no rolling state)
//   * J = 4 consecutive windows share the (K-3)-mer that starts at the last of them, and every SUNK was
//     entered into the filters under each of its 4 sub-mers.  Per group of 4 windows ONE word of the
//     L2-resident presence filter is tested; the groups that pass (a few % / ~20 % for a whole genome)
//     are compacted across the warp and only their windows are hashed (canonical = min(fwd, rc)) and
//     tested against the group's 16-byte block of the blocked Bloom filter (4 bits per key, one per
//     word) -- one window per lane, so the ALU work per base follows the pass rate, not the read length
//   * filter-positive windows (~1 %) are compacted into a per-warp queue in position order and looked
//     up in the exact table (32-byte bucket in HBM) 32 at a time
//   * work is handed out in spans of a few hundred tiles through one atomic counter (no tail: a warp
//     that drew hit-poor reads simply takes more spans); runs of hits on one SUNK group collapse into one
//     record (first hit + follower count: ~6 hits per group crossing at 94 % read identity); every span
//     appends its records to its own region (position order, no per-hit atomics); a scan of the per-span
//     counts + one coalesced copy give the dense ordered list
#include "table.cuh"
#include <stdlib.h>
#include <vector>

#ifndef PW_WARPS
#define PW_WARPS 8     // warps per block
#endif
#ifndef PW_BLOCKS
#define PW_BLOCKS 4    // resident blocks per SM (PW_WARPS * PW_BLOCKS warps of 65536 / (32 * PW_WARPS * PW_BLOCKS) registers per thread)
#endif
#define PW_TILE 512    // window starts per warp tile
static_assert(PW_TILE == GVS_TILE_BASES, "ctx.cu sizes the copy segments in probe tiles");
#define PW_RING 64     // packed words in the ring: two tile slots of 32 words (16 bases each)
#define PW_MAXB 32

#define FLAG_KEYERROR 1u
#define FLAG_OVERFLOW 2u

// ASCII -> 2-bit codes for 4 bytes at once (mapping pinned by tests/golden/kat_bytes: A/a 0, C/c 1,
// G/g 2, T/t/U/u 3, bytes 0x01..0x03 themselves, everything else 0)
__device__ __forceinline__ u32 p_codes4(u32 x) {
  u32 f = ((x >> 1) ^ (x >> 2)) & 0x03030303u;
  u32 l = x | 0x20202020u;
  u32 letter = __vcmpeq4(l, 0x63636363u) | __vcmpeq4(l, 0x67676767u) | __vcmpeq4(l, 0x74747474u) |
               __vcmpeq4(l, 0x75757575u);
  u32 low = __vcmpeq4(x & 0xFCFCFCFCu, 0u);
  return (f & letter) | (x & low & 0x03030303u);
}
// Fast path for the overwhelmingly common tile that holds nothing but A/C/G/T (any case): the code of a
// letter is ((x >> 1) ^ (x >> 2)) & 3; `bad` collects a non-zero value when a byte is something else
// (the codes are turned back into letters with one PRMT and compared with the upper-cased input).
__device__ __forceinline__ u32 p_codes4_fast(u32 x, u32& bad) {
  u32 f = ((x >> 1) ^ (x >> 2)) & 0x03030303u;
  u32 t = f | (f >> 4);                      // byte 0 = f1:f0, byte 2 = f3:f2 (nibbles)
  u32 sel = __byte_perm(t, 0u, 0x4420);      // low 16 bits = f3:f2:f1:f0
  u32 letters = __byte_perm(0x54474341u, 0u, sel);  // "ACGT"[f] per byte
  bad |= letters ^ (x & 0xDFDFDFDFu);
  return f;
}
// 4 code bytes (first base in byte 0) -> 8 bits big-endian (first base in bits 7:6), left in the TOP byte
__device__ __forceinline__ u32 p_be8_top(u32 c) { return c * 0x40100401u; }
__device__ __forceinline__ u32 p_gather_top(u32 px, u32 py, u32 pz, u32 pw) {
  u32 t1 = __byte_perm(py, px, 0x0073);  // low 16 bits = top(px):top(py)
  u32 t2 = __byte_perm(pw, pz, 0x0073);
  return __byte_perm(t2, t1, 0x5410);
}
__device__ __forceinline__ u32 p_pack16_be(uint4 v) {
  return p_gather_top(p_be8_top(p_codes4(v.x)), p_be8_top(p_codes4(v.y)), p_be8_top(p_codes4(v.z)), p_be8_top(p_codes4(v.w)));
}
__device__ __forceinline__ u32 p_pack16_be_fast(uint4 v, u32& bad) {
  return p_gather_top(p_be8_top(p_codes4_fast(v.x, bad)), p_be8_top(p_codes4_fast(v.y, bad)),
                      p_be8_top(p_codes4_fast(v.z, bad)), p_be8_top(p_codes4_fast(v.w, bad)));
}
// reverse complement of 16 packed bases
__device__ __forceinline__ u32 p_rc16(u32 w) {
  u32 x = __brev(~w);
  return ((x >> 1) & 0x55555555u) | ((x & 0x55555555u) << 1);
}
// 2*LEN bits starting at base offset `off` (0..15) of the big-endian string a:b:c
template <int LEN>
__device__ __forceinline__ u64 p_extract(u32 a, u32 b, u32 c, int off) {
  int s = 2 * off;
  u32 hi = __funnelshift_l(b, a, s);
  u32 lo = __funnelshift_l(c, b, s);
  u64 v = ((u64)hi << 32) | lo;
  return v >> (64 - 2 * LEN);
}

struct __align__(16) WarpSmem {
  u32 fw[PW_RING];   // forward packed words, ring index = (slot base + word) & 63
  u32 rc[PW_RING];   // rc[i] = reverse complement of fw[i] (same index)
  uint4 raw[32];     // landing zone of the tile's bulk copy (TMA): 16 ASCII bases per lane (PACKED: one word per lane)
  u64 bar;           // mbarrier the bulk copy of a tile completes on (one per warp; the phase flips per tile)
  u32 bound[20];
  u32 shrt[20];
  u32 bpos[PW_MAXB];
  u32 bidx[PW_MAXB];
  u32 cand[PW_TILE / 32];  // filter-positive windows of the tile (bit p)
  u16 inv[32];             // per lane: invalid windows among its 16
  u32 q_row[PW_TILE];      // group queue: block hash of the passing group
  u16 q_p[PW_TILE];        // group queue: group index inside the tile; later: window of a candidate
  u32 s_blk[32][3];        // large databases: key words of the blocks whose fingerprint bit was set (one round)
  u16 s_p[32];             // ... and their group index inside the tile
};

// forward / reverse-complement k-mer of window p (0..511) of the tile whose ring base is `rb`
template <int K>
__device__ __forceinline__ u64 p_fwd_at(const WarpSmem& sm, u32 rb, u32 p) {
  u32 wi = rb + (p >> 4);
  return p_extract<K>(sm.fw[wi & 63], sm.fw[(wi + 1) & 63], sm.fw[(wi + 2) & 63], p & 15);
}
template <int K>
__device__ __forceinline__ u64 p_rc_at(const WarpSmem& sm, u32 rb, u32 p) {
  // the window ends at base e = p + K (exclusive); its reverse complement starts inside the rc of
  // word c-1 (c = ceil(e/16)) at base offset 16c - e and continues through DEscending word indices
  u32 e = p + K, c = (e + 15) >> 4;
  u32 wi = rb + c - 1;
  return p_extract<K>(sm.rc[wi & 63], sm.rc[(wi - 1) & 63], sm.rc[(wi - 2) & 63], 16 * c - e);
}
template <int K>
__device__ __forceinline__ u64 p_canon_at(const WarpSmem& sm, u32 rb, u32 p, bool force_last_a) {
  u64 f = p_fwd_at<K>(sm, rb, p), r = p_rc_at<K>(sm, rb, p);
  if (force_last_a) {  // the bogus window of a (k-1)-long read: last base read as A (Q6)
    f &= ~3ull;
    r |= 3ull << (2 * (K - 1));
  }
  return f < r ? f : r;
}

struct Probe2Params {
  const u8* __restrict__ seq;
  u64 total;
  const u64* __restrict__ read_off;
  u64 n_reads;
  u64 tile_begin, tile_stop;  // this launch covers tiles [tile_begin, tile_stop)
  u64 span_base;              // global index of this launch's first span (hit region / count slot)
  u32 span_tiles, n_spans;    // spans of span_tiles tiles, handed out through *span_ctr
  u32* span_ctr;
  u32 blk_stream;             // blocked filter too large for L2: fetch its blocks with evict_first
  const u32* __restrict__ filt;
  u32 filt_mask;
  const u32* __restrict__ filt1;  // presence filter of the sub-mers
  u32 filt1_words;  // presence filter size in 32-bit words (any number)
  TabView tab;
  u32* hit_read;  // hit records (first hit of a run on one group + number of followers), see common.cuh
  u32* hit_w;
  u32* hit_row;
  u32* hit_gidx;
  u8* hit_nf;
  u64 hit_cap;
  u32* flags;
  u32* warp_cnt;  // hits found in each span (they sit at span * cap_w in the hit arrays)
  u64 cap_w;
};

// L2 residency: the reads stream through once (evict_first), the filter that every window group touches
// must survive that stream (evict_last).  Without the hints the 4-12 GB read stream keeps evicting the
// 32-64 MiB filter and every filter access becomes a 64-byte HBM fetch (profiles/k_probe2_h3100_r1k.txt).
__device__ __forceinline__ u64 p_policy_stream() {
  u64 p;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ u64 p_policy_keep() {
  u64 p;
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ uint4 p_ldg_v4(const uint4* ptr, u64 pol) {
  uint4 v;
  // .L2::64B: a sector miss fills 64 bytes of the line instead of all 128 (profiles/microbench/fetch_granularity.cu:
  // 61 instead of 118 bytes of DRAM traffic per random 16-byte read, at the same 40 G reads/s)
  asm volatile("ld.global.nc.L2::cache_hint.L2::64B.v4.u32 {%0,%1,%2,%3}, [%4], %5;"
               : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w)
               : "l"(ptr), "l"(pol));
  return v;
}
__device__ __forceinline__ u32 p_ldg_u32(const u32* ptr, u64 pol) {
  u32 v;
  asm volatile("ld.global.nc.L2::cache_hint.L2::64B.u32 %0, [%1], %2;" : "=r"(v) : "l"(ptr), "l"(pol));
  return v;
}

// ---- tile staging: ONE 1-D bulk copy (TMA, cp.async.bulk + mbarrier) per warp tile -------------------------
// A tile is 512 consecutive bases = 512 B of ASCII (128 B of 2-bit words when PACKED), contiguous in HBM and
// 16-byte aligned: lane 0 arms the warp's mbarrier with the byte count and issues the copy (evict_first: the
// reads stream through L2 once), all lanes wait on the barrier's phase when they need the bytes.  Replaces
// 32 cp.async (LDGSTS) + commit / wait_group per tile.
__device__ __forceinline__ u32 p_smem_addr(const void* p) { return (u32)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void p_bar_init(u64* bar) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;\n" ::"r"(p_smem_addr(bar)) : "memory");
  asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
}
__device__ __forceinline__ void p_bar_wait(u64* bar, u32 phase) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "PW_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra PW_DONE;\n"
      "bra PW_WAIT;\n"
      "PW_DONE:\n"
      "}\n" ::"r"(p_smem_addr(bar)),
      "r"(phase)
      : "memory");
}
// bytes of `tile` that exist in the batch's sequence buffer, rounded up to the 16 bytes a bulk copy moves (the
// buffer carries >= 64 bytes of slack); 0 beyond the end
template <bool PACKED>
__device__ __forceinline__ u32 p_tile_bytes(u64 tile, u64 total) {
  const u64 unit = PACKED ? PW_TILE / 4 : PW_TILE;
  const u64 have = PACKED ? 4 * ((total + 15) >> 4) : total;
  const u64 b0 = tile * unit;
  if (b0 >= have) return 0;
  const u64 r = have - b0;
  return r >= unit ? (u32)unit : (u32)((r + 15) & ~15ull);
}
// FULL: the caller knows that the tile lies entirely inside the batch (every tile of a span but the batch's last few)
template <bool PACKED, bool FULL = false>
__device__ __forceinline__ void p_stage_issue(WarpSmem& sm, const u8* __restrict__ seq, u64 tile, u64 total, int lane, u64 pol) {
  const u32 bytes = FULL ? (PACKED ? PW_TILE / 4 : PW_TILE) : p_tile_bytes<PACKED>(tile, total);
  if (lane == 0 && bytes) {
    const u32 bar = p_smem_addr(&sm.bar), dst = p_smem_addr(&sm.raw[0]);
    const u8* src = seq + tile * (PACKED ? PW_TILE / 4 : PW_TILE);
    // the lanes' reads of the previous tile in sm.raw (generic proxy; a __syncwarp lies in between) come before the
    // copy engine's writes (async proxy)
    asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(bar), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;\n" ::"r"(dst),
                 "l"(src), "r"(bytes), "r"(bar), "l"(pol)
                 : "memory");
  }
}
// wait for the tile's bytes and pack them into ring slot `rb` (forward + reverse complement); `phase` is the
// warp's barrier phase (flips whenever a copy was waited for)
template <bool PACKED, bool FULL = false>
__device__ __forceinline__ void p_stage_finish(WarpSmem& sm, u32 rb, u64 tile, u64 total, int lane, u32& phase) {
  if (FULL) {
    p_bar_wait(&sm.bar, phase);
    phase ^= 1u;
    u32 w;
    if (PACKED) {
      w = ((const u32*)sm.raw)[lane];
    } else {
      const uint4 v = sm.raw[lane];
      u32 bad = 0;
      w = p_pack16_be_fast(v, bad);
      if (__any_sync(0xFFFFFFFFu, bad != 0)) w = p_pack16_be(v);  // N runs, U, control bytes: the exact byte map
    }
    sm.fw[(rb + lane) & 63] = w;
    sm.rc[(rb + lane) & 63] = p_rc16(w);
    return;
  }
  const u32 bytes = p_tile_bytes<PACKED>(tile, total);
  if (bytes) {
    p_bar_wait(&sm.bar, phase);
    phase ^= 1u;
  }
  u32 w = 0;
  if (PACKED) {
    if (4u * lane < bytes) w = ((const u32*)sm.raw)[lane];  // the word array is zero-padded to whole words
  } else {
    uint4 v = make_uint4(0u, 0u, 0u, 0u);
    const u64 g = tile * PW_TILE + 16ull * lane;
    const bool tail = g + 16 > total;  // the last bases of the batch: bytes beyond the end read as 0 (-> A; their windows are invalid)
    if (16u * lane < bytes) {
      v = sm.raw[lane];
      if (tail) {
        const u32 nv = g < total ? (u32)(total - g) : 0u;
        u32 x[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int i = 0; i < 4; i++) {
          const u32 left = nv > 4u * i ? nv - 4u * i : 0u;
          x[i] &= left >= 4u ? 0xFFFFFFFFu : ((1u << (8 * left)) - 1u);
        }
        v = make_uint4(x[0], x[1], x[2], x[3]);
      }
    }
    u32 bad = 0;
    w = p_pack16_be_fast(v, bad);
    if (__any_sync(0xFFFFFFFFu, (bad != 0) | tail)) w = p_pack16_be(v);  // N runs, U, control bytes, the batch's tail: the exact byte map
  }
  sm.fw[(rb + lane) & 63] = w;
  sm.rc[(rb + lane) & 63] = p_rc16(w);
}

// SMALL: the blocked filter is L2-resident (<= 32 MiB): few groups pass the presence gate, one window round
// is the rule and gets a path without the multi-round bookkeeping
template <int K, bool PACKED, bool SMALL>
__global__ void __launch_bounds__(PW_WARPS * 32, PW_BLOCKS) k_probe2(const Probe2Params P) {
  __shared__ WarpSmem sm_all[PW_WARPS];
  const int lane = threadIdx.x & 31;
  WarpSmem& sm = sm_all[threadIdx.x >> 5];
  constexpr int CMAX = (K + 15 + 15) / 16;
  constexpr u32 ALL = 0xFFFFFFFFu;
  // Filter groups: J consecutive windows share the (K-J+1)-mer that starts at the last of them, and
  // every SUNK was inserted under each of its J sub-mers (table.cu)
  constexpr int J = GVS_FJ(K);
  constexpr int L = K - J + 1;
  constexpr int NG = 16 / J;
  const u64 pol_keep = p_policy_keep();
  const u64 pol_stream = p_policy_stream();
  const u64 pol_blk = P.blk_stream ? pol_stream : pol_keep;
  if (lane == 0) p_bar_init(&sm.bar);
  __syncwarp();
  u32 phase = 0;  // parity of the warp's mbarrier: flips with every tile copy waited for

  for (;;) {
    // ---- next span of tiles ----
    u32 span = 0;
    if (lane == 0) span = atomicAdd(P.span_ctr, 1u);
    span = __shfl_sync(ALL, span, 0);
    if (span >= P.n_spans) break;
    const u64 tile0 = P.tile_begin + (u64)span * P.span_tiles;
    u64 tile_end = tile0 + P.span_tiles;
    if (tile_end > P.tile_stop) tile_end = P.tile_stop;
    const u64 region = P.span_base + span;

    // cursor: first boundary index j >= 1 with read_off[j] > tile start; prev_off = start of the read
    // that contains the tile start
    u64 cur;
    {
      u64 ts0 = tile0 * PW_TILE;
      u64 lo = 1, hi = P.n_reads;
      while (lo < hi) {
        u64 mid = (lo + hi) >> 1;
        if (__ldg(P.read_off + mid) > ts0) hi = mid; else lo = mid + 1;
      }
      cur = lo;
    }
    u64 next_off = __ldg(P.read_off + cur);
    u64 prev_off = __ldg(P.read_off + cur - 1);

    // prologue: tiles T0 and T0+1 into ring slots 0 and 1
    __syncwarp();
    p_stage_issue<PACKED>(sm, P.seq, tile0, P.total, lane, pol_stream);
    p_stage_finish<PACKED>(sm, 0, tile0, P.total, lane, phase);
    __syncwarp();
    p_stage_issue<PACKED>(sm, P.seq, tile0 + 1, P.total, lane, pol_stream);
    p_stage_finish<PACKED>(sm, 32, tile0 + 1, P.total, lane, phase);
    __syncwarp();

    // all tiles this span stages (its own and the two prefetched past its end) lie entirely inside the batch: no tail handling
    const bool span_full = (tile_end + 2) * PW_TILE <= P.total;
    u32 wcount = 0;  // hits of this span so far
    for (u64 tile = tile0; tile < tile_end; tile++) {
      const u64 ts = tile * PW_TILE;
      const u32 rb = (u32)((tile - tile0) & 1) * 32;  // ring base of this tile
      // prefetch tile T+2 (lands in sm.raw while this tile is processed)
      if (span_full) p_stage_issue<PACKED, true>(sm, P.seq, tile + 2, P.total, lane, pol_stream);
      else p_stage_issue<PACKED>(sm, P.seq, tile + 2, P.total, lane, pol_stream);

      // ---- read boundaries in (ts, ts + 512 + K - 2] ----
      const u64 limit = ts + PW_TILE + (K > 1 ? K - 1 : 1);
      const u64 cur0 = cur;
      u32 nb = 0;
      const bool has_bound = next_off < limit;
      // the read that starts exactly at ts (its boundary belongs to the previous tile) may be (K-1) long
      const bool start_short = K >= 2 && prev_off == ts && next_off - prev_off == (u64)(K - 1);
      if (has_bound) {
        if (lane < 20) { sm.bound[lane] = 0; sm.shrt[lane] = 0; }
        __syncwarp();
        u64 j = cur + lane;
        for (;;) {
          u64 o = (j <= P.n_reads) ? __ldg(P.read_off + j) : ~0ull;
          bool inr = o < limit;
          bool intile = inr && (o - ts) < PW_TILE;
          u32 bal_tile = __ballot_sync(ALL, intile);
          if (inr) {
            u32 rel = (u32)(o - ts);
            atomicOr(&sm.bound[rel >> 5], 1u << (rel & 31));
            if (intile) {
              u32 slot = nb + __popc(bal_tile & ((1u << lane) - 1));
              if (slot < PW_MAXB) { sm.bpos[slot] = rel; sm.bidx[slot] = (u32)j; }
              if (K >= 2 && j < P.n_reads && __ldg(P.read_off + j + 1) - o == (u64)(K - 1))
                atomicOr(&sm.shrt[rel >> 5], 1u << (rel & 31));
            }
          }
          nb += __popc(bal_tile);
          u32 bal_adv = __ballot_sync(ALL, o <= ts + PW_TILE);
          cur += __popc(bal_adv);
          u32 bal_in = __ballot_sync(ALL, inr);
          if (bal_in != ALL) break;
          j += 32;
        }
        next_off = (cur <= P.n_reads) ? __ldg(P.read_off + cur) : ~0ull;
        prev_off = __ldg(P.read_off + cur - 1);
        __syncwarp();
      }

      // ---- per lane: its 16 windows in NG groups; presence test of every group's shared sub-mer ----
      u32 cm = 0;  // candidate (filter-positive) windows of this lane
      u32 S16 = 0;
      u32 pass = 0;  // groups whose sub-mer is (probably) a sub-mer of some SUNK
      u32 hbv[NG];
      {
        const u32 wb = rb + lane;
        const u32 f0 = sm.fw[wb & 63], f1 = sm.fw[(wb + 1) & 63], f2 = sm.fw[(wb + 2) & 63];
        // rc words in DEscending ring order: r_j = rc of forward word (lane + CMAX - 1 - j)
        const u32 r0 = sm.rc[(wb + CMAX - 1) & 63], r1 = sm.rc[(wb + CMAX - 2) & 63], r2 = sm.rc[(wb + CMAX - 3) & 63],
                  r3 = sm.rc[(wb + CMAX - 4) & 63];
        // validity: no boundary inside (p, p+K-1], p < total
        u32 inval = 0;
        if (has_bound) {
          int idx = lane >> 1, sh = (lane & 1) * 16;
          u64 B = ((u64)sm.bound[idx] | ((u64)sm.bound[idx + 1] << 32)) >> sh;
          if (sh) B |= (u64)sm.bound[idx + 2] << 48;
          u64 x = 0;
          if (K >= 2) {
            x = B >> 1;
            int c = 1;
#pragma unroll
            for (int it = 0; it < 6; it++) {
              if (c < K - 1) {
                int step = (K - 1 - c) < c ? (K - 1 - c) : c;
                x |= x >> step;
                c += step;
              }
            }
          }
          inval = (u32)x & 0xFFFFu;
          S16 = (sm.shrt[idx] >> sh) & 0xFFFFu;
        }
        if (start_short && lane == 0) S16 |= 1u;
        {
          u64 p0 = ts + 16ull * lane;
          if (p0 + 16 > P.total) {
            u32 nv = p0 < P.total ? (u32)(P.total - p0) : 0u;
            inval |= 0xFFFFu & ~((1u << nv) - 1);
          }
        }
        sm.inv[lane] = (u16)inval;
        if (lane < PW_TILE / 32) sm.cand[lane] = 0;
        u32 w1[NG];
#pragma unroll
        for (int g = 0; g < NG; g++) {
          const int o = J * g + (J - 1);  // lane-relative base offset of the shared sub-mer
          u64 sf = p_extract<L>(f0, f1, f2, o);
          const int e = o + L;            // = J*g + K, inside [K, K+15] like the windows' own ends
          const int c = (e + 15) / 16;
          const int j0 = CMAX - c;
          const int off = 16 * c - e;
          u64 sr = (j0 == 0) ? p_extract<L>(r0, r1, r2, off) : p_extract<L>(r1, r2, r3, off);
          hbv[g] = gvs_bhash(sf < sr ? sf : sr);
          const u32 gm = (1u << J) - 1;
          const bool any_valid = ((inval >> (J * g)) & gm) != gm;
          w1[g] = any_valid ? p_ldg_u32(P.filt1 + gvs_p1_word(hbv[g], P.filt1_words), pol_keep) : 0u;
        }
#pragma unroll
        for (int g = 0; g < NG; g++)  // both bits of gvs_p1_bits(hb) set in the word (the funnel shift wraps mod 32)
          pass |= (__funnelshift_r(w1[g], 0u, hbv[g]) & __funnelshift_r(w1[g], 0u, hbv[g] >> 5) & 1u) << g;
      }
      auto read_of = [&](u32 prel) -> u32 {
        if (!has_bound) return (u32)(cur0 - 1);
        if (nb <= PW_MAXB) {
          u32 rd = (u32)(cur0 - 1), bestpos = 0;
          bool any = false;
          for (u32 q = 0; q < nb; q++) {
            u32 bp = sm.bpos[q], bj = sm.bidx[q];
            if (bp <= prel && (!any || bp > bestpos || (bp == bestpos && bj > rd))) {
              any = true;
              bestpos = bp;
              rd = bj;
            }
          }
          return rd;
        }
        u64 p = ts + prel;
        u64 l = 1, h2 = P.n_reads;
        while (l < h2) {
          u64 mid = (l + h2) >> 1;
          if (__ldg(P.read_off + mid) > p) h2 = mid; else l = mid + 1;
        }
        return (u32)(l - 1);
      };
      // The hits of a lookup round (lane order = position order) are written out at once: runs of
      // consecutive hits on one group inside one read collapse into ONE record (first hit + number of
      // followers) -- kmerpos_annot3 prints only the first (nim:92), the others just shift the positions
      // reported later in the read (Q3).  Runs are cut at round and tile boundaries; the emit pass
      // (match.cu) merges what was cut.
      auto emit_round = [&](u32 row, u32 gi, u32 pp) {
        u32 rd = 0;
        const bool hit = row != GVS_NOHIT;
        const u32 bal = __ballot_sync(ALL, hit);
        if (bal == 0) return;  // warp-uniform
        if (hit) rd = read_of(pp);
        const u32 below = bal & ((1u << lane) - 1);
        const int prev = below ? 31 - __clz(below) : lane;  // the hit before this one in the round
        const u32 gi_prev = __shfl_sync(ALL, gi, prev), rd_prev = __shfl_sync(ALL, rd, prev);
        const bool head = hit && (below == 0 || gi != gi_prev || rd != rd_prev);
        const u32 hb = __ballot_sync(ALL, head);
        const u32 nrec = __popc(hb);
        const bool fits = (u64)wcount + nrec <= P.cap_w;
        if (!fits && lane == 0) atomicOr(P.flags, FLAG_OVERFLOW);
        if (head && fits) {
          const u32 above = lane == 31 ? 0u : (hb >> (lane + 1)) << (lane + 1);
          const u32 upto = above ? ((1u << (__ffs(above) - 1)) - 1) : 0xFFFFFFFFu;  // lanes below the next head
          const u32 after = lane == 31 ? 0u : ~((2u << lane) - 1);                    // lanes above this one
          const u64 o = region * P.cap_w + wcount + __popc(hb & ((1u << lane) - 1));
          P.hit_read[o] = rd;
          // low word of the hit's batch position: the gather pass (match.cu) subtracts the read's start, so that no
          // dependent load of read_off[rd] sits on the warp's path
          P.hit_w[o] = (u32)(ts + pp);
          P.hit_row[o] = row;
          P.hit_gidx[o] = gi;
          P.hit_nf[o] = (u8)__popc(bal & upto & after);
        }
        wcount += nrec;
      };
      const bool any_s16 = SMALL && __any_sync(ALL, S16 != 0);
      bool fused = false;  // SMALL: the tile's hits were already written by the single-round path
      // ---- passing groups -> warp queue (position order); their windows are tested one per lane ----
      if (__any_sync(ALL, pass != 0)) {
        const u32 np_lane = __popc(pass);
        u32 incl = np_lane;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
          u32 o = __shfl_up_sync(ALL, incl, d);
          if (lane >= d) incl += o;
        }
        const u32 n_grp = __shfl_sync(ALL, incl, 31);
        u32 qo = incl - np_lane;
#pragma unroll
        for (int g = 0; g < NG; g++) {
          if ((pass >> g) & 1u) {
            sm.q_p[qo] = (u16)(lane * NG + g);
            sm.q_row[qo] = hbv[g];
            qo++;
          }
        }
        __syncwarp();
        const u32 n_ent = n_grp * J;
        // (2, not more: a tile seldom queues more than 32 groups, and every extra round of loads held in registers
        // costs the whole kernel -- measured 24.3 ms with 2 or 1 against 24.6 ms with 4)
        constexpr int RB = 2;  // rounds whose block loads are issued back to back before any window math
        if (SMALL && n_ent <= 32 && !any_s16) {
          // one round, and the queue order is the position order: test, exact lookup and record output in
          // one go (no candidate bitmap, no second extraction of the k-mer)
          u32 row = GVS_NOHIT, gi = 0, p = 0;
          if ((u32)lane < n_ent) {
            const u32 q = lane / J, w = lane % J;
            p = (u32)sm.q_p[q] * J + w;
            const uint4 b4 = p_ldg_v4((const uint4*)P.filt + (sm.q_row[q] & P.filt_mask), pol_blk);
            const bool valid = !((sm.inv[p >> 4] >> (p & 15)) & 1u);
            const u64 canon = p_canon_at<K>(sm, rb, p, false);
            const u32 h = gvs_fhash(canon);
            const u32 t = __funnelshift_r(b4.x, 0u, h) & __funnelshift_r(b4.y, 0u, h >> 5) & __funnelshift_r(b4.z, 0u, h >> 10) &
                          __funnelshift_r(b4.w, 0u, h >> 15);
            if (valid && (t & 1u)) {
              row = tab_lookup(P.tab, canon, gvs_mix(canon), &gi);
              if (row == GVS_ROW_MISSING) {
                atomicOr(P.flags, FLAG_KEYERROR);
                row = GVS_NOHIT;
              } else if (row >= GVS_NOHIT) {
                row = GVS_NOHIT;
              }
            }
          }
          emit_round(row, gi, p);
          fused = true;
        } else if (SMALL) {
        for (u32 base = 0; base < n_ent; base += 32 * RB) {
          uint4 b4[RB];
          u32 pw[RB];
#pragma unroll
          for (int r = 0; r < RB; r++) {
            const u32 e = base + 32 * r + lane;
            pw[r] = 0xFFFFFFFFu;
            b4[r] = make_uint4(0, 0, 0, 0);
            if (e < n_ent) {
              const u32 q = e / J, w = e % J;
              pw[r] = (u32)sm.q_p[q] * J + w;  // window inside the tile
              b4[r] = p_ldg_v4((const uint4*)P.filt + (sm.q_row[q] & P.filt_mask), pol_blk);
            }
          }
#pragma unroll
          for (int r = 0; r < RB; r++) {
            if (base + 32 * r >= n_ent) break;  // warp-uniform
            const u32 p = pw[r];
            if (p != 0xFFFFFFFFu) {
              const bool valid = !((sm.inv[p >> 4] >> (p & 15)) & 1u);
              const u32 h = gvs_fhash(p_canon_at<K>(sm, rb, p, false));
              const u32 t = __funnelshift_r(b4[r].x, 0u, h) & __funnelshift_r(b4[r].y, 0u, h >> 5) &
                            __funnelshift_r(b4[r].z, 0u, h >> 10) & __funnelshift_r(b4[r].w, 0u, h >> 15);
              if (valid && (t & 1u)) atomicOr(&sm.cand[p >> 5], 1u << (p & 31));
            }
          }
        }
        } else {
        // Large database: ONE lane per passing group fetches the group's block (the loads of up to RB rounds
        // are issued together) and tests the fingerprint bit of the group's sub-mer in word 3 -- most passing
        // groups are false positives of the saturated presence filter and end here.  Only the windows of the
        // surviving groups are extracted, hashed and tested against the key words, which by then sit in
        // shared memory.
        for (u32 gbase = 0; gbase < n_grp; gbase += 32 * RB) {
          uint4 b4[RB];
          u32 hq[RB];
#pragma unroll
          for (int r = 0; r < RB; r++) {
            const u32 q = gbase + 32 * r + lane;
            hq[r] = 0;
            b4[r] = make_uint4(0, 0, 0, 0);
            if (q < n_grp) {
              hq[r] = sm.q_row[q];
              b4[r] = p_ldg_v4((const uint4*)P.filt + (hq[r] & P.filt_mask), pol_blk);
            }
          }
#pragma unroll
          for (int r = 0; r < RB; r++) {
            if (gbase + 32 * r >= n_grp) break;  // warp-uniform
            const u32 q = gbase + 32 * r + lane;
            const bool ok = q < n_grp && ((b4[r].w >> gvs_fp_bit(hq[r])) & 1u);
            const u32 bal = __ballot_sync(ALL, ok);
            if (bal == 0) continue;  // warp-uniform
            if (ok) {
              const u32 slot = __popc(bal & ((1u << lane) - 1));
              sm.s_p[slot] = sm.q_p[q];
              sm.s_blk[slot][0] = b4[r].x;
              sm.s_blk[slot][1] = b4[r].y;
              sm.s_blk[slot][2] = b4[r].z;
            }
            __syncwarp();
            const u32 n_win = __popc(bal) * J;
            for (u32 base = 0; base < n_win; base += 32) {
              const u32 e = base + lane;
              if (e < n_win) {
                const u32 sq = e / J, w = e % J;
                const u32 p = (u32)sm.s_p[sq] * J + w;
                const bool valid = !((sm.inv[p >> 4] >> (p & 15)) & 1u);
                const u32 h = gvs_fhash(p_canon_at<K>(sm, rb, p, false));
                const u32 t = __funnelshift_r(sm.s_blk[sq][0], 0u, h) & __funnelshift_r(sm.s_blk[sq][1], 0u, h >> 5) &
                              __funnelshift_r(sm.s_blk[sq][2], 0u, h >> 10);
                if (valid && (t & 1u)) atomicOr(&sm.cand[p >> 5], 1u << (p & 31));
              }
            }
            __syncwarp();
          }
        }
        }
        __syncwarp();
        if (!fused) cm = (sm.cand[lane >> 1] >> ((lane & 1) * 16)) & 0xFFFFu;
      }
      if (S16) {  // bogus windows of (K-1)-long reads: last base read as A, always "valid"
        for (u32 s16 = S16; s16; s16 &= s16 - 1) {
          int i = __ffs(s16) - 1;
          u32 p = 16u * lane + i;
          u64 canon = p_canon_at<K>(sm, rb, p, true);
          // its own first sub-mer (real bases only) selects the block
          u64 sub = (p_fwd_at<K>(sm, rb, p) & ~3ull) >> (2 * (K - L));
          u64 subr = gvs_revcomp(sub, L);
          uint4 b4 = __ldg((const uint4*)P.filt + (gvs_bhash(sub < subr ? sub : subr) & P.filt_mask));
          u32 h = gvs_fhash(canon);
          u32 t = __funnelshift_r(b4.x, 0u, h) & __funnelshift_r(b4.y, 0u, h >> 5) & __funnelshift_r(b4.z, 0u, h >> 10);
          if (SMALL) t &= __funnelshift_r(b4.w, 0u, h >> 15);  // large databases keep sub-mer fingerprints in word 3
          if (t & 1u) cm |= 1u << i; else cm &= ~(1u << i);
        }
      }
      cm |= (S16 << 16);  // remember which candidates are forced-A windows
      // ---- queue candidates in position order ----
      if (__any_sync(ALL, (cm & 0xFFFFu) != 0)) {
        u32 ncand_lane = __popc(cm & 0xFFFFu);
        u32 incl = ncand_lane;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
          u32 o = __shfl_up_sync(ALL, incl, d);
          if (lane >= d) incl += o;
        }
        const u32 ncand = __shfl_sync(ALL, incl, 31);
        u32 qo = incl - ncand_lane;
        for (u32 s = cm & 0xFFFFu; s; s &= s - 1) {
          int i = __ffs(s) - 1;
          sm.q_p[qo++] = (u16)((16u * lane + i) | (((cm >> (16 + i)) & 1) << 15));
        }
        __syncwarp();
        // ---- exact lookups, 32 candidates per round ----
        for (u32 base = 0; base < ncand; base += 32) {
          u32 row = GVS_NOHIT, gi = 0;
          u32 pp = 0;
          if (base + lane < ncand) {
            u32 e = sm.q_p[base + lane];
            pp = e & 0x7FFFu;
            u64 canon = p_canon_at<K>(sm, rb, pp, (e >> 15) != 0);
            row = tab_lookup(P.tab, canon, gvs_mix(canon), &gi);
            if (row == GVS_ROW_MISSING) {
              atomicOr(P.flags, FLAG_KEYERROR);
              row = GVS_NOHIT;
            } else if (row >= GVS_NOHIT) {
              row = GVS_NOHIT;
            }
          }
          emit_round(row, gi, pp);
        }
      }
      // ---- tile T is done: its ring slot receives tile T+2 ----
      __syncwarp();
      if (span_full) p_stage_finish<PACKED, true>(sm, rb, tile + 2, P.total, lane, phase);
      else p_stage_finish<PACKED>(sm, rb, tile + 2, P.total, lane, phase);
      __syncwarp();
    }
    if (lane == 0) P.warp_cnt[region] = wcount;
  }
}

typedef void (*probe_fn)(const Probe2Params);
static probe_fn probe_table(int k, bool packed, bool small) {
  switch (k) {
#ifdef GVS_PROBE_ONLY_K  // experiment builds: one SUNK_len, seconds instead of minutes
#define PK(n) case n: if (n != GVS_PROBE_ONLY_K) return nullptr; return packed ? (small ? k_probe2<GVS_PROBE_ONLY_K, true, true> : k_probe2<GVS_PROBE_ONLY_K, true, false>) \
                                    : (small ? k_probe2<GVS_PROBE_ONLY_K, false, true> : k_probe2<GVS_PROBE_ONLY_K, false, false>);
#else
#define PK(n) case n: return packed ? (small ? k_probe2<n, true, true> : k_probe2<n, true, false>) \
                                    : (small ? k_probe2<n, false, true> : k_probe2<n, false, false>);
#endif
    PK(1) PK(2) PK(3) PK(4) PK(5) PK(6) PK(7) PK(8) PK(9) PK(10) PK(11) PK(12) PK(13) PK(14) PK(15) PK(16)
    PK(17) PK(18) PK(19) PK(20) PK(21) PK(22) PK(23) PK(24) PK(25) PK(26) PK(27) PK(28) PK(29) PK(30) PK(31)
#undef PK
  }
  return nullptr;
}

// launches the probe over ctx's reads; span s's hits land at s * cap_w in ctx->hit_*, its count in
// ctx->tile_cnt[s] (zeroed here); flags to the CNT_FLAGS counter
int gvs_probe_launch(gvs_ctx* ctx, u64* n_warps_out, u64* cap_w_out) {
  u64 total = ctx->total_bases;
  u64 n_tiles = cdiv(total, PW_TILE);
  probe_fn fn = probe_table(ctx->k, ctx->seq_packed, !ctx->filt_fp);  // the variant follows the block layout (table.cu)
  if (!fn) return gvs_fail(ctx, GVS_E_ARG, "no probe kernel for k=%d", ctx->k);
  Probe2Params P;
  P.seq = ctx->seq;
  P.total = total;
  P.read_off = ctx->read_off;
  P.n_reads = ctx->n_reads;
  // launch plan: one launch for resident reads; for a host batch that is still arriving (ctx.cu) one
  // launch per copy segment, each released by the segment's event.  Inside a launch the tiles are cut
  // into spans (~32 per resident warp) that the warps draw from an atomic counter.
  struct Seg { u64 t0, t1, span_base, ev; u32 span_tiles, n_spans, blocks; };
  std::vector<Seg> plan;
  const bool piped = !ctx->seg_tile_end.empty() && ctx->seq == ctx->own_seq.as<u8>();
  const u64 n_launch = piped ? ctx->seg_tile_end.size() : 1;
  const u64 resident_warps = (u64)ctx->n_sm * PW_BLOCKS * PW_WARPS;
  u64 spans = 0;
  for (u64 s = 0, t0 = 0; s < n_launch; s++) {
    u64 t1 = piped ? ctx->seg_tile_end[s] : n_tiles;
    if (t1 > t0) {
      u64 st = cdiv(t1 - t0, resident_warps * 32);
      if (st < 8) st = 8;
      if (st > 1024) st = 1024;
      u64 ns = cdiv(t1 - t0, st);
      u64 blocks = cdiv(ns, PW_WARPS);
      if (blocks > (u64)ctx->n_sm * PW_BLOCKS) blocks = (u64)ctx->n_sm * PW_BLOCKS;
      plan.push_back({t0, t1, spans, s, (u32)st, (u32)ns, (u32)blocks});
      spans += ns;
    }
    t0 = t1;
  }
  if (spans >= 0xFFFFFFF0ull) return gvs_fail(ctx, GVS_E_OVERFLOW, "too many probe spans");
  *n_warps_out = spans;
  CKR(gvs_reserve(ctx, ctx->tile_cnt, spans * 4));
  CKR(gvs_reserve(ctx, ctx->tile_dst, spans * 8));
  CKR(gvs_reserve(ctx, ctx->tile_off, (plan.size() + 1) * 4));  // one span counter per launch
  CK(cudaMemsetAsync(ctx->tile_cnt.p, 0, spans * 4, ctx->stream));
  CK(cudaMemsetAsync(ctx->tile_off.p, 0, (plan.size() + 1) * 4, ctx->stream));
  P.cap_w = ctx->hit_cap / spans;
  *cap_w_out = P.cap_w;
  P.filt = ctx->filt.as<u32>();
  P.filt_mask = (u32)(ctx->filt_words - 1);
  P.filt1 = ctx->filt1.as<u32>();
  P.filt1_words = (u32)ctx->filt1_words;
  P.blk_stream = ctx->filt_words * 16 > (32ull << 20) ? 1u : 0u;
  P.tab.kv = ctx->tab_kv.as<u64>();
  P.tab.slots = ctx->tab_slots;
  P.hit_read = ctx->hit_read.as<u32>();
  P.hit_w = ctx->hit_w.as<u32>();
  P.hit_row = ctx->hit_row.as<u32>();
  P.hit_gidx = ctx->hit_gidx.as<u32>();
  P.hit_nf = ctx->hit_nf.as<u8>();
  P.hit_cap = ctx->hit_cap;
  P.flags = counter(ctx, CNT_FLAGS);
  P.warp_cnt = ctx->tile_cnt.as<u32>();
  // L2 persistence: the structure every window group touches (the presence filter) is pinned in the
  // persisting carve-out of L2; everything outside the window (reads, exact table, hit lists) is
  // treated as streaming.
  if (ctx->l2_persist_max < 0) {
    cudaDeviceGetAttribute(&ctx->l2_persist_max, cudaDevAttrMaxPersistingL2CacheSize, ctx->device);
    cudaDeviceGetAttribute(&ctx->l2_window_max, cudaDevAttrMaxAccessPolicyWindowSize, ctx->device);
    if (ctx->l2_persist_max < 0) ctx->l2_persist_max = 0;
  }
  const int persist_max = ctx->l2_persist_max, window_max = ctx->l2_window_max;
  {
    static bool said = false;
    if (!said && getenv("GVS_EXP_VERBOSE")) {
      said = true;
      fprintf(stderr, "[gvs] L2 persisting max %d B, access window max %d B, presence filter %llu B, block filter %llu B, table %llu slots\n",
              persist_max, window_max, (unsigned long long)ctx->filt1_words * 4, (unsigned long long)ctx->filt_words * 16,
              (unsigned long long)ctx->tab_slots);
    }
  }
  const void* hot = ctx->filt1.p;
  size_t hot_bytes = ctx->filt1_words * 4;
  cudaLaunchConfig_t cfg = {};
  cfg.blockDim = dim3(PW_WARPS * 32);
  cfg.dynamicSmemBytes = 0;
  cfg.stream = ctx->stream;
  cudaLaunchAttribute attr[1];
  int n_attr = 0;
  static const int exp_no_persist = getenv("GVS_EXP_NO_PERSIST") ? atoi(getenv("GVS_EXP_NO_PERSIST")) : 0;  // experiments
  if (persist_max > 0 && window_max > 0 && exp_no_persist != 1) {
    size_t carve = hot_bytes < (size_t)persist_max ? hot_bytes : (size_t)persist_max;
    if (exp_no_persist == 2) carve = (size_t)persist_max;
    if (ctx->l2_carve_set != carve) {
      cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, carve);
      ctx->l2_carve_set = carve;
    }
    size_t win = hot_bytes < (size_t)window_max ? hot_bytes : (size_t)window_max;
    attr[0].id = cudaLaunchAttributeAccessPolicyWindow;
    attr[0].val.accessPolicyWindow.base_ptr = const_cast<void*>(hot);
    attr[0].val.accessPolicyWindow.num_bytes = win;
    attr[0].val.accessPolicyWindow.hitRatio = win <= carve ? 1.0f : (float)carve / (float)win;
    attr[0].val.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
    attr[0].val.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
    n_attr = 1;
  }
  cfg.attrs = attr;
  cfg.numAttrs = n_attr;
  for (size_t s = 0; s < plan.size(); s++) {
    probe_fn fn_s = fn;
    P.seq = ctx->seq;
    if (piped) {
      // a segment of an ASCII host batch may have been packed on the host (ctx.cu HostPipe): wait until the
      // submitter has queued it, then scan it with the variant of its kind
      CKR(gvs_pipe_wait(ctx, plan[s].ev));
      if (!ctx->seg_packed.empty() && ctx->seg_packed[plan[s].ev]) {
        fn_s = probe_table(ctx->k, true, !ctx->filt_fp);
        P.seq = ctx->own_words.as<u8>();
      }
      CK(cudaStreamWaitEvent(ctx->stream, ctx->seg_ev[plan[s].ev], 0));
    }
    cfg.gridDim = dim3(plan[s].blocks);
    P.tile_begin = plan[s].t0;
    P.tile_stop = plan[s].t1;
    P.span_tiles = plan[s].span_tiles;
    P.n_spans = plan[s].n_spans;
    P.span_base = plan[s].span_base;
    P.span_ctr = ctx->tile_off.as<u32>() + s;
    cudaError_t e = cudaLaunchKernelEx(&cfg, fn_s, P);
    ctx->launches++;
    if (e == cudaSuccess) e = cudaGetLastError();
    if (e != cudaSuccess) return gvs_fail(ctx, GVS_E_CUDA, "k_probe2 launch: %s", cudaGetErrorString(e));
  }
  if (piped) CKR(gvs_pipe_join(ctx));
  return 0;
}
