// common.cuh -- context, device-buffer arena, error handling and the device-wide scan primitive
// shared by every stage of libgavisunk_b200.so.  sm_100a only.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <string>
#include <vector>

#include "../../include/gavisunk_b200.h"

typedef uint8_t u8;
typedef uint16_t u16;
typedef uint32_t u32;
typedef uint64_t u64;
typedef int32_t i32;
typedef int64_t i64;

#define GVS_NSM_DEFAULT 148
#define GVS_TILE_BASES 512                 // window starts per probe tile (probe.cu PW_TILE)
#define GVS_SEG_COUNT 16                   // copy/probe pipeline depth for host batches
#define GVS_SEG_COUNT_PACK 48              // ... when segments may be packed on the host (finer hand-over between link and cores)
#define GVS_SEG_MIN_BYTES (256ull << 20)   // smaller host batches are copied in one piece

// grow-only device buffer: stages re-use their scratch across calls so that the timed loop of
// bench.py never allocates after the first (warm-up) step.
struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  template <typename T>
  T* as() const { return (T*)p; }
};

struct Rows {  // sunkpos rows, structure of arrays (24 B per row)
  DevBuf read, pos, contig, start, group, gidx;
  u64 n = 0;
};

// a result table: u32 columns `stride` entries apart in one buffer, the first n entries of each filled; `ready` once the
// stage that writes it has run (rec_reserve / rec_get below)
struct RecTable {
  DevBuf buf;
  u64 n = 0, stride = 0;
  bool ready = false;
  u32* col(u32 t) const { return buf.as<u32>() + t * stride; }
};

struct gvs_ctx {
  int device = 0;
  int k = 20;
  int n_sm = GVS_NSM_DEFAULT;
  cudaStream_t stream = 0;
  std::string err;
  u64 launches = 0;
  bool profiling = false;
  cudaEvent_t ev0[GVS_ST_COUNT], ev1[GVS_ST_COUNT];
  bool ev_valid[GVS_ST_COUNT];
  std::vector<void*> pinned;  // small pinned host staging blocks
  // side streams for independent launches of one stage (e.g. the row-count tiers of the validation):
  // gvs_fork makes them wait for everything queued on `stream`, gvs_join makes `stream` wait for them
  cudaStream_t aux[2] = {nullptr, nullptr};
  // per-device one-time settings (a process may drive one context per GPU: no function-level statics)
  bool val_attr_set = false;                  // dynamic shared memory opt-in of k_validate
  int l2_persist_max = -1, l2_window_max = 0;  // L2 persistence limits of this device
  size_t l2_carve_set = 0;
  cudaEvent_t ev_fork = nullptr, ev_join[2] = {nullptr, nullptr};

  // ---- database ----
  bool db_ready = false;
  u64 n_loc = 0, n_groups = 0;
  u32 n_contigs = 0;
  DevBuf loc_kmer, loc_contig, loc_start, loc_group, loc_gidx;  // per .loc row
  DevBuf loc_pack;                                               // per .loc row: (contig, start, group, 0) in one 16-byte word for the emit pass
  DevBuf grp_contig, grp_start;                                  // per group (index = gidx)
  u64 grp_gen = 0;                                               // bumped whenever the group table is rebuilt
  DevBuf tab_keys, tab_rows, tab_kv;                             // open-addressed probe table: (build only) keys and rows; buckets of 4 keys + 4 (group index << 32 | row) words
  u64 tab_slots = 0;                                             // power of two, buckets of 4
  DevBuf filt;                                                   // 32-bit-word blocked Bloom filter
  u64 filt_words = 0;                                            // number of 16-byte blocks, power of two
  bool filt_fp = false;                                          // block layout: word 3 = sub-mer fingerprints (gvs_fp_bit), keys in words 0..2
  int probe_variant = 0;                                         // gvs_set_probe_variant: 0 by size, 1 small-database, 2 large-database
  DevBuf filt1;                                                  // presence filter of the sub-mers (large databases)
  u64 filt1_words = 0;                                           // 0 = single-level filter
  DevBuf contig_hap, contig_hash, contig_len;

  // ---- reads ----
  bool reads_ready = false;
  const u8* seq = nullptr;     // device: ASCII bases, or (seq_packed) 2-bit words of 16 bases, big-endian
  bool seq_packed = false;
  const u64* read_off = nullptr;  // device, n_reads+1
  u64 n_reads = 0, total_bases = 0;
  DevBuf own_seq, own_off;     // when copied from the host
  // host batches are copied in segments on a second stream; the probe of segment s is launched as soon
  // as its bytes (+ a two-tile halo) have landed, so the PCIe transfer hides the compute
  cudaStream_t copy_stream = nullptr;
  cudaEvent_t ev_reads_free = nullptr;  // everything that read the previous batch has finished
  std::vector<cudaEvent_t> seg_ev;      // seg_ev[s]: bytes of segments 0..s are in HBM
  std::vector<u64> seg_tile_end;        // tile index (512 bases) where segment s ends; empty = one launch
  u64 seg_min_bytes = GVS_SEG_MIN_BYTES;
  u32 seg_count = GVS_SEG_COUNT;
  bool seg_count_set = false;           // gvs_set_copy_pipeline was called
  // host batches of ASCII bases: a segment travels either as it is or 2-bit packed by host threads
  // (hostpack.cpp) through a page-locked staging buffer -- the PCIe link and the host cores work side by
  // side (ctx.cu HostPipe).  seg_packed[s] selects the probe variant and the device buffer of segment s.
  DevBuf own_words;
  std::vector<u8> seg_packed;           // empty: every segment lives in `seq` as seq_packed says
  struct HostPipe* pipe = nullptr;
  int pack_mode = GVS_PACK_ADAPTIVE;
  int pack_threads = 0;                 // 0 = the cores this process may run on, at most 16
  u64 h2d_bytes = 0;                    // sequence bytes the last host batch put on the link
  u32 h2d_segs = 0, h2d_segs_packed = 0;
  DevBuf chunk_first, chunk_hap;  // device copies
  std::vector<u64> h_chunk_first;
  std::vector<u8> h_chunk_hap;
  u32 n_chunks = 0;
  DevBuf read_len;             // explicit lengths (gvs_reads_meta) when there are no sequences
  bool have_read_len = false;
  DevBuf gt_keys, gt_val;      // (contig, group) -> group index lookup for gvs_rows_set
  u64 gt_slots = 0;
  bool groups_ready = false;   // grp_contig / grp_start / n_groups valid (database or rows-derived)

  // ---- match ----
  DevBuf tile_first;                  // DB build: first contig of every tile
  DevBuf tile_cnt, tile_off, tile_dst;  // probe spans: record count, span counters of the launches, dense destination
  // hit records: the first hit of a run of consecutive hits on ONE group inside one read (and one probe
  // tile), with the number of hits that follow it in the run -- kmerpos_annot3 prints only the first
  // (nim:92) and the others merely shift later positions (Q3)
  DevBuf hit_read, hit_w, hit_row, hit_gidx, hit_nf;       // per probe span
  DevBuf ohit_read, ohit_w, ohit_row, ohit_gidx, ohit_nf;  // dense, position order
  u64 hit_cap = 0, n_hits = 0;
  DevBuf counters;                     // small block of device counters / flags
  void* mailbox = nullptr;             // 256 page-locked bytes: where read_dev() lands the scalars the host needs (sizes, flags)
  DevBuf scan_tmp, scan_tmp2, flags_a, flags_b, flags_c;
  Rows rows;                           // gvs_match output
  bool match_ready = false;

  // ---- diag ----
  DevBuf seg_start;     // per segment (read with rows): first row, n_seg+1
  u64 n_seg = 0;
  DevBuf seg_ndist, seg_cap, seg_best, seg_good, seg_dir;
  DevBuf diag_scratch;
  Rows kept;
  DevBuf best_read, best_contig, best_good, best_dir;
  u64 n_best = 0;
  bool diag_ready = false;
  // kept rows + read lengths of the batches of one run (batches.cu): read indices count through the batches
  Rows stash;
  DevBuf stash_len;
  u64 stash_reads = 0;
  // haplotype mode of the diag filter (diag.cu): per segment the best contig of both haplotypes, and the records
  DevBuf rh_scratch;
  RecTable rh;       // records of the last diag filter in haplotype mode; after gvs_batches_bind those of the run
  RecTable rh_run;   // records of the run's batches so far (run-wide read indices), appended by gvs_batch_stash

  // ---- histogram / bad groups ----
  DevBuf hist, cnt_hist, bad_flag, bad_list;
  u64 n_bad = 0;
  bool hist_ready = false, bad_ready = false;

  // ---- validation ----
  DevBuf kseg_start;  // segments of kept rows
  u64 n_kseg = 0;
  DevBuf val_scratch;
  // gvs_validate's outputs per kept row (the read's validated IDs, from its first row on) and per segment (their count
  // and their offset in the pairs)
  const u32 *val_id = nullptr, *val_seg_cnt = nullptr, *val_seg_off = nullptr;
  DevBuf pair_read, pair_contig, pair_group, pair_gidx;
  DevBuf seg_orient;  // per segment: orientation majority of the read (0: positions rise with starts)
  u64 n_pairs = 0;
  bool val_ready = false;

  // ---- support tracks (support.cu) ----
  u64 rank_gen = ~0ull;             // grp_gen the rank below was computed for
  u64 order_gen = ~0ull;            // grp_gen rank_identity was found for
  bool rank_identity = false;       // group index order is already (contig, start) order
  DevBuf rank_of, rank_grp;         // group index -> rank in (contig, start) order, and back (unless identity)
  DevBuf sup_diff;                  // int32[n_groups] by rank: +1 at a placement's first group, -1 at its last
  RecTable pl;                      // placements: read, contig, start, end, IDs
  DevBuf pl_strand, pl_tmp;         // per placement its strand (u8); per segment (start, end, IDs, strand)
  DevBuf sup_depth, sup_gx, sup_cstat;
  RecTable sup;                     // runs of gvs_support: contig, start, end, depth

  // ---- gap evidence (gap_evidence.cu) ----
  DevBuf ge_seg_start;              // segments of the kept rows when gvs_validate's are not current
  DevBuf ge_cgap, ge_seg, ge_cand, ge_res;  // per contig gap range, per segment (first gap, count), candidates, their results
  RecTable ge;                      // records: 8 columns, one entry per candidate

  // ---- junctions (junctions.cu) ----
  Rows jn_stash;                    // rows gvs_junction_screen kept (run-wide read indices), input of gvs_junctions
  u64 jn_reads = 0;                 // reads in jn_stash
  bool jn_in_run = false;           // between gvs_batches_begin and gvs_batches_bind: a screen appends to jn_stash
  DevBuf jn_seg_start, jn_row_seg, jn_seg_cnt;  // segments of the screened / stashed rows, per segment count or offset
  DevBuf jn_flags, jn_scr;          // per-row flags (2 bytes) and per-row u32 scratch of gvs_junctions
  RecTable jn;                      // records: 13 columns

  // ---- discordance (discordance.cu) ----
  DevBuf dc_diff;                   // int32[3][n_groups] by rank: spans, longer, shorter (+1 at a span's first group, -1 at its last)
  DevBuf dc_scr, dc_seg;            // per kept row u32 scratch (4 arrays); per segment usable rows, records, record offset
  RecTable dc;                      // span records of gvs_spans: 8 columns
  RecTable dc_runs;                 // runs of gvs_discordance: contig, start, end, spans, longer, shorter

  // ---- components / intervals / gaps ----
  DevBuf parent, present, comp_min, comp_max, comp_cnt;
  DevBuf comp_rank;  // unsorted group tables only: [smallest member rank per root | root per interval rank]
  DevBuf iv_contig, iv_start, iv_end;
  u64 n_iv = 0;
  DevBuf gap_contig, gap_start, gap_end, nodata_contig;
  u64 n_gaps = 0, n_nodata = 0;
  bool comp_ready = false, iv_ready = false, gaps_ready = false;
};

// -------------------------------------------------------------------------------------------
// error handling
// -------------------------------------------------------------------------------------------
static inline int gvs_fail(gvs_ctx* c, int code, const char* fmt, ...) __attribute__((format(printf, 3, 4)));
#include <stdarg.h>
static inline int gvs_fail(gvs_ctx* c, int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  if (c) c->err = buf;
  return code;
}

#define CK(call)                                                                            \
  do {                                                                                      \
    cudaError_t e__ = (call);                                                               \
    if (e__ != cudaSuccess)                                                                 \
      return gvs_fail(ctx, GVS_E_CUDA, "%s:%d %s: %s", __FILE__, __LINE__, #call,           \
                      cudaGetErrorString(e__));                                             \
  } while (0)

#define CKR(call)            \
  do {                       \
    int r__ = (call);        \
    if (r__ != 0) return r__; \
  } while (0)

// kernel launch with launch counting + error check
#define LAUNCH(kern, grid, block, smem, ...)                                                \
  do {                                                                                      \
    kern<<<(grid), (block), (smem), ctx->stream>>>(__VA_ARGS__);                            \
    ctx->launches++;                                                                        \
    cudaError_t e__ = cudaGetLastError();                                                   \
    if (e__ != cudaSuccess)                                                                 \
      return gvs_fail(ctx, GVS_E_CUDA, "%s:%d launch %s: %s", __FILE__, __LINE__, #kern,    \
                      cudaGetErrorString(e__));                                             \
  } while (0)

#define LAUNCH_ON(strm, kern, grid, block, smem, ...)                                       \
  do {                                                                                      \
    kern<<<(grid), (block), (smem), (strm)>>>(__VA_ARGS__);                                 \
    ctx->launches++;                                                                        \
    cudaError_t e__ = cudaGetLastError();                                                   \
    if (e__ != cudaSuccess)                                                                 \
      return gvs_fail(ctx, GVS_E_CUDA, "%s:%d launch %s: %s", __FILE__, __LINE__, #kern,    \
                      cudaGetErrorString(e__));                                             \
  } while (0)

static inline int gvs_fork(gvs_ctx* ctx) {
  if (!ctx->aux[0]) {
    for (int i = 0; i < 2; i++) {
      CK(cudaStreamCreateWithFlags(&ctx->aux[i], cudaStreamNonBlocking));
      CK(cudaEventCreateWithFlags(&ctx->ev_join[i], cudaEventDisableTiming));
    }
    CK(cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming));
  }
  CK(cudaEventRecord(ctx->ev_fork, ctx->stream));
  for (int i = 0; i < 2; i++) CK(cudaStreamWaitEvent(ctx->aux[i], ctx->ev_fork, 0));
  return 0;
}
static inline int gvs_join(gvs_ctx* ctx) {
  for (int i = 0; i < 2; i++) {
    CK(cudaEventRecord(ctx->ev_join[i], ctx->aux[i]));
    CK(cudaStreamWaitEvent(ctx->stream, ctx->ev_join[i], 0));
  }
  return 0;
}

static inline int gvs_reserve(gvs_ctx* ctx, DevBuf& b, size_t bytes) {
  if (bytes == 0) bytes = 16;
  if (b.cap >= bytes) return 0;
  // stream-ordered work may still use the old block: wait before freeing
  if (b.p) {
    CK(cudaStreamSynchronize(ctx->stream));
    CK(cudaFree(b.p));
    b.p = nullptr;
    b.cap = 0;
  }
  size_t want = bytes + bytes / 8 + 256;  // slack so that slightly larger batches do not realloc
  cudaError_t e = cudaMalloc(&b.p, want);
  if (e != cudaSuccess) {
    b.p = nullptr;
    return gvs_fail(ctx, GVS_E_NOMEM, "cudaMalloc(%zu bytes): %s", want, cudaGetErrorString(e));
  }
  b.cap = want;
  return 0;
}

static inline void gvs_release(DevBuf& b) {
  if (b.p) cudaFree(b.p);
  b.p = nullptr;
  b.cap = 0;
}

struct StageTimer {
  gvs_ctx* c;
  int st;
  StageTimer(gvs_ctx* c_, int st_) : c(c_), st(st_) {
    if (c->profiling) cudaEventRecord(c->ev0[st], c->stream);
  }
  ~StageTimer() {
    if (c->profiling) {
      cudaEventRecord(c->ev1[st], c->stream);
      c->ev_valid[st] = true;
    }
  }
};

// ctx.cu: segment `seg` of a host batch has been handed to the copy stream (its event is recorded);
// blocks while the submitter thread is still packing it
int gvs_pipe_wait(gvs_ctx* ctx, u64 seg);
// the submitter thread of the last host batch has finished (called before the batch's buffers change)
int gvs_pipe_join(gvs_ctx* ctx);

static inline u64 next_pow2(u64 x) {
  u64 p = 1;
  while (p < x) p <<= 1;
  return p;
}
static inline u64 cdiv(u64 a, u64 b) { return (a + b - 1) / b; }

// -------------------------------------------------------------------------------------------
// hashing shared by table build and probe
// -------------------------------------------------------------------------------------------
#define GVS_EMPTY_KEY 0xFFFFFFFFFFFFFFFFull
#define GVS_ROW_MISSING 0xFFFFFFFFu  // db k-mer without a .loc row (reference: KeyError)
#define GVS_ROW_NOTINDB 0xFFFFFFFEu  // .loc k-mer that is not in the db set (never a hit)

__host__ __device__ __forceinline__ u64 gvs_mix(u64 x) {
  x *= 0x9E3779B97F4A7C15ull;
  x ^= x >> 32;
  x *= 0xD6E8FEB86659FD93ull;
  x ^= x >> 32;
  return x;
}
// filter: 32-bit hash of the canonical k-mer (two IMADs + two xorshift-multiply rounds); the word
// index is h & mask, the two bit positions inside the 32-bit word come from one more multiply
__host__ __device__ __forceinline__ u32 gvs_fhash(u64 key) {
  u32 lo = (u32)key, hi = (u32)(key >> 32);
  u32 h = (lo * 0x9E3779B1u) ^ (hi * 0x85EBCA77u + 0xC2B2AE3Du);
  h ^= h >> 15;
  h *= 0x2C1B3C6Du;
  h ^= h >> 12;
  return h;
}
// Blocked filter: a block is 4 x u32; a key sets bit (h >> 5i) & 31 of word i (h = gvs_fhash(key)).
// The block is selected by the canonical form of a sub-mer of length K-J+1 of the key; a key is
// inserted once per sub-mer offset (J times), so J consecutive read windows share one block.
#define GVS_FJ(K) ((K) >= 4 ? 4 : 1)
__host__ __device__ __forceinline__ u32 gvs_bhash(u64 sub) {
  u32 lo = (u32)sub, hi = (u32)(sub >> 32);
  u32 h = (lo * 0xCC9E2D51u) ^ (hi * 0x1B873593u + 0x7F4A7C15u);
  h ^= h >> 16;
  h *= 0x85EBCA6Bu;
  h ^= h >> 13;
  return h;
}
// Large databases (blocked filter beyond L2): word 3 of a block does not hold key bits but one fingerprint bit
// per sub-mer that selected the block (~2 distinct sub-mers per block), so that a window group whose sub-mer
// merely collided in the presence filter is dropped by ONE bit test on the block before any of its windows is
// extracted and hashed; the keys keep words 0..2.
__host__ __device__ __forceinline__ u32 gvs_fp_bit(u32 hb) { return (hb * 0x85EBCA6Bu) >> 27; }
// Presence filter in front of the blocked filter: one 32-bit word per sub-mer hash, 2 bits; answers "is
// this (K-J+1)-mer a sub-mer of any SUNK" from L2, so that only the window groups that pass (a few % for
// a 150 Mbp database, ~20 % for a whole genome whose 1.4e8 sub-mers saturate the 64 MiB that L2 can hold)
// go on to hash their windows and fetch their 16-byte block.
// (any number of words: multiply-shift range reduction of a re-mixed hash, so that the filter can be sized to what stays
// resident in L2 instead of to a power of two)
__host__ __device__ __forceinline__ u32 gvs_p1_word(u32 hb, u32 n_words) { return (u32)(((u64)(hb * 0x9E3779B1u) * n_words) >> 32); }
__host__ __device__ __forceinline__ u32 gvs_p1_bits(u32 hb) { return (1u << (hb & 31)) | (1u << ((hb >> 5) & 31)); }
// reverse complement of an L-mer in 2-bit big-endian packing
__host__ __device__ __forceinline__ u64 gvs_revcomp(u64 x, int L) {
  u64 y = ~x;
  y = ((y >> 2) & 0x3333333333333333ull) | ((y & 0x3333333333333333ull) << 2);
  y = ((y >> 4) & 0x0F0F0F0F0F0F0F0Full) | ((y & 0x0F0F0F0F0F0F0F0Full) << 4);
  y = ((y >> 8) & 0x00FF00FF00FF00FFull) | ((y & 0x00FF00FF00FF00FFull) << 8);
  y = ((y >> 16) & 0x0000FFFF0000FFFFull) | ((y & 0x0000FFFF0000FFFFull) << 16);
  y = (y >> 32) | (y << 32);
  return y >> (64 - 2 * L);
}
// table: bucket (4 slots = one 32-byte sector of keys) from bits 24.. of the hash
__host__ __device__ __forceinline__ u64 gvs_tab_bucket(u64 h, u64 tab_slots) { return (h >> 24) & ((tab_slots >> 2) - 1); }

// -------------------------------------------------------------------------------------------
// device-wide exclusive scan (3 launches: tile reduce, scan of tile sums, tile scan + write)
// The input is produced by a functor so that flag arrays never have to be materialised.
// -------------------------------------------------------------------------------------------
#define SCAN_THREADS 256
#define SCAN_ITEMS 8
#define SCAN_TILE (SCAN_THREADS * SCAN_ITEMS)

struct OpSum {
  template <typename T>
  __device__ __forceinline__ T operator()(T a, T b) const { return a + b; }
  template <typename T>
  __device__ __forceinline__ T identity() const { return (T)0; }
};
struct OpMax {
  template <typename T>
  __device__ __forceinline__ T operator()(T a, T b) const { return a > b ? a : b; }
  template <typename T>
  __device__ __forceinline__ T identity() const { return (T)0; }  // unsigned inputs only
};

template <typename T, typename Op>
__device__ __forceinline__ T warp_incl_scan(T v, Op op) {
  int lane = threadIdx.x & 31;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    T o = __shfl_up_sync(0xFFFFFFFFu, v, d);
    if (lane >= d) v = op(o, v);
  }
  return v;
}

// block-wide exclusive scan of one value per thread; returns exclusive prefix, *total = block sum
template <typename T, typename Op>
__device__ __forceinline__ T block_excl_scan(T v, Op op, T* total, T* smem /* >= 33 entries */) {
  int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
  T inc = warp_incl_scan(v, op);
  if (lane == 31) smem[wid] = inc;
  __syncthreads();
  if (wid == 0) {
    T w = (lane < nw) ? smem[lane] : op.template identity<T>();
    T winc = warp_incl_scan(w, op);
    smem[lane] = winc;  // inclusive per-warp sums
  }
  __syncthreads();
  T wprefix = (wid == 0) ? op.template identity<T>() : smem[wid - 1];
  T tot = smem[nw - 1];
  T excl_in_warp = __shfl_up_sync(0xFFFFFFFFu, inc, 1);
  if (lane == 0) excl_in_warp = op.template identity<T>();
  __syncthreads();
  if (total) *total = tot;
  return op(wprefix, excl_in_warp);
}

template <typename T, typename Op, typename F>
__global__ void __launch_bounds__(SCAN_THREADS) k_scan_reduce(F f, u64 n, T* tile_sums, Op op) {
  __shared__ T sm[33];
  u64 base = (u64)blockIdx.x * SCAN_TILE + (u64)threadIdx.x * SCAN_ITEMS;
  T acc = op.template identity<T>();
#pragma unroll
  for (int i = 0; i < SCAN_ITEMS; i++) {
    u64 j = base + i;
    if (j < n) acc = op(acc, f(j));
  }
  T tot;
  block_excl_scan(acc, op, &tot, sm);
  if (threadIdx.x == 0) tile_sums[blockIdx.x] = tot;
}

template <typename T, typename Op>
__global__ void __launch_bounds__(1024) k_scan_sums(T* tile_sums, u64 n_tiles, T* total_out, Op op) {
  __shared__ T sm[33];
  __shared__ T carry_s;
  if (threadIdx.x == 0) carry_s = op.template identity<T>();
  __syncthreads();
  for (u64 base = 0; base < n_tiles; base += 1024) {
    u64 j = base + threadIdx.x;
    T v = (j < n_tiles) ? tile_sums[j] : op.template identity<T>();
    T tot;
    T ex = block_excl_scan(v, op, &tot, sm);
    T carry = carry_s;
    if (j < n_tiles) tile_sums[j] = op(carry, ex);
    __syncthreads();
    if (threadIdx.x == 0) carry_s = op(carry, tot);
    __syncthreads();
  }
  if (threadIdx.x == 0 && total_out) *total_out = carry_s;
}

template <typename T, typename Op, typename F, typename G>
__global__ void __launch_bounds__(SCAN_THREADS) k_scan_apply(F f, G g, u64 n, const T* tile_sums, Op op) {
  __shared__ T sm[33];
  u64 base = (u64)blockIdx.x * SCAN_TILE + (u64)threadIdx.x * SCAN_ITEMS;
  T v[SCAN_ITEMS];
  T acc = op.template identity<T>();
#pragma unroll
  for (int i = 0; i < SCAN_ITEMS; i++) {
    u64 j = base + i;
    v[i] = (j < n) ? f(j) : op.template identity<T>();
    acc = op(acc, v[i]);
  }
  T ex = block_excl_scan(acc, op, (T*)nullptr, sm);
  T run = op(tile_sums[blockIdx.x], ex);
#pragma unroll
  for (int i = 0; i < SCAN_ITEMS; i++) {
    u64 j = base + i;
    if (j < n) g(j, run, v[i]);  // g(index, exclusive prefix, own value)
    run = op(run, v[i]);
  }
}

// exclusive scan: out via g(j, excl, v).  total_dev (may be null) receives the grand total.
template <typename T, typename Op, typename F, typename G>
static int device_scan(gvs_ctx* ctx, u64 n, F f, G g, Op op, T* total_dev) {
  u64 n_tiles = cdiv(n, SCAN_TILE);
  if (n_tiles == 0) n_tiles = 1;
  CKR(gvs_reserve(ctx, ctx->scan_tmp, n_tiles * sizeof(T)));
  T* sums = ctx->scan_tmp.as<T>();
  LAUNCH((k_scan_reduce<T, Op, F>), (unsigned)n_tiles, SCAN_THREADS, 0, f, n, sums, op);
  LAUNCH((k_scan_sums<T, Op>), 1, 1024, 0, sums, n_tiles, total_dev, op);
  LAUNCH((k_scan_apply<T, Op, F, G>), (unsigned)n_tiles, SCAN_THREADS, 0, f, g, n, sums, op);
  return 0;
}

// *err |= 4 unless groups 0..ng-1 are in strictly ascending (contig, start) order (covprob's lookup, support tracks)
static __global__ void __launch_bounds__(256) k_groups_sorted(const u32* __restrict__ g_contig, const u32* __restrict__ g_id, u64 ng, u32* err) {
  u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (i + 1 >= ng) return;
  u32 a = g_contig[i], b = g_contig[i + 1];
  if (a > b || (a == b && g_id[i] >= g_id[i + 1])) atomicOr(err, 4u);
}

// the validation's ratio test on two rows (pos, start): 9*|dstart| < 10*|dpos| < 11*|dstart|
// (process-by-contig_lowmem_AR.py:145-147, Q12); gap evidence and junctions anchor rows with it
__device__ __forceinline__ bool gvs_ratio_ok(u32 pi, u32 si, u32 pj, u32 sj) {
  const u64 ds = si > sj ? si - sj : sj - si;
  const u64 dp = pi > pj ? pi - pj : pj - pi;
  return 9 * ds < 10 * dp && 10 * dp < 11 * ds;
}

// small helpers to read device scalars (synchronises the stream)
template <typename T>
static int read_dev(gvs_ctx* ctx, const T* d, T* h, size_t n = 1) {
  if (ctx->mailbox && n * sizeof(T) <= 256) {  // page-locked landing zone: the copy is a plain DMA, no staging by the driver
    CK(cudaMemcpyAsync(ctx->mailbox, d, n * sizeof(T), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    memcpy(h, ctx->mailbox, n * sizeof(T));
    return 0;
  }
  CK(cudaMemcpyAsync(h, d, n * sizeof(T), cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return 0;
}

// Slots of the 64-word ctx->counters block (reserved in ctx.cu and table.cu): flags a kernel sets for the host, and
// totals the host reads later or several at once.  A total read back right after its scan goes through scan_total.
enum CounterSlot : u32 {
  CNT_HITS,         // match: hits                                   } cleared and read back together (match.cu)
  CNT_FLAGS,        // match: probe flags (key error, overflow)      }
  CNT_EMIT,         // match: (rows << 32) + suppressed hits         }
  CNT_HIT_MAX,      // match: most hits of one probe span            }
  CNT_SCAN,         // scan_total
  CNT_VOTE_BIG,     // diag: candidates left to the block-wide vote
  CNT_KEPT,         // diag: kept rows  } one read-back
  CNT_BEST,         // diag: best rows  }
  CNT_MISS,         // gvs_rows_set: rows whose (contig, group) is not in the database
  CNT_HIST_MAX,     // gvs_hist_mode: largest group count
  CNT_MODE,         // gvs_hist_mode: int64 mode per haplotype (two words)
  CNT_VAL_STATS = CNT_MODE + 2,  // gvs_validate: reads whose clean-up removed every edge
  CNT_COVPROB_ERR,  // gvs_covprob_gaps
  CNT_ORDER_ERR,    // gvs_check_group_order
  CNT_RUNS_ERR,     // gvs_rank_runs
  CNT_COUNT
};
static_assert(CNT_COUNT <= 64, "ctx->counters holds 64 words");
template <typename T = u32>
static inline T* counter(gvs_ctx* ctx, CounterSlot s) { return (T*)(ctx->counters.as<u64>() + s); }

// device_scan whose grand total the host needs at once: *total receives it (one read-back)
template <typename T, typename Op, typename F, typename G>
static int scan_total(gvs_ctx* ctx, u64 n, F f, G g, Op op, T* total) {
  T* d = counter<T>(ctx, CNT_SCAN);
  CKR((device_scan<T>(ctx, n, f, g, op, d)));
  return read_dev(ctx, d, total);
}

// the kept rows of a Rows cut into segments (one per read), as the per-read kernels see them
struct SegRows {
  const u32 *read, *pos, *contig, *start, *group, *gidx;
  const u32* seg_start;  // n_seg + 1
  u32 n_seg;
  const u8* bad;         // per group index (null: nothing is bad)
  __device__ __forceinline__ bool is_bad(u32 i) const { return bad && bad[gidx[i]]; }
};
static inline SegRows seg_rows(const gvs_ctx* ctx, const Rows& r, const DevBuf& seg_start, u64 n_seg) {
  return {r.read.as<u32>(), r.pos.as<u32>(), r.contig.as<u32>(), r.start.as<u32>(), r.group.as<u32>(), r.gidx.as<u32>(),
          seg_start.as<u32>(), (u32)n_seg, ctx->bad_ready ? ctx->bad_flag.as<u8>() : nullptr};
}

// read lengths: explicit (gvs_reads_meta, a batches run) or from the offsets of the batch, clamped to 32 bits
struct ReadLens {
  const u64* off;
  const u32* len;  // null: from off
  __device__ __forceinline__ u32 operator()(u32 rd) const {
    return len ? len[rd] : (u32)min(off[rd + 1] - off[rd], (u64)0xFFFFFFFFu);
  }
};
static inline ReadLens read_lens(const gvs_ctx* ctx) {
  return {ctx->read_off, ctx->have_read_len ? ctx->read_len.as<u32>() : nullptr};
}

static inline int rec_reserve(gvs_ctx* ctx, RecTable& t, u32 n_cols, u64 stride) {
  t.stride = stride;
  return gvs_reserve(ctx, t.buf, stride * n_cols * 4);
}
// a record getter: the first n entries of the table's columns to host buffers (null ones skipped); returns when the
// copies (and any queued before them) have finished
template <int N>
static int rec_get(gvs_ctx* ctx, const RecTable& t, const char* before, uint32_t* const (&dst)[N]) {
  if (!t.ready) return gvs_fail(ctx, GVS_E_STATE, "%s", before);
  CK(cudaSetDevice(ctx->device));
  if (t.n == 0) return 0;
  for (int c = 0; c < N; c++)
    if (dst[c]) CK(cudaMemcpyAsync(dst[c], t.col(c), t.n * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return 0;
}
template <typename T>
static int to_dev(gvs_ctx* ctx, DevBuf& b, const T* h, size_t n) {
  CKR(gvs_reserve(ctx, b, n * sizeof(T)));
  if (n) CK(cudaMemcpyAsync(b.p, h, n * sizeof(T), cudaMemcpyHostToDevice, ctx->stream));
  return 0;
}

// stage entry points implemented in the other translation units
int gvs_tab_build_impl(gvs_ctx* ctx, const u64* d_db_kmer, u64 n_db);  // table.cu
int gvs_tab_attach_gidx(gvs_ctx* ctx);                                 // table.cu (after loc_gidx exists)
int gvs_group_index_rows(gvs_ctx* ctx, const u32* contig, const u32* group, u64 n, u32* gidx_out);  // table.cu
int gvs_build_segments(gvs_ctx* ctx, const u32* read, u64 n, DevBuf& seg_start, DevBuf& row_seg, u64* n_seg_out);  // diag.cu
int gvs_reserve_rows(gvs_ctx* ctx, Rows& r, u64 n);
// support.cu: group ranks in (contig, start) order (rank_of / rank_grp unless rank_identity), cached per group table
int gvs_ensure_rank(gvs_ctx* ctx);
// support.cu: rank_identity of a freshly built group table (one launch; called by every table build, so that the
// rank of a sorted table costs the later stages nothing)
int gvs_check_group_order(gvs_ctx* ctx);
// support.cu: runs of equal values over the groups in rank order that tile [0, contig_len) of every contig: diff = nv
// difference arrays of n_groups int32 by rank, prefix-summed here; out receives 3 + nv columns: contig, start, end, values
int gvs_rank_runs(gvs_ctx* ctx, const i32* diff, u32 nv, const uint32_t* contig_len, RecTable& out, const char* who);
int grow_keep(gvs_ctx* ctx, DevBuf& b, size_t need, size_t keep);  // batches.cu: grow to `need` bytes keeping the first `keep`
