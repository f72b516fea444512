// validate.cu -- bad-SUNK histogram (workflow/scripts/badsunks_AR.py:20-103) and the per-read
// inter-SUNK distance validation (workflow/scripts/process-by-contig_lowmem_AR.py:50-207).
// SURVEY.md A.5, A.6 (steps 1-5), quirks Q12-Q14.
//
//   k_hist / k_cnt_hist / k_mode / k_bad_flag
//       rows per (contig, group); per haplotype the smallest mode m of the non-zero counts;
//       bad <=> count > m + 4*sqrt(m) or count < 2 (threshold passed in as an integer floor)
//   k_validate<BIG>
//       one thread block per read.  Rows minus bad groups, stable rank-sort by assembly start,
//       then every pair (i<j) is tested with the integer form of the reference's float64 ratio
//       test (0.9 < dpos/dstart < 1.1  <=>  9*ds < 10*dp < 11*ds, exact for 32-bit inputs),
//       orientation majority, "multipos" clean-up, union-find over group IDs in shared memory,
//       largest component (ties: the component holding the earliest vertex in graph-tool's
//       insertion order), output in vertex order.
#include "common.cuh"
#include <algorithm>

// ---------------------------------------------------------------------------------------------
// histogram / bad groups
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_hist(const u32* __restrict__ gidx, u64 n, i32* hist) {
  u64 j = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (j < n) atomicAdd(&hist[gidx[j]], 1);
}
__global__ void __launch_bounds__(256) k_hist_max(const i32* __restrict__ hist, u64 ng, u32* maxv) {
  u32 m = 0;
  for (u64 g = (u64)blockIdx.x * blockDim.x + threadIdx.x; g < ng; g += (u64)gridDim.x * blockDim.x) m = max(m, (u32)hist[g]);
  for (int d = 16; d; d >>= 1) m = max(m, __shfl_xor_sync(0xFFFFFFFFu, m, d));
  if ((threadIdx.x & 31) == 0 && m) atomicMax(maxv, m);
}
__global__ void __launch_bounds__(256) k_cnt_hist(const i32* __restrict__ hist, const u32* __restrict__ grp_contig,
                                                  const u8* __restrict__ contig_hap, u64 ng, u32 M, u32* cnt_hist) {
  // almost all groups share a handful of count values: privatise the low bins per block
  constexpr u32 LOW = 2048;
  __shared__ u32 s_low[2 * LOW];
  for (u32 i = threadIdx.x; i < 2 * LOW; i += blockDim.x) s_low[i] = 0;
  __syncthreads();
  for (u64 g = (u64)blockIdx.x * blockDim.x + threadIdx.x; g < ng; g += (u64)gridDim.x * blockDim.x) {
    u32 c = (u32)hist[g];
    if (!c) continue;
    u8 h = contig_hap[grp_contig[g]];
    if (h > 1) continue;
    if (c < LOW) atomicAdd(&s_low[h * LOW + c], 1u);
    else atomicAdd(&cnt_hist[(u64)h * (M + 1) + c], 1u);
  }
  __syncthreads();
  for (u32 i = threadIdx.x; i < 2 * LOW; i += blockDim.x) {
    u32 v = s_low[i];
    u32 h = i / LOW, c = i % LOW;
    if (v && c <= M) atomicAdd(&cnt_hist[(u64)h * (M + 1) + c], v);
  }
}
// pandas .mode()[0]: the smallest of the most frequent values
__global__ void __launch_bounds__(1024) k_mode(const u32* __restrict__ cnt_hist, u32 M, i64* mode) {
  __shared__ unsigned long long best;
  const u32* ch = cnt_hist + (u64)blockIdx.x * (M + 1);
  if (threadIdx.x == 0) best = 0;
  __syncthreads();
  unsigned long long loc = 0;
  for (u32 v = 1 + threadIdx.x; v <= M; v += blockDim.x) {
    u32 f = ch[v];
    if (f) {
      unsigned long long key = ((unsigned long long)f << 32) | (0xFFFFFFFFu - v);  // max freq, then min v
      if (key > loc) loc = key;
    }
  }
  atomicMax(&best, loc);
  __syncthreads();
  if (threadIdx.x == 0) mode[blockIdx.x] = best ? (i64)(0xFFFFFFFFu - (u32)best) : 0;
}
__global__ void __launch_bounds__(256) k_bad_flag(const i32* __restrict__ hist, const u32* __restrict__ grp_contig,
                                                  const u8* __restrict__ contig_hap, u64 ng, i64 lim0, i64 lim1, u8* bad) {
  u64 g = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= ng) return;
  i64 c = hist[g];
  u8 h = contig_hap[grp_contig[g]];
  bool b = false;
  if (c > 0 && h <= 1) b = c > (h ? lim1 : lim0) || c < 2;  // badsunks_AR.py:48
  else if (c > 0 && h <= 3) b = c > (h == 3 ? lim1 : lim0);  // contig of the other haplotype: only the upper limit (:51)
  bad[g] = b ? 1 : 0;
}

extern "C" int gvs_contigs_set(gvs_ctx* ctx, const uint8_t* contig_hap, const uint32_t* contig_hash, uint32_t n_contigs) {
  if (!ctx || !contig_hap) return GVS_E_ARG;
  CK(cudaSetDevice(ctx->device));
  if (ctx->n_contigs && n_contigs != ctx->n_contigs) return gvs_fail(ctx, GVS_E_ARG, "n_contigs mismatch (%u vs %u)", n_contigs, ctx->n_contigs);
  ctx->n_contigs = n_contigs;
  CKR(to_dev(ctx, ctx->contig_hap, contig_hap, n_contigs));
  if (contig_hash) CKR(to_dev(ctx, ctx->contig_hash, contig_hash, n_contigs));
  CK(cudaStreamSynchronize(ctx->stream));
  return 0;
}

extern "C" int gvs_group_hist(gvs_ctx* ctx, int accumulate, int32_t** hist_dev) {
  if (!ctx) return GVS_E_ARG;
  if (!ctx->diag_ready) return gvs_fail(ctx, GVS_E_STATE, "gvs_group_hist before gvs_diag_filter / gvs_rows_set(1)");
  if (!ctx->groups_ready) return gvs_fail(ctx, GVS_E_STATE, "gvs_group_hist: no group index");
  CK(cudaSetDevice(ctx->device));
  StageTimer tm(ctx, GVS_ST_HIST);
  u64 ng = ctx->n_groups;
  bool fresh = ctx->hist.cap < (ng ? ng : 1) * 4;
  CKR(gvs_reserve(ctx, ctx->hist, (ng ? ng : 1) * 4));
  if (!accumulate || fresh || !ctx->hist_ready) CK(cudaMemsetAsync(ctx->hist.p, 0, (ng ? ng : 1) * 4, ctx->stream));
  u64 n = ctx->kept.n;
  if (n) LAUNCH(k_hist, (unsigned)cdiv(n, 256), 256, 0, ctx->kept.gidx.as<u32>(), n, ctx->hist.as<i32>());
  ctx->hist_ready = true;
  ctx->bad_ready = false;
  if (hist_dev) *hist_dev = ctx->hist.as<i32>();
  return 0;
}

extern "C" int gvs_hist_mode(gvs_ctx* ctx, int64_t mode[2]) {
  if (!ctx || !mode) return GVS_E_ARG;
  if (!ctx->hist_ready) return gvs_fail(ctx, GVS_E_STATE, "gvs_hist_mode before gvs_group_hist");
  if (ctx->contig_hap.cap == 0) return gvs_fail(ctx, GVS_E_STATE, "gvs_hist_mode: contig haplotypes unknown (gvs_contigs_set)");
  CK(cudaSetDevice(ctx->device));
  StageTimer tm(ctx, GVS_ST_MODE);
  u64 ng = ctx->n_groups;
  mode[0] = mode[1] = 0;
  if (ng == 0) return 0;
  u32* mx = counter(ctx, CNT_HIST_MAX);
  CK(cudaMemsetAsync(mx, 0, 4, ctx->stream));
  u64 grid = cdiv(ng, 256);
  if (grid > (u64)ctx->n_sm * 8) grid = (u64)ctx->n_sm * 8;
  LAUNCH(k_hist_max, (unsigned)grid, 256, 0, ctx->hist.as<i32>(), ng, mx);
  u32 M = 0;
  CKR(read_dev(ctx, mx, &M));
  if (M == 0) return 0;
  if (M > (1u << 28)) return gvs_fail(ctx, GVS_E_OVERFLOW, "group hit count %u too large for the mode table", M);
  CKR(gvs_reserve(ctx, ctx->cnt_hist, 2ull * (M + 1) * 4 + 16));
  CK(cudaMemsetAsync(ctx->cnt_hist.p, 0, 2ull * (M + 1) * 4 + 16, ctx->stream));
  LAUNCH(k_cnt_hist, (unsigned)(cdiv(ng, 256) < (u64)ctx->n_sm * 4 ? cdiv(ng, 256) : (u64)ctx->n_sm * 4), 256, 0, ctx->hist.as<i32>(), ctx->grp_contig.as<u32>(), ctx->contig_hap.as<u8>(), ng,
         M, ctx->cnt_hist.as<u32>());
  i64* dm = counter<i64>(ctx, CNT_MODE);
  LAUNCH(k_mode, 2, 1024, 0, ctx->cnt_hist.as<u32>(), M, dm);
  i64 hm[2];
  CKR(read_dev(ctx, dm, hm, 2));
  mode[0] = hm[0];
  mode[1] = hm[1];
  return 0;
}

extern "C" int gvs_bad_groups(gvs_ctx* ctx, const int64_t limit_floor[2], uint64_t* n_bad) {
  if (!ctx || !limit_floor) return GVS_E_ARG;
  if (!ctx->hist_ready) return gvs_fail(ctx, GVS_E_STATE, "gvs_bad_groups before gvs_group_hist");
  CK(cudaSetDevice(ctx->device));
  StageTimer tm(ctx, GVS_ST_BAD);
  u64 ng = ctx->n_groups;
  CKR(gvs_reserve(ctx, ctx->bad_flag, ng ? ng : 1));
  CKR(gvs_reserve(ctx, ctx->bad_list, (ng ? ng : 1) * 4));
  ctx->n_bad = 0;
  if (ng) {
    LAUNCH(k_bad_flag, (unsigned)cdiv(ng, 256), 256, 0, ctx->hist.as<i32>(), ctx->grp_contig.as<u32>(), ctx->contig_hap.as<u8>(), ng,
           limit_floor[0], limit_floor[1], ctx->bad_flag.as<u8>());
    const u8* bf = ctx->bad_flag.as<u8>();
    u32* bl = ctx->bad_list.as<u32>();
    auto f = [bf] __device__(u64 g) -> u32 { return bf[g]; };
    auto g2 = [bl] __device__(u64 g, u32 ex, u32 v) { if (v) bl[ex] = (u32)g; };
    u32 nb = 0;
    CKR(scan_total(ctx, ng, f, g2, OpSum(), &nb));
    ctx->n_bad = nb;
  }
  ctx->bad_ready = true;
  if (n_bad) *n_bad = ctx->n_bad;
  return 0;
}

extern "C" int gvs_bad_get(gvs_ctx* ctx, uint32_t* group_index) {
  if (!ctx) return GVS_E_ARG;
  if (!ctx->bad_ready) return gvs_fail(ctx, GVS_E_STATE, "gvs_bad_get before gvs_bad_groups");
  CK(cudaSetDevice(ctx->device));
  if (ctx->n_bad && group_index) {
    CK(cudaMemcpyAsync(group_index, ctx->bad_list.p, ctx->n_bad * 4, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
  }
  return 0;
}


// groups named in a bad_sunks.txt (process-by-contig_lowmem_AR.py:66-72): keys = sorted (contig << 32 | group)
__global__ void __launch_bounds__(256) k_bad_from_keys(const u32* __restrict__ grp_contig, const u32* __restrict__ grp_start, u64 ng,
                                                       const u64* __restrict__ keys, u64 nk, u8* bad) {
  u64 g = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= ng) return;
  u64 key = ((u64)grp_contig[g] << 32) | grp_start[g];
  u64 lo = 0, hi = nk;
  while (lo < hi) {
    u64 mid = (lo + hi) >> 1;
    if (keys[mid] < key) lo = mid + 1; else hi = mid;
  }
  bad[g] = (lo < nk && keys[lo] == key) ? 1 : 0;
}

extern "C" int gvs_bad_set(gvs_ctx* ctx, const uint32_t* contig, const uint32_t* group, uint64_t n, uint64_t* n_bad) {
  if (!ctx || (n && (!contig || !group))) return GVS_E_ARG;
  if (!ctx->groups_ready) return gvs_fail(ctx, GVS_E_STATE, "gvs_bad_set: no group index (database or gvs_rows_set first)");
  CK(cudaSetDevice(ctx->device));
  u64 ng = ctx->n_groups;
  CKR(gvs_reserve(ctx, ctx->bad_flag, ng ? ng : 1));
  CKR(gvs_reserve(ctx, ctx->bad_list, (ng ? ng : 1) * 4));
  ctx->n_bad = 0;
  if (ng) {
    std::vector<u64> keys(n);
    for (u64 i = 0; i < n; i++) keys[i] = ((u64)contig[i] << 32) | group[i];
    std::sort(keys.begin(), keys.end());
    DevBuf dk;
    int rc = to_dev(ctx, dk, keys.data(), keys.size());
    if (!rc) {
      k_bad_from_keys<<<(unsigned)cdiv(ng, 256), 256, 0, ctx->stream>>>(ctx->grp_contig.as<u32>(), ctx->grp_start.as<u32>(), ng,
                                                                        dk.as<u64>(), n, ctx->bad_flag.as<u8>());
      ctx->launches++;
      const u8* bf = ctx->bad_flag.as<u8>();
      u32* bl = ctx->bad_list.as<u32>();
      auto f = [bf] __device__(u64 g) -> u32 { return bf[g]; };
      auto g2 = [bl] __device__(u64 g, u32 ex, u32 v) { if (v) bl[ex] = (u32)g; };
      u32 nb = 0;
      rc = scan_total(ctx, ng, f, g2, OpSum(), &nb);
      ctx->n_bad = nb;
    }
    cudaStreamSynchronize(ctx->stream);
    gvs_release(dk);
    if (rc) return rc;
  }
  ctx->bad_ready = true;
  if (n_bad) *n_bad = ctx->n_bad;
  return 0;
}

extern "C" int gvs_groups_get(gvs_ctx* ctx, uint32_t* contig, uint32_t* group, int32_t* hist) {
  if (!ctx) return GVS_E_ARG;
  if (!ctx->groups_ready) return gvs_fail(ctx, GVS_E_STATE, "gvs_groups_get: no group index");
  if (hist && !ctx->hist_ready) return gvs_fail(ctx, GVS_E_STATE, "gvs_groups_get: no histogram (gvs_group_hist)");
  CK(cudaSetDevice(ctx->device));
  u64 ng = ctx->n_groups;
  if (ng == 0) return 0;
  if (contig) CK(cudaMemcpyAsync(contig, ctx->grp_contig.p, ng * 4, cudaMemcpyDeviceToHost, ctx->stream));
  if (group) CK(cudaMemcpyAsync(group, ctx->grp_start.p, ng * 4, cudaMemcpyDeviceToHost, ctx->stream));
  if (hist) CK(cudaMemcpyAsync(hist, ctx->hist.p, ng * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return 0;
}

extern "C" int gvs_groups_count(gvs_ctx* ctx, uint64_t* n_groups) {
  if (!ctx || !n_groups) return GVS_E_ARG;
  if (!ctx->groups_ready) return gvs_fail(ctx, GVS_E_STATE, "gvs_groups_count: no group index");
  *n_groups = ctx->n_groups;
  return 0;
}
