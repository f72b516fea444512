// diag.cu -- best contig per read by diagonal band vote + row filter: the GPU replacement of
// diag_filter_v3 (workflow/src/diag_filter_v3.nim:18-229) and diag_filter_step2
// (workflow/src/diag_filter_step2.nim:13-66).  SURVEY.md A.4, quirks Q8-Q11.
//
// Flat decomposition over global scratch arrays (rows are ~1 per kb of read, so this stage moves
// ~1 % of the bytes of the probe kernel):
//   segments      consecutive rows of one read
//   k_row_first   first row of every distinct contig of a read (Table insertion order) + its hit count
//   candidates    first rows whose contig is in the read's haplotype .fai and has >= 2 hits
//   k_cand_gather (pos, start, group) of a candidate's rows, contiguous
//   k_cand_vote   both orientations: interpolated median, truncation toward zero, distinct groups
//                 with |n - median| < 2500
//   k_seg_best    argmax (good desc, hitlen asc); cross-contig ties are flagged ...
//   k_seg_tie     ... and resolved by replaying Nim's Table[string, _] slot order (murmur3 & mask,
//                 linear probing, growth at count*3 > cap*2, capacity sticky within a chunk)
//   k_keep_rows   rows on the best contig survive (all of them, Q11)
// Haplotype mode (gvs_diag_filter_haps): candidates on the contigs of both haplotypes, k_seg_best_haps keeps the best
// of each, k_seg_tie<true> replays the ties per (read, haplotype), k_seg_pick keeps the chunk's or the assigned
// haplotype's choice, and the records of the reads with a vote on either are written by one scan.
#include "common.cuh"

#define NOBEST 0xFFFFFFFFu
#define BANDWIDTH 2500

int gvs_build_segments(gvs_ctx* ctx, const u32* read, u64 n, DevBuf& seg_start, DevBuf& row_seg, u64* n_seg_out);

__global__ void __launch_bounds__(256) k_seg_fill(const u32* __restrict__ read, const u32* __restrict__ row_seg, u64 n,
                                                  u32* seg_start, u32 n_seg) {
  u64 j = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (j > n) return;
  if (j == n) { seg_start[n_seg] = (u32)n; return; }
  if (j == 0 || read[j] != read[j - 1]) seg_start[row_seg[j]] = (u32)j;
}

int gvs_build_segments(gvs_ctx* ctx, const u32* read, u64 n, DevBuf& seg_start, DevBuf& row_seg, u64* n_seg_out) {
  CKR(gvs_reserve(ctx, row_seg, n * 4));
  u32* rs = row_seg.as<u32>();
  auto f = [read] __device__(u64 j) -> u32 { return (j == 0 || read[j] != read[j - 1]) ? 1u : 0u; };
  auto g = [rs] __device__(u64 j, u32 ex, u32 v) { rs[j] = ex + v - 1; };
  u32 ns = 0;
  CKR(scan_total(ctx, n, f, g, OpSum(), &ns));
  CKR(gvs_reserve(ctx, seg_start, ((u64)ns + 1) * 4));
  LAUNCH(k_seg_fill, (unsigned)cdiv(n + 1, 256), 256, 0, read, rs, n, seg_start.as<u32>(), ns);
  *n_seg_out = ns;
  return 0;
}

__global__ void __launch_bounds__(256) k_seg_info(const u32* __restrict__ read, const u32* __restrict__ seg_start, u32 n_seg,
                                                  const u64* __restrict__ chunk_first, const u8* __restrict__ chunk_hap,
                                                  u32 n_chunks, u32* seg_chunk, u8* seg_hap, u32* seg_ndist) {
  u32 s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n_seg) return;
  u32 c = chunk_of_read(chunk_first, n_chunks, read[seg_start[s]]);
  seg_chunk[s] = c;
  seg_hap[s] = chunk_hap[c];
  seg_ndist[s] = 0;
}

// row_cnt[j] = number of rows of j's contig in j's read if j is the first such row, else 0
__global__ void __launch_bounds__(256) k_row_first(const u32* __restrict__ contig, const u32* __restrict__ row_seg,
                                                   const u32* __restrict__ seg_start, u64 n, u32* row_cnt, u32* seg_ndist) {
  u64 j = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n) return;
  u32 s = row_seg[j];
  u32 a = seg_start[s], b = seg_start[s + 1];
  u32 c = contig[j];
  // (a read's rows come in long runs of one contig: the row before almost always settles it)
  if ((u32)j > a && contig[j - 1] == c) { row_cnt[j] = 0; return; }
  for (u32 i = a; i + 1 < (u32)j; i++)
    if (contig[i] == c) { row_cnt[j] = 0; return; }
  u32 cnt = 1;
  for (u32 i = (u32)j + 1; i < b; i++) cnt += contig[i] == c;
  row_cnt[j] = cnt;
  atomicAdd(&seg_ndist[s], 1u);
}

// (pos, start, group) of the candidate's rows, in read order
__global__ void __launch_bounds__(256) k_cand_gather(const u32* __restrict__ cand_row, const u32* __restrict__ cand_voff,
                                                     u32 n_cand, const u32* __restrict__ contig, const u32* __restrict__ pos,
                                                     const u32* __restrict__ start, const u32* __restrict__ group,
                                                     const u32* __restrict__ row_seg, const u32* __restrict__ seg_start,
                                                     u32* v_pos, u32* v_start, u32* v_group) {
  u32 w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  int lane = threadIdx.x & 31;
  if (w >= n_cand) return;
  u32 j = cand_row[w];
  u32 b = seg_start[row_seg[j] + 1];
  u32 c = contig[j];
  u32 o = cand_voff[w];
  for (u32 base = j; base < b; base += 32) {
    u32 i = base + lane;
    bool m = i < b && contig[i] == c;
    u32 bal = __ballot_sync(0xFFFFFFFFu, m);
    if (m) {
      u32 d = o + __popc(bal & ((1u << lane) - 1));
      v_pos[d] = pos[i];
      v_start[d] = start[i];
      v_group[d] = group[i];
    }
    o += __popc(bal);
  }
}

// warp per candidate (<= VOTE_WARP_MAX rows): the diagonals of both orientations are staged in shared
// memory once, ranks / medians / band membership / distinct groups are computed for both in one sweep
#define VOTE_WARP_MAX 256
#define VOTE_WARPS 4
__global__ void __launch_bounds__(VOTE_WARPS * 32) k_cand_vote_warp(const u32* __restrict__ cand_row, const u32* __restrict__ cand_voff,
                                                                    u32 n_cand, const u32* __restrict__ row_cnt,
                                                                    const u32* __restrict__ v_pos, const u32* __restrict__ v_start,
                                                                    const u32* __restrict__ v_group, u32* cand_good, u8* cand_dir,
                                                                    u32* big_list, u32* n_big) {
  __shared__ i64 s_n0[VOTE_WARPS][VOTE_WARP_MAX], s_n1[VOTE_WARPS][VOTE_WARP_MAX];
  __shared__ u32 s_g[VOTE_WARPS][VOTE_WARP_MAX];
  __shared__ u8 s_f[VOTE_WARPS][VOTE_WARP_MAX];
  __shared__ i64 s_med[VOTE_WARPS][4];
  const int grp = threadIdx.x >> 5, tid = threadIdx.x & 31;
  const u32 ci = blockIdx.x * VOTE_WARPS + grp;
  if (ci >= n_cand) return;
  const u32 cnt = row_cnt[cand_row[ci]];
  if (cnt > VOTE_WARP_MAX) {  // k_cand_vote<1024> takes it
    if (tid == 0) big_list[atomicAdd(n_big, 1u)] = ci;
    return;
  }
  const u32 o = cand_voff[ci];
  i64 *n0 = s_n0[grp], *n1 = s_n1[grp];
  u32* sg = s_g[grp];
  u8* sf = s_f[grp];
  for (u32 i = tid; i < cnt; i += 32) {
    i64 st = v_start[o + i], ps = v_pos[o + i];
    n0[i] = st + ps;  // reverse strand: pos + start is constant along the diagonal (nim:84-86)
    n1[i] = st - ps;  // forward strand (nim:111-113)
    sg[i] = v_group[o + i];
  }
  if (tid < 4) s_med[grp][tid] = 0;
  __syncwarp();
  const u32 lo = (cnt - 1) >> 1;
  // A read that follows one strand of its contig has one diagonal sorted along its rows (pos + start for a forward
  // read, start - pos for a reverse one) and its group ids strictly monotone: the sorted diagonal's median elements are
  // read off by index, and only the other one (the jittery true diagonal) needs rank counting.
  bool up0 = true, dn0 = true, up1 = true, dn1 = true, gup = true, gdn = true;
  for (u32 i = tid; i + 1 < cnt; i += 32) {
    const i64 x0 = n0[i], y0 = n0[i + 1], x1 = n1[i], y1 = n1[i + 1];
    const u32 g0 = sg[i], g1 = sg[i + 1];
    up0 &= x0 <= y0; dn0 &= x0 >= y0;
    up1 &= x1 <= y1; dn1 &= x1 >= y1;
    gup &= g0 < g1; gdn &= g0 > g1;
  }
  up0 = __all_sync(0xFFFFFFFFu, up0); dn0 = __all_sync(0xFFFFFFFFu, dn0);
  up1 = __all_sync(0xFFFFFFFFu, up1); dn1 = __all_sync(0xFFFFFFFFu, dn1);
  const bool groups_distinct = __all_sync(0xFFFFFFFFu, gup) || __all_sync(0xFFFFFFFFu, gdn);
  const bool sorted0 = up0 || dn0, sorted1 = up1 || dn1;
  if (tid == 0) {
    const u32 hi = lo + 1 < cnt ? lo + 1 : lo;  // (rank lo + 1 exists whenever it is used: even cnt)
    if (sorted0) { s_med[grp][0] = up0 ? n0[lo] : n0[cnt - 1 - lo]; s_med[grp][1] = up0 ? n0[hi] : n0[cnt - 1 - hi]; }
    if (sorted1) { s_med[grp][2] = up1 ? n1[lo] : n1[cnt - 1 - lo]; s_med[grp][3] = up1 ? n1[hi] : n1[cnt - 1 - hi]; }
  }
  // Unsorted diagonal of a larger candidate: elements of rank lo and lo + 1 by bisection on the value (one counting pass
  // per bit of the diagonal's spread) instead of ranking every row against every other
  auto select2 = [&](const i64* x, i64* out) {
    i64 mn = 0x7FFFFFFFFFFFFFFFll, mx = -0x7FFFFFFFFFFFFFFFll - 1;
    for (u32 i = tid; i < cnt; i += 32) {
      const i64 v = x[i];
      mn = v < mn ? v : mn;
      mx = v > mx ? v : mx;
    }
#pragma unroll
    for (int d = 16; d; d >>= 1) {
      const i64 a = __shfl_xor_sync(0xFFFFFFFFu, mn, d), b = __shfl_xor_sync(0xFFFFFFFFu, mx, d);
      mn = a < mn ? a : mn;
      mx = b > mx ? b : mx;
    }
    auto count_le = [&](i64 v) -> u32 {
      u32 c = 0;
      for (u32 i = tid; i < cnt; i += 32) c += x[i] <= v;
      return __reduce_add_sync(0xFFFFFFFFu, c);
    };
    i64 vlo = mn, vhi = mx;
    while (vlo < vhi) {  // warp-uniform
      const i64 mid = vlo + (i64)(((u64)vhi - (u64)vlo) >> 1);
      if (count_le(mid) >= lo + 1) vhi = mid; else vlo = mid + 1;
    }
    i64 nxt = vlo;
    if (count_le(vlo) < lo + 2) {  // rank lo + 1 is the smallest larger value
      i64 best = 0x7FFFFFFFFFFFFFFFll;
      for (u32 i = tid; i < cnt; i += 32) {
        const i64 v = x[i];
        if (v > vlo && v < best) best = v;
      }
#pragma unroll
      for (int d = 16; d; d >>= 1) {
        const i64 a = __shfl_xor_sync(0xFFFFFFFFu, best, d);
        best = a < best ? a : best;
      }
      nxt = best;
    }
    if (tid == 0) { out[0] = vlo; out[1] = nxt; }
  };
  const bool bisect = cnt > 48;
  if (bisect) {
    if (!sorted0) select2(n0, &s_med[grp][0]);
    if (!sorted1) select2(n1, &s_med[grp][2]);
  } else if (!sorted0 || !sorted1) {
    for (u32 i = tid; i < cnt; i += 32) {
      const i64 a0 = n0[i], a1 = n1[i];
      u32 r0 = 0, r1 = 0;
      if (!sorted0 && !sorted1) {
        for (u32 j = 0; j < cnt; j++) {
          const i64 b0 = n0[j], b1 = n1[j];
          const bool before = j < i;
          r0 += (b0 < a0) || (b0 == a0 && before);
          r1 += (b1 < a1) || (b1 == a1 && before);
        }
      } else if (!sorted0) {
        for (u32 j = 0; j < cnt; j++) {
          const i64 b0 = n0[j];
          r0 += (b0 < a0) || (b0 == a0 && j < i);
        }
      } else {
        for (u32 j = 0; j < cnt; j++) {
          const i64 b1 = n1[j];
          r1 += (b1 < a1) || (b1 == a1 && j < i);
        }
      }
      if (!sorted0 && r0 == lo) s_med[grp][0] = a0;
      if (!sorted0 && r0 == lo + 1) s_med[grp][1] = a0;
      if (!sorted1 && r1 == lo) s_med[grp][2] = a1;
      if (!sorted1 && r1 == lo + 1) s_med[grp][3] = a1;
    }
  }
  __syncwarp();
  i64 med[2];
#pragma unroll
  for (int orient = 0; orient < 2; orient++) {
    // arraymancer percentile(n, 50): linear interpolation in float64, then int() truncation toward
    // zero (diag_filter_v3.nim:86,113; Q8)
    i64 alo = s_med[grp][2 * orient], m = alo;
    if (!(cnt & 1)) {
      i64 d = s_med[grp][2 * orient + 1] - alo;  // >= 0
      m = alo + (d >> 1);
      if ((d & 1) && m < 0) m += 1;  // x.5 below zero truncates up
    }
    med[orient] = m;
  }
  for (u32 i = tid; i < cnt; i += 32) {
    i64 d0 = n0[i] - med[0], d1 = n1[i] - med[1];
    if (d0 < 0) d0 = -d0;
    if (d1 < 0) d1 = -d1;
    sf[i] = (u8)((d0 < BANDWIDTH ? 1 : 0) | (d1 < BANDWIDTH ? 2 : 0));
  }
  __syncwarp();
  u32 good0 = 0, good1 = 0;
  for (u32 i = tid; i < cnt; i += 32) {
    const u32 f = sf[i];
    if (!f) continue;
    u32 seen = 0;  // orientations in which an earlier in-band row already carries this group
    if (!groups_distinct) {
      const u32 gi = sg[i];
      for (u32 j = 0; j < i; j++)
        if (sg[j] == gi) seen |= sf[j];
    }
    good0 += (f & ~seen) & 1u;
    good1 += ((f & ~seen) >> 1) & 1u;
  }
#pragma unroll
  for (int d = 16; d; d >>= 1) {
    good0 += __shfl_xor_sync(0xFFFFFFFFu, good0, d);
    good1 += __shfl_xor_sync(0xFFFFFFFFu, good1, d);
  }
  if (tid == 0) {
    // reverse is tried first; forward replaces it only on a strictly larger count (nim:98-138)
    const bool fwd = good1 > good0;
    cand_good[ci] = fwd ? good1 : good0;
    cand_dir[ci] = fwd ? 1 : 0;
  }
}

// one thread group (NT threads) per candidate; NT = 32 (a warp, 4 per block) or 1024 (a block)
// one block per LARGE candidate (> VOTE_WARP_MAX rows), taken from the list the warp kernel left behind
template <int NT>
__global__ void __launch_bounds__(NT) k_cand_vote(const u32* __restrict__ cand_row, const u32* __restrict__ cand_voff,
                                                  const u32* __restrict__ big_list, const u32* __restrict__ n_big,
                                                  const u32* __restrict__ row_cnt, const u32* __restrict__ v_pos,
                                                  const u32* __restrict__ v_start, const u32* __restrict__ v_group,
                                                  u32* cand_good, u8* cand_dir) {
  __shared__ i64 s_alo, s_ahi;
  __shared__ u32 s_good;
  const int tid = threadIdx.x;
  const u32 nbig = *n_big;
  for (u32 q = blockIdx.x; q < nbig; q += gridDim.x) {
    const u32 ci = big_list[q];
    const u32 cnt = row_cnt[cand_row[ci]];
    const u32 o = cand_voff[ci];
    u32 good2[2] = {0, 0};
    // strictly monotone group ids are all distinct: the duplicate scan of the band count is not needed then
    bool gup = true, gdn = true;
    for (u32 i = tid; i + 1 < cnt; i += NT) {
      const u32 g0 = v_group[o + i], g1 = v_group[o + i + 1];
      gup &= g0 < g1;
      gdn &= g0 > g1;
    }
    const bool groups_distinct = __syncthreads_and(gup) || __syncthreads_and(gdn);
    for (int orient = 0; orient < 2; orient++) {  // 0: reverse (pos + start), 1: forward (start - pos)
      if (tid == 0) { s_alo = 0; s_ahi = 0; s_good = 0; }
      __syncthreads();
      const u32 lo = (cnt - 1) >> 1;
      auto val = [&](u32 i) -> i64 {
        return orient == 0 ? (i64)v_start[o + i] + (i64)v_pos[o + i] : (i64)v_start[o + i] - (i64)v_pos[o + i];
      };
      // a diagonal that is sorted along the rows (the one across the read's strand) gives its median elements by index
      bool up = true, dn = true;
      for (u32 i = tid; i + 1 < cnt; i += NT) {
        const i64 x = val(i), y = val(i + 1);
        up &= x <= y;
        dn &= x >= y;
      }
      const bool is_up = __syncthreads_and(up), is_dn = __syncthreads_and(dn);
      if (is_up || is_dn) {
        if (tid == 0) {
          const u32 hi = lo + 1 < cnt ? lo + 1 : lo;
          s_alo = is_up ? val(lo) : val(cnt - 1 - lo);
          s_ahi = is_up ? val(hi) : val(cnt - 1 - hi);
        }
      } else {
        // Elements of rank lo and lo + 1 by bisection on the value (~30 counting passes over the candidate's rows)
        // instead of ranking every row against every other: these candidates have hundreds to thousands of rows.
        i64 mn = 0x7FFFFFFFFFFFFFFFll, mx = -0x7FFFFFFFFFFFFFFFll - 1;
        for (u32 i = tid; i < cnt; i += NT) {
          const i64 v = val(i);
          mn = v < mn ? v : mn;
          mx = v > mx ? v : mx;
        }
        if (tid == 0) { s_alo = 0x7FFFFFFFFFFFFFFFll; s_ahi = -0x7FFFFFFFFFFFFFFFll - 1; }
        __syncthreads();
        atomicMin((long long*)&s_alo, (long long)mn);
        atomicMax((long long*)&s_ahi, (long long)mx);
        __syncthreads();
        i64 vlo = s_alo, vhi = s_ahi;  // the value of rank lo lies in [vlo, vhi]
        __syncthreads();
        auto count_le = [&](i64 x) -> u32 {  // rows with value <= x (block-uniform result)
          u32 c = 0;
          for (u32 base = 0; base < cnt; base += NT) {
            const u32 i = base + tid;
            c += (u32)__syncthreads_count(i < cnt && val(i) <= x);
          }
          return c;
        };
        while (vlo < vhi) {
          const i64 mid = vlo + (i64)(((u64)vhi - (u64)vlo) >> 1);
          if (count_le(mid) >= lo + 1) vhi = mid; else vlo = mid + 1;
        }
        // rank lo + 1: the same value if it occurs often enough, else the smallest larger one
        i64 nxt = vlo;
        if (count_le(vlo) < lo + 2) {
          i64 best = 0x7FFFFFFFFFFFFFFFll;
          for (u32 i = tid; i < cnt; i += NT) {
            const i64 v = val(i);
            if (v > vlo && v < best) best = v;
          }
          if (tid == 0) s_ahi = 0x7FFFFFFFFFFFFFFFll;
          __syncthreads();
          atomicMin((long long*)&s_ahi, (long long)best);
          __syncthreads();
          nxt = s_ahi;  // (only used when cnt is even, i.e. when rank lo + 1 exists)
          __syncthreads();
        }
        if (tid == 0) { s_alo = vlo; s_ahi = nxt; }
      }
      __syncthreads();
      // arraymancer percentile(n, 50): linear interpolation in float64, then int() truncation
      // toward zero (diag_filter_v3.nim:86,113; Q8)
      i64 alo = s_alo, med = alo;
      if (!(cnt & 1)) {
        i64 d = s_ahi - alo;  // >= 0
        med = alo + (d >> 1);
        if ((d & 1) && med < 0) med += 1;  // x.5 below zero truncates up
      }
      for (u32 i = tid; i < cnt; i += NT) {
        i64 ni = orient == 0 ? (i64)v_start[o + i] + (i64)v_pos[o + i] : (i64)v_start[o + i] - (i64)v_pos[o + i];
        i64 dv = ni - med;
        if (dv < 0) dv = -dv;
        if (dv >= BANDWIDTH) continue;
        u32 gi = v_group[o + i];
        bool dup = false;
        for (u32 j = 0; j < i && !dup && !groups_distinct; j++) {
          if (v_group[o + j] != gi) continue;
          i64 nj = orient == 0 ? (i64)v_start[o + j] + (i64)v_pos[o + j] : (i64)v_start[o + j] - (i64)v_pos[o + j];
          i64 dj = nj - med;
          if (dj < 0) dj = -dj;
          dup = dj < BANDWIDTH;
        }
        if (!dup) atomicAdd(&s_good, 1u);
      }
      __syncthreads();
      good2[orient] = s_good;
      __syncthreads();
    }
    if (tid == 0) {
      // reverse is tried first; forward replaces it only on a strictly larger count (nim:98-138)
      bool fwd = good2[1] > good2[0];
      cand_good[ci] = fwd ? good2[1] : good2[0];
      cand_dir[ci] = fwd ? 1 : 0;
    }
  }
}

// smallest power-of-two capacity >= 64 that holds n distinct keys without growing
// (tables.nim mustRehash: cap*2 < count*3 checked before each insert, count = keys so far)
__host__ __device__ __forceinline__ u32 cap_needed(u32 n) {
  u32 cap = 64;
  while (n > 0 && (u64)cap * 2 < (u64)(n - 1) * 3) cap <<= 1;
  return cap;
}

__global__ void __launch_bounds__(256) k_seg_best(u32 n_seg, const u32* __restrict__ seg_start,
                                                  const u32* __restrict__ cidx_excl, const u32* __restrict__ cand_row,
                                                  const u32* __restrict__ row_cnt, const u32* __restrict__ contig,
                                                  const u32* __restrict__ cand_good, const u8* __restrict__ cand_dir,
                                                  u32* seg_best, u32* seg_good, u8* seg_dir, u8* seg_tie) {
  u32 s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n_seg) return;
  u32 c0 = cidx_excl[seg_start[s]], c1 = cidx_excl[seg_start[s + 1]];
  u32 maxgood = 0, maxhit = 0, best = NOBEST, ties = 0;
  u8 dir = 0;
  for (u32 ci = c0; ci < c1; ci++) {
    u32 g = cand_good[ci], h = row_cnt[cand_row[ci]];
    if (g > maxgood || (g == maxgood && g > 0 && h < maxhit)) {
      maxgood = g; maxhit = h; best = contig[cand_row[ci]]; dir = cand_dir[ci]; ties = 1;
    } else if (g == maxgood && g > 0 && h == maxhit) {
      ties++;
    }
  }
  bool ok = maxgood > 1;  // `if maxgood>1: echo ...` (nim:141)
  seg_best[s] = ok ? best : NOBEST;
  seg_good[s] = maxgood;
  seg_dir[s] = dir;
  seg_tie[s] = (ok && ties > 1) ? 1 : 0;
}

// replay Nim's Table for the reads whose optimum is shared by several contigs.  HAPS: a tie entry is 2 * segment +
// haplotype, only that haplotype's candidates compete, and best / dir are written per entry
template <bool HAPS>
__global__ void __launch_bounds__(64) k_seg_tie(const u32* __restrict__ tie_seg, u32 n_tie, const u32* __restrict__ seg_start,
                                                const u32* __restrict__ seg_cap, const u32* __restrict__ cidx_excl,
                                                const u32* __restrict__ cand_row, const u32* __restrict__ row_cnt,
                                                const u32* __restrict__ contig, const u32* __restrict__ contig_hash,
                                                const u32* __restrict__ cand_good, const u8* __restrict__ cand_dir,
                                                const u8* __restrict__ contig_hap, u32* scratch, u32 maxcap, u32* seg_best,
                                                u8* seg_dir) {
  u32 t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_tie) return;
  const u32 e = tie_seg[t];
  const u32 s = HAPS ? e >> 1 : e;
  auto mine = [&](u32 ci) { return !HAPS || contig_hap[contig[cand_row[ci]]] == (e & 1); };
  u32 a = seg_start[s], b = seg_start[s + 1];
  u32* A = scratch + (u64)t * 2 * maxcap;
  u32* B = A + maxcap;
  u32 cap = seg_cap[s], count = 0;
  for (u32 i = 0; i < cap; i++) A[i] = NOBEST;
  for (u32 j = a; j < b; j++) {
    if (row_cnt[j] == 0) continue;  // not the first row of its contig
    u32 c = contig[j];
    if ((u64)cap * 2 < (u64)count * 3 || cap - count < 4) {  // enlarge: re-insert in old slot order
      u32 ncap = cap * 2;
      for (u32 i = 0; i < ncap; i++) B[i] = NOBEST;
      for (u32 i = 0; i < cap; i++) {
        u32 x = A[i];
        if (x == NOBEST) continue;
        u32 h = contig_hash[x] & (ncap - 1);
        while (B[h] != NOBEST) h = (h + 1) & (ncap - 1);
        B[h] = x;
      }
      u32* tmp = A; A = B; B = tmp;
      cap = ncap;
    }
    u32 h = contig_hash[c] & (cap - 1);
    while (A[h] != NOBEST) h = (h + 1) & (cap - 1);
    A[h] = c;
    count++;
  }
  // optimum of this read
  u32 c0 = cidx_excl[a], c1 = cidx_excl[b];
  u32 maxgood = 0, maxhit = 0;
  for (u32 ci = c0; ci < c1; ci++) {
    if (!mine(ci)) continue;
    u32 g = cand_good[ci], h = row_cnt[cand_row[ci]];
    if (g > maxgood || (g == maxgood && h < maxhit)) { maxgood = g; maxhit = h; }
  }
  for (u32 i = 0; i < cap; i++) {  // `for k,v in posStarts.pairs()`: slot order
    u32 x = A[i];
    if (x == NOBEST) continue;
    for (u32 ci = c0; ci < c1; ci++) {
      if (contig[cand_row[ci]] == x && cand_good[ci] == maxgood && row_cnt[cand_row[ci]] == maxhit && mine(ci)) {
        seg_best[e] = x;
        seg_dir[e] = cand_dir[ci];
        return;
      }
    }
  }
}

// haplotype mode: k_seg_best with one accumulator per haplotype, results at 2 * segment + haplotype
__global__ void __launch_bounds__(256) k_seg_best_haps(u32 n_seg, const u32* __restrict__ seg_start,
                                                       const u32* __restrict__ cidx_excl, const u32* __restrict__ cand_row,
                                                       const u32* __restrict__ row_cnt, const u32* __restrict__ contig,
                                                       const u8* __restrict__ contig_hap, const u32* __restrict__ cand_good,
                                                       const u8* __restrict__ cand_dir, u32* hap_best, u32* hap_good,
                                                       u8* hap_dir, u8* hap_tie) {
  u32 s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n_seg) return;
  struct Acc {
    u32 maxgood = 0, maxhit = 0, best = NOBEST, ties = 0;
    u8 dir = 0;
  } acc[2];
  auto upd = [](Acc& a, u32 g, u32 h, u32 c, u8 d) {
    if (g > a.maxgood || (g == a.maxgood && g > 0 && h < a.maxhit)) {
      a.maxgood = g; a.maxhit = h; a.best = c; a.dir = d; a.ties = 1;
    } else if (g == a.maxgood && g > 0 && h == a.maxhit) {
      a.ties++;
    }
  };
  u32 c0 = cidx_excl[seg_start[s]], c1 = cidx_excl[seg_start[s + 1]];
  for (u32 ci = c0; ci < c1; ci++) {
    const u32 c = contig[cand_row[ci]], g = cand_good[ci], h = row_cnt[cand_row[ci]];
    if (contig_hap[c]) upd(acc[1], g, h, c, cand_dir[ci]);
    else upd(acc[0], g, h, c, cand_dir[ci]);
  }
#pragma unroll
  for (int k = 0; k < 2; k++) {
    const bool ok = acc[k].maxgood > 1;
    hap_best[2 * s + k] = ok ? acc[k].best : NOBEST;
    hap_good[2 * s + k] = ok ? acc[k].maxgood : 0;
    hap_dir[2 * s + k] = acc[k].dir;
    hap_tie[2 * s + k] = (ok && acc[k].ties > 1) ? 1 : 0;
  }
}

// assignment of a read from its two votes (n = 0 without a vote): 0 / 1, 2 = tie, 3 = none
__device__ __forceinline__ u32 hap_assign(u32 n0, u32 n1) { return n0 > n1 ? 0u : n1 > n0 ? 1u : n0 ? 2u : 3u; }

// the kept haplotype's choice becomes the segment's: the chunk's haplotype, or the assigned one of an unbinned read
__global__ void __launch_bounds__(256) k_seg_pick(u32 n_seg, const u8* __restrict__ seg_hap, const u32* __restrict__ hap_best,
                                                  const u32* __restrict__ hap_good, const u8* __restrict__ hap_dir,
                                                  u32* seg_best, u32* seg_good, u8* seg_dir) {
  u32 s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n_seg) return;
  const u32 sh = seg_hap[s];
  const u32 k = sh < GVS_HAP_ANY ? sh : hap_assign(hap_good[2 * s], hap_good[2 * s + 1]);
  seg_best[s] = k < 2 ? hap_best[2 * s + k] : NOBEST;
  seg_good[s] = k < 2 ? hap_good[2 * s + k] : 0;
  seg_dir[s] = k < 2 ? hap_dir[2 * s + k] : 0;
}

__global__ void __launch_bounds__(256) k_keep_rows(u64 n, const u32* __restrict__ keep_excl, const u32* __restrict__ row_seg,
                                                   const u32* __restrict__ seg_best, const u32* __restrict__ read,
                                                   const u32* __restrict__ pos, const u32* __restrict__ contig,
                                                   const u32* __restrict__ start, const u32* __restrict__ group,
                                                   const u32* __restrict__ gidx, u32* o_read, u32* o_pos, u32* o_contig,
                                                   u32* o_start, u32* o_group, u32* o_gidx) {
  u64 j = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n) return;
  u32 c = contig[j];
  if (seg_best[row_seg[j]] != c) return;
  u32 o = keep_excl[j];
  o_read[o] = read[j];
  o_pos[o] = pos[j];
  o_contig[o] = c;
  o_start[o] = start[j];
  o_group[o] = group[j];
  o_gidx[o] = gidx[j];
}

__global__ void __launch_bounds__(256) k_best_rows(u32 n_seg, const u32* __restrict__ best_excl,
                                                   const u32* __restrict__ seg_best, const u32* __restrict__ seg_good,
                                                   const u8* __restrict__ seg_dir, const u32* __restrict__ seg_start,
                                                   const u32* __restrict__ read, u32* o_read, u32* o_contig, u32* o_good,
                                                   u8* o_dir) {
  u32 s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n_seg || seg_best[s] == NOBEST) return;
  u32 o = best_excl[s];
  o_read[o] = read[seg_start[s]];
  o_contig[o] = seg_best[s];
  o_good[o] = seg_good[s];
  o_dir[o] = seg_dir[s];
}


// scratch layout inside ctx->diag_scratch (u32 units)
struct DiagScratch {
  u32 *row_seg, *row_cnt, *cidx, *keep_excl, *cand_row, *cand_voff, *v_pos, *v_start, *v_group, *cand_good;
  u32 *seg_chunk, *seg_ndist, *seg_cap, *seg_best, *seg_good, *best_excl, *tie_seg;
  u8 *seg_hap, *seg_dir, *seg_tie, *cand_dir;
};

static int diag_impl(gvs_ctx* ctx, bool haps, u64* n_best_out, u64* n_kept_out) {
  Rows& R = ctx->rows;
  u64 n = R.n;
  ctx->kept.n = 0;
  ctx->n_best = 0;
  ctx->n_seg = 0;
  ctx->rh.n = 0;
  ctx->rh.ready = haps;
  if (n == 0) return 0;
  StageTimer tm(ctx, GVS_ST_DIAG);
  const u32 *read = R.read.as<u32>(), *pos = R.pos.as<u32>(), *contig = R.contig.as<u32>(), *start = R.start.as<u32>(),
            *group = R.group.as<u32>(), *gidx = R.gidx.as<u32>();
  u64 n_seg = 0;
  CKR(gvs_build_segments(ctx, read, n, ctx->seg_start, ctx->flags_c, &n_seg));
  ctx->n_seg = n_seg;
  const u32* row_seg = ctx->flags_c.as<u32>();
  const u32* seg_start = ctx->seg_start.as<u32>();
  // carve scratch
  u64 words = n * 9 + (n_seg + 1) * 8 + 64;
  CKR(gvs_reserve(ctx, ctx->diag_scratch, words * 4 + n * 2 + (n_seg + 1) * 4));
  u32* w = ctx->diag_scratch.as<u32>();
  DiagScratch D;
  D.row_cnt = w; w += n;
  D.cidx = w; w += n + 1;
  D.keep_excl = w; w += n;
  D.cand_row = w; w += n;
  D.cand_voff = w; w += n;
  D.v_pos = w; w += n;
  D.v_start = w; w += n;
  D.v_group = w; w += n;
  D.cand_good = w; w += n;
  D.seg_chunk = w; w += n_seg;
  D.seg_ndist = w; w += n_seg;
  D.seg_cap = w; w += n_seg;
  D.seg_best = w; w += n_seg;
  D.seg_good = w; w += n_seg;
  D.best_excl = w; w += n_seg + 1;
  D.tie_seg = w; w += n_seg;
  u8* bb = (u8*)(ctx->diag_scratch.as<u32>() + words);
  D.cand_dir = bb; bb += n;
  D.seg_hap = bb; bb += n_seg;
  D.seg_dir = bb; bb += n_seg;
  D.seg_tie = bb; bb += n_seg;

  LAUNCH(k_seg_info, (unsigned)cdiv(n_seg, 256), 256, 0, read, seg_start, (u32)n_seg, ctx->chunk_first.as<u64>(),
         ctx->chunk_hap.as<u8>(), ctx->n_chunks, D.seg_chunk, D.seg_hap, D.seg_ndist);
  LAUNCH(k_row_first, (unsigned)cdiv(n, 256), 256, 0, contig, row_seg, seg_start, n, D.row_cnt, D.seg_ndist);
  // candidates: first rows whose contig is in the read's haplotype and has >= 2 hits (nim:82,147)
  const u8* contig_hap = ctx->contig_hap.as<u8>();
  u64 packed = 0;
  {
    const u32* rc = D.row_cnt;
    const u8* sh = D.seg_hap;
    u32 *cidx = D.cidx, *crow = D.cand_row, *cvoff = D.cand_voff;
    auto g = [cidx, crow, cvoff] __device__(u64 j, u64 ex, u64 v) {
      cidx[j] = (u32)(ex >> 32);
      if (v) {
        crow[ex >> 32] = (u32)j;
        cvoff[ex >> 32] = (u32)ex;
      }
    };
    if (haps) {  // the contigs of either haplotype
      auto f = [rc, contig, contig_hap] __device__(u64 j) -> u64 {
        u32 c = rc[j];
        return (c >= 2 && contig_hap[contig[j]] <= 1) ? ((1ull << 32) | c) : 0ull;
      };
      CKR(scan_total(ctx, n, f, g, OpSum(), &packed));
    } else {
      auto f = [rc, contig, contig_hap, sh, row_seg] __device__(u64 j) -> u64 {
        u32 c = rc[j];
        return (c >= 2 && contig_hap[contig[j]] == sh[row_seg[j]]) ? ((1ull << 32) | c) : 0ull;
      };
      CKR(scan_total(ctx, n, f, g, OpSum(), &packed));
    }
  }
  u32 n_cand = (u32)(packed >> 32);
  CK(cudaMemcpyAsync(D.cidx + n, &n_cand, 4, cudaMemcpyHostToDevice, ctx->stream));
  if (n_cand) {
    LAUNCH(k_cand_gather, (unsigned)cdiv((u64)n_cand * 32, 256), 256, 0, D.cand_row, D.cand_voff, n_cand, contig, pos, start,
           group, row_seg, seg_start, D.v_pos, D.v_start, D.v_group);
    u32* n_big = counter(ctx, CNT_VOTE_BIG);
    CK(cudaMemsetAsync(n_big, 0, 4, ctx->stream));
    u32* big_list = D.keep_excl;  // free until the keep scan below
    LAUNCH(k_cand_vote_warp, (unsigned)cdiv(n_cand, VOTE_WARPS), VOTE_WARPS * 32, 0, D.cand_row, D.cand_voff, n_cand, D.row_cnt,
           D.v_pos, D.v_start, D.v_group, D.cand_good, D.cand_dir, big_list, n_big);
    LAUNCH(k_cand_vote<1024>, (unsigned)ctx->n_sm * 2, 1024, 0, D.cand_row, D.cand_voff, big_list, n_big, D.row_cnt, D.v_pos,
           D.v_start, D.v_group, D.cand_good, D.cand_dir);
  }
  // haplotype mode: per segment and haplotype best, good, dir, tie at 2 * s + h, and the tie list over those entries
  u32 *hap_best = nullptr, *hap_good = nullptr, *hap_tie_seg = nullptr;
  u8 *hap_dir = nullptr, *hap_tie = nullptr;
  if (haps) {
    CKR(gvs_reserve(ctx, ctx->rh_scratch, (n_seg + 1) * 2 * (4 * 3 + 2)));
    hap_best = ctx->rh_scratch.as<u32>();
    hap_good = hap_best + 2 * n_seg;
    hap_tie_seg = hap_good + 2 * n_seg;
    hap_dir = (u8*)(hap_tie_seg + 2 * n_seg);
    hap_tie = hap_dir + 2 * n_seg;
    StageTimer th(ctx, GVS_ST_READHAPS);
    LAUNCH(k_seg_best_haps, (unsigned)cdiv(n_seg, 256), 256, 0, (u32)n_seg, seg_start, D.cidx, D.cand_row, D.row_cnt, contig,
           contig_hap, D.cand_good, D.cand_dir, hap_best, hap_good, hap_dir, hap_tie);
  } else {
    LAUNCH(k_seg_best, (unsigned)cdiv(n_seg, 256), 256, 0, (u32)n_seg, seg_start, D.cidx, D.cand_row, D.row_cnt, contig,
           D.cand_good, D.cand_dir, D.seg_best, D.seg_good, D.seg_dir, D.seg_tie);
  }
  // ---- ties: Table capacity at the start of each read (sticky within a chunk) ----
  u32 n_tie = 0;
  {
    const u8* st = haps ? hap_tie : D.seg_tie;
    u32* ts = haps ? hap_tie_seg : D.tie_seg;
    auto f = [st] __device__(u64 s) -> u32 { return st[s]; };
    auto g = [ts] __device__(u64 s, u32 ex, u32 v) { if (v) ts[ex] = (u32)s; };
    CKR(scan_total(ctx, haps ? 2 * n_seg : n_seg, f, g, OpSum(), &n_tie));
  }
  if (n_tie) {
    const u32 *sc = D.seg_chunk, *nd = D.seg_ndist;
    u32* cap = D.seg_cap;
    auto f = [sc, nd] __device__(u64 s) -> u64 { return ((u64)(sc[s] + 1) << 32) | cap_needed(nd[s]); };
    auto g = [sc, cap] __device__(u64 s, u64 ex, u64 v) {
      cap[s] = ((u32)(ex >> 32) == sc[s] + 1) ? (u32)ex : 64u;  // capacity left by earlier reads of the chunk
    };
    u64 mxv = 0;
    CKR(scan_total(ctx, n_seg, f, g, OpMax(), &mxv));
    // any read may itself grow the table while it is replayed: bound by the largest need overall
    u32 maxcap = 64;
    {
      // the u64 max is dominated by the chunk id; take a safe bound from the largest segment instead
      u32 max_nd = 0;
      const u32* ndp = D.seg_ndist;
      auto f2 = [ndp] __device__(u64 s) -> u32 { return ndp[s]; };
      auto g2 = [] __device__(u64 s, u32 ex, u32 v) {};
      CKR(scan_total(ctx, n_seg, f2, g2, OpMax(), &max_nd));
      maxcap = cap_needed(max_nd) * 2;
    }
    DevBuf& sb = ctx->scan_tmp2;
    CKR(gvs_reserve(ctx, sb, (u64)n_tie * 2 * maxcap * 4));
    if (haps)
      LAUNCH(k_seg_tie<true>, (unsigned)cdiv(n_tie, 64), 64, 0, hap_tie_seg, n_tie, seg_start, D.seg_cap, D.cidx, D.cand_row,
             D.row_cnt, contig, ctx->contig_hash.as<u32>(), D.cand_good, D.cand_dir, contig_hap, sb.as<u32>(), maxcap, hap_best,
             hap_dir);
    else
      LAUNCH(k_seg_tie<false>, (unsigned)cdiv(n_tie, 64), 64, 0, D.tie_seg, n_tie, seg_start, D.seg_cap, D.cidx, D.cand_row,
             D.row_cnt, contig, ctx->contig_hash.as<u32>(), D.cand_good, D.cand_dir, contig_hap, sb.as<u32>(), maxcap, D.seg_best,
             D.seg_dir);
  }
  if (haps) {
    StageTimer th(ctx, GVS_ST_READHAPS);
    LAUNCH(k_seg_pick, (unsigned)cdiv(n_seg, 256), 256, 0, (u32)n_seg, D.seg_hap, hap_best, hap_good, hap_dir, D.seg_best,
           D.seg_good, D.seg_dir);
    // records: one per segment with a vote on either haplotype, in segment (read) order
    CKR(rec_reserve(ctx, ctx->rh, 8, n_seg));
    RecTable& T = ctx->rh;
    u32* cols[8];
    for (u32 c = 0; c < 8; c++) cols[c] = T.col(c);
    u32 *r_read = cols[0], *r_c1 = cols[1], *r_n1 = cols[2], *r_s1 = cols[3], *r_c2 = cols[4], *r_n2 = cols[5], *r_s2 = cols[6],
        *r_hap = cols[7];
    const u32 *hb = hap_best, *hg = hap_good;
    const u8* hd = hap_dir;
    auto f = [hb] __device__(u64 s) -> u32 { return (hb[2 * s] != NOBEST || hb[2 * s + 1] != NOBEST) ? 1u : 0u; };
    auto g = [=] __device__(u64 s, u32 ex, u32 v) {
      if (!v) return;
      r_read[ex] = read[seg_start[s]];
      r_c1[ex] = hb[2 * s];
      r_n1[ex] = hg[2 * s];
      r_s1[ex] = hb[2 * s] != NOBEST ? hd[2 * s] ^ 1u : 0u;  // dir 1 = '+' -> strand 0
      r_c2[ex] = hb[2 * s + 1];
      r_n2[ex] = hg[2 * s + 1];
      r_s2[ex] = hb[2 * s + 1] != NOBEST ? hd[2 * s + 1] ^ 1u : 0u;
      r_hap[ex] = hap_assign(hg[2 * s], hg[2 * s + 1]);
    };
    u32 n_rec = 0;
    CKR(scan_total(ctx, n_seg, f, g, OpSum(), &n_rec));
    T.n = n_rec;
  }
  // ---- kept rows + best list ----
  u32* kt = counter(ctx, CNT_KEPT);
  {
    const u32* sbest = D.seg_best;
    u32* ke = D.keep_excl;
    auto f = [sbest, row_seg, contig] __device__(u64 j) -> u32 { return sbest[row_seg[j]] == contig[j] ? 1u : 0u; };
    auto g = [ke] __device__(u64 j, u32 ex, u32 v) { ke[j] = ex; };
    CKR((device_scan<u32>(ctx, n, f, g, OpSum(), kt)));
  }
  u32* bt = counter(ctx, CNT_BEST);
  {
    const u32* sbest = D.seg_best;
    u32* be = D.best_excl;
    auto f = [sbest] __device__(u64 s) -> u32 { return sbest[s] != NOBEST ? 1u : 0u; };
    auto g = [be] __device__(u64 s, u32 ex, u32 v) { be[s] = ex; };
    CKR((device_scan<u32>(ctx, n_seg, f, g, OpSum(), bt)));
  }
  u64 kb[2] = {0, 0};  // one read-back for both totals
  CKR(read_dev(ctx, counter<u64>(ctx, CNT_KEPT), kb, 2));
  const u32 n_kept = (u32)kb[0], n_best = (u32)kb[1];
  CKR(gvs_reserve_rows(ctx, ctx->kept, n_kept));
  CKR(gvs_reserve(ctx, ctx->best_read, (u64)n_best * 4));
  CKR(gvs_reserve(ctx, ctx->best_contig, (u64)n_best * 4));
  CKR(gvs_reserve(ctx, ctx->best_good, (u64)n_best * 4));
  CKR(gvs_reserve(ctx, ctx->best_dir, (u64)n_best));
  LAUNCH(k_keep_rows, (unsigned)cdiv(n, 256), 256, 0, n, D.keep_excl, row_seg, D.seg_best, read, pos, contig, start, group, gidx,
         ctx->kept.read.as<u32>(), ctx->kept.pos.as<u32>(), ctx->kept.contig.as<u32>(), ctx->kept.start.as<u32>(),
         ctx->kept.group.as<u32>(), ctx->kept.gidx.as<u32>());
  LAUNCH(k_best_rows, (unsigned)cdiv(n_seg, 256), 256, 0, (u32)n_seg, D.best_excl, D.seg_best, D.seg_good, D.seg_dir, seg_start,
         read, ctx->best_read.as<u32>(), ctx->best_contig.as<u32>(), ctx->best_good.as<u32>(), ctx->best_dir.as<u8>());
  ctx->kept.n = n_kept;
  ctx->n_best = n_best;
  *n_best_out = n_best;
  *n_kept_out = n_kept;
  return 0;
}

extern "C" int gvs_diag_filter(gvs_ctx* ctx, const uint8_t* contig_hap, const uint32_t* contig_hash, uint64_t* n_best,
                               uint64_t* n_kept) {
  return gvs_diag_filter_haps(ctx, contig_hap, contig_hash, 0, n_best, n_kept);
}

extern "C" int gvs_diag_filter_haps(gvs_ctx* ctx, const uint8_t* contig_hap, const uint32_t* contig_hash, int read_haps,
                                    uint64_t* n_best, uint64_t* n_kept) {
  if (!ctx) return GVS_E_ARG;
  if (!ctx->match_ready) return gvs_fail(ctx, GVS_E_STATE, "gvs_diag_filter before gvs_match");
  if (!contig_hap || !contig_hash) return gvs_fail(ctx, GVS_E_ARG, "null contig tables");
  CK(cudaSetDevice(ctx->device));
  ctx->diag_ready = false;
  ctx->val_ready = false;
  CKR(to_dev(ctx, ctx->contig_hap, contig_hap, ctx->n_contigs));
  CKR(to_dev(ctx, ctx->contig_hash, contig_hash, ctx->n_contigs));
  bool haps = read_haps != 0;
  for (u8 h : ctx->h_chunk_hap) haps |= h == GVS_HAP_ANY;
  u64 nb = 0, nk = 0;
  CKR(diag_impl(ctx, haps, &nb, &nk));
  if (n_best) *n_best = nb;
  if (n_kept) *n_kept = nk;
  ctx->diag_ready = true;
  return 0;
}

extern "C" int gvs_read_haps(gvs_ctx* ctx, uint64_t* n_records) {
  if (!ctx) return GVS_E_ARG;
  if (!ctx->rh.ready) return gvs_fail(ctx, GVS_E_STATE, "gvs_read_haps without a diag filter in haplotype mode");
  if (n_records) *n_records = ctx->rh.n;
  return 0;
}

extern "C" int gvs_read_haps_get(gvs_ctx* ctx, uint32_t* read, uint32_t* contig1, uint32_t* n1, uint32_t* strand1,
                                 uint32_t* contig2, uint32_t* n2, uint32_t* strand2, uint32_t* hap) {
  return ctx ? rec_get(ctx, ctx->rh, "gvs_read_haps_get without a diag filter in haplotype mode",
                       {read, contig1, n1, strand1, contig2, n2, strand2, hap})
             : GVS_E_ARG;
}

extern "C" int gvs_best_get(gvs_ctx* ctx, uint32_t* read_idx, uint32_t* contig, uint32_t* ngood, uint8_t* dir) {
  if (!ctx) return GVS_E_ARG;
  if (!ctx->diag_ready) return gvs_fail(ctx, GVS_E_STATE, "gvs_best_get before gvs_diag_filter");
  CK(cudaSetDevice(ctx->device));
  u64 n = ctx->n_best;
  if (n == 0) return 0;
  if (read_idx) CK(cudaMemcpyAsync(read_idx, ctx->best_read.p, n * 4, cudaMemcpyDeviceToHost, ctx->stream));
  if (contig) CK(cudaMemcpyAsync(contig, ctx->best_contig.p, n * 4, cudaMemcpyDeviceToHost, ctx->stream));
  if (ngood) CK(cudaMemcpyAsync(ngood, ctx->best_good.p, n * 4, cudaMemcpyDeviceToHost, ctx->stream));
  if (dir) CK(cudaMemcpyAsync(dir, ctx->best_dir.p, n, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return 0;
}

// ---------------------------------------------------------------------------------------------
// diag_filter_step2 on its own (workflow/src/diag_filter_step2.nim:13-66): the best contig per read
// comes from a `_diag.sunkpos` file instead of the vote; rows whose contig equals it survive.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_keep_by_table(u64 n, const u32* __restrict__ keep_excl, const u32* __restrict__ best_of_read,
                                                       const u32* __restrict__ read, const u32* __restrict__ pos,
                                                       const u32* __restrict__ contig, const u32* __restrict__ start,
                                                       const u32* __restrict__ group, const u32* __restrict__ gidx, u32* o_read,
                                                       u32* o_pos, u32* o_contig, u32* o_start, u32* o_group, u32* o_gidx) {
  u64 j = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n) return;
  u32 c = contig[j];
  if (best_of_read[read[j]] != c) return;
  u32 o = keep_excl[j];
  o_read[o] = read[j];
  o_pos[o] = pos[j];
  o_contig[o] = c;
  o_start[o] = start[j];
  o_group[o] = group[j];
  o_gidx[o] = gidx[j];
}

extern "C" int gvs_filter_best(gvs_ctx* ctx, const uint32_t* best_contig_of_read, uint64_t* n_kept) {
  if (!ctx || !best_contig_of_read) return GVS_E_ARG;
  if (!ctx->match_ready) return gvs_fail(ctx, GVS_E_STATE, "gvs_filter_best before gvs_match / gvs_rows_set(0)");
  CK(cudaSetDevice(ctx->device));
  Rows& R = ctx->rows;
  u64 n = R.n;
  ctx->kept.n = 0;
  ctx->n_best = 0;
  CKR(to_dev(ctx, ctx->seg_best, best_contig_of_read, ctx->n_reads ? ctx->n_reads : 1));
  CKR(gvs_reserve(ctx, ctx->flags_b, (n ? n : 1) * 4));
  u32 nk = 0;
  if (n) {
    const u32* best = ctx->seg_best.as<u32>();
    const u32 *read = R.read.as<u32>(), *contig = R.contig.as<u32>();
    u32* ke = ctx->flags_b.as<u32>();
    auto f = [best, read, contig] __device__(u64 j) -> u32 { return best[read[j]] == contig[j] ? 1u : 0u; };
    auto g = [ke] __device__(u64 j, u32 ex, u32 v) { ke[j] = ex; };
    CKR(scan_total(ctx, n, f, g, OpSum(), &nk));
    CKR(gvs_reserve_rows(ctx, ctx->kept, nk));
    LAUNCH(k_keep_by_table, (unsigned)cdiv(n, 256), 256, 0, n, ke, best, read, R.pos.as<u32>(), contig, R.start.as<u32>(),
           R.group.as<u32>(), R.gidx.as<u32>(), ctx->kept.read.as<u32>(), ctx->kept.pos.as<u32>(), ctx->kept.contig.as<u32>(),
           ctx->kept.start.as<u32>(), ctx->kept.group.as<u32>(), ctx->kept.gidx.as<u32>());
    CK(cudaStreamSynchronize(ctx->stream));
  }
  ctx->kept.n = nk;
  ctx->diag_ready = true;
  ctx->val_ready = false;
  if (n_kept) *n_kept = nk;
  return 0;
}
