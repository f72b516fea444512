// validate_reads.cu -- per-read inter-SUNK distance validation
// (workflow/scripts/process-by-contig_lowmem_AR.py:50-207; SURVEY.md A.6 steps 1-5, Q12-Q14).
//
// One thread group per read: a warp for reads with <= 64 rows (8 reads per 256-thread block, no block
// barriers), a 256-thread block with shared memory up to 512 rows, a 1024-thread block with global
// scratch beyond.  Rows minus bad groups -> rank-sort by (assembly start, read position) -> every
// pair (i<j) tested with the integer form of the reference's float64 ratio test (0.9 < dpos/dstart <
// 1.1  <=>  9*ds < 10*dp < 11*ds, exact for 32-bit inputs) -> orientation majority -> "multipos"
// clean-up -> connected components of the graph on group IDs -> largest component (ties: the
// component holding the earliest vertex in graph-tool's insertion order) -> output in vertex order.
//
// Every pass is row-centric and branch-free: the thread that owns row r walks all rows q with
// shared-memory broadcast reads and predicated arithmetic; the pair predicate is recomputed instead
// of stored (the edge list of a read is O(rows^2)).  Components come from min-label propagation over
// the recomputed edge predicate (a few rounds: these graphs are dense), not from per-edge atomics.
#include "common.cuh"

#define VCAP_WARP 64      // rows per read handled by one warp
#define VCAP 512          // rows per read handled in shared memory by one block
#define VROW_BYTES 80     // bytes of working storage per row
#define NOV 0xFFFFFFFFu
#define NOT64 0xFFFFFFFFFFFFFFFFull

#define F_MULTI 1u   // the row's ID occurs at more than one read position among the oriented edges
#define F_GOOD 2u    // ... and this row is the ID's most frequent position
#define F_PRES 4u    // the row has at least one surviving edge

struct VWork {
  u32 *P, *S, *ID, *G;        // rows sorted by (assembly start, read position)
  u32 *uP, *uS, *uID, *uG;    // rows after bad-group removal (any order)
  u32 *deg, *rep, *label, *csize, *flags;
  u64 *key, *tv, *ct;
};

__device__ __forceinline__ void vwork_carve(VWork& w, u8* base, u32 cap) {
  u64* q = (u64*)base;
  w.key = q; q += cap;
  w.tv = q; q += cap;
  w.ct = q; q += cap;
  u32* p = (u32*)q;
  w.P = p; p += cap; w.S = p; p += cap; w.ID = p; p += cap; w.G = p; p += cap;
  w.uP = p; p += cap; w.uS = p; p += cap; w.uID = p; p += cap; w.uG = p; p += cap;
  w.deg = p; p += cap; w.rep = p; p += cap; w.label = p; p += cap; w.csize = p; p += cap; w.flags = p; p += cap;
}

// 0.9 < dpos/dstart < 1.1 in float64 (process-by-contig_lowmem_AR.py:145-147) as exact integers (Q12)
__device__ __forceinline__ bool pair_ok(u32 pi, u32 si, u32 pj, u32 sj) {
  u64 ds = si > sj ? si - sj : sj - si;
  u64 dp = pi > pj ? pi - pj : pj - pi;
  return 9 * ds < 10 * dp && 10 * dp < 11 * ds;
}

struct ValParams : SegRows {  // kept rows
  ReadLens len;
  u32 min_len;
  u32* out_id;               // per kept row slot: validated IDs of the read, from its first row on
  u32* out_gidx;
  u32* seg_cnt;              // validated IDs per segment
  u8* orient;                // orientation majority per segment with validated IDs (0: read positions rise with starts)
  u32 m_lo, m_hi;            // this launch handles reads with m_lo < rows <= m_hi
  u8* gscratch;              // global-scratch variant: per block VROW_BYTES * big_cap
  u32 big_cap;
  u32* stats;                // [0] reads whose clean-up removed every edge (reference would raise)
};

// NT threads per read, GROUPS reads per block; GLOBAL: working arrays in global scratch
template <int NT, int GROUPS, bool GLOBAL>
__global__ void __launch_bounds__(NT* GROUPS) k_validate(const ValParams V) {
  extern __shared__ __align__(16) u8 smem[];
  __shared__ u32 s_n0[GROUPS], s_n1[GROUPS], s_m[GROUPS], s_kept[GROUPS], s_bestroot[GROUPS], s_flag[GROUPS], s_dup[GROUPS];
  __shared__ u32 s_pmin[GROUPS], s_pmax[GROUPS];  // span of the read's positions (all threads of the group)
  __shared__ u32 s_up[GROUPS], s_dn[GROUPS];      // some position step up / down along ascending starts
  __shared__ unsigned long long s_best[GROUPS];
  __shared__ u32 s_wtot[GROUPS][NT / 32];  // per-warp counts of the order-preserving compaction
  const int grp = threadIdx.x / NT;
  const int tid = threadIdx.x % NT;
  auto gsync = [&]() {
    if (NT == 32) __syncwarp(); else __syncthreads();
  };
  VWork w;
  const u32 cap = GLOBAL ? V.big_cap : (NT == 32 ? VCAP_WARP : VCAP);
  if (GLOBAL) vwork_carve(w, V.gscratch + (u64)blockIdx.x * VROW_BYTES * cap, cap);
  else vwork_carve(w, smem + (u64)grp * VROW_BYTES * cap, cap);

  for (u32 s = blockIdx.x * GROUPS + grp; s < V.n_seg; s += gridDim.x * GROUPS) {
    const u32 a = V.seg_start[s], b = V.seg_start[s + 1];
    const u32 mrows = b - a;
    if (mrows <= V.m_lo || mrows > V.m_hi) continue;  // another launch owns this read (group-uniform)
    gsync();
    if (tid == 0) { s_m[grp] = 0; s_n0[grp] = 0; s_n1[grp] = 0; s_kept[grp] = 0; s_best[grp] = 0; s_bestroot[grp] = NOV; s_flag[grp] = 0; s_dup[grp] = 0; s_pmin[grp] = 0xFFFFFFFFu; s_pmax[grp] = 0; s_up[grp] = 0; s_dn[grp] = 0; }
    gsync();
    // read length filter (hard-coded 10000 in the reference, :106-108; Q13)
    const u32 rd = V.read[a];
    const u32 rlen = V.len(rd);
    const bool skip = rlen < V.min_len || mrows < 2;
    // ---- rows minus bad groups (:70-72), input order preserved (a read's rows come in increasing pos) ----
    if (!skip) {
      u32 kept_so_far = 0;
      for (u32 base = 0; base < mrows; base += NT) {
        const u32 i = base + tid;
        bool keep = false;
        u32 gi = 0;
        if (i < mrows) {
          gi = V.gidx[a + i];
          keep = !(V.bad && V.bad[gi]);
        }
        const u32 bal = __ballot_sync(0xFFFFFFFFu, keep);
        if (NT > 32) {
          if ((tid & 31) == 0) s_wtot[grp][tid >> 5] = __popc(bal);
          gsync();
        }
        u32 before = 0, total = __popc(bal);
        if (NT > 32) {
          total = 0;
          for (int wv = 0; wv < NT / 32; wv++) {
            u32 c = s_wtot[grp][wv];
            before += wv < (tid >> 5) ? c : 0u;
            total += c;
          }
        }
        if (keep) {
          const u32 d = kept_so_far + before + __popc(bal & ((1u << (tid & 31)) - 1));
          w.uP[d] = V.pos[a + i];
          w.uS[d] = V.start[a + i];
          w.uID[d] = V.group[a + i];
          w.uG[d] = gi;
        }
        kept_so_far += total;
        if (NT > 32) gsync();
      }
      if (tid == 0) s_m[grp] = kept_so_far;
    }
    gsync();
    const u32 m = s_m[grp];
    if (skip || m < 2) {
      if (tid == 0) V.seg_cnt[s] = 0;
      continue;
    }
    // ---- sort by (start, pos): sort_values(['rname','start']) is stable and rows of a read come in
    //      increasing pos (:100).  Reads follow one strand: their starts are usually already strictly
    //      ascending or strictly descending, which makes the sort a copy; otherwise rank sort. ----
    {
      u32 not_asc = 0, not_desc = 0;
      for (u32 i = tid; i + 1 < m; i += NT) {
        const u32 s0 = w.uS[i], s1 = w.uS[i + 1];
        not_asc |= s0 >= s1;
        not_desc |= s0 <= s1;
      }
      if (not_asc) s_n0[grp] = 1;
      if (not_desc) s_n1[grp] = 1;
      gsync();
      const u32 mono = s_n0[grp] == 0 ? 1u : (s_n1[grp] == 0 ? 2u : 0u);
      gsync();
      if (tid == 0) { s_n0[grp] = 0; s_n1[grp] = 0; }
      for (u32 i = tid; i < m; i += NT) {
        const u32 si = w.uS[i], pi = w.uP[i];
        u32 rank = mono == 1 ? i : m - 1 - i;
        if (mono == 0) {
          rank = 0;
          for (u32 j = 0; j < m; j++) {
            u32 sj = w.uS[j], pj = w.uP[j];
            rank += (sj < si) | ((sj == si) & (pj < pi));
          }
        }
        w.P[rank] = pi;
        w.S[rank] = si;
        w.ID[rank] = w.uID[i];
        w.G[rank] = w.uG[i];
        w.csize[i] = 0;
        w.tv[i] = NOT64;
        w.ct[i] = NOT64;
      }
    }
    gsync();
    // some group ID on more than one row (rare: the general path below).  IDs are group starts, so along
    // ascending SUNK starts they do not decrease and equal IDs are neighbours; rows that break this
    // (hand-made input) are sent down the general path as well.
    {
      u32 dupl = 0;
      for (u32 i = tid; i + 1 < m; i += NT) dupl |= w.ID[i] >= w.ID[i + 1];
      if (dupl) s_dup[grp] = 1;
    }
    // at least two distinct groups (:91-97)
    {
      const u32 id0 = w.ID[0];
      u32 any = 0;
      for (u32 i = tid; i < m; i += NT) any |= w.ID[i] != id0;
      if (any) s_flag[grp] = 1;
    }
    gsync();
    if (!s_flag[grp]) {
      if (tid == 0) V.seg_cnt[s] = 0;
      continue;
    }
    // ---- pass AB: masked pairs by sign (:140-152) and, for BOTH candidate orientations at once, the
    //      incidence of every row in the oriented edge list (the (ID,pos) multiset M) with its order of
    //      first appearance in M = [all left ends in edge order] + [all right ends]; the orientation is
    //      only known after the whole read has been seen, so both variants are kept until then.
    //      Rows are sorted by start, so |ds| needs no abs; partners below and above the row are walked
    //      separately (the row is the right / the left end of the pair); when starts and positions of
    //      the read span < 2^28 the ratio test 9*ds < 10*dp < 11*ds runs in 32-bit arithmetic. ----
    {
      // span of the positions (starts are sorted: S[m-1] - S[0])
      u32 pmin = 0xFFFFFFFFu, pmax = 0;
      for (u32 r = tid; r < m; r += NT) {
        u32 p = w.P[r];
        pmin = p < pmin ? p : pmin;
        pmax = p > pmax ? p : pmax;
      }
      // a thread sees only its strided rows: the span is that of the whole group (warp shuffle, then shared atomics)
      for (int d = 16; d; d >>= 1) {
        pmin = min(pmin, __shfl_xor_sync(0xFFFFFFFFu, pmin, d));
        pmax = max(pmax, __shfl_xor_sync(0xFFFFFFFFu, pmax, d));
      }
      if ((tid & 31) == 0 && pmax >= pmin) {
        atomicMin(&s_pmin[grp], pmin);
        atomicMax(&s_pmax[grp], pmax);
      }
      gsync();
      if (tid == 0 && (s_pmax[grp] - s_pmin[grp] >= (1u << 28) || w.S[m - 1] - w.S[0] >= (1u << 28))) s_flag[grp] = 2;  // (s_flag is 1 here; 2 = wide read)
      gsync();
      const bool narrow = s_flag[grp] != 2;
      u32 n0 = 0, n1 = 0;
      // Reads follow one strand of one locus: along ascending starts their positions then never decrease (or never
      // increase), every pair has the same sign, and with one row per ID nothing downstream needs the number of
      // masked pairs -- only, per row, whether it has a partner and which partner comes first on either side
      // (presence, first appearance in the edge list, first label).  Those are found by a search that stops at the
      // first hit: O(rows) per read instead of O(rows^2) pair tests.
      u32 p_up = 0, p_dn = 0;
      if (!s_dup[grp]) {
        for (u32 i = tid; i + 1 < m; i += NT) {
          const u32 a0 = w.P[i], a1 = w.P[i + 1];
          p_up |= a0 < a1;
          p_dn |= a0 > a1;
        }
        if (p_up) s_up[grp] = 1;
        if (p_dn) s_dn[grp] = 1;
      }
      gsync();
      const bool steps_up = s_up[grp] != 0, steps_dn = s_dn[grp] != 0;
      const u32 psign = (!s_dup[grp] && !(steps_up && steps_dn)) ? (steps_dn ? 2u : 1u) : 0u;  // 1: never decreases, 2: never increases
      auto search = [&](auto ok_fn) {
        for (u32 r = tid; r < m; r += NT) {
          const u32 pr = w.P[r], sr = w.S[r];
          u32 fp = NOV, fh = NOV;
          for (u32 q = 0; q < r; q++) {
            const u32 pq = w.P[q];
            if (ok_fn(sr - w.S[q], pq > pr ? pq - pr : pr - pq)) { fp = q; break; }
          }
          for (u32 q = r + 1; q < m; q++) {
            const u32 pq = w.P[q];
            if (ok_fn(w.S[q] - sr, pq > pr ? pq - pr : pr - pq)) { fh = q; break; }
          }
          const u32 d = (fp != NOV) + (fh != NOV);
          if (psign == 1) { w.uP[r] = fp; w.uS[r] = fh; w.uID[r] = NOV; w.uG[r] = NOV; w.deg[r] = d; w.label[r] = 0; n0 += fh != NOV; }
          else { w.uP[r] = NOV; w.uS[r] = NOV; w.uID[r] = fp; w.uG[r] = fh; w.deg[r] = 0; w.label[r] = d; n1 += fh != NOV; }
        }
      };
      auto walk = [&](auto ok_fn) {
        for (u32 r = tid; r < m; r += NT) {
          const u32 pr = w.P[r], sr = w.S[r];
          u32 dlo0 = 0, dlo1 = 0, dhi0 = 0, dhi1 = 0, fp0 = NOV, fp1 = NOV, fh0 = NOV, fh1 = NOV;
          for (u32 q = 0; q < r; q++) {  // pair (q, r): r is the right end; sign = pos_q > pos_r
            const u32 pq = w.P[q], sq = w.S[q];
            const u32 sg = pq > pr;
            const u32 ok = ok_fn(sr - sq, sg ? pq - pr : pr - pq);
            const u32 e1 = ok & sg, e0 = ok & (sg ^ 1u);
            dlo0 += e0;
            dlo1 += e1;
            fp0 = min(fp0, q | (e0 - 1u));  // first edge (q, r) with r as the right end
            fp1 = min(fp1, q | (e1 - 1u));
          }
          for (u32 q = r + 1; q < m; q++) {  // pair (r, q): r is the left end; sign = pos_r > pos_q
            const u32 pq = w.P[q], sq = w.S[q];
            const u32 sg = pr > pq;
            const u32 ok = ok_fn(sq - sr, sg ? pr - pq : pq - pr);
            const u32 e1 = ok & sg, e0 = ok & (sg ^ 1u);
            dhi0 += e0;
            dhi1 += e1;
            fh0 = min(fh0, q | (e0 - 1u));  // first edge (r, q) with r as the left end
            fh1 = min(fh1, q | (e1 - 1u));
          }
          // the unsorted copies are dead after the sort: they keep the first partners of both orientations
          w.uP[r] = fp0; w.uS[r] = fh0; w.uID[r] = fp1; w.uG[r] = fh1;
          n0 += dhi0;
          n1 += dhi1;
          w.deg[r] = dlo0 + dhi0;
          w.label[r] = dlo1 + dhi1;
          w.key[r] = dhi0 ? (u64)r : ((1ull << 63) | ((u64)fp0 * m + r));
          w.ct[r] = dhi1 ? (u64)r : ((1ull << 63) | ((u64)fp1 * m + r));
        }
      };
      // 0.9 < dpos/dstart < 1.1 in float64 (:145-147) as exact integers (Q12)
      if (psign) {
        if (narrow) search([](u32 ds, u32 dp) -> bool { return (9u * ds < 10u * dp) & (10u * dp < 11u * ds); });
        else search([](u32 ds, u32 dp) -> bool { return (9ull * ds < 10ull * dp) & (10ull * dp < 11ull * ds); });
      } else if (narrow) walk([](u32 ds, u32 dp) -> u32 { return (9u * ds < 10u * dp) & (10u * dp < 11u * ds); });
      else walk([](u32 ds, u32 dp) -> u32 { return (9ull * ds < 10ull * dp) & (10ull * dp < 11ull * ds); });
      for (int d = 16; d; d >>= 1) {
        n0 += __shfl_xor_sync(0xFFFFFFFFu, n0, d);
        n1 += __shfl_xor_sync(0xFFFFFFFFu, n1, d);
      }
      if ((tid & 31) == 0) {
        if (n0) atomicAdd(&s_n0[grp], n0);
        if (n1) atomicAdd(&s_n1[grp], n1);
      }
    }
    gsync();
    if (s_n0[grp] + s_n1[grp] < 1) {  // `if sum(mask) < 1: continue` (:148)
      if (tid == 0) V.seg_cnt[s] = 0;
      continue;
    }
    const u32 orient = s_n1[grp] > s_n0[grp];  // np.unique sorted + argmax: a tie keeps 0 (:151-152)
    if (!s_dup[grp]) {
      // Every ID sits on exactly one row: the multipos clean-up (:161-181) cannot drop anything, a vertex is
      // a row, and what pass C would derive follows from the first partners found in pass AB -- presence
      // = degree > 0, first appearance in the edge list = the earlier of (r, first right partner) as a
      // source and (first left partner, r) as a target, first label = smallest neighbour or itself.
      for (u32 r = tid; r < m; r += NT) {
        const u32 deg = orient ? w.label[r] : w.deg[r];
        const u32 fp = orient ? w.uID[r] : w.uP[r], fh = orient ? w.uG[r] : w.uS[r];
        const u32 present = deg > 0;
        u64 tmin = NOT64;
        if (fh != NOV) tmin = 2 * ((u64)r * m + fh);
        if (fp != NOV) {
          u64 et = 2 * ((u64)fp * m + r) + 1;
          tmin = et < tmin ? et : tmin;
        }
        w.rep[r] = r;
        w.flags[r] = present ? F_PRES : 0u;
        w.label[r] = present ? (fp != NOV ? fp : r) : NOV;
        w.tv[r] = present ? tmin : NOT64;
        w.ct[r] = NOT64;
      }
      if (tid == 0) s_kept[grp] = orient ? s_n1[grp] : s_n0[grp];
    } else {
      for (u32 r = tid; r < m; r += NT) {
        if (orient) {
          w.deg[r] = w.label[r];
          w.key[r] = w.ct[r];
        }
        w.ct[r] = NOT64;
      }
      gsync();
      // ---- multipos (:161-181): IDs seen at more than one read position keep their most frequent one ----
      for (u32 r = tid; r < m; r += NT) {
        const u32 id = w.ID[r], dr = w.deg[r];
        const u64 kr = w.key[r];
        u32 first = r, multi = 0, good = dr > 0;
        for (u32 q = 0; q < m; q++) {
          u32 same = (w.ID[q] == id);
          u32 dq = w.deg[q];
          first = (same & (q < first)) ? q : first;
          u32 other = same & (q != r) & (dq > 0);
          multi |= other;
          u32 beats = other & ((dq > dr) | ((dq == dr) & (w.key[q] < kr)));
          good &= beats ^ 1u;
        }
        w.rep[r] = first;
        w.flags[r] = ((multi & (dr > 0)) ? F_MULTI : 0u) | (good ? F_GOOD : 0u);
      }
      gsync();
      // ---- pass C: surviving edges (:189-192): presence, first appearance, first label ----
      // edge (lo, hi) is dropped iff the LEFT row's ID is multi-positioned, lo is not that ID's good row and
      // hi is not that ID's good row either (left end only: Q14)
      {
        u32 nk = 0;
        for (u32 r = tid; r < m; r += NT) {
          const u32 pr = w.P[r], sr = w.S[r], idr = w.ID[r], fr = w.flags[r];
          u64 tmin = NOT64;
          u32 lab = NOV;
          for (u32 q = 0; q < m; q++) {
            u32 pq = w.P[q], sq = w.S[q], idq = w.ID[q], fq = w.flags[q];
            u32 hi = q > r;
            u32 sg = hi ? (pr > pq) : (pq > pr);
            u32 e = pair_ok(pr, sr, pq, sq) & (q != r) & (sg == orient);
            u32 fl = hi ? fr : fq, fh = hi ? fq : fr;  // flags of the left / right row of the pair
            u32 drop = ((fl & F_MULTI) != 0) & ((fl & F_GOOD) == 0) & (((fh & F_GOOD) == 0) | (idq != idr));
            u32 kept = e & (drop ^ 1u);
            u32 lo_row = hi ? r : q, hi_row = hi ? q : r;
            u64 et = 2 * ((u64)lo_row * m + hi_row) + (hi ^ 1u);  // source before target
            tmin = (kept && et < tmin) ? et : tmin;
            nk += kept & hi;
            u32 rq = w.rep[q];
            lab = (kept && rq < lab) ? rq : lab;
          }
          u32 present = tmin != NOT64;
          u32 rr = w.rep[r];
          w.flags[r] = fr | (present ? F_PRES : 0u);
          w.label[r] = present ? (rr < lab ? rr : lab) : NOV;
          if (present) atomicMin((unsigned long long*)&w.tv[rr], (unsigned long long)tmin);
        }
        if (nk) atomicAdd(&s_kept[grp], nk);
      }
    }
    gsync();
    if (s_kept[grp] == 0) {  // graph-tool would raise on the empty graph; counted, read skipped (A.6 step 5)
      if (tid == 0) {
        V.seg_cnt[s] = 0;
        atomicAdd(&V.stats[0], 1u);
      }
      continue;
    }
    // Shortcut for the common case: pass C already took one propagation step (label = min rep over the
    // row's own ID and its neighbours); if every present row now carries the same label L, each of them
    // is in or adjacent to vertex L, i.e. the graph is one component and no further round is needed.
    if (tid == 0) { s_n0[grp] = NOV; s_n1[grp] = 0; }
    gsync();
    for (u32 r = tid; r < m; r += NT)
      if (w.flags[r] & F_PRES) atomicMin(&s_n0[grp], w.label[r]);
    gsync();
    {
      const u32 l0 = s_n0[grp];
      u32 differs = 0;
      for (u32 r = tid; r < m; r += NT) differs |= ((w.flags[r] & F_PRES) != 0) & (w.label[r] != l0);
      if (differs) s_n1[grp] = 1;
    }
    gsync();
    // one row per ID and a single component found by the shortcut: every present row but the first has that first
    // row as its first left partner, so the vertices were inserted in row order (see the output pass below)
    const bool in_row_order = !s_dup[grp] && s_n1[grp] == 0;
    // ---- components: min-label propagation over surviving edges and same-ID rows until stable ----
    for (int round = 0; s_n1[grp] && round < 4096; round++) {
      if (tid == 0) s_flag[grp] = 0;
      gsync();
      u32 changed = 0;
      for (u32 r = tid; r < m; r += NT) {
        const u32 fr = w.flags[r];
        if (!(fr & F_PRES)) continue;
        const u32 pr = w.P[r], sr = w.S[r], idr = w.ID[r];
        u32 lab = w.label[r];
        const u32 lab0 = lab;
        for (u32 q = 0; q < m; q++) {
          u32 pq = w.P[q], sq = w.S[q], idq = w.ID[q], fq = w.flags[q];
          u32 hi = q > r;
          u32 sg = hi ? (pr > pq) : (pq > pr);
          u32 e = pair_ok(pr, sr, pq, sq) & (q != r) & (sg == orient);
          u32 fl = hi ? fr : fq, fh = hi ? fq : fr;
          u32 drop = ((fl & F_MULTI) != 0) & ((fl & F_GOOD) == 0) & (((fh & F_GOOD) == 0) | (idq != idr));
          u32 link = (e & (drop ^ 1u)) | ((idq == idr) & ((fq & F_PRES) != 0));  // edge, or same vertex
          u32 lq = w.label[q];  // may already be this round's value: only speeds convergence up
          lab = (link && lq < lab) ? lq : lab;
        }
        if (lab != lab0) {
          w.label[r] = lab;
          changed = 1;
        }
      }
      if (changed) s_flag[grp] = 1;
      gsync();
      if (!s_flag[grp]) break;
      gsync();
    }
    // ---- component sizes (distinct IDs) and earliest vertex ----
    for (u32 r = tid; r < m; r += NT) {
      u32 fr = w.flags[r];
      if (!(fr & F_PRES)) continue;
      // the first present row of an ID represents the vertex
      const u32 idr = w.ID[r];
      u32 firstp = r;
      if (s_dup[grp])  // (with one row per ID every present row is its own vertex)
        for (u32 q = 0; q < r; q++)
          if (w.ID[q] == idr && (w.flags[q] & F_PRES)) { firstp = q; break; }
      if (firstp != r) continue;
      u32 lab = w.label[r];
      atomicAdd(&w.csize[lab], 1u);
      atomicMin((unsigned long long*)&w.ct[lab], (unsigned long long)w.tv[w.rep[r]]);
      w.flags[r] = fr | 8u;  // vertex representative
    }
    gsync();
    // largest component; ties -> lowest label = the one holding the earliest-inserted vertex
    for (u32 r = tid; r < m; r += NT) {
      if (w.csize[r]) {
        unsigned long long key = ((unsigned long long)w.csize[r] << 42) | ((1ull << 42) - 1 - w.ct[r]);
        atomicMax(&s_best[grp], key);
      }
    }
    gsync();
    for (u32 r = tid; r < m; r += NT) {
      if (w.csize[r]) {
        unsigned long long key = ((unsigned long long)w.csize[r] << 42) | ((1ull << 42) - 1 - w.ct[r]);
        if (key == s_best[grp]) s_bestroot[grp] = r;
      }
    }
    gsync();
    const u32 broot = s_bestroot[grp];
    // ---- output in vertex order (first appearance in the edge list, source before target) ----
    if (in_row_order) {
      // vertex order == row order: the first vertex v0 enters as the source of its first edge (v0, r1), every other
      // row r as the target of (v0, r), and edges are listed by (left row, right row); rank = vertices before the row
      u32 done = 0;
      for (u32 base = 0; base < m; base += NT) {
        const u32 r = base + tid;
        const bool mem = r < m && (w.flags[r] & 8u);
        const u32 bal = __ballot_sync(0xFFFFFFFFu, mem);
        if (NT > 32) {
          if ((tid & 31) == 0) s_wtot[grp][tid >> 5] = __popc(bal);
          gsync();
        }
        u32 before = 0, total = __popc(bal);
        if (NT > 32) {
          total = 0;
          for (int wv = 0; wv < NT / 32; wv++) {
            const u32 c = s_wtot[grp][wv];
            before += wv < (tid >> 5) ? c : 0u;
            total += c;
          }
        }
        if (mem) {
          const u32 rank = done + before + __popc(bal & ((1u << (tid & 31)) - 1));
          V.out_id[a + rank] = w.ID[r];
          V.out_gidx[a + rank] = w.G[r];
        }
        done += total;
        if (NT > 32) gsync();
      }
    } else
    for (u32 r = tid; r < m; r += NT) {
      if ((w.flags[r] & 8u) && w.label[r] == broot) {
        const u64 t = w.tv[w.rep[r]];
        u32 rank = 0;
        for (u32 q = 0; q < m; q++) rank += ((w.flags[q] & 8u) != 0) & (w.label[q] == broot) & (w.tv[w.rep[q]] < t);
        V.out_id[a + rank] = w.ID[r];
        V.out_gidx[a + rank] = w.G[r];
      }
    }
    if (tid == 0) {
      V.seg_cnt[s] = w.csize[broot];
      V.orient[s] = (u8)orient;
    }
  }
}

__global__ void __launch_bounds__(256) k_pairs_compact(const u32* __restrict__ seg_start, const u32* __restrict__ seg_cnt,
                                                       const u32* __restrict__ seg_off, u32 n_seg, const u32* __restrict__ out_id,
                                                       const u32* __restrict__ out_gidx, const u32* __restrict__ read,
                                                       const u32* __restrict__ contig, u32* p_read, u32* p_contig, u32* p_group,
                                                       u32* p_gidx) {
  u32 wv = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  int lane = threadIdx.x & 31;
  if (wv >= n_seg) return;
  u32 c = seg_cnt[wv];
  if (!c) return;
  u32 a = seg_start[wv], o = seg_off[wv];
  u32 rd = read[a], ct = contig[a];
  for (u32 i = lane; i < c; i += 32) {
    p_read[o + i] = rd;
    p_contig[o + i] = ct;
    p_group[o + i] = out_id[a + i];
    p_gidx[o + i] = out_gidx[a + i];
  }
}

extern "C" int gvs_validate(gvs_ctx* ctx, uint32_t min_read_len, uint64_t* n_pairs_out) {
  if (!ctx) return GVS_E_ARG;
  if (!ctx->diag_ready) return gvs_fail(ctx, GVS_E_STATE, "gvs_validate before gvs_diag_filter / gvs_rows_set(1)");
  if (!ctx->read_off && !ctx->have_read_len) return gvs_fail(ctx, GVS_E_STATE, "gvs_validate: read lengths unknown");
  CK(cudaSetDevice(ctx->device));
  StageTimer tm(ctx, GVS_ST_VALIDATE);
  ctx->val_ready = false;
  ctx->pl.ready = ctx->sup.ready = false;
  ctx->dc.ready = ctx->dc_runs.ready = false;
  ctx->n_pairs = 0;
  if (n_pairs_out) *n_pairs_out = 0;
  Rows& R = ctx->kept;
  u64 n = R.n;
  if (n == 0) {
    ctx->val_ready = true;
    return 0;
  }
  u64 n_seg = 0;
  CKR(gvs_build_segments(ctx, R.read.as<u32>(), n, ctx->kseg_start, ctx->flags_c, &n_seg));
  ctx->n_kseg = n_seg;
  const u32* seg_start = ctx->kseg_start.as<u32>();
  // scratch: out_id[n], out_gidx[n], seg_cnt[n_seg], seg_off[n_seg]
  CKR(gvs_reserve(ctx, ctx->val_scratch, (2 * n + 2 * n_seg + 16) * 4));
  u32* out_id = ctx->val_scratch.as<u32>();
  u32* out_gidx = out_id + n;
  u32* seg_cnt = out_gidx + n;
  u32* seg_off = seg_cnt + n_seg;
  ctx->val_id = out_id; ctx->val_seg_cnt = seg_cnt; ctx->val_seg_off = seg_off;
  CKR(gvs_reserve(ctx, ctx->seg_orient, n_seg));
  // largest read (rows) decides which launches are needed
  u32 max_m = 0;
  {
    auto f2 = [seg_start] __device__(u64 s) -> u32 { return seg_start[s + 1] - seg_start[s]; };
    auto g2 = [] __device__(u64 s, u32 ex, u32 v) {};
    CKR(scan_total(ctx, n_seg, f2, g2, OpMax(), &max_m));
  }
  u32* stats = counter(ctx, CNT_VAL_STATS);
  CK(cudaMemsetAsync(stats, 0, 8, ctx->stream));
  ValParams V;
  (SegRows&)V = seg_rows(ctx, R, ctx->kseg_start, n_seg);
  V.len = read_lens(ctx);
  V.min_len = min_read_len;
  V.out_id = out_id; V.out_gidx = out_gidx; V.seg_cnt = seg_cnt; V.orient = ctx->seg_orient.as<u8>();
  V.gscratch = nullptr; V.big_cap = 0; V.stats = stats;
  const size_t sm_warp = (size_t)VROW_BYTES * VCAP_WARP * 8, sm_blk = (size_t)VROW_BYTES * VCAP;
  if (!ctx->val_attr_set) {
    CK(cudaFuncSetAttribute((k_validate<32, 8, false>), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm_warp));
    CK(cudaFuncSetAttribute((k_validate<256, 1, false>), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm_blk));
    ctx->val_attr_set = true;
  }
  // the three row-count tiers touch disjoint reads and outputs: they run side by side (the few very long
  // reads of the last tier would otherwise be a serial tail)
  const bool tiers = max_m > VCAP_WARP;
  if (tiers) CKR(gvs_fork(ctx));
  if (max_m > VCAP) {  // the few very long reads first: their blocks get placed before the SMs fill up
    u32 blocks = (u32)ctx->n_sm;
    u32 bcap = (max_m + 15) & ~15u;
    CKR(gvs_reserve(ctx, ctx->scan_tmp2, (u64)blocks * VROW_BYTES * bcap));
    V.gscratch = ctx->scan_tmp2.as<u8>();
    V.big_cap = bcap;
    V.m_lo = VCAP; V.m_hi = 0xFFFFFFFFu;
    LAUNCH_ON(ctx->aux[1], (k_validate<1024, 1, true>), blocks, 1024, 0, V);
    V.gscratch = nullptr; V.big_cap = 0;
  }
  if (max_m > VCAP_WARP) {
    V.m_lo = VCAP_WARP; V.m_hi = VCAP;
    u64 grid = n_seg;
    u64 capg = (u64)ctx->n_sm * 5;
    if (grid > capg) grid = capg;
    LAUNCH_ON(ctx->aux[0], (k_validate<256, 1, false>), (unsigned)grid, 256, sm_blk, V);
  }
  {  // reads with <= 64 rows: one warp each (includes the reads with < 2 rows, which just report 0)
    V.m_lo = 0; V.m_hi = VCAP_WARP;
    u64 grid = cdiv(n_seg, 8);
    u64 capg = (u64)ctx->n_sm * 5;
    if (grid > capg) grid = capg;
    LAUNCH((k_validate<32, 8, false>), (unsigned)grid, 256, sm_warp, V);
  }
  if (tiers) CKR(gvs_join(ctx));
  // compaction of the validated (ID, read) pairs
  u32 np = 0;
  {
    auto f = [seg_cnt] __device__(u64 s) -> u32 { return seg_cnt[s]; };
    auto g = [seg_off] __device__(u64 s, u32 ex, u32 v) { seg_off[s] = ex; };
    CKR(scan_total(ctx, n_seg, f, g, OpSum(), &np));
  }
  CKR(gvs_reserve(ctx, ctx->pair_read, (u64)np * 4));
  CKR(gvs_reserve(ctx, ctx->pair_contig, (u64)np * 4));
  CKR(gvs_reserve(ctx, ctx->pair_group, (u64)np * 4));
  CKR(gvs_reserve(ctx, ctx->pair_gidx, (u64)np * 4));
  if (np)
    LAUNCH(k_pairs_compact, (unsigned)cdiv(n_seg * 32, 256), 256, 0, seg_start, seg_cnt, seg_off, (u32)n_seg, out_id, out_gidx,
           R.read.as<u32>(), R.contig.as<u32>(), ctx->pair_read.as<u32>(), ctx->pair_contig.as<u32>(),
           ctx->pair_group.as<u32>(), ctx->pair_gidx.as<u32>());
  ctx->n_pairs = np;
  ctx->val_ready = true;
  if (n_pairs_out) *n_pairs_out = np;
  return 0;
}

extern "C" int gvs_pairs_get(gvs_ctx* ctx, uint32_t* read_idx, uint32_t* contig, uint32_t* group, uint32_t* group_index) {
  if (!ctx) return GVS_E_ARG;
  if (!ctx->val_ready) return gvs_fail(ctx, GVS_E_STATE, "gvs_pairs_get before gvs_validate");
  CK(cudaSetDevice(ctx->device));
  u64 n = ctx->n_pairs;
  if (n == 0) return 0;
  if (read_idx) CK(cudaMemcpyAsync(read_idx, ctx->pair_read.p, n * 4, cudaMemcpyDeviceToHost, ctx->stream));
  if (contig) CK(cudaMemcpyAsync(contig, ctx->pair_contig.p, n * 4, cudaMemcpyDeviceToHost, ctx->stream));
  if (group) CK(cudaMemcpyAsync(group, ctx->pair_group.p, n * 4, cudaMemcpyDeviceToHost, ctx->stream));
  if (group_index) CK(cudaMemcpyAsync(group_index, ctx->pair_gidx.p, n * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return 0;
}
