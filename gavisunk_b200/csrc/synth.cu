// synth.cu -- deterministic synthetic workloads generated on the device (bench.py / tests only;
// SURVEY.md 8d): a diploid assembly (hap1 i.i.d. ACGT + segmental duplications + N runs, hap2 =
// hap1 + SNPs) and ONT-like reads (log-normal lengths, both strands, 3 % substitutions, 2 %
// deletions, 1 % insertions, occasional N runs).  Counter-based hashing (no RNG state), so any
// position can be regenerated independently.
#include "common.cuh"

__host__ __device__ __forceinline__ u64 sm64(u64 x) {  // splitmix64 finaliser
  x += 0x9E3779B97F4A7C15ull;
  x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
  x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
  return x ^ (x >> 31);
}
__host__ __device__ __forceinline__ u64 h3(u64 seed, u64 a, u64 b) { return sm64(sm64(seed ^ (a * 0xD1342543DE82EF95ull)) + b); }

struct DupEvent { u64 tgt, src, len; };  // hap-local coordinates (concatenated hap1 contigs)
struct NRun { u64 pos, len; };

__device__ __forceinline__ u32 raw_base(u64 seed, u64 pos) { return (u32)(h3(seed, 1, pos) >> 17) & 3; }

__global__ void __launch_bounds__(256) k_synth_asm(u8* seq, u64 hap_len, u64 seed, u64 snp_thr,
                                                   const DupEvent* __restrict__ dups, u32 n_dups,
                                                   const NRun* __restrict__ nruns, u32 n_nruns) {
  const char ACGT[4] = {'A', 'C', 'G', 'T'};
  for (u64 p = (u64)blockIdx.x * blockDim.x + threadIdx.x; p < hap_len; p += (u64)gridDim.x * blockDim.x) {
    u64 src = p;
    // duplication targets are sorted and disjoint: binary search
    {
      u32 lo = 0, hi = n_dups;
      while (lo < hi) {
        u32 mid = (lo + hi) >> 1;
        if (dups[mid].tgt + dups[mid].len <= p) lo = mid + 1; else hi = mid;
      }
      if (lo < n_dups && dups[lo].tgt <= p) src = dups[lo].src + (p - dups[lo].tgt);
    }
    u32 b1 = raw_base(seed, src);
    u32 b2 = b1;
    u64 hs = h3(seed, 2, p);
    if ((hs >> 32) < snp_thr) b2 = (b1 + 1 + (u32)(hs % 3)) & 3;
    u8 c1 = ACGT[b1], c2 = ACGT[b2];
    {
      u32 lo = 0, hi = n_nruns;
      while (lo < hi) {
        u32 mid = (lo + hi) >> 1;
        if (nruns[mid].pos + nruns[mid].len <= p) lo = mid + 1; else hi = mid;
      }
      if (lo < n_nruns && nruns[lo].pos <= p) c1 = c2 = 'N';
    }
    seq[p] = c1;
    seq[hap_len + p] = c2;
  }
}

extern "C" int gvs_synth_assembly(gvs_ctx* ctx, uint8_t* seq_dev, const uint64_t* contig_len, uint32_t n_contigs_per_hap,
                                  double snp_rate, double dup_frac, uint64_t seed) {
  if (!ctx || !seq_dev || !contig_len || n_contigs_per_hap == 0) return GVS_E_ARG;
  CK(cudaSetDevice(ctx->device));
  u64 hap_len = 0;
  for (u32 c = 0; c < n_contigs_per_hap; c++) hap_len += contig_len[c];
  // duplication events: blocks of 10-100 kb (scaled down for tiny assemblies) copied from elsewhere
  std::vector<DupEvent> dups;
  std::vector<NRun> nruns;
  u64 st = sm64(seed ^ 0xABCDEF);
  auto rnd = [&st]() { st = sm64(st); return st; };
  u64 blk_min = 10000, blk_max = 100000;
  if (hap_len < 4000000) { blk_min = hap_len / 400 + 50; blk_max = hap_len / 40 + 100; }
  u64 want = (u64)(dup_frac * (double)hap_len), have = 0;
  // place targets left to right with random gaps so that they are sorted and disjoint
  if (want > 0 && hap_len > 4 * blk_max) {
    u64 n_ev = want / ((blk_min + blk_max) / 2) + 1;
    u64 stride = hap_len / n_ev;
    for (u64 e = 0; e < n_ev && have < want; e++) {
      u64 len = blk_min + rnd() % (blk_max - blk_min + 1);
      if (len + 2 > stride) len = stride / 2;
      if (len == 0) continue;
      u64 tgt = e * stride + rnd() % (stride - len);
      u64 src = rnd() % (hap_len - len);
      dups.push_back({tgt, src, len});
      have += len;
    }
  }
  // N runs: 0.01 % of the sequence in runs of 50..500 (scaled for tiny assemblies)
  {
    u64 n_want = hap_len / 10000;
    u64 n_ev = n_want / 275 + (hap_len >= 20000 ? 1 : 0);
    u64 stride = n_ev ? hap_len / n_ev : 0;
    for (u64 e = 0; e < n_ev; e++) {
      u64 len = 50 + rnd() % 451;
      if (len * 4 > stride) continue;
      u64 pos = e * stride + rnd() % (stride - len);
      nruns.push_back({pos, len});
    }
  }
  DevBuf dd, dn;
  int rc = to_dev(ctx, dd, dups.data(), dups.size());
  if (!rc) rc = to_dev(ctx, dn, nruns.data(), nruns.size());
  if (!rc) {
    u64 snp_thr = (u64)(snp_rate * 4294967296.0);
    u64 grid = cdiv(hap_len, 256);
    if (grid > (u64)ctx->n_sm * 32) grid = (u64)ctx->n_sm * 32;
    k_synth_asm<<<(unsigned)grid, 256, 0, ctx->stream>>>(seq_dev, hap_len, seed, snp_thr, dd.as<DupEvent>(), (u32)dups.size(),
                                                        dn.as<NRun>(), (u32)nruns.size());
    ctx->launches++;
    if (cudaGetLastError() != cudaSuccess) rc = gvs_fail(ctx, GVS_E_CUDA, "k_synth_asm launch failed");
  }
  cudaStreamSynchronize(ctx->stream);
  gvs_release(dd);
  gvs_release(dn);
  return rc;
}

// ---------------------------------------------------------------------------------------------
// reads
// ---------------------------------------------------------------------------------------------
#define RSEG 1024  // source bases per generation segment

struct ReadPlan {
  u64 src;      // global assembly coordinate of the first source base
  u32 len;      // source bases
  u32 flags;    // bit0 = reverse strand, bit1 = carries an N run
  u32 n_pos, n_len;
};

struct SynthState {
  DevBuf plan, seg_first, seg_out, seg_off;
  u64 n_reads = 0, n_segs = 0, seed = 0;
};
static SynthState g_synth;  // one plan at a time (bench / tests helper, not part of the engine state)
int gvs_synth_plan_scans(gvs_ctx* ctx, DevBuf& segcount, u64 n_reads, u64* read_off_dev, u64* total_bases);

// error model thresholds out of 65536
#define DEL_THR 1311   // 2 %
#define SUB_THR 1966   // 3 %
#define INS_THR 655    // 1 %

__device__ __forceinline__ u32 src_emit_count(u64 seed, u64 r, u32 j) {
  u64 h = h3(seed, 16 + r, j);
  u32 del = (u32)(h & 0xFFFF) < DEL_THR;
  u32 ins = (u32)((h >> 32) & 0xFFFF) < INS_THR;
  return (del ? 0u : 1u) + ins;
}

__global__ void __launch_bounds__(256) k_reads_sample(ReadPlan* plan, u32* segcount, u64 n_reads,
                                                      const u64* __restrict__ contig_off, u32 clo, u32 chi, double mu,
                                                      double sigma, u32 lmin, u32 lmax, u64 seed) {
  u64 r = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n_reads) return;
  u64 g0 = contig_off[clo], g1 = contig_off[chi];
  u64 span = g1 - g0;
  u64 h = h3(seed, 3, r);
  u64 pos = g0 + __umul64hi(h, span);
  // contig of pos
  u32 lo = clo, hi = chi;
  while (hi - lo > 1) {
    u32 mid = (lo + hi) >> 1;
    if (contig_off[mid] <= pos) lo = mid; else hi = mid;
  }
  u64 cend = contig_off[lo + 1];
  // log-normal length (Box-Muller on hashed uniforms)
  u64 h2 = h3(seed, 4, r);
  double u1 = ((double)(h2 >> 11) + 0.5) * (1.0 / 9007199254740992.0);
  double u2 = ((double)(h3(seed, 5, r) >> 11) + 0.5) * (1.0 / 9007199254740992.0);
  double z = sqrt(-2.0 * log(u1)) * cos(6.283185307179586 * u2);
  double L = exp(mu + sigma * z);
  u64 len = (u64)L;
  if (len < lmin) len = lmin;
  if (len > lmax) len = lmax;
  if (pos + len > cend) len = cend - pos;
  u64 h6 = h3(seed, 6, r);
  ReadPlan p;
  p.src = pos;
  p.len = (u32)len;
  p.flags = (u32)(h6 & 1);
  p.n_pos = 0;
  p.n_len = 0;
  if (((h6 >> 8) % 1000) == 0 && len > 400) {  // 0.1 % of the reads carry an N run
    p.flags |= 2;
    p.n_len = 1 + (u32)((h6 >> 24) % 40);
    p.n_pos = (u32)((h6 >> 32) % (len - p.n_len));
  }
  plan[r] = p;
  segcount[r] = (u32)((len + RSEG - 1) / RSEG);
}

__device__ __forceinline__ u64 seg_read(const u64* __restrict__ seg_first, u64 n_reads, u64 seg) {
  u64 lo = 0, hi = n_reads;  // last r with seg_first[r] <= seg
  while (hi - lo > 1) {
    u64 mid = (lo + hi) >> 1;
    if (seg_first[mid] <= seg) lo = mid; else hi = mid;
  }
  return lo;
}

__global__ void __launch_bounds__(256) k_seg_count(const ReadPlan* __restrict__ plan, const u64* __restrict__ seg_first,
                                                   u64 n_reads, u64 n_segs, u64 seed, u32* seg_out) {
  u64 s = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n_segs) return;
  u64 r = seg_read(seg_first, n_reads, s);
  u32 j0 = (u32)(s - seg_first[r]) * RSEG;
  u32 j1 = min(plan[r].len, j0 + RSEG);
  u32 c = 0;
  for (u32 j = j0; j < j1; j++) c += src_emit_count(seed, r, j);
  seg_out[s] = c;
}

__global__ void __launch_bounds__(256) k_read_offsets(const u64* __restrict__ seg_first, const u64* __restrict__ seg_off,
                                                      u64 n_reads, u64 n_segs, u64 total, u64* read_off) {
  u64 r = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (r > n_reads) return;
  if (r == n_reads) { read_off[r] = total; return; }
  u64 s = seg_first[r];
  read_off[r] = s < n_segs ? seg_off[s] : total;
}

__global__ void __launch_bounds__(256) k_seg_fill(const ReadPlan* __restrict__ plan, const u64* __restrict__ seg_first,
                                                  const u64* __restrict__ seg_off, const u64* __restrict__ read_off,
                                                  u64 n_reads, u64 n_segs, u64 seed, const u8* __restrict__ asm_seq,
                                                  u8* out) {
  u64 s = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n_segs) return;
  const char ACGT[4] = {'A', 'C', 'G', 'T'};
  u64 r = seg_read(seg_first, n_reads, s);
  ReadPlan p = plan[r];
  u32 j0 = (u32)(s - seg_first[r]) * RSEG;
  u32 j1 = min(p.len, j0 + RSEG);
  u64 rstart = read_off[r], rend = read_off[r + 1];
  u64 o = seg_off[s] - seg_off[seg_first[r]];  // forward output index inside the read
  bool rev = p.flags & 1;
  for (u32 j = j0; j < j1; j++) {
    u64 h = h3(seed, 16 + r, j);
    bool del = (u32)(h & 0xFFFF) < DEL_THR;
    bool sub = (u32)((h >> 16) & 0xFFFF) < SUB_THR;
    bool ins = (u32)((h >> 32) & 0xFFFF) < INS_THR;
    u8 c = asm_seq[p.src + j];
    if (!del) {
      if (sub) {
        u32 x = ((c >> 1) ^ (c >> 2)) & 3;
        c = ACGT[(x + 1 + (u32)((h >> 48) % 3)) & 3];
      }
      if ((p.flags & 2) && j >= p.n_pos && j < p.n_pos + p.n_len) c = 'N';
      u8 w = c;
      if (rev) {  // reverse complement: mirrored index, complemented base (non-ACGT -> N)
        u8 l = c | 0x20;
        w = l == 'a' ? 'T' : l == 'c' ? 'G' : l == 'g' ? 'C' : l == 't' ? 'A' : 'N';
      }
      out[rstart + (rev ? (rend - rstart - 1 - o) : o)] = w;
      o++;
    }
    if (ins) {
      u8 w = ACGT[(h >> 52) & 3];
      out[rstart + (rev ? (rend - rstart - 1 - o) : o)] = w;
      o++;
    }
  }
}

extern "C" int gvs_synth_reads_plan(gvs_ctx* ctx, const uint64_t* contig_off_dev, uint32_t contig_lo, uint32_t contig_hi,
                                    uint64_t n_reads, double len_mu, double len_sigma, uint32_t len_min,
                                    uint32_t len_max, uint64_t seed, uint64_t* read_off_dev, uint64_t* total_bases) {
  if (!ctx || !contig_off_dev || !read_off_dev || contig_hi <= contig_lo) return GVS_E_ARG;
  CK(cudaSetDevice(ctx->device));
  SynthState& S = g_synth;
  S.n_reads = n_reads;
  S.seed = seed;
  CKR(gvs_reserve(ctx, S.plan, n_reads * sizeof(ReadPlan)));
  CKR(gvs_reserve(ctx, S.seg_first, (n_reads + 1) * 8));
  DevBuf segcount;
  CKR(gvs_reserve(ctx, segcount, n_reads * 4));
  int rc = 0;
  if (n_reads) {
    k_reads_sample<<<(unsigned)cdiv(n_reads, 256), 256, 0, ctx->stream>>>(S.plan.as<ReadPlan>(), segcount.as<u32>(), n_reads,
        contig_off_dev, contig_lo, contig_hi, len_mu, len_sigma, len_min, len_max, seed);
    ctx->launches++;
    if (cudaGetLastError() != cudaSuccess) rc = gvs_fail(ctx, GVS_E_CUDA, "k_reads_sample launch failed");
  }
  if (!rc) rc = gvs_synth_plan_scans(ctx, segcount, n_reads, read_off_dev, total_bases);
  cudaStreamSynchronize(ctx->stream);
  gvs_release(segcount);
  return rc;
}

int gvs_synth_plan_scans(gvs_ctx* ctx, DevBuf& segcount, u64 n_reads, u64* read_off_dev, u64* total_bases) {
  SynthState& S = g_synth;
  const u32* sc = segcount.as<u32>();
  u64* sf = S.seg_first.as<u64>();
  u64 n_segs = 0;
  {
    auto f = [sc] __device__(u64 i) -> u64 { return (u64)sc[i]; };
    auto g = [sf] __device__(u64 i, u64 ex, u64 v) { sf[i] = ex; };
    CKR(scan_total(ctx, n_reads, f, g, OpSum(), &n_segs));
  }
  S.n_segs = n_segs;
  CK(cudaMemcpyAsync(sf + n_reads, counter<u64>(ctx, CNT_SCAN), 8, cudaMemcpyDeviceToDevice, ctx->stream));
  CKR(gvs_reserve(ctx, S.seg_out, n_segs * 4));
  CKR(gvs_reserve(ctx, S.seg_off, (n_segs + 1) * 8));
  if (n_segs)
    LAUNCH(k_seg_count, (unsigned)cdiv(n_segs, 256), 256, 0, S.plan.as<ReadPlan>(), sf, n_reads, n_segs, S.seed,
           S.seg_out.as<u32>());
  const u32* so = S.seg_out.as<u32>();
  u64* sof = S.seg_off.as<u64>();
  u64 total = 0;
  {
    auto f = [so] __device__(u64 i) -> u64 { return (u64)so[i]; };
    auto g = [sof] __device__(u64 i, u64 ex, u64 v) { sof[i] = ex; };
    CKR(scan_total(ctx, n_segs, f, g, OpSum(), &total));
  }
  LAUNCH(k_read_offsets, (unsigned)cdiv(n_reads + 1, 256), 256, 0, sf, sof, n_reads, n_segs, total, read_off_dev);
  if (total_bases) *total_bases = total;
  return 0;
}

extern "C" int gvs_synth_reads_fill(gvs_ctx* ctx, const uint8_t* asm_seq_dev, uint8_t* reads_dev,
                                    const uint64_t* read_off_dev, uint64_t n_reads) {
  if (!ctx || !asm_seq_dev || !reads_dev || !read_off_dev) return GVS_E_ARG;
  CK(cudaSetDevice(ctx->device));
  SynthState& S = g_synth;
  if (S.n_reads != n_reads) return gvs_fail(ctx, GVS_E_STATE, "gvs_synth_reads_fill: plan first");
  if (S.n_segs)
    LAUNCH(k_seg_fill, (unsigned)cdiv(S.n_segs, 256), 256, 0, S.plan.as<ReadPlan>(), S.seg_first.as<u64>(),
           S.seg_off.as<u64>(), read_off_dev, n_reads, S.n_segs, S.seed, asm_seq_dev, reads_dev);
  CK(cudaStreamSynchronize(ctx->stream));
  return 0;
}
