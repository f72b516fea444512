// format.cu -- text egress at the reference's file boundary (SURVEY.md Appendix C): .sunkpos / .rlen / kmer.loc /
// jellyfish.db / jellyfish.fa / inter_outs / BED rows formatted from column arrays on host threads.  The reference
// writes these with `writeLine` (workflow/src/kmerpos_annot3.nim:93), awk / bedtools (workflow/rules/defineSUNKs.smk:59-60,
// 124-126) and pandas to_csv (process-by-contig_lowmem_AR.py:203-207,260); a whole-genome sample has 1.2e8 kmer.loc
// rows and ~7e7 sunkpos rows, far too many for per-row Python formatting.  Host code only (no kernel).
#include <string.h>

#include <thread>
#include <vector>

#include "../../include/gavisunk_b200.h"

namespace {

static const char DIGIT_PAIRS[201] =
    "00010203040506070809101112131415161718192021222324252627282930313233343536373839404142434445464748495051525354555657585960616263646566"
    "676869707172737475767778798081828384858687888990919293949596979899";

static inline unsigned dec_len32(uint32_t v) {
  return v < 100000u ? (v < 100u ? (v < 10u ? 1 : 2) : (v < 1000u ? 3 : (v < 10000u ? 4 : 5)))
                     : (v < 10000000u ? (v < 1000000u ? 6 : 7) : (v < 100000000u ? 8 : (v < 1000000000u ? 9 : 10)));
}
static inline unsigned dec_len(uint64_t v) {
  if (v <= 0xFFFFFFFFull) return dec_len32((uint32_t)v);
  unsigned n = 0;
  while (v > 0xFFFFFFFFull) { v /= 10; n++; }
  return n + dec_len32((uint32_t)v);
}
// digits written backwards from p + len, two at a time
static inline void put_digits32(char* end, uint32_t v) {
  while (v >= 100u) {
    const uint32_t q = v / 100u, r = v - q * 100u;
    end -= 2;
    end[0] = DIGIT_PAIRS[2 * r];
    end[1] = DIGIT_PAIRS[2 * r + 1];
    v = q;
  }
  if (v >= 10u) {
    end -= 2;
    end[0] = DIGIT_PAIRS[2 * v];
    end[1] = DIGIT_PAIRS[2 * v + 1];
  } else {
    *--end = (char)('0' + v);
  }
}
static inline char* put_dec(char* p, uint64_t v) {
  const unsigned n = dec_len(v);
  char* end = p + n;
  while (v > 0xFFFFFFFFull) {
    *--end = (char)('0' + v % 10);
    v /= 10;
  }
  put_digits32(end, (uint32_t)v);
  return p + n;
}

static inline uint64_t cell_len(const gvs_col& c, uint64_t r) {
  uint64_t n = (c.prefix ? 1 : 0) + 1;  // + separator
  switch (c.kind) {
    case GVS_COL_U32: return n + dec_len(((const uint32_t*)c.data)[r]);
    case GVS_COL_U64: return n + dec_len(((const uint64_t*)c.data)[r]);
    case GVS_COL_I64: { int64_t v = ((const int64_t*)c.data)[r]; return n + (v < 0 ? 1 + dec_len((uint64_t)(-(v + 1)) + 1) : dec_len((uint64_t)v)); }
    case GVS_COL_NAME: { uint32_t i = ((const uint32_t*)c.data)[r]; return n + (c.name_off[i + 1] - c.name_off[i]); }
    case GVS_COL_KMER: return n + (uint64_t)c.k;
    default: return n;
  }
}
static inline char* put_cell(char* p, const gvs_col& c, uint64_t r) {
  if (c.prefix) *p++ = c.prefix;
  switch (c.kind) {
    case GVS_COL_U32: p = put_dec(p, ((const uint32_t*)c.data)[r]); break;
    case GVS_COL_U64: p = put_dec(p, ((const uint64_t*)c.data)[r]); break;
    case GVS_COL_I64: {
      int64_t v = ((const int64_t*)c.data)[r];
      if (v < 0) { *p++ = '-'; p = put_dec(p, (uint64_t)(-(v + 1)) + 1); } else p = put_dec(p, (uint64_t)v);
      break;
    }
    case GVS_COL_NAME: {
      uint32_t i = ((const uint32_t*)c.data)[r];
      uint64_t a = c.name_off[i], n = c.name_off[i + 1] - a;
      memcpy(p, c.names + a, n);
      p += n;
      break;
    }
    case GVS_COL_KMER: {
      uint64_t v = ((const uint64_t*)c.data)[r];
      for (int j = c.k - 1; j >= 0; j--) *p++ = "ACGT"[(v >> (2 * j)) & 3];
      break;
    }
    default: break;
  }
  *p++ = c.sep;
  return p;
}

}  // namespace

extern "C" int64_t gvs_format_rows(const gvs_col* cols, uint32_t n_cols, uint64_t n_rows, const uint64_t* sel, uint64_t n_sel,
                                   char* out, uint64_t cap, int threads) {
  if ((n_cols && !cols) || n_cols > 32) return GVS_E_ARG;  // junctions.reads.tsv has 19 columns
  const uint64_t n = sel ? n_sel : n_rows;
  for (uint32_t c = 0; c < n_cols; c++) {
    if (cols[c].kind < GVS_COL_U32 || cols[c].kind > GVS_COL_KMER) return GVS_E_ARG;
    if (n && !cols[c].data) return GVS_E_ARG;
    if (cols[c].kind == GVS_COL_NAME && (!cols[c].names || !cols[c].name_off)) return GVS_E_ARG;
    if (cols[c].kind == GVS_COL_KMER && (cols[c].k < 1 || cols[c].k > 32)) return GVS_E_ARG;
  }
  if (threads < 1) threads = 1;
  if ((uint64_t)threads > n / 4096 + 1) threads = (int)(n / 4096 + 1);
  std::vector<uint64_t> part((size_t)threads + 1, 0);
  auto range = [&](int t, uint64_t& a, uint64_t& b) { a = n * (uint64_t)t / threads; b = n * (uint64_t)(t + 1) / threads; };
  auto size_pass = [&](int t) {
    uint64_t a, b, s = 0;
    range(t, a, b);
    for (uint64_t i = a; i < b; i++) {
      const uint64_t r = sel ? sel[i] : i;
      for (uint32_t c = 0; c < n_cols; c++) s += cell_len(cols[c], r);
    }
    part[(size_t)t + 1] = s;
  };
  {
    std::vector<std::thread> pool;
    for (int t = 1; t < threads; t++) pool.emplace_back(size_pass, t);
    size_pass(0);
    for (auto& th : pool) th.join();
  }
  for (int t = 0; t < threads; t++) part[(size_t)t + 1] += part[(size_t)t];
  const uint64_t total = part[(size_t)threads];
  if (!out) return (int64_t)total;  // size query
  if (cap < total) return GVS_E_OVERFLOW;
  auto write_pass = [&](int t) {
    uint64_t a, b;
    range(t, a, b);
    char* p = out + part[(size_t)t];
    for (uint64_t i = a; i < b; i++) {
      const uint64_t r = sel ? sel[i] : i;
      for (uint32_t c = 0; c < n_cols; c++) p = put_cell(p, cols[c], r);
    }
  };
  {
    std::vector<std::thread> pool;
    for (int t = 1; t < threads; t++) pool.emplace_back(write_pass, t);
    write_pass(0);
    for (auto& th : pool) th.join();
  }
  return (int64_t)total;
}
