// table.cuh -- device-side view of the SUNK probe structures (shared by build and probe kernels)
//
// Layout in HBM (DESIGN.md "Data layout"):
//   filt      u32[filt_words]   word-blocked Bloom filter, 2 bits per key inside ONE 32-bit word;
//                               sized to stay L2-resident (<= 64 MiB), probed once per read base
//   tab_kv    u64[2 tab_slots]  open-addressed canonical k-mers, buckets of 4 slots, load factor <= 0.5, EMPTY =
//                               all ones (k <= 31 => < 2^62; at k = 32 the all-T k-mer's
//                               canonical form is all-A); a bucket is 64 bytes: 4 keys, then their 4 value
//                               words (low: .loc row or GVS_ROW_MISSING / GVS_ROW_NOTINDB, high: the row's dense
//                               group index) -- one HBM access per lookup
//                               (tab_keys u64[tab_slots] / tab_rows u32[tab_slots] only exist while the table is built)
#pragma once
#include "common.cuh"

struct TabView {
  // probe-side layout: bucket b = 64 bytes = its 4 keys followed by its 4 value words (low word: .loc row or GVS_ROW_*,
  // high word: dense group index of the row), so that a lookup is ONE 64-byte access to HBM: the keys decide, and the
  // value of a match has arrived with them (the probe's warps used to wait for two dependent random accesses)
  const u64* __restrict__ kv;
  u64 slots;
};

#define GVS_NOHIT 0xFFFFFFFDu

// 16 bytes of a bucket; .L2::64B: a miss fills half a line, not the whole 128 bytes (the buckets are scattered over
// gigabytes: profiles/microbench/fetch_granularity.cu)
__device__ __forceinline__ ulonglong2 tab_ld16(const ulonglong2* p) {
  ulonglong2 v;
  asm volatile("ld.global.nc.L2::64B.v2.u64 {%0,%1}, [%2];" : "=l"(v.x), "=l"(v.y) : "l"(p));
  return v;
}
// returns row, GVS_ROW_MISSING / GVS_ROW_NOTINDB, or GVS_NOHIT; *gidx = group index of the row (valid for a real row)
__device__ __forceinline__ u32 tab_lookup(const TabView& t, u64 key, u64 h, u32* gidx) {
  const u64 nb = t.slots >> 2;
  u64 b = gvs_tab_bucket(h, t.slots);
  for (u64 it = 0; it < nb; it++) {
    const ulonglong2* p = (const ulonglong2*)(t.kv + (b << 3));
    const ulonglong2 a = tab_ld16(p), c = tab_ld16(p + 1);
    const ulonglong2 va = tab_ld16(p + 2), vc = tab_ld16(p + 3);
    u64 v;
    bool found = true;
    if (a.x == key) v = va.x;
    else if (a.y == key) v = va.y;
    else if (c.x == key) v = vc.x;
    else if (c.y == key) v = vc.y;
    else found = false;
    if (found) {
      *gidx = (u32)(v >> 32);
      return (u32)v;
    }
    if (a.x == GVS_EMPTY_KEY || a.y == GVS_EMPTY_KEY || c.x == GVS_EMPTY_KEY || c.y == GVS_EMPTY_KEY) return GVS_NOHIT;
    b = (b + 1) & (nb - 1);
  }
  return GVS_NOHIT;
}

// find-or-insert; returns slot index (never fails while load < 1)
__device__ __forceinline__ u64 tab_insert(u64* keys, u64 slots, u64 key, u64 h) {
  u64 nb = slots >> 2;
  u64 b = gvs_tab_bucket(h, slots);
  for (;;) {
#pragma unroll
    for (int j = 0; j < 4; j++) {
      u64 s = (b << 2) + j;
      u64 cur = keys[s];
      if (cur == key) return s;
      if (cur == GVS_EMPTY_KEY) {
        u64 old = atomicCAS((unsigned long long*)&keys[s], (unsigned long long)GVS_EMPTY_KEY,
                            (unsigned long long)key);
        if (old == GVS_EMPTY_KEY || old == key) return s;
      }
    }
    b = (b + 1) & (nb - 1);
  }
}
