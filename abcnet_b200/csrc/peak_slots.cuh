// Slot layout of the sparse-heads path: where peak i of group g = n * 2 + which (image n, which = 0 atom centres /
// 1 bond centres) sits in the compact tensors that the gathered patches, hidden maps and class logits share.
//   fixed  (off == nullptr): slot = g * cap + i, at most `cap` peaks per group -- a crowded image is truncated;
//   pooled (off != nullptr): slot = off[g] + i, off = exclusive prefix sums of the untruncated counts over the groups, one
//                            pool of `pool` slots for the whole batch -- a peak whose slot would be >= pool is dropped, so
//                            the batch's records are complete exactly when off[groups] (the total) <= pool.
// The find step, the patch gather and the record step all go through these functions, so the two layouts share one code
// path. Compiles for the host too (tests/test_peak_slots_cpu.py probes it there).
#pragma once
#include <cstdint>

#if defined(__CUDACC__)
#define ABC_SLOT_FN __host__ __device__ __forceinline__
#else
#define ABC_SLOT_FN inline
#endif

namespace abc {

struct SlotLayout {
  const int32_t* off;  // pooled: exclusive slot offsets [groups + 1]; nullptr selects the fixed layout
  int cap;             // fixed: slots per group
  int pool;            // pooled: slots in the pool
  int list_stride;     // entries per group in the peak lists: cap (fixed, truncated) or H * W (pooled, never truncated)
};

ABC_SLOT_FN int slot_base(const SlotLayout& L, int g) { return L.off ? L.off[g] : g * L.cap; }

// Peaks of group g (untruncated count `raw`) that own a slot; the rest are neither read nor written.
ABC_SLOT_FN int slot_count(const SlotLayout& L, int g, int raw) {
  if (!L.off) return raw < L.cap ? raw : L.cap;
  const int room = L.pool - L.off[g];
  return room <= 0 ? 0 : (raw < room ? raw : room);
}

// Group that owns `slot` (0 <= slot < number of slots): slot / cap, or the last g with off[g] <= slot (an empty group shares
// its offset with the next one, which then owns the slot). The index is slot - slot_base(L, g); it is a peak only when it is
// below slot_count(L, g, cnt[g]).
ABC_SLOT_FN int slot_group(const SlotLayout& L, int slot, int groups) {
  if (!L.off) return slot / L.cap;
  int lo = 0, hi = groups - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (L.off[mid] <= slot) lo = mid;
    else hi = mid - 1;
  }
  return lo;
}

// off[i] = base + cnt[0] + ... + cnt[i - 1] for i < n; returns base + the sum of all n counts. The offsets kernel runs it
// on consecutive runs of groups, each thread with the block-scanned base of its run.
ABC_SLOT_FN int slot_offsets(const int32_t* cnt, int n, int base, int32_t* off) {
  for (int i = 0; i < n; ++i) {
    off[i] = base;
    base += cnt[i];
  }
  return base;
}

}  // namespace abc
