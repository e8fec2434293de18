// raven_b200 — seed lookup and hit expansion, shared by the single-GPU path
// (map.cu) and the key-partitioned multi-GPU path (dist.cu).
//
//   probe   one thread per query minimizer: bucket table -> sorted run ->
//           (first kept posting, kept count) or "filtered" if the run is
//           longer than the occurrence threshold
//   expand  hits (ram "Match": group = (rhs_id<<1|same_strand)<<32|diagonal,
//           positions = lhs_pos<<32|rhs_pos) written per query read
//
// The postings of a key are in read order (the index sort is stable over
// records in (read, position) order), so with avoid_equal && avoid_symmetric
// the kept postings (rhs_id > lhs_id) are a SUFFIX of the run - and with both
// flags off they are the whole run. The probe then only needs the first kept
// posting (a binary search in the run), and the expansion can be done by whole
// warps with fully coalesced stores. Other flags filter every posting.
#pragma once

#include "engine.cuh"

namespace rvn {

struct IndexView {
  ValView val;  // sorted values, u32 or u64
  const uint64_t* org;
  const uint32_t* bucket;
  uint64_t n;
  int shift;
  uint32_t occurrence;
  uint64_t limit;  // values beyond it are not indexed (tiered build)
};

inline IndexView IndexViewOf(const Ctx& c) {
  return IndexView{ValView{c.i_val.get(), c.i_is32 ? 1 : 0}, c.i_org.get(), c.i_bucket.get(),
                   c.i_n, c.i_shift, c.occurrence, c.i_limit};
}

// the kept postings of every run are contiguous (a suffix or the whole run)
inline bool KeptContiguous(const Ctx& c, bool avoid_equal, bool avoid_symmetric) {
  return (avoid_equal && avoid_symmetric && c.i_sorted_ids) || (!avoid_equal && !avoid_symmetric);
}

// first record with value v and the run length capped at occurrence+1
__device__ __forceinline__ void Lookup(const IndexView& ix, uint64_t v,
                                       uint32_t* first, uint32_t* count) {
  if (v > ix.limit) {
    *first = 0;
    *count = 0;
    return;
  }
  const uint64_t b = v >> ix.shift;
  uint32_t lo = ix.bucket[b], hi = ix.bucket[b + 1];
  while (hi - lo > 8) {  // long buckets: bisect down to a short scan
    const uint32_t mid = lo + (hi - lo) / 2;
    if (ix.val[mid] < v) {
      lo = mid + 1;
    } else {
      hi = mid;
    }
  }
  // here every record before lo is < v; the run (if any) starts in [lo, hi]
  const uint32_t end = ix.bucket[b + 1];
  while (lo < end && ix.val[lo] < v) ++lo;
  if (lo >= end || ix.val[lo] != v) {
    *first = 0;
    *count = 0;
    return;
  }
  *first = lo;
  if (ix.occurrence != 0xFFFFFFFFu &&
      static_cast<uint64_t>(lo) + ix.occurrence < ix.n &&
      ix.val[static_cast<uint64_t>(lo) + ix.occurrence] == v) {
    *count = ix.occurrence + 1;  // over the threshold, exact length not needed
    return;
  }
  uint32_t n = 1;
  while (static_cast<uint64_t>(lo) + n < ix.n && ix.val[lo + n] == v) ++n;
  *count = n;
}

__device__ __forceinline__ bool KeepPosting(uint32_t lhs_id, uint64_t origin,
                                            bool avoid_equal,
                                            bool avoid_symmetric) {
  const uint32_t rhs_id = static_cast<uint32_t>(origin >> 32);
  if (avoid_equal && lhs_id == rhs_id) return false;
  if (avoid_symmetric && lhs_id > rhs_id) return false;
  return true;
}

// which postings of its run a query keeps
enum class Kept { kFiltered, kSuffix, kWholeRun };

// first posting and kept count of the query with value v; lhs_read() gives its
// read id, loaded only where the kept postings depend on it. Returns whether the
// run is over the occurrence threshold (it then keeps nothing).
// kFiltered: *first = the run's first posting, the kept ones are among the run;
// kSuffix (rhs_id > lhs_id) and kWholeRun: the kept postings are [*first, +kept).
template <typename ReadId>
__device__ __forceinline__ bool Probe(const IndexView& ix, uint64_t v, ReadId lhs_read,
                                      Kept mode, bool avoid_equal, bool avoid_symmetric,
                                      uint32_t* first, uint32_t* kept) {
  uint32_t f, n;
  Lookup(ix, v, &f, &n);
  *first = f;
  *kept = 0;
  if (n > ix.occurrence) return true;
  if (n == 0) return false;
  const uint32_t lhs_id = mode == Kept::kWholeRun ? 0 : lhs_read();
  if (mode == Kept::kFiltered) {
    uint32_t k = 0;
    for (uint32_t j = 0; j < n; ++j) {
      k += KeepPosting(lhs_id, ix.org[f + j], avoid_equal, avoid_symmetric);
    }
    *kept = k;
    return false;
  }
  uint32_t lo = f;
  if (mode == Kept::kSuffix) {  // first posting with rhs_id > lhs_id
    uint32_t hi = f + n;
    while (lo < hi) {
      const uint32_t mid = lo + (hi - lo) / 2;
      if (static_cast<uint32_t>(ix.org[mid] >> 32) <= lhs_id) lo = mid + 1; else hi = mid;
    }
  }
  *first = lo;
  *kept = f + n - lo;
  return false;
}

// ram's Match: the hit of a query (origin lo) on a posting (origin o)
struct Match {
  uint64_t group, positions;
};

__device__ __forceinline__ Match EncodeHit(uint64_t lo, uint64_t o) {
  const uint32_t lhs_pos = static_cast<uint32_t>(lo) >> 1;
  const uint64_t rhs_pos = static_cast<uint32_t>(o) >> 1;
  const uint64_t rhs_id = o >> 32;
  const uint64_t strand = (lo & 1) == (o & 1);
  const uint64_t diagonal = !strand ? rhs_pos + lhs_pos : rhs_pos - lhs_pos + (3ULL << 30);
  return Match{(((rhs_id << 1) | strand) << 32) | diagonal,
               (static_cast<uint64_t>(lhs_pos) << 32) | rhs_pos};
}

// One thread per query (value v, origin lo): its `left` kept postings among the
// run from `first` on, written to [dst, dst + left). h_lhs, if not null, gets
// the query read of every hit.
__device__ __forceinline__ void ExpandQuery(const IndexView& ix, uint64_t v, uint64_t lo,
                                            uint32_t first, uint32_t left, bool avoid_equal,
                                            bool avoid_symmetric, uint64_t dst, uint64_t* h_grp,
                                            uint64_t* h_pos, uint32_t* h_lhs) {
  const uint32_t lhs_id = static_cast<uint32_t>(lo >> 32);
  for (uint64_t j = first; left > 0 && j < ix.n && ix.val[j] == v; ++j) {
    const uint64_t o = ix.org[j];
    if (!KeepPosting(lhs_id, o, avoid_equal, avoid_symmetric)) continue;
    const Match m = EncodeHit(lo, o);
    h_grp[dst] = m.group;
    h_pos[dst] = m.positions;
    if (h_lhs) h_lhs[dst] = lhs_id;
    ++dst;
    --left;
  }
}

// One whole warp for the queries of its 32 lanes, each with `cnt` hits on the
// contiguous postings org[first, first + cnt), written to [dst, dst + cnt).
// Hit t of the warp is located by a shuffle search over the 32 exclusive
// prefixes of the counts, so the loads and stores of a pass are coalesced when
// the destinations of consecutive lanes follow each other. Every lane of the
// warp must call it; lanes without a query pass cnt = 0. h_lhs as ExpandQuery.
__device__ __forceinline__ void ExpandWarp(const uint64_t* org, uint32_t cnt, uint32_t first,
                                           uint64_t lo, uint64_t dst, uint64_t* h_grp,
                                           uint64_t* h_pos, uint32_t* h_lhs) {
  const uint32_t lane = threadIdx.x & 31;
  uint32_t incl = cnt;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const uint32_t o = __shfl_up_sync(0xFFFFFFFFu, incl, d);
    if (lane >= static_cast<uint32_t>(d)) incl += o;
  }
  const uint32_t rel = incl - cnt;
  const uint32_t total = __shfl_sync(0xFFFFFFFFu, incl, 31);
  for (uint32_t t0 = 0; t0 < total; t0 += 32) {
    const uint32_t t = t0 + lane;
    uint32_t q = 0;  // largest q with rel[q] <= t
#pragma unroll
    for (uint32_t step = 16; step > 0; step >>= 1) {
      const uint32_t r = __shfl_sync(0xFFFFFFFFu, rel, q + step);
      if (r <= t) q += step;
    }
    const uint32_t qrel = __shfl_sync(0xFFFFFFFFu, rel, q);
    const uint32_t qfirst = __shfl_sync(0xFFFFFFFFu, first, q);
    const uint64_t qlo = __shfl_sync(0xFFFFFFFFu, lo, q);
    const uint64_t qdst = __shfl_sync(0xFFFFFFFFu, dst, q);
    if (t < total) {
      const uint64_t at = qdst + (t - qrel);
      const Match m = EncodeHit(qlo, org[qfirst + (t - qrel)]);
      h_grp[at] = m.group;
      h_pos[at] = m.positions;
      if (h_lhs) h_lhs[at] = static_cast<uint32_t>(qlo >> 32);
    }
  }
}

}  // namespace rvn
