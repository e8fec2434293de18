// raven_b200 — multi-GPU building blocks of the stage-1 overlap path.
//
// One context per rank; the collectives themselves are the caller's
// (raven_b200/distributed.py: torch.distributed over NCCL). With N ranks:
//   reads     sketched by contiguous ranges of equal bases (the caller's choice);
//   index     partitioned by KEY: owner(value) = value mod N (minimizers are
//             minima of hashes - their high bits are skewed towards zero, the
//             low bits stay uniform). Every key's postings live on exactly one
//             rank, in the reference's order: records arrive in read order and
//             the build sort is stable;
//   reads as queries / piles / overlap lists: read r belongs to rank r mod N
//             (with avoid_symmetric a read only meets higher ids, so contiguous
//             ranges would be triangular; the interleave gives every rank the
//             same mix).
// Steps per index batch of raven::FindOverlapsAndCreatePiles
// (RavenLib/src/construct.cc:36-112):
//   1. DistSketchSplit   sketch, stable radix partition of the records by owner
//        -> all-to-all of 16-byte minimizer records
//   2. BuildIndexFrom the received records; IndexHistogram -> all-reduce ->
//        ONE global occurrence threshold per batch (SURVEY.md App. B#3)
//   3. DistHitsSplit     probe + expand the received queries, hits written
//        straight into per-destination runs (owner of the query read)
//        -> all-to-all of seed hits ("minimizer-bucket hits", the north star)
//   4. DistChainOwned    merge the runs by read, chain (the single-GPU kernels)
//   5. DistOverlapsSplit every overlap also goes to the owner of its rhs read
//        -> all-to-all of overlaps (32 B each)
//   6. DistStage1Add     merge by query, then piles + lists of the OWNED reads
//        with the reference's flush schedule; End compacts them for the host.
#include <algorithm>
#include <cstring>

#include "engine.cuh"
#include "seed.cuh"

namespace rvn {

namespace {

constexpr int kThreads = 256;
constexpr uint32_t kMaxParts = 16;

// ---------------------------------------------------------------------------
// stable partition of (value, origin) records by value % parts
// ---------------------------------------------------------------------------
constexpr uint32_t kPartRounds = 8;
constexpr uint32_t kPartTile = kThreads * kPartRounds;

__global__ void __launch_bounds__(kThreads)
PartitionCount(ValView val, uint64_t n, uint32_t parts,
               uint64_t n_tiles, uint32_t* __restrict__ hist) {
  __shared__ uint32_t cnt[kMaxParts];
  if (threadIdx.x < kMaxParts) cnt[threadIdx.x] = 0;
  __syncthreads();
  const uint64_t base = static_cast<uint64_t>(blockIdx.x) * kPartTile;
#pragma unroll
  for (uint32_t r = 0; r < kPartRounds; ++r) {
    const uint64_t i = base + r * kThreads + threadIdx.x;
    const uint32_t owner = i < n ? static_cast<uint32_t>(val[i] % parts) : 0xFFFFFFFFu;
    const uint32_t mask = __match_any_sync(0xFFFFFFFFu, owner);
    if (owner != 0xFFFFFFFFu && (threadIdx.x & 31) == __ffs(mask) - 1) {
      atomicAdd(&cnt[owner], __popc(mask));
    }
  }
  __syncthreads();
  if (threadIdx.x < parts) hist[threadIdx.x * n_tiles + blockIdx.x] = cnt[threadIdx.x];
}

__global__ void __launch_bounds__(kThreads)
PartitionScatter(ValView val, const uint64_t* __restrict__ org,
                 uint64_t n, uint32_t parts, uint64_t n_tiles,
                 const uint64_t* __restrict__ tile_base, uint64_t* __restrict__ out_val,
                 uint64_t* __restrict__ out_org) {
  __shared__ uint32_t warp_cnt[kThreads / 32][kMaxParts];
  __shared__ uint64_t running[kMaxParts];
  const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x < kMaxParts) {
    running[threadIdx.x] =
        threadIdx.x < parts ? tile_base[threadIdx.x * n_tiles + blockIdx.x] : 0;
  }
  const uint64_t base = static_cast<uint64_t>(blockIdx.x) * kPartTile;
  for (uint32_t r = 0; r < kPartRounds; ++r) {
    if (threadIdx.x < (kThreads / 32) * kMaxParts) {
      (&warp_cnt[0][0])[threadIdx.x] = 0;
    }
    __syncthreads();
    const uint64_t i = base + r * kThreads + threadIdx.x;
    uint64_t v = 0, o = 0;
    uint32_t owner = 0xFFFFFFFFu;
    if (i < n) {
      v = val[i];
      o = org[i];
      owner = static_cast<uint32_t>(v % parts);
    }
    const uint32_t mask = __match_any_sync(0xFFFFFFFFu, owner);
    const uint32_t rank = __popc(mask & ((1u << lane) - 1));
    if (owner != 0xFFFFFFFFu && rank == 0) warp_cnt[warp][owner] = __popc(mask);
    __syncthreads();
    if (owner != 0xFFFFFFFFu) {
      uint64_t at = running[owner] + rank;
      for (uint32_t w = 0; w < warp; ++w) at += warp_cnt[w][owner];
      out_val[at] = v;
      out_org[at] = o;
    }
    __syncthreads();
    if (threadIdx.x < parts) {
      uint32_t s = 0;
      for (uint32_t w = 0; w < kThreads / 32; ++w) s += warp_cnt[w][threadIdx.x];
      running[threadIdx.x] += s;
    }
    __syncthreads();
  }
}

// out[p] = src[p * stride] for p in [0, parts]
__global__ void GatherBoundaries(const uint64_t* __restrict__ src, uint64_t stride,
                                 uint32_t parts, uint64_t* __restrict__ out) {
  const uint32_t p = threadIdx.x;
  if (p <= parts) out[p] = src[p * stride];
}

// ---------------------------------------------------------------------------
// seed lookup of received queries, hits written into per-destination runs
// ---------------------------------------------------------------------------
// the received query records are sorted by read id:
// start[r] = first query record of a read >= r, for r in [0, n_reads]
__global__ void QueryReadStarts(const uint64_t* __restrict__ q_org, uint64_t n_q,
                                uint32_t n_reads, uint64_t* __restrict__ start) {
  const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r > n_reads) return;
  uint64_t lo = 0, hi = n_q;
  while (lo < hi) {
    const uint64_t mid = lo + (hi - lo) / 2;
    if (static_cast<uint32_t>(q_org[mid] >> 32) < r) lo = mid + 1; else hi = mid;
  }
  start[r] = lo;
}

// destination-major slot of read r: (r % parts) * per_part + r / parts
__device__ __forceinline__ uint64_t Slot(uint32_t r, uint32_t parts, uint32_t per_part) {
  return static_cast<uint64_t>(r % parts) * per_part + r / parts;
}

__global__ void ReadHitTotals(const uint64_t* __restrict__ start,
                              const uint64_t* __restrict__ hit_off, uint32_t n_reads,
                              uint32_t parts, uint32_t per_part, uint32_t* __restrict__ tot,
                              uint32_t* __restrict__ bad) {
  const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n_reads) return;
  const uint64_t t = hit_off[start[r + 1]] - hit_off[start[r]];
  if (t >= 0x7FFFFFFFULL) *bad = 3;
  tot[Slot(r, parts, per_part)] = static_cast<uint32_t>(t);
}

__global__ void __launch_bounds__(kThreads)
ExpandOwned(IndexView ix, const uint64_t* __restrict__ q_val,
            const uint64_t* __restrict__ q_org, uint64_t n_q, bool ae, bool as,
            const uint32_t* __restrict__ cnt, const uint32_t* __restrict__ first,
            const uint64_t* __restrict__ hit_off, const uint64_t* __restrict__ start,
            const uint64_t* __restrict__ read_base, uint32_t n_reads, uint32_t parts,
            uint32_t per_part, uint64_t* __restrict__ h_grp, uint64_t* __restrict__ h_pos,
            uint32_t* __restrict__ h_lhs, uint32_t* __restrict__ bad) {
  const uint64_t i = static_cast<uint64_t>(blockIdx.x) * kThreads + threadIdx.x;
  if (i >= n_q) return;
  const uint64_t lo = q_org[i];
  const uint32_t lhs_id = static_cast<uint32_t>(lo >> 32);
  if (lhs_id >= n_reads || i < start[lhs_id] || i >= start[lhs_id + 1]) {
    *bad = 2;  // query records not sorted by read (or a read out of range)
    return;
  }
  uint32_t left = cnt[i];
  if (left == 0) return;
  const uint64_t v = q_val[i];
  const uint64_t dst =
      read_base[Slot(lhs_id, parts, per_part)] + (hit_off[i] - hit_off[start[lhs_id]]);
  // (h_lhs is always given: without the hint the shared loop tests it per hit, and its
  //  postings are no longer loaded through the read-only path)
  __builtin_assume(h_lhs != nullptr);
  ExpandQuery(ix, v, lo, first[i], left, ae, as, dst, h_grp, h_pos, h_lhs);
}

// the kept postings are contiguous (seed.cuh): whole warps, coalesced loads
__global__ void __launch_bounds__(kThreads)
ExpandOwnedWarp(IndexView ix, const uint64_t* __restrict__ q_org, uint64_t n_q,
                const uint32_t* __restrict__ cnt, const uint32_t* __restrict__ first,
                const uint64_t* __restrict__ hit_off, const uint64_t* __restrict__ start,
                const uint64_t* __restrict__ read_base, uint32_t n_reads, uint32_t parts,
                uint32_t per_part, uint64_t* __restrict__ h_grp, uint64_t* __restrict__ h_pos,
                uint32_t* __restrict__ h_lhs, uint32_t* __restrict__ bad) {
  const uint64_t i = static_cast<uint64_t>(blockIdx.x) * kThreads + threadIdx.x;
  uint32_t my_cnt = 0, my_first = 0;
  uint64_t my_org = 0, my_dst = 0;
  if (i < n_q) {
    my_org = q_org[i];
    const uint32_t lhs_id = static_cast<uint32_t>(my_org >> 32);
    if (lhs_id >= n_reads || i < start[lhs_id] || i >= start[lhs_id + 1]) {
      *bad = 2;  // query records not sorted by read (or a read out of range)
    } else {
      my_cnt = cnt[i];
      my_first = first[i];
      my_dst = read_base[Slot(lhs_id, parts, per_part)] + (hit_off[i] - hit_off[start[lhs_id]]);
    }
  }
  __builtin_assume(h_lhs != nullptr);  // (see ExpandOwned)
  ExpandWarp(ix.org, my_cnt, my_first, my_org, my_dst, h_grp, h_pos, h_lhs);
}

// ---------------------------------------------------------------------------
// k-way merge of runs sorted by a u32 key (stride = u32 words per record)
// start[p * (nk + 1) + k] = first record of run p with key / div >= k
// ---------------------------------------------------------------------------
__global__ void RunStarts(const uint32_t* __restrict__ keys, uint32_t stride, uint32_t div,
                          const uint64_t* __restrict__ seg_off, uint32_t n_seg, uint32_t nk,
                          uint64_t* __restrict__ start) {
  const uint64_t t = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (t >= static_cast<uint64_t>(n_seg) * (nk + 1ULL)) return;
  const uint32_t p = static_cast<uint32_t>(t / (nk + 1ULL));
  const uint32_t want = static_cast<uint32_t>(t % (nk + 1ULL));
  uint64_t lo = seg_off[p], hi = seg_off[p + 1];
  while (lo < hi) {
    const uint64_t mid = lo + (hi - lo) / 2;
    if (keys[mid * stride] / div < want) lo = mid + 1; else hi = mid;
  }
  start[t] = lo;
}

__global__ void RunCounts(const uint64_t* __restrict__ start, uint32_t n_seg, uint32_t nk,
                          uint32_t* __restrict__ cnt) {
  const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= nk) return;
  uint64_t n = 0;
  for (uint32_t p = 0; p < n_seg; ++p) {
    n += start[p * (nk + 1ULL) + k + 1] - start[p * (nk + 1ULL) + k];
  }
  cnt[k] = static_cast<uint32_t>(n);
}

// base[p][k] = destination of the first record with key k that came in run p
__global__ void RunBases(const uint64_t* __restrict__ start, const uint64_t* __restrict__ koff,
                         uint32_t n_seg, uint32_t nk, uint64_t* __restrict__ base) {
  const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= nk) return;
  uint64_t at = koff[k];
  for (uint32_t p = 0; p < n_seg; ++p) {
    base[p * (nk + 1ULL) + k] = at;
    at += start[p * (nk + 1ULL) + k + 1] - start[p * (nk + 1ULL) + k];
  }
}

__device__ __forceinline__ bool MergeSlot(const uint32_t* keys, uint32_t stride, uint32_t div,
                                          uint32_t mod, uint32_t rem,
                                          const uint64_t* seg_off, uint32_t n_seg, uint32_t nk,
                                          const uint64_t* start, const uint64_t* base,
                                          uint64_t i, uint64_t* at, uint32_t* bad) {
  uint32_t p = 0;
  while (p + 1 < n_seg && i >= seg_off[p + 1]) ++p;
  const uint32_t id = keys[i * stride];
  if (id % mod != rem || id / div >= nk) {
    *bad = 1;  // a record of a read this rank does not own
    return false;
  }
  const uint64_t s = p * (nk + 1ULL) + id / div;
  if (i < start[s] || i >= start[s + 1]) {
    *bad = 2;  // run not sorted by key
    return false;
  }
  *at = base[s] + (i - start[s]);
  return true;
}

// (a read's hits end up run after run; the chain result is a function of the
// hit multiset, and its cost was measured insensitive to this order)
__global__ void MergeHits(const uint64_t* __restrict__ grp, const uint64_t* __restrict__ pos,
                          const uint32_t* __restrict__ lhs, uint32_t mod, uint32_t rem,
                          const uint64_t* __restrict__ seg_off, uint32_t n_seg, uint32_t nk,
                          const uint64_t* __restrict__ start, const uint64_t* __restrict__ base,
                          uint64_t n, uint64_t* __restrict__ out_grp,
                          uint64_t* __restrict__ out_pos, uint32_t* __restrict__ bad) {
  const uint64_t i = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint64_t at;
  if (!MergeSlot(lhs, 1, mod, mod, rem, seg_off, n_seg, nk, start, base, i, &at, bad)) return;
  out_grp[at] = grp[i];
  out_pos[at] = pos[i];
}

// two threads per 32-byte overlap record, keyed by lhs_id (word 0)
__global__ void MergeOverlaps(const rvn_overlap* __restrict__ in,
                              const uint64_t* __restrict__ seg_off, uint32_t n_seg,
                              uint32_t nk, const uint64_t* __restrict__ start,
                              const uint64_t* __restrict__ base, uint64_t n,
                              rvn_overlap* __restrict__ out, uint32_t* __restrict__ bad) {
  const uint64_t t = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  const uint64_t i = t >> 1;
  if (i >= n) return;
  uint64_t at;
  if (!MergeSlot(reinterpret_cast<const uint32_t*>(in), 8, 1, 1, 0, seg_off, n_seg, nk, start,
                 base, i, &at, bad)) {
    return;
  }
  reinterpret_cast<uint4*>(out + at)[t & 1] = reinterpret_cast<const uint4*>(in + i)[t & 1];
}

__global__ void StridedIds(const uint32_t* __restrict__ ids, uint32_t mod, uint32_t rem,
                           uint32_t n, uint32_t* __restrict__ out) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = ids[rem + static_cast<uint64_t>(i) * mod];
}

// ---------------------------------------------------------------------------
// overlaps -> destination runs: part d gets the overlaps whose rhs read it
// owns, the own part (self) gets every overlap
// ---------------------------------------------------------------------------
__global__ void OverlapFlags(const rvn_overlap* __restrict__ ovl, uint64_t n, uint32_t parts,
                             uint32_t p, uint32_t self, uint32_t* __restrict__ flag) {
  const uint64_t i = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  flag[i] = (p == self || ovl[i].rhs_id % parts == p) ? 1u : 0u;
}

__global__ void OverlapScatter(const rvn_overlap* __restrict__ ovl,
                               const uint32_t* __restrict__ flag,
                               const uint64_t* __restrict__ pos, uint64_t n, uint64_t base,
                               rvn_overlap* __restrict__ out) {
  const uint64_t t = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  const uint64_t i = t >> 1;
  if (i >= n || !flag[i]) return;
  reinterpret_cast<uint4*>(out + base + pos[i])[t & 1] =
      reinterpret_cast<const uint4*>(ovl + i)[t & 1];
}

__global__ void RelativeOffsets(const uint64_t* __restrict__ off, uint32_t k0, uint32_t n,
                                uint64_t* __restrict__ rel) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) rel[i] = off[k0 + i] - off[k0];
}

// ---------------------------------------------------------------------------
// results of the owned reads, compacted for the host
// ---------------------------------------------------------------------------
__global__ void OwnedCounts(const uint32_t* __restrict__ cnt, uint32_t mod, uint32_t rem,
                            uint32_t n_own, uint32_t* __restrict__ out) {
  const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j < n_own) out[j] = cnt[rem + static_cast<uint64_t>(j) * mod];
}

__global__ void __launch_bounds__(kThreads)
OwnedLists(const rvn_overlap* __restrict__ lists, const uint64_t* __restrict__ g_off,
           const uint32_t* __restrict__ cnt, uint32_t mod, uint32_t rem, uint32_t n_own,
           const uint64_t* __restrict__ own_off, rvn_overlap* __restrict__ out) {
  const uint32_t j = blockIdx.x * (kThreads / 32) + (threadIdx.x >> 5);
  if (j >= n_own) return;
  const uint64_t r = rem + static_cast<uint64_t>(j) * mod;
  const uint4* s = reinterpret_cast<const uint4*>(lists + g_off[r]);
  uint4* d = reinterpret_cast<uint4*>(out + own_off[j]);
  for (uint32_t i = threadIdx.x & 31; i < cnt[r] * 2; i += 32) d[i] = s[i];
}

__global__ void __launch_bounds__(kThreads)
OwnedPiles(const uint16_t* __restrict__ data, const uint64_t* __restrict__ bin_off,
           uint32_t mod, uint32_t rem, uint32_t n_own, const uint64_t* __restrict__ own_off,
           uint16_t* __restrict__ out) {
  const uint32_t j = blockIdx.x * (kThreads / 32) + (threadIdx.x >> 5);
  if (j >= n_own) return;
  const uint64_t r = rem + static_cast<uint64_t>(j) * mod;
  const uint64_t b = bin_off[r], bins = bin_off[r + 1] - b;
  for (uint64_t i = threadIdx.x & 31; i < bins; i += 32) out[own_off[j] + i] = data[b + i];
}

void CheckParts(uint32_t parts, uint32_t rank) {
  if (parts == 0 || parts > kMaxParts) throw InvalidArgument("1..16 partitions");
  if (rank >= parts) throw InvalidArgument("rank outside the partition");
}

uint32_t OwnedBelow(uint32_t n, uint32_t mod, uint32_t rem) {
  return n > rem ? (n - rem + mod - 1) / mod : 0;
}

void ThrowBad(uint32_t bad) {
  if (bad == 1) throw InvalidArgument("a record belongs to a read this rank does not own");
  if (bad == 2) throw InvalidArgument("records must arrive sorted by query read");
  if (bad == 3) throw LimitError("a query has 2^31 or more hits");
}

}  // namespace

void DistSketchSplit(Ctx& c, uint32_t first, uint32_t last, int which, uint32_t parts,
                     const uint64_t** d_val, const uint64_t** d_org, uint64_t* counts) {
  CheckParts(parts, 0);
  EnsureSketch(c, first, last);
  ValView sv{c.s_val.get(), c.s_is32 ? 1 : 0};
  const uint64_t* so = c.s_org.get();
  uint64_t n = c.s_n;
  if (which == 1) {
    EnsureMicromizers(c, first, last);
    sv = ValView{c.q_val.get(), c.q_is32 ? 1 : 0};
    so = c.q_org.get();
    n = c.q_n;
  }
  if ((parts == 1 && !sv.is32) || n == 0) {  // nothing to move
    for (uint32_t p = 0; p < parts; ++p) counts[p] = 0;
    counts[0] = n;
    *d_val = static_cast<const uint64_t*>(sv.p);
    *d_org = so;
    return;
  }
  // (one part with u32 sketch values: the partition below is the widening copy
  //  to the 16-byte exchange format)
  DevBuf<uint64_t>& ov = which == 1 ? c.ds_qsplit_val : c.ds_split_val;
  DevBuf<uint64_t>& oo = which == 1 ? c.ds_qsplit_org : c.ds_split_org;
  uint64_t* out_val = ov.reserve(n + 1);
  uint64_t* out_org = oo.reserve(n + 1);
  const uint64_t n_tiles = CeilDiv(n, kPartTile);
  if (n_tiles >= 0x7FFFFFFFULL) throw LimitError("too many partition tiles");
  uint32_t* hist = c.m_cnt.reserve(parts * n_tiles + 1);
  uint64_t* base = c.m_hit_off.reserve(parts * n_tiles + 2);
  uint64_t* bnd = c.ds_bounds.reserve(64 + 2);
  TimerBegin(c, "dist_split");
  PartitionCount<<<static_cast<unsigned>(n_tiles), kThreads, 0, c.stream>>>(sv, n, parts,
                                                                           n_tiles, hist);
  ExclusiveScanU32(c, hist, base, parts * n_tiles);
  GatherBoundaries<<<1, 32, 0, c.stream>>>(base, n_tiles, parts, bnd);
  PartitionScatter<<<static_cast<unsigned>(n_tiles), kThreads, 0, c.stream>>>(
      sv, so, n, parts, n_tiles, base, out_val, out_org);
  RVN_LAUNCH_CHECK();
  c.launches += 3;
  TimerEnd(c);
  uint64_t h_bnd[kMaxParts + 1];
  RVN_CUDA(cudaMemcpyAsync(h_bnd, bnd, (parts + 1) * 8, cudaMemcpyDeviceToHost, c.stream));
  RVN_CUDA(cudaStreamSynchronize(c.stream));
  for (uint32_t p = 0; p < parts; ++p) counts[p] = h_bnd[p + 1] - h_bnd[p];
  *d_val = out_val;
  *d_org = out_org;
}

void DistHitsSplit(Ctx& c, const uint64_t* d_qval, const uint64_t* d_qorg, uint64_t n_q,
                   bool ae, bool as, uint32_t parts, uint32_t n_query,
                   const uint64_t** d_grp, const uint64_t** d_pos, const uint32_t** d_lhs,
                   uint64_t* counts) {
  if (!c.i_valid) throw StateError("no index");
  CheckParts(parts, 0);
  if (n_query > c.n_reads) throw InvalidArgument("query range out of bounds");
  const IndexView ix = IndexViewOf(c);
  const uint32_t per_part = CeilDiv(n_query, parts);
  const uint64_t slots = static_cast<uint64_t>(per_part) * parts;
  uint32_t* cnt = c.m_cnt.reserve(n_q + 1);
  uint32_t* frst = c.m_first.reserve(n_q + 1);
  uint64_t* off = c.m_hit_off.reserve(n_q + 2);
  uint64_t* start = c.ds_seg_start.reserve(n_query + 2ULL);
  uint32_t* tot = c.ds_masked.reserve(slots + 1);
  uint64_t* rbase = c.ds_seg_base.reserve(slots + 2);
  uint64_t* bnd = c.ds_bounds.reserve(64 + 2);
  uint32_t* bad = c.ds_flag.reserve(4);
  RVN_CUDA(cudaMemsetAsync(bad, 0, 4, c.stream));
  RVN_CUDA(cudaMemsetAsync(tot, 0, (slots + 1) * 4, c.stream));
  TimerBegin(c, "probe");
  ProbeQueries(c, ValView{d_qval, 0}, d_qorg, 0, n_q, ae, as, cnt, frst, nullptr);
  ExclusiveScanU32(c, cnt, off, n_q);
  TimerEnd(c);
  TimerBegin(c, "expand");
  QueryReadStarts<<<CeilDiv(n_query + 1ULL, kThreads), kThreads, 0, c.stream>>>(d_qorg, n_q,
                                                                               n_query, start);
  if (n_query) {
    ReadHitTotals<<<CeilDiv(n_query, kThreads), kThreads, 0, c.stream>>>(
        start, off, n_query, parts, per_part, tot, bad);
  }
  ExclusiveScanU32(c, tot, rbase, slots);
  GatherBoundaries<<<1, 32, 0, c.stream>>>(rbase, per_part, parts, bnd);
  RVN_LAUNCH_CHECK();
  c.launches += 3;
  uint64_t h_bnd[kMaxParts + 1];
  RVN_CUDA(cudaMemcpyAsync(h_bnd, bnd, (parts + 1) * 8, cudaMemcpyDeviceToHost, c.stream));
  RVN_CUDA(cudaStreamSynchronize(c.stream));
  const uint64_t n_hits = h_bnd[parts];
  uint64_t* hg = c.h_grp.reserve(n_hits + 1);
  uint64_t* hp = c.h_pos.reserve(n_hits + 1);
  uint32_t* hl = c.ds_hit_lhs.reserve(n_hits + 1);
  if (n_q) {
    if (KeptContiguous(c, ae, as)) {
      ExpandOwnedWarp<<<CeilDiv(n_q, kThreads), kThreads, 0, c.stream>>>(
          ix, d_qorg, n_q, cnt, frst, off, start, rbase, n_query, parts, per_part, hg, hp, hl, bad);
    } else {
      ExpandOwned<<<CeilDiv(n_q, kThreads), kThreads, 0, c.stream>>>(
          ix, d_qval, d_qorg, n_q, ae, as, cnt, frst, off, start, rbase, n_query, parts,
          per_part, hg, hp, hl, bad);
    }
    RVN_LAUNCH_CHECK();
    ++c.launches;
  }
  TimerEnd(c);
  uint32_t h_bad = 0;
  RVN_CUDA(cudaMemcpyAsync(&h_bad, bad, 4, cudaMemcpyDeviceToHost, c.stream));
  RVN_CUDA(cudaStreamSynchronize(c.stream));
  ThrowBad(h_bad);
  for (uint32_t p = 0; p < parts; ++p) counts[p] = h_bnd[p + 1] - h_bnd[p];
  c.stats.query_records += n_q;
  c.stats.hits += n_hits;
  *d_grp = hg;
  *d_pos = hp;
  *d_lhs = hl;
}

// hits of the owned reads (r % mod == rem, r < n_query) as n_seg runs, each
// sorted by query read (what the all-to-all delivers) -> overlaps in query order
void DistChainOwned(Ctx& c, const uint64_t* d_grp, const uint64_t* d_pos,
                    const uint32_t* d_lhs, uint64_t n_hits, uint32_t n_seg,
                    const uint64_t* h_seg_off, uint32_t mod, uint32_t rem, uint32_t n_query,
                    const rvn_overlap** d_ovl, uint64_t* n_ovl) {
  CheckParts(mod, rem);
  if (n_query > c.n_reads) throw InvalidArgument("query range out of bounds");
  if (n_seg == 0 || n_seg > 64) throw InvalidArgument("1..64 hit runs");
  if (h_seg_off[0] != 0 || h_seg_off[n_seg] != n_hits) {
    throw InvalidArgument("run offsets do not cover the hits");
  }
  const uint32_t nr = OwnedBelow(n_query, mod, rem);
  TimerBegin(c, "dist_merge");
  uint32_t* rcnt = c.ds_read_cnt.reserve(nr + 2ULL);
  uint64_t* roff = c.m_read_hit_off.reserve(nr + 2ULL);
  uint64_t* gg = c.ds_grouped_grp.reserve(n_hits + 1);
  uint64_t* gp = c.ds_grouped_pos.reserve(n_hits + 1);
  const uint64_t cells = static_cast<uint64_t>(n_seg) * (nr + 1ULL);
  uint64_t* start = c.ds_seg_start.reserve(cells + 1);
  uint64_t* base = c.ds_seg_base.reserve(cells + 1);
  uint64_t* d_seg = c.ds_bounds.reserve(64 + 2);
  uint32_t* ids = c.ds_own_ids.reserve(nr + 1ULL);
  uint32_t* bad = c.ds_flag.reserve(4);
  RVN_CUDA(cudaMemcpyAsync(d_seg, h_seg_off, (n_seg + 1ULL) * 8, cudaMemcpyHostToDevice,
                           c.stream));
  RVN_CUDA(cudaMemsetAsync(bad, 0, 4, c.stream));
  RVN_CUDA(cudaMemsetAsync(rcnt, 0, (nr + 1ULL) * 4, c.stream));
  RunStarts<<<CeilDiv(cells, kThreads), kThreads, 0, c.stream>>>(d_lhs, 1, mod, d_seg, n_seg, nr,
                                                               start);
  if (nr) {
    RunCounts<<<CeilDiv(nr, kThreads), kThreads, 0, c.stream>>>(start, n_seg, nr, rcnt);
    StridedIds<<<CeilDiv(nr, kThreads), kThreads, 0, c.stream>>>(c.d_ids.get(), mod, rem, nr, ids);
  }
  ExclusiveScanU32(c, rcnt, roff, nr);
  if (nr) {
    RunBases<<<CeilDiv(nr, kThreads), kThreads, 0, c.stream>>>(start, roff, n_seg, nr, base);
  }
  if (n_hits) {
    MergeHits<<<CeilDiv(n_hits, kThreads), kThreads, 0, c.stream>>>(
        d_grp, d_pos, d_lhs, mod, rem, d_seg, n_seg, nr, start, base, n_hits, gg, gp, bad);
  }
  RVN_LAUNCH_CHECK();
  c.launches += 5;
  uint32_t h_bad = 0;
  RVN_CUDA(cudaMemcpyAsync(&h_bad, bad, 4, cudaMemcpyDeviceToHost, c.stream));
  std::vector<uint64_t> h_rho(nr + 1ULL);
  RVN_CUDA(cudaMemcpyAsync(h_rho.data(), roff, (nr + 1ULL) * 8, cudaMemcpyDeviceToHost, c.stream));
  RVN_CUDA(cudaStreamSynchronize(c.stream));
  TimerEnd(c);
  ThrowBad(h_bad);
  const uint64_t n = ChainGroupedHits(c, gg, gp, roff, h_rho, ids, nr, n_hits, 0);
  RVN_CUDA(cudaStreamSynchronize(c.stream));
  uint64_t qbases = 0;
  for (uint64_t r = rem; r < n_query; r += mod) qbases += c.h_len[r];
  c.stats.query_bases += qbases;
  c.stats.overlaps += n;
  c.r_n_ovl = n;
  *d_ovl = c.m_ovl.get();
  *n_ovl = n;
}

// the overlaps of the last DistChainOwned as `parts` runs: run d != self holds
// the overlaps whose rhs read d owns, run self holds all of them
void DistOverlapsSplit(Ctx& c, uint32_t parts, uint32_t self, const rvn_overlap** d_out,
                       uint64_t* counts) {
  CheckParts(parts, self);
  const uint64_t n = c.r_n_ovl;
  const rvn_overlap* ovl = c.m_ovl.get();
  if (parts == 1 || n == 0) {
    for (uint32_t p = 0; p < parts; ++p) counts[p] = 0;
    counts[self] = n;
    *d_out = ovl;
    return;
  }
  rvn_overlap* out = c.ds_ovl_split.reserve(2 * n + 1);
  uint32_t* flag = c.m_cnt.reserve(n + 1);
  uint64_t* pos = c.m_hit_off.reserve(n + 2);
  TimerBegin(c, "dist_ovl_split");
  uint64_t base = 0;
  for (uint32_t p = 0; p < parts; ++p) {
    OverlapFlags<<<CeilDiv(n, kThreads), kThreads, 0, c.stream>>>(ovl, n, parts, p, self, flag);
    ExclusiveScanU32(c, flag, pos, n);
    const uint64_t cnt = ReadU64(c, pos + n);
    OverlapScatter<<<CeilDiv(2 * n, kThreads), kThreads, 0, c.stream>>>(ovl, flag, pos, n, base,
                                                                       out);
    RVN_LAUNCH_CHECK();
    c.launches += 2;
    counts[p] = cnt;
    base += cnt;
  }
  TimerEnd(c);
  RVN_CUDA(cudaStreamSynchronize(c.stream));
  *d_out = out;
}

// ---- stage-1 tail of the owned reads (construct.cc:51-112) ----
void DistStage1Begin(Ctx& c, uint32_t parts, uint32_t rank) {
  CheckParts(parts, rank);
  if (!c.ids_identity) throw StateError("stage 1 needs read ids equal to their index");
  c.own_mod = parts;
  c.own_rem = rank;
  c.ds_results_valid = false;
  const uint32_t n = c.n_reads;
  c.st_valid = false;
  c.st_pile_off.assign(n + 1ULL, 0);
  for (uint32_t i = 0; i < n; ++i) c.st_pile_off[i + 1] = c.st_pile_off[i] + (c.h_len[i] >> 4);
  const uint64_t total_bins = c.st_pile_off[n];
  uint16_t* d_pile = c.p_data.reserve(total_bins + 1);
  uint64_t* d_poff = c.p_off.reserve(n + 1ULL);
  RVN_CUDA(cudaMemsetAsync(d_pile, 0, (total_bins + 1) * 2, c.stream));
  RVN_CUDA(cudaMemcpyAsync(d_poff, c.st_pile_off.data(), (n + 1ULL) * 8, cudaMemcpyHostToDevice,
                           c.stream));
  GatherReset(c);
  c.st_mapped = 0;
}

// `d_ovl`: n_seg runs (h_seg_off), each sorted by query (lhs) read: every overlap
// of one index batch that touches an owned read, queries [0, n_query)
void DistStage1Add(Ctx& c, const rvn_overlap* d_ovl, uint64_t n_ovl, uint32_t n_seg,
                   const uint64_t* h_seg_off, uint32_t n_query, uint64_t kmax, uint64_t qb) {
  if (qb == 0) qb = 1ULL << 30;
  if (n_query > c.n_reads) throw InvalidArgument("query range out of bounds");
  if (n_seg == 0 || n_seg > 64) throw InvalidArgument("1..64 overlap runs");
  if (h_seg_off[0] != 0 || h_seg_off[n_seg] != n_ovl) {
    throw InvalidArgument("run offsets do not cover the overlaps");
  }
  const uint32_t n = c.n_reads;
  // ---- merge the runs into global query order, offsets per query ----
  TimerBegin(c, "dist_merge");
  const uint64_t cells = static_cast<uint64_t>(n_seg) * (n_query + 1ULL);
  uint64_t* start = c.ds_seg_start.reserve(cells + 1);
  uint64_t* base = c.ds_seg_base.reserve(cells + 1);
  uint64_t* d_seg = c.ds_bounds.reserve(64 + 2);
  uint32_t* qcnt = c.ds_read_cnt.reserve(n_query + 2ULL);
  uint64_t* qoff = c.ds_q_off.reserve(n_query + 2ULL);
  uint32_t* bad = c.ds_flag.reserve(4);
  rvn_overlap* merged = c.ds_merged.reserve(n_ovl + 1);
  RVN_CUDA(cudaMemcpyAsync(d_seg, h_seg_off, (n_seg + 1ULL) * 8, cudaMemcpyHostToDevice,
                           c.stream));
  RVN_CUDA(cudaMemsetAsync(bad, 0, 4, c.stream));
  RVN_CUDA(cudaMemsetAsync(qcnt, 0, (n_query + 1ULL) * 4, c.stream));
  RunStarts<<<CeilDiv(cells, kThreads), kThreads, 0, c.stream>>>(
      reinterpret_cast<const uint32_t*>(d_ovl), 8, 1, d_seg, n_seg, n_query, start);
  if (n_query) {
    RunCounts<<<CeilDiv(n_query, kThreads), kThreads, 0, c.stream>>>(start, n_seg, n_query, qcnt);
  }
  ExclusiveScanU32(c, qcnt, qoff, n_query);
  if (n_query) {
    RunBases<<<CeilDiv(n_query, kThreads), kThreads, 0, c.stream>>>(start, qoff, n_seg, n_query,
                                                                   base);
  }
  if (n_ovl) {
    MergeOverlaps<<<CeilDiv(2 * n_ovl, kThreads), kThreads, 0, c.stream>>>(
        d_ovl, d_seg, n_seg, n_query, start, base, n_ovl, merged, bad);
  }
  RVN_LAUNCH_CHECK();
  c.launches += 4;
  uint32_t h_bad = 0;
  RVN_CUDA(cudaMemcpyAsync(&h_bad, bad, 4, cudaMemcpyDeviceToHost, c.stream));
  std::vector<uint64_t> h_off(n_query + 1ULL);
  RVN_CUDA(cudaMemcpyAsync(h_off.data(), qoff, (n_query + 1ULL) * 8, cudaMemcpyDeviceToHost,
                           c.stream));
  RVN_CUDA(cudaStreamSynchronize(c.stream));
  TimerEnd(c);
  ThrowBad(h_bad);
  if (h_off[n_query] != n_ovl) throw InvalidArgument("an overlap of a query outside the batch");

  // ---- the reference's flush schedule over the merged list ----
  uint64_t* d_rel = c.ds_rel_off.reserve(n + 2ULL);
  uint64_t bases = 0;
  for (uint32_t k = 0, k0 = 0; k < n_query; ++k) {
    bases += c.h_len[k];
    if (k != n_query - 1 && bases < qb) continue;
    bases = 0;
    const uint64_t b = h_off[k0], e = h_off[k + 1];
    if (e > b) {
      RelativeOffsets<<<CeilDiv(k + 2 - k0, kThreads), kThreads, 0, c.stream>>>(qoff, k0,
                                                                              k + 2 - k0, d_rel);
      PileAddLayersDevice(c, c.p_data.get(), c.p_off.get(), c.st_pile_off.data(), n, merged + b,
                          e - b);
      GatherFlush(c, merged + b, d_rel, e - b, k0, k + 1, kmax);
    }
    k0 = k + 1;
  }
}

void DistStage1End(Ctx& c) {
  const uint32_t n = c.n_reads, mod = c.own_mod, rem = c.own_rem;
  const uint32_t n_own = OwnedBelow(n, mod, rem);
  TimerBegin(c, "dist_results");
  // lists of the owned reads
  uint32_t* ocnt = c.ds_read_cnt.reserve(n_own + 2ULL);
  uint64_t* ooff = c.ds_q_off.reserve(n_own + 2ULL);
  RVN_CUDA(cudaMemsetAsync(ocnt, 0, (n_own + 1ULL) * 4, c.stream));
  if (n_own) {
    OwnedCounts<<<CeilDiv(n_own, kThreads), kThreads, 0, c.stream>>>(c.g_cnt.get(), mod, rem,
                                                                   n_own, ocnt);
  }
  ExclusiveScanU32(c, ocnt, ooff, n_own);
  const uint64_t n_kept = ReadU64(c, ooff + n_own);
  rvn_overlap* d_lists = c.ds_merged.reserve(n_kept + 1);
  if (n_own && n_kept) {
    OwnedLists<<<CeilDiv(n_own, kThreads / 32), kThreads, 0, c.stream>>>(
        c.g_list[c.g_cur].get(), c.g_off.get(), c.g_cnt.get(), mod, rem, n_own, ooff, d_lists);
  }
  // piles of the owned reads
  uint64_t* h_poff = c.ds_r_pile_off.reserve(n_own + 1ULL);
  h_poff[0] = 0;
  for (uint32_t j = 0; j < n_own; ++j) {
    h_poff[j + 1] = h_poff[j] + (c.h_len[rem + static_cast<uint64_t>(j) * mod] >> 4);
  }
  const uint64_t own_bins = h_poff[n_own];
  uint64_t* d_poff = c.ds_rel_off.reserve(std::max<uint64_t>(n_own + 2ULL, n + 2ULL));
  uint16_t* d_piles = reinterpret_cast<uint16_t*>(c.ds_grouped_grp.reserve(own_bins / 4 + 2));
  RVN_CUDA(cudaMemcpyAsync(d_poff, h_poff, (n_own + 1ULL) * 8, cudaMemcpyHostToDevice, c.stream));
  if (n_own) {
    OwnedPiles<<<CeilDiv(n_own, kThreads / 32), kThreads, 0, c.stream>>>(
        c.p_data.get(), c.p_off.get(), mod, rem, n_own, d_poff, d_piles);
  }
  RVN_LAUNCH_CHECK();
  c.launches += 3;
  rvn_overlap* h_lists = c.ds_r_ovl.reserve(n_kept + 1);
  uint64_t* h_ooff = c.ds_r_ovl_off.reserve(n_own + 1ULL);
  uint16_t* h_piles = c.ds_r_pile.reserve(own_bins + 1);
  RVN_CUDA(cudaMemcpyAsync(h_ooff, ooff, (n_own + 1ULL) * 8, cudaMemcpyDeviceToHost, c.stream));
  if (n_kept) {
    RVN_CUDA(cudaMemcpyAsync(h_lists, d_lists, n_kept * sizeof(rvn_overlap),
                             cudaMemcpyDeviceToHost, c.stream));
  }
  if (own_bins) {
    RVN_CUDA(cudaMemcpyAsync(h_piles, d_piles, own_bins * 2, cudaMemcpyDeviceToHost, c.stream));
  }
  TimerEnd(c);
  RVN_CUDA(cudaStreamSynchronize(c.stream));
  c.ds_n_own = n_own;
  c.st_mapped = c.stats.overlaps;
  TimerCollect(c);
  c.stats.occurrence = c.occurrence;
  c.ds_results_valid = true;
  c.own_mod = 1;
  c.own_rem = 0;
}

// ---------------------------------------------------------------------------
// Peer-memory exchange: every rank owns a receive arena that its peers map
// through CUDA IPC; an all-to-all is then one DMA write per (array, peer)
// straight into the destination's arena over NVLink (copy engines, no staging,
// no NCCL). The caller (raven_b200/distributed.py: P2PComm) agrees on the
// layout from the exchanged count matrix and brackets the writes with barriers.
// ---------------------------------------------------------------------------
void ArenaClosePeers(Ctx& c) {
  for (uint32_t p = 0; p < c.x_peers.size(); ++p) {
    if (p != c.x_rank && c.x_peers[p]) cudaIpcCloseMemHandle(c.x_peers[p]);
  }
  c.x_peers.clear();
}

void ArenaExport(Ctx& c, uint64_t bytes, void* handle64) {
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
  ArenaClosePeers(c);
  if (c.x_arena) {
    RVN_CUDA(cudaFree(c.x_arena));
    c.x_arena = nullptr;
    c.x_cap = 0;
  }
  if (bytes == 0) throw InvalidArgument("empty arena");
  RVN_CUDA(cudaMalloc(&c.x_arena, bytes));
  c.x_cap = bytes;
  cudaIpcMemHandle_t h;
  RVN_CUDA(cudaIpcGetMemHandle(&h, c.x_arena));
  std::memcpy(handle64, &h, 64);
}

void ArenaImport(Ctx& c, uint32_t parts, uint32_t rank, const void* handles) {
  CheckParts(parts, rank);
  if (!c.x_arena) throw StateError("export the arena first");
  ArenaClosePeers(c);
  c.x_rank = rank;
  c.x_peers.assign(parts, nullptr);
  for (uint32_t p = 0; p < parts; ++p) {
    if (p == rank) {
      c.x_peers[p] = c.x_arena;
      continue;
    }
    cudaIpcMemHandle_t h;
    std::memcpy(&h, static_cast<const char*>(handles) + 64ULL * p, 64);
    RVN_CUDA(cudaIpcOpenMemHandle(&c.x_peers[p], h, cudaIpcMemLazyEnablePeerAccess));
  }
  while (c.x_streams.size() < parts) {
    cudaStream_t st;
    RVN_CUDA(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
    c.x_streams.push_back(st);
  }
}

void ArenaPut(Ctx& c, uint32_t dest, uint64_t dst_off, const void* d_src, uint64_t bytes) {
  if (dest >= c.x_peers.size() || !c.x_peers[dest]) throw StateError("no such peer arena");
  if (bytes == 0) return;
  if (!d_src) throw InvalidArgument("null source");
  RVN_CUDA(cudaMemcpyAsync(static_cast<char*>(c.x_peers[dest]) + dst_off, d_src, bytes,
                           cudaMemcpyDefault, c.x_streams[dest]));
}

void ArenaFlush(Ctx& c) {
  for (auto st : c.x_streams) RVN_CUDA(cudaStreamSynchronize(st));
}

void ArenaRelease(Ctx& c) {
  ArenaClosePeers(c);
  if (c.x_arena) cudaFree(c.x_arena);
  c.x_arena = nullptr;
  c.x_cap = 0;
  for (auto st : c.x_streams) cudaStreamDestroy(st);
  c.x_streams.clear();
}

}  // namespace rvn
