// raven_b200 — seed lookup, hit expansion and chaining on sm_100a.
//
// Replaces ram::MinimizerEngine::Map + Chain (un-vendored; call sites
// RavenLib/src/construct.cc:59-64 -> Map(seq,1,1,1) and :377-381 ->
// Map(seq,1,1,0,&filtered); algorithm SURVEY.md App. A.2).
//
//   probe, expand   see seed.cuh
//   chain   ONE CTA PER QUERY READ, hits resident in shared memory:
//           bitonic sort by (group, positions) -> diagonal-band intervals by
//           binary searches + block scans -> second sort by (band, positions)
//           -> one thread per band runs ram's patience/LIS with its exact
//           binary-search predicate, gap split and covered-bases test ->
//           overlaps written through a reserved slab, then re-ordered by
//           query id so that the output order equals the reference's.
//   Reads whose hits do not fit in shared memory take the same code path
//   over a global-memory scratch slab.
//
// The chain result is a pure function of the MULTISET of hits of a query
// (both reference sorts are total orders here: equal (group, positions)
// pairs cannot occur), so hit generation order is free (DESIGN.md).
#include <algorithm>

#include "engine.cuh"
#include "seed.cuh"

namespace rvn {

namespace {

constexpr int kThreads = 256;

__global__ void __launch_bounds__(kThreads)
ProbeKernel(IndexView ix, ValView q_val,
            const uint64_t* __restrict__ q_org, uint64_t q_begin, uint64_t n_q,
            bool avoid_equal, bool avoid_symmetric,
            uint32_t* __restrict__ cnt, uint32_t* __restrict__ first,
            uint8_t* __restrict__ filt) {
  const uint64_t i = static_cast<uint64_t>(blockIdx.x) * kThreads + threadIdx.x;
  if (i >= n_q) return;
  uint32_t f, kept;
  const bool over = Probe(ix, q_val[q_begin + i], [&] { return static_cast<uint32_t>(q_org[q_begin + i] >> 32); },
                          Kept::kFiltered, avoid_equal, avoid_symmetric, &f, &kept);
  cnt[i] = kept;
  first[i] = f;
  if (filt) filt[i] = over;
  // the posting count is re-derived in ExpandKernel from the run itself
}

__global__ void __launch_bounds__(kThreads)
ExpandKernel(IndexView ix, ValView q_val,
             const uint64_t* __restrict__ q_org, uint64_t q_begin, uint64_t n_q,
             bool avoid_equal, bool avoid_symmetric,
             const uint32_t* __restrict__ cnt,
             const uint32_t* __restrict__ first,
             const uint64_t* __restrict__ hit_off, uint64_t* __restrict__ h_grp,
             uint64_t* __restrict__ h_pos) {
  const uint64_t i = static_cast<uint64_t>(blockIdx.x) * kThreads + threadIdx.x;
  if (i >= n_q) return;
  const uint32_t left = cnt[i];
  if (left == 0) return;
  ExpandQuery(ix, q_val[q_begin + i], q_org[q_begin + i], first[i], left, avoid_equal,
              avoid_symmetric, hit_off[i], h_grp, h_pos, nullptr);
}

// ---- fast path of probe + expand: the kept postings are contiguous ----
// strict_above: they are the suffix rhs_id > lhs_id, else the whole run
__global__ void __launch_bounds__(kThreads)
ProbeSuffixKernel(IndexView ix, ValView q_val,
                  const uint64_t* __restrict__ q_org, uint64_t q_begin, uint64_t n_q,
                  bool strict_above, uint32_t* __restrict__ cnt,
                  uint32_t* __restrict__ first, uint8_t* __restrict__ filt) {
  const uint64_t i = static_cast<uint64_t>(blockIdx.x) * kThreads + threadIdx.x;
  if (i >= n_q) return;
  uint32_t fk, kept;
  const bool over = Probe(ix, q_val[q_begin + i], [&] { return static_cast<uint32_t>(q_org[q_begin + i] >> 32); },
                          strict_above ? Kept::kSuffix : Kept::kWholeRun, true, true, &fk, &kept);
  cnt[i] = kept;
  first[i] = fk;
  if (filt) filt[i] = over;
}

// the same probe over queries sorted by value: neighbouring threads walk
// neighbouring parts of the bucket table and of the postings (coalesced,
// TLB-friendly) instead of 67 M independent random probes into 12 GB
__global__ void __launch_bounds__(kThreads)
ProbeSortedKernel(IndexView ix, ValView sorted_val,
                  const uint32_t* __restrict__ sorted_idx,
                  const uint64_t* __restrict__ q_org, uint64_t q_begin, uint64_t n_q,
                  bool strict_above, uint64_t* __restrict__ packed) {
  const uint64_t t = static_cast<uint64_t>(blockIdx.x) * kThreads + threadIdx.x;
  if (t >= n_q) return;
  const uint32_t i = sorted_idx[t];
  uint32_t fk, kept;
  const bool over = Probe(ix, sorted_val[t], [&] { return static_cast<uint32_t>(q_org[q_begin + i] >> 32); },
                          strict_above ? Kept::kSuffix : Kept::kWholeRun, true, true, &fk, &kept);
  // ONE scattered store per query (a partial-sector write costs a read-modify-
  // write in HBM): first kept posting | over-threshold flag | kept count
  packed[i] = (static_cast<uint64_t>(fk) << 32) | (static_cast<uint64_t>(over) << 31) | kept;
}

__global__ void UnpackProbe(const uint64_t* __restrict__ packed, uint64_t n,
                            uint32_t* __restrict__ cnt, uint32_t* __restrict__ first,
                            uint8_t* __restrict__ filt) {
  const uint64_t i = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint64_t p = packed[i];
  cnt[i] = static_cast<uint32_t>(p) & 0x7FFFFFFFu;
  first[i] = static_cast<uint32_t>(p >> 32);
  filt[i] = static_cast<uint8_t>((p >> 31) & 1);
}


__global__ void __launch_bounds__(kThreads)
ExpandWarpKernel(IndexView ix, const uint64_t* __restrict__ q_org, uint64_t q_begin,
                 uint64_t n_q, const uint32_t* __restrict__ cnt,
                 const uint32_t* __restrict__ first, const uint64_t* __restrict__ hit_off,
                 uint64_t* __restrict__ h_grp, uint64_t* __restrict__ h_pos) {
  const uint64_t i = (static_cast<uint64_t>(blockIdx.x) * kThreads + threadIdx.x);
  const bool valid = i < n_q;
  ExpandWarp(ix.org, valid ? cnt[i] : 0, valid ? first[i] : 0, valid ? q_org[q_begin + i] : 0,
             valid ? hit_off[i] : 0, h_grp, h_pos, nullptr);
}

// ---- stage-1 hits by a self-join over the index ----
// In stage 1 (construct.cc:59-64) the queries of a flush are the micromizers of reads
// that are themselves in the index, so every query IS a posting of the run of its
// value: a posting (value v, read r, position p) is a query iff it passes r's
// selection rule (thr_val, thr_pos; sketch.cu), and its hits are the postings of the
// same run with a larger read id - the ones that follow it, the run being in read
// order. No query sort, no table probe, no binary search: two sweeps over the sorted
// postings (count, then emit through per-read cursors; the order of the hits inside
// a read is free, see the header). Runs longer than `occurrence` give no hits.
struct JoinView {
  ValView val;
  const uint64_t* org;
  uint64_t n;
  uint32_t occurrence;
  const uint64_t* thr_val;  // of reads [thr_first, ...)
  const uint32_t* thr_pos;
  uint32_t thr_first;
  uint32_t first, last;     // query reads of this flush
};

// number of hits of posting i (read r, value v) and the offset of the first one
__device__ __forceinline__ uint32_t JoinKept(const JoinView& jv, uint64_t i, uint64_t v,
                                             uint32_t r, uint32_t* skip) {
  uint32_t fw = 0, same = 0;
  for (uint64_t j = i + 1; j < jv.n && jv.val[j] == v; ++j) {
    ++fw;
    if (fw > jv.occurrence) return 0;
    if (static_cast<uint32_t>(jv.org[j] >> 32) == r) ++same;
  }
  if (fw == same) return 0;
  if (jv.occurrence != 0xFFFFFFFFu) {
    uint32_t len = fw + 1;
    if (len > jv.occurrence) return 0;
    for (uint64_t j = i; j > 0 && jv.val[j - 1] == v; --j) {
      if (++len > jv.occurrence) return 0;
    }
  }
  *skip = same;
  return fw - same;
}

__device__ __forceinline__ bool JoinIsQuery(const JoinView& jv, uint64_t v, uint64_t o) {
  const uint32_t r = static_cast<uint32_t>(o >> 32);
  if (r < jv.first || r >= jv.last) return false;
  const uint64_t t = jv.thr_val[r - jv.thr_first];
  return v < t || (v == t && (static_cast<uint32_t>(o) >> 1) < jv.thr_pos[r - jv.thr_first]);
}

// sweep over the sorted postings: every query posting with hits takes the next free
// slot of its read (slots [q_off[r], q_off[r + 1]) - one per micromizer - in any
// order) and leaves (posting index, number of hits) there
__global__ void __launch_bounds__(kThreads)
JoinProbeKernel(JoinView jv, const uint64_t* __restrict__ q_off, uint64_t q_begin,
                uint32_t* __restrict__ cursor, uint64_t* __restrict__ packed) {
  const uint64_t i = static_cast<uint64_t>(blockIdx.x) * kThreads + threadIdx.x;
  if (i >= jv.n) return;
  const uint64_t v = jv.val[i], o = jv.org[i];
  if (!JoinIsQuery(jv, v, o)) return;
  const uint32_t r = static_cast<uint32_t>(o >> 32);
  uint32_t skip;
  const uint32_t kept = JoinKept(jv, i, v, r, &skip);
  if (!kept) return;
  const uint64_t slot = q_off[r - jv.thr_first] - q_begin + atomicAdd(cursor + (r - jv.first), 1u);
  packed[slot] = (i << 32) | kept;
}

__global__ void UnpackJoin(const uint64_t* __restrict__ packed, uint64_t n,
                           uint32_t* __restrict__ cnt) {
  const uint64_t i = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i < n) cnt[i] = static_cast<uint32_t>(packed[i]);
}

// ExpandWarpKernel over the slots of JoinProbeKernel: the query's own posting gives
// its origin, its hits follow it in the run (after the postings of the same read)
__global__ void __launch_bounds__(kThreads)
ExpandJoinKernel(const uint64_t* __restrict__ i_org, const uint64_t* __restrict__ packed,
                 uint64_t n_q, const uint64_t* __restrict__ hit_off,
                 uint64_t* __restrict__ h_grp, uint64_t* __restrict__ h_pos) {
  const uint64_t i = (static_cast<uint64_t>(blockIdx.x) * kThreads + threadIdx.x);
  const bool valid = i < n_q;
  const uint64_t pk = valid ? packed[i] : 0;
  const uint32_t my_cnt = static_cast<uint32_t>(pk);
  uint32_t my_first = 0;
  uint64_t my_org = 0;
  if (my_cnt) {
    const uint32_t post = static_cast<uint32_t>(pk >> 32);
    my_org = i_org[post];
    my_first = post + 1;
    while ((i_org[my_first] >> 32) == (my_org >> 32)) ++my_first;  // same read: not a hit
  }
  ExpandWarp(i_org, my_cnt, my_first, my_org, valid ? hit_off[i] : 0, h_grp, h_pos, nullptr);
}

// per-read offsets out of per-record offsets
__global__ void GatherU64(const uint64_t* __restrict__ src,
                          const uint64_t* __restrict__ idx, uint64_t idx_base,
                          uint64_t n, uint64_t* __restrict__ dst) {
  const uint64_t i = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  dst[i] = src[idx[i] - idx_base];
}

// positions of over-frequent query minimizers, compacted in sketch order
__global__ void FilteredFlagsToU32(const uint8_t* __restrict__ filt, uint64_t n,
                                   uint32_t* __restrict__ out) {
  const uint64_t i = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i < n) out[i] = filt[i];
}
__global__ void ScatterFiltered(const uint8_t* __restrict__ filt,
                                const uint64_t* __restrict__ pos,
                                const uint64_t* __restrict__ q_org,
                                uint64_t q_begin, uint64_t n,
                                uint32_t* __restrict__ out) {
  const uint64_t i = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n || !filt[i]) return;
  out[pos[i]] = static_cast<uint32_t>(q_org[q_begin + i]) >> 1;
}

// ---------------------------------------------------------------------------
// chaining
// ---------------------------------------------------------------------------

struct ChainParams {
  uint32_t k, bandwidth, chain, matches, gap;
};

// sorts (A[i], B[i]) pairs ascending by (A, B); npad is a power of two
template <int THREADS>
__device__ void BitonicSortPairs(uint64_t* A, uint64_t* B, uint32_t npad) {
  for (uint32_t size = 2; size <= npad; size <<= 1) {
    for (uint32_t stride = size >> 1; stride > 0; stride >>= 1) {
      for (uint32_t t = threadIdx.x; t < (npad >> 1); t += THREADS) {
        const uint32_t i = 2 * t - (t & (stride - 1));
        const uint32_t j = i + stride;
        const bool up = (i & size) == 0;
        const uint64_t ai = A[i], aj = A[j], bi = B[i], bj = B[j];
        const bool gt = ai > aj || (ai == aj && bi > bj);
        if (gt == up) {
          A[i] = aj;
          A[j] = ai;
          B[i] = bj;
          B[j] = bi;
        }
      }
      __syncthreads();
    }
  }
}

// Everything a CTA needs to chain the hits of one query read. IdxT = u16 for
// the shared-memory path (n <= 65534), u32 for the global scratch path.
template <typename IdxT>
struct ChainWork {
  uint64_t* G;   // npad   group, later band tag
  uint64_t* P;   // npad   positions
  IdxT* LB;      // n + 1  lower bounds, later LIS "minimal"+indices (n + nb + 1)
  IdxT* PD;      // n      predecessor
  IdxT* IB;      // n/4+1  band begin
  IdxT* IE;      // n/4+1  band end
  uint32_t* CNT; // n/4+1  overlaps per band
};

template <typename IdxT, int THREADS>
__device__ uint32_t ChainRead(const ChainWork<IdxT>& wk, uint32_t n,
                              uint32_t npad, uint32_t lhs_id,
                              const ChainParams& cp, uint32_t* sm32,
                              rvn_overlap* __restrict__ ovl_raw,
                              unsigned long long* __restrict__ ovl_counter,
                              uint64_t ovl_cap, uint64_t* out_base,
                              uint64_t* __restrict__ ovl_key = nullptr, uint64_t key_hi = 0) {
  uint64_t* G = wk.G;
  uint64_t* P = wk.P;
  __shared__ unsigned long long sh_base;

  // 1. order by (group, positions); padding is all-ones and sorts last, and
  //    G[n] doubles as the reference's stop dummy
  BitonicSortPairs<THREADS>(G, P, npad);

  // 2. lower bounds: LB[i] = first j with G[i] - G[j] <= bandwidth
  for (uint32_t i = threadIdx.x; i <= n; i += THREADS) {
    const uint64_t gi = i < n ? G[i] : ~0ULL;
    uint32_t lo = 0, hi = i;
    while (lo < hi) {
      const uint32_t mid = lo + (hi - lo) / 2;
      if (gi - G[mid] <= cp.bandwidth) {
        hi = mid;
      } else {
        lo = mid + 1;
      }
    }
    wk.LB[i] = static_cast<IdxT>(lo);
  }
  __syncthreads();

  // 3. events: at i (1..n) the window [LB[i-1], i) closes; it qualifies with
  //    >= 4 hits; a qualifying window overlapping the previous qualifying
  //    one extends it. Done chunk-wise with carried state.
  uint32_t carry_prevq = 0;  // last qualifying event index so far (0 = none)
  uint32_t carry_nb = 0;     // bands opened so far
  for (uint32_t base = 1; base <= n; base += THREADS) {
    const uint32_t i = base + threadIdx.x;
    uint32_t e = 0, jp = 0;
    if (i <= n) {
      jp = wk.LB[i - 1];
      const uint64_t gi = i < n ? G[i] : ~0ULL;
      e = (gi - G[jp] > cp.bandwidth) && (i - jp >= 4);
    }
    // previous qualifying event (exclusive max-scan of e ? i : 0)
    const uint32_t incl = BlockInclusiveMax<uint32_t, THREADS>(e ? i : 0u, sm32);
    uint32_t prevq_incl_before;  // max over lanes < this one
    {
      // shift by one lane: recompute exclusive from inclusive of neighbours
      __shared__ uint32_t sh_incl[THREADS];
      sh_incl[threadIdx.x] = incl;
      __syncthreads();
      prevq_incl_before = threadIdx.x ? sh_incl[threadIdx.x - 1] : 0u;
      __syncthreads();
    }
    const uint32_t prevq = max(carry_prevq, prevq_incl_before);
    const uint32_t start = e && (prevq == 0 || prevq <= jp);
    uint32_t tot;
    const uint32_t ex = BlockExclusiveSum<uint32_t, THREADS>(start, sm32, &tot);
    if (e) {
      const uint32_t band = carry_nb + ex + start - 1;  // band this event feeds
      if (start) {
        wk.IB[band] = static_cast<IdxT>(jp);
        // the previous band (if any) ended at the previous qualifying event
        if (prevq != 0) wk.IE[band - 1] = static_cast<IdxT>(prevq);
      }
    }
    carry_nb += tot;
    // last qualifying event of the chunk
    {
      __shared__ uint32_t sh_last;
      if (threadIdx.x == THREADS - 1) sh_last = max(carry_prevq, incl);
      __syncthreads();
      carry_prevq = sh_last;
      __syncthreads();
    }
  }
  const uint32_t nb = carry_nb;
  if (threadIdx.x == 0 && nb) wk.IE[nb - 1] = static_cast<IdxT>(carry_prevq);
  __syncthreads();
  if (nb == 0) return 0;

  // 4. tag hits with their band (2b+1) or the gap before band b (2b), then
  //    order each band by positions with one more (tag, positions) sort
  for (uint32_t i = threadIdx.x; i < npad; i += THREADS) {
    if (i >= n) {
      G[i] = ~0ULL;
      continue;
    }
    // band with the largest begin <= i
    uint32_t lo = 0, hi = nb;
    while (lo < hi) {
      const uint32_t mid = lo + (hi - lo) / 2;
      if (wk.IB[mid] <= i) {
        lo = mid + 1;
      } else {
        hi = mid;
      }
    }
    // lo = number of bands beginning at or before i
    uint64_t tag;
    if (lo == 0) {
      tag = 0;
    } else if (i < wk.IE[lo - 1]) {
      tag = 2ULL * (lo - 1) + 1;
    } else {
      tag = 2ULL * lo;
    }
    // keep rhs_id/strand of the band reachable after the sort: stash the
    // top 32 group bits in the low half of the tag word
    G[i] = (tag << 32) | (G[i] >> 32);
  }
  __syncthreads();
  BitonicSortPairs<THREADS>(G, P, npad);

  // 5. one thread per band: LIS + gap split + covered bases
  IdxT* MINI = wk.LB;  // re-used: per band (len + 1) entries at IB[b] + b
  for (uint32_t b = threadIdx.x; b < nb; b += THREADS) {
    const uint32_t jb = wk.IB[b], ie = wk.IE[b];
    const uint32_t len = ie - jb;
    uint32_t emitted = 0;
    uint32_t longest = 0;
    if (len >= cp.chain) {
      const uint64_t* Pb = P + jb;
      IdxT* minimal = MINI + jb + b;
      IdxT* pred = wk.PD + jb;
      const bool strand = G[jb] & 1;
      minimal[0] = 0;
      for (uint32_t t = 0; t < len; ++t) {
        const uint32_t cl = static_cast<uint32_t>(Pb[t] >> 32);
        const uint32_t cr = static_cast<uint32_t>(Pb[t]);
        uint32_t lo = 1, hi = longest;
        while (lo <= hi) {
          const uint32_t mid = lo + (hi - lo) / 2;
          const uint64_t tail = Pb[minimal[mid]];
          const uint32_t tl = static_cast<uint32_t>(tail >> 32);
          const uint32_t tr = static_cast<uint32_t>(tail);
          if (tl < cl && (strand ? tr < cr : tr > cr)) {
            lo = mid + 1;
          } else {
            hi = mid - 1;
          }
        }
        pred[t] = minimal[lo - 1];
        minimal[lo] = static_cast<IdxT>(t);
        longest = max(longest, lo);
      }
      if (longest >= cp.chain) {
        // unroll the chain into minimal[0 .. longest)
        uint32_t j = minimal[longest];
        for (uint32_t i = 0; i < longest; ++i) {
          const uint32_t pj = pred[j];
          minimal[longest - 1 - i] = static_cast<IdxT>(j);
          j = pj;
        }
      } else {
        longest = 0;
      }
    }
    // count the overlaps this band emits (walk repeated when writing)
    if (longest) {
      const uint64_t* Pb = P + jb;
      const IdxT* idx = MINI + jb + b;
      const bool strand = G[jb] & 1;
      for (uint32_t kk = 1, l = 0; kk <= longest; ++kk) {
        const uint32_t prev = static_cast<uint32_t>(Pb[idx[kk - 1]] >> 32);
        const uint32_t cur =
            kk < longest ? static_cast<uint32_t>(Pb[idx[kk]] >> 32) : 0xFFFFFFFFu;
        if (cur - prev > cp.gap) {
          if (kk - l >= cp.chain) {
            uint32_t lm = 0, lb_ = 0, le = 0, rm = 0, rb_ = 0, re = 0;
            for (uint32_t m = l; m < kk; ++m) {
              const uint64_t pp = Pb[idx[m]];
              const uint32_t lp = static_cast<uint32_t>(pp >> 32);
              if (lp > le) {
                lm += le - lb_;
                lb_ = lp;
              }
              le = lp + cp.k;
              uint32_t rp = static_cast<uint32_t>(pp);
              rp = strand ? rp : (1U << 31) - (rp + cp.k - 1);
              if (rp > re) {
                rm += re - rb_;
                rb_ = rp;
              }
              re = rp + cp.k;
            }
            lm += le - lb_;
            rm += re - rb_;
            if (min(lm, rm) >= cp.matches) ++emitted;
          }
          l = kk;
        }
      }
    }
    wk.CNT[b] = emitted;
    // stash the chain length where the writer finds it
    wk.IE[b] = static_cast<IdxT>(longest);
  }
  __syncthreads();

  // 6. place the overlaps of all bands in band order
  uint32_t carry = 0;
  __shared__ uint32_t sh_total;
  // first pass: total
  {
    uint32_t local = 0;
    for (uint32_t b = threadIdx.x; b < nb; b += THREADS) local += wk.CNT[b];
    uint32_t tot;
    BlockExclusiveSum<uint32_t, THREADS>(local, sm32, &tot);
    if (threadIdx.x == 0) {
      sh_total = tot;
      sh_base = tot ? atomicAdd(ovl_counter, static_cast<unsigned long long>(tot))
                    : 0ULL;
    }
    __syncthreads();
  }
  const uint32_t total = sh_total;
  const uint64_t base = sh_base;
  *out_base = base;
  if (total == 0 || base + total > ovl_cap) return total;

  for (uint32_t b0 = 0; b0 < nb; b0 += THREADS) {
    const uint32_t b = b0 + threadIdx.x;
    const uint32_t mine = b < nb ? wk.CNT[b] : 0;
    uint32_t tot;
    const uint32_t ex = BlockExclusiveSum<uint32_t, THREADS>(mine, sm32, &tot);
    if (mine) {
      rvn_overlap* dst = ovl_raw + base + carry + ex;
      // (pair-at-a-time callers: emission sequence number of every overlap)
      uint64_t* kdst = ovl_key ? ovl_key + base + carry + ex : nullptr;
      uint32_t seq = carry + ex;
      const uint32_t jb = wk.IB[b];
      const uint32_t longest = wk.IE[b];
      const uint64_t* Pb = P + jb;
      const IdxT* idx = MINI + jb + b;
      const bool strand = G[jb] & 1;
      const uint32_t rhs_id = static_cast<uint32_t>(G[jb] & 0xFFFFFFFFu) >> 1;
      for (uint32_t kk = 1, l = 0; kk <= longest; ++kk) {
        const uint32_t prev = static_cast<uint32_t>(Pb[idx[kk - 1]] >> 32);
        const uint32_t cur =
            kk < longest ? static_cast<uint32_t>(Pb[idx[kk]] >> 32) : 0xFFFFFFFFu;
        if (cur - prev > cp.gap) {
          if (kk - l >= cp.chain) {
            uint32_t lm = 0, lb_ = 0, le = 0, rm = 0, rb_ = 0, re = 0;
            for (uint32_t m = l; m < kk; ++m) {
              const uint64_t pp = Pb[idx[m]];
              const uint32_t lp = static_cast<uint32_t>(pp >> 32);
              if (lp > le) {
                lm += le - lb_;
                lb_ = lp;
              }
              le = lp + cp.k;
              uint32_t rp = static_cast<uint32_t>(pp);
              rp = strand ? rp : (1U << 31) - (rp + cp.k - 1);
              if (rp > re) {
                rm += re - rb_;
                rb_ = rp;
              }
              re = rp + cp.k;
            }
            lm += le - lb_;
            rm += re - rb_;
            if (min(lm, rm) >= cp.matches) {
              const uint64_t pf = Pb[idx[l]], pl = Pb[idx[kk - 1]];
              rvn_overlap o;
              o.lhs_id = lhs_id;
              o.lhs_begin = static_cast<uint32_t>(pf >> 32);
              o.lhs_end = cp.k + static_cast<uint32_t>(pl >> 32);
              o.rhs_id = rhs_id;
              o.rhs_begin = strand ? static_cast<uint32_t>(pf)
                                   : static_cast<uint32_t>(pl);
              o.rhs_end = cp.k + (strand ? static_cast<uint32_t>(pl)
                                         : static_cast<uint32_t>(pf));
              o.score = min(lm, rm);
              o.strand = strand;
              *dst++ = o;
              if (kdst) *kdst++ = key_hi | seq++;
            }
          }
          l = kk;
        }
      }
    }
    carry += tot;
  }
  return total;
}

constexpr uint32_t kChainSmemCap = 65535;  // hits per read on the split path (16-bit offsets)
constexpr uint32_t kSplitMaxTable = 8192;  // pair hash table entries per read, at most
constexpr uint32_t kPairMaxHits = 8191;    // hits of one pair PairChainKernel holds on chip
constexpr uint32_t kThreadPairMax = 48;   // larger (rhs, strand) pairs get a CTA each

// ---------------------------------------------------------------------------
// Fast path, two kernels.
//
// Bands never span two (rhs_id, strand) pairs (group keys of different pairs
// differ by >= 2^30 > bandwidth), so the reference's per-query sort by group is
// not needed.
//  SplitKernel  one CTA per query read: the read's hits are split by pair with
//               a shared-memory hash table; pairs with < 4 hits (about half of
//               all hits: spurious key matches) are dropped on the spot; the
//               rest is written pair-contiguous to HBM with one descriptor per
//               pair, pairs of a read in ascending key order (= the reference's
//               emission order).
//  GroupChainKernel  ONE THREAD PER PAIR over all pairs of all reads, largest
//               pairs first (size-sorted, so the lanes of a warp carry similar
//               work and nothing waits at a barrier): (diagonal, positions)
//               order by binary insertion, the reference's window loop, per
//               band the position order, ram's patience/LIS recurrence with
//               its exact probe sequence, gap split, covered bases. Overlaps go
//               to a global list keyed (pair index, sequence number) and are
//               put back in emission order by a radix sort of the keys.
// ---------------------------------------------------------------------------
struct GroupDesc {
  uint32_t hit_off, cnt, gid, lhs_id;
};

struct SplitLayout {
  uint32_t hs, gpad;
  size_t hk, hc, gl, bytes;
};

__host__ __device__ inline SplitLayout MakeSplitLayout(uint32_t n) {
  SplitLayout L;
  // open addressing, never full: distinct pairs <= n < hs. (A smaller table
  // does fill up: a random key match drags in every read covering that locus,
  // so single-hit pairs are about as many as half the hits.)
  uint32_t hs = 64;
  while (hs < n + 1 && hs < kSplitMaxTable) hs <<= 1;
  L.hs = hs;  // (reads beyond 8191 hits: a full table sends the read to the generic path)
  uint32_t gpad = 2;
  while (gpad < n / 4 + 1 && gpad < hs) gpad <<= 1;
  L.gpad = gpad;
  size_t o = 0;
  L.hk = o; o += 4ULL * hs;
  L.hc = o; o += 4ULL * hs;
  L.gl = o; o += 8ULL * gpad;
  L.bytes = (o + 15) & ~size_t(15);
  return L;
}

__device__ __forceinline__ uint32_t HashGid(uint32_t x) {
  x ^= x >> 16;
  x *= 0x7feb352dU;
  x ^= x >> 15;
  x *= 0x846ca68bU;
  x ^= x >> 16;
  return x;
}

template <int THREADS, int MINB>
__global__ void __launch_bounds__(THREADS, MINB)
SplitKernel(const uint64_t* __restrict__ h_grp, const uint64_t* __restrict__ h_pos,
            const uint64_t* __restrict__ read_hit_off,
            const uint32_t* __restrict__ lhs_ids,
            const uint32_t* __restrict__ read_list,
            unsigned long long* __restrict__ totals,  // [0] pairs, [1] kept hits
            GroupDesc* __restrict__ desc, uint32_t* __restrict__ desc_cnt,
            uint32_t* __restrict__ desc_idx, uint32_t* __restrict__ g_diag,
            uint64_t* __restrict__ g_pos, uint64_t* __restrict__ group_loc,
            uint32_t* __restrict__ fallback_list,
            unsigned int* __restrict__ fallback_cnt) {
  extern __shared__ __align__(16) unsigned char smem[];
  __shared__ uint32_t sm32[34];
  __shared__ uint32_t sh_bail;
  __shared__ unsigned long long sh_gbase, sh_hbase;
  const uint32_t r = read_list[blockIdx.x];
  const uint64_t hb = read_hit_off[r];
  const uint32_t n = static_cast<uint32_t>(read_hit_off[r + 1] - hb);
  const SplitLayout L = MakeSplitLayout(n);
  uint32_t* HK = reinterpret_cast<uint32_t*>(smem + L.hk);
  uint32_t* HC = reinterpret_cast<uint32_t*>(smem + L.hc);
  uint64_t* GL = reinterpret_cast<uint64_t*>(smem + L.gl);
  const uint32_t hmask = L.hs - 1;
  const uint64_t* hg = h_grp + hb;
  const uint64_t* hp = h_pos + hb;

  // ---- hash table of (rhs_id, strand) pairs with their hit counts ----
  for (uint32_t i = threadIdx.x; i < L.hs; i += THREADS) {
    HK[i] = 0xFFFFFFFFu;
    HC[i] = 0;
  }
  if (threadIdx.x == 0) sh_bail = 0;
  __syncthreads();
  for (uint32_t i = threadIdx.x; i < n; i += THREADS) {
    const uint32_t gid = static_cast<uint32_t>(hg[i] >> 32);
    uint32_t s = HashGid(gid) & hmask;
    uint32_t probes = 0;
    while (true) {
      const uint32_t prev = atomicCAS(&HK[s], 0xFFFFFFFFu, gid);
      if (prev == 0xFFFFFFFFu || prev == gid) break;
      s = (s + 1) & hmask;
      if (++probes > hmask) {  // table full (only possible beyond 8191 hits)
        sh_bail = 1;
        break;
      }
    }
    if (probes <= hmask) atomicAdd(&HC[s], 1u);
  }
  __syncthreads();
  if (sh_bail) {  // more distinct pairs than the table holds: the generic kernel
    if (threadIdx.x == 0) fallback_list[atomicAdd(fallback_cnt, 1u)] = r;
    return;
  }

  // ---- pairs with >= 4 hits: list + offsets inside the read's kept hits ----
  uint32_t carry = 0;  // low 16: pairs so far, high 16: kept hits so far
  for (uint32_t b = 0; b < L.hs; b += THREADS) {
    const uint32_t s = b + threadIdx.x;
    const uint32_t cnt = s < L.hs ? HC[s] : 0;
    const uint32_t keep = cnt >= 4;
    if (cnt > kPairMaxHits) sh_bail = 1;  // (a pair PairChainKernel cannot hold on chip)
    uint32_t tot;
    const uint32_t ex = BlockExclusiveSum<uint32_t, THREADS>(
        keep ? ((cnt << 16) | 1u) : 0u, sm32, &tot);
    if (s < L.hs) {
      if (keep) {
        const uint32_t at = carry + ex;
        GL[at & 0xFFFF] = (static_cast<uint64_t>(HK[s]) << 32) | s;
        HC[s] = (cnt << 16) | (at >> 16);  // (count, offset)
      } else {
        HC[s] = 0xFFFFFFFFu;  // dropped
      }
    }
    carry += tot;
  }
  const uint32_t ng = carry & 0xFFFF, nh = carry >> 16;
  __syncthreads();
  if (sh_bail) {  // a very large pair: the generic kernel takes this read
    if (threadIdx.x == 0) fallback_list[atomicAdd(fallback_cnt, 1u)] = r;
    return;
  }
  if (ng == 0) {
    if (threadIdx.x == 0) group_loc[r] = 0;
    return;
  }

  // ---- pairs in ascending key order; reserve descriptor and hit space ----
  uint32_t gpad = 2;
  while (gpad < ng) gpad <<= 1;
  for (uint32_t i = ng + threadIdx.x; i < gpad; i += THREADS) GL[i] = ~0ULL;
  if (threadIdx.x == 0) {
    sh_gbase = atomicAdd(&totals[0], static_cast<unsigned long long>(ng));
    sh_hbase = atomicAdd(&totals[1], static_cast<unsigned long long>(nh));
  }
  __syncthreads();
  for (uint32_t size = 2; size <= gpad; size <<= 1) {
    for (uint32_t stride = size >> 1; stride > 0; stride >>= 1) {
      for (uint32_t t = threadIdx.x; t < (gpad >> 1); t += THREADS) {
        const uint32_t i = 2 * t - (t & (stride - 1));
        const uint32_t j = i + stride;
        const uint64_t a = GL[i], c2 = GL[j];
        if ((a > c2) == ((i & size) == 0)) {
          GL[i] = c2;
          GL[j] = a;
        }
      }
      __syncthreads();
    }
  }
  const uint64_t gbase = sh_gbase, hbase = sh_hbase;
  const uint32_t lhs_id = lhs_ids[r];
  for (uint32_t q = threadIdx.x; q < ng; q += THREADS) {
    const uint64_t e = GL[q];
    const uint32_t s = static_cast<uint32_t>(e);
    const uint32_t v = HC[s];
    GroupDesc d;
    d.hit_off = static_cast<uint32_t>(hbase) + (v & 0xFFFF);
    d.cnt = v >> 16;
    d.gid = static_cast<uint32_t>(e >> 32);
    d.lhs_id = lhs_id;
    desc[gbase + q] = d;
    desc_cnt[gbase + q] = d.cnt;
    desc_idx[gbase + q] = static_cast<uint32_t>(gbase + q);
    HC[s] = v & 0xFFFF;  // fill cursor
  }
  if (threadIdx.x == 0) group_loc[r] = (gbase << 24) | ng;
  __syncthreads();

  // ---- scatter the hits of kept pairs (order inside a pair is free) ----
  for (uint32_t i = threadIdx.x; i < n; i += THREADS) {
    const uint64_t g = hg[i];
    const uint32_t gid = static_cast<uint32_t>(g >> 32);
    uint32_t s = HashGid(gid) & hmask;
    while (HK[s] != gid) s = (s + 1) & hmask;
    if (HC[s] == 0xFFFFFFFFu) continue;
    const uint64_t at = hbase + atomicAdd(&HC[s], 1u);
    g_diag[at] = static_cast<uint32_t>(g);
    g_pos[at] = hp[i];
  }
}

// A pair's hits live in shared memory, interleaved across the CTA's threads
// (element i of thread t at [i * T + t]): every thread walks its own column,
// same-index accesses of a warp are conflict-free, and no barrier is needed.
struct Column {
  uint64_t* P;  // positions column (already offset by the thread index)
  uint32_t* D;  // diagonal column; per band re-used as (minimal, predecessor) u16 pairs
  uint32_t T;   // column stride = threads per CTA
  __device__ __forceinline__ uint64_t& p(uint32_t i) const { return P[i * T]; }
  __device__ __forceinline__ uint32_t& d(uint32_t i) const { return D[i * T]; }
};

// one band [jb, ie) of a pair: position order, LIS, gap split, emit
__device__ __forceinline__ void BandChain(const Column& c, uint32_t jb, uint32_t ie,
                                          bool strand, uint32_t lhs_id,
                                          uint32_t rhs_id, const ChainParams& cp,
                                          uint64_t key_hi, uint32_t* seq,
                                          rvn_overlap* __restrict__ out,
                                          uint64_t* __restrict__ out_key,
                                          unsigned long long* __restrict__ out_cnt,
                                          uint64_t out_cap) {
  const uint32_t len = ie - jb;
  if (len < cp.chain) return;
  for (uint32_t a = 1; a < len; ++a) {  // binary insertion sort by positions
    const uint64_t pv = c.p(jb + a);
    if (c.p(jb + a - 1) <= pv) continue;
    uint32_t lo = 0, hi = a - 1;  // first element > pv lies in [lo, hi]
    while (lo < hi) {
      const uint32_t mid = (lo + hi) >> 1;
      if (c.p(jb + mid) > pv) {
        hi = mid;
      } else {
        lo = mid + 1;
      }
    }
    for (uint32_t b = a; b > lo; --b) c.p(jb + b) = c.p(jb + b - 1);
    c.p(jb + lo) = pv;
  }
  // the band's diagonals are dead: word x of the band now holds
  // minimal[x + 1] (low half) and predecessor[x] (high half); minimal[0] = 0
  auto mini_get = [&](uint32_t x) -> uint32_t { return c.d(jb + x) & 0xFFFFu; };
  auto mini_set = [&](uint32_t x, uint32_t v) {
    c.d(jb + x) = (c.d(jb + x) & 0xFFFF0000u) | v;
  };
  auto pred_get = [&](uint32_t x) -> uint32_t { return c.d(jb + x) >> 16; };
  auto pred_set = [&](uint32_t x, uint32_t v) {
    c.d(jb + x) = (c.d(jb + x) & 0xFFFFu) | (v << 16);
  };
  uint32_t longest = 0;
  for (uint32_t t = 0; t < len; ++t) {
    const uint64_t cur = c.p(jb + t);
    const uint32_t cl = static_cast<uint32_t>(cur >> 32);
    const uint32_t cr = static_cast<uint32_t>(cur);
    uint32_t lo = 1, hi = longest;
    while (lo <= hi) {
      const uint32_t mid = lo + (hi - lo) / 2;
      const uint64_t tail = c.p(jb + mini_get(mid - 1));
      const uint32_t tl = static_cast<uint32_t>(tail >> 32);
      const uint32_t tr = static_cast<uint32_t>(tail);
      if (tl < cl && (strand ? tr < cr : tr > cr)) {
        lo = mid + 1;
      } else {
        hi = mid - 1;
      }
    }
    pred_set(t, lo > 1 ? mini_get(lo - 2) : 0u);
    mini_set(lo - 1, t);
    longest = max(longest, lo);
  }
  if (longest < cp.chain) return;
  {
    uint32_t j = mini_get(longest - 1);
    for (uint32_t i = 0; i < longest; ++i) {
      const uint32_t pj = pred_get(j);
      mini_set(longest - 1 - i, j);
      j = pj;
    }
  }
  for (uint32_t kk = 1, l = 0; kk <= longest; ++kk) {
    const uint32_t prev = static_cast<uint32_t>(c.p(jb + mini_get(kk - 1)) >> 32);
    const uint32_t cur = kk < longest
                             ? static_cast<uint32_t>(c.p(jb + mini_get(kk)) >> 32)
                             : 0xFFFFFFFFu;
    if (cur - prev > cp.gap) {
      if (kk - l >= cp.chain) {
        uint32_t lm = 0, lb_ = 0, le = 0, rm = 0, rb_ = 0, re = 0;
        for (uint32_t m = l; m < kk; ++m) {
          const uint64_t pp = c.p(jb + mini_get(m));
          const uint32_t lp = static_cast<uint32_t>(pp >> 32);
          if (lp > le) {
            lm += le - lb_;
            lb_ = lp;
          }
          le = lp + cp.k;
          uint32_t rp = static_cast<uint32_t>(pp);
          rp = strand ? rp : (1U << 31) - (rp + cp.k - 1);
          if (rp > re) {
            rm += re - rb_;
            rb_ = rp;
          }
          re = rp + cp.k;
        }
        lm += le - lb_;
        rm += re - rb_;
        if (min(lm, rm) >= cp.matches) {
          const uint64_t pf = c.p(jb + mini_get(l)), pl = c.p(jb + mini_get(kk - 1));
          rvn_overlap o;
          o.lhs_id = lhs_id;
          o.lhs_begin = static_cast<uint32_t>(pf >> 32);
          o.lhs_end = cp.k + static_cast<uint32_t>(pl >> 32);
          o.rhs_id = rhs_id;
          o.rhs_begin = strand ? static_cast<uint32_t>(pf) : static_cast<uint32_t>(pl);
          o.rhs_end = cp.k + (strand ? static_cast<uint32_t>(pl)
                                     : static_cast<uint32_t>(pf));
          o.score = min(lm, rm);
          o.strand = strand;
          const unsigned long long slot = atomicAdd(out_cnt, 1ULL);
          if (slot < out_cap) {
            out[slot] = o;
            out_key[slot] = key_hi | (*seq)++;
          }
        }
      }
      l = kk;
    }
  }
}

// thread t of the launch handles pair order[first + t]; every pair of this
// launch has at most m_cap hits (the launch is one size class)
__global__ void GroupChainKernel(const GroupDesc* __restrict__ desc,
                                 const uint32_t* __restrict__ order, uint64_t first,
                                 uint64_t last, uint32_t m_cap,
                                 const uint32_t* __restrict__ g_diag,
                                 const uint64_t* __restrict__ g_pos, ChainParams cp,
                                 rvn_overlap* __restrict__ out,
                                 uint64_t* __restrict__ out_key,
                                 unsigned long long* __restrict__ out_cnt,
                                 uint64_t out_cap) {
  extern __shared__ __align__(16) unsigned char smem[];
  const uint32_t T = blockDim.x;
  const uint64_t t = first + static_cast<uint64_t>(blockIdx.x) * T + threadIdx.x;
  if (t >= last) return;
  Column c;
  c.P = reinterpret_cast<uint64_t*>(smem) + threadIdx.x;
  c.D = reinterpret_cast<uint32_t*>(smem + 8ULL * m_cap * T) + threadIdx.x;
  c.T = T;
  const uint32_t g = order[t];
  const GroupDesc d = desc[g];
  const uint32_t m = d.cnt;
  for (uint32_t i = 0; i < m; ++i) {
    c.p(i) = g_pos[d.hit_off + i];
    c.d(i) = g_diag[d.hit_off + i];
  }
  for (uint32_t a = 1; a < m; ++a) {  // binary insertion by (diagonal, positions)
    const uint32_t dv = c.d(a);
    const uint64_t pv = c.p(a);
    uint32_t lo = 0, hi = a;  // first element > (dv, pv) lies in [lo, hi]
    while (lo < hi) {
      const uint32_t mid = (lo + hi) >> 1;
      const uint32_t dm = c.d(mid);
      if (dm > dv || (dm == dv && c.p(mid) > pv)) {
        hi = mid;
      } else {
        lo = mid + 1;
      }
    }
    for (uint32_t b = a; b > lo; --b) {
      c.d(b) = c.d(b - 1);
      c.p(b) = c.p(b - 1);
    }
    c.d(lo) = dv;
    c.p(lo) = pv;
  }
  // the reference's window loop; index m plays the stop dummy
  const bool strand = d.gid & 1;
  const uint32_t rhs_id = d.gid >> 1;
  const uint64_t key_hi = static_cast<uint64_t>(g) << 16;
  uint32_t seq = 0;
  bool open = false;
  uint32_t ob = 0, oe = 0;
  for (uint32_t i = 1, j = 0; i <= m; ++i) {
    if (i == m || c.d(i) - c.d(j) > cp.bandwidth) {
      if (i - j >= 4) {
        if (open && oe > j) {
          oe = i;
        } else {
          if (open) {
            BandChain(c, ob, oe, strand, d.lhs_id, rhs_id, cp, key_hi, &seq, out,
                      out_key, out_cnt, out_cap);
          }
          ob = j;
          oe = i;
          open = true;
        }
      }
      ++j;
      while (j < i && (i == m || c.d(i) - c.d(j) > cp.bandwidth)) ++j;
    }
  }
  if (open) {
    BandChain(c, ob, oe, strand, d.lhs_id, rhs_id, cp, key_hi, &seq, out, out_key,
              out_cnt, out_cap);
  }
}

// One CTA per (query, rhs, strand) pair with more than kThreadPairMax hits - the
// true overlaps, above all on HiFi reads where a pair holds hundreds of hits: the
// pair's hits live in shared memory, both orders come from parallel bitonic
// sorts and the bands from block scans (ChainRead); only the LIS of a band is one
// thread's work. CTA blockIdx.x handles pair order[first + blockIdx.x]; every
// pair of a launch has at most npad - 1 hits.
constexpr int kPairThreads = 64;

__host__ __device__ inline size_t PairChainSmem(uint32_t npad) {
  const uint32_t n = npad - 1, nb = n / 4 + 1;
  size_t o = 16ULL * npad;                        // G, P
  o += 2ULL * (n + nb + 2) + 2ULL * (n + 1) + 2ULL * 2 * nb;  // LB, PD, IB, IE (u16)
  o = (o + 3) & ~size_t(3);
  o += 4ULL * nb;                                 // CNT
  return (o + 15) & ~size_t(15);
}

__global__ void __launch_bounds__(kPairThreads)
PairChainKernel(const GroupDesc* __restrict__ desc, const uint32_t* __restrict__ order,
                uint64_t first, uint32_t npad, const uint32_t* __restrict__ g_diag,
                const uint64_t* __restrict__ g_pos, ChainParams cp,
                rvn_overlap* __restrict__ out, uint64_t* __restrict__ out_key,
                unsigned long long* __restrict__ out_cnt, uint64_t out_cap) {
  extern __shared__ __align__(16) unsigned char smem[];
  __shared__ uint32_t sm32[34];
  const uint32_t g = order[first + blockIdx.x];
  const GroupDesc d = desc[g];
  const uint32_t n = d.cnt;
  const uint32_t ncap = npad - 1, nbmax = ncap / 4 + 1;
  ChainWork<uint16_t> wk;
  wk.G = reinterpret_cast<uint64_t*>(smem);
  wk.P = wk.G + npad;
  wk.LB = reinterpret_cast<uint16_t*>(wk.P + npad);
  wk.PD = wk.LB + (ncap + nbmax + 2);
  wk.IB = wk.PD + (ncap + 1);
  wk.IE = wk.IB + nbmax;
  wk.CNT = reinterpret_cast<uint32_t*>(
      (reinterpret_cast<uintptr_t>(wk.IE + nbmax) + 3) & ~uintptr_t(3));
  // padding beyond the pair's hits sorts last (all ones), like the reference's dummy
  uint32_t np2 = 8;
  while (np2 < n + 1) np2 <<= 1;
  for (uint32_t i = threadIdx.x; i < np2; i += kPairThreads) {
    wk.G[i] = i < n ? (static_cast<uint64_t>(d.gid) << 32) | g_diag[d.hit_off + i] : ~0ULL;
    wk.P[i] = i < n ? g_pos[d.hit_off + i] : ~0ULL;
  }
  __syncthreads();
  uint64_t base = 0;
  ChainRead<uint16_t, kPairThreads>(wk, n, np2, d.lhs_id, cp, sm32, out, out_cnt, out_cap, &base,
                                    out_key, static_cast<uint64_t>(g) << 16);
}

// first index of a descending-sorted count array with count <= bound[i]
__global__ void SizeClassStarts(const uint32_t* __restrict__ sorted_cnt, uint64_t n,
                                const uint32_t* __restrict__ bound, uint32_t n_bounds,
                                uint64_t* __restrict__ start) {
  const uint32_t i = threadIdx.x;
  if (i >= n_bounds) return;
  const uint32_t bnd = bound[i];
  uint64_t lo = 0, hi = n;
  while (lo < hi) {
    const uint64_t mid = lo + (hi - lo) / 2;
    if (sorted_cnt[mid] > bnd) {
      lo = mid + 1;
    } else {
      hi = mid;
    }
  }
  start[i] = lo;
}

__global__ void IotaU32(uint32_t* __restrict__ out, uint64_t n) {
  const uint64_t i = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i < n) out[i] = static_cast<uint32_t>(i);
}

__global__ void GatherOverlapsByIndex(const rvn_overlap* __restrict__ src,
                                      const uint32_t* __restrict__ idx, uint64_t n,
                                      rvn_overlap* __restrict__ dst) {
  const uint64_t i = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n * 2) return;
  const uint4* s = reinterpret_cast<const uint4*>(src);
  reinterpret_cast<uint4*>(dst)[i] = s[static_cast<uint64_t>(idx[i >> 1]) * 2 + (i & 1)];
}

// per listed read: where its overlaps sit in the key-sorted list
__global__ void LocateReadOverlaps(const uint64_t* __restrict__ sorted_key,
                                   uint64_t n_keys,
                                   const uint32_t* __restrict__ read_list,
                                   uint32_t n_list,
                                   const uint64_t* __restrict__ group_loc,
                                   uint64_t base0, uint64_t* __restrict__ ovl_loc) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_list) return;
  const uint32_t r = read_list[i];
  const uint64_t gl = group_loc[r];
  const uint64_t gbase = gl >> 24, ng = gl & 0xFFFFFF;
  if (ng == 0) {
    ovl_loc[r] = 0;
    return;
  }
  auto lower = [&](uint64_t key) {
    uint64_t lo = 0, hi = n_keys;
    while (lo < hi) {
      const uint64_t mid = lo + (hi - lo) / 2;
      if (sorted_key[mid] < key) {
        lo = mid + 1;
      } else {
        hi = mid;
      }
    }
    return lo;
  };
  const uint64_t a = lower(gbase << 16), b = lower((gbase + ng) << 16);
  ovl_loc[r] = b > a ? ((base0 + a) << 24) | (b - a) : 0;
}

// global-memory path for reads with more hits than shared memory holds: one
// CTA per listed read, arrays in a scratch slab (u32 indices)
__global__ void __launch_bounds__(kThreads)
ChainKernelGlobal(const uint64_t* __restrict__ h_grp,
                  const uint64_t* __restrict__ h_pos,
                  const uint64_t* __restrict__ read_hit_off,
                  const uint32_t* __restrict__ lhs_ids,
                  const uint32_t* __restrict__ big_reads,
                  const uint64_t* __restrict__ slab64_off,
                  const uint64_t* __restrict__ slab32_off,
                  uint64_t* __restrict__ slab64, uint32_t* __restrict__ slab32,
                  ChainParams cp, rvn_overlap* __restrict__ ovl_raw,
                  unsigned long long* __restrict__ ovl_counter,
                  uint64_t ovl_cap, uint64_t* __restrict__ ovl_loc) {
  __shared__ uint32_t sm32[34];
  const uint32_t r = big_reads[blockIdx.x];
  const uint64_t hb = read_hit_off[r];
  const uint32_t n = static_cast<uint32_t>(read_hit_off[r + 1] - hb);
  uint32_t npad = 8;
  while (npad < n + 1) npad <<= 1;

  ChainWork<uint32_t> wk;
  wk.G = slab64 + slab64_off[blockIdx.x];
  wk.P = wk.G + npad;
  const uint32_t nbmax = n / 4 + 1;
  wk.LB = slab32 + slab32_off[blockIdx.x];
  wk.PD = wk.LB + (n + nbmax + 2);
  wk.IB = wk.PD + (n + 1);
  wk.IE = wk.IB + nbmax;
  wk.CNT = wk.IE + nbmax;

  for (uint32_t i = threadIdx.x; i < npad; i += kThreads) {
    wk.G[i] = i < n ? h_grp[hb + i] : ~0ULL;
    wk.P[i] = i < n ? h_pos[hb + i] : ~0ULL;
  }
  __syncthreads();
  uint64_t base = 0;
  const uint32_t total = ChainRead<uint32_t, kThreads>(
      wk, n, npad, lhs_ids[r], cp, sm32, ovl_raw, ovl_counter, ovl_cap,
      &base);
  if (threadIdx.x == 0) ovl_loc[r] = total ? (base << 24) | total : 0;
}

__global__ void OverlapCounts(const uint64_t* __restrict__ ovl_loc, uint64_t n,
                              uint32_t* __restrict__ cnt) {
  const uint64_t i = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i < n) cnt[i] = static_cast<uint32_t>(ovl_loc[i] & 0xFFFFFF);
}

// move every read's overlaps from its reserved slab to query order
__global__ void ReorderOverlaps(const rvn_overlap* __restrict__ raw,
                                const uint64_t* __restrict__ ovl_loc,
                                const uint64_t* __restrict__ ovl_off,
                                uint32_t n_reads, rvn_overlap* __restrict__ out) {
  const uint32_t r = blockIdx.x * (blockDim.x / 32) + (threadIdx.x >> 5);
  if (r >= n_reads) return;
  const uint64_t loc = ovl_loc[r];
  const uint32_t cnt = static_cast<uint32_t>(loc & 0xFFFFFF);
  const uint64_t src = loc >> 24, dst = ovl_off[r];
  const uint4* s = reinterpret_cast<const uint4*>(raw + src);
  uint4* d = reinterpret_cast<uint4*>(out + dst);
  for (uint32_t i = threadIdx.x & 31; i < cnt * 2; i += 32) d[i] = s[i];
}

}  // namespace

// Chains hits that are already grouped by query read: hits of read i of the
// range are h_grp/h_pos[read_hit_off[i] .. read_hit_off[i+1]) (any order inside
// a read). Leaves the overlaps in query order in c.m_ovl / c.m_ovl_off.
uint64_t ChainGroupedHits(Ctx& c, const uint64_t* hg, const uint64_t* hp,
                          const uint64_t* read_hit_off,
                          const std::vector<uint64_t>& h_rho, const uint32_t* lhs_ids,
                          uint32_t nr, uint64_t n_hits, uint64_t n_q) {
  TimerBegin(c, "chain");
  ChainParams cp{c.prm.k, c.prm.bandwidth, c.prm.chain, c.prm.matches, c.prm.gap};
  const uint64_t ovl_cap = n_hits / std::max(1u, std::min(c.prm.chain, 4u)) + 16;
  rvn_overlap* raw = c.m_ovl_raw.reserve(ovl_cap);
  uint64_t* loc = c.m_ovl_loc.reserve(nr + 1ULL);
  uint64_t* counter = c.m_counter.reserve((1u << 16) + 8);
  RVN_CUDA(cudaMemsetAsync(counter, 0, sizeof(uint64_t), c.stream));
  RVN_CUDA(cudaMemsetAsync(loc, 0, (nr + 1ULL) * sizeof(uint64_t), c.stream));

  // ---- fast path: split by (rhs, strand) pair, then one thread per pair ----
  static const uint32_t kBounds[] = {256, 512, 1024, 2048, 4096, 8192, 65536};
  constexpr int kClasses = sizeof(kBounds) / sizeof(kBounds[0]);
  std::vector<uint32_t> cls[kClasses];
  std::vector<uint32_t> big;
  const bool fast_ok = c.prm.chain >= 1;
  for (uint32_t i = 0; i < nr; ++i) {
    const uint64_t n = h_rho[i + 1] - h_rho[i];
    if (n < 4) continue;  // cannot form a band; ovl_loc stays 0
    if (n > kChainSmemCap || !fast_ok) {
      big.push_back(i);
      continue;
    }
    int k = 0;
    while (kBounds[k] < n + 1) ++k;
    cls[k].push_back(i);
  }
  uint64_t n_fast_ovl = 0;
  {
    size_t total = 0;
    for (auto& v : cls) total += v.size();
    uint32_t* d_list = c.m_first.reserve(std::max<size_t>(total, n_q) + 1);
    uint32_t* d_fb = c.m_fallback.reserve(nr + 4ULL);
    RVN_CUDA(cudaMemsetAsync(d_fb, 0, 2 * sizeof(uint32_t), c.stream));
    std::vector<uint32_t> flat;
    flat.reserve(total);
    for (int k = kClasses - 1; k >= 0; --k) {
      flat.insert(flat.end(), cls[k].begin(), cls[k].end());
    }
    if (total) {
      RVN_CUDA(cudaMemcpyAsync(d_list, flat.data(), total * sizeof(uint32_t),
                               cudaMemcpyHostToDevice, c.stream));
      RVN_CUDA(cudaStreamSynchronize(c.stream));  // flat goes out of scope

      const uint64_t max_groups = n_hits / 4 + 1;
      GroupDesc* desc = reinterpret_cast<GroupDesc*>(
          c.m_desc.reserve(max_groups * (sizeof(GroupDesc) / 4)));
      uint32_t* dcnt = c.m_desc_cnt.reserve(max_groups);
      uint32_t* didx = c.m_desc_idx.reserve(max_groups);
      uint32_t* dcnt2 = c.m_desc_cnt2.reserve(max_groups);
      uint32_t* didx2 = c.m_desc_idx2.reserve(max_groups);
      uint32_t* g_diag = c.m_gdiag.reserve(n_hits + 1);
      uint64_t* g_pos = c.m_gpos.reserve(n_hits + 1);
      uint64_t* group_loc = c.m_group_loc.reserve(nr + 1ULL);
      // counters: [0] overlaps (generic path), [1] pairs, [2] kept hits,
      // [3] overlaps of the fast path
      RVN_CUDA(cudaMemsetAsync(counter, 0, 4 * sizeof(uint64_t), c.stream));
      auto* ctr = reinterpret_cast<unsigned long long*>(counter);

      size_t off = 0;
      for (int k = kClasses - 1; k >= 0; --k) {  // largest class first
        const unsigned cnt = static_cast<unsigned>(cls[k].size());
        if (cnt == 0) continue;
        const size_t smem = MakeSplitLayout(kBounds[k] - 1).bytes;
        const uint32_t* lst = d_list + off;
        off += cnt;
        if (kBounds[k] > 2048) {
          auto kern = SplitKernel<256, 2>;
          RVN_CUDA(cudaFuncSetAttribute(
              kern, cudaFuncAttributeMaxDynamicSharedMemorySize,
              static_cast<int>(MakeSplitLayout(kChainSmemCap).bytes)));
          kern<<<cnt, 256, smem, c.stream>>>(hg, hp, read_hit_off, lhs_ids, lst,
                                             ctr + 1, desc, dcnt, didx, g_diag, g_pos,
                                             group_loc, d_fb + 2, d_fb);
        } else {
          auto kern = SplitKernel<128, 8>;
          kern<<<cnt, 128, smem, c.stream>>>(hg, hp, read_hit_off, lhs_ids, lst,
                                             ctr + 1, desc, dcnt, didx, g_diag, g_pos,
                                             group_loc, d_fb + 2, d_fb);
        }
        RVN_LAUNCH_CHECK();
        ++c.launches;
      }
      // pair count, reads handed back (pair table full / a pair beyond kPairMaxHits)
      uint64_t* hpin = c.pin64.reserve(8);
      RVN_CUDA(cudaMemcpyAsync(hpin, counter, 4 * sizeof(uint64_t),
                               cudaMemcpyDeviceToHost, c.stream));
      std::vector<uint32_t> fb(2);
      RVN_CUDA(cudaMemcpyAsync(fb.data(), d_fb, 2 * sizeof(uint32_t),
                               cudaMemcpyDeviceToHost, c.stream));
      RVN_CUDA(cudaStreamSynchronize(c.stream));
      const uint64_t n_groups = hpin[1];
      const uint32_t nfb = fb[0];
      if (nfb) {
        fb.resize(nfb);
        RVN_CUDA(cudaMemcpyAsync(fb.data(), d_fb + 2, nfb * sizeof(uint32_t),
                                 cudaMemcpyDeviceToHost, c.stream));
        RVN_CUDA(cudaStreamSynchronize(c.stream));
        std::sort(fb.begin(), fb.end());
        big.insert(big.end(), fb.begin(), fb.end());
      }
      if (n_groups >= 0xFFFFFFFFULL) throw LimitError("2^32 or more seed pairs");
      // GroupDesc::hit_off is 32 bits wide
      if (hpin[2] >= 0xFFFFFFFFULL) throw LimitError("2^32 or more chained seed hits in one flush");

      if (n_groups) {
        // largest pairs first: lanes of a warp get pairs of similar size
        // (stable descending radix sort on the 13 count bits, radix.cu)
        const int w_desc = RadixSortPairs(c, dcnt, dcnt2, dcnt, didx, didx2, didx, n_groups, 0, 13,
                                          /*descending=*/true);
        const uint32_t* sorted_cnt = w_desc == 0 ? dcnt2 : dcnt;
        const uint32_t* sorted_idx = w_desc == 0 ? didx2 : didx;
        rvn_overlap* tmp_ovl = c.m_ovl_tmp.reserve(ovl_cap);
        uint64_t* key = c.m_okey.reserve(ovl_cap);
        uint64_t* key2 = c.m_okey2.reserve(ovl_cap);
        uint32_t* oidx = c.m_oidx.reserve(ovl_cap);
        uint32_t* oidx2 = c.m_oidx2.reserve(ovl_cap);
        // One launch per size class of the (descending) pair order. Pairs with more
        // than kThreadPairMax hits get a CTA each (PairChainKernel, shared memory
        // by class); the many small ones a thread each (GroupChainKernel: shared
        // memory per CTA = threads x class bound x 12 B).
        static const uint32_t kGB[] = {8191, 4095, 2047, 1023, 511, 255, 127, 63,
                                       kThreadPairMax, 32, 24, 16, 8};
        constexpr uint32_t kNB = sizeof(kGB) / sizeof(kGB[0]);
        constexpr uint32_t kFirstThreadClass = 8;  // kGB[8] == kThreadPairMax
        uint32_t* d_bounds = c.m_bounds.reserve(kNB);
        uint64_t* d_starts = c.m_starts.reserve(kNB + 1);
        RVN_CUDA(cudaMemcpyAsync(d_bounds, kGB, sizeof(kGB), cudaMemcpyHostToDevice,
                                 c.stream));
        SizeClassStarts<<<1, 32, 0, c.stream>>>(sorted_cnt, n_groups, d_bounds, kNB, d_starts);
        uint64_t h_starts[kNB + 1];
        RVN_CUDA(cudaMemcpyAsync(h_starts, d_starts, kNB * sizeof(uint64_t),
                                 cudaMemcpyDeviceToHost, c.stream));
        RVN_CUDA(cudaStreamSynchronize(c.stream));
        h_starts[kNB] = n_groups;
        h_starts[0] = 0;  // (a read has at most kChainSmemCap = 8191 hits on this path)
        RVN_CUDA(cudaFuncSetAttribute(GroupChainKernel,
                                      cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      200 * 1024));
        RVN_CUDA(cudaFuncSetAttribute(PairChainKernel,
                                      cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      static_cast<int>(PairChainSmem(8192))));
        for (uint32_t b = 0; b < kNB; ++b) {
          // pairs with bound[b+1] < count <= bound[b]
          const uint64_t lo = h_starts[b], hi = h_starts[b + 1];
          if (hi <= lo) continue;
          if (b < kFirstThreadClass) {
            const uint32_t npad = kGB[b] + 1;
            PairChainKernel<<<static_cast<unsigned>(hi - lo), kPairThreads, PairChainSmem(npad),
                              c.stream>>>(desc, sorted_idx, lo, npad, g_diag, g_pos, cp, tmp_ovl,
                                          key, ctr + 3, ovl_cap);
          } else {
            uint32_t threads = 128;
            while (threads > 8 && 12ULL * kGB[b] * threads > 196 * 1024) threads >>= 1;
            const size_t smem = 12ULL * kGB[b] * threads;
            GroupChainKernel<<<CeilDiv(hi - lo, threads), threads, smem, c.stream>>>(
                desc, sorted_idx, lo, hi, kGB[b], g_diag, g_pos, cp, tmp_ovl, key, ctr + 3,
                ovl_cap);
          }
          RVN_LAUNCH_CHECK();
          ++c.launches;
        }
        n_fast_ovl = ReadU64(c, counter + 3);
        if (n_fast_ovl > ovl_cap) throw LimitError("overlap slab overflow");
        if (n_fast_ovl >= 0xFFFFFFFFULL) throw LimitError("2^32 or more overlaps");
        if (n_fast_ovl) {
          // emission order = (pair index, sequence number)
          IotaU32<<<CeilDiv(n_fast_ovl, kThreads), kThreads, 0, c.stream>>>(
              oidx, n_fast_ovl);
          int key_bits = 17;
          while (key_bits < 64 && (1ULL << (key_bits - 16)) < n_groups) ++key_bits;
          const int w_ovl = RadixSortPairs(c, key, key2, key, oidx, oidx2, oidx, n_fast_ovl, 0,
                                           key_bits);
          const uint64_t* sorted_key = w_ovl == 0 ? key2 : key;
          const uint32_t* sorted_oidx = w_ovl == 0 ? oidx2 : oidx;
          GatherOverlapsByIndex<<<CeilDiv(n_fast_ovl * 2, kThreads), kThreads, 0,
                                  c.stream>>>(tmp_ovl, sorted_oidx, n_fast_ovl, raw);
          LocateReadOverlaps<<<CeilDiv(total, kThreads), kThreads, 0, c.stream>>>(
              sorted_key, n_fast_ovl, d_list, static_cast<uint32_t>(total),
              group_loc, 0, loc);
          RVN_LAUNCH_CHECK();
          c.launches += 3;
        }
      }
      // the generic kernel appends behind the fast path's overlaps
      RVN_CUDA(cudaMemcpyAsync(counter, &n_fast_ovl, sizeof(uint64_t),
                               cudaMemcpyHostToDevice, c.stream));
      RVN_CUDA(cudaStreamSynchronize(c.stream));
    }
  }
  if (!big.empty()) {
    std::vector<uint64_t> off64(big.size() + 1, 0), off32(big.size() + 1, 0);
    for (size_t i = 0; i < big.size(); ++i) {
      const uint64_t n = h_rho[big[i] + 1] - h_rho[big[i]];
      if (n >= 0x7FFFFFFFULL) throw LimitError("a query has 2^31 or more hits");
      uint64_t npad = 8;
      while (npad < n + 1) npad <<= 1;
      const uint64_t nbmax = n / 4 + 1;
      off64[i + 1] = off64[i] + 2 * npad;
      off32[i + 1] = off32[i] + (n + nbmax + 2) + (n + 1) + 3 * nbmax + 4;
    }
    uint64_t* slab64 = c.m_scratch64.reserve(off64.back() + 2 * (big.size() + 1) + 8);
    uint32_t* slab32 = c.m_scratch32.reserve(off32.back() + big.size() + 8);
    // offsets and the read list ride at the tail of the slabs
    uint64_t* d_off64 = slab64 + off64.back();
    uint64_t* d_off32 = d_off64 + big.size() + 1;
    uint32_t* d_big = slab32 + off32.back();
    RVN_CUDA(cudaMemcpyAsync(d_off64, off64.data(), (big.size() + 1) * 8,
                             cudaMemcpyHostToDevice, c.stream));
    RVN_CUDA(cudaMemcpyAsync(d_off32, off32.data(), (big.size() + 1) * 8,
                             cudaMemcpyHostToDevice, c.stream));
    RVN_CUDA(cudaMemcpyAsync(d_big, big.data(), big.size() * 4,
                             cudaMemcpyHostToDevice, c.stream));
    ChainKernelGlobal<<<static_cast<unsigned>(big.size()), kThreads, 0,
                        c.stream>>>(
        hg, hp, read_hit_off, lhs_ids, d_big, d_off64, d_off32, slab64, slab32, cp,
        raw, reinterpret_cast<unsigned long long*>(counter), ovl_cap, loc);
    RVN_LAUNCH_CHECK();
    ++c.launches;
    RVN_CUDA(cudaStreamSynchronize(c.stream));  // host vectors go out of scope
  }

  // ---- query order ----
  uint32_t* ocnt = c.m_cnt.reserve(nr + 1ULL);
  uint64_t* ooff = c.m_ovl_off.reserve(nr + 2ULL);
  uint64_t n_ovl = 0;
  if (nr > 0) {
    OverlapCounts<<<CeilDiv(nr, kThreads), kThreads, 0, c.stream>>>(loc, nr, ocnt);
    RVN_LAUNCH_CHECK();
    ++c.launches;
    ExclusiveScanU32(c, ocnt, ooff, nr);
    n_ovl = ReadU64(c, ooff + nr);
  } else {
    RVN_CUDA(cudaMemsetAsync(ooff, 0, sizeof(uint64_t), c.stream));
  }
  if (n_ovl > ovl_cap) throw LimitError("overlap slab overflow");
  rvn_overlap* ordered = c.m_ovl.reserve(n_ovl + 1);
  if (n_ovl > 0) {
    ReorderOverlaps<<<CeilDiv(nr, kThreads / 32), kThreads, 0, c.stream>>>(
        raw, loc, ooff, nr, ordered);
    RVN_LAUNCH_CHECK();
    ++c.launches;
  }
  TimerEnd(c);
  return n_ovl;
}

void ProbeQueries(Ctx& c, ValView q_val, const uint64_t* q_org, uint64_t q_begin, uint64_t n_q,
                  bool avoid_equal, bool avoid_symmetric, uint32_t* cnt, uint32_t* first,
                  uint8_t* filt) {
  if (n_q == 0) return;
  const IndexView ix = IndexViewOf(c);
  if (KeptContiguous(c, avoid_equal, avoid_symmetric)) {
    ProbeSuffixKernel<<<CeilDiv(n_q, kThreads), kThreads, 0, c.stream>>>(
        ix, q_val, q_org, q_begin, n_q, avoid_equal, cnt, first, filt);
  } else {
    ProbeKernel<<<CeilDiv(n_q, kThreads), kThreads, 0, c.stream>>>(
        ix, q_val, q_org, q_begin, n_q, avoid_equal, avoid_symmetric, cnt, first, filt);
  }
  RVN_LAUNCH_CHECK();
  ++c.launches;
}

void MapRange(Ctx& c, uint32_t first, uint32_t last, bool avoid_equal,
              bool avoid_symmetric, bool minhash, bool want_filtered,
              bool fetch) {
  if (!c.i_valid) throw StateError("Map before Minimize");
  c.r_valid = false;
  const uint32_t nr = last - first;

  // ---- stage 1 with the query reads inside the index batch: self-join ----
  const bool join = c.self_join && minhash && avoid_equal && avoid_symmetric && !want_filtered &&
                    c.i_from_sketch && c.i_sorted_ids && c.ids_identity && first >= c.i_first &&
                    last <= c.i_last;
  if (join && !(c.qt_valid && c.qt_first <= first && last <= c.qt_last)) {
    EnsureThresholds(c, first, last);  // (e.g. after a flush of reads outside the batch)
  }
  uint64_t n_q = 0, n_hits = 0;
  uint64_t *hg = nullptr, *hp = nullptr;
  uint64_t* read_hit_off = c.m_read_hit_off.reserve(nr + 2ULL);
  std::vector<uint64_t> h_rho(nr + 1ULL);
  if (join) {
    JoinView jv{ValView{c.i_val.get(), c.i_is32 ? 1 : 0}, c.i_org.get(), c.i_n, c.occurrence,
                c.qt_val.get(), c.qt_pos.get(), c.qt_first, first, last};
    TimerBegin(c, "probe");
    const uint64_t b0 = first - c.qt_first;
    const uint64_t q_begin = c.h_q_off[b0];
    n_q = c.h_q_off[b0 + nr] - q_begin;
    uint32_t* cnt = c.m_cnt.reserve(n_q + 1);
    uint32_t* cursor = c.m_first.reserve(nr + 1ULL);
    uint64_t* packed = c.m_sq_key.reserve(n_q + 2);
    uint64_t* hit_off = c.m_hit_off.reserve(n_q + 2);
    RVN_CUDA(cudaMemsetAsync(cursor, 0, (nr + 1ULL) * sizeof(uint32_t), c.stream));
    RVN_CUDA(cudaMemsetAsync(packed, 0, (n_q + 1) * sizeof(uint64_t), c.stream));
    if (c.i_n > 0 && n_q > 0) {
      JoinProbeKernel<<<CeilDiv(c.i_n, kThreads), kThreads, 0, c.stream>>>(
          jv, c.q_off.get(), q_begin, cursor, packed);
      UnpackJoin<<<CeilDiv(n_q, kThreads), kThreads, 0, c.stream>>>(packed, n_q, cnt);
      RVN_LAUNCH_CHECK();
      c.launches += 2;
    }
    if (n_q > 0) {
      ExclusiveScanU32(c, cnt, hit_off, n_q);
      n_hits = ReadU64(c, hit_off + n_q);
    } else {
      RVN_CUDA(cudaMemsetAsync(hit_off, 0, sizeof(uint64_t), c.stream));
    }
    TimerEnd(c);
    TimerBegin(c, "expand");
    hg = c.h_grp.reserve(n_hits + 1);
    hp = c.h_pos.reserve(n_hits + 1);
    if (n_hits > 0) {
      ExpandJoinKernel<<<CeilDiv(n_q, kThreads), kThreads, 0, c.stream>>>(
          c.i_org.get(), packed, n_q, hit_off, hg, hp);
      RVN_LAUNCH_CHECK();
      ++c.launches;
    }
    GatherU64<<<CeilDiv(nr + 1ULL, kThreads), kThreads, 0, c.stream>>>(
        hit_off, c.q_off.get() + b0, q_begin, nr + 1ULL, read_hit_off);
    RVN_LAUNCH_CHECK();
    ++c.launches;
    RVN_CUDA(cudaMemcpyAsync(h_rho.data(), read_hit_off, (nr + 1ULL) * sizeof(uint64_t),
                             cudaMemcpyDeviceToHost, c.stream));
    RVN_CUDA(cudaStreamSynchronize(c.stream));
    TimerEnd(c);
    c.r_filt_off.reserve(nr + 2ULL);
    for (uint32_t i = 0; i <= nr; ++i) c.r_filt_off.get()[i] = 0;
  } else {
  // ---- query records ----
  const uint64_t *qo, *d_read_off;
  ValView qv;  // query values: u32 for full sketches of k <= 15, else u64
  const std::vector<uint64_t>* h_read_off;
  uint64_t off_base_read;  // index of `first` inside the offsets arrays
  if (minhash) {
    if (!(c.q_valid && c.q_first <= first && last <= c.q_last)) {
      EnsureMicromizers(c, first, last);
    }
    qv = ValView{c.q_val.get(), c.q_is32 ? 1 : 0};
    qo = c.q_org.get();
    d_read_off = c.q_off.get();
    h_read_off = &c.h_q_off;
    off_base_read = first - c.q_first;
  } else {
    if (!(c.s_valid && c.s_first <= first && last <= c.s_last)) {
      EnsureSketch(c, first, last);
    }
    qv = ValView{c.s_val.get(), c.s_is32 ? 1 : 0};
    qo = c.s_org.get();
    d_read_off = c.s_off.get();
    h_read_off = &c.h_s_off;
    off_base_read = first - c.s_first;
  }
  const uint64_t q_begin = (*h_read_off)[off_base_read];
  n_q = (*h_read_off)[off_base_read + nr] - q_begin;

  const IndexView ix = IndexViewOf(c);

  // ---- probe + expand ----
  TimerBegin(c, "probe");
  uint32_t* cnt = c.m_cnt.reserve(n_q + 1);
  uint32_t* frst = c.m_first.reserve(n_q + 1);
  uint8_t* filt = c.m_filt.reserve(n_q + 1);
  uint64_t* hit_off = c.m_hit_off.reserve(n_q + 2);
  const bool suffix = KeptContiguous(c, avoid_equal, avoid_symmetric);
  if (n_q > 0) {
    if (suffix && n_q >= (1u << 16) && n_q < 0xFFFFFFFFULL) {
      // sort the queries by value, probe in that order, results back by index
      uint64_t* k1 = c.m_sq_key.reserve(n_q + 2);
      uint64_t* k2 = c.m_sq_key2.reserve(n_q);
      uint32_t* v1 = c.m_sq_idx.reserve(n_q);
      uint32_t* v2 = c.m_sq_idx2.reserve(n_q);
      IotaU32<<<CeilDiv(n_q, kThreads), kThreads, 0, c.stream>>>(v1, n_q);
      // FULL value order: consecutive probes then walk consecutive buckets, values
      // and postings (the reads of a warp fall into a few hundred bytes instead of
      // one 32-byte sector per probe per array)
      const int hi_bit = static_cast<int>(2 * c.prm.k);
      int w_q;
      ValView sorted_qv;
      if (qv.is32) {
        const uint32_t* src = static_cast<const uint32_t*>(qv.p) + q_begin;
        uint32_t* a32 = reinterpret_cast<uint32_t*>(k1);
        uint32_t* b32 = a32 + n_q + (n_q & 1);  // second half of k1 (8-byte aligned)
        w_q = RadixSortPairs(c, src, a32, b32, v1, v2, v1, n_q, 0, hi_bit);
        sorted_qv = ValView{w_q < 0 ? src : (w_q == 0 ? a32 : b32), 1};
      } else {
        const uint64_t* src = static_cast<const uint64_t*>(qv.p) + q_begin;
        w_q = RadixSortPairs(c, src, k1, k2, v1, v2, v1, n_q, 0, hi_bit);
        sorted_qv = ValView{w_q < 0 ? src : (w_q == 0 ? k1 : k2), 0};
      }
      const uint32_t* sorted_qi = w_q == 0 ? v2 : v1;
      // (a key buffer the sort did not end in receives the packed results)
      uint64_t* packed = (qv.is32 || w_q == 0) ? k2 : k1;
      ProbeSortedKernel<<<CeilDiv(n_q, kThreads), kThreads, 0, c.stream>>>(
          ix, sorted_qv, sorted_qi, qo, q_begin, n_q, avoid_equal, packed);
      UnpackProbe<<<CeilDiv(n_q, kThreads), kThreads, 0, c.stream>>>(packed, n_q, cnt, frst, filt);
      RVN_LAUNCH_CHECK();
      c.launches += (2 * c.prm.k + 7) / 8 + 6;
    } else {
      ProbeQueries(c, qv, qo, q_begin, n_q, avoid_equal, avoid_symmetric, cnt, frst, filt);
    }
    ExclusiveScanU32(c, cnt, hit_off, n_q);
    n_hits = ReadU64(c, hit_off + n_q);
  } else {
    RVN_CUDA(cudaMemsetAsync(hit_off, 0, sizeof(uint64_t), c.stream));
  }
  TimerEnd(c);
  TimerBegin(c, "expand");
  hg = c.h_grp.reserve(n_hits + 1);
  hp = c.h_pos.reserve(n_hits + 1);
  if (n_hits > 0) {
    if (suffix) {
      ExpandWarpKernel<<<CeilDiv(n_q, kThreads), kThreads, 0, c.stream>>>(
          ix, qo, q_begin, n_q, cnt, frst, hit_off, hg, hp);
    } else {
      ExpandKernel<<<CeilDiv(n_q, kThreads), kThreads, 0, c.stream>>>(
          ix, qv, qo, q_begin, n_q, avoid_equal, avoid_symmetric, cnt, frst,
          hit_off, hg, hp);
    }
    RVN_LAUNCH_CHECK();
    ++c.launches;
  }
  // per-read hit ranges
  GatherU64<<<CeilDiv(nr + 1ULL, kThreads), kThreads, 0, c.stream>>>(
      hit_off, d_read_off + off_base_read, q_begin, nr + 1ULL, read_hit_off);
  RVN_LAUNCH_CHECK();
  ++c.launches;
  RVN_CUDA(cudaMemcpyAsync(h_rho.data(), read_hit_off,
                           (nr + 1ULL) * sizeof(uint64_t),
                           cudaMemcpyDeviceToHost, c.stream));
  RVN_CUDA(cudaStreamSynchronize(c.stream));
  TimerEnd(c);

  // ---- filtered positions (stage 2 only) ----
  c.r_filt_off.reserve(nr + 2ULL);
  for (uint32_t i = 0; i <= nr; ++i) c.r_filt_off.get()[i] = 0;
  uint64_t n_filtered = 0;
  if (want_filtered && n_q > 0) {
    uint32_t* f32 = c.m_first.get();  // `first` is dead after ExpandKernel
    FilteredFlagsToU32<<<CeilDiv(n_q, kThreads), kThreads, 0, c.stream>>>(
        filt, n_q, f32);
    uint64_t* fpos = c.m_filt_off.reserve(n_q + 2);
    ExclusiveScanU32(c, f32, fpos, n_q);
    n_filtered = ReadU64(c, fpos + n_q);
    uint32_t* fout = c.m_filtered.reserve(n_filtered + 1);
    ScatterFiltered<<<CeilDiv(n_q, kThreads), kThreads, 0, c.stream>>>(
        filt, fpos, qo, q_begin, n_q, fout);
    RVN_LAUNCH_CHECK();
    c.launches += 2;
    // per-read offsets of the filtered list
    uint64_t* froff = c.m_ovl_off.reserve(nr + 2ULL);
    GatherU64<<<CeilDiv(nr + 1ULL, kThreads), kThreads, 0, c.stream>>>(
        fpos, d_read_off + off_base_read, q_begin, nr + 1ULL, froff);
    RVN_LAUNCH_CHECK();
    ++c.launches;
    uint32_t* hf = c.r_filtered.reserve(n_filtered + 1);
    RVN_CUDA(cudaMemcpyAsync(hf, fout, n_filtered * sizeof(uint32_t),
                             cudaMemcpyDeviceToHost, c.stream));
    RVN_CUDA(cudaMemcpyAsync(c.r_filt_off.get(), froff,
                             (nr + 1ULL) * sizeof(uint64_t),
                             cudaMemcpyDeviceToHost, c.stream));
    RVN_CUDA(cudaStreamSynchronize(c.stream));
  }

  }  // (probe path)

  if (c.keep_hits) {
    uint64_t* g = c.r_hit_grp.reserve(n_hits + 1);
    uint64_t* p = c.r_hit_pos.reserve(n_hits + 1);
    uint64_t* o = c.r_hit_off.reserve(nr + 2ULL);
    RVN_CUDA(cudaMemcpyAsync(g, hg, n_hits * sizeof(uint64_t),
                             cudaMemcpyDeviceToHost, c.stream));
    RVN_CUDA(cudaMemcpyAsync(p, hp, n_hits * sizeof(uint64_t),
                             cudaMemcpyDeviceToHost, c.stream));
    for (uint32_t i = 0; i <= nr; ++i) o[i] = h_rho[i];
    RVN_CUDA(cudaStreamSynchronize(c.stream));
    c.r_n_hits = n_hits;
  }

  // ---- chain ----
  const uint64_t n_ovl =
      ChainGroupedHits(c, hg, hp, read_hit_off, h_rho, c.d_ids.get() + first, nr, n_hits, n_q);
  const rvn_overlap* ordered = c.m_ovl.get();
  const uint64_t* ooff = c.m_ovl_off.get();

  // ---- results to the host ----
  if (fetch) {
    rvn_overlap* ho = c.r_ovl.reserve(n_ovl + 1);
    uint64_t* hoff = c.r_ovl_off.reserve(nr + 2ULL);
    RVN_CUDA(cudaMemcpyAsync(ho, ordered, n_ovl * sizeof(rvn_overlap),
                             cudaMemcpyDeviceToHost, c.stream));
    RVN_CUDA(cudaMemcpyAsync(hoff, ooff, (nr + 1ULL) * sizeof(uint64_t),
                             cudaMemcpyDeviceToHost, c.stream));
    RVN_CUDA(cudaStreamSynchronize(c.stream));
  }
  c.r_n_ovl = n_ovl;
  c.m_hits = n_hits;
  c.m_first_read = first;
  c.m_last_read = last;
  c.r_valid = fetch;

  uint64_t qbases = 0;
  for (uint32_t r = first; r < last; ++r) qbases += c.h_len[r];
  c.stats.query_bases += qbases;
  c.stats.query_records += n_q;
  c.stats.hits += n_hits;
  c.stats.overlaps += n_ovl;
}

}  // namespace rvn
