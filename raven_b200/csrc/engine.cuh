// raven_b200 — overlap engine context and stage entry points (host side).
//
// Data layout in HBM (all SoA, 8-byte fields, see DESIGN.md):
//   reads      words[]           2-bit packed, biosoup layout, 0.25 B/base
//   sketch     s_val[], s_org[]  minimizer records in (read, position) order
//   queries    q_val[], q_org[]  micromizers (len/k smallest per read)
//   index      i_val[], i_org[]  sketch stably sorted by value + bucket table
//   hits       h_grp[], h_pos[]  ram "Match" records grouped by query read
//   overlaps   rvn_overlap[]     32 B records grouped by query read
#pragma once

#include <string>
#include <vector>

#include "../../include/raven_b200.h"
#include "common.cuh"

namespace rvn {

struct Params {
  uint32_t k = 15, w = 5, bandwidth = 500, chain = 4, matches = 100;
  uint32_t gap = 10000;
};

// k-mer positions handled by one CTA of the sketch kernels
constexpr uint32_t kSketchTile = 2048;
constexpr uint32_t kSketchThreads = 256;
constexpr uint32_t kMaxWindow = 256;  // w limit (halo staged in shared memory)

struct PhaseTimer {
  std::vector<const char*> names;
  std::vector<float> ms;
  std::vector<std::pair<cudaEvent_t, cudaEvent_t>> pending;
  std::vector<cudaEvent_t> pool;
};

struct Ctx {
  int device = 0;
  cudaStream_t stream = nullptr;
  bool own_stream = false;
  // option "async_upload": the packed bases travel on a copy stream in chunks; the
  // sketch kernel of the next call starts on the reads that have arrived
  int64_t async_upload = 0;
  cudaStream_t copy_stream = nullptr;
  cudaEvent_t up_fence = nullptr;
  std::vector<cudaEvent_t> up_events;   // one per chunk (reused)
  std::vector<uint32_t> up_read_end;    // reads [.., up_read_end[i]) are complete after chunk i
  uint32_t up_chunks = 0;
  bool up_pending = false;
  bool p_off_uploaded = false;  // stage-1 pile offsets already on the device
  std::string err;
  Params prm;
  bool keep_hits = false;
  rvn_stats stats{};

  // ---- reads ----
  uint32_t n_reads = 0;
  uint64_t n_words = 0;
  DevBuf<uint64_t> d_words, d_woff;
  DevBuf<uint32_t> d_len, d_ids;
  std::vector<uint64_t> h_woff;
  std::vector<uint32_t> h_len, h_ids;
  bool ids_identity = true;  // id == index (needed by the device-side gather)
  uint32_t res_first = 0, res_last = 0;  // reads whose bases are in HBM
  // sketch tiles: tile_off[r] = first tile of read r (depends on k)
  std::vector<uint64_t> h_tile_off;
  DevBuf<uint64_t> d_tile_off;
  DevBuf<uint32_t> d_tile_read;  // read of every tile
  uint32_t tiles_k = 0;

  // ---- current sketch (full minimizers of reads [s_first, s_last)) ----
  bool s_valid = false;
  uint32_t s_first = 0, s_last = 0;
  uint64_t s_n = 0;
  DevBuf<uint64_t> s_val, s_org, s_off;  // s_off: (s_last-s_first)+1
  bool s_is32 = false;  // s_val holds u32 values (2k <= 30 bits)
  std::vector<uint64_t> h_s_off;
  DevBuf<uint32_t> tile_cnt;
  DevBuf<uint64_t> tile_out, tile_status;

  // ---- current micromizer set (of reads [q_first, q_last)) ----
  bool q_valid = false;
  uint32_t q_first = 0, q_last = 0;
  uint64_t q_n = 0;
  DevBuf<uint64_t> q_val, q_org, q_off;
  bool q_is32 = false;  // q_val holds u32 values
  std::vector<uint64_t> h_q_off;
  // micromizer thresholds of reads [qt_first, qt_last): record (value, position) of read r
  // is a micromizer iff value < qt_val[r] || (value == qt_val[r] && position < qt_pos[r])
  bool qt_valid = false;
  uint32_t qt_first = 0, qt_last = 0;
  DevBuf<uint64_t> qt_val;
  DevBuf<uint32_t> qt_pos;
  int t_b_low = 0;  // the bare keys of the upper tier are sorted above this many low bits
  uint64_t group_count_min = 0;  // fewer keys per group of equal upper bits: full sort instead
  bool i_from_sketch = false;  // the index holds the FULL sketches of reads [i_first, i_last)
  int64_t self_join = 1;       // option: stage-1 hits by a self-join over the index

  // ---- index ----
  bool i_valid = false;
  uint32_t i_first = 0, i_last = 0;
  uint64_t i_n = 0, i_keys = 0;
  DevBuf<uint64_t> i_val, i_org, i_val_alt, i_org_alt;
  bool i_is32 = false;  // i_val holds u32 values
  int i_shift = 0;             // bucket = value >> i_shift
  uint64_t i_limit = ~0ULL;    // tiered build: only values <= i_limit are in the index
  // tiers (index.cu): staging of the probe-able tier and the bare keys beyond it
  DevBuf<uint32_t> t_cnt;
  DevBuf<uint64_t> t_off, t_aval, t_aorg, t_b0, t_b1, t_b2, t_narrow;
  const uint32_t* t_sorted_b = nullptr;
  uint64_t t_nb = 0;
  uint64_t tier_min_records = 1ULL << 18;  // smaller index batches are not worth a partition
  DevBuf<uint32_t> i_bucket;
  int i_bucket_bits = 0;
  DevBuf<uint64_t> i_gaps;  // long empty stretches of the bucket table (index.cu)
  DevBuf<uint64_t> i_hist;  // run-length histogram of the keys + #keys (index.cu)
  uint32_t occurrence = 0xFFFFFFFFu;
  bool i_sorted_ids = false;  // postings of a key are in ascending read-id order
  bool ids_ascending = true;  // read ids never decrease with the read index
  DevBuf<uint8_t> sort_tmp;

  // ---- map ----
  DevBuf<uint32_t> m_cnt, m_first;
  DevBuf<uint8_t> m_filt;
  DevBuf<uint64_t> m_hit_off;  // per query record (+1)
  DevBuf<uint64_t> m_sq_key, m_sq_key2;  // queries sorted by value (probe order)
  DevBuf<uint32_t> m_sq_idx, m_sq_idx2;
  DevBuf<uint64_t> h_grp, h_pos;
  DevBuf<uint64_t> m_read_hit_off;  // per query read (+1)
  DevBuf<uint64_t> m_scratch64;     // oversize chain scratch
  DevBuf<uint32_t> m_scratch32, m_fallback;
  // split chain path: pair descriptors, pair-contiguous hits, overlap keys
  DevBuf<uint32_t> m_desc, m_desc_cnt, m_desc_idx, m_desc_cnt2, m_desc_idx2, m_gdiag,
      m_oidx, m_oidx2;
  DevBuf<uint64_t> m_gpos, m_group_loc, m_okey, m_okey2, m_starts;
  DevBuf<uint32_t> m_bounds;
  DevBuf<rvn_overlap> m_ovl_raw, m_ovl, m_ovl_tmp;
  DevBuf<uint64_t> m_ovl_loc;  // per read: base<<24 | count  (raw placement)
  DevBuf<uint64_t> m_ovl_off;
  DevBuf<uint64_t> m_counter;
  DevBuf<uint32_t> m_filtered;
  DevBuf<uint64_t> m_filt_off;
  DevBuf<uint64_t> scan_tmp;
  uint64_t m_hits = 0;
  uint32_t m_first_read = 0, m_last_read = 0;

  // host-side results of the last map
  PinBuf<rvn_overlap> r_ovl;
  PinBuf<uint64_t> r_ovl_off;
  PinBuf<uint32_t> r_filtered;
  PinBuf<uint64_t> r_filt_off;
  uint64_t r_n_ovl = 0;
  bool r_valid = false;
  PinBuf<uint64_t> r_hit_grp, r_hit_pos, r_hit_off;
  uint64_t r_n_hits = 0;

  // introspection staging
  PinBuf<uint64_t> x_val, x_org, x_off;

  // ---- piles ----
  DevBuf<int32_t> p_diff;
  DevBuf<uint16_t> p_data;
  DevBuf<uint64_t> p_off;
  DevBuf<rvn_overlap> p_ovl;

  // ---- per-read overlap lists (gather.cu) ----
  int g_cur = 0;
  uint64_t g_total = 0;
  DevBuf<rvn_overlap> g_list[2], g_stage;
  DevBuf<uint64_t> g_off, g_off_alt, g_rhs_off, g_t_off, g_pairs;
  DevBuf<uint32_t> g_cnt, g_kept, g_key, g_idx, g_key2, g_idx2, g_rhs_cnt,
      g_total_cnt;

  // ---- POA (poa.cu) ----
  DevBuf<uint32_t> po_win_first, po_seq_begin, po_seq_end, po_cons_len, po_cov, po_list;
  DevBuf<uint64_t> po_seq_off, po_d_cons_off;
  DevBuf<uint8_t> po_bases, po_quals, po_cons, po_status, po_scratch;
  std::vector<uint64_t> po_cons_off, po_out_off;
  std::vector<uint8_t> po_h_status, po_h_cons, po_out_cons;
  std::vector<uint32_t> po_h_clen, po_h_cov, po_out_cov;
  uint64_t po_cells = 0;
  uint32_t po_n_windows = 0;
  bool po_has_cov = false, poa_valid = false;

  // ---- stage-1 results ----
  PinBuf<rvn_overlap> st_ovl;  // pinned: the D2H of the results runs at link speed
  PinBuf<uint64_t> st_ovl_off;
  PinBuf<uint16_t> st_pile;
  std::vector<uint64_t> st_pile_off;
  uint64_t st_mapped = 0;
  bool st_valid = false;
  bool st_piles_on_device = false;  // c.p_data / c.p_off still hold the piles of that call

  // ---- read ownership of the stage-1 tail: read r is owned iff r % own_mod ==
  // own_rem (1 / 0 = every read: the single-GPU path) ----
  uint32_t own_mod = 1, own_rem = 0;

  // ---- multi-GPU partition / exchange staging (dist.cu) ----
  DevBuf<uint64_t> ds_split_val, ds_split_org, ds_qsplit_val, ds_qsplit_org;
  DevBuf<uint64_t> ds_grouped_grp, ds_grouped_pos, ds_rel_off, ds_seg_start, ds_seg_base,
      ds_bounds, ds_q_off;
  DevBuf<uint32_t> ds_masked, ds_hit_lhs, ds_read_cnt, ds_flag, ds_own_ids;
  DevBuf<rvn_overlap> ds_ovl_split, ds_merged;
  // results of the owned reads (pinned host)
  PinBuf<rvn_overlap> ds_r_ovl;
  PinBuf<uint64_t> ds_r_ovl_off, ds_r_pile_off;
  PinBuf<uint16_t> ds_r_pile;
  uint32_t ds_n_own = 0;
  bool ds_results_valid = false;
  // peer-memory exchange: own receive arena + the peers' arenas (CUDA IPC)
  void* x_arena = nullptr;
  uint64_t x_cap = 0;
  uint32_t x_rank = 0;
  std::vector<void*> x_peers;
  std::vector<cudaStream_t> x_streams;

  // pinned scalars for small D2H reads
  PinBuf<uint64_t> pin64;

  PhaseTimer timer;
  uint64_t launches = 0;
};

// ---- utilities (scan.cu) ----
// out[i] = sum_{j<i} in[j] for i in [0, n]; out has n + 1 entries.
void ExclusiveScanU32(Ctx& c, const uint32_t* in, uint64_t* out, uint64_t n);
uint64_t ReadU64(Ctx& c, const uint64_t* dptr);  // sync D2H of one value

void TimerBegin(Ctx& c, const char* name);
void TimerEnd(Ctx& c);
void TimerCollect(Ctx& c);
void TimerReset(Ctx& c);

// ---- sketch.cu ----
void EnsureTiles(Ctx& c);
// full minimizers of reads [first,last) into c.s_* (no-op if already there)
void EnsureSketch(Ctx& c, uint32_t first, uint32_t last);
// micromizers of reads [first,last) into c.q_* (needs the sketch of a range
// that contains [first,last))
void WaitUpload(Ctx& c);  // the context's stream waits for an asynchronous upload
void EnsureMicromizers(Ctx& c, uint32_t first, uint32_t last);
void EnsureThresholds(Ctx& c, uint32_t first, uint32_t last);

// ---- index.cu ----
// value_limit: records whose value exceeds it are counted (occurrence threshold)
// but not indexed - the caller guarantees that no query value is larger
void BuildIndex(Ctx& c, uint32_t first, uint32_t last, bool minhash,
                uint64_t value_limit = ~0ULL);
uint64_t MaxMicromizerValue(Ctx& c, uint32_t first, uint32_t last);
// index from device records already in (read, position) order (values as u32
// or u64, see ValView)
void BuildIndexFrom(Ctx& c, ValView src_val, const uint64_t* src_org, uint64_t n,
                    uint64_t index_bases, uint64_t value_limit = ~0ULL);

// ---- radix.cu ---- stable LSD radix sort on key bits [begin_bit, end_bit).
// The source arrays are only read (src may alias buffer b: it is dead once the
// first pass is through); the result lands in buffer a (return 0) or b (return
// 1); -1 = nothing to do, the source order is the result.
int RadixSortPairs(Ctx& c, const uint32_t* src_keys, uint32_t* keys_a, uint32_t* keys_b,
                   const uint64_t* src_vals, uint64_t* vals_a, uint64_t* vals_b, uint64_t n,
                   int begin_bit, int end_bit, bool descending = false);
int RadixSortPairs(Ctx& c, const uint64_t* src_keys, uint64_t* keys_a, uint64_t* keys_b,
                   const uint64_t* src_vals, uint64_t* vals_a, uint64_t* vals_b, uint64_t n,
                   int begin_bit, int end_bit, bool descending = false);
int RadixSortPairs(Ctx& c, const uint32_t* src_keys, uint32_t* keys_a, uint32_t* keys_b,
                   const uint32_t* src_vals, uint32_t* vals_a, uint32_t* vals_b, uint64_t n,
                   int begin_bit, int end_bit, bool descending = false);
int RadixSortPairs(Ctx& c, const uint64_t* src_keys, uint64_t* keys_a, uint64_t* keys_b,
                   const uint32_t* src_vals, uint32_t* vals_a, uint32_t* vals_b, uint64_t n,
                   int begin_bit, int end_bit, bool descending = false);
int RadixSortKeys(Ctx& c, const uint32_t* src_keys, uint32_t* keys_a, uint32_t* keys_b,
                  uint64_t n, int begin_bit, int end_bit);
// run-length histogram of the index keys (c.i_hist: 65536 u64 bins + #keys), filled by the build
uint64_t* IndexHistogram(Ctx& c);
uint32_t ThresholdFromHistogram(Ctx& c, const uint64_t* h_hist, uint64_t n_keys,
                                double frequency, bool* needs_long_runs);
uint32_t FilterIndex(Ctx& c, double frequency);

// ---- map.cu ----
// fetch = copy the ordered overlaps to the host (rvn_map); stage 1 keeps them
// on the device (c.m_ovl, c.m_ovl_off, c.r_n_ovl)
void MapRange(Ctx& c, uint32_t first, uint32_t last, bool avoid_equal,
              bool avoid_symmetric, bool minhash, bool want_filtered,
              bool fetch = true);

// seed lookup of the queries [q_begin, q_begin + n_q) in their own order (seed.cuh): per
// query the kept count and the first posting; the over-threshold flags go to filt
// unless it is null
void ProbeQueries(Ctx& c, ValView q_val, const uint64_t* q_org, uint64_t q_begin, uint64_t n_q,
                  bool avoid_equal, bool avoid_symmetric, uint32_t* cnt, uint32_t* first,
                  uint8_t* filt);

// chains hits grouped by query read (see map.cu); overlaps land in c.m_ovl
// lhs_ids[i] = id of query read i of the batch (device)
uint64_t ChainGroupedHits(Ctx& c, const uint64_t* hg, const uint64_t* hp,
                          const uint64_t* read_hit_off,
                          const std::vector<uint64_t>& h_rho, const uint32_t* lhs_ids,
                          uint32_t nr, uint64_t n_hits, uint64_t n_q);

// ---- gather.cu ----
void GatherReset(Ctx& c);
void GatherFlush(Ctx& c, const rvn_overlap* ovl, const uint64_t* q_ovl_off,
                 uint64_t m, uint32_t k0, uint32_t k1, uint64_t kmax);
void GatherFetch(Ctx& c);

// ---- dist.cu ---- key-partitioned index, reads owned by id mod parts
// which: 0 = full minimizers, 1 = micromizers; records of reads [first,last)
// stably partitioned by value % parts; counts[parts]
void DistSketchSplit(Ctx& c, uint32_t first, uint32_t last, int which, uint32_t parts,
                     const uint64_t** d_val, const uint64_t** d_org, uint64_t* counts);
void DistHitsSplit(Ctx& c, const uint64_t* d_qval, const uint64_t* d_qorg, uint64_t n_q,
                   bool avoid_equal, bool avoid_symmetric, uint32_t parts, uint32_t n_query,
                   const uint64_t** d_grp, const uint64_t** d_pos, const uint32_t** d_lhs,
                   uint64_t* counts);
void DistChainOwned(Ctx& c, const uint64_t* d_grp, const uint64_t* d_pos,
                    const uint32_t* d_lhs, uint64_t n_hits, uint32_t n_seg,
                    const uint64_t* h_seg_off, uint32_t mod, uint32_t rem, uint32_t n_query,
                    const rvn_overlap** d_ovl, uint64_t* n_ovl);
void DistOverlapsSplit(Ctx& c, uint32_t parts, uint32_t self, const rvn_overlap** d_out,
                       uint64_t* counts);
void DistStage1Begin(Ctx& c, uint32_t parts, uint32_t rank);
void DistStage1Add(Ctx& c, const rvn_overlap* d_ovl, uint64_t n_ovl, uint32_t n_seg,
                   const uint64_t* h_seg_off, uint32_t n_query, uint64_t kmax, uint64_t qb);
void DistStage1End(Ctx& c);
void ArenaClosePeers(Ctx& c);
void ArenaExport(Ctx& c, uint64_t bytes, void* handle64);
void ArenaImport(Ctx& c, uint32_t parts, uint32_t rank, const void* handles);
void ArenaPut(Ctx& c, uint32_t dest, uint64_t dst_off, const void* d_src, uint64_t bytes);
void ArenaFlush(Ctx& c);
void ArenaRelease(Ctx& c);

// ---- editdist.cu ---- batched global edit distance of read substrings
void StagePileRegions(Ctx& c, uint32_t coverage, uint32_t* h_begin, uint32_t* h_end,
                      uint16_t* h_median, uint8_t* h_invalid);
void AlignBreakingPoints(Ctx& c, uint64_t n, const uint32_t* q_read, const uint32_t* q_begin,
                         const uint32_t* q_len, const uint8_t* strand, const uint32_t* t_read,
                         const uint32_t* t_begin, const uint32_t* t_len, uint32_t window,
                         const uint64_t* bp_off, int32_t* distance, uint32_t* bp);
void EditDistanceBatch(Ctx& c, uint64_t n, const uint32_t* lhs_read, const uint32_t* lhs_begin,
                       const uint32_t* lhs_len, const uint32_t* rhs_read,
                       const uint32_t* rhs_begin, const uint32_t* rhs_len,
                       const uint8_t* strand, const int32_t* limit, int32_t* out);

// ---- pile.cu ----
// data: device u16 bins, off: device u64 offsets (n_piles + 1)
void PileAddLayersDevice(Ctx& c, uint16_t* d_data, const uint64_t* d_off,
                         const uint64_t* h_off, uint32_t n_piles,
                         const rvn_overlap* d_ovl, uint64_t n_ovl);

// ---- poa.cu ---- racon window consensus over a flat batch of windows
void PoaBatch(Ctx& c, uint32_t n_windows, const uint32_t* h_win_first,
              const uint64_t* h_seq_off, const uint8_t* h_bases, const uint8_t* h_quals,
              const uint32_t* h_seq_begin, const uint32_t* h_seq_end, int m, int n,
              int gap, bool trim, bool tgs, bool want_coverage);

// Pile::AddKmers low-complexity test for (read index, position) pairs
void KmerComplexity(Ctx& c, const uint32_t* h_read_idx, const uint32_t* h_pos,
                    uint64_t n, uint32_t k, uint8_t* h_keep);

}  // namespace rvn
