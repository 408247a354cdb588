// Device-side data layout and warp-level building blocks of the B200 query path.
//
// What each piece replaces in the reference (paths relative to /root/reference):
//   decode_block        BlockSegmentPostings::load_block -> BlockDecoder::uncompress_block_sorted /
//                       uncompress_block_unsorted (src/postings/block_segment_postings.rs:343-391,
//                       src/postings/compression/mod.rs:105-150; BitPacker4x of crate bitpacking)
//   bm25_score          Bm25Weight::score / tf_factor (src/query/bm25.rs:158-175) +
//                       FieldNormReader::fieldnorm_id (src/fieldnorm/reader.rs:128-136)
//   TopK (CTA buffer)   TopNHeap (src/collector/sort_key/sort_by_score.rs:121-161): same accepted set,
//                       obtained by threshold filtering + exact selection instead of a binary heap
//   first_block_ge      SkipReader::seek (src/postings/skip.rs:263-275) — random access over the
//                       block table instead of a linear walk
//
// No tensor cores: the path is integer unpack + one f32 divide per posting (SURVEY.md §8d).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace tq {

constexpr uint32_t kTerminated = 0x7FFFFFFFu;  // src/docset.rs:12
constexpr uint32_t kNoList = 0xFFFFFFFFu;
constexpr unsigned kFull = 0xFFFFFFFFu;

constexpr int kThreads = 256;                 // 8 warps per CTA
constexpr int kWarps = kThreads / 32;
constexpr uint32_t kCap = 2048;               // CTA candidate buffer (u64 keys), power of two
constexpr uint32_t kRoundMargin = kWarps * 128;  // most keys one round of 8 warps can push
constexpr uint32_t kTileDocs = 8192;          // OR: doc-id tile width held in shared memory
constexpr uint32_t kTfRows = 17;              // term frequencies below this use the precomputed factor table (tf_bits <= 4 => tf <= 16)

// One posting list of one (segment, field, term), device resident.  Built once per term by
// k_build_tables from the raw tantivy bytes and cached for the life of the segment (segments
// are immutable, ARCHITECTURE.md "Searcher").
struct ListDesc {
  const uint8_t* blocks;      // the list's bit-packed blocks, copied 16-byte aligned when the table is built
                              // (posting lists start at arbitrary byte offsets inside the .idx body)
  const uint32_t* last_doc;   // [n_total] last doc id of every block; entry n_blocks = last tail doc
  const uint2* blk;           // [n_blocks + 1] .x byte offset from `blocks`, .y packed meta
  const uint4* tab4;          // [n_total] {last_doc, byte offset, meta, last doc of the previous block (0xFFFFFFFF: none)}
                              // one 16-byte record per block so that a 32-wide probe yields position AND record
  const uint32_t* tail_docs;  // [tail_n] the VInt tail, decoded at build time
  const uint32_t* tail_tfs;   // [tail_n]
  const uint8_t* fieldnorm;   // the segment's fieldnorm ids for this field; null => constant id 1
  uint32_t n_blocks;          // full 128-doc blocks
  uint32_t tail_n;            // docs in the VInt tail (0..127)
  uint32_t n_total;           // n_blocks + (tail_n ? 1 : 0)
  uint32_t doc_freq;
  uint32_t has_freq;          // term frequencies are stored (else tf = 1)
  uint32_t build_status;      // 0 ok, else corrupt
};
// meta bits: [0:5) doc_bits, bit 6 strict-delta, [8:14) tf_bits, [16:24) block-max fieldnorm id,
// [24:32) block-max tf code (255 = saturated), see src/postings/skip.rs:16-22,205-253.

struct QList {  // one clause of one query in one segment
  uint32_t list_id;
  float weight;        // Bm25Weight.weight
  uint32_t cache_idx;  // which 256-entry tf-norm table
  uint32_t pad;        // k_or_strip: thin-clause cache slot; k_bool: role | group << 2
};
struct QSeg {  // one (query, segment): what Collector::collect_segment sees
  uint32_t query;
  uint32_t lists_base;  // index into qlists; AND: ascending doc_freq (leader first); OR/TERM: clause order
  uint32_t n_lists;
  uint32_t max_doc;
  uint32_t segment_ord;
  uint32_t flags;        // bit 0: every clause reads the same fieldnorm array (`fieldnorm` below), bit 1: every weight finite and >= 0;
                         // k_bool: [8:16) MUST groups, [16:24) SHOULD clauses needed
  const uint8_t* alive;  // alive bitset bytes or null
  const uint8_t* fieldnorm;  // shared fieldnorm ids (padded to a multiple of kTileDocs) when flags&1
};
struct Unit {  // one CTA's share of a QSeg
  uint32_t qseg;
  uint32_t begin, end;  // TERM/AND: block range of the (leader) list; OR: tile range
  uint32_t pad;
};
struct DQuery {
  uint32_t k;
  uint32_t cand_base;  // first slot of this query's candidate region
  uint32_t cand_cap;
  uint32_t op;
};
struct QState {  // zeroed before every run
  unsigned int theta;       // score key: lower bound of the final k-th best score
  unsigned int cand_count;
};
struct Cand { uint32_t score_key, segment_ord, doc, pad; };

struct BatchParams {
  const ListDesc* lists;
  const float* caches;  // [n_caches][256] tf-norm tables (bm25.rs:58-69)
  const float* tf_tables;  // [n_caches][kTfRows][256]: tf / (tf + norm[id]) for tf < kTfRows
  const QList* qlists;
  const QSeg* qsegs;
  const Unit* units;
  const DQuery* queries;
  QState* qstate;
  Cand* cands;
  float* res_scores;
  uint32_t* res_segs;
  uint32_t* res_docs;
  uint32_t* res_counts;
  uint32_t res_stride;
  uint32_t n_queries;
  unsigned long long* counters;  // [8] k_or_strip diagnostics, tq_stats.or_windows
  // Unused.  Every kernel takes BatchParams by value; with 16 bytes less, ptxas schedules k_tile's parameter loads
  // differently and the default workload measured 0.2 % slower (B200, 1000 W power limit).
  uint32_t reserved[4];
  uint32_t* ovf;                // set by k_final when a query was handed more candidates than its region holds (tile engine only), or null
};

// ---- small helpers ---------------------------------------------------------------------------
__device__ __forceinline__ uint32_t score_to_key(float f) {  // order preserving for every float
  const uint32_t u = __float_as_uint(f);
  return u ^ ((u >> 31) ? 0xFFFFFFFFu : 0x80000000u);
}
__device__ __forceinline__ float key_to_score(uint32_t k) {
  return __uint_as_float((k & 0x80000000u) ? (k ^ 0x80000000u) : ~k);
}
// Float lower bound equivalent to a key threshold, for cheap pre-filtering: every score whose key is
// >= (k << 32) satisfies score >= threshold_score(k). No threshold yet (k == 0, or a NaN pattern) => -inf.
__device__ __forceinline__ float threshold_score(uint32_t k) {
  const float f = key_to_score(k);
  return (k == 0u || f != f) ? __int_as_float(0xff800000) : f;
}
__device__ __forceinline__ unsigned long long make_key(float score, uint32_t doc) {
  // larger key = better hit: higher score, then LOWER doc id (sort_by_score.rs:104-110)
  return ((unsigned long long)score_to_key(score) << 32) | (unsigned long long)(0xFFFFFFFFu - doc);
}
__device__ __forceinline__ uint32_t lanemask_lt(uint32_t lane) { return (1u << lane) - 1u; }

__device__ __forceinline__ uint32_t warp_incl_scan(uint32_t v, uint32_t lane) {
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const uint32_t n = __shfl_up_sync(kFull, v, o);
    if ((int)lane >= o) v += n;
  }
  return v;
}
__device__ __forceinline__ uint32_t warp_min(uint32_t v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = min(v, __shfl_xor_sync(kFull, v, o));
  return v;
}

// ---- K1: one warp decodes one 128-doc block ----------------------------------------------------
// Split in two so that the HBM round trips of block b+1 overlap the scoring of block b:
//   fetch_issue   block-table record -> the two 16-byte vectors of doc bits and of tf bits this lane needs
//   fetch_decode  funnel-shift the 4+4 fields out, add 1 to tf (v7), inclusive prefix sum of the doc gaps
// BitPacker4x layout: value j sits in bit stream j&3 at bit (j>>2)*b; word w of stream c is the c-th word of
// 16-byte vector w.  Lane L takes values 4L..4L+3 = row L of the four streams = ONE vector (plus the next one
// when the field straddles a word).  Blocks are 16-byte aligned in the cached copy, so these are plain
// LDG.128; a warp's 32 loads cover the block's b vectors contiguously.
// Packed posting vectors are read exactly once: fetch them around L1 so that they do not evict what IS re-used
// there (the tf-factor table, block records, fieldnorm lines).
__device__ __forceinline__ uint4 ldg_stream(const uint4* p) {
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
  return r;
}

struct BlockFetch {
  uint4 dlo, dhi, tlo, thi;
  uint32_t meta;  // 0xFFFFFFFF marks the VInt tail pseudo block
  uint32_t prev;  // last doc of the previous block
};

__device__ __forceinline__ void fetch_issue(const ListDesc& L, uint32_t b, uint32_t lane, BlockFetch& f) {
  if (b >= L.n_blocks) { f.meta = 0xFFFFFFFFu; return; }
  const uint2 rec = __ldg(L.blk + b);
  f.meta = rec.y;
  f.prev = b ? __ldg(L.last_doc + b - 1) : 0u;
  const uint32_t db = rec.y & 31u, tb = (rec.y >> 8) & 63u;
  const uint4* v = reinterpret_cast<const uint4*>(L.blocks + rec.x);
  const uint32_t wd = (lane * db) >> 5;
  f.dlo = ldg_stream(v + wd);
  f.dhi = ldg_stream(v + wd + 1);  // may belong to the next field/block; masked out when not needed (copy is padded)
  if (L.has_freq) {
    const uint32_t wt = db + ((lane * tb) >> 5);
    f.tlo = ldg_stream(v + wt);
    f.thi = ldg_stream(v + wt + 1);
  }
}

__device__ __forceinline__ void fetch_decode(const ListDesc& L, uint32_t b, const BlockFetch& f, uint32_t lane,
                                             uint32_t (&doc)[4], uint32_t (&tf)[4]) {
  if (f.meta == 0xFFFFFFFFu) {  // VInt tail, decoded when the table was built
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const uint32_t j = lane * 4 + i;
      const bool v = j < L.tail_n;
      doc[i] = v ? __ldg(L.tail_docs + j) : kTerminated;
      tf[i] = v ? __ldg(L.tail_tfs + j) : 1u;
    }
    return;
  }
  const uint32_t meta = f.meta;
  const uint32_t db = meta & 31u, strict = (meta >> 6) & 1u, tb = (meta >> 8) & 63u;
  uint32_t d0, d1, d2, d3;
  {
    const uint32_t sh = (lane * db) & 31u;
    const uint32_t mask = (1u << db) - 1u;  // db < 32 (skip.rs:16-22)
    d0 = __funnelshift_r(f.dlo.x, f.dhi.x, sh) & mask;
    d1 = __funnelshift_r(f.dlo.y, f.dhi.y, sh) & mask;
    d2 = __funnelshift_r(f.dlo.z, f.dhi.z, sh) & mask;
    d3 = __funnelshift_r(f.dlo.w, f.dhi.w, sh) & mask;
  }
  if (L.has_freq) {
    const uint32_t sh = (lane * tb) & 31u;
    const uint32_t mask = tb >= 32u ? 0xFFFFFFFFu : ((1u << tb) - 1u);
    tf[0] = (__funnelshift_r(f.tlo.x, f.thi.x, sh) & mask) + strict;  // v7: tf-1 stored (mod.rs:134-150)
    tf[1] = (__funnelshift_r(f.tlo.y, f.thi.y, sh) & mask) + strict;
    tf[2] = (__funnelshift_r(f.tlo.z, f.thi.z, sh) & mask) + strict;
    tf[3] = (__funnelshift_r(f.tlo.w, f.thi.w, sh) & mask) + strict;
  } else {
    tf[0] = tf[1] = tf[2] = tf[3] = 1u;
  }
  // inclusive prefix sum of the (strict) deltas across the 128 values
  const uint32_t s0 = d0 + strict, s1 = s0 + d1 + strict, s2 = s1 + d2 + strict, s3 = s2 + d3 + strict;
  const uint32_t incl = warp_incl_scan(s3, lane);
  // offset 0 means "no previous doc" for strict deltas: predecessor is -1 (mod.rs:112-113)
  const uint32_t base = ((strict && f.prev == 0u) ? 0xFFFFFFFFu : f.prev) + (incl - s3);
  doc[0] = base + s0; doc[1] = base + s1; doc[2] = base + s2; doc[3] = base + s3;
}

__device__ __forceinline__ void decode_block(const ListDesc& L, uint32_t b, uint32_t lane, uint32_t (&doc)[4], uint32_t (&tf)[4]) {
  BlockFetch f;
  fetch_issue(L, b, lane, f);
  fetch_decode(L, b, f, lane, doc, tf);
}

// ---- K2: BM25 of one posting (f32, reference operation order, no contraction) -------------------
// score = weight * (tf / (tf + norm[fieldnorm_id]))  (bm25.rs:158-175).  The inner factor depends only on
// (tf, fieldnorm id) for a given average fieldnorm, so it is tabulated per batch for tf < kTfRows with the
// very same IEEE operations (k_build_tf_tables); larger tfs take the divide.
struct Scorer {
  float weight;
  const float* cache;     // [256] norms
  const float* tf_table;  // [kTfRows][256]
};
__device__ __noinline__ float bm25_factor_large_tf(const float* __restrict__ cache, uint32_t id, uint32_t tf) {
  const float t = __uint2float_rn(tf);
  return __fdiv_rn(t, __fadd_rn(t, __ldg(cache + id)));
}
__device__ __forceinline__ float bm25_score_id(const Scorer& sc, uint32_t id, uint32_t tf) {
  const float fac = tf < kTfRows ? __ldg(sc.tf_table + (tf << 8) + id) : bm25_factor_large_tf(sc.cache, id, tf);
  return __fmul_rn(sc.weight, fac);
}
__device__ __forceinline__ float bm25_score(const Scorer& sc, const uint8_t* __restrict__ fieldnorm, uint32_t doc, uint32_t tf) {
  const uint32_t id = fieldnorm ? (uint32_t)__ldg(fieldnorm + doc) : 1u;  // constant fieldnorm 1 -> id 1
  return bm25_score_id(sc, id, tf);
}
__device__ __forceinline__ Scorer make_scorer(const BatchParams& P, const QList& ql) {
  return Scorer{ql.weight, P.caches + 256u * ql.cache_idx, P.tf_tables + (size_t)(kTfRows * 256u) * ql.cache_idx};
}

// ---- first block whose last_doc >= target, searching [from, n) (SkipReader::seek) ---------------
// Warp-cooperative: one coalesced probe of 32 entries at `from`, then a 32-ary search.
// Returns n if there is none.
__device__ __noinline__ uint32_t first_block_ge(const uint32_t* __restrict__ last_doc, uint32_t from, uint32_t n,
                                                   uint32_t target, uint32_t lane) {
  if (from >= n) return n;
  {
    const uint32_t idx = from + lane;
    const uint32_t v = idx < n ? __ldg(last_doc + idx) : 0xFFFFFFFFu;
    const unsigned m = __ballot_sync(kFull, v >= target);
    if (m) { const uint32_t j = from + (uint32_t)__ffs(m) - 1u; return j < n ? j : n; }
  }
  uint32_t lo = from + 32u, hi = n;  // answer in [lo, hi] (hi == n means none)
  if (lo >= hi) return n;
  if (__ldg(last_doc + (n - 1)) < target) return n;
  // invariant: last_doc[hi-1] >= target, every index < lo is < target
  while (hi - lo > 32u) {
    const uint32_t step = (hi - lo + 31u) / 32u;
    uint32_t idx = lo + (lane + 1u) * step - 1u;
    if (idx > hi - 1u) idx = hi - 1u;
    const uint32_t v = __ldg(last_doc + idx);
    const unsigned m = __ballot_sync(kFull, v >= target);  // non-empty: lane 31 probes hi-1
    const uint32_t f = (uint32_t)__ffs(m) - 1u;
    uint32_t nhi = lo + (f + 1u) * step;
    if (nhi > hi) nhi = hi;
    lo = lo + f * step;
    hi = nhi;
  }
  {
    const uint32_t idx = lo + lane;
    const uint32_t v = idx < hi ? __ldg(last_doc + idx) : 0xFFFFFFFFu;
    const unsigned m = __ballot_sync(kFull, v >= target);
    return lo + (uint32_t)__ffs(m) - 1u;
  }
}

// ---- K6a: CTA-level exact top-k buffer ----------------------------------------------------------
struct TopKScratch {  // shared memory used by the histogram compaction
  unsigned int hist[256];
  unsigned short holes[kCap / 2];
  unsigned int kmin, kmax, hole_n, mover_n, keep, cut;
};
struct TopK {
  unsigned long long* keys;   // [kCap] shared
  unsigned int* count;        // shared
  unsigned long long* theta;  // shared: keys below it can no longer enter the top-k
  TopKScratch* scratch;       // shared
  unsigned nthreads;          // threads of the CTA
};

// All lanes of a warp call this together (pass may differ per lane).
__device__ __forceinline__ void topk_push(const TopK& t, bool pass, unsigned long long key, uint32_t lane) {
  const unsigned m = __ballot_sync(kFull, pass);
  if (m == 0) return;
  const int leader = __ffs(m) - 1;
  unsigned base = 0;
  if ((int)lane == leader) base = atomicAdd(t.count, (unsigned)__popc(m));
  base = __shfl_sync(kFull, base, leader);
  if (pass) t.keys[base + __popc(m & lanemask_lt(lane))] = key;
}

// Whole CTA. Sorts the buffer (descending) and keeps the best k; publishes the k-th score.
__device__ __noinline__ void topk_compact(const TopK& t, uint32_t k, unsigned int* theta_global) {
  __syncthreads();
  const unsigned n = *t.count;
  unsigned size = 2;
  while (size < n) size <<= 1;
  for (unsigned i = threadIdx.x; i < size; i += t.nthreads)
    if (i >= n) t.keys[i] = 0ull;
  __syncthreads();
  for (unsigned kk = 2; kk <= size; kk <<= 1) {
    for (unsigned j = kk >> 1; j > 0; j >>= 1) {
      for (unsigned i = threadIdx.x; i < size; i += t.nthreads) {
        const unsigned ixj = i ^ j;
        if (ixj > i) {
          const unsigned long long a = t.keys[i], b = t.keys[ixj];
          const bool desc = (i & kk) == 0;
          if (desc ? (a < b) : (a > b)) { t.keys[i] = b; t.keys[ixj] = a; }
        }
      }
      __syncthreads();
    }
  }
  if (threadIdx.x == 0 && n > k) {
    *t.count = k;
    const unsigned long long kth = t.keys[k - 1];
    if (kth > *t.theta) *t.theta = kth;
    atomicMax(theta_global, (unsigned)(kth >> 32));
  }
  __syncthreads();
}

// Cheap compaction.  The CTA only has to keep a SUPERSET of its k best keys and a threshold that is a valid
// lower bound of its k-th best score (k_final selects exactly).  One histogram of the score keys (256 bins
// between the smallest and largest key in the buffer) finds the highest bin edge with >= k keys at or above
// it; keys below that edge are dropped by moving the survivors of the upper part into the holes of the lower
// part.  Falls back to the exact sort when the boundary bin is too crowded (ties) to make room.
__device__ __noinline__ void topk_compact_hist(const TopK& t, uint32_t k, uint32_t keep_max, unsigned int* theta_global) {
  TopKScratch& sc = *t.scratch;
  __syncthreads();
  const unsigned n = *t.count;
  if (n <= k) return;  // uniform
  for (unsigned i = threadIdx.x; i < 256; i += t.nthreads) sc.hist[i] = 0;
  if (threadIdx.x == 0) { sc.kmin = 0xFFFFFFFFu; sc.kmax = 0; sc.hole_n = 0; sc.mover_n = 0; }
  __syncthreads();
  unsigned lmin = 0xFFFFFFFFu, lmax = 0;
  for (unsigned i = threadIdx.x; i < n; i += t.nthreads) {
    const unsigned sk = (unsigned)(t.keys[i] >> 32);
    lmin = min(lmin, sk); lmax = max(lmax, sk);
  }
  lmin = __reduce_min_sync(kFull, lmin);
  lmax = __reduce_max_sync(kFull, lmax);
  if ((threadIdx.x & 31u) == 0) { atomicMin(&sc.kmin, lmin); atomicMax(&sc.kmax, lmax); }
  __syncthreads();
  const unsigned kmin = sc.kmin, span = sc.kmax - kmin;
  const unsigned shift = span < 256u ? 0u : (unsigned)(32 - __clz(span)) - 8u;  // (key - kmin) >> shift in [0, 255]
  for (unsigned i = threadIdx.x; i < n; i += t.nthreads) atomicAdd(&sc.hist[((unsigned)(t.keys[i] >> 32) - kmin) >> shift], 1u);
  __syncthreads();
  if (threadIdx.x < 32) {  // suffix sums over the 256 bins: 8 per lane
    const unsigned lane = threadIdx.x;
    unsigned loc[8], tot = 0;
#pragma unroll
    for (int j = 7; j >= 0; --j) { tot += sc.hist[lane * 8 + j]; loc[j] = tot; }  // inclusive suffix within the lane's bins
    // inclusive suffix sum of the lane totals, then what lies above this lane's bins
    unsigned run = tot;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned v = __shfl_down_sync(kFull, run, o);
      if (lane + o < 32) run += v;
    }
    const unsigned above = run - tot;
    // the boundary bin: the highest bin b with (#keys in bins >= b) >= k
    int cut = -1; unsigned keep = 0;
#pragma unroll
    for (int j = 7; j >= 0; --j) {
      const unsigned ge = above + loc[j];
      if (cut < 0 && ge >= k) { cut = (int)(lane * 8 + j); keep = ge; }
    }
    const unsigned has = __ballot_sync(kFull, cut >= 0);
    const int src = 31 - __clz(has);  // highest lane that found one (n > k guarantees at least one)
    cut = __shfl_sync(kFull, cut, src);
    keep = __shfl_sync(kFull, keep, src);
    if (lane == 0) { sc.cut = (unsigned)cut; sc.keep = keep; }
  }
  __syncthreads();
  const unsigned keep = sc.keep;
  if (keep > keep_max || keep == n) {  // crowded boundary bin (ties) or nothing to drop: exact route
    topk_compact(t, k, theta_global);
    return;
  }
  const unsigned edge = kmin + (sc.cut << shift);  // every survivor has score key >= edge, and there are >= k of them
  for (unsigned i = threadIdx.x; i < keep; i += t.nthreads)
    if ((unsigned)(t.keys[i] >> 32) < edge) sc.holes[atomicAdd(&sc.hole_n, 1u)] = (unsigned short)i;
  __syncthreads();
  for (unsigned i = keep + threadIdx.x; i < n; i += t.nthreads) {
    const unsigned long long key = t.keys[i];
    if ((unsigned)(key >> 32) >= edge) t.keys[sc.holes[atomicAdd(&sc.mover_n, 1u)]] = key;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    *t.count = keep;
    const unsigned long long th = (unsigned long long)edge << 32;
    if (th > *t.theta) *t.theta = th;
    atomicMax(theta_global, edge);
  }
  __syncthreads();
}

// End of a round of the CTA: refresh the shared threshold from the query-wide one and make room.
// `limit`: compact as soon as this many keys are buffered (a pruning kernel wants its threshold early).
__device__ __forceinline__ void topk_round_end(const TopK& t, uint32_t k, unsigned int* theta_global, uint32_t limit = kCap - kRoundMargin) {
  __syncthreads();
  if (*t.count > limit) topk_compact_hist(t, k, kCap - kRoundMargin, theta_global);
  if (threadIdx.x == 0) {
    const unsigned long long g = (unsigned long long)(*(volatile unsigned int*)theta_global) << 32;
    if (g > *t.theta) *t.theta = g;
  }
  __syncthreads();
}

// End of a unit: the CTA's survivors go to the query's candidate region (at most 2k of them).
__device__ __noinline__ void topk_flush(const TopK& t, const DQuery& q, QState* qs, Cand* cands, uint32_t segment_ord) {
  __syncthreads();
  if (*t.count > 2u * q.k) topk_compact_hist(t, q.k, min(2u * q.k, kCap / 2u), &qs->theta);
  __shared__ unsigned s_base;
  const unsigned n = *t.count;
  if (threadIdx.x == 0) s_base = n ? atomicAdd(&qs->cand_count, n) : 0u;
  __syncthreads();
  const unsigned base = s_base;
  for (unsigned i = threadIdx.x; i < n; i += t.nthreads) {
    if (base + i < q.cand_cap) {
      const unsigned long long key = t.keys[i];
      Cand c;
      c.score_key = (uint32_t)(key >> 32);
      c.segment_ord = segment_ord;
      c.doc = 0xFFFFFFFFu - (uint32_t)key;
      c.pad = 0;
      cands[q.cand_base + base + i] = c;
    }
  }
}

__device__ __forceinline__ bool is_alive(const uint8_t* __restrict__ alive, uint32_t doc) {
  return alive == nullptr || ((__ldg(alive + (doc >> 3)) >> (doc & 7u)) & 1u);
}

}  // namespace tq
