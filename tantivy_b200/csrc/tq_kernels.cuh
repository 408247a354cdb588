// The sm_100a kernels of the query path.  One CTA (8 warps) per work unit; one warp per 128-doc
// posting block; exact per-CTA top-k buffers reduced per query by k_final.
//
//   k_build_tables  SkipReader::read_block_info/advance as ONE exclusive scan (src/postings/skip.rs:205-302)
//                   + decode_vint_block for the tail (src/postings/block_segment_postings.rs:56-76)
//   k_term          block_wand_single_scorer's result set (block_wand_union.rs:226-265), exhaustive form
//   k_and           block_wand_intersection's result set (block_wand_intersection.rs:19-179): leader =
//                   rarest list, secondaries probed through their block tables; score summed
//                   leader first, then secondaries by ascending doc_freq (:27,146-158)
//   k_or            BufferedUnionScorer's shape (union/buffered_union.rs:63-151): a doc-id window of
//                   score slots in shared memory, clauses accumulated in clause order
//   k_bool          BooleanWeight::complex_scorer's result set for mixed Occurs (boolean_weight.rs:236-431):
//                   k_or's windows with per-group presence bitmaps, SHOULD counts and a MUST_NOT mask
//   k_final         TopBySortKeyCollector::merge_fruits / merge_top_k (sort_key_top_collector.rs:54-95)
#pragma once
#include "tq_device.cuh"

namespace tq {

struct BuildJob {
  const uint8_t* bytes;  // the term's postings range
  uint32_t len;
  uint32_t doc_freq;
  uint32_t record_option;  // 0/1/2; bit 8: ignore term frequencies (score with tf = 1)
  uint32_t list_id;
};

__device__ __forceinline__ uint32_t load_u32_unaligned(const uint8_t* p) {
  return (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24);
}

// One CTA per posting list.  Fills last_doc / blk / tail arrays of its ListDesc.
__global__ void __launch_bounds__(kThreads) k_build_tables(const BuildJob* __restrict__ jobs, const ListDesc* __restrict__ init,
                                                           ListDesc* __restrict__ lists, uint32_t* __restrict__ status_out) {
  const BuildJob J = jobs[blockIdx.x];
  ListDesc& L = lists[J.list_id];
  if (threadIdx.x == 0) L = init[blockIdx.x];  // (list ids are recycled: the slot may hold an unregistered segment's table)
  __syncthreads();
  uint32_t* last_doc = const_cast<uint32_t*>(L.last_doc);
  uint2* blk = const_cast<uint2*>(L.blk);
  uint4* tab4 = const_cast<uint4*>(L.tab4);
  uint32_t* tail_docs = const_cast<uint32_t*>(L.tail_docs);
  uint32_t* tail_tfs = const_cast<uint32_t*>(L.tail_tfs);
  const uint32_t n_blocks = J.doc_freq / 128u, tail_n = J.doc_freq % 128u;
  __shared__ uint32_t s_hdr, s_skip_len, s_rec, s_status, s_carry;
  __shared__ uint32_t s_wsum[kWarps];
  const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
  if (tid == 0) {
    const uint32_t ro = J.record_option & 0xFFu;
    uint32_t hdr = 0, skip_len = 0, rec = ro == 0 ? 5u : (ro == 1 ? 8u : 12u), status = 0;
    if (J.doc_freq >= 128u) {  // split_into_skips_and_postings (block_segment_postings.rs:78-88)
      uint64_t v = 0;
      uint32_t shift = 0;
      bool done = false;
      while (hdr < J.len && hdr < 10u) {
        const uint8_t b = J.bytes[hdr++];
        v |= (uint64_t)(b & 127u) << shift;
        shift += 7;
        if (b & 128u) { done = true; break; }
      }
      if (!done || v > (uint64_t)J.len - hdr) status = 1;
      skip_len = (uint32_t)v;
      // a field indexed with freqs can hold terms written without (block_segment_postings.rs:116-123)
      if (rec != 5u && skip_len < 8u * n_blocks) rec = 5u;
      if ((uint64_t)rec * n_blocks > skip_len) status = 1;
    }
    s_hdr = hdr; s_skip_len = skip_len; s_rec = rec; s_status = status; s_carry = 0;
  }
  __syncthreads();
  const uint32_t rec = s_rec;
  const uint8_t* skip = J.bytes + s_hdr;
  const uint8_t* blocks = skip + s_skip_len;
  const uint32_t avail = J.len - s_hdr - s_skip_len;
  if (s_status == 0) {
    for (uint32_t base = 0; base < n_blocks; base += kThreads) {
      const uint32_t i = base + tid;
      uint32_t size = 0, meta = 0, last = 0;
      if (i < n_blocks) {
        const uint8_t* r = skip + (size_t)i * rec;
        last = load_u32_unaligned(r);
        const uint32_t bw = r[4];
        const uint32_t db = bw & 31u, strict = (bw >> 6) & 1u;
        uint32_t tb = 0, bm_fn = 0, bm_tf = 0;
        if (rec == 8u) { tb = r[5]; bm_fn = r[6]; bm_tf = r[7]; }
        else if (rec == 12u) { tb = r[5]; bm_fn = r[10]; bm_tf = r[11]; }
        if (tb > 32u) { tb = 32u; s_status = 1; }
        size = 16u * (db + tb);
        meta = db | (strict << 6) | (tb << 8) | (bm_fn << 16) | (bm_tf << 24);
      }
      const uint32_t incl = warp_incl_scan(size, lane);
      if (lane == 31) s_wsum[warp] = incl;
      __syncthreads();
      uint32_t woff = 0;
#pragma unroll
      for (int w = 0; w < kWarps; ++w) woff += (w < (int)warp) ? s_wsum[w] : 0u;
      const uint32_t excl = s_carry + woff + incl - size;
      if (i < n_blocks) {
        last_doc[i] = last;
        blk[i] = make_uint2(excl, meta);
        const uint32_t prev_last = i ? load_u32_unaligned(skip + (size_t)(i - 1) * rec) : 0xFFFFFFFFu;
        tab4[i] = make_uint4(last, excl, meta, prev_last);
      }
      __syncthreads();
      if (tid == kThreads - 1) s_carry = excl + size;
      __syncthreads();
    }
  }
  if (tid == 0) {
    uint32_t status = s_status;
    const uint32_t total = s_carry;
    blk[n_blocks] = make_uint2(total, 0u);
    if (total > avail) status = 1;
    if (tail_n && status == 0) {
      // decode_vint_block: plain deltas from last_doc_in_previous_block, tfs raw (serializer.rs:456-468)
      const uint8_t* p = blocks + total;
      uint32_t remaining = avail - total, pos = 0;
      uint32_t result = n_blocks ? load_u32_unaligned(skip + (size_t)(n_blocks - 1) * rec) : 0u;
      for (uint32_t i = 0; i < tail_n && status == 0; ++i) {
        uint32_t shift = 0;
        for (;;) {
          if (pos >= remaining) { status = 1; break; }
          const uint8_t b = p[pos++];
          result += (uint32_t)(b & 127u) << shift;
          if (b & 128u) break;
          shift += 7;
        }
        tail_docs[i] = result;
      }
      const bool read_freq = (rec != 5u) && pos < remaining && !(J.record_option & 0x100u);  // block_segment_postings.rs:66-75
      for (uint32_t i = 0; i < tail_n && status == 0; ++i) {
        uint32_t v = 1u;
        if (read_freq) {
          v = 0;
          uint32_t shift = 0;
          for (;;) {
            if (pos >= remaining) { status = 1; break; }
            const uint8_t b = p[pos++];
            v += (uint32_t)(b & 127u) << shift;
            if (b & 128u) break;
            shift += 7;
          }
        }
        tail_tfs[i] = v;
      }
      if (status == 0) {
        last_doc[n_blocks] = tail_docs[tail_n - 1];
        const uint32_t prev_last = n_blocks ? load_u32_unaligned(skip + (size_t)(n_blocks - 1) * rec) : 0xFFFFFFFFu;
        tab4[n_blocks] = make_uint4(tail_docs[tail_n - 1], total, 0xFFFFFFFFu, prev_last);
      }
    }
    L.has_freq = rec != 5u && !(J.record_option & 0x100u);  // SkipFreq: the tf bits stay in the block sizes, nobody reads them
    L.build_status = status;
    status_out[blockIdx.x] = status;
  }
  // 16-byte aligned copy of the bit-packed blocks (L.blocks was pre-set by the host to an arena region of
  // >= len + 64 bytes): posting lists start at arbitrary byte offsets inside the .idx body; the copy lets
  // every lane fetch its vectors with plain LDG.128.
  __syncthreads();
  if (s_status == 0 && s_carry <= avail) {
    const uint32_t total_words = s_carry / 4u + 16u;  // + 64 bytes of slack after the last block
    const uint32_t mis = (uint32_t)((uintptr_t)blocks & 3u);
    const uint32_t* src32 = reinterpret_cast<const uint32_t*>(blocks - mis);
    uint32_t* dst32 = reinterpret_cast<uint32_t*>(const_cast<uint8_t*>(L.blocks));
    const uint32_t sh = mis * 8u;
    for (uint32_t i = tid; i < total_words; i += kThreads) {
      const uint32_t w0 = src32[i], w1 = src32[i + 1];  // the segment body is padded by 256 bytes on the device
      dst32[i] = mis ? __funnelshift_r(w0, w1, sh) : w0;
    }
  }
}

// tf / (tf + norm[id]) for tf < kTfRows, one table per tf-norm cache of the batch; same IEEE operations and
// order as Bm25Weight::tf_factor (bm25.rs:170-175).
__global__ void k_build_tf_tables(const float* __restrict__ caches, float* __restrict__ tables, uint32_t n_caches) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_caches * kTfRows * 256u) return;
  const uint32_t c = i / (kTfRows * 256u), tf = (i >> 8) % kTfRows, id = i & 255u;
  const float t = __uint2float_rn(tf);
  tables[i] = __fdiv_rn(t, __fadd_rn(t, caches[c * 256u + id]));
}

// ---- K1 stand-alone: whole-list decode (parity tests, decode micro-benchmark) ------------------
__global__ void __launch_bounds__(kThreads) k_decode_list(const ListDesc* __restrict__ lists, uint32_t list_id,
                                                          uint32_t* __restrict__ out_docs, uint32_t* __restrict__ out_tfs) {
  const ListDesc L = lists[list_id];
  const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
  const uint32_t b = blockIdx.x * kWarps + warp;
  if (b >= L.n_total) return;
  uint32_t doc[4], tf[4];
  decode_block(L, b, lane, doc, tf);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const uint32_t j = b * 128u + lane * 4u + i;
    if (j < L.doc_freq) { out_docs[j] = doc[i]; if (out_tfs) out_tfs[j] = tf[i]; }
  }
}

// Block-max score of every full block (SkipReader::block_max_score, skip.rs:175-184).
__global__ void k_block_max(const ListDesc* __restrict__ lists, uint32_t list_id, float weight, const float* __restrict__ cache,
                            uint32_t* __restrict__ out_last_doc, float* __restrict__ out_block_max) {
  const ListDesc L = lists[list_id];
  const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= L.n_blocks) return;
  const uint32_t meta = L.blk[b].y;
  const uint32_t code = meta >> 24;
  const uint32_t tf = code == 255u ? 0xFFFFFFFFu : code;
  out_last_doc[b] = L.last_doc[b];
  const float t = __uint2float_rn(tf);
  out_block_max[b] = __fmul_rn(weight, __fdiv_rn(t, __fadd_rn(t, __ldg(cache + ((meta >> 16) & 255u)))));
}

// ---- shared CTA scaffolding ------------------------------------------------------------------------
struct CtaTopK {
  unsigned long long keys[kCap];
  unsigned int count;
  unsigned long long theta;
  TopKScratch scratch;
};

// ---- single term ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads) k_term(const BatchParams P, uint32_t unit_base) {
  __shared__ CtaTopK s_top;
  const Unit U = P.units[unit_base + blockIdx.x];
  const QSeg S = P.qsegs[U.qseg];
  const DQuery Q = P.queries[S.query];
  QState* qs = P.qstate + S.query;
  const QList ql = P.qlists[S.lists_base];
  const ListDesc L = P.lists[ql.list_id];
  const Scorer sc = make_scorer(P, ql);
  const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
  if (threadIdx.x == 0) { s_top.count = 0; s_top.theta = (unsigned long long)qs->theta << 32; }
  __syncthreads();
  const TopK T{s_top.keys, &s_top.count, &s_top.theta, &s_top.scratch, (unsigned)kThreads};
  BlockFetch f;
  if (U.begin + warp < U.end) fetch_issue(L, U.begin + warp, lane, f);
  for (uint32_t r = U.begin; r < U.end; r += kWarps) {
    const uint32_t b = r + warp;
    if (b < U.end) {
      uint32_t doc[4], tf[4];
      fetch_decode(L, b, f, lane, doc, tf);
      if (b + kWarps < U.end) fetch_issue(L, b + kWarps, lane, f);  // next round's block travels while this one is scored
      const unsigned long long theta = *T.theta;
      const float theta_f = threshold_score((uint32_t)(theta >> 32));
      bool pass[4];
      float score[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const bool valid = doc[i] < S.max_doc;  // also rejects the kTerminated padding of the tail
        score[i] = valid ? bm25_score(sc, L.fieldnorm, doc[i], tf[i]) : 0.0f;
        pass[i] = valid && score[i] >= theta_f;  // cheap float test first; the exact key test only on survivors
      }
      if (__ballot_sync(kFull, pass[0] | pass[1] | pass[2] | pass[3])) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const unsigned long long key = make_key(score[i], doc[i]);
          bool p = pass[i] && key >= theta;
          if (p && S.alive) p = is_alive(S.alive, doc[i]);
          topk_push(T, p, key, lane);
        }
      }
    }
    topk_round_end(T, Q.k, &qs->theta);
  }
  topk_flush(T, Q, qs, P.cands, S.segment_ord);
}

// ---- intersection ----------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads) k_and(const BatchParams P, uint32_t unit_base) {
  __shared__ uint32_t s_dec[kWarps][256];  // a decoded secondary block: 128 docs, 128 tfs
  __shared__ CtaTopK s_top;
  const Unit U = P.units[unit_base + blockIdx.x];
  const QSeg S = P.qsegs[U.qseg];
  const DQuery Q = P.queries[S.query];
  QState* qs = P.qstate + S.query;
  const QList ql0 = P.qlists[S.lists_base];
  const ListDesc L0 = P.lists[ql0.list_id];
  const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
  uint32_t* dec = s_dec[warp];
  if (threadIdx.x == 0) { s_top.count = 0; s_top.theta = (unsigned long long)qs->theta << 32; }
  __syncthreads();
  const TopK T{s_top.keys, &s_top.count, &s_top.theta, &s_top.scratch, (unsigned)kThreads};
  // MaxScore for the conjunction (exact): a leader doc whose own score plus the secondaries' bounds (score < weight)
  // cannot reach the threshold is dropped BEFORE its secondary blocks are looked up and decoded -- the lookups are
  // what this kernel spends its time on (block_wand_intersection.rs:60-120 prunes on block maxima for the same reason).
  const bool prunable = (S.flags & 2u) != 0;
  const Scorer sc0 = make_scorer(P, ql0);
  float ub_secondaries = 0.0f;
  for (uint32_t s = 1; s < S.n_lists; ++s) ub_secondaries += P.qlists[S.lists_base + s].weight;
  // Without a threshold the first round would look up every leader doc of 8 blocks; one block (one warp) is enough to
  // get a first threshold, the other seven then start pruned.
  bool narrow = prunable && s_top.theta == 0ull;
  for (uint32_t r = U.begin; r < U.end;) {
    const uint32_t width = narrow ? 1u : (uint32_t)kWarps;
    const uint32_t b = r + warp;
    if (warp < width && b < U.end) {
      uint32_t doc[4], tf0[4];
      decode_block(L0, b, lane, doc, tf0);
      uint32_t alive_m = 0;
#pragma unroll
      for (int i = 0; i < 4; ++i) alive_m |= (doc[i] < S.max_doc) ? (1u << i) : 0u;  // rejects tail padding
      float total[4] = {0.f, 0.f, 0.f, 0.f};
      float ub = ub_secondaries;
      const float theta_f = prunable ? threshold_score((uint32_t)(*(volatile unsigned long long*)T.theta >> 32)) : 0.0f;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        if ((alive_m >> i) & 1u) {
          total[i] = bm25_score(sc0, L0.fieldnorm, doc[i], tf0[i]);
          if (theta_f > 0.0f && (total[i] + ub) * 1.00001f < theta_f) alive_m &= ~(1u << i);
        }
      }
      for (uint32_t s = 1; s < S.n_lists; ++s) {
        if (__ballot_sync(kFull, alive_m != 0) == 0) break;
        const QList qls = P.qlists[S.lists_base + s];
        const ListDesc Ls = P.lists[qls.list_id];
        const Scorer sc_s = make_scorer(P, qls);
        uint32_t pending = alive_m;
        uint32_t stf[4] = {1u, 1u, 1u, 1u};
        uint32_t cur = 0;
        for (;;) {
          // smallest unresolved candidate of the warp (candidates ascend with lane*4+i)
          const uint32_t c = (pending & 1u) ? doc[0] : (pending & 2u) ? doc[1] : (pending & 4u) ? doc[2] : (pending & 8u) ? doc[3] : 0xFFFFFFFFu;
          const uint32_t cmin = warp_min(c);
          if (cmin == 0xFFFFFFFFu) break;
          const uint32_t j = first_block_ge(Ls.last_doc, cur, Ls.n_total, cmin, lane);
          if (j >= Ls.n_total) { alive_m &= ~pending; pending = 0; break; }  // past the end of this list
          const uint32_t blk_last = __ldg(Ls.last_doc + j);
          uint32_t sd[4], st[4];
          decode_block(Ls, j, lane, sd, st);
          __syncwarp();
#pragma unroll
          for (int i = 0; i < 4; ++i) { dec[lane * 4 + i] = sd[i]; dec[128 + lane * 4 + i] = st[i]; }
          __syncwarp();
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            if (((pending >> i) & 1u) && doc[i] <= blk_last) {
              uint32_t lo = 0;
#pragma unroll
              for (uint32_t step = 64; step > 0; step >>= 1)
                if (dec[lo + step - 1] < doc[i]) lo += step;
              if (dec[lo] == doc[i]) stf[i] = dec[128 + lo]; else alive_m &= ~(1u << i);
              pending &= ~(1u << i);
            }
          }
          cur = j + 1;
        }
        ub -= qls.weight;  // what the clauses still to come can add at most
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          if ((alive_m >> i) & 1u) {
            total[i] = __fadd_rn(total[i], bm25_score(sc_s, Ls.fieldnorm, doc[i], stf[i]));
            if (theta_f > 0.0f && s + 1u < S.n_lists && (total[i] + ub) * 1.00001f < theta_f) alive_m &= ~(1u << i);
          }
        }
      }
      const unsigned long long theta = *T.theta;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const unsigned long long key = make_key(total[i], doc[i]);
        bool pass = ((alive_m >> i) & 1u) && key >= theta;
        if (pass && S.alive) pass = is_alive(S.alive, doc[i]);
        topk_push(T, pass, key, lane);
      }
    }
    topk_round_end(T, Q.k, &qs->theta, !prunable ? kCap - kRoundMargin : (narrow ? Q.k : min(max(4u * Q.k, 128u), kCap - kRoundMargin)));
    r += width;
    narrow = false;
  }
  topk_flush(T, Q, qs, P.cands, S.segment_ord);
}

// ---- union -------------------------------------------------------------------------------------------------
// Shared memory per CTA: kTileDocs f32 score slots (dynamic) + kTileDocs fieldnorm bytes.
// A slot holding -0.0f has not been touched: -0.0 + s == 0.0 + s bit for bit for every s except
// s == -0.0 (SumCombiner starts from 0.0, score_combiner.rs:39-57).
//
// The general per-query union (any number of clauses, any k): per window of kTileDocs doc ids every clause's blocks
// are decoded and added in clause order, then the window is harvested.  A window is skipped when no clause has a
// block in it, or when the clause maxima together cannot reach the threshold.
struct OrShared {
  uint32_t blo[2][32], bhi[2][32];  // per clause: block range overlapping the tile (double buffered)
  uint32_t cur[32];                 // per clause: search cursor
  uint32_t any[2];
  uint32_t npass;
  float bound;                      // no doc of the segment scores above this
  uint32_t skip;                    // the current window holds nothing that can enter the top-k
};

__device__ __forceinline__ void or_tile_ranges(const BatchParams& P, const QSeg& S, OrShared& sh, int buf, uint32_t tile,
                                               uint32_t warp, uint32_t lane) {
  const uint32_t lo = tile * kTileDocs;
  const uint32_t hi = min(lo + kTileDocs, S.max_doc);
  for (uint32_t t = warp; t < S.n_lists; t += kWarps) {
    const QList ql = P.qlists[S.lists_base + t];
    const uint32_t* last_doc = P.lists[ql.list_id].last_doc;
    const uint32_t n_total = P.lists[ql.list_id].n_total;
    uint32_t blo = 1, bhi = 0;
    const uint32_t j_lo = first_block_ge(last_doc, sh.cur[t], n_total, lo, lane);
    if (j_lo < n_total) {
      // the last block that can hold a doc < hi is the first one whose last doc is >= hi-1
      uint32_t j_hi = first_block_ge(last_doc, j_lo, n_total, hi - 1u, lane);
      if (j_hi >= n_total) j_hi = n_total - 1u;
      blo = j_lo; bhi = j_hi;
    }
    if (lane == 0) { sh.blo[buf][t] = blo; sh.bhi[buf][t] = bhi; sh.cur[t] = j_lo; if (blo <= bhi) sh.any[buf] = 1; }
  }
}

// Blocks of clause t are dealt to the warps rotated by the clause ordinal: the single block of a rare
// clause lands on warp (t mod 8), so the rare clauses of a window are fetched by different warps at the same
// time instead of queueing on warp 0.
__device__ __forceinline__ uint32_t or_first_block(const OrShared& sh, int buf, uint32_t t, uint32_t warp) {
  return sh.blo[buf][t] + ((warp + kWarps - (t & (kWarps - 1))) & (kWarps - 1));
}
// next (clause, block) of this warp at or after (t, b) in tile buffer `buf`; t == n_lists when none
__device__ __forceinline__ void or_next_item(const OrShared& sh, int buf, uint32_t n_lists, uint32_t warp, uint32_t& t, uint32_t& b) {
  while (t < n_lists) {
    if (b <= sh.bhi[buf][t] && sh.blo[buf][t] <= sh.bhi[buf][t]) return;
    ++t;
    if (t < n_lists) b = or_first_block(sh, buf, t, warp);
  }
}

__global__ void __launch_bounds__(kThreads, 3) k_or(const BatchParams P, uint32_t unit_base) {
  extern __shared__ __align__(16) float s_acc[];                  // [kTileDocs]
  uint8_t* s_fn = reinterpret_cast<uint8_t*>(s_acc + kTileDocs);  // [kTileDocs]
  __shared__ CtaTopK s_top;
  __shared__ OrShared sh;
  const Unit U = P.units[unit_base + blockIdx.x];
  const QSeg S = P.qsegs[U.qseg];
  const DQuery Q = P.queries[S.query];
  QState* qs = P.qstate + S.query;
  const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
  const float neg_zero = __uint_as_float(0x80000000u);
  const bool staged_fn = (S.flags & 1u) && S.fieldnorm != nullptr;
  for (uint32_t i = threadIdx.x; i < kTileDocs; i += kThreads) s_acc[i] = neg_zero;
  if (threadIdx.x < 32) sh.cur[threadIdx.x] = 0;
  if (threadIdx.x == 0) {
    s_top.count = 0; s_top.theta = (unsigned long long)qs->theta << 32;
    sh.any[0] = sh.any[1] = 0; sh.npass = 0;
    // a clause can add at most its weight (tf/(tf+norm) < 1, bm25.rs:170-175); the maxima are summed smallest first
    float mx[32];
    for (uint32_t t = 0; t < S.n_lists; ++t) {
      const float m = fmaxf(P.qlists[S.lists_base + t].weight, 0.0f);
      uint32_t j = t;
      while (j > 0 && mx[j - 1] > m) { mx[j] = mx[j - 1]; --j; }
      mx[j] = m;
    }
    float sum = 0.0f;
    for (uint32_t t = 0; t < S.n_lists; ++t) sum += mx[t];
    sh.bound = sum * 1.00001f;  // f32 sums of up to 32 terms differ by < 4e-6 relative
  }
  __syncthreads();
  const TopK T{s_top.keys, &s_top.count, &s_top.theta, &s_top.scratch, (unsigned)kThreads};
  or_tile_ranges(P, S, sh, 0, U.begin, warp, lane);
  unsigned int theta_g_seen = 0;  // thread 0: query-wide threshold sampled one window ago
  __syncthreads();
  for (uint32_t tile = U.begin; tile < U.end; ++tile) {
    const int buf = (int)((tile - U.begin) & 1u);
    const uint32_t lo = tile * kTileDocs;
    const uint32_t hi = min(lo + kTileDocs, S.max_doc);
    if (threadIdx.x == 0) {
      const unsigned long long g = (unsigned long long)theta_g_seen << 32;
      if (g > s_top.theta) s_top.theta = g;
      theta_g_seen = *(volatile unsigned int*)&qs->theta;  // consumed at the next window
      sh.skip = !sh.any[buf] || sh.bound < threshold_score((uint32_t)(s_top.theta >> 32));
    }
    __syncthreads();
    const bool skip = sh.skip != 0;
    const unsigned long long theta = *T.theta;
    const float theta_f = threshold_score((uint32_t)(theta >> 32));

    if (!skip) {
      // ---- accumulate ----------------------------------------------------------------------------------
      // fieldnorm bytes of the window: one coalesced 16-byte row per thread pair instead of a byte gather per posting
      if (staged_fn) {
        const uint4* src = reinterpret_cast<const uint4*>(S.fieldnorm + lo);
        uint4* dst = reinterpret_cast<uint4*>(s_fn);
        for (uint32_t i = threadIdx.x; i < kTileDocs / 16; i += kThreads) dst[i] = __ldg(src + i);
      }
      // first work item of this warp, fetched before the barrier
      uint32_t t = 0, b = or_first_block(sh, buf, 0, warp);
      or_next_item(sh, buf, S.n_lists, warp, t, b);
      BlockFetch f;
      QList ql;
      ListDesc L;
      if (t < S.n_lists) { ql = P.qlists[S.lists_base + t]; L = P.lists[ql.list_id]; fetch_issue(L, b, lane, f); }
      __syncthreads();  // s_fn ready
      for (uint32_t tt = 0; tt < S.n_lists; ++tt) {
        while (t == tt) {
          uint32_t doc[4], tf[4];
          fetch_decode(L, b, f, lane, doc, tf);
          const Scorer scr = make_scorer(P, ql);
          const uint8_t* fn_global = L.fieldnorm;
          // next item (same clause or a later one) starts travelling now
          uint32_t nt = t, nb = b + kWarps;
          or_next_item(sh, buf, S.n_lists, warp, nt, nb);
          if (nt < S.n_lists) {
            if (nt != t) { ql = P.qlists[S.lists_base + nt]; L = P.lists[ql.list_id]; }
            fetch_issue(L, nb, lane, f);
          }
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            if (doc[i] >= lo && doc[i] < hi) {
              const uint32_t slot = doc[i] - lo;
              const uint32_t id = staged_fn ? (uint32_t)s_fn[slot] : (fn_global ? (uint32_t)__ldg(fn_global + doc[i]) : 1u);
              const float sc = bm25_score_id(scr, id, tf[i]);
              s_acc[slot] = __fadd_rn(s_acc[slot], sc);
            }
          }
          t = nt; b = nb;
        }
        __syncthreads();  // clause order is the f32 summation order
      }
    }

    // ranges of the next window: the searches overlap the harvest below
    if (tile + 1 < U.end) {
      if (threadIdx.x == 0) sh.any[buf ^ 1] = 0;
      __syncthreads();
      or_tile_ranges(P, S, sh, buf ^ 1, tile + 1, warp, lane);
    }

    if (!skip) {
      // harvest: count what passes, then push in one go when it fits.
      // A float compare against the threshold score rejects nearly every slot (untouched slots hold
      // -0.0, which is below any positive threshold); the exact key test runs only on the survivors.
      uint32_t passmask = 0;
#pragma unroll 1
      for (int j = 0; j < (int)(kTileDocs / (kThreads * 4)); ++j) {
        const uint32_t idx = (j * kThreads + threadIdx.x) * 4;
        const float4 v = *reinterpret_cast<const float4*>(s_acc + idx);
        if (v.x >= theta_f || v.y >= theta_f || v.z >= theta_f || v.w >= theta_f) {
          const float vv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            const uint32_t d = lo + idx + c;
            bool pass = vv[c] >= theta_f && __float_as_uint(vv[c]) != 0x80000000u && make_key(vv[c], d) >= theta;
            if (pass && S.alive) pass = is_alive(S.alive, d);
            passmask |= pass ? (1u << (j * 4 + c)) : 0u;
          }
        }
      }
      const uint32_t wsum = __reduce_add_sync(kFull, (uint32_t)__popc(passmask));
      if (lane == 0 && wsum) atomicAdd(&sh.npass, wsum);
      __syncthreads();
      const uint32_t npass = sh.npass;
      const bool fits = *T.count + npass <= kCap;
      __syncthreads();
      if (fits) {
#pragma unroll 1
        for (int j = 0; j < (int)(kTileDocs / (kThreads * 4)); ++j) {
          const uint32_t idx = (j * kThreads + threadIdx.x) * 4;
          const uint32_t sub = (passmask >> (j * 4)) & 15u;
          if (__ballot_sync(kFull, sub != 0)) {
            const float4 v = *reinterpret_cast<const float4*>(s_acc + idx);
            const float vv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
            for (int c = 0; c < 4; ++c) topk_push(T, (sub >> c) & 1u, make_key(vv[c], lo + idx + c), lane);
          }
          *reinterpret_cast<float4*>(s_acc + idx) = make_float4(neg_zero, neg_zero, neg_zero, neg_zero);
        }
        if (threadIdx.x == 0) sh.npass = 0;
        topk_round_end(T, Q.k, &qs->theta);
      } else {  // cold start: more survivors than the buffer holds; go in rounds with compaction between
        if (threadIdx.x == 0) sh.npass = 0;
        topk_round_end(T, Q.k, &qs->theta);  // leaves at most kCap - kRoundMargin keys
#pragma unroll 1
        for (int j = 0; j < (int)(kTileDocs / (kThreads * 4)); ++j) {
          const uint32_t idx = (j * kThreads + threadIdx.x) * 4;
          const float4 v = *reinterpret_cast<const float4*>(s_acc + idx);
          const float vv[4] = {v.x, v.y, v.z, v.w};
          const unsigned long long th = *T.theta;
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            const unsigned long long key = make_key(vv[c], lo + idx + c);
            topk_push(T, ((passmask >> (j * 4 + c)) & 1u) && key >= th, key, lane);
          }
          *reinterpret_cast<float4*>(s_acc + idx) = make_float4(neg_zero, neg_zero, neg_zero, neg_zero);
          topk_round_end(T, Q.k, &qs->theta);
        }
      }
    } else {
      __syncthreads();
    }
  }
  topk_flush(T, Q, qs, P.cands, S.segment_ord);
}

// ---- union, strip form ----------------------------------------------------------------------------------------
// The same result as k_or, organised for latency tolerance: NO block-wide barrier in the loop.  Every warp owns a
// contiguous strip of doc ids and walks it in windows of kWin docs with private score slots, private fieldnorm
// bytes, a private candidate buffer and its own threshold (plus the query-wide one).  Clause order inside a warp
// is program order, so the f32 sum is still taken clause by clause.
//  * thick clauses (>= 1 block per window on average) are decoded window by window: one 32-wide probe of the
//    16-byte block records gives position and record, the packed vectors follow (2 dependent loads);
//  * thinner clauses keep their current block DECODED AND SCORED in shared memory (docs + scores); a window only
//    looks at it when the block's next unread doc falls inside the window, so a block is decoded once per strip.
// Eligible when k <= kStripMaxK, <= kStripMaxLists clauses and <= kMaxCached thin clauses; otherwise k_or.
#ifndef TQ_KWIN
#define TQ_KWIN 1024
#endif
constexpr uint32_t kWin = TQ_KWIN;  // docs per window (multiple of 512)
constexpr uint32_t kWBuf = 256;
constexpr uint32_t kMaxCached = 6;
constexpr uint32_t kStripWarps = 4;
constexpr uint32_t kStripThreads = kStripWarps * 32;
constexpr uint32_t kStripMaxLists = 8;
constexpr uint32_t kStripNeDiv = 8;    // clauses with >= 1 posting per this many docs may turn non-essential
constexpr uint32_t kStripNeDiv2 = 64;  // ...and the densest clause of a union without such a clause, under this looser bound
constexpr uint32_t kStripMaxK = 128;
constexpr uint32_t kNoDoc = 0xFFFFFFFFu;

struct StripWarpFixed {  // per warp, dynamic shared memory; followed by n_cached x StripCache
  float acc[kWin + 32];               // + one private dummy slot per lane for postings outside the window
  unsigned long long keys[kWBuf];
  uint8_t fn[kWin];
  uint32_t cur[kStripMaxLists];       // thick: first block that can still matter; thin: block held in the cache
  uint32_t next_doc[kStripMaxLists];  // thin: smallest cached doc not applied yet (kNoDoc: clause exhausted)
  uint32_t pos[kStripMaxLists];       // thin: its index in the cached block (entries are in doc order)
  uint32_t stat[8];                   // lane 0: windows by route (1 exhaustive, 2 hot, 3 cold), [5] 16-byte units read
};
struct StripCache {
  uint32_t doc[128];
  float score[128];
};
__host__ __device__ constexpr size_t strip_smem_bytes(uint32_t n_cached) {
  return kStripWarps * (sizeof(StripWarpFixed) + (size_t)n_cached * sizeof(StripCache));
}

__device__ __forceinline__ void fetch_issue_rec(const ListDesc& L, const uint4 rec, uint32_t lane, BlockFetch& f) {
  f.meta = rec.z;
  if (rec.z == 0xFFFFFFFFu) return;  // VInt tail
  f.prev = rec.w == 0xFFFFFFFFu ? 0u : rec.w;
  const uint32_t db = rec.z & 31u, tb = (rec.z >> 8) & 63u;
  const uint4* v = reinterpret_cast<const uint4*>(L.blocks + rec.y);
  const uint32_t wd = (lane * db) >> 5;
  f.dlo = ldg_stream(v + wd);
  f.dhi = ldg_stream(v + wd + 1);
  if (L.has_freq) {
    const uint32_t wt = db + ((lane * tb) >> 5);
    f.tlo = ldg_stream(v + wt);
    f.thi = ldg_stream(v + wt + 1);
  }
}

// warp-level: sort the candidate buffer (descending) and keep the best k
__device__ __noinline__ void strip_compact(unsigned long long* keys, uint32_t& cnt, uint32_t k, unsigned long long& theta,
                                              unsigned int* theta_global, uint32_t lane) {
  for (uint32_t i = cnt + lane; i < kWBuf; i += 32) keys[i] = 0ull;
  __syncwarp();
  for (uint32_t kk = 2; kk <= kWBuf; kk <<= 1) {
    for (uint32_t j = kk >> 1; j > 0; j >>= 1) {
      for (uint32_t p = lane; p < kWBuf / 2; p += 32) {
        const uint32_t i = ((p & ~(j - 1u)) << 1) | (p & (j - 1u));
        const uint32_t ixj = i | j;
        const unsigned long long a = keys[i], b = keys[ixj];
        const bool desc = (i & kk) == 0;
        if (desc ? (a < b) : (a > b)) { keys[i] = b; keys[ixj] = a; }
      }
      __syncwarp();
    }
  }
  if (cnt > k) {
    cnt = k;
    const unsigned long long kth = keys[k - 1];
    if (kth > theta) theta = kth;
    if (lane == 0) atomicMax(theta_global, (unsigned)(kth >> 32));
  }
  __syncwarp();
}

// Decodes block j of a thin clause into the warp's cache, scored (one conflict-free 16-byte store per lane and array).
__device__ __noinline__ uint32_t strip_cache_block(const ListDesc& L, uint32_t j, const Scorer sc, uint32_t max_doc, StripCache& cc, uint32_t lane) {
  uint32_t doc[4], tf[4];
  decode_block(L, j, lane, doc, tf);
  uint32_t cd[4];
  float cs[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const bool valid = doc[i] < max_doc;
    cd[i] = valid ? doc[i] : kNoDoc;
    cs[i] = valid ? bm25_score(sc, L.fieldnorm, doc[i], tf[i]) : 0.0f;
  }
  reinterpret_cast<uint4*>(cc.doc)[lane] = make_uint4(cd[0], cd[1], cd[2], cd[3]);
  reinterpret_cast<float4*>(cc.score)[lane] = make_float4(cs[0], cs[1], cs[2], cs[3]);
  __syncwarp();
  // bytes this touched, in 16-byte units: the packed block (or the decoded tail) + one fieldnorm byte per posting
  return (j < L.n_blocks ? (__ldg(&L.blk[j + 1].x) - __ldg(&L.blk[j].x)) / 16u : L.tail_n / 2u) + 8u;
}

// Positions a thin clause on the first posting >= lo: keeps the cached block when it still reaches lo, else seeks through
// the block table (SkipReader::seek) and caches that block.  cur = block in the cache (n_total: exhausted).
__device__ __noinline__ uint32_t strip_thin_seek(const ListDesc& L, const Scorer sc, uint32_t max_doc, StripCache& cc, bool cache_valid,
                                                    uint32_t lo, uint32_t lane, uint32_t& cur, uint32_t& pos, uint32_t& next_doc) {
  uint32_t j = cur, touched16 = 0;
  if (!(cache_valid && j < L.n_total && __ldg(L.last_doc + j) >= lo)) {
    j = first_block_ge(L.last_doc, cache_valid ? j + 1u : 0u, L.n_total, lo, lane);
    cur = j;
    if (j >= L.n_total) { pos = 128u; next_doc = kNoDoc; return 0; }
    touched16 = strip_cache_block(L, j, sc, max_doc, cc, lane);
  }
  uint32_t below = 0;  // entries are in doc order, padding is kNoDoc: count what lies before lo
#pragma unroll
  for (uint32_t g = 0; g < 4; ++g) below += (uint32_t)__popc(__ballot_sync(kFull, cc.doc[g * 32u + lane] < lo));
  pos = below;
  next_doc = below < 128u ? cc.doc[below] : kNoDoc;
  return touched16;
}

// MaxScore on top of the strips (exact).  The planner orders a union's clauses by descending Bm25Weight.weight — that is
// the order the f32 sum is taken in — so the clauses whose upper bounds (score < weight, since tf/(tf+norm) < 1) add up
// to less than the current threshold are always a SUFFIX of the clause list: the non-essential clauses.  Per window the
// warp applies the essential prefix; if the largest partial sum plus the non-essential bound cannot reach the threshold,
// the window is cold and the non-essential clauses (the dense, expensive ones) are not decoded at all; otherwise they
// are added on top, in order, which continues the very same f32 sum.  A doc without any essential posting scores below
// the threshold by construction.  Non-essential clauses fall behind while windows stay cold and catch up through the
// block table when a window turns hot.
__global__ void __launch_bounds__(kStripThreads) k_or_strip(const BatchParams P, uint32_t unit_base, uint32_t n_cached_max) {
  extern __shared__ __align__(16) unsigned char s_dyn[];
  __shared__ ListDesc s_list[kStripMaxLists];
  __shared__ QList s_ql[kStripMaxLists];
  const Unit U = P.units[unit_base + blockIdx.x];
  const QSeg S = P.qsegs[U.qseg];
  const DQuery Q = P.queries[S.query];
  QState* qs = P.qstate + S.query;
  const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
  if (threadIdx.x < S.n_lists) {
    s_ql[threadIdx.x] = P.qlists[S.lists_base + threadIdx.x];
    s_list[threadIdx.x] = P.lists[s_ql[threadIdx.x].list_id];
  }
  __syncthreads();  // the only block-wide barrier
  const size_t per_warp = sizeof(StripWarpFixed) + (size_t)n_cached_max * sizeof(StripCache);
  StripWarpFixed& W = *reinterpret_cast<StripWarpFixed*>(s_dyn + warp * per_warp);
  StripCache* C = reinterpret_cast<StripCache*>(s_dyn + warp * per_warp + sizeof(StripWarpFixed));
  const float neg_zero = __uint_as_float(0x80000000u);
  // this warp's windows
  const uint32_t n_win = U.end - U.begin;
  const uint32_t w_begin = U.begin + (uint32_t)(((unsigned long long)n_win * warp) / kStripWarps);
  const uint32_t w_end = U.begin + (uint32_t)(((unsigned long long)n_win * (warp + 1)) / kStripWarps);
  for (uint32_t i = lane; i < kWin; i += 32) W.acc[i] = neg_zero;
  const bool staged_fn = (S.flags & 1u) && S.fieldnorm != nullptr;
  const bool prunable = (S.flags & 2u) != 0;  // every weight finite and >= 0
  uint32_t thick_mask = 0;
  uint32_t n_e_min = 0;  // only the thick clauses at the end of the list may turn non-essential: thin ones are cheap to
                         // apply and every clause kept essential tightens the cold-window test
  uint32_t cnt = 0;
  if (lane < 8) W.stat[lane] = 0;  // [5]: postings and fieldnorm bytes actually read, in 16-byte units (SURVEY.md §8d: pruned kernels)
  __syncwarp();
  unsigned long long theta = (unsigned long long)(*(volatile unsigned int*)&qs->theta) << 32;
  if (w_begin < w_end) {
    // ---- strip start: position every clause -------------------------------------------------------------
    const uint32_t lo0 = w_begin * kWin;
    for (uint32_t t = 0; t < S.n_lists; ++t) {
      const ListDesc& L = s_list[t];
      const bool thin = (s_ql[t].pad & 1u) != 0;
      if (!thin) {
        thick_mask |= 1u << t;
        const uint32_t j = first_block_ge(L.last_doc, 0, L.n_total, lo0, lane);
        if (lane == 0) { W.cur[t] = j; W.next_doc[t] = 0; }
      } else {
        uint32_t cur = 0, pos = 0, nd = kNoDoc;
        const uint32_t t16 = strip_thin_seek(L, make_scorer(P, s_ql[t]), S.max_doc, C[s_ql[t].pad >> 1], false, lo0, lane, cur, pos, nd);
        if (lane == 0) { W.cur[t] = cur; W.pos[t] = pos; W.next_doc[t] = nd; W.stat[5] += t16; }
      }
    }
    __syncwarp();
    {  // a clause may turn non-essential when it has at least one posting per kStripNeDiv docs
      n_e_min = S.n_lists;
      while (n_e_min > 0 && (unsigned long long)s_list[n_e_min - 1u].doc_freq * kStripNeDiv >= S.max_doc) --n_e_min;
      // no such clause: the single densest one may still go if it is dense enough to matter (kStripNeDiv2)
      if (n_e_min == S.n_lists && n_e_min > 1 && (unsigned long long)s_list[n_e_min - 1u].doc_freq * kStripNeDiv2 >= S.max_doc) --n_e_min;
    }
    // ---- the windows ---------------------------------------------------------------------------------------
    uint32_t since_refresh = 0;
    for (uint32_t w = w_begin; w < w_end; ++w) {
      const float theta_f = threshold_score((uint32_t)(theta >> 32));
      // essential prefix [0, n_e) / non-essential suffix and its score bound under the current threshold
      uint32_t n_e = S.n_lists;
      float ne_bound = 0.0f;
      if (prunable && theta_f > 0.0f) {
        while (n_e > n_e_min) {
          const float nb = ne_bound + s_ql[n_e - 1u].weight;
          if (!(nb * 1.00001f < theta_f)) break;
          ne_bound = nb;
          --n_e;
        }
        if (n_e == 0) break;  // no doc of this segment can reach the threshold any more
      }
      if (!(thick_mask & ((1u << n_e) - 1u))) {  // only thin essential clauses: jump to the window of their next unread doc
        uint32_t nd = lane < n_e ? W.next_doc[lane] : kNoDoc;
        nd = warp_min(nd);
        if (nd == kNoDoc) break;
        const uint32_t wj = nd / kWin;
        if (wj >= w_end) break;
        if (wj > w) w = wj;
      }
      const uint32_t lo = w * kWin;
      const uint32_t hi = min(lo + kWin, S.max_doc);
      if (++since_refresh == 16u) {  // pick up the query-wide threshold now and then
        since_refresh = 0;
        unsigned int g = lane == 0 ? *(volatile unsigned int*)&qs->theta : 0u;
        g = __shfl_sync(kFull, g, 0);
        const unsigned long long gt = (unsigned long long)g << 32;
        if (gt > theta) theta = gt;
      }
      bool fn_ready = false;  // the window's fieldnorm bytes are staged when the first thick clause needs them
      bool dirty = false;     // the window received at least one score
      bool cold = false;
      float wmax = 0.0f;      // largest partial sum written by this lane (scores are non-negative: it bounds the final sums)
      for (uint32_t t = 0; t < S.n_lists; ++t) {
        if (t >= n_e) {  // can the clauses still to come lift a doc of this window over the threshold?  (asked again
                         // after every non-essential clause: the densest ones come last)
          const float mx = __uint_as_float(__reduce_max_sync(kFull, __float_as_uint(wmax)));
          if ((mx + ne_bound) * 1.00001f < theta_f) { cold = true; break; }
          ne_bound -= s_ql[t].weight;  // (rounding stays far inside the 1e-5 margin of the test)
        }
        const ListDesc& L = s_list[t];
        const bool thin = (s_ql[t].pad & 1u) != 0;
        if (!thin) {
          // ---- thick clause: decode the blocks that overlap [lo, hi) ---------------------------------------
          uint32_t cur = W.cur[t];
          if (cur >= L.n_total) continue;
          uint4 r;
          unsigned m;
          {
            const uint32_t idx = cur + lane;
            r = idx < L.n_total ? __ldg(L.tab4 + idx) : make_uint4(0xFFFFFFFFu, 0, 0, 0);
            m = __ballot_sync(kFull, r.x >= lo);
            if (!m) {  // the clause sat out many windows: seek through the block table
              cur = first_block_ge(L.last_doc, cur + 32u, L.n_total, lo, lane);
              const uint32_t idx2 = cur + lane;
              r = idx2 < L.n_total ? __ldg(L.tab4 + idx2) : make_uint4(0xFFFFFFFFu, 0, 0, 0);
              m = __ballot_sync(kFull, r.x >= lo);
            }
          }
          uint32_t src = (uint32_t)__ffs(m) - 1u;
          uint32_t j = cur + src;
          __syncwarp();  // every lane has read W.cur[t]
          if (lane == 0) W.cur[t] = j;
          if (j >= L.n_total) continue;
          const Scorer sc = make_scorer(P, s_ql[t]);
          uint4 rec;
          rec.x = __shfl_sync(kFull, r.x, src); rec.y = __shfl_sync(kFull, r.y, src);
          rec.z = __shfl_sync(kFull, r.z, src); rec.w = __shfl_sync(kFull, r.w, src);
          if (rec.w != 0xFFFFFFFFu && rec.w + 1u >= hi) continue;  // the block starts at or after the window's end
          BlockFetch f;
          fetch_issue_rec(L, rec, lane, f);
          if (staged_fn && !fn_ready) {
            const uint4* fsrc = reinterpret_cast<const uint4*>(S.fieldnorm + lo);
            uint4* dst = reinterpret_cast<uint4*>(W.fn);
            for (uint32_t i = lane; i < kWin / 16u; i += 32) dst[i] = __ldg(fsrc + i);
            __syncwarp();
            fn_ready = true;
            if (lane == 0) W.stat[5] += kWin / 16u;
          }
          dirty = true;
          uint32_t t16 = 0;  // 16-byte units of packed postings read for this clause and window
          for (;;) {
            uint32_t doc[4], tf[4];
            const bool small_tf = ((f.meta >> 8) & 63u) <= 4u;  // (the VInt tail's marker reads as 63 bits)
            t16 += f.meta == 0xFFFFFFFFu ? L.tail_n / 2u : (f.meta & 31u) + ((f.meta >> 8) & 63u);
            fetch_decode(L, j, f, lane, doc, tf);
            // the next block is needed iff this one ends before the window does
            const bool more = rec.x < hi - 1u && j + 1u < L.n_total;
            if (more) {
              ++j; ++src;
              if (src == 32u) {  // ran off the probe: fetch the next 32 records
                cur = j; src = 0;
                const uint32_t idx = cur + lane;
                r = idx < L.n_total ? __ldg(L.tab4 + idx) : make_uint4(0xFFFFFFFFu, 0, 0, 0);
              }
              rec.x = __shfl_sync(kFull, r.x, src); rec.y = __shfl_sync(kFull, r.y, src);
              rec.z = __shfl_sync(kFull, r.z, src); rec.w = __shfl_sync(kFull, r.w, src);
              fetch_issue_rec(L, rec, lane, f);
            }
            // Branch-free: the four postings of a lane form four independent load chains (fieldnorm byte -> factor
            // table -> score slot) that overlap instead of running one after the other behind divergent branches.
            // Postings outside the window are steered to the lane's dummy slot behind the window (its value is never read back
            // for a result: all four loads precede the four stores).
            bool in[4];
            uint32_t slot[4], id[4];
            float fac[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              in[i] = doc[i] >= lo && doc[i] < hi;
              slot[i] = in[i] ? doc[i] - lo : kWin + lane;
              id[i] = staged_fn ? (uint32_t)W.fn[in[i] ? slot[i] : 0u]
                                : (L.fieldnorm ? (uint32_t)__ldg(L.fieldnorm + (in[i] ? doc[i] : 0u)) : 1u);
            }
            if (small_tf) {  // tf_bits <= 4: every term frequency of the block is inside the factor table
#pragma unroll
              for (int i = 0; i < 4; ++i) fac[i] = __ldg(sc.tf_table + (tf[i] << 8) + id[i]);
            } else {
              bool big = false;
#pragma unroll
              for (int i = 0; i < 4; ++i) {
                fac[i] = __ldg(sc.tf_table + (min(tf[i], kTfRows - 1u) << 8) + id[i]);
                big |= in[i] && tf[i] >= kTfRows;
              }
              if (__ballot_sync(kFull, big)) {  // a term frequency beyond the table: take the divide for those
#pragma unroll
                for (int i = 0; i < 4; ++i)
                  if (in[i] && tf[i] >= kTfRows) fac[i] = bm25_factor_large_tf(sc.cache, id[i], tf[i]);
              }
            }
            float a[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) a[i] = W.acc[slot[i]];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const float nv = __fadd_rn(a[i], __fmul_rn(sc.weight, fac[i]));
              W.acc[slot[i]] = nv;
              wmax = in[i] ? fmaxf(wmax, nv) : wmax;
            }
            if (!more) break;
          }
          if (lane == 0) W.stat[5] += t16;
          __syncwarp();
        } else {
          // ---- thin clause: the decoded block lives in shared memory ---------------------------------------
          StripCache& cc = C[s_ql[t].pad >> 1];
          if (W.next_doc[t] < lo) {  // it sat out some windows as a non-essential clause: skip what lies before this one
            uint32_t cur = W.cur[t], pos = 0, nd = kNoDoc;
            const uint32_t t16 = strip_thin_seek(L, make_scorer(P, s_ql[t]), S.max_doc, cc, cur < L.n_total, lo, lane, cur, pos, nd);
            __syncwarp();
            if (lane == 0) { W.cur[t] = cur; W.pos[t] = pos; W.next_doc[t] = nd; W.stat[5] += t16; }
            __syncwarp();
          }
          for (;;) {
            if (W.next_doc[t] >= hi) break;  // nothing of this clause in the window (also: clause exhausted)
            // entries are in doc order: the window's postings are the next few entries, one per lane
            uint32_t pos = W.pos[t];
            const uint32_t e = pos + lane;
            const uint32_t d = e < 128u ? cc.doc[e] : kNoDoc;
            const bool in = d < hi;  // d >= lo: everything before the cursor is consumed
            const uint32_t napp = (uint32_t)__popc(__ballot_sync(kFull, in));
            if (in) {
              const uint32_t slot = d - lo;
              const float nv = __fadd_rn(W.acc[slot], cc.score[e]);
              W.acc[slot] = nv;
              wmax = fmaxf(wmax, nv);
            }
            dirty = true;
            pos += napp;
            const uint32_t nxt = napp < 32u ? __shfl_sync(kFull, d, napp) : (pos < 128u ? cc.doc[pos] : kNoDoc);
            __syncwarp();
            if (nxt != kNoDoc) {  // the block still holds unread docs (in this window only if all 32 lanes applied)
              if (lane == 0) { W.pos[t] = pos; W.next_doc[t] = nxt; }
              __syncwarp();
              continue;
            }
            // block used up: bring in the next one
            const uint32_t jb = W.cur[t] + 1u;
            __syncwarp();  // every lane has read W.cur[t]
            if (jb >= L.n_total) { if (lane == 0) { W.cur[t] = L.n_total; W.next_doc[t] = kNoDoc; } __syncwarp(); break; }
            const uint32_t t16 = strip_cache_block(L, jb, make_scorer(P, s_ql[t]), S.max_doc, cc, lane);
            const uint32_t first = cc.doc[0];  // a block's first entry is always a real doc
            if (lane == 0) { W.cur[t] = jb; W.next_doc[t] = first; W.pos[t] = 0; W.stat[5] += t16; }
            __syncwarp();
          }
        }
      }
      if (lane == 0) ++W.stat[n_e == S.n_lists ? 1 : (cold ? 3 : 2)];
      // ---- harvest -----------------------------------------------------------------------------------------------
      if (dirty) {
        // the largest partial sum any lane wrote bounds every final score of the window (scores >= 0; a negative
        // one makes the uint compare fail safe): when it is below the threshold the window is only cleared
        const uint32_t mx = __reduce_max_sync(kFull, __float_as_uint(wmax));
        const bool may_pass = !cold && (!(theta_f > 0.0f) || mx >= __float_as_uint(theta_f));
        for (uint32_t g = 0; g < kWin / 128; ++g) {
          const uint32_t idx = g * 128 + lane * 4;
          float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
          if (may_pass) v = *reinterpret_cast<const float4*>(W.acc + idx);
          *reinterpret_cast<float4*>(W.acc + idx) = make_float4(neg_zero, neg_zero, neg_zero, neg_zero);
          // float test first (nearly everything fails it); keys are built for the survivors only
          if (may_pass && __ballot_sync(kFull, v.x >= theta_f || v.y >= theta_f || v.z >= theta_f || v.w >= theta_f)) {
            const float vv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
            for (int c = 0; c < 4; ++c) {
              const uint32_t d = lo + idx + c;
              const unsigned long long key = make_key(vv[c], d);
              bool pass = vv[c] >= theta_f && __float_as_uint(vv[c]) != 0x80000000u && key >= theta;
              if (pass && S.alive) pass = is_alive(S.alive, d);
              unsigned mm = __ballot_sync(kFull, pass);
              if (mm) {
                if (cnt + 32u > kWBuf) {  // make room for one key per lane; the threshold may rise
                  strip_compact(W.keys, cnt, Q.k, theta, &qs->theta, lane);
                  pass = pass && key >= theta;
                  mm = __ballot_sync(kFull, pass);
                }
                if (pass) W.keys[cnt + __popc(mm & lanemask_lt(lane))] = key;
                cnt += __popc(mm);
              }
            }
            __syncwarp();
          }
        }
      }
      __syncwarp();  // cursor updates of this window are visible to the next one
    }
  }
  __syncwarp();
  if (P.counters && (lane == 1 || lane == 2 || lane == 3 || lane == 5) && W.stat[lane])
    atomicAdd(&P.counters[lane], (unsigned long long)W.stat[lane] * (lane == 5 ? 16ull : 1ull));
  // ---- hand the survivors over ------------------------------------------------------------------------------
  if (cnt > Q.k) strip_compact(W.keys, cnt, Q.k, theta, &qs->theta, lane);
  unsigned base = 0;
  if (lane == 0 && cnt) base = atomicAdd(&qs->cand_count, cnt);
  base = __shfl_sync(kFull, base, 0);
  for (uint32_t i = lane; i < cnt; i += 32) {
    if (base + i < Q.cand_cap) {
      const unsigned long long key = W.keys[i];
      Cand c;
      c.score_key = (uint32_t)(key >> 32);
      c.segment_ord = S.segment_ord;
      c.doc = 0xFFFFFFFFu - (uint32_t)key;
      c.pad = 0;
      P.cands[Q.cand_base + base + i] = c;
    }
  }
}

// ---- final per-query selection -----------------------------------------------------------------------------
// Keys: a = score_key:32 | (0xFFFFFFFF - segment_ord):32, b = ~doc; descending (a, b) is
// (score desc, segment_ord asc, doc asc) = compare_for_top_k (top_score_collector.rs:591-600).
__device__ __noinline__ void sort_pairs_desc(unsigned long long* a, uint32_t* b, unsigned n) {
  unsigned size = 2;
  while (size < n) size <<= 1;
  for (unsigned i = threadIdx.x; i < size; i += blockDim.x)
    if (i >= n) { a[i] = 0ull; b[i] = 0u; }
  __syncthreads();
  for (unsigned kk = 2; kk <= size; kk <<= 1) {
    for (unsigned j = kk >> 1; j > 0; j >>= 1) {
      for (unsigned i = threadIdx.x; i < size; i += blockDim.x) {
        const unsigned ixj = i ^ j;
        if (ixj > i) {
          const unsigned long long a1 = a[i], a2 = a[ixj];
          const uint32_t b1 = b[i], b2 = b[ixj];
          const bool first_less = a1 < a2 || (a1 == a2 && b1 < b2);
          const bool first_greater = a1 > a2 || (a1 == a2 && b1 > b2);
          const bool desc = (i & kk) == 0;
          if (desc ? first_less : first_greater) { a[i] = a2; a[ixj] = a1; b[i] = b2; b[ixj] = b1; }
        }
      }
      __syncthreads();
    }
  }
}

// ---- Count collector (N4): how many alive docs match, no scores ----------------------------------------------------
// src/collector/count_collector.rs + Weight::count (term_weight.rs:179-219, boolean_weight.rs): one CTA walks its share
// of a (query, segment)'s doc-id tiles; a tile is a bitmap in shared memory, a clause sets the bits of its postings
// (OR: into the result, AND: into a scratch bitmap that is then intersected), the alive bitset is and-ed in, popcount.
struct CountSeg {
  uint32_t query, lists_base, n_lists, max_doc;
  const uint8_t* alive;
  uint32_t op, pad;
};
struct CountParams {
  const ListDesc* lists;
  const uint32_t* list_ids;
  const CountSeg* segs;
  const Unit* units;
  unsigned long long* counts;
};

__global__ void __launch_bounds__(kThreads) k_count(const CountParams P) {
  constexpr uint32_t kWords = kTileDocs / 32u;
  __shared__ uint32_t s_acc[kWords], s_tmp[kWords];
  __shared__ uint32_t s_part[kWarps];
  const Unit U = P.units[blockIdx.x];
  const CountSeg S = P.segs[U.qseg];
  const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
  uint32_t total = 0;
  for (uint32_t tile = U.begin; tile < U.end; ++tile) {
    const uint32_t lo = tile * kTileDocs, hi = min(lo + kTileDocs, S.max_doc);
    for (uint32_t c = 0; c < S.n_lists; ++c) {
      uint32_t* bitmap = (S.op == 1u && c > 0) ? s_tmp : s_acc;  // 1 == TQ_OP_AND
      if (c == 0 || S.op == 1u)
        for (uint32_t w = threadIdx.x; w < kWords; w += blockDim.x) bitmap[w] = 0;
      __syncthreads();
      const ListDesc L = P.lists[P.list_ids[S.lists_base + c]];
      const uint32_t j0 = first_block_ge(L.last_doc, 0, L.n_total, lo, lane);
      for (uint32_t j = j0 + warp; j < L.n_total; j += kWarps) {
        const uint32_t prev = __ldg(&L.tab4[j].w);
        if (prev != 0xFFFFFFFFu && prev + 1u >= hi) break;  // the block starts at or after the tile's end
        uint32_t doc[4], tf[4];
        decode_block(L, j, lane, doc, tf);
#pragma unroll
        for (int i = 0; i < 4; ++i)
          if (doc[i] >= lo && doc[i] < hi) atomicOr(&bitmap[(doc[i] - lo) >> 5], 1u << ((doc[i] - lo) & 31u));
      }
      __syncthreads();
      if (S.op == 1u && c > 0) {
        for (uint32_t w = threadIdx.x; w < kWords; w += blockDim.x) s_acc[w] &= s_tmp[w];
        __syncthreads();
      }
    }
    for (uint32_t w = threadIdx.x; w < kWords; w += blockDim.x) {
      uint32_t bits = s_acc[w];
      if (bits && S.alive) bits &= __ldg(reinterpret_cast<const uint32_t*>(S.alive) + ((lo >> 5) + w));  // 32 docs per word, little endian
      total += (uint32_t)__popc(bits);
    }
    __syncthreads();
  }
  total = __reduce_add_sync(kFull, total);
  if (lane == 0) s_part[warp] = total;
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned long long sum = 0;
    for (int w = 0; w < kWarps; ++w) sum += s_part[w];
    if (sum) atomicAdd(&P.counts[S.query], sum);
  }
}

// Count for mixed boolean shapes (TQ_OP_BOOL; Weight::count over BooleanWeight::complex_scorer's scorer, boolean_weight.rs:236-431):
// per 8192-doc tile a result bitmap = AND over the MUST groups of (OR of the group's clauses), SHOULD clauses counted per doc
// (byte counters, four to a word) against `need`, MUST_NOT clauses cleared, alive bits and-ed in, popcount.
// words = [n_groups, need, n_should, n_not, (len, list ids..) per group, should list ids.., not list ids..] (32-bit).
struct CountBoolSeg {
  uint32_t query, words_base, max_doc, pad;
  const uint8_t* alive;
};
struct CountBoolParams {
  const ListDesc* lists;
  const uint32_t* words;
  const CountBoolSeg* segs;
  const Unit* units;
  unsigned long long* counts;
};

template <class F>
__device__ __forceinline__ void count_for_each_posting(const ListDesc& L, uint32_t lo, uint32_t hi, uint32_t lane, uint32_t warp, F f) {
  const uint32_t j0 = first_block_ge(L.last_doc, 0, L.n_total, lo, lane);
  for (uint32_t j = j0 + warp; j < L.n_total; j += kWarps) {
    const uint32_t prev = __ldg(&L.tab4[j].w);
    if (prev != 0xFFFFFFFFu && prev + 1u >= hi) break;  // the block starts at or after the tile's end
    uint32_t doc[4], tf[4];
    decode_block(L, j, lane, doc, tf);
#pragma unroll
    for (int i = 0; i < 4; ++i)
      if (doc[i] >= lo && doc[i] < hi) f(doc[i] - lo);
  }
}

__global__ void __launch_bounds__(kThreads) k_count_bool(const CountBoolParams P) {
  constexpr uint32_t kWords = kTileDocs / 32u;
  __shared__ uint32_t s_acc[kWords], s_tmp[kWords];
  __shared__ uint32_t s_cnt[kTileDocs / 4u];
  __shared__ uint32_t s_part[kWarps];
  const Unit U = P.units[blockIdx.x];
  const CountBoolSeg S = P.segs[U.qseg];
  const uint32_t* __restrict__ W = P.words + S.words_base;
  const uint32_t ng = W[0], need = W[1], ns = W[2], nn = W[3];
  const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
  uint32_t total = 0;
  for (uint32_t tile = U.begin; tile < U.end; ++tile) {
    const uint32_t lo = tile * kTileDocs, hi = min(lo + kTileDocs, S.max_doc);
    for (uint32_t w = threadIdx.x; w < kWords; w += blockDim.x) s_acc[w] = 0xFFFFFFFFu;
    uint32_t x = 4;
    for (uint32_t g = 0; g < ng; ++g) {
      const uint32_t glen = W[x++];
      for (uint32_t w = threadIdx.x; w < kWords; w += blockDim.x) s_tmp[w] = 0;
      __syncthreads();
      for (uint32_t e = 0; e < glen; ++e, ++x) {
        const ListDesc L = P.lists[W[x]];
        count_for_each_posting(L, lo, hi, lane, warp, [&](uint32_t o) { atomicOr(&s_tmp[o >> 5], 1u << (o & 31u)); });
      }
      __syncthreads();
      for (uint32_t w = threadIdx.x; w < kWords; w += blockDim.x) s_acc[w] &= s_tmp[w];
      __syncthreads();
    }
    if (need) {
      for (uint32_t w = threadIdx.x; w < kTileDocs / 4u; w += blockDim.x) s_cnt[w] = 0;
      __syncthreads();
      for (uint32_t e = 0; e < ns; ++e) {
        const ListDesc L = P.lists[W[x + e]];
        count_for_each_posting(L, lo, hi, lane, warp, [&](uint32_t o) { atomicAdd(&s_cnt[o >> 2], 1u << ((o & 3u) * 8u)); });  // <= 32 clauses: no carry
      }
      __syncthreads();
      for (uint32_t w = threadIdx.x; w < kWords; w += blockDim.x) {
        uint32_t m = 0;
#pragma unroll
        for (uint32_t b = 0; b < 8; ++b) {
          const uint32_t c4 = s_cnt[w * 8u + b];
#pragma unroll
          for (uint32_t k = 0; k < 4; ++k) m |= (((c4 >> (8u * k)) & 255u) >= need ? 1u : 0u) << (b * 4u + k);
        }
        s_acc[w] &= m;
      }
      __syncthreads();
    }
    x += ns;
    if (nn) {
      for (uint32_t w = threadIdx.x; w < kWords; w += blockDim.x) s_tmp[w] = 0;
      __syncthreads();
      for (uint32_t e = 0; e < nn; ++e) {
        const ListDesc L = P.lists[W[x + e]];
        count_for_each_posting(L, lo, hi, lane, warp, [&](uint32_t o) { atomicOr(&s_tmp[o >> 5], 1u << (o & 31u)); });
      }
      __syncthreads();
      for (uint32_t w = threadIdx.x; w < kWords; w += blockDim.x) s_acc[w] &= ~s_tmp[w];
      __syncthreads();
    }
    __syncthreads();
    for (uint32_t w = threadIdx.x; w < kWords; w += blockDim.x) {
      uint32_t bits = s_acc[w];
      const uint32_t first = lo + w * 32u;
      if (first >= hi) bits = 0;
      else if (hi - first < 32u) bits &= (1u << (hi - first)) - 1u;  // docs beyond max_doc
      if (bits && S.alive) bits &= __ldg(reinterpret_cast<const uint32_t*>(S.alive) + ((lo >> 5) + w));
      total += (uint32_t)__popc(bits);
    }
    __syncthreads();
  }
  total = __reduce_add_sync(kFull, total);
  if (lane == 0) s_part[warp] = total;
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned long long sum = 0;
    for (int w = 0; w < kWarps; ++w) sum += s_part[w];
    if (sum) atomicAdd(&P.counts[S.query], sum);
  }
}

// ---- mixed boolean shapes (TQ_OP_BOOL), per query ----------------------------------------------------------------------
// The per-query form of tile_eval_bool (tq_tile.cuh): BooleanWeight::complex_scorer for term leaves (boolean_weight.rs:236-431),
// evaluated window by window like k_count_bool matches and k_or scores.  The QSeg's clauses are laid out
//   MUST groups (ascending cost; each group's clauses by descending weight), SHOULD clauses, MUST_NOT clauses
// with QList.pad = role | group << 2 and QSeg.flags bits [8:16) = number of groups, [16:24) = SHOULD clauses needed.
// Per window: each group's clauses are added into a per-doc group score (first match assigned, clause order), folded into the
// running total (group order) and its presence bits and-ed into the match mask; an empty mask ends the window.  Then the SHOULD
// clauses (a second sum + per-doc counts), the MUST_NOT clauses (cleared from the mask), and the harvest of k_or.
// score = ng ? (cnt ? total + ss : total) : ss, the f32 operations and order of tile_eval_bool and of the oracle's bool_for_each.
constexpr uint32_t kBoolDocs = 4096;  // doc ids per window
constexpr uint32_t kBoolWords = kBoolDocs / 32u;
constexpr uint32_t kBoolMust = 0, kBoolShould = 1, kBoolNot = 2;  // QList.pad & 3
constexpr size_t kBoolDynSmem = 2u * kBoolDocs * sizeof(float) + 2u * kBoolDocs + 2u * kBoolWords * 4u;

struct BoolShared {
  uint32_t blo[32], bhi[32];  // per clause: block range overlapping the window (blo > bhi: none)
  uint32_t cur[32];           // per clause: search cursor
  uint32_t npass;
  float bound;                // no doc of the segment scores above this (prunable shapes)
  uint32_t skip;
};

// Every posting of the clause's blocks [blo, bhi] that falls in [lo, hi): f(slot, score) (kScore: false passes 0).  Warps take
// the blocks round robin; the next block of a warp travels while this one is scored.
template <bool kScore, class F>
__device__ __forceinline__ void bool_for_each_posting(const BatchParams& P, const QList& ql, uint32_t blo, uint32_t bhi, uint32_t lo, uint32_t hi,
                                                      const uint8_t* s_fn, bool staged_fn, uint32_t warp, uint32_t lane, F f) {
  if (blo > bhi || blo + warp > bhi) return;
  const ListDesc L = P.lists[ql.list_id];
  const Scorer scr = make_scorer(P, ql);
  BlockFetch fch;
  fetch_issue(L, blo + warp, lane, fch);
  for (uint32_t b = blo + warp; b <= bhi; b += kWarps) {
    uint32_t doc[4], tf[4];
    fetch_decode(L, b, fch, lane, doc, tf);
    if (b + kWarps <= bhi) fetch_issue(L, b + kWarps, lane, fch);
    float sc[4] = {0.f, 0.f, 0.f, 0.f};
    if (kScore) {
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        if (doc[i] >= lo && doc[i] < hi) {
          const uint32_t id = staged_fn ? (uint32_t)s_fn[doc[i] - lo] : (L.fieldnorm ? (uint32_t)__ldg(L.fieldnorm + doc[i]) : 1u);
          sc[i] = bm25_score_id(scr, id, tf[i]);
        }
      }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i)
      if (doc[i] >= lo && doc[i] < hi) f(doc[i] - lo, sc[i]);
  }
}

__global__ void __launch_bounds__(kThreads, 2) k_bool(const BatchParams P, uint32_t unit_base) {
  extern __shared__ __align__(16) float s_tot[];                          // [kBoolDocs] sum of the group scores
  float* s_part = s_tot + kBoolDocs;                                      // [kBoolDocs] the current group's score, then the SHOULD sum
  uint32_t* s_mask = reinterpret_cast<uint32_t*>(s_part + kBoolDocs);     // [kBoolWords] docs still matching
  uint32_t* s_pres = s_mask + kBoolWords;                                 // [kBoolWords] docs the current group lists
  uint8_t* s_cnt = reinterpret_cast<uint8_t*>(s_pres + kBoolWords);       // [kBoolDocs] SHOULD clauses listing the doc
  uint8_t* s_fn = s_cnt + kBoolDocs;                                      // [kBoolDocs] fieldnorm ids of the window
  __shared__ CtaTopK s_top;
  __shared__ BoolShared sh;
  const Unit U = P.units[unit_base + blockIdx.x];
  const QSeg S = P.qsegs[U.qseg];
  const DQuery Q = P.queries[S.query];
  QState* qs = P.qstate + S.query;
  const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
  const float neg_zero = __uint_as_float(0x80000000u);  // -0.0 + s == s bit for bit: a slot holding it takes its first score as is
  const bool staged_fn = (S.flags & 1u) && S.fieldnorm != nullptr;
  const bool prunable = (S.flags & 2u) != 0;
  const uint32_t ng = (S.flags >> 8) & 255u, need = (S.flags >> 16) & 255u;
  if (threadIdx.x < 32) sh.cur[threadIdx.x] = 0;
  if (threadIdx.x == 0) {
    s_top.count = 0; s_top.theta = (unsigned long long)qs->theta << 32;
    sh.npass = 0;
    // a doc scores less than the sum of the MUST and SHOULD weights: a clause adds less than its weight (tf/(tf+norm) < 1,
    // bm25.rs:170-175); used only when every weight is finite and >= 0
    float sum = 0.0f;
    for (uint32_t t = 0; t < S.n_lists; ++t) {
      const QList ql = P.qlists[S.lists_base + t];
      if ((ql.pad & 3u) != kBoolNot) sum += ql.weight;
    }
    sh.bound = sum * 1.00001f;  // f32 sums of up to 32 non-negative terms differ by < 4e-6 relative, whatever the order
  }
  __syncthreads();
  const TopK T{s_top.keys, &s_top.count, &s_top.theta, &s_top.scratch, (unsigned)kThreads};
  for (uint32_t win = U.begin; win < U.end; ++win) {
    const uint32_t lo = win * kBoolDocs;
    const uint32_t hi = min(lo + kBoolDocs, S.max_doc);
    // ---- block ranges of every clause in this window ---------------------------------------------------------------
    for (uint32_t t = warp; t < S.n_lists; t += kWarps) {
      const QList ql = P.qlists[S.lists_base + t];
      const uint32_t* last_doc = P.lists[ql.list_id].last_doc;
      const uint32_t n_total = P.lists[ql.list_id].n_total;
      uint32_t blo = 1, bhi = 0;
      const uint32_t j_lo = first_block_ge(last_doc, sh.cur[t], n_total, lo, lane);
      if (j_lo < n_total) {
        uint32_t j_hi = first_block_ge(last_doc, j_lo, n_total, hi - 1u, lane);  // the last block that can hold a doc < hi
        if (j_hi >= n_total) j_hi = n_total - 1u;
        blo = j_lo; bhi = j_hi;
      }
      if (lane == 0) { sh.blo[t] = blo; sh.bhi[t] = bhi; sh.cur[t] = j_lo; }
    }
    __syncthreads();
    // ---- skip: a MUST group without a block here, too few SHOULD clauses with one, or a bound under the threshold ------
    if (threadIdx.x == 0) {
      const unsigned long long g = (unsigned long long)(*(volatile unsigned int*)&qs->theta) << 32;
      if (g > s_top.theta) s_top.theta = g;
      bool skip = prunable && sh.bound < threshold_score((uint32_t)(s_top.theta >> 32));
      uint32_t n_should = 0, group = 0, group_any = 0;
      for (uint32_t t = 0; t < S.n_lists && !skip; ++t) {
        const uint32_t pad = P.qlists[S.lists_base + t].pad;
        const bool has = sh.blo[t] <= sh.bhi[t];
        if ((pad & 3u) == kBoolMust) {
          if ((pad >> 2) != group) { skip = !group_any; group = pad >> 2; group_any = 0; }
          group_any |= has;
        } else if ((pad & 3u) == kBoolShould) {
          n_should += has;
        }
      }
      if (ng && !group_any) skip = true;  // the last group
      sh.skip = skip || n_should < need;
    }
    __syncthreads();
    if (sh.skip) continue;  // (uniform: read between two barriers; the next write is behind the next window's barrier)

    if (staged_fn) {
      const uint4* src = reinterpret_cast<const uint4*>(S.fieldnorm + lo);
      uint4* dst = reinterpret_cast<uint4*>(s_fn);
      for (uint32_t i = threadIdx.x; i < kBoolDocs / 16; i += kThreads) dst[i] = __ldg(src + i);
    }
    for (uint32_t i = threadIdx.x; i < kBoolDocs; i += kThreads) s_part[i] = neg_zero;
    for (uint32_t w = threadIdx.x; w < kBoolWords; w += kThreads) {
      const uint32_t first = lo + w * 32u;
      s_mask[w] = first >= hi ? 0u : (hi - first >= 32u ? 0xFFFFFFFFu : (1u << (hi - first)) - 1u);  // docs below max_doc
      s_pres[w] = 0;
    }
    __syncthreads();
    // ---- MUST groups ------------------------------------------------------------------------------------------------
    uint32_t t = 0;
    bool matching = true;
    for (uint32_t g = 0; g < ng && matching; ++g) {
      for (; t < S.n_lists; ++t) {
        const QList ql = P.qlists[S.lists_base + t];
        if ((ql.pad & 3u) != kBoolMust || (ql.pad >> 2) != g) break;
        bool_for_each_posting<true>(P, ql, sh.blo[t], sh.bhi[t], lo, hi, s_fn, staged_fn, warp, lane, [&](uint32_t slot, float sc) {
          s_part[slot] = __fadd_rn(s_part[slot], sc);
          atomicOr(&s_pres[slot >> 5], 1u << (slot & 31u));
        });
        __syncthreads();  // clause order is the f32 summation order
      }
      for (uint32_t i = threadIdx.x; i < kBoolDocs; i += kThreads) {
        const float v = s_part[i];
        s_tot[i] = g ? __fadd_rn(s_tot[i], v) : v;
        s_part[i] = neg_zero;
      }
      uint32_t any = 0;
      for (uint32_t w = threadIdx.x; w < kBoolWords; w += kThreads) {
        const uint32_t m = s_mask[w] & s_pres[w];
        s_mask[w] = m;
        s_pres[w] = 0;
        any |= m;
      }
      matching = __syncthreads_or(any != 0) != 0;
    }
    if (!matching) continue;  // no doc of the window has every MUST group
    // ---- SHOULD clauses: their sum (s_part) and how many list the doc ------------------------------------------------
    const uint32_t should_begin = t;
    for (; t < S.n_lists && (P.qlists[S.lists_base + t].pad & 3u) == kBoolShould; ++t) {
      if (t == should_begin) {
        for (uint32_t i = threadIdx.x; i < kBoolDocs / 16; i += kThreads) reinterpret_cast<uint4*>(s_cnt)[i] = make_uint4(0, 0, 0, 0);
        __syncthreads();
      }
      bool_for_each_posting<true>(P, P.qlists[S.lists_base + t], sh.blo[t], sh.bhi[t], lo, hi, s_fn, staged_fn, warp, lane, [&](uint32_t slot, float sc) {
        s_part[slot] = __fadd_rn(s_part[slot], sc);
        s_cnt[slot] = (uint8_t)(s_cnt[slot] + 1u);  // one posting per doc and clause: no other thread writes this byte now
      });
      __syncthreads();
    }
    const bool has_should = t > should_begin;
    // ---- MUST_NOT clauses ---------------------------------------------------------------------------------------------
    for (; t < S.n_lists; ++t)
      bool_for_each_posting<false>(P, P.qlists[S.lists_base + t], sh.blo[t], sh.bhi[t], lo, hi, s_fn, staged_fn, warp, lane, [&](uint32_t slot, float) {
        atomicAnd(&s_mask[slot >> 5], ~(1u << (slot & 31u)));
      });
    __syncthreads();

    // ---- harvest: final scores, the float pre-filter, the exact key test on the survivors (as k_or) ------------------
    const unsigned long long theta = *T.theta;
    const float theta_f = threshold_score((uint32_t)(theta >> 32));
    uint32_t passmask = 0;
#pragma unroll 1
    for (int j = 0; j < (int)(kBoolDocs / (kThreads * 4)); ++j) {
      const uint32_t idx = (j * kThreads + threadIdx.x) * 4;
      const uint32_t bits = (s_mask[idx >> 5] >> (idx & 31u)) & 15u;
      if (bits) {
        const float4 tv = *reinterpret_cast<const float4*>(s_tot + idx);
        const float4 sv = *reinterpret_cast<const float4*>(s_part + idx);
        const uint32_t cnt4 = has_should ? *reinterpret_cast<const uint32_t*>(s_cnt + idx) : 0u;
        const float tt[4] = {tv.x, tv.y, tv.z, tv.w}, ss[4] = {sv.x, sv.y, sv.z, sv.w};
        float vv[4];
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          const uint32_t cnt = (cnt4 >> (8 * c)) & 255u;
          vv[c] = ng ? (cnt ? __fadd_rn(tt[c], ss[c]) : tt[c]) : ss[c];
          const uint32_t d = lo + idx + c;
          bool pass = ((bits >> c) & 1u) && cnt >= need && vv[c] >= theta_f && make_key(vv[c], d) >= theta;
          if (pass && S.alive) pass = is_alive(S.alive, d);
          passmask |= pass ? (1u << (j * 4 + c)) : 0u;
        }
        *reinterpret_cast<float4*>(s_tot + idx) = make_float4(vv[0], vv[1], vv[2], vv[3]);  // read back by the push below
      }
    }
    const uint32_t wsum = __reduce_add_sync(kFull, (uint32_t)__popc(passmask));
    if (lane == 0 && wsum) atomicAdd(&sh.npass, wsum);
    __syncthreads();
    const uint32_t npass = sh.npass;
    const bool fits = *T.count + npass <= kCap;
    __syncthreads();
    if (threadIdx.x == 0) sh.npass = 0;
    if (!fits) topk_round_end(T, Q.k, &qs->theta);  // cold start: more survivors than the buffer holds; rounds with compaction between
#pragma unroll 1
    for (int j = 0; j < (int)(kBoolDocs / (kThreads * 4)); ++j) {
      const uint32_t idx = (j * kThreads + threadIdx.x) * 4;
      const uint32_t sub = (passmask >> (j * 4)) & 15u;
      if (__ballot_sync(kFull, sub != 0)) {
        const float4 v = *reinterpret_cast<const float4*>(s_tot + idx);
        const float vv[4] = {v.x, v.y, v.z, v.w};
        const unsigned long long th = fits ? 0ull : *T.theta;
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          const unsigned long long key = make_key(vv[c], lo + idx + c);
          topk_push(T, ((sub >> c) & 1u) && key >= th, key, lane);
        }
      }
      if (!fits) topk_round_end(T, Q.k, &qs->theta);
    }
    if (fits) topk_round_end(T, Q.k, &qs->theta);
  }
  topk_flush(T, Q, qs, P.cands, S.segment_ord);
}

// The exact k-th largest score key among a query's candidates so far (4-pass radix select) becomes a lower bound of
// its threshold: run between the sampled windows and the main launch of k_or_strip.
__global__ void __launch_bounds__(kThreads) k_theta(const BatchParams P) {
  __shared__ uint32_t s_hist[256];
  __shared__ uint32_t s_prefix, s_need;
  const uint32_t q = blockIdx.x;
  const DQuery Q = P.queries[q];
  if (Q.op == 3u) return;  // TQ_OP_PHRASE: one launch, possibly still running on the batch's second stream
  const uint32_t C = min(P.qstate[q].cand_count, Q.cand_cap);
  if (C < Q.k) return;  // fewer than k hits so far: no bound
  const Cand* cands = P.cands + Q.cand_base;
  if (threadIdx.x == 0) { s_prefix = 0; s_need = Q.k; }
  uint32_t mask = 0;
  for (int pass = 0; pass < 4; ++pass) {
    const int shift = 24 - 8 * pass;
    for (uint32_t i = threadIdx.x; i < 256; i += blockDim.x) s_hist[i] = 0;
    __syncthreads();
    const uint32_t prefix = s_prefix;
    for (uint32_t i = threadIdx.x; i < C; i += blockDim.x) {
      const uint32_t key = cands[i].score_key;
      if ((key & mask) == prefix) atomicAdd(&s_hist[(key >> shift) & 255u], 1u);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      uint32_t need = s_need, bsel = 0;
      for (int bin = 255; bin >= 0; --bin) {
        const uint32_t h = s_hist[bin];
        if (h >= need) { bsel = (uint32_t)bin; break; }
        need -= h;
      }
      s_need = need;
      s_prefix = prefix | (bsel << shift);
    }
    mask |= 0xFFu << shift;
    __syncthreads();
  }
  if (threadIdx.x == 0) atomicMax(&P.qstate[q].theta, s_prefix);
}

__global__ void k_theta_export(const QState* __restrict__ qs, long long* __restrict__ out, uint32_t n) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = (long long)qs[i].theta;
}
__global__ void k_theta_import(QState* __restrict__ qs, const long long* __restrict__ in, uint32_t n) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) atomicMax(&qs[i].theta, (unsigned int)in[i]);
}

// Exact top-k of a query's candidates. Small sets are sorted directly; large ones go through a
// 4-pass radix select on the score key (O(C)), then only the survivors and the boundary ties are sorted.
__global__ void __launch_bounds__(kThreads) k_final(const BatchParams P) {
  __shared__ unsigned long long s_a[kCap];
  __shared__ uint32_t s_b[kCap];
  __shared__ uint32_t s_hist[256];
  __shared__ uint32_t s_prefix, s_need, s_n, s_ties;
  const uint32_t q = blockIdx.x;
  const DQuery Q = P.queries[q];
  const uint32_t C = min(P.qstate[q].cand_count, Q.cand_cap);
  if (threadIdx.x == 0 && P.ovf && P.qstate[q].cand_count > Q.cand_cap) atomicExch(P.ovf, 1u);  // candidates were dropped: the host repeats the run
  const Cand* cands = P.cands + Q.cand_base;
  uint32_t have = 0;
  if (C <= kCap) {
    for (uint32_t i = threadIdx.x; i < C; i += blockDim.x) {
      const Cand c = cands[i];
      s_a[i] = ((unsigned long long)c.score_key << 32) | (unsigned long long)(0xFFFFFFFFu - c.segment_ord);
      s_b[i] = ~c.doc;
    }
    __syncthreads();
    sort_pairs_desc(s_a, s_b, C);
    have = min(C, Q.k);
  } else {
    // k-th largest score key (C > kCap >= k)
    if (threadIdx.x == 0) { s_prefix = 0; s_need = Q.k; s_n = 0; }  // (s_n: set here, behind the loop's barriers -- the four
                                                                    // words share one vector load further down)
    uint32_t mask = 0;
    for (int pass = 0; pass < 4; ++pass) {
      const int shift = 24 - 8 * pass;
      for (uint32_t i = threadIdx.x; i < 256; i += blockDim.x) s_hist[i] = 0;
      __syncthreads();
      const uint32_t prefix = s_prefix;
      for (uint32_t i = threadIdx.x; i < C; i += blockDim.x) {
        const uint32_t key = cands[i].score_key;
        if ((key & mask) == prefix) atomicAdd(&s_hist[(key >> shift) & 255u], 1u);
      }
      __syncthreads();
      if (threadIdx.x == 0) {
        uint32_t need = s_need, bsel = 0;
        for (int bin = 255; bin >= 0; --bin) {
          const uint32_t h = s_hist[bin];
          if (h >= need) { bsel = (uint32_t)bin; s_ties = h; break; }
          need -= h;
        }
        s_need = need;
        s_prefix = prefix | (bsel << shift);
      }
      mask |= 0xFFu << shift;
      __syncthreads();
    }
    const uint32_t kth = s_prefix;       // exactly the k-th largest score key
    const uint32_t ties_total = s_ties;   // how many candidates carry exactly that key
    const uint32_t above_total = Q.k - s_need;  // strictly better ones (< k)
    if (above_total + ties_total <= kCap) {  // the usual case: one sweep, one sort
      for (uint32_t i = threadIdx.x; i < C; i += blockDim.x) {
        const Cand c = cands[i];
        if (c.score_key >= kth) {
          const uint32_t slot = atomicAdd(&s_n, 1u);
          s_a[slot] = ((unsigned long long)c.score_key << 32) | (unsigned long long)(0xFFFFFFFFu - c.segment_ord);
          s_b[slot] = ~c.doc;
        }
      }
      __syncthreads();
      const uint32_t n = s_n;
      __syncthreads();
      sort_pairs_desc(s_a, s_b, n);
      have = min(n, Q.k);
    } else {  // a flood of equal scores: keep the best (segment, doc) of the ties slab by slab
      for (uint32_t i = threadIdx.x; i < C; i += blockDim.x) {
        const Cand c = cands[i];
        if (c.score_key > kth) {
          const uint32_t slot = atomicAdd(&s_n, 1u);
          s_a[slot] = ((unsigned long long)c.score_key << 32) | (unsigned long long)(0xFFFFFFFFu - c.segment_ord);
          s_b[slot] = ~c.doc;
        }
      }
      __syncthreads();
      have = s_n;
      uint32_t next = 0;
      for (;;) {
        __syncthreads();
        if (threadIdx.x == 0) s_n = have;
        __syncthreads();
        const uint32_t slab_end = min(C, next + (kCap - have));
        for (uint32_t i = next + threadIdx.x; i < slab_end; i += blockDim.x) {
          const Cand c = cands[i];
          if (c.score_key == kth) {
            const uint32_t slot = atomicAdd(&s_n, 1u);
            s_a[slot] = ((unsigned long long)c.score_key << 32) | (unsigned long long)(0xFFFFFFFFu - c.segment_ord);
            s_b[slot] = ~c.doc;
          }
        }
        __syncthreads();
        const uint32_t n = s_n;
        __syncthreads();
        sort_pairs_desc(s_a, s_b, n);
        have = min(n, Q.k);
        next = slab_end;
        if (next >= C) break;
      }
    }
  }
  for (uint32_t i = threadIdx.x; i < have; i += blockDim.x) {
    const size_t o = (size_t)q * P.res_stride + i;
    P.res_scores[o] = key_to_score((uint32_t)(s_a[i] >> 32));
    P.res_segs[o] = 0xFFFFFFFFu - (uint32_t)s_a[i];
    P.res_docs[o] = ~s_b[i];
  }
  if (threadIdx.x == 0) P.res_counts[q] = have;
}

// K7 (device half): merge_fruits across result sets gathered from several GPUs.
// in: n_lists result sets, each [nq][stride] rows sorted like k_final's output (+ [nq] counts), `row_pitch` / `count_pitch`
// elements apart (contiguous [n_lists][nq][stride] arrays: nq * stride / nq; one packed buffer per shard: its size);
// out: [nq][stride].
__global__ void __launch_bounds__(kThreads) k_merge(uint32_t n_lists, uint32_t nq, uint32_t stride, uint32_t k, size_t row_pitch, size_t count_pitch,
                                                    const float* __restrict__ in_scores, const uint32_t* __restrict__ in_segs,
                                                    const uint32_t* __restrict__ in_docs, const uint32_t* __restrict__ in_counts,
                                                    float* __restrict__ out_scores, uint32_t* __restrict__ out_segs,
                                                    uint32_t* __restrict__ out_docs, uint32_t* __restrict__ out_counts) {
  __shared__ unsigned long long s_a[kCap];
  __shared__ uint32_t s_b[kCap];
  const uint32_t q = blockIdx.x;
  uint32_t have = 0;
  for (uint32_t l = 0; l < n_lists; ++l) {
    const uint32_t cnt = min(min(in_counts[(size_t)l * count_pitch + q], stride), k);
    // have <= k <= 1024 and cnt <= 1024, so have + cnt <= kCap
    for (uint32_t i = threadIdx.x; i < cnt; i += blockDim.x) {
      const size_t o = (size_t)l * row_pitch + (size_t)q * stride + i;
      s_a[have + i] = ((unsigned long long)score_to_key(in_scores[o]) << 32) | (unsigned long long)(0xFFFFFFFFu - in_segs[o]);
      s_b[have + i] = ~in_docs[o];
    }
    const uint32_t n = have + cnt;
    __syncthreads();
    sort_pairs_desc(s_a, s_b, n);
    have = min(n, k);
  }
  for (uint32_t i = threadIdx.x; i < have; i += blockDim.x) {
    const size_t o = (size_t)q * stride + i;
    out_scores[o] = key_to_score((uint32_t)(s_a[i] >> 32));
    out_segs[o] = 0xFFFFFFFFu - (uint32_t)s_a[i];
    out_docs[o] = ~s_b[i];
  }
  if (threadIdx.x == 0) out_counts[q] = have;
}

}  // namespace tq
