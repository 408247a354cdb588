// Phrase queries on the device (SURVEY.md §8f N3): PhraseScorer; slop for two-term phrases (intersection_count_with_slop).
//
//   k_build_pos_tables  PositionReader::open + advance_num_blocks as ONE exclusive scan over the term's bit-width bytes
//                       (src/positions/reader.rs:43-80), the VInt rest decoded once (reader.rs:82-102), and the position
//                       offset of every posting block = the running sum of the skip records' tf_sum (src/postings/skip.rs:236-249,285)
//   k_phrase            Intersection over the phrase's terms (leader = rarest list, the others probed through their block tables
//                       exactly like k_and) + for every doc that holds all terms the phrase count: every term's positions shifted
//                       by (max_offset - its offset), size of the intersection of the shifted sets
//                       (phrase_scorer.rs:349-398,431-497 compute_phrase_count; intersection_count :60-90);
//                       score = Bm25Weight(for_terms).score(fieldnorm_id, phrase_count) (phrase_scorer.rs:576-589, bm25.rs:95-129)
//
// Position blocks are BitPacker4x blocks of 128 deltas (unsorted, not minus-one: positions/serializer.rs:66, reader.rs:94-95), read
// in place from the `.pos` bytes at arbitrary alignment.  A doc's positions are the `tf` deltas that start at
// (position offset of its posting block) + (sum of the tfs before it in the block) (segment_postings.rs:232-254).
#pragma once
#include "tq_kernels.cuh"

namespace tq {

constexpr uint32_t kPhraseMaxTerms = 8;
constexpr uint32_t kPhraseWarps = 4;
constexpr uint32_t kPhraseThreads = kPhraseWarps * 32;

struct PosDesc {  // one term's position stream in one segment, built on first use and cached with the segment
  const uint8_t* widths;                 // [n_blocks] bit width of every bit-packed block
  const uint32_t* blk_off;               // [n_blocks + 1] byte offset of block b from `blocks`
  const uint8_t* blocks;                 // the bit-packed blocks (in the `.pos` body, any alignment)
  const uint32_t* tail;                  // [tail_n] the VInt-encoded rest, decoded
  const unsigned long long* post_off;    // [n_posting_blocks + 1] positions that precede posting block b (last entry: the VInt tail block)
  uint32_t n_blocks, tail_n, status, pad;
};
struct PosJob {
  const uint8_t* pos_bytes;   // the term's positions range
  uint32_t pos_len;
  const uint8_t* list_bytes;  // the term's postings range (for the skip records)
  uint32_t list_len;
  uint32_t doc_freq;
  uint32_t pos_id;
  unsigned char* pool;        // the segment's table pool ...
  unsigned long long* pool_cursor;  // ... bump-allocated on the device (the sizes are in the data)
  unsigned long long pool_cap;
};
struct PhraseAux { uint32_t pos_id, offset, slop = 0; };  // per clause of a phrase (parallel to qlists): its position table, max_offset - its offset, the phrase's slop

__global__ void __launch_bounds__(kThreads) k_build_pos_tables(const PosJob* __restrict__ jobs, PosDesc* __restrict__ descs, uint32_t* __restrict__ status_out) {
  const PosJob J = jobs[blockIdx.x];
  PosDesc& D = descs[J.pos_id];
  __shared__ uint32_t s_hdr, s_nblocks, s_status, s_carry, s_skip_hdr;
  __shared__ unsigned long long s_base, s_carry64;
  __shared__ uint32_t s_wsum[kWarps];
  __shared__ unsigned long long s_wsum64[kWarps];
  const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
  const uint32_t n_post_blocks = J.doc_freq / 128u;
  if (tid == 0) {
    uint32_t status = 0, hdr = 0;
    unsigned long long v = 0;
    uint32_t shift = 0;
    bool done = false;
    while (hdr < J.pos_len && hdr < 10u) {  // VInt(number of bit-packed blocks), stop bit on the last byte (common/src/vint.rs)
      const uint8_t b = J.pos_bytes[hdr++];
      v |= (unsigned long long)(b & 127u) << shift;
      shift += 7;
      if (b & 128u) { done = true; break; }
    }
    if (!done || v > (unsigned long long)J.pos_len - hdr) status = 1;
    const uint32_t n_blocks = status ? 0u : (uint32_t)v;
    // skip section of the postings (12-byte records: ..., u32 tf_sum at byte 6)
    uint32_t shdr = 0;
    if (J.doc_freq >= 128u) {
      unsigned long long sl = 0;
      shift = 0;
      done = false;
      while (shdr < J.list_len && shdr < 10u) {
        const uint8_t b = J.list_bytes[shdr++];
        sl |= (unsigned long long)(b & 127u) << shift;
        shift += 7;
        if (b & 128u) { done = true; break; }
      }
      if (!done || sl > (unsigned long long)J.list_len - shdr || sl < 12ull * n_post_blocks) status = 1;
    }
    const unsigned long long need = (((unsigned long long)n_blocks + 1u) * 4u + 128u * 4u + ((unsigned long long)n_post_blocks + 2u) * 8u + 63u) & ~63ull;
    unsigned long long base = 0;
    if (!status) {
      base = atomicAdd(J.pool_cursor, need);
      if (base + need > J.pool_cap) status = 2;  // the segment's position-table pool is exhausted
    }
    s_hdr = hdr; s_nblocks = n_blocks; s_status = status; s_carry = 0; s_carry64 = 0; s_base = base; s_skip_hdr = shdr;
  }
  __syncthreads();
  const uint32_t n_blocks = s_nblocks;
  if (s_status == 0) {
    unsigned long long* post_off = reinterpret_cast<unsigned long long*>(J.pool + s_base);
    uint32_t* blk_off = reinterpret_cast<uint32_t*>(post_off + n_post_blocks + 2u);
    uint32_t* tail = blk_off + n_blocks + 1u;  // (the three arrays start 8-byte aligned: n_blocks + 1 words may leave `tail` 4-byte aligned, fine)
    const uint8_t* widths = J.pos_bytes + s_hdr;
    const uint8_t* blocks = widths + n_blocks;
    // byte offsets of the position blocks: exclusive scan of 16 * width
    for (uint32_t base = 0; base < n_blocks; base += kThreads) {
      const uint32_t i = base + tid;
      uint32_t size = 0;
      if (i < n_blocks) { size = 16u * (uint32_t)widths[i]; if (widths[i] > 32u) s_status = 1; }
      const uint32_t incl = warp_incl_scan(size, lane);
      if (lane == 31) s_wsum[warp] = incl;
      __syncthreads();
      uint32_t woff = 0;
#pragma unroll
      for (int w = 0; w < kWarps; ++w) woff += (w < (int)warp) ? s_wsum[w] : 0u;
      const uint32_t excl = s_carry + woff + incl - size;
      if (i < n_blocks) blk_off[i] = excl;
      __syncthreads();
      if (tid == kThreads - 1) s_carry = excl + size;
      __syncthreads();
    }
    // positions before every posting block: exclusive scan of the skip records' tf_sum
    const uint8_t* skip = J.list_bytes + s_skip_hdr;
    for (uint32_t base = 0; base < n_post_blocks; base += kThreads) {
      const uint32_t i = base + tid;
      unsigned long long v = 0;
      if (i < n_post_blocks) v = load_u32_unaligned(skip + (size_t)i * 12u + 6u);
      unsigned long long incl = v;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const unsigned long long nb = __shfl_up_sync(kFull, incl, o);
        if ((int)lane >= o) incl += nb;
      }
      if (lane == 31) s_wsum64[warp] = incl;
      __syncthreads();
      unsigned long long woff = 0;
#pragma unroll
      for (int w = 0; w < kWarps; ++w) woff += (w < (int)warp) ? s_wsum64[w] : 0ull;
      const unsigned long long excl = s_carry64 + woff + incl - v;
      if (i < n_post_blocks) post_off[i] = excl;
      __syncthreads();
      if (tid == kThreads - 1) s_carry64 = excl + v;
      __syncthreads();
    }
    if (tid == 0) {
      blk_off[n_blocks] = s_carry;
      post_off[n_post_blocks] = s_carry64;  // the VInt tail block of the postings starts after all full blocks
      uint32_t status = s_status, tail_n = 0;
      const uint32_t avail = J.pos_len - s_hdr - n_blocks;
      if (s_carry > avail) status = 1;
      if (!status) {  // the rest: VInt deltas until the range ends, fewer than 128 of them (reader.rs:96-101)
        const uint8_t* p = blocks + s_carry;
        const uint32_t remaining = avail - s_carry;
        uint32_t pos = 0;
        while (pos < remaining && tail_n < 128u) {
          uint32_t result = 0, shift = 0;
          for (;;) {
            if (pos >= remaining) { status = 1; break; }
            const uint8_t b = p[pos++];
            result += (uint32_t)(b & 127u) << shift;
            if (b & 128u) break;
            shift += 7;
          }
          if (status) break;
          tail[tail_n++] = result;
        }
      }
      D.widths = widths; D.blk_off = blk_off; D.blocks = blocks; D.tail = tail; D.post_off = post_off;
      D.n_blocks = n_blocks; D.tail_n = tail_n; D.status = status; D.pad = 0;
      status_out[blockIdx.x] = status;
    }
  } else if (tid == 0) {
    D.status = s_status;
    status_out[blockIdx.x] = s_status;
  }
}

// Delta number g of a term's position stream.
__device__ __forceinline__ uint32_t pos_delta(const PosDesc& D, unsigned long long g) {
  const unsigned long long b = g >> 7;
  if (b >= D.n_blocks) {
    const unsigned long long r = g - (unsigned long long)D.n_blocks * 128ull;
    return r < D.tail_n ? __ldg(D.tail + r) : 0u;
  }
  const uint32_t w = (uint32_t)__ldg(D.widths + b);
  if (w == 0u) return 0u;
  const uint32_t r = (uint32_t)(g & 127u);
  const uint32_t stream = r & 3u, bit = (r >> 2) * w;  // BitPacker4x: value j in stream j & 3 at bit (j >> 2) * w; word k of a stream is the stream-th word of vector k
  const uint8_t* base = D.blocks + __ldg(D.blk_off + b) + ((bit >> 5) * 4u + stream) * 4u;
  const uint32_t sh = bit & 31u;
  uint32_t v = load_u32_unaligned(base) >> sh;
  if (sh + w > 32u) v |= load_u32_unaligned(base + 16) << (32u - sh);
  return w >= 32u ? v : (v & ((1u << w) - 1u));
}

struct PhraseCand { uint32_t pos_lo, pos_hi, tf; };  // first delta of the doc in the term's stream (64-bit), its term frequency

// Two terms with slop: intersection_count_with_slop (phrase_scorer.rs:145-186) over the two position streams, left = the term the
// Intersection puts first (ascending size_hint).  A left position within `slop` of the right one matches; the left cursor first moves
// to the LAST left position that is not beyond the right one ("there could be a better match"), then both advance.
__device__ __noinline__ uint32_t phrase_count_slop2(const PosDesc* __restrict__ pdescs, const PhraseAux* __restrict__ aux, const PhraseCand* __restrict__ cand,
                                                    uint32_t slop) {
  const PosDesc& DL = pdescs[aux[0].pos_id];
  const PosDesc& DR = pdescs[aux[1].pos_id];
  unsigned long long gl = ((unsigned long long)cand[0].pos_hi << 32) | cand[0].pos_lo, gr = ((unsigned long long)cand[1].pos_hi << 32) | cand[1].pos_lo;
  uint32_t ll = cand[0].tf, rl = cand[1].tf;  // positions not read yet
  if (ll == 0u || rl == 0u) return 0u;
  uint32_t lv = aux[0].offset + pos_delta(DL, gl), rv = aux[1].offset + pos_delta(DR, gr);
  ++gl; --ll; ++gr; --rl;
  uint32_t count = 0;
  for (;;) {
    const uint32_t distance = lv > rv ? lv - rv : rv - lv;
    if (distance <= slop) {
      while (ll) {  // there could be a better match
        const uint32_t nxt = lv + pos_delta(DL, gl);
        if (nxt > rv) break;
        lv = nxt; ++gl; --ll;
      }
      ++count;
      if (ll == 0u || rl == 0u) return count;
      lv += pos_delta(DL, gl); ++gl; --ll;
      rv += pos_delta(DR, gr); ++gr; --rl;
    } else if (lv < rv) {
      if (ll == 0u) return count;
      lv += pos_delta(DL, gl); ++gl; --ll;
    } else {
      if (rl == 0u) return count;
      rv += pos_delta(DR, gr); ++gr; --rl;
    }
  }
}

// |intersection of the terms' shifted position sets| for one doc (k-way leap-frog; the sets are strictly ascending).
__device__ __noinline__ uint32_t phrase_count(const PosDesc* __restrict__ pdescs, const PhraseAux* __restrict__ aux, const PhraseCand* __restrict__ cand,
                                              uint32_t n_terms) {
  if (aux[0].slop != 0u) return phrase_count_slop2(pdescs, aux, cand, aux[0].slop);  // (the planner admits slop for two terms only)
  unsigned long long g[kPhraseMaxTerms];
  uint32_t left[kPhraseMaxTerms], pos[kPhraseMaxTerms];
  for (uint32_t t = 0; t < n_terms; ++t) {
    g[t] = ((unsigned long long)cand[t].pos_hi << 32) | cand[t].pos_lo;
    left[t] = cand[t].tf;
    if (left[t] == 0u) return 0u;
    pos[t] = aux[t].offset + pos_delta(pdescs[aux[t].pos_id], g[t]);
    ++g[t]; --left[t];
  }
  uint32_t count = 0;
  for (;;) {
    uint32_t target = 0;
    for (uint32_t t = 0; t < n_terms; ++t) target = max(target, pos[t]);
    bool all = true;
    for (uint32_t t = 0; t < n_terms; ++t) {
      while (pos[t] < target) {
        if (left[t] == 0u) return count;
        pos[t] += pos_delta(pdescs[aux[t].pos_id], g[t]);
        ++g[t]; --left[t];
      }
      all = all && pos[t] == target;
    }
    if (!all) continue;
    ++count;
    for (uint32_t t = 0; t < n_terms; ++t) {
      if (left[t] == 0u) return count;
      pos[t] += pos_delta(pdescs[aux[t].pos_id], g[t]);
      ++g[t]; --left[t];
    }
  }
}

// exclusive prefix sums of a decoded block's 128 term frequencies (4 per lane) -> where each doc's positions start inside the block
__device__ __forceinline__ void tf_prefix(const uint32_t (&tf)[4], uint32_t lane, uint32_t (&pre)[4]) {
  const uint32_t s = tf[0] + tf[1] + tf[2] + tf[3];
  const uint32_t incl = warp_incl_scan(s, lane);
  pre[0] = incl - s; pre[1] = pre[0] + tf[0]; pre[2] = pre[1] + tf[1]; pre[3] = pre[2] + tf[2];
}

// dynamic shared memory: per warp [128][ct] PhraseCand (ct = most terms of a phrase in the batch) + [128 docs | 128 tfs | 128 prefixes]
// of a decoded secondary block (reused for the compacted matches)
__host__ __device__ constexpr size_t phrase_smem_bytes(uint32_t ct) { return kPhraseWarps * (128u * ct * sizeof(PhraseCand) + 384u * 4u); }

__global__ void __launch_bounds__(kPhraseThreads, 5) k_phrase(const BatchParams P, const PosDesc* __restrict__ pdescs, const PhraseAux* __restrict__ aux_all,
                                                           uint32_t unit_base, uint32_t ct) {
  extern __shared__ __align__(16) unsigned char s_dyn[];
  __shared__ CtaTopK s_top;
  const Unit U = P.units[unit_base + blockIdx.x];
  const QSeg S = P.qsegs[U.qseg];
  const DQuery Q = P.queries[S.query];
  QState* qs = P.qstate + S.query;
  const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
  PhraseCand* cands = reinterpret_cast<PhraseCand*>(s_dyn) + (size_t)warp * 128u * ct;
  uint32_t* dec = reinterpret_cast<uint32_t*>(s_dyn + kPhraseWarps * 128u * ct * sizeof(PhraseCand)) + warp * 384u;
  const PhraseAux* aux = aux_all + S.lists_base;
  const QList ql0 = P.qlists[S.lists_base];
  const ListDesc L0 = P.lists[ql0.list_id];
  const Scorer sc = make_scorer(P, ql0);  // the phrase's single Bm25Weight
  if (threadIdx.x == 0) { s_top.count = 0; s_top.theta = (unsigned long long)qs->theta << 32; }
  __syncthreads();
  const TopK T{s_top.keys, &s_top.count, &s_top.theta, &s_top.scratch, (unsigned)kPhraseThreads};
  for (uint32_t r = U.begin; r < U.end; r += kPhraseWarps) {
    const uint32_t b = r + warp;
    if (b < U.end) {
      uint32_t doc[4], tf0[4], pre[4];
      decode_block(L0, b, lane, doc, tf0);
      uint32_t alive_m = 0;
#pragma unroll
      for (int i = 0; i < 4; ++i) alive_m |= (doc[i] < S.max_doc) ? (1u << i) : 0u;  // rejects tail padding
#pragma unroll
      for (int i = 0; i < 4; ++i) if (!((alive_m >> i) & 1u)) tf0[i] = 0u;
      tf_prefix(tf0, lane, pre);
      {
        const unsigned long long base = __ldg(pdescs[aux[0].pos_id].post_off + min(b, L0.n_blocks));
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const unsigned long long g = base + pre[i];
          cands[(lane * 4 + i) * ct] = PhraseCand{(uint32_t)g, (uint32_t)(g >> 32), tf0[i]};
        }
      }
      for (uint32_t s = 1; s < S.n_lists; ++s) {
        if (__ballot_sync(kFull, alive_m != 0) == 0) break;
        const QList qls = P.qlists[S.lists_base + s];
        const ListDesc Ls = P.lists[qls.list_id];
        const PosDesc& Ds = pdescs[aux[s].pos_id];
        uint32_t pending = alive_m;
        uint32_t cur = 0;
        for (;;) {
          const uint32_t c = (pending & 1u) ? doc[0] : (pending & 2u) ? doc[1] : (pending & 4u) ? doc[2] : (pending & 8u) ? doc[3] : 0xFFFFFFFFu;
          const uint32_t cmin = warp_min(c);
          if (cmin == 0xFFFFFFFFu) break;
          const uint32_t j = first_block_ge(Ls.last_doc, cur, Ls.n_total, cmin, lane);
          if (j >= Ls.n_total) { alive_m &= ~pending; pending = 0; break; }  // past the end of this list
          const uint32_t blk_last = __ldg(Ls.last_doc + j);
          uint32_t sd[4], st[4], sp[4];
          decode_block(Ls, j, lane, sd, st);
#pragma unroll
          for (int i = 0; i < 4; ++i) if (sd[i] >= S.max_doc) st[i] = 0u;
          tf_prefix(st, lane, sp);
          __syncwarp();
#pragma unroll
          for (int i = 0; i < 4; ++i) { dec[lane * 4 + i] = sd[i]; dec[128 + lane * 4 + i] = st[i]; dec[256 + lane * 4 + i] = sp[i]; }
          __syncwarp();
          const unsigned long long base = __ldg(Ds.post_off + min(j, Ls.n_blocks));
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            if (((pending >> i) & 1u) && doc[i] <= blk_last) {
              uint32_t lo = 0;
#pragma unroll
              for (uint32_t step = 64; step > 0; step >>= 1)
                if (dec[lo + step - 1] < doc[i]) lo += step;
              if (dec[lo] == doc[i]) {
                const unsigned long long g = base + dec[256 + lo];
                cands[(lane * 4 + i) * ct + s] = PhraseCand{(uint32_t)g, (uint32_t)(g >> 32), dec[128 + lo]};
              } else {
                alive_m &= ~(1u << i);
              }
              pending &= ~(1u << i);
            }
          }
          cur = j + 1;
        }
      }
      __syncwarp();
      // the docs that hold every term, compacted (a block of the rarest list keeps few of its 128 docs): their phrase counts, one
      // doc per lane -- the position deltas are read with dependent loads, so the fewer sequential rounds the better
      uint32_t n_match = 0;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const bool m = (alive_m >> i) & 1u;
        const unsigned bal = __ballot_sync(kFull, m);
        if (m) {
          const uint32_t at = n_match + (uint32_t)__popc(bal & lanemask_lt(lane));
          dec[at] = lane * 4u + (uint32_t)i;
          dec[128u + at] = doc[i];
        }
        n_match += (uint32_t)__popc(bal);
      }
      __syncwarp();
      const unsigned long long theta = *T.theta;
      for (uint32_t base = 0; base < n_match; base += 32u) {
        bool pass = false;
        unsigned long long key = 0;
        if (base + lane < n_match) {
          const uint32_t c = dec[base + lane], d = dec[128u + base + lane];
          const uint32_t cnt = phrase_count(pdescs, aux, cands + c * ct, S.n_lists);
          if (cnt) {
            const float score = bm25_score(sc, L0.fieldnorm, d, cnt);
            key = make_key(score, d);
            pass = key >= theta;
            if (pass && S.alive) pass = is_alive(S.alive, d);
          }
        }
        topk_push(T, pass, key, lane);
      }
    }
    topk_round_end(T, Q.k, &qs->theta);
  }
  topk_flush(T, Q, qs, P.cands, S.segment_ord);
}

}  // namespace tq
