// Host engine behind the C ABI of include/tantivy_b200.h: segment registry in HBM, per-term
// block-table cache, batch planning, kernel launches, result fetch.
//
// Replaces, for TermQuery / all-MUST / all-SHOULD BooleanQuery of TermQuerys collected by
// TopDocs::order_by_score, the reference's per-segment loop
//   Searcher::search_with_executor            src/core/searcher.rs:220-237
//   SortBySimilarityScore::collect_segment_top_k   src/collector/sort_key/sort_by_score.rs:35-66
//   Weight::for_each_pruning                  src/query/weight.rs:123-132
//   TopBySortKeyCollector::merge_fruits       src/collector/sort_key_top_collector.rs:54-60
// There is NO CPU fallback: without a CUDA device every entry point fails with TQ_ERR_CUDA.
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <string>
#include <unordered_map>
#include <vector>

#include "../../include/tantivy_b200.h"
#include "bm25_host.hpp"
#include "segment_writer.hpp"
#include "tq_tile.cuh"
#include "tq_phrase.cuh"

using namespace tq;

static constexpr size_t kOrDynSmem = kTileDocs * sizeof(float) + kTileDocs;  // score slots + fieldnorm bytes

namespace {

thread_local std::string g_err;

struct DevBuf {
  uint8_t* p = nullptr;
  size_t cap = 0;
  cudaError_t ensure(size_t n) {
    if (n <= cap) return cudaSuccess;
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
    const size_t want = std::max<size_t>(n + n / 4, 1 << 20);
    cudaError_t e = cudaMalloc(&p, want);
    if (e == cudaSuccess) cap = want;
    return e;
  }
  void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};
struct PinBuf {
  uint8_t* p = nullptr;
  size_t cap = 0;
  cudaError_t ensure(size_t n) {
    if (n <= cap) return cudaSuccess;
    if (p) cudaFreeHost(p);
    p = nullptr;
    cap = 0;
    const size_t want = std::max<size_t>(n + n / 4, 1 << 16);
    cudaError_t e = cudaMallocHost(&p, want);
    if (e == cudaSuccess) cap = want;
    return e;
  }
  void release() { if (p) cudaFreeHost(p); p = nullptr; cap = 0; }
};

struct ListKey {
  uint32_t segment_ord, field;
  uint64_t postings_start;  // bit 63: the table was built with term frequencies ignored (TQ_TERM_IGNORE_FREQ)
  bool operator==(const ListKey& o) const { return segment_ord == o.segment_ord && field == o.field && postings_start == o.postings_start; }
};
struct ListKeyHash {
  size_t operator()(const ListKey& k) const {
    uint64_t h = k.postings_start * 0x9E3779B97F4A7C15ull ^ ((uint64_t)k.segment_ord << 32 | k.field) * 0xC2B2AE3D27D4EB4Full;
    return (size_t)(h ^ (h >> 29));
  }
};

// Bump allocator over big cudaMalloc chunks for the per-term block tables (immutable, never freed
// individually; dropped with the context).
struct Arena {
  std::vector<uint8_t*> chunks;
  size_t chunk_size = 1u << 20, cap = 0, used = 0;  // chunks double up to 64 MiB: a small segment holds a small arena
  uint8_t* alloc(size_t n, cudaError_t* err) {
    n = (n + 255) & ~(size_t)255;
    if (chunks.empty() || used + n > cap) {
      const size_t sz = std::max(chunk_size, n);
      uint8_t* p = nullptr;
      *err = cudaMalloc(&p, sz);
      if (*err != cudaSuccess) return nullptr;
      chunks.push_back(p);
      cap = sz;
      used = 0;
      chunk_size = std::min<size_t>(chunk_size * 2, 64u << 20);
    }
    uint8_t* r = chunks.back() + used;
    used += n;
    *err = cudaSuccess;
    return r;
  }
  void release() { for (auto* c : chunks) cudaFree(c); chunks.clear(); used = 0; cap = 0; }
};

struct Segment {
  uint32_t segment_ord, field, max_doc;
  int record_option;
  uint8_t* d_idx = nullptr;  // field body incl. the 8-byte header, padded
  size_t idx_len = 0;
  uint8_t* d_fieldnorm = nullptr;
  uint8_t* d_alive = nullptr;
  uint32_t doc_lo = 0, doc_hi = 0;  // the docs this context evaluates (tq_segment_set_doc_range; [0, max_doc) by default)
  Arena arena;  // block tables + aligned block copies of this segment's posting lists; freed with the segment
  uint8_t* d_pos = nullptr;  // the field's `.pos` sub-file (phrase queries), padded
  size_t pos_len = 0;
  uint8_t* d_pos_pool = nullptr;  // position tables of this segment's terms, bump-allocated by k_build_pos_tables
  size_t pos_pool_cap = 0;        // (the first 8 bytes of the pool are the cursor)
};

uint32_t env_u32(const char* name, uint32_t def) {
  const char* v = getenv(name);
  if (!v || !*v) return def;
  return (uint32_t)strtoul(v, nullptr, 10);
}

}  // namespace

struct tq_ctx {
  int device = 0;
  std::mutex mu;  // guards segments, list cache, arena, batch pool, stats
  std::map<std::pair<uint32_t, uint32_t>, Segment> segments;
  ListDesc* d_lists = nullptr;
  uint32_t lists_cap = 0, n_lists = 0;
  std::unordered_map<ListKey, uint32_t, ListKeyHash> list_cache;
  std::vector<uint32_t> free_ids;  // list ids of unregistered segments (and of rolled-back builds), reused first
  PosDesc* d_pos_descs = nullptr;  // position tables (phrase queries), same life cycle as the block tables
  uint32_t pos_cap = 0, n_pos = 0;
  std::unordered_map<ListKey, uint32_t, ListKeyHash> pos_cache;  // (segment, field, positions_start) -> pos id
  std::vector<uint32_t> free_pos_ids;
  cudaStream_t build_stream = nullptr;
  PinBuf build_pin;
  DevBuf build_dev;
  std::vector<tq_batch*> pool;
  tq_stats stats{};
  uint32_t term_blocks_per_unit, and_blocks_per_unit;
  unsigned long long* d_counters = nullptr;  // [0..8) k_or_strip diagnostics (or_windows), [8..16) k_tile diagnostics
  uint32_t tile = 1, tile_scratch_mb = 24576, tile_sample_div = 16, tile_round_div1 = 8, tile_round_div2 = 2, tile_light_max = 96, tile_counters = 0;
  uint32_t tile_ops = 7;  // bit per TQ_OP_*: which query shapes the tile engine takes
  uint32_t tile_seg_cap_hook = 0;
  uint32_t tile_windows = 0;
  uint32_t phrase_side = 1;
  uint32_t tile_terms = 2;
  uint32_t tile_max_slots = kTileMaxSlots, tile_max_queries = kTileMaxQueries, tile_wide_queries = 256;
  uint64_t tile_smem_last = 0;
  uint32_t tile_cand_floor = 32768, tile_max_dens_x1000 = 0, tile_pcap_hook = 0, tile_big_min = 6, tile_units = 148 * 6;
};

constexpr int kTileRounds = 4;  // launches of k_tile per run: the sample launch + three exact ones

// Deep copy of a batch's queries (only kept when the tile engine runs them: an overflowing run is repeated on the per-query kernels).
struct OwnedQueries {
  std::vector<tq_query> q;
  std::vector<tq_term_seg> ts;
  std::vector<float> w, avg, cache;
  std::vector<uint8_t> flags;
  std::vector<tq_term_pos> tp;
  std::vector<uint32_t> toff;
};

struct tq_batch {
  struct Span { cudaEvent_t a = nullptr, b = nullptr; int kind = 0; };
  struct TileGroup {
    TileParams params{};
    uint32_t n_chunks = 0;
    uint32_t unit_base[kTileRounds] = {0, 0, 0, 0}, n_units[kTileRounds] = {0, 0, 0, 0};
    size_t smem = 0;
  };
  tq_ctx* ctx = nullptr;
  cudaStream_t stream = nullptr;
  cudaStream_t side = nullptr;             // k_phrase runs here, next to the tile engine's launches on `stream`
  cudaEvent_t ev_side0 = nullptr, ev_side1 = nullptr;
  bool side_pending = false;               // `stream` has not waited for ev_side1 yet
  cudaEvent_t ev_start = nullptr, ev_k0 = nullptr, ev_k1 = nullptr, ev_end = nullptr;
  std::vector<Span> spans;  // per-kind kernel times of the current run (events are created once and reused)
  size_t n_spans = 0;
  std::vector<TileGroup> groups;
  OwnedQueries owned;
  DevBuf tile_dev;  // pair arrays, tile indexes, samples, flags of the tile engine
  uint32_t* flags_pin = nullptr;  // [0] tile buffer overflow, [1] candidate region overflow (read back after the last phase)
  size_t tile_zero_off = 0, tile_zero_bytes = 0, tile_flags_off = 0;
  bool finalized = false, is_fallback = false, last_round_sampled = false;
  PinBuf pin;      // staged descriptors (H2D source)
  DevBuf dev;      // descriptors on device
  DevBuf scratch;  // qstate + candidates + results
  PinBuf res_pin;  // results (D2H target)
  BatchParams params{};
  size_t desc_bytes = 0;
  uint32_t nq = 0, kmax = 0;
  uint32_t n_units[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};  // term, and, or (window kernel), or (strip kernel), strip threshold rounds 1..3, phrase, mixed boolean
  uint32_t unit_base[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
  uint32_t phrase_ct = 2;                 // most terms of a phrase in the batch (k_phrase's candidate stride)
  const PhraseAux* phrase_aux = nullptr;  // device: per clause of the batch's phrase queries (parallel to qlists)
  uint32_t strip_cached_max = 0;
  size_t qinit_off = 0;
  int next_phase = 0;  // of the current run (0: none started)
  size_t qstate_off = 0, cands_off = 0, res_off = 0, res_bytes = 0, n_cands = 0;
  tq_stats stats{};
  bool ran = false;
};

#define TQ_CUDA(expr)                                                                         \
  do {                                                                                        \
    cudaError_t _e = (expr);                                                                  \
    if (_e != cudaSuccess) {                                                                  \
      g_err = std::string(#expr) + ": " + cudaGetErrorString(_e);                             \
      return TQ_ERR_CUDA;                                                                     \
    }                                                                                         \
  } while (0)

static int fail(int code, const std::string& msg) { g_err = msg; return code; }

// host twin of score_to_key (tq_device.cuh): order-preserving u32 image of a float
static uint32_t host_score_key(float f) {
  uint32_t u;
  memcpy(&u, &f, 4);
  return u ^ ((u >> 31) ? 0xFFFFFFFFu : 0x80000000u);
}

extern "C" {

const char* tq_last_error(tq_ctx*) { return g_err.c_str(); }

int tq_ctx_create(int device, tq_ctx** out) {
  if (!out) return fail(TQ_ERR_INVALID_ARGUMENT, "out is null");
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0)
    return fail(TQ_ERR_CUDA, std::string("no CUDA device: the B200 path has no CPU fallback (") + cudaGetErrorString(e) + ")");
  if (device < 0 || device >= n) return fail(TQ_ERR_INVALID_ARGUMENT, "bad device ordinal");
  TQ_CUDA(cudaSetDevice(device));
  auto* c = new tq_ctx();
  c->device = device;
  c->lists_cap = env_u32("TQ_MAX_LISTS", 1u << 20);
  c->term_blocks_per_unit = env_u32("TQ_TERM_BLOCKS_PER_UNIT", 512);
  c->and_blocks_per_unit = env_u32("TQ_AND_BLOCKS_PER_UNIT", 128);
  c->tile = env_u32("TQ_TILE", 1);                          // unions take the shared-decode tile engine (tq_tile.cuh); 0 = per-query kernels only
  c->tile_scratch_mb = env_u32("TQ_TILE_SCRATCH_MB", 24576);  // (doc, score) pairs one batch may materialise
  c->tile_sample_div = env_u32("TQ_TILE_SAMPLE_DIV", 16);    // share of the tiles in the sample launch (0/1: none)
  c->tile_round_div1 = env_u32("TQ_TILE_ROUND_DIV1", 8);     // the exact launches end at 1/8, 1/2 and all of a segment's tiles
  c->tile_round_div2 = env_u32("TQ_TILE_ROUND_DIV2", 2);
  c->tile_light_max = env_u32("TQ_TILE_LIGHT_MAX", 96);      // essential postings up to which a (query, tile) pair is evaluated posting by posting
  c->tile_counters = env_u32("TQ_TILE_COUNTERS", 0);         // diagnostics (tile_counters of tq_stats)
  c->tile_ops = env_u32("TQ_TILE_OPS", 7);                  // bit 0 term, 1 AND, 2 OR
  c->tile_cand_floor = env_u32("TQ_TILE_CAND_FLOOR", 32768);  // smallest candidate region of a tile query (test hook: tiny regions overflow)
  c->tile_max_dens_x1000 = env_u32("TQ_TILE_MAX_DENS_X1000", 0);  // test hook: cap on a group's pairs per 1000 docs (forces several groups)
  c->tile_pcap_hook = env_u32("TQ_TILE_PCAP", 0);            // test hook: tile buffer size (forces overflowing tiles)
  c->tile_seg_cap_hook = env_u32("TQ_TILE_SEG_CAP", 0);      // test hook: entries of the per-tile work list (forces extra routing rounds)
  c->tile_max_slots = std::min<uint32_t>(kTileMaxSlots, std::max<uint32_t>(64u, env_u32("TQ_TILE_MAX_SLOTS", kTileMaxSlots)));  // distinct lists of one segment per group (shared memory per CTA grows by 20 B per list)
  c->tile_max_queries = std::min<uint32_t>(kTileMaxQueries, std::max<uint32_t>(1u, env_u32("TQ_TILE_MAX_QUERIES", kTileMaxQueries)));  // queries of one segment per group
  c->tile_wide_queries = std::max<uint32_t>(1u, env_u32("TQ_TILE_WIDE_QUERIES", 256));  // ... for queries of more than 8 terms
  c->tile_terms = env_u32("TQ_TILE_TERMS", 2);               // single-term queries on the tile engine: 0 never, 1 always, 2 when the batch has multi-term queries
  c->phrase_side = env_u32("TQ_PHRASE_SIDE_STREAM", 1);      // k_phrase on the batch's second stream, next to the tile engine
  c->tile_windows = env_u32("TQ_TILE_WINDOWS", 0);           // warps with a window for the heavy pairs (0 = kTileExactWindows)
  c->tile_big_min = env_u32("TQ_TILE_BIG_MIN", 6);          // expected pairs per tile from which a list gets a tile index
  c->tile_units = env_u32("TQ_TILE_UNITS", 148u * 6u);       // CTAs an exact launch aims for
  cudaError_t err = cudaMalloc(&c->d_lists, (size_t)c->lists_cap * sizeof(ListDesc));
  if (err == cudaSuccess) err = cudaMemset(c->d_lists, 0, (size_t)c->lists_cap * sizeof(ListDesc));
  c->pos_cap = env_u32("TQ_MAX_POS_LISTS", 1u << 18);
  if (err == cudaSuccess) err = cudaMalloc(&c->d_pos_descs, (size_t)c->pos_cap * sizeof(PosDesc));
  if (err == cudaSuccess) err = cudaMemset(c->d_pos_descs, 0, (size_t)c->pos_cap * sizeof(PosDesc));
  if (err == cudaSuccess) err = cudaFuncSetAttribute(k_phrase, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)phrase_smem_bytes(kPhraseMaxTerms));
  if (err == cudaSuccess) err = cudaMalloc(&c->d_counters, 16 * sizeof(unsigned long long));
  if (err == cudaSuccess) err = cudaMemset(c->d_counters, 0, 16 * sizeof(unsigned long long));
  if (err == cudaSuccess) err = cudaStreamCreateWithFlags(&c->build_stream, cudaStreamNonBlocking);
  if (err == cudaSuccess) err = cudaFuncSetAttribute(k_or, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kOrDynSmem);
  if (err == cudaSuccess) err = cudaFuncSetAttribute(k_bool, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kBoolDynSmem);  // (+ its static smem: > 48 KB)
  if (err == cudaSuccess) err = cudaFuncSetAttribute(k_or_strip, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)strip_smem_bytes(kMaxCached));
  if (err == cudaSuccess) err = cudaFuncSetAttribute(k_tile, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
  if (err != cudaSuccess) { delete c; return fail(TQ_ERR_CUDA, cudaGetErrorString(err)); }
  *out = c;
  return TQ_OK;
}

void tq_batch_destroy_real(tq_batch* b) {
  if (!b) return;
  cudaSetDevice(b->ctx->device);
  if (b->stream) cudaStreamSynchronize(b->stream);
  if (b->side) { cudaStreamSynchronize(b->side); cudaStreamDestroy(b->side); }
  if (b->ev_side0) cudaEventDestroy(b->ev_side0);
  if (b->ev_side1) cudaEventDestroy(b->ev_side1);
  b->pin.release(); b->dev.release(); b->scratch.release(); b->res_pin.release(); b->tile_dev.release();
  if (b->flags_pin) cudaFreeHost(b->flags_pin);
  if (b->ev_start) cudaEventDestroy(b->ev_start);
  if (b->ev_k0) cudaEventDestroy(b->ev_k0);
  if (b->ev_k1) cudaEventDestroy(b->ev_k1);
  if (b->ev_end) cudaEventDestroy(b->ev_end);
  for (auto& sp : b->spans) { if (sp.a) cudaEventDestroy(sp.a); if (sp.b) cudaEventDestroy(sp.b); }
  if (b->stream) cudaStreamDestroy(b->stream);
  delete b;
}

void tq_ctx_destroy(tq_ctx* c) {
  if (!c) return;
  cudaSetDevice(c->device);
  cudaDeviceSynchronize();
  for (auto* b : c->pool) tq_batch_destroy_real(b);
  for (auto& kv : c->segments) {
    cudaFree(kv.second.d_idx); cudaFree(kv.second.d_fieldnorm); cudaFree(kv.second.d_alive);
    cudaFree(kv.second.d_pos); cudaFree(kv.second.d_pos_pool);
    kv.second.arena.release();
  }
  cudaFree(c->d_pos_descs);
  c->build_pin.release(); c->build_dev.release();
  if (c->build_stream) cudaStreamDestroy(c->build_stream);
  cudaFree(c->d_lists);
  cudaFree(c->d_counters);
  delete c;
}

int tq_get_stats(tq_ctx* c, tq_stats* out) {
  if (!c || !out) return fail(TQ_ERR_INVALID_ARGUMENT, "null");
  std::lock_guard<std::mutex> g(c->mu);
  *out = c->stats;
  out->lists_cached = c->list_cache.size();
  cudaSetDevice(c->device);
  unsigned long long h[16];
  if (cudaMemcpy(h, c->d_counters, sizeof(h), cudaMemcpyDeviceToHost) == cudaSuccess)
    for (int i = 0; i < 8; ++i) { out->or_windows[i] = h[i]; out->tile_counters[i] = h[8 + i]; }
  out->tile_counters[7] = c->tile_smem_last;
  return TQ_OK;
}

int tq_segment_register(tq_ctx* c, uint32_t segment_ord, uint32_t field, uint32_t max_doc, int record_option,
                        const uint8_t* idx_body, size_t idx_len, const uint8_t* fieldnorm, size_t fieldnorm_len,
                        const uint8_t* alive_bitset, size_t alive_len) {
  if (!c || !idx_body || idx_len < 8) return fail(TQ_ERR_INVALID_ARGUMENT, "idx_body must hold the 8-byte header");
  if (record_option < 0 || record_option > 2) return fail(TQ_ERR_INVALID_ARGUMENT, "record_option");
  if (max_doc >= TQ_TERMINATED) return fail(TQ_ERR_INVALID_ARGUMENT, "max_doc");
  if (fieldnorm && fieldnorm_len < max_doc) return fail(TQ_ERR_INVALID_ARGUMENT, "fieldnorm shorter than max_doc");
  if (alive_bitset && alive_len * 8 < max_doc) return fail(TQ_ERR_INVALID_ARGUMENT, "alive bitset shorter than max_doc");
  TQ_CUDA(cudaSetDevice(c->device));
  std::lock_guard<std::mutex> g(c->mu);
  if (c->segments.count({segment_ord, field})) return fail(TQ_ERR_INVALID_ARGUMENT, "segment/field already registered");
  Segment s;
  s.segment_ord = segment_ord; s.field = field; s.max_doc = max_doc; s.record_option = record_option; s.idx_len = idx_len;
  s.doc_lo = 0; s.doc_hi = max_doc;
  const size_t pad = 256;  // decode_block reads one word past a block; the aligned block copy of k_build_tables reads 64 + 8 bytes past the last block
  cudaError_t e = cudaMalloc(&s.d_idx, idx_len + pad);
  if (e == cudaSuccess) e = cudaMemset(s.d_idx + idx_len, 0, pad);
  if (e == cudaSuccess) e = cudaMemcpy(s.d_idx, idx_body, idx_len, cudaMemcpyHostToDevice);
  if (e == cudaSuccess && fieldnorm) {
    const size_t padded = ((size_t)max_doc + kTileDocs - 1) / kTileDocs * kTileDocs + kTileDocs;  // k_or stages whole windows
    e = cudaMalloc(&s.d_fieldnorm, padded);
    if (e == cudaSuccess) e = cudaMemset(s.d_fieldnorm, 0, padded);
    if (e == cudaSuccess) e = cudaMemcpy(s.d_fieldnorm, fieldnorm, max_doc, cudaMemcpyHostToDevice);
  }
  if (e == cudaSuccess && alive_bitset) {
    const size_t alive_padded = ((alive_len + 7) & ~(size_t)7) + 8;  // k_count reads whole 32-bit words
    e = cudaMalloc(&s.d_alive, alive_padded);
    if (e == cudaSuccess) e = cudaMemset(s.d_alive, 0, alive_padded);
    if (e == cudaSuccess) e = cudaMemcpy(s.d_alive, alive_bitset, alive_len, cudaMemcpyHostToDevice);
  }
  if (e != cudaSuccess) {  // nothing of a half-registered segment stays behind
    cudaFree(s.d_idx); cudaFree(s.d_fieldnorm); cudaFree(s.d_alive);
    return fail(TQ_ERR_CUDA, std::string("segment upload: ") + cudaGetErrorString(e));
  }
  c->segments[{segment_ord, field}] = s;
  return TQ_OK;
}

int tq_segment_register_positions(tq_ctx* c, uint32_t segment_ord, uint32_t field, const uint8_t* pos_body, size_t pos_len) {
  if (!c || (!pos_body && pos_len)) return fail(TQ_ERR_INVALID_ARGUMENT, "null");
  TQ_CUDA(cudaSetDevice(c->device));
  std::lock_guard<std::mutex> g(c->mu);
  auto it = c->segments.find({segment_ord, field});
  if (it == c->segments.end()) return fail(TQ_ERR_NOT_FOUND, "segment/field not registered");
  Segment& s = it->second;
  if (s.record_option != TQ_RECORD_FREQS_POSITIONS) return fail(TQ_ERR_INVALID_ARGUMENT, "the field was not indexed with positions");
  if (s.d_pos) return fail(TQ_ERR_INVALID_ARGUMENT, "positions already registered");
  // table pool: 4 bytes per position block (<= 1 per 16 bytes of `.pos`), 8 per posting block, 512 + slack per term that is
  // ever queried as part of a phrase
  const size_t pool = pos_len / 4 + s.idx_len / 8 + (4u << 20);
  uint8_t *d_pos = nullptr, *d_pool = nullptr;
  cudaError_t e = cudaMalloc(&d_pos, pos_len + 256);
  if (e == cudaSuccess) e = cudaMemset(d_pos + pos_len, 0, 256);
  if (e == cudaSuccess && pos_len) e = cudaMemcpy(d_pos, pos_body, pos_len, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMalloc(&d_pool, pool);
  if (e == cudaSuccess) e = cudaMemset(d_pool, 0, 64);
  if (e == cudaSuccess) {
    const unsigned long long first = 64;  // the cursor lives in the pool's first word; tables start behind it
    e = cudaMemcpy(d_pool, &first, 8, cudaMemcpyHostToDevice);
  }
  if (e != cudaSuccess) { cudaFree(d_pos); cudaFree(d_pool); return fail(TQ_ERR_CUDA, std::string("positions upload: ") + cudaGetErrorString(e)); }
  s.d_pos = d_pos; s.pos_len = pos_len; s.d_pos_pool = d_pool; s.pos_pool_cap = pool;
  return TQ_OK;
}

// A single huge segment split by doc-id range over several contexts / GPUs (SURVEY.md §8e: every block's first and last doc is known
// from the skip list, so any doc range of a segment is a unit of work of its own; the reference's own parallel axis stops at whole
// segments, src/core/executor.rs:60-100).  Correctness rests on the alive bitset (docs outside the range are "deleted" for this
// context: every kernel already honours it); the speed-up comes from the tile engine, which only visits the tiles of the range.
int tq_segment_set_doc_range(tq_ctx* c, uint32_t segment_ord, uint32_t field, uint32_t doc_lo, uint32_t doc_hi) {
  if (!c) return fail(TQ_ERR_INVALID_ARGUMENT, "null");
  TQ_CUDA(cudaSetDevice(c->device));
  std::lock_guard<std::mutex> g(c->mu);
  auto it = c->segments.find({segment_ord, field});
  if (it == c->segments.end()) return fail(TQ_ERR_NOT_FOUND, "segment/field not registered");
  Segment& s = it->second;
  if (doc_lo > doc_hi || doc_hi > s.max_doc) return fail(TQ_ERR_INVALID_ARGUMENT, "doc range must satisfy lo <= hi <= max_doc");
  if (doc_lo < s.doc_lo || doc_hi > s.doc_hi) return fail(TQ_ERR_INVALID_ARGUMENT, "a doc range can only be narrowed");
  TQ_CUDA(cudaDeviceSynchronize());  // batches in flight read the bitset
  const size_t nbytes = ((size_t)s.max_doc + 7) / 8;
  if (!s.d_alive) {
    for (auto& kv : c->list_cache)  // prepared batches keep the segment's (null) alive pointer: set the range before the first search
      if (kv.first.segment_ord == segment_ord && kv.first.field == field) return fail(TQ_ERR_INVALID_ARGUMENT, "set the doc range before the segment is searched");
    const size_t padded = ((nbytes + 7) & ~(size_t)7) + 8;
    uint8_t* d = nullptr;
    TQ_CUDA(cudaMalloc(&d, padded));
    cudaError_t e = cudaMemset(d, 0, padded);
    if (e == cudaSuccess && nbytes) e = cudaMemset(d, 0xFF, nbytes);
    if (e != cudaSuccess) { cudaFree(d); return fail(TQ_ERR_CUDA, cudaGetErrorString(e)); }
    s.d_alive = d;
  }
  auto patch = [&](size_t byte, uint8_t keep) -> cudaError_t {  // alive[byte] &= keep
    uint8_t v = 0;
    cudaError_t e = cudaMemcpy(&v, s.d_alive + byte, 1, cudaMemcpyDeviceToHost);
    v &= keep;
    if (e == cudaSuccess) e = cudaMemcpy(s.d_alive + byte, &v, 1, cudaMemcpyHostToDevice);
    return e;
  };
  auto clear_bits = [&](uint32_t a, uint32_t b) -> cudaError_t {  // docs [a, b) are not alive here (bit d & 7 of byte d >> 3)
    if (a >= b) return cudaSuccess;
    const size_t fb = ((size_t)a + 7) / 8, lb = (size_t)b / 8;  // whole bytes [fb, lb)
    cudaError_t e = cudaSuccess;
    if (fb > lb) return patch(a / 8, (uint8_t)~(((1u << (b - a)) - 1u) << (a & 7u)));  // a and b inside one byte
    if (lb > fb) e = cudaMemset(s.d_alive + fb, 0, lb - fb);
    if (e == cudaSuccess && (a & 7u)) e = patch(a / 8, (uint8_t)((1u << (a & 7u)) - 1u));
    if (e == cudaSuccess && (b & 7u)) e = patch(b / 8, (uint8_t)~((1u << (b & 7u)) - 1u));
    return e;
  };
  cudaError_t e = clear_bits(s.doc_lo, doc_lo);
  if (e == cudaSuccess) e = clear_bits(doc_hi, s.doc_hi);
  if (e != cudaSuccess) return fail(TQ_ERR_CUDA, std::string("doc range: ") + cudaGetErrorString(e));
  s.doc_lo = doc_lo; s.doc_hi = doc_hi;
  return TQ_OK;
}

int tq_segment_unregister(tq_ctx* c, uint32_t segment_ord, uint32_t field) {
  if (!c) return fail(TQ_ERR_INVALID_ARGUMENT, "null");
  cudaSetDevice(c->device);
  std::lock_guard<std::mutex> g(c->mu);
  auto it = c->segments.find({segment_ord, field});
  if (it == c->segments.end()) return fail(TQ_ERR_NOT_FOUND, "segment/field not registered");
  cudaDeviceSynchronize();
  cudaFree(it->second.d_idx); cudaFree(it->second.d_fieldnorm); cudaFree(it->second.d_alive);
  cudaFree(it->second.d_pos); cudaFree(it->second.d_pos_pool);
  for (auto pi = c->pos_cache.begin(); pi != c->pos_cache.end();)
    if (pi->first.segment_ord == segment_ord && pi->first.field == field) { c->free_pos_ids.push_back(pi->second); pi = c->pos_cache.erase(pi); } else ++pi;
  it->second.arena.release();  // the segment's block tables and aligned block copies go with it ...
  c->segments.erase(it);
  for (auto li = c->list_cache.begin(); li != c->list_cache.end();)
    if (li->first.segment_ord == segment_ord && li->first.field == field) { c->free_ids.push_back(li->second); li = c->list_cache.erase(li); } else ++li;  // ... and their ids are reused
  return TQ_OK;
}

}  // extern "C"

// ---- list cache ---------------------------------------------------------------------------------
namespace {

struct PendingBuild { BuildJob job; ListDesc desc; ListKey key; };

// Takes back every list that was scheduled but not built (an error path of the caller, or a corrupt list): its cache
// entry would otherwise hand an uninitialised ListDesc to the next query on the same term.  ctx->mu held.
void rollback_builds(tq_ctx* c, std::vector<PendingBuild>& pending) {
  for (auto& pb : pending) {
    auto it = c->list_cache.find(pb.key);
    if (it != c->list_cache.end() && it->second == pb.job.list_id) c->list_cache.erase(it);
    c->free_ids.push_back(pb.job.list_id);
  }
  pending.clear();
}
struct PendingScope {  // pending builds never outlive the call that scheduled them
  tq_ctx* c;
  std::vector<PendingBuild>& pending;
  ~PendingScope() { if (!pending.empty()) rollback_builds(c, pending); }
};

// Looks a posting list up in the cache or schedules its table build. ctx->mu held.
int get_list(tq_ctx* c, const tq_term_seg& ts, bool ignore_freq, std::vector<PendingBuild>& pending, uint32_t* list_id, const Segment** seg_out) {
  auto sit = c->segments.find({ts.segment_ord, ts.field});
  if (sit == c->segments.end()) return fail(TQ_ERR_NOT_FOUND, "term_seg names a segment/field that is not registered");
  Segment& seg = sit->second;
  *seg_out = &seg;
  if (ts.postings_end < ts.postings_start || ts.postings_end + 8 > seg.idx_len) return fail(TQ_ERR_INVALID_ARGUMENT, "postings range outside the field body");
  if (ts.postings_end - ts.postings_start > 0xFFFFFFFFull) return fail(TQ_ERR_UNSUPPORTED, "posting list larger than 4 GiB");
  ignore_freq = ignore_freq && seg.record_option != 0;
  const ListKey key{ts.segment_ord, ts.field, ts.postings_start | (ignore_freq ? 1ull << 63 : 0ull)};
  auto it = c->list_cache.find(key);
  if (it != c->list_cache.end()) { *list_id = it->second; return TQ_OK; }
  if (c->free_ids.empty() && c->n_lists >= c->lists_cap) return fail(TQ_ERR_OOM, "posting-list table cache full (TQ_MAX_LISTS)");
  const uint32_t n_blocks = ts.doc_freq / 128u, tail_n = ts.doc_freq % 128u;
  cudaError_t e;
  const size_t n_last = (size_t)n_blocks + 1, n_blk = (size_t)n_blocks + 1;
  const size_t len = (size_t)(ts.postings_end - ts.postings_start);
  const size_t copy_bytes = ((len + 15) & ~(size_t)15) + 128;  // 16-byte aligned copy of the blocks + slack
  uint8_t* mem = seg.arena.alloc(copy_bytes + n_last * 16 + n_last * 4 + 12 + n_blk * 8 + (size_t)tail_n * 8 + 16, &e);
  if (!mem) return fail(TQ_ERR_OOM, std::string("block table alloc: ") + cudaGetErrorString(e));
  PendingBuild pb;
  ListDesc& d = pb.desc;
  memset(&d, 0, sizeof(d));
  uint8_t* p = mem;
  d.blocks = p; p += copy_bytes;  // filled by k_build_tables
  d.tab4 = reinterpret_cast<const uint4*>(p); p += n_last * 16;
  d.blk = reinterpret_cast<const uint2*>(p); p += n_blk * 8;
  d.last_doc = reinterpret_cast<const uint32_t*>(p); p += n_last * 4;
  d.tail_docs = reinterpret_cast<const uint32_t*>(p); p += (size_t)tail_n * 4;
  d.tail_tfs = reinterpret_cast<const uint32_t*>(p);
  d.fieldnorm = seg.d_fieldnorm;
  d.n_blocks = n_blocks; d.tail_n = tail_n; d.n_total = n_blocks + (tail_n ? 1u : 0u); d.doc_freq = ts.doc_freq;
  d.build_status = 1;  // until k_build_tables says otherwise
  pb.job.bytes = seg.d_idx + 8 + ts.postings_start;
  pb.job.len = (uint32_t)(ts.postings_end - ts.postings_start);
  pb.job.doc_freq = ts.doc_freq;
  pb.job.record_option = (uint32_t)seg.record_option | (ignore_freq ? 0x100u : 0u);
  if (!c->free_ids.empty()) { pb.job.list_id = c->free_ids.back(); c->free_ids.pop_back(); }
  else pb.job.list_id = c->n_lists++;
  pb.key = key;
  *list_id = pb.job.list_id;
  c->list_cache.emplace(key, *list_id);  // later clauses of the same batch share the id; rolled back if the build does not happen
  pending.push_back(pb);
  return TQ_OK;
}

// Builds every pending table and waits for it (first use of a term only). ctx->mu held.  On any failure the
// pending lists are rolled back (no cache entry survives for a list that was not built).
int flush_builds(tq_ctx* c, std::vector<PendingBuild>& pending, uint64_t* built) {
  if (pending.empty()) return TQ_OK;
  const size_t n = pending.size();
  struct Fail { tq_ctx* c; std::vector<PendingBuild>& p; bool ok = false; ~Fail() { if (!ok) rollback_builds(c, p); } } guard{c, pending};
  TQ_CUDA(c->build_pin.ensure(n * (sizeof(ListDesc) + sizeof(BuildJob) + 4)));
  TQ_CUDA(c->build_dev.ensure(n * (sizeof(ListDesc) + sizeof(BuildJob) + 4)));
  ListDesc* hd = reinterpret_cast<ListDesc*>(c->build_pin.p);
  BuildJob* hj = reinterpret_cast<BuildJob*>(c->build_pin.p + n * sizeof(ListDesc));
  uint32_t* hs = reinterpret_cast<uint32_t*>(c->build_pin.p + n * (sizeof(ListDesc) + sizeof(BuildJob)));
  for (size_t i = 0; i < n; ++i) { hd[i] = pending[i].desc; hj[i] = pending[i].job; hs[i] = 1; }
  const ListDesc* dd = reinterpret_cast<const ListDesc*>(c->build_dev.p);
  const BuildJob* dj = reinterpret_cast<const BuildJob*>(c->build_dev.p + n * sizeof(ListDesc));
  uint32_t* ds = reinterpret_cast<uint32_t*>(c->build_dev.p + n * (sizeof(ListDesc) + sizeof(BuildJob)));
  TQ_CUDA(cudaMemcpyAsync(c->build_dev.p, c->build_pin.p, n * (sizeof(ListDesc) + sizeof(BuildJob) + 4), cudaMemcpyHostToDevice, c->build_stream));
  k_build_tables<<<(unsigned)n, kThreads, 0, c->build_stream>>>(dj, dd, c->d_lists, ds);
  TQ_CUDA(cudaGetLastError());
  TQ_CUDA(cudaMemcpyAsync(hs, ds, n * 4, cudaMemcpyDeviceToHost, c->build_stream));
  TQ_CUDA(cudaStreamSynchronize(c->build_stream));
  for (size_t i = 0; i < n; ++i)
    if (hs[i] != 0) return fail(TQ_ERR_CORRUPT, "posting list bytes are not a valid tantivy posting list");
  *built += n;
  guard.ok = true;
  pending.clear();
  return TQ_OK;
}

struct PendingPos { PosJob job; ListKey key; };

void rollback_pos(tq_ctx* c, std::vector<PendingPos>& pending) {
  for (auto& pp : pending) {
    auto it = c->pos_cache.find(pp.key);
    if (it != c->pos_cache.end() && it->second == pp.job.pos_id) c->pos_cache.erase(it);
    c->free_pos_ids.push_back(pp.job.pos_id);
  }
  pending.clear();
}
struct PendingPosScope {
  tq_ctx* c;
  std::vector<PendingPos>& pending;
  ~PendingPosScope() { if (!pending.empty()) rollback_pos(c, pending); }
};

// The position table of one (term, segment): cached, or scheduled.  ctx->mu held.
int get_pos(tq_ctx* c, const tq_term_seg& ts, const tq_term_pos& tp, std::vector<PendingPos>& pending, uint32_t* pos_id) {
  auto sit = c->segments.find({ts.segment_ord, ts.field});
  if (sit == c->segments.end()) return fail(TQ_ERR_NOT_FOUND, "term_seg names a segment/field that is not registered");
  Segment& seg = sit->second;
  if (!seg.d_pos) return fail(TQ_ERR_INVALID_ARGUMENT, "phrase query on a segment without registered positions (tq_segment_register_positions)");
  if (tp.positions_end < tp.positions_start || tp.positions_end > seg.pos_len) return fail(TQ_ERR_INVALID_ARGUMENT, "positions range outside the `.pos` body");
  if (tp.positions_end - tp.positions_start > 0xFFFFFFFFull) return fail(TQ_ERR_UNSUPPORTED, "position stream larger than 4 GiB");
  const ListKey key{ts.segment_ord, ts.field, tp.positions_start ^ (ts.postings_start << 1) ^ (1ull << 62)};
  auto it = c->pos_cache.find(key);
  if (it != c->pos_cache.end()) { *pos_id = it->second; return TQ_OK; }
  if (c->free_pos_ids.empty() && c->n_pos >= c->pos_cap) return fail(TQ_ERR_OOM, "position table cache full (TQ_MAX_POS_LISTS)");
  PendingPos pp;
  pp.job.pos_bytes = seg.d_pos + tp.positions_start;
  pp.job.pos_len = (uint32_t)(tp.positions_end - tp.positions_start);
  pp.job.list_bytes = seg.d_idx + 8 + ts.postings_start;
  pp.job.list_len = (uint32_t)(ts.postings_end - ts.postings_start);
  pp.job.doc_freq = ts.doc_freq;
  pp.job.pool = seg.d_pos_pool;
  pp.job.pool_cursor = reinterpret_cast<unsigned long long*>(seg.d_pos_pool);
  pp.job.pool_cap = seg.pos_pool_cap;
  if (!c->free_pos_ids.empty()) { pp.job.pos_id = c->free_pos_ids.back(); c->free_pos_ids.pop_back(); }
  else pp.job.pos_id = c->n_pos++;
  pp.key = key;
  *pos_id = pp.job.pos_id;
  c->pos_cache.emplace(key, *pos_id);
  pending.push_back(pp);
  return TQ_OK;
}

int flush_pos_builds(tq_ctx* c, std::vector<PendingPos>& pending) {
  if (pending.empty()) return TQ_OK;
  const size_t n = pending.size();
  struct Fail { tq_ctx* c; std::vector<PendingPos>& p; bool ok = false; ~Fail() { if (!ok) rollback_pos(c, p); } } guard{c, pending};
  TQ_CUDA(c->build_pin.ensure(n * (sizeof(PosJob) + 4)));
  TQ_CUDA(c->build_dev.ensure(n * (sizeof(PosJob) + 4)));
  PosJob* hj = reinterpret_cast<PosJob*>(c->build_pin.p);
  uint32_t* hs = reinterpret_cast<uint32_t*>(c->build_pin.p + n * sizeof(PosJob));
  for (size_t i = 0; i < n; ++i) { hj[i] = pending[i].job; hs[i] = 1; }
  uint32_t* ds = reinterpret_cast<uint32_t*>(c->build_dev.p + n * sizeof(PosJob));
  TQ_CUDA(cudaMemcpyAsync(c->build_dev.p, c->build_pin.p, n * (sizeof(PosJob) + 4), cudaMemcpyHostToDevice, c->build_stream));
  k_build_pos_tables<<<(unsigned)n, kThreads, 0, c->build_stream>>>(reinterpret_cast<const PosJob*>(c->build_dev.p), c->d_pos_descs, ds);
  TQ_CUDA(cudaGetLastError());
  TQ_CUDA(cudaMemcpyAsync(hs, ds, n * 4, cudaMemcpyDeviceToHost, c->build_stream));
  TQ_CUDA(cudaStreamSynchronize(c->build_stream));
  for (size_t i = 0; i < n; ++i) {
    if (hs[i] == 2) return fail(TQ_ERR_OOM, "the segment's position-table pool is exhausted");
    if (hs[i] != 0) return fail(TQ_ERR_CORRUPT, "position bytes are not a valid tantivy position stream");
  }
  guard.ok = true;
  pending.clear();
  return TQ_OK;
}

struct CacheKey {
  std::vector<float> table;
};

}  // namespace

// ---- batches ---------------------------------------------------------------------------------------
// Kernel time by kind: CUDA events recorded on the batch's stream around every launch (group of launches) of that kind.
enum SpanKind { SPAN_TERM = 0, SPAN_AND, SPAN_OR, SPAN_FINAL, SPAN_SCORE, SPAN_TILE, SPAN_THETA, SPAN_PHRASE, SPAN_BOOL, SPAN_KINDS };

static int span_begin(tq_batch* b, int kind, cudaStream_t on = nullptr) {
  if (b->n_spans == b->spans.size()) {
    tq_batch::Span s;
    s.kind = kind;
    if (cudaEventCreate(&s.a) != cudaSuccess || cudaEventCreate(&s.b) != cudaSuccess) return -1;
    b->spans.push_back(s);
  }
  tq_batch::Span& s = b->spans[b->n_spans];
  s.kind = kind;
  cudaEventRecord(s.a, on ? on : b->stream);
  return (int)b->n_spans++;
}
static void span_end(tq_batch* b, int idx, cudaStream_t on = nullptr) {
  if (idx >= 0) cudaEventRecord(b->spans[idx].b, on ? on : b->stream);
}

static void collect_times(tq_batch* b) {
  float ms = 0;
  if (cudaEventElapsedTime(&ms, b->ev_k0, b->ev_k1) == cudaSuccess) b->stats.kernel_ms = ms;
  float by_kind[SPAN_KINDS] = {0};
  for (size_t i = 0; i < b->n_spans; ++i)
    if (cudaEventElapsedTime(&ms, b->spans[i].a, b->spans[i].b) == cudaSuccess) by_kind[b->spans[i].kind] += ms;
  b->stats.term_ms = by_kind[SPAN_TERM];
  b->stats.and_ms = by_kind[SPAN_AND];
  b->stats.or_ms = by_kind[SPAN_OR];
  b->stats.final_ms = by_kind[SPAN_FINAL];
  b->stats.score_ms = by_kind[SPAN_SCORE];
  b->stats.tile_ms = by_kind[SPAN_TILE];
  b->stats.theta_ms = by_kind[SPAN_THETA];
  b->stats.phrase_ms = by_kind[SPAN_PHRASE];
  b->stats.bool_ms = by_kind[SPAN_BOOL];
}

static tq_batch* acquire_batch(tq_ctx* c) {
  {
    std::lock_guard<std::mutex> g(c->mu);
    if (!c->pool.empty()) { tq_batch* b = c->pool.back(); c->pool.pop_back(); return b; }
  }
  auto* b = new tq_batch();
  b->ctx = c;
  if (cudaStreamCreateWithFlags(&b->stream, cudaStreamNonBlocking) != cudaSuccess || cudaStreamCreateWithFlags(&b->side, cudaStreamNonBlocking) != cudaSuccess ||
      cudaEventCreateWithFlags(&b->ev_side0, cudaEventDisableTiming) != cudaSuccess || cudaEventCreateWithFlags(&b->ev_side1, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreate(&b->ev_start) != cudaSuccess ||
      cudaEventCreate(&b->ev_k0) != cudaSuccess || cudaEventCreate(&b->ev_k1) != cudaSuccess || cudaEventCreate(&b->ev_end) != cudaSuccess ||
      cudaMallocHost(&b->flags_pin, 64) != cudaSuccess) {
    tq_batch_destroy_real(b);
    return nullptr;
  }
  return b;
}

namespace {

// One (query, segment) of the plan: its clauses in evaluation order with their block tables resolved.
struct SegPlan {
  uint32_t segment_ord = 0;
  const Segment* seg = nullptr;
  struct Clause { uint32_t first; QList second; uint32_t range_len; };  // doc_freq, clause, bytes of its postings range
  std::vector<Clause> here;
  std::vector<uint32_t> term_idx;  // clause ordinals in arrival order (phrases: before `here` is sorted)
  std::vector<uint16_t> bool_words;  // TQ_OP_BOOL: [n_groups, need_should, n_should, n_not, (len, clauses..) per group, shoulds.., nots..],
                                     // clauses as indices into `here` (tile_admit turns them into slots)
  const uint8_t* fn0 = nullptr;
  bool uniform_fn = true, prunable = false;
};

// A group of queries that k_tile evaluates together (shared decode, see tq_tile.cuh), while it is being planned.
struct TileGroupBuild {
  struct SegB {
    uint32_t segment_ord = 0, max_doc = 0;
    uint32_t t_lo = 0, t_hi = 0;  // tiles that overlap the segment's doc range (tq_segment_set_doc_range)
    const uint8_t* alive = nullptr;
    std::vector<TSlot> slots;  // (TSlot::pad chains the slots of one list: several weights / tables of a list are rare)
    std::vector<TQuery> queries;
    std::vector<uint16_t> clauses;
    double dens = 0;  // sum of doc_freq / max_doc over the slots: expected pairs per doc
  };
  std::vector<SegB> segs;
  std::unordered_map<uint32_t, uint32_t> seg_of;  // segment_ord -> index in segs
  std::vector<uint32_t> slot_head;                 // list id -> first slot of that list in its segment (kNoSlot: none); a list lives in one segment
  uint32_t find_slot(const SegB& sb, const QList& ql) const {
    if (ql.list_id >= slot_head.size()) return kNoSlot;
    for (uint32_t s = slot_head[ql.list_id]; s != kNoSlot; s = sb.slots[s].pad) {
      const TSlot& sl = sb.slots[s];
      if (memcmp(&sl.weight, &ql.weight, 4) == 0 && sl.cache_idx == ql.cache_idx) return s;
    }
    return kNoSlot;
  }
  uint64_t pairs = 0;                              // elements of the pair arrays (doc_freq rounded up to 128 per slot)
  uint64_t list_bytes = 0;                         // postings-range bytes of the distinct lists
};

// BooleanWeight::complex_scorer for ONE segment (boolean_weight.rs:236-431), term leaves only: `here` = the clauses that have
// postings in the segment (term_idx / doc_freq / weight per entry).  Clauses without postings are EmptyScorers -- removed before
// anything is counted; an empty MUST group empties the query in this segment.  Writes
//   [n_groups, need_should, n_should, n_not, (len, entries..) per MUST group, SHOULD entries.., MUST_NOT entries..]
// (entries = indices into `here`; groups by ascending cost = Intersection's order, entries by descending weight = the union order)
// and returns 1; 0 when nothing can match in this segment; -1 on a bad Occur.
int bool_structure(const tq_query& q, const uint32_t* term_idx, const uint32_t* dfs, const float* ws, size_t n_here, std::vector<uint16_t>& words) {
  struct Grp { uint32_t id, first; uint64_t cost; std::vector<uint16_t> cl; };
  std::vector<Grp> groups;
  std::vector<uint16_t> shoulds, nots;
  for (uint32_t t = 0; t < q.n_terms; ++t) {  // declared MUST groups, present or not
    if (q.term_occur[t] > TQ_OCCUR_MUST_NOT) return -1;
    if (q.term_occur[t] != TQ_OCCUR_MUST) continue;
    const uint32_t id = q.term_group ? q.term_group[t] : 256u + t;
    bool known = false;
    for (auto& g : groups) known = known || g.id == id;
    if (!known) groups.push_back(Grp{id, t, 0, {}});
  }
  for (size_t a = 0; a < n_here; ++a) {
    const uint32_t t = term_idx[a];
    if (q.term_occur[t] == TQ_OCCUR_MUST) {
      const uint32_t id = q.term_group ? q.term_group[t] : 256u + t;
      for (auto& g : groups) if (g.id == id) { g.cl.push_back((uint16_t)a); g.cost += dfs[a]; }
    } else (q.term_occur[t] == TQ_OCCUR_SHOULD ? shoulds : nots).push_back((uint16_t)a);
  }
  for (auto& g : groups) if (g.cl.empty()) return 0;
  uint32_t m = q.min_should_match;
  if (m > shoulds.size()) return 0;
  if (m >= 2 && m == shoulds.size()) {  // as many as there are SHOULD clauses: they are MUST clauses (boolean_weight.rs:287-292)
    for (uint16_t a : shoulds) groups.push_back(Grp{512u + a, term_idx[a], dfs[a], {a}});
    shoulds.clear();
    m = 0;
  }
  if (groups.empty() && shoulds.empty()) return 0;
  const uint32_t need = m >= 1 ? m : (groups.empty() ? 1u : 0u);
  auto by_weight = [&](std::vector<uint16_t>& v) { std::stable_sort(v.begin(), v.end(), [&](uint16_t x, uint16_t y) { return ws[x] > ws[y]; }); };
  std::stable_sort(groups.begin(), groups.end(), [](const Grp& x, const Grp& y) { return x.cost < y.cost; });
  words.clear();
  words.push_back((uint16_t)groups.size());
  words.push_back((uint16_t)need);
  words.push_back((uint16_t)shoulds.size());
  words.push_back((uint16_t)nots.size());
  for (auto& g : groups) {
    by_weight(g.cl);
    words.push_back((uint16_t)g.cl.size());
    for (uint16_t a : g.cl) words.push_back(a);
  }
  by_weight(shoulds);
  for (uint16_t a : shoulds) words.push_back(a);
  for (uint16_t a : nots) words.push_back(a);
  return 1;
}

// Would the group still satisfy k_tile's limits with this query added?  Returns the number of NEW pair elements, or -1.
int64_t tile_admit_cost(const TileGroupBuild& g, const SegPlan* plans, size_t n_plans, uint32_t max_dens_x1000, uint32_t max_slots, uint32_t max_queries) {
  int64_t new_pairs = 0;
  for (size_t pi = 0; pi < n_plans; ++pi) {
    const SegPlan& sp = plans[pi];
    auto it = g.seg_of.find(sp.segment_ord);
    const TileGroupBuild::SegB* sb = it == g.seg_of.end() ? nullptr : &g.segs[it->second];
    if (sb && sb->queries.size() + 1 > max_queries) return -1;
    size_t n_slots = sb ? sb->slots.size() : 0;
    double dens = sb ? sb->dens : 0.0;
    for (auto& h : sp.here) {
      const bool found = sb && g.find_slot(*sb, h.second) != kNoSlot;
      if (!found) {
        ++n_slots;
        dens += (double)h.first / std::max(1u, sp.seg->max_doc);
        new_pairs += ((int64_t)h.first + 127) / 128 * 128;
      }
    }
    if (n_slots > max_slots) return -1;
    if (dens * kTile * 1.5 + 256.0 > (double)kTileMaxPairs || (max_dens_x1000 && dens * 1000.0 > max_dens_x1000)) return -1;
  }
  return new_pairs;
}

// Cheap sufficient test (every clause counted as a new list): most queries pass it and skip the exact cost.
bool tile_admit_surely_fits(const TileGroupBuild& g, const SegPlan* plans, size_t n_plans, uint32_t max_dens_x1000, uint32_t max_slots, uint32_t max_queries) {
  for (size_t pi = 0; pi < n_plans; ++pi) {
    const SegPlan& sp = plans[pi];
    auto it = g.seg_of.find(sp.segment_ord);
    const TileGroupBuild::SegB* sb = it == g.seg_of.end() ? nullptr : &g.segs[it->second];
    if (sb && sb->queries.size() + 1 > max_queries) return false;
    double dens = sb ? sb->dens : 0.0;
    for (auto& h : sp.here) dens += (double)h.first / std::max(1u, sp.seg->max_doc);
    if ((sb ? sb->slots.size() : 0) + sp.here.size() > max_slots) return false;
    if (dens * kTile * 1.5 + 256.0 > (double)kTileMaxPairs || (max_dens_x1000 && dens * 1000.0 > max_dens_x1000)) return false;
  }
  return true;
}

// Adds the query to the group; returns the number of new pair elements it brought.
uint64_t tile_admit(TileGroupBuild& g, uint32_t query, int op, const SegPlan* plans, size_t n_plans) {
  const uint64_t pairs_before = g.pairs;
  for (size_t pi = 0; pi < n_plans; ++pi) {
    const SegPlan& sp = plans[pi];
    auto it = g.seg_of.find(sp.segment_ord);
    if (it == g.seg_of.end()) {
      it = g.seg_of.emplace(sp.segment_ord, (uint32_t)g.segs.size()).first;
      g.segs.emplace_back();
      g.segs.back().segment_ord = sp.segment_ord;
      g.segs.back().max_doc = sp.seg->max_doc;
      g.segs.back().alive = sp.seg->d_alive;
      g.segs.back().t_lo = sp.seg->doc_lo / kTile;
      g.segs.back().t_hi = (uint32_t)(((uint64_t)sp.seg->doc_hi + kTile - 1) / kTile);
    }
    TileGroupBuild::SegB& sb = g.segs[it->second];
    TQuery tq;
    tq.query = query;
    tq.clause_base = (uint32_t)sb.clauses.size();
    tq.n_clauses = (uint16_t)(op == TQ_OP_BOOL ? sp.bool_words.size() : sp.here.size());
    tq.op = (uint8_t)(op == TQ_OP_BOOL ? kTileOpBool : op);
    tq.flags = sp.prunable ? 1u : 0u;
    uint16_t slot_of_here[TQ_MAX_TERMS];
    size_t hi_idx = 0;
    for (auto& h : sp.here) {
      uint32_t slot = g.find_slot(sb, h.second);
      if (slot == kNoSlot) {
        slot = (uint32_t)sb.slots.size();
        TSlot sl{};
        sl.list_id = h.second.list_id; sl.weight = h.second.weight; sl.cache_idx = h.second.cache_idx; sl.doc_freq = h.first;
        sl.big = kNoSlot;
        if (h.second.list_id >= g.slot_head.size()) g.slot_head.resize((size_t)h.second.list_id + 1024, kNoSlot);
        sl.pad = g.slot_head[h.second.list_id];  // chain
        g.slot_head[h.second.list_id] = slot;
        sb.slots.push_back(sl);
        sb.dens += (double)h.first / std::max(1u, sp.seg->max_doc);
        g.pairs += ((uint64_t)h.first + 127) / 128 * 128;
        g.list_bytes += h.range_len;
      }
      slot_of_here[hi_idx++] = (uint16_t)slot;
      if (op != TQ_OP_BOOL) sb.clauses.push_back((uint16_t)slot);
    }
    if (op == TQ_OP_BOOL) {  // the structure words stay, the clause indices become slots
      const std::vector<uint16_t>& w = sp.bool_words;
      size_t x = 0;
      for (int k = 0; k < 4; ++k) sb.clauses.push_back(w[x++]);
      for (uint32_t g = 0; g < w[0]; ++g) {
        const uint16_t len = w[x++];
        sb.clauses.push_back(len);
        for (uint16_t e = 0; e < len; ++e) sb.clauses.push_back(slot_of_here[w[x++]]);
      }
      while (x < w.size()) sb.clauses.push_back(slot_of_here[w[x++]]);
    }
    sb.queries.push_back(tq);
  }
  return g.pairs - pairs_before;
}

}  // namespace

static int batch_prepare_impl(tq_ctx* c, const tq_query* queries, size_t nq, bool force_legacy, tq_batch** out);

extern "C" {

void tq_batch_destroy(tq_batch* b) {
  if (!b) return;
  cudaSetDevice(b->ctx->device);
  cudaStreamSynchronize(b->stream);
  b->next_phase = 0;
  b->ran = false;
  std::lock_guard<std::mutex> g(b->ctx->mu);
  b->ctx->pool.push_back(b);  // buffers are recycled by the next batch
}

int tq_batch_prepare(tq_ctx* c, const tq_query* queries, size_t nq, tq_batch** out) {
  return batch_prepare_impl(c, queries, nq, false, out);
}

}  // extern "C"

static int batch_prepare_impl(tq_ctx* c, const tq_query* queries, size_t nq, bool force_legacy, tq_batch** out) {
  if (!c || !out || (!queries && nq)) return fail(TQ_ERR_INVALID_ARGUMENT, "null");
  TQ_CUDA(cudaSetDevice(c->device));
  tq_batch* b = acquire_batch(c);
  if (!b) return fail(TQ_ERR_CUDA, "stream/event creation failed");
  struct Guard { tq_batch* b; bool ok = false; ~Guard() { if (!ok) tq_batch_destroy(b); } } guard{b};
  b->ran = false;
  b->finalized = false;
  b->next_phase = 0;  // a recycled batch may have been abandoned in the middle of a phased run
  b->nq = (uint32_t)nq;
  b->stats = tq_stats{};
  b->n_spans = 0;
  b->groups.clear();
  b->owned = OwnedQueries{};
  b->is_fallback = force_legacy;

  std::vector<QList> qlists;
  std::vector<QSeg> qsegs;
  std::vector<Unit> units[9];
  std::vector<PhraseAux> qaux;  // parallel to qlists once a phrase query shows up
  std::vector<PendingPos> pending_pos;
  std::vector<DQuery> dq(nq);
  std::vector<float> caches;  // n_caches * 256
  std::unordered_map<uint32_t, uint32_t> cache_by_avg;  // avg bits -> cache idx
  std::vector<PendingBuild> pending;
  uint64_t built = 0, alg_bytes = 0, postings = 0, op_bytes[3] = {0, 0, 0};
  uint32_t kmax = 1;
  size_t n_cands = 0;
  std::vector<int> qseg_op;
  std::vector<uint32_t> qseg_total;
  uint32_t n_qsegs_op[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};  // (query, segment) pairs per unit class
  std::vector<char> qseg_sample;  // strip pairs that get a threshold sample pass (MaxScore can then skip their dense clauses)
  uint32_t strip_cached_max = 0, phrase_ct = 2;
  std::vector<TileGroupBuild> tgroups;
  std::vector<size_t> q_cands(nq, 0);
  const bool tile_on = c->tile != 0 && !force_legacy;
  const uint64_t tile_pair_budget = (uint64_t)c->tile_scratch_mb * (1u << 20) / 8u;
  uint64_t tile_pairs_total = 0;
  // Single-term queries ride along on the tile engine when the batch has multi-term queries whose decoded lists they share
  // (mixed workload: 32.6 K q/s against 28.6 K with them on k_term); a batch of nothing but single-term queries has nothing to
  // share and streams its lists through k_term (configs[0]: 1.39 M q/s against 0.49 M).  TQ_TILE_TERMS: 0 never, 1 always, 2 this rule.
  bool terms_on_tile = c->tile_terms == 1;
  if (c->tile_terms >= 2)
    for (size_t qi = 0; qi < nq && !terms_on_tile; ++qi)
      terms_on_tile = queries[qi].n_terms >= 2 && queries[qi].op != TQ_OP_PHRASE;
  {
    std::lock_guard<std::mutex> g(c->mu);
    PendingScope pending_scope{c, pending};  // an early error return leaves no half-built list in the cache
    PendingPosScope pending_pos_scope{c, pending_pos};
    std::vector<const tq_term_seg*> order;
    std::vector<SegPlan> plans;  // reused from query to query (n_plans live entries)
    uint32_t last_avg_bits = 0, last_avg_idx = 0xFFFFFFFFu;
    for (size_t qi = 0; qi < nq; ++qi) {
      const tq_query& q = queries[qi];
      if (q.k == 0 || q.k > TQ_MAX_K) return fail(TQ_ERR_INVALID_ARGUMENT, "k must be in 1..TQ_MAX_K");
      if (q.n_terms == 0 || q.n_terms > TQ_MAX_TERMS) return fail(TQ_ERR_INVALID_ARGUMENT, "n_terms must be in 1..TQ_MAX_TERMS");
      const bool is_bool = q.op == TQ_OP_BOOL;
      if (is_bool && !q.term_occur) return fail(TQ_ERR_INVALID_ARGUMENT, "TQ_OP_BOOL needs term_occur");
      if (q.op != TQ_OP_TERM && q.op != TQ_OP_AND && q.op != TQ_OP_OR && q.op != TQ_OP_PHRASE && !is_bool) return fail(TQ_ERR_INVALID_ARGUMENT, "op");
      if (q.op == TQ_OP_TERM && q.n_terms != 1) return fail(TQ_ERR_INVALID_ARGUMENT, "TQ_OP_TERM takes one term");
      if (!q.weight || (!q.avg_fieldnorm && !q.tf_cache) || (!q.term_segs && q.n_term_segs)) return fail(TQ_ERR_INVALID_ARGUMENT, "query arrays");
      const bool is_phrase = q.op == TQ_OP_PHRASE;
      if (is_phrase) {
        if (q.n_terms < 2 || q.n_terms > TQ_MAX_PHRASE_TERMS) return fail(TQ_ERR_UNSUPPORTED, "a phrase takes 2..TQ_MAX_PHRASE_TERMS terms on the device path");
        // slop: two terms take intersection_count_with_slop on the device; three and more carry per-position slops through
        // growing buffers (intersection_count_with_carrying_slop, phrase_scorer.rs:236-345) and stay on the reference's CPU path
        if (q.slop != 0 && q.n_terms != 2) return fail(TQ_ERR_UNSUPPORTED, "phrase slop with more than two terms stays on the reference's CPU path");
        if ((!q.term_pos && q.n_term_segs) || !q.term_offset) return fail(TQ_ERR_INVALID_ARGUMENT, "a phrase needs term_pos and term_offset");
      }
      kmax = std::max(kmax, q.k);
      alg_bytes += 12ull * q.k;
      op_bytes[is_phrase ? TQ_OP_AND : (is_bool ? TQ_OP_OR : (q.n_terms == 1 ? TQ_OP_TERM : q.op))] += 12ull * q.k;
      // tf-norm tables of this query's clauses
      uint32_t cache_idx[TQ_MAX_TERMS];
      for (uint32_t t = 0; t < q.n_terms; ++t) {
        if (q.tf_cache) {
          cache_idx[t] = (uint32_t)(caches.size() / 256);
          caches.insert(caches.end(), q.tf_cache + 256 * (size_t)t, q.tf_cache + 256 * (size_t)(t + 1));
        } else {
          uint32_t bits;
          memcpy(&bits, &q.avg_fieldnorm[t], 4);
          if (bits == last_avg_bits && last_avg_idx != 0xFFFFFFFFu) { cache_idx[t] = last_avg_idx; continue; }  // (nearly always the same field)
          auto it = cache_by_avg.find(bits);
          if (it == cache_by_avg.end()) {
            float tab[256];
            bm25_tf_cache(q.avg_fieldnorm[t], tab);
            it = cache_by_avg.emplace(bits, (uint32_t)(caches.size() / 256)).first;
            caches.insert(caches.end(), tab, tab + 256);
          }
          cache_idx[t] = it->second;
          last_avg_bits = bits; last_avg_idx = it->second;
        }
      }
      // effective shape: an AND / OR of one clause is that clause (boolean_weight.rs:57-68, block_wand_union.rs:154-157)
      const int op = is_phrase ? TQ_OP_PHRASE : (is_bool ? TQ_OP_BOOL : (q.n_terms == 1 ? TQ_OP_TERM : q.op));
      dq[qi].k = q.k;
      dq[qi].op = (uint32_t)op;
      // group the (clause, segment) lists by segment
      order.clear();
      for (uint32_t i = 0; i < q.n_term_segs; ++i) {
        if (q.term_segs[i].term_idx >= q.n_terms) return fail(TQ_ERR_INVALID_ARGUMENT, "term_idx out of range");
        if (q.term_segs[i].doc_freq) order.push_back(&q.term_segs[i]);
      }
      std::stable_sort(order.begin(), order.end(), [](const tq_term_seg* a, const tq_term_seg* b) {
        return a->segment_ord != b->segment_ord ? a->segment_ord < b->segment_ord : a->term_idx < b->term_idx;
      });
      size_t n_plans = 0;
      uint64_t q_postings = 0;
      for (size_t i = 0; i < order.size();) {
        size_t j = i;
        while (j < order.size() && order[j]->segment_ord == order[i]->segment_ord) ++j;
        // lists of this (query, segment), clause order
        const size_t n_here = j - i;
        bool dup = false;
        for (size_t a = i + 1; a < j; ++a) dup |= order[a]->term_idx == order[a - 1]->term_idx;
        if (dup) return fail(TQ_ERR_INVALID_ARGUMENT, "duplicate (term_idx, segment_ord)");
        if ((op == TQ_OP_AND || op == TQ_OP_PHRASE) && n_here != q.n_terms) { i = j; continue; }  // a clause is absent: empty intersection
        if (n_plans == plans.size()) plans.emplace_back();
        SegPlan& sp = plans[n_plans++];
        sp.here.clear();
        sp.term_idx.clear();
        sp.uniform_fn = true;
        sp.segment_ord = order[i]->segment_ord;
        for (size_t a = i; a < j; ++a) {
          uint32_t id;
          int rc = get_list(c, *order[a], q.term_flags && (q.term_flags[order[a]->term_idx] & TQ_TERM_IGNORE_FREQ), pending, &id, &sp.seg);
          if (rc != TQ_OK) return rc;
          if (a == i) sp.fn0 = sp.seg->d_fieldnorm; else sp.uniform_fn &= (sp.seg->d_fieldnorm == sp.fn0);
          QList ql{id, q.weight[is_phrase ? 0 : order[a]->term_idx], cache_idx[is_phrase ? 0 : order[a]->term_idx], 0};
          if (is_phrase) {  // the clause's position table; QList.pad carries its id to the aux array below
            if (sp.seg->record_option != TQ_RECORD_FREQS_POSITIONS) return fail(TQ_ERR_INVALID_ARGUMENT, "phrase query on a field without positions");
            rc = get_pos(c, *order[a], q.term_pos[order[a] - q.term_segs], pending_pos, &ql.pad);
            if (rc != TQ_OK) return rc;
          }
          sp.here.push_back(SegPlan::Clause{order[a]->doc_freq, ql, (uint32_t)(order[a]->postings_end - order[a]->postings_start)});
          sp.term_idx.push_back(order[a]->term_idx);
          alg_bytes += (order[a]->postings_end - order[a]->postings_start) + order[a]->doc_freq;
          op_bytes[is_phrase ? TQ_OP_AND : (is_bool ? TQ_OP_OR : op)] += (order[a]->postings_end - order[a]->postings_start) + order[a]->doc_freq;
          postings += order[a]->doc_freq;
          q_postings += order[a]->doc_freq;
        }
        if (op == TQ_OP_PHRASE) {
          // PhraseScorer keeps its terms by ascending size_hint (intersection.rs:40-52); every clause carries
          // (max_offset - its offset), the shift that lines the terms' positions up (phrase_scorer.rs:349-398)
          uint32_t max_offset = 0;
          for (uint32_t t = 0; t < q.n_terms; ++t) max_offset = std::max(max_offset, q.term_offset[t]);
          for (size_t a = 0; a < sp.here.size(); ++a) sp.here[a].range_len = max_offset - q.term_offset[sp.term_idx[a]];  // (range_len is free here)
          std::stable_sort(sp.here.begin(), sp.here.end(), [](const SegPlan::Clause& a, const SegPlan::Clause& b) { return a.first < b.first; });
        }
        if (op == TQ_OP_AND)  // leader = rarest, then ascending doc_freq; stable (block_wand_intersection.rs:27)
          std::stable_sort(sp.here.begin(), sp.here.end(), [](const SegPlan::Clause& a, const SegPlan::Clause& b) { return a.first < b.first; });
        if (op == TQ_OP_OR)
          // Canonical union order = descending Bm25Weight.weight, ties in clause order (the reference's own order is
          // data dependent, block_wand_union.rs:205-208): the f32 sum is taken in this order, and the clauses with the
          // smallest score bounds form a suffix, which is what the MaxScore splits of k_tile / k_or_strip need.
          std::stable_sort(sp.here.begin(), sp.here.end(), [](const SegPlan::Clause& a, const SegPlan::Clause& b) { return a.second.weight > b.second.weight; });
        sp.prunable = true;
        for (auto& h : sp.here) sp.prunable = sp.prunable && std::isfinite(h.second.weight) && h.second.weight >= 0.0f;
        if (op == TQ_OP_BOOL) {
          uint32_t dfs[TQ_MAX_TERMS];
          float ws[TQ_MAX_TERMS];
          for (size_t a = 0; a < sp.here.size(); ++a) { dfs[a] = sp.here[a].first; ws[a] = sp.here[a].second.weight; }
          const int st = bool_structure(q, sp.term_idx.data(), dfs, ws, sp.here.size(), sp.bool_words);
          if (st < 0) return fail(TQ_ERR_INVALID_ARGUMENT, "term_occur");
          if (st == 0) { --n_plans; i = j; continue; }
        }
        i = j;
      }
      // ---- route: the shared-decode tile engine, or the per-query kernels -------------------------------------------------
      bool on_tile = false;
      if (tile_on && (((c->tile_ops >> op) & 1u) || op == TQ_OP_BOOL) && (op != TQ_OP_TERM || terms_on_tile) && n_plans) {
        if (tgroups.empty()) tgroups.emplace_back();
        // wide unions: every query brings its clause words, work-list entries and (mostly distinct) lists into the CTA's shared
        // memory; smaller groups keep two CTAs per SM (configs[4]: 1.64 s -> 1.05 s per 512 20-term queries on 500M docs)
        const uint32_t max_q = q.n_terms > 8 ? std::min(c->tile_max_queries, c->tile_wide_queries) : c->tile_max_queries;
        bool fits = tile_admit_surely_fits(tgroups.back(), plans.data(), n_plans, c->tile_max_dens_x1000, c->tile_max_slots, max_q);
        if (!fits) fits = tile_admit_cost(tgroups.back(), plans.data(), n_plans, c->tile_max_dens_x1000, c->tile_max_slots, max_q) >= 0;
        if (!fits && !tgroups.back().segs.empty()) {  // the current group is full: open the next one
          TileGroupBuild fresh;
          if (tile_admit_cost(fresh, plans.data(), n_plans, c->tile_max_dens_x1000, c->tile_max_slots, max_q) >= 0) { tgroups.emplace_back(); fits = true; }
        }
        if (fits && tile_pairs_total + q_postings + 128ull * n_plans * q.n_terms <= tile_pair_budget) {
          tile_pairs_total += tile_admit(tgroups.back(), (uint32_t)qi, op, plans.data(), n_plans);
          on_tile = true;
          // every doc at or above the running threshold is handed over: the sample launch and the k_theta passes keep that
          // near k; a query that still overflows sends the batch to the per-query kernels (flags[1])
          const uint32_t cand_floor = c->tile_cand_floor;  // (test hook: tiny regions overflow)
          q_cands[qi] += (size_t)std::min<uint64_t>(q_postings, std::max<uint64_t>((cand_floor >= 8192 ? 128ull : 1ull) * q.k, cand_floor));
        }
      }
      if (on_tile) continue;
      for (size_t pi = 0; pi < n_plans; ++pi) {
        SegPlan& sp = plans[pi];
        auto& here = sp.here;
        QSeg qs;
        memset(&qs, 0, sizeof(qs));
        qs.query = (uint32_t)qi;
        qs.lists_base = (uint32_t)qlists.size();
        qs.segment_ord = sp.segment_ord;
        qs.max_doc = sp.seg->max_doc;
        qs.alive = sp.seg->d_alive;
        qs.fieldnorm = sp.uniform_fn ? sp.fn0 : nullptr;
        const bool prunable = sp.prunable && op != TQ_OP_TERM;
        qs.flags = (sp.uniform_fn ? 1u : 0u) | (prunable ? 2u : 0u);
        int unit_class = op == TQ_OP_PHRASE ? 7 : (op == TQ_OP_BOOL ? 8 : op);
        if (op == TQ_OP_PHRASE) {
          if (qaux.size() < qlists.size()) qaux.resize(qlists.size(), PhraseAux{0, 0, 0});
          for (auto& h : here) { qaux.push_back(PhraseAux{h.second.pad, h.range_len, q.slop}); h.second.pad = 0; }
          phrase_ct = std::max<uint32_t>(phrase_ct, (uint32_t)here.size());
        }
        if (op == TQ_OP_OR && q.k <= kStripMaxK && here.size() <= kStripMaxLists) {
          // strip kernel: clauses with less than one block per kWin-doc window keep their current block decoded in shared memory
          uint32_t n_thin = 0;
          auto is_thin = [&](uint32_t df) { return (uint64_t)df * (kWin / 128u) < (uint64_t)qs.max_doc; };
          for (auto& h : here) if (is_thin(h.first)) ++n_thin;
          if (n_thin <= kMaxCached) {
            uint32_t slot = 0;
            for (auto& h : here) h.second.pad = is_thin(h.first) ? (1u | (slot++ << 1)) : 0u;
            strip_cached_max = std::max(strip_cached_max, n_thin);
            unit_class = 3;
          }
        }
        if (op == TQ_OP_BOOL) {
          // k_bool: the clauses in bool_structure's order (groups, SHOULD, MUST_NOT); QList.pad = role | group << 2,
          // QSeg.flags [8:16) = number of groups, [16:24) = SHOULD clauses needed
          const std::vector<uint16_t>& w = sp.bool_words;
          const uint32_t ng = w[0], ns = w[2], nn = w[3];
          qs.flags |= (ng << 8) | ((uint32_t)w[1] << 16);
          size_t x = 4;
          for (uint32_t g = 0; g < ng; ++g) {
            const uint16_t len = w[x++];
            for (uint16_t e = 0; e < len; ++e) { QList ql = here[w[x++]].second; ql.pad = kBoolMust | (g << 2); qlists.push_back(ql); }
          }
          for (uint32_t e = 0; e < ns; ++e) { QList ql = here[w[x++]].second; ql.pad = kBoolShould; qlists.push_back(ql); }
          for (uint32_t e = 0; e < nn; ++e) { QList ql = here[w[x++]].second; ql.pad = kBoolNot; qlists.push_back(ql); }
        } else {
          for (auto& h : here) qlists.push_back(h.second);
        }
        qs.n_lists = (uint32_t)here.size();
        const uint32_t lead_total = here[0].first / 128u + ((here[0].first % 128u) ? 1u : 0u);
        qsegs.push_back(qs);
        qseg_op.push_back(unit_class);
        {
          bool any_thick = false;
          for (auto& h : here) any_thick = any_thick || (uint64_t)h.first * std::max(kStripNeDiv, kStripNeDiv2) >= qs.max_doc;
          qseg_sample.push_back(unit_class == 3 && prunable && any_thick);
        }
        qseg_total.push_back(unit_class == 3 ? (qs.max_doc + kWin - 1) / kWin
                                             : (op == TQ_OP_OR ? (qs.max_doc + kTileDocs - 1) / kTileDocs
                                                               : (op == TQ_OP_BOOL ? (qs.max_doc + kBoolDocs - 1) / kBoolDocs : lead_total)));
        ++n_qsegs_op[unit_class == 7 ? TQ_OP_AND : unit_class];
      }
    }
    // Work units. A unit is one CTA's share of a (query, segment). With few (query, segment) pairs in the
    // batch every pair is cut into many units (latency); with many, units grow so that a CTA's local
    // top-k threshold gets tight and few candidates reach k_final (throughput).
    const uint32_t target_units = env_u32("TQ_TARGET_UNITS", 148u * 4u * 32u);
    for (size_t s = 0; s < qsegs.size(); ++s) {
      const int op = qseg_op[s];
      const uint32_t total = qseg_total[s];
      // (k_bool: 32 of its 4096-doc windows, the docs of k_or's 16 8192-doc windows)
      const uint32_t min_per = op == TQ_OP_TERM ? c->term_blocks_per_unit
                                                : ((op == TQ_OP_AND || op == 7) ? c->and_blocks_per_unit : (op == 3 ? kStripWarps * 64u : (op == 8 ? 32u : 16u)));
      const uint32_t n_same = n_qsegs_op[op == 7 ? TQ_OP_AND : op];
      const uint32_t want_units = std::max<uint32_t>(1u, (target_units + n_same - 1) / n_same);
      const uint32_t per = std::max<uint32_t>(min_per, (total + want_units - 1) / want_units);
      const uint32_t k = dq[qsegs[s].query].k;
      // Threshold rounds: the first 1/32, then up to 1/8 and up to 1/2 of a strip pair's windows run in launches of their
      // own; the exact k-th best score over all windows run so far of the query (k_theta) then seeds the threshold of the
      // next launch, whose MaxScore split drops the dense clauses from the first window on.  Nothing is scored twice.
      uint32_t first = 0;
      if (op == 3 && qseg_sample[s] && total >= 8u * 32u) {
        const uint32_t cut1 = std::max<uint32_t>(kStripWarps, total / 32u);
        const uint32_t cut2 = std::max(cut1, total / 8u);
        const uint32_t cut3 = std::max(cut2, total / 2u);
        const uint32_t cuts[4] = {0, cut1, cut2, cut3};
        for (int r = 0; r < 3; ++r)  // round r covers [cuts[r], cuts[r+1]); a k_theta pass follows each round
          for (uint32_t b0 = cuts[r]; b0 < cuts[r + 1]; b0 += per) {
            units[4 + r].push_back(Unit{(uint32_t)s, b0, std::min(cuts[r + 1], b0 + per), 0});
            q_cands[qsegs[s].query] += (size_t)kStripWarps * k;
          }
        first = cut3;
      }
      for (uint32_t b0 = first; b0 < total; b0 += per) {
        units[op].push_back(Unit{(uint32_t)s, b0, std::min(total, b0 + per), 0});
        q_cands[qsegs[s].query] += op == 3 ? (size_t)kStripWarps * k : 2u * (size_t)k;  // what one unit may hand over
      }
    }
    for (size_t qi = 0; qi < nq; ++qi) {
      dq[qi].cand_base = (uint32_t)n_cands;
      dq[qi].cand_cap = (uint32_t)q_cands[qi];
      n_cands += q_cands[qi];
      if (n_cands > 0xFFFFFFF0ull) return fail(TQ_ERR_UNSUPPORTED, "batch too large: split it");
    }
    int rc = flush_builds(c, pending, &built);
    if (rc == TQ_OK) rc = flush_pos_builds(c, pending_pos);
    if (rc != TQ_OK) return rc;
  }
  if (caches.empty()) caches.resize(256, 0.0f);
  if (!qaux.empty() && qaux.size() < qlists.size()) qaux.resize(qlists.size(), PhraseAux{0, 0, 0});

  // ---- tile groups: slot order, pair bases, score chunks, tile ranges of the launches -------------------------------------------
  struct GroupStage {
    std::vector<TSlot> slots;
    std::vector<TSeg> segs;
    std::vector<TQuery> queries;
    std::vector<uint16_t> clauses;
    std::vector<TUnit> units[kTileRounds];
    std::vector<SChunk> chunks;
    uint32_t max_slots = 1, p_cap = 1024, max_big = 1, max_queries = 1, max_clause_words = 0, max_clauses = 1;
    size_t tix_words = 0;
  };
  std::vector<GroupStage> gstage(tgroups.size());
  uint64_t pair_cursor = 0;
  size_t tix_total_words = 0;
  uint64_t tile_postings = 0, tile_units = 0;
  const uint32_t big_min = c->tile_big_min;
  for (size_t gi = 0; gi < tgroups.size(); ++gi) {
    TileGroupBuild& tg = tgroups[gi];
    GroupStage& gs = gstage[gi];
    double dens_max = 0;
    uint64_t tiles_total = 0;
    uint32_t kmax_g = 1;
    for (auto& sb : tg.segs) {
      // dense lists first (they get a tile index and whole warps), then the rest; clause ordinals follow the permutation
      std::vector<uint32_t> perm(sb.slots.size());
      for (uint32_t i = 0; i < perm.size(); ++i) perm[i] = i;
      auto is_big = [&](const TSlot& sl) { return (uint64_t)sl.doc_freq * kTile >= (uint64_t)big_min * std::max(1u, sb.max_doc); };
      // (by descending doc_freq throughout: the threads of a warp that stage sparse slots then see similar lists)
      std::stable_sort(perm.begin(), perm.end(), [&](uint32_t a, uint32_t b2) { return sb.slots[a].doc_freq > sb.slots[b2].doc_freq; });
      std::vector<uint32_t> new_of(perm.size());
      for (uint32_t i = 0; i < perm.size(); ++i) new_of[perm[i]] = i;
      TSeg G{};
      G.slot_base = (uint32_t)gs.slots.size();
      G.n_slots = (uint32_t)sb.slots.size();
      G.query_base = (uint32_t)gs.queries.size();
      G.n_queries = (uint32_t)sb.queries.size();
      G.max_doc = sb.max_doc;
      G.segment_ord = sb.segment_ord;
      G.n_tiles = (sb.max_doc + kTile - 1) / kTile;
      G.alive = sb.alive;
      uint32_t n_big = 0;
      for (uint32_t i = 0; i < perm.size(); ++i) {
        TSlot sl = sb.slots[perm[i]];
        sl.tseg = (uint32_t)gs.segs.size();
        sl.pair_base = (uint32_t)pair_cursor;
        if (is_big(sl) && n_big < kTileMaxBig) sl.big = n_big++;  // (the densest ones: the order above is by descending doc_freq)
        const uint32_t n_total = sl.doc_freq / 128u + ((sl.doc_freq % 128u) ? 1u : 0u);
        for (uint32_t b0 = 0; b0 < n_total; b0 += 64u) gs.chunks.push_back(SChunk{(uint32_t)gs.slots.size(), b0, std::min(n_total, b0 + 64u)});
        pair_cursor += ((uint64_t)sl.doc_freq + 127) / 128 * 128;
        tile_postings += sl.doc_freq;
        gs.slots.push_back(sl);
      }
      G.n_big = n_big;
      G.tix = reinterpret_cast<uint32_t*>(tix_total_words + gs.tix_words);  // offset for now, rebased below
      gs.tix_words += (size_t)(G.n_tiles + 1) * n_big;
      const uint32_t clause_shift = (uint32_t)gs.clauses.size();
      G.clause_base = clause_shift;
      G.n_clause_words = (uint32_t)sb.clauses.size();
      gs.max_clause_words = std::max(gs.max_clause_words, G.n_clause_words);
      for (auto& tq : sb.queries) {
        TQuery t2 = tq;
        t2.clause_base += clause_shift;
        gs.queries.push_back(t2);
        kmax_g = std::max(kmax_g, dq[tq.query].k);
        gs.max_clauses = std::max<uint32_t>(gs.max_clauses, tq.n_clauses);
      }
      {  // clause slots follow the permutation (the structure words of TQ_OP_BOOL queries do not)
        const size_t c0 = gs.clauses.size();
        for (uint16_t cl : sb.clauses) gs.clauses.push_back(cl);
        for (auto& tq : sb.queries) {
          uint16_t* w = gs.clauses.data() + c0 + tq.clause_base;
          if (tq.op != kTileOpBool) { for (uint32_t e = 0; e < tq.n_clauses; ++e) w[e] = (uint16_t)new_of[w[e]]; continue; }
          size_t x = 4;
          for (uint32_t g = 0; g < w[0]; ++g) { const uint16_t len = w[x++]; for (uint16_t e = 0; e < len; ++e, ++x) w[x] = (uint16_t)new_of[w[x]]; }
          for (; x < tq.n_clauses; ++x) w[x] = (uint16_t)new_of[w[x]];
        }
      }
      gs.max_slots = std::max(gs.max_slots, G.n_slots);
      gs.max_big = std::max(gs.max_big, G.n_big);
      gs.max_queries = std::max(gs.max_queries, G.n_queries);
      dens_max = std::max(dens_max, sb.dens);
      tiles_total += sb.t_hi - sb.t_lo;
      gs.segs.push_back(G);
    }
    tix_total_words += gs.tix_words;
    gs.p_cap = (uint32_t)std::min<double>(kTileMaxPairs, std::max(1024.0, dens_max * kTile * 1.25 + 192.0));
    gs.p_cap = (gs.p_cap + 63u) & ~63u;
    if (c->tile_pcap_hook) gs.p_cap = c->tile_pcap_hook;  // (test hook: overflowing tiles)
    // Launches: [0] samples scores on a spread of short tile runs, [1..3] are exact and cover every tile once.
    const uint32_t target = std::max(1u, c->tile_units);
    const uint32_t sample_div = std::max<uint32_t>(2u, c->tile_sample_div);
    // enough sampled tiles for k_max samples to exist: each (query, tile) contributes at most kSamplePerTile
    const uint64_t want_sample_tiles = std::min<uint64_t>(tiles_total / 2, std::max<uint64_t>(tiles_total / sample_div, (uint64_t)kmax_g / 2u + 8u));
    for (uint32_t si = 0; si < gs.segs.size(); ++si) {
      const uint32_t tl = tg.segs[si].t_lo, nt = tg.segs[si].t_hi - tl;  // (the whole segment unless a doc range was set)
      if (nt == 0) continue;
      if (c->tile_sample_div > 1 && nt >= 8 && tiles_total) {
        // short runs of tiles spread over the segment, one CTA each (a sample launch has few tiles: it needs them all in flight)
        const uint32_t seg_sample = (uint32_t)std::max<uint64_t>(1, want_sample_tiles * nt / tiles_total);
        const uint32_t len = std::max<uint32_t>(1u, std::min<uint32_t>(4u, seg_sample / 64u + 1u));
        const uint32_t runs = std::max<uint32_t>(1u, seg_sample / len);
        for (uint32_t r = 0; r < runs; ++r) {
          const uint32_t start = (uint32_t)(((uint64_t)(2 * r + 1) * nt) / (2 * runs));
          const uint32_t t0 = std::min(start, nt - 1), t1 = std::min(nt, t0 + len);
          gs.units[0].push_back(TUnit{si, tl + t0, tl + t1, 0});
        }
      }
      const uint32_t cut1 = nt >= 16 ? nt / std::max(2u, c->tile_round_div1) : 0, cut2 = nt >= 16 ? std::max(cut1, nt / std::max(2u, c->tile_round_div2)) : 0;
      const uint32_t cuts[4] = {0, cut1, cut2, nt};
      for (int r = 0; r < 3; ++r) {
        const uint32_t span = cuts[r + 1] - cuts[r];
        if (!span) continue;
        // this launch's share of the target, by its share of all tiles; at least 8 tiles per unit (cursor start-up)
        const uint64_t round_tiles_all = std::max<uint64_t>(1, (uint64_t)tiles_total * span / nt);
        const uint32_t per = (uint32_t)std::max<uint64_t>(tiles_total >= 16ull * target ? 8 : 2, (round_tiles_all + target - 1) / target);
        for (uint32_t t0 = cuts[r]; t0 < cuts[r + 1]; t0 += per) gs.units[1 + r].push_back(TUnit{si, tl + t0, tl + std::min(cuts[r + 1], t0 + per), 0});
      }
    }
    for (int r = 0; r < kTileRounds; ++r) tile_units += gs.units[r].size();
  }
  if (pair_cursor > 0xFFFFFF00ull) return fail(TQ_ERR_UNSUPPORTED, "batch decodes more than 4G postings: split it");

  // ---- stage descriptors -------------------------------------------------------------------------
  auto align = [](size_t x) { return (x + 255) & ~(size_t)255; };
  size_t off = 0;
  const size_t o_caches = off; off = align(off + caches.size() * 4);
  const size_t n_caches = caches.size() / 256;
  const size_t o_tftab = off; off = align(off + n_caches * kTfRows * 256 * 4);  // device only (built by k_build_tf_tables)
  const size_t o_qlists = off; off = align(off + qlists.size() * sizeof(QList));
  const size_t o_qsegs = off; off = align(off + qsegs.size() * sizeof(QSeg));
  const size_t o_qaux = off; off = align(off + qaux.size() * sizeof(PhraseAux));
  const size_t n_units_total = units[0].size() + units[1].size() + units[2].size() + units[3].size() + units[4].size() + units[5].size() + units[6].size() + units[7].size() +
                               units[8].size();
  b->strip_cached_max = strip_cached_max;
  b->phrase_ct = std::min<uint32_t>(phrase_ct, kPhraseMaxTerms);
  const size_t o_units = off; off = align(off + n_units_total * sizeof(Unit));
  const size_t o_queries = off; off = align(off + dq.size() * sizeof(DQuery));
  const size_t o_qinit = off; off = align(off + std::max<size_t>(nq, 1) * sizeof(QState));  // per-run initial state (threshold keys)
  struct GroupOff { size_t slots, segs, queries, clauses, units, chunks; };
  std::vector<GroupOff> goff(gstage.size());
  for (size_t gi = 0; gi < gstage.size(); ++gi) {
    GroupStage& gs = gstage[gi];
    size_t nu = 0;
    for (int r = 0; r < kTileRounds; ++r) nu += gs.units[r].size();
    goff[gi].slots = off; off = align(off + gs.slots.size() * sizeof(TSlot));
    goff[gi].segs = off; off = align(off + gs.segs.size() * sizeof(TSeg));
    goff[gi].queries = off; off = align(off + gs.queries.size() * sizeof(TQuery));
    goff[gi].clauses = off; off = align(off + gs.clauses.size() * 2);
    goff[gi].units = off; off = align(off + nu * sizeof(TUnit));
    goff[gi].chunks = off; off = align(off + gs.chunks.size() * sizeof(SChunk));
  }
  b->desc_bytes = off;
  TQ_CUDA(b->pin.ensure(off + 256));
  TQ_CUDA(b->dev.ensure(off + 256));

  // ---- tile scratch: pair arrays | tile indexes | samples | sample counts | flags + counters --------------------------------
  uint32_t sample_cap = 0;
  size_t to_docs = 0, to_scores = 0, to_tix = 0, to_samples = 0, to_scount = 0, to_flags = 0, tile_bytes = 0;
  if (!gstage.empty()) {
    uint64_t sample_units_tiles = 0;
    for (auto& gs : gstage) for (auto& u : gs.units[0]) sample_units_tiles += u.t1 - u.t0;
    sample_cap = (uint32_t)std::min<uint64_t>(1u << 16, std::max<uint64_t>(256, sample_units_tiles * 8u));
    size_t so2 = 0;
    to_docs = so2; so2 = align(so2 + (size_t)pair_cursor * 4);
    to_scores = so2; so2 = align(so2 + (size_t)pair_cursor * 4);
    to_tix = so2; so2 = align(so2 + tix_total_words * 4);
    to_samples = so2; so2 = align(so2 + (size_t)std::max<size_t>(nq, 1) * sample_cap * 4);
    to_scount = so2; so2 = align(so2 + std::max<size_t>(nq, 1) * 4);
    to_flags = so2; so2 = align(so2 + 256);
    tile_bytes = so2;
    TQ_CUDA(b->tile_dev.ensure(tile_bytes));
  }
  b->tile_zero_off = to_scount;
  b->tile_zero_bytes = gstage.empty() ? 0 : (to_flags + 256 - to_scount);
  b->tile_flags_off = to_flags;

  memcpy(b->pin.p + o_caches, caches.data(), caches.size() * 4);
  if (!qlists.empty()) memcpy(b->pin.p + o_qlists, qlists.data(), qlists.size() * sizeof(QList));
  if (!qsegs.empty()) memcpy(b->pin.p + o_qsegs, qsegs.data(), qsegs.size() * sizeof(QSeg));
  if (!qaux.empty()) memcpy(b->pin.p + o_qaux, qaux.data(), qaux.size() * sizeof(PhraseAux));
  b->phrase_aux = reinterpret_cast<const PhraseAux*>(b->dev.p + o_qaux);
  {
    Unit* u = reinterpret_cast<Unit*>(b->pin.p + o_units);
    uint32_t base = 0;
    for (int op = 0; op < 9; ++op) {
      b->unit_base[op] = base;
      b->n_units[op] = (uint32_t)units[op].size();
      if (!units[op].empty()) memcpy(u + base, units[op].data(), units[op].size() * sizeof(Unit));
      base += (uint32_t)units[op].size();
    }
  }
  if (!dq.empty()) memcpy(b->pin.p + o_queries, dq.data(), dq.size() * sizeof(DQuery));
  {
    QState* qi0 = reinterpret_cast<QState*>(b->pin.p + o_qinit);
    for (size_t qi = 0; qi < std::max<size_t>(nq, 1); ++qi) {
      qi0[qi].theta = 0; qi0[qi].cand_count = 0;
      if (qi < nq && (queries[qi].flags & TQ_QUERY_HAS_THRESHOLD)) {
        // collect score > threshold: the smallest accepted key is the next representable score (NaN: no filter)
        float th = queries[qi].threshold;
        if (th == 0.0f) th = 0.0f;  // -0.0 and +0.0 are the same threshold
        if (th == th) { const uint32_t key = host_score_key(th); qi0[qi].theta = key == 0xFFFFFFFFu ? key : key + 1u; }
      }
    }
  }
  b->qinit_off = o_qinit;
  size_t tix_cursor = 0;
  for (size_t gi = 0; gi < gstage.size(); ++gi) {
    GroupStage& gs = gstage[gi];
    tq_batch::TileGroup run;
    for (auto& G : gs.segs) {  // rebase the tile-index offsets to device addresses
      const size_t w = reinterpret_cast<size_t>(G.tix);
      G.tix = reinterpret_cast<uint32_t*>(b->tile_dev.p + to_tix) + w;
    }
    tix_cursor += gs.tix_words;
    if (!gs.slots.empty()) memcpy(b->pin.p + goff[gi].slots, gs.slots.data(), gs.slots.size() * sizeof(TSlot));
    if (!gs.segs.empty()) memcpy(b->pin.p + goff[gi].segs, gs.segs.data(), gs.segs.size() * sizeof(TSeg));
    if (!gs.queries.empty()) memcpy(b->pin.p + goff[gi].queries, gs.queries.data(), gs.queries.size() * sizeof(TQuery));
    if (!gs.clauses.empty()) memcpy(b->pin.p + goff[gi].clauses, gs.clauses.data(), gs.clauses.size() * 2);
    {
      TUnit* u = reinterpret_cast<TUnit*>(b->pin.p + goff[gi].units);
      uint32_t base = 0;
      for (int r = 0; r < kTileRounds; ++r) {
        run.unit_base[r] = base;
        run.n_units[r] = (uint32_t)gs.units[r].size();
        if (!gs.units[r].empty()) memcpy(u + base, gs.units[r].data(), gs.units[r].size() * sizeof(TUnit));
        base += (uint32_t)gs.units[r].size();
      }
    }
    if (!gs.chunks.empty()) memcpy(b->pin.p + goff[gi].chunks, gs.chunks.data(), gs.chunks.size() * sizeof(SChunk));
    run.n_chunks = (uint32_t)gs.chunks.size();
    TileParams& TP = run.params;
    TP.slots = reinterpret_cast<const TSlot*>(b->dev.p + goff[gi].slots);
    TP.segs = reinterpret_cast<const TSeg*>(b->dev.p + goff[gi].segs);
    TP.queries = reinterpret_cast<const TQuery*>(b->dev.p + goff[gi].queries);
    TP.clauses = reinterpret_cast<const uint16_t*>(b->dev.p + goff[gi].clauses);
    TP.units = reinterpret_cast<const TUnit*>(b->dev.p + goff[gi].units);
    TP.chunks = reinterpret_cast<const SChunk*>(b->dev.p + goff[gi].chunks);
    TP.p_docs = reinterpret_cast<uint32_t*>(b->tile_dev.p + to_docs);
    TP.p_scores = reinterpret_cast<float*>(b->tile_dev.p + to_scores);
    TP.samples = reinterpret_cast<uint32_t*>(b->tile_dev.p + to_samples);
    TP.sample_count = reinterpret_cast<uint32_t*>(b->tile_dev.p + to_scount);
    TP.flags = reinterpret_cast<uint32_t*>(b->tile_dev.p + to_flags);
    TP.counters = c->tile_counters ? c->d_counters + 8 : nullptr;
    TP.sample_cap = sample_cap;
    TP.p_cap = gs.p_cap;
    TP.max_slots = gs.max_slots;
    TP.max_big = gs.max_big;
    TP.max_queries = (gs.max_queries + 1u) & ~1u;
    // per-tile work list: about two (query, essential clause) entries per query, more for wide unions; a tile that needs more
    // takes another round of routing + expansion
    TP.seg_cap = std::min<uint32_t>(4096u, std::max<uint32_t>(256u, std::max<uint32_t>(2u, gs.max_clauses / 4u) * TP.max_queries));
    if (c->tile_seg_cap_hook) TP.seg_cap = c->tile_seg_cap_hook;
    TP.light_max = c->tile_light_max;
    TP.cl_cap = gs.max_clause_words <= 16384u ? ((gs.max_clause_words + 3u) & ~3u) : 0u;
    TP.n_win = c->tile_windows ? std::min<uint32_t>(c->tile_windows, kTileWarps) : kTileExactWindows;
    run.smem = tile_smem_bytes(gs.p_cap, gs.max_slots, TP.max_big, TP.max_queries, TP.seg_cap, TP.cl_cap, TP.n_win);
    c->tile_smem_last = run.smem;
    if (run.smem > 200u * 1024u) return fail(TQ_ERR_UNSUPPORTED, "tile group needs more shared memory than an SM has");
    b->groups.push_back(run);
  }
  (void)tix_cursor;
  if (!b->groups.empty()) {  // the queries are kept: an overflowing run is repeated on the per-query kernels
    OwnedQueries& o = b->owned;
    o.q.assign(queries, queries + nq);
    size_t n_ts = 0, n_t = 0;
    for (size_t qi = 0; qi < nq; ++qi) { n_ts += queries[qi].n_term_segs; n_t += queries[qi].n_terms; }
    o.ts.reserve(n_ts); o.w.reserve(n_t); o.avg.reserve(n_t); o.flags.reserve(n_t);
    size_t n_cache = 0;
    for (size_t qi = 0; qi < nq; ++qi) if (queries[qi].tf_cache) n_cache += 256 * (size_t)queries[qi].n_terms;
    o.cache.reserve(n_cache);
    o.tp.reserve(n_ts); o.toff.reserve(n_t);
    for (size_t qi = 0; qi < nq; ++qi) {
      const tq_query& q = queries[qi];
      tq_query& d = o.q[qi];
      d.term_pos = nullptr;
      if (q.term_pos) { d.term_pos = reinterpret_cast<const tq_term_pos*>(o.tp.size() + 1); o.tp.insert(o.tp.end(), q.term_pos, q.term_pos + q.n_term_segs); }
      d.term_offset = nullptr;
      if (q.term_offset) { d.term_offset = reinterpret_cast<const uint32_t*>(o.toff.size() + 1); o.toff.insert(o.toff.end(), q.term_offset, q.term_offset + q.n_terms); }
      d.term_segs = reinterpret_cast<const tq_term_seg*>(o.ts.size());  // offsets for now (the vectors do not move again: reserved)
      o.ts.insert(o.ts.end(), q.term_segs, q.term_segs + q.n_term_segs);
      d.weight = reinterpret_cast<const float*>(o.w.size());
      o.w.insert(o.w.end(), q.weight, q.weight + q.n_terms);
      d.avg_fieldnorm = nullptr;
      if (q.avg_fieldnorm) { d.avg_fieldnorm = reinterpret_cast<const float*>(o.avg.size() + 1); o.avg.insert(o.avg.end(), q.avg_fieldnorm, q.avg_fieldnorm + q.n_terms); }
      d.tf_cache = nullptr;
      if (q.tf_cache) { d.tf_cache = reinterpret_cast<const float*>(o.cache.size() + 1); o.cache.insert(o.cache.end(), q.tf_cache, q.tf_cache + 256 * (size_t)q.n_terms); }
      d.term_flags = nullptr;
      if (q.term_flags) { d.term_flags = reinterpret_cast<const uint8_t*>(o.flags.size() + 1); o.flags.insert(o.flags.end(), q.term_flags, q.term_flags + q.n_terms); }
    }
    for (size_t qi = 0; qi < nq; ++qi) {
      tq_query& d = o.q[qi];
      d.term_segs = o.ts.data() + reinterpret_cast<size_t>(d.term_segs);
      d.weight = o.w.data() + reinterpret_cast<size_t>(d.weight);
      if (d.avg_fieldnorm) d.avg_fieldnorm = o.avg.data() + (reinterpret_cast<size_t>(d.avg_fieldnorm) - 1);
      if (d.tf_cache) d.tf_cache = o.cache.data() + (reinterpret_cast<size_t>(d.tf_cache) - 1);
      if (d.term_flags) d.term_flags = o.flags.data() + (reinterpret_cast<size_t>(d.term_flags) - 1);
      if (d.term_pos) d.term_pos = o.tp.data() + (reinterpret_cast<size_t>(d.term_pos) - 1);
      if (d.term_offset) d.term_offset = o.toff.data() + (reinterpret_cast<size_t>(d.term_offset) - 1);
    }
  }

  // ---- scratch: qstate | candidates | results ------------------------------------------------------
  b->kmax = kmax;
  b->n_cands = n_cands;
  size_t so = 0;
  b->qstate_off = so; so = align(so + std::max<size_t>(nq, 1) * sizeof(QState));
  b->cands_off = so; so = align(so + std::max<size_t>(n_cands, 1) * sizeof(Cand));
  b->res_off = so;
  const size_t rows = std::max<size_t>(nq, 1) * kmax;
  const size_t o_rs = 0, o_rg = align(rows * 4), o_rd = o_rg + align(rows * 4), o_rc = o_rd + align(rows * 4);
  b->res_bytes = o_rc + align(std::max<size_t>(nq, 1) * 4);
  so += b->res_bytes;
  TQ_CUDA(b->scratch.ensure(so));
  TQ_CUDA(b->res_pin.ensure(b->res_bytes));

  BatchParams& P = b->params;
  P.lists = c->d_lists;
  P.caches = reinterpret_cast<const float*>(b->dev.p + o_caches);
  P.tf_tables = reinterpret_cast<const float*>(b->dev.p + o_tftab);
  P.qlists = reinterpret_cast<const QList*>(b->dev.p + o_qlists);
  P.qsegs = reinterpret_cast<const QSeg*>(b->dev.p + o_qsegs);
  P.units = reinterpret_cast<const Unit*>(b->dev.p + o_units);
  P.queries = reinterpret_cast<const DQuery*>(b->dev.p + o_queries);
  P.qstate = reinterpret_cast<QState*>(b->scratch.p + b->qstate_off);
  P.cands = reinterpret_cast<Cand*>(b->scratch.p + b->cands_off);
  uint8_t* r = b->scratch.p + b->res_off;
  P.res_scores = reinterpret_cast<float*>(r + o_rs);
  P.res_segs = reinterpret_cast<uint32_t*>(r + o_rg);
  P.res_docs = reinterpret_cast<uint32_t*>(r + o_rd);
  P.res_counts = reinterpret_cast<uint32_t*>(r + o_rc);
  P.res_stride = kmax;
  P.n_queries = (uint32_t)nq;
  P.counters = c->d_counters;
  P.ovf = b->groups.empty() ? nullptr : reinterpret_cast<uint32_t*>(b->tile_dev.p + to_flags) + 1;

  TQ_CUDA(cudaEventRecord(b->ev_start, b->stream));
  TQ_CUDA(cudaMemcpyAsync(b->dev.p, b->pin.p, b->desc_bytes, cudaMemcpyHostToDevice, b->stream));
  {
    const unsigned n = (unsigned)(n_caches * kTfRows * 256);
    k_build_tf_tables<<<(n + 255) / 256, 256, 0, b->stream>>>(P.caches, reinterpret_cast<float*>(b->dev.p + o_tftab), (uint32_t)n_caches);
    TQ_CUDA(cudaGetLastError());
  }
  b->stats.lists_built = built;
  b->stats.units = n_units_total + tile_units;
  b->stats.h2d_bytes = b->desc_bytes;
  b->stats.algorithmic_bytes = alg_bytes;
  b->stats.postings = postings;
  b->stats.units_term = units[0].size(); b->stats.units_and = units[1].size(); b->stats.units_or = units[2].size() + units[3].size() + units[4].size() + units[5].size() + units[6].size(); b->stats.units_or_strip = units[3].size() + units[4].size() + units[5].size() + units[6].size();
  b->stats.bytes_term = op_bytes[0]; b->stats.bytes_and = op_bytes[1]; b->stats.bytes_or = op_bytes[2];
  b->stats.units_tile = tile_units;
  b->stats.units_phrase = units[7].size();
  b->stats.units_bool = units[8].size();
  b->stats.tile_groups = b->groups.size();
  b->stats.tile_postings = tile_postings;
  for (auto& tg : tgroups) b->stats.tile_list_bytes += tg.list_bytes;
  b->stats.tile_scratch_bytes = tile_bytes;
  guard.ok = true;
  *out = b;
  return TQ_OK;
}

// Phases of a run: 0 = term / AND / window-union kernels + the decode-and-score pass and the sample launch of the tile engine
// + the strips' first threshold round, 1 and 2 = the next (exact) tile launches / threshold rounds, 3 = the last tile launch,
// the strips' main launch and k_final.  Every phase but the last ends with the per-query thresholds refreshed (k_theta).
// Sharded callers exchange keys in between.
constexpr int kPhases = 4;

static int launch_tile_round(tq_batch* b, int r, uint64_t* launches) {
  bool any = false;
  for (auto& g : b->groups) any = any || g.n_units[r];
  if (!any) return TQ_OK;
  const int sp = span_begin(b, SPAN_TILE);
  for (auto& g : b->groups) {
    if (!g.n_units[r]) continue;
    k_tile<<<g.n_units[r], kTileThreads, g.smem, b->stream>>>(b->params, g.params, g.unit_base[r], r == 0 ? 1u : 0u);
    ++*launches;
  }
  span_end(b, sp);
  TQ_CUDA(cudaGetLastError());
  return TQ_OK;
}

static int run_phase(tq_batch* b, int phase) {
  TQ_CUDA(cudaSetDevice(b->ctx->device));
  const BatchParams& P = b->params;
  uint64_t launches = 0;
  if (phase != b->next_phase) return fail(TQ_ERR_INVALID_ARGUMENT, "phases run in order, each once per run");
  const bool tiles = !b->groups.empty();
  if (phase == 0) {
    b->n_spans = 0;
    b->finalized = false;
    if (b->side_pending) { TQ_CUDA(cudaStreamWaitEvent(b->stream, b->ev_side1, 0)); b->side_pending = false; }  // (a run that was abandoned)
    TQ_CUDA(cudaMemcpyAsync(P.qstate, b->dev.p + b->qinit_off, std::max<size_t>(b->nq, 1) * sizeof(QState), cudaMemcpyDeviceToDevice, b->stream));
    if (tiles) TQ_CUDA(cudaMemsetAsync(b->tile_dev.p + b->tile_zero_off, 0, b->tile_zero_bytes, b->stream));
    TQ_CUDA(cudaEventRecord(b->ev_k0, b->stream));
    if (b->n_units[TQ_OP_TERM]) {
      const int sp = span_begin(b, SPAN_TERM);
      k_term<<<b->n_units[TQ_OP_TERM], kThreads, 0, b->stream>>>(P, b->unit_base[TQ_OP_TERM]); ++launches;
      span_end(b, sp);
    }
    if (b->n_units[TQ_OP_AND]) {
      const int sp = span_begin(b, SPAN_AND);
      k_and<<<b->n_units[TQ_OP_AND], kThreads, 0, b->stream>>>(P, b->unit_base[TQ_OP_AND]); ++launches;
      span_end(b, sp);
    }
    if (b->n_units[7]) {
      // phrase queries share nothing with the tile engine's launches (their own candidate regions; k_theta and the key export
      // skip them) and k_phrase waits on dependent position loads most of the time: it runs on a second stream next to them
      const bool aside = tiles && b->ctx->phrase_side;
      cudaStream_t on = aside ? b->side : b->stream;
      if (aside) {
        TQ_CUDA(cudaEventRecord(b->ev_side0, b->stream));
        TQ_CUDA(cudaStreamWaitEvent(b->side, b->ev_side0, 0));
      }
      const int sp = span_begin(b, SPAN_PHRASE, on);
      k_phrase<<<b->n_units[7], kPhraseThreads, phrase_smem_bytes(b->phrase_ct), on>>>(P, b->ctx->d_pos_descs, b->phrase_aux, b->unit_base[7], b->phrase_ct); ++launches;
      span_end(b, sp, on);
      if (aside) {
        TQ_CUDA(cudaEventRecord(b->ev_side1, b->side));
        b->side_pending = true;
      }
    }
    if (b->n_units[TQ_OP_OR]) {
      const int sp = span_begin(b, SPAN_OR);
      k_or<<<b->n_units[TQ_OP_OR], kThreads, kOrDynSmem, b->stream>>>(P, b->unit_base[TQ_OP_OR]); ++launches;
      span_end(b, sp);
    }
    if (b->n_units[8]) {
      const int sp = span_begin(b, SPAN_BOOL);
      k_bool<<<b->n_units[8], kThreads, kBoolDynSmem, b->stream>>>(P, b->unit_base[8]); ++launches;
      span_end(b, sp);
    }
    if (tiles) {  // K1 + K2 once for every distinct list of the batch
      const int sp = span_begin(b, SPAN_SCORE);
      for (auto& g : b->groups)
        if (g.n_chunks) { k_score_lists<<<g.n_chunks, kThreads, 0, b->stream>>>(P, g.params, 0u); ++launches; }
      span_end(b, sp);
      TQ_CUDA(cudaGetLastError());
    }
    b->stats.kernel_launches = 0;
  }
  if (phase < kPhases - 1) {
    // tile engine: phase 0 = sample launch, then exact launches; strips: threshold round `phase`
    if (tiles) {
      const int rc = launch_tile_round(b, phase, &launches);
      if (rc != TQ_OK) return rc;
      if (phase == 0 && (kTileRounds == kPhases + 0)) {}  // (rounds 1..3 belong to phases 1..3)
    }
    const int r = 4 + phase;
    if (b->n_units[r]) {
      const int sp = span_begin(b, SPAN_OR);
      k_or_strip<<<b->n_units[r], kStripThreads, strip_smem_bytes(b->strip_cached_max), b->stream>>>(P, b->unit_base[r], b->strip_cached_max);
      ++launches;
      span_end(b, sp);
    }
    bool tile_round = false;
    for (auto& g : b->groups) tile_round = tile_round || g.n_units[phase];
    if ((b->n_units[r] || (tile_round && phase > 0)) && b->nq) {
      const int sp = span_begin(b, SPAN_THETA);
      k_theta<<<(unsigned)b->nq, kThreads, 0, b->stream>>>(P);
      ++launches;
      span_end(b, sp);
    }
    if (tile_round && phase == 0 && b->nq) {
      const int sp = span_begin(b, SPAN_THETA);
      const TileParams& TP = b->groups[0].params;
      k_theta_samples<<<(unsigned)b->nq, kThreads, 0, b->stream>>>(P, TP.samples, TP.sample_count, TP.sample_cap);
      ++launches;
      span_end(b, sp);
    }
    TQ_CUDA(cudaGetLastError());
    b->stats.kernel_launches += launches;
    b->next_phase = phase + 1;
    b->last_round_sampled = tile_round && phase == 0;
    return TQ_OK;
  }
  if (tiles) {
    const int rc = launch_tile_round(b, kTileRounds - 1, &launches);
    if (rc != TQ_OK) return rc;
  }
  if (b->n_units[3]) {
    const int sp = span_begin(b, SPAN_OR);
    k_or_strip<<<b->n_units[3], kStripThreads, strip_smem_bytes(b->strip_cached_max), b->stream>>>(P, b->unit_base[3], b->strip_cached_max); ++launches;
    span_end(b, sp);
  }
  TQ_CUDA(cudaGetLastError());
  if (b->side_pending) { TQ_CUDA(cudaStreamWaitEvent(b->stream, b->ev_side1, 0)); b->side_pending = false; }
  if (b->nq) {
    const int sp = span_begin(b, SPAN_FINAL);
    k_final<<<b->nq, kThreads, 0, b->stream>>>(P); ++launches;
    span_end(b, sp);
  }
  TQ_CUDA(cudaGetLastError());
  if (tiles) TQ_CUDA(cudaMemcpyAsync(b->flags_pin, b->tile_dev.p + b->tile_flags_off, 16, cudaMemcpyDeviceToHost, b->stream));
  TQ_CUDA(cudaEventRecord(b->ev_k1, b->stream));
  b->stats.kernel_launches += launches;
  b->next_phase = 0;
  b->ran = true;
  return TQ_OK;
}

// After the last phase: wait for the stream; a run whose tile engine overflowed (a tile with more pairs than its buffer, or a
// query with more candidates than its region) is repeated on the per-query kernels and its rows replace ours.  Exactness
// never depends on the fast path's capacity guesses.
static int finalize_run(tq_batch* b) {
  if (!b->ran) return fail(TQ_ERR_INVALID_ARGUMENT, "batch has not run");
  if (b->finalized) return TQ_OK;
  TQ_CUDA(cudaStreamSynchronize(b->stream));
  b->finalized = true;
  if (b->groups.empty() || b->is_fallback) return TQ_OK;
  if (b->flags_pin[0] == 0 && b->flags_pin[1] == 0) return TQ_OK;
  tq_batch* fb = nullptr;
  int rc = batch_prepare_impl(b->ctx, b->owned.q.data(), b->owned.q.size(), true, &fb);
  if (rc != TQ_OK) return rc;
  rc = tq_batch_run(fb);
  if (rc == TQ_OK) {
    cudaError_t e = cudaStreamSynchronize(fb->stream);
    if (e == cudaSuccess && fb->res_bytes == b->res_bytes)
      e = cudaMemcpyAsync(b->scratch.p + b->res_off, fb->scratch.p + fb->res_off, b->res_bytes, cudaMemcpyDeviceToDevice, b->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(b->stream);
    if (e != cudaSuccess) rc = fail(TQ_ERR_CUDA, cudaGetErrorString(e));
    else if (fb->res_bytes != b->res_bytes) rc = fail(TQ_ERR_CUDA, "fallback batch layout differs");
  }
  tq_batch_destroy(fb);
  b->stats.tile_fallbacks = 1;
  return rc;
}

extern "C" {

int tq_batch_run(tq_batch* b) {
  if (!b) return fail(TQ_ERR_INVALID_ARGUMENT, "null");
  for (int p = b->next_phase; p < kPhases; ++p) {
    const int rc = run_phase(b, p);
    if (rc != TQ_OK) { b->next_phase = 0; return rc; }
  }
  return TQ_OK;
}

int tq_batch_phases(tq_batch* b) { return b ? kPhases : 0; }

int tq_batch_run_phase(tq_batch* b, int phase) {
  if (!b || phase < 0 || phase >= kPhases) return fail(TQ_ERR_INVALID_ARGUMENT, "batch / phase");
  const int rc = run_phase(b, phase);
  if (rc != TQ_OK && rc != TQ_ERR_INVALID_ARGUMENT) b->next_phase = 0;  // a failed run starts over
  return rc;
}

int tq_batch_stream(tq_batch* b, void** stream_out) {
  if (!b || !stream_out) return fail(TQ_ERR_INVALID_ARGUMENT, "null");
  *stream_out = (void*)b->stream;
  return TQ_OK;
}

int tq_batch_thresholds_export_dev(tq_batch* b, int64_t* keys_dev) {
  if (!b || !keys_dev || b->next_phase == 0) return fail(TQ_ERR_INVALID_ARGUMENT, "export needs a batch between two phases of a run");
  TQ_CUDA(cudaSetDevice(b->ctx->device));
  if (b->nq) k_theta_export<<<(unsigned)((b->nq + 255) / 256), 256, 0, b->stream>>>(b->params.qstate, reinterpret_cast<long long*>(keys_dev), (uint32_t)b->nq);
  TQ_CUDA(cudaGetLastError());
  TQ_CUDA(cudaStreamSynchronize(b->stream));  // the caller's collective runs on its own stream
  return TQ_OK;
}

int tq_batch_thresholds_import_dev(tq_batch* b, const int64_t* keys_dev) {
  if (!b || !keys_dev || b->next_phase == 0) return fail(TQ_ERR_INVALID_ARGUMENT, "import needs a batch between two phases of a run");
  TQ_CUDA(cudaSetDevice(b->ctx->device));
  if (b->nq) k_theta_import<<<(unsigned)((b->nq + 255) / 256), 256, 0, b->stream>>>(b->params.qstate, reinterpret_cast<const long long*>(keys_dev), (uint32_t)b->nq);
  TQ_CUDA(cudaGetLastError());
  return TQ_OK;
}

int tq_batch_topkeys_export_dev(tq_batch* b, uint32_t* keys_dev, uint32_t k_stride) {
  if (!b || !keys_dev || !k_stride || b->next_phase == 0) return fail(TQ_ERR_INVALID_ARGUMENT, "export needs a batch between two phases of a run");
  TQ_CUDA(cudaSetDevice(b->ctx->device));
  if (b->nq) {
    const bool from_samples = b->last_round_sampled && !b->groups.empty();
    const TileParams* TP = b->groups.empty() ? nullptr : &b->groups[0].params;
    k_topkeys_export<<<(unsigned)b->nq, kThreads, 0, b->stream>>>(b->params, TP ? TP->samples : nullptr, TP ? TP->sample_count : nullptr,
                                                                  TP ? TP->sample_cap : 0u, from_samples ? 1u : 0u, keys_dev, k_stride);
  }
  TQ_CUDA(cudaGetLastError());
  return TQ_OK;  // enqueued on the batch's stream (tq_batch_stream): the caller's collective must be ordered behind it
}

int tq_batch_thresholds_from_keys_dev(tq_batch* b, const uint32_t* gathered_dev, uint32_t n_shards, uint32_t k_stride) {
  if (!b || !gathered_dev || !n_shards || !k_stride || b->next_phase == 0) return fail(TQ_ERR_INVALID_ARGUMENT, "import needs a batch between two phases of a run");
  if ((size_t)n_shards * k_stride * 4 > 200u * 1024u) return fail(TQ_ERR_UNSUPPORTED, "n_shards * k_stride too large for one CTA");
  TQ_CUDA(cudaSetDevice(b->ctx->device));
  if (b->nq) {
    const size_t smem = (size_t)n_shards * k_stride * 4;
    if (smem > 48u * 1024u) TQ_CUDA(cudaFuncSetAttribute(k_theta_from_keys, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k_theta_from_keys<<<(unsigned)b->nq, kThreads, smem, b->stream>>>(b->params, gathered_dev, n_shards, (uint32_t)b->nq, k_stride);
  }
  TQ_CUDA(cudaGetLastError());
  return TQ_OK;
}

int tq_batch_results_dev(tq_batch* b, const float** scores_dev, const uint32_t** segment_ord_dev, const uint32_t** doc_dev,
                         const uint32_t** count_dev, uint32_t* stride) {
  if (!b || !b->ran) return fail(TQ_ERR_INVALID_ARGUMENT, "batch has not run");
  TQ_CUDA(cudaSetDevice(b->ctx->device));
  { const int rc = finalize_run(b); if (rc != TQ_OK) return rc; }
  if (scores_dev) *scores_dev = b->params.res_scores;
  if (segment_ord_dev) *segment_ord_dev = b->params.res_segs;
  if (doc_dev) *doc_dev = b->params.res_docs;
  if (count_dev) *count_dev = b->params.res_counts;
  if (stride) *stride = b->kmax;
  collect_times(b);
  std::lock_guard<std::mutex> g(b->ctx->mu);
  b->ctx->stats = b->stats;
  return TQ_OK;
}

int tq_batch_results_copy_dev(tq_batch* b, float* scores_dev, uint32_t* segment_ord_dev, uint32_t* doc_dev, uint32_t* count_dev) {
  if (!b || !b->ran) return fail(TQ_ERR_INVALID_ARGUMENT, "batch has not run");
  if (!scores_dev || !segment_ord_dev || !doc_dev || !count_dev) return fail(TQ_ERR_INVALID_ARGUMENT, "null output");
  TQ_CUDA(cudaSetDevice(b->ctx->device));
  { const int rc = finalize_run(b); if (rc != TQ_OK) return rc; }
  const size_t rows = (size_t)b->nq * b->kmax * 4;
  TQ_CUDA(cudaMemcpyAsync(scores_dev, b->params.res_scores, rows, cudaMemcpyDeviceToDevice, b->stream));
  TQ_CUDA(cudaMemcpyAsync(segment_ord_dev, b->params.res_segs, rows, cudaMemcpyDeviceToDevice, b->stream));
  TQ_CUDA(cudaMemcpyAsync(doc_dev, b->params.res_docs, rows, cudaMemcpyDeviceToDevice, b->stream));
  TQ_CUDA(cudaMemcpyAsync(count_dev, b->params.res_counts, (size_t)b->nq * 4, cudaMemcpyDeviceToDevice, b->stream));
  TQ_CUDA(cudaStreamSynchronize(b->stream));
  collect_times(b);
  std::lock_guard<std::mutex> g(b->ctx->mu);
  b->ctx->stats = b->stats;
  return TQ_OK;
}

int tq_batch_fetch(tq_batch* b, uint32_t out_stride, float* out_scores, uint32_t* out_segment_ord, uint32_t* out_doc, uint32_t* out_count) {
  if (!b || !b->ran) return fail(TQ_ERR_INVALID_ARGUMENT, "batch has not run");
  if (!out_scores || !out_segment_ord || !out_doc || !out_count) return fail(TQ_ERR_INVALID_ARGUMENT, "null output");
  TQ_CUDA(cudaSetDevice(b->ctx->device));
  if (!b->groups.empty()) { const int rc = finalize_run(b); if (rc != TQ_OK) return rc; }  // (a run without tile groups cannot overflow: one sync below)
  TQ_CUDA(cudaMemcpyAsync(b->res_pin.p, b->scratch.p + b->res_off, b->res_bytes, cudaMemcpyDeviceToHost, b->stream));
  TQ_CUDA(cudaEventRecord(b->ev_end, b->stream));
  TQ_CUDA(cudaStreamSynchronize(b->stream));
  const size_t rows = std::max<size_t>(b->nq, 1) * b->kmax;
  auto align = [](size_t x) { return (x + 255) & ~(size_t)255; };
  const float* rs = reinterpret_cast<const float*>(b->res_pin.p);
  const uint32_t* rg = reinterpret_cast<const uint32_t*>(b->res_pin.p + align(rows * 4));
  const uint32_t* rd = reinterpret_cast<const uint32_t*>(b->res_pin.p + 2 * align(rows * 4));
  const uint32_t* rc = reinterpret_cast<const uint32_t*>(b->res_pin.p + 3 * align(rows * 4));
  for (uint32_t q = 0; q < b->nq; ++q) {
    const uint32_t n = std::min(std::min(rc[q], b->kmax), out_stride);
    out_count[q] = rc[q];
    memcpy(out_scores + (size_t)q * out_stride, rs + (size_t)q * b->kmax, n * 4);
    memcpy(out_segment_ord + (size_t)q * out_stride, rg + (size_t)q * b->kmax, n * 4);
    memcpy(out_doc + (size_t)q * out_stride, rd + (size_t)q * b->kmax, n * 4);
  }
  collect_times(b);
  float ms = 0;
  if (cudaEventElapsedTime(&ms, b->ev_start, b->ev_end) == cudaSuccess) b->stats.total_ms = ms;
  b->stats.d2h_bytes = b->res_bytes;
  std::lock_guard<std::mutex> g(b->ctx->mu);
  b->ctx->stats = b->stats;
  return TQ_OK;
}

int tq_search_batch(tq_ctx* c, const tq_query* queries, size_t nq, uint32_t out_stride, float* out_scores, uint32_t* out_segment_ord,
                    uint32_t* out_doc, uint32_t* out_count) {
  tq_batch* b = nullptr;
  int rc = tq_batch_prepare(c, queries, nq, &b);
  if (rc != TQ_OK) return rc;
  rc = tq_batch_run(b);
  if (rc == TQ_OK) rc = tq_batch_fetch(b, out_stride, out_scores, out_segment_ord, out_doc, out_count);
  tq_batch_destroy(b);
  return rc;
}

int tq_merge_topk_dev(tq_ctx* c, uint32_t n_lists, uint32_t nq, uint32_t stride, uint32_t k, const float* scores_dev,
                      const uint32_t* segment_ord_dev, const uint32_t* doc_dev, const uint32_t* count_dev, float* out_scores_dev,
                      uint32_t* out_segment_ord_dev, uint32_t* out_doc_dev, uint32_t* out_count_dev) {
  if (!c) return fail(TQ_ERR_INVALID_ARGUMENT, "null");
  if (k == 0 || k > TQ_MAX_K || stride < 1) return fail(TQ_ERR_INVALID_ARGUMENT, "k / stride");
  TQ_CUDA(cudaSetDevice(c->device));
  if (nq == 0) return TQ_OK;
  k_merge<<<nq, kThreads, 0, 0>>>(n_lists, nq, stride, std::min(k, stride), (size_t)nq * stride, (size_t)nq, scores_dev, segment_ord_dev, doc_dev,
                                  count_dev, out_scores_dev, out_segment_ord_dev, out_doc_dev, out_count_dev);
  TQ_CUDA(cudaGetLastError());
  TQ_CUDA(cudaStreamSynchronize(0));
  return TQ_OK;
}

// Packed form for sharded callers: one buffer per shard = [nq*stride scores | nq*stride segment ords | nq*stride docs | nq counts]
// (32-bit words, what tq_batch_results_pack_dev writes), `n_lists` of them `pitch_words` apart -- the layout ONE all-gather
// produces.  Enqueued on `cuda_stream` (a cudaStream_t; e.g. the batch's, tq_batch_stream) without any host synchronisation.
int tq_merge_topk_packed_dev(tq_ctx* c, void* cuda_stream, uint32_t n_lists, uint32_t nq, uint32_t stride, uint32_t k, const uint32_t* packed_dev,
                             size_t pitch_words, uint32_t* out_packed_dev) {
  if (!c || !packed_dev || !out_packed_dev) return fail(TQ_ERR_INVALID_ARGUMENT, "null");
  if (k == 0 || k > TQ_MAX_K || stride < 1 || pitch_words < (size_t)3 * nq * stride + nq) return fail(TQ_ERR_INVALID_ARGUMENT, "k / stride / pitch");
  TQ_CUDA(cudaSetDevice(c->device));
  if (nq == 0) return TQ_OK;
  const size_t rows = (size_t)nq * stride;
  k_merge<<<nq, kThreads, 0, (cudaStream_t)cuda_stream>>>(n_lists, nq, stride, std::min(k, stride), pitch_words, pitch_words,
                                                          reinterpret_cast<const float*>(packed_dev), packed_dev + rows, packed_dev + 2 * rows,
                                                          packed_dev + 3 * rows, reinterpret_cast<float*>(out_packed_dev), out_packed_dev + rows,
                                                          out_packed_dev + 2 * rows, out_packed_dev + 3 * rows);
  TQ_CUDA(cudaGetLastError());
  return TQ_OK;
}

// The result rows of a finished run in the packed layout above (row stride = k_max of the batch), into a caller-owned DEVICE buffer
// of 3 * nq * k_max + nq words.  Waits for the run (a tile-engine overflow is resolved first), then copies on the batch's stream.
int tq_batch_results_pack_dev(tq_batch* b, uint32_t* packed_dev) {
  if (!b || !b->ran) return fail(TQ_ERR_INVALID_ARGUMENT, "batch has not run");
  if (!packed_dev) return fail(TQ_ERR_INVALID_ARGUMENT, "null output");
  TQ_CUDA(cudaSetDevice(b->ctx->device));
  { const int rc = finalize_run(b); if (rc != TQ_OK) return rc; }
  const size_t rows = (size_t)b->nq * b->kmax;
  TQ_CUDA(cudaMemcpyAsync(packed_dev, b->params.res_scores, rows * 4, cudaMemcpyDeviceToDevice, b->stream));
  TQ_CUDA(cudaMemcpyAsync(packed_dev + rows, b->params.res_segs, rows * 4, cudaMemcpyDeviceToDevice, b->stream));
  TQ_CUDA(cudaMemcpyAsync(packed_dev + 2 * rows, b->params.res_docs, rows * 4, cudaMemcpyDeviceToDevice, b->stream));
  TQ_CUDA(cudaMemcpyAsync(packed_dev + 3 * rows, b->params.res_counts, (size_t)b->nq * 4, cudaMemcpyDeviceToDevice, b->stream));
  collect_times(b);
  std::lock_guard<std::mutex> g(b->ctx->mu);
  b->ctx->stats = b->stats;
  return TQ_OK;
}

// The same rows WITHOUT waiting for the run: everything is enqueued on the batch's stream right behind the run's last kernel, so a
// sharded caller can queue pack -> all-gather -> merge -> the next batch's run and only then wait for this one (two batches in
// flight).  packed_dev holds 3 * nq * k_max + nq + 4 words; the last four are the run's overflow flags -- all zero: the rows are
// final; anything else: the tile engine overflowed a buffer and the caller must take tq_batch_results_pack_dev (which repeats the
// run on the per-query kernels) instead.  The flags travel with the rows, so every shard sees every shard's.
int tq_batch_results_pack_dev_async(tq_batch* b, uint32_t* packed_dev) {
  if (!b || !b->ran) return fail(TQ_ERR_INVALID_ARGUMENT, "batch has not run");
  if (!packed_dev) return fail(TQ_ERR_INVALID_ARGUMENT, "null output");
  TQ_CUDA(cudaSetDevice(b->ctx->device));
  const size_t rows = (size_t)b->nq * b->kmax;
  TQ_CUDA(cudaMemcpyAsync(packed_dev, b->params.res_scores, rows * 4, cudaMemcpyDeviceToDevice, b->stream));
  TQ_CUDA(cudaMemcpyAsync(packed_dev + rows, b->params.res_segs, rows * 4, cudaMemcpyDeviceToDevice, b->stream));
  TQ_CUDA(cudaMemcpyAsync(packed_dev + 2 * rows, b->params.res_docs, rows * 4, cudaMemcpyDeviceToDevice, b->stream));
  TQ_CUDA(cudaMemcpyAsync(packed_dev + 3 * rows, b->params.res_counts, (size_t)b->nq * 4, cudaMemcpyDeviceToDevice, b->stream));
  uint32_t* flags = packed_dev + 3 * rows + b->nq;
  if (!b->groups.empty() && !b->is_fallback && !b->finalized)
    TQ_CUDA(cudaMemcpyAsync(flags, b->tile_dev.p + b->tile_flags_off, 16, cudaMemcpyDeviceToDevice, b->stream));
  else
    TQ_CUDA(cudaMemsetAsync(flags, 0, 16, b->stream));  // (per-query kernels cannot overflow; a finalized run has been repaired already)
  return TQ_OK;
}

// ---- Count collector -------------------------------------------------------------------------------------------
int tq_count_batch(tq_ctx* c, const tq_query* queries, size_t nq, uint64_t* out_counts) {
  if (!c || (!queries && nq) || (!out_counts && nq)) return fail(TQ_ERR_INVALID_ARGUMENT, "null");
  TQ_CUDA(cudaSetDevice(c->device));
  for (size_t qi = 0; qi < nq; ++qi) out_counts[qi] = 0;
  if (!nq) return TQ_OK;
  tq_batch* b = acquire_batch(c);
  if (!b) return fail(TQ_ERR_CUDA, "stream/event creation failed");
  struct Guard { tq_batch* b; ~Guard() { tq_batch_destroy(b); } } guard{b};
  std::vector<uint32_t> list_ids;
  std::vector<CountSeg> segs;
  std::vector<Unit> units;
  std::vector<uint32_t> bool_words;  // TQ_OP_BOOL (query, segment) pairs: their structure words with list ids
  std::vector<CountBoolSeg> bool_segs;
  std::vector<Unit> bool_units;
  {
    std::lock_guard<std::mutex> g(c->mu);
    std::vector<PendingBuild> pending;
    PendingScope pending_scope{c, pending};
    uint64_t built = 0;
    std::vector<const tq_term_seg*> order;
    for (size_t qi = 0; qi < nq; ++qi) {
      const tq_query& q = queries[qi];
      if (q.n_terms == 0 || q.n_terms > TQ_MAX_TERMS) return fail(TQ_ERR_INVALID_ARGUMENT, "n_terms must be in 1..TQ_MAX_TERMS");
      if (q.op != TQ_OP_TERM && q.op != TQ_OP_AND && q.op != TQ_OP_OR && q.op != TQ_OP_BOOL) return fail(TQ_ERR_INVALID_ARGUMENT, "op");
      if (q.op == TQ_OP_TERM && q.n_terms != 1) return fail(TQ_ERR_INVALID_ARGUMENT, "TQ_OP_TERM takes one term");
      if (!q.term_segs && q.n_term_segs) return fail(TQ_ERR_INVALID_ARGUMENT, "query arrays");
      if (q.op == TQ_OP_BOOL && (!q.term_occur || !q.weight)) return fail(TQ_ERR_INVALID_ARGUMENT, "TQ_OP_BOOL needs term_occur and weights");
      order.clear();
      for (uint32_t i = 0; i < q.n_term_segs; ++i) {
        if (q.term_segs[i].term_idx >= q.n_terms) return fail(TQ_ERR_INVALID_ARGUMENT, "term_idx out of range");
        if (q.term_segs[i].doc_freq) order.push_back(&q.term_segs[i]);
      }
      std::stable_sort(order.begin(), order.end(), [](const tq_term_seg* a, const tq_term_seg* b) {
        return a->segment_ord != b->segment_ord ? a->segment_ord < b->segment_ord : a->term_idx < b->term_idx;
      });
      for (size_t i = 0; i < order.size();) {
        size_t j = i;
        while (j < order.size() && order[j]->segment_ord == order[i]->segment_ord) ++j;
        const uint32_t n_here = (uint32_t)(j - i);
        if (q.op == TQ_OP_BOOL) {  // mixed shapes: the structure of this segment, with list ids in place of the clause indices
          uint32_t tix_[TQ_MAX_TERMS], dfs_[TQ_MAX_TERMS], ids_[TQ_MAX_TERMS];
          float ws_[TQ_MAX_TERMS];
          const Segment* seg = nullptr;
          for (size_t a = i; a < j; ++a) {
            int rc = get_list(c, *order[a], false, pending, &ids_[a - i], &seg);
            if (rc != TQ_OK) return rc;
            tix_[a - i] = order[a]->term_idx; dfs_[a - i] = order[a]->doc_freq; ws_[a - i] = q.weight[order[a]->term_idx];
          }
          std::vector<uint16_t> words;
          const int st = bool_structure(q, tix_, dfs_, ws_, n_here, words);
          if (st < 0) return fail(TQ_ERR_INVALID_ARGUMENT, "term_occur");
          if (st > 0) {
            CountBoolSeg bs{};
            bs.query = (uint32_t)qi; bs.words_base = (uint32_t)bool_words.size(); bs.max_doc = seg->max_doc; bs.alive = seg->d_alive;
            size_t x = 0;
            for (int k4 = 0; k4 < 4; ++k4) bool_words.push_back(words[x++]);
            for (uint32_t g2 = 0; g2 < words[0]; ++g2) { const uint16_t len = words[x++]; bool_words.push_back(len); for (uint16_t e = 0; e < len; ++e) bool_words.push_back(ids_[words[x++]]); }
            while (x < words.size()) bool_words.push_back(ids_[words[x++]]);
            const uint32_t tiles = (bs.max_doc + kTileDocs - 1) / kTileDocs, per = 8;
            for (uint32_t t0 = 0; t0 < tiles; t0 += per) bool_units.push_back(Unit{(uint32_t)bool_segs.size(), t0, std::min(tiles, t0 + per), 0});
            bool_segs.push_back(bs);
          }
          i = j;
          continue;
        }
        if (q.op == TQ_OP_AND && n_here < q.n_terms) { i = j; continue; }  // a clause without postings: empty intersection
        CountSeg cs{};
        cs.query = (uint32_t)qi; cs.lists_base = (uint32_t)list_ids.size(); cs.n_lists = n_here; cs.op = (uint32_t)q.op;
        const Segment* seg = nullptr;
        uint64_t df_single = 0;
        for (size_t a = i; a < j; ++a) {
          uint32_t id;
          int rc = get_list(c, *order[a], false, pending, &id, &seg);
          if (rc != TQ_OK) return rc;
          list_ids.push_back(id);
          df_single = order[a]->doc_freq;
        }
        cs.max_doc = seg->max_doc;
        cs.alive = seg->d_alive;
        if (n_here == 1 && !seg->d_alive) {  // TermWeight::count without deletes: the term's doc_freq (term_weight.rs:179-190)
          out_counts[qi] += df_single;
          list_ids.resize(cs.lists_base);
        } else {
          const uint32_t tiles = (cs.max_doc + kTileDocs - 1) / kTileDocs, per = 8;
          for (uint32_t t0 = 0; t0 < tiles; t0 += per) units.push_back(Unit{(uint32_t)segs.size(), t0, std::min(tiles, t0 + per), 0});
          segs.push_back(cs);
        }
        i = j;
      }
    }
    int rc = flush_builds(c, pending, &built);
    if (rc != TQ_OK) return rc;
  }
  if (!bool_units.empty()) {  // mixed boolean shapes: their own kernel, counts added to out_counts
    auto align2 = [](size_t x) { return (x + 255) & ~(size_t)255; };
    size_t o2 = 0;
    const size_t o_w = o2; o2 = align2(o2 + bool_words.size() * 4);
    const size_t o_s = o2; o2 = align2(o2 + bool_segs.size() * sizeof(CountBoolSeg));
    const size_t o_u = o2; o2 = align2(o2 + bool_units.size() * sizeof(Unit));
    const size_t o_c = o2; o2 = align2(o2 + nq * 8);
    TQ_CUDA(b->pin.ensure(o2 + 256));
    TQ_CUDA(b->dev.ensure(o2 + 256));
    memcpy(b->pin.p + o_w, bool_words.data(), bool_words.size() * 4);
    memcpy(b->pin.p + o_s, bool_segs.data(), bool_segs.size() * sizeof(CountBoolSeg));
    memcpy(b->pin.p + o_u, bool_units.data(), bool_units.size() * sizeof(Unit));
    memset(b->pin.p + o_c, 0, nq * 8);
    TQ_CUDA(cudaMemcpyAsync(b->dev.p, b->pin.p, o2, cudaMemcpyHostToDevice, b->stream));
    CountBoolParams BP;
    BP.lists = c->d_lists;
    BP.words = reinterpret_cast<const uint32_t*>(b->dev.p + o_w);
    BP.segs = reinterpret_cast<const CountBoolSeg*>(b->dev.p + o_s);
    BP.units = reinterpret_cast<const Unit*>(b->dev.p + o_u);
    BP.counts = reinterpret_cast<unsigned long long*>(b->dev.p + o_c);
    k_count_bool<<<(unsigned)bool_units.size(), kThreads, 0, b->stream>>>(BP);
    TQ_CUDA(cudaGetLastError());
    TQ_CUDA(cudaMemcpyAsync(b->pin.p + o_c, b->dev.p + o_c, nq * 8, cudaMemcpyDeviceToHost, b->stream));
    TQ_CUDA(cudaStreamSynchronize(b->stream));
    const unsigned long long* dc = reinterpret_cast<const unsigned long long*>(b->pin.p + o_c);
    for (size_t qi = 0; qi < nq; ++qi) out_counts[qi] += dc[qi];
  }
  if (units.empty()) return TQ_OK;
  auto align = [](size_t x) { return (x + 255) & ~(size_t)255; };
  size_t off = 0;
  const size_t o_ids = off; off = align(off + list_ids.size() * 4);
  const size_t o_segs = off; off = align(off + segs.size() * sizeof(CountSeg));
  const size_t o_units = off; off = align(off + units.size() * sizeof(Unit));
  const size_t o_counts = off; off = align(off + nq * 8);
  TQ_CUDA(b->pin.ensure(off + 256));
  TQ_CUDA(b->dev.ensure(off + 256));
  memcpy(b->pin.p + o_ids, list_ids.data(), list_ids.size() * 4);
  memcpy(b->pin.p + o_segs, segs.data(), segs.size() * sizeof(CountSeg));
  memcpy(b->pin.p + o_units, units.data(), units.size() * sizeof(Unit));
  memset(b->pin.p + o_counts, 0, nq * 8);
  TQ_CUDA(cudaMemcpyAsync(b->dev.p, b->pin.p, off, cudaMemcpyHostToDevice, b->stream));
  CountParams P;
  P.lists = c->d_lists;
  P.list_ids = reinterpret_cast<const uint32_t*>(b->dev.p + o_ids);
  P.segs = reinterpret_cast<const CountSeg*>(b->dev.p + o_segs);
  P.units = reinterpret_cast<const Unit*>(b->dev.p + o_units);
  P.counts = reinterpret_cast<unsigned long long*>(b->dev.p + o_counts);
  k_count<<<(unsigned)units.size(), kThreads, 0, b->stream>>>(P);
  TQ_CUDA(cudaGetLastError());
  TQ_CUDA(cudaMemcpyAsync(b->pin.p + o_counts, b->dev.p + o_counts, nq * 8, cudaMemcpyDeviceToHost, b->stream));
  TQ_CUDA(cudaStreamSynchronize(b->stream));
  const unsigned long long* dc = reinterpret_cast<const unsigned long long*>(b->pin.p + o_counts);
  for (size_t qi = 0; qi < nq; ++qi) out_counts[qi] += dc[qi];
  return TQ_OK;
}

// ---- codec-level access ---------------------------------------------------------------------------
static int resolve_single(tq_ctx* c, const tq_term_seg* list, uint32_t* id) {
  std::lock_guard<std::mutex> g(c->mu);
  std::vector<PendingBuild> pending;
  PendingScope pending_scope{c, pending};
  const Segment* seg;
  uint64_t built = 0;
  int rc = get_list(c, *list, false, pending, id, &seg);
  if (rc != TQ_OK) return rc;
  return flush_builds(c, pending, &built);
}

int tq_decode_postings(tq_ctx* c, const tq_term_seg* list, uint32_t* out_docs, uint32_t* out_tfs) {
  if (!c || !list || !out_docs) return fail(TQ_ERR_INVALID_ARGUMENT, "null");
  TQ_CUDA(cudaSetDevice(c->device));
  if (list->doc_freq == 0) return TQ_OK;
  uint32_t id;
  int rc = resolve_single(c, list, &id);
  if (rc != TQ_OK) return rc;
  uint32_t *d_docs = nullptr, *d_tfs = nullptr;
  const size_t bytes = (size_t)list->doc_freq * 4;
  TQ_CUDA(cudaMalloc(&d_docs, bytes));
  TQ_CUDA(cudaMalloc(&d_tfs, bytes));
  const uint32_t n_total = list->doc_freq / 128u + ((list->doc_freq % 128u) ? 1u : 0u);
  k_decode_list<<<(n_total + kWarps - 1) / kWarps, kThreads>>>(c->d_lists, id, d_docs, d_tfs);
  cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess) e = cudaMemcpy(out_docs, d_docs, bytes, cudaMemcpyDeviceToHost);
  if (e == cudaSuccess && out_tfs) e = cudaMemcpy(out_tfs, d_tfs, bytes, cudaMemcpyDeviceToHost);
  cudaFree(d_docs); cudaFree(d_tfs);
  if (e != cudaSuccess) return fail(TQ_ERR_CUDA, cudaGetErrorString(e));
  return TQ_OK;
}

int tq_block_table(tq_ctx* c, const tq_term_seg* list, float weight, float avg_fieldnorm, uint32_t* out_last_doc, float* out_block_max) {
  if (!c || !list || !out_last_doc || !out_block_max) return fail(TQ_ERR_INVALID_ARGUMENT, "null");
  TQ_CUDA(cudaSetDevice(c->device));
  const uint32_t n = list->doc_freq / 128u;
  if (n == 0) return TQ_OK;
  uint32_t id;
  int rc = resolve_single(c, list, &id);
  if (rc != TQ_OK) return rc;
  float tab[256];
  bm25_tf_cache(avg_fieldnorm, tab);
  float *d_cache = nullptr, *d_bm = nullptr;
  uint32_t* d_last = nullptr;
  TQ_CUDA(cudaMalloc(&d_cache, 1024));
  TQ_CUDA(cudaMalloc(&d_bm, (size_t)n * 4));
  TQ_CUDA(cudaMalloc(&d_last, (size_t)n * 4));
  cudaError_t e = cudaMemcpy(d_cache, tab, 1024, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) {
    k_block_max<<<(n + 255) / 256, 256>>>(c->d_lists, id, weight, d_cache, d_last, d_bm);
    e = cudaGetLastError();
  }
  if (e == cudaSuccess) e = cudaMemcpy(out_last_doc, d_last, (size_t)n * 4, cudaMemcpyDeviceToHost);
  if (e == cudaSuccess) e = cudaMemcpy(out_block_max, d_bm, (size_t)n * 4, cudaMemcpyDeviceToHost);
  cudaFree(d_cache); cudaFree(d_bm); cudaFree(d_last);
  if (e != cudaSuccess) return fail(TQ_ERR_CUDA, cudaGetErrorString(e));
  return TQ_OK;
}

// ---- BM25 scalars --------------------------------------------------------------------------------------
float tq_bm25_idf(uint64_t doc_freq, uint64_t doc_count) { return bm25_idf(doc_freq, doc_count); }
float tq_bm25_weight(uint64_t doc_freq, uint64_t doc_count, float boost) { return bm25_weight(doc_freq, doc_count, boost); }
void tq_bm25_tf_cache(float avg_fieldnorm, float out[256]) { bm25_tf_cache(avg_fieldnorm, out); }
uint32_t tq_id_to_fieldnorm(uint8_t id) { return id_to_fieldnorm(id); }
uint8_t tq_fieldnorm_to_id(uint32_t fieldnorm) { return fieldnorm_to_id(fieldnorm); }

// ---- segment writer ----------------------------------------------------------------------------------
struct tq_field_writer {
  uint32_t max_doc = 0;
  std::vector<uint8_t> fieldnorm_ids;
  FieldPostingsWriter* w = nullptr;
};

int tq_field_writer_create(int record_option, uint64_t total_num_tokens, const uint8_t* fieldnorm_ids, uint32_t max_doc, tq_field_writer** out) {
  if (!out || record_option < 0 || record_option > 2) return fail(TQ_ERR_INVALID_ARGUMENT, "args");
  auto* fw = new tq_field_writer();
  fw->max_doc = max_doc;
  if (fieldnorm_ids) fw->fieldnorm_ids.assign(fieldnorm_ids, fieldnorm_ids + max_doc);
  fw->w = new FieldPostingsWriter(record_option, total_num_tokens, fieldnorm_ids ? fw->fieldnorm_ids.data() : nullptr, max_doc);
  *out = fw;
  return TQ_OK;
}
int tq_field_writer_add_term(tq_field_writer* fw, const uint32_t* docs, const uint32_t* tfs, uint32_t doc_freq, uint64_t* postings_start,
                             uint64_t* postings_end) {
  if (!fw || (!docs && doc_freq)) return fail(TQ_ERR_INVALID_ARGUMENT, "args");
  for (uint32_t i = 0; i < doc_freq; ++i) {
    if (i && docs[i] <= docs[i - 1]) return fail(TQ_ERR_INVALID_ARGUMENT, "docs must be strictly ascending");
    if (docs[i] >= TQ_TERMINATED || docs[i] >= fw->max_doc) return fail(TQ_ERR_INVALID_ARGUMENT, "doc id out of range (>= max_doc)");
    if (tfs && tfs[i] == 0) return fail(TQ_ERR_INVALID_ARGUMENT, "term frequency 0");
  }
  const TermInfoOut ti = fw->w->add_term(docs, tfs, doc_freq);
  if (postings_start) *postings_start = ti.postings_start;
  if (postings_end) *postings_end = ti.postings_end;
  return TQ_OK;
}
int tq_field_writer_body(tq_field_writer* fw, const uint8_t** body, size_t* len) {
  if (!fw || !body || !len) return fail(TQ_ERR_INVALID_ARGUMENT, "args");
  *body = fw->w->body().data();
  *len = fw->w->body().size();
  return TQ_OK;
}
void tq_field_writer_destroy(tq_field_writer* fw) {
  if (!fw) return;
  delete fw->w;
  delete fw;
}

}  // extern "C"

// ---- several GPUs behind one handle -------------------------------------------------------------------------------------
// The reference fans a search out over segments inside one process (Executor::map, src/core/executor.rs:60-100;
// Searcher::search_with_executor, src/core/searcher.rs:220-237).  tq_multi is that shape for GPUs: one tq_ctx per device,
// every segment lives on one of them, a search runs the devices' shares concurrently (one host thread per device), exchanges
// the exact k-th best score keys between the phases (so that every device prunes like a single device holding everything),
// and merges the per-device rows on the host (merge_fruits / merge_top_k, sort_key_top_collector.rs:54-95).
#include <condition_variable>
#include <thread>

struct tq_multi {
  std::vector<tq_ctx*> ctxs;
  std::map<std::pair<uint32_t, uint32_t>, std::vector<int>> owner;  // (segment_ord, field) -> indices into ctxs (several: the segment is split by doc range)
  std::vector<uint64_t> load;                           // bytes registered per device
  std::mutex mu;
  std::string err;
};

namespace {
struct HostBarrier {
  std::mutex m;
  std::condition_variable cv;
  int n, waiting = 0;
  uint64_t gen = 0;
  explicit HostBarrier(int n_) : n(n_) {}
  template <class F> void arrive(F&& last) {  // `last` runs on exactly one thread while the others wait
    std::unique_lock<std::mutex> lk(m);
    const uint64_t g = gen;
    if (++waiting == n) { last(); waiting = 0; ++gen; cv.notify_all(); }
    else cv.wait(lk, [&] { return gen != g; });
  }
};
}  // namespace

extern "C" {

int tq_multi_create(const int* devices, int n_devices, tq_multi** out) {
  if (!devices || n_devices <= 0 || !out) return fail(TQ_ERR_INVALID_ARGUMENT, "devices");
  auto* m = new tq_multi();
  for (int i = 0; i < n_devices; ++i) {
    tq_ctx* c = nullptr;
    const int rc = tq_ctx_create(devices[i], &c);
    if (rc != TQ_OK) { for (auto* x : m->ctxs) tq_ctx_destroy(x); delete m; return rc; }
    m->ctxs.push_back(c);
  }
  m->load.assign(n_devices, 0);
  *out = m;
  return TQ_OK;
}

void tq_multi_destroy(tq_multi* m) {
  if (!m) return;
  for (auto* c : m->ctxs) tq_ctx_destroy(c);
  delete m;
}

const char* tq_multi_last_error(tq_multi* m) { return m ? m->err.c_str() : g_err.c_str(); }

int tq_multi_num_devices(tq_multi* m) { return m ? (int)m->ctxs.size() : 0; }

int tq_multi_segment_register(tq_multi* m, int device_index, uint32_t segment_ord, uint32_t field, uint32_t max_doc, int record_option,
                              const uint8_t* idx_body, size_t idx_len, const uint8_t* fieldnorm, size_t fieldnorm_len,
                              const uint8_t* alive_bitset, size_t alive_len) {
  if (!m) return fail(TQ_ERR_INVALID_ARGUMENT, "null");
  std::lock_guard<std::mutex> g(m->mu);
  if (device_index >= (int)m->ctxs.size()) { m->err = "device_index"; return TQ_ERR_INVALID_ARGUMENT; }
  if (device_index < 0) {  // least loaded device: segments shard naturally (SURVEY.md §8e)
    device_index = 0;
    for (size_t i = 1; i < m->load.size(); ++i) if (m->load[i] < m->load[device_index]) device_index = (int)i;
  }
  const int rc = tq_segment_register(m->ctxs[device_index], segment_ord, field, max_doc, record_option, idx_body, idx_len, fieldnorm, fieldnorm_len,
                                     alive_bitset, alive_len);
  if (rc != TQ_OK) { m->err = g_err; return rc; }
  m->owner[{segment_ord, field}] = std::vector<int>{device_index};
  m->load[device_index] += idx_len + fieldnorm_len;
  return TQ_OK;
}

// One segment over ALL devices of the handle, device i evaluating the docs [i, i + 1) * ceil(max_doc / n / 1024) * 1024 (whole
// tiles of the tile engine): the intra-segment split of SURVEY.md §8(e) for an index of one (or few) huge segments.
int tq_multi_segment_register_split(tq_multi* m, uint32_t segment_ord, uint32_t field, uint32_t max_doc, int record_option,
                                    const uint8_t* idx_body, size_t idx_len, const uint8_t* fieldnorm, size_t fieldnorm_len,
                                    const uint8_t* alive_bitset, size_t alive_len) {
  if (!m) return fail(TQ_ERR_INVALID_ARGUMENT, "null");
  std::lock_guard<std::mutex> g(m->mu);
  const uint32_t nd = (uint32_t)m->ctxs.size();
  const uint32_t per = (uint32_t)((((uint64_t)max_doc + nd - 1) / nd + kTile - 1) / kTile * kTile);
  std::vector<int> owners;
  for (uint32_t d = 0; d < nd; ++d) {
    const uint32_t lo = (uint32_t)std::min<uint64_t>((uint64_t)d * per, max_doc), hi = (uint32_t)std::min<uint64_t>((uint64_t)(d + 1) * per, max_doc);
    int rc = tq_segment_register(m->ctxs[d], segment_ord, field, max_doc, record_option, idx_body, idx_len, fieldnorm, fieldnorm_len, alive_bitset, alive_len);
    if (rc == TQ_OK) rc = tq_segment_set_doc_range(m->ctxs[d], segment_ord, field, lo, hi);
    if (rc != TQ_OK) {
      m->err = g_err;
      tq_segment_unregister(m->ctxs[d], segment_ord, field);
      for (int o : owners) tq_segment_unregister(m->ctxs[o], segment_ord, field);
      g_err = m->err;
      return rc;
    }
    owners.push_back((int)d);
    m->load[d] += idx_len + fieldnorm_len;
  }
  m->owner[{segment_ord, field}] = owners;
  return TQ_OK;
}

int tq_multi_search_batch(tq_multi* m, const tq_query* queries, size_t nq, uint32_t out_stride, float* out_scores, uint32_t* out_segment_ord,
                          uint32_t* out_doc, uint32_t* out_count) {
  if (!m || (!queries && nq) || !out_scores || !out_segment_ord || !out_doc || !out_count) return fail(TQ_ERR_INVALID_ARGUMENT, "null");
  const int nd = (int)m->ctxs.size();
  uint32_t kmax = 1;
  for (size_t q = 0; q < nq; ++q) kmax = std::max(kmax, queries[q].k);
  // every device's share of every query: the (clause, segment) lists of the segments it owns
  std::vector<std::vector<tq_query>> dq(nd, std::vector<tq_query>(queries, queries + nq));
  std::vector<std::vector<tq_term_seg>> dts(nd);
  {
    std::lock_guard<std::mutex> g(m->mu);
    std::vector<std::vector<size_t>> first(nd, std::vector<size_t>(nq + 1, 0));
    for (size_t q = 0; q < nq; ++q) {
      for (int d = 0; d < nd; ++d) first[d][q] = dts[d].size();
      for (uint32_t i = 0; i < queries[q].n_term_segs; ++i) {
        const tq_term_seg& ts = queries[q].term_segs[i];
        auto it = m->owner.find({ts.segment_ord, ts.field});
        if (it == m->owner.end()) { m->err = "term_seg names a segment/field that is not registered"; return TQ_ERR_NOT_FOUND; }
        for (int d : it->second) dts[d].push_back(ts);
      }
    }
    for (int d = 0; d < nd; ++d) {
      first[d][nq] = dts[d].size();
      for (size_t q = 0; q < nq; ++q) {
        dq[d][q].term_segs = dts[d].data() + first[d][q];
        dq[d][q].n_term_segs = (uint32_t)(first[d][q + 1] - first[d][q]);
      }
    }
  }
  const size_t rows = std::max<size_t>(nq, 1) * kmax;
  std::vector<std::vector<float>> r_sc(nd, std::vector<float>(rows));
  std::vector<std::vector<uint32_t>> r_sg(nd, std::vector<uint32_t>(rows)), r_dc(nd, std::vector<uint32_t>(rows)), r_ct(nd, std::vector<uint32_t>(std::max<size_t>(nq, 1)));
  std::vector<std::vector<uint32_t>> keys(nd, std::vector<uint32_t>(rows));  // [device][query][kmax] best keys so far
  std::vector<long long> bound(std::max<size_t>(nq, 1), 0);                   // exact k-th best of the union, per query
  std::vector<int> rcs(nd, TQ_OK);
  std::vector<std::string> errs(nd);
  HostBarrier bar(nd);
  bool abort_all = false;
  auto worker = [&](int d) {
    tq_batch* b = nullptr;
    uint32_t* d_keys = nullptr;
    long long* d_bound = nullptr;
    int rc = tq_batch_prepare(m->ctxs[d], dq[d].data(), nq, &b);
    if (rc == TQ_OK && (cudaMalloc(&d_keys, rows * 4) != cudaSuccess || cudaMalloc(&d_bound, std::max<size_t>(nq, 1) * 8) != cudaSuccess)) rc = fail(TQ_ERR_OOM, "exchange buffers");
    const int phases = kPhases;
    for (int p = 0; p < phases; ++p) {
      if (rc == TQ_OK) rc = tq_batch_run_phase(b, p);
      if (p + 1 == phases) break;
      if (rc == TQ_OK) rc = tq_batch_topkeys_export_dev(b, d_keys, kmax);
      if (rc == TQ_OK && (cudaMemcpyAsync(keys[d].data(), d_keys, rows * 4, cudaMemcpyDeviceToHost, b->stream) != cudaSuccess ||
                          cudaStreamSynchronize(b->stream) != cudaSuccess)) rc = fail(TQ_ERR_CUDA, "key export");
      if (rc != TQ_OK) { std::lock_guard<std::mutex> g(m->mu); abort_all = true; }
      bar.arrive([&] {  // one thread: the exact k-th best key of the union of all devices' keys
        std::vector<uint32_t> all((size_t)nd * kmax);
        for (size_t q = 0; q < nq; ++q) {
          for (int e = 0; e < nd; ++e) memcpy(all.data() + (size_t)e * kmax, keys[e].data() + q * kmax, (size_t)kmax * 4);
          const uint32_t k = queries[q].k;
          std::nth_element(all.begin(), all.begin() + (k - 1), all.end(), std::greater<uint32_t>());
          bound[q] = (long long)all[k - 1];
        }
      });
      if (abort_all) { if (rc == TQ_OK) rc = TQ_ERR_CUDA; break; }
      if (rc == TQ_OK && cudaMemcpyAsync(d_bound, bound.data(), nq * 8, cudaMemcpyHostToDevice, b->stream) != cudaSuccess) rc = fail(TQ_ERR_CUDA, "bound import");
      if (rc == TQ_OK && nq) rc = tq_batch_thresholds_import_dev(b, reinterpret_cast<const int64_t*>(d_bound));
    }
    if (rc == TQ_OK) rc = tq_batch_fetch(b, kmax, r_sc[d].data(), r_sg[d].data(), r_dc[d].data(), r_ct[d].data());
    if (rc != TQ_OK) errs[d] = g_err;
    rcs[d] = rc;
    if (b) tq_batch_destroy(b);
    cudaFree(d_keys);
    cudaFree(d_bound);
  };
  std::vector<std::thread> th;
  for (int d = 0; d < nd; ++d) th.emplace_back(worker, d);
  for (auto& t : th) t.join();
  for (int d = 0; d < nd; ++d)
    if (rcs[d] != TQ_OK) { m->err = errs[d]; g_err = errs[d]; return rcs[d]; }
  // merge_fruits: (score desc, segment_ord asc, doc asc), keep k (top_score_collector.rs:591-600)
  struct Row { float s; uint32_t g, d; };
  std::vector<Row> all;
  for (size_t q = 0; q < nq; ++q) {
    all.clear();
    for (int d = 0; d < nd; ++d) {
      const uint32_t n = std::min(r_ct[d][q], kmax);
      for (uint32_t i = 0; i < n; ++i) all.push_back(Row{r_sc[d][q * kmax + i], r_sg[d][q * kmax + i], r_dc[d][q * kmax + i]});
    }
    std::sort(all.begin(), all.end(), [](const Row& a, const Row& b) {
      if (a.s != b.s) return a.s > b.s;
      if (a.g != b.g) return a.g < b.g;
      return a.d < b.d;
    });
    const uint32_t n = (uint32_t)std::min<size_t>(all.size(), queries[q].k);
    out_count[q] = n;
    for (uint32_t i = 0; i < std::min(n, out_stride); ++i) {
      out_scores[q * out_stride + i] = all[i].s;
      out_segment_ord[q * out_stride + i] = all[i].g;
      out_doc[q * out_stride + i] = all[i].d;
    }
  }
  return TQ_OK;
}

}  // extern "C"
