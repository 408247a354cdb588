// Tests of the C++ host mirror (tantivy_b200/host/tantivy_host.hpp), written in the shape of the reference's own
// tests for this path.  Every test names the reference test it restates; the expected scores are the reference's.
//
//   host_mirror_tests               run every search test on cuda:0 (needs a GPU)
//   host_mirror_tests --dump DIR    write the segment bytes of every test index under DIR (CPU only; the Python
//                                   suite feeds them to the oracle and checks the same golden scores there)
//   host_mirror_tests --cpu         host-only checks: tokenizer, fieldnorms, statistics, file framing, error kinds,
//                                   and that a search without a CUDA device raises (no CPU fallback; with one, it answers)
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <fstream>
#include <functional>
#include <iostream>
#include <sstream>

#include "../../tantivy_b200/host/tantivy_host.hpp"

using namespace tantivy_b200;

static int g_failed = 0;
#define CHECK(cond)                                                                  \
  do {                                                                               \
    if (!(cond)) {                                                                   \
      std::printf("    CHECK failed %s:%d: %s\n", __FILE__, __LINE__, #cond);        \
      ++g_failed;                                                                    \
    }                                                                                \
  } while (0)
// the reference's assert_nearly_equals! uses |l - r| <= 0.0005 (src/lib.rs:406-427); this port is 500x tighter
#define CHECK_NEARLY(left, right)                                                                              \
  do {                                                                                                         \
    const double l_ = (left), r_ = (right);                                                                    \
    if (!(std::fabs(l_ - r_) <= 1e-6 * std::max(std::fabs(l_), std::fabs(r_)))) {                                 \
      std::printf("    CHECK_NEARLY failed %s:%d: %.9g vs %.9g\n", __FILE__, __LINE__, l_, r_);               \
      ++g_failed;                                                                                              \
    }                                                                                                          \
  } while (0)

static Document doc(Field f, const std::string& text) {
  Document d;
  d.add_text(f, text);
  return d;
}
static QueryBox term_query(Field f, const std::string& text, IndexRecordOption opt) {
  return std::make_unique<TermQuery>(Term::from_field_text(f, text), opt);
}

// ---- index builders shared by the search tests and by --dump -------------------------------------------------
struct Named { std::string name; Index index; };

// term_query/mod.rs:21-44
static Index index_one_doc_string() {
  SchemaBuilder sb;
  Field text = sb.add_text_field("text", STRING);
  Index index = Index::create_in_ram(sb.build());
  IndexWriter w = index.writer_for_tests();
  w.add_document(doc(text, "a"));
  w.commit();
  return index;
}
// term_query/mod.rs:46-78
static Index index_block_len_docs() {
  SchemaBuilder sb;
  Field text = sb.add_text_field("text", STRING);
  Index index = Index::create_in_ram(sb.build());
  IndexWriter w = index.writer_for_tests();
  for (int i = 0; i < 128; ++i) w.add_document(doc(text, "a"));
  w.commit();
  return index;
}
// term_query/mod.rs:80-100
static Index index_term_weight() {
  SchemaBuilder sb;
  Field left = sb.add_text_field("left", TEXT);
  Field right = sb.add_text_field("right", TEXT);
  Field large = sb.add_text_field("large", TEXT);
  Index index = Index::create_in_ram(sb.build());
  IndexWriter w = index.writer_for_tests();
  std::string big;
  for (int i = 0; i <= 286; ++i) big += (i ? " large" : "large") + std::to_string(i);
  Document d;
  d.add_text(left, "left1 left2 left2 left2f2 left2f2 left3 abcde abcde abcde abcde abcde abcde abcde abcde abcde abcewde abcde abcde");
  d.add_text(right, "right1 right2");
  d.add_text(large, big);
  w.add_document(d);
  w.add_document(doc(left, "left4 left1"));
  w.commit();
  return index;
}
// boolean_query/mod.rs:27-44 (aux_test_helper)
static Index index_boolean_aux() {
  SchemaBuilder sb;
  Field text = sb.add_text_field("text", TEXT);
  Index index = Index::create_in_ram(sb.build());
  IndexWriter w = index.writer_for_tests();
  for (const char* t : {"a b c", "a c", "b c", "a b c d", "d"}) w.add_document(doc(text, t));
  w.commit();
  return index;
}
// boolean_query/mod.rs:221-233
static Index index_boolean_weight() {
  SchemaBuilder sb;
  Field text = sb.add_text_field("text", TEXT);
  Index index = Index::create_in_ram(sb.build());
  IndexWriter w = index.writer_for_tests();
  for (const char* t : {"a b c", "a c", "b c"}) w.add_document(doc(text, t));
  w.commit();
  return index;
}
// top_score_collector.rs:718-729 (make_index)
static Index index_droopy() {
  SchemaBuilder sb;
  Field text = sb.add_text_field("text", TEXT);
  Index index = Index::create_in_ram(sb.build());
  IndexWriter w = index.writer_for_tests();
  w.add_document(doc(text, "Hello happy tax payer."));
  w.add_document(doc(text, "Droopy says hello happy tax payer"));
  w.add_document(doc(text, "I like Droopy"));
  w.commit();
  return index;
}
// several commits -> several segments, a delete in between, multi-block lists with tf > 1
static Index index_multi_segment() {
  SchemaBuilder sb;
  Field body = sb.add_text_field("body", TEXT);
  Index index = Index::create_in_ram(sb.build());
  IndexWriter w = index.writer_for_tests();
  uint32_t x = 12345;
  auto next = [&]() { x = x * 1664525u + 1013904223u; return x >> 8; };
  for (int seg = 0; seg < 3; ++seg) {
    for (int d = 0; d < 700 + 111 * seg; ++d) {
      std::string t = "w" + std::to_string(next() % 7);
      const int len = 1 + (int)(next() % 30);
      for (int i = 0; i < len; ++i) t += " w" + std::to_string(next() % (4 + 13 * (i % 3)));
      if (next() % 5 == 0) t += " rare";
      w.add_document(doc(body, t));
    }
    if (seg == 1) w.delete_term(Term::from_field_text(body, "rare"));
    w.commit();
  }
  return index;
}

// phrase_query/mod.rs:24-38 create_index(texts): one TEXT field "text", one doc per text, one commit
static Index index_from_texts(std::initializer_list<const char*> texts) {
  SchemaBuilder sb;
  Field text = sb.add_text_field("text", TEXT);
  Index index = Index::create_in_ram(sb.build());
  IndexWriter w = index.writer_for_tests();
  for (const char* t : texts) w.add_document(doc(text, t));
  w.commit();
  return index;
}

static std::vector<Named> all_indexes() {
  std::vector<Named> v;
  // the indexes of the reference's phrase tests (phrase_query/mod.rs:41-275): dumped for the oracle's PhraseScorer
  v.push_back({"phrase_query", index_from_texts({"b b b d c g c", "a b b d c g c", "a b a b c", "c a b a d ga a", "a b c"})});
  v.push_back({"phrase_simple", index_from_texts({"a b b d c g c", "a b a b c"})});
  v.push_back({"phrase_score", index_from_texts({"a b c", "a b c a b"})});
  v.push_back({"phrase_slop_bug", index_from_texts({"asdf asdf Captain Subject Wendy", "Captain"})});
  v.push_back({"phrase_slop_bug_2a", index_from_texts({"a x b x c", "a a c"})});
  v.push_back({"phrase_slop_bug_2b", index_from_texts({"a x b x c", "b c c"})});
  v.push_back({"phrase_slop_repeating", index_from_texts({"wendy subject subject captain", "Captain"})});
  v.push_back({"phrase_slop_size", index_from_texts({"a b e c", "a e e e c", "a e e e e c"})});
  v.push_back({"phrase_slop_1", index_from_texts({"a x b c"})});
  v.push_back({"phrase_slop_2", index_from_texts({"a x b x c"})});
  v.push_back({"phrase_slop_3", index_from_texts({"a b"})});
  v.push_back({"phrase_slop_ordering", index_from_texts({"a e b e c", "a e e e e e b e e e e c", "a c b", "a c e b e", "a e c b", "a e b c"})});
  v.push_back({"one_doc_string", index_one_doc_string()});
  v.push_back({"block_len_docs", index_block_len_docs()});
  v.push_back({"term_weight", index_term_weight()});
  v.push_back({"boolean_aux", index_boolean_aux()});
  v.push_back({"boolean_weight", index_boolean_weight()});
  v.push_back({"droopy", index_droopy()});
  v.push_back({"multi_segment", index_multi_segment()});
  return v;
}

// ---- search tests (GPU) --------------------------------------------------------------------------------------------
static void test_term_query_no_freq() {  // term_query/mod.rs:21-44
  Index index = index_one_doc_string();
  Field text = *index.schema().get_field("text");
  Searcher searcher = index.reader().searcher();
  TermQuery q(Term::from_field_text(text, "a"), IndexRecordOption::Basic);
  auto top = searcher.search(q, TopDocs::with_limit(1));
  CHECK(top.size() == 1);
  CHECK(top[0].second == DocAddress(0, 0));
  CHECK_NEARLY(top[0].first, 0.28768212);
}

static void test_term_query_multiple_of_block_len() {  // term_query/mod.rs:46-78: the scorer visits docs 0..127, then TERMINATED
  Index index = index_block_len_docs();
  Field text = *index.schema().get_field("text");
  Searcher searcher = index.reader().searcher();
  TermQuery q(Term::from_field_text(text, "a"), IndexRecordOption::Basic);
  auto top = searcher.search(q, TopDocs::with_limit(200));
  CHECK(top.size() == 128);
  for (uint32_t i = 0; i < top.size(); ++i) CHECK(top[i].second == DocAddress(0, i));  // equal scores: ascending doc
}

static void test_term_weight() {  // term_query/mod.rs:80-129
  Index index = index_term_weight();
  Field left = *index.schema().get_field("left");
  Searcher searcher = index.reader().searcher();
  {
    TermQuery q(Term::from_field_text(left, "left2"), IndexRecordOption::WithFreqs);
    auto top = searcher.search(q, TopDocs::with_limit(2).order_by_score());
    CHECK(top.size() == 1);
    CHECK_NEARLY(top[0].first, 0.77802235);
  }
  {
    TermQuery q(Term::from_field_text(left, "left1"), IndexRecordOption::WithFreqs);
    auto top = searcher.search(q, TopDocs::with_limit(2).order_by_score());
    CHECK(top.size() == 2);
    CHECK_NEARLY(top[0].first, 0.27101856);
    CHECK_NEARLY(top[1].first, 0.13736556);
  }
  {
    QueryParser parser = QueryParser::for_index(index, {});
    QueryBox q = parser.parse_query("left:left2 left:left1");
    auto top = searcher.search(*q, TopDocs::with_limit(2).order_by_score());
    CHECK(top.size() == 2);
    CHECK_NEARLY(top[0].first, 0.9153879);
    CHECK_NEARLY(top[1].first, 0.27101856);
  }
}

static void test_boolean_query_with_weight() {  // boolean_query/mod.rs:221-259
  Index index = index_boolean_weight();
  Field text = *index.schema().get_field("text");
  Searcher searcher = index.reader().searcher();
  std::vector<std::pair<Occur, QueryBox>> clauses;
  clauses.emplace_back(Occur::Should, term_query(text, "a", IndexRecordOption::WithFreqs));
  clauses.emplace_back(Occur::Should, term_query(text, "b", IndexRecordOption::WithFreqs));
  BooleanQuery q(std::move(clauses));
  {
    auto top = searcher.search(q, TopDocs::with_limit(3));
    CHECK(top.size() == 3);
    CHECK(top[0].second == DocAddress(0, 0));
    CHECK_NEARLY(top[0].first, 0.84163445);
  }
  {  // boolean_weight.scorer(reader, 2.0): the boost multiplies every clause's weight
    BoostQuery boosted(q.box_clone(), 2.0f);
    auto top = searcher.search(boosted, TopDocs::with_limit(3));
    CHECK(top[0].second == DocAddress(0, 0));
    CHECK_NEARLY(top[0].first, 1.6832689);
  }
}

static void test_intersection_score() {  // boolean_query/mod.rs:262-291
  Index index = index_boolean_aux();
  Field text = *index.schema().get_field("text");
  Searcher searcher = index.reader().searcher();
  std::vector<std::pair<Occur, QueryBox>> clauses;
  clauses.emplace_back(Occur::Must, term_query(text, "a", IndexRecordOption::Basic));
  clauses.emplace_back(Occur::Must, term_query(text, "b", IndexRecordOption::Basic));
  BooleanQuery q(std::move(clauses));
  auto top = searcher.search(q, TopDocs::with_limit(10));
  CHECK(top.size() == 2);
  CHECK(top[0].second == DocAddress(0, 0));
  CHECK_NEARLY(top[0].first, 0.977973);
  CHECK(top[1].second == DocAddress(0, 3));
  CHECK_NEARLY(top[1].first, 0.84699446);
}

static void check_results(const std::vector<std::pair<Score, DocAddress>>& got, const std::vector<std::pair<Score, DocAddress>>& want) {
  CHECK(got.size() == want.size());
  for (size_t i = 0; i < std::min(got.size(), want.size()); ++i) {
    CHECK(got[i].second == want[i].second);
    CHECK_NEARLY(got[i].first, want[i].first);
  }
}

static void test_top_collector() {  // top_score_collector.rs:838-921 (the four capacity / offset cases)
  Index index = index_droopy();
  Field text = *index.schema().get_field("text");
  QueryBox q = QueryParser::for_index(index, {text}).parse_query("droopy tax");
  Searcher searcher = index.reader().searcher();
  check_results(searcher.search(*q, TopDocs::with_limit(4).order_by_score()),
                {{0.81221175f, DocAddress(0, 1)}, {0.5376842f, DocAddress(0, 2)}, {0.48527452f, DocAddress(0, 0)}});
  check_results(searcher.search(*q, TopDocs::with_limit(4).and_offset(2).order_by_score()), {{0.48527452f, DocAddress(0, 0)}});
  check_results(searcher.search(*q, TopDocs::with_limit(2).order_by_score()),
                {{0.81221175f, DocAddress(0, 1)}, {0.5376842f, DocAddress(0, 2)}});
  check_results(searcher.search(*q, TopDocs::with_limit(2).and_offset(1).order_by_score()),
                {{0.5376842f, DocAddress(0, 2)}, {0.48527452f, DocAddress(0, 0)}});
}

static void test_multi_segment_deletes_and_paging() {
  // top_score_collector.rs:923-957 (stable sorting: growing pages are prefixes of each other), on three segments
  // with deleted docs; and Searcher statistics (searcher.rs:133-141, bm25.rs:27-50)
  Index index = index_multi_segment();
  Field body = *index.schema().get_field("body");
  Searcher searcher = index.reader().searcher();
  CHECK(searcher.segment_readers().size() == 3);
  CHECK(searcher.total_num_docs() == 700 + 811 + 922);
  CHECK(searcher.num_docs() < searcher.total_num_docs());
  CHECK(searcher.segment_reader(2).num_deleted_docs() == 0);  // the delete preceded the third commit's docs
  const Term rare = Term::from_field_text(body, "rare");
  CHECK(searcher.doc_freq(rare) > 0);  // doc_freq still counts deleted docs
  {
    TermQuery q(rare, IndexRecordOption::WithFreqs);
    auto top = searcher.search(q, TopDocs::with_limit(1000));
    CHECK(!top.empty());
    for (auto& h : top) CHECK(h.second.segment_ord == 2);  // every "rare" doc of segments 0 and 1 is deleted
    CHECK(top.size() == searcher.segment_reader(2).inverted_index(body).doc_freq(rare));
  }
  std::vector<std::pair<Occur, QueryBox>> clauses;
  for (const char* t : {"w0", "w3", "w11"}) clauses.emplace_back(Occur::Should, term_query(body, t, IndexRecordOption::WithFreqs));
  BooleanQuery q(std::move(clauses));
  auto page3 = searcher.search(q, TopDocs::with_limit(300));
  auto page2 = searcher.search(q, TopDocs::with_limit(120));
  auto tail = searcher.search(q, TopDocs::with_limit(100).and_offset(200));
  CHECK(page3.size() == 300 && page2.size() == 120 && tail.size() == 100);
  for (size_t i = 0; i < page2.size(); ++i) CHECK(page2[i] == page3[i]);
  for (size_t i = 0; i < tail.size(); ++i) CHECK(tail[i] == page3[200 + i]);
  for (size_t i = 1; i < page3.size(); ++i)  // (score desc, DocAddress asc), top_score_collector.rs:591-600
    CHECK(page3[i - 1].first > page3[i].first || (page3[i - 1].first == page3[i].first && page3[i - 1].second < page3[i].second));
  for (auto& h : page3) CHECK(!searcher.segment_reader(h.second.segment_ord).is_deleted(h.second.doc_id));
  // the same queries as one device batch give the same rows
  TermQuery tq1(rare, IndexRecordOption::WithFreqs);
  auto batch = searcher.search_batch({&q, &tq1, &q}, TopDocs::with_limit(120));
  CHECK(batch.size() == 3 && batch[0] == page2 && batch[2] == page2);
  // a conjunction never returns more than its rarest clause
  std::vector<std::pair<Occur, QueryBox>> must;
  must.emplace_back(Occur::Must, term_query(body, "rare", IndexRecordOption::WithFreqs));
  must.emplace_back(Occur::Must, term_query(body, "w1", IndexRecordOption::WithFreqs));
  auto both = searcher.search(BooleanQuery(std::move(must)), TopDocs::with_limit(1000));
  CHECK(!both.empty() && both.size() <= searcher.doc_freq(rare));
}

static void test_count_collector() {  // boolean_query/mod.rs:46-75 shapes on the aux index: searcher.search(&query, &Count)
  Index index = index_boolean_aux();   // docs: "a b c", "a c", "b c", "a b c d", "d"
  Field text = *index.schema().get_field("text");
  Searcher searcher = index.reader().searcher();
  QueryParser parser = QueryParser::for_index(index, {text});
  CHECK(searcher.search(*parser.parse_query("+a"), Count{}) == 3);
  CHECK(searcher.search(*parser.parse_query("+a +b"), Count{}) == 2);
  CHECK(searcher.search(*parser.parse_query("a d"), Count{}) == 4);
  CHECK(searcher.search(*parser.parse_query("a b c d"), Count{}) == 5);
  CHECK(searcher.search(*parser.parse_query("+a +d"), Count{}) == 1);
  CHECK(searcher.search(*parser.parse_query("zzz"), Count{}) == 0);
  Index multi = index_multi_segment();  // deletes in two of the three segments
  Field body = *multi.schema().get_field("body");
  Searcher s2 = multi.reader().searcher();
  const Term rare = Term::from_field_text(body, "rare");
  const size_t alive_rare = s2.search(TermQuery(rare, IndexRecordOption::Basic), Count{});
  CHECK(alive_rare == s2.segment_reader(2).inverted_index(body).doc_freq(rare));  // segments 0 and 1 lost theirs
  CHECK(alive_rare < s2.doc_freq(rare));
  auto top = s2.search(TermQuery(Term::from_field_text(body, "w5"), IndexRecordOption::WithFreqs), TopDocs::with_limit(1000));
  CHECK(top.size() == std::min<size_t>(1000, s2.search(TermQuery(Term::from_field_text(body, "w5"), IndexRecordOption::Basic), Count{})));
}

static void test_absent_terms_and_unsupported_shapes() {
  Index index = index_boolean_aux();
  Field text = *index.schema().get_field("text");
  Searcher searcher = index.reader().searcher();
  CHECK(searcher.search(TermQuery(Term::from_field_text(text, "zzz"), IndexRecordOption::WithFreqs), TopDocs::with_limit(5)).empty());
  CHECK(searcher.search(BooleanQuery(), TopDocs::with_limit(5)).empty());
  {
    std::vector<std::pair<Occur, QueryBox>> c;  // a Must clause without postings: nothing matches
    c.emplace_back(Occur::Must, term_query(text, "a", IndexRecordOption::WithFreqs));
    c.emplace_back(Occur::Must, term_query(text, "zzz", IndexRecordOption::WithFreqs));
    CHECK(searcher.search(BooleanQuery(std::move(c)), TopDocs::with_limit(5)).empty());
  }
  auto throws = [&](const Query& q, TantivyError::Kind kind) {
    try {
      searcher.search(q, TopDocs::with_limit(5));
    } catch (const TantivyError& e) {
      return e.kind() == kind;
    }
    return false;
  };
  {
    std::vector<std::pair<Occur, QueryBox>> c;  // boolean_query/mod.rs:186-216 shapes stay on the reference's CPU path
    c.emplace_back(Occur::Must, term_query(text, "d", IndexRecordOption::Basic));
    c.emplace_back(Occur::MustNot, term_query(text, "a", IndexRecordOption::Basic));
    CHECK(throws(BooleanQuery(std::move(c)), TantivyError::Unsupported));
  }
  {
    QueryBox mixed = QueryParser::for_index(index, {text}).parse_query("+a b");
    CHECK(throws(*mixed, TantivyError::Unsupported));
  }
  bool limit_zero = false;
  try { TopDocs::with_limit(0); } catch (const TantivyError& e) { limit_zero = e.kind() == TantivyError::InvalidArgument; }
  CHECK(limit_zero);
}

// ---- host-only checks ------------------------------------------------------------------------------------------------
static void test_host_tokenizer_and_statistics() {
  auto toks = tokenize("default", "Hello, happy tax-payer! ÜBER x" + std::string(45, 'y') + " Z9");
  // "x" + 45 x 'y' is dropped by RemoveLongFilter(40); only ASCII letters are lower-cased (the U-umlaut's bytes stay)
  CHECK((toks == std::vector<std::string>{"hello", "happy", "tax", "payer", "\xC3\x9C" "ber", "z9"}));
  CHECK(tokenize("raw", "Hello World").size() == 1);
  {  // two values of one field: positions of the second value start POSITION_GAP = 1 after the first (postings_writer.rs:19,162)
    SchemaBuilder sb;
    Field f = sb.add_text_field("f", TEXT);
    Index ix = Index::create_in_ram(sb.build());
    IndexWriter w = ix.writer_for_tests();
    w.add_document(Document().add_text(f, "a b").add_text(f, "c a"));
    w.commit();
    const FieldSegmentData& fd = ix.segments()[0]->fields[f.id];
    CHECK(fd.fieldnorms[0] == 4 && fd.total_num_tokens() == 4);
    const TermInfo a = fd.term_dict.at("a"), c = fd.term_dict.at("c");
    // "a": positions 0 and 4 -> VInt(0 blocks), VInt(0), VInt(4);  "c": position 3
    CHECK(a.positions_end - a.positions_start == 3 && fd.positions[a.positions_start] == 0x80 && fd.positions[a.positions_start + 1] == 0x80 &&
          fd.positions[a.positions_start + 2] == 0x84);
    CHECK(c.positions_end - c.positions_start == 2 && fd.positions[c.positions_start + 1] == 0x83);
  }
  Index index = index_term_weight();
  Field left = *index.schema().get_field("left"), large = *index.schema().get_field("large");
  Searcher searcher = index.reader().searcher();
  CHECK(searcher.total_num_docs() == 2 && searcher.num_docs() == 2);
  CHECK(searcher.total_num_tokens(left) == 18 + 2);
  CHECK(searcher.total_num_tokens(large) == 287);
  CHECK(searcher.doc_freq(Term::from_field_text(left, "left1")) == 2);
  CHECK(searcher.doc_freq(Term::from_field_text(left, "left2")) == 1);
  const SegmentData& seg = searcher.segment_reader(0).data();
  CHECK(seg.fields[left.id].fieldnorms[0] == 18 && seg.fields[left.id].fieldnorms[1] == 2);  // ids < 24 are exact (code.rs)
  CHECK(seg.fields[large.id].fieldnorms[0] == tq::fieldnorm_to_id(287) && seg.fields[large.id].fieldnorms[1] == 0);
  CHECK(tq::id_to_fieldnorm(seg.fields[large.id].fieldnorms[0]) == 280);  // fieldnorm/reader.rs:168-193 (300 -> 280 bucket)
  auto ti = searcher.segment_reader(0).inverted_index(left).get_term_info(Term::from_field_text(left, "abcde"));
  CHECK(ti && ti->doc_freq == 1);
  // a 1-doc list with freqs: VInt(doc delta) + VInt(tf), stop bit on the last byte (vint.rs)
  const auto& body = seg.fields[left.id].idx_body;
  CHECK(ti->postings_end - ti->postings_start == 2);
  CHECK(body[8 + ti->postings_start] == (0x80 | 0) && body[8 + ti->postings_start + 1] == (0x80 | 11));
}

// TermInfoStoreWriter restated for the test (term_info_store.rs:160-294): blocks of 256, the first entry verbatim in the
// 39-byte block meta, the others bit-packed as (postings start, positions start, doc_freq) deltas, the block's end offsets last.
static std::vector<uint8_t> write_term_info_store(const std::vector<TermInfo>& infos) {
  auto nbits = [](uint64_t v) { uint8_t n = 0; while (v) { ++n; v >>= 1; } return n; };
  std::vector<uint8_t> metas, bits;
  auto put = [](std::vector<uint8_t>& out, const void* p, size_t n) { const uint8_t* b = (const uint8_t*)p; out.insert(out.end(), b, b + n); };
  for (size_t b0 = 0; b0 < infos.size(); b0 += 256) {
    const size_t n = std::min<size_t>(256, infos.size() - b0);
    const TermInfo& ref = infos[b0];
    const TermInfo& last = infos[b0 + n - 1];
    const uint64_t post_end = last.postings_end - ref.postings_start, pos_end = last.positions_end - ref.positions_start;
    uint32_t max_df = 0;
    for (size_t i = 1; i < n; ++i) max_df = std::max(max_df, infos[b0 + i].doc_freq);
    const uint8_t df_bits = nbits(max_df), post_bits = nbits(post_end), pos_bits = nbits(pos_end);
    const uint64_t offset = bits.size();
    const uint32_t post_len = (uint32_t)(ref.postings_end - ref.postings_start), pos_len = (uint32_t)(ref.positions_end - ref.positions_start);
    put(metas, &offset, 8); put(metas, &ref.doc_freq, 4); put(metas, &ref.postings_start, 8); put(metas, &post_len, 4);
    put(metas, &ref.positions_start, 8); put(metas, &pos_len, 4);
    metas.push_back(df_bits); metas.push_back(post_bits); metas.push_back(pos_bits);
    unsigned __int128 acc = 0;  // LSB-first bit packer (tantivy_bitpacker::BitPacker)
    int filled = 0;
    auto write_bits = [&](uint64_t v, uint8_t nb) {
      acc |= (unsigned __int128)v << filled;
      filled += nb;
      while (filled >= 8) { bits.push_back((uint8_t)acc); acc >>= 8; filled -= 8; }
    };
    for (size_t i = 1; i < n; ++i) {
      write_bits(infos[b0 + i].postings_start - ref.postings_start, post_bits);
      write_bits(infos[b0 + i].positions_start - ref.positions_start, pos_bits);
      write_bits(infos[b0 + i].doc_freq, df_bits);
    }
    write_bits(post_end, post_bits);
    write_bits(pos_end, pos_bits);
    if (filled) { bits.push_back((uint8_t)acc); acc = 0; filled = 0; }  // a block ends on a byte boundary
  }
  std::vector<uint8_t> out;
  const uint64_t len = metas.size(), num = infos.size();
  put(out, &len, 8); put(out, &num, 8);
  out.insert(out.end(), metas.begin(), metas.end());
  out.insert(out.end(), bits.begin(), bits.end());
  return out;
}

static void test_host_term_info_store() {
  // term_info_store.rs:308-324 test_bitpacked: 321 in 9 bits, 2 in 2 bits, 51 in 6 bits -> 3 bytes
  const uint8_t packed[3] = {(uint8_t)(321 & 0xFF), (uint8_t)((321 >> 8) | (2 << 1) | ((51 & 0x1F) << 3)), (uint8_t)(51 >> 5)};
  CHECK(files::extract_bits(packed, 3, 0, 9) == 321 && files::extract_bits(packed, 3, 9, 2) == 2 && files::extract_bits(packed, 3, 11, 6) == 51);
  // term_info_store.rs:349-380 test_pack shape: consecutive postings / positions ranges, 1000 terms = 4 blocks
  std::vector<TermInfo> infos;
  uint64_t post = 0, pos = 0;
  uint32_t x = 7;
  for (int i = 0; i < 1000; ++i) {
    x = x * 1664525u + 1013904223u;
    TermInfo ti;
    ti.doc_freq = 1 + (x >> 8) % 5000;
    ti.postings_start = post; post += 1 + (x >> 12) % 700; ti.postings_end = post;
    ti.positions_start = pos; pos += (x >> 20) % 3000; ti.positions_end = pos;
    infos.push_back(ti);
  }
  const std::vector<uint8_t> bytes = write_term_info_store(infos);
  files::TermInfoStore store(bytes.data(), bytes.size());
  CHECK(store.num_terms() == 1000);
  bool all = true;
  for (size_t i = 0; i < infos.size(); ++i) all = all && store.get(i) == infos[i];
  CHECK(all);
  bool range = false;
  try { store.get(1000); } catch (const TantivyError& e) { range = e.kind() == TantivyError::InvalidArgument; }
  CHECK(range);
}

// No CPU fallback: the search raises SystemError exactly when no CUDA device can be opened; where one can, it answers.
static void test_host_search_without_device_raises() {
  tq_ctx* probe = nullptr;
  const bool device = tq_ctx_create(0, &probe) == TQ_OK;
  if (device) tq_ctx_destroy(probe);
  Index index = index_one_doc_string();
  Field text = *index.schema().get_field("text");
  Searcher searcher = index.reader().searcher();
  bool raised = false, answered = false;
  try {
    answered = searcher.search(TermQuery(Term::from_field_text(text, "a"), IndexRecordOption::Basic), TopDocs::with_limit(1)).size() == 1;
  } catch (const TantivyError& e) {
    raised = e.kind() == TantivyError::SystemError;
    std::printf("    (raised: %s)\n", e.what());
  }
  if (device) {
    CHECK(answered);
  } else {
    CHECK(raised);
  }
}

static std::vector<uint8_t> read_file(const std::string& path) {
  std::ifstream f(path, std::ios::binary);
  return std::vector<uint8_t>((std::istreambuf_iterator<char>(f)), std::istreambuf_iterator<char>());
}

// N1: the reference's compat fixtures (tests/compat_tests_data/index_v{6,7}, src/compat_tests.rs:39-56), handed over
// as files by the Python suite (hex in tests/golden/reference_fixtures.json): DIR/<version>/meta.json and the segment's
// files under their own names.  One doc: label = "dateformat".
static Index index_from_compat_files(const std::string& dir, const std::string& version) {
  const std::string base = dir + "/" + version + "/";
  const auto meta_bytes = read_file(base + "meta.json");
  Index index = files::open_index_in_dir(dir + "/" + version);  // Index::open_in_dir
  // the `.term` file: its framing and TermInfoStore are read (term ordinal 0 -> TermInfo); the FST that maps term
  // bytes to the ordinal is crate tantivy-fst (N2, not decoded): the dictionary has exactly one term, "dateformat"
  Field label = *index.schema().get_field("label");
  const files::IndexMeta meta = files::read_meta(std::string(meta_bytes.begin(), meta_bytes.end()));
  const auto term_file = read_file(base + meta.segments[0].file_stem() + ".term");
  const files::Footer tf = files::read_footer(term_file.data(), term_file.size());
  auto parts = files::open_composite(term_file.data(), tf.body_len);
  const files::FileSlice sl = parts.at({label.id, 0});
  const files::TermDictionaryParts dict = files::open_term_dictionary(term_file.data() + sl.offset, sl.len);
  if (dict.store.num_terms() != 1) throw TantivyError(TantivyError::DataCorruption, "compat fixture: one term expected");
  auto seg = std::make_shared<SegmentData>(*index.segments()[0]);
  seg->fields[label.id].term_dict["dateformat"] = dict.store.get(0);
  return Index::from_segments(index.schema(), {seg});
}

static void test_host_compat_framing(const std::string& dir) {
  for (const std::string version : {"index_v6", "index_v7"}) {
    const auto meta_bytes = read_file(dir + "/" + version + "/meta.json");
    const files::IndexMeta meta = files::read_meta(std::string(meta_bytes.begin(), meta_bytes.end()));
    CHECK(meta.segments.size() == 1 && meta.segments[0].max_doc == 1 && !meta.segments[0].has_deletes && meta.opstamp == 2);
    CHECK(meta.schema.num_fields() == 2);
    const FieldEntry& label = meta.schema.get_field_entry(Field{0});
    CHECK(label.name == "label" && label.options.indexing && label.options.indexing->record == IndexRecordOption::WithFreqsAndPositions &&
          label.options.indexing->fieldnorms && label.options.indexing->tokenizer == "default");
    CHECK(meta.schema.get_field_entry(Field{1}).name == "date" && !meta.schema.get_field_entry(Field{1}).options.indexing);
    const auto idx = read_file(dir + "/" + version + "/" + meta.segments[0].file_stem() + ".idx");
    CHECK(!idx.empty());
    const files::Footer f = files::read_footer(idx.data(), idx.size());
    CHECK(f.index_format_version == (version == "index_v6" ? 6u : 7u));
    auto parts = files::open_composite(idx.data(), f.body_len);
    CHECK(parts.size() == 2);  // label (text) and date fields
    Index index = index_from_compat_files(dir, version);
    const SegmentData& seg = *index.segments()[0];
    CHECK(seg.max_doc == 1 && seg.fields.size() == 2 && !seg.fields[1].indexed);
    CHECK(seg.fields[0].total_num_tokens() == 1);
    CHECK(seg.fields[0].idx_body.size() == 10 && seg.fields[0].idx_body[8] == 0x80 && seg.fields[0].idx_body[9] == 0x81);
    CHECK(seg.fields[0].fieldnorms.size() == 1 && seg.fields[0].fieldnorms[0] == 1);
    // the TermInfo read from the `.term` file: 1 doc, postings bytes 0..2, positions bytes 0..2
    const TermInfo ti = seg.fields[0].term_dict.at("dateformat");
    CHECK(ti.doc_freq == 1 && ti.postings_start == 0 && ti.postings_end == 2 && ti.positions_start == 0 && ti.positions_end == 2);
    auto corrupted = idx;
    corrupted[0] ^= 1;
    bool crc = false;
    try { files::read_footer(corrupted.data(), corrupted.size()); } catch (const TantivyError& e) { crc = e.kind() == TantivyError::DataCorruption; }
    CHECK(crc);
  }
  bool bad_meta = false;
  try { files::read_meta("{\"segments\": 3}"); } catch (const TantivyError& e) { bad_meta = e.kind() == TantivyError::DataCorruption; }
  CHECK(bad_meta);
  bool missing = false;
  try { files::open_index_in_dir(dir + "/no_such_index"); } catch (const TantivyError& e) { missing = e.kind() == TantivyError::SystemError; }
  CHECK(missing);
}

// A segment with deletes: meta.json's DeleteMeta + `<uuid>.<opstamp>.del` (BitSet::serialize + footer).  The byte layout is pinned by
// the reference's own (de)serialisation code (common/src/bitset.rs:217-224,362-367,404-409) and by alive_bitset.rs:107-156, whose
// cases are replayed here; the compat index is opened with its only doc deleted.
static void test_host_alive_bitset_file(const std::string& dir) {
  auto from_deleted = [](std::vector<uint32_t> deleted, uint32_t max_doc) {  // AliveBitSet::for_test_from_deleted_docs
    std::vector<uint8_t> w(((size_t)max_doc + 63) / 64 * 8, 0);
    for (uint32_t d = 0; d < max_doc; ++d) w[d >> 3] |= (uint8_t)(1u << (d & 7u));  // BitSet::with_max_value_and_full: padding bits stay 0
    for (uint32_t d : deleted) w[d >> 3] &= (uint8_t)~(1u << (d & 7u));
    return files::write_alive_bitset(w, max_doc);
  };
  {
    const auto file = from_deleted({1, 9}, 10);  // test_alive_bitset
    CHECK(file.size() > 12 && file[0] == 10 && file[1] == 0 && file[4] == 0xFD && file[5] == 0x01 && file[6] == 0);  // 4 + 8 bytes of body
    uint32_t alive = 0;
    const auto words = files::read_alive_bitset(file.data(), file.size(), 10, &alive);
    CHECK(words.size() == 8 && alive == 8);
    for (uint32_t d = 0; d < 10; ++d) CHECK((((words[d >> 3] >> (d & 7u)) & 1u) == 1u) == (d != 1 && d != 9));
  }
  {
    const auto file = from_deleted({0, 1, 1000}, 1001);  // test_alive_bitset_iter
    uint32_t alive = 0;
    const auto words = files::read_alive_bitset(file.data(), file.size(), 1001, &alive);
    CHECK(words.size() == 16 * 8 && alive == 998);
    bool wrong_max = false, bad_crc = false;
    try { files::read_alive_bitset(file.data(), file.size(), 1000); } catch (const TantivyError& e) { wrong_max = e.kind() == TantivyError::DataCorruption; }
    auto corrupted = file;
    corrupted[5] ^= 4;
    try { files::read_alive_bitset(corrupted.data(), corrupted.size(), 1001); } catch (const TantivyError& e) { bad_crc = e.kind() == TantivyError::DataCorruption; }
    CHECK(wrong_max && bad_crc);
  }
  // Index::open_in_dir over the compat files + a DeleteMeta: the segment's only doc is deleted
  const std::string base = dir + "/index_v7/";
  const auto meta_bytes = read_file(base + "meta.json");
  std::string meta_json(meta_bytes.begin(), meta_bytes.end());
  const files::IndexMeta meta0 = files::read_meta(meta_json);
  const std::string none = "\"deletes\": null";
  const size_t at = meta_json.find(none);
  CHECK(at != std::string::npos);
  if (at == std::string::npos) return;
  meta_json.replace(at, none.size(), "\"deletes\": {\"num_deleted_docs\": 1, \"opstamp\": 5}");
  const std::string del_name = meta0.segments[0].file_stem() + ".5.del";
  int asked = 0;
  auto read = [&](const std::string& name) {
    if (name == del_name) { ++asked; return from_deleted({0}, 1); }
    return read_file(base + name);
  };
  Index index = files::open_index(meta_json, read);
  CHECK(asked == 1);
  const SegmentData& seg = *index.segments()[0];
  CHECK(seg.alive.size() == 8 && !seg.is_alive(0));
  CHECK(index.reader().searcher().num_docs() == 0);
  bool mismatch = false;  // meta.json and the bitset must agree on the number of deleted docs
  try { files::open_index(meta_json, [&](const std::string& name) { return name == del_name ? from_deleted({}, 1) : read_file(base + name); }); }
  catch (const TantivyError& e) { mismatch = e.kind() == TantivyError::DataCorruption; }
  CHECK(mismatch);
}

// N2, SSTable kind: the term dictionary of the `quickwit` feature, specified inside the reference tree (sstable/).  Golden bytes:
// sstable/src/lib.rs:417-448 (test_simple_sstable); value block: sstable_termdict/mod.rs:117-150 (test_block_terminfos); long keys:
// lib.rs:394-414 (test_long_key_diff).
static void test_host_sstable_term_dictionary(const std::string& dir) {
  const std::vector<uint8_t> golden = {8, 0, 0, 0, 0, 16, 17, 33, 18, 19, 17, 20, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0,
                                       16, 0, 0, 0, 0, 0, 0, 0, 3, 0, 0, 0, 0, 0, 0, 0, 3, 0, 0, 0};
  {
    const auto keys = files::read_sstable(golden.data(), golden.size(), false);
    CHECK(keys.size() == 3 && keys[0].key == std::string("\x11") && keys[1].key == std::string("\x11\x12\x13") && keys[2].key == std::string("\x11\x14"));
    CHECK(files::write_single_block_sstable(keys, false) == golden);  // the test-side writer reproduces the reference's bytes
    auto bad = golden;
    bad[40] = 4;  // version
    bool unsupported = false;
    try { files::read_sstable(bad.data(), bad.size(), false); } catch (const TantivyError& e) { unsupported = e.kind() == TantivyError::Unsupported; }
    CHECK(unsupported);
    bad = golden;
    bad[32] = 2;  // num_terms
    bool corrupt = false;
    try { files::read_sstable(bad.data(), bad.size(), false); } catch (const TantivyError& e) { corrupt = e.kind() == TantivyError::DataCorruption; }
    CHECK(corrupt);
  }
  auto ti = [](uint32_t df, uint64_t ps, uint64_t pe, uint64_t qs, uint64_t qe) { TermInfo t; t.doc_freq = df; t.postings_start = ps; t.postings_end = pe; t.positions_start = qs; t.positions_end = qe; return t; };
  {  // test_block_terminfos' three TermInfos under three keys
    std::vector<files::SSTableEntry> in = {{"abba", ti(120, 17, 45, 10, 122)}, {"bjork", ti(10, 45, 450, 122, 1100)}, {"blur", ti(17, 450, 462, 1100, 1302)}};
    const auto bytes = files::write_single_block_sstable(in);
    // values: VInt(3) VInt(17) VInt(10) (120, 28, 112) (10, 405, 978) (17, 12, 202), common::VInt (stop bit on the last byte)
    const std::vector<uint8_t> values = {0x83, 0x91, 0x8A, 0xF8, 0x9C, 0xF0, 0x8A, 0x15, 0x83, 0x52, 0x87, 0x91, 0x8C, 0x4A, 0x81};
    CHECK(bytes.size() > 5 + values.size() && std::equal(values.begin(), values.end(), bytes.begin() + 5));
    // deltas: (keep 0, add 4) "abba", (0, 5) "bjork", (1, 3) "lur"
    const std::vector<uint8_t> deltas = {0x40, 'a', 'b', 'b', 'a', 0x50, 'b', 'j', 'o', 'r', 'k', 0x31, 'l', 'u', 'r'};
    CHECK(std::equal(deltas.begin(), deltas.end(), bytes.begin() + 5 + (long)values.size()));
    const auto out = files::read_sstable(bytes.data(), bytes.size());
    CHECK(out.size() == 3);
    for (size_t i = 0; i < out.size() && i < in.size(); ++i) CHECK(out[i].key == in[i].key && out[i].info == in[i].info);
    // as a field's `.term` sub-file: + the dictionary type (SSTable = 2)
    auto sub = bytes;
    sub.insert(sub.end(), {2, 0, 0, 0});
    CHECK(files::term_dictionary_type(sub.data(), sub.size()) == 2u);
    CHECK(files::open_sstable_term_dictionary(sub.data(), sub.size()).size() == 3);
    bool not_fst = false;  // ... which the FST reader refuses
    try { files::open_term_dictionary(sub.data(), sub.size()); } catch (const TantivyError& e) { not_fst = e.kind() == TantivyError::Unsupported; }
    CHECK(not_fst);
  }
  {  // test_long_key_diff: keep / add beyond 15 take the vint form
    std::string k1, k3;
    for (int x = 0; x < 1024; ++x) k1.push_back((char)(x % 255));
    for (int x = 1; x < 300; ++x) k3.push_back((char)(x % 255));
    std::vector<files::SSTableEntry> in = {{k1, ti(1, 0, 2, 0, 0)}, {std::string("\x00\x03\x04", 3), ti(2, 2, 9, 0, 0)}, {k3, ti(3, 9, 11, 0, 0)}};
    const auto bytes = files::write_single_block_sstable(in);
    const auto out = files::read_sstable(bytes.data(), bytes.size());
    CHECK(out.size() == 3);
    for (size_t i = 0; i < out.size() && i < in.size(); ++i) CHECK(out[i].key == in[i].key && out[i].info == in[i].info);
  }
  {  // two blocks + an index the reader does not need (v3 with a block-address store): keys restart at every block
    std::vector<files::SSTableEntry> a = {{"aa", ti(1, 0, 2, 0, 0)}, {"ab", ti(2, 2, 4, 0, 0)}}, b = {{"ba", ti(3, 4, 9, 0, 0)}};
    const auto ba = files::write_single_block_sstable(a), bb = files::write_single_block_sstable(b);
    auto body_of = [](const std::vector<uint8_t>& t) { return std::vector<uint8_t>(t.begin(), t.end() - 4 - 28); };  // block without terminator + footer
    std::vector<uint8_t> two = body_of(ba);
    const auto second = body_of(bb);
    two.insert(two.end(), second.begin(), second.end());
    two.insert(two.end(), {0, 0, 0, 0});
    const uint64_t index_offset = two.size();
    two.insert(two.end(), {0xDE, 0xAD, 0xBE, 0xEF});                      // "index" bytes (an FST map + block addresses in a real file)
    auto u64le = [&](uint64_t v) { const uint8_t* p = reinterpret_cast<const uint8_t*>(&v); two.insert(two.end(), p, p + 8); };
    u64le(index_offset + 2);                                              // store_offset != 0: a real index
    u64le(index_offset);
    u64le(3);
    two.insert(two.end(), {3, 0, 0, 0});
    const auto out = files::read_sstable(two.data(), two.size());
    CHECK(out.size() == 3 && out[0].key == "aa" && out[1].key == "ab" && out[2].key == "ba" && out[2].info == b[0].info);
  }
  // Index::open_in_dir over the compat segment with its `.term` swapped for an SSTable dictionary of the same term: term_dict is filled
  // by open_index itself (the FST kind leaves it to the caller)
  const std::string base = dir + "/index_v7/";
  const auto meta_bytes = read_file(base + "meta.json");
  const std::string meta_json(meta_bytes.begin(), meta_bytes.end());
  const files::IndexMeta meta = files::read_meta(meta_json);
  const std::string term_name = meta.segments[0].file_stem() + ".term";
  {  // (the fixture's own `.term` is of the FST kind: read too, see test_host_fst_term_dictionary)
    Index plain = files::open_index(meta_json, [&](const std::string& name) { return read_file(base + name); });
    CHECK(plain.segments()[0]->fields[0].term_dict.size() == 1);
  }
  std::vector<uint8_t> sub = files::write_single_block_sstable({{"dateformat", ti(1, 0, 2, 0, 2)}});
  sub.insert(sub.end(), {2, 0, 0, 0});
  // composite file with one sub-file (field 0): body ‖ VInt(1) ‖ VInt(0) u32 field VInt(0) ‖ u32 footer_len, then the directory footer
  std::vector<uint8_t> file = sub;
  const std::vector<uint8_t> cfoot = {0x81, 0x80, 0, 0, 0, 0, 0x80};
  file.insert(file.end(), cfoot.begin(), cfoot.end());
  const uint32_t cfoot_len = (uint32_t)cfoot.size();
  file.insert(file.end(), reinterpret_cast<const uint8_t*>(&cfoot_len), reinterpret_cast<const uint8_t*>(&cfoot_len) + 4);
  const std::string json = "{\"version\":{\"major\":0,\"minor\":26,\"patch\":0,\"index_format_version\":7},\"crc\":" + std::to_string(files::crc32(file.data(), file.size())) + "}";
  const uint32_t json_len = (uint32_t)json.size(), magic = 1337u;
  file.insert(file.end(), json.begin(), json.end());
  file.insert(file.end(), reinterpret_cast<const uint8_t*>(&json_len), reinterpret_cast<const uint8_t*>(&json_len) + 4);
  file.insert(file.end(), reinterpret_cast<const uint8_t*>(&magic), reinterpret_cast<const uint8_t*>(&magic) + 4);
  Index index = files::open_index(meta_json, [&](const std::string& name) { return name == term_name ? file : read_file(base + name); });
  const auto& dict = index.segments()[0]->fields[0].term_dict;
  CHECK(dict.size() == 1 && dict.count("dateformat") == 1);
  if (dict.count("dateformat")) CHECK(dict.at("dateformat") == ti(1, 0, 2, 0, 2));
  CHECK(index.reader().searcher().doc_freq(Term::from_field_text(*index.schema().get_field("label"), "dateformat")) == 1);
}

// N2, FST kind: crate tantivy-fst's map (term -> ordinal), restated from its published layout (tantivy_host.hpp, class files::Fst).
// What the reference tree pins: the compat fixtures' one-term dictionary.  Everything else is checked for self-consistency only,
// against a test-side compiler of the same layout (a plain trie: valid, not minimal).
namespace {
struct TrieNode { std::map<uint8_t, int> next; bool is_final = false; uint64_t value = 0; };
struct FstCompiler {
  std::vector<uint8_t> out;
  size_t last_addr = 0;  // address (last byte) of the node compiled most recently
  static int code_of(uint8_t b) {
    static const char kInv[] = "te/oasripcnw.hlm-du012g=:bf3y5&_4v9678k%?xCDASFIBEjPTzRNM+LOqHG";
    for (int i = 0; i < 63; ++i) if ((uint8_t)kInv[i] == b) return i + 1;
    return 0;
  }
  static uint8_t bytes_for(uint64_t v) { uint8_t n = 0; while (v) { ++n; v >>= 8; } return n; }
  void put(uint64_t v, uint8_t n) { for (uint8_t k = 0; k < n; ++k) out.push_back((uint8_t)(v >> (8 * k))); }
  struct T { uint8_t input; uint64_t output; size_t addr; };
  // compiles one state whose targets are compiled already; returns its address
  size_t compile(const std::vector<T>& ts, bool is_final, uint64_t final_output) {
    if (ts.empty() && is_final && final_output == 0) return 0;  // the empty final state
    const size_t cur = out.size();
    if (ts.size() == 1 && !is_final) {
      const T& t = ts[0];
      const int code = code_of(t.input);
      if (t.addr == last_addr && t.addr != 0 && t.output == 0 && t.addr + 1 == cur) {  // 11cccccc: the target is the node just before
        if (!code) out.push_back(t.input);
        out.push_back((uint8_t)(0xC0 | code));
      } else {
        const uint64_t delta = t.addr ? cur - t.addr : 0;
        const uint8_t tsize = std::max<uint8_t>(1, bytes_for(delta)), osize = bytes_for(t.output);
        put(t.output, osize);
        put(delta, tsize);
        out.push_back((uint8_t)((tsize << 4) | osize));
        if (!code) out.push_back(t.input);
        out.push_back((uint8_t)(0x80 | code));
      }
      return last_addr = out.size() - 1;
    }
    uint64_t max_delta = 0, max_out = is_final ? final_output : 0;
    for (auto& t : ts) { max_delta = std::max<uint64_t>(max_delta, t.addr ? cur - t.addr : 0); max_out = std::max(max_out, t.output); }
    const uint8_t tsize = std::max<uint8_t>(1, bytes_for(max_delta)), osize = bytes_for(max_out);
    const size_t n = ts.size();
    if (is_final) put(final_output, osize);
    for (size_t i = n; i-- > 0;) put(ts[i].output, osize);
    for (size_t i = n; i-- > 0;) put(ts[i].addr ? cur - ts[i].addr : 0, tsize);
    for (size_t i = n; i-- > 0;) out.push_back(ts[i].input);
    if (n > 32) {  // the 256-byte input index of version 2
      std::vector<uint8_t> index(256, 255);
      for (size_t i = 0; i < n; ++i) index[ts[i].input] = (uint8_t)i;
      out.insert(out.end(), index.begin(), index.end());
    }
    out.push_back((uint8_t)((tsize << 4) | osize));
    const bool inline_count = n >= 1 && n <= 63;
    if (!inline_count) out.push_back((uint8_t)(n == 256 ? 1 : n));
    out.push_back((uint8_t)((is_final ? 0x40 : 0) | (inline_count ? n : 0)));
    return last_addr = out.size() - 1;
  }
};
// keys sorted ascending, value of key i = i (what TermDictionaryBuilder inserts)
std::vector<uint8_t> compile_fst(const std::vector<std::string>& keys) {
  std::vector<TrieNode> trie(1);
  for (size_t k = 0; k < keys.size(); ++k) {
    int at = 0;
    for (unsigned char b : keys[k]) {
      auto it = trie[at].next.find(b);
      if (it == trie[at].next.end()) { trie.emplace_back(); it = trie[at].next.emplace(b, (int)trie.size() - 1).first; }
      at = it->second;
    }
    trie[at].is_final = true;
    trie[at].value = k;
  }
  FstCompiler c;
  c.out.assign(16, 0);
  c.out[0] = 2;  // version 2, type 0
  // post-order; a leaf's value rides on the transition that reaches it (the leaf is the empty final state), a key that is a prefix of
  // others keeps its value as the final output of its node
  std::function<size_t(int)> emit = [&](int id) -> size_t {
    std::vector<FstCompiler::T> ts;
    for (auto& kv : trie[id].next) {
      const TrieNode& child = trie[kv.second];
      if (child.next.empty()) ts.push_back({kv.first, child.value, 0});
      else ts.push_back({kv.first, 0, emit(kv.second)});
    }
    return c.compile(ts, trie[id].is_final, trie[id].is_final ? trie[id].value : 0);
  };
  const size_t root = emit(0);
  auto u64le = [&](uint64_t v) { for (int k = 0; k < 8; ++k) c.out.push_back((uint8_t)(v >> (8 * k))); };
  u64le(keys.size());
  u64le(root);
  return c.out;
}
}  // namespace

static void test_host_fst_term_dictionary(const std::string& dir) {
  // (1) what the reference tree pins: the compat fixtures' dictionaries (one term each), through the whole `.term` framing
  for (const std::string version : {"index_v6", "index_v7"}) {
    const std::string base = dir + "/" + version + "/";
    const auto meta_bytes = read_file(base + "meta.json");
    const files::IndexMeta meta = files::read_meta(std::string(meta_bytes.begin(), meta_bytes.end()));
    const auto term_file = read_file(base + meta.segments[0].file_stem() + ".term");
    const files::Footer tf = files::read_footer(term_file.data(), term_file.size());
    auto parts = files::open_composite(term_file.data(), tf.body_len);
    const files::FileSlice sl = parts.at({0u, 0u});
    const auto entries = files::open_fst_term_dictionary(term_file.data() + sl.offset, sl.len);
    CHECK(entries.size() == 1 && entries[0].key == "dateformat");
    if (!entries.empty()) CHECK(entries[0].info.doc_freq == 1 && entries[0].info.postings_start == 0 && entries[0].info.postings_end == 2);
    const files::TermDictionaryParts dict = files::open_term_dictionary(term_file.data() + sl.offset, sl.len);
    const files::Fst fst(dict.fst.data(), dict.fst.size());
    CHECK(fst.len() == 1 && fst.get("dateformat") == std::optional<uint64_t>(0));
    CHECK(!fst.get("dateforma") && !fst.get("dateformats") && !fst.get("") && !fst.get("x"));
    // Index::open_in_dir alone now answers a term look-up
    Index index = files::open_index_in_dir(dir + "/" + version);
    CHECK(index.reader().searcher().doc_freq(Term::from_field_text(*index.schema().get_field("label"), "dateformat")) == 1);
    // the test-side compiler writes the fixture's FST byte for byte (single-transition nodes, input codes, header, footer)
    CHECK(compile_fst({"dateformat"}) == dict.fst);
  }
  // (2) self-consistency beyond the fixture: prefixes that are keys, shared prefixes, explicit input bytes, outputs of several bytes
  {
    std::vector<std::string> keys = {"a", "ab", "abc", "abd", "b", "ba", "date", "dateformat", "dates", "zz", std::string("zz\xC3\xA9"), "zzz"};
    std::sort(keys.begin(), keys.end());
    const auto bytes = compile_fst(keys);
    const files::Fst fst(bytes.data(), bytes.size());
    CHECK(fst.len() == keys.size());
    for (size_t i = 0; i < keys.size(); ++i) CHECK(fst.get(keys[i]) == std::optional<uint64_t>(i));
    CHECK(!fst.get("") && !fst.get("dat") && !fst.get("abcd") && !fst.get("c") && !fst.get("zzzz"));
    std::vector<std::string> seen;
    fst.for_each([&](const std::string& k, uint64_t v) { CHECK(v == seen.size()); seen.push_back(k); });
    CHECK(seen == keys);
  }
  {  // a root with more than 32 transitions (the 256-byte index), 3000 keys (two-byte outputs), all byte values
    std::vector<std::string> keys;
    uint64_t x = 0x9E3779B97F4A7C15ull;
    auto rnd = [&]() { x ^= x << 7; x ^= x >> 9; return x; };
    for (int i = 0; i < 3000; ++i) {
      std::string k;
      const int n = 1 + (int)(rnd() % 9);
      for (int j = 0; j < n; ++j) k.push_back((char)(j == 0 ? rnd() % 256 : "etaoinshrdlu0123456789XYZ_\xC3\xA9\x01"[rnd() % 29]));
      keys.push_back(k);
    }
    std::sort(keys.begin(), keys.end());
    keys.erase(std::unique(keys.begin(), keys.end()), keys.end());
    const auto bytes = compile_fst(keys);
    const files::Fst fst(bytes.data(), bytes.size());
    size_t n = 0;
    bool ordered = true;
    fst.for_each([&](const std::string& k, uint64_t v) { ordered = ordered && n < keys.size() && k == keys[n] && v == n; ++n; });
    CHECK(n == keys.size() && ordered);
    for (size_t i = 0; i < keys.size(); i += 37) CHECK(fst.get(keys[i]) == std::optional<uint64_t>(i));
    // a truncated / damaged file is refused, not misread
    bool refused = false;
    try { files::Fst bad(bytes.data(), 20); (void)bad; } catch (const TantivyError& e) { refused = e.kind() == TantivyError::DataCorruption; }
    CHECK(refused);
  }
  {  // damaged dictionaries: an error or an answer, never a crash or a runaway walk (2000 random byte flips each, FST and SSTable)
    const auto fst_bytes = compile_fst({"a", "ab", "abc", "b", "date", "dateformat", "dates", "zz", "zzz"});
    std::vector<files::SSTableEntry> es;
    for (int i = 0; i < 40; ++i) { TermInfo t; t.doc_freq = (uint32_t)i + 1; t.postings_start = (uint64_t)i * 7; t.postings_end = t.postings_start + 7; es.push_back({"k" + std::to_string(100 + i), t}); }
    const auto sst_bytes = files::write_single_block_sstable(es);
    uint64_t x = 88172645463325252ull;
    auto rnd = [&]() { x ^= x << 13; x ^= x >> 7; x ^= x << 17; return x; };
    size_t survived = 0;
    for (int it = 0; it < 2000; ++it) {
      auto f = fst_bytes;
      for (int k = 0; k < 1 + (int)(rnd() % 3); ++k) f[rnd() % f.size()] ^= (uint8_t)(1u << (rnd() % 8));
      try { files::Fst t(f.data(), f.size()); size_t n = 0; t.for_each([&](const std::string&, uint64_t) { ++n; }); (void)t.get("dateformat"); ++survived; } catch (const TantivyError&) {}
      auto s2 = sst_bytes;
      for (int k = 0; k < 1 + (int)(rnd() % 3); ++k) s2[rnd() % s2.size()] ^= (uint8_t)(1u << (rnd() % 8));
      try { (void)files::read_sstable(s2.data(), s2.size()); ++survived; } catch (const TantivyError&) {}
    }
    CHECK(survived > 0);
  }
}

static void test_compat_index_search(const std::string& dir) {  // GPU: segments the reference wrote, searched on the device
  for (const std::string version : {"index_v6", "index_v7"}) {
    Index index = index_from_compat_files(dir, version);
    Field label = *index.schema().get_field("label");
    Searcher searcher = index.reader().searcher();
    // assert_date_time_precision (compat_tests.rs:57-80): parse_query("dateformat"), TopDocs::with_limit(1) -> 1 hit
    QueryBox q = QueryParser::for_index(index, {label}).parse_query("dateformat");
    auto top = searcher.search(*q, TopDocs::with_limit(1).order_by_score());
    CHECK(top.size() == 1);
    CHECK(top[0].second == DocAddress(0, 0));
    CHECK_NEARLY(top[0].first, 0.28768212);  // one doc, one token: idf(1,1) * 2.2 * 1/(1+1.2)
    CHECK(searcher.search(*q, Count{}) == 1);
  }
}

// ---- --dump -------------------------------------------------------------------------------------------------------------
static void write_file(const std::string& path, const uint8_t* p, size_t n) {
  std::ofstream f(path, std::ios::binary);
  f.write(reinterpret_cast<const char*>(p), (std::streamsize)n);
}
static std::string json_escape(const std::string& s) {
  std::string o;
  for (unsigned char c : s) {
    if (c == '"' || c == '\\') { o += '\\'; o += (char)c; }
    else if (c < 0x20 || c >= 0x7F) { char b[8]; std::snprintf(b, sizeof b, "\\u%04x", c); o += b; }
    else o += (char)c;
  }
  return o;
}
static void dump_all(const std::string& dir) {
  std::ostringstream m;
  m << "{\n";
  auto all = all_indexes();
  for (size_t n = 0; n < all.size(); ++n) {
    const Index& ix = all[n].index;
    m << "  \"" << all[n].name << "\": {\"fields\": [";
    for (uint32_t f = 0; f < ix.schema().num_fields(); ++f) m << (f ? ", " : "") << "\"" << ix.schema().get_field_entry(Field{f}).name << "\"";
    m << "], \"segments\": [\n";
    for (size_t s = 0; s < ix.segments().size(); ++s) {
      const SegmentData& sd = *ix.segments()[s];
      m << "    {\"max_doc\": " << sd.max_doc << ", \"alive\": ";
      if (sd.alive.empty()) m << "null";
      else {
        const std::string p = all[n].name + ".seg" + std::to_string(s) + ".alive";
        write_file(dir + "/" + p, sd.alive.data(), sd.alive.size());
        m << "\"" << p << "\"";
      }
      m << ", \"fields\": [";
      for (uint32_t f = 0; f < sd.fields.size(); ++f) {
        const FieldSegmentData& fd = sd.fields[f];
        const std::string base = all[n].name + ".seg" + std::to_string(s) + ".f" + std::to_string(f);
        write_file(dir + "/" + base + ".idx", fd.idx_body.data(), fd.idx_body.size());
        if (fd.has_fieldnorms) write_file(dir + "/" + base + ".fieldnorm", fd.fieldnorms.data(), fd.fieldnorms.size());
        write_file(dir + "/" + base + ".pos", fd.positions.data(), fd.positions.size());
        m << (f ? ", " : "") << "{\"record\": " << (int)fd.record << ", \"idx\": \"" << base << ".idx\", \"fieldnorm\": "
          << (fd.has_fieldnorms ? "\"" + base + ".fieldnorm\"" : std::string("null")) << ", \"terms\": {";
        bool first = true;
        for (auto& kv : fd.term_dict) {
          m << (first ? "" : ", ") << "\"" << json_escape(kv.first) << "\": [" << kv.second.doc_freq << ", " << kv.second.postings_start << ", "
            << kv.second.postings_end << ", " << kv.second.positions_start << ", " << kv.second.positions_end << "]";
          first = false;
        }
        m << "}}";
      }
      m << "]}" << (s + 1 < ix.segments().size() ? "," : "") << "\n";
    }
    m << "  ]}" << (n + 1 < all.size() ? "," : "") << "\n";
  }
  m << "}\n";
  const std::string text = m.str();
  write_file(dir + "/manifest.json", reinterpret_cast<const uint8_t*>(text.data()), text.size());
}

int main(int argc, char** argv) {
  std::string mode = argc > 1 ? argv[1] : "";
  std::string dir = argc > 2 ? argv[2] : "";
  if (mode == "--dump") {
    dump_all(dir);
    return 0;
  }
  std::vector<std::pair<std::string, std::function<void()>>> tests;
  if (mode == "--cpu") {
    tests = {{"host_tokenizer_and_statistics", test_host_tokenizer_and_statistics},
             {"host_term_info_store", test_host_term_info_store},
             {"host_search_without_device_raises", test_host_search_without_device_raises}};
    if (!dir.empty()) tests.push_back({"host_compat_framing", [dir]() { test_host_compat_framing(dir); }});
    if (!dir.empty()) tests.push_back({"host_alive_bitset_file", [dir]() { test_host_alive_bitset_file(dir); }});
    if (!dir.empty()) tests.push_back({"host_sstable_term_dictionary", [dir]() { test_host_sstable_term_dictionary(dir); }});
    if (!dir.empty()) tests.push_back({"host_fst_term_dictionary", [dir]() { test_host_fst_term_dictionary(dir); }});
  } else {
    tests = {{"term_query_no_freq", test_term_query_no_freq},
             {"term_query_multiple_of_block_len", test_term_query_multiple_of_block_len},
             {"term_weight", test_term_weight},
             {"boolean_query_with_weight", test_boolean_query_with_weight},
             {"intersection_score", test_intersection_score},
             {"top_collector", test_top_collector},
             {"multi_segment_deletes_and_paging", test_multi_segment_deletes_and_paging},
             {"count_collector", test_count_collector},
             {"absent_terms_and_unsupported_shapes", test_absent_terms_and_unsupported_shapes},
             {"host_tokenizer_and_statistics", test_host_tokenizer_and_statistics}};
    if (mode == "--compat" && !dir.empty()) tests.push_back({"compat_index_search", [dir]() { test_compat_index_search(dir); }});
  }
  int bad = 0;
  for (auto& t : tests) {
    const int before = g_failed;
    try {
      t.second();
    } catch (const std::exception& e) {
      std::printf("    exception: %s\n", e.what());
      ++g_failed;
    }
    std::printf("%s %s\n", g_failed == before ? "ok  " : "FAIL", t.first.c_str());
    bad += g_failed != before;
  }
  std::printf("%d test(s) failed\n", bad);
  return bad ? 1 : 0;
}
