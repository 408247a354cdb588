"""GPU parity tests: the CUDA path, called through the C ABI, against the CPU oracle on the same
seeded inputs.  Doc ids and segment ordinals must be bit-exact; scores are compared bit-exact too
(the device computes BM25 with the reference's f32 operation order; tolerance stated where the
reference itself is order dependent).  Edge cases follow the reference's tests: empty / one-doc /
127 / 128 / 129-doc lists, blocks starting at doc 0, every bit width, deletes, absent terms."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import tantivy_b200 as T  # noqa: E402
from oracle import tq_oracle as O  # noqa: E402
from tantivy_b200._abi import (TQ_OP_AND, TQ_OP_OR, TQ_OP_TERM, TQ_RECORD_BASIC, TQ_RECORD_FREQS,  # noqa: E402
                               TQ_RECORD_FREQS_POSITIONS, QueryBatch)
from tests.helpers import OracleSegment, hits, make_query  # noqa: E402


import os  # noqa: E402


def _ctx_with_env(**env):
    """tq_ctx_create reads its tuning knobs from the environment."""
    old = {k: os.environ.get(k) for k in env}
    os.environ.update({k: str(v) for k, v in env.items()})
    try:
        return T.Context(0)
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


# every test runs on both union engines: "tile" = the shared-decode tile engine (k_score_lists + k_tile, the default),
# "legacy" = the per-query kernels (k_or_strip, and k_or for > 8 clauses or k > 128) that the tile engine falls back to
@pytest.fixture(scope="module", params=["tile", "legacy"])
def ctx(request):
    # (TQ_TILE_TERMS=1: single-term batches stay on the tile engine here; the default rule has a test of its own)
    c = _ctx_with_env(TQ_TILE=1 if request.param == "tile" else 0, TQ_TILE_TERMS=1)
    c.engine = request.param
    yield c
    c.close()


_next_seg = [1000]


def fresh_ord():
    _next_seg[0] += 1
    return _next_seg[0]


def both(ctx, segments):
    oi = O.OracleIndex()
    for s in segments:
        s.register(oi)
        s.register(ctx)
    return oi


def assert_same(gpu_res, cpu_res, nq, exact_scores=True):
    for i in range(nq):
        g, c = hits(gpu_res, i), hits(cpu_res, i)
        assert [(s, d) for _, s, d in g] == [(s, d) for _, s, d in c], f"query {i}: doc ids differ\n gpu={g[:8]}\n cpu={c[:8]}"
        for (sg, _, _), (sc, _, _) in zip(g, c):
            if exact_scores:
                assert sg == sc, f"query {i}: score {sg!r} != {sc!r}"
            else:
                assert abs(sg - sc) <= 1e-5 * max(abs(sg), abs(sc))


# ---- K1: block decode -------------------------------------------------------------------------------
def _lists_all_widths(rng, max_doc):
    lists = []
    for bits in list(range(0, 21)) + [24]:
        n = 128 * 3 + int(rng.integers(0, 128))
        gaps = rng.integers(1, 2 ** bits + 1, size=n, dtype=np.uint64)
        gaps[5] = 2 ** bits  # force the width
        start = int(rng.integers(0, 3))
        docs = start + np.cumsum(gaps) - gaps[0]
        docs = docs[docs < max_doc].astype(np.uint32)
        tf_bits = int(rng.integers(0, 12))
        tfs = rng.integers(1, 2 ** tf_bits + 1, size=len(docs), dtype=np.uint64).astype(np.uint32)
        lists.append((docs, tfs))
    for n in (1, 2, 127, 128, 129, 255, 256, 257):
        docs = np.sort(rng.choice(max_doc, size=n, replace=False)).astype(np.uint32)
        lists.append((docs, rng.integers(1, 9, size=n).astype(np.uint32)))
    lists.append((np.arange(0, 300, dtype=np.uint32), np.ones(300, np.uint32)))  # 0-bit deltas from doc 0
    big = np.ones(200, np.uint32)
    big[17] = 0xFFFFFFFF  # 32-bit tf width
    lists.append((np.arange(5, 205, dtype=np.uint32), big))
    # doc bit widths 25..31 (skip.rs:16-22 allows up to 31): one gap of 2^(bits-1) + 1 in a full block (doc ids stay below
    # TERMINATED = 2^31 - 1), both as the first block of a list and behind another block / in front of a VInt tail
    for bits in range(25, 32):
        for n, at in ((128 + int(rng.integers(0, 100)), 5), (256 + int(rng.integers(1, 128)), 128 + 77)):
            gaps = rng.integers(1, 40, size=n, dtype=np.uint64)
            gaps[at] = 2 ** (bits - 1) + 1
            docs = (int(rng.integers(0, 3)) + np.cumsum(gaps) - gaps[0])
            assert docs[-1] < max_doc
            lists.append((docs.astype(np.uint32), rng.integers(1, 2 ** int(rng.integers(1, 12)) + 1, size=n, dtype=np.uint64).astype(np.uint32)))
    return lists


@pytest.mark.parametrize("record_option", [TQ_RECORD_BASIC, TQ_RECORD_FREQS, TQ_RECORD_FREQS_POSITIONS])
def test_decode_every_width_and_alignment(ctx, record_option):
    rng = np.random.default_rng(42 + record_option)
    max_doc = 0x7FFFFFFE  # the largest max_doc there is (TERMINATED - 1): widths 25..31 need doc ids up to 2^31
    lists = _lists_all_widths(rng, max_doc)
    if record_option == TQ_RECORD_BASIC:
        lists = [(d, None) for d, _ in lists]
    so = fresh_ord()
    seg = OracleSegment(lists, None, record_option=record_option, segment_ord=so, writer_cls=T.FieldWriter, max_doc=max_doc)
    oi = both(ctx, [seg])
    starts = set()
    for t, (docs, tfs) in enumerate(lists):
        ts = seg.term_seg(t)
        starts.add(ts[4] % 4)
        d_g, f_g = ctx.decode_postings(ts)
        d_c, f_c = oi.decode_postings(ts)
        assert (d_g == d_c).all() and (d_g == docs).all(), f"term {t}"
        assert (f_g == f_c).all(), f"term {t}"
    assert len(starts) > 1  # both aligned and misaligned block starts were exercised


def test_block_table_matches_skip_reader(ctx):
    rng = np.random.default_rng(9)
    max_doc = 400_000
    fieldnorms = rng.integers(1, 2000, size=max_doc)
    lists = []
    for p in (0.3, 0.02, 0.004):
        docs = np.nonzero(rng.random(max_doc) < p)[0].astype(np.uint32)
        tfs = np.minimum(rng.geometric(0.7, size=len(docs)), 300).astype(np.uint32)
        tfs[::97] = 300  # saturated block-max tf codes
        lists.append((docs, tfs))
    seg = OracleSegment(lists, fieldnorms, segment_ord=fresh_ord(), writer_cls=T.FieldWriter)
    oi = both(ctx, [seg])
    w, avg = O.bm25_weight(len(lists[0][0]), max_doc), float(np.float32(seg.total_num_tokens) / np.float32(max_doc))
    for t in range(3):
        lg, bg = ctx.block_table(seg.term_seg(t), w, avg)
        lc, bc = oi.block_table(seg.term_seg(t), w, avg)
        assert (lg == lc).all()
        assert (bg == bc).all()


# ---- queries on small random segments ------------------------------------------------------------------
def _random_segments(rng, n_segments, n_terms, max_doc_range=(300, 40_000), dens=(0.5, 0.2, 0.05, 0.01, 0.002), deletes=False):
    segs = []
    for _ in range(n_segments):
        max_doc = int(rng.integers(*max_doc_range))
        fieldnorms = np.clip(np.round(np.exp(rng.normal(np.log(40), 0.7, size=max_doc))), 1, 4096).astype(np.uint32)
        lists = []
        for t in range(n_terms):
            p = dens[t % len(dens)] * float(rng.uniform(0.5, 1.5))
            docs = np.nonzero(rng.random(max_doc) < p)[0].astype(np.uint32)
            tfs = np.minimum(rng.geometric(0.6, size=len(docs)), 10).astype(np.uint32)
            lists.append((docs, tfs))
        alive = None
        if deletes:
            alive_bits = rng.random(max_doc) > 0.2
            alive = np.packbits(alive_bits, bitorder="little")
        segs.append(OracleSegment(lists, fieldnorms, segment_ord=fresh_ord(), writer_cls=T.FieldWriter, alive=alive))
    return segs


def _run_both(ctx, segs, queries):
    oi = both(ctx, segs)
    qb = QueryBatch(queries)
    return ctx.search_batch(qb), oi.search_batch(qb, mode=0), qb.nq


@pytest.mark.parametrize("n_segments", [1, 3])
def test_term_queries(ctx, n_segments):
    rng = np.random.default_rng(100 + n_segments)
    segs = _random_segments(rng, n_segments, 5)
    queries = [make_query(TQ_OP_TERM, segs, [t], k) for t in range(5) for k in (1, 10, 100, 1000)]
    g, c, nq = _run_both(ctx, segs, queries)
    assert_same(g, c, nq)


@pytest.mark.parametrize("n_segments", [1, 3])
def test_and_queries(ctx, n_segments):
    rng = np.random.default_rng(200 + n_segments)
    segs = _random_segments(rng, n_segments, 5)
    combos = [[0, 1], [0, 4], [3, 0], [4, 3], [0, 1, 2], [4, 0, 2], [0, 1, 2, 3, 4], [2, 2 - 1]]
    queries = [make_query(TQ_OP_AND, segs, terms, k) for terms in combos for k in (1, 10, 300)]
    g, c, nq = _run_both(ctx, segs, queries)
    assert_same(g, c, nq)


@pytest.mark.parametrize("n_segments", [1, 3])
def test_or_queries(ctx, n_segments):
    rng = np.random.default_rng(300 + n_segments)
    segs = _random_segments(rng, n_segments, 5)
    combos = [[0, 1], [4, 3], [3, 0], [0, 1, 2], [0, 1, 2, 3, 4], [4, 2, 0]]
    queries = [make_query(TQ_OP_OR, segs, terms, k) for terms in combos for k in (1, 10, 100, 1024)]
    g, c, nq = _run_both(ctx, segs, queries)
    assert_same(g, c, nq)


def test_many_term_union_and_wide_segments(ctx):
    rng = np.random.default_rng(400)
    segs = _random_segments(rng, 2, 20, max_doc_range=(100_000, 200_000), dens=(0.05, 0.01, 0.002, 0.0005))
    queries = [make_query(TQ_OP_OR, segs, list(range(20)), 10), make_query(TQ_OP_OR, segs, list(range(0, 20, 3)), 100),
               make_query(TQ_OP_AND, segs, [0, 4, 8], 10), make_query(TQ_OP_TERM, segs, [3], 50)]
    g, c, nq = _run_both(ctx, segs, queries)
    assert_same(g, c, nq)


def test_deletes_and_absent_terms(ctx):
    rng = np.random.default_rng(500)
    segs = _random_segments(rng, 3, 4, deletes=True)
    # make term 3 absent from segment 1 and term 2 absent everywhere but segment 0
    segs[1].terms[3] = (0, 0, 0)
    segs[1].terms[2] = (0, 0, 0)
    segs[2].terms[2] = (0, 0, 0)
    queries = [make_query(op, segs, terms, k) for op, terms in
               [(TQ_OP_TERM, [3]), (TQ_OP_TERM, [2]), (TQ_OP_AND, [0, 3]), (TQ_OP_AND, [2, 1]), (TQ_OP_OR, [3, 2]), (TQ_OP_OR, [0, 2, 3])]
               for k in (5, 50)]
    g, c, nq = _run_both(ctx, segs, queries)
    assert_same(g, c, nq)


def test_basic_record_option_and_no_fieldnorm(ctx):
    rng = np.random.default_rng(600)
    max_doc = 20_000
    lists = [(np.nonzero(rng.random(max_doc) < p)[0].astype(np.uint32), None) for p in (0.3, 0.05)]
    seg = OracleSegment(lists, None, record_option=TQ_RECORD_BASIC, segment_ord=fresh_ord(), writer_cls=T.FieldWriter, max_doc=max_doc)
    oi = both(ctx, [seg])  # constant fieldnorm 1
    qb = QueryBatch([make_query(TQ_OP_TERM, [seg], [0], 10), make_query(TQ_OP_AND, [seg], [0, 1], 10), make_query(TQ_OP_OR, [seg], [0, 1], 10)])
    assert_same(ctx.search_batch(qb), oi.search_batch(qb, mode=0), qb.nq)


def test_basic_option_requested_on_a_field_with_freqs(ctx):
    """TermQuery::new(term, IndexRecordOption::Basic) on a WithFreqs field: tf blocks are skipped and
    every posting scores with tf = 1 (FreqReadingOption::SkipFreq, block_segment_postings.rs:97-140)."""
    rng = np.random.default_rng(650)
    segs = _random_segments(rng, 2, 4)
    queries = []
    for op, terms in [(TQ_OP_TERM, [0]), (TQ_OP_TERM, [3]), (TQ_OP_AND, [0, 1]), (TQ_OP_OR, [0, 2, 3]), (TQ_OP_OR, [1, 0])]:
        for flags in ([1] * len(terms), [1] + [0] * (len(terms) - 1)):
            q = make_query(op, segs, terms, 25)
            q["term_flags"] = flags
            queries.append(q)
    plain = make_query(TQ_OP_TERM, segs, [0], 25)  # the same list WITH freqs, in the same batch
    g, c, nq = _run_both(ctx, segs, queries + [plain])
    assert_same(g, c, nq)
    assert [s for s, _, _ in hits(g, 0)] != [s for s, _, _ in hits(g, nq - 1)]  # the flag changes the scores


def test_initial_threshold_like_for_each_pruning(ctx):
    """tq_query.threshold = the `threshold` argument of Weight::for_each_pruning (weight.rs:123-132): only docs scoring
    strictly above it are collected; passing the k-th score of a finished search returns the k-1 docs above it."""
    rng = np.random.default_rng(660)
    segs = _random_segments(rng, 3, 5)
    base = [make_query(op, segs, terms, 20) for op, terms in
            [(TQ_OP_TERM, [1]), (TQ_OP_AND, [0, 1]), (TQ_OP_OR, [0, 1, 2, 3, 4]), (TQ_OP_OR, [4, 2]), (TQ_OP_OR, [0, 3, 4])]]
    oi = both(ctx, segs)
    qb0 = QueryBatch(base)
    g0, c0 = ctx.search_batch(qb0), oi.search_batch(qb0, mode=0)
    assert_same(g0, c0, qb0.nq)
    queries = []
    for i, q in enumerate(base):
        h = hits(g0, i)
        for thr in (h[len(h) // 2][0], h[-1][0], h[0][0], 0.0, -1.0, 1e9):
            q2 = dict(q)
            q2["threshold"] = float(thr)
            q2["k"] = 50
            queries.append(q2)
    qb = QueryBatch(queries)
    g, c, nq = ctx.search_batch(qb), oi.search_batch(qb, mode=0), qb.nq
    assert_same(g, c, nq)
    for i, q in enumerate(queries):
        assert all(s > np.float32(q["threshold"]) for s, _, _ in hits(g, i))
    mid = hits(g0, 2)[10][0]  # the OR query again, threshold = its 11th score: exactly the hits above it come back
    above = [h for h in hits(g0, 2) if h[0] > mid]
    assert hits(g, 2 * 6)[:len(above)] == above


def test_ties_pick_lowest_doc(ctx):
    # every doc has the same length and tf: all scores tie; the top-k must be the k lowest doc ids
    max_doc = 5000
    docs = np.arange(7, max_doc, 3, dtype=np.uint32)
    segs = [OracleSegment([(docs, np.ones(len(docs), np.uint32))], np.full(max_doc, 10), segment_ord=fresh_ord(), writer_cls=T.FieldWriter)
            for _ in range(2)]
    g, c, nq = _run_both(ctx, segs, [make_query(TQ_OP_TERM, segs, [0], k) for k in (1, 7, 200)])
    assert_same(g, c, nq)
    assert [d for _, _, d in hits(g, 1)] == list(range(7, 7 + 21, 3))
    assert len({s for _, s, _ in hits(g, 1)}) == 1  # all from the lower segment ordinal


def test_explicit_tf_cache_and_boost(ctx):
    rng = np.random.default_rng(700)
    segs = _random_segments(rng, 1, 3)
    q = make_query(TQ_OP_OR, segs, [0, 1, 2], 20, boost=2.5)
    q2 = dict(q)
    q2["tf_cache"] = np.stack([O.bm25_tf_cache(np.float32(a)) for a in q["avg_fieldnorm"]])
    g, c, nq = _run_both(ctx, segs, [q, q2])
    assert_same(g, c, nq)
    assert hits(g, 0) == hits(g, 1)


def test_batch_split_and_idempotence(ctx):
    rng = np.random.default_rng(800)
    segs = _random_segments(rng, 2, 5)
    for s in segs:
        s.register(ctx)
    queries = [make_query(op, segs, terms, 10) for op, terms in [(TQ_OP_TERM, [0]), (TQ_OP_AND, [0, 1]), (TQ_OP_OR, [1, 2, 3])] * 20]
    qb = QueryBatch(queries)
    a = ctx.search_batch(qb)
    b = ctx.search_batch(qb)
    for x, y in zip(a, b):
        assert (x == y).all()
    bt = ctx.prepare(qb)
    bt.run()
    bt.run()  # a prepared batch can be re-run
    c3 = bt.fetch()
    bt.close()
    for x, y in zip(a, c3):
        assert (x == y).all()
    single = [ctx.search_batch(QueryBatch([q])) for q in queries[:6]]
    for i, r in enumerate(single):
        assert hits(r, 0) == hits(a, i)


def test_invalid_arguments(ctx):
    rng = np.random.default_rng(900)
    segs = _random_segments(rng, 1, 2)
    segs[0].register(ctx)
    q = make_query(TQ_OP_TERM, segs, [0], 10)
    bad = dict(q); bad["k"] = 0
    with pytest.raises(T.TqError):
        ctx.search_batch(QueryBatch([bad]))
    bad = dict(q); bad["k"] = 5000
    with pytest.raises(T.TqError):
        ctx.search_batch(QueryBatch([bad]))
    bad = dict(q); bad["term_segs"] = [(0, 999_999, 0, 10, 0, 10)]
    with pytest.raises(T.TqError):
        ctx.search_batch(QueryBatch([bad]))
    # corrupt bytes: a list that claims a skip section but is two bytes long
    df, s, e = segs[0].terms[0]
    bad = dict(q); bad["term_segs"] = [(0, segs[0].segment_ord, 0, 1000, s, s + 2)]
    with pytest.raises(T.TqError):
        ctx.search_batch(QueryBatch([bad]))


# ---- larger synthetic index (SURVEY.md §8d generator) ---------------------------------------------------------
@pytest.fixture(scope="module")
def synth(ctx):
    dens = [0.3, 0.15, 0.05, 0.01, 0.002, 0.0001]
    ix = T.SynthIndex(3, 1_000_000, dens, seed=77)
    base = 5000
    ix.register(ctx, segment_base=base)
    oi = O.OracleIndex()
    ix.register(oi, segment_base=base)
    return ix, oi, base


def test_synth_mixed_batch(ctx, synth):
    ix, oi, base = synth
    queries = []
    for t in range(6):
        queries.append(ix.query(TQ_OP_TERM, [t], 10, segment_base=base))
    for terms in ([0, 1], [0, 3], [1, 4], [0, 5], [2, 3, 4], [0, 1, 2]):
        queries.append(ix.query(TQ_OP_AND, terms, 10, segment_base=base))
    for terms in ([0, 1], [3, 4], [4, 5], [0, 1, 2, 3, 4], [2, 5]):
        queries.append(ix.query(TQ_OP_OR, terms, 100, segment_base=base))
    qb = QueryBatch(queries)
    g = ctx.search_batch(qb)
    c = oi.search_batch(qb, mode=0, n_threads=8)
    assert_same(g, c, qb.nq)
    st = ctx.stats()
    assert st["units"] > 0 and st["kernel_launches"] >= 3 and st["algorithmic_bytes"] > 0


def test_synth_union_pruning_is_exact(ctx, synth):
    """Unions of dense and rare terms with small k: the tile engine prunes on its per-tile maxima, and on the legacy
    engine k_or_strip splits off the non-essential clauses (MaxScore) and runs its threshold rounds; the result must
    stay identical to the exhaustive oracle, hit for hit."""
    ix, oi, base = synth
    queries = []
    for k in (1, 3, 10, 50):
        for terms in ([0, 5], [0, 4, 5], [1, 0, 5, 3], [5, 4, 3, 2, 1, 0], [0, 1, 2], [2, 3, 4], [0, 3]):
            queries.append(ix.query(TQ_OP_OR, terms, k, segment_base=base))
    qb = QueryBatch(queries)
    g = ctx.search_batch(qb)
    c = oi.search_batch(qb, mode=0, n_threads=8)
    assert_same(g, c, qb.nq)
    # single-query batches use small units (many cold starts + threshold sharing between CTAs)
    for q in queries[:8]:
        qb1 = QueryBatch([q])
        assert_same(ctx.search_batch(qb1), oi.search_batch(qb1, mode=0), 1)


def test_synth_pruned_reference_path_agrees(ctx, synth):
    """The reference-faithful CPU path (Block-WAND + TopNHeap) returns the same hits as the GPU for
    term and AND queries (fixed summation order); for OR the reference's order-dependent f32 sum may
    differ in the last bits: tolerance 1e-5 relative (BASELINE.json north_star)."""
    ix, oi, base = synth
    q_exact = [ix.query(TQ_OP_TERM, [2], 10, segment_base=base), ix.query(TQ_OP_AND, [1, 3], 10, segment_base=base)]
    qb = QueryBatch(q_exact)
    assert_same(ctx.search_batch(qb), oi.search_batch(qb, mode=1), qb.nq)
    q_or = [ix.query(TQ_OP_OR, [1, 3, 4], 10, segment_base=base)]
    qb = QueryBatch(q_or)
    g, c = ctx.search_batch(qb), oi.search_batch(qb, mode=1)
    gs, cs = hits(g), hits(c)
    assert len(gs) == len(cs)
    for (sg, _, _), (sc, _, _) in zip(gs, cs):
        assert abs(sg - sc) <= 1e-5 * max(abs(sg), abs(sc))


def test_merge_topk_dev_matches_merge_fruits(ctx, synth):
    torch = pytest.importorskip("torch")
    ix, oi, base = synth
    queries = [ix.query(TQ_OP_OR, [1, 3], 50, segment_base=base), ix.query(TQ_OP_TERM, [2], 50, segment_base=base)]
    per_seg = []
    for s in range(ix.n_segments):
        qs = [ix.query(q["op"], terms, 50, segment_base=base, segments=[s]) for q, terms in zip(queries, ([1, 3], [2]))]
        per_seg.append(ctx.search_batch(QueryBatch(qs)))
    full = ctx.search_batch(QueryBatch(queries))
    dev = torch.device("cuda:0")
    sc = torch.tensor(np.stack([r[0] for r in per_seg]), device=dev)
    sg = torch.tensor(np.stack([r[1] for r in per_seg]).astype(np.int64), device=dev).to(torch.int32)
    dc = torch.tensor(np.stack([r[2] for r in per_seg]).astype(np.int64), device=dev).to(torch.int32)
    ct = torch.tensor(np.stack([r[3] for r in per_seg]).astype(np.int64), device=dev).to(torch.int32)
    o_sc = torch.zeros((2, 50), dtype=torch.float32, device=dev)
    o_sg = torch.zeros((2, 50), dtype=torch.int32, device=dev)
    o_dc = torch.zeros((2, 50), dtype=torch.int32, device=dev)
    o_ct = torch.zeros((2,), dtype=torch.int32, device=dev)
    torch.cuda.synchronize()
    ctx.merge_topk_dev(ix.n_segments, 2, 50, 50, sc.data_ptr(), sg.data_ptr(), dc.data_ptr(), ct.data_ptr(), o_sc.data_ptr(),
                       o_sg.data_ptr(), o_dc.data_ptr(), o_ct.data_ptr())
    assert (o_sc.cpu().numpy() == full[0]).all()
    assert (o_sg.cpu().numpy().astype(np.uint32) == full[1]).all()
    assert (o_dc.cpu().numpy().astype(np.uint32) == full[2]).all()
    assert (o_ct.cpu().numpy().astype(np.uint32) == full[3]).all()


def test_two_phase_run_with_threshold_exchange(ctx, synth):
    """tq_batch_run_phase(0) / thresholds export + import / phase(1): the split run returns what the plain run returns,
    and a foreign bound that is valid (another shard's k-th best, here: this shard's own final k-th score) only prunes."""
    import torch
    ix, oi, base = synth
    qb = QueryBatch([ix.query(TQ_OP_OR, terms, k, segment_base=base)
                     for terms, k in [([0, 1, 2, 3, 4], 100), ([0, 3, 5], 100), ([1, 2], 10), ([0, 4, 5], 50), ([2, 3, 4, 5], 100)]])
    plain = ctx.search_batch(qb)
    keys = torch.zeros(qb.nq, dtype=torch.int64, device="cuda:0")
    b = ctx.prepare(qb)
    n_phases = b.phases()
    assert n_phases >= 2
    sampled = None
    for phase in range(n_phases):
        b.run_phase(phase)
        if phase + 1 < n_phases:
            b.thresholds_export_dev(keys.data_ptr())
            now = keys.cpu().numpy().copy()
            assert sampled is None or (now >= sampled).all()  # thresholds only rise
            sampled = now
            b.thresholds_import_dev(keys.data_ptr())
    split = b.fetch()
    for a, c in zip(plain, split):
        assert (a == c).all()
    # the exported keys are lower bounds of the final k-th score keys
    final_kth = np.array([plain[0][i, plain[3][i] - 1] if plain[3][i] == qb.q["k"][i] else -np.inf for i in range(qb.nq)], dtype=np.float32)
    u = final_kth.view(np.uint32).astype(np.int64)
    final_keys = np.where(final_kth == -np.inf, 0, u ^ np.where(u >> 31, 0xFFFFFFFF, 0x80000000))
    assert (sampled <= final_keys).all()
    # hand the final k-th keys in as if another rank had found them: same rows again
    b.run_phase(0)
    keys2 = torch.from_numpy(final_keys.astype(np.int64)).to("cuda:0")
    b.thresholds_import_dev(keys2.data_ptr())
    for phase in range(1, n_phases):
        b.run_phase(phase)
    again = b.fetch()
    for a, c in zip(plain, again):
        assert (a == c).all()
    b.close()


def test_count_collector(ctx):
    """tq_count_batch = searcher.search(&query, &Count) (src/collector/count_collector.rs): alive matching docs, over
    several segments, with and without deletes, for term / AND / OR, absent terms included."""
    rng = np.random.default_rng(900)
    for deletes in (False, True):
        segs = _random_segments(rng, 3, 5, deletes=deletes)
        segs[1].terms[3] = (0, 0, 0)  # term 3 absent from one segment
        oi = both(ctx, segs)
        queries = [make_query(TQ_OP_TERM, segs, [t], 1) for t in range(5)]
        queries += [make_query(TQ_OP_AND, segs, ts, 1) for ts in ([0, 1], [0, 3], [1, 2, 4], [4, 3], [0, 1, 2, 3, 4])]
        queries += [make_query(TQ_OP_OR, segs, ts, 1) for ts in ([0, 1], [3], [3, 4], [0, 1, 2, 3, 4], [2, 4])]
        qb = QueryBatch(queries)
        g, c = ctx.count_batch(qb), oi.count_batch(qb)
        assert (g == c).all(), (g, c)
        assert g[:5].sum() > 0 and (g[5:10] <= g[0]).any()
        if not deletes:  # a term query without deletes is its doc_freq (term_weight.rs:179-190)
            assert [int(x) for x in g[:5]] == [sum(s.terms[t][0] for s in segs) for t in range(5)]


def test_count_collector_synth(ctx, synth):
    ix, oi, base = synth
    qb = QueryBatch([ix.query(op, terms, 1, segment_base=base) for op, terms in
                     [(TQ_OP_OR, [0, 1, 2, 3, 4, 5]), (TQ_OP_AND, [0, 1]), (TQ_OP_AND, [2, 0, 3]), (TQ_OP_OR, [4, 5]), (TQ_OP_TERM, [1])]])
    assert (ctx.count_batch(qb) == oi.count_batch(qb)).all()


# ---- tile engine specifics -------------------------------------------------------------------------------------------
def _tile_queries(ix, base):
    qs = []
    for k in (1, 10, 100, 1000):
        for terms in ([0, 5], [0, 4, 5], [1, 0, 5, 3], [5, 4, 3, 2, 1, 0], [0, 1, 2], [2, 3, 4], [3, 5], [4, 5]):
            qs.append(ix.query(TQ_OP_OR, terms, k, segment_base=base))
    return qs


def test_tile_engine_is_what_runs(ctx, synth):
    ix, oi, base = synth
    qb = QueryBatch(_tile_queries(ix, base))
    g = ctx.search_batch(qb)
    assert_same(g, oi.search_batch(qb, mode=0, n_threads=8), qb.nq)
    st = ctx.stats()
    if ctx.engine == "tile":
        assert st["tile_groups"] == 1 and st["units_tile"] > 0 and st["tile_postings"] > 0 and st["tile_fallbacks"] == 0
        assert st["units_or"] == 0  # no per-query union kernel ran
    else:
        assert st["tile_groups"] == 0 and st["units_or"] > 0
        # k <= 128: k_or_strip; the k = 1000 queries take k_or
        assert st["units_or"] > st["units_or_strip"] > 0


@pytest.mark.parametrize("hook", [dict(TQ_TILE_PCAP=64), dict(TQ_TILE_CAND_FLOOR=4), dict(TQ_TILE_SAMPLE_DIV=0, TQ_TILE_CAND_FLOOR=64)])
def test_tile_overflow_is_repeated_on_the_per_query_kernels(synth, hook):
    """A tile with more pairs than its shared-memory buffer, or a query with more candidates than its region, never costs
    exactness: the run is repeated on the per-query kernels (tile_fallbacks == 1) and returns the oracle's rows."""
    ix, oi, base = synth
    c = _ctx_with_env(TQ_TILE=1, **hook)
    try:
        ix.register(c, segment_base=base)
        qb = QueryBatch(_tile_queries(ix, base))
        g = c.search_batch(qb)
        assert_same(g, oi.search_batch(qb, mode=0, n_threads=8), qb.nq)
        assert c.stats()["tile_fallbacks"] == 1
        bt = c.prepare(qb)  # device-resident results take the same route
        bt.run()
        bt.results_dev()
        assert_same(bt.fetch(), g, qb.nq)
        bt.close()
    finally:
        c.close()


@pytest.mark.parametrize("hook", [dict(TQ_TILE_SEG_CAP=8), dict(TQ_TILE_SEG_CAP=3), dict(TQ_TILE_LIGHT_MAX=0), dict(TQ_TILE_LIGHT_MAX=0, TQ_TILE_WINDOWS=8), dict(TQ_TILE_LIGHT_MAX=100000), dict(TQ_TILE_SAMPLE_DIV=0),
                                  dict(TQ_TILE_BIG_MIN=1), dict(TQ_TILE_BIG_MIN=100000), dict(TQ_TILE_UNITS=1), dict(TQ_TILE_ROUND_DIV1=2, TQ_TILE_ROUND_DIV2=2)])
def test_tile_paths_agree(synth, hook):
    """Every route through k_tile gives the same rows: a full work list (further routing rounds per tile; with 3 entries the
    wider unions take the window path), window path only (2 or 8 window warps),
    flat path only, no sample launch, every list dense (bitmap lookups) / every list sparse (binary searches), one CTA per launch,
    other launch cuts."""
    ix, oi, base = synth
    c = _ctx_with_env(TQ_TILE=1, **hook)
    try:
        ix.register(c, segment_base=base)
        qs = _tile_queries(ix, base)
        qs += [ix.query(TQ_OP_AND, terms, k, segment_base=base) for k in (10, 200) for terms in ([0, 1], [0, 3], [1, 4], [0, 5], [2, 3, 4], [0, 1, 2])]
        qs += [ix.query(TQ_OP_TERM, [t], 10, segment_base=base) for t in range(6)]
        qb = QueryBatch(qs)
        assert_same(c.search_batch(qb), oi.search_batch(qb, mode=0, n_threads=8), qb.nq)
        st = c.stats()
        assert st["tile_groups"] == 1
        # without a sample launch the first exact launch hands over every match of its tiles: k = 1000 overflows its candidate
        # region and the batch is repeated on the per-query kernels (still the oracle's rows, asserted above)
        assert st["tile_fallbacks"] == (1 if "TQ_TILE_SAMPLE_DIV" in hook else 0)
    finally:
        c.close()


def test_single_term_batches_take_k_term_unless_they_can_share(synth):
    """Default routing (TQ_TILE_TERMS=2): a batch of nothing but single-term queries streams its lists through k_term; as soon
    as the batch holds a multi-term query the single-term queries ride along on the tile engine.  Same rows either way."""
    ix, oi, base = synth
    c = _ctx_with_env(TQ_TILE=1)
    try:
        ix.register(c, segment_base=base)
        terms = [ix.query(TQ_OP_TERM, [t], k, segment_base=base) for t in range(6) for k in (10, 100)]
        qb = QueryBatch(terms)
        assert_same(c.search_batch(qb), oi.search_batch(qb, mode=0, n_threads=8), qb.nq)
        st = c.stats()
        assert st["tile_groups"] == 0 and st["units_tile"] == 0
        qb = QueryBatch(terms + [ix.query(TQ_OP_OR, [0, 3], 10, segment_base=base)])
        assert_same(c.search_batch(qb), oi.search_batch(qb, mode=0, n_threads=8), qb.nq)
        st = c.stats()
        assert st["tile_groups"] == 1 and st["units_tile"] > 0
    finally:
        c.close()


def test_tile_groups_split_on_capacity(synth):
    """More distinct dense lists than one tile buffer holds: the planner opens further groups (one decode pass each)."""
    ix, oi, base = synth
    c = _ctx_with_env(TQ_TILE=1, TQ_TILE_MAX_DENS_X1000=320)  # {0,5},{0,4,5},{3,5},{4,5} fill the first group; {2,3,4} opens the second
    try:
        ix.register(c, segment_base=base)
        qb = QueryBatch(_tile_queries(ix, base))
        g = c.search_batch(qb)
        assert_same(g, oi.search_batch(qb, mode=0, n_threads=8), qb.nq)
        st = c.stats()
        assert st["tile_groups"] > 1 and st["tile_fallbacks"] == 0
    finally:
        c.close()


def test_topkeys_exchange_matches_plain_run(ctx, synth):
    """The exact cross-shard threshold exchange on one shard: export the k best keys after every phase, feed them back as if
    gathered from n_shards = 1 (and duplicated, n_shards = 2): the rows equal the plain run's."""
    import torch
    ix, oi, base = synth
    qb = QueryBatch(_tile_queries(ix, base)[:16])
    plain = ctx.search_batch(qb)
    kmax = qb.kmax
    for shards in (1, 2):
        keys = torch.zeros((shards, qb.nq, kmax), dtype=torch.int32, device="cuda:0")
        b = ctx.prepare(qb)
        n_phases = b.phases()
        for phase in range(n_phases):
            b.run_phase(phase)
            if phase + 1 < n_phases:
                b.topkeys_export_dev(keys[0].data_ptr(), kmax)
                b.thresholds_from_keys_dev(keys.data_ptr(), shards, kmax)  # shard 1 (if any) reports nothing: zeros
        out = b.fetch()
        b.close()
        for a, c in zip(plain, out):
            assert (a == c).all()


# ---- BASELINE.json configurations at full size (SURVEY.md §8d), one segment of each ------------------------------------
def _zipf_queries(rng, n, n_terms, max_rank):
    ranks = np.arange(1, max_rank + 1)
    prob = (1.0 / ranks) / (1.0 / ranks).sum()
    return [sorted(int(r) for r in rng.choice(ranks, size=n_terms, replace=False, p=prob)) for _ in range(n)]


def test_bench_config_or5_top100_one_full_segment(ctx):
    """configs[2] at its real segment size: 12.5M docs, 5-term unions of Zipf-drawn ranks from {1..1000} (density 0.3 / rank),
    top-100 -- threshold rounds, MaxScore splits and tile maxima all active -- vs the exhaustive oracle, bit for bit."""
    rng = np.random.default_rng(0x7A6E)
    qranks = _zipf_queries(rng, 48, 5, 1000)
    ranks = sorted({r for q in qranks for r in q})
    dens = [min(0.5, 0.3 / r) for r in ranks]
    ix = T.SynthIndex(1, 12_500_000, dens, seed=0x7A6E7469)
    base = fresh_ord()
    ix.register(ctx, segment_base=base)
    oi = O.OracleIndex()
    ix.register(oi, segment_base=base)
    qb = QueryBatch([ix.query(TQ_OP_OR, [ranks.index(r) for r in q], 100, segment_base=base) for q in qranks])
    g = ctx.search_batch(qb)
    assert_same(g, oi.search_batch(qb, mode=0, n_threads=32), qb.nq)
    assert ctx.stats()["tile_fallbacks"] == 0
    ctx.segment_unregister(base, 0)


def test_bench_config_and2_top10_10M(ctx):
    """configs[1]: 10M docs, one segment, the three density pairs of benches/intersection_bench.rs:107-113, top-10."""
    pairs = [(0.10, 0.10), (0.50, 0.02), (0.80, 0.005)]
    dens = [p for ab in pairs for p in ab]
    ix = T.SynthIndex(1, 10_000_000, dens, seed=0x7A6E7469)
    base = fresh_ord()
    ix.register(ctx, segment_base=base)
    oi = O.OracleIndex()
    ix.register(oi, segment_base=base)
    qb = QueryBatch([ix.query(TQ_OP_AND, [2 * i, 2 * i + 1], k, segment_base=base) for i in range(3) for k in (10, 100)])
    assert_same(ctx.search_batch(qb), oi.search_batch(qb, mode=0, n_threads=32), qb.nq)
    ctx.segment_unregister(base, 0)


# ---- the boundary under concurrency, and several devices behind one handle -------------------------------------------
def test_concurrent_callers_on_one_ctx(ctx, synth):
    """rayon threads call collect_segment concurrently (src/core/executor.rs:60-100): 8 host threads x tq_search_batch on ONE
    ctx, new terms (block-table builds), cached terms, an invalid batch in the middle -- every call returns what it returns
    alone, and the failing call poisons nothing."""
    import threading
    ix, oi, base = synth
    batches = []
    for t in range(8):
        qs = [ix.query(TQ_OP_OR, [(t + i) % 6, (t + 2 * i + 1) % 6, 5], 10 + 7 * t, segment_base=base) for i in range(6) if (t + i) % 6 != (t + 2 * i + 1) % 6]
        qs += [ix.query(TQ_OP_AND, [t % 6, (t + 1) % 6], 10, segment_base=base), ix.query(TQ_OP_TERM, [t % 6], 20, segment_base=base)]
        batches.append(QueryBatch(qs))
    expected = [ctx.search_batch(qb) for qb in batches]
    fresh = _ctx_with_env(TQ_TILE=1 if ctx.engine == "tile" else 0)  # nothing cached: the threads race on the table builds
    try:
        ix.register(fresh, segment_base=base)
        results, errors = [None] * 8, []
        bad = dict(ix.query(TQ_OP_TERM, [0], 10, segment_base=base))
        bad["term_segs"] = [(0, 424242, 0, 10, 0, 10)]  # unknown segment: the whole batch fails, after valid queries scheduled builds
        bad_batch = QueryBatch([ix.query(TQ_OP_TERM, [4], 10, segment_base=base), bad])

        def work(t):
            try:
                for rep in range(3):
                    if t == 3 and rep == 1:
                        with pytest.raises(T.TqError):
                            fresh.search_batch(bad_batch)
                    results[t] = fresh.search_batch(batches[t])
            except Exception as e:  # noqa: BLE001
                errors.append(repr(e))

        threads = [threading.Thread(target=work, args=(t,)) for t in range(8)]
        for th in threads:
            th.start()
        for th in threads:
            th.join()
        assert not errors, errors
        for t in range(8):
            for a, b in zip(results[t], expected[t]):
                assert (a == b).all()
        # the term the failing batch had scheduled is searchable afterwards
        assert_same(fresh.search_batch(QueryBatch([ix.query(TQ_OP_TERM, [4], 10, segment_base=base)])),
                    oi.search_batch(QueryBatch([ix.query(TQ_OP_TERM, [4], 10, segment_base=base)]), mode=0), 1)
    finally:
        fresh.close()


def test_segment_churn_recycles_list_ids(ctx):
    """register -> search -> unregister many times (merges): block tables and list ids are reclaimed with the segment."""
    rng = np.random.default_rng(4242)
    before = ctx.stats()["lists_cached"]
    for _ in range(6):
        segs = _random_segments(rng, 2, 4)
        g, c, nq = _run_both(ctx, segs, [make_query(TQ_OP_OR, segs, [0, 1, 2, 3], 10), make_query(TQ_OP_AND, segs, [0, 1], 10)])
        assert_same(g, c, nq)
        for s in segs:
            ctx.segment_unregister(s.segment_ord, 0)
    assert ctx.stats()["lists_cached"] == before


def _multi_check(devices, synth_ix, oi, base):
    m = T.MultiContext(devices)
    try:
        for s in range(synth_ix.n_segments):
            m.segment_register(base + s, 0, synth_ix.max_doc[s], synth_ix.record_option, synth_ix.body(s), synth_ix.fieldnorm(s), None)
        qs = _tile_queries(synth_ix, base)[:24] + [synth_ix.query(TQ_OP_AND, [0, 1], 10, segment_base=base), synth_ix.query(TQ_OP_TERM, [2], 50, segment_base=base)]
        qb = QueryBatch(qs)
        assert_same(m.search_batch(qb), oi.search_batch(qb, mode=0, n_threads=8), qb.nq)
    finally:
        m.close()


def test_multi_handle_two_contexts_one_device(synth):
    """tq_multi with two contexts (here on the same device): segments spread over them, concurrent phases, exact key exchange,
    host merge -- the rows of a single process holding everything."""
    ix, oi, base = synth
    _multi_check([0, 0], ix, oi, base)


def test_multi_handle_two_devices(synth):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    ix, oi, base = synth
    _multi_check([0, 1], ix, oi, base)


# ---- SURVEY.md §8(e): one segment split by doc-id range ---------------------------------------------------------------
def _range_ctx(engine):
    return _ctx_with_env(TQ_TILE=1 if engine == "tile" else 0, TQ_TILE_TERMS=1)


@pytest.mark.parametrize("cuts", [[0, 101_376, 202_752, 300_000], [0, 1, 77_777, 77_780, 262_144, 299_999, 300_000], [0, 0, 300_000]])
def test_doc_range_parts_merge_to_the_whole_segment(ctx, cuts):
    """tq_segment_set_doc_range: every part of a segment (one context each, as on several GPUs) returns the top-k / the Count of its
    docs; merged like segment fruits (merge_fruits) they are the rows of the whole segment.  Cuts inside tiles, inside bytes of the
    alive bitset, one-doc and empty parts; with and without deletes."""
    from tantivy_b200.sharding import merge_rows_host
    ix = T.SynthIndex(1, 300_000, [0.3, 0.05, 0.01, 0.002, 0.0004], seed=31)
    for deletes in (False, True):
        alive = None
        if deletes:
            alive = np.packbits(np.random.default_rng(5).random(300_000) > 0.3, bitorder="little")
        base = fresh_ord()
        oi = O.OracleIndex()
        oi.segment_register(base, 0, ix.max_doc[0], ix.record_option, ix.body(0), ix.fieldnorm(0), alive)
        qs = [ix.query(TQ_OP_TERM, [t], 10, segment_base=base) for t in range(5)]
        qs += [ix.query(TQ_OP_AND, ts, 10, segment_base=base) for ts in ([0, 1], [1, 2], [0, 3])]
        qs += [ix.query(TQ_OP_OR, ts, 50, segment_base=base) for ts in ([0, 1, 2, 3, 4], [3, 4], [1, 4], [2, 3])]
        qb = QueryBatch(qs)
        want = oi.search_batch(qb, mode=0, n_threads=8)
        want_counts = oi.count_batch(qb)
        rows, counts = [], np.zeros(qb.nq, dtype=np.uint64)
        for lo, hi in zip(cuts[:-1], cuts[1:]):
            c = _range_ctx(ctx.engine)
            try:
                c.segment_register(base, 0, ix.max_doc[0], ix.record_option, ix.body(0), ix.fieldnorm(0), alive)
                c.segment_set_doc_range(base, 0, lo, hi)
                r = c.search_batch(qb)
                for q in range(qb.nq):
                    assert all(lo <= d < hi for _, _, d in hits(r, q))
                rows.append([np.array(x) for x in r])
                counts += c.count_batch(qb)
                if ctx.engine == "tile":
                    assert c.stats()["tile_fallbacks"] == 0
            finally:
                c.close()
        assert (counts == want_counts).all(), (counts, want_counts)
        kmax = max(q["k"] for q in qs)
        m = merge_rows_host(np.stack([r[0] for r in rows]), np.stack([r[1] for r in rows]), np.stack([r[2] for r in rows]), np.stack([r[3] for r in rows]), kmax)
        for q in range(qb.nq):
            n = int(want[3][q])
            assert int(m[3][q]) >= n
            assert (m[1][q, :n] == want[1][q, :n]).all() and (m[2][q, :n] == want[2][q, :n]).all()
            assert (m[0][q, :n].view(np.uint32) == want[0][q, :n].view(np.uint32)).all()


def test_doc_range_argument_checks(ctx):
    ix = T.SynthIndex(1, 5000, [0.2], seed=3)
    base = fresh_ord()
    ctx.segment_register(base, 0, ix.max_doc[0], ix.record_option, ix.body(0), ix.fieldnorm(0), None)
    with pytest.raises(T.TqError):
        ctx.segment_set_doc_range(base + 1, 0, 0, 10)      # not registered
    with pytest.raises(T.TqError):
        ctx.segment_set_doc_range(base, 0, 10, 5001)       # beyond max_doc
    with pytest.raises(T.TqError):
        ctx.segment_set_doc_range(base, 0, 20, 10)         # lo > hi
    ctx.segment_set_doc_range(base, 0, 1000, 4000)
    with pytest.raises(T.TqError):
        ctx.segment_set_doc_range(base, 0, 0, 4000)        # a range can only be narrowed
    ctx.segment_set_doc_range(base, 0, 1024, 3000)
    r = ctx.search_batch(QueryBatch([ix.query(TQ_OP_TERM, [0], 1000, segment_base=base)]))
    docs = [d for _, _, d in hits(r, 0)]
    assert docs and min(docs) >= 1024 and max(docs) < 3000
    base2 = fresh_ord()
    ctx.segment_register(base2, 0, ix.max_doc[0], ix.record_option, ix.body(0), ix.fieldnorm(0), None)
    ctx.search_batch(QueryBatch([ix.query(TQ_OP_TERM, [0], 5, segment_base=base2)]))
    with pytest.raises(T.TqError):
        ctx.segment_set_doc_range(base2, 0, 0, 100)        # after the first search on a segment without deletes
    ctx.segment_unregister(base, 0)
    ctx.segment_unregister(base2, 0)


def test_multi_handle_split_segment(synth):
    """tq_multi_segment_register_split: ONE segment over the handle's devices by doc range (here two contexts on one device, and
    next to a whole segment on one of them) -- the rows of a single context holding everything."""
    ix, oi, base = synth
    m = T.MultiContext([0, 0])
    try:
        m.segment_register_split(base + 0, 0, ix.max_doc[0], ix.record_option, ix.body(0), ix.fieldnorm(0), None)
        m.segment_register(base + 1, 0, ix.max_doc[1], ix.record_option, ix.body(1), ix.fieldnorm(1), None)
        m.segment_register_split(base + 2, 0, ix.max_doc[2], ix.record_option, ix.body(2), ix.fieldnorm(2), None)
        qs = _tile_queries(ix, base)[:24] + [ix.query(TQ_OP_AND, [0, 1], 10, segment_base=base), ix.query(TQ_OP_TERM, [2], 50, segment_base=base)]
        qb = QueryBatch(qs)
        assert_same(m.search_batch(qb), oi.search_batch(qb, mode=0, n_threads=8), qb.nq)
    finally:
        m.close()


# ---- N4: mixed boolean shapes (TQ_OP_BOOL) --------------------------------------------------------------------------
def _bool_query(ix_query, occurs, groups=None, msm=0):
    q = dict(ix_query)
    q["op"] = T.TQ_OP_BOOL
    q["term_occur"] = occurs
    if groups is not None:
        q["term_group"] = groups
    q["min_should_match"] = msm
    return q


_BOOL_SHAPES = [  # (terms, occurs, groups, msm): the shapes of benches/and_or_queries.rs:142-155 and of boolean_query/mod.rs
    ([2, 1, 3], [1, 1, 1], [0, 1, 1], 0),            # +c +(b OR d)
    ([0, 2, 5], [1, 1, 1], [0, 1, 1], 0),            # +e +(c OR a)
    ([2, 1, 3, 0], [1, 1, 1, 1], [0, 0, 1, 1], 0),   # +(c OR b) +(d OR e)
    ([0, 1, 4], [1, 0, 0], None, 0),                 # +a b e   (RequiredOptionalScorer)
    ([1, 2, 0], [0, 0, 2], None, 0),                 # b c -a
    ([3, 0, 1], [1, 2, 2], None, 0),                 # +d -a -b (Exclude with two scorers)
    ([1, 2, 3, 4], [1, 1, 0, 2], [7, 7, 9, 9], 0),   # +(b OR c) d -e
    ([0, 1, 2, 3], [1, 0, 0, 0], None, 2),           # +a and at least two of b c d
    ([1, 2, 3, 4], [0, 0, 0, 0], None, 2),           # at least two of b c d e (Disjunction with minimum match)
    ([1, 2], [0, 0], None, 2),                       # as many as there are: they act as MUST clauses
    ([0, 1], [1, 1], None, 0),                       # plain conjunction
    ([3, 4, 5], [0, 0, 0], None, 0),                 # plain union
    ([2], [1], None, 0),                             # +c
    ([2], [2], None, 0),                             # -c alone: nothing
]


def test_mixed_boolean_shapes(ctx, synth):
    if ctx.engine != "tile":
        pytest.skip("TQ_OP_BOOL runs on the tile engine only")
    ix, oi, base = synth
    qs = []
    for k in (1, 10, 300):
        for terms, occ, grp, msm in _BOOL_SHAPES:
            qs.append(_bool_query(ix.query(TQ_OP_OR, terms, k, segment_base=base), occ, grp, msm))
    qb = QueryBatch(qs)
    g, c = ctx.search_batch(qb), oi.search_batch(qb, mode=0, n_threads=8)
    assert_same(g, c, qb.nq)
    n = len(_BOOL_SHAPES)
    assert len(hits(g, 2 * n + 0)) > 0 and hits(g, 2 * n + 13) == []
    # pure shapes return the rows of the specialised paths
    plain = ctx.search_batch(QueryBatch([ix.query(TQ_OP_AND, [0, 1], 300, segment_base=base), ix.query(TQ_OP_OR, [3, 4, 5], 300, segment_base=base)]))
    assert hits(g, 2 * n + 10) == hits(plain, 0) and hits(g, 2 * n + 11) == hits(plain, 1)


def test_mixed_boolean_small_segments_with_deletes_and_absent_terms(ctx):
    if ctx.engine != "tile":
        pytest.skip("TQ_OP_BOOL runs on the tile engine only")
    rng = np.random.default_rng(4711)
    segs = _random_segments(rng, 3, 6, deletes=True)
    segs[1].terms[3] = (0, 0, 0)  # term 3 absent from one segment: an EmptyScorer there
    segs[2].terms[1] = (0, 0, 0)
    queries = []
    for terms, occ, grp, msm in _BOOL_SHAPES:
        for k in (5, 1000):
            queries.append(_bool_query(make_query(TQ_OP_OR, segs, terms, k), occ, grp, msm))
    g, c, nq = _run_both(ctx, segs, queries)
    assert_same(g, c, nq)


def test_count_mixed_boolean_shapes(ctx, synth):
    """searcher.search(&query, &Count) for the mixed shapes (k_count_bool): alive docs matching, vs the oracle's Count."""
    ix, oi, base = synth
    qs = [_bool_query(ix.query(TQ_OP_OR, terms, 1, segment_base=base), occ, grp, msm) for terms, occ, grp, msm in _BOOL_SHAPES]
    qb = QueryBatch(qs)
    g, c = ctx.count_batch(qb), oi.count_batch(qb)
    assert (g == c).all(), (g, c)
    assert g[0] > 0 and g[13] == 0
    rng = np.random.default_rng(815)
    segs = _random_segments(rng, 3, 6, deletes=True)
    segs[0].terms[2] = (0, 0, 0)
    oi2 = both(ctx, segs)
    qb2 = QueryBatch([_bool_query(make_query(TQ_OP_OR, segs, terms, 1), occ, grp, msm) for terms, occ, grp, msm in _BOOL_SHAPES])
    assert (ctx.count_batch(qb2) == oi2.count_batch(qb2)).all()
