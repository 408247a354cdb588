"""Mixed boolean queries (TQ_OP_BOOL) on the per-query kernel k_bool: with TQ_TILE=0, for queries that fit no tile group, and
when an overflowing tile-engine run is repeated.  Every comparison is against the oracle's exhaustive path (mode 0): doc ids,
segment ordinals and scores bit-equal."""
import os
from contextlib import contextmanager

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import tantivy_b200 as T  # noqa: E402
from oracle import tq_oracle as O  # noqa: E402
from tantivy_b200._abi import TQ_OP_AND, TQ_OP_OR, TQ_OP_TERM, QueryBatch  # noqa: E402
from tests.helpers import OracleSegment, hits, make_query  # noqa: E402
from tests.test_gpu_parity import _BOOL_SHAPES, _bool_query, _ctx_with_env, _random_segments, assert_same, fresh_ord  # noqa: E402

_DENS = [0.3, 0.15, 0.05, 0.01, 0.002, 0.0001]


@pytest.fixture(scope="module")
def setup():
    """3 x 1M docs with positions (phrases ride along in the overflow test), on a per-query context, a tile context and the oracle."""
    ix = T.SynthIndex(3, 1_000_000, _DENS, seed=77, record_option=2)
    base = fresh_ord() * 10
    legacy, tile = _ctx_with_env(TQ_TILE=0), _ctx_with_env(TQ_TILE=1)
    oi = O.OracleIndex()
    for target in (legacy, tile, oi):
        ix.register(target, segment_base=base)
    yield ix, oi, base, legacy, tile
    legacy.close()
    tile.close()


def _bool_batch(ix, base, ks):
    return [_bool_query(ix.query(TQ_OP_OR, terms, k, segment_base=base), occ, grp, msm) for k in ks for terms, occ, grp, msm in _BOOL_SHAPES]


def test_shapes_on_the_per_query_kernel(setup):
    ix, oi, base, legacy, _ = setup
    qb = QueryBatch(_bool_batch(ix, base, (1, 10, 300, 1000)))
    g = legacy.search_batch(qb)
    assert_same(g, oi.search_batch(qb, mode=0, n_threads=8), qb.nq)
    st = legacy.stats()
    assert st["units_bool"] > 0 and st["tile_groups"] == 0 and st["units_tile"] == 0 and st["bool_ms"] > 0
    n = len(_BOOL_SHAPES)
    assert len(hits(g, 3 * n)) == 1000 and hits(g, 3 * n + 13) == []


def test_both_engines_return_the_same_rows(setup):
    ix, _, base, legacy, tile = setup
    qb = QueryBatch(_bool_batch(ix, base, (10, 300)))
    a = tile.search_batch(qb)
    st = tile.stats()
    assert st["tile_groups"] >= 1 and st["units_bool"] == 0 and st["tile_fallbacks"] == 0
    b = legacy.search_batch(qb)
    for x, y in zip(a, b):
        assert x.tobytes() == y.tobytes()


def _edge_segment(rng):
    """Lists of 1 / 127 / 128 / 129 docs and two dense ones, docs on both sides of the 4096-doc window edges, max_doc not a multiple
    of the window, and the whole second window deleted."""
    max_doc = 3 * 4096 + 77
    fieldnorms = np.clip(np.round(np.exp(rng.normal(np.log(40), 0.7, size=max_doc))), 1, 4096).astype(np.uint32)
    edge = np.arange(4096 - 63, 4096 + 64, dtype=np.uint32)                                    # 127 docs across the first edge
    lists = [np.array([4095], dtype=np.uint32),
             edge,
             np.unique(np.concatenate([[0, 8191, 8192, max_doc - 1], rng.choice(np.arange(1, 8191), 124, replace=False)])).astype(np.uint32),
             np.concatenate([np.arange(8192 - 64, 8192 + 64), [max_doc - 1]]).astype(np.uint32),
             np.nonzero(rng.random(max_doc) < 0.3)[0].astype(np.uint32),
             np.nonzero(rng.random(max_doc) < 0.6)[0].astype(np.uint32)]
    assert [len(x) for x in lists[:4]] == [1, 127, 128, 129]
    lists = [(d, np.minimum(rng.geometric(0.6, size=len(d)), 40).astype(np.uint32)) for d in lists]
    alive_bits = rng.random(max_doc) > 0.1
    alive_bits[4096:8192] = False
    return OracleSegment(lists, fieldnorms, segment_ord=fresh_ord(), writer_cls=T.FieldWriter, alive=np.packbits(alive_bits, bitorder="little"))


def test_small_segments_window_edges_deletes_and_non_prunable_weights(setup):
    """Random small segments with deletes and absent terms plus the edge segment; every shape also with a weight-0 clause and
    with a negative boost on one clause, so that the bound skip is off (not every weight finite and >= 0)."""
    _, _, _, legacy, _ = setup
    rng = np.random.default_rng(4712)
    segs = _random_segments(rng, 3, 6, deletes=True) + [_edge_segment(rng)]
    segs[1].terms[3] = (0, 0, 0)  # term 3 absent from one segment
    segs[2].terms[1] = (0, 0, 0)
    oi = O.OracleIndex()
    for s in segs:
        s.register(oi)
        s.register(legacy)
    queries = []
    for terms, occ, grp, msm in _BOOL_SHAPES:
        for k in (5, 1000):
            q = _bool_query(make_query(TQ_OP_OR, segs, terms, k), occ, grp, msm)
            queries.append(q)
            zero = dict(q, weights=list(q["weights"]))
            zero["weights"][-1] = 0.0
            queries.append(zero)
            neg = dict(q, weights=list(q["weights"]))
            neg["weights"][0] = -neg["weights"][0]
            queries.append(neg)
    for tail in ([3, 4], [0, 2, 5], [1, 3]):  # the 1- / 127- / 128- / 129-doc lists against the dense ones
        queries.append(_bool_query(make_query(TQ_OP_OR, segs, tail + [4, 5], 50), [1] * len(tail) + [0, 2], None, 0))
        queries.append(_bool_query(make_query(TQ_OP_OR, segs, [5] + tail, 50), [1] + [0] * len(tail), None, 0))
    qb = QueryBatch(queries)
    g = legacy.search_batch(qb)
    assert_same(g, oi.search_batch(qb, mode=0), qb.nq)
    assert legacy.stats()["units_bool"] > 0
    for s in segs:
        legacy.segment_unregister(s.segment_ord, 0)


def _mixed_batch(ix, base):
    qs = [ix.query(TQ_OP_TERM, [t], 10, segment_base=base) for t in (1, 4)]
    qs += [ix.query(TQ_OP_AND, terms, k, segment_base=base) for terms, k in (([0, 1], 10), ([1, 3], 100))]
    qs += [ix.query(TQ_OP_OR, terms, k, segment_base=base) for k in (10, 1000) for terms in ([0, 5], [1, 0, 5, 3], [2, 3, 4])]
    qs += _bool_batch(ix, base, (10, 1000))
    qs += [ix.phrase_query(terms, k, segment_base=base) for terms, k in (([0, 1], 10), ([1, 0, 2], 100))]
    return qs


@pytest.mark.parametrize("hook", [dict(TQ_TILE_PCAP=64), dict(TQ_TILE_CAND_FLOOR=4)])
def test_overflow_is_repeated_exactly_with_bool_queries(setup, hook):
    """A tile-engine run that overflows a tile buffer or a candidate region is repeated on the per-query kernels, BOOL queries
    included (k_bool): the oracle's rows, through search_batch and through prepare / run / results_dev / fetch."""
    ix, oi, base, _, _ = setup
    c = _ctx_with_env(TQ_TILE=1, **hook)
    try:
        ix.register(c, segment_base=base)
        qb = QueryBatch(_mixed_batch(ix, base))
        g = c.search_batch(qb)
        assert_same(g, oi.search_batch(qb, mode=0, n_threads=8), qb.nq)
        # (the counters describe the tile-engine run; the repeat on the per-query kernels only sets tile_fallbacks)
        assert c.stats()["tile_fallbacks"] == 1
        bt = c.prepare(qb)
        bt.run()
        bt.results_dev()
        assert_same(bt.fetch(), g, qb.nq)
        bt.close()
    finally:
        c.close()


def test_query_that_fits_no_tile_group(setup):
    """A BOOL query too dense for any tile group (here: a cap on a group's expected pairs per doc; the slot cap cannot go below
    64 lists, more than a query holds) runs on k_bool next to the queries the tile engine took."""
    ix, oi, base, _, _ = setup
    c = _ctx_with_env(TQ_TILE=1, TQ_TILE_MAX_DENS_X1000=100)  # {3,4}, {4,5}, {3,5} and +d e f fit; the shapes over a, b, c do not
    try:
        ix.register(c, segment_base=base)
        qs = [ix.query(TQ_OP_OR, terms, 10, segment_base=base) for terms in ([3, 4], [4, 5], [3, 5])]
        qs += _bool_batch(ix, base, (10, 100))
        qb = QueryBatch(qs)
        assert_same(c.search_batch(qb), oi.search_batch(qb, mode=0, n_threads=8), qb.nq)
        st = c.stats()
        assert st["tile_groups"] >= 1 and st["units_bool"] > 0 and st["tile_fallbacks"] == 0
    finally:
        c.close()


def test_initial_threshold_on_bool_queries(setup):
    """TQ_QUERY_HAS_THRESHOLD (a `threshold` entry): only docs scoring strictly above it are collected."""
    ix, oi, base, legacy, _ = setup
    base_queries = _bool_batch(ix, base, (20,))
    g0 = legacy.search_batch(QueryBatch(base_queries))
    queries = []
    for i, q in enumerate(base_queries):
        h = hits(g0, i)
        for thr in ([h[len(h) // 2][0], h[-1][0]] if h else []) + [0.0, -1.0, 1e9]:
            queries.append(dict(q, k=50, threshold=float(thr)))
    qb = QueryBatch(queries)
    g = legacy.search_batch(qb)
    assert_same(g, oi.search_batch(qb, mode=0, n_threads=8), qb.nq)
    for i, q in enumerate(queries):
        assert all(s > np.float32(q["threshold"]) for s, _, _ in hits(g, i))


def test_topkeys_exchange_matches_plain_run(setup):
    import torch
    ix, _, base, legacy, _ = setup
    qb = QueryBatch(_bool_batch(ix, base, (10, 300)))
    plain = legacy.search_batch(qb)
    kmax = qb.kmax
    for shards in (1, 2):
        keys = torch.zeros((shards, qb.nq, kmax), dtype=torch.int32, device="cuda:0")
        b = legacy.prepare(qb)
        n_phases = b.phases()
        for phase in range(n_phases):
            b.run_phase(phase)
            if phase + 1 < n_phases:
                b.topkeys_export_dev(keys[0].data_ptr(), kmax)
                b.thresholds_from_keys_dev(keys.data_ptr(), shards, kmax)
        out = b.fetch()
        b.close()
        for a, c in zip(plain, out):
            assert (a == c).all()


@contextmanager
def _env(**env):
    old = {k: os.environ.get(k) for k in env}
    os.environ.update({k: str(v) for k, v in env.items()})
    try:
        yield
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


def test_multi_context_whole_and_split_segments(setup):
    ix, oi, base, _, _ = setup
    with _env(TQ_TILE=0):
        m = T.MultiContext([0, 0])
    try:
        m.segment_register_split(base + 0, 0, ix.max_doc[0], ix.record_option, ix.body(0), ix.fieldnorm(0), None)
        m.segment_register(base + 1, 0, ix.max_doc[1], ix.record_option, ix.body(1), ix.fieldnorm(1), None)
        m.segment_register(base + 2, 0, ix.max_doc[2], ix.record_option, ix.body(2), ix.fieldnorm(2), None)
        qb = QueryBatch(_bool_batch(ix, base, (10, 300)))
        assert_same(m.search_batch(qb), oi.search_batch(qb, mode=0, n_threads=8), qb.nq)
    finally:
        m.close()


def test_doc_range_parts_merge_to_the_whole_segment():
    from tantivy_b200.sharding import merge_rows_host
    ix = T.SynthIndex(1, 300_000, [0.3, 0.05, 0.01, 0.002, 0.0004, 0.15], seed=31)
    alive = np.packbits(np.random.default_rng(5).random(300_000) > 0.3, bitorder="little")
    base = fresh_ord()
    oi = O.OracleIndex()
    oi.segment_register(base, 0, ix.max_doc[0], ix.record_option, ix.body(0), ix.fieldnorm(0), alive)
    qb = QueryBatch(_bool_batch(ix, base, (10, 100)))
    want = oi.search_batch(qb, mode=0, n_threads=8)
    cuts = [0, 1, 77_777, 77_780, 262_144, 299_999, 300_000]
    rows = []
    for lo, hi in zip(cuts[:-1], cuts[1:]):
        c = _ctx_with_env(TQ_TILE=0)
        try:
            c.segment_register(base, 0, ix.max_doc[0], ix.record_option, ix.body(0), ix.fieldnorm(0), alive)
            c.segment_set_doc_range(base, 0, lo, hi)
            r = c.search_batch(qb)
            for q in range(qb.nq):
                assert all(lo <= d < hi for _, _, d in hits(r, q))
            rows.append([np.array(x) for x in r])
        finally:
            c.close()
    m = merge_rows_host(np.stack([r[0] for r in rows]), np.stack([r[1] for r in rows]), np.stack([r[2] for r in rows]), np.stack([r[3] for r in rows]), qb.kmax)
    for q in range(qb.nq):
        n = int(want[3][q])
        assert int(m[3][q]) >= n
        assert (m[1][q, :n] == want[1][q, :n]).all() and (m[2][q, :n] == want[2][q, :n]).all()
        assert (m[0][q, :n].view(np.uint32) == want[0][q, :n].view(np.uint32)).all()


def _probe_shapes(terms):
    """The four shapes of profiles/probe_bool.py over four term ordinals a, b, c, d: (name, terms, occurs, groups, msm)."""
    a, b, c, d = terms
    return [("+a +(b OR c)", [a, b, c], [1, 1, 1], [0, 1, 1], 0),
            ("+a b c", [a, b, c], [1, 0, 0], None, 0),
            ("a b c -d", [a, b, c, d], [0, 0, 0, 2], None, 0),
            ("2 of a b c d", [a, b, c, d], [0, 0, 0, 0], None, 2)]


def test_bench_sized_segment(setup):
    """One 12.5M-doc segment at the benchmark's densities (0.3 / Zipf rank, ranks 1..1000), 48 BOOL queries of the four probe
    shapes, k = 10 and 100, on k_bool."""
    _, _, _, legacy, _ = setup
    rng = np.random.default_rng(0xB001)
    ranks_all = np.arange(1, 1001)
    prob = (1.0 / ranks_all) / (1.0 / ranks_all).sum()
    qranks = [[int(r) for r in rng.choice(ranks_all, size=4, replace=False, p=prob)] for _ in range(12)]
    ranks = sorted({r for q in qranks for r in q})
    ix = T.SynthIndex(1, 12_500_000, [min(0.5, 0.3 / r) for r in ranks], seed=0x7A6E7469)
    base = fresh_ord()
    ix.register(legacy, segment_base=base)
    oi = O.OracleIndex()
    ix.register(oi, segment_base=base)
    queries = []
    for i, q in enumerate(qranks):
        for _, terms, occ, grp, msm in _probe_shapes([ranks.index(r) for r in q]):
            queries.append(_bool_query(ix.query(TQ_OP_OR, terms, (10, 100)[i % 2], segment_base=base), occ, grp, msm))
    assert len(queries) == 48
    qb = QueryBatch(queries)
    g = legacy.search_batch(qb)
    assert_same(g, oi.search_batch(qb, mode=0, n_threads=8), qb.nq)
    assert legacy.stats()["units_bool"] > 0
    legacy.segment_unregister(base, 0)
