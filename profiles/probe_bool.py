"""Mixed boolean queries (TQ_OP_BOOL) on the default 100M-doc index (the or5_top100_100M_8seg segments), in 256-query batches of
four shapes over Zipf-drawn terms a, b, c, d: `+a +(b OR c)`, `+a b c`, `a b c -d` and two of `a b c d` (min_should_match), k = 100.
Two contexts in one process, alternated step by step: TQ_TILE=0 (the per-query kernel k_bool) and TQ_TILE=1 (the tile engine).
Per shape: the median bool_ms of k_bool, the median tile_ms + score_ms of the tile engine, units_bool, tile_groups, and a check
of the first `check` queries of both engines against the oracle (exhaustive path, bit-equal scores).  The card's name and power
limit are read in the same run.
usage: python profiles/probe_bool.py [steps] [check]"""
import json
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench as B  # noqa: E402
import tantivy_b200 as T  # noqa: E402

steps = int(sys.argv[1]) if len(sys.argv) > 1 else 5
check = int(sys.argv[2]) if len(sys.argv) > 2 else 16
seed, nq, k = 0x7A6E7469, 256, 100
wl = dict(B.WORKLOADS["or5_top100_100M_8seg"])
dens, batches = B.build_query_plan(dict(wl, n_terms=4, k=k), nq, 1, seed)  # four distinct Zipf-drawn terms per query
SHAPES = {  # name: (terms used of a, b, c, d; Occur per term; MUST group per term; min_should_match)
    "+a +(b OR c)": (3, [1, 1, 1], [0, 1, 1], 0),
    "+a b c": (3, [1, 0, 0], None, 0),
    "a b c -d": (4, [0, 0, 0, 2], None, 0),
    "2 of a b c d": (4, [0, 0, 0, 0], None, 2),
}
card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                      capture_output=True, text=True).stdout.strip()
shard = B.make_shard(wl, dens, 0, 1, seed)


def context(tile):
    """tq_ctx_create reads TQ_TILE from the environment."""
    old = os.environ.get("TQ_TILE")
    os.environ["TQ_TILE"] = str(tile)
    try:
        return T.Context(0)
    finally:
        if old is None:
            os.environ.pop("TQ_TILE")
        else:
            os.environ["TQ_TILE"] = old


def bool_batch(n_terms, occurs, groups, msm, count=nq):
    """The batch's queries as one shape, with the global statistics of the index (as ShardedIndex.marshal weighs them)."""
    out = []
    for _, terms, kk in batches[0][:count]:
        terms = terms[:n_terms]
        term_segs = [(clause, g, 0) + tuple(shard.ix.term_info[i][t]) for clause, t in enumerate(terms)
                     for i, g in enumerate(shard.global_ords) if shard.ix.term_info[i][t][0]]
        q = dict(op=T.TQ_OP_BOOL, k=kk, weights=[T.bm25_weight(int(shard.df[t]), shard.total_docs, 1.0) for t in terms],
                 avg_fieldnorm=[shard.avg] * n_terms, term_segs=term_segs, term_occur=occurs, min_should_match=msm)
        if groups is not None:
            q["term_group"] = groups
        out.append(q)
    return T.QueryBatch(out)


def mismatches(rows, ref, n):
    bad = 0
    for q in range(n):
        m = int(ref[3][q])
        bad += not (int(rows[3][q]) == m and (rows[1][q, :m] == ref[1][q, :m]).all() and (rows[2][q, :m] == ref[2][q, :m]).all()
                    and (rows[0][q, :m].view(np.uint32) == ref[0][q, :m].view(np.uint32)).all())
    return bad


per_query, tile = context(0), context(1)
shard.register(per_query)
shard.register(tile)
oi = None
if check:
    from oracle import tq_oracle as O
    oi = O.OracleIndex()
    shard.register(oi)
for name, (n_terms, occurs, groups, msm) in SHAPES.items():
    qb = bool_batch(n_terms, occurs, groups, msm)
    for c in (per_query, tile):
        for _ in range(2):  # block tables built, modules loaded
            c.search_batch(qb)
    bool_ms, tile_ms = [], []
    for _ in range(steps):
        rows_pq = per_query.search_batch(qb)
        st_pq = per_query.stats()
        bool_ms.append(st_pq["bool_ms"])
        rows_t = tile.search_batch(qb)
        st_t = tile.stats()
        tile_ms.append(st_t["tile_ms"] + st_t["score_ms"])
    line = {"shape": name, "k": k, "nq": nq, "bool_ms_median": round(float(np.median(bool_ms)), 3),
            "tile_plus_score_ms_median": round(float(np.median(tile_ms)), 3), "bool_ms": [round(x, 3) for x in bool_ms],
            "units_bool": st_pq["units_bool"], "tile_groups": st_t["tile_groups"], "tile_fallbacks": st_t["tile_fallbacks"],
            "engines_byte_identical": all(a.tobytes() == b.tobytes() for a, b in zip(rows_pq, rows_t)), "card": card}
    if oi is not None:
        ref = oi.search_batch(bool_batch(n_terms, occurs, groups, msm, check), mode=0, n_threads=B.host_info()["threads"])
        line["oracle"] = {"checked": check, "mismatches_k_bool": mismatches(rows_pq, ref, check), "mismatches_tile": mismatches(rows_t, ref, check)}
    print(json.dumps(line), flush=True)
per_query.close()
tile.close()
