"""The per-query union kernels on the default 100M-doc index, in 256-query batches of three shapes: 5-term unions with
k = 100 (k_or_strip), 5-term unions with k = 1000 and 20-term unions with k = 10 (k_or).  Per shape: or_ms of every timed
batch, units_or and units_or_strip, and a check of the first `check` queries against the oracle (exhaustive path, bit-equal
scores).  With an output directory the rows go to <out>/<shape>/*.npy (bench.dump_outputs), so that two builds
(TANTIVY_B200_LIB) can be compared output for output.  Run with TQ_TILE=0, else the tile engine takes the unions.
usage: TQ_TILE=0 python profiles/probe_or_routes.py [out_dir] [steps] [check]"""
import json
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench as B  # noqa: E402
import tantivy_b200 as T  # noqa: E402

out_dir = sys.argv[1] if len(sys.argv) > 1 else None
steps = int(sys.argv[2]) if len(sys.argv) > 2 else 5
check = int(sys.argv[3]) if len(sys.argv) > 3 else 256
seed, nq = 0x7A6E7469, 256
wl = dict(B.WORKLOADS["or5_top100_100M_8seg"])
shapes = {"or5_k100": (5, 100), "or5_k1000": (5, 1000), "or20_k10": (20, 10)}
# one index for every shape: each shape's query plan, its terms mapped into one density list
dens, batches = [], {}
for name, (n_terms, k) in shapes.items():
    d, b = B.build_query_plan(dict(wl, n_terms=n_terms, k=k), nq, 1, seed)
    for p in d:
        if p not in dens:
            dens.append(p)
    batches[name] = [(op, [dens.index(d[t]) for t in terms], k) for op, terms, k in b[0]]
shard = B.make_shard(wl, dens, 0, 1, seed)
ctx = T.Context(0)
shard.register(ctx)
oi = None
if check:
    from oracle import tq_oracle as O
    oi = O.OracleIndex()
    shard.register(oi)
for name, queries in batches.items():
    qb = B.marshal(shard, queries)
    for _ in range(2):  # block tables built, modules loaded
        ctx.search_batch(qb)
    or_ms = []
    for _ in range(steps):
        rows = ctx.search_batch(qb)
        st = ctx.stats()
        or_ms.append(st["or_ms"])
    line = {"shape": name, "or_ms_median": round(float(np.median(or_ms)), 3), "or_ms": [round(x, 3) for x in or_ms],
            "units_or": st["units_or"], "units_or_strip": st["units_or_strip"], "tile_groups": st["tile_groups"]}
    if oi is not None:
        ref = oi.search_batch(B.marshal(shard, queries[:check]), mode=0, n_threads=B.host_info()["threads"])
        bad = 0
        for q in range(min(check, nq)):
            n = int(ref[3][q])
            bad += not (int(rows[3][q]) == n and (rows[1][q, :n] == ref[1][q, :n]).all() and (rows[2][q, :n] == ref[2][q, :n]).all()
                        and (rows[0][q, :n].view(np.uint32) == ref[0][q, :n].view(np.uint32)).all())
        line["oracle"] = {"checked": min(check, nq), "mismatches": bad}
    if out_dir:
        B.dump_outputs(os.path.join(out_dir, name), rows, seed)
    print(json.dumps(line), flush=True)
ctx.close()
