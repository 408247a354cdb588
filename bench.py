#!/usr/bin/env python
"""bench.py — queries/sec of the posting-decode -> AND/OR -> BM25 -> top-k hot path on B200.

One "step" = one batch of synthetic queries through the whole hot path.  Default workload =
BASELINE.json configs[2], the configuration the metric is quoted on (100M-doc index):
5-term OR (Zipf-drawn ranks from {1..1000}), top-100, 100M docs in 8 segments, on ONE B200.
With --gpus N (torchrun, one rank per GPU) the SAME index is sharded by segment over the ranks
(strong scaling); every step ends with an NCCL all-gather of the ranks' top-k rows and a device
merge (merge_fruits).

value : whole-job queries/s with the batch descriptors already resident in HBM (kernels only).
e2e   : the same through tq_search_batch with HOST buffers (H2D descriptors + D2H results inside
        the timed region) — the number to compare with the reference arm.
parity: after the timed legs a sample of the queries the bench just timed is re-run on the CPU oracle's
        exhaustive path over the WHOLE index (all segments, also at N > 1) and compared row by row
        (doc, segment: equal; score: bit-equal) with what the GPU arm returned.
--impl reference : the reference's CPU algorithm (oracle/ restatement of tantivy's Block-WAND path;
        the Rust crate itself cannot be built here) on all host cores, same workload/metric.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (op, n_segments, docs_per_segment, k, description)
    "or5_top100_100M_8seg": dict(op="or", n_segments=8, docs_per_segment=12_500_000, k=100, n_terms=5, max_rank=1000,
                                 desc="BASELINE.json configs[2]: 5-term OR, top-100, 100M docs, 8 segments"),
    "and2_top10_10M_1seg": dict(op="and", n_segments=1, docs_per_segment=10_000_000, k=10, n_terms=2, max_rank=0,
                                desc="BASELINE.json configs[1]: 2-term AND, top-10, 10M docs, 1 segment"),
    "term_top10_1M_1seg": dict(op="term", n_segments=1, docs_per_segment=1_000_000, k=10, n_terms=1, max_rank=0,
                               desc="BASELINE.json configs[0]: single-term top-10, 1M docs, 1 segment"),
    "or20_top10_500M_64seg": dict(op="or", n_segments=64, docs_per_segment=7_812_500, k=10, n_terms=20, max_rank=10_000,
                                  desc="BASELINE.json configs[4]: 20-term OR, top-10, 500M docs, 64 segments (8 per GPU at N=8)"),
    "mixed_top10_100M_8seg": dict(op="mixed", n_segments=8, docs_per_segment=12_500_000, k=10, n_terms=0, max_rank=1000, record_option=2,
                                  desc="BASELINE.json configs[3]: search-benchmark-game shape, 35% 2-term AND, 35% 2-4-term OR, 15% term, 15% 2-3-term phrase, top-10, "
                                       "100M docs with positions, 8 segments"),
}
AND_PAIRS = [(0.10, 0.10), (0.50, 0.02), (0.80, 0.005)]     # benches/intersection_bench.rs:107-113
TERM_LADDER = [0.0001, 0.01, 0.05, 0.15, 0.30]              # benches/and_or_queries.rs:134-140
ZIPF_C = 0.30                                               # rank 1 ~ 30 % (SURVEY.md §8d)


def zipf_density(rank):
    return min(0.5, ZIPF_C / rank)


def build_query_plan(wl, nq, n_batches, seed):
    """Returns (densities list, batches) where a batch is a list of (op, [term indices], k)."""
    rng = np.random.default_rng(seed)
    dens, index_of = [], {}

    def term(p):
        key = round(p, 12)
        if key not in index_of:
            index_of[key] = len(dens)
            dens.append(p)
        return index_of[key]

    if wl["max_rank"]:
        ranks = np.arange(1, wl["max_rank"] + 1)
        prob = (1.0 / ranks) / (1.0 / ranks).sum()
    batches = []
    for _ in range(n_batches):
        qs = []
        for _ in range(nq):
            op = wl["op"]
            if op == "mixed":
                u = rng.random()
                op = "and" if u < 0.35 else ("or" if u < 0.70 else ("term" if u < 0.85 else "phrase"))
                nt = 2 if op == "and" else (int(rng.integers(2, 5)) if op == "or" else (1 if op == "term" else int(rng.integers(2, 4))))
            else:
                nt = wl["n_terms"]
            if wl["max_rank"]:
                rs = rng.choice(ranks, size=nt, replace=False, p=prob)
                terms = [term(zipf_density(int(r))) for r in rs]
            elif op == "and":
                a, b = AND_PAIRS[int(rng.integers(0, len(AND_PAIRS)))]
                terms = [term(a), term(b * (1 + 1e-9))]  # distinct lists even when a == b
            else:
                terms = [term(TERM_LADDER[int(rng.integers(0, len(TERM_LADDER)))])]
            qs.append((op, terms, wl["k"]))
        batches.append(qs)
    return dens, batches


OPS = {"term": 0, "and": 1, "or": 2, "phrase": 3}


def make_shard(wl, dens, rank, world, seed, dist=None, device=None):
    """This rank's segments of the synthetic index (segment s always has seed base+s) + global statistics."""
    import tantivy_b200 as T
    from tantivy_b200.sharding import ShardedIndex, assign_parts
    units = assign_parts(wl["n_segments"], world, rank)  # whole segments round-robin; fewer segments than ranks: doc-range parts
    ords = [u[0] for u in units]
    t0 = time.time()
    # (segment s of the index always has seed base + s: local segment i is global segment ords[0] + i * stride)
    stride = world if wl["n_segments"] >= world else wl["n_segments"]
    ix = T.SynthIndex(len(ords), wl["docs_per_segment"], dens, seed=seed, segment_base=ords[0], segment_stride=stride,
                      record_option=wl.get("record_option", 1)) if ords else None
    shard = ShardedIndex(ix, ords, len(dens), dist, device, parts=[(u[1], u[2]) for u in units])
    shard.gen_s = time.time() - t0
    return shard


def marshal(shard, queries):
    return shard.marshal([(OPS[op], terms, k) for op, terms, k in queries])


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    def __init__(self, device):
        self.device, self.rows, self.proc = device, [], None

    def start(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown," \
            "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.device}", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = [float(r[0]) for r in self.rows if len(r) >= 8 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 8 and r[1].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 8:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm)}


def host_info():
    """Threads this process may use (affinity / cgroup quota), CPU model."""
    try:
        threads = len(os.sched_getaffinity(0))
    except AttributeError:
        threads = os.cpu_count() or 1
    quota = None
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            quota = float(q) / float(per)
            threads = max(1, min(threads, int(quota)))
    except Exception:
        pass
    model = "unknown"
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                model = line.split(":", 1)[1].strip()
                break
    except Exception:
        pass
    return {"threads": threads, "cpu_model": model, "cpu_count": os.cpu_count(), "cgroup_cpu_quota": quota}


def parity_check(wl, dens, seed, queries, rows, threads):
    """rows = (scores, segs, docs, counts) the GPU arm returned for `queries` (a prefix of a timed batch).  The oracle's
    exhaustive path (mode 0: canonical truth, DESIGN.md §5) runs over the whole index; docs and segments must be equal and
    scores bit-equal."""
    from oracle import tq_oracle as O
    full = make_shard(wl, dens, 0, 1, seed)
    oi = O.OracleIndex()
    full.register(oi)
    qb = marshal(full, queries)
    t0 = time.perf_counter()
    ref = oi.search_batch(qb, mode=0, n_threads=threads)
    mism, rows_checked = 0, 0
    first = None
    for q in range(len(queries)):
        n = int(ref[3][q])
        rows_checked += n
        ok = int(rows[3][q]) == n and (np.asarray(rows[1][q][:n], dtype=np.uint32) == ref[1][q, :n]).all() and \
            (np.asarray(rows[2][q][:n], dtype=np.uint32) == ref[2][q, :n]).all() and \
            (np.asarray(rows[0][q][:n], dtype=np.float32).view(np.uint32) == ref[0][q, :n].view(np.uint32)).all()
        if not ok:
            mism += 1
            first = q if first is None else first
    return {"checked": len(queries), "rows": rows_checked, "mismatches": mism, "first_mismatch": first, "oracle": "oracle/ mode 0 (exhaustive, canonical order), whole index",
            "score_compare": "bit-equal", "oracle_s": round(time.perf_counter() - t0, 2)}


DUMP_LIMIT_BYTES = 64_000_000 - 4096  # 64 MB in all, the five .npy headers included


def dump_outputs(path, rows, seed):
    """Writes one step's result rows so that two builds can be compared output for output: scores.npy (float32 [n, k]),
    segment_ords.npy, docs.npy (float64 [n, k], exact for u32), counts.npy and queries.npy (float64 [n]: the rows' positions in
    the batch).  Entries past a query's count are zero.  When the batch's rows exceed DUMP_LIMIT_BYTES, n is a sample of the
    queries drawn from `seed`, the same for every run with the same arguments."""
    scores, segs, docs, counts = (np.asarray(a) for a in rows)
    nq, k = scores.shape
    row_bytes = k * (4 + 8 + 8) + 8 + 8
    queries = np.arange(nq)
    if nq * row_bytes > DUMP_LIMIT_BYTES:
        queries = np.sort(np.random.default_rng(seed).choice(nq, DUMP_LIMIT_BYTES // row_bytes, replace=False))
    valid = np.arange(k)[None, :] < np.minimum(counts[queries], k)[:, None]
    os.makedirs(path, exist_ok=True)
    out = {"scores": np.where(valid, scores[queries], 0).astype(np.float32),
           "segment_ords": np.where(valid, segs[queries], 0).astype(np.float64),
           "docs": np.where(valid, docs[queries], 0).astype(np.float64),
           "counts": counts[queries].astype(np.float64),
           "queries": queries.astype(np.float64)}
    for name, a in out.items():
        np.save(os.path.join(path, name + ".npy"), a)


def cpu_reference_run(wl, shard, batches, steps, warmup, sample_queries, threads):
    """The reference CPU algorithm (oracle restatement, Block-WAND + TopNHeap + merge_top_k), all host
    cores, on a bounded sample of the same query stream. One step = `sample_queries` queries."""
    from oracle import tq_oracle as O
    oi = O.OracleIndex()
    shard.register(oi)
    flat = [q for b in batches for q in b]
    times = []
    for i in range(warmup + steps):
        qs = [flat[(i * sample_queries + j) % len(flat)] for j in range(sample_queries)]
        qb = marshal(shard, qs)
        t0 = time.perf_counter()
        oi.search_batch(qb, mode=1, n_threads=threads)
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    total = sum(times)
    return sample_queries * len(times) / total, 1000.0 * total / len(times)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=12)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="or5_top100_100M_8seg", choices=sorted(WORKLOADS))
    ap.add_argument("--nq", type=int, default=512, help="queries per step (batch)")
    ap.add_argument("--batches", type=int, default=4, help="distinct query batches cycled through the steps")
    ap.add_argument("--docs-per-segment", type=int, default=0, help="override (smoke runs); 0 = the workload's size")
    ap.add_argument("--seed", type=int, default=0x7A6E7469)
    ap.add_argument("--cpu-sample", type=int, default=0, help="queries in the cpu_baseline sample (0 = auto, ~10-30 s)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--parity-queries", type=int, default=32, help="queries of the first timed batch re-checked on the oracle (0 = off)")
    ap.add_argument("--in-flight", type=int, default=0, choices=[0, 1, 2],
                    help="batches in flight per GPU in the timed legs (2: step i+1 is queued on its own stream before the host waits for step i; "
                         "0 = auto: 2 on one GPU, 1 at N > 1, where queueing step i+1 early skews the ranks between the key exchanges of step i "
                         "and measured 4 %% slower at N = 2)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the rows the last timed step returned (scores, segment ords, docs, counts) as DIR/<name>.npy, "
                         "float32 / float64, at most 64 MB (a seeded sample of the queries beyond that)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the product arm's rows; the reference arm times a sample of the query stream")
    if args.warmup < 3:
        args.warmup = 3

    wl = dict(WORKLOADS[args.workload])
    if args.docs_per_segment:
        wl["docs_per_segment"] = args.docs_per_segment
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    hinfo = host_info()
    host_threads = hinfo["threads"]
    dens, batches = build_query_plan(wl, args.nq, args.batches, args.seed)
    # identical in both arms (the driver compares them); everything measured goes to `workload_stats`
    config = {"workload": args.workload, "desc": wl["desc"], "queries_per_step": args.nq, "docs": wl["n_segments"] * wl["docs_per_segment"],
              "segments": wl["n_segments"], "k": wl["k"], "vocab_terms_materialised": len(dens),
              "sharding": f"segments round-robin over {args.gpus} rank(s)" if wl["n_segments"] >= args.gpus else
                          f"{wl['n_segments']} segment(s) split by doc-id range into {args.gpus // wl['n_segments']} parts each, one per rank",
              "l2_policy": "inputs larger than L2: every step streams the index's posting bytes plus its (doc, score) pair scratch (see workload_stats)"}

    # ------------------------------------------------------------------ reference arm (CPU)
    if args.impl == "reference":
        if rank != 0:
            return 0
        shard = make_shard(wl, dens, 0, 1, args.seed)
        # several queries per host thread, so that the threads stay busy while the heavy queries of the sample finish
        sample = args.cpu_sample or min(512, max(64, 4 * host_threads))
        qps, ms = cpu_reference_run(wl, shard, batches, args.steps, args.warmup, sample, host_threads)
        line = {"metric": "queries/sec", "value": qps, "unit": "queries/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "impl": "reference", "config": config,
                "cpu_baseline": {"value": qps, "unit": "queries/s", "cores": host_threads, "kind": "port", "host": hinfo,
                                 "sample": f"{sample} queries per step of the same query stream, all host threads, "
                                           "Block-WAND + TopNHeap + merge_top_k restatement (oracle/, mode=1)"},
                "e2e": {"value": qps, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return 0

    # ------------------------------------------------------------------ our arm (B200)
    import torch
    import tantivy_b200 as T
    dist = None
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    else:
        torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)

    def barrier_sync():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    shard = make_shard(wl, dens, rank, world, args.seed, dist, dev)
    ctx = T.Context(local_rank)
    shard.register(ctx)
    qbs = [marshal(shard, b) for b in batches]
    k = wl["k"]
    nq = args.nq
    n_total = args.warmup + args.steps

    depth = args.in_flight or (2 if world == 1 else 1)  # (both timed legs)
    mergers = []
    if world > 1:
        from tantivy_b200.sharding import CrossGpuMerger
        # NCCL all-gathers + device merge (K7); one set of exchange buffers per batch in flight, ONE process group: every rank
        # issues the collectives of the batches in the same program order
        mergers = [CrossGpuMerger(ctx, dist, dev, nq, k) for _ in range(depth)]
    cross_gpu_merge = mergers[0] if mergers else None

    # ---- leg 1: `value` — descriptors resident, kernels only -----------------------------------------
    prepared = [ctx.prepare(qb) for qb in qbs]  # also warms the block-table cache; cycled through the steps
    n_prep = len(prepared)
    assert n_prep >= depth or depth == 1

    def run_step(bt):
        if world > 1:
            cross_gpu_merge.run(bt)      # phases + exact threshold exchange (NCCL on the batch's stream)
            rows = cross_gpu_merge(bt)   # packed all-gather + device merge
            torch.cuda.synchronize()
            return rows
        bt.run()
        bt.results_dev()  # waits for the step
        return None

    def submit(bt, slot):
        """Queues one whole step on the batch's own stream and returns without waiting."""
        if world > 1:
            mergers[slot].run(bt)            # phases + key exchanges
            mergers[slot].finish_async(bt)   # pack + all-gather + merge (+ every rank's overflow flags)
        else:
            bt.run()

    def complete(bt, slot, out=None, rows_to_host=False):
        """Waits for a submitted step; rows to host buffers when asked (e2e leg)."""
        if world > 1:
            return mergers[slot].complete(bt, rows_to_host=rows_to_host)
        if out is not None:
            return bt.fetch(out)[0:4]
        bt.results_dev()
        return None

    barrier_sync()
    for i in range(args.warmup):
        run_step(prepared[i % n_prep])
    barrier_sync()
    # (a) serialised steps (one batch at a time, a synchronisation per step): the per-kind device times of the kernels come from
    # here -- CUDA events recorded by the library on the stream each kernel is launched on; the intervals of a step do not overlap
    kinds = ("score_ms", "tile_ms", "theta_ms", "phrase_ms", "term_ms", "and_ms", "or_ms", "final_ms", "kernel_ms")
    kern = {name: [] for name in kinds}
    launches = 0
    stats = None
    touched0 = ctx.stats()["or_windows"][5]  # cumulative bytes the pruned per-query union kernel actually read
    fallbacks = 0
    t0 = time.perf_counter()
    for i in range(args.warmup, n_total):
        run_step(prepared[i % n_prep])
        stats = ctx.stats()
        for key in kern:
            kern[key].append(stats[key])
        fallbacks += stats["tile_fallbacks"]
        launches += stats["kernel_launches"] + (7 if world > 1 else 0)  # + 3 x (key export + threshold import), cross-GPU merge
    barrier_sync()
    dt_value_serial = time.perf_counter() - t0
    # (b) the timed `value` steps: the same K steps with `depth` batches in flight -- step i+1 (another prepared batch, its own stream
    # and scratch) is queued before the host waits for step i, so the GPU fills the tails of step i's launches and the waits of
    # its cross-rank exchanges with step i+1's first kernels.  Every step still runs every kernel; nothing is cached across steps.
    def pipelined_steps(first, count):
        pending = []
        for j in range(count):
            bt, slot = prepared[(first + j) % n_prep], j % depth
            submit(bt, slot)
            pending.append((bt, slot))
            if len(pending) >= depth:
                complete(*pending.pop(0))
        while pending:
            complete(*pending.pop(0))

    pipelined_steps(0, args.warmup)
    barrier_sync()
    sampler = ClockSampler(local_rank) if rank == 0 else None  # one sampler per job, not per rank
    if sampler:
        sampler.start()
    t0 = time.perf_counter()
    pipelined_steps(args.warmup, args.steps)
    barrier_sync()
    dt_value = time.perf_counter() - t0
    touched_per_step = (stats["or_windows"][5] - touched0) / max(args.steps, 1) if stats else 0
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0:  # the rows of the last timed step, read back after the timed region
        if world > 1:
            m = mergers[(args.steps - 1) % depth]
            last_rows = m._host_views(m.rows_o.cpu().numpy())
        else:
            last_rows = prepared[(args.warmup + args.steps - 1) % n_prep].fetch()
        dump_outputs(args.dump_outputs, last_rows, args.seed)
    for b in prepared:
        b.close()

    # ---- leg 2: `e2e` — public API with host buffers ---------------------------------------------------
    outs = [qbs[i % len(qbs)].alloc_out() for i in range(2)]
    h2d = d2h = 0
    parity_rows = None
    barrier_sync()
    for i in range(args.warmup):
        ctx.search_batch(qbs[i % len(qbs)], outs[i % 2])
    barrier_sync()
    # (a) one call per step, nothing overlapped: tq_search_batch (N=1) / prepare + phases + exchange + merge + read-back (N>1)
    def e2e_serial_step(bt):
        cross_gpu_merge.run(bt)
        cross_gpu_merge(bt)
        if rank == 0:
            cross_gpu_merge.fetch_host(bt)
        else:
            torch.cuda.synchronize()
        bt.close()

    t0 = time.perf_counter()
    for i in range(args.steps):
        if world == 1:
            ctx.search_batch(qbs[i % len(qbs)], outs[i % 2])
        else:
            e2e_serial_step(ctx.prepare(qbs[i % len(qbs)]))
    barrier_sync()
    dt_e2e_serial = time.perf_counter() - t0
    # (b) the same work with `depth` batches in flight: while step i runs on the GPU the host plans step i+1 (tq_batch_prepare: host
    # planning + H2D of its descriptors) and queues it, then waits for step i and reads its rows back (D2H).  Every step still
    # plans, copies its descriptors up and its rows down inside the timed region.
    def e2e_pipelined(count):
        nonlocal h2d, d2h, parity_rows
        cur = ctx.prepare(qbs[0])
        submit(cur, 0)
        for i in range(count):
            nxt = ctx.prepare(qbs[(i + 1) % len(qbs)]) if i + 1 < count else None  # host planning + H2D while step i runs
            if nxt is not None and depth > 1:
                submit(nxt, (i + 1) % depth)
            res = complete(cur, i % depth, out=outs[i % 2], rows_to_host=(rank == 0))
            st = ctx.stats()
            h2d = st["h2d_bytes"]
            d2h = st["d2h_bytes"] if world == 1 else (sum(a.nbytes for a in res) if res is not None else 0)
            if i == 0 and args.parity_queries and (world == 1 or res is not None):
                rows = outs[0][1:] if world == 1 else res
                parity_rows = [np.array(x[:args.parity_queries]) for x in rows]
            cur.close()
            if nxt is not None and depth == 1:
                submit(nxt, 0)
            cur = nxt

    t0 = time.perf_counter()
    e2e_pipelined(args.steps)
    barrier_sync()
    dt_e2e = time.perf_counter() - t0

    # max over ranks
    if dist is not None:
        t = torch.tensor([dt_value, dt_e2e, dt_e2e_serial, dt_value_serial], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dt_value, dt_e2e, dt_e2e_serial, dt_value_serial = float(t[0]), float(t[1]), float(t[2]), float(t[3])

    if rank == 0:
        value = nq * args.steps / dt_value
        e2e = nq * args.steps / dt_e2e
        # roofline of the dominant kernel (this rank's launches; at N > 1 every rank runs the same kernels on its shard)
        peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
        if os.path.exists(peaks_path):
            peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (of measured)"
        else:
            peak, peak_src = 6650.0, "B200_PROFILING.md fallback 6.65 TB/s (of fallback)"
        ms = {name[:-3]: float(np.mean(kern[name])) for name in kinds}
        per_kernel = {k2: v for k2, v in ms.items() if k2 != "kernel"}
        dominant = max(per_kernel, key=per_kernel.get)
        n_tile_launches = 4  # the sample launch + three exact launches per step and group
        tile_groups = max(1, int(stats["tile_groups"]))
        # SURVEY.md §8(d) per kernel.  k_score_lists: every distinct list of the batch is read once (packed blocks + skip data =
        # its postings range, + one fieldnorm byte per posting) and written once as 8-byte (doc, score) pairs.  k_tile: the pairs
        # are read once per launch that covers their tile (the three exact launches partition the tiles, the sample launch re-reads
        # 1/16 of them) + 16 B per candidate handed over.  Per-query kernels: exhaustive formula / device byte counter as before.
        score_bytes = float(stats["tile_list_bytes"] + stats["tile_postings"] + 8 * stats["tile_postings"])
        tile_bytes = float(8 * stats["tile_postings"]) * (1.0 + 1.0 / 16.0) + 12.0 * wl["k"] * nq
        table = {
            "score": ("k_score_lists", score_bytes, tile_groups, "postings ranges + 1 B fieldnorm + 8 B pair written per posting, every distinct list once"),
            "tile": ("k_tile", tile_bytes, n_tile_launches * tile_groups, "8 B (doc, score) pair read per posting per covering launch + result rows"),
            "or": ("k_or_strip" if stats.get("units_or_strip", 0) * 2 > stats["units_or"] else "k_or_pipe", float(touched_per_step) + 12.0 * wl["k"] * nq if touched_per_step else float(stats["bytes_or"]), 4, "bytes the kernel decoded (device counter)"),
            "and": ("k_and", float(stats["bytes_and"]), 1, "exhaustive formula; k_and prunes leader docs, so this is an exhaustive-equivalent figure"),
            "phrase": ("k_phrase", float(stats["bytes_and"]), 1, "postings ranges + fieldnorm bytes of the phrases' terms (position bytes of the matching docs not counted)"),
            "term": ("k_term", float(stats["bytes_term"]), 1, "exhaustive formula (the kernel reads every posting)"),
            "final": ("k_final", 16.0 * 8192 * nq, 1, "candidate regions (upper bound)"),
            "theta": ("k_theta", 16.0 * 8192 * nq, 3, "candidate regions (upper bound)"),
        }
        kernel_name, step_bytes, n_launch, basis = table[dominant]
        step_ms = per_kernel[dominant]
        achieved = step_bytes / (step_ms * 1e-3) / 1e9 if step_ms > 0 else 0.0
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tpath) and world == 1:
            traffic = json.load(open(tpath)).get(args.workload, {}).get(kernel_name)  # dram bytes per launch, one ncu --set full capture
        exh = float(stats["algorithmic_bytes"])
        roofline = {"bound": "hbm", "kernel": kernel_name, "achieved": achieved, "peak": peak, "unit": "GB/s",
                    "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                    "algorithmic_bytes_per_launch": step_bytes / n_launch, "avg_launch_ms": step_ms / n_launch,
                    "launches_per_step_of_this_kernel": n_launch, "algorithmic_bytes_per_step": step_bytes, "kernel_ms_per_step": step_ms,
                    "achieved_basis": basis,
                    "exhaustive_algorithmic_bytes_per_step": exh,
                    "exhaustive_equivalent_gbs": exh / (ms["kernel"] * 1e-3) / 1e9 if ms["kernel"] > 0 else 0.0,
                    "exhaustive_equivalent_frac": exh / (ms["kernel"] * 1e-3) / 1e9 / peak if ms["kernel"] > 0 else 0.0,
                    "exhaustive_note": "SURVEY.md §8(d) exhaustive bytes of the step (every posting of every clause of every query) / device time of ALL kernels of the step",
                    "all_kernels_ms_per_step": {k2: round(v, 4) for k2, v in ms.items()},
                    "second_kernel": None}
        others = sorted(((v, k2) for k2, v in per_kernel.items() if k2 != dominant), reverse=True)
        if others and others[0][0] > 0:
            k2 = others[0][1]
            n2, b2, l2, basis2 = table[k2]
            roofline["second_kernel"] = {"kernel": n2, "kernel_ms_per_step": others[0][0], "algorithmic_bytes_per_step": b2, "launches_per_step": l2,
                                         "achieved": b2 / (others[0][0] * 1e-3) / 1e9, "frac": b2 / (others[0][0] * 1e-3) / 1e9 / peak, "achieved_basis": basis2}
        workload_stats = {"index_bytes_this_rank": shard.index_bytes, "step_bytes_algorithmic_exhaustive": stats["algorithmic_bytes"],
                          "postings_per_step_exhaustive": stats["postings"], "postings_decoded_per_step": stats["tile_postings"],
                          "pair_scratch_bytes": stats["tile_scratch_bytes"], "units_per_step": stats["units"], "tile_groups": stats["tile_groups"],
                          "tile_fallback_steps": int(fallbacks), "index_generation_s": round(shard.gen_s, 2), "host": hinfo}
        line = {"metric": "queries/sec", "value": value, "unit": "queries/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": 1000.0 * dt_value / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic", "config": config, "workload_stats": workload_stats, "roofline": roofline, "clocks": clocks,
                "e2e": {"value": e2e, "unit": "queries/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                        "ms_per_step": 1000.0 * dt_e2e / args.steps,
                        "mode": f"{depth} batch(es) in flight: step i+1 is planned (tq_batch_prepare: host planning + H2D) while step i runs" +
                                (" and queued behind it" if depth > 1 else "") + "; the host then waits for step i and reads its rows back (D2H); "
                                "serial_* = one step at a time, nothing overlapped",
                        "serial_value": nq * args.steps / dt_e2e_serial, "serial_ms_per_step": 1000.0 * dt_e2e_serial / args.steps},
                "pipeline": {"batches_in_flight": depth,
                             "note": "value / ms_per_step: K steps with `batches_in_flight` prepared batches queued on their own streams (the host waits "
                                     "for step i after queueing step i+1); serial_* and every per-kernel time of `roofline`: the same K steps one at a "
                                     "time with a synchronisation per step",
                             "serial_value": nq * args.steps / dt_value_serial, "serial_ms_per_step": 1000.0 * dt_value_serial / args.steps,
                             "overflow_repeats": int(sum(getattr(m, "repeats", 0) for m in mergers))},
                "gpu_launches": int(launches)}
        if args.parity_queries and parity_rows is not None:
            line["parity"] = parity_check(wl, dens, args.seed, batches[0][:args.parity_queries], parity_rows, host_threads)
            line["parity"]["rows_from"] = "the first timed e2e step (tq_batch_prepare + run + fetch)" if world == 1 else f"rank 0's merged rows of the first timed e2e step ({world} ranks)"
        if world == 1 and not args.no_cpu_baseline:
            sample = args.cpu_sample or min(512, max(64, 4 * host_threads))
            # bounded: a few seconds per step; several queries per host thread keep the threads busy
            qps, ms_c = cpu_reference_run(wl, shard, batches, 2, 1, sample, host_threads)
            line["cpu_baseline"] = {"value": qps, "unit": "queries/s", "cores": host_threads, "kind": "port", "host": hinfo,
                                    "sample": f"3 x {sample} queries of the same stream (1 warm-up), all host threads, oracle/ "
                                              "restatement of tantivy's Block-WAND + TopNHeap + merge_top_k (mode=1)",
                                    "ms_per_sample": ms_c}
        print(json.dumps(line))
    ctx.close()
    if dist is not None:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
