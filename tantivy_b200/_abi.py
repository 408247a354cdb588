"""ctypes mirror of include/tantivy_b200.h (structs and constants only; no library is loaded here).

Shared by the product binding (tantivy_b200/lib.py) and by the test-only oracle binding
(oracle/tq_oracle.py) so that one marshalled query batch can be handed to either side.
"""
import ctypes as C

import numpy as np

TQ_OK = 0
TQ_RECORD_BASIC, TQ_RECORD_FREQS, TQ_RECORD_FREQS_POSITIONS = 0, 1, 2
TQ_OP_TERM, TQ_OP_AND, TQ_OP_OR, TQ_OP_PHRASE, TQ_OP_BOOL = 0, 1, 2, 3, 4
TQ_OCCUR_SHOULD, TQ_OCCUR_MUST, TQ_OCCUR_MUST_NOT = 0, 1, 2
TERMINATED = 0x7FFFFFFF
TQ_MAX_K = 1024
TQ_MAX_TERMS = 32
TQ_TERM_IGNORE_FREQ = 1
TQ_QUERY_HAS_THRESHOLD = 1

u8p = C.POINTER(C.c_uint8)
u32p = C.POINTER(C.c_uint32)
u64p = C.POINTER(C.c_uint64)
f32p = C.POINTER(C.c_float)


class TermSeg(C.Structure):
    """tq_term_seg — postings::TermInfo of one (clause, segment) (src/postings/term_info.rs:9-16)."""
    _fields_ = [
        ("term_idx", C.c_uint32),
        ("segment_ord", C.c_uint32),
        ("field", C.c_uint32),
        ("doc_freq", C.c_uint32),
        ("postings_start", C.c_uint64),
        ("postings_end", C.c_uint64),
    ]


TERM_SEG_DTYPE = np.dtype(
    [("term_idx", "<u4"), ("segment_ord", "<u4"), ("field", "<u4"), ("doc_freq", "<u4"),
     ("postings_start", "<u8"), ("postings_end", "<u8")]
)
assert TERM_SEG_DTYPE.itemsize == C.sizeof(TermSeg) == 32


class TermPos(C.Structure):
    """tq_term_pos — TermInfo::positions_range of one (clause, segment)."""
    _fields_ = [("positions_start", C.c_uint64), ("positions_end", C.c_uint64)]


TERM_POS_DTYPE = np.dtype([("positions_start", "<u8"), ("positions_end", "<u8")])


class Query(C.Structure):
    """tq_query — one Weight for all segments (src/core/searcher.rs:226)."""
    _fields_ = [
        ("op", C.c_int32),
        ("n_terms", C.c_uint32),
        ("k", C.c_uint32),
        ("n_term_segs", C.c_uint32),
        ("term_segs", C.POINTER(TermSeg)),
        ("weight", f32p),
        ("avg_fieldnorm", f32p),
        ("tf_cache", f32p),
        ("term_flags", u8p),
        ("flags", C.c_uint32),
        ("threshold", C.c_float),
        ("term_pos", C.POINTER(TermPos)),
        ("term_offset", u32p),
        ("slop", C.c_uint32),
        ("min_should_match", C.c_uint32),
        ("term_occur", u8p),
        ("term_group", u8p),
    ]


QUERY_DTYPE = np.dtype(
    [("op", "<i4"), ("n_terms", "<u4"), ("k", "<u4"), ("n_term_segs", "<u4"),
     ("term_segs", "<u8"), ("weight", "<u8"), ("avg_fieldnorm", "<u8"), ("tf_cache", "<u8"), ("term_flags", "<u8"),
     ("flags", "<u4"), ("threshold", "<f4"), ("term_pos", "<u8"), ("term_offset", "<u8"), ("slop", "<u4"), ("min_should_match", "<u4"),
     ("term_occur", "<u8"), ("term_group", "<u8")]
)
assert QUERY_DTYPE.itemsize == C.sizeof(Query) == 104


class Stats(C.Structure):
    """tq_stats."""
    _fields_ = [
        ("lists_cached", C.c_uint64),
        ("lists_built", C.c_uint64),
        ("units", C.c_uint64),
        ("kernel_launches", C.c_uint64),
        ("h2d_bytes", C.c_uint64),
        ("d2h_bytes", C.c_uint64),
        ("algorithmic_bytes", C.c_uint64),
        ("postings", C.c_uint64),
        ("kernel_ms", C.c_float),
        ("total_ms", C.c_float),
        ("term_ms", C.c_float),
        ("and_ms", C.c_float),
        ("or_ms", C.c_float),
        ("final_ms", C.c_float),
        ("units_term", C.c_uint64),
        ("units_and", C.c_uint64),
        ("units_or", C.c_uint64),
        ("bytes_term", C.c_uint64),
        ("bytes_and", C.c_uint64),
        ("bytes_or", C.c_uint64),
        ("or_windows", C.c_uint64 * 8),
        ("units_or_strip", C.c_uint64),
        ("score_ms", C.c_float),
        ("tile_ms", C.c_float),
        ("theta_ms", C.c_float),
        ("phrase_ms", C.c_float),
        ("units_tile", C.c_uint64),
        ("units_phrase", C.c_uint64),
        ("tile_groups", C.c_uint64),
        ("tile_postings", C.c_uint64),
        ("tile_list_bytes", C.c_uint64),
        ("tile_scratch_bytes", C.c_uint64),
        ("tile_fallbacks", C.c_uint64),
        ("tile_counters", C.c_uint64 * 8),
        ("units_bool", C.c_uint64),
        ("bool_ms", C.c_float),
    ]


def ptr(arr, typ):
    """numpy array -> ctypes pointer (array must stay alive while the pointer is used)."""
    if arr is None:
        return typ()
    return arr.ctypes.data_as(typ)


class QueryBatch:
    """A marshalled array of tq_query with everything it points to kept alive.

    `queries` is an iterable of dicts / objects with fields
      op, k, weights[n_terms], avg_fieldnorm[n_terms], term_segs: list of
      (term_idx, segment_ord, field, doc_freq, postings_start, postings_end),
      tf_cache (optional [n_terms,256]), term_flags (optional [n_terms] bytes, TQ_TERM_IGNORE_FREQ),
      threshold (optional float: only docs scoring above it are collected),
      phrase queries (op TQ_OP_PHRASE): term_pos = list of (positions_start, positions_end) parallel to term_segs,
      term_offset = [n_terms] offsets in the phrase, slop (optional, must be 0 on the device path);
      boolean queries (op TQ_OP_BOOL): term_occur = [n_terms] TQ_OCCUR_*, term_group = optional [n_terms] group ids of the MUST
      clauses, min_should_match (optional).
    Built with numpy so that a batch of thousands of queries marshals in milliseconds.
    """

    def __init__(self, queries):
        queries = list(queries)
        self.nq = len(queries)
        n_ts = sum(len(q["term_segs"]) for q in queries)
        n_terms = sum(len(q["weights"]) for q in queries)
        self.term_segs = np.zeros(max(n_ts, 1), dtype=TERM_SEG_DTYPE)
        self.weights = np.zeros(max(n_terms, 1), dtype=np.float32)
        self.avgs = np.zeros(max(n_terms, 1), dtype=np.float32)
        self.caches = []
        self.q = np.zeros(max(self.nq, 1), dtype=QUERY_DTYPE)
        ts_base = self.term_segs.ctypes.data
        w_base = self.weights.ctypes.data
        a_base = self.avgs.ctypes.data
        its, iw = 0, 0
        self.kmax = 1
        for i, q in enumerate(queries):
            nt = len(q["weights"])
            ts = q["term_segs"]
            if len(ts):
                block = np.asarray(ts, dtype=np.uint64).reshape(-1, 6)
                v = self.term_segs[its:its + len(ts)]
                v["term_idx"] = block[:, 0]
                v["segment_ord"] = block[:, 1]
                v["field"] = block[:, 2]
                v["doc_freq"] = block[:, 3]
                v["postings_start"] = block[:, 4]
                v["postings_end"] = block[:, 5]
            self.weights[iw:iw + nt] = q["weights"]
            self.avgs[iw:iw + nt] = q["avg_fieldnorm"]
            row = self.q[i]
            row["op"] = q["op"]
            row["n_terms"] = nt
            row["k"] = q["k"]
            row["n_term_segs"] = len(ts)
            row["term_segs"] = ts_base + its * TERM_SEG_DTYPE.itemsize
            row["weight"] = w_base + iw * 4
            row["avg_fieldnorm"] = a_base + iw * 4
            cache = q.get("tf_cache")
            if cache is not None:
                cache = np.ascontiguousarray(cache, dtype=np.float32).reshape(nt, 256)
                self.caches.append(cache)
                row["tf_cache"] = cache.ctypes.data
            if q.get("threshold") is not None:
                row["flags"] = TQ_QUERY_HAS_THRESHOLD
                row["threshold"] = q["threshold"]
            tpos = q.get("term_pos")
            if tpos is not None:
                tp = np.zeros(max(len(tpos), 1), dtype=TERM_POS_DTYPE)
                if len(tpos):
                    blockp = np.asarray(tpos, dtype=np.uint64).reshape(-1, 2)
                    tp["positions_start"][:len(tpos)] = blockp[:, 0]
                    tp["positions_end"][:len(tpos)] = blockp[:, 1]
                toff = np.ascontiguousarray(q["term_offset"], dtype=np.uint32).reshape(nt)
                self.caches += [tp, toff]
                row["term_pos"] = tp.ctypes.data
                row["term_offset"] = toff.ctypes.data
                row["slop"] = int(q.get("slop", 0))
            occ = q.get("term_occur")
            if occ is not None:
                occ = np.ascontiguousarray(occ, dtype=np.uint8).reshape(nt)
                self.caches.append(occ)
                row["term_occur"] = occ.ctypes.data
                grp = q.get("term_group")
                if grp is not None:
                    grp = np.ascontiguousarray(grp, dtype=np.uint8).reshape(nt)
                    self.caches.append(grp)
                    row["term_group"] = grp.ctypes.data
                row["min_should_match"] = int(q.get("min_should_match", 0))
            flags = q.get("term_flags")
            if flags is not None:
                flags = np.ascontiguousarray(flags, dtype=np.uint8).reshape(nt)
                self.caches.append(flags)
                row["term_flags"] = flags.ctypes.data
            self.kmax = max(self.kmax, int(q["k"]))
            its += len(ts)
            iw += nt

    @property
    def ptr(self):
        return C.cast(self.q.ctypes.data, C.POINTER(Query))

    def alloc_out(self, stride=None):
        stride = stride or self.kmax
        n = max(self.nq, 1)
        return (
            stride,
            np.zeros((n, stride), dtype=np.float32),
            np.zeros((n, stride), dtype=np.uint32),
            np.zeros((n, stride), dtype=np.uint32),
            np.zeros(n, dtype=np.uint32),
        )
