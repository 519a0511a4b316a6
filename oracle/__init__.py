"""ORACLE — TEST INFRASTRUCTURE ONLY.

ctypes binding of ``oracle/liboracle.so`` (the CPU restatement of the reference's hot path, see the
headers of ``distance.hpp`` / ``hnsw.hpp`` / ``segment.hpp`` / ``bm25.hpp`` for the reference
file:line each function follows).  Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s
``cpu_baseline`` / ``--impl reference`` legs may import this package; the product package
``nucliadb_b200`` never does.

Parity status: distances / brute force / HNSW are pinned to the reference's own known-answer tests
(one-hot fixtures, tolerances; tests/test_oracle_*.py); BM25 is **parity unpinned** (tantivy is a
third-party crate absent from /root/reference and no reference test asserts a BM25 value).
"""
from __future__ import annotations

import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
NIL = 0xFFFFFFFF
SIM_DOT, SIM_COSINE, SIM_L2 = 0, 1, 2
BM25_OR, BM25_AND = 0, 1

_lib = None
_native_path = None


def build(native: bool = False) -> str:
    """Compile the oracle (gcc only).  Returns the path of the shared object.  The -march=native build is only valid on the
    machine that compiles it, so it goes to a temporary directory of this process (removed at exit), never into the source tree,
    which may be read-only; it is compiled once per process and must load here."""
    global _native_path
    if not native:
        subprocess.run(["make", "-s", "-C", _HERE, "liboracle.so"], check=True)
        return os.path.join(_HERE, "liboracle.so")
    if _native_path is None:
        tmp = tempfile.mkdtemp(prefix="oracle_native_")
        atexit.register(shutil.rmtree, tmp, True)
        path = os.path.join(tmp, "liboracle_native.so")
        subprocess.run(["make", "-s", "-C", _HERE, "native", f"NATIVE_OUT={path}"], check=True)
        C.CDLL(path)
        _native_path = path
    return _native_path


def lib(native: bool = False):
    global _lib
    if _lib is not None and not native:
        return _lib
    path = build(True) if native else os.path.join(_HERE, "liboracle.so")
    if not os.path.exists(path):
        build()
    L = C.CDLL(path)
    L.oracle_dot.restype = C.c_float
    L.oracle_dot_f64.restype = C.c_double
    L.oracle_norm.restype = C.c_float
    L.oracle_cosine.restype = C.c_float
    L.oracle_graph_layout.restype = C.c_uint64
    L.oracle_hnsw_build.restype = C.c_double
    L.oracle_fssc_new.restype = C.c_void_p
    L.oracle_fieldnorm_to_id.restype = C.c_uint8
    L.oracle_fieldnorm_id_to_value.restype = C.c_uint32
    L.oracle_bm25_idf.restype = C.c_float
    L.oracle_bm25_term_score.restype = C.c_float
    if not native:
        _lib = L
    return L


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


def dot(a, b) -> float:
    a, b = _f32(a), _f32(b)
    return float(lib().oracle_dot(_p(a), _p(b), C.c_int(a.size)))


def dot_f64(a, b) -> float:
    a, b = _f32(a), _f32(b)
    return float(lib().oracle_dot_f64(_p(a), _p(b), C.c_int(a.size)))


def cosine(a, b) -> float:
    a, b = _f32(a), _f32(b)
    return float(lib().oracle_cosine(_p(a), _p(b), C.c_int(a.size)))


def normalize(a) -> np.ndarray:
    a = _f32(a)
    out = np.empty_like(a)
    lib().oracle_normalize(_p(a), _p(out), C.c_int(a.size))
    return out


def norms(vecs, nthreads=1) -> np.ndarray:
    vecs = _f32(vecs)
    n, d = vecs.shape
    out = np.empty(n, dtype=np.float32)
    lib().oracle_norms(_p(vecs), C.c_uint32(n), C.c_int(d), C.c_int(d), _p(out), C.c_int(nthreads))
    return out


def use_hnsw(total, matching, top_k, has_rabitq=False, M=30) -> bool:
    return bool(lib().oracle_use_hnsw(C.c_uint64(total), C.c_uint64(matching), C.c_uint64(top_k), C.c_int(int(has_rabitq)), C.c_int(M)))


def assign_levels(n, M=30, seed=2) -> np.ndarray:
    out = np.empty(n, dtype=np.uint8)
    lib().oracle_assign_levels(C.c_uint32(n), C.c_int(M), C.c_uint64(seed), _p(out))
    return out


def brute_force(vecs, queries, k, sim=SIM_COSINE, min_score=-1.0, alive_bits=None, first_vec=None, num_vec=None, nthreads=1, native=False):
    """segment.rs:569-623 for a batch of queries -> (ids [nq,k] u32, scores [nq,k] f32, count [nq])."""
    vecs, queries = _f32(vecs), _f32(np.atleast_2d(queries))
    n, d = vecs.shape
    nq = queries.shape[0]
    nrm = norms(vecs, nthreads) if sim != SIM_DOT else None
    n_par = n if first_vec is None else len(first_vec)
    ids = np.empty((nq, k), dtype=np.uint32)
    sc = np.empty((nq, k), dtype=np.float32)
    cnt = np.empty(nq, dtype=np.int32)
    lib(native).oracle_brute_force(_p(vecs), _p(nrm), C.c_uint32(n), C.c_int(d), C.c_int(d), C.c_int(sim), _p(queries), C.c_int(nq), C.c_int(d),
                                   C.c_int(k), C.c_float(min_score), _p(alive_bits), C.c_uint32(n_par), _p(first_vec), _p(num_vec), _p(ids),
                                   _p(sc), _p(cnt), C.c_int(nthreads))
    return ids, sc, cnt


def maxsim_similarity(query_vectors, doc_vectors, sim=SIM_COSINE) -> float:
    """multivector.rs:34-46: sum over query vectors of max(0, best similarity to a vector of the document), f32 fold."""
    total = np.float32(0.0)
    for vq in query_vectors:
        best = np.float32(0.0)
        for vd in doc_vectors:
            s = np.float32(cosine(vd, vq) if sim == SIM_COSINE else dot(vd, vq))
            if s > best:
                best = s
        total = np.float32(total + best)
    return float(total)


def multi_vector_search(paragraphs, query_vectors, k, min_score, sim=SIM_COSINE):
    """searcher.rs:345-394 on one exhaustive segment: every query vector retrieves (exact scan, duplicates allowed, no
    min_score, at least 10 results) the paragraphs of its best vectors; the union is re-scored with MaxSim, filtered with a
    strict `> min_score`, sorted and truncated.  paragraphs: list of [n_i, d] arrays.  -> [(paragraph index, score)]."""
    first = np.cumsum([0] + [len(p) for p in paragraphs]).astype(np.uint32)
    vecs = _f32(np.concatenate(paragraphs))
    ids, _, counts = brute_force(vecs, _f32(query_vectors), max(k, 10), sim=sim, min_score=float(np.finfo(np.float32).min), first_vec=first[:-1],
                                 num_vec=np.diff(first).astype(np.uint32))
    cand = sorted({int(np.searchsorted(first, a, side="right") - 1) for qi in range(len(query_vectors)) for a in ids[qi, : counts[qi]]})
    scored = [(p, maxsim_similarity(query_vectors, paragraphs[p], sim)) for p in cand]
    scored = [(p, s) for p, s in scored if s > min_score]
    scored.sort(key=lambda t: -t[1])
    return scored[:k]


class Graph:
    """Flat HNSW graph (the layout shared with the CUDA library, DESIGN.md)."""

    def __init__(self, n, M, M0, level):
        L = lib()
        self.n, self.M, self.M0 = int(n), int(M), int(M0)
        self.s0, self.su = L.oracle_stride0(C.c_int(M0)), L.oracle_strideU(C.c_int(M))
        self.level = np.ascontiguousarray(level, dtype=np.uint8)
        self.upper_off = np.zeros(max(n, 1), dtype=np.uint64)
        en, el = C.c_uint32(0), C.c_uint32(0)
        self.upper_rows = int(L.oracle_graph_layout(C.c_uint32(n), _p(self.level), _p(self.upper_off), C.byref(en), C.byref(el)))
        self.entry_node, self.entry_layer = en.value, el.value
        self.adj0 = np.full((n, self.s0), NIL, dtype=np.uint32)
        self.w0 = np.zeros((n, self.s0), dtype=np.float32)
        self.adjU = np.full((max(self.upper_rows, 1), self.su), NIL, dtype=np.uint32)
        self.wU = np.zeros((max(self.upper_rows, 1), self.su), dtype=np.float32)

    def edges(self, node, layer):
        row = self.adj0[node] if layer == 0 else self.adjU[int(self.upper_off[node]) + layer - 1]
        return row[row != NIL]


def default_schedule(n, entry_node, max_batch=1, growth=16):
    """Insertion order (entry point first, then ascending id) and batch ends: batch size
    min(max_batch, max(1, inserted // growth))."""
    order = np.concatenate([[entry_node], np.delete(np.arange(n, dtype=np.uint32), entry_node)]).astype(np.uint32)
    ends, done = [], 0
    while done < n:
        b = min(max_batch, max(1, done // growth), n - done)
        done += b
        ends.append(done)
    return order, np.asarray(ends, dtype=np.uint32)


def hnsw_build(vecs, sim=SIM_COSINE, M=30, M0=60, efC=100, seed=2, max_batch=1, nthreads=1, levels=None, native=False):
    vecs = _f32(vecs)
    n, d = vecs.shape
    level = assign_levels(n, M, seed) if levels is None else np.ascontiguousarray(levels, dtype=np.uint8)
    g = Graph(n, M, M0, level)
    nrm = norms(vecs, nthreads) if sim != SIM_DOT else None
    order, ends = default_schedule(n, g.entry_node, max_batch)
    counters = np.zeros(3, dtype=np.uint64)
    secs = lib(native).oracle_hnsw_build(_p(vecs), _p(nrm), C.c_uint32(n), C.c_int(d), C.c_int(d), C.c_int(sim), C.c_int(M), C.c_int(M0),
                                         C.c_int(efC), _p(g.level), C.c_uint32(g.entry_node), C.c_uint32(g.entry_layer), _p(g.adj0), _p(g.w0),
                                         _p(g.upper_off), _p(g.adjU), _p(g.wU), _p(order), _p(ends), C.c_uint32(len(ends)), C.c_int(nthreads),
                                         _p(counters))
    g.build_seconds, g.build_counters = secs, counters
    return g


def fix_broken_links(g: Graph) -> int:
    """ram_hnsw.rs:52-64,118-123: in every layer above 0 drop the links that point at a node not present in that layer
    (graphs written by an old version can hold them).  Rows stay left-packed.  -> number of links removed."""
    removed = 0
    for node in np.nonzero(g.level > 0)[0]:
        base = int(g.upper_off[node])
        for layer in range(1, int(g.level[node]) + 1):
            row, wrow = g.adjU[base + layer - 1], g.wU[base + layer - 1]
            valid = row != NIL
            keep = valid & (g.level[np.where(valid, row, 0)] >= layer)
            if (keep != valid).any():
                removed += int(valid.sum() - keep.sum())
                ids, ws = row[keep].copy(), wrow[keep].copy()
                row[:], wrow[:] = NIL, 0
                row[: len(ids)], wrow[: len(ids)] = ids, ws
    return removed


def hnsw_extend(vecs, g0: Graph, sim=SIM_COSINE, efC=100, seed=2, max_batch=1, nthreads=1):
    """merge_indexes' fast path (segment.rs:143-167): keep g0 (the graph of the first g0.n vectors) and insert the remaining
    vectors; new levels from a fresh RNG (build.rs:36-55), entry point moved only if a higher layer appears."""
    vecs = _f32(vecs)
    n, d = vecs.shape
    n0 = g0.n
    level = np.concatenate([g0.level, assign_levels(n - n0, g0.M, seed)]).astype(np.uint8)
    g = Graph(n, g0.M, g0.M0, level)
    raised = (g.entry_node, g.entry_layer)      # lowest id of the global top layer
    raises = raised[1] > g0.entry_layer and raised[0] >= n0
    if raised[1] > g0.entry_layer and not raises:
        g.entry_node, g.entry_layer = raised    # g0's entry point was below its own top layer
    else:
        g.entry_node, g.entry_layer = g0.entry_node, g0.entry_layer
    g.adj0[:n0], g.w0[:n0] = g0.adj0, g0.w0
    rows0 = int(g0.level.astype(np.int64).sum())
    g.adjU[:rows0], g.wU[:rows0] = g0.adjU[:rows0], g0.wU[:rows0]
    fix_broken_links(g)                         # merge_indexes: index.fix_broken_graph() (segment.rs:162)
    nrm = norms(vecs, nthreads) if sim != SIM_DOT else None
    # Deviation from the reference, shared with the CUDA path (see nidx_vec_extend_hnsw): a new node that raises the top layer
    # is inserted first, from the old entry point, and only then becomes the entry point -- the reference moves the entry point
    # to the still unlinked node up front (build.rs:49-55), which cuts the reused graph off.
    order = ([raised[0]] if raises else []) + [i for i in range(n0, n) if not (raises and i == raised[0])]
    order = np.asarray(order, dtype=np.uint32)
    ends, done = ([1] if raises else []), n0 + (1 if raises else 0)
    while done < n:
        b = min(max_batch, max(1, done // 16), n - done)
        done += b
        ends.append(done - n0)
    counters = np.zeros(3, dtype=np.uint64)

    def run(order_part, ends_part):
        e = np.asarray(ends_part, dtype=np.uint32)
        o = np.ascontiguousarray(order_part, dtype=np.uint32)
        lib().oracle_hnsw_build(_p(vecs), _p(nrm), C.c_uint32(n), C.c_int(d), C.c_int(d), C.c_int(sim), C.c_int(g.M), C.c_int(g.M0), C.c_int(efC), _p(g.level),
                                C.c_uint32(g.entry_node), C.c_uint32(g.entry_layer), _p(g.adj0), _p(g.w0), _p(g.upper_off), _p(g.adjU), _p(g.wU), _p(o), _p(e),
                                C.c_uint32(len(e)), C.c_int(nthreads), _p(counters))

    if raises:
        run(order[:1], [1])
        g.entry_node, g.entry_layer = raised
        if len(order) > 1:
            run(order[1:], [x - 1 for x in ends[1:]])
    elif len(order):
        run(order, ends)
    return g


def hnsw_search(vecs, g: Graph, queries, k, ef, sim=SIM_COSINE, min_score=-1.0, with_duplicates=True, multi_vector=False, filter_bits=None,
                paragraph_of=None, nthreads=1, native=False, norms_=None):
    """search.rs:306-383 for a batch -> (ids, scores, count, counters[n_dist, n_expand, n_edges_read])."""
    vecs, queries = _f32(vecs), _f32(np.atleast_2d(queries))
    n, d = vecs.shape
    nq = queries.shape[0]
    nrm = (norms(vecs, nthreads) if norms_ is None else norms_) if sim != SIM_DOT else None
    ids = np.empty((nq, k), dtype=np.uint32)
    sc = np.empty((nq, k), dtype=np.float32)
    cnt = np.empty(nq, dtype=np.int32)
    counters = np.zeros(3, dtype=np.uint64)
    lib(native).oracle_hnsw_search(_p(vecs), _p(nrm), C.c_uint32(n), C.c_int(d), C.c_int(d), C.c_int(sim), C.c_int(g.M), C.c_int(g.M0),
                                   _p(g.level), C.c_uint32(g.entry_node), C.c_uint32(g.entry_layer), _p(g.adj0), _p(g.upper_off), _p(g.adjU),
                                   _p(queries), C.c_int(nq), C.c_int(d), C.c_int(k), C.c_int(ef), C.c_float(min_score),
                                   C.c_int(int(with_duplicates)), C.c_int(int(multi_vector)), _p(filter_bits), _p(paragraph_of), _p(ids), _p(sc),
                                   _p(cnt), _p(counters), C.c_int(nthreads))
    return ids, sc, cnt, counters


def layer_search(vecs, g: Graph, query, layer, k, eps, sim=SIM_COSINE):
    vecs, query = _f32(vecs), _f32(query)
    n, d = vecs.shape
    nrm = norms(vecs) if sim != SIM_DOT else None
    eps = np.ascontiguousarray(eps, dtype=np.uint32)
    cap = max(k, len(eps))
    ids = np.empty(cap, dtype=np.uint32)
    sc = np.empty(cap, dtype=np.float32)
    r = lib().oracle_layer_search(_p(vecs), _p(nrm), C.c_uint32(n), C.c_int(d), C.c_int(d), C.c_int(sim), C.c_int(g.M), C.c_int(g.M0),
                                  _p(g.level), _p(g.adj0), _p(g.upper_off), _p(g.adjU), _p(query), C.c_int(layer), C.c_int(k), _p(eps),
                                  C.c_int(len(eps)), _p(ids), _p(sc))
    return ids[:r].copy(), sc[:r].copy()


def select_neighbours(vecs, k, cand_ids, cand_scores, sim=SIM_COSINE):
    vecs = _f32(vecs)
    n, d = vecs.shape
    nrm = norms(vecs) if sim != SIM_DOT else None
    cand_ids = np.ascontiguousarray(cand_ids, dtype=np.uint32)
    cand_scores = _f32(cand_scores)
    ids = np.empty(len(cand_ids), dtype=np.uint32)
    sc = np.empty(len(cand_ids), dtype=np.float32)
    r = lib().oracle_select_neighbours(_p(vecs), _p(nrm), C.c_uint32(n), C.c_int(d), C.c_int(d), C.c_int(sim), C.c_int(k), _p(cand_ids),
                                       _p(cand_scores), C.c_int(len(cand_ids)), _p(ids), _p(sc))
    return ids[:r].copy(), sc[:r].copy()


class Fssc:
    """searcher.rs:150-199."""

    def __init__(self, size, with_duplicates):
        self._h = C.c_void_p(lib().oracle_fssc_new(C.c_int(size), C.c_int(int(with_duplicates))))
        self._size = size

    def add(self, pid: str, score: float, segment: int, addr: int, vec_bytes: bytes):
        lib().oracle_fssc_add(self._h, pid.encode(), C.c_float(score), C.c_uint32(segment), C.c_uint32(addr), vec_bytes, C.c_int(len(vec_bytes)))

    def result(self):
        seg = np.empty(self._size, dtype=np.uint32)
        addr = np.empty(self._size, dtype=np.uint32)
        sc = np.empty(self._size, dtype=np.float32)
        r = lib().oracle_fssc_result(self._h, _p(seg), _p(addr), _p(sc))
        return seg[:r], addr[:r], sc[:r]

    def __del__(self):
        try:
            lib().oracle_fssc_free(self._h)
        except Exception:
            pass


# ---- BM25 -------------------------------------------------------------------------------------------
def fieldnorm_to_id(v: int) -> int:
    return int(lib().oracle_fieldnorm_to_id(C.c_uint32(v)))


def fieldnorm_id_to_value(i: int) -> int:
    return int(lib().oracle_fieldnorm_id_to_value(C.c_uint32(i)))


def bm25_idf(df, n) -> float:
    return float(lib().oracle_bm25_idf(C.c_uint64(df), C.c_uint64(n)))


def bm25_term_score(df, n_docs, total_tokens, fieldnorm_id, tf) -> float:
    return float(lib().oracle_bm25_term_score(C.c_uint64(df), C.c_uint64(n_docs), C.c_uint64(total_tokens), C.c_uint32(fieldnorm_id), C.c_uint32(tf)))


class Postings:
    """One segment's inverted index built from token-id documents (CPU, numpy)."""

    def __init__(self, doc_off, tokens, n_terms):
        doc_off = np.asarray(doc_off, dtype=np.int64)
        tokens = np.asarray(tokens, dtype=np.uint32)
        self.n_docs = len(doc_off) - 1
        self.n_terms = int(n_terms)
        lens = np.diff(doc_off)
        self.total_tokens = int(lens.sum())
        self.fieldnorm_id = np.array([fieldnorm_to_id(int(x)) for x in np.unique(lens)], dtype=np.uint8)[np.searchsorted(np.unique(lens), lens)] \
            if self.n_docs else np.zeros(0, dtype=np.uint8)
        doc_of_tok = np.repeat(np.arange(self.n_docs, dtype=np.uint32), lens)
        key = tokens.astype(np.uint64) * np.uint64(max(self.n_docs, 1)) + doc_of_tok.astype(np.uint64)
        uniq, tf = np.unique(key, return_counts=True)
        self.post_term = (uniq // np.uint64(max(self.n_docs, 1))).astype(np.uint32)
        self.post_doc = (uniq % np.uint64(max(self.n_docs, 1))).astype(np.uint32)
        self.post_tf = tf.astype(np.uint32)
        self.term_off = np.zeros(self.n_terms + 1, dtype=np.uint64)
        np.add.at(self.term_off, self.post_term.astype(np.int64) + 1, 1)
        self.term_off = np.cumsum(self.term_off).astype(np.uint64)
        self.doc_freq = np.diff(self.term_off.astype(np.int64)).astype(np.uint64)


def bm25_search(P: Postings, queries, k, mode=BM25_OR, use_tf=True, alive_bits=None, total_docs=None, total_tokens=None, doc_freq=None,
                nthreads=1, native=False):
    """queries: list of term-id lists.  Statistics default to the segment's own (single-segment index)."""
    q_off = np.zeros(len(queries) + 1, dtype=np.uint32)
    q_off[1:] = np.cumsum([len(q) for q in queries])
    q_terms = np.ascontiguousarray(np.concatenate([np.asarray(q, dtype=np.uint32) for q in queries]) if len(queries) else np.zeros(0, np.uint32))
    nq = len(queries)
    docs = np.empty((nq, k), dtype=np.uint32)
    sc = np.empty((nq, k), dtype=np.float32)
    cnt = np.empty(nq, dtype=np.int32)
    total = np.empty(nq, dtype=np.uint64)
    df = P.doc_freq if doc_freq is None else np.ascontiguousarray(doc_freq, dtype=np.uint64)
    lib(native).oracle_bm25_search(C.c_uint32(P.n_docs), C.c_uint32(P.n_terms), _p(P.term_off), _p(P.post_doc), _p(P.post_tf), _p(P.fieldnorm_id),
                                   _p(alive_bits), C.c_uint64(P.n_docs if total_docs is None else total_docs),
                                   C.c_uint64(P.total_tokens if total_tokens is None else total_tokens), _p(df), _p(q_terms), _p(q_off),
                                   C.c_int(nq), C.c_int(mode), C.c_int(int(use_tf)), C.c_int(k), _p(docs), _p(sc), _p(cnt), _p(total),
                                   C.c_int(nthreads))
    return docs, sc, cnt, total


# ---- RaBitQ (rabitq.rs) ---------------------------------------------------------------------------------
def rabitq_encoded_len(d: int) -> int:
    lib().oracle_rabitq_encoded_len.restype = C.c_uint64
    return int(lib().oracle_rabitq_encoded_len(C.c_int(d)))


def rabitq_encode(vecs, nthreads=1) -> np.ndarray:
    """[n][d] f32 -> [n][d/8 + 8] bytes: [f32 dot_quant_original][u32 sum_bits][sign bits] (rabitq.rs:75-106)."""
    vecs = _f32(np.atleast_2d(vecs))
    n, d = vecs.shape
    out = np.empty((n, rabitq_encoded_len(d)), dtype=np.uint8)
    lib().oracle_rabitq_encode(_p(vecs), C.c_uint32(n), C.c_int(d), C.c_int(d), _p(out), C.c_int(nthreads))
    return out


def rabitq_estimate(enc, d, queries, nthreads=1):
    """-> (estimate [nq][n], error [nq][n]) (rabitq.rs:202-218)."""
    enc = np.ascontiguousarray(enc, dtype=np.uint8)
    queries = _f32(np.atleast_2d(queries))
    n, nq = enc.shape[0], queries.shape[0]
    est = np.empty((nq, n), dtype=np.float32)
    err = np.empty((nq, n), dtype=np.float32)
    lib().oracle_rabitq_estimate(_p(enc), C.c_uint32(n), C.c_int(d), _p(queries), C.c_int(nq), C.c_int(queries.shape[1]), _p(est), _p(err), C.c_int(nthreads))
    return est, err


def rabitq_query(q):
    q = _f32(q)
    d = q.size
    planes = np.empty((4, d // 64), dtype=np.uint64)
    low, delta, sq = C.c_float(), C.c_float(), C.c_uint32()
    lib().oracle_rabitq_query(_p(q), C.c_int(d), _p(planes), C.byref(low), C.byref(delta), C.byref(sq))
    return planes, low.value, delta.value, sq.value


def rabitq_brute_force(vecs, enc, queries, k, min_score=0.0, nthreads=1):
    """segment.rs:581-608 with a RaBitQ query: estimates -> upper bound filter -> rerank_top (exact dot)."""
    vecs, queries = _f32(vecs), _f32(np.atleast_2d(queries))
    enc = np.ascontiguousarray(enc, dtype=np.uint8)
    n, d = vecs.shape
    nq = queries.shape[0]
    ids = np.empty((nq, k), dtype=np.uint32)
    sc = np.empty((nq, k), dtype=np.float32)
    cnt = np.empty(nq, dtype=np.int32)
    evals = np.empty(nq, dtype=np.uint64)
    lib().oracle_rabitq_brute_force(_p(vecs), C.c_uint32(n), C.c_int(d), C.c_int(d), _p(enc), _p(queries), C.c_int(nq), C.c_int(d), C.c_int(k),
                                    C.c_float(min_score), _p(ids), _p(sc), _p(cnt), _p(evals), C.c_int(nthreads))
    return ids, sc, cnt, evals


def hnsw_search_rabitq(vecs, enc, g: Graph, queries, k, min_score=0.0, with_duplicates=True, filter_bits=None, nthreads=1):
    """hnsw/search.rs:306-383 with a SearchVector::RabitQ query (Dot similarity): the walk ranks by the RaBitQ estimate, layer 0
    asks for min(k * 100, 2000) nodes, rerank_top re-scores with the raw vectors, closest_up_nodes works on exact similarities.
    -> (ids, scores, count, counters[exact similarities, expansions, edges read, quantised estimates])."""
    vecs, queries = _f32(vecs), _f32(np.atleast_2d(queries))
    enc = np.ascontiguousarray(enc, dtype=np.uint8)
    n, d = vecs.shape
    nq = queries.shape[0]
    ids = np.empty((nq, k), dtype=np.uint32)
    sc = np.empty((nq, k), dtype=np.float32)
    cnt = np.empty(nq, dtype=np.int32)
    counters = np.zeros(4, dtype=np.uint64)
    lib().oracle_hnsw_search_rabitq(_p(vecs), C.c_uint32(n), C.c_int(d), C.c_int(d), _p(enc), C.c_int(g.M), C.c_int(g.M0), _p(g.level),
                                    C.c_uint32(g.entry_node), C.c_uint32(g.entry_layer), _p(g.adj0), _p(g.upper_off), _p(g.adjU), _p(queries),
                                    C.c_int(nq), C.c_int(d), C.c_int(k), C.c_float(min_score), C.c_int(int(with_duplicates)), _p(filter_bits),
                                    _p(ids), _p(sc), _p(cnt), _p(counters), C.c_int(nthreads))
    return ids, sc, cnt, counters
