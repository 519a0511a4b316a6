"""The constants the hot path takes from the reference, as read from the reference's own Rust sources into
tests/golden/reference_facts.json (tests/golden/make_reference_facts.py), compared with what the mirror, the oracle and the CUDA
sources use."""
import json
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = json.load(open(os.path.join(ROOT, "tests", "golden", "reference_facts.json")))["nidx_vector"]


def test_hnsw_parameters():
    """hnsw/params.rs:34-46: M, M_MAX, M_MAX_0, EF_CONSTRUCTION, EF_SEARCH and prune_m = m * 95 / 100 = the mirror's and the library's defaults."""
    from nucliadb_b200 import vector as V

    p = REF["hnsw_params"]
    cfg = V.VectorConfig(dimension=8)
    assert cfg.m == p["M"] == p["M_MAX"]
    assert cfg.m0 == p["M_MAX_0"]
    assert cfg.ef_construction == p["EF_CONSTRUCTION"]
    assert cfg.ef_search == p["EF_SEARCH"]
    num, den = p["prune_m_ratio"]
    assert f"mmax * {num} / {den}" in open(os.path.join(ROOT, "nucliadb_b200", "csrc", "hnsw_build.cuh")).read()
    header = open(os.path.join(ROOT, "include", "nidx_b200.h")).read()
    for field, want in (("m;", p["M"]), ("m0;", p["M_MAX_0"]), ("ef_construction;", p["EF_CONSTRUCTION"]), ("ef_search;", p["EF_SEARCH"])):
        assert re.search(rf"int32_t {re.escape(field)}[^\n]*0 => {want} \*/", header), field


def test_rabitq_constants():
    """vector_types/rabitq.rs:30-36: EPSILON, RERANKING_FACTOR, RERANKING_LIMIT in the kernels, the host code and the oracle."""
    eps, fac, lim = REF["rabitq"]["EPSILON"], REF["rabitq"]["RERANKING_FACTOR"], REF["rabitq"]["RERANKING_LIMIT"]
    cu = open(os.path.join(ROOT, "nucliadb_b200", "csrc", "rabitq.cuh")).read()
    assert float(re.search(r"RABITQ_EPSILON = ([0-9.]+)f", cu).group(1)) == eps
    assert float(re.search(r"RABITQ_EPSILON = ([0-9.]+)f", open(os.path.join(ROOT, "oracle", "rabitq.hpp")).read()).group(1)) == eps
    api = open(os.path.join(ROOT, "nucliadb_b200", "csrc", "api.cu")).read()
    m = re.search(r"last_k = \(int\)std::min<size_t>\(\(size_t\)k \* (\d+), (\d+)\)", api)
    assert (float(m.group(1)), float(m.group(2))) == (fac, lim)
    assert float(re.search(r"const size_t RERANKING_FACTOR = (\d+);", api).group(1)) == fac


def test_cost_model_matches_the_reference_source():
    """segment.rs:626-660 use_hnsw: the constants of the reference's function body (16, * 3 / 4, / 2, ln - 2.0) as stored, and the
    oracle's restatement agrees with a literal Python transcription of the Rust, built from those constants, on a grid."""
    import numpy as np

    import oracle as O

    c = REF["use_hnsw"]
    rq, plain = c["with_rabitq"], c["without_rabitq"]
    assert (rq["full_cost"], rq["search_mult_of_reranking_factor"], rq["rerank_divisor_of_reranking_factor"]) == (16, [3, 4], 2)
    assert (plain["full_cost"], plain["search_mult"], plain["rerank_mult"]) == (1, 1, 0) and (c["log_offset"], c["log_power"]) == (2.0, 2)
    fac = REF["rabitq"]["RERANKING_FACTOR"]

    def ref(total, matching, k, has_rq, M=30):
        if has_rq:
            num, den = rq["search_mult_of_reranking_factor"]
            full, smul, rmul = rq["full_cost"], fac * num // den, fac // rq["rerank_divisor_of_reranking_factor"]
        else:
            full, smul, rmul = plain["full_cost"], plain["search_mult"], plain["rerank_mult"]
        hnsw_rq = (np.log(np.float32(total)) - np.float32(c["log_offset"])) ** c["log_power"] * np.log(np.float32(k)) * np.float32(smul)
        hnsw_full = k * rmul + k * M * total // matching
        hnsw_cost = (int(hnsw_rq) if hnsw_rq > 0 else 0) + hnsw_full * full
        return hnsw_cost < matching + k * rmul * full

    for total in (100, 10_000, 200_000, 10_000_000):
        for frac in (1.0, 0.3, 0.01, 0.0001):
            matching = max(1, int(total * frac))
            for k in (1, 10, 100):
                for has_rq in (False, True):
                    assert bool(O.use_hnsw(total, matching, k, has_rabitq=has_rq, M=30)) == bool(ref(total, matching, k, has_rq)), (total, matching, k, has_rq)


def test_segment_file_names():
    """The v2 segment directory's file names (hnsw/disk/v2.rs:64-65, data_store/v2/*.rs): what the library and the mirror read and write."""
    want = {"hnsw.graph": "hnsw/disk/v2.rs:GRAPH_FILENAME", "hnsw.edges": "hnsw/disk/v2.rs:EDGES_FILENAME",
            "vectors.bin": "data_store/v2/vector_store.rs:FILENAME", "vectors.quant": "data_store/v2/quant_vector_store.rs:FILENAME",
            "paragraphs.bin": "data_store/v2/paragraph_store.rs:FILENAME_DATA", "paragraphs.pos": "data_store/v2/paragraph_store.rs:FILENAME_POS"}
    ours = open(os.path.join(ROOT, "nucliadb_b200", "csrc", "segment_io.hpp")).read() + open(os.path.join(ROOT, "nucliadb_b200", "csrc", "api.cu")).read() + \
        open(os.path.join(ROOT, "nucliadb_b200", "paragraph_store.py")).read() + open(os.path.join(ROOT, "nucliadb_b200", "vector.py")).read()
    for name, const in want.items():
        assert REF["segment_file_names"][const] == name, const
        assert f'"/{name}"' in ours or f'"{name}"' in ours, name
