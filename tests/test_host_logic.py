"""Host-side logic of the reference-interface mirror (no GPU): field keys, label filters, Fssc, BM25
host helpers, use of the oracle only as the checker."""
import os
import uuid

import numpy as np
import pytest

import oracle as O
from nucliadb_b200 import text as T
from nucliadb_b200 import vector as V


def _segment(keys, labels):
    cfg = V.VectorConfig(dimension=4)
    return V.OpenSegment(cfg, None, keys, labels, [None] * len(keys), list(range(len(keys) + 1)))


RID = "9cb39c75f8d9498d8f82d92b173011f5"


def test_field_key_matches_reference_layout():  # utils.rs:80-117
    fk = V.field_key(f"{RID}/f/file/0-100")
    assert fk == uuid.UUID(RID).bytes + b"f/file"
    assert V.field_key(RID) == uuid.UUID(RID).bytes
    assert V.field_key(f"{RID}/f") is None and V.field_key("not-a-uuid/f/x") is None


def test_label_filter_prefix_at_segment_boundary():  # inverted_index/paragraph.rs:64-66, segment/tests.rs:343-381
    seg = _segment([f"{RID}/f/a/0-1", f"{RID}/f/a/1-2", f"{RID}/f/b/0-1"], [["/l/labelset/LABEL"], ["/l/labelset/LABEL_0"], ["/l/other/x"]])
    assert seg._clause(V.Literal("/l/labelset")).tolist() == [True, True, False]
    assert seg._clause(V.Literal("/l/labelset/LABEL")).tolist() == [True, False, False]
    assert seg._clause(V.Not(V.Literal("/l/labelset"))).tolist() == [False, False, True]
    both = V.Operation("or", (V.Literal("/l/labelset/LABEL_0"), V.Literal("/l/other")))
    assert seg._clause(both).tolist() == [False, True, True]
    assert seg.filter_bitset([V.Literal("/l/labelset"), V.Literal("/l/other")], operator_and=True).tolist() == [False, False, False]
    assert seg.filter_bitset([V.Literal("/l/labelset"), V.Literal("/l/other")], operator_and=False).tolist() == [True, True, True]


def test_key_prefix_set_is_an_exact_field_lookup():  # paragraph.rs:150-155 uses field_index.get (exact)
    other = "00000000000000000000000000000001"
    seg = _segment([f"{RID}/f/a/0-1", f"{RID}/f/b/0-1", f"{other}/f/a/0-1"], [[], [], []])
    assert seg._clause(V._KeyPrefixSet(frozenset([f"{RID}/f/a"]))).tolist() == [True, False, False]
    assert seg._clause(V._KeyPrefixSet(frozenset([RID]))).tolist() == [False, False, False]


def test_fssc_matches_oracle_restatement():
    rng = np.random.default_rng(0)
    for with_dups in (True, False):
        mine, theirs = V._Fssc(5, with_dups), O.Fssc(5, with_dups)
        for i in range(60):
            pid = f"p{rng.integers(0, 20)}"
            score = float(np.float32(rng.random()))
            vb = bytes([int(rng.integers(0, 12))])
            mine.add(pid, score, i, vb)
            theirs.add(pid, score, 0, i, vb)
        seg, addr, sc = theirs.result()
        got = mine.result()
        assert [p for _, _, p in got] == list(addr)
        assert np.allclose([s for s, _, _ in got], sc)


def test_fieldnorm_code_matches_oracle_table():
    for n in list(range(0, 3000)) + [10_000, 65_535, 1_000_000, 2_013_265_944]:
        assert T.fieldnorm_to_id(n) == O.fieldnorm_to_id(n), n


def test_tokenizer_is_lowercase_alnum():
    assert T.tokenize("Hello, World! it's 42") == ["hello", "world", "it", "s", "42"]
    assert T.tokenize("x" * 41) == []
    assert T.tokenize("x" * 40) == [] and T.tokenize("x" * 39) == ["x" * 39]      # RemoveLongFilter: len < 40 ...
    assert T.tokenize("é" * 20) == [] and T.tokenize("é" * 19) == ["é" * 19]      # ... counted in UTF-8 bytes


# ---- paragraphs.bin / paragraphs.pos (data_store/v2/paragraph_store.rs; bincode 2 standard config, utils.rs:25-28) ---------
def test_bincode_varint_boundaries():
    from nucliadb_b200 import paragraph_store as PS

    cases = {0: b"\x00", 250: b"\xfa", 251: b"\xfb\xfb\x00", 65535: b"\xfb\xff\xff", 65536: b"\xfc\x00\x00\x01\x00",
             2 ** 32 - 1: b"\xfc\xff\xff\xff\xff", 2 ** 32: b"\xfd\x00\x00\x00\x00\x01\x00\x00\x00"}
    for value, enc in cases.items():
        assert PS.encode_varint(value) == enc and PS.decode_varint(enc, 0) == (value, len(enc))


def test_stored_paragraph_bytes_and_store_round_trip(tmp_path):
    from nucliadb_b200 import paragraph_store as PS

    # StoredParagraph {key: "k", labels: ["/l/a"], metadata: [1, 2], first_vector: 300, num_vectors: 1}, hand-encoded
    want = b"\x01k" + b"\x01" + b"\x04/l/a" + b"\x02\x01\x02" + b"\xfb\x2c\x01" + b"\x01"
    assert PS.encode_paragraph("k", ["/l/a"], b"\x01\x02", 300, 1) == want
    assert PS.decode_paragraph(want) == (("k", ["/l/a"], b"\x01\x02", 300, 1), len(want))
    paragraphs = [(f"9cb39c75f8d9498d8f82d92b173011f5/f/field/{i}-{i + 1}", [f"/l/set/{j}" for j in range(i % 3)], None if i % 2 else bytes(range(i % 7)), 2 * i, 2)
                  for i in range(300)]
    paragraphs.append(("x" * 300, ["y" * 70000], b"z" * 260, 2 ** 31, 7))       # lengths and integers past one byte / two bytes
    assert PS.write_paragraphs(str(tmp_path), paragraphs) == 301
    back = PS.read_paragraphs(str(tmp_path))
    assert back == [(k, list(l), (m or None), f, n) for k, l, m, f, n in paragraphs]
    assert os.path.getsize(tmp_path / "paragraphs.pos") == 301 * 4                # stored_elements = len / 4 (paragraph_store.rs:109)
    with open(tmp_path / "paragraphs.pos", "ab") as f:
        f.write(b"\xff\xff\xff\x7f")
    with pytest.raises(ValueError):
        PS.read_paragraphs(str(tmp_path))


# ---- the octet map of bm25_kernel (csrc/bm25.cuh resolve() / load_round()), restated in Python ------------------------------------
def test_bm25_octet_map_covers_every_posting_once():
    """resolve(): run r of a tile has ceil(len_r / 8) octets; pre8[] is the exclusive prefix of the octet counts in TERM order
    (the warp scans lanes, then carries over the 32-term groups), omap[o] names the run of octet o.  load_round(): thread t owns
    slots round * 4096 + u * 256 + t (u < 16); slot s is posting (s >> 3 - pre8[r]) * 8 + (s & 7) of run r = omap[s >> 3] (one
    round) or of the last run with pre8[r] <= s >> 3 (several rounds).  Every posting of the tile must be visited exactly once."""
    rng = np.random.default_rng(12)
    threads, pt = 256, 16
    slots = threads * pt
    for trial in range(40):
        nt = int(rng.integers(1, 129))
        scale = 40 if trial % 3 else 700                  # every third trial needs several rounds
        lens = (rng.integers(0, scale, nt) * (rng.random(nt) < 0.7)).astype(np.int64)
        if trial == 0:
            lens[:] = 0
        octs = (lens + 7) >> 3
        pre = np.zeros(nt + 1, dtype=np.int64)
        run = 0
        for j in range(0, nt, 32):                       # the kernel's order: 32 terms per shuffle scan, carry `run`
            c = octs[j:j + 32]
            pre[j:j + len(c)] = run + np.cumsum(c) - c
            run += int(c.sum())
        pre[nt] = run
        noct = run
        one_round = noct <= slots // 8
        omap = np.full(max(noct, 1), -1)
        for r in range(nt):
            omap[pre[r]:pre[r] + octs[r]] = r
        seen = [np.zeros(n, dtype=np.int64) for n in lens]
        for rnd in range(-(-noct // (slots // 8))):
            for s in range(rnd * slots, (rnd + 1) * slots):
                o = s >> 3
                if o >= noct:
                    continue
                if one_round:
                    r = omap[o]
                else:
                    lo, hi = 0, nt - 1
                    while lo < hi:
                        mid = (lo + hi + 1) >> 1
                        if pre[mid] <= o:
                            lo = mid
                        else:
                            hi = mid - 1
                    r = lo
                    assert r == omap[o]
                within = (o - pre[r]) * 8 + (s & 7)
                if within < lens[r]:
                    seen[r][within] += 1
        assert all((x == 1).all() for x in seen)


# ---- bench.py's CPU-side pieces (they run on the GPU box's host cores; exercised here on a small graph) -----------------------------
def test_bench_cpu_baseline_block():
    import bench
    from conftest import make_queries, make_vectors

    v = make_vectors(3000, 32, seed=50)
    g = O.hnsw_build(v, M=8, M0=16, efC=40, max_batch=64, nthreads=4)
    nq, k, ef = 64, 10, 32
    hq0 = np.concatenate([make_queries(v, nq, seed=60 + i) for i in range(3)])        # three "timed batches"
    gpu_ids, _, _, _ = O.hnsw_search(v, g, hq0[:nq], k, ef, nthreads=2)               # stands in for the GPU's first batch
    line = bench.run_cpu_baseline(O, v, g, hq0, gpu_ids.astype(np.int32), nq, k, ef, cores=2, cpu_seconds=0.2)
    assert line["kind"] == "port" and line["cores"] == 2 and line["unit"] == "queries/s"
    assert line["value"] > 0 and line["single_thread_qps"] > 0 and line["ids_identical_to_gpu"] == 1.0
    assert "repeated" in line["sample"]                                               # 192 queries do not last 0.2 s: the batches repeat
    assert bench.effective_cores() >= 1
    assert bench.recall_at_k(gpu_ids, gpu_ids) == 1.0


def test_bench_generators_and_clock_sampler_degrade_gracefully():
    import torch

    import bench

    dev = torch.device("cpu")
    v = bench.gen_vectors(2000, 48, dev, seed=1, latent=8, noise=0.15)
    assert v.shape == (2000, 48) and v.dtype == torch.float32
    assert torch.allclose(v.norm(dim=1), torch.ones(2000), atol=1e-5)                  # L2-normalised
    q = bench.gen_queries(v, 16, seed=2)
    assert q.shape == (16, 48) and torch.allclose(q.norm(dim=1), torch.ones(16), atol=1e-5)
    assert (q @ v.T).max(dim=1).values.min() > 0.9                                     # queries sit next to data points
    clocks = bench.ClockSampler(0)                                                      # no NVML / no GPU here: must not raise
    with clocks:
        pass
    s = clocks.summary()
    assert isinstance(s, dict) and "reasons" in s


def test_paragraph_store_round_trip_property():
    from hypothesis import given, settings
    from hypothesis import strategies as st

    from nucliadb_b200 import paragraph_store as PS

    paragraph = st.tuples(st.text(max_size=40), st.lists(st.text(max_size=12), max_size=4), st.one_of(st.none(), st.binary(min_size=1, max_size=300)),
                          st.integers(0, 2 ** 32 - 1), st.integers(0, 2 ** 32 - 1))

    @settings(max_examples=150, deadline=None)
    @given(st.lists(paragraph, max_size=6), st.integers(0, 2 ** 64 - 1))
    def check(paragraphs, u):
        blob = b"".join(PS.encode_paragraph(*p) for p in paragraphs)
        pos, back = 0, []
        for _ in paragraphs:
            p, pos = PS.decode_paragraph(blob, pos)
            back.append(p)
        assert pos == len(blob) and back == [(k, list(l), m, f, n) for k, l, m, f, n in paragraphs]
        enc = PS.encode_varint(u)
        assert PS.decode_varint(enc, 0) == (u, len(enc)) and len(enc) in (1, 3, 5, 9)

    check()


def test_nidx_binding_has_the_reference_surface():
    """nidx/nidx_binding/nidx_binding.pyi:15-71, as read into tests/golden/reference_facts.json: every method of the reference's
    NidxBinding exists with the same parameter names, and both port attributes are declared."""
    import inspect
    import json

    import nidx_binding

    ref = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_facts.json")))["nidx_binding"]["NidxBinding"]
    assert ref["methods"]
    for name, want in ref["methods"].items():
        got = list(inspect.signature(getattr(nidx_binding.NidxBinding, name)).parameters)
        assert got == want, (name, got, want)
    assert sorted(ref["attributes"]) == ["api_port", "searcher_port"]
    src = inspect.getsource(nidx_binding.NidxBinding.__init__)
    assert "self.searcher_port" in src and "self.api_port" in src
