#!/usr/bin/env python
"""bench.py — k-NN QPS of the nidx_vector HNSW search hot path on B200 (BASELINE.json configs[1]:
"HNSW search 10M×768 cosine, ef=128 k=10, batch=1024 on 1×B200").

A step = one batch of `--batch` queries through OpenSegment::search (segment.rs:477-567 -> hnsw/search.rs:306-383)
on one HBM-resident segment.  Contract (driver): `python bench.py --gpus N --steps K --warmup W [--impl reference]`
prints ONE JSON line on rank 0.  See DESIGN.md §measurement for what each key means.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--vectors", dest="n", type=int, default=10_000_000, help="vectors per segment (per GPU)")
    ap.add_argument("--dim", type=int, default=768)
    ap.add_argument("--batch", type=int, default=1024)
    ap.add_argument("--k", type=int, default=10)
    ap.add_argument("--ef", type=int, default=128)
    ap.add_argument("--m", type=int, default=16)
    ap.add_argument("--efc", type=int, default=200)
    ap.add_argument("--max-batch", type=int, default=8192, help="insertion batch of the GPU HNSW build")
    ap.add_argument("--data", default="latent", choices=["latent", "gauss", "clustered"],
                    help="synthetic embeddings: 'latent' (default, DESIGN.md 5) = 16-d gaussian latent -> linear map + 15 %% noise; 'gauss' = BASELINE.md 3's "
                         "N(0,1) normalised; 'clustered' = BASELINE.md 3's 4 096 centres, points = normalise(centre + 0.1 * unit noise) (segment.rs:697-706)")
    ap.add_argument("--hybrid", action="store_true",
                    help="BASELINE configs[4]: after the vector measurement every rank also indexes --hybrid-docs / N documents (BM25, doc-partitioned, global "
                         "statistics by all_reduce) and the line gains a `hybrid` block: sharded BM25 top-100 and vector + BM25 back to back per batch")
    ap.add_argument("--hybrid-docs", type=int, default=5_000_000)
    ap.add_argument("--no-extra", action="store_true", help="skip the `extra` block (BASELINE configs 1 and 4 + the quantised walk at N = 1)")
    ap.add_argument("--latent", type=int, default=16)
    ap.add_argument("--noise", type=float, default=0.15)
    ap.add_argument("--cpu-seconds", type=float, default=15.0, help="target wall time of the cpu_baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--exchange", default="lib", choices=["lib", "torch"],
                    help="N>1: 'lib' = nidx_vec_search_sharded (search -> ncclAllGather -> Fssc merge inside the library, one stream, no host code "
                         "in between); 'torch' = round 1's torch.distributed all_gather + nidx_merge_topk")
    ap.add_argument("--pipeline", action="store_true",
                    help="N>1: two batches in flight (exchange of batch i under the search of batch i+1) instead of search -> exchange -> merge back to "
                         "back; measured 1.5 %% SLOWER at N=2 (profiles/r01c_bench_2M_n2_pipelined.json): the in-line exchange costs 0.02 ms of a 1.63 ms step")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="--impl ours: after the timed steps, rank 0 writes what the last timed step returned (ids, scores, counts; parts when N>1) as DIR/<name>.npy "
                         "in float64 (ids and counts) or float32 (scores), so that two builds can be compared output for output on the same inputs")
    return ap.parse_args()


def dump_outputs(directory, names, tensors):
    """The tensors of one search result as DIR/<name>.npy: integer arrays as float64 (exact for every int32), float32 as is."""
    os.makedirs(directory, exist_ok=True)
    for name, t in zip(names, tensors):
        a = t.cpu().numpy()
        np.save(os.path.join(directory, f"{name}.npy"), a if a.dtype == np.float32 else a.astype(np.float64))


# ---- synthetic data (BASELINE.md §3 "synthetic embeddings of the named shape") ----------------------
def gen_vectors(n, d, device, seed, latent, noise, chunk=500_000):
    """Low-intrinsic-dimension embeddings: gaussian latent -> fixed random linear map + isotropic noise, L2-normalised."""
    import torch

    g = torch.Generator(device=device)
    g.manual_seed(99)
    w = torch.randn((latent, d), generator=g, device=device, dtype=torch.float32)
    g.manual_seed(seed)
    out = torch.empty((n, d), device=device, dtype=torch.float32)
    for i in range(0, n, chunk):
        m = min(chunk, n - i)
        z = torch.randn((m, latent), generator=g, device=device, dtype=torch.float32)
        v = z @ w
        v += noise * (latent ** 0.5) * torch.randn((m, d), generator=g, device=device, dtype=torch.float32)
        v /= v.norm(dim=1, keepdim=True)
        out[i:i + m] = v
    return out


def gen_vectors_gauss(n, d, device, seed, chunk=500_000):
    """BASELINE.md 3 / SURVEY 8d: standard normal f32, L2-normalised (isotropic: no neighbourhood structure at d = 768)."""
    import torch

    g = torch.Generator(device=device)
    g.manual_seed(seed)
    out = torch.empty((n, d), device=device, dtype=torch.float32)
    for i in range(0, n, chunk):
        m = min(chunk, n - i)
        v = torch.randn((m, d), generator=g, device=device, dtype=torch.float32)
        v /= v.norm(dim=1, keepdim=True)
        out[i:i + m] = v
    return out


def gen_vectors_clustered(n, d, device, seed, centres=4096, sigma=0.1, chunk=500_000):
    """BASELINE.md 3's clustered variant: 4 096 random unit centres; a point = normalise(centre + sigma * unit fuzz), the
    reference's random_nearby_vector (segment.rs:697-706, fuzz = U(-1, 1)^d normalised)."""
    import torch

    g = torch.Generator(device=device)
    g.manual_seed(4096)
    c = torch.rand((centres, d), generator=g, device=device, dtype=torch.float32) * 2 - 1
    c /= c.norm(dim=1, keepdim=True)
    g.manual_seed(seed)
    out = torch.empty((n, d), device=device, dtype=torch.float32)
    for i in range(0, n, chunk):
        m = min(chunk, n - i)
        which = torch.randint(0, centres, (m,), generator=g, device=device)
        fuzz = torch.rand((m, d), generator=g, device=device, dtype=torch.float32) * 2 - 1
        fuzz /= fuzz.norm(dim=1, keepdim=True)
        v = c[which] + sigma * fuzz
        v /= v.norm(dim=1, keepdim=True)
        out[i:i + m] = v
    return out


def make_vectors(args, n, d, device, seed):
    if args.data == "gauss":
        return gen_vectors_gauss(n, d, device, seed)
    if args.data == "clustered":
        return gen_vectors_clustered(n, d, device, seed)
    return gen_vectors(n, d, device, seed=seed, latent=args.latent, noise=args.noise)


def gen_queries(vecs, nq, seed, distance=0.05):
    """Queries near data points (segment.rs:880-883)."""
    import torch

    g = torch.Generator(device=vecs.device)
    g.manual_seed(seed)
    idx = torch.randint(0, vecs.shape[0], (nq,), generator=g, device=vecs.device)
    fuzz = torch.rand((nq, vecs.shape[1]), generator=g, device=vecs.device) * 2 - 1
    fuzz /= fuzz.norm(dim=1, keepdim=True)
    q = vecs[idx] + distance * fuzz
    q /= q.norm(dim=1, keepdim=True)
    return q.contiguous()


class ClockSampler:
    """SM clock / throttle reasons sampled DURING the timed regions (B200_PROFILING.md) through NVML (the same
    counters nvidia-smi prints; a 2 ms period needs the library, the CLI takes ~50 ms per call)."""

    def __init__(self, index):
        self.index, self.sm, self.max_sm, self.reasons, self._stop, self._t = index, [], None, set(), threading.Event(), None
        self.power, self.power_limit = [], None
        self.nv = None
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self._physical_index(index))
            self.max_sm = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            try:
                self.power_limit = pynvml.nvmlDeviceGetEnforcedPowerLimit(self.h) / 1000.0
            except Exception:
                pass
        except Exception:
            self.nv = None

    @staticmethod
    def _physical_index(i):
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            try:
                return int(vis.split(",")[i])
            except Exception:
                return i
        return i

    def _run(self):
        nv = self.nv
        names = {"hw_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
                 "hw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
                 "sw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
                 "sw_power_cap": getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4)}
        while not self._stop.is_set():
            try:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                try:
                    self.power.append(nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0)
                except Exception:
                    pass
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            self._stop.wait(0.002)

    def __enter__(self):
        if self.nv is not None:
            self._stop.clear()
            self._t = threading.Thread(target=self._run, daemon=True)
            self._t.start()
        return self

    def __exit__(self, *a):
        if self._t is not None:
            self._stop.set()
            self._t.join(timeout=2)
            self._t = None

    def summary(self):
        return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.max_sm, "reasons": sorted(self.reasons),
                "samples": len(self.sm), "source": "nvml" if self.nv is not None else "unavailable",
                "power_w": float(np.median(self.power)) if self.power else None, "power_limit_w": self.power_limit}


def effective_cores() -> int:
    """Host threads the CPU arm can really use: min(os.cpu_count(), the affinity mask, the cgroup CPU quota).  On this pool's
    GPU boxes os.cpu_count() is 128 but cpu.max is 16 CPUs: 128 threads run 2.7x SLOWER than 16 (scripts/cpu_scaling_check.py)."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = min(n, max(1, int(int(quota) / int(period))))
    except Exception:
        try:
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            p = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                n = min(n, max(1, q // p))
        except Exception:
            pass
    return n


def recall_at_k(found, truth):
    return float(np.mean([len(set(a.tolist()) & set(b.tolist())) / len(b) for a, b in zip(found, truth)]))


def export_graph_for_oracle(seg, O, n, m, m0):
    g = seg.get_graph()
    og = O.Graph(n, m, m0, g["level"])
    og.adj0, og.adjU = g["adj0"], g["adjU"]
    og.entry_node, og.entry_layer = g["entry_node"], g["entry_layer"]
    return og


def cpu_search_rate(O, host_vecs, og, host_q, k, ef, norms, threads, native):
    t0 = time.perf_counter()
    ids, sc, cnt, counters = O.hnsw_search(host_vecs, og, host_q, k, ef, nthreads=threads, native=native, norms_=norms)
    dt = time.perf_counter() - t0
    return len(host_q) / dt, ids, dt


def run_cpu_baseline(O, host_vecs, og, hq0, gpu_ids_first_batch, nq, k, ef, cores, cpu_seconds):
    """The `cpu_baseline` object: the oracle's hnsw_search on `cores` host threads over a sample of the timed batches sized for
    about `cpu_seconds` (the batches are repeated if they are too few), plus the single-thread rate and the agreement with the
    GPU's ids on the first timed batch."""
    try:
        O.build(native=True)
        native = True
    except Exception:
        native = False
    norms = O.norms(host_vecs, nthreads=cores)
    rate, _, _ = cpu_search_rate(O, host_vecs, og, hq0[:256], k, ef, norms, cores, native)
    ns = int(max(256, rate * cpu_seconds))
    reps = -(-ns // len(hq0))                              # the timed batches, repeated until the sample is ~cpu_seconds long
    sample_q = np.concatenate([hq0] * reps)[:ns] if reps > 1 else hq0[:ns]
    rate, cids, dt = cpu_search_rate(O, host_vecs, og, sample_q, k, ef, norms, cores, native)
    m = min(ns, nq, len(gpu_ids_first_batch))
    same = float(np.mean(cids[:m] == gpu_ids_first_batch[:m].astype(np.uint32)))
    rate1, _, _ = cpu_search_rate(O, host_vecs, og, hq0[:128], k, ef, norms, 1, native)      # one core, for the per-core figure
    return {"value": rate, "unit": "queries/s", "cores": cores, "kind": "port", "sample": f"{ns} queries (the timed batches{', repeated' if reps > 1 else ''}), {dt:.1f} s",
            "native_isa": native, "ids_identical_to_gpu": same, "single_thread_qps": rate1}


def run_hybrid(args, rank, world, local_rank, dev, comm, seg, queries, k, ef, multi):
    """configs[4]: every rank holds one vector segment AND the postings of its own documents.  Per batch: sharded vector search
    (search -> ncclAllGather -> Fssc merge) and sharded BM25 (local top-100 + Count -> ncclAllGather + ncclAllReduce -> merge), both
    inside the C ABI on one stream.  Statistics (N, df, tokens) are those of the union of the parts (nidx_tantivy index_reader.rs:39-77)."""
    import torch
    import torch.distributed as dist

    import bench_extra as BX
    from nucliadb_b200 import _lib
    from nucliadb_b200.dist import ShardComm
    from nucliadb_b200.segment import TextSegment
    from nucliadb_b200.text import fieldnorm_to_id

    own_comm = comm is None
    if own_comm:
        comm = ShardComm(rank, world, local_rank, exchange=(lambda b: b) if not multi else None)
    n_terms, nq, kt = 1_000_000, args.batch, 100
    per = args.hybrid_docs // world
    t0 = time.perf_counter()
    c = BX.make_corpus(per, n_terms, dev, seed=7 + rank)
    lut = np.asarray([fieldnorm_to_id(i) for i in range(int(c["lens"].max()) + 1)], dtype=np.uint8)
    fieldnorm = lut[c["lens"]]
    df = torch.from_numpy(np.diff(c["term_off"].astype(np.int64))).to(dev)
    tot = torch.tensor([per, c["total_tokens"]], dtype=torch.int64, device=dev)
    if multi:
        dist.all_reduce(df)
        dist.all_reduce(tot)
    df_h = df.cpu().numpy().astype(np.uint64)
    ts = TextSegment.create(per, n_terms, c["term_off"], c["post_doc"], c["post_tf"], fieldnorm, device=local_rank)
    ts.set_stats(int(tot[0].item()), int(tot[1].item()), df_h)
    t_setup = time.perf_counter() - t0
    rng = np.random.default_rng(11)
    band = np.nonzero((df_h >= 1_000) & (df_h <= 100_000))[0]
    qs = [rng.choice(band, 50, replace=False).astype(np.uint32) for _ in range(nq)]
    qoff = torch.tensor(np.concatenate([[0], np.cumsum([len(x) for x in qs])]), dtype=torch.int32, device=dev)
    qt = torch.tensor(np.concatenate(qs).astype(np.int64), dtype=torch.int32, device=dev)
    if multi:
        dist.broadcast(qt, src=0)
    t_out = (torch.empty((nq, kt), dtype=torch.int32, device=dev), torch.empty((nq, kt), dtype=torch.float32, device=dev),
             torch.empty((nq, kt), dtype=torch.int32, device=dev), torch.empty((nq,), dtype=torch.int32, device=dev), torch.empty((nq,), dtype=torch.int64, device=dev))
    v_out = (torch.empty((nq, k), dtype=torch.int32, device=dev), torch.empty((nq, k), dtype=torch.float32, device=dev),
             torch.empty((nq, k), dtype=torch.int32, device=dev), torch.empty((nq,), dtype=torch.int32, device=dev))

    def text_step():
        comm.search_text(ts, qt, qoff, kt, mode=_lib.NIDX_BM25_OR, use_tf=False, out=t_out)

    def both_step(i):
        comm.search_vectors(seg, queries[i % len(queries)], k, ef=ef, dedup=True, out=v_out)
        text_step()

    def timed_ms(fn, steps):
        for i in range(3):
            fn(i)
        torch.cuda.synchronize()
        if multi:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            fn(i)
        e1.record()
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if multi:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()) / steps

    ms_text = timed_ms(lambda i: text_step(), args.steps)
    ms_both = timed_ms(both_step, args.steps)
    postings = float(sum(int(df_h[t]) for q in qs for t in q)) / nq
    out = {"workload": f"hybrid: {world} x ({len(seg)} x {args.dim} vectors + {per} docs), 50-term OR queries top-{kt} + k-NN k={k} ef={ef}, batch {nq}",
           "bm25_sharded": {"ms_per_step": ms_text, "queries_per_s": nq / (ms_text * 1e-3), "docs_total": per * world, "postings_per_query": postings,
                            "note": "every query is scored on all parts; Count = ncclAllReduce, top-100 = ncclAllGather + merge (shard_merge.rs:227-231)"},
           "vector_plus_bm25": {"ms_per_step": ms_both, "hybrid_queries_per_s": nq / (ms_both * 1e-3)},
           "text_setup_seconds": t_setup}
    ts.close()
    if own_comm:
        comm.close()
    return out


def main():
    args = parse_args()
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference" and rank != 0:
        return 0
    multi = world > 1 and args.impl == "ours"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if multi:
        opts = None
        if args.pipeline:   # the exchange kernel of batch i has to slip in between the CTAs of the search of batch i + 1
            try:
                opts = dist.ProcessGroupNCCL.Options()
                opts.is_high_priority_stream = True
            except Exception:
                opts = None
        if opts is not None:
            dist.init_process_group("nccl", device_id=dev, pg_options=opts)
        else:
            dist.init_process_group("nccl", device_id=dev)

    from nucliadb_b200 import _lib
    from nucliadb_b200.dist import ShardedSearcher
    from nucliadb_b200.segment import VectorSegment

    L = _lib.require_device()
    n, d, nq, k, ef = args.n, args.dim, args.batch, args.k, args.ef
    m, m0 = args.m, 2 * args.m

    # ---- setup (untimed): data, segment, GPU HNSW build, ground truth -------------------------------
    t0 = time.perf_counter()
    vecs = make_vectors(args, n, d, dev, seed=1234567890 + rank)
    n_batches = args.steps + args.warmup
    queries = [gen_queries(vecs, nq, seed=123 + i) for i in range(n_batches)]  # same on every rank for a given i? no: per-rank data
    if multi:  # every rank must search the SAME queries: take rank 0's
        for q in queries:
            dist.broadcast(q, src=0)
    host_vecs = None
    if args.impl == "reference" or (rank == 0 and not args.no_cpu_baseline and not multi):
        host_vecs = vecs.cpu().numpy()
    seg = VectorSegment.create(vecs, d, similarity=_lib.NIDX_SIM_COSINE, m=m, m0=m0, ef_construction=args.efc, ef_search=ef, device=local_rank)
    del vecs
    torch.cuda.empty_cache()
    t_data = time.perf_counter() - t0
    t0 = time.perf_counter()
    seg.build_hnsw(seed=2, max_batch=args.max_batch)
    torch.cuda.synchronize()
    t_build = time.perf_counter() - t0
    build_counters = seg.counters()

    # exact ground truth for the first timed batch (the scan kernel, segment.rs:569-623)
    gt_ids, _, _ = seg.search(queries[args.warmup], k, method=_lib.NIDX_METHOD_BRUTE)
    torch.cuda.synchronize()
    gt = gt_ids.cpu().numpy()

    out = (torch.empty((nq, k), dtype=torch.int32, device=dev), torch.empty((nq, k), dtype=torch.float32, device=dev),
           torch.empty((nq,), dtype=torch.int32, device=dev))
    cores = effective_cores()

    if args.impl == "reference":
        # The reference's own CPU implementation of the path (oracle port; Rust cannot be built here), all host cores.
        import oracle as O

        try:
            O.build(native=True)
            native = True
        except Exception:
            native = False
        og = export_graph_for_oracle(seg, O, n, m, m0)
        norms = O.norms(host_vecs, nthreads=cores)
        sample = nq   # the whole batch: ~0.3 s of CPU work per step on the box's 16 usable cores
        host_q = [q[:sample].cpu().numpy() for q in queries]
        for i in range(args.warmup):
            cpu_search_rate(O, host_vecs, og, host_q[i], k, ef, norms, cores, native)
        t0 = time.perf_counter()
        ids0 = None
        for i in range(args.warmup, n_batches):
            _, ids, _ = cpu_search_rate(O, host_vecs, og, host_q[i], k, ef, norms, cores, native)
            if ids0 is None:
                ids0 = ids
        dt = time.perf_counter() - t0
        qps = sample * args.steps / dt
        line = {"metric": "k-NN QPS @ recall@10", "value": qps, "unit": "queries/s", "n_gpus": 1, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
                "data": "synthetic", "impl": "reference",
                "config": {"workload": f"HNSW search {n}x{d} cosine, ef={ef} k={k}, batch={nq}", "sample": f"{sample} queries of each batch per step",
                           "graph": "built by the GPU builder during setup (untimed); the timed region runs only the CPU oracle",
                           "M": m, "M0": m0, "efC": args.efc},
                "recall_at_10": recall_at_k(ids0, gt[:sample]),
                "cpu_baseline": {"value": qps, "unit": "queries/s", "cores": cores, "kind": "port", "sample": f"{sample * args.steps} queries",
                                 "native_isa": native},
                "e2e": {"value": qps, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return 0

    pipelined = multi and args.pipeline
    use_lib = multi and args.exchange == "lib" and not pipelined
    sharded = ShardedSearcher(seg, nq, k, local_rank) if multi and not use_lib else None
    comm = sh_out = None
    if use_lib:   # the library's own NCCL communicator (the id travels over the torch group, the data path does not touch torch)
        from nucliadb_b200.dist import ShardComm

        comm = ShardComm(rank, world, local_rank)
        sh_out = (torch.empty((nq, k), dtype=torch.int32, device=dev), torch.empty((nq, k), dtype=torch.float32, device=dev),
                  torch.empty((nq, k), dtype=torch.int32, device=dev), torch.empty((nq,), dtype=torch.int32, device=dev))

    def step(i):
        if use_lib:  # local search -> ncclAllGather of the partials over NVLink -> Fssc merge (segments of ONE index), all inside the C ABI call
            return comm.search_vectors(seg, queries[i], k, ef=ef, dedup=True, out=sh_out)
        if multi:  # local search -> ONE all_gather of the [2, nq, k] partials over NVLink -> in-place merge kernel
            return sharded.search(queries[i], ef)
        return seg.search(queries[i], k, ef=ef, method=_lib.NIDX_METHOD_HNSW, out=out)

    def run_steps(first, last):
        """-> the result of the last step when pipelined."""
        if not pipelined:
            for i in range(first, last):
                step(i)
            return
        for i in range(first, last):   # two batches in flight: the exchange of batch i overlaps the search of batch i + 1
            sharded.submit(queries[i], ef)
            if i > first:
                sharded.collect()
        return sharded.collect()

    # ---- warm-up + timed region: inputs resident in HBM (value) --------------------------------------
    # Everything with a host-side cost that differs between ranks (NVML initialisation: 8 processes contend for it on an
    # 8-GPU node, event creation, the sampler thread) happens BEFORE the warm-up; the barrier + synchronize sit immediately
    # before the first event, so no rank's clock runs while it waits for a slower rank's set-up.  (Round 1's N = 8 point
    # had the NVML init between the barrier and the first event: 6.4 ms/step of skew against 1.8 ms/step of work.)
    clocks = ClockSampler(local_rank)
    step_ev = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]   # step i = step_ev[i] .. step_ev[i + 1]
    run_steps(0, args.warmup)
    torch.cuda.synchronize()
    launches0 = L.nidx_launch_count()
    with clocks:
        if multi:
            dist.barrier()
        torch.cuda.synchronize()
        torch.cuda.cudart().cudaProfilerStart()  # `ncu --profile-from-start off` captures exactly the timed region
        step_ev[0].record()
        if pipelined:
            last = run_steps(args.warmup, n_batches)
        else:
            for i in range(args.warmup, n_batches):
                last = step(i)
                step_ev[i - args.warmup + 1].record()
        step_ev[-1].record()
        torch.cuda.synchronize()
        torch.cuda.cudart().cudaProfilerStop()
    if args.dump_outputs and rank == 0:   # before anything else reuses the output buffers of the timed steps
        dump_outputs(args.dump_outputs, ("ids", "scores", "parts", "counts") if use_lib else ("ids", "scores", "parts") if multi else ("ids", "scores", "counts"), last)
    ms_total = step_ev[0].elapsed_time(step_ev[-1])
    per_step = None if pipelined else [step_ev[i].elapsed_time(step_ev[i + 1]) for i in range(args.steps)]
    launches = L.nidx_launch_count() - launches0
    if multi:
        t = torch.tensor([ms_total], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total = float(t.item())
        if per_step is not None:   # per-step spread: the slowest rank's time of every step
            ps = torch.tensor(per_step, device=dev)
            dist.all_reduce(ps, op=dist.ReduceOp.MAX)
            per_step = [float(x) for x in ps.tolist()]
        dist.barrier()
    ms_step = ms_total / args.steps
    step_ms = None if per_step is None else {"min": float(np.min(per_step)), "median": float(np.median(per_step)), "max": float(np.max(per_step))}
    inline_ms = None
    if pipelined:   # context: the same steps with search -> exchange -> merge back to back (what the pipelining removes)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        dist.barrier()
        e0.record()
        for i in range(args.warmup, n_batches):
            step(i)
        e1.record()
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1)], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        inline_ms = float(t.item()) / args.steps
        dist.barrier()

    # ---- the same steps with TWO batches in flight (N = 1) ----------------------------------------------
    # A batch of 1024 queries runs as 592 + 432 CTAs (4 resident per SM): while the second wave drains, 27 % of the CTA slots are
    # empty.  The reference's searcher serves concurrent requests against one shared index (shard_search.rs:139-155); with the next
    # batch issued on a second stream its CTAs fill those slots.  Same K steps, inputs in HBM, events across both streams.
    two_streams = None
    if not multi and not pipelined:
        st2 = [torch.cuda.Stream(device=dev) for _ in range(2)]
        outs2 = [out, (torch.empty_like(out[0]), torch.empty_like(out[1]), torch.empty_like(out[2]))]
        for i in range(args.warmup):
            with torch.cuda.stream(st2[i % 2]):
                seg.search(queries[i], k, ef=ef, method=_lib.NIDX_METHOD_HNSW, out=outs2[i % 2])
        torch.cuda.synchronize()
        e0 = torch.cuda.Event(enable_timing=True)
        e_end = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        launches_a = L.nidx_launch_count()
        with clocks:
            e0.record(st2[0])
            st2[1].wait_event(e0)
            for i in range(args.warmup, n_batches):
                j = (i - args.warmup) % 2
                with torch.cuda.stream(st2[j]):
                    seg.search(queries[i], k, ef=ef, method=_lib.NIDX_METHOD_HNSW, out=outs2[j])
            for j in range(2):
                e_end[j].record(st2[j])
            torch.cuda.synchronize()
        ms2 = max(e0.elapsed_time(e_end[0]), e0.elapsed_time(e_end[1]))
        two_streams = {"value": nq * args.steps / (ms2 * 1e-3), "unit": "queries/s", "ms_per_step": ms2 / args.steps, "steps": args.steps,
                       "gpu_launches": int(L.nidx_launch_count() - launches_a),
                       "note": "the same K steps issued on two streams alternately: batch i + 1 starts while the second wave of batch i drains"}

    # ---- recall + roofline accounting (separate, synchronous passes) ----------------------------------
    ids, _, _ = seg.search(queries[args.warmup], k, ef=ef, method=_lib.NIDX_METHOD_HNSW)
    torch.cuda.synchronize()
    ids_np = ids.cpu().numpy()
    recall = recall_at_k(ids_np, gt)
    # the reference's compile-time operating point (params.rs:46 EF_SEARCH = 30) on the same graph, for context
    ef30 = None
    if not multi:
        i30, _, _ = seg.search(queries[args.warmup], k, ef=30, method=_lib.NIDX_METHOD_HNSW)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(args.warmup, min(n_batches, args.warmup + 5)):
            seg.search(queries[i], k, ef=30, method=_lib.NIDX_METHOD_HNSW, out=out)
        e1.record()
        torch.cuda.synchronize()
        n30 = min(n_batches, args.warmup + 5) - args.warmup
        ef30 = {"recall_at_10": recall_at_k(i30.cpu().numpy(), gt), "qps": nq * n30 / (e0.elapsed_time(e1) * 1e-3)}
    kernel_ms, alg_bytes = [], []
    ld = (d + 3) // 4 * 4
    for i in range(args.warmup, min(n_batches, args.warmup + 8)):
        seg.search(queries[i], k, ef=ef, method=_lib.NIDX_METHOD_HNSW, out=out)
        kernel_ms.append(seg.last_kernel_ms())
        c = seg.counters()
        alg_bytes.append(c["similarities"] * (ld * 4 + 4) + c["expansions"] * (2 * m) * 4)
        overflow = c["overflows"]
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    # The kernel's duration for the roofline comes from the TIMED REGION itself when it can: at N = 1 a step is memset + row norms
    # (~5 us) + hnsw_search_kernel, so the median per-step device time is an upper bound of the kernel's launch duration under the
    # very conditions the value was measured in (the separate accounting pass below the timed region runs after the CPU baseline
    # and the extra measurements, and on power-capped boxes comes out slower than the timed steps).  The counters are those of the
    # same query batches.  Multi-GPU steps contain the exchange, so they keep the accounting pass' kernel-only events.
    kernel_ms_accounting = float(np.mean(kernel_ms))
    kernel_ms_roof = kernel_ms_accounting if (multi or step_ms is None) else min(kernel_ms_accounting, step_ms["median"])
    achieved = float(np.mean(alg_bytes)) / (kernel_ms_roof * 1e-3) / 1e9
    workload = f"HNSW search {n}x{d} cosine, ef={ef} k={k}, batch={nq}"
    traffic = None            # DRAM bytes per launch from the committed ncu capture of this exact workload, if there is one
    try:
        traffic = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json"))).get(workload, {}).get("dram_bytes_per_launch")
    except Exception:
        pass

    # ---- e2e: the same metric through the host-buffer C ABI call (H2D + D2H inside the timed region) --
    hq = [torch.empty((nq, d), dtype=torch.float32).pin_memory() for _ in range(n_batches)]
    for h, q in zip(hq, queries):
        h.copy_(q)
    torch.cuda.synchronize()
    hq_np = [h.numpy() for h in hq]
    for i in range(args.warmup):
        seg.search(hq_np[i], k, ef=ef, method=_lib.NIDX_METHOD_HNSW)
    e2e_steps = []
    dq = torch.empty((nq, d), dtype=torch.float32, device=dev)
    host_out = (torch.empty((nq, k), dtype=torch.int32).pin_memory(), torch.empty((nq, k), dtype=torch.float32).pin_memory())
    e2e_host_out = (np.empty((nq, k), dtype=np.uint32), np.empty((nq, k), dtype=np.float32), np.empty((nq, k), dtype=np.int32), np.empty(nq, dtype=np.int32))
    if use_lib:
        for i in range(args.warmup):
            comm.search_vectors(seg, hq_np[i], k, ef=ef, dedup=True, out=e2e_host_out)
    if multi:
        dist.barrier()
    def to_host(r):
        host_out[0].copy_(r[0], non_blocking=True)
        host_out[1].copy_(r[1], non_blocking=True)

    with clocks:
        t0 = time.perf_counter()
        if pipelined:   # pinned host queries -> device, search, exchange (overlapping the next batch's search), merge, result -> pinned host
            for i in range(args.warmup, n_batches):
                dq.copy_(hq[i], non_blocking=True)
                sharded.submit(dq, ef)
                if i > args.warmup:
                    to_host(sharded.collect())
            to_host(sharded.collect())
            torch.cuda.synchronize()
            e2e_steps = [(time.perf_counter() - t0) / args.steps]
        else:
            for i in range(args.warmup, n_batches):
                t1 = time.perf_counter()
                if use_lib:  # host queries in, merged host results out: H2D, search, exchange, merge and D2H inside ONE C ABI call
                    comm.search_vectors(seg, hq_np[i], k, ef=ef, dedup=True, out=e2e_host_out)
                elif multi:  # pinned host queries -> device, sharded search + exchange + merge, merged result -> pinned host
                    dq.copy_(hq[i], non_blocking=True)
                    to_host(sharded.search(dq, ef))
                    torch.cuda.synchronize()
                else:
                    e_ids, e_sc, e_cnt = seg.search(hq_np[i], k, ef=ef, method=_lib.NIDX_METHOD_HNSW)
                e2e_steps.append(time.perf_counter() - t1)
        torch.cuda.synchronize()
        e2e_dt = time.perf_counter() - t0
    print(f"[bench] e2e per-step ms: min {min(e2e_steps) * 1e3:.3f} median {np.median(e2e_steps) * 1e3:.3f} max {max(e2e_steps) * 1e3:.3f}", file=sys.stderr)
    if multi:
        t = torch.tensor([e2e_dt], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_dt = float(t.item())
    e2e_qps = world * nq * args.steps / e2e_dt
    e2e_mode = {"calls_in_flight": 1, "one_call_at_a_time_qps": e2e_qps}
    if not multi:
        # The reference serves every request on its own blocking thread against a shared searcher (shard_search.rs:139-155); the
        # same here: two to four host threads, each with its own stream, call the re-entrant entry point on alternate batches so that
        # one call's copies and its second-wave tail overlap the other calls' kernels.  Every step still carries its own H2D and D2H inside the timed region.
        import threading

        errors = []
        names = {2: "two_calls_in_flight_qps", 3: "three_calls_in_flight_qps", 4: "four_calls_in_flight_qps"}
        for nth in (2, 3, 4):                      # concurrent blocking callers, each on its own stream (every step: H2D + kernel + D2H + sync)
            streams = [torch.cuda.Stream(device=dev) for _ in range(nth)]

            def worker(j, nth=nth, streams=streams):
                try:
                    for i in range(args.warmup + j, n_batches, nth):
                        seg.search(hq_np[i], k, ef=ef, method=_lib.NIDX_METHOD_HNSW, stream=streams[j].cuda_stream)
                except Exception as e:  # noqa: BLE001
                    errors.append(e)

            def warm(j, nth=nth, streams=streams):
                for i in range(j, min(max(args.warmup, nth), n_batches), nth):
                    seg.search(hq_np[i], k, ef=ef, method=_lib.NIDX_METHOD_HNSW, stream=streams[j].cuda_stream)

            threads = [threading.Thread(target=warm, args=(j,)) for j in range(nth)]   # workspaces allocated outside the timed region
            for th in threads:
                th.start()
            for th in threads:
                th.join()
            torch.cuda.synchronize()
            with clocks:
                threads = [threading.Thread(target=worker, args=(j,)) for j in range(nth)]
                t0 = time.perf_counter()
                for th in threads:
                    th.start()
                for th in threads:
                    th.join()
                torch.cuda.synchronize()
                dtn = time.perf_counter() - t0
            if errors:
                raise errors[0]
            qpsn = nq * args.steps / dtn
            e2e_mode[names[nth]] = qpsn
            if qpsn > e2e_qps:
                e2e_qps, e2e_mode["calls_in_flight"] = qpsn, nth

    # ---- CPU baseline (rank 0, N=1): the oracle on the host cores, bounded sample ---------------------
    cpu = None
    if rank == 0 and host_vecs is not None:
        import oracle as O

        og = export_graph_for_oracle(seg, O, n, m, m0)
        hq0 = torch.cat(queries[args.warmup:]).cpu().numpy()   # the timed batches, in order
        cpu = run_cpu_baseline(O, host_vecs, og, hq0, ids_np, nq, k, ef, cores, args.cpu_seconds)

    # ---- BASELINE configs[2] (the build that made this index): roofline of the whole build + the CPU port on a bounded sample ----
    build_extra = {}
    try:
        alg_build = float(build_counters["similarities"]) * (ld * 4 + 4)
        build_extra["roofline"] = {"bound": "hbm", "achieved": alg_build / t_build / 1e9, "peak": peak, "unit": "GB/s", "frac": alg_build / t_build / 1e9 / peak,
                                   "note": "similarities x row bytes of the whole build (search + select + reverse-link + sort) / wall seconds"}
        if rank == 0 and host_vecs is not None:
            import oracle as O

            ns = min(n, 20_000)       # the CPU port's sequential-semantics build (rayon-like parallel insertion, segment.rs:254-256) on a prefix
            secs = O.hnsw_build(host_vecs[:ns], sim=O.SIM_COSINE, M=m, M0=m0, efC=args.efc, seed=2, max_batch=256, nthreads=cores,
                                native=bool(cpu and cpu.get("native_isa"))).build_seconds
            build_extra["cpu_baseline"] = {"value": ns / secs, "unit": "vectors/s", "cores": cores, "kind": "port",
                                           "sample": f"the first {ns} vectors ({secs:.1f} s); the cost per insertion grows with log n, so the sample favours the CPU"}
    except Exception as e:  # noqa: BLE001
        build_extra["error"] = f"{type(e).__name__}: {e}"

    # ---- BASELINE configs[4]: hybrid vector + BM25 over the same ranks (doc-partitioned text index, NCCL merge inside the library) ----
    hybrid = None
    if args.hybrid and args.impl == "ours":
        hybrid = run_hybrid(args, rank, world, local_rank, dev, comm, seg, queries, k, ef, multi)

    # ---- the other BASELINE configs, N = 1 only: exact scan (configs[0]), BM25 (configs[3]), the quantised walk (SURVEY 8f rank 1) ----
    extra = None
    if rank == 0 and not multi and not args.no_extra:
        try:
            import bench_extra as BX

            host_vecs = None
            seg.close()                      # 33 GB of vectors + graph back to the allocator first
            del seg
            torch.cuda.empty_cache()
            extra = BX.driver_extras(steps=max(3, min(args.steps, 10)), warmup=max(3, min(args.warmup, 5)))
        except Exception as e:  # noqa: BLE001  (the headline line must survive a failure of the side measurements)
            extra = {"error": f"{type(e).__name__}: {e}"}

    if rank == 0:
        qps_units = world * nq * args.steps / (ms_total * 1e-3)
        line = {
            "metric": "k-NN QPS @ recall@10", "value": qps_units, "unit": "queries/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_step, "step_ms": step_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload, "segments": world, "vectors_per_segment": n, "exchange": ("pipelined, 2 batches in flight (torch)" if pipelined else ("in line, nidx_vec_search_sharded (ncclAllGather + Fssc merge in the library)" if use_lib else "in line, torch all_gather + nidx_merge_topk")) if multi else None,
                       "M": m, "M0": m0, "efC": args.efc, "l2": f"inputs larger than L2 ({n * d * 4 / 1e9:.1f} GB of vectors per GPU, fresh queries every step)",
                       "unit_note": "one unit = one query searched on one segment; merged_qps = user-visible queries/s over all segments",
                       "data_gen": ({"latent": f"latent={args.latent} noise={args.noise} normalised", "gauss": "N(0,1) normalised (BASELINE.md 3)",
                                     "clustered": "4096 centres, normalise(centre + 0.1 * unit fuzz) (BASELINE.md 3)"}[args.data]
                                    + "; queries = data point + 0.05 * unit noise")},
            "two_batches_in_flight": two_streams,
            "merged_qps": nq * args.steps / (ms_total * 1e-3),
            "exchange_in_line_ms_per_step": inline_ms,
            "recall_at_10": recall,
            "ef30": ef30,
            "build": {"workload": f"HNSW index build {n}x{d}, M={m} M0={m0} efC={args.efc}", "seconds": t_build, "vectors_per_s": n / t_build,
                      "similarities": build_counters["similarities"], "max_batch": args.max_batch, "data_seconds": t_data, **build_extra},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                         "traffic_source": "profiles/ncu_traffic.json" if traffic else None, "kernel": "hnsw_search_kernel", "kernel_ms": kernel_ms_roof, "kernel_ms_accounting_pass": kernel_ms_accounting,
                         "kernel_ms_source": "min(median device time of the timed steps (upper bound: includes memset + row norms), mean kernel-only time of the accounting pass)" if not multi else "kernel-only events of the accounting pass",
                         "alg_bytes_per_launch": float(np.mean(alg_bytes)),
                         "peak_source": "MEASURED_PEAKS.json hbm_gbs" if peaks else "fallback"},
            "cpu_baseline": cpu,
            "e2e": {"value": e2e_qps, "unit": "queries/s", "h2d_bytes_per_step": nq * d * 4, "d2h_bytes_per_step": nq * k * (12 if use_lib else 8) + nq * 4, **e2e_mode},
            "gpu_launches": int(launches),
            "hybrid": hybrid,
            "extra": extra,
            "visited_overflows": int(overflow),
            "clocks": clocks.summary(),
        }
        print(json.dumps(line))
    if comm is not None:
        comm.close()
    if multi:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.dont_write_bytecode = True   # the benchmark writes nothing into the source tree, which may be read-only
    sys.exit(main())
