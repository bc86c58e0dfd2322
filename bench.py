#!/usr/bin/env python
"""bench.py — queries/sec @ recall@10, DBpedia-1M-shaped d=768 top-10 (BASELINE.json), on 1/2/4/8 B200.

A "step" is one pass of the hot path over one batch of Q independent single-query HNSW traversals
(config C2: 1M x 768 f32, cosine, m=16/m0=32/ef_construction=200, ef=100, k=10; no cross-query sharing).

  value   : whole-job queries/sec, queries already resident in HBM (hx_search_device), CUDA-event timed.
  e2e     : the same metric through the reference-facing C-ABI call hx_search with HOST (pinned) buffers:
            H2D of the queries and D2H of ids/scores/counts are inside the timed region.
  roofline: k_hnsw_search, algorithmic bytes E*(5+8*32) + Dc*(4+4d) per launch (SURVEY §8d) / CUDA-event kernel time,
            against the measured HBM peak in MEASURED_PEAKS.json.
  cpu_baseline / --impl reference: the CPU oracle (restatement of the reference's algorithm without its KV layer)
            traversing the IDENTICAL graph on all host cores, one query per thread.
  N > 1   : one process per GPU (torchrun).  `value` is the "replica" mode: the QUERIES are partitioned across full
            replicas (no data-path collective; weak scaling: Q queries per GPU per step).  The same line carries a
            "sharded" object: the 1M corpus split by id range, every rank searching every query on its shard through
            hx_search_sharded_device (C ABI: local search into the send block, ONE ncclAllGather issued by the library,
            (score,id) merge kernel), per-shard ef tuned to iso-recall with the unsharded index; and "dense_c4": the
            C4 shape (1.25M x 768 bf16 rows per GPU, batch 1024) through the tensor-core path, sharded the same way.
  N = 1   : the line also carries driver-visible sub-results for the other BASELINE configs, each with its own
            roofline / e2e / cpu_baseline / parity flags: "prefilter" (C3 label sets + the reference's contiguous
            100/1k/10k/100k shapes), "dense_c4" (one C4 shard), "concurrent_callers" (the reference's calling pattern:
            1..256 callers x one query per call through hx_service), "euclid_d1536" (the reference's own traversal
            fixture shape: 1M x 1536, Euclidean).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

SEED = 0x0DB9ED1A          # SURVEY §8(d)
N_CENTROIDS = 1024
K = 10
EF = 100
# Synthetic corpus recipes (no network => no DBpedia download):
#  "embedding" (default): 1024-component Gaussian mixture in a 32-d latent space (sigma 1.0: overlapping clusters) pushed
#      through a fixed random 768x32 projection + 2 % isotropic noise, unit-normalised.  Intrinsic dimension ~32 like real
#      sentence embeddings; HNSW (m=16, ef=100) reaches recall@10 ~0.97 on it, as it does on DBpedia-OpenAI-1M.
#  "survey": SURVEY §8(d)'s literal example — 1024 isolated isotropic clusters in full 768-d (sigma 0.3).  Its landscape is
#      flat between clusters, so ANY greedy HNSW descent (reference algorithm included) lands in a wrong cluster for ~7 %
#      of the queries at 1M (profiles/r01_recall_diag_survey_mixture.json): recall@10 0.89 at ef=100, 0.91 at ef=200.
RECIPES = {"embedding": dict(kind=32, sigma=1.0), "survey": dict(kind=0, sigma=0.3)}
KIND = 32
SIGMA = 1.0


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--n", "--rows", dest="n", type=int, default=1_000_000)
    ap.add_argument("--dim", type=int, default=768)
    ap.add_argument("--queries-per-step", type=int, default=32768)
    ap.add_argument("--metric", default="cosine", choices=["cosine", "euclidean"])
    ap.add_argument("--recall-queries", type=int, default=512)
    ap.add_argument("--cpu-seconds", type=float, default=15.0)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-sharded", action="store_true")
    ap.add_argument("--no-default-mode", action="store_true")
    ap.add_argument("--workload", default="hnsw", choices=["hnsw", "prefilter", "dense"])
    ap.add_argument("--no-subresults", action="store_true", help="skip the prefilter / dense / callers / d1536 sub-results")
    ap.add_argument("--no-d1536", action="store_true")
    ap.add_argument("--d1536-rows", type=int, default=1_000_000)
    ap.add_argument("--dense-rows-per-gpu", type=int, default=1_250_000)
    ap.add_argument("--dense-batch", type=int, default=1024)
    ap.add_argument("--callers-seconds", type=float, default=1.0)
    ap.add_argument("--recipe", default="embedding", choices=sorted(RECIPES))
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write rank 0's results of the last timed step (ids, scores, counts) to DIR/<name>.npy")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and (a.impl != "ours" or a.workload != "hnsw"):
        ap.error("--dump-outputs applies to the default workload (--impl ours --workload hnsw)")
    global KIND, SIGMA
    KIND, SIGMA = RECIPES[a.recipe]["kind"], RECIPES[a.recipe]["sigma"]
    return a


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""

    def __init__(self, device_index: int):
        self.idx = device_index
        self.proc = None
        self.lines = []

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms",
                                          "50", "-i", str(self.idx)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], 0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            p = [x.strip() for x in ln.split(",")]
            if len(p) < 7:
                continue
            try:
                sm.append(float(p[0]))
                mx = max(mx, float(p[1]))
            except ValueError:
                continue
            for nm, v in zip(names, p[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx or None, "samples": len(sm),
                "reasons": sorted(reasons)}


def available_cores():
    """Host threads this process can really use: affinity mask capped by the cgroup CPU quota (cpu.max)."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    try:
        txt = Path("/sys/fs/cgroup/cpu.max").read_text().split()
        if txt[0] != "max":
            n = max(1, min(n, int(float(txt[0]) / float(txt[1]) + 0.5)))
    except Exception:
        pass
    return n


def measured_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic(kernel: str, shape: dict):
    """Per-launch DRAM bytes of the dominant kernel from the committed ncu summary — only when the capture was taken on
    a launch of this very shape (a number for another launch size would not be "per launch like achieved"), else None."""
    p = ROOT / "profiles" / "ncu_summary.json"
    if p.exists():
        try:
            e = json.loads(p.read_text()).get(kernel, {})
            return e.get("dram_bytes_per_launch") if e.get("shape") == shape else None
        except Exception:
            return None
    return None


# ------------------------------------------------------------------------------------------------------------------
def build_index(hx, args, device, first_id, n, storage=0):
    metric = hx.Metric.Cosine if args.metric == "cosine" else hx.Metric.Euclidean
    cfg = hx.VectorIndexConfig("dbpedia_1m_synthetic", "embedding", args.dim)   # m=16, m0=32, ef_c=200 defaults
    ix = hx.VectorIndex(metric, cfg, device=device, storage=storage)
    t0 = time.perf_counter()
    ix.generate_vectors(first_id, n, SEED, N_CENTROIDS, SIGMA, KIND)
    t1 = time.perf_counter()
    ix.build(seed=SEED)
    t2 = time.perf_counter()
    return ix, {"generate_s": round(t1 - t0, 2), "build_s": round(t2 - t1, 2)}


def oracle_from_device(hxo, ix, args):
    """Mirror the device index (vectors + graph) into the CPU oracle so both traverse identical adjacency."""
    metric = hxo.COSINE if args.metric == "cosine" else hxo.EUCLIDEAN
    ora = hxo.Index(metric, args.dim)
    g = ix.download_graph()
    n = g["n"]
    chunk = 65536
    for lo in range(0, n, chunk):
        ids, rows = ix.download_vectors(lo, min(chunk, n - lo))
        ora.put_vectors(ids, rows)
    ora.import_graph(g["levels"], g["deg0"], g["nbr0"], g["layer0_stride"], g["upper_node"], g["upper_layer"],
                     g["upper_deg"], g["upper_nbr"], g["upper_stride"], g["entry_point"], g["max_layer"])
    return ora


def exact_topk_device_full(hx, torch, ix, queries, n, first_id, k):
    """Ground truth by the exact scan kernel over ALL rows (same metric, same (score,id) tie rule).  The restricted
    entry point accepts at most 1e6 candidates (the reference's bound), so larger shards are scanned in 1M-row ranges
    whose top-k lists are merged by the (score,id) merge kernel.  Returns (ids u64 [B,k], scores f32 [B,k], counts)."""
    dev = torch.device("cuda", ix.device)
    B = len(queries)
    dq = torch.from_numpy(queries).to(dev)
    stream = torch.cuda.current_stream(dev).cuda_stream
    R = 1_000_000
    ranges = [(a, min(n, a + R)) for a in range(0, n, R)]
    a_ids = torch.zeros((len(ranges), B, k), dtype=torch.int64, device=dev)
    a_sc = torch.zeros((len(ranges), B, k), dtype=torch.float32, device=dev)
    a_cnt = torch.zeros((len(ranges), B), dtype=torch.int32, device=dev)
    step = 64
    for ri, (a, b) in enumerate(ranges):
        slots = torch.arange(a, b, dtype=torch.int32, device=dev)
        for lo in range(0, B, step):
            bb = min(step, B - lo)
            ix.search_restricted_device(dq[lo:lo + bb].data_ptr(), bb, hx.SearchParams.strict(k), slots.data_ptr(), 0,
                                        b - a, b - a, a_ids[ri, lo:lo + bb].data_ptr(), a_sc[ri, lo:lo + bb].data_ptr(),
                                        a_cnt[ri, lo:lo + bb].data_ptr(), stream)
        torch.cuda.synchronize(dev)
    ix.last_kernel_ms()
    if len(ranges) == 1:
        return a_ids[0].cpu().numpy().view(np.uint64), a_sc[0].cpu().numpy(), a_cnt[0].cpu().numpy()
    o_ids = torch.zeros((B, k), dtype=torch.int64, device=dev)
    o_sc = torch.zeros((B, k), dtype=torch.float32, device=dev)
    o_cnt = torch.zeros((B,), dtype=torch.int32, device=dev)
    hx.merge_topk_device(ix.device, a_ids.data_ptr(), a_sc.data_ptr(), a_cnt.data_ptr(), len(ranges), B, k,
                         o_ids.data_ptr(), o_sc.data_ptr(), o_cnt.data_ptr(), stream)
    torch.cuda.synchronize(dev)
    return o_ids.cpu().numpy().view(np.uint64), o_sc.cpu().numpy(), o_cnt.cpu().numpy()


def exact_topk_device(hx, torch, ix, queries, n, first_id, k):
    return exact_topk_device_full(hx, torch, ix, queries, n, first_id, k)[0]


def c2_config(args, world):
    """The `config` object of the C2 line — shared verbatim by our arm and the --impl reference arm."""
    n, dim, Q = args.n, args.dim, args.queries_per_step
    cfg = {
        "workload": f"C2: {n}x{dim} f32 {args.metric} HNSW top-10 (m=16, m0=32, ef_construction=200, ef={EF}), "
                    f"independent single-query traversals (batch=1 semantics, no cross-query sharing), "
                    f"{Q} queries per GPU per step",
        "queries_per_step_per_gpu": Q,
        "parallelism": "single GPU" if world == 1 else f"{world} full replicas, queries partitioned, no data-path collective",
        "value_mode": "single GPU" if world == 1 else "replicas (the id-range-sharded path is the `sharded` object)",
        "l2": f"corpus {n * dim * 4 / 1e9:.2f} GB >> 126 MB L2; distinct queries every step and rank",
        "graph": "built on the device (hx_index_build), identical adjacency mirrored into the CPU oracle",
        "data_recipe": (f"{args.recipe}: unit-normalised {N_CENTROIDS}-component Gaussian mixture, sigma={SIGMA}, "
                        + (f"rank-{KIND} latent space -> fixed random projection to {dim}-d + 2% noise"
                           if KIND else f"isolated isotropic clusters in {dim}-d") + ", seed=0x0DB9ED1A"),
    }
    return cfg


def recall_at_k(found, truth):
    hit = 0
    for f, t in zip(found, truth):
        hit += len(set(f.tolist()) & set(t.tolist()))
    return hit / float(truth.size)


QUERY_RING = 16


def step_sets(n_sets, make):
    """The query set of each of n_sets steps (warm-up included), make(set index) called at most QUERY_RING times so that
    memory does not grow with --steps.  Step 0 keeps set 0 (the recall and parity checks read it) and the last
    QUERY_RING - 1 steps keep their own sets; the steps in between cycle through those, so consecutive steps never share a
    set and up to QUERY_RING steps every step has a set of its own."""
    r = QUERY_RING - 1
    order = [0] + [s + (n_sets - 1 - s) // r * r for s in range(1, n_sets)]
    made = {}
    for i in order:
        if i not in made:
            made[i] = make(i)
    return [made[i] for i in order]


def map_sets(sets, f):
    """[f(q) for q in sets], f applied once per distinct set: steps that share a set share its copy."""
    done = {}
    for q in sets:
        if id(q) not in done:
            done[id(q)] = f(q)
    return [done[id(q)] for q in sets]


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, ids, scores, counts):
    """Writes one step's answer as the caller receives it: ids [B,k] as float64 (exact below 2^53), scores [B,k] and
    counts [B] as float32.  Above DUMP_BYTES a fixed seeded sample of query rows stands for the batch; the sampled row
    indices are written as sample_rows.npy."""
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    rows = np.arange(len(counts))
    row_bytes = ids.shape[1] * 8 + scores.shape[1] * 4 + 4 + 8
    if len(rows) * row_bytes > DUMP_BYTES:
        rows = np.sort(np.random.default_rng(SEED).choice(len(rows), (DUMP_BYTES - 4096) // row_bytes, replace=False))
        np.save(out / "sample_rows.npy", rows.astype(np.float64))
    np.save(out / "ids.npy", ids[rows].astype(np.float64))
    np.save(out / "scores.npy", scores[rows].astype(np.float32))
    np.save(out / "counts.npy", counts[rows].astype(np.float32))


# ------------------------------------------------------------------------------------------------------------------
# Sub-results carried by the default line (driver-visible evidence for every BASELINE config, VERDICT r1 item 1c)
REF_PREFILTER_SHAPES = [("prefilter-100", 0, 100), ("prefilter-1000", 100, 1_000), ("prefilter-10000", 1_100, 10_000),
                        ("prefilter-100000", 11_100, 100_000)]   # index_lifecycle_scale.rs:583-613 (contiguous id ranges)


def _timed_device(torch, dev, steps, warmup, fn):
    for s in range(warmup):
        fn(s)
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for s in range(steps):
        fn(warmup + s)
    e1.record()
    torch.cuda.synchronize(dev)
    return e0.elapsed_time(e1)


def measure_prefilter(hx, torch, ix, args, dev, stream, n, dim, ora=None):
    """Config C3 on an index whose ids are 0..n-1: (a) the graph-label filter — 100 queries per step, query b restricted to
    {id : id mod 100 == b} (1 % each: one step streams every row once), (b) the reference's own prefilter shapes — one
    contiguous id range of 100 / 1k / 10k / 100k candidates shared by 64 queries.  Exact scan (k_scan + k_select);
    the oracle's restricted_exact_scan checks ids and score bits."""
    import ctypes as C
    k, sel = K, 100
    B = sel
    steps = args.steps
    hbm_peak, peak_src = measured_peaks()
    n_sets = steps + args.warmup
    qsets = step_sets(n_sets, lambda s: ix.generate_queries(SEED, B, first_query=20_000_000 + s * B, n_centroids=N_CENTROIDS,
                                                            sigma=SIGMA, kind=KIND))
    cand_lists = [np.arange(b, n, sel, dtype=np.uint64) for b in range(B)]
    cand_ids = np.concatenate(cand_lists)
    offs = np.zeros(B + 1, dtype=np.uint64)
    offs[1:] = np.cumsum([len(c) for c in cand_lists])
    per_q = int(max(len(c) for c in cand_lists))
    total = int(offs[-1])
    d_slots = torch.from_numpy(cand_ids.astype(np.uint32).view(np.int32)).to(dev)      # ids == slots here (first_id 0)
    d_offs = torch.from_numpy(offs.view(np.int64)).to(dev)
    d_q = map_sets(qsets, lambda q: torch.from_numpy(q).to(dev))
    o_ids = torch.zeros((B, k), dtype=torch.int64, device=dev)
    o_sc = torch.zeros((B, k), dtype=torch.float32, device=dev)
    o_cnt = torch.zeros((B,), dtype=torch.int32, device=dev)
    params = hx.SearchParams.strict(k)
    hdr = 4 if args.metric == "cosine" else 0

    def step_device(s):
        ix.search_restricted_device(d_q[s].data_ptr(), B, params, d_slots.data_ptr(), d_offs.data_ptr(), total, per_q,
                                    o_ids.data_ptr(), o_sc.data_ptr(), o_cnt.data_ptr(), stream)

    ix.last_kernel_ms()
    for s in range(args.warmup):
        step_device(s)
    torch.cuda.synchronize(dev)
    ix.last_kernel_ms()
    ms_total = _timed_device(torch, dev, steps, 0, lambda s: step_device(args.warmup + s))
    kms, kl = ix.last_kernel_ms()
    value = steps * B / (ms_total / 1e3)
    bytes_per_launch = total * (4 * dim + hdr)
    kernel_ms = kms / max(kl, 1)
    achieved = bytes_per_launch / (kernel_ms * 1e-3) / 1e9
    dev_ids = o_ids.cpu().numpy().view(np.uint64).copy()
    dev_sc = o_sc.cpu().numpy().copy()
    last_q = qsets[args.warmup + steps - 1]
    L = hx.load_library()
    cp = params._c()
    h_q = map_sets(qsets, lambda q: torch.from_numpy(q).pin_memory())
    h_c = torch.from_numpy(cand_ids.view(np.int64)).pin_memory()
    h_o = torch.from_numpy(offs.view(np.int64)).pin_memory()
    h_ids = torch.zeros((B, k), dtype=torch.int64).pin_memory()
    h_sc = torch.zeros((B, k), dtype=torch.float32).pin_memory()
    h_cnt = torch.zeros((B,), dtype=torch.int32).pin_memory()

    def step_host(s):
        rc = L.hx_search_restricted_multi(ix.h, C.cast(h_q[s].data_ptr(), C.POINTER(C.c_float)), B, C.byref(cp),
                                          C.cast(h_c.data_ptr(), C.POINTER(C.c_uint64)),
                                          C.cast(h_o.data_ptr(), C.POINTER(C.c_uint64)),
                                          C.cast(h_ids.data_ptr(), C.POINTER(C.c_uint64)),
                                          C.cast(h_sc.data_ptr(), C.POINTER(C.c_float)),
                                          C.cast(h_cnt.data_ptr(), C.POINTER(C.c_uint32)), None)
        if rc != 0:
            raise RuntimeError(L.hx_last_error().decode())

    for s in range(args.warmup):
        step_host(s)
    t0 = time.perf_counter()
    for s in range(steps):
        step_host(args.warmup + s)
    e2e_value = steps * B / (time.perf_counter() - t0)
    same = bool(h_ids.numpy().view(np.uint64).tolist() == dev_ids.tolist() and h_sc.numpy().tobytes() == dev_sc.tobytes())
    # label sets resident on the device (hx_candidates: uploaded + mapped once, like a label bitmap cached per snapshot)
    t0 = time.perf_counter()
    dsets = [ix.cache_candidates(hx.RestrictedVectorCandidates(c)) for c in cand_lists]
    cache_s = time.perf_counter() - t0
    set_arr = (C.c_void_p * B)(*[d.h for d in dsets])

    def step_host_sets(s):
        rc = L.hx_search_restricted_sets(ix.h, C.cast(h_q[s].data_ptr(), C.POINTER(C.c_float)), B, C.byref(cp), set_arr, B,
                                         C.cast(h_ids.data_ptr(), C.POINTER(C.c_uint64)),
                                         C.cast(h_sc.data_ptr(), C.POINTER(C.c_float)),
                                         C.cast(h_cnt.data_ptr(), C.POINTER(C.c_uint32)), None)
        if rc != 0:
            raise RuntimeError(L.hx_last_error().decode())

    for s in range(args.warmup):
        step_host_sets(s)
    t0 = time.perf_counter()
    for s in range(steps):
        step_host_sets(args.warmup + s)
    e2e_sets = steps * B / (time.perf_counter() - t0)
    same_sets = bool(h_ids.numpy().view(np.uint64).tolist() == dev_ids.tolist() and h_sc.numpy().tobytes() == dev_sc.tobytes())
    for d in dsets:
        d.close()

    # ---- the reference's contiguous shapes: one candidate range shared by 64 queries ----
    # each shape is answered twice: exactly (scan) and by the reference's own plan for |C| > 256, the filter-aware (ACORN)
    # walk (restricted.rs:837-1148; needs node fingerprints: a stand-in hyperplane table when none is loaded)
    shapes = []
    SB = 64
    acorn_ready = False
    try:
        ix.download_simhash(0, 1)
        acorn_ready = True
    except Exception:
        try:
            ix._bench_planes = np.random.default_rng(42).standard_normal((64, dim)).astype(np.float32)
            ix.set_simhash_planes(ix._bench_planes)
            ix.compute_simhash()
            acorn_ready = True
        except Exception:
            acorn_ready = False
    ora_sim = False

    def hxo_simhash(planes, v):
        from oracle import hxo as _h
        return _h.simhash_from_planes(planes, v)
    sq = ix.generate_queries(SEED, SB, first_query=21_000_000, n_centroids=N_CENTROIDS, sigma=SIGMA, kind=KIND)
    d_sq = torch.from_numpy(sq).to(dev)
    s_ids = torch.zeros((SB, k), dtype=torch.int64, device=dev)
    s_sc = torch.zeros((SB, k), dtype=torch.float32, device=dev)
    s_cnt = torch.zeros((SB,), dtype=torch.int32, device=dev)
    for name, start, count in REF_PREFILTER_SHAPES:
        if start + count > n:
            continue
        cids = np.arange(start, start + count, dtype=np.uint64)
        dsl = torch.from_numpy(cids.astype(np.uint32).view(np.int32)).to(dev)

        def step_shape(_s):
            ix.search_restricted_device(d_sq.data_ptr(), SB, params, dsl.data_ptr(), 0, count, count, s_ids.data_ptr(),
                                        s_sc.data_ptr(), s_cnt.data_ptr(), stream)

        ix.last_kernel_ms()
        ms = _timed_device(torch, dev, steps, args.warmup, step_shape)
        kms2, kl2 = ix.last_kernel_ms()
        g_ids = s_ids.cpu().numpy().view(np.uint64).copy()
        g_sc = s_sc.cpu().numpy().copy()
        t0 = time.perf_counter()
        for _ in range(steps):
            hi, hs, hc = ix.search_restricted_batch(sq, params, hx.RestrictedVectorCandidates(cids))
        e2e = steps * SB / (time.perf_counter() - t0)
        ent = {"shape": name, "candidates": count, "id_range": [start, start + count], "queries_per_step": SB,
               "value": round(steps * SB / (ms / 1e3), 1), "e2e": round(e2e, 1), "unit": "queries/s",
               "kernel_ms_per_launch": round(kms2 / max(kl2, 1), 4),
               "scan_GBps": round(SB * count * (4 * dim + hdr) / (kms2 / max(kl2, 1) * 1e-3) / 1e9, 1) if kms2 else None,
               "reference_plan": hx.restricted_plan(count, dim),
               "note": "one candidate range shared by the 64 queries of a step: rows are re-read from L2, so scan_GBps can exceed the HBM peak",
               "host_path_identical_to_device_path": bool(hi.tolist() == g_ids.tolist() and hs.tobytes() == g_sc.tobytes())}
        if ora is not None:
            nchk = 8 if count <= 10_000 else 2
            ok = True
            t0 = time.perf_counter()
            for b in range(nchk):
                ei, es = ora.search_restricted(sq[b], k, cids)
                ok = ok and g_ids[b, :len(ei)].tolist() == ei.tolist() and g_sc[b, :len(ei)].tobytes() == es.tobytes()
            ent["oracle_bit_exact"] = bool(ok)
            ent["cpu_port_qps_1thread"] = round(nchk / (time.perf_counter() - t0), 1)
        if acorn_ready and count > 256 and ix.graph_info()["max_layer"] > 0:   # the walk needs a real graph
            pa = hx.SearchParams.new(k)                              # ef = 100 -> ef_filtered 150, <= 800 vectors scored
            cset = hx.RestrictedVectorCandidates(cids)
            fst = hx.FilteredStats()
            try:
                # one CTA per query: 296 queries per call fill the 148 SMs twice over (the 64-query step above would leave
                # more than half of them idle); both plans are timed through the same host entry points on the same queries
                AB = 296
                aq = ix.generate_queries(SEED, AB, first_query=22_000_000, n_centroids=N_CENTROIDS, sigma=SIGMA, kind=KIND)
                x_ids, _, x_cnt = ix.search_restricted_batch(aq, params, cset)
                t0 = time.perf_counter()
                for _ in range(steps):
                    ix.search_restricted_batch(aq, params, cset)
                x_qps = steps * AB / (time.perf_counter() - t0)
                a_ids, a_sc, a_cnt = ix.search_filtered_graph(aq, pa, cset, stats=fst)
                t0 = time.perf_counter()
                for _ in range(steps):
                    ix.search_filtered_graph(aq, pa, cset)
                a_qps = steps * AB / (time.perf_counter() - t0)
                hit = sum(len(set(a_ids[b, :a_cnt[b]].tolist()) & set(x_ids[b, :x_cnt[b]].tolist())) for b in range(AB))
                ac = {"qps": round(a_qps, 1), "exact_scan_qps_same_queries": round(x_qps, 1), "queries_per_call": AB,
                      "recall_at_10_vs_exact": round(hit / float(AB * k), 4),
                      "vectors_scored_per_query": round(fst.vector_payload_requests / AB, 1),
                      "bridge_rows_per_query": round(fst.bridge_rows / AB, 1),
                      "kernel": "k_filtered_walk (one CTA per query)", "faster_than_exact_scan": bool(a_qps > x_qps)}
                if ora is not None:
                    if not ora_sim:
                        nn = n
                        ora.put_simhash(np.arange(nn, dtype=np.uint64), ix.download_simhash(0, nn))
                        ora_sim = True
                    okw = True
                    for b in range(2):
                        # the device projected the query fingerprints from the planes; project the same way on the host
                        pl = getattr(ix, "_bench_planes", None)
                        if pl is None:
                            break
                        oi, osc, _ = ora.search_filtered_graph(aq[b], k, cids, hxo_simhash(pl, aq[b]), ef=100)
                        okw = okw and a_ids[b, :a_cnt[b]].tolist() == oi.tolist() and a_sc[b, :a_cnt[b]].tobytes() == osc.tobytes()
                    else:
                        ac["oracle_bit_exact"] = bool(okw)
                ent["acorn_walk"] = ac
            except hx.HelixDbError as e:
                ent["acorn_walk"] = {"error": str(e)}
        shapes.append(ent)

    cpu = None
    if ora is not None:
        cores = available_cores()
        ci, cs, cc, secs = ora.search_restricted_batch(last_q, k, cand_ids, offs, threads=cores)
        parity = bool(ci.tolist() == dev_ids.tolist() and cs.tobytes() == dev_sc.tobytes())
        cpu = {"value": round(B / secs, 1), "unit": "queries/s", "cores": cores, "kind": "port",
               "sample": f"the last step's {B} queries x {per_q} candidates, one query per thread, {cores} threads",
               "bit_exact_vs_device": parity}
    out = {
        "metric": "queries/sec, DBpedia-1M d=768 prefiltered top-10 (graph-label filter), exact scan (config C3)",
        "value": round(value, 1), "unit": "queries/s", "steps": steps, "ms_per_step": round(ms_total / steps, 4),
        "recall_at_10": 1.0, "dtype": "f32",
        "config": {"workload": f"C3: {n}x{dim} f32 {args.metric}, {B} queries per step, query b restricted to "
                               f"{{id : id mod {sel} == b}} ({per_q} candidates each): every row read once per step",
                   "l2": f"{n * dim * 4 / 1e9:.2f} GB streamed per step >> 126 MB L2"},
        "e2e": {"value": round(e2e_value, 1), "unit": "queries/s", "h2d_bytes_per_step": B * dim * 4 + total * 8 + (B + 1) * 8,
                "d2h_bytes_per_step": B * (k * 12 + 4) + B * 4 + 4, "api": "hx_search_restricted_multi (C ABI, pinned host)",
                "identical_to_device_path": same},
        "e2e_device_resident_sets": {"value": round(e2e_sets, 1), "unit": "queries/s",
                                     "h2d_bytes_per_step": B * dim * 4 + B * 24, "d2h_bytes_per_step": B * (k * 12 + 4) + B * 4 + 4,
                                     "api": "hx_search_restricted_sets (label sets uploaded once with hx_candidates_create)",
                                     "sets_upload_s": round(cache_s, 3), "identical_to_device_path": same_sets},
        "gpu_launches": steps * 2, "launches_per_step": {"k_validate_and_header": 1, "k_scan_topk": 1},
        "roofline": {"bound": "hbm", "kernel": "k_scan_topk (bit-exact scan + warp-shuffle top-k, one launch)", "achieved": round(achieved, 1), "peak": hbm_peak, "unit": "GB/s",
                     "frac": round(achieved / hbm_peak, 4),
                     "traffic": ncu_traffic("k_scan_topk", {"queries": B, "candidates": per_q, "dim": dim}), "peak_source": peak_src,
                     "algorithmic_bytes_per_launch": int(bytes_per_launch), "kernel_ms_per_launch": round(kernel_ms, 4)},
        "reference_shapes": shapes,
    }
    if cpu:
        out["cpu_baseline"] = cpu
    return out


def measure_callers(hx, ix, queries, k, ef, seconds):
    """The reference's calling pattern (read_index.rs:81-101: one query per call, one call per tokio task, many tasks):
    N concurrent callers through hx_service, driven by the C++ host harness (host/hx_callers.cpp).  `blocking` = N OS
    threads each in hx_service_search; `tasks` = N logical callers multiplexed on 8 threads with submit / poll."""
    from helix_db_b200 import callers
    ref_ids, ref_sc, ref_cnt = ix.search_batch(queries, hx.SearchParams.strict(k, ef))
    svc = ix.service(k, ef, capacity=2048, max_batch=128)
    info = svc.stats()
    rows = []
    all_exact = True
    for mode, ncall, nthr in (("blocking", 1, 0), ("blocking", 16, 0), ("blocking", 64, 0), ("blocking", 256, 0),
                              ("tasks", 256, 8), ("tasks", 1024, 8)):
        rep, ids, sc, cnt = callers.run(svc, ix, queries, k, ef, ncall, mode=mode, n_threads=nthr, seconds=seconds)
        exact = bool(ids.tolist() == ref_ids.tolist() and sc.tobytes() == ref_sc.tobytes() and cnt.tolist() == ref_cnt.tolist())
        all_exact = all_exact and exact and rep["errors"] == 0
        rows.append({"mode": mode, "callers": ncall, "host_threads": rep["threads"], "qps": round(rep["qps"], 1),
                     "p50_us": rep["p50_us"], "p99_us": rep["p99_us"], "max_us": rep["max_us"],
                     "completed": rep["completed"], "bit_exact_vs_hx_search": exact})
    st = svc.stats()
    svc.close()
    direct = []
    for ncall in (1, 16):   # round-1 path for comparison: a blocking B = 1 hx_search per caller thread, no service
        rep, _, _, _ = callers.run(None, ix, queries[:1024], k, ef, ncall, mode="direct", seconds=min(seconds, 0.5))
        direct.append({"callers": ncall, "qps": round(rep["qps"], 1), "p50_us": rep["p50_us"], "p99_us": rep["p99_us"]})
    best256 = max((r for r in rows if r["callers"] == 256), key=lambda r: r["qps"])
    return {"api": "hx_service_submit / hx_service_poll / hx_service_search (C ABI), one query per call",
            "kernel": "k_hnsw_search_cta_ring, one CTA per query, results written to host-mapped slots",
            "launch_shape": {x: info[x] for x in ("cta_warps", "rows_in_flight", "visited_cap", "smem_bytes", "ctas_per_sm")},
            "queries_pool": int(len(queries)), "runs": rows, "at_256_callers": {"qps": best256["qps"], "p99_us": best256["p99_us"],
                                                                              "mode": best256["mode"]},
            "launches": st["launches"], "queries_per_launch_avg": round(st["completed"] / max(st["launches"], 1), 2),
            "max_batch_seen": st["max_batch_seen"], "all_bit_exact": all_exact,
            "direct_hx_search_b1_per_thread": direct}


def measure_dense(hx, torch, args, world, rank, local_rank, dev, stream, uid):
    """C4 shape: exhaustive top-10 of a 1024-query batch against 1.25M x 768 bf16 rows PER GPU through the tensor cores
    (k_dense_scores: tcgen05 + TMEM + TMA), nominees re-ranked by the exact fp32 scan; with N > 1 the corpus is the
    id-range union of the ranks' shards (8 GPUs = C4's 10M rows) and every step ends with ONE ncclAllGather + merge
    (hx_search_sharded*, issued by the library)."""
    from helix_db_b200 import sharding as sh
    rows, dim, k, B = args.dense_rows_per_gpu, args.dim, K, args.dense_batch
    lo = rank * rows
    metric = hx.Metric.Cosine if args.metric == "cosine" else hx.Metric.Euclidean
    ix = hx.VectorIndex(metric, hx.VectorIndexConfig("dense_c4", "embedding", dim), device=local_rank, storage=1)
    t0 = time.perf_counter()
    ix.generate_vectors(lo, rows, SEED, N_CENTROIDS, SIGMA, KIND)
    ix.load_graph(0, np.array([lo], np.uint64), np.array([0, 0], np.uint32), np.zeros(0, np.uint64))
    ix.set_entry(lo, 0)
    gen_s = time.perf_counter() - t0
    if world > 1:   # one NCCL unique id per communicator: never reuse the id of another group
        uid = sh.exchange_unique_id(rank, device=dev)
    g = sh.ShardGroup(ix, world, rank, uid)
    peaks = json.loads((ROOT / "MEASURED_PEAKS.json").read_text()) if (ROOT / "MEASURED_PEAKS.json").exists() else {}
    tf_peak = float(peaks.get("bf16_tflops", 1590.0))
    steps = args.steps
    qsets = step_sets(steps + args.warmup,          # every rank answers the SAME queries
                      lambda s: ix.generate_queries(SEED, B, first_query=30_000_000 + s * B, n_centroids=N_CENTROIDS,
                                                    sigma=SIGMA, kind=KIND))
    params = hx.SearchParams.strict(k)
    d_q = map_sets(qsets, lambda q: torch.from_numpy(q).to(dev))
    o_ids = torch.zeros((B, k), dtype=torch.int64, device=dev)
    o_sc = torch.zeros((B, k), dtype=torch.float32, device=dev)
    o_cnt = torch.zeros((B,), dtype=torch.int32, device=dev)

    def step_device(s):
        g.search_device(sh.DENSE, d_q[s].data_ptr(), B, params, k, o_ids.data_ptr(), o_sc.data_ptr(), o_cnt.data_ptr(), stream)

    ms_total = _timed_device(torch, dev, steps, args.warmup, step_device)
    import torch.distributed as dist
    t = torch.tensor([ms_total], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total = float(t.item())
    dev_ids = o_ids.cpu().numpy().view(np.uint64).copy()
    # e2e: host buffers through hx_search_sharded (H2D queries, D2H merged results, one stream sync)
    h_q = map_sets(qsets, lambda q: torch.from_numpy(q).pin_memory().numpy())
    for s in range(args.warmup):
        g.search(sh.DENSE, h_q[s], params, k)
    if world > 1:
        dist.barrier()
    kms = lms = cms = 0.0
    t0 = time.perf_counter()
    for s in range(steps):
        e_ids, e_sc, e_cnt = g.search(sh.DENSE, h_q[args.warmup + s], params, k)
        a, b = g.last_ms()
        lms += a
        cms += b
        kms += ix.last_kernel_ms()[0]
    wall = time.perf_counter() - t0
    tw = torch.tensor([wall], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tw, op=dist.ReduceOp.MAX)
    wall = float(tw.item())
    same = bool(e_ids.tolist() == dev_ids.tolist())
    ldb = (dim + 63) // 64 * 64
    flop = 2.0 * B * rows * ldb
    kernel_ms = kms / steps
    # recall of the merged answer vs the exact scan of every shard merged the same way
    rq = min(64, B)
    last = qsets[args.warmup + steps - 1]
    gi, gs, gc = exact_topk_device_full(hx, torch, ix, last[:rq], rows, lo, k)
    if world > 1:
        lay = sh.block_layout(rq, k)
        blk = np.zeros(lay["bytes"], dtype=np.uint8)
        bi, bs, bc = sh.block_views(blk, rq, k)
        bi[:], bs[:], bc[:] = gi, gs, gc.astype(np.uint32)
        allb = torch.zeros((world, lay["bytes"]), dtype=torch.uint8, device=dev)
        dist.all_gather_into_tensor(allb.view(-1), torch.from_numpy(blk).to(dev))
        truth = sh.merge_blocks_reference([allb[r].cpu().numpy() for r in range(world)], rq, k, k)[0]
    else:
        truth = gi
    rec = recall_at_k(dev_ids[:rq], truth)
    out = {"metric": "queries/sec, exhaustive top-10 through the tensor cores (config C4 shape)",
           "value": round(steps * B / (ms_total / 1e3), 1), "unit": "queries/s", "n_gpus": world, "steps": steps,
           "ms_per_step": round(ms_total / steps, 3), "scaling": "weak (rows per GPU fixed; 8 GPUs = C4's 10M rows)",
           "dtype": "bf16 (fp32 accumulate in TMEM) + f32 exact re-rank", "recall_at_10_vs_exact_scan": round(rec, 4),
           "config": {"workload": f"C4 shard shape: {B} queries x {rows} rows per GPU x d={dim} (total {rows * world} rows on "
                                  f"{world} GPU(s)), k={k}", "setup": {"generate_s": round(gen_s, 2)}},
           "e2e": {"value": round(steps * B / wall, 1), "unit": "queries/s", "ms_per_step": round(wall / steps * 1e3, 3),
                   "h2d_bytes_per_step": B * dim * 4, "d2h_bytes_per_step": B * (k * 12 + 4),
                   "api": "hx_search_sharded(HX_SHARD_DENSE) (C ABI, pinned host buffers, blocking)",
                   "identical_to_device_path": same},
           "step_breakdown_ms": {"local_search": round(lms / steps, 3), "all_gather_and_merge": round(cms / steps, 3),
                                 "k_dense_scores": round(kernel_ms, 4)},
           "collective": (f"1 x ncclAllGather of {sh.block_layout(B, k)['bytes']} B per rank per step (issued by "
                          f"libhelix_b200 through dlopen'ed NCCL) + merge kernel") if world > 1 else "none (single shard)",
           "roofline": {"bound": "tensor", "kernel": "k_dense_scores", "achieved": round(flop / (kernel_ms * 1e-3) / 1e12, 1) if kernel_ms else None,
                        "peak": tf_peak, "unit": "TFLOP/s", "frac": round(flop / (kernel_ms * 1e-3) / 1e12 / tf_peak, 4) if kernel_ms else None,
                        "traffic": ncu_traffic("k_dense_scores", {"queries": B, "rows": rows, "dim": dim}),
                        "flop_per_launch_per_gpu": flop, "kernel_ms_per_launch": round(kernel_ms, 4),
                        "peak_source": "MEASURED_PEAKS.json bf16_tflops (burst); per GPU"},
           "gpu_launches": steps * 8}
    if world == 1 and rank == 0 and not args.no_cpu:
        # the oracle's exact scan (search_exact = restricted_exact_scan over every id) on a bounded sample: parity + CPU rate
        from oracle import hxo
        om = hxo.COSINE if args.metric == "cosine" else hxo.EUCLIDEAN
        ora = hxo.Index(om, dim)
        for a0 in range(0, rows, 65536):
            ids_, rows_ = ix.download_vectors(a0, min(65536, rows - a0))
            ora.put_vectors(ids_, rows_)
        ora.set_entry(lo, 0)
        cores = available_cores()
        ns = 2 * cores
        t0 = time.perf_counter()
        ci, cs, cc, _ = ora.search_exact_batch(last[:ns], k, threads=cores)
        secs = time.perf_counter() - t0
        out["cpu_baseline"] = {"value": round(ns / secs, 2), "unit": "queries/s", "cores": cores, "kind": "port",
                               "sample": f"{ns} queries of the last step, exact scan of all {rows} rows (oracle search_exact)",
                               "bit_exact_vs_device": bool(ci.tolist() == dev_ids[:ns].tolist() and
                                                           cs.tobytes() == o_sc.cpu().numpy()[:ns].tobytes())}
    g.close()
    ix.close()
    return out


def measure_d1536(hx, torch, args, local_rank, dev, stream):
    """The reference's own million-row traversal fixture shape (index_lifecycle_scale.rs:1407-1430: d=1536, Euclidean,
    m=16, m0=32, ef_construction=200) on synthetic vectors of that shape: HNSW top-10 + its four prefilter ranges."""
    import argparse as _ap
    a2 = _ap.Namespace(**vars(args))
    a2.dim, a2.metric, a2.n = 1536, "euclidean", args.d1536_rows
    n, dim, k = a2.n, a2.dim, K
    Q = 16384
    steps = args.steps
    ix, setup = build_index(hx, a2, local_rank, 0, n)
    hbm_peak, peak_src = measured_peaks()
    qsets = step_sets(steps + args.warmup, lambda s: ix.generate_queries(SEED, Q, first_query=40_000_000 + s * Q,
                                                                         n_centroids=N_CENTROIDS, sigma=SIGMA, kind=KIND))
    params = hx.SearchParams.strict(k, EF)
    d_q = map_sets(qsets, lambda q: torch.from_numpy(q).to(dev))
    o_ids = torch.zeros((Q, k), dtype=torch.int64, device=dev)
    o_sc = torch.zeros((Q, k), dtype=torch.float32, device=dev)
    o_cnt = torch.zeros((Q,), dtype=torch.int32, device=dev)

    def step_device(s):
        ix.search_device(d_q[s].data_ptr(), Q, params, o_ids.data_ptr(), o_sc.data_ptr(), o_cnt.data_ptr(), stream)

    rq = 256
    truth = exact_topk_device(hx, torch, ix, qsets[0][:rq], n, 0, k)
    step_device(0)
    torch.cuda.synchronize(dev)
    first_ids = o_ids.cpu().numpy().view(np.uint64).copy()
    first_sc = o_sc.cpu().numpy().copy()
    recall = recall_at_k(first_ids[:rq], truth)
    ix.last_kernel_ms()
    for s in range(args.warmup):
        step_device(s)
    torch.cuda.synchronize(dev)
    ix.last_kernel_ms()
    ms_total = _timed_device(torch, dev, steps, 0, lambda s: step_device(args.warmup + s))
    kms, kl = ix.last_kernel_ms()
    pst = hx.SearchParams.strict(k, EF)
    pst.collect_stats = True
    st = hx.SearchStats()
    ix.search_device(d_q[0].data_ptr(), Q, pst, o_ids.data_ptr(), o_sc.data_ptr(), o_cnt.data_ptr(), stream, st)
    ix.last_kernel_ms()
    kernel_ms = kms / max(kl, 1)
    achieved = st.algorithmic_bytes / (kernel_ms * 1e-3) / 1e9 if kernel_ms else 0.0
    flags, fstatus = ix.device_flags(stream)
    # e2e: hx_search through the C ABI with pinned host buffers (the same call as the C2 line's e2e)
    import ctypes as C
    L = hx.load_library()
    cp = params._c()
    h_q = map_sets(qsets[args.warmup:], lambda q: torch.from_numpy(q).pin_memory())
    h_ids = torch.zeros((Q, k), dtype=torch.int64).pin_memory()
    h_sc = torch.zeros((Q, k), dtype=torch.float32).pin_memory()
    h_cnt = torch.zeros((Q,), dtype=torch.int32).pin_memory()

    def step_host(s):
        rc = L.hx_search(ix.h, C.cast(h_q[s].data_ptr(), C.POINTER(C.c_float)), Q, C.byref(cp),
                         C.cast(h_ids.data_ptr(), C.POINTER(C.c_uint64)), C.cast(h_sc.data_ptr(), C.POINTER(C.c_float)),
                         C.cast(h_cnt.data_ptr(), C.POINTER(C.c_uint32)), None)
        if rc != 0:
            raise RuntimeError(f"hx_search failed: {L.hx_last_error().decode()}")

    step_host(0)
    t0 = time.perf_counter()
    for s in range(steps):
        step_host(s)
    e2e = steps * Q / (time.perf_counter() - t0)
    out = {"metric": "queries/sec @ recall@10, 1M x 1536 Euclidean HNSW top-10 (the reference's traversal fixture shape)",
           "value": round(steps * Q / (ms_total / 1e3), 1), "unit": "queries/s", "steps": steps,
           "ms_per_step": round(ms_total / steps, 3), "recall_at_10": round(recall, 4), "dtype": "f32",
           "config": {"workload": f"{n}x{dim} f32 euclidean HNSW top-10 (m=16, m0=32, ef_construction=200, ef={EF}), {Q} "
                                  f"independent single-query traversals per step", "setup": setup},
           "e2e": {"value": round(e2e, 1), "unit": "queries/s", "h2d_bytes_per_step": Q * dim * 4,
                   "d2h_bytes_per_step": Q * (k * 12 + 4) + Q * 8 + 4, "api": "hx_search (C ABI, pinned host buffers, blocking)"},
           "roofline": {"bound": "hbm", "kernel": "k_hnsw_search_ring", "achieved": round(achieved, 1), "peak": hbm_peak,
                        "unit": "GB/s", "frac": round(achieved / hbm_peak, 4), "traffic": None, "peak_source": peak_src,
                        "algorithmic_bytes_per_launch": int(st.algorithmic_bytes), "kernel_ms_per_launch": round(kernel_ms, 4),
                        "distance_computations_per_query": round(st.distance_computations / Q, 1)},
           "device_flags": flags}
    if not args.no_cpu:
        from oracle import hxo
        t0 = time.perf_counter()
        ora = oracle_from_device(hxo, ix, a2)
        mirror_s = time.perf_counter() - t0
        cores = available_cores()
        ns = 1024
        ci, cs, cc, cst, secs = ora.search_batch(qsets[0][:ns], k, EF, threads=cores)
        out["cpu_baseline"] = {"value": round(ns / secs, 1), "unit": "queries/s", "cores": cores, "kind": "port",
                               "sample": f"{ns} queries of the first step, one query per thread, identical graph and vectors",
                               "ids_identical_to_device": bool(ci.tolist() == first_ids[:ns].tolist()),
                               "scores_identical_to_device": bool(cs.tobytes() == first_sc[:ns].tobytes()),
                               "mirror_s": round(mirror_s, 1)}
        pf = measure_prefilter(hx, torch, ix, a2, dev, stream, n, dim, ora=ora)
        out["prefilter_reference_shapes"] = pf["reference_shapes"]
        out["prefilter_label_sets"] = {"value": pf["value"], "roofline_frac": pf["roofline"]["frac"],
                                       "bit_exact_vs_oracle": pf.get("cpu_baseline", {}).get("bit_exact_vs_device")}
        del ora
    ix.close()
    return out


# ------------------------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist

    import helix_db_b200 as hx

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    stream = torch.cuda.current_stream(dev).cuda_stream
    n, dim, Q, k = args.n, args.dim, args.queries_per_step, K
    hbm_peak, peak_src = measured_peaks()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # ---- setup (untimed): corpus on the device, graph built on the device ---------------------------------------
    ix, setup = build_index(hx, args, local_rank, 0, n)
    n_sets = args.steps + args.warmup
    # distinct queries every rank and in consecutive steps (nothing can be answered from a previous step's cache lines)
    qsets = step_sets(n_sets, lambda s: ix.generate_queries(SEED, Q, first_query=(rank * n_sets + s) * Q,
                                                            n_centroids=N_CENTROIDS, sigma=SIGMA, kind=KIND))
    params = hx.SearchParams.strict(k, EF)
    d_q = map_sets(qsets, lambda q: torch.from_numpy(q).to(dev))
    o_ids = torch.zeros((Q, k), dtype=torch.int64, device=dev)
    o_sc = torch.zeros((Q, k), dtype=torch.float32, device=dev)
    o_cnt = torch.zeros((Q,), dtype=torch.int32, device=dev)

    def step_device(s):
        ix.search_device(d_q[s].data_ptr(), Q, params, o_ids.data_ptr(), o_sc.data_ptr(), o_cnt.data_ptr(), stream)

    # recall@10 on the first query set vs the exact scan
    rq = min(args.recall_queries, Q)
    truth = exact_topk_device(hx, torch, ix, qsets[0][:rq], n, 0, k)
    step_device(0)
    torch.cuda.synchronize(dev)
    strict_ids0 = o_ids.cpu().numpy().view(np.uint64).copy()     # the device's strict answer for query set 0 (parity check)
    strict_sc0 = o_sc.cpu().numpy().copy()
    strict_cnt0 = o_cnt.cpu().numpy().copy()
    recall = recall_at_k(strict_ids0[:rq], truth)

    # ---- value: W warm-up steps, then exactly K timed steps, barrier + synchronize on both sides ----------------------
    for s in range(args.warmup):
        step_device(s)
    barrier()
    ix.last_kernel_ms()                       # drop warm-up launches from the kernel-time accumulator
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for s in range(args.steps):
        step_device(args.warmup + s)
    e1.record()
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    last_step = None
    if args.dump_outputs and rank == 0:       # the last timed step's answer, copied after the timed region closed
        last_step = (o_ids.cpu().numpy().view(np.uint64).copy(), o_sc.cpu().numpy().copy(), o_cnt.cpu().numpy().copy())
    ms_total = e0.elapsed_time(e1)
    kernel_ms_total, kernel_launches = ix.last_kernel_ms()
    dev_flags, dev_flag_status = ix.device_flags(stream)   # error flags ORed over the timed launches (ADVICE r1): must be 0
    if dev_flags != 0:
        raise RuntimeError(f"device error flags {dev_flags:#x} raised inside the timed region (status {dev_flag_status})")
    t = torch.tensor([ms_total], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total = float(t.item())
    value = world * args.steps * Q / (ms_total / 1e3)

    # algorithmic bytes per launch: replay the timed query sets with the reference's counters switched on (untimed)
    st_sum = dict(expansion_steps=0, distance_computations=0, neighbors_examined=0, algorithmic_bytes=0)
    params_st = hx.SearchParams.strict(k, EF)
    params_st.collect_stats = True
    for s in range(args.steps):
        st = hx.SearchStats()
        ix.search_device(d_q[args.warmup + s].data_ptr(), Q, params_st, o_ids.data_ptr(), o_sc.data_ptr(),
                         o_cnt.data_ptr(), stream, st)
        for f in st_sum:
            st_sum[f] += int(getattr(st, f))
    ix.last_kernel_ms()
    bytes_per_launch = st_sum["algorithmic_bytes"] / args.steps
    kernel_ms = kernel_ms_total / max(kernel_launches, 1)
    achieved = bytes_per_launch / (kernel_ms * 1e-3) / 1e9 if kernel_ms > 0 else 0.0

    # ---- e2e: reference-facing C-ABI call with host (pinned) buffers -------------------------------------------------
    h_q = map_sets(qsets, lambda q: torch.from_numpy(q).pin_memory())
    h_ids = torch.zeros((Q, k), dtype=torch.int64).pin_memory()
    h_sc = torch.zeros((Q, k), dtype=torch.float32).pin_memory()
    h_cnt = torch.zeros((Q,), dtype=torch.int32).pin_memory()
    import ctypes as C
    L = hx.load_library()
    cp = params._c()

    def step_host(s):
        rc = L.hx_search(ix.h, C.cast(h_q[s].data_ptr(), C.POINTER(C.c_float)), Q, C.byref(cp),
                         C.cast(h_ids.data_ptr(), C.POINTER(C.c_uint64)), C.cast(h_sc.data_ptr(), C.POINTER(C.c_float)),
                         C.cast(h_cnt.data_ptr(), C.POINTER(C.c_uint32)), None)
        if rc != 0:
            raise RuntimeError(f"hx_search failed: {L.hx_last_error().decode()}")

    for s in range(args.warmup):
        step_host(s)
    barrier()
    t0 = time.perf_counter()
    for s in range(args.steps):
        step_host(args.warmup + s)
    torch.cuda.synchronize(dev)
    t1 = time.perf_counter()
    te = torch.tensor([t1 - t0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_value = world * args.steps * Q / float(te.item())

    # ---- batch-1 single-stream latency (one query per call, sequential) ------------------------------------------------
    nb1 = 200
    for i in range(20):
        ix.search_device(d_q[0][i:i + 1].data_ptr(), 1, params, o_ids.data_ptr(), o_sc.data_ptr(), o_cnt.data_ptr(), stream)
    torch.cuda.synchronize(dev)
    b0, b1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    b0.record()
    for i in range(nb1):
        ix.search_device(d_q[0][i:i + 1].data_ptr(), 1, params, o_ids.data_ptr(), o_sc.data_ptr(), o_cnt.data_ptr(), stream)
    b1.record()
    torch.cuda.synchronize(dev)
    batch1_us = b0.elapsed_time(b1) / nb1 * 1e3
    ix.last_kernel_ms()

    # ---- production-default mode: SearchParams::new = SimHashMode::Adaptive (SimHash gate + sampling policy) ----------------
    # No network => no way to obtain the reference's StdRng(42) hyperplanes; a Gaussian table from numpy's seed 42 stands in
    # (the fingerprints are data to the kernel either way).  Host buffers through hx_search_ex, fingerprints of the queries
    # projected on the device inside the timed region.
    default_mode = None
    default_planes = None
    d_ids_first = None
    if not args.no_default_mode and args.metric == "cosine":
        planes = np.random.default_rng(42).standard_normal((64, dim)).astype(np.float32)
        ix._bench_planes = planes
        ix.set_simhash_planes(planes)
        t0 = time.perf_counter()
        ix.compute_simhash()
        simhash_s = time.perf_counter() - t0
        pnew = hx.SearchParams.new(k)
        pnew.collect_stats = True
        st_d, ps_d = hx.SearchStats(), hx.PolicyStats()
        d_ids, _, d_cnt = ix.search_ex(qsets[0], pnew, stats=st_d, policy_stats=ps_d)
        d_ids_first = d_ids
        d_recall = recall_at_k(d_ids[:rq], truth)
        pnew.collect_stats = False
        cpn, poln = pnew._c(), pnew._policy()

        def step_default(s):
            rc = L.hx_search_ex(ix.h, C.cast(h_q[s].data_ptr(), C.POINTER(C.c_float)), Q, C.byref(cpn), C.byref(poln), None,
                                C.cast(h_ids.data_ptr(), C.POINTER(C.c_uint64)), C.cast(h_sc.data_ptr(), C.POINTER(C.c_float)),
                                C.cast(h_cnt.data_ptr(), C.POINTER(C.c_uint32)), None, None)
            if rc != 0:
                raise RuntimeError(f"hx_search_ex failed: {L.hx_last_error().decode()}")

        for s in range(args.warmup):
            step_default(s)
        barrier()
        kms_sum = 0.0
        t0 = time.perf_counter()
        for s in range(args.steps):
            step_default(args.warmup + s)
            kms_sum += ix.last_kernel_ms()[0]
        td = time.perf_counter() - t0
        # one query per call (the reference's usage: one query per tokio task)
        for i in range(10):
            ix.search_ex(qsets[0][i:i + 1], pnew)
        t0 = time.perf_counter()
        for i in range(100):
            ix.search_ex(qsets[0][i:i + 1], pnew)
        single_us = (time.perf_counter() - t0) / 100 * 1e6
        # recall of the production default against the beam width (the reference ships ef = max(k, 100); its own recall gate
        # for this mode is 0.92, tests/production_support/vector/search.rs): where does 0.95 sit?
        ef_study = []
        for ef_d in (100, 150, 200, 300):
            pe = hx.SearchParams.new(k).with_ef(ef_d)
            e_ids, _, _ = ix.search_ex(qsets[0][:rq], pe)
            ef_study.append({"ef": ef_d, "recall_at_10": round(recall_at_k(e_ids, truth), 4)})
        default_mode = {
            "params": "SearchParams::new(10): ef=100, SimHashMode::Adaptive, threshold 43, sampling 0.8, failure 0.1",
            "recall_vs_ef": ef_study,
            "e2e_qps": round(args.steps * Q / td, 1), "kernel": "k_hnsw_search_policy",
            "kernel_ms_per_launch": round(kms_sum / args.steps, 4), "kernel_qps": round(args.steps * Q / (kms_sum / 1e3), 1),
            "recall_at_10": round(d_recall, 4),
            "distance_computations_per_query": round(st_d.distance_computations / Q, 1),
            "simhash_examined_per_query": round(ps_d.simhash_examined / Q, 1),
            "simhash_filtered_per_query": round(ps_d.simhash_filtered / Q, 1),
            "rng_draws_per_query": round(ps_d.rng_draws / Q, 2),
            "alg_GBps": round(st_d.algorithmic_bytes / (kms_sum / args.steps * 1e-3) / 1e9, 1) if kms_sum else None,
            "simhash_projection_s": round(simhash_s, 3),
            "single_query_us": round(single_us, 1),
            "note": "hyperplanes: numpy default_rng(42) Gaussian stand-in for the reference's StdRng(42) table",
        }
        default_planes = planes

    # ---- sharded path (north_star): id-range shards of the SAME corpus behind the C ABI ------------------------------------
    # hx_search_sharded_device: local search writes into the send block -> ONE ncclAllGather issued by the library -> merge.
    sharded = None
    uid = None
    if world > 1:
        from helix_db_b200 import sharding as sh
        uid = sh.exchange_unique_id(rank, device=dev)
    if world > 1 and not args.no_sharded:
        lo, hi = rank * n // world, (rank + 1) * n // world
        sx, s_setup = build_index(hx, args, local_rank, lo, hi - lo)
        grp = sh.ShardGroup(sx, world, rank, uid)
        # every rank searches the SAME queries (rank 0's sets) against its shard
        sq = step_sets(n_sets, lambda s: ix.generate_queries(SEED, Q, first_query=s * Q, n_centroids=N_CENTROIDS, sigma=SIGMA,
                                                             kind=KIND))
        d_sq = map_sets(sq, lambda q: torch.from_numpy(q).to(dev))
        truth_s = exact_topk_device(hx, torch, ix, sq[0][:rq], n, 0, k)
        step_device(0)   # the unsharded index on the same queries: the recall the shards have to match
        ix.search_device(d_sq[0].data_ptr(), Q, params, o_ids.data_ptr(), o_sc.data_ptr(), o_cnt.data_ptr(), stream)
        torch.cuda.synchronize(dev)
        target = recall_at_k(o_ids[:rq].cpu().numpy().view(np.uint64), truth_s)

        def run_sharded(s, p_local):
            grp.search_device(sh.HNSW, d_sq[s].data_ptr(), Q, p_local, k, o_ids.data_ptr(), o_sc.data_ptr(), o_cnt.data_ptr(), stream)

        # iso-recall tuning of the per-shard beam: a shard is 1/world of the corpus, so the unsharded ef is over-provisioned
        tuning, chosen = [], None
        for ef_s in (10, 12, 16, 20, 24, 32, 40, 48, 56, 64, 72, 80, 90, EF):
            p_loc = hx.SearchParams.strict(k, ef_s)
            run_sharded(0, p_loc)
            torch.cuda.synchronize(dev)
            r = recall_at_k(o_ids[:rq].cpu().numpy().view(np.uint64), truth_s)
            tuning.append({"ef_per_shard": ef_s, "recall_at_10": round(r, 4)})
            if chosen is None and r >= target:
                chosen = ef_s
                break
        chosen = chosen or EF
        p_loc = hx.SearchParams.strict(k, chosen)
        run_sharded(0, p_loc)
        torch.cuda.synchronize(dev)
        s_recall = recall_at_k(o_ids[:rq].cpu().numpy().view(np.uint64), truth_s)
        for s in range(args.warmup):
            run_sharded(s, p_loc)
        barrier()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record()
        for s in range(args.steps):
            run_sharded(args.warmup + s, p_loc)
        g1.record()
        barrier()
        ts = torch.tensor([g0.elapsed_time(g1)], dtype=torch.float64, device=dev)
        dist.all_reduce(ts, op=dist.ReduceOp.MAX)
        sflags, _ = sx.device_flags(stream)
        # the same per-shard parameters at the unsharded beam width, for reference
        p_full = hx.SearchParams.strict(k, EF)
        for s in range(2):
            run_sharded(s, p_full)
        barrier()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record()
        for s in range(args.steps):
            run_sharded(args.warmup + s, p_full)
        f1.record()
        barrier()
        tf_ = torch.tensor([f0.elapsed_time(f1)], dtype=torch.float64, device=dev)
        dist.all_reduce(tf_, op=dist.ReduceOp.MAX)
        blk = sh.block_layout(Q, k)["bytes"]
        sharded = {"value": round(args.steps * Q / (float(ts.item()) / 1e3), 1), "unit": "queries/s",
                   "recall_at_10": round(s_recall, 4), "unsharded_recall_at_10_same_queries": round(target, 4),
                   "ef_per_shard": chosen, "k_per_shard": k, "iso_recall_tuning": tuning,
                   "value_at_unsharded_ef": round(args.steps * Q / (float(tf_.item()) / 1e3), 1),
                   "shard_vectors": hi - lo,
                   "api": "hx_search_sharded_device (C ABI): local search into the send block, ncclAllGather, merge kernel",
                   "collective": f"1 x ncclAllGather of {blk} B per rank per step (issued by libhelix_b200 via dlopen'ed NCCL)",
                   "ms_per_step": round(float(ts.item()) / args.steps, 3), "shard_build_s": s_setup["build_s"],
                   "device_flags": sflags}
        grp.close()
        sx.close()

    # ---- the other BASELINE configs as sub-results of the same line --------------------------------------------------------------
    dense_c4 = None
    if not args.no_subresults:
        dense_c4 = measure_dense(hx, torch, args, world, rank, local_rank, dev, stream, uid)

    # ---- CPU baseline: the oracle on the box's host cores, same graph, bounded sample (rank 0, N = 1 only) -------------------
    cpu = None
    ora = None
    parity = None
    if rank == 0 and world == 1 and not args.no_cpu:
        cpu, ora = cpu_baseline(args, ix, qsets[0], truth[:rq] if rq else None,
                                default_planes if default_mode is not None else None)
        if default_mode is not None and "default_mode_qps" in cpu:
            default_mode["cpu_port_qps"] = cpu.pop("default_mode_qps")
            default_mode["cpu_port_recall_at_10"] = cpu.pop("default_mode_recall")
            pi = cpu.pop("_default_ids")
            cpu.pop("default_mode_sample", None)
            default_mode["cpu_port_identical_to_device"] = bool(d_ids_first is not None and
                                                                pi.tolist() == d_ids_first[:len(pi)].tolist())
        # id-level parity on the headline config (VERDICT r1 weak #1): every CPU-sampled query, ids + score bytes + counts
        ci, cs, cc = cpu.pop("_ids"), cpu.pop("_scores"), cpu.pop("_counts")
        m = len(ci)
        parity = {"queries_checked": int(m),
                  "ids_identical_to_device": bool(ci.tolist() == strict_ids0[:m].tolist() and cc.tolist() == strict_cnt0[:m].tolist()),
                  "scores_identical_to_device": bool(cs.tobytes() == strict_sc0[:m].tobytes()),
                  "oracle": "C restatement of search.rs / restricted.rs traversing the identical graph and vectors"}
        # and the recall ground truth itself: the device's exact scan against the oracle's exact scan
        ng = min(2 * available_cores(), rq)
        ei, es, ec, _ = ora.search_exact_batch(qsets[0][:ng], k, threads=available_cores())
        parity["ground_truth_vs_oracle_exact_scan"] = {"queries": int(ng), "identical": bool(ei.tolist() == truth[:ng].tolist())}
        cpu["parity"] = parity

    prefilter = callers_res = d1536 = None
    if rank == 0 and world == 1 and not args.no_subresults:
        prefilter = measure_prefilter(hx, torch, ix, args, dev, stream, n, dim, ora=ora)
        callers_res = measure_callers(hx, ix, qsets[0][:8192], k, EF, args.callers_seconds)
    del ora

    hnsw_kernel = "k_hnsw_search_ring"
    line = None
    if rank == 0:
        line = {
            "metric": "queries/sec @ recall@10, DBpedia-1M d=768 top-10, 1/2/4/8 B200 vs CPU ref",
            "value": round(value, 1), "unit": "queries/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": round(ms_total / args.steps, 4), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "recall_at_10": round(recall, 4),
            "config": c2_config(args, world),
            "setup": setup,                                    # timings of the untimed setup: outside `config`, which both arms share verbatim
            "e2e": {"value": round(e2e_value, 1), "unit": "queries/s", "h2d_bytes_per_step": Q * dim * 4,
                    "d2h_bytes_per_step": Q * (k * 12 + 4) + Q * 8 + 4,
                    "api": "hx_search (C ABI, pinned host buffers, blocking)"},
            "gpu_launches": args.steps,
            "launches_per_step": {hnsw_kernel: 1},
            "roofline": {"bound": "hbm", "kernel": hnsw_kernel, "achieved": round(achieved, 1), "peak": hbm_peak,
                         "unit": "GB/s", "frac": round(achieved / hbm_peak, 4), "traffic": ncu_traffic("k_hnsw_search", {"queries": Q, "rows": n, "dim": dim, "ef": EF}),
                         "peak_source": peak_src, "algorithmic_bytes_per_launch": int(bytes_per_launch),
                         "kernel_ms_per_launch": round(kernel_ms, 4),
                         "expansions_per_query": round(st_sum["expansion_steps"] / (args.steps * Q), 1),
                         "distance_computations_per_query": round(st_sum["distance_computations"] / (args.steps * Q), 1)},
            "single_stream_batch1": {"latency_us": round(batch1_us, 1), "qps": round(1e6 / batch1_us, 1),
                                     "note": "one query per hx_search_device call, calls issued back to back"},
            "device_flags_in_timed_region": dev_flags,
            "clocks": clocks,
        }
        if cpu is not None:
            line["cpu_baseline"] = cpu
        if parity is not None:
            line["parity"] = parity
        if sharded is not None:
            line["sharded"] = sharded
        if default_mode is not None:
            line["default_mode"] = default_mode
        if callers_res is not None:
            line["concurrent_callers"] = callers_res
        if prefilter is not None:
            line["prefilter"] = prefilter
        if dense_c4 is not None:
            line["dense_c4"] = dense_c4
    ix.close()
    if rank == 0 and world == 1 and not args.no_subresults and not args.no_d1536:
        line["euclid_d1536"] = measure_d1536(hx, torch, args, local_rank, dev, stream)
    if last_step is not None:
        dump_outputs(args.dump_outputs, *last_step)
    if rank == 0:
        print(json.dumps(line), flush=True)
        if parity is not None and not (parity["ids_identical_to_device"] and parity["scores_identical_to_device"]):
            print("PARITY FAILURE: device ids / scores differ from the oracle on the headline config", file=sys.stderr)
            sys.exit(3)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def cpu_baseline(args, ix, queries, truth, planes=None):
    """The oracle (C restatement of the reference, no KV layer => an upper bound on the reference's CPU throughput)."""
    from oracle import hxo

    cores = available_cores()
    t0 = time.perf_counter()
    ora = oracle_from_device(hxo, ix, args)
    mirror_s = time.perf_counter() - t0
    probe = min(256, len(queries))
    _, _, _, _, secs = ora.search_batch(queries[:probe], K, EF, threads=cores)
    qps_probe = probe / max(secs, 1e-9)
    sample = int(max(probe, min(len(queries), qps_probe * args.cpu_seconds)))
    ids, sc, cnt, st, secs = ora.search_batch(queries[:sample], K, EF, threads=cores)
    rec = recall_at_k(ids[:len(truth)], truth) if truth is not None and len(truth) <= sample else None
    _, _, _, _, secs1 = ora.search_batch(queries[:min(sample, 256)], K, EF, threads=1)
    extra = {}
    if planes is not None:   # the production-default mode on the CPU: same fingerprints, same policy
        n = args.n
        ora.put_simhash(np.arange(n, dtype=np.uint64), ix.download_simhash(0, n))
        dq = min(sample, 4096)
        qsim = np.array([hxo.simhash_from_planes(planes, q) for q in queries[:dq]], dtype=np.uint64)
        cfg = hxo.policy_defaults()
        pi, _, pc, psecs = ora.search_policy_batch(queries[:dq], K, EF, cfg, qsim, threads=cores)
        extra["default_mode_qps"] = round(dq / psecs, 1)
        extra["default_mode_recall"] = round(recall_at_k(pi[:len(truth)], truth), 4) if truth is not None and len(truth) <= dq else None
        extra["default_mode_sample"] = dq
        extra["_default_ids"] = pi
    out = {"value": round(sample / secs, 1), "unit": "queries/s", "cores": cores, "kind": "port",
            "sample": f"{sample} queries of the first step's set, one query per thread, {cores} threads, "
                      f"identical graph and vectors",
            "single_thread_qps": round(min(sample, 256) / secs1, 1), "recall_at_10": None if rec is None else round(rec, 4),
            "distance_computations_per_query": round(st["distance_computations"] / sample, 1),
            "mirror_s": round(mirror_s, 1),
            "build_flags": "gcc -O2 -ffp-contract=off, AVX+FMA distance kernels via target attributes (oracle/Makefile); no -march=native: the traversal is DRAM-latency bound",
            "_ids": ids, "_scores": sc, "_counts": cnt}
    out.update(extra)
    return out, ora


# ------------------------------------------------------------------------------------------------------------------
def run_prefilter(args):
    """--workload prefilter: config C3 alone (the default line carries the same object as `prefilter`)."""
    import torch

    import helix_db_b200 as hx

    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    stream = torch.cuda.current_stream(dev).cuda_stream
    n, dim = args.n, args.dim
    # the exact scan needs no graph; the filter-aware walk reported next to the reference's shapes does: build it
    ix, _setup = build_index(hx, args, local_rank, 0, n)
    ora = None
    if not args.no_cpu:
        from oracle import hxo
        ora = oracle_from_device(hxo, ix, args)
    sampler = ClockSampler(local_rank)
    sampler.start()
    line = measure_prefilter(hx, torch, ix, args, dev, stream, n, dim, ora=ora)
    line.update({"n_gpus": 1, "warmup": args.warmup, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                 "data": "synthetic", "clocks": sampler.stop()})
    print(json.dumps(line), flush=True)
    ix.close()


# ------------------------------------------------------------------------------------------------------------------
def run_dense(args):
    """--workload dense: the C4 shape alone (the default line carries the same object as `dense_c4`)."""
    import torch

    import helix_db_b200 as hx

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    uid = None
    if world > 1:
        import torch.distributed as dist
        from helix_db_b200 import sharding as sh
        dist.init_process_group("nccl", device_id=dev)
        uid = sh.exchange_unique_id(rank, device=dev)
    stream = torch.cuda.current_stream(dev).cuda_stream
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    line = measure_dense(hx, torch, args, world, rank, local_rank, dev, stream, uid)
    if rank == 0:
        line.update({"warmup": args.warmup, "higher_is_better": True, "vs_baseline": None, "data": "synthetic",
                     "clocks": sampler.stop()})
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------------------------
def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path (oracle port; the Rust reference cannot be built
    here: no rustc/cargo, un-vendored SlateDB fork) on all host cores, same config, metric and unit."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch

    import helix_db_b200 as hx
    from oracle import hxo

    if not torch.cuda.is_available():
        print(json.dumps({"impl": "reference", "unavailable": "the graph of config C2 is built on the device "
                          "(hours on the CPU); no GPU visible in this process"}))
        return
    n, dim, Q = args.n, args.dim, args.queries_per_step
    ix, setup = build_index(hx, args, 0, 0, n)
    cores = available_cores()
    queries = ix.generate_queries(SEED, Q, first_query=0, n_centroids=N_CENTROIDS, sigma=SIGMA, kind=KIND)
    rq = min(args.recall_queries, Q)
    truth = exact_topk_device(hx, torch, ix, queries[:rq], n, 0, K)
    ora = oracle_from_device(hxo, ix, args)
    ix.close()
    # a step = a bounded sample of the workload sized so that the whole run ends within a few minutes
    _, _, _, _, secs = ora.search_batch(queries[:256], K, EF, threads=cores)
    per_step = int(max(256, min(Q, (256 / max(secs, 1e-9)) * (args.cpu_seconds / max(args.steps, 1)))))
    for _ in range(args.warmup):
        ora.search_batch(queries[:per_step], K, EF, threads=cores)
    total = 0.0
    last = None
    for _ in range(args.steps):
        last = ora.search_batch(queries[:per_step], K, EF, threads=cores)
        total += last[4]
    value = args.steps * per_step / total
    rec = recall_at_k(last[0][:min(rq, per_step)], truth[:min(rq, per_step)])
    line = {
        "impl": "reference",
        "metric": "queries/sec @ recall@10, DBpedia-1M d=768 top-10, 1/2/4/8 B200 vs CPU ref",
        "value": round(value, 1), "unit": "queries/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": round(total / args.steps * 1e3, 3), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic", "recall_at_10": round(rec, 4),
        "config": c2_config(args, args.gpus),              # the config of OUR arm at this N, verbatim (rank 0 alone runs the CPU arm)
        "setup": setup,
        "sample": f"each step = {per_step} of the workload's {Q} queries per step (a bounded sample: throughput metric), one "
                  f"query per host thread, {cores} threads; the graph both arms traverse is built on the device as untimed setup",
        "cpu_baseline": {"value": round(value, 1), "unit": "queries/s", "cores": cores, "kind": "port",
                         "sample": f"{per_step} queries per step x {args.steps} steps, {cores} threads"},
        "e2e": {"value": round(value, 1), "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    elif a.workload == "prefilter":
        run_prefilter(a)
    elif a.workload == "dense":
        run_dense(a)
    else:
        run_ours(a)
