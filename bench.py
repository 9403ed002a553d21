#!/usr/bin/env python
"""bench.py -- queries/sec of the multi-vector MaxSim scan (BASELINE.json metric) on N GPUs.

    python bench.py --gpus 1 --steps 10 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 \
        --master-port 29500 bench.py --gpus 8 --steps 10 --warmup 3
    python bench.py --impl reference ...      # the reference's CPU arithmetic on the host cores
    python bench.py ... --dump-outputs DIR    # also write the last timed step's results as DIR/*.npy

Workload (default ``c4shard``): BASELINE configs[3] -- 10M chunks x 12 vecs x 1024-d fp32, row-sharded
over 8 GPUs -- run as its per-GPU shard: every rank holds 1.25M chunks (15.36M vectors, 61.4 GB) and
scans them for the same batch of queries; ranks all-gather their per-shard hits over NCCL and merge.
Weak scaling: per-GPU work is fixed, the corpus grows with N (10M chunks at N = 8).

``value`` is in queries/sec over 10M chunks: ``batch / t_step * (chunks_scanned / 10M)`` -- at N = 8
it is literally queries/sec over the 10M-chunk corpus; at smaller N a query that only had to scan a
fraction of 10M chunks counts for that fraction (``queries_per_sec_raw`` is the unnormalised rate).
One "step" = one batch of ``--batch`` queries through adapter-less ``vector_search`` semantics
(top-num_hits vectors -> GROUP BY chunk max -> top-k, _search.py:65-79,143-153).
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
for p in (ROOT, ROOT / "tests"):
    if str(p) not in sys.path:
        sys.path.insert(0, str(p))

TEN_M = 10_000_000
WORKLOADS = {
    # name: chunks per GPU, vecs per chunk, dim, batch, k
    "c4shard": dict(chunks=1_250_000, vecs=12, dim=1024, batch=256, k=100,
                    desc="BASELINE configs[3] per-GPU shard: 1.25M chunks x 12 vecs x 1024-d fp32 per GPU (10M chunks at 8 GPUs)"),
    "c3": dict(chunks=1_000_000, vecs=8, dim=1024, batch=1024, k=100,
               desc="BASELINE configs[2]: 1M chunks x 8 vecs x 1024-d, batch 1024, top-100, query adapter"),
    "c2": dict(chunks=100_000, vecs=8, dim=384, batch=256, k=20,
               desc="BASELINE configs[1]: 100k chunks x 8 vecs x 384-d fp32, batch 256, top-20"),
    "tiny": dict(chunks=20_000, vecs=8, dim=128, batch=64, k=10, desc="debug"),
    "pool": dict(chunks=0, vecs=0, dim=1024, batch=2048, k=0,
                 desc="late-chunking pool (_embed.py:119-140): 2048 segments x 496 token rows x 1024-d fp32 -> per-sentence mean, L2, fp16"),
    "c5": dict(chunks=0, vecs=0, dim=384, batch=1024, k=100,
               desc="BASELINE configs[4]: cross-encoder rerank, MiniLM-L12-H384, 1024 queries x 100 candidates (seeded weights)"),
}


def positive_int(text: str) -> int:
    v = int(text)
    if v < 1:
        raise argparse.ArgumentTypeError(f"must be at least 1, got {v}")
    return v


def parse_args() -> argparse.Namespace:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=positive_int, default=10, help="timed steps")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c4shard", choices=sorted(WORKLOADS))
    ap.add_argument("--batch", type=int, default=0)
    ap.add_argument("--k", type=int, default=0)
    ap.add_argument("--chunks", type=int, default=0, help="chunks per GPU (override)")
    ap.add_argument("--oversample", type=int, default=4)
    ap.add_argument("--exact-maxsim", action="store_true")
    ap.add_argument("--adapter", default="auto", choices=["auto", "on", "off"], help="query adapter apply (on for c3)")
    ap.add_argument("--algo", default="auto")
    ap.add_argument("--sample-stride", type=int, default=0, help="override the sampling stride (0 = library heuristic)")
    ap.add_argument("--storage", default="fp32", choices=["fp32", "fp16"],
                    help="fp16: corpus rounded to float16 and stored as such (lossless layout for RAGLite data)")
    ap.add_argument("--inflight", type=int, default=2, help="batches in flight in the end-to-end loop (1: serial vector_search_batch calls)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-check", action="store_true")
    ap.add_argument("--cpu-sample-chunks", type=int, default=0)
    ap.add_argument("--data", default="gaussian", choices=["gaussian", "clustered"],
                    help="clustered: tight clusters of near-duplicates + low-rank background, float16-rounded (tests/synth.py)")
    ap.add_argument("--check-queries", type=int, default=16, help="queries compared with the oracle after the timed region")
    ap.add_argument("--burst-probe", action="store_true",
                    help="after the timed loop: the same step launched after 250 ms of idle, six times (is the scan slower inside a "
                         "loop of steps than timed alone?)")
    ap.add_argument("--filtered", action="store_true", help="also time metadata-filtered searches (both reference branches)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step returned as DIR/<name>.npy (float32 or "
                         "float64, at most 64 MB in all) so that two builds can be compared on identical seeded inputs")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs records the GPU path; the reference arm times a host-side sample of the workload")
    return args


DUMP_MAX_BYTES = 64 << 20


def dump_outputs(out_dir: str, arrays: dict[str, np.ndarray]) -> None:
    """``out_dir/<name>.npy`` per array: float16/float32 as float32, everything else (float64, integer ids and
    counts, exact below 2**53) as float64."""
    conv = {name: a.astype(np.float32 if a.dtype in (np.float16, np.float32) else np.float64) for name, a in arrays.items()}
    total = sum(a.nbytes for a in conv.values())
    if total > DUMP_MAX_BYTES:
        raise ValueError(f"--dump-outputs: {total} bytes of outputs exceed the {DUMP_MAX_BYTES}-byte limit")
    d = Path(out_dir)
    d.mkdir(parents=True, exist_ok=True)
    for name, a in conv.items():
        np.save(d / f"{name}.npy", a)


def resolve(args: argparse.Namespace) -> dict:
    w = dict(WORKLOADS[args.workload])
    if args.batch:
        w["batch"] = args.batch
    if args.k:
        w["k"] = args.k
    if args.chunks:
        w["chunks"] = args.chunks
    w["name"] = args.workload
    w["num_hits"] = 0 if args.exact_maxsim else round(args.oversample * 2048 / 2048) * max(w["k"], 10)
    return w


# ---- clocks sampler (B200_PROFILING.md "clocks line") ---------------------------------------------
class ClockSampler:
    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
              "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc: subprocess.Popen | None = None
        self.lines: list[str] = []
        self.thread: threading.Thread | None = None

    def start(self) -> None:
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "50",
                 "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None
            return
        def pump() -> None:
            assert self.proc is not None and self.proc.stdout is not None
            for line in self.proc.stdout:
                self.lines.append((time.perf_counter(), line.strip()))
        self.thread = threading.Thread(target=pump, daemon=True)
        self.thread.start()

    def wait_first_sample(self, timeout: float = 5.0) -> None:
        t0 = time.perf_counter()
        while not self.lines and time.perf_counter() - t0 < timeout and self.proc is not None:
            time.sleep(0.05)

    def stop(self, windows: list[tuple[float, float]] | None = None) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, power, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for stamp, line in self.lines:
            if windows and not any(w0 - 0.05 <= stamp <= w1 + 0.15 for w0, w1 in windows):
                continue
            parts = [x.strip() for x in line.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1])); mx.append(float(parts[2])); power.append(float(parts[3]))
            except ValueError:
                continue
            for name, val in zip(names, parts[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


# ---- CPU arm: the reference's arithmetic (oracle port) on the host cores ----------------------------
def cpu_reference_rate(w: dict, sample_chunks: int, reps: int, seed: int = 0, warmup: int = 0) -> dict:
    """Time ``oracle.vector_search.blas_batch_topk`` (sgemm on all host cores -> cosine scaling ->
    top-num_hits / group max / top-k) on a bounded sample of the workload, ``reps`` timed runs after
    ``warmup`` untimed ones, and extrapolate linearly in the number of vectors."""
    from oracle.vector_search import blas_batch_topk  # the ONLY product-side use of the oracle: the CPU baseline
    from synth import make_corpus, make_queries

    # torchrun exports OMP_NUM_THREADS=1; the CPU arm is meant to use every host core it can.
    import contextlib
    want = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        from threadpoolctl import threadpool_info, threadpool_limits
        limiter = threadpool_limits(limits=want)
    except Exception:  # noqa: BLE001
        threadpool_info, limiter = None, contextlib.nullcontext()
    E, _ = make_corpus(sample_chunks, w["vecs"], w["dim"], seed=seed)
    Q = make_queries(E, w["batch"], seed=seed + 1)
    times = []
    with limiter:
        # threads actually used: the BLAS pool after the limit (never more than the cores this process may run on)
        threads = min(want, max([i.get("num_threads", 1) for i in threadpool_info()] + [1])) if threadpool_info else want
        blas_batch_topk(E[: 1024 * w["vecs"]], w["vecs"], Q[:8], min(w["k"], 64), num_hits=w["num_hits"])  # warm BLAS
        for _ in range(warmup):
            blas_batch_topk(E, w["vecs"], Q, w["k"], num_hits=w["num_hits"])
        for _ in range(reps):
            t0 = time.perf_counter()
            blas_batch_topk(E, w["vecs"], Q, w["k"], num_hits=w["num_hits"])
            times.append(time.perf_counter() - t0)
    t = float(np.median(times))
    raw_qps_sample = w["batch"] / t
    return {"t_sample_s": t, "reps": reps, "threads": int(threads), "sample_chunks": sample_chunks,
            "qps_over_10M": raw_qps_sample * sample_chunks / TEN_M}


def run_reference(args: argparse.Namespace, w: dict) -> None:
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    sample = args.cpu_sample_chunks or max(2048, min(w["chunks"], 16_384))
    t0 = time.perf_counter()
    r = cpu_reference_rate(w, sample, reps=args.steps, warmup=args.warmup)   # the median of the timed steps is the per-step figure
    value = r["qps_over_10M"]
    line = {
        "impl": "reference", "metric": "queries/sec multi-vector MaxSim over 10M chunks", "value": value,
        "unit": "queries/s (10M-chunk equivalent)", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": r["t_sample_s"] * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": w["desc"], "batch": w["batch"], "k": w["k"], "num_hits": w["num_hits"],
                   "metric": "cosine", "cpu_sample": f"{sample} chunks x {w['vecs']} vecs x {w['dim']}-d per step, "
                   "extrapolated linearly in vectors to 10M chunks"},
        "cpu_baseline": {"value": value, "unit": "queries/s (10M-chunk equivalent)", "cores": r["threads"],
                         "kind": "port", "sample": f"{sample} chunks ({sample * w['vecs']} vectors) x batch {w['batch']}; "
                         "NumPy sgemm + top-num_hits/group-max/top-k (oracle.vector_search.blas_batch_topk)"},
        "e2e": {"value": value, "unit": "queries/s (10M-chunk equivalent)", "h2d_bytes_per_step": 0,
                "d2h_bytes_per_step": 0},
        "wall_s": time.perf_counter() - t0,
    }
    print(json.dumps(line), flush=True)


# ---- GPU arm -------------------------------------------------------------------------------------------
def build_shard(w: dict, rank: int, device, storage: str = "fp32", data: str = "gaussian"):  # noqa: ANN001, ANN201
    """Synthetic unit-norm corpus shard generated on the device (seeded per rank); float32, or rounded
    to float16 (what RAGLite stores, _embed.py:140) for the fp16 layout.  ``clustered``: tight clusters of
    near-duplicates + low-rank background (tests/synth.py), float16-rounded values in either storage."""
    import torch

    n_rows = w["chunks"] * w["vecs"]
    dtype = torch.float16 if storage == "fp16" else torch.float32
    if data == "clustered":
        from synth_torch import clustered_corpus_torch

        E, _ = clustered_corpus_torch(n_rows, w["dim"], seed=1234 + rank, device=device, dtype=dtype)
        return E
    g = torch.Generator(device=device)
    g.manual_seed(1234 + rank)
    E = torch.empty((n_rows, w["dim"]), dtype=dtype, device=device)
    step = 1 << 20
    for r0 in range(0, n_rows, step):
        r1 = min(n_rows, r0 + step)
        blk = torch.randn((r1 - r0, w["dim"]), generator=g, device=device, dtype=torch.float32)
        blk /= blk.norm(dim=1, keepdim=True)
        E[r0:r1] = blk
    return E


def make_batch_queries(E, w: dict, seed: int):  # noqa: ANN001, ANN201
    """Queries near random rows of rank 0's shard (identical on every rank) + 25% random directions."""
    import torch

    g = torch.Generator(device="cpu")
    g.manual_seed(seed)
    B, d = w["batch"], w["dim"]
    noise = torch.randn((B, d), generator=g)
    noise /= noise.norm(dim=1, keepdim=True)
    rows = torch.randint(0, min(E.shape[0], 1 << 20), (B,), generator=g)
    return noise, rows


def run_rerank(args: argparse.Namespace, w: dict) -> None:
    """configs[4]: data-parallel over queries, one process per GPU, scores all-gathered at the end."""
    import torch
    import torch.distributed as dist

    from raglite_b200._xenc import CrossEncoderEngine, random_minilm_state_dict

    world, rank = int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    n_q, n_c = w["batch"], w["k"]
    rng = np.random.default_rng(0)
    lens = np.clip(rng.normal(200, 60, size=n_q * n_c).astype(int), 32, 512)
    if args.impl == "reference":
        if rank != 0:
            return
        from oracle import rerank as orr     # the CPU arm: float32 transformers forward
        model = orr.seeded_model(seed=0)
        n = 64
        ids = [rng.integers(1000, 30000, size=L).astype(np.int32) for L in lens[:n]]
        types = [np.r_[np.zeros(12, np.int32), np.ones(L - 12, np.int32)] for L in lens[:n]]
        torch.set_num_threads(len(os.sched_getaffinity(0)))
        orr.hf_logits(model, ids[:4], types[:4])     # first call pays thread-pool / allocator start-up
        t0 = time.perf_counter()
        for _ in range(args.steps):
            orr.hf_logits(model, ids, types)
        dt = (time.perf_counter() - t0) / args.steps
        v = n / dt
        print(json.dumps({"impl": "reference", "metric": "cross-encoder pairs/sec", "value": v, "unit": "pairs/s", "n_gpus": args.gpus,
                          "steps": args.steps, "warmup": 0, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "strong",
                          "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": {"workload": w["desc"]},
                          "cpu_baseline": {"value": v, "unit": "pairs/s", "cores": torch.get_num_threads(), "kind": "port",
                                           "sample": f"{n} pairs, transformers BertForSequenceClassification fp32"},
                          "e2e": {"value": v, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}), flush=True)
        return
    sys.stdout.flush(); saved = os.dup(1); os.dup2(2, 1)
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    eng = CrossEncoderEngine(random_minilm_state_dict(0), n_layers=12, hidden=384, n_heads=12, ffn=1536, max_pos=512)
    mine = np.arange(rank, n_q, world)                       # this rank's queries
    sel = np.concatenate([np.arange(q * n_c, (q + 1) * n_c) for q in mine])
    ids = [rng.integers(1000, 30000, size=L).astype(np.int32) for L in lens[sel]]
    types = [np.r_[np.zeros(12, np.int32), np.ones(L - 12, np.int32)] for L in lens[sel]]
    eng.score_tokens(ids[:256], types[:256])
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        logits, scores = eng.score_tokens(ids, types)              # host ids in -> host scores out
        order = np.argsort(-scores.reshape(len(mine), n_c), axis=1, kind="stable")   # rerank_chunks' reorder
    torch.cuda.synchronize()
    dt = torch.tensor([(time.perf_counter() - t0) / args.steps], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(dt, op=dist.ReduceOp.MAX)
    if args.dump_outputs and rank == 0:   # this rank's queries (all of them on one GPU)
        dump_outputs(args.dump_outputs, {"logits": logits, "scores": scores, "order": order})
    if rank == 0:
        total = n_q * n_c
        v = total / float(dt.item())
        tok = int(lens.sum())
        line = {"metric": "cross-encoder pairs/sec", "value": v, "unit": "pairs/s", "n_gpus": world, "steps": args.steps, "warmup": 1,
                "ms_per_step": float(dt.item()) * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": "f16", "data": "synthetic (seeded weights, random token pairs, mean 200 tokens)",
                "config": {"workload": w["desc"], "pairs": total, "tokens": tok, "parallelism": f"dp{world} over queries"},
                "e2e": {"value": v, "unit": "pairs/s", "h2d_bytes_per_step": int(tok * 12 // world), "d2h_bytes_per_step": int(total * 8 // world)},
                "gpu_launches": int(87 * np.ceil(tok / world / eng.max_tokens_per_call)) * args.steps, "reordered": int(order.shape[0])}
        # Tensor-pipe roofline of the whole forward (it is one fused sequence of GEMM-shaped kernels):
        # per layer 2*T*(4H^2 + 2HF) for the linears + 4*sum(L^2)*H for QK^T and PV (SURVEY 8d).
        Hh, Ff, Ly = 384, 1536, 12
        flops = Ly * (2.0 * tok * (4 * Hh * Hh + 2 * Hh * Ff) + 4.0 * float((lens.astype(np.float64) ** 2).sum()) * Hh)
        peaks = {}
        try:
            peaks = json.loads((ROOT / "MEASURED_PEAKS.json").read_text())
        except (OSError, ValueError):
            pass
        peak_tf = float(peaks.get("bf16_tflops", 1720.0))
        ach = flops / float(dt.item()) / 1e12
        line["roofline"] = {"bound": "tensor", "achieved": ach, "peak": peak_tf * world, "unit": "TFLOP/s", "frac": ach / (peak_tf * world),
                            "traffic": None, "kernel": "whole cross-encoder forward (linear_tcgen05 + attention + LayerNorm), wall clock incl. host packing",
                            "peak_source": "MEASURED_PEAKS.json bf16_tflops" if peaks else "fallback 1720 TFLOP/s"}
        if world == 1 and not args.no_cpu_baseline:
            from oracle import rerank as orr     # checker / CPU arm only: float32 transformers forward on a bounded sample
            model = orr.seeded_model(seed=0)
            n = 64
            torch.set_num_threads(len(os.sched_getaffinity(0)))
            orr.hf_logits(model, ids[:4], types[:4])     # first call pays thread-pool / allocator start-up
            t1 = time.perf_counter(); orr.hf_logits(model, ids[:n], types[:n]); cdt = time.perf_counter() - t1
            line["cpu_baseline"] = {"value": n / cdt, "unit": "pairs/s", "cores": torch.get_num_threads(), "kind": "port",
                                    "sample": f"{n} pairs, transformers BertForSequenceClassification fp32 (oracle.rerank.hf_logits)"}
        sys.stdout.flush(); os.dup2(saved, 1); print(json.dumps(line), flush=True); os.dup2(2, 1)
    if world > 1:
        dist.barrier(); dist.destroy_process_group()


def oracle_check(local, index, Q_raw, adapter, ids, sims, counts, *, w: dict, n_check: int, world: int, rank: int,  # noqa: ANN001, PLR0913
                 exact_maxsim: bool) -> dict:
    """Correctness gate outside the timed region, at every N: ``n_check`` queries against the ORACLE
    (``oracle.vector_search.vector_search_sql``, float64 distances, FLOAT ties -- the restatement of
    _search.py:65-79,143-153) over the whole sharded corpus.

    The oracle cannot hold a 61 GB shard per rank on the host, so every rank first shortlists, with a plain
    float32 matmul on its device, the ``take`` = selection size + 64 rows of its shard nearest to each query
    (a superset of that shard's share of the true selection unless more than 64 rows tie with the cut to
    within float32 rounding), the shortlisted rows (vectors, global chunk ids, global row order) are
    all-gathered, and rank 0 runs the oracle on that gathered table exactly as on any other table."""
    import torch
    import torch.distributed as dist

    from oracle import vector_search as ovs   # checker only: never on the timed / product path

    n = min(n_check, int(Q_raw.shape[0]))
    k, num_hits, V = w["k"], w["num_hits"], w["vecs"]
    sel = num_hits if num_hits else (k - 1) * V + 1
    take = min(local.n_rows, sel + 64)
    Qa = local.apply_adapter(Q_raw[:n].contiguous(), round_fp16=False) if adapter is not None else Q_raw[:n]
    Qn = Qa / Qa.norm(dim=1, keepdim=True)
    best_v = torch.full((n, take), -float("inf"), device=local.device)
    best_r = torch.zeros((n, take), dtype=torch.int64, device=local.device)
    step = 1 << 20
    for r0 in range(0, local.n_rows, step):
        blk = local.E[r0:r0 + step].float()
        s = (Qn @ blk.T) * local.inv_norm[r0:r0 + step][None, :]
        v, i = torch.topk(s, min(take, s.shape[1]), dim=1)
        cv, ci = torch.cat([best_v, v], 1), torch.cat([best_r, i + r0], 1)
        best_v, o = torch.topk(cv, take, dim=1)
        best_r = torch.gather(ci, 1, o)
    rows = best_r.reshape(-1)
    Esel = local.E[rows].float().reshape(n, take, -1)
    chunk = (local.row_chunk[rows].to(torch.int64) + local.chunk_base).reshape(n, take)
    order = (best_r + (rank << 40)).reshape(n, take)
    if world > 1:
        def gather(t):  # noqa: ANN001, ANN202
            out = torch.empty((world, *t.shape), dtype=t.dtype, device=t.device)
            dist.all_gather_into_tensor(out, t.contiguous())
            return out
        Esel, chunk, order = gather(Esel), gather(chunk), gather(order)
        Esel = Esel.permute(1, 0, 2, 3).reshape(n, world * take, -1)
        chunk = chunk.permute(1, 0, 2).reshape(n, world * take)
        order = order.permute(1, 0, 2).reshape(n, world * take)
    if rank != 0:
        return {"checked_queries": n}
    Esel, chunk, order, Qh = Esel.cpu().numpy(), chunk.cpu().numpy(), order.cpu().numpy(), Q_raw[:n].cpu().numpy()
    exact_sets, exact_order, sim_err = 0, 0, 0.0
    for b in range(n):
        o = np.argsort(order[b], kind="stable")          # the gathered table in global row order
        Eb, cb = Esel[b][o], chunk[b][o]
        if exact_maxsim:
            dist64 = ovs.vector_distances_f64(Eb, ovs.apply_query_adapter(adapter, Qh[b]), "cosine")
            oo = np.argsort(dist64, kind="stable")
            ref_ids, ref_s = ovs.group_hits(dist64[oo], cb[oo], k)
        else:
            ref_ids, ref_s, _ = ovs.vector_search_sql(Eb, None, Qh[b], num_results=k, oversample=w["oversample"], metric="cosine",
                                                      adapter=adapter, f64=True, f32_ties=True, row_chunk=cb)
        m = int(counts[b])
        got = ids[b, :m]
        exact_sets += int(m == len(ref_ids) and set(got.tolist()) == set(ref_ids.tolist()))
        exact_order += int(got.tolist() == ref_ids.tolist())
        mm = min(m, len(ref_s))
        sim_err = max(sim_err, float(np.abs(sims[b, :mm] - np.asarray(ref_s[:mm], np.float64)).max()) if mm else 0.0)
    return {"checked_queries": n, "identical_topk_sets": exact_sets, "identical_order": exact_order, "max_abs_score_err": sim_err,
            "oracle": "oracle.vector_search.vector_search_sql(f64, FLOAT ties) over the gathered per-shard shortlists",
            "shortlist_rows_per_shard": take}


def run_pool(args: argparse.Namespace, w: dict) -> None:
    """SURVEY 8a-4: the late-chunking pool (_embed.py:119-140).  A "step" pools ``batch`` segments of 496
    token rows x d float32 (bge-m3 at n_ctx 512, _embed.py:99) into per-sentence mean / L2 / fp16 rows in
    ONE launch of ``rl_segment_mean_pool``; the token matrices stay on the device for ``value`` and come
    from pinned host memory for ``e2e``."""
    import torch

    from raglite_b200 import _embed

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:      # the pool does not shard a document: replicas only; rank 0 reports
        return
    T_seg, d, n_seg = 496, w["dim"], w["batch"]
    rng = np.random.default_rng(0)
    seg_tokens, begins, ends, n_pre = [], [], [], []
    base = 0
    for _ in range(n_seg):          # ~24-token sentences; the first ~38% of a segment is preamble (not pooled)
        toks = np.maximum(rng.poisson(24, size=32), 1)
        toks = toks[: max(2, int(np.searchsorted(np.cumsum(toks), T_seg)))]
        sizes = _embed.largest_remainder_sizes(T_seg, toks)
        cuts = np.concatenate([[0], np.cumsum(sizes)]) + base
        first = int(np.searchsorted(np.cumsum(toks), 0.382 * T_seg))
        begins.append(cuts[first:-1]); ends.append(cuts[first + 1:])
        seg_tokens.append(toks); n_pre.append(first); base += T_seg
    rb, re_ = np.concatenate(begins), np.concatenate(ends)
    S, T = len(rb), n_seg * T_seg
    if args.impl == "reference":
        from oracle import pool as opool     # CPU arm: the NumPy restatement (pinned to the reference's goldens)

        n = 64
        X = rng.standard_normal((n * T_seg, d)).astype(np.float32)
        mats = [X[i * T_seg:(i + 1) * T_seg].astype(np.float64) for i in range(n)]
        t0 = time.perf_counter()
        reps = max(1, args.steps)
        for _ in range(reps):
            for i, m in enumerate(mats):
                opool.late_chunk_pool([m], seg_tokens[i], [(0, n_pre[i], len(seg_tokens[i]))])
        dt = (time.perf_counter() - t0) / reps
        v = n * T_seg / dt
        print(json.dumps({"impl": "reference", "metric": "late-chunking pool token rows/sec", "value": v, "unit": "token rows/s",
                          "n_gpus": args.gpus, "steps": reps, "warmup": 0, "ms_per_step": dt * 1e3, "higher_is_better": True,
                          "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                          "config": {"workload": w["desc"]},
                          "cpu_baseline": {"value": v, "unit": "token rows/s", "cores": 1, "kind": "port",
                                           "sample": f"{n} segments x {T_seg} x {d} (oracle.pool.late_chunk_pool, NumPy float64)"},
                          "e2e": {"value": v, "unit": "token rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}), flush=True)
        return
    sys.stdout.flush(); saved = os.dup(1); os.dup2(2, 1)
    torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", "0")))
    dev = torch.device("cuda")
    X = torch.randn((T, d), device=dev, generator=torch.Generator(device=dev).manual_seed(0))
    X_host = torch.empty((T, d), dtype=torch.float32, pin_memory=True)
    X_host.copy_(X)
    sampler = ClockSampler(torch.cuda.current_device()); sampler.start()
    for _ in range(max(args.warmup, 3)):
        out = _embed.segment_mean_pool(X, rb, re_, normalize=1)
    torch.cuda.synchronize(); sampler.wait_first_sample()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    w0 = time.perf_counter()
    # row ranges live on the device for the timed region (what pool_segments uploads once per document)
    rbd, red = torch.from_numpy(rb.astype(np.int32)).to(dev), torch.from_numpy(re_.astype(np.int32)).to(dev)
    outd = torch.empty((S, d), dtype=torch.float16, device=dev)
    from raglite_b200 import _lib
    lib = _lib.load()
    ev0.record()
    for _ in range(args.steps):
        _lib.check(lib.rl_segment_mean_pool(X.data_ptr(), d, d, rbd.data_ptr(), red.data_ptr(), S, 1, outd.data_ptr(),
                                            torch.cuda.current_stream().cuda_stream), "rl_segment_mean_pool")
    ev1.record(); torch.cuda.synchronize()
    windows = [(w0, time.perf_counter())]
    ms = ev0.elapsed_time(ev1) / args.steps
    if args.dump_outputs:   # a seeded sample of the pooled rows: all of them (S x 1024) would exceed the dump limit
        pick = np.sort(np.random.default_rng(0).choice(S, size=min(S, 8192), replace=False))
        dump_outputs(args.dump_outputs, {"pooled": outd[torch.from_numpy(pick).to(dev)].cpu().numpy(), "pooled_rows": pick})
    pooled_rows = int((re_ - rb).sum())
    alg_bytes = pooled_rows * d * 4 + S * d * 2 + S * 8
    t0 = time.perf_counter()
    for _ in range(args.steps):
        Xd = X_host.to(dev, non_blocking=True)
        o = _embed.segment_mean_pool(Xd, rb, re_, normalize=1)
        oh = o.cpu()
    e2e_ms = (time.perf_counter() - t0) * 1e3 / args.steps
    windows.append((t0, time.perf_counter()))
    clocks = sampler.stop(windows)
    # parity of the timed configuration against the oracle on a few segments
    from oracle import pool as opool
    got = outd.cpu().numpy()
    ulp_max, pos = 0, 0
    for i in range(4):
        ns = len(begins[i])
        want = opool.late_chunk_pool([X_host[i * T_seg:(i + 1) * T_seg].numpy().astype(np.float64)], seg_tokens[i],
                                     [(0, n_pre[i], len(seg_tokens[i]))])
        ulp = np.abs(got[pos:pos + ns].view(np.int16).astype(np.int32) - want.view(np.int16).astype(np.int32))
        ulp_max = max(ulp_max, int(ulp.max())); pos += ns
    assert ulp_max <= 1, ulp_max
    peaks = {}
    try:
        peaks = json.loads((ROOT / "MEASURED_PEAKS.json").read_text())
    except (OSError, ValueError):
        pass
    hbm = float(peaks.get("hbm_gbs", 6650.0))
    ach = alg_bytes / (ms * 1e-3) / 1e9
    line = {"metric": "late-chunking pool token rows/sec", "value": T / (ms * 1e-3), "unit": "token rows/s", "n_gpus": 1,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": w["desc"], "segments": n_seg, "token_rows": T, "pooled_rows": pooled_rows, "sentences": S, "dim": d,
                       "l2": "token matrix (%.1f GB) >> L2" % (T * d * 4 / 1e9)},
            "e2e": {"value": T / (e2e_ms * 1e-3), "unit": "token rows/s", "ms_per_step": e2e_ms, "h2d_bytes_per_step": int(T * d * 4),
                    "d2h_bytes_per_step": int(S * d * 2), "api": "raglite_b200._embed.segment_mean_pool (pinned host matrix in, host fp16 out)"},
            "gpu_launches": args.steps, "roofline": {"bound": "hbm", "achieved": ach, "peak": hbm, "unit": "GB/s", "frac": ach / hbm,
                                                     "traffic": None, "kernel": "segment_mean_pool_kernel", "kernel_ms": ms,
                                                     "algorithmic_bytes": alg_bytes,
                                                     "peak_source": "MEASURED_PEAKS.json hbm_gbs" if peaks else "fallback 6650 GB/s"},
            "clocks": clocks, "check": {"segments": 4, "max_fp16_ulp": ulp_max}}
    if not args.no_cpu_baseline:
        n = 32
        t1 = time.perf_counter()
        for i in range(n):
            opool.late_chunk_pool([X_host[i * T_seg:(i + 1) * T_seg].numpy().astype(np.float64)], seg_tokens[i],
                                  [(0, n_pre[i], len(seg_tokens[i]))])
        cdt = time.perf_counter() - t1
        line["cpu_baseline"] = {"value": n * T_seg / cdt, "unit": "token rows/s", "cores": 1, "kind": "port",
                                "sample": f"{n} segments x {T_seg} x {d} (oracle.pool.late_chunk_pool, NumPy float64, 1 thread of pooling)"}
    sys.stdout.flush(); os.dup2(saved, 1); print(json.dumps(line), flush=True); os.dup2(2, 1)
    _ = world


def main() -> None:  # noqa: PLR0915
    args = parse_args()
    w = resolve(args)
    w["oversample"] = args.oversample
    if w["name"] == "c5":
        run_rerank(args, w)
        return
    if w["name"] == "pool":
        run_pool(args, w)
        return
    if args.impl == "reference":
        run_reference(args, w)
        return

    # Keep stdout to the one JSON line: library chatter (e.g. "NCCL version ...") goes to stderr.
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    import torch
    import torch.distributed as dist

    import raglite_b200 as rl
    from raglite_b200._dist import ShardedIndex
    from raglite_b200._lib import RL_FLAG_TIME_KERNELS

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world} (launch with torch.distributed.run)"
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)

    B, k, num_hits, d = w["batch"], w["k"], w["num_hits"], w["dim"]
    E = build_shard(w, rank, device, args.storage, args.data)
    chunk_off = np.arange(0, E.shape[0] + 1, w["vecs"], dtype=np.int64)
    meta = None
    if args.filtered:   # two tags per chunk: "half" matches every other chunk (> 100k rows: rank-then-filter), "rare" 1 in 512
        meta = [{"half": c & 1, "rare": int(c % 512 == 0)} for c in range(w["chunks"])]
    local = rl.CorpusIndex(E, chunk_off, chunk_base=rank * w["chunks"], device=device, storage=args.storage, chunk_metadata=meta)
    esize = 2 if args.storage == "fp16" else 4
    del E
    index = ShardedIndex(local, group=dist.group.WORLD if world > 1 else None)

    # Queries: built from rank 0's rows so that every rank sees the same batch.
    noise, rows = make_batch_queries(local.E, w, seed=99)
    base = local.E[rows.to(device)].float().clone()
    if world > 1:
        dist.broadcast(base, src=0)
    Qd = base + 0.3 * noise.to(device)
    n_rand = B // 4
    Qd[:n_rand] = noise[:n_rand].to(device)
    Qd /= Qd.norm(dim=1, keepdim=True)
    Q_host = torch.empty((B, d), dtype=torch.float32, pin_memory=True)
    Q_host.copy_(Qd.cpu())
    torch.cuda.synchronize()

    total_chunks = w["chunks"] * world
    norm = total_chunks / TEN_M

    use_adapter = args.adapter == "on" or (args.adapter == "auto" and w["name"] == "c3")
    A_np = None
    if use_adapter:  # orthogonal d x d float64 adapter as the cosine fit produces (_query_adapter.py:204-205)
        Ad = torch.linalg.svd(torch.randn((d, d), dtype=torch.float64, generator=torch.Generator().manual_seed(2)))
        A_np = (Ad[0] @ Ad[2]).numpy()
        local.set_query_adapter(A_np)

    def device_step(flags: int = 0):  # noqa: ANN202
        Qa = local.apply_adapter(Qd, round_fp16=False) if use_adapter else Qd     # _search.py:58-62
        return index.search_pipeline(Qa, k=k, num_hits=num_hits, metric="cosine", algo=args.algo, flags=flags,
                                     sample_stride=args.sample_stride)

    def barrier() -> None:
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident throughput ("value") ----
    sampler = ClockSampler(local_rank)
    sampler.start()
    for _ in range(max(args.warmup, 3)):
        out = device_step()
    barrier()
    status = out[3].cpu().numpy()
    overflow_in_timed_config = bool((status & 1).any())
    sampler.wait_first_sample()
    windows = []
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    w0 = time.perf_counter()
    ev0.record()
    for _ in range(args.steps):
        out = device_step(flags=RL_FLAG_TIME_KERNELS)
    ev1.record()
    barrier()
    windows.append((w0, time.perf_counter()))
    if args.dump_outputs and rank == 0:   # the merged result of the last timed step: every rank holds the same one
        sim, chunk, count, status = (t.cpu().numpy() for t in out)
        dump_outputs(args.dump_outputs, {"sim": sim, "chunk": chunk, "count": count, "status": status})
    ms_total = ev0.elapsed_time(ev1)
    t = torch.tensor([ms_total], dtype=torch.float64, device=device)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_per_step = float(t.item()) / args.steps
    # Stage times averaged over the timed steps themselves (CUDA events recorded on the launch stream
    # inside rl_maxsim_topk; the library keeps a ring of 32 event sets, read after the loop).
    stage_ms = local.kernel_times_ms()
    stats = local.scan_stats()
    n_rows = local.n_rows
    scan_ms = float(stage_ms["main_scan"])
    burst = None
    if args.burst_probe:   # the emit-mode launch timed alone: 250 ms of idle GPU before every step (CUDA events, as above)
        alone = []
        for _ in range(6):
            torch.cuda.synchronize()
            time.sleep(0.25)
            device_step(flags=RL_FLAG_TIME_KERNELS)
            alone.append(float(local.kernel_times_ms()["main_scan"]))
        burst = {"main_scan_ms_after_250ms_idle": alone, "main_scan_ms_in_loop": scan_ms,
                 "note": "same launch, same inputs; only the load before it differs"}
    comm_ms = None
    if world > 1:   # where does the multi-GPU step go: scan pipeline vs all-gather vs merge (CUDA events, this rank)
        from raglite_b200._index import merge_packed
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        acc = np.zeros(3)
        H = num_hits if num_hits else k
        for _ in range(5):
            evs[0].record()
            res = local.scan(Qd, k=k, num_hits=num_hits, metric="cosine", algo=args.algo)
            evs[1].record()
            allb = torch.empty(world * res.packed.numel(), dtype=torch.uint8, device=device)
            dist.all_gather_into_tensor(allb, res.packed)
            evs[2].record()
            merge_packed(allb, world, B, H, num_hits=num_hits, k=k)
            evs[3].record()
            torch.cuda.synchronize()
            acc += np.array([evs[i].elapsed_time(evs[i + 1]) for i in range(3)]) / 5
        comm_ms = {"scan_pipeline": float(acc[0]), "all_gather": float(acc[1]), "merge": float(acc[2])}
    S = max(1, stats["sample_stride"])
    n_blocks = (n_rows + 127) // 128
    main_rows = min(n_rows, (n_blocks - (n_blocks + S - 1) // S) * 128)
    groups = (B + 255) // 256
    alg_bytes = main_rows * d * esize + main_rows * 4 + B * d * 4    # corpus rows once + inv_norm + queries (SURVEY 8d)
    peaks = {}
    try:
        peaks = json.loads((ROOT / "MEASURED_PEAKS.json").read_text())
    except Exception:  # noqa: BLE001
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    traffic = None
    try:   # dram__bytes_read.sum + dram__bytes_write.sum of this kernel from the committed ncu --set full capture
        for name in ("r02_traffic.json", "r01_traffic.json"):
            f = ROOT / "profiles" / name
            if not f.exists():
                continue
            tr = json.loads(f.read_text()).get(w["name"])
            if (tr and w["chunks"] == WORKLOADS[w["name"]]["chunks"] and B == WORKLOADS[w["name"]]["batch"]
                    and not args.exact_maxsim and args.storage == "fp32" and args.data == "gaussian"):
                traffic = tr["traffic_bytes_per_launch"]
                break
    except Exception:  # noqa: BLE001
        pass
    achieved = alg_bytes / (scan_ms * 1e-3) / 1e9 if scan_ms > 0 else 0.0
    flops = 2.0 * B * main_rows * d
    tensor_peak = peaks.get("bf16_tflops_sustained") or peaks.get("bf16_tflops")
    roofline = {"bound": "hbm", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak,
                "traffic": traffic, "kernel": "main scan (emit mode), algo=%s" % {1: "fp32", 2: "tcgen05"}.get(stats["algo"], "?"),
                "kernel_ms": scan_ms, "algorithmic_bytes": alg_bytes, "query_groups_per_launch": groups,
                "peak_source": "MEASURED_PEAKS.json hbm_gbs (of measured)" if peaks else "fallback 6650 GB/s (of fallback)",
                "tensor_tflops": flops / (scan_ms * 1e-3) / 1e12 if scan_ms > 0 else 0.0,
                "tensor_peak_tflops": tensor_peak,
                "tensor_frac": (flops / (scan_ms * 1e-3) / 1e12 / tensor_peak) if (tensor_peak and scan_ms > 0) else None}
    # Which roof binds: the arithmetic intensity of the launch (2*B*d flop per row of esize*d bytes) against the ridge of
    # the measured peaks.  fp32 corpus, B = 256: 128 flop/B, below the ridge (~229) -> HBM.  configs[2] (B = 1024) and the
    # fp16 layout at B = 256 (256 flop/B; ncu: tensor pipe 81 % active at the power-capped clock) are past it -> tensor.
    ridge = (tensor_peak * 1e12) / (hbm_peak * 1e9) if tensor_peak else None
    roofline["flop_per_byte"] = flops / alg_bytes
    roofline["ridge_flop_per_byte"] = ridge
    if tensor_peak and flops / alg_bytes > ridge:
        roofline.update({"bound": "tensor", "achieved": roofline["tensor_tflops"], "peak": tensor_peak, "unit": "TFLOP/s",
                         "frac": roofline["tensor_frac"], "hbm_gbs": achieved, "hbm_frac": achieved / hbm_peak,
                         "peak_source": "MEASURED_PEAKS.json bf16_tflops_sustained (kernel timed inside a long step)"})

    # ---- end to end through the public API: host queries in, host results out, every step ----
    cfg = rl.RAGLiteConfig(db_url=f"bench://rank{rank}", reranker=None, vector_search_query_adapter=use_adapter)
    rl.register_index(cfg, index)

    def timed_e2e(inflight: int = 1, **kw):  # noqa: ANN003, ANN202
        """K searches through the public API, host queries in -> host results out for every one of them.
        inflight = 1: vector_search_batch, one call after the other (each waits for its result);
        inflight > 1: vector_search_batch_async with that many batches in flight (each on its own stream with its own
        upload, kernels and pinned download; results collected in order) -- how a server drives the index."""
        from collections import deque

        common = dict(num_results=k, oversample=args.oversample, config=cfg, exact_maxsim=args.exact_maxsim, algo=args.algo, **kw)

        def run(n: int):  # noqa: ANN202
            r = None
            if inflight <= 1:
                for _ in range(n):
                    r = rl.vector_search_batch(Q_host, **common)
                return r
            pend: deque = deque()
            for _ in range(n):
                pend.append(rl.vector_search_batch_async(Q_host, **common))
                if len(pend) >= inflight:
                    r = pend.popleft().result()
            while pend:
                r = pend.popleft().result()
            return r

        run(3)
        barrier()
        t0 = time.perf_counter()
        r = run(args.steps)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        windows.append((t0, t0 + dt))
        tt = torch.tensor([dt], dtype=torch.float64, device=device)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        return r, float(tt.item()) * 1e3 / args.steps

    (ids_s, sims_s, counts_s), e2e_serial_ms = timed_e2e(1)
    (ids, sims, counts), e2e_ms = timed_e2e(args.inflight) if args.inflight > 1 else ((ids_s, sims_s, counts_s), e2e_serial_ms)
    assert np.array_equal(ids, ids_s) and np.array_equal(counts, counts_s), "pipelined and serial searches disagree"
    e2e_value = B / (e2e_ms * 1e-3) * norm
    filtered = None
    probe_calls = {"n": 0}
    if args.filtered:
        _orig_count = type(local).count_at_least

        def _counting(self, *a, **kw):  # noqa: ANN001, ANN002, ANN003, ANN202
            probe_calls["n"] += 1
            return _orig_count(self, *a, **kw)

        type(local).count_at_least = _counting
    if args.filtered:   # both reference branches (_search.py:96-143), same batch, same API
        _, ms_rare = timed_e2e(1, metadata_filter={"rare": 1})      # <= 100k matching rows: filter, then rank
        _, ms_half = timed_e2e(1, metadata_filter={"half": 1})      # > 100k rows in a > 1M-vector table: rank, then filter
        filtered = {"filter_first_ms": ms_rare, "rank_then_filter_ms": ms_half, "unfiltered_ms": e2e_serial_ms,
                    "rank_probe_passes_over_the_corpus": probe_calls["n"], "matching_rows_rare": int(local.filter_chunks({"rare": [1]})[1]),
                    "matching_rows_half": int(local.filter_chunks({"half": [1]})[1]),
                    "filter_first_vs_unfiltered": ms_rare / e2e_serial_ms, "rank_then_filter_vs_unfiltered": ms_half / e2e_serial_ms}
    clocks = sampler.stop(windows)
    clocks["windows"] = "timed device steps + timed e2e steps"

    # ---- correctness gate outside the timed region, at every N: the oracle over the whole sharded corpus ----
    check = {"checked_queries": 0}
    if not args.no_check:
        check = oracle_check(local, index, Qd, A_np, ids, sims, counts, w=w, n_check=args.check_queries, world=world, rank=rank,
                             exact_maxsim=args.exact_maxsim)
        if rank == 0 and args.data == "gaussian":
            assert check["identical_topk_sets"] == check["checked_queries"] and check["max_abs_score_err"] < 1e-4, check

    if rank == 0:
        qps_raw = B / (ms_per_step * 1e-3)
        line = {
            "metric": "queries/sec multi-vector MaxSim over 10M chunks", "value": qps_raw * norm,
            "unit": "queries/s (10M-chunk equivalent)", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32" if args.storage == "fp32" else "f16", "data": "synthetic" if args.data == "gaussian" else "synthetic (clustered)",
            "config": {"workload": w["desc"], "chunks_per_gpu": w["chunks"], "vecs_per_chunk": w["vecs"], "dim": d,
                       "batch": B, "k": k, "num_hits": num_hits, "metric": "cosine", "query_adapter": use_adapter,
                       "corpus_storage": args.storage, "corpus_data": args.data,
                       "semantics": "exact MaxSim" if args.exact_maxsim else "reference SQL (top-num_hits vectors -> group max -> top-k)",
                       "chunks_scanned": total_chunks, "normalisation": "value = batch / t_step * chunks_scanned / 10M",
                       "parallelism": f"row-sharded x{world}, NCCL all-gather of per-shard hits" if world > 1 else "single GPU shard",
                       "l2": "corpus shard (%.1f GB) >> L2, no flush needed" % (n_rows * d * esize / 1e9)},
            "queries_per_sec_raw": qps_raw,
            "e2e": {"value": e2e_value, "unit": "queries/s (10M-chunk equivalent)", "ms_per_step": e2e_ms,
                    "h2d_bytes_per_step": int(B * d * 4), "d2h_bytes_per_step": int(B * k * 12 + B * 4 + 4),
                    "api": ("raglite_b200.vector_search_batch_async, %d batches in flight (each: pinned host queries in -> its own stream "
                            "-> pinned host results out)" % args.inflight) if args.inflight > 1 else
                           "raglite_b200.vector_search_batch (pinned host queries in -> host numpy out, one sync)",
                    "batches_in_flight": max(1, args.inflight),
                    "serial_ms_per_step": e2e_serial_ms, "serial_api": "raglite_b200.vector_search_batch, one call after the other"},
            "gpu_launches": int((stats["launches"] + 1 + (1 if use_adapter else 0)) * args.steps),
            "launches_per_step": {"scan_pipeline": stats["launches"], "merge": 1, "adapter_apply": 1 if use_adapter else 0},
            "roofline": roofline,
            "stage_ms": stage_ms, "multi_gpu_stage_ms": comm_ms,
            "scan_stats": stats, "clocks": clocks, "check": check,
            "robustness": {"fp32_fallback_queries": 0, "candidate_overflow_in_timed_config": overflow_in_timed_config,
                           "streamed_survivor_queries": int(stats.get("survivors_max", 0) > 4096)},
        }
        if filtered is not None:
            line["filtered"] = filtered
        if burst is not None:
            line["burst_probe"] = burst
        if not args.no_cpu_baseline and world == 1:
            sample = args.cpu_sample_chunks or max(2048, min(w["chunks"], 16_384))
            r = cpu_reference_rate(w, sample, reps=3)
            line["cpu_baseline"] = {
                "value": r["qps_over_10M"], "unit": "queries/s (10M-chunk equivalent)", "cores": r["threads"], "kind": "port",
                "sample": f"{sample} chunks ({sample * w['vecs']} vectors) x batch {B}, {r['reps']} reps, median "
                          f"{r['t_sample_s']:.3f} s; extrapolated linearly in vectors"}
        sys.stdout.flush()
        os.dup2(saved_stdout, 1)
        print(json.dumps(line), flush=True)
        os.dup2(2, 1)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
