#!/usr/bin/env python
"""bench.py — headline benchmark of the hot path (contract in the task statement).

Default workload (BASELINE.json configs[1]): FLAT 10M x 768 fp32, cosine, k=10, batch=256 queries.
A "step" is one pass of the KNN hot path over one batch of 256 synthetic queries.

  value   true queries/s on the WHOLE corpus with queries and corpus resident in HBM, timed with CUDA events on the
          launching stream, max over ranks.
  e2e     the same through the host-facing C-ABI with HOST buffers: VecSimB200_TopKQueryBatch (N = 1) /
          VecSimB200_ShardGroup_TopKBatch (N > 1: H2D, shard scan, the ONE ncclAllGather, device merge, D2H — all inside).
  roofline  the dominant kernel (main pass of the tcgen05 coarse scan), timed with CUDA events inside the library.  The
            batched pass is tensor-bound (2*B*N*D flop against the measured dense bf16 peak of MEASURED_PEAKS.json); the
            HBM view sits beside it under roofline.hbm.  The single-query leg is HBM-bound.
  parity_at_config  after the timed region, 16+ of the 256 queries are checked at the FULL size against the reference's
            own distance kernels + heap (oracle/_ref) run over the device's corpus copied back to the host:
            ids and score bits.
  cpu_baseline  that same CPU scan, timed (one query per host thread over the full 10M x 768 corpus).

N > 1 (torchrun), --scaling strong (default): the 10M-row corpus of BASELINE configs[1] is row-sharded over the N GPUs
(10M / N rows each); a step = local scan + one all-gather of the packed per-shard top-k + device merge, all inside
VecSimB200_ShardGroup_TopKBatchDevice.  value = 256 / step time = QPS on exactly the BASELINE corpus at every N.
--scaling weak: every GPU holds its own 10M rows (corpus = N x 10M); value is still true QPS (on the N x 10M corpus),
`shard_query_rate` carries the additive figure (queries x 10M-row shards per second).

--config 3 | 5: BASELINE configs[2] (50M x 768 fp16, IP, k=100, batch 1024, sharded) and configs[4] (hybrid filtered
KNN: 10M x 768 fp32 pre-filtered by a 2-term posting-list intersection, k=10), same contract.

--impl reference: the reference's own BruteForceIndex::topKQuery (oracle/_ref, compiled from /root/reference) on the host
cores over the FULL 10M x 768 corpus (rank 0 only).

--dump-outputs DIR (configs 2 and 3): after the timed steps, rank 0 writes what the last timed step returned — labels.npy (float64)
and scores.npy (float32), one row per query — so that two builds can be compared output for output on the same seeded inputs.
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "KNN QPS @k=10 on 10M x 768 fp32 (cosine, batch=256)"
N_ROWS, DIM, K, BATCH = 10_000_000, 768, 10, 256
SEED_ROWS, SEED_QUERIES = 42, 43


def usable_cores():
    """Threads this process may really use: scheduler affinity, capped by the cgroup CPU quota."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:
            quota, period = f.read().split()[:2]
        if quota != "max":
            n = max(1, min(n, int(int(quota) / int(period))))
    except (OSError, ValueError):
        pass
    return n


def load_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def load_tensor_peak():
    """Dense bf16/fp16 tensor throughput (TFLOP/s): the burst figure, for a kernel timed alone."""
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return float(p["bf16_tflops"]), float(p.get("bf16_tflops_sustained", p["bf16_tflops"])), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 2250.0, 2250.0, "fallback (nominal dense bf16, B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region."""

    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.samples = []
        self.stop = threading.Event()
        self.t = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        while not self.stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.FIELDS}",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                parts = [x.strip() for x in out.strip().split(",")]
                if len(parts) >= 7:
                    self.samples.append(parts)
            except Exception:
                pass
            self.stop.wait(0.1)

    def __enter__(self):
        self.t.start()
        return self

    def __exit__(self, *a):
        self.stop.set()
        self.t.join(timeout=3)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no nvidia-smi samples"]}
        sm = [float(s[0]) for s in self.samples if s[0].replace(".", "").isdigit()]
        mx = [float(s[1]) for s in self.samples if s[1].replace(".", "").isdigit()]
        pw = [float(s[2]) for s in self.samples if s[2].replace(".", "").isdigit()]
        reasons = set()
        for s in self.samples:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), s[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "reasons": sorted(reasons), "samples": len(self.samples)}


DUMP_CAP_BYTES = 64 << 20


def dump_outputs(out_dir, **arrays):
    """Writes each (queries x k) device tensor as out_dir/<name>.npy in float32 or float64 (labels below 2^53 stay exact).  Past
    64 MB in all, a fixed seeded sample of query rows is kept, listed in rows.npy."""
    import numpy as np

    host = {name: t.cpu().numpy() for name, t in arrays.items()}
    host = {name: a.astype(np.float32 if a.dtype == np.float32 else np.float64) for name, a in host.items()}
    n = next(iter(host.values())).shape[0]
    total = sum(a.nbytes for a in host.values())
    if total > DUMP_CAP_BYTES:
        keep = np.sort(np.random.default_rng(0).choice(n, max(1, DUMP_CAP_BYTES // (total // n + 8)), replace=False))
        host = {name: a[keep] for name, a in host.items()}
        host["rows"] = keep.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in host.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def knn_config(rows_total, nq, k, world, scaling, dtype="fp32", metric="cosine"):
    """The `config` object: identical for our arm and the reference arm (nothing run-dependent in here)."""
    rows_gpu = rows_total // world if scaling == "strong" else rows_total
    corpus = rows_total if scaling == "strong" else rows_total * world
    shard = "" if world == 1 else f", row-sharded over {world} GPUs ({rows_gpu} rows each): one NCCL all-gather of per-shard top-k + device merge"
    return {"workload": f"FLAT {corpus} x {DIM} {dtype} {metric} k={k} batch={nq}{shard}", "corpus_rows": corpus, "rows_per_gpu": rows_gpu,
            "dim": DIM, "k": k, "batch": nq, "scaling": scaling,
            "l2_policy": "the corpus (GBs per GPU) is far larger than the 126 MB L2: every step re-reads it from HBM, no flush needed"}


# ------------------------------------------------------------------------------------------------
# reference arm: the reference's own CPU code on the host cores, FULL corpus
# ------------------------------------------------------------------------------------------------
def build_reference_index(ol, rows_total, threads, log):
    """10M x 768 fp32 cosine rows into the reference's BruteForceIndex.  Rows are generated by `threads` workers (the
    generator call releases the GIL) and added 250K at a time; blockSize 65536 (a BFParams knob of the reference) keeps
    brute_force.h's per-block resize of idToLabelMapping from going quadratic at 10M rows."""
    import numpy as np
    from concurrent.futures import ThreadPoolExecutor

    ix = ol.RefIndex(ol.F32, DIM, ol.COS, block_size=65536) if ol.ref_vecsim() is not None else None
    kind = "reference"
    if ix is None:
        kind = "port"
        ix = ol.PortIndex(ol.F32, DIM, ol.COS, tier=ol.TIER_AVX512)
    chunk = 250_000
    t0 = time.perf_counter()
    with ThreadPoolExecutor(max_workers=threads) as ex:
        done = 0
        while done < rows_total:
            n = min(chunk, rows_total - done)
            buf = np.empty((n, DIM), dtype=np.float32)
            parts = max(1, min(threads, n // 4096))
            bounds = [(done + n * i // parts, done + n * (i + 1) // parts) for i in range(parts)]
            list(ex.map(lambda b: ol.port().orc_synth_rows(ol.F32, SEED_ROWS, b[0], b[1] - b[0], DIM, ol._p(buf[b[0] - done:b[1] - done])), bounds))
            ix.add_many(buf, done + 1)
            done += n
    log["build_seconds"] = round(time.perf_counter() - t0, 1)
    return ix, kind


def run_reference_arm(args, rank, world):
    if rank != 0:
        return
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import numpy as np

    import oracle_lib as ol

    threads = usable_cores()
    rows_total = args.rows if args.scaling == "strong" else args.rows * world
    log = {}
    t_all = time.perf_counter()
    ix, kind = build_reference_index(ol, rows_total, threads, log)
    qs_all = ol.synth_rows(ol.F32, SEED_QUERIES, 0, args.batch, DIM)

    def run(nq_step, first):
        qs = np.ascontiguousarray(qs_all[[(first + i) % args.batch for i in range(nq_step)]])
        th = min(threads, nq_step)
        if kind == "reference":
            return ol.ref_vecsim().Ref_TimeTopK(ix.h, ol._p(qs), qs.strides[0], nq_step, K, th, None, None)
        return ol.port().orc_index_time_topk(ix.h, ol._p(qs), qs.strides[0], nq_step, K, th, None, None)

    # a step = nq_step queries, one per host thread (brute_force.h:243-291 is one thread per query), sized from a
    # calibration pass so that a step takes ~8 s; every step scans the full corpus
    cal_n = min(threads, 16)
    cal_s = run(cal_n, 0)
    nq_step = int(max(4, min(4 * threads, round(cal_n / cal_s * 8.0))))
    budget_s = 150.0
    warm = max(1, min(args.warmup, 2))
    for w in range(warm):
        run(nq_step, w * nq_step)
    times = []
    for i in range(args.steps):
        times.append(run(nq_step, (warm + i) * nq_step))
        if sum(times) > budget_s:
            break
    secs = sum(times)
    qps = nq_step * len(times) / secs
    cfg = knn_config(args.rows, args.batch, K, world, args.scaling)
    line = {"impl": "reference", "metric": METRIC, "value": qps, "unit": "queries/s", "n_gpus": args.gpus,
            "steps": len(times), "warmup": warm, "ms_per_step": 1000.0 * secs / len(times),
            "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": cfg,
            "cpu_baseline": {"value": qps, "unit": "queries/s", "cores": min(threads, nq_step), "kind": kind,
                             "sample": f"{len(times)} steps x {nq_step} queries over the FULL {rows_total} x {DIM} fp32 cosine corpus in the "
                                       f"reference's BruteForceIndex (blockSize 65536), one query per thread, {min(threads, nq_step)} threads "
                                       f"(usable cores: {threads}, os.cpu_count {os.cpu_count()}); a step is a bounded sample of the batch-{args.batch} workload",
                             "sample_seconds": secs, "queries_per_step": nq_step, "index_build_seconds": log.get("build_seconds"),
                             "wall_seconds": round(time.perf_counter() - t_all, 1)},
            "e2e": {"value": qps, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------
# second half of the metric: BM25 intersect docs/sec (BASELINE.json configs[3])
# ------------------------------------------------------------------------------------------------
from bench_postings import bench_postings, cpu_postings_baseline  # noqa: E402


# ------------------------------------------------------------------------------------------------
# helpers of our arm
# ------------------------------------------------------------------------------------------------
class Env:
    """torch / NCCL plumbing + the library handles for one rank."""

    def __init__(self):
        import torch

        self.torch = torch
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a CUDA device: the product has no CPU fallback")
        torch.cuda.set_device(self.local_rank)
        self.dev = torch.device("cuda", self.local_rank)
        self.dist = None
        if self.world > 1:
            import torch.distributed as dist

            dist.init_process_group("nccl", device_id=self.dev)
            self.dist = dist
        from redisearch_b200 import vecsim as vs
        from redisearch_b200._lib import load_library

        self.vs = vs
        self.L = vs.lib()
        S = load_library("libsynth_b200.so")
        S.Synth_FillRows.argtypes = [C.c_void_p, C.c_size_t, C.c_int, C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint32, C.c_void_p]
        S.Synth_NormalizeRowsF32.argtypes = [C.c_void_p, C.c_size_t, C.c_uint64, C.c_uint32, C.c_void_p]
        self.S = S
        # an explicit stream: a NULL handle would mean CUDA's legacy default stream
        self.stream = torch.cuda.Stream(device=self.dev)
        torch.cuda.set_stream(self.stream)
        self.sp = C.c_void_p(self.stream.cuda_stream)
        self.group = None

    def barrier(self):
        if self.dist is not None:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, x):
        if self.dist is None:
            return x
        t = self.torch.tensor([x], dtype=self.torch.float64, device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def shard_group(self):
        """The library's own NCCL communicator: rank 0 draws the id, torch.distributed (plumbing) ships the 128 bytes."""
        if self.group is None:
            import numpy as np

            idbuf = np.zeros(128, dtype=np.uint8)
            if self.world > 1:
                if self.rank == 0:
                    assert self.L.VecSimB200_ShardGroup_UniqueId(idbuf.ctypes.data) == 0, "cannot load NCCL"
                t = self.torch.from_numpy(idbuf).to(self.dev)
                self.dist.broadcast(t, 0)
                idbuf = t.cpu().numpy()
            self.group = self.L.VecSimB200_ShardGroup_New(idbuf.ctypes.data, self.rank, self.world)
            assert self.group, "VecSimB200_ShardGroup_New failed"
        return self.group

    def close(self):
        if self.group:
            self.L.VecSimB200_ShardGroup_Free(self.group)
            self.group = None
        if self.dist is not None:
            self.dist.destroy_process_group()


def build_shard(env, vtype, metric, rows, row0_global, dim=DIM, normalize=True):
    """Generate + (cosine fp32) normalise on device, ingest device-to-device.  Labels = global row + 1."""
    vs, L, S, torch = env.vs, env.L, env.S, env.torch
    index = vs.VecSimIndex(vtype, dim, metric)
    assert L.VecSimB200_Reserve(index.h, rows) == 0, "cannot reserve HBM for the corpus"
    es = {vs.VecSimType_FLOAT32: 4, vs.VecSimType_FLOAT16: 2, vs.VecSimType_BFLOAT16: 2}[vtype]
    tdt = {4: torch.float32, 2: torch.float16}[es]
    chunk = min(rows, 1_000_000)
    buf = torch.empty((chunk, dim), dtype=tdt, device=env.dev)
    t0 = time.perf_counter()
    done = 0
    while done < rows:
        n = min(chunk, rows - done)
        assert S.Synth_FillRows(buf.data_ptr(), dim * es, vtype, SEED_ROWS, row0_global + done, n, dim, env.sp) == 0
        if normalize and vtype == vs.VecSimType_FLOAT32 and metric == vs.VecSimMetric_Cosine:
            assert S.Synth_NormalizeRowsF32(buf.data_ptr(), dim * 4, n, dim, env.sp) == 0
        torch.cuda.synchronize()
        assert L.VecSimB200_AddVectorsDevice(index.h, buf.data_ptr(), n, row0_global + done + 1) == n
        done += n
    del buf
    return index, time.perf_counter() - t0


def bench_clustered(env, rows, nq, k, steps, check):
    """The proof tiers on a corpus that is NOT uniform: a mixture of tight Gaussians (every centre has ~rows / centres members
    within sigma, i.e. hundreds of near-duplicates of whatever a query is close to), queries drawn near centres.  On such data
    a query's admission bound lets far more than `keep` rows of one row range through, so the first tier overflows and the second
    (adaptive lists of 128) or, failing that, the exact scan answers.  Reports which tier proved how many queries, the step time,
    and parity of a few queries against the reference's kernels over the device's own rows."""
    import numpy as np

    vs, L, torch = env.vs, env.L, env.torch
    dev = env.dev
    centres_n, sigma = 2000, 0.015
    g = torch.Generator(device=dev)
    g.manual_seed(4242)
    centres = torch.rand((centres_n, DIM), generator=g, device=dev) * 2 - 1
    centres = centres / centres.norm(dim=1, keepdim=True)
    index = vs.VecSimIndex(vs.VecSimType_FLOAT32, DIM, vs.VecSimMetric_Cosine)
    assert L.VecSimB200_Reserve(index.h, rows) == 0
    done, chunk = 0, 250_000
    while done < rows:
        n = min(chunk, rows - done)
        # the members of a centre are CONTIGUOUS in row order (documents of one topic ingested together): ~1000 near-duplicates land
        # in ONE row range of the scan, far more than the 96 slots a first-tier list has under the bound
        which = (torch.arange(done, done + n, device=dev) // max(1, rows // centres_n)) % centres_n
        buf = centres[which] + sigma * torch.randn((n, DIM), generator=g, device=dev)
        buf = (buf / buf.norm(dim=1, keepdim=True)).contiguous()
        torch.cuda.synchronize()
        assert L.VecSimB200_AddVectorsDevice(index.h, buf.data_ptr(), n, done + 1) == n
        done += n
    qwhich = torch.randint(0, centres_n, (nq,), generator=g, device=dev)
    q = centres[qwhich] + sigma * torch.randn((nq, DIM), generator=g, device=dev)
    q = (q / q.norm(dim=1, keepdim=True)).contiguous()
    out_labels = torch.empty((nq, k), dtype=torch.int64, device=dev)
    out_scores = torch.empty((nq, k), dtype=torch.float32, device=dev)

    def step():
        assert L.VecSimB200_TopKQueryBatchDevice(index.h, q.data_ptr(), nq, k, out_labels.data_ptr(), out_scores.data_ptr(), env.sp) == 0

    for _ in range(3):
        step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    flags = np.zeros(nq, dtype=np.uint32)
    tiers = None
    if L.VecSimB200_LastCoarseFlags(index.h, flags.ctypes.data, nq) == 0:
        tiers = {"tier1": int((flags == 1).sum()), "tier2": int((flags == 2).sum()), "exact_scan": int((flags == 0).sum())}
    parity = None
    if check:
        pick = [(i * nq) // 8 for i in range(8)]
        qh = q.cpu().numpy()
        chk, _, kind = reference_scan_of_device_rows(env, index, rows, 0, np.ascontiguousarray(qh[pick]), k, 0, 2, usable_cores())
        dl, ds = out_labels.cpu().numpy(), out_scores.cpu().numpy()
        ids_ok = all(dl[qq].tolist() == chk.result(i)[0].tolist() for i, qq in enumerate(pick))
        bits_ok = all(ds[qq].tobytes() == chk.result(i)[1].astype(np.float32).tobytes() for i, qq in enumerate(pick))
        parity = {"queries": 8, "ids_equal": bool(ids_ok), "score_bits_equal": bool(bits_ok), "checker": kind}
    del index
    torch.cuda.empty_cache()
    return {"workload": f"FLAT {rows} x {DIM} fp32 cosine k={k} batch={nq}; corpus = {centres_n} unit centres + N(0, {sigma}^2) noise per coordinate "
                        f"(~{rows // centres_n} near-duplicates per centre, contiguous in row order), queries drawn the same way",
            "value": nq / (ms / 1000.0), "unit": "queries/s", "ms_per_step": ms, "proven_by_tier": tiers, "parity": parity,
            }


def reference_scan_of_device_rows(env, index, rows, row0_global, q_stored, k, vtype_code, metric_code, threads):
    """The parity checker at full size: copy this rank's stored rows back from HBM 500K at a time and feed them to the
    reference's own distance kernels + heap (tests/oracle_lib.StreamingTopK -> oracle/_ref Ref_ScanTopKChunk).  Returns
    (checker, cpu seconds spent in the scan, checker kind)."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import numpy as np

    import oracle_lib as ol

    st = ol.StreamingTopK(vtype_code, metric_code, DIM, q_stored, k, threads)
    es = q_stored.dtype.itemsize
    chunk = 500_000
    host = np.empty((chunk, DIM), dtype=q_stored.dtype)
    secs, done = 0.0, 0
    while done < rows:
        n = min(chunk, rows - done)
        assert env.L.VecSimB200_ReadRows(index.h, done, n, host.ctypes.data) == 0
        t0 = time.perf_counter()
        st.feed(host[:n], row0_global + done + 1)
        secs += time.perf_counter() - t0
        done += n
    assert es * DIM == host.strides[0]
    return st, secs, st.kind


# ------------------------------------------------------------------------------------------------
# our arm, config 2 (default): FLAT 10M x 768 fp32 cosine k=10 batch=256
# ------------------------------------------------------------------------------------------------
def run_knn(args):
    import numpy as np

    env = Env()
    torch, L, vs, S = env.torch, env.L, env.vs, env.S
    rank, world, dev, sp = env.rank, env.world, env.dev, env.sp
    warmup = max(3, args.warmup)
    nq = args.batch
    if args.scaling == "strong":
        lo = (args.rows * rank) // world
        hi = (args.rows * (rank + 1)) // world
        rows, row0 = hi - lo, lo
        corpus_rows = args.rows
    else:
        rows, row0 = args.rows, rank * args.rows
        corpus_rows = args.rows * world
    index, build_s = build_shard(env, vs.VecSimType_FLOAT32, vs.VecSimMetric_Cosine, rows, row0)
    group = env.shard_group()

    # ---- queries: same generator, normalised like VecSimIndex_TopKQuery would (preprocessors.h:121-131)
    qdev = torch.empty((nq, DIM), dtype=torch.float32, device=dev)
    assert S.Synth_FillRows(qdev.data_ptr(), DIM * 4, 0, SEED_QUERIES, 0, nq, DIM, sp) == 0
    q_host_raw = qdev.cpu().numpy().copy()  # raw (un-normalised) host blobs for the e2e arm
    assert S.Synth_NormalizeRowsF32(qdev.data_ptr(), DIM * 4, nq, DIM, sp) == 0
    torch.cuda.synchronize()
    q_stored = qdev.cpu().numpy().copy()
    out_labels = torch.empty((nq, K), dtype=torch.int64, device=dev)
    out_scores = torch.empty((nq, K), dtype=torch.float32, device=dev)

    def step_device():  # world > 1: local scan -> ONE all-gather of the packed per-shard top-k -> device merge, inside the library
        assert L.VecSimB200_ShardGroup_TopKBatchDevice(group, index.h, qdev.data_ptr(), nq, K, out_labels.data_ptr(),
                                                       out_scores.data_ptr(), sp) == 0

    for _ in range(warmup):
        step_device()
    env.barrier()
    index.stats(reset=True)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(env.local_rank) as clocks:
        env.barrier()
        ev0.record(env.stream)
        for _ in range(args.steps):
            step_device()
        ev1.record(env.stream)
        env.barrier()
    st = index.stats(reset=True)
    ms_step = env.max_over_ranks(ev0.elapsed_time(ev1)) / args.steps
    value = nq / (ms_step / 1000.0)  # true QPS: every step answers nq queries over the whole corpus
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, labels=out_labels, scores=out_scores)

    # ---- sustained: the same loop for >= 3 s (the short timed region above is a burst; the pass draws ~1 kW)
    sustained = None
    if args.sustained_seconds > 0:
        n_long = max(args.steps, int(args.sustained_seconds * 1000.0 / ms_step))
        with ClockSampler(env.local_rank) as clocks_long:
            env.barrier()
            ev0.record(env.stream)
            for _ in range(n_long):
                step_device()
            ev1.record(env.stream)
            env.barrier()
        ms_long = env.max_over_ranks(ev0.elapsed_time(ev1)) / n_long
        sustained = {"steps": n_long, "ms_per_step": ms_long, "value": nq / (ms_long / 1000.0), "clocks": clocks_long.summary()}
        index.stats(reset=True)

    # ---- e2e through the host-facing C-ABI: host blobs in, host results out (all ranks: it is a collective)
    h_labels = np.empty((nq, K), dtype=np.uint64)
    h_scores = np.empty((nq, K), dtype=np.float64)
    qh = np.ascontiguousarray(q_host_raw)

    def step_e2e():
        if world == 1:
            assert L.VecSimB200_TopKQueryBatch(index.h, qh.ctypes.data, qh.strides[0], nq, K, None, h_labels.ctypes.data, h_scores.ctypes.data) == 0
        else:
            assert L.VecSimB200_ShardGroup_TopKBatch(group, index.h, qh.ctypes.data, qh.strides[0], nq, K, h_labels.ctypes.data,
                                                     h_scores.ctypes.data) == 0

    for _ in range(3):
        step_e2e()
    e2e_steps = max(3, min(args.steps, 20))
    env.barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        step_e2e()
    torch.cuda.synchronize()
    e2e_s = env.max_over_ranks((time.perf_counter() - t0) / e2e_steps)
    e2e_value = nq / e2e_s
    dl, ds = out_labels.cpu().numpy(), out_scores.cpu().numpy()
    agree = bool((dl == h_labels.astype(np.int64)).all())

    # ---- proof statistics of the last device batch (tier 1 = sample pass + fixed bound, tier 2 = lists of 128, 0 = exact scan)
    step_device()
    torch.cuda.synchronize()
    flags = np.zeros(nq, dtype=np.uint32)
    tiers = None
    if world == 1 and L.VecSimB200_LastCoarseFlags(index.h, flags.ctypes.data, nq) == 0:
        tiers = {"tier1": int((flags == 1).sum()), "tier2": int((flags == 2).sum()), "exact_scan": int((flags == 0).sum())}

    # ---- parity at the quoted size + the CPU baseline: the reference's distance kernels + heap over the device's rows
    parity, cpu_base = None, None
    if not args.no_parity:
        threads = usable_cores()
        n_check = max(16, min(threads, 64, nq)) if world == 1 else 16
        pick = [(i * nq) // n_check for i in range(n_check)]
        chk, scan_s, chk_kind = reference_scan_of_device_rows(env, index, rows, row0, np.ascontiguousarray(q_stored[pick]), K, 0, 2, threads)
        local = [chk.result(i) for i in range(n_check)]
        if world > 1:  # merge the per-shard reference answers by (score, label) like the coordinator
            gathered = [None] * world
            env.dist.all_gather_object(gathered, local)
            local = []
            for i in range(n_check):
                ids = np.concatenate([g[i][0] for g in gathered])
                sc = np.concatenate([g[i][1] for g in gathered])
                order = np.lexsort((ids, sc))[:K]
                local.append((ids[order], sc[order]))
        ids_equal = all(dl[q].tolist() == local[i][0].tolist() for i, q in enumerate(pick))
        bits_equal = all(ds[q].tobytes() == local[i][1].astype(np.float32).tobytes() for i, q in enumerate(pick))
        parity = {"queries": n_check, "ids_equal": bool(ids_equal), "score_bits_equal": bool(bits_equal), "rows": corpus_rows,
                  "checker": f"{chk_kind}: the reference's dispatched distance kernel + its heap (oracle/_ref Ref_ScanTopKChunk) over the "
                             f"device's own stored rows copied back from HBM" + ("; per-shard answers merged by (score, label)" if world > 1 else ""),
                  "proven_by_tier": tiers}
        if world == 1:
            cpu_base = {"value": n_check / scan_s, "unit": "queries/s", "cores": min(threads, n_check), "kind": chk_kind,
                        "sample": f"{n_check} of the {nq} queries, one per host thread, each scanning the FULL {rows} x {DIM} fp32 corpus with the "
                                  f"reference's distance kernel + heap (the loop of brute_force.h:262-281 over flat 500K-row chunks); "
                                  f"usable cores {threads}",
                        "sample_seconds": scan_s}

    # ---- B=1 through the stock VecSimIndex_TopKQuery (what hybrid_reader.c:374 calls), N = 1 only.  Two legs: as served
    # (the fp16 shadow built by the batches above is current, so a single query rides the tensor-core route too) and the
    # exact HBM-bound scan alone (coarse mode off) — the north_star's ">= 10x CPU at >= 70% of HBM roofline" figure
    single = {}
    if world == 1:
        def single_query_leg():
            index.stats(reset=True)
            q1 = np.ascontiguousarray(q_host_raw[0])
            for _ in range(3):
                index.topk(q1, K)
            index.stats(reset=True)
            n1 = 20
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for i in range(n1):
                index.topk(np.ascontiguousarray(q_host_raw[i % nq]), K)
            dt = (time.perf_counter() - t0) / n1
            st1 = index.stats(reset=True)
            return dt, st1.scan_device_us / max(1, st1.scan_launches), int(L.VecSimB200_LastBatchPath(index.h))

        b1s_s, b1s_scan_us, b1s_path = single_query_leg()
        L.VecSimB200_SetCoarseMode(0)
        b1_s, b1_scan_us, _ = single_query_leg()
        L.VecSimB200_SetCoarseMode(-1)
        b1_bytes = rows * DIM * 4 + DIM * 4 + K * 12
        peak, _ = load_peaks()
        single = {"single_query_as_served": {"api": "VecSimIndex_TopKQuery with the fp16 shadow current", "value": 1.0 / b1s_s,
                                             "unit": "queries/s", "ms_per_query": b1s_s * 1000.0, "route": b1s_path,
                                             "dominant_kernel_us": b1s_scan_us},
                  "single_query": {"api": "VecSimIndex_TopKQuery (host blob in, reply out), exact scan only", "value": 1.0 / b1_s,
                                   "unit": "queries/s", "ms_per_query": b1_s * 1000.0,
                                   "roofline": {"bound": "hbm", "achieved": b1_bytes / (b1_scan_us * 1e-6) / 1e9, "peak": peak, "unit": "GB/s",
                                                "frac": b1_bytes / (b1_scan_us * 1e-6) / 1e9 / peak, "kernel": "scan_topk_kernel<f32,IP,4,1>",
                                                "avg_launch_us": b1_scan_us, "algorithmic_bytes_per_launch": b1_bytes}}}

    # ---- roofline of the dominant kernel: the library brackets it with CUDA events on the launch stream
    # (VecSimB200_GetStats); one launch per synchronised call so that every interval is one kernel
    peak, peak_src = load_peaks()
    index.stats(reset=True)
    per_launch = []
    for _ in range(max(3, min(args.steps, 10))):
        step_device()
        torch.cuda.synchronize()
        s_i = index.stats(reset=True)
        if s_i.scan_launches:
            per_launch.append(s_i.scan_device_us / s_i.scan_launches)
    scan_us = float(np.mean(per_launch)) if per_launch else None
    coarse_mode = int(os.environ.get("VECSIM_B200_COARSE", "1"))
    dom_kernel = {0: "scan_topk_kernel<f32,IP,4,8>",
                  1: "coarse_qtmem_kernel<fixed bound> (tcgen05 kind::f16 TS-mode, queries in TMEM, fp16 shadow rows; main pass)",
                  2: "coarse_kernel<CfgTF32> (tcgen05 kind::tf32)"}.get(coarse_mode, "?")
    traffic = None
    try:
        with open(os.path.join(ROOT, "profiles", "r2_traffic.json")) as f:
            t = json.load(f).get(dom_kernel.split(" ")[0].split("<")[0])
        if t and (t["rows"], t["dim"], t["batch"]) == (rows, DIM, nq):
            traffic = t["dram_bytes_per_launch"]
    except (OSError, ValueError, KeyError):
        pass
    alg_bytes = rows * DIM * 4 + nq * DIM * 4 + nq * K * 12  # SURVEY.md §8(d): N*D*s per corpus pass
    read_bytes = rows * DIM * (2 if coarse_mode == 1 else 4)   # what this kernel has to pull from HBM once
    achieved = alg_bytes / (scan_us * 1e-6) / 1e9 if scan_us else None
    hbm_view = {"achieved": achieved, "peak": peak, "unit": "GB/s", "frac": (achieved / peak) if achieved else None,
                "algorithmic_bytes_per_launch": alg_bytes, "hbm_bytes_read_per_launch": read_bytes,
                "frac_on_bytes_read": (read_bytes / (scan_us * 1e-6) / 1e9 / peak) if scan_us else None}
    common = {"traffic": traffic, "kernel": dom_kernel, "avg_launch_us": scan_us, "launch_us_samples": per_launch,
              "share_of_step": (scan_us / 1000.0 / ms_step) if scan_us else None}
    if coarse_mode in (1, 2) and scan_us:
        # batch of 256: 128 flop per fp32 corpus byte — the pass is tensor-bound (SURVEY.md §8d), HBM view kept beside it
        flops = 2.0 * nq * rows * DIM
        tpeak, tsust, tsrc = load_tensor_peak()
        if coarse_mode == 2:
            tpeak, tsust = tpeak / 2, tsust / 2  # TF32 runs at half the 16-bit rate
        tf = flops / (scan_us * 1e-6) / 1e12
        roofline = dict(common, bound="tensor", achieved=tf, peak=tpeak, unit="TFLOP/s", frac=tf / tpeak,
                        flops_per_launch=flops, peak_source=tsrc + " — burst dense bf16 (cuBLAS), kernel timed alone",
                        peak_sustained=tsust, hbm=dict(hbm_view, peak_source=peak_src),
                        note="per GPU; long runs sit at the 1000 W board power cap (see `sustained`)")
    else:
        roofline = dict(common, bound="hbm", peak_source=peak_src, **hbm_view)

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": "queries/s", "n_gpus": world, "steps": args.steps,
            "warmup": warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": args.scaling,
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": knn_config(args.rows, nq, K, world, args.scaling),
            "run_info": {"build_seconds": round(build_s, 2), "host_device_results_agree": agree,
                         "exchange": None if world == 1 else "VecSimB200_ShardGroup (library-owned NCCL communicator): one ncclAllGather of "
                                                             f"{L.VecSimB200_ShardBlockBytes(nq, K)} B per rank + merge_shards_kernel"},
            "e2e": {"value": e2e_value, "unit": "queries/s", "h2d_bytes_per_step": int(nq * DIM * 4),
                    "d2h_bytes_per_step": int(nq * K * 12), "ms_per_step": e2e_s * 1000.0,
                    "api": "VecSimB200_TopKQueryBatch" if world == 1 else "VecSimB200_ShardGroup_TopKBatch (includes the all-gather and the merge)"},
            "gpu_launches": int(st.kernel_launches),
            "roofline": roofline,
            "clocks": clocks.summary(),
            "sustained": sustained,
            "parity_at_config": parity,
        }
        if args.scaling == "weak" and world > 1:
            line["shard_query_rate"] = {"value": world * value, "unit": "queries x 10M-row shards / s"}
        line.update(single)
        if world == 1 and not args.no_clustered:
            del index
            index = None
            torch.cuda.empty_cache()
            try:
                line["clustered_corpus"] = bench_clustered(env, args.clustered_rows, nq, K, max(3, min(args.steps, 10)), check=not args.no_parity)
            except Exception as e:
                line["clustered_corpus"] = {"value": None, "error": repr(e)}
        if world == 1 and not args.no_postings:
            index = None
            torch.cuda.empty_cache()
            try:
                line["bm25_intersect"] = bench_postings(torch, dev, sp, args.posting_docs, max(1, min(args.steps, 5)), load_peaks()[0],
                                                        check=not args.no_parity)
            except Exception as e:
                line["bm25_intersect"] = {"value": None, "error": repr(e)}
        bm = line.get("bm25_intersect") if isinstance(line.get("bm25_intersect"), dict) else None
        gpu_rows = bm.pop("_gpu_rows", None) if bm else None
        doc_len = bm.pop("_doc_len", None) if bm else None
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_base if cpu_base else {"value": None, "error": "parity scan skipped (--no-parity)"}
            try:
                if bm and bm.get("value"):
                    cb = cpu_postings_baseline(args.posting_docs, usable_cores(), doc_len=doc_len, gpu_rows=gpu_rows)
                    bm["parity_at_config"] = cb.pop("parity_at_config", None)
                    bm["cpu_baseline"] = cb
            except Exception as e:  # the baseline is a reported side number; never fail the bench on it
                bm["cpu_baseline"] = {"value": None, "error": repr(e)}
        print(json.dumps(line))
    env.close()


# ------------------------------------------------------------------------------------------------
# config 3: FLAT 50M x 768 fp16, IP, k=100, batch=1024, row-sharded over the GPUs (BASELINE configs[2])
# ------------------------------------------------------------------------------------------------
def run_config3(args):
    import numpy as np

    env = Env()
    torch, L, vs, S = env.torch, env.L, env.vs, env.S
    rank, world, dev, sp = env.rank, env.world, env.dev, env.sp
    total, k, nq = args.rows3, 100, 1024
    lo, hi = (total * rank) // world, (total * (rank + 1)) // world
    rows = hi - lo
    index, build_s = build_shard(env, vs.VecSimType_FLOAT16, vs.VecSimMetric_IP, rows, lo)
    group = env.shard_group()
    qdev = torch.empty((nq, DIM), dtype=torch.float16, device=dev)
    assert S.Synth_FillRows(qdev.data_ptr(), DIM * 2, vs.VecSimType_FLOAT16, SEED_QUERIES, 0, nq, DIM, sp) == 0
    torch.cuda.synchronize()
    q_host = qdev.cpu().numpy().copy()
    out_labels = torch.empty((nq, k), dtype=torch.int64, device=dev)
    out_scores = torch.empty((nq, k), dtype=torch.float32, device=dev)

    def step_device():
        assert L.VecSimB200_ShardGroup_TopKBatchDevice(group, index.h, qdev.data_ptr(), nq, k, out_labels.data_ptr(), out_scores.data_ptr(), sp) == 0

    warmup = max(3, args.warmup)
    for _ in range(warmup):
        step_device()
    env.barrier()
    assert L.VecSimB200_LastBatchPath(index.h) == 2, "the batch did not take the tensor-core direct route"
    index.stats(reset=True)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(env.local_rank) as clocks:
        env.barrier()
        ev0.record(env.stream)
        for _ in range(args.steps):
            step_device()
        ev1.record(env.stream)
        env.barrier()
    st = index.stats(reset=True)
    ms_step = env.max_over_ranks(ev0.elapsed_time(ev1)) / args.steps
    scan_us = st.scan_device_us / max(1, st.scan_launches)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, labels=out_labels, scores=out_scores)
    h_labels = np.empty((nq, k), dtype=np.uint64)
    h_scores = np.empty((nq, k), dtype=np.float64)
    for _ in range(2):
        assert L.VecSimB200_ShardGroup_TopKBatch(group, index.h, q_host.ctypes.data, q_host.strides[0], nq, k, h_labels.ctypes.data, h_scores.ctypes.data) == 0
    e2e_steps = max(3, min(args.steps, 10))
    env.barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        assert L.VecSimB200_ShardGroup_TopKBatch(group, index.h, q_host.ctypes.data, q_host.strides[0], nq, k, h_labels.ctypes.data, h_scores.ctypes.data) == 0
    torch.cuda.synchronize()
    e2e_s = env.max_over_ranks((time.perf_counter() - t0) / e2e_steps)
    # parity at the quoted size: 8 queries against the reference's fp16 kernels over the device's rows (bar 1e-2)
    parity = None
    if not args.no_parity:
        threads = usable_cores()
        pick = [(i * nq) // 8 for i in range(8)]
        chk, scan_s, chk_kind = reference_scan_of_device_rows(env, index, rows, lo, np.ascontiguousarray(q_host[pick]), k, 3, 1, threads)
        local = [chk.result(i) for i in range(8)]
        if world > 1:
            gathered = [None] * world
            env.dist.all_gather_object(gathered, local)
            local = []
            for i in range(8):
                ids = np.concatenate([g[i][0] for g in gathered])
                sc = np.concatenate([g[i][1] for g in gathered])
                order = np.lexsort((ids, sc))[:k]
                local.append((ids[order], sc[order]))
        dl, ds = out_labels.cpu().numpy(), out_scores.cpu().numpy()
        # SURVEY §8(d): |delta| <= tol * max(|d_ref|, scale), tol = 1e-2 for fp16; scale = |q||x| for raw inner products (~256 for
        # these rows).  The check below uses the STRICTER scale 1: a pass here is a pass of the survey's bar.  (The reference's own
        # tiers differ from each other at this level: the AVX512-FP16 tier accumulates in half precision, SURVEY finding 5.)
        worst, worst_rel, id_overlap = 0.0, 0.0, 1.0
        for i, q in enumerate(pick):
            ref = local[i][1].astype(np.float32)
            diff = np.abs(ds[q] - ref)
            worst = max(worst, float(diff.max()))
            worst_rel = max(worst_rel, float((diff / np.maximum(np.abs(ref), 1.0)).max()))
            id_overlap = min(id_overlap, len(set(dl[q].tolist()) & set(local[i][0].tolist())) / k)
        parity = {"queries": 8, "max_abs_score_diff": worst, "max_rel_score_diff": worst_rel, "tolerance": 1e-2,
                  "tolerance_is": "relative: |delta| <= 1e-2 * max(|d_ref|, 1)", "within_tolerance": worst_rel <= 1e-2,
                  "min_id_overlap": id_overlap,
                  "checker": f"{chk_kind}: reference fp16 distance kernel (the CPU's own tier) + heap over the device's rows"}
    tpeak, tsust, tsrc = load_tensor_peak()
    flops = 2.0 * nq * rows * DIM
    tf = flops / (scan_us * 1e-6) / 1e12
    if rank == 0:
        print(json.dumps({
            "metric": "KNN QPS @k=100 on 50M x 768 fp16 (IP, batch=1024)", "value": nq / (ms_step / 1000.0), "unit": "queries/s", "n_gpus": world,
            "steps": args.steps, "warmup": warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f16", "data": "synthetic",
            "config": {"workload": f"FLAT {total} x {DIM} fp16 IP k={k} batch={nq}, row-sharded over {world} GPU(s) ({rows} rows each), one NCCL "
                                   f"all-gather of per-shard top-k + device merge", "corpus_rows": total, "rows_per_gpu": rows, "dim": DIM, "k": k, "batch": nq},
            "run_info": {"build_seconds": round(build_s, 2)},
            "e2e": {"value": nq / e2e_s, "unit": "queries/s", "h2d_bytes_per_step": int(nq * DIM * 2), "d2h_bytes_per_step": int(nq * k * 12),
                    "ms_per_step": e2e_s * 1000.0, "api": "VecSimB200_ShardGroup_TopKBatch"},
            "gpu_launches": int(st.kernel_launches),
            "roofline": {"bound": "tensor", "achieved": tf, "peak": tpeak, "unit": "TFLOP/s", "frac": tf / tpeak, "peak_sustained": tsust,
                         "peak_source": tsrc, "kernel": "coarse_qtmem_kernel<direct 16-bit> (tcgen05 kind::f16, rows through a 128B-swizzle tensor map)",
                         "avg_launch_us": scan_us, "flops_per_launch": flops, "share_of_step": scan_us / 1000.0 / ms_step, "traffic": None,
                         "hbm": {"algorithmic_bytes_per_launch": rows * DIM * 2, "achieved": rows * DIM * 2 / (scan_us * 1e-6) / 1e9,
                                 "peak": load_peaks()[0], "unit": "GB/s"}},
            "clocks": clocks.summary(), "parity_at_config": parity}))
    env.close()


# ------------------------------------------------------------------------------------------------
# config 5: hybrid filtered KNN — 10M x 768 fp32 FLAT scan pre-filtered by a 2-term posting intersection, k=10
# ------------------------------------------------------------------------------------------------
from bench_postings import run_config5  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=[2, 3, 5], help="2 = BASELINE configs[1] (default, the metric), 3 = configs[2], 5 = configs[4]")
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"])
    ap.add_argument("--rows", type=int, default=N_ROWS, help="corpus rows (strong scaling: total; weak: per GPU)")
    ap.add_argument("--rows3", type=int, default=50_000_000, help="config 3 corpus rows")
    ap.add_argument("--batch", type=int, default=BATCH)
    ap.add_argument("--sustained-seconds", type=float, default=3.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-postings", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--no-clustered", action="store_true", help="skip the clustered-corpus leg (proof tiers on non-uniform data)")
    ap.add_argument("--clustered-rows", type=int, default=2_000_000)
    ap.add_argument("--posting-docs", type=int, default=50_000_000)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's labels / scores as DIR/<name>.npy (configs 2 and 3)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or args.config == 5):
        ap.error("--dump-outputs covers the device KNN of configs 2 and 3")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        if args.config != 2:
            if rank == 0:
                print(json.dumps({"impl": "reference", "unavailable": f"the reference arm covers the metric's config only (config 2); config {args.config} has its CPU leg inside the line"}))
            return
        run_reference_arm(args, rank, world)
        return
    if args.config == 3:
        run_config3(args)
    elif args.config == 5:
        run_config5(args, Env, build_shard, ClockSampler, load_peaks, usable_cores)
    else:
        run_knn(args)


if __name__ == "__main__":
    main()
