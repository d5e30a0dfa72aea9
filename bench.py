#!/usr/bin/env python
"""bench.py -- exact kNN queries/sec on the BASELINE.json headline workload, plus BASELINE configs 1-5.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--configs all|none|c1,c3,...] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Headline workload (BASELINE.json metric): 10M x 768 fp32 rows, cosine, k=10, batch-1 queries; with N GPUs the rows are
sharded over the ranks (strong scaling: total work fixed) and every query ends with the exchange of the ranks'
candidates fused into the scan kernel (NVLink peer memory).  A "step" is ``--queries-per-step`` consecutive batch-1
queries (each a full pass over the stored rows).

One JSON line on rank 0:
  value     queries/s with queries and results resident in HBM (device pointers through the C ABI, CUDA-event timed,
            max over ranks).  Every query is its own search (own launch, own result); two are in flight on two streams
            so one query's scan fills the SMs the previous one's tail has left (roofline.one_query_in_flight has the
            strictly serial rate)
  e2e       the same through the reference-shaped public API: ``search(VectorDTO, top_k, namespace, metric) ->
            List[SearchResult]`` -- ``GpuIndex`` at N=1, ``ShardedGpuIndex`` (one process per GPU) at N>1; host query in,
            host results out, copies inside; two requests in flight (``search_async``), and
            e2e.one_request_at_a_time is the plain synchronous ``search`` call
  parity    UNTIMED gate: some of the timed queries, taken from the device path AND from the e2e path, are checked on
            rank 0 against the streamed C oracle over all 10M rows (oracle/exact_scan.c::orc_knn_synthetic, the full
            parity rule of oracle/exact.py::check_topk_parity).  A mismatch makes every rank exit non-zero.
  roofline  scan kernel: algorithmic bytes per launch / average launch duration over the timed region (region device
            time / scan launches in it) vs the measured HBM copy peak; kernel_alone = CUDA events around every scan
            launch with one query in flight
  configs   BASELINE.json configs[0..4] timed after the headline region (each with its own roofline and parity entry):
            c1 10k x 128 single-query latency, c2 1M x 768 batch-1, c3 10M x 768 l2 k=100 4096-query batches on N GPUs
            (tensor-core path), c4 10M x 384 filtered at 1 / 10 / 50 %, c5 100M x 128 ip kNN + range search on N GPUs
  cpu_baseline  the oracle's C port of hnswlib's brute-force arithmetic on the host cores, on a bounded row sample,
            scaled to the full row count (N=1, rank 0 only)

``--impl reference`` times that CPU implementation as the reference arm (the reference's own search is the absent
hnswlib wheel; see DESIGN.md) with every host core it may use and prints the same line with impl=reference.

``--dump-outputs DIR`` writes what the device path returned for the queries of the last timed headline step:
distances.npy [nq, k] float32, rows.npy [nq, k] and counts.npy [nq] as float64, and query_index.npy (which queries of the
step they are; all of them unless the step's results exceed 60 MB).  Rows and queries come from fixed seeds, so two runs
with the same arguments see the same inputs.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "exact_knn_queries_per_sec"
UNIT = "queries/s"
SEED = 42
PART_SHIFT = 40


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10,
                    help="timed steps of the headline region and of its e2e measurement (configs c1-c5 time fixed repetitions)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--rows", type=int, default=10_000_000)
    ap.add_argument("--dim", type=int, default=768)
    ap.add_argument("--k", type=int, default=10)
    ap.add_argument("--space", default="cosine")
    ap.add_argument("--queries-per-step", type=int, default=32)
    ap.add_argument("--inflight", type=int, default=2,
                    help="independent batch-1 queries in flight (one CUDA stream each); 1 = strictly one at a time")
    ap.add_argument("--e2e-inflight", type=int, default=4,
                    help="requests in flight through the asynchronous public API in the e2e measurement (1..4: the handle's async slots)")
    ap.add_argument("--cpu-sample-rows", type=int, default=1_000_000)
    ap.add_argument("--cpu-queries", type=int, default=48)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--parity-queries", type=int, default=4, help="timed queries checked against the streamed oracle (0 = skip)")
    ap.add_argument("--configs", default="all", help="all | none | comma list of c1,c2,c3,c4,c5")
    ap.add_argument("--configs-scale", type=float, default=1.0, help="scale the configs' row counts (development runs)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the results of the last timed headline step to DIR/<name>.npy (float32/float64) so that "
                         "two builds can be compared output for output")
    a = ap.parse_args()
    if a.steps < 1 or a.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if a.dump_outputs and a.impl == "reference":
        ap.error("--dump-outputs writes the device path's results; the reference arm has none to write")
    return a


def workload_config(a, n_gpus):
    return {
        "workload": f"{a.rows}x{a.dim} fp32 {a.space} exact kNN k={a.k}, batch-1 queries "
                    f"(BASELINE.json metric config; rows sharded over {n_gpus} GPU(s))",
        "rows": a.rows, "dim": a.dim, "k": a.k, "space": a.space, "batch": 1,
        "queries_per_step": a.queries_per_step, "queries_in_flight": a.inflight,
        "parallelism": f"row-shard x{n_gpus}" if n_gpus > 1 else "single GPU",
        "l2": f"no flush needed: every query streams {a.rows * a.dim * 4 / n_gpus / 1e9:.2f} GB per GPU (> 126 MB L2)",
    }


def make_queries(nq, dim):
    return np.random.default_rng(SEED + 1).standard_normal((nq, dim), dtype=np.float32)


DUMP_MAX_BYTES = 60_000_000      # data; the four .npy headers add 512 bytes, the whole dump stays under 64 MB


def dump_outputs(out_dir, dists, rows, counts):
    """Write one step's results (dists [nq, k] fp32, global rows [nq, k], counts [nq]) as .npy files.  Ids go out as
    float64 (exact below 2**53).  Past DUMP_MAX_BYTES a fixed seeded sample of the queries is written;
    query_index.npy says which."""
    nq, k = dists.shape
    per_query = k * (4 + 8) + 8 + 8
    keep = np.arange(nq)
    if nq * per_query > DUMP_MAX_BYTES:
        keep = np.sort(np.random.default_rng(SEED).choice(nq, DUMP_MAX_BYTES // per_query, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    for name, arr in (("distances", dists[keep].astype(np.float32)), ("rows", rows[keep].astype(np.float64)),
                      ("counts", counts[keep].astype(np.float64)), ("query_index", keep.astype(np.float64))):
        np.save(os.path.join(out_dir, f"{name}.npy"), arr)


def hbm_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            j = json.load(f)
        return float(j["hbm_gbs"]), float(j.get("bf16_tflops", 1621.8)), "measured (MEASURED_PEAKS.json)"
    return 6650.0, 1621.8, "fallback (B200_PROFILING.md)"


# --------------------------------------------------------------------------- clocks sampler
class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons of one GPU during the timed region (NVML)."""

    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
               0x80: "hw_power_brake_slowdown"}

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu_index = gpu_index
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop_evt = threading.Event()
        self.error = None

    def run(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(self.gpu_index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
            while not self._stop_evt.is_set():
                self.samples.append(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM))
                mask = pynvml.nvmlDeviceGetCurrentClocksEventReasons(h)
                for bit, name in self.REASONS.items():
                    if mask & bit:
                        self.reasons.add(name)
                time.sleep(0.05)
        except Exception as e:  # noqa: BLE001
            self.error = repr(e)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=2)

    def summary(self):
        out = {"sm_mhz": statistics.median(self.samples) if self.samples else None, "sm_max_mhz": self.max_mhz,
               "reasons": sorted(self.reasons), "samples": len(self.samples)}
        if self.error:
            out["error"] = self.error
        return out


def physical_gpu_index(local_rank):
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    if vis:
        try:
            return int(vis.split(",")[local_rank])
        except (ValueError, IndexError):
            pass
    return local_rank


# --------------------------------------------------------------------------- CPU arm (oracle)
def cpu_knn_qps(a, steps, warmup, queries_per_step):
    """Oracle C port (hnswlib brute-force arithmetic, SIMD16 summation order, EVERY host core this process may use --
    torchrun's OMP_NUM_THREADS=1 is overridden) on a bounded prefix of the rows; queries/s scaled linearly to the full
    row count."""
    from oracle import cscan

    cores = cscan.use_all_cores()
    n = min(a.cpu_sample_rows, a.rows)
    X = cscan.fill_synthetic(SEED, 0, n, a.dim, True)
    if a.space == "cosine":
        X = cscan.normalize(X)
    Q = make_queries(queries_per_step, a.dim)
    if a.space == "cosine":
        Q = cscan.normalize(Q)
    for _ in range(warmup):
        cscan.knn(X, Q[:2], a.k, a.space)
    t0 = time.perf_counter()
    for _ in range(steps):
        for j in range(queries_per_step):
            cscan.knn(X, Q[j:j + 1], a.k, a.space)
    dt = time.perf_counter() - t0
    qps_sample = steps * queries_per_step / dt
    frac = n / a.rows
    return {
        "value": qps_sample * frac, "unit": UNIT, "cores": cores, "kind": "port",
        "sample": f"first {n} of {a.rows} rows (a {frac:g} prefix), {steps} x {queries_per_step} batch-1 queries in {dt:.1f} s "
                  f"({qps_sample:.2f} q/s on the sample, {dt / (steps * queries_per_step) * 1e3:.1f} ms per query); "
                  f"scaled by {frac:g} (a scan is linear in rows)",
        "row_prefix_used": n < a.rows, "ms_per_query_on_sample": dt / (steps * queries_per_step) * 1e3,
        "impl": "oracle/exact_scan.c orc_knn (hnswlib 0.8.0 arithmetic restated; hnswlib itself is not installable here)",
    }, dt


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # the same step as the GPU arm (queries_per_step batch-1 queries), each query over a bounded row prefix
    base, dt = cpu_knn_qps(a, a.steps, max(a.warmup, 1), a.queries_per_step)
    line = {
        "impl": "reference", "metric": METRIC, "value": base["value"], "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps,
        "warmup": a.warmup, "ms_per_step": dt / a.steps * 1e3, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(a, a.gpus),
        "cpu_baseline": base,
        "e2e": {"value": base["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit_result(line)


# --------------------------------------------------------------------------- GPU arm
class Ctx:
    """Process-wide plumbing of the GPU arm: ranks, device, collectives, device timing."""

    def __init__(self):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device; the product has no CPU path (use --impl reference for the CPU arm)")
        torch.cuda.set_device(self.local_rank)
        self.device = torch.device("cuda", self.local_rank)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.device)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()

    def reduce(self, x, op):
        if self.world == 1:
            return x
        t = self.torch.tensor([x], dtype=self.torch.float64, device=self.device)
        self.dist.all_reduce(t, op=op)
        return float(t.item())

    def max_over_ranks(self, x):
        return self.reduce(x, self.dist.ReduceOp.MAX)

    def sum_over_ranks(self, x):
        return self.reduce(x, self.dist.ReduceOp.SUM)

    def timed(self, fn, n, streams=()):
        """n calls of fn between two events on the current stream that every lane stream is fenced by; max over ranks."""
        torch = self.torch
        cur = torch.cuda.current_stream(self.device)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        self.barrier()
        torch.cuda.synchronize()
        e0.record(cur)
        for st in streams:
            st.wait_event(e0)
        for _ in range(n):
            fn()
        for st in streams:
            cur.wait_stream(st)
        e1.record(cur)
        torch.cuda.synchronize()
        self.barrier()
        return self.max_over_ranks(e0.elapsed_time(e1))

    def agree(self, ok: bool) -> bool:
        """True only when every rank says ok."""
        return self.reduce(0.0 if ok else 1.0, self.dist.ReduceOp.MAX) == 0.0 if self.world > 1 else ok


def gen_row_of(global_rows, n_rows, world):
    """ShardedGpuIndex.add_synthetic layout: global row = rank << 40 | local row, generator row = rank * ceil(n/world) + local."""
    g = np.asarray(global_rows, dtype=np.int64)
    if world == 1:
        return g
    per = -(-n_rows // world)
    return np.where(g >= 0, (g >> PART_SHIFT) * per + (g & ((1 << PART_SHIFT) - 1)), -1)


def global_row_of(gen_row, n_rows, world):
    if world == 1:
        return int(gen_row)
    per = -(-n_rows // world)
    return ((int(gen_row) // per) << PART_SHIFT) | (int(gen_row) % per)


def run_ours(a):
    ctx = Ctx()
    torch = ctx.torch
    from mlvectordb_b200 import GpuIndex, VectorDTO
    from mlvectordb_b200.sharded_index import ShardedGpuIndex

    world, rank, device = ctx.world, ctx.rank, ctx.device
    # ---- data: generated on the device, rows sharded over ranks ------------------------------
    ns = "bench"
    if world == 1:
        index = GpuIndex(space=a.space, device=ctx.local_rank, capacity=a.rows)
        index.add_synthetic(ns, a.rows, a.dim, SEED, scaled=True)
        shard = index._ns[ns].shard
        searcher = None
        local_rows = a.rows
    else:
        index = ShardedGpuIndex(space=a.space, device=device, capacity=a.rows)
        index.add_synthetic(ns, a.rows, a.dim, SEED, scaled=True)
        searcher = index._ns[ns].searcher
        shard = searcher.shard
        local_rows = shard.rows
    qps_step = a.queries_per_step
    Q = make_queries(qps_step, a.dim)
    Qd = torch.from_numpy(Q).to(device)
    k = a.k
    inflight = max(1, min(a.inflight, 2))
    streams = [torch.cuda.Stream(device) for _ in range(inflight)]
    # one result buffer per query of a step, so that the whole last step is still there when it is read back
    outs = [(torch.empty((1, k), dtype=torch.float32, device=device), torch.empty((1, k), dtype=torch.int64, device=device),
             torch.empty((1,), dtype=torch.int32, device=device)) for _ in range(qps_step)]
    step_results = [None] * qps_step

    def device_query(j, st, o):
        """ONE batch-1 search through the C ABI with device pointers, on stream st, results into o."""
        with torch.cuda.stream(st):
            if searcher is None:
                shard.search_device(Qd[j:j + 1].data_ptr(), 1, k, o[0].data_ptr(), o[1].data_ptr(), o[2].data_ptr(),
                                    stream=st.cuda_stream)
                return o
            return searcher.search_device(Qd[j:j + 1], k)

    def step_device(lanes=inflight):
        # every query is its own search (own launch, own result); `lanes` of them are in flight, each
        # on its own stream, so one query's scan fills the SMs the previous one's tail has left
        for j in range(qps_step):
            step_results[j] = device_query(j, streams[j % lanes], outs[j])

    def api_search(j):
        return index.search(VectorDTO(values=Q[j], metadata={}), top_k=k, namespace=ns, metric=a.space)

    e2e_depth = max(1, min(a.e2e_inflight, 4))

    def step_e2e(depth=e2e_depth):
        # host query in, host List[SearchResult] out, per query; `depth` requests in flight through the asynchronous
        # public API (search_async / .result()), 1 = the plain synchronous search() call
        last, pending = None, []
        for j in range(qps_step):
            if depth <= 1:
                last = api_search(j)
                continue
            pending.append(index.search_async(VectorDTO(values=Q[j], metadata={}), top_k=k, namespace=ns, metric=a.space))
            if len(pending) >= depth:
                last = pending.pop(0).result()
        for p in pending:
            last = p.result()
        return last

    # ---- device-resident timing ----------------------------------------------------------------
    for _ in range(a.warmup):
        step_device()
    torch.cuda.synchronize()
    launches0 = shard.kernel_launches()
    merges0 = searcher.merge_launches if searcher else 0
    half0 = shard.gemm_stats()
    sampler = ClockSampler(physical_gpu_index(ctx.local_rank))
    sampler.start()
    ms_total = ctx.timed(step_device, a.steps, streams)
    sampler.stop()
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, *(torch.cat([r[i] for r in step_results]).cpu().numpy() for i in range(3)))
    half1 = shard.gemm_stats()
    half_q = half1["half_scan_queries"] - half0["half_scan_queries"]           # searches that read the fp16 shadow
    half_u = half1["half_scan_uncertified"] - half0["half_scan_uncertified"]   # ... re-run by the fp32 launch behind
    launches = shard.kernel_launches() - launches0 + ((searcher.merge_launches - merges0) if searcher else 0)
    total_launches = int(ctx.sum_over_ranks(launches))
    n_queries = a.steps * qps_step
    value = n_queries / (ms_total / 1e3)
    # the scan kernel alone: one query at a time, CUDA events around every scan launch
    shard.set_timing(True)
    shard.scan_time_ms()
    alone_steps = max(1, min(a.steps, 3))
    alone_ms = ctx.timed(lambda: step_device(1), alone_steps, streams)
    scan_ms, scan_n = shard.scan_time_ms()
    shard.set_timing(False)

    # ---- end-to-end timing through the public host API -----------------------------------------
    def time_e2e(depth):
        for _ in range(a.warmup):
            step_e2e(depth)
        ctx.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(a.steps):
            out = step_e2e(depth)
        torch.cuda.synchronize()
        dt = ctx.max_over_ranks(time.perf_counter() - t0)
        ctx.barrier()
        return n_queries / dt, out

    e2e_value, last = time_e2e(e2e_depth)
    e2e_sync_value, last_sync = time_e2e(1)

    # ---- parity gate (untimed): timed queries vs the streamed oracle over ALL rows -----------------------------------
    parity = {"queries": 0, "ok": None, "how": "skipped (--parity-queries 0)"}
    n_par = min(max(a.parity_queries, 0), qps_step)
    if n_par:
        # every rank re-runs the first n_par timed queries on both paths (the searches are collective at N > 1)
        dev_rows, dev_d, dev_c, api_hits = [], [], [], []
        for j in range(n_par):
            o = device_query(j, streams[0], outs[0])
            torch.cuda.synchronize()
            dev_d.append(o[0].cpu().numpy()[0]); dev_rows.append(o[1].cpu().numpy()[0]); dev_c.append(int(o[2].cpu().numpy()[0]))
            api_hits.append(api_search(j))
        problems = []
        t_or = 0.0
        if rank == 0:
            from oracle import cscan, exact
            cores = cscan.use_all_cores()
            t0 = time.perf_counter()
            L, D, Cn = cscan.knn_synthetic(SEED, 0, a.rows, a.dim, True, Q[:n_par], k, a.space)
            t_or = time.perf_counter() - t0
            nsobj = index._ns[ns]
            for j in range(n_par):
                adjud = lambda l, j=j: float(cscan.distances_synthetic(SEED, [l], a.dim, True, Q[j], a.space)[0])  # noqa: E731
                c = int(Cn[j])
                if dev_c[j] != c:
                    problems.append(f"device path q{j}: count {dev_c[j]} vs oracle {c}")
                    continue
                msg = exact.check_topk_parity(gen_row_of(dev_rows[j][:c], a.rows, world), dev_d[j][:c], L[j, :c], D[j, :c], all_ref_scores=adjud)
                if msg:
                    problems.append(f"device path q{j}: {msg}")
                hits = api_hits[j]
                if len(hits) != c:
                    problems.append(f"api q{j}: {len(hits)} hits vs oracle {c}")
                    continue
                # SearchResult carries a UUID: map it back through the id table of the rows the device path returned
                by_uuid = {nsobj.uuid_of(int(r)): int(g) for r, g in zip(dev_rows[j][:c], gen_row_of(dev_rows[j][:c], a.rows, world))}
                api_rows = [by_uuid.get(h.vector_id, -1) for h in hits]
                api_d = np.array([(1.0 - h.score) if a.space == "cosine" else h.score for h in hits])
                if -1 in api_rows or api_rows != gen_row_of(dev_rows[j][:c], a.rows, world).tolist():
                    problems.append(f"api q{j}: ids differ from the device path's")
                msg = exact.check_topk_parity(api_rows, api_d, L[j, :c], D[j, :c], all_ref_scores=adjud)
                if msg:
                    problems.append(f"api q{j}: {msg}")
            parity = {"queries": n_par, "ok": not problems, "paths": ["device pointers (value)", "public API (e2e)"],
                      "how": f"streamed C oracle over all {a.rows} generator rows (orc_knn_synthetic, {cores} threads, {t_or:.1f} s), "
                             "oracle.exact.check_topk_parity: scores within 1e-5*max+1e-6, id sets equal except ties with the k-th",
                      "problems": problems[:8]}
        ok = ctx.agree(not problems)
        if not ok:
            if rank == 0:
                emit_result({"metric": METRIC, "value": None, "unit": UNIT, "n_gpus": world, "parity": parity,
                             "error": "parity gate failed: results differ from the oracle; no number is reported"})
            index.close()
            if world > 1:
                ctx.dist.destroy_process_group()
            sys.exit(3)

    # ---- roofline of the dominant kernel ---------------------------------------------------------
    peak, bf16_peak, peak_src = hbm_peak()
    bytes_per_launch = local_rows * a.dim * 4          # SURVEY.md 8d: R*d*4; rows pre-normalised, no bitmap
    # average launch duration over the timed region: queries overlap (2 in flight), so it is the
    # region's device time divided by the scan launches in it -- fold, final select, the multi-GPU
    # exchange wait and every launch gap included
    launch_ms = ms_total / n_queries
    achieved = bytes_per_launch / (launch_ms * 1e-3) / 1e9
    scan_ms_avg = scan_ms / max(scan_n, 1)
    traffic = None
    ncu_path = os.path.join(ROOT, "profiles", "scan_ncu_summary.json")
    if os.path.exists(ncu_path):
        try:
            with open(ncu_path) as f:
                traffic = json.load(f).get("dram_bytes_per_launch_at_bench_shape", {}).get(str(local_rows * a.dim * 4))
        except Exception:  # noqa: BLE001
            traffic = None
    shadow = half_q * 2 >= n_queries      # the shadow scan answered (most of) the timed searches
    kernel = "mlv::scan_kernel<ip,NQ=1,R> (TMA ring scan + fused top-k, final select"
    moved = None
    if shadow:
        kernel = ("mlv::scan_kernel_half<ip,R> (TMA ring scan of the fp16 shadow of the rows + fused top-32, exact fp32 re-rank + "
                  "certificate in the last CTA; an fp32 scan_kernel launch queued behind it returns at once unless the certificate failed")
        ld16 = (a.dim + 7) // 8 * 8
        # what the pass actually reads: the halves, the 32 re-ranked fp32 rows, and the fp32 pass of every uncertified query
        moved = local_rows * ld16 * 2 + 32 * a.dim * 4 + (half_u / max(half_q, 1)) * bytes_per_launch
        traffic_key = "dram_bytes_per_launch_shadow_scan"
    else:
        traffic_key = "dram_bytes_per_launch_at_bench_shape"
    if os.path.exists(ncu_path):
        try:
            with open(ncu_path) as f:
                traffic = json.load(f).get(traffic_key, {}).get(str(local_rows * a.dim * 4))
        except Exception:  # noqa: BLE001
            traffic = None
    roofline = {
        "bound": "hbm", "kernel": kernel + (", peer-memory exchange" if searcher is not None else "") + ")",
        "achieved": achieved, "peak": peak, "unit": "GB/s",
        "frac": achieved / peak, "peak_source": peak_src + " hbm_gbs, copy read+write", "traffic": traffic,
        "bytes_per_launch": bytes_per_launch, "launches_timed": n_queries, "mean_launch_ms": launch_ms,
        "how": "algorithmic bytes (SURVEY 8d: rows * dim * 4, the fp32 matrix) per search / (timed-region device time / searches in it)"
               + ("; the shadow scan moves about half of them (bytes_moved_per_launch), so frac exceeds 1 by construction: "
                  "frac_of_bytes_moved is the fraction of the HBM peak the pass actually sustains" if shadow else ""),
        "bytes_moved_per_launch": moved,
        "frac_of_bytes_moved": (moved / (launch_ms * 1e-3) / 1e9 / peak) if moved else None,
        "shadow_scan": {"searches": int(half_q), "uncertified_rerun_in_fp32": int(half_u), "of_timed_searches": n_queries},
        "frac_of_nominal_8000": achieved / 8000.0,
        "one_query_in_flight": {"value": alone_steps * qps_step / (alone_ms / 1e3), "unit": UNIT,
                                "how": "the same searches strictly one after another on one stream (device-timed)"},
        "kernel_alone": {"mean_launch_ms": scan_ms_avg, "GBps": (bytes_per_launch / (scan_ms_avg * 1e-3) / 1e9) if scan_n else None,
                         "launches": scan_n, "share_of_its_step": (scan_ms / alone_ms) if scan_n else None,
                         "how": "CUDA events around every scan launch, one query in flight"},
    }
    api = ("GpuIndex" if searcher is None else "ShardedGpuIndex (one process per GPU)")
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
        "ms_per_step": ms_total / a.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "config": workload_config(a, world),
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": qps_step * a.dim * 4,
                "d2h_bytes_per_step": qps_step * (k * 12 + 4),
                "api": f"{api}.search_async(VectorDTO, top_k, namespace, metric).result() -> List[SearchResult], {e2e_depth} requests in flight",
                "one_request_at_a_time": {"value": e2e_sync_value, "unit": UNIT,
                                          "api": f"{api}.search(VectorDTO, top_k, namespace, metric) -> List[SearchResult]"}},
        "parity": parity, "roofline": roofline, "clocks": sampler.summary(), "gpu_launches": total_launches,
    }
    index.close()
    del Qd, outs
    torch.cuda.empty_cache()

    # ---- BASELINE configs 1-5 (after the headline region; failures are recorded, never fatal) -----------------------
    wanted = [] if a.configs == "none" else (["c1", "c2", "c3", "c4", "c5"] if a.configs == "all" else a.configs.split(","))
    if wanted:
        import bench_configs
        line["configs"] = bench_configs.run(ctx, a, wanted, peak, bf16_peak, peak_src)

    if rank == 0 and world == 1 and not a.no_cpu_baseline:
        base, _ = cpu_knn_qps(a, 1, 1, a.cpu_queries)
        line["cpu_baseline"] = base
    if rank == 0:
        emit_result(line)
    if world > 1:
        ctx.dist.destroy_process_group()


_RESULT_FD = None


def emit_result(line: dict) -> None:
    """THE one JSON line of the contract, on the process's original stdout."""
    text = json.dumps(line) + "\n"
    if _RESULT_FD is None:
        sys.stdout.write(text)
        sys.stdout.flush()
    else:
        os.write(_RESULT_FD, text.encode())


def main():
    # Libraries below us write to file descriptor 1 on their own (NCCL prints "NCCL version ..." there when
    # NCCL_DEBUG=VERSION is set in the environment): keep stdout for the result line, send the rest to stderr.
    global _RESULT_FD
    sys.stdout.flush()
    _RESULT_FD = os.dup(1)
    os.dup2(2, 1)
    a = parse_args()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)


if __name__ == "__main__":
    main()
