#!/usr/bin/env python
"""bench.py — BASELINE.json headline: queries/s (+ GB/s scanned) of single-query brute-force cosine search over
10M x 768 f32 vectors, sharded over N B200s, next to the reference's CPU path on the same box.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config all|c2|c3|c4|c5]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

A step = one query (BASELINE configs[1]: single-query streaming scan) answered over the WHOLE data set: every rank
scans its shard (10M/N rows, strong scaling); the shards' top-10 lists cross GPUs through peer-mapped buffers inside the merge
kernel (qb_comm.cu; consecutive steps are pipelined across GPUs), every rank ends up with the merged list.
  value  : queries/s with the query already resident in HBM (CUDA events on the launch stream, max over ranks)
  e2e    : the same through the public host API — qb_search_batch (N=1) / qb_multi_search_batch (N>1): host
           query in (H2D inside), host top-k out (D2H inside), wall clock, max over ranks.  The data set itself is
           resident state of the storage (uploaded once, like the reference's vectors in RAM), not a per-step input.
  roofline: the dominant kernel timed live with CUDA events on its stream (qb_profile_enable).  Shards of >= 2^19 rows are
           scanned through the int8 shadow plane (dense_q8_filter_kernel, qb_prefilter.cu) with exact rescoring — results
           bit-identical to the f32 scan, asserted inside the run; achieved = ALGORITHMIC bytes (rows_per_rank*768*4, SURVEY 8d)
           / avg launch time against MEASURED_PEAKS.json hbm_gbs, so it exceeds the peak; bytes_moved_per_launch /
           hbm_frac_of_bytes_moved describe the kernel's own traffic.  QB_DISABLE_PREFILTER=1 measures the f32 scan itself.
  cpu_baseline: the oracle's restatement of the reference's AVX2+FMA path (peek_top_iter loop) on this box's cores: the FULL
           10M rows per query when RAM allows (pinned threads, one first-touched segment each, oracle/mt.c).
`--impl reference` times only that CPU path and prints the same JSON shape.

The default run (`--config all`) prints ONE JSON line: the C2 headline fields above plus `configs.{c3,c4,c5}` — the other
BASELINE configs measured in the same process (each with value / e2e / roofline / parity / cpu_baseline): C3 10Mx768 SQ8 batch
1024 on the int8 tensor cores, C4 one 6.25M-row PQ shard per GPU, C5 HNSW M=16 ef=128 with the traversal on the device.
At N > 1 only the sharded configs (C2, C4) run.  --steps sets the number of timed steps of every config.

`--dump-outputs DIR` writes, after the timed steps, the top-k lists each config's timed path returned in its last timed step:
DIR/<config>_ids.npy (float64) and DIR/<config>_scores.npy (float32), [query, rank], -1 / NaN past a query's count.  Every
input is generated from fixed seeds, so two builds run with the same arguments can be compared output for output.  C5 is
left out: its graph comes from the multi-threaded builder, whose links depend on thread timing, so its lists vary from run
to run.
"""
from __future__ import annotations

import argparse
import concurrent.futures as cf
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_ROWS = 10_000_000
DIM = 768
TOP = 10
N_QUERIES = 100
CPU_SAMPLE_ROWS = 0          # 0 = the full data set when host RAM allows, else ~8 GB
METRIC = "queries/sec, 10Mx768 f32 brute-force cosine top-10, single query (GB/s scanned = value * 30.72)"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--rows", type=int, default=N_ROWS, help="total rows (debug only; the headline is 10M)")
    ap.add_argument("--dim", type=int, default=DIM)
    ap.add_argument("--cpu-sample-rows", type=int, default=CPU_SAMPLE_ROWS)
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--config", default="all", choices=["all", "c2", "c3", "c4", "c5"],
                    help="all = C2 headline + configs.{c3,c4,c5} in one line (default); cN = that config alone")
    ap.add_argument("--c5-rows", type=int, default=1_000_000, help="points of the HNSW index (BASELINE says 10M; the graph is built on the host cores inside the run)")
    ap.add_argument("--c5-queries", type=int, default=4096)
    ap.add_argument("--batch", type=int, default=1024, help="queries per batch (c3)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the results of the last timed step of each config as DIR/<name>.npy")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    return a


# the top-k lists each config's timed path returned in its last timed step (--dump-outputs)
OUTPUTS: dict[str, np.ndarray] = {}
OUTPUTS_MAX_BYTES = 64 << 20


def keep_lists(name: str, lists, top: int) -> None:
    """Per-query ScoredPointOffset lists -> [query, rank] ids (float64: exact for any row id) and scores (float32)."""
    ids = np.full((len(lists), top), -1.0, np.float64)
    scores = np.full((len(lists), top), np.nan, np.float32)
    for i, l in enumerate(lists):
        ids[i, : l.size] = l["idx"]
        scores[i, : l.size] = l["score"]
    OUTPUTS[name + "_ids"], OUTPUTS[name + "_scores"] = ids, scores


def device_lists(d_out, d_cnt):
    """The lists a qb_*_search_batch_device call left in (d_out, d_cnt); the caller has synchronised the device."""
    from qdrant_b200.scorer import SCORED_POINT_OFFSET

    rec = d_out.cpu().numpy().view(SCORED_POINT_OFFSET)
    cnt = d_cnt.cpu().numpy()
    return [rec[i, : cnt[i]] for i in range(rec.shape[0])]


def write_outputs(path: str) -> None:
    total = sum(a.nbytes for a in OUTPUTS.values())
    assert total <= OUTPUTS_MAX_BYTES, f"{total} bytes of outputs"
    os.makedirs(path, exist_ok=True)
    for name, a in OUTPUTS.items():
        np.save(os.path.join(path, name + ".npy"), a)


def ncu_traffic(name):
    """(bytes per launch, source) of the largest launch in a profiles/ summary: dram read + write."""
    try:
        best = None
        rd = None
        for ln in open(os.path.join(ROOT, "profiles", name)):
            f = ln.split()
            if len(f) >= 3 and f[0] == "dram__bytes_read.sum":
                rd = float(f[1]) * {"Gbyte": 1e9, "Mbyte": 1e6, "Kbyte": 1e3, "byte": 1.0}[f[2]]
            elif len(f) >= 3 and f[0] == "dram__bytes_write.sum" and rd is not None:
                tot = rd + float(f[1]) * {"Gbyte": 1e9, "Mbyte": 1e6, "Kbyte": 1e3, "byte": 1.0}[f[2]]
                best = tot if best is None or tot > best else best
                rd = None
        return best, ("profiles/" + name if best else None)
    except Exception:
        return None, None


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    def __init__(self, index: int):
        self.index, self.proc, self.lines, self.mark_at = index, None, [], 0

    def mark(self):
        """Call at the start of the timed region: only samples taken after this point are reported."""
        self.mark_at = len(self.lines)

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
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
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        lines = self.lines[self.mark_at:] or self.lines[-3:]   # a region shorter than one sampling period: nearest samples
        for l in lines:
            f = [x.strip() for x in l.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx = float(f[1])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------ CPU reference arm
def c2_config(rows: int, dim: int) -> dict:
    return {"workload": f"{rows}x{dim} f32 cosine brute-force, single query, top {TOP} (BASELINE configs[1])", "rows": rows, "dim": dim, "top": TOP}


def cpu_rows_that_fit(total_rows: int, dim: int, want: int) -> int:
    """The full data set when the host has the RAM for it (30.7 GB at 10M x 768), else ~8 GB of it."""
    if want:
        return min(want, total_rows)
    try:
        import psutil

        avail = psutil.virtual_memory().available
    except Exception:
        avail = 0
    full = total_rows * dim * 4
    if avail > full * 1.4 + (8 << 30):
        return total_rows
    return min(total_rows, max(100_000, (8 << 30) // (dim * 4)))


def cpu_reference_run(queries_pre: np.ndarray, steps: int, warmup: int, total_rows: int, dim: int, sample_rows: int = 0):
    """The reference's CPU path for C2 on this box's cores: T pinned threads, each owning (allocating, first-touching, scanning)
    one contiguous segment — one blocking task per segment, segments_searcher.rs:255 — every task the peek_top_iter loop of the
    oracle (AVX2+FMA dot, 64-id chunks, binary heap), lists merged on the host.  All of it inside oracle/mt.c: no Python per
    segment.  Rows are generated by the owning threads (seeded standard normal, cosine-preprocessed): same shape, dtype and
    distribution as the GPU arm's rows."""
    from oracle import oracle as o

    threads = os.cpu_count() or 1
    rows = cpu_rows_that_fit(total_rows, dim, sample_rows)
    pool = o.CpuPool(threads)
    t0 = time.perf_counter()
    pool.load_f32(rows, dim, o.COSINE, seed=42)
    load_s = time.perf_counter() - t0
    nq = queries_pre.shape[0]
    for i in range(warmup):
        pool.scan_f32(queries_pre[i % nq : i % nq + 1], TOP)
    t0 = time.perf_counter()
    for i in range(steps):
        res = pool.scan_f32(queries_pre[i % nq : i % nq + 1], TOP)
    dt = (time.perf_counter() - t0) / steps
    assert res[0].size == TOP and np.all(res[0]["score"][:-1] >= res[0]["score"][1:])
    pool.close()
    # one thread, one segment (how the reference scans a single segment): the many-thread figure must be a multiple of it
    one = o.CpuPool(1)
    r1 = min(rows, 400_000)
    one.load_f32(r1, dim, o.COSINE, seed=42)
    one.scan_f32(queries_pre[:1], TOP)
    t0 = time.perf_counter()
    for i in range(3):
        one.scan_f32(queries_pre[i % nq : i % nq + 1], TOP)
    dt1 = (time.perf_counter() - t0) / 3
    one.close()
    gbs, gbs1 = rows * dim * 4 / dt / 1e9, r1 * dim * 4 / dt1 / 1e9
    scale = total_rows / rows
    out = {"value": 1.0 / (dt * scale), "unit": "queries/s", "cores": threads, "kind": "port", "threads": threads,
           "rows_scanned_per_query": rows, "same_config": rows == total_rows, "ms_per_scan": dt * 1e3, "gb_per_s": gbs, "gb_per_s_1thread": gbs1,
           "speedup_vs_1thread": gbs / gbs1, "load_s": load_s,
           "sample": (f"{'the full' if rows == total_rows else 'first'} {rows} of {total_rows} rows x {dim} f32, {steps} single-query scans, {threads} pinned threads each "
                      f"scanning its own first-touched segment (oracle/mt.c) + host merge: {dt * 1e3:.1f} ms/scan = {gbs:.1f} GB/s ({gbs / gbs1:.1f}x the 1-thread "
                      f"{gbs1:.1f} GB/s)" + ("" if rows == total_rows else f", extrapolated linearly to {total_rows} rows"))}
    if threads >= 8 and gbs < 4 * gbs1:
        out["note"] = f"{threads}-thread scan is only {gbs / gbs1:.1f}x one thread: host DRAM bandwidth (not cores) bounds this arm"
    return out


def main_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    from oracle import oracle as o

    o.ensure_built()
    q = np.random.default_rng(43).standard_normal((N_QUERIES, args.dim)).astype(np.float32)
    qp = np.stack([o.preprocess_f32(o.COSINE, x) for x in q])
    W = max(args.warmup, 3)
    r = cpu_reference_run(qp, args.steps, W, args.rows, args.dim, args.cpu_sample_rows)
    ms = 1e3 / r["value"]
    line = {"impl": "reference", "metric": METRIC, "value": r["value"], "unit": "queries/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": W,
            "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": c2_config(args.rows, args.dim),
            "cpu_baseline": r,
            "e2e": {"value": r["value"], "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gb_per_s_scanned": r["gb_per_s"]}
    print(json.dumps(line))
    return 0


# ------------------------------------------------------------------------------------------------ GPU arm
def dist_ctx():
    """(world, rank, local_rank, device); initialises the NCCL process group once under torchrun."""
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl ours needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1 and not dist.is_initialized():
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    return world, rank, local_rank, dev


def main_ours(args):
    """C2, the headline.  Returns the JSON line as a dict on rank 0 (None elsewhere)."""
    import torch
    import torch.distributed as dist

    world, rank, local_rank, dev = dist_ctx()

    from qdrant_b200 import scorer as qb
    from qdrant_b200._capi import lib
    from qdrant_b200.sharded import ShardedSegmentSearcher, shard_ranges

    b, e = shard_ranges(args.rows, world)[rank]
    n_local = e - b
    # ---- synthetic data generated on the device, shard by shard (no 30 GB host copy); cosine => normalise like
    # Distance::preprocess_vector does at insert time (qb_metric_preprocess_device runs cosine_preprocess_avx arithmetic)
    st = qb.DenseVectorStorage(None, qb.Distance.Cosine, count=n_local, dim=args.dim, device=local_rank)
    gen = torch.Generator(device=dev)
    gen.manual_seed(42 + rank)
    chunk = 500_000
    from qdrant_b200._capi import check, vp

    for r0 in range(0, n_local, chunk):
        n = min(chunk, n_local - r0)
        x = torch.randn((n, args.dim), generator=gen, device=dev, dtype=torch.float32)
        check(lib().qb_metric_preprocess_device(local_rank, int(qb.Distance.Cosine), args.dim, n, vp(x.data_ptr()), args.dim * 4))
        st.write_rows_device(r0, n, x.data_ptr(), args.dim * 4)
        del x
    torch.cuda.synchronize()
    torch.cuda.empty_cache()

    queries = np.random.default_rng(43).standard_normal((N_QUERIES, args.dim)).astype(np.float32)
    searcher = ShardedSegmentSearcher(st, id_base=b, top=TOP, max_queries=1, device=dev)
    d_all_q = torch.from_numpy(queries).to(dev)
    stream = searcher.stream

    def step_device(i):
        with torch.cuda.stream(stream):
            searcher.d_queries[:1].copy_(d_all_q[i % N_QUERIES : i % N_QUERIES + 1], non_blocking=True)
        searcher.search_device(1)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    W, K = max(args.warmup, 3), args.steps
    for i in range(W):
        step_device(i)
    barrier()
    # ---- timed region 1: device-resident queries, CUDA events on the launch stream
    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
        time.sleep(0.3)   # nvidia-smi start-up
    for i in range(3):
        step_device(i)       # every rank (collective inside): keep the GPUs under load while the first samples arrive
    barrier()
    if rank == 0:
        clocks.mark()
    st.profile(True)
    launches0 = int(lib().qb_kernel_launch_count())
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record(stream)
    for i in range(K):
        step_device(W + i)
    searcher.drain()         # N > 1: every step's exchange + merge (communicator stream) completes inside the timed region
    ev1.record(stream)
    barrier()
    dev_ms = ev0.elapsed_time(ev1)
    launches = int(lib().qb_kernel_launch_count()) - launches0
    n_prof, prof_ms = st.profile_read(reset=True)
    st.profile(False)
    clk = clocks.stop() if rank == 0 else None
    # sanity: the result of the last step must be a valid top-k
    last = searcher.results_host(1)[0]
    assert last.size == TOP and np.all(last["score"][:-1] >= last["score"][1:]), "invalid top-k from the timed region"
    keep_lists("c2", [last], TOP)

    # ---- timed region 2: end to end through the public host API (H2D query, D2H results inside)
    for i in range(3):
        searcher.search(queries[i : i + 1])
    barrier()
    t0 = time.perf_counter()
    for i in range(K):
        searcher.search(queries[(W + i) % N_QUERIES : (W + i) % N_QUERIES + 1])
    barrier()
    e2e_s = time.perf_counter() - t0

    t = torch.tensor([dev_ms, e2e_s * 1e3], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms, e2e_ms = float(t[0]), float(t[1])

    # ---- parity inside the bench (the driver sees it): every rank checks its shard's fused scan against the oracle on the very rows
    # the GPU holds (a prefix read back from HBM), and at N > 1 rank 0 re-merges the ranks' LOCAL lists on the host
    # (BatchResultAggregator restated in numpy) and compares with what the device exchange + merge produced.
    parity = {"checked": False}
    if not args.no_cpu:
        from oracle import oracle as o
        from qdrant_b200.sharded import merge_topk_host

        rows = min(200_000, n_local)
        ids = np.arange(rows, dtype=np.uint32) + np.uint32(b)
        base = st.get_dense(ids)
        qp0 = o.preprocess_f32(o.COSINE, queries[0])
        got = st.search_batch(queries[0], TOP, id_list=ids)[0]
        want = o.scan_f32(o.COSINE, base, qp0[None], TOP)[0]
        assert np.array_equal(got["score"].view(np.uint32), want["score"].view(np.uint32)), "bench parity spot-check failed: GPU scan != oracle scan"
        assert np.array_equal(got["idx"], want["idx"] + np.uint32(b))
        parity = {"checked": True, "rows_checked_per_rank": rows, "scan_vs_oracle": "bit-exact"}
        if world > 1:
            with torch.cuda.stream(stream):
                searcher.d_queries[:1].copy_(d_all_q[:1], non_blocking=True)      # on the storage's stream: ordered before the scan
            searcher.search_device(1)
            merged = searcher.results_host(1)[0]
            local = st.search_batch(queries[0], TOP)[0]          # this rank's own top-k through the plain C-ABI call (global ids)
            gathered = [None] * world
            dist.all_gather_object(gathered, local)
            if rank == 0:
                want_m = merge_topk_host(gathered, TOP)
                assert np.array_equal(merged, want_m), "sharded search != host merge of the shards' lists"
                parity["sharded_equals_merge_of_shards"] = True
    searches, reruns = st.search_stats()
    assert reruns == 0, f"{reruns} fallback reruns in the C2 path"
    # single-query searches on >= 2^19 rows stream the bf16 shadow plane and re-score the survivors exactly (qb_prefilter.cu): the timed path
    # must return what the exact f32 scan returns, bit for bit, on the whole shard
    prefilter = n_local >= (1 << 19) and not os.environ.get("QB_DISABLE_PREFILTER")
    plane_q8 = prefilter and os.environ.get("QB_PREFILTER_PLANE", "0") != "1" and args.dim <= 1024   # int8 codes + per-row scale, else bf16
    if prefilter:
        from qdrant_b200.scorer import set_option
        fast = [st.search_batch(queries[i], TOP)[0] for i in range(3)]
        set_option("disable_prefilter", 1)
        slow = [st.search_batch(queries[i], TOP)[0] for i in range(3)]
        set_option("disable_prefilter", 0)
        for a_, b_ in zip(fast, slow):
            assert np.array_equal(a_["idx"], b_["idx"]) and np.array_equal(a_["score"].view(np.uint32), b_["score"].view(np.uint32)), \
                "C2: the bf16-prefilter path differs from the exact f32 scan"
        assert st.search_stats()[1] == 0, "C2: the prefilter fell back to the exact scan"
        parity["prefilter_equals_exact_scan"] = f"bit-exact on 3 queries x {n_local} rows"
    exchange = {"peer": "peer-mapped buffers over NVLink, fused into the merge kernel; steps pipelined (window 2): merge of step i overlaps the scan of step i+1", "nccl": "NCCL all-gather", "none": "single GPU"}[searcher.exchange]
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        qp = np.stack([o.preprocess_f32(o.COSINE, x) for x in queries])
        cpu = cpu_reference_run(qp, steps=5, warmup=2, total_rows=args.rows, dim=args.dim, sample_rows=args.cpu_sample_rows)

    line = None
    if rank == 0:
        peak, peak_src = peaks()
        qps = K / (dev_ms / 1e3)
        algo_bytes = n_local * args.dim * 4
        kern_ms = prof_ms / max(n_prof, 1)
        achieved = algo_bytes / (kern_ms / 1e3) / 1e9 if n_prof else None
        # dram__bytes_read.sum + dram__bytes_write.sum of this kernel's main pass from the committed `ncu --set full` capture; it
        # was taken on the 10M x 768 single-GPU workload, so it is only quoted for that shape
        traffic, traffic_src = ncu_traffic(("ncu_q8_filter_kernel_r02.txt" if plane_q8 else "ncu_bf16_filter_kernel_r02.txt") if prefilter else "ncu_stream_kernel_r01_localk.txt") if (n_local == 10_000_000 and args.dim == 768) else (None, None)
        line = {
            "metric": METRIC, "value": qps, "unit": "queries/s", "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": dev_ms / K,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": ("f32 results (exact reference arithmetic); the scan itself runs on an " + ("int8" if plane_q8 else "bf16") + " shadow plane and re-scores the survivors in f32") if prefilter else "f32",
            "data": "synthetic",
            "config": dict(c2_config(args.rows, args.dim), rows_per_gpu=n_local, parallelism=f"row-sharded x{world}, top-k exchange ({exchange}) + device merge",
                           l2="inputs larger than L2 (shard = %.1f GB >> 126 MB), no flush needed" % (algo_bytes / 1e9)),
            "gb_per_s_scanned": qps * args.rows * args.dim * 4 / 1e9,
            "e2e": {"value": K / (e2e_ms / 1e3), "unit": "queries/s", "h2d_bytes_per_step": args.dim * 4, "d2h_bytes_per_step": TOP * 8 + 4,
                    "ms_per_step": e2e_ms / K},
            "gpu_launches": launches,
            "clocks": clk,
            "roofline": {"bound": "hbm", "kernel": (("dense_q8_filter_kernel (the scan reads the int8 shadow plane: 1 byte per element + 16 bytes per row for its scale; "
                                                     if plane_q8 else "dense_bf16_filter_kernel (the scan reads the bf16 shadow plane: 2 bytes per element; ") +
                                                    "exact f32 sample scan before, exact rescoring of the survivors after)") if prefilter else "dense_f32_stream_kernel (main pass)",
                         "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": (achieved / peak) if achieved else None, "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": algo_bytes, "avg_launch_ms": kern_ms, "launches_timed": n_prof},
        }
        if prefilter and n_prof:
            # algorithmic bytes (SURVEY 8d: dim x 4 per row) / time exceeds the HBM peak because the kernel moves half of them
            moved = n_local * (((args.dim + 15) // 16) * 16 + 16) if plane_q8 else algo_bytes // 2
            line["roofline"]["bytes_moved_per_launch"] = moved
            line["roofline"]["hbm_frac_of_bytes_moved"] = moved / (kern_ms / 1e3) / 1e9 / peak
            line["roofline"]["note"] = ("achieved = algorithmic f32 bytes / kernel time; the kernel itself streams the shadow plane (bytes_moved_per_launch) at "
                                        "hbm_frac_of_bytes_moved of the measured copy peak; results are bit-identical to the f32 scan (parity.prefilter_equals_exact_scan)")
        line["parity"] = parity
        line["fallback_reruns"] = reruns
        if cpu is not None:
            line["cpu_baseline"] = cpu
    # ---- the same storage, 1024 f32 queries at once (north_star: "batched multi-query x segment scoring on tensor cores"): bf16 tcgen05
    # prefilter + exact rescoring.  Reported as configs.f32_batch of the default line.
    if rank == 0 and world == 1 and getattr(args, "with_f32_batch", False):
        line["_f32_batch"] = f32_batch_on(st, args, dev)
    # orderly teardown: torch tensors / streams first, then the storage (the process group outlives this config)
    searcher.close()
    del searcher, d_all_q
    torch.cuda.synchronize()
    st.close()
    torch.cuda.empty_cache()
    return line if rank == 0 else None


def f32_batch_on(st, args, dev):
    """1024-query f32 batches over the C2 storage: device-timed steps, host-API steps, tensor-core == CUDA-core lists, no fallback rerun."""
    import torch

    from qdrant_b200 import scorer as qb
    from qdrant_b200._capi import check, lib, vp

    nq, top = args.batch, TOP
    queries = np.random.default_rng(46).standard_normal((nq, args.dim)).astype(np.float32)
    d_q = torch.from_numpy(queries).to(dev)
    d_out = torch.empty((nq, top), dtype=torch.int64, device=dev); d_cnt = torch.empty((nq,), dtype=torch.int32, device=dev)
    stream = torch.cuda.ExternalStream(st.stream_ptr(), device=dev)

    def step():
        check(lib().qb_search_batch_device(st._h, vp(d_q.data_ptr()), nq, top, vp(d_out.data_ptr()), vp(d_cnt.data_ptr())))

    for _ in range(3):
        step()                                   # the first one builds the bf16 shadow plane
    torch.cuda.synchronize()
    st.search_stats(reset=True); st.profile_read(reset=True); st.profile(True)
    launches0 = int(lib().qb_kernel_launch_count())
    K = args.steps
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(stream)
    for _ in range(K):
        step()
    ev1.record(stream)
    torch.cuda.synchronize()
    dev_ms = ev0.elapsed_time(ev1)
    launches = int(lib().qb_kernel_launch_count()) - launches0
    n_prof, prof_ms = st.profile_read(reset=True)
    st.profile(False)
    keep_lists("f32_batch", device_lists(d_out, d_cnt), top)
    t0 = time.perf_counter()
    for _ in range(K):
        res = st.search_batch(queries, top)
    e2e_ms = (time.perf_counter() - t0) * 1e3 / K
    searches, reruns = st.search_stats(reset=True)
    assert reruns == 0, f"f32 batch: {reruns} fallback reruns"
    qb.set_option("disable_mma", 1)
    try:
        res_cc = st.search_batch(queries[:32], top)
    finally:
        qb.set_option("disable_mma", 0)
    for a_, b_ in zip(res[:32], res_cc):
        assert np.array_equal(a_, b_), "f32 batch: tensor-core prefilter path and CUDA-core path disagree"
    try:
        peak = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["bf16_tflops"]); peak_src = "measured (MEASURED_PEAKS.json bf16_tflops)"
    except Exception:
        peak, peak_src = 2250.0, "fallback (nominal dense bf16)"
    n = st.count
    flops = 2.0 * nq * n * args.dim
    kern_ms = prof_ms / max(n_prof, 1)
    ach = flops / (kern_ms / 1e3) / 1e12 if n_prof else None
    return {"metric": f"queries/sec, {n}x{args.dim} f32 cosine brute-force top-{top}, batch={nq}, bf16 tensor-core prefilter + exact rescoring", "value": nq * K / (dev_ms / 1e3),
            "unit": "queries/s", "n_gpus": 1, "steps": K, "warmup": 3, "ms_per_step": dev_ms / K, "higher_is_better": True, "dtype": "f32 (bf16 prefilter, f32 exact rescoring)",
            "data": "synthetic", "config": {"workload": f"{n}x{args.dim} f32 cosine, batch={nq}", "rows": n, "dim": args.dim, "batch": nq},
            "e2e": {"value": nq / (e2e_ms / 1e3), "unit": "queries/s", "h2d_bytes_per_step": nq * args.dim * 4, "d2h_bytes_per_step": nq * top * 8 + nq * 4, "ms_per_step": e2e_ms},
            "gpu_launches": launches,
            "roofline": {"bound": "tensor", "kernel": "sq8_mma_kernel<1,1> (tcgen05.mma kind::f16 prefilter) + f32_rescore_kernel, main pass", "achieved": ach, "peak": peak, "unit": "TFLOP/s",
                         "frac": (ach / peak) if ach else None, "traffic": None, "peak_source": peak_src, "avg_launch_ms": kern_ms, "launches_timed": n_prof,
                         "algorithmic_flops_per_launch": flops},
            "parity": {"checked": True, "tensor_core_equals_cuda_core": "bit-exact on 32 queries x all rows", "fallback_reruns": reruns}}


# ------------------------------------------------------------------------------------------------ C3: batched SQ8 (1 GPU)
def main_c3(args):
    """BASELINE configs[2]: 10M x 768 SQ8 cosine, batch = 1024 queries, int8 tensor-core GEMM scorer, 1 GPU.
    A step = one 1024-query batch over the whole segment.  Not the default bench line (that is c2)."""
    import torch

    from qdrant_b200 import scorer as qb
    from qdrant_b200._capi import check, lib, vp

    dev = torch.device("cuda", 0)
    torch.cuda.set_device(0)
    n, dim, nq, top = args.rows, args.dim, args.batch, TOP
    ad = dim + (16 - dim % 16) % 16
    chunk = 500_000

    def gen_chunk(i, cn):
        g = torch.Generator(device=dev)
        g.manual_seed(1000 + i)
        x = torch.randn((cn, dim), generator=g, device=dev, dtype=torch.float32)
        check(lib().qb_metric_preprocess_device(0, int(qb.Distance.Cosine), dim, cn, vp(x.data_ptr()), dim * 4))
        return x

    mn, mx = float("inf"), float("-inf")
    for i, r0 in enumerate(range(0, n, chunk)):
        x = gen_chunk(i, min(chunk, n - r0))
        a, b = torch.aminmax(x)
        mn, mx = min(mn, float(a)), max(mx, float(b))
        del x
    alpha, offset = np.float32((np.float32(mx) - np.float32(mn)) / np.float32(127.0)), np.float32(mn)
    multiplier = np.float32(alpha * alpha)
    rows = torch.empty((n, 4 + ad), dtype=torch.uint8, device=dev)
    for i, r0 in enumerate(range(0, n, chunk)):
        cn = min(chunk, n - r0)
        x = gen_chunk(i, cn)
        # EncodedVectorsU8::encode on the device (qb_sq8_encode_rows_device), straight into the storage's row format
        qb.sq8_encode_rows(x.data_ptr(), cn, dim, alpha, offset, qb.Distance.Cosine, rows[r0:].data_ptr())
        if i == 0 and not args.no_cpu:
            from oracle import oracle as o

            torch.cuda.synchronize()
            want = o.SQ8.encode(x[:2000].cpu().numpy(), o.QD_DOT, False, alpha=alpha, offset=offset)
            assert np.array_equal(rows[:2000].cpu().numpy(), want.rows), "bench parity spot-check failed: device SQ8 encode != oracle encode"
        torch.cuda.synchronize()
        del x
    torch.cuda.synchronize()
    st = qb.ScalarQuantizedVectors(None, dim, float(alpha), float(offset), float(multiplier), qb.Distance.Cosine, rows_ptr=rows.data_ptr(), count=n)
    sample_rows = min(65536, n)
    h_sample = rows[:sample_rows].cpu().numpy()
    del rows
    torch.cuda.empty_cache()

    queries = np.random.default_rng(44).standard_normal((nq, dim)).astype(np.float32)
    stream = torch.cuda.ExternalStream(st.stream_ptr(), device=dev)
    d_q = torch.from_numpy(queries).to(dev)
    d_out = torch.empty((nq, top), dtype=torch.int64, device=dev)
    d_cnt = torch.empty((nq,), dtype=torch.int32, device=dev)

    def step_device():
        check(lib().qb_search_batch_device(st._h, vp(d_q.data_ptr()), nq, top, vp(d_out.data_ptr()), vp(d_cnt.data_ptr())))

    W, K = max(args.warmup, 3), args.steps
    for _ in range(W):
        step_device()
    torch.cuda.synchronize()
    st.profile(True)
    launches0 = int(lib().qb_kernel_launch_count())
    clocks = ClockSampler(0)
    clocks.start()
    time.sleep(0.3)
    for _ in range(2):
        step_device()
    torch.cuda.synchronize()
    clocks.mark()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(stream)
    for _ in range(K):
        step_device()
    ev1.record(stream)
    torch.cuda.synchronize()
    dev_ms = ev0.elapsed_time(ev1)
    launches = int(lib().qb_kernel_launch_count()) - launches0
    n_prof, prof_ms = st.profile_read(reset=True)
    st.profile(False)
    clk = clocks.stop()
    keep_lists("c3", device_lists(d_out, d_cnt), top)
    for _ in range(2):
        st.search_batch(queries, top)
    t0 = time.perf_counter()
    for _ in range(K):
        res = st.search_batch(queries, top)
    e2e_ms = (time.perf_counter() - t0) * 1e3
    searches, reruns = st.search_stats(reset=True)
    assert reruns == 0, f"C3: {reruns} fallback reruns in {searches} searches — the tensor-core fast path did not produce these results"
    # the tensor-core path must agree with the lane-exact CUDA-core path (bit-exact), on a slice of the batch
    qb.set_option("disable_mma", 1)
    try:
        res_cc = st.search_batch(queries[:48], top)
    finally:
        qb.set_option("disable_mma", 0)
    for a, b in zip(res[:48], res_cc):
        assert np.array_equal(a, b), "tensor-core and CUDA-core SQ8 paths disagree"
    parity = {"checked": True, "tensor_core_equals_cuda_core": "bit-exact on 48 queries x all rows", "fallback_reruns": reruns}

    cpu = None
    if not args.no_cpu:
        from oracle import oracle as o

        meta = o.SQ8Meta(dim, ad, float(alpha), float(offset), float(multiplier), o.QD_DOT, 0)
        sq = o.SQ8(meta, h_sample)
        enc = [sq.encode_query(o.preprocess_f32(o.COSINE, q)) for q in queries]
        codes = np.ascontiguousarray(np.stack([e[0] for e in enc])); offs = np.array([e[1] for e in enc], np.float32)
        # oracle == GPU on the sample rows (same codes, same query encodings): bit-exact scores
        want = sq.scan(codes[:8], offs[:8], top)
        got = st.search_batch(queries[:8], top, id_list=np.arange(sample_rows, dtype=np.uint32))
        for a_, b_ in zip(got, want):
            assert np.array_equal(a_["score"].view(np.uint32), b_["score"].view(np.uint32)), "C3 parity spot-check failed: GPU SQ8 scan != oracle"
        parity["scan_vs_oracle"] = f"bit-exact on 8 queries x {sample_rows} rows"
        pool = o.CpuPool()
        pool.scan_sq8(meta, h_sample, codes, offs, top)
        t0 = time.perf_counter()
        reps = 3
        for _ in range(reps):
            pool.scan_sq8(meta, h_sample, codes, offs, top)
        dt = (time.perf_counter() - t0) / reps
        threads = pool.threads
        pool.close()
        cpu = {"value": nq / (dt * n / sample_rows), "unit": "queries/s", "cores": threads, "kind": "reference+port",
               "sample": f"{sample_rows} of {n} rows x {nq} queries: impl_score_dot_avx arithmetic + postprocess + heap (oracle qo_scan_sq8), {threads} pinned threads over row "
                         f"segments (oracle/mt.c), {dt*1e3:.0f} ms per sample batch, extrapolated linearly to {n} rows (compute-bound: every row meets every query)"}
    # MEASURED_PEAKS.json has no int8 figure (its tensor number is cuBLAS bf16, 1645.8 TF/s); the denominator here is the stricter
    # one: the tcgen05.mma kind::i8 issue rate measured on this pool by tools/mma_rate.cu (8190 MAC/clk/SM x 148 SMs x 1.965 GHz)
    peak_i8 = 4539.0
    try:
        for ln in open(os.path.join(ROOT, "profiles", "mma_rate_r01.jsonl")):
            r = json.loads(ln)
            if r.get("kind") == "i8" and r.get("n") == 256:
                peak_i8 = float(r["chip_tera_ops_per_s"])
                break
    except Exception:
        pass
    ops = 2.0 * nq * n * ad
    kern_ms = prof_ms / max(n_prof, 1)
    achieved = ops / (kern_ms / 1e3) / 1e12 if n_prof else None
    line = {"metric": f"queries/sec, {n}x{dim} SQ8 cosine brute-force top-{top}, batch={nq} (BASELINE configs[2])", "value": nq * K / (dev_ms / 1e3), "unit": "queries/s",
            "n_gpus": 1, "steps": K, "warmup": W, "ms_per_step": dev_ms / K, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u8 (s32 accumulate)",
            "data": "synthetic", "config": {"workload": f"{n}x{dim} SQ8 cosine, batch={nq}, int8 tensor-core GEMM scorer + fused top-{top}", "rows": n, "dim": dim, "batch": nq,
                                            "l2": "code plane 7.68 GB >> 126 MB L2"},
            "e2e": {"value": nq * K / (e2e_ms / 1e3), "unit": "queries/s", "h2d_bytes_per_step": nq * dim * 4, "d2h_bytes_per_step": nq * top * 8 + nq * 4, "ms_per_step": e2e_ms / K},
            "gpu_launches": launches, "clocks": clk,
            "roofline": {"bound": "tensor", "kernel": "sq8_mma_kernel (tcgen05.mma kind::i8, main pass)", "achieved": achieved, "peak": peak_i8, "unit": "TOP/s",
                         "frac": (achieved / peak_i8) if achieved else None, "traffic": None,
                         "peak_source": "measured tcgen05.mma kind::i8 issue rate (profiles/mma_rate_r01.jsonl, tools/mma_rate.cu); MEASURED_PEAKS.json holds no int8 figure "
                                        "(2 x its cuBLAS bf16 number would be 3291.6)", "avg_launch_ms": kern_ms,
                         "launches_timed": n_prof, "algorithmic_ops_per_launch": ops}}
    line["parity"] = parity
    if cpu:
        line["cpu_baseline"] = cpu
    st.close()
    del d_q, d_out, d_cnt
    torch.cuda.empty_cache()
    return line


# ------------------------------------------------------------------------------------------------ C4: PQ LUT scorer
def main_c4(args):
    """BASELINE configs[3]: 50M x 1536 PQ (m=96, 256 centroids), batch = 256, rows sharded over 8 GPUs.  Each rank holds
    50M/8 = 6.25M rows; with --gpus 1 this measures ONE such shard (1/8 of the job) and says so.  Codes and centroids are
    random (scoring cost does not depend on their values; parity is covered by tests/test_gpu_quant.py)."""
    import torch
    import torch.distributed as dist

    from qdrant_b200 import scorer as qb
    from qdrant_b200._capi import check, lib, vp
    from qdrant_b200.sharded import ShardedSegmentSearcher

    world, rank, local_rank, dev = dist_ctx()
    total_rows, dim, chunk, nq, top = 50_000_000, 1536, 16, 256, TOP
    if args.rows != N_ROWS:
        total_rows = args.rows
    n_local = total_rows // 8   # one of eight shards per rank, whatever N is
    m = dim // chunk
    rng = np.random.default_rng(100 + rank)
    codes = rng.integers(0, 256, (n_local, m), dtype=np.uint8)
    cents = np.random.default_rng(7).standard_normal((256, dim)).astype(np.float32) * 0.05
    st = qb.ProductQuantizedVectors(codes, cents, chunk, dim, qb.Distance.Dot, device=local_rank)
    sample_rows = min(200_000, n_local)
    h_sample = np.ascontiguousarray(codes[:sample_rows])
    del codes
    queries = np.random.default_rng(45).standard_normal((nq, dim)).astype(np.float32)
    searcher = ShardedSegmentSearcher(st, id_base=rank * n_local, top=top, max_queries=nq, device=dev)
    searcher.d_queries.copy_(torch.from_numpy(queries).to(dev))
    torch.cuda.synchronize()          # the copy ran on torch's stream, the searches run on the storage's
    W, K = max(args.warmup, 3), args.steps

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(W):
        searcher.search_device(nq)
    barrier()
    st.profile(True)
    launches0 = int(lib().qb_kernel_launch_count())
    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
        time.sleep(0.3)
        clocks.mark()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record(searcher.stream)
    for _ in range(K):
        searcher.search_device(nq)
    searcher.drain()                 # N > 1: the last steps' exchange + merge (communicator stream) are inside the timed region
    ev1.record(searcher.stream)
    barrier()
    dev_ms = ev0.elapsed_time(ev1)
    launches = int(lib().qb_kernel_launch_count()) - launches0
    n_prof, prof_ms = st.profile_read(reset=True)
    st.profile(False)
    clk = clocks.stop() if rank == 0 else None
    keep_lists("c4", searcher.results_host(nq), top)
    for _ in range(2):
        searcher.search(queries)
    barrier()
    t0 = time.perf_counter()
    for _ in range(K):
        searcher.search(queries)
    barrier()
    e2e_ms = (time.perf_counter() - t0) * 1e3
    t = torch.tensor([dev_ms, e2e_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms, e2e_ms = float(t[0]), float(t[1])
    searches, reruns = st.search_stats(reset=True)
    # the timed path (sixteen queries per gather through u8 tables + exact rescoring) against the single-query f32 kernel, all rows
    from qdrant_b200.scorer import set_option
    fast = st.search_batch(queries[:24], top)
    set_option("pq_queries_per_pass", 1)
    slow = st.search_batch(queries[:24], top)
    set_option("pq_queries_per_pass", 0)
    for a_, b_ in zip(fast, slow):
        assert np.array_equal(a_["idx"], b_["idx"]) and np.array_equal(a_["score"].view(np.uint32), b_["score"].view(np.uint32)), \
            "C4: the batched prefilter + rescoring path differs from the single-query f32 kernel"
    st.search_stats(reset=True)
    parity, cpu = {"checked": False, "fallback_reruns": reruns, "batched_equals_single_query_kernel": f"bit-exact on 24 queries x {n_local} rows"}, None
    if rank == 0 and not args.no_cpu:
        from oracle import oracle as o

        pq = o.PQ(dim, chunk, cents, h_sample, o.QD_DOT, False)
        luts = np.ascontiguousarray(np.stack([pq.encode_query(q).reshape(-1) for q in queries]))   # Dot: Metric::preprocess is the identity
        ids = np.arange(sample_rows, dtype=np.uint32) + np.uint32(rank * n_local)
        got = st.search_batch(queries[:4], top, id_list=ids)
        pool = o.CpuPool()
        want = pool.scan_pq(h_sample, 256, luts[:4], top)
        for a_, b_ in zip(got, want):
            assert np.array_equal(a_["score"].view(np.uint32), b_["score"].view(np.uint32)), "C4 parity spot-check failed: GPU PQ scan != oracle (LUT build + score_point_sse order)"
        parity.update({"checked": True, "scan_vs_oracle": f"bit-exact on 4 queries x {sample_rows} rows (device LUT build + scan)"})
        pool.scan_pq(h_sample, 256, luts, top)
        t0 = time.perf_counter()
        pool.scan_pq(h_sample, 256, luts, top)
        dt = time.perf_counter() - t0
        cpu = {"value": nq / (dt * n_local / sample_rows) , "unit": "queries/s", "cores": pool.threads, "kind": "port",
               "sample": f"{sample_rows} of {n_local} rows x {nq} queries: score_point_sse summation order + heap (oracle qo_scan_pq), {pool.threads} pinned threads over row segments, "
                         f"{dt*1e3:.0f} ms per sample batch, extrapolated linearly to one {n_local}-row shard (per-GPU figure; x{world} shards for the whole job)"}
        pool.close()
    line = None
    if rank == 0:
        lookups = float(nq) * n_local * m
        kern_ms = prof_ms / max(n_prof, 1)
        # shared-memory gather peak: 148 SMs x 32 banks x 4 B per clock at clocks.max.sm
        smem_peak_glookups = 148 * 32 * 1.965
        line = {"metric": f"queries/sec, {total_rows}x{dim} PQ(m={m},256) LUT scorer top-{top}, batch={nq}, {world} of 8 shards resident (BASELINE configs[3])",
                "value": nq * K / (dev_ms / 1e3), "unit": "queries/s", "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": dev_ms / K, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "u8 codes, f32 LUT sums", "data": "synthetic (random codes / centroids)",
                "config": {"workload": f"PQ m={m} chunk={chunk}, {n_local} rows per GPU (= 50M/8), batch={nq}", "rows_per_gpu": n_local, "dim": dim, "m": m, "batch": nq,
                           "l2": "code plane 600 MB per GPU > 126 MB L2"},
                "e2e": {"value": nq * K / (e2e_ms / 1e3), "unit": "queries/s", "h2d_bytes_per_step": nq * dim * 4, "d2h_bytes_per_step": nq * top * 8 + nq * 4, "ms_per_step": e2e_ms / K},
                "gpu_launches": launches, "clocks": clk,
                "roofline": {"bound": "smem-gather", "kernel": "pq16_prep_kernel + pq_scan16_kernel (sixteen queries per 16-byte gather through u8 tables, integer thresholds) + "
                                                               "pq_rescore_kernel (exact f32 sums of the survivors)", "achieved": (lookups / (kern_ms / 1e3) / 1e9) if n_prof else None,
                             "peak": smem_peak_glookups, "unit": "Glookup/s", "frac": (lookups / (kern_ms / 1e3) / 1e9 / smem_peak_glookups) if n_prof else None, "traffic": None,
                             "peak_source": "148 SMs x 32 banks x clocks.max.sm = one 4-byte table entry per bank per clock (the exact kernels' conflict-free gather rate, the "
                                            "denominator of rounds 1-2; no such figure in MEASURED_PEAKS.json).  A (row, query, chunk) lookup of the batched kernel moves ONE byte "
                                            "(sixteen queries share a 16-byte gather), so frac > 1 is possible; see frac_of_16B_gather_peak and profiles/ncu_pq16_kernel_r02.txt "
                                            "(shared-memory pipe 88 % busy, 9.6 wavefronts per LDS.128 on random codes where 4 is conflict-free)",
                             "frac_of_16B_gather_peak": (lookups / (kern_ms / 1e3) / 1e9 / (148 * 8 * 16 * 1.965)) if n_prof else None,
                             "avg_launch_ms": kern_ms, "launches_timed": n_prof, "hbm_gb_per_s": (float(nq) * n_local * m / (kern_ms / 1e3) / 1e9) if n_prof else None}}
        line["parity"] = parity
        if cpu:
            line["cpu_baseline"] = cpu
    searcher.close()
    del searcher
    torch.cuda.synchronize()
    st.close()
    torch.cuda.empty_cache()
    return line


# ------------------------------------------------------------------------------------------------ C5: HNSW, traversal on the device
def main_c5(args):
    """BASELINE configs[4]: HNSW (M=16, ef=128) graph search on the GPU scorer, recall@10 vs the CPU HNSW.
    The traversal itself runs on the device (qb_hnsw_search_batch: one persistent CTA per in-flight query, graph links in HBM);
    the CPU arm is the reference traversal (oracle/hnsw.c restating graph_layers.rs) on ALL host cores, one search per thread,
    over the SAME graph.  A step = one batch of --c5-queries queries.  The graph is built inside the run by the oracle's
    multi-threaded builder (the reference builds with rayon + per-point locks too), so the index size is bounded by build
    time: --c5-rows (default 1M of BASELINE's 10M) and the line says so."""
    import torch

    from oracle import oracle as o
    from qdrant_b200 import scorer as qb
    from qdrant_b200._capi import check, lib, vp

    dev = torch.device("cuda", 0)
    torch.cuda.set_device(0)
    n, dim, top, ef, nq = args.c5_rows, args.dim, TOP, 128, args.c5_queries
    threads = os.cpu_count() or 1
    # clustered synthetic data (1024 Gaussian clusters): i.i.d. Gaussian vectors in 768-d are the degenerate worst case for any
    # graph index (all points nearly equidistant, recall ~0.1), which says nothing about the scorer under test.  Generated on the
    # device, normalised with the reference's cosine preprocess, then copied to the host for the CPU builder.
    g = torch.Generator(device=dev); g.manual_seed(42)
    centers = torch.randn((1024, dim), generator=g, device=dev)
    base_d = torch.empty((n, dim), dtype=torch.float32, device=dev)
    for r0 in range(0, n, 250_000):
        cn = min(250_000, n - r0)
        idx = torch.randint(0, 1024, (cn,), generator=g, device=dev)
        x = centers[idx] + 0.5 * torch.randn((cn, dim), generator=g, device=dev)
        check(lib().qb_metric_preprocess_device(0, int(qb.Distance.Cosine), dim, cn, vp(x.data_ptr()), dim * 4))
        base_d[r0 : r0 + cn] = x
    qi = torch.randint(0, 1024, (nq,), generator=g, device=dev)
    queries = (centers[qi] + 0.5 * torch.randn((nq, dim), generator=g, device=dev)).cpu().numpy()
    base = base_d.cpu().numpy()
    st = qb.DenseVectorStorage(None, qb.Distance.Cosine, count=n, dim=dim)
    st.write_rows_device(0, n, base_d.data_ptr(), dim * 4)
    del base_d, centers
    torch.cuda.empty_cache()
    t0 = time.perf_counter()
    graph = o.HNSW(base, o.COSINE, m=16, ef_construct=100, seed=42, threads=threads)
    build_s = time.perf_counter() - t0
    entry, entry_level, m, m0 = graph.entry()
    hg = qb.HnswGraph(st, graph.export_plain(), m, m0)
    qp = o.preprocess_rows_f32(o.COSINE, queries)
    d_q = torch.from_numpy(queries).to(dev)
    d_out = torch.empty((nq, top), dtype=torch.int64, device=dev)
    d_cnt = torch.empty((nq,), dtype=torch.int32, device=dev)
    stream = torch.cuda.ExternalStream(st.stream_ptr(), device=dev)

    def step_device():
        check(lib().qb_hnsw_search_batch_device(hg._h, vp(d_q.data_ptr()), nq, top, ef, entry, entry_level, vp(d_out.data_ptr()), vp(d_cnt.data_ptr())))

    W, K = 3, args.steps
    for _ in range(W):
        step_device()
    torch.cuda.synchronize()
    hg.stats(reset=True)
    st.profile(True)
    launches0 = int(lib().qb_kernel_launch_count())
    clocks = ClockSampler(0)
    clocks.start(); time.sleep(0.3); clocks.mark()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(stream)
    for _ in range(K):
        step_device()
    ev1.record(stream)
    torch.cuda.synchronize()
    dev_ms = ev0.elapsed_time(ev1)
    launches = int(lib().qb_kernel_launch_count()) - launches0
    n_prof, prof_ms = st.profile_read(reset=True)
    st.profile(False)
    clk = clocks.stop()
    hops, evals = hg.stats(reset=True)
    hops /= K * nq; evals /= K * nq
    gpu = hg.search(queries, top, ef, entry, entry_level)
    t0 = time.perf_counter()
    for _ in range(K):
        gpu = hg.search(queries, top, ef, entry, entry_level)
    e2e_ms = (time.perf_counter() - t0) * 1e3
    # ---- CPU arm: the reference traversal with the CPU scorer, same graph, all cores (one search per thread at a time)
    graph.search_batch(qp[:256], top, ef, threads=threads)
    t0 = time.perf_counter()
    cpu = graph.search_batch(qp, top, ef, threads=threads)
    cpu_s = time.perf_counter() - t0
    t0 = time.perf_counter()
    graph.search_batch(qp[:128], top, ef, threads=1)
    cpu1_s = (time.perf_counter() - t0) / 128
    # ---- parity: identical lists (scores bit-equal; ids equal except inside equal-score runs) => recall difference 0
    same = sum(int(np.array_equal(a["score"].view(np.uint32), b["score"].view(np.uint32)) and
                   (np.array_equal(a["idx"], b["idx"]) or np.array_equal(np.sort(a["idx"]), np.sort(b["idx"])))) for a, b in zip(gpu, cpu))
    ne = min(nq, 500)
    exact = st.search_batch(queries[:ne], top)

    def recall(res):
        return float(np.mean([np.mean(r["score"] >= e["score"][-1]) for r, e in zip(res[:ne], exact)]))
    r_cpu, r_gpu = recall(cpu), recall(gpu)
    assert same == nq, f"C5: device traversal differs from the CPU traversal on {nq - same} of {nq} queries"
    assert abs(r_cpu - r_gpu) <= 1e-4
    peak, peak_src = peaks()
    kern_ms = prof_ms / max(n_prof, 1)
    algo_bytes = evals * nq * dim * 4      # every scored point is one dim*4-byte row read
    achieved = algo_bytes / (kern_ms / 1e3) / 1e9 if n_prof else None
    line = {"metric": f"queries/sec, HNSW M=16 ef={ef} top-{top}, {n}x{dim} cosine, traversal + scoring on the GPU (BASELINE configs[4]; {n} of its 10M points)",
            "value": nq * K / (dev_ms / 1e3), "unit": "queries/s", "n_gpus": 1, "steps": K, "warmup": W, "ms_per_step": dev_ms / K, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic (1024 Gaussian clusters)",
            "config": {"workload": f"HNSW graph search, {nq} concurrent queries per batch, {hops:.0f} hops / {evals:.0f} scored points per query", "rows": n, "dim": dim, "ef": ef, "m": m,
                       "batch": nq, "graph_build_s": build_s, "graph_build_threads": threads, "l2": f"vectors {n * dim * 4 / 1e9:.1f} GB >> 126 MB L2"},
            "e2e": {"value": nq * K / (e2e_ms / 1e3), "unit": "queries/s", "h2d_bytes_per_step": nq * dim * 4, "d2h_bytes_per_step": nq * top * 8 + nq * 4, "ms_per_step": e2e_ms / K},
            "gpu_launches": launches, "clocks": clk,
            "roofline": {"bound": "hbm", "kernel": "hnsw_search_kernel (random 3-KB row reads)", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": (achieved / peak) if achieved else None,
                         "traffic": None, "peak_source": peak_src, "algorithmic_bytes_per_launch": algo_bytes, "avg_launch_ms": kern_ms, "launches_timed": n_prof},
            "cpu_baseline": {"value": nq / cpu_s, "unit": "queries/s", "cores": threads, "kind": "port", "single_thread_qps": 1.0 / cpu1_s,
                             "sample": f"same {nq} queries, same graph, reference traversal + AVX2 f32 scorer (oracle/hnsw.c), {threads} threads each running one search at a time"},
            "parity": {"checked": True, "identical_result_lists": same, "of": nq, "recall_at_10": {"cpu_traversal": r_cpu, "gpu_traversal": r_gpu, "vs_exact_on": ne}},
            "recall_at_10": {"cpu_traversal": r_cpu, "gpu_traversal": r_gpu}}
    hg.close(); graph.close()
    del d_q, d_out, d_cnt
    st.close()
    torch.cuda.empty_cache()
    return line


def main_all(args):
    """Default run: C2 headline + configs.{c3,c4,c5} in ONE JSON line (rank 0)."""
    import torch.distributed as dist

    world, rank, _, _ = dist_ctx()
    if args.config == "all":
        args.with_f32_batch = True
    line = main_ours(args) if args.config in ("all", "c2") else None
    extras = {}
    if line is not None and "_f32_batch" in line:
        extras["f32_batch"] = line.pop("_f32_batch")
    if args.config == "all":
        small = args.rows != N_ROWS     # debug sizes: shrink the other configs along
        sub = argparse.Namespace(**vars(args))
        if small:
            sub.c5_rows = min(args.c5_rows, max(20_000, args.rows // 10)); sub.c5_queries = min(args.c5_queries, 512)
        if world == 1:
            extras["c3"] = main_c3(sub)
        extras["c4"] = main_c4(sub)
        if world == 1:
            extras["c5"] = main_c5(sub)
    elif args.config != "c2":
        line = {"c3": main_c3, "c4": main_c4, "c5": main_c5}[args.config](args)
    if rank == 0 and line is not None:
        if extras:
            line["configs"] = extras
        print(json.dumps(line))
    if rank == 0 and args.dump_outputs:
        write_outputs(args.dump_outputs)
    sys.stdout.flush()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        sys.exit(main_reference(a))
    sys.exit(main_all(a))
