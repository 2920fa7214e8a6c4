#!/usr/bin/env python
"""bench.py — kNN queries/sec + achieved HBM GB/s of the fused distance+top-k path (BASELINE.json metric).

    python bench.py --gpus 1 --steps K --warmup W                (default workload: "headline")
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...                          (the reference's CPU path, timed on host cores)
    python bench.py ... --dump-outputs DIR                        (+ the last timed step's indices / scores as DIR/*.npy)

A "step" = one batch of Q queries searched against the whole HBM-resident corpus (one pass of the hot path).
Workload "headline" = BASELINE.json's metric shape: N=10M x d=1024 fp32, k=10, with configs[1]'s Q=64 cosine.
Multi-GPU: the corpus is row-sharded over the ranks (rank g owns rows [g*N/G, (g+1)*N/G)), every rank scans its
shard with the same fused kernel, and the per-rank candidate lists (Q*k*8 B) cross GPUs by plain peer stores over
NVLink into IPC-mapped buffers (csrc/exchange.cu, behind the C ABI: nk_search_sharded_device) where a fused
wait+merge+decode kernel folds them with the same (score desc, row asc) rule — no NCCL on the data path (NCCL only
carries the barriers and the MAX-over-ranks of the timings).  Total work is fixed, so scaling is "strong".

One JSON line on stdout (rank 0).  `value` = device-resident throughput (queries already in HBM), `e2e` = the
same metric through the reference-facing C-ABI call with HOST buffers (H2D of the queries and D2H of the
results inside the timed region).  `roofline` is for the dominant kernel (the scan), timed with CUDA events
inside the library on the launching stream.  `cpu_baseline` = the oracle's AVX2 restatement of the reference's
pkg/simd brute force timed on this box's host cores, single-threaded (how the reference runs a query) and on all
cores, on a bounded >= 1 GB sample (N=1, rank 0 only).  `parity_check` = an UNTIMED post-check of the results of
this very run (planted neighbours, exact fp64 recomputation of every returned score, uniqueness / order, and for
N > 1 bit-equality with the in-process multi-device search).  `also` (default N=1 line) = the rest of the north_star grid
measured by the same rules: configs[1..3], Q=1, k=100, the fp32-row scans and the clustered corpus; on the default 8-GPU
line `also.c5` = configs[4] (N=100M, the one config that needs 8 GPUs), with its own parity_check."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (N_total, dim, dtype, Q, k, metric, description)
    "headline": (10_000_000, 1024, "f32", 64, 10, "cosine",
                 "N=10M d=1024 fp32 Q=64 k=10 cosine (BASELINE.json metric shape: d=1024 N=10M k=10; Q/metric of configs[1])"),
    "c2": (1_000_000, 1024, "f32", 64, 10, "cosine", "configs[1]: N=1M d=1024 (bge-m3) fp32 Q=64 k=10 cosine"),
    "c3": (10_000_000, 1024, "f32", 1024, 100, "dot", "configs[2]: N=10M d=1024 fp32 Q=1024 k=100 inner-product"),
    "c4": (10_000_000, 768, "f16", 1, 10, "euclidean", "configs[3]: N=10M d=768 fp16 Q=1 k=10 L2"),
    "c5": (100_000_000, 1024, "f32", 1024, 10, "cosine",
           "configs[4]: N=100M d=1024 fp32 Q=1024 k=10 cosine, row-sharded (needs >= 4 GPUs: 410 GB of corpus)"),
    "c1": (100_000, 128, "f32", 1, 10, "cosine", "configs[0]: N=100k d=128 fp32 Q=1 k=10 cosine"),
    "q1": (10_000_000, 1024, "f32", 1, 10, "cosine", "N=10M d=1024 fp32 Q=1 k=10 cosine (single-query latency)"),
    "clustered": (10_000_000, 1024, "f32", 64, 10, "cosine",
                  "N=10M d=1024 fp32 Q=64 k=10 cosine on the Gaussian-mixture corpus of SURVEY.md 8(d) (1000 centres, sigma=0.1)"),
}
CORPUS_SEED, QUERY_SEED = 42, 1337
SCAN_DESC = {
    "shadow": "filter scan streams the 16-bit image of the corpus (BF16 shadow of fp32 rows: +50% HBM held, half the bytes read; "
              "fp16/bf16 corpora in place); survivors re-scored exactly in fp32 from the stored rows: results identical to a full-precision scan",
    "filter": "1xTF32 filter scan over the fp32 rows + exact fp32 rescoring",
    "tensor": "exact 3xTF32 scan over the fp32 rows",
    "simt": "CUDA-core scan over the stored rows",
}
KERNEL_NAME = {"tensor": "knn_scan_tc_kernel<3> (tcgen05/TMEM/TMA, 3xTF32 exact)",
               "filter": "knn_scan_tc_kernel<1> (tcgen05/TMEM/TMA, 1xTF32 filter + exact fp32 rescoring)",
               "shadow": "knn_scan_shadow_kernel (tcgen05/TMEM/TMA over the 16-bit corpus image + exact fp32 rescoring)",
               "simt": "knn_scan_simt_kernel"}


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="headline", choices=sorted(WORKLOADS))
    ap.add_argument("--path", default="auto", choices=["auto", "simt", "tensor", "filter", "shadow"])
    ap.add_argument("--rows", type=int, default=0, help="override N_total (debug)")
    ap.add_argument("--k", type=int, default=0, help="override k (debug)")
    ap.add_argument("--q", type=int, default=0, help="override Q (debug)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-also", action="store_true", help="skip the secondary north_star-grid measurements")
    ap.add_argument("--no-parity", action="store_true", help="skip the untimed parity post-check")
    ap.add_argument("--exchange", default="peer", choices=["peer", "nccl"],
                    help="N>1 candidate exchange: peer-memory kernels behind the C ABI (default) or NCCL all-gather + merge")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the result of the last timed step to DIR/indices.npy (row ids, float64) and DIR/scores.npy "
                         "(float32), [Q x k]; inputs are seeded, so two builds can be compared output for output")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the GPU search's results: it needs --impl ours")
    return args


# ------------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self) -> dict:
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); pw.append(float(f[3]))
            except ValueError:
                continue
            for nm, val in zip(names, f[4:8]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(mx), "power_w_max": max(pw), "samples": len(sm),
                "reasons": sorted(reasons)}


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return json.load(open(p))
        except Exception:
            return None
    return None


def load_peaks():
    d = _peaks()
    if d and "hbm_gbs" in d:
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def load_tensor_peak(bf16=False):
    """Dense tensor TFLOP/s of the arithmetic the scan uses: BF16 / FP16 (16-bit path), or TF32 = half the bf16 figure
    (tf32 : bf16 = 1.1 : 2.25 PFLOP/s nominal, B200_PROFILING.md table).  Sustained, because the scan runs inside a
    long, power-capped step."""
    div = 1.0 if bf16 else 2.0
    what = "" if bf16 else " / 2: dense TF32 runs at half the bf16 rate"
    d = _peaks()
    if d and ("bf16_tflops_sustained" in d or "bf16_tflops" in d):
        return float(d.get("bf16_tflops_sustained", d.get("bf16_tflops"))) / div, \
            f"measured (MEASURED_PEAKS.json bf16_tflops_sustained{what})"
    return 1590.0 / div, f"fallback (B200_PROFILING.md 1.59 PFLOP/s bf16{what})"


def load_traffic(workload: str, path: str):
    """dram bytes per scan launch from the committed ncu --set full capture (profiles/traffic.json), or None."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return d.get(f"{workload}:{path}", d.get(workload))
        except Exception:
            return None
    return None


def scan_bytes(path: str, n: int, dim: int, dtype: str) -> int:
    """Algorithmic bytes ONE scan launch streams (DESIGN.md §3): the stored rows, or — shadow path over fp32 rows — their
    BF16 shadow (rows padded to 64 elements) plus the two per-row norm floats; a 16-bit corpus is scanned in place
    (+ 4 B/row of |x|^2)."""
    elem = 4 if dtype == "f32" else 2
    if path == "shadow":
        if dtype == "f32":
            return n * ((dim + 63) // 64 * 64) * 2 + n * 8
        return n * dim * 2 + n * 4
    return n * dim * elem


# ------------------------------------------------------------------------------------------------------
def cpu_reference_run(N_total, dim, dtype, Q, k, metric, budget_s=25.0, min_passes=5):
    """The reference's CPU brute force (oracle/simd_baseline.c: AVX2+FMA kernels in the simd.Batch* loop shape +
    bounded insertion top-k) on a bounded >= 1 GB sample of the workload: (i) single-threaded — how the reference
    executes a query (vector_index.go:330-342, no goroutine fan-out) — and (ii) all host threads (an upper bound the
    reference does not implement).  Threads pinned (OMP_PROC_BIND=close, set in main before libgomp starts); the
    median of >= 5 passes is reported.  Returns the JSON fields."""
    import numpy as np
    import oracle  # loads the liboracle.so that build() made; never recompiles it (the tree may be read-only)
    hw = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    # bounded sample: S rows of the same synthetic corpus (>= 1 GB of fp32 rows where the corpus is that large), Qs queries
    row_bytes = dim * 4
    S = min(N_total, max(131072, -(-(1 << 30) // row_bytes)))
    Qs = min(Q, 8)
    rows = oracle.fill_uniform(S, dim, CORPUS_SEED, dtype="f16" if dtype == "f16" else "f32")
    if dtype != "f32":
        rows = rows.astype(np.float32)  # the reference has no 16-bit path: widen once (pkg/simd is float32-only)
    q = oracle.fill_uniform(Qs, dim, QUERY_SEED)

    def timed(threads, nq, budget):
        oracle.simd_knn(rows, q[:1], k, metric, threads=threads)  # warm-up (page-in, thread pool)
        ts, t_start = [], time.perf_counter()
        while len(ts) < min_passes or (time.perf_counter() - t_start < budget and len(ts) < 15):
            t0 = time.perf_counter()
            oracle.simd_knn(rows, q[:nq], k, metric, threads=threads)
            ts.append(time.perf_counter() - t0)
            if time.perf_counter() - t_start > 2.5 * budget:
                break
        ts.sort()
        return ts[len(ts) // 2], len(ts), ts[0], ts[-1]

    # all-core: fastest of {all, 1/2} hardware threads (containers often report more logical CPUs than their quota)
    best = None
    for cand in sorted({hw, max(hw // 2, 1)}, reverse=True):
        med, n_p, lo, hi = timed(cand, Qs, budget_s * 0.25)
        if best is None or med < best[0]:
            best = (med, n_p, lo, hi, cand)
    med_all, n_all, lo_all, hi_all, threads = best
    # single thread: fewer queries per pass keep it inside the budget (the scan is linear in queries)
    q1n = 1 if S * row_bytes > (1 << 29) else Qs
    med_1, n_1, lo_1, hi_1 = timed(1, q1n, budget_s * 0.35)
    scale = N_total / S
    qps_all = Qs / (med_all * scale)
    qps_1 = q1n / (med_1 * scale)
    return {
        "value": qps_all, "unit": "queries/s", "cores": threads, "kind": "port",
        "sample": (f"{Qs} queries x first {S} rows ({S * row_bytes / 1e9:.2f} GB) of the same synthetic corpus (d={dim}); median of {n_all} "
                   f"passes = {med_all * 1e3:.1f} ms (min {lo_all * 1e3:.1f}, max {hi_all * 1e3:.1f}), scaled linearly to N={N_total}; AVX2+FMA "
                   f"-ffast-math restatement of pkg/simd (vek32) + insertion top-k, OpenMP over rows, {threads} of {hw} hardware "
                   f"threads, OMP_PROC_BIND=close"),
        "ms_per_pass": med_all * 1e3, "steps_timed": n_all,
        "single_thread": {"value": qps_1, "unit": "queries/s", "cores": 1,
                          "sample": f"{q1n} quer{'y' if q1n == 1 else 'ies'} x the same {S} rows, median of {n_1} passes = {med_1 * 1e3:.1f} ms "
                                    f"(min {lo_1 * 1e3:.1f}, max {hi_1 * 1e3:.1f}); this is how the reference executes one query "
                                    f"(pkg/search/vector_index.go:330-342: a single goroutine)"},
    }


# ------------------------------------------------------------------------------------------------------
class Runner:
    """One GPU rank: index + exchange context + the timed loops (shared by the headline and the `also` entries)."""

    def __init__(self, args, G, rank, local_rank):
        import torch
        self.torch = torch
        self.args, self.G, self.rank, self.local_rank = args, G, rank, local_rank
        self.dev = torch.device("cuda", local_rank)
        self.dist = None
        if G > 1:
            import torch.distributed as dist
            dist.init_process_group("nccl", device_id=self.dev)
            self.dist = dist
        # An explicit non-default stream: torch's default stream handle is 0, which the C ABI reads as "use the
        # index's own stream"; the CUDA events below must sit on the stream the kernels are launched on.
        self.tstream = torch.cuda.Stream(device=self.dev)
        torch.cuda.set_stream(self.tstream)
        self.stream = self.tstream.cuda_stream
        assert self.stream != 0
        self.comm = None

    def barrier(self):
        if self.dist is not None:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, v: float) -> float:
        if self.dist is None:
            return v
        t = self.torch.tensor([v], dtype=self.torch.float64, device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(self, v: int) -> int:
        if self.dist is None:
            return v
        t = self.torch.tensor([v], dtype=self.torch.int64, device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM)
        return int(t.item())

    def ensure_comm(self, slot_bytes: int):
        """Peer-memory exchange context (nk_comm_*): IPC handles travel once over torch.distributed (setup only)."""
        from nornicdb_b200.knn import Comm
        if self.comm is not None and self.comm_slot >= slot_bytes:
            return self.comm
        if self.comm is not None:
            self.barrier()
            self.comm.release()
        self.comm = Comm(self.local_rank, self.rank, self.G, slot_bytes)
        self.comm_slot = slot_bytes
        handles = [None] * self.G
        self.dist.all_gather_object(handles, self.comm.export())
        self.comm.connect(handles)
        self.barrier()
        return self.comm

    def timed_steps(self, step, steps, flush=None):
        """K steps bracketed by barrier + synchronize; CUDA events on the launching stream; returns total ms (MAX over
        ranks).  With an L2 flush between steps every step has its own event pair (the flush is not timed)."""
        torch = self.torch
        self.barrier()
        if flush is None:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for s in range(steps):
                step(s)
            e1.record()
            self.barrier()
            ms = e0.elapsed_time(e1)
        else:
            ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
            for s in range(steps):
                flush.zero_()
                ev[s][0].record()
                step(s)
                ev[s][1].record()
            self.barrier()
            ms = sum(a.elapsed_time(b) for a, b in ev)
        return self.max_over_ranks(ms)


def measure(run: Runner, ix, n_shard, N_total, dim, dtype, Q, k, metric, steps, warmup, want_e2e=True, sample_clocks=False):
    """Device-resident and end-to-end throughput of one workload on an already filled index (all ranks call this)."""
    import numpy as np
    torch = run.torch
    from nornicdb_b200.knn import fill_uniform_device, merge_keys_device
    G, dev, stream, lr = run.G, run.dev, run.stream, run.local_rank
    n_all = warmup + steps
    q_all = torch.empty((n_all, Q, dim), dtype=torch.float32, device=dev)
    fill_uniform_device(lr, q_all.data_ptr(), n_all * Q, dim, QUERY_SEED, 0, stream)
    out_idx = torch.empty((Q, k), dtype=torch.int32, device=dev)
    out_score = torch.empty((Q, k), dtype=torch.float32, device=dev)
    peer = G > 1 and run.args.exchange == "peer"
    comm = run.ensure_comm(Q * k * 8) if peer else None
    keys_local = torch.empty((Q, k), dtype=torch.int64, device=dev) if G > 1 and not peer else None
    keys_all = torch.empty((G, Q, k), dtype=torch.int64, device=dev) if G > 1 and not peer else None
    elem = 4 if dtype == "f32" else 2
    flush = None
    if n_shard * dim * elem <= 512e6:
        flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)
    torch.cuda.synchronize()

    def search_dev(qp):
        if G == 1:
            ix.search_device(qp, Q, k, out_idx.data_ptr(), out_score.data_ptr(), stream)
        elif peer:
            ix.search_sharded_device(comm, qp, Q, k, out_idx.data_ptr(), out_score.data_ptr(), stream)
        else:
            ix.search_keys_device(qp, Q, k, keys_local.data_ptr(), stream)
            run.dist.all_gather_into_tensor(keys_all.view(-1), keys_local.view(-1))
            merge_keys_device(lr, keys_all.data_ptr(), G, Q, k, metric, out_idx.data_ptr(), out_score.data_ptr(), stream)

    for i in range(warmup):
        search_dev(q_all[i].data_ptr())
    run.barrier()
    launches0 = ix.stats()["kernel_launches"]
    ix.enable_timing(True)
    ix.scan_time_ms()
    sampler = None
    if sample_clocks:
        sampler = ClockSampler(lr)
        sampler.start()
    t_wall0 = time.perf_counter()
    total_ms = run.timed_steps(lambda s: search_dev(q_all[warmup + s].data_ptr()), steps, flush)
    t_wall = time.perf_counter() - t_wall0
    last = (out_idx.clone(), out_score.clone())  # the untimed searches below write into out_idx / out_score again
    scan_ms, scan_launches = ix.scan_time_ms()
    ix.enable_timing(False)
    launches = ix.stats()["kernel_launches"] - launches0 + (steps if G > 1 and not peer else 0)
    clocks = None
    if sampler is not None:
        note = "sampled during the timed region"
        if t_wall < 0.6:
            # nvidia-smi cannot sample faster than ~100 ms: keep the identical step loop running (untimed) until the
            # sampler has seen ~0.6 s of this load, so the clock / throttle record describes the measured workload
            note = ("timed region %.0f ms is shorter than the sampler period: sampled over it plus an untimed continuation of the "
                    "same step loop" % (t_wall * 1e3))
            n_extra = 0
            while time.perf_counter() - t_wall0 < 0.6 and n_extra < 100000:
                search_dev(q_all[warmup + (n_extra % steps)].data_ptr())
                n_extra += 1
                if n_extra % 8 == 0:
                    torch.cuda.current_stream().synchronize()
            run.barrier()
        clocks = sampler.stop()
        clocks["note"] = note
    used_path = ix.last_path()
    res = {"value": Q * steps / (total_ms / 1e3), "ms_per_step": total_ms / steps, "steps": steps, "path": used_path,
           "scan_ms": scan_ms, "scan_launches": scan_launches, "launches": int(launches), "wall_s": t_wall, "clocks": clocks,
           "l2": "L2 flushed between steps (256 MB memset, untimed)" if flush is not None
                 else "corpus shard per GPU >> 126 MB L2 (inputs larger than L2; no flush needed)",
           "out_idx": out_idx, "out_score": out_score, "q_all": q_all, "search_dev": search_dev, "last": last}

    if want_e2e:
        # e2e: the reference-facing call with HOST buffers (H2D queries + D2H results inside the timed region)
        q_host = torch.empty((n_all, Q, dim), dtype=torch.float32).pin_memory()
        q_host.copy_(q_all.cpu())
        res_idx_h = torch.empty((Q, k), dtype=torch.int32).pin_memory()
        res_sc_h = torch.empty((Q, k), dtype=torch.float32).pin_memory()
        q_np = q_host.numpy()
        q_stage = torch.empty((Q, dim), dtype=torch.float32, device=dev)

        def step_e2e(i):
            if G == 1:
                ix.search(q_np[i], k)  # nk_search: H2D + fused scan + D2H, synchronous
                return
            q_stage.copy_(q_host[i], non_blocking=True)  # pinned host -> preallocated device staging
            search_dev(q_stage.data_ptr())
            res_idx_h.copy_(out_idx, non_blocking=True)
            res_sc_h.copy_(out_score, non_blocking=True)
            torch.cuda.current_stream().synchronize()

        for i in range(min(warmup, 3)):
            step_e2e(i)
        t0 = time.perf_counter()
        ev_ms = run.timed_steps(lambda s: step_e2e(warmup + s), steps, None)
        wall_ms = run.max_over_ranks((time.perf_counter() - t0) * 1e3)
        # G == 1: nk_search runs on the index's own stream and returns synchronously — the events on this stream see none
        # of it, the wall clock around the K calls is the honest figure.  G > 1: everything is ordered on the timed stream.
        e2e_ms = wall_ms if G == 1 else ev_ms
        res["e2e"] = {"value": Q * steps / (e2e_ms / 1e3), "unit": "queries/s", "h2d_bytes_per_step": Q * dim * 4,
                      "d2h_bytes_per_step": Q * k * 8, "ms_per_step": e2e_ms / steps, "steps": steps,
                      "timing": "wall clock around K synchronous nk_search calls (bracketed by barrier + synchronize)" if G == 1
                                else "CUDA events on the launching stream around K steps (H2D, search, exchange, D2H, sync), MAX over ranks",
                      "api": "nk_search (C ABI, host buffers)" if G == 1 else
                             ("pinned host -> H2D -> nk_search_sharded_device (scan + peer-memory exchange + merge) -> D2H" if peer else
                              "pinned host -> H2D -> nk_search_keys_device -> ncclAllGather -> nk_merge_keys_device -> D2H")}
    return res


def roofline_of(res, n_shard, dim, dtype, Q, workload, peak, peak_src):
    path = res["path"]
    algo = scan_bytes(path, n_shard, dim, dtype)
    launches = max(res["scan_launches"], 1)
    avg_ms = res["scan_ms"] / launches
    achieved = algo / (avg_ms / 1e3) / 1e9
    r = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
         "traffic": load_traffic(workload, path), "peak_source": peak_src, "kernel": KERNEL_NAME.get(path, path),
         "algorithmic_bytes_per_launch": algo, "avg_launch_ms": avg_ms, "scan_launches_per_step": launches / res["steps"],
         "scan_share_of_step": res["scan_ms"] / (res["ms_per_step"] * res["steps"])}
    fp32_bytes = n_shard * dim * (4 if dtype == "f32" else 2)
    if path == "shadow" and dtype == "f32":
        r["note"] = ("the scan streams the BF16 shadow (n*dpad*2 + 8n bytes per launch), not the fp32 rows: `achieved` counts the bytes "
                     "actually read; SURVEY.md 8(d)'s fp32 figure n*d*4 is reported as fp32_equivalent_gbs; the like-for-like scans over "
                     "the fp32 rows are in also.headline_filter / also.q1_simt")
        r["fp32_corpus_bytes_per_launch"] = fp32_bytes
        r["fp32_equivalent_gbs"] = fp32_bytes / (avg_ms / 1e3) / 1e9
    if path in ("tensor", "filter", "shadow"):
        # SURVEY.md §8(d): roofline fraction = max(bytes/t / BW, flops/t / tensor peak).  Large batches (several query
        # blocks per corpus pass) are bound by the tensor pipes, not by HBM: report whichever bound is tighter.
        tpeak, tsrc = load_tensor_peak(bf16=path == "shadow")
        flops = 2.0 * Q * n_shard * dim * res["steps"] / launches  # algorithmic: one product per (query, row, dim)
        tflops = flops / (avg_ms / 1e3) / 1e12
        r["tensor"] = {"achieved": tflops, "peak": tpeak, "unit": "TFLOP/s", "frac": tflops / tpeak, "peak_source": tsrc,
                       "algorithmic_flops_per_launch": flops}
        if tflops / tpeak > achieved / peak:
            r.update({"bound": "tensor", "achieved": tflops, "peak": tpeak, "unit": "TFLOP/s", "frac": tflops / tpeak, "peak_source": tsrc,
                      "hbm": {"achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak}})
    return r


def dump_outputs(out_dir, out_idx, out_score, k_eff):
    """--dump-outputs: the [Q x k'] result a caller of the device-resident search receives (k' = min(k, N)).  Row ids are
    written as float64 (exact for 32-bit ids).  Results above 60 MB keep a fixed, seeded sample of the queries, whose
    positions in the batch go to query_rows.npy."""
    import numpy as np
    idx = out_idx[:, :k_eff].cpu().numpy().view(np.uint32).astype(np.float64)
    score = out_score[:, :k_eff].cpu().numpy()
    os.makedirs(out_dir, exist_ok=True)
    keep = (60 << 20) // (k_eff * 12 + 8)
    if idx.shape[0] > keep:
        rows = np.sort(np.random.default_rng(0).choice(idx.shape[0], keep, replace=False))
        idx, score = idx[rows], score[rows]
        np.save(os.path.join(out_dir, "query_rows.npy"), rows.astype(np.float64))
    np.save(os.path.join(out_dir, "indices.npy"), idx)
    np.save(os.path.join(out_dir, "scores.npy"), score)


def also_entry(res, n, dim, dtype, Q, desc, peak, peak_src, workload):
    r = roofline_of(res, n, dim, dtype, Q, workload, peak, peak_src)
    e = {"workload": desc, "value": res["value"], "unit": "queries/s", "ms_per_step": res["ms_per_step"], "steps": res["steps"],
         "path": res["path"], "scan_kernel_ms": r["avg_launch_ms"], "scan_launches_per_step": r["scan_launches_per_step"],
         "scan_share_of_step": r["scan_share_of_step"], "gpu_launches_per_step": res["launches"] / res["steps"],
         "algorithmic_bytes_per_launch": r["algorithmic_bytes_per_launch"], "bound": r["bound"], "roofline_frac": r["frac"],
         "achieved": r["achieved"], "achieved_unit": r["unit"], "l2": res["l2"]}
    if "hbm" in r:
        e["hbm_frac"] = r["hbm"]["frac"]
    if "fp32_equivalent_gbs" in r:
        e["fp32_equivalent_gbs"] = r["fp32_equivalent_gbs"]
    if "e2e" in res:
        e["e2e"] = res["e2e"]
    return e


# ------------------------------------------------------------------------------------------------------
def parity_check(run: Runner, ix, lo, hi, N_total, dim, dtype, Q, k, metric, res, clustered=False):
    """UNTIMED post-check of this very run (every rank count): (1) 8 planted queries = corpus rows at known global
    indices (+ tiny noise) must come back first; (2) every returned score is recomputed in fp64 from the rows read back
    from HBM (each rank checks the rows it owns); (3) indices unique, order correct; (4) N > 1: the exchanged result
    must be bit-identical with the in-process multi-device search (nk_index_create over devices 0..N-1 + nk_search)."""
    import numpy as np
    torch = run.torch
    from nornicdb_b200.knn import KnnIndex, fill_uniform_device
    G, dev, stream, lr = run.G, run.dev, run.stream, run.local_rank
    out = {"ok": True, "checks": []}

    def fail(msg):
        out["ok"] = False
        out.setdefault("errors", []).append(msg)

    # ---- (1) planted near-copies
    P = min(8, Q)
    planted = [(N_total * (2 * i + 1)) // (2 * P) for i in range(P)]  # spread over all shards
    q = res["q_all"][0].clone()
    if dtype == "f32" and not clustered:
        for i, r in enumerate(planted):
            fill_uniform_device(lr, q[i].data_ptr(), 1, dim, CORPUS_SEED, r, stream)  # generator row r == corpus row r
        noise = torch.empty((P, dim), dtype=torch.float32, device=dev)
        fill_uniform_device(lr, noise.data_ptr(), P, dim, 99, 0, stream)
        torch.cuda.current_stream().synchronize()
        q[:P] += 1e-3 * noise
        res["search_dev"](q.data_ptr())
        run.barrier()
        gi = res["out_idx"].cpu().numpy().view(np.uint32)
        top1 = gi[:P, 0].tolist()
        if top1 != planted:
            fail(f"planted rows {planted} came back as {top1}")
        out["checks"].append(f"planted: {P} near-copies of rows spread over all shards returned first")
    else:
        res["search_dev"](q.data_ptr())
        run.barrier()
    gi = res["out_idx"].cpu().numpy().view(np.uint32)
    gs = res["out_score"].cpu().numpy()
    qh = q.cpu().numpy().astype(np.float64)

    # ---- (3) uniqueness / order
    for qi in range(Q):
        row = gi[qi]
        if len(set(row.tolist())) != k:
            fail(f"query {qi}: duplicate rows")
            break
        d = np.diff(gs[qi].astype(np.float64))
        if (metric == "euclidean" and (d < -1e-6 * np.maximum(1, np.abs(gs[qi][1:]))).any()) or \
           (metric != "euclidean" and (d > 1e-6 * np.maximum(1, np.abs(gs[qi][1:]))).any()):
            fail(f"query {qi}: scores out of order")
            break
    out["checks"].append("unique indices, scores ordered")

    # ---- (2) exact fp64 recomputation from rows read back (each rank: the rows it owns; at most 4096 per rank)
    mine = [(qi, j) for qi in range(Q) for j in range(k) if lo <= int(gi[qi, j]) < hi][:4096]
    bad, worst = 0, 0.0
    for qi, j in mine:
        x = ix.read_rows(int(gi[qi, j]) - lo, 1)[0]
        if dtype == "bf16":
            from nornicdb_b200.knn import from_bf16_bits
            x = from_bf16_bits(x)
        x = x.astype(np.float64)
        if metric == "dot":
            s = float(x @ qh[qi])
        elif metric == "cosine":
            den = np.linalg.norm(x) * np.linalg.norm(qh[qi])
            s = float(x @ qh[qi] / den) if den > 0 else 0.0
        else:
            s = float(np.sqrt(((x - qh[qi]) ** 2).sum()))
        err = abs(s - float(gs[qi, j])) / max(abs(s), 1e-2)
        worst = max(worst, err)
        if err > 1e-4:
            bad += 1
    total_checked = run.sum_over_ranks(len(mine))
    total_bad = run.sum_over_ranks(bad)
    worst = run.max_over_ranks(worst)
    if total_bad:
        fail(f"{total_bad} returned scores differ from the fp64 recomputation by > 1e-4 relative")
    out["scores_recomputed_fp64"] = total_checked
    out["worst_rel_err"] = worst
    out["checks"].append(f"{total_checked} of {Q * k} returned scores recomputed in fp64 from rows read back (1e-4 relative)")

    # ---- (4) exchanged result == in-process multi-device search (the form a single Go host process would call)
    if G > 1 and not clustered:
        run.barrier()
        if run.rank == 0:
            try:
                shard_gb = (N_total // G) * dim * (4 if dtype == "f32" else 2) / 1e9
                tight = shard_gb * 3.0 > 140  # a second shard + shadow would not fit beside this rank's own rows + shadow
                if tight:
                    os.environ["NK_SHADOW"] = "0"  # read at index creation: rows only (TF32 filter path, same exact results)
                mix = KnnIndex(dim, metric=metric, dtype=dtype, devices=tuple(range(G)))
                os.environ.pop("NK_SHADOW", None)
                mix.fill_uniform(N_total, CORPUS_SEED)
                mi, ms = mix.search(q.cpu().numpy(), k)
                mix.release()
                same_i = bool((mi == gi).all())
                same_s = bool((ms.view(np.uint32) == gs.view(np.uint32)).all())
                if not (same_i and same_s):
                    fail(f"exchange result differs from the in-process multi-device nk_search (indices equal: {same_i}, scores bit-equal: {same_s})")
                out["checks"].append(f"bit-identical to nk_index_create(devices=0..{G - 1}) + nk_search on rank 0"
                                     + (" (shadow-less index: TF32 filter path)" if tight else ""))
            except Exception as e:  # e.g. out of memory next to the other ranks' shards
                out["checks"].append(f"in-process multi-device comparison skipped: {e}")
        run.barrier()
    try:
        ix.status(stream)
        if run.comm is not None:
            run.comm.status(stream)
    except Exception as e:
        fail(str(e))
    all_bad = run.sum_over_ranks(0 if out["ok"] else 1)
    if run.rank != 0 and not out["ok"]:
        sys.stderr.write(f"[rank {run.rank}] parity_check: {out.get('errors')}\n")
    if all_bad and out["ok"]:
        fail(f"{all_bad} other rank(s) reported a parity failure (see stderr)")
    return out


# ------------------------------------------------------------------------------------------------------
def main():
    args = parse_args()
    # torchrun exports OMP_NUM_THREADS=1 for every rank; the CPU baseline (oracle/liboracle.so, OpenMP) must be
    # free to use every core this process may run on, pinned.  Must happen before libgomp initialises.
    ncpu = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    runs_cpu_baseline = args.impl == "reference" or (int(os.environ.get("WORLD_SIZE", "1")) == 1 and not args.no_cpu_baseline)
    if runs_cpu_baseline and int(os.environ.get("RANK", "0")) == 0:
        if os.environ.get("OMP_NUM_THREADS", "1") == "1":
            os.environ["OMP_NUM_THREADS"] = str(ncpu)
        os.environ.setdefault("OMP_PROC_BIND", "close")
        os.environ.setdefault("OMP_PLACES", "cores")
    N_total, dim, dtype, Q, k, metric, desc = WORKLOADS[args.workload]
    if args.rows:
        N_total = args.rows
    if args.k:
        k = args.k
    if args.q:
        Q = args.q
    overridden = bool(args.rows or args.k or args.q)
    if overridden:
        desc += f" [debug override: N={N_total} Q={Q} k={k}]"
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    G = args.gpus
    if world != G:
        if world == 1 and G > 1:
            print(f"bench.py: --gpus {G} needs torchrun with {G} ranks", file=sys.stderr)
            sys.exit(2)
        G = world
    elem = 2 if dtype != "f32" else 4
    if N_total // max(G, 1) * dim * elem > 150e9:
        if rank == 0:
            print(json.dumps({"error": f"workload {args.workload} needs more GPUs: {N_total // max(G, 1) * dim * elem / 1e9:.0f} GB per GPU"}))
        return
    config = {"workload": desc, "N": N_total, "dim": dim, "corpus_dtype": dtype, "Q": Q, "k": k, "metric": metric,
              "sharding": f"row-range x{G}" if G > 1 else "single GPU",
              "l2": "corpus shard per GPU >> 126 MB L2 (inputs larger than L2; no flush needed)"
              if N_total // G * dim * elem > 512e6 else "L2 flushed between steps (256 MB memset)"}

    # ------------------------------------------------------------------ reference arm (CPU)
    if args.impl == "reference":
        if rank != 0:
            return
        r = cpu_reference_run(N_total, dim, dtype, Q, k, metric)
        line = {
            "impl": "reference", "metric": "kNN queries/sec", "value": r["value"], "unit": "queries/s", "n_gpus": G,
            "steps": r["steps_timed"], "warmup": 1, "ms_per_step": r["ms_per_pass"],
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config,
            "cpu_baseline": {"value": r["value"], "unit": "queries/s", "cores": r["cores"], "kind": r["kind"],
                             "sample": r["sample"], "single_thread": r["single_thread"]},
            "e2e": {"value": r["value"], "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0,
        }
        print(json.dumps(line))
        return

    # ------------------------------------------------------------------ our arm (GPU)
    import torch
    from nornicdb_b200 import build as knn_build
    from nornicdb_b200 import cuda as ncuda
    from nornicdb_b200.knn import KnnIndex
    from nornicdb_b200.sharding import shard_range

    if rank == 0 or local_rank == 0:
        knn_build.build()
    if not ncuda.IsAvailable():
        raise RuntimeError("bench.py needs a CUDA device: the product has no CPU fallback")
    torch.cuda.set_device(local_rank)
    run = Runner(args, G, rank, local_rank)
    peak, peak_src = load_peaks()

    # ---- corpus: this rank's row range, generated in HBM by the counter-based generator
    lo, hi = shard_range(N_total, G, rank)
    n_shard = hi - lo
    clustered = args.workload == "clustered"
    ix = KnnIndex(dim, metric=metric, dtype=dtype, devices=(local_rank,))
    ix.set_path(args.path)
    ix.set_row_base(lo)
    if clustered:
        ix.fill_clustered(n_shard, CORPUS_SEED, 1000, 0.1)
    else:
        ix.fill_uniform(n_shard, CORPUS_SEED)

    res = measure(run, ix, n_shard, N_total, dim, dtype, Q, k, metric, args.steps, args.warmup, want_e2e=True, sample_clocks=True)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, *res["last"], min(k, N_total))
    used_path = res["path"]
    roofline = roofline_of(res, n_shard, dim, dtype, Q, args.workload, peak, peak_src)
    algo = roofline["algorithmic_bytes_per_launch"]
    line = {
        "metric": "kNN queries/sec", "value": res["value"], "unit": "queries/s", "n_gpus": G, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": res["ms_per_step"], "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32" if dtype == "f32" else f"{dtype} corpus / f32 accumulate", "data": "synthetic",
        "config": config, "scan": SCAN_DESC.get(used_path, used_path),
        "hbm_gbs_whole_step": G * algo * roofline["scan_launches_per_step"] / (res["ms_per_step"] / 1e3) / 1e9,
        "roofline": roofline, "clocks": res["clocks"], "e2e": res["e2e"],
        "gpu_launches": res["launches"], "gpu_launches_per_step": res["launches"] / args.steps, "path": used_path,
        "wall_s_timed_region": res["wall_s"],
        "timing": "value: one CUDA event pair on the launching stream around the K steps, barrier + synchronize on both sides, MAX over "
                  "ranks; e2e: " + res["e2e"]["timing"],
        "exchange": None if G == 1 else ("peer-memory push + fused wait/merge/decode (nk_search_sharded_device, csrc/exchange.cu)"
                                         if args.exchange == "peer" else "ncclAllGather + nk_merge_keys_device"),
    }
    if clustered or used_path in ("shadow", "filter"):
        c = ix.debug_counters()
        searches = max(ix.stats()["searches"], 1)
        line["filter_retries"] = {"bf16_stage_retry_rate": c["bf16_stage_retries"] / searches, "exact_stage_rate": c["exact_stage_runs"] / searches,
                                  "searches": searches, "longest_survivor_list_last_search": c["longest_list"], "overflow_bits": c["overflow_bits"],
                                  "note": "asynchronous API: a first-stage overflow goes straight to the exact stage (exact_stage_rate); the TF32 retry stage belongs to the host-synchronous nk_search"}
    if not args.no_parity:
        line["parity_check"] = parity_check(run, ix, lo, hi, N_total, dim, dtype, Q, k, metric, res, clustered=clustered)
    for key in ("out_idx", "out_score", "q_all", "search_dev", "last"):
        res.pop(key, None)

    # ---- the rest of the north_star grid (default N=1 line only), same timing rules, device-resident + e2e where cheap
    if G == 1 and args.workload == "headline" and not overridden and not args.no_also and args.path == "auto":
        also = {}

        def sub(name, index, n, d, dt, q_, k_, m_, desc_, steps, warm, path="auto", e2e=False, wl=None):
            try:
                index.set_metric(m_)
                index.set_path(path)
                c0, s0 = index.debug_counters(), index.stats()["searches"]
                r = measure(run, index, n, n, d, dt, q_, k_, m_, steps, warm, want_e2e=e2e)
                for key in ("out_idx", "out_score", "q_all", "search_dev", "last"):
                    r.pop(key, None)
                also[name] = also_entry(r, n, d, dt, q_, desc_, peak, peak_src, wl or name)
                if r["path"] in ("shadow", "filter"):
                    c1, s1 = index.debug_counters(), index.stats()["searches"]
                    also[name]["filter_retries"] = {"first_stage_retry_rate": (c1["bf16_stage_retries"] - c0["bf16_stage_retries"]) / max(s1 - s0, 1),
                                                    "exact_stage_rate": (c1["exact_stage_runs"] - c0["exact_stage_runs"]) / max(s1 - s0, 1),
                                                    "searches": s1 - s0, "longest_survivor_list_last_search": c1["longest_list"],
                                                    "overflow_bits_so_far": c1["overflow_bits"]}
                return r
            except Exception as e:  # never let a secondary measurement break the contract line
                also[name] = {"error": str(e)}
                return None

        n10, d10 = N_total, dim
        sub("c3", ix, n10, d10, "f32", 1024, 100, "dot", WORKLOADS["c3"][6], 5, 3, e2e=True)
        sub("c3_k10", ix, n10, d10, "f32", 1024, 10, "dot", "configs[2] with k=10: N=10M d=1024 fp32 Q=1024 k=10 inner-product", 5, 3)
        sub("q1024_cos_k10", ix, n10, d10, "f32", 1024, 10, "cosine", "configs[4]'s per-GPU shape at N=10M: Q=1024 k=10 cosine", 5, 3)
        sub("q1", ix, n10, d10, "f32", 1, 10, "cosine", WORKLOADS["q1"][6], 20, 3, e2e=True, wl="q1")
        sub("k100", ix, n10, d10, "f32", 64, 100, "cosine", "headline with k=100: N=10M d=1024 fp32 Q=64 k=100 cosine", 10, 3)
        sub("headline_filter", ix, n10, d10, "f32", 64, 10, "cosine",
            "headline on the fp32 ROWS (1xTF32 filter, no shadow): the like-for-like scan of SURVEY.md 8(d)'s n*d*4 bytes", 10, 3,
            path="filter", wl="headline")
        sub("q1_simt", ix, n10, d10, "f32", 1, 10, "cosine", "Q=1 CUDA-core scan over the fp32 rows (n*d*4 bytes per query)", 10, 3,
            path="simt", wl="q1")
        sub("headline_l2", ix, n10, d10, "f32", 64, 10, "euclidean", "headline shape, L2 metric", 10, 3)
        ix.release()
        ix = None
        try:
            cx = KnnIndex(dim, metric="cosine", dtype="f32", devices=(local_rank,))
            cx.fill_clustered(N_total, CORPUS_SEED, 1000, 0.1)
            r = sub("headline_clustered", cx, N_total, dim, "f32", 64, 10, "cosine", WORKLOADS["clustered"][6], 10, 3, wl="clustered")
            sub("clustered_filter", cx, N_total, dim, "f32", 64, 10, "cosine",
                "clustered corpus through the TF32 filter over the fp32 rows", 5, 2, path="filter", wl="clustered")
            cx.release()
        except Exception as e:
            also["headline_clustered"] = {"error": str(e)}
        for name, wl in (("c4", "c4"), ("c2", "c2"), ("c1", "c1")):
            n2, d2, dt2, Q2, k2, m2, desc2 = WORKLOADS[wl]
            try:
                ix2 = KnnIndex(d2, metric=m2, dtype=dt2, devices=(local_rank,))
                ix2.fill_uniform(n2, CORPUS_SEED)
                sub(name, ix2, n2, d2, dt2, Q2, k2, m2, desc2, 50 if n2 <= 1_000_000 else 20, 5, e2e=True, wl=wl)
                if wl == "c4":
                    sub("c4_q64", ix2, n2, d2, dt2, 64, k2, m2, "configs[3]'s fp16 corpus with a batch: Q=64 (16-bit tensor pass in place)", 10, 3)
                ix2.release()
            except Exception as e:
                also[name] = {"error": str(e)}
        line["also"] = also
    # ---- configs[4] under the same run (8 GPUs, default workload only): N=100M needs the 8-way row sharding, so this is the
    # one north_star config that only exists at N=8 — measured and parity-checked here so that the driver's own 8-GPU
    # record carries it.  51 GB of rows + 26 GB of shadow per GPU; ~15 s on top of the headline run.
    if G >= 8 and args.workload == "headline" and not overridden and not args.no_also and args.path == "auto":
        n5, d5, dt5, Q5, k5, m5, desc5 = WORKLOADS["c5"]
        entry = {}
        try:
            ix.release()
            ix = None
            lo5, hi5 = shard_range(n5, G, rank)
            ix = KnnIndex(d5, metric=m5, dtype=dt5, devices=(local_rank,))
            ix.set_row_base(lo5)
            ix.fill_uniform(hi5 - lo5, CORPUS_SEED)
            r5 = measure(run, ix, hi5 - lo5, n5, d5, dt5, Q5, k5, m5, 5, 2, want_e2e=True)
            entry = also_entry(r5, hi5 - lo5, d5, dt5, Q5, desc5, peak, peak_src, "c5")
            entry["n_gpus"] = G
            entry["rows_per_gpu"] = hi5 - lo5
            if not args.no_parity:
                entry["parity_check"] = parity_check(run, ix, lo5, hi5, n5, d5, dt5, Q5, k5, m5, r5)
        except Exception as e:  # every rank takes the same path up to here; a failure must not lose the headline line
            entry = {"error": str(e)}
        line["also"] = {"c5": entry}
    if G == 1 and rank == 0 and not args.no_cpu_baseline:
        r = cpu_reference_run(N_total, dim, dtype, Q, k, metric, budget_s=18.0)
        line["cpu_baseline"] = {"value": r["value"], "unit": "queries/s", "cores": r["cores"], "kind": r["kind"],
                                "sample": r["sample"], "single_thread": r["single_thread"]}
    if rank == 0:
        print(json.dumps(line))
    if ix is not None:
        ix.release()
    if run.comm is not None:
        run.barrier()
        run.comm.release()
    if run.dist is not None:
        run.dist.destroy_process_group()


if __name__ == "__main__":
    main()
