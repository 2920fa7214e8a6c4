"""Times k-means++ seeding on the device (nk_index_kmeanspp) on the corpora of SURVEY.md 8(d): N = 10M, d = 1024 fp32, generated
on the device, clustered (1000 centres, sigma 0.1) and uniform; K = 1000.  Per corpus it reports:
  * the whole seeding (host clock around the call, which ends in a device synchronise), a cold and a warm call;
  * per-kernel times from a torch.profiler run of its own: the first update pass (no bound yet: every row is read) with its
    bytes and fraction of the device-to-device copy peak measured in the same run, and the update / select / cc times of
    the last 50 steps;
  * rows_scored / ((K-1) N): the share of (row, step) distances computed rather than skipped by the triangle-inequality bound;
  * the Lloyd loop of ClusterIndex.Cluster (assign_nearest + cluster_means until nothing changes or --max-iter passes,
    capped at --lloyd-cap seconds) after the seeding, and the cluster sizes after 4 passes (the 4 passes of DESIGN.md §3.7's
    random-init clustering) and at the end.
Then, for the before/after comparison, the host seeding ClusterIndex._init_kmeanspp (numpy) against the device at
--host-n x d, K = --host-K.

    python profiles/experiments/time_kmeanspp.py [--n 10000000] [--out FILE.json]"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", ".."))
from nornicdb_b200.cluster_index import ClusterIndex  # noqa: E402
from nornicdb_b200.knn import KnnIndex  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--n", type=int, default=10_000_000)
ap.add_argument("--d", type=int, default=1024)
ap.add_argument("--K", type=int, default=1000)
ap.add_argument("--max-iter", type=int, default=100)
ap.add_argument("--lloyd-cap", type=float, default=90.0)
ap.add_argument("--host-n", type=int, default=200_000)
ap.add_argument("--host-K", type=int, default=100)
ap.add_argument("--out", default="")
args = ap.parse_args()
n, d, K = args.n, args.d, args.K
res = {"n": n, "d": d, "K": K}

card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                      capture_output=True, text=True).stdout.strip().splitlines()[0]
print(f"card: {card}")
res["card"] = card

# device-to-device copy peak (read + write bytes), 4 GB buffers
src = torch.empty(1 << 30, dtype=torch.float32, device="cuda")
dst = torch.empty_like(src)
for _ in range(3):
    dst.copy_(src)
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
for _ in range(20):
    dst.copy_(src)
e1.record()
torch.cuda.synchronize()
peak = 2 * src.numel() * 4 * 20 / (e0.elapsed_time(e1) * 1e-3) / 1e9
del src, dst
torch.cuda.empty_cache()
print(f"copy peak: {peak:.0f} GB/s (read + write)")
res["copy_peak_gbs"] = peak


def kernel_times(ix, first, draws):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        ix.kmeanspp(K, first, draws)
    ev = sorted((e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA), key=lambda e: e.time_range.start)
    out = {}
    for name in ("kpp_update_kernel", "kpp_select_kernel", "kpp_cc_kernel"):
        out[name] = [e.device_time_total * 1e-3 for e in ev if name in e.name]  # ms, in launch order
    return out


for corpus in ("clustered", "uniform"):
    ix = KnnIndex(d, metric="euclidean")
    if corpus == "clustered":
        ix.fill_clustered(n, seed=7, n_centres=1000, sigma=0.1)
    else:
        ix.fill_uniform(n, seed=7)
    rng = np.random.default_rng(0)
    first, draws = int(rng.integers(n)), rng.random(K - 1)
    r = {}
    t0 = time.perf_counter()
    cen, picked, scored = ix.kmeanspp(K, first, draws)
    r["seed_s_cold"] = time.perf_counter() - t0
    t0 = time.perf_counter()
    cen2, picked2, scored2 = ix.kmeanspp(K, first, draws)
    r["seed_s"] = time.perf_counter() - t0
    assert (picked == picked2).all() and scored == scored2 and np.array_equal(cen, cen2)
    r["scored_fraction"] = scored / ((K - 1) * n)
    r["distinct_rows"] = int(np.unique(picked).size)
    kt = kernel_times(ix, first, draws)
    up = kt["kpp_update_kernel"]
    first_bytes = n * d * 4 + n * 12 + (n // 1024) * 8  # rows read; d2 + near written; block sums
    r["first_step_ms"] = up[0]
    r["first_step_bytes"] = first_bytes
    r["first_step_gbs"] = first_bytes / (up[0] * 1e-3) / 1e9
    r["first_step_peak_fraction"] = r["first_step_gbs"] / peak
    r["update_ms_last50"] = float(np.mean(up[-50:]))
    r["select_ms_last50"] = float(np.mean(kt["kpp_select_kernel"][-50:]))
    r["cc_ms_last50"] = float(np.mean(kt["kpp_cc_kernel"][-50:]))
    r["kernel_ms_total"] = float(sum(up) + sum(kt["kpp_select_kernel"]) + sum(kt["kpp_cc_kernel"]))
    r["update_ms_by_step"] = [float(np.mean(up[i:i + 50])) for i in range(0, len(up), 50)]
    print(f"[{corpus}] seeding {r['seed_s']:.2f} s (cold {r['seed_s_cold']:.2f} s), kernels {r['kernel_ms_total']:.0f} ms; "
          f"first step {up[0]:.2f} ms = {r['first_step_gbs']:.0f} GB/s = {r['first_step_peak_fraction']:.2f} of the copy peak; "
          f"scored {r['scored_fraction']:.4f}; last 50 steps: update {r['update_ms_last50']:.3f} ms, select "
          f"{r['select_ms_last50']:.3f} ms, cc {r['cc_ms_last50']:.3f} ms")
    print(f"[{corpus}] update ms per 50-step window: {[round(x, 3) for x in r['update_ms_by_step']]}")
    # the Lloyd loop of ClusterIndex.Cluster after this seeding
    assign = np.zeros(n, np.int32)
    t0 = time.perf_counter()
    it, changed, c = 0, -1, cen
    while it < args.max_iter and time.perf_counter() - t0 < args.lloyd_cap:
        changed = ix.assign_nearest(c, assign)
        c, counts = ix.cluster_means(assign, c)
        it += 1
        if it == 4:
            r["sizes_after_4"] = [int(counts.min()), int(counts.max())]
        if changed == 0:
            break
    r["lloyd_s"] = time.perf_counter() - t0
    r["lloyd_iterations"] = it
    r["lloyd_converged"] = changed == 0
    r["sizes_final"] = [int(counts.min()), int(counts.max())]
    r["cluster_s"] = r["seed_s"] + r["lloyd_s"]
    print(f"[{corpus}] Cluster(): seeding + {it} Lloyd passes ({'converged' if changed == 0 else f'{changed} still changing'}) "
          f"= {r['cluster_s']:.1f} s; cluster sizes after 4 passes {r.get('sizes_after_4')}, final {r['sizes_final']}")
    res[corpus] = r
    if corpus == "clustered":
        host_rows = ix.read_rows(0, args.host_n)
    ix.release()

# before / after: the host seeding at a size it can finish, and the device on the same rows
hn, hK = args.host_n, args.host_K
ci = ClusterIndex(d, rng=np.random.default_rng(1))
t0 = time.perf_counter()
ci._init_kmeanspp(hK, host_rows)
host_s = time.perf_counter() - t0
hx = KnnIndex(d, metric="euclidean")
hx.upload(host_rows)
rng = np.random.default_rng(1)
hfirst, hdraws = int(rng.integers(hn)), rng.random(hK - 1)
hx.kmeanspp(hK, hfirst, hdraws)
t0 = time.perf_counter()
hx.kmeanspp(hK, hfirst, hdraws)
dev_s = time.perf_counter() - t0
hx.release()
res["host_vs_device"] = {"n": hn, "K": hK, "host_init_kmeanspp_s": host_s, "device_s": dev_s, "cpus": os.cpu_count()}
print(f"host _init_kmeanspp at n={hn}, K={hK}: {host_s:.2f} s on {os.cpu_count()} CPUs; device: {dev_s * 1e3:.1f} ms")
if args.out:
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
