"""Times the cluster-routed search (nk_search_clusters_device) on the clustered corpus of SURVEY.md 8(d): N = 10M, d = 1024
fp32 (1000 centres, sigma 0.1, generated on the device), K = 1000 from a few device Lloyd passes.  For Q in {1, 64, 1024},
n_probe in {3, 10}, k = 10 it reports ms per batch (CUDA events around many device-resident calls after warm-up), the
algorithmic bytes (distinct probed clusters' rows + their member ids, from the returned probe lists), GB/s and the fraction of
a device-to-device copy peak measured in the same run, the scan kernel's own time (nk_index_scan_time_ms), nk_search_device on
the same queries and recall@k against it (routed search is approximate by definition).  Untimed checks: every returned score
equals an fp64 recomputation, and the device-resident and host-synchronous results are identical.

    python profiles/experiments/time_cluster_search.py [--n 10000000] [--out FILE.json]"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", ".."))
from nornicdb_b200.knn import KnnIndex  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--n", type=int, default=10_000_000)
ap.add_argument("--d", type=int, default=1024)
ap.add_argument("--K", type=int, default=1000)
ap.add_argument("--iters", type=int, default=50)
ap.add_argument("--out", default="")
args = ap.parse_args()
n, d, K, k = args.n, args.d, args.K, 10

card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                      capture_output=True, text=True).stdout.strip().splitlines()[0]
print(f"card: {card}")

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
print(f"copy peak: {peak:.0f} GB/s (read + write)")

ix = KnnIndex(d, metric="cosine")
ix.fill_clustered(n, seed=7, n_centres=1000, sigma=0.1)
rng = np.random.default_rng(0)
cen = ix.read_rows(0, 20 * K)[rng.choice(20 * K, K, replace=False)].astype(np.float32)
assign = np.zeros(n, np.int32)
for it in range(4):
    changed = ix.assign_nearest(cen, assign)
    cen, counts = ix.cluster_means(assign, cen)
    print(f"Lloyd pass {it}: {changed} changed, cluster sizes {counts.min()}..{counts.max()}")
ix.set_clusters(cen, assign)
sizes = np.bincount(assign, minlength=K)

results = []
for Q in (1, 64, 1024):
    qh = (ix.read_rows(int(rng.integers(0, n - Q)), Q) + rng.standard_normal((Q, d)).astype(np.float32) * 0.05).astype(np.float32)
    qd = torch.from_numpy(qh).cuda()
    oi = torch.empty((Q, k), dtype=torch.int32, device="cuda")
    os_ = torch.empty((Q, k), dtype=torch.float32, device="cuda")
    fi, fs = torch.empty_like(oi), torch.empty_like(os_)
    stream = torch.cuda.Stream()
    st = stream.cuda_stream
    for P in (3, 10):
        op = torch.empty((Q, P), dtype=torch.int32, device="cuda")
        for _ in range(5):
            ix.search_clusters_device(qd.data_ptr(), Q, k, P, oi.data_ptr(), os_.data_ptr(), op.data_ptr(), st)
        ix.status(st)
        e0.record(stream)
        for _ in range(args.iters):
            ix.search_clusters_device(qd.data_ptr(), Q, k, P, oi.data_ptr(), os_.data_ptr(), op.data_ptr(), st)
        e1.record(stream)
        ix.status(st)
        ms = e0.elapsed_time(e1) / args.iters
        ix.scan_time_ms()
        ix.enable_timing(True)  # the scan kernel alone, in a run of its own (the event pairs cost host time per call)
        for _ in range(args.iters):
            ix.search_clusters_device(qd.data_ptr(), Q, k, P, oi.data_ptr(), os_.data_ptr(), op.data_ptr(), st)
        ix.status(st)
        scan_ms, scans = ix.scan_time_ms()
        ix.enable_timing(False)
        scan_ms /= max(scans, 1)
        probes = op.cpu().numpy()
        distinct = np.unique(probes)
        nbytes = int(sizes[distinct].sum()) * (d * 4 + 4)
        for _ in range(3):
            ix.search_device(qd.data_ptr(), Q, k, fi.data_ptr(), fs.data_ptr(), st)
        e0.record(stream)
        for _ in range(max(5, args.iters // 5)):
            ix.search_device(qd.data_ptr(), Q, k, fi.data_ptr(), fs.data_ptr(), st)
        e1.record(stream)
        ix.status(st)
        full_ms = e0.elapsed_time(e1) / max(5, args.iters // 5)
        gi, gs = oi.cpu().numpy().view(np.uint32), os_.cpu().numpy()
        full = fi.cpu().numpy().view(np.uint32)
        recall = float(np.mean([len(set(gi[i]) & set(full[i])) / k for i in range(Q)]))
        # untimed checks: fp64 recomputation of every score, host-synchronous call identical
        hi, hs, hp = ix.search_clusters(qh, k, P, return_probes=True)
        same = bool((hi == gi).all() and (hs == gs).all() and (hp == probes).all())
        worst = 0.0
        for i in range(Q):
            rowsx = np.stack([ix.read_rows(int(r), 1)[0] for r in gi[i]]).astype(np.float64)
            qq = qh[i].astype(np.float64)
            ex = rowsx @ qq / (np.linalg.norm(rowsx, axis=1) * np.linalg.norm(qq))
            worst = max(worst, float((np.abs(ex - gs[i]) / np.maximum(np.abs(ex), 1e-6)).max()))
        r = dict(Q=Q, n_probe=P, k=k, ms=round(ms, 4), scan_ms=round(scan_ms, 4), bytes=nbytes, distinct_clusters=int(len(distinct)),
                 GBps=round(nbytes / (ms * 1e-3) / 1e9, 1), scan_GBps=round(nbytes / (scan_ms * 1e-3) / 1e9, 1),
                 frac_copy_peak_scan=round(nbytes / (scan_ms * 1e-3) / 1e9 / peak, 3), full_scan_ms=round(full_ms, 4),
                 recall_at_k=round(recall, 4), max_rel_score_err=worst, device_equals_host=same)
        results.append(r)
        print(json.dumps(r))

if args.out:
    os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(dict(card=card, copy_peak_GBps=peak, n=n, d=d, K=K, results=results), f, indent=1)
ix.release()
