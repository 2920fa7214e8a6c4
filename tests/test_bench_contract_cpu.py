"""bench.py's output contract, checked without a GPU: helpers import, every workload BASELINE.json names is defined, and
the committed bench lines (profiles/bench_r1.jsonl, profiles/bench_r2.jsonl, produced by bench.py on B200 boxes) carry every
key the driver reads — round 2 also the in-run parity check and the north_star grid."""
import json
import os

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REQUIRED = ["metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
            "dtype", "data", "config", "roofline", "e2e", "clocks", "gpu_launches"]


def test_bench_helpers_and_workloads():
    import bench
    assert set(["headline", "c1", "c2", "c3", "c4", "c5", "q1"]) <= set(bench.WORKLOADS)
    n, d, dt, Q, k, metric, _ = bench.WORKLOADS["headline"]
    assert (n, d, dt, Q, k, metric) == (10_000_000, 1024, "f32", 64, 10, "cosine")   # BASELINE.json metric shape
    assert bench.WORKLOADS["c3"][:6] == (10_000_000, 1024, "f32", 1024, 100, "dot")
    assert bench.WORKLOADS["c4"][:6] == (10_000_000, 768, "f16", 1, 10, "euclidean")
    assert bench.WORKLOADS["c5"][:6] == (100_000_000, 1024, "f32", 1024, 10, "cosine")
    peak, src = bench.load_peaks()
    assert 3000 < peak < 9000 and ("measured" in src or "fallback" in src)
    tf32, _ = bench.load_tensor_peak()
    bf16, _ = bench.load_tensor_peak(bf16=True)
    assert abs(bf16 - 2 * tf32) < 1e-6
    assert bench.load_traffic("headline", "shadow") > 2.0e10 and bench.load_traffic("headline", "filter") > 4.0e10


def test_committed_bench_lines_follow_the_contract():
    lines = [json.loads(l) for l in open(os.path.join(ROOT, "profiles", "bench_r1.jsonl"))]
    ours = [d for d in lines if d.get("impl") != "reference"]
    ref = [d for d in lines if d.get("impl") == "reference"]
    assert ours and ref
    for d in ours:
        for key in REQUIRED:
            assert key in d, (d.get("run"), key)
        assert d["metric"] == "kNN queries/sec" and d["unit"] == "queries/s" and d["higher_is_better"] is True
        assert d["vs_baseline"] is None and d["data"] == "synthetic" and d["scaling"] == "strong"
        r = d["roofline"]
        assert r["bound"] in ("hbm", "tensor") and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9 and r["unit"] in ("GB/s", "TFLOP/s")
        e = d["e2e"]
        assert e["unit"] == "queries/s" and e["h2d_bytes_per_step"] > 0 and e["d2h_bytes_per_step"] > 0 and e["value"] > 0
        assert d["gpu_launches"] > 0 and "workload" in d["config"] and "model" not in d["config"]
        assert "sm_mhz" in d["clocks"] and "reasons" in d["clocks"]
        assert not set(d["clocks"]["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}
    default = [d for d in ours if d.get("run", "").startswith("default")][0]
    cb = default["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["unit"] == "queries/s" and "sample" in cb
    for d in ref:
        assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0 and d["cpu_baseline"]["value"] == d["value"]


def test_round2_bench_lines_carry_parity_check_and_grid():
    lines = [json.loads(l) for l in open(os.path.join(ROOT, "profiles", "bench_r2.jsonl"))]
    by = {d["run"]: d for d in lines}
    for d in lines:
        for key in REQUIRED + ["scan", "timing"]:
            assert key in d, (d["run"], key)
        assert "scan" not in d["config"]  # moved to the top level so the two arms' configs compare equal
        pc = d.get("parity_check")
        if pc is None:  # the NCCL-exchange comparison run was taken with --no-parity
            assert "nccl" in d["run"], d["run"]
            continue
        # every returned score is recomputed (bounded at 4096 row read-backs per rank for the Q=1024, k=100 shape)
        assert pc["ok"] is True and pc["scores_recomputed_fp64"] >= min(d["config"]["Q"] * d["config"]["k"], 4096 * d["n_gpus"]), (d["run"], pc)
        assert d["e2e"]["value"] <= d["value"] * 1.02, d["run"]  # one clock per quantity: e2e never beats device-resident
        r = d["roofline"]
        assert abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9
    one = by["default_1gpu"]
    want = {"c3", "c3_k10", "q1", "k100", "headline_filter", "q1_simt", "headline_clustered", "c4", "c4_q64", "c2", "c1"}
    assert want <= set(one["also"]), sorted(set(one["also"]))
    for name, e in one["also"].items():
        assert "error" not in e, (name, e)
        assert e["ms_per_step"] > 0 and 0 < e["roofline_frac"] < 1.25 and e["bound"] in ("hbm", "tensor")
    assert one["also"]["headline_clustered"]["filter_retries"]["first_stage_retry_rate"] <= 0.05  # the round-1 cliff
    assert one["also"]["headline_clustered"]["filter_retries"]["exact_stage_rate"] <= 0.05
    st = one["cpu_baseline"]["single_thread"]
    assert st["cores"] == 1 and st["value"] > 0 and one["cpu_baseline"]["value"] >= st["value"] * 0.9
    for name in ("headline_8gpu_peer", "c5_8gpu_peer"):
        checks = " ".join(by[name]["parity_check"]["checks"])
        assert "bit-identical to nk_index_create(devices=0..7) + nk_search" in checks, name
    assert by["headline_8gpu_peer"]["exchange"].startswith("peer-memory")
    c5 = by["default_8gpu"]["also"]["c5"]  # configs[4] rides on the default 8-GPU command
    assert c5["parity_check"]["ok"] is True and c5["rows_per_gpu"] == 12_500_000 and c5["value"] > 0


def test_dump_outputs_writes_the_result_as_npy(tmp_path):
    import numpy as np
    import torch
    import bench
    idx = torch.arange(12, dtype=torch.int32).reshape(3, 4)
    idx[0, 0] = -1  # row id 2**32 - 1, as the C ABI's uint32 lands in the int32 buffer
    score = torch.linspace(1, 0, 12).reshape(3, 4)
    bench.dump_outputs(str(tmp_path / "a"), idx, score, 3)  # k' = min(k, N) = 3: the 4th column is never written
    i, s = np.load(tmp_path / "a" / "indices.npy"), np.load(tmp_path / "a" / "scores.npy")
    assert i.dtype == np.float64 and s.dtype == np.float32 and i.shape == s.shape == (3, 3)
    assert i[0, 0] == 2 ** 32 - 1 and i[1].tolist() == [4, 5, 6] and (s == score[:, :3].numpy()).all()
    assert not (tmp_path / "a" / "query_rows.npy").exists()
    # above the size limit: the same seeded sample of queries every time, within 64 MB in all
    Q, k = 600_000, 10
    idx = torch.arange(Q * k, dtype=torch.int32).reshape(Q, k)
    score = idx.float()
    for d in ("b", "c"):
        bench.dump_outputs(str(tmp_path / d), idx, score, k)
    files = sorted(p.name for p in (tmp_path / "b").iterdir())
    assert files == ["indices.npy", "query_rows.npy", "scores.npy"]
    assert sum((tmp_path / "b" / f).stat().st_size for f in files) <= 64 << 20
    rows = np.load(tmp_path / "b" / "query_rows.npy")
    assert (np.diff(rows) > 0).all() and (rows == np.load(tmp_path / "c" / "query_rows.npy")).all()
    i = np.load(tmp_path / "b" / "indices.npy")
    assert (i == rows[:, None] * k + np.arange(k)).all()
