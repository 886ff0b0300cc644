"""The measurement contract of bench.py, checked without a GPU: the committed bench lines under profiles/ (real B200 output of the
current bench.py) carry every key the driver reads, and the reference arm runs here on the CPU and prints its line."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def _line(name):
    return json.loads(open(os.path.join(ROOT, "profiles", name)).read().strip().splitlines()[-1])


def test_committed_bench_line_has_the_contract_keys():
    d = _line("r01d_bench.json")
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data",
              "config", "clocks", "gpu_launches", "e2e", "roofline", "cpu_baseline"):
        assert k in d, k
    assert d["unit"] == "pairs/s" and d["n_gpus"] == 1 and d["warmup"] >= 3 and d["higher_is_better"] is True and d["scaling"] == "weak"
    assert d["vs_baseline"] is None and d["data"] == "synthetic" and "workload" in d["config"] and "8192" in d["config"]["workload"]
    assert d["gpu_launches"] > 0 and d["config"]["exactness_errors"] == 0
    e = d["e2e"]
    assert e["unit"] == "pairs/s" and 0 < e["value"] < d["value"] and e["h2d_bytes_per_step"] == 100 * 8192 * 128 * 4 and e["d2h_bytes_per_step"] > 0
    r = d["roofline"]
    assert r["bound"] == "tensor" and r["unit"] == "TFLOP/s" and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9 and r["traffic"] > 0
    flop = d["value"] * r["flop_per_pair"] / 1e12
    assert 0.9 * r["achieved"] < flop <= r["achieved"] * 1.001          # kernel time <= step time
    c = d["cpu_baseline"]
    assert c["kind"] in ("reference", "port") and c["cores"] >= 1 and c["unit"] == "pairs/s" and c["value"] > 0 and c["sample"]
    assert d["clocks"]["sm_mhz"] and not {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"} & set(d["clocks"]["reasons"])
    assert d["cpu_baseline_cascade_hashing"]["value"] > c["value"]
    for n, name in ((2, "r01d_bench_2gpu.json"), (4, "r01d_bench_4gpu.json")):
        m = _line(name)
        assert m["n_gpus"] == n and m["value"] > 0.9 * n * d["value"] * 0.95 and abs(m["config"]["pairs_per_gpu"] - 4950) < 60
    h = _line("r01d_bench_hamming_40img.json")
    assert h["roofline"]["bound"] == "hbm" and h["roofline"]["unit"] == "GB/s" and h["dtype"] == "u32-popcount"


def test_round2_bench_lines():
    """Round-2 lines (same contract, `value` now timed until the records are in pinned host memory): single GPU, real-valued, multi-GPU, fixed lists."""
    d = _line("r02_bench.json")
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data",
              "config", "clocks", "gpu_launches", "e2e", "roofline", "cpu_baseline"):
        assert k in d, k
    assert d["n_gpus"] == 1 and d["warmup"] >= 3 and d["scaling"] == "weak" and d["vs_baseline"] is None and "8192" in d["config"]["workload"]
    assert d["config"]["exactness_errors"] == 0 and "pinned host memory" in d["config"]["value_timing"]
    e = d["e2e"]
    assert 0 < e["value"] < d["value"] and e["h2d_bytes_per_step"] == 100 * 8192 * (128 + 8) and e["d2h_bytes_per_step"] > 0     # uchar staging + positions
    r = d["roofline"]
    assert r["bound"] == "tensor" and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9 and r["traffic"] > 0
    assert 0.9 * r["achieved"] < d["value"] * r["flop_per_pair"] / 1e12 <= r["achieved"] * 1.001
    c = d["cpu_baseline"]
    assert c["kind"] == "reference" and c["cores"] == c["host"]["threads_used"] <= c["host"]["affinity_cpus"] and c["value"] > 0
    assert d["clocks"]["sm_mhz"] and not {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"} & set(d["clocks"]["reasons"])
    real = _line("r02_bench_real.json")
    assert real["config"]["real_valued_tensor_core_pairs"] == 4950 and real["config"]["tensor_core_pairs"] == 0 and real["config"]["exactness_errors"] == 0
    assert 0 < real["config"]["fallback_rows_fraction_of_queries"] < 0.01 and real["value"] > 0.5 * d["value"]
    ref = _line("r02_bench_reference_arm.json")
    assert ref["impl"] == "reference" and "100 synthetic images" in ref["config"]["workload"] and ref["cpu_baseline_cascade_hashing"]["value"] > ref["value"]
    for n, name in ((4, "r02_bench_4gpu.json"), (8, "r02_bench_8gpu.json")):
        m = _line(name)
        assert m["n_gpus"] == n and m["scaling"] == "weak" and abs(m["config"]["pairs_per_gpu"] - 4950) < 60
        assert m["config"]["max_views_on_a_gpu"] <= {4: 0.76, 8: 0.51}[n] * bench_images(n) + 1
        assert m["e2e"]["value"] > {4: 0.80, 8: 0.75}[n] * n * d["e2e"]["value"]          # the 4-GPU line predates the last kernel change (its own 1-GPU e2e was 73 k)
    c2 = _line("r02_bench_config2_8gpu.json"); c3 = _line("r02_bench_config3_4gpu.json")
    assert c2["n_gpus"] == 8 and c2["scaling"] == "strong" and "1000 synthetic images" in c2["config"]["workload"] and c2["config"]["max_views_on_a_gpu"] == 500
    assert c3["n_gpus"] == 4 and c3["scaling"] == "strong" and "500 synthetic images" in c3["config"]["workload"] and c3["roofline"]["bound"] == "hbm"


def bench_images(n):
    import bench
    return bench.IMAGES_FOR_GPUS[n]


def test_reference_arm_runs_on_the_cpu():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1", "--images", "4",
                        "--features", "256", "--cpu-seconds", "2"], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads(r.stdout.strip().splitlines()[-1])
    assert d["impl"] == "reference" and d["unit"] == "pairs/s" and d["value"] > 0 and d["higher_is_better"] is True
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"] == {"value": d["value"], "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    # under torchrun only rank 0 works: the others exit 0 without output
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"], capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_dump_outputs(tmp_path):
    """--dump-outputs: float32 / float64 arrays only; the sampled match lists are the returned records of the sampled pairs, the
    per-pair sums cover every record, and the sample is the same on every run."""
    import numpy as np
    import bench
    from alicevision_b200 import synth
    from alicevision_b200.matching import MATCH_DTYPE
    rng = np.random.default_rng(1)
    pairs = synth.exhaustive_pairs(40)
    offsets = np.concatenate([[0], np.cumsum(rng.integers(0, 30, len(pairs)))]).astype(np.int64)
    m = np.zeros(int(offsets[-1]), MATCH_DTYPE)
    m["i"] = rng.integers(0, 1 << 32, len(m)); m["j"] = rng.integers(0, 1 << 32, len(m)); m["ratio"] = rng.random(len(m)); m["dist"] = rng.random(len(m)) * 1e5
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), pairs, offsets, m, max_features=200000)
    got = {f[:-4]: np.load(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")}
    assert all(a.dtype in (np.float32, np.float64) for a in got.values())
    assert all(np.array_equal(a, np.load(tmp_path / "b" / f"{k}.npy")) for k, a in got.items())
    assert np.array_equal(got["pair_ids"], pairs) and np.array_equal(got["offsets"], offsets)
    sums = [m["dist"][a:b].astype(np.float64).sum() for a, b in zip(offsets[:-1], offsets[1:])]
    assert np.allclose(got["dist_sum_per_pair"], sums, rtol=1e-12)
    sample = got["sample_pair_index"].astype(np.int64)
    assert 0 < len(sample) < len(pairs) and np.all(np.diff(sample) > 0)      # 48 MB / (24 B x 200000 features): 10 pairs
    so = got["sample_offsets"].astype(np.int64)
    for k, p in enumerate(sample):
        want = m[offsets[p]:offsets[p + 1]]
        assert np.array_equal(got["sample_i"][so[k]:so[k + 1]], want["i"]) and np.array_equal(got["sample_j"][so[k]:so[k + 1]], want["j"])
        assert np.array_equal(got["sample_ratio"][so[k]:so[k + 1]], want["ratio"]) and np.array_equal(got["sample_dist"][so[k]:so[k + 1]], want["dist"])
