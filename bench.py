#!/usr/bin/env python
"""bench.py — image-pairs matched/sec on the descriptor-matching hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config 1|2|3|sweep]
                    [--features M] [--images I] [--dtype f32|u8|bin] [--data int|real] [--cpu-seconds S] [--dump-outputs DIR]

One "step" = one pass of the hot path over the rank's shard of the pair list.  Default (N=1): BASELINE configs[1],
100 synthetic images x 8192 SIFT features, exhaustive 4950 pairs.  Printed by rank 0 as ONE JSON line:

  value        whole-job pairs/s with the descriptors resident in HBM: CUDA-event time from the first enqueue of the step to
               the moment its LAST MATCH LIST HAS LANDED IN PINNED HOST MEMORY (search + exactness + packing + finishing
               kernels, D2H of the records); max over ranks
  e2e          the same pairs through the reference-facing C-ABI call chain with HOST buffers, wall clock:
               b200m_clear_views + b200m_upload_views_async (H2D inside) + b200m_match_pairs(STAGE_FULL) + result arrays
  roofline     dominant kernel (tcgen05 distance GEMM + fused top-2): 2*M^2*128 FLOP per pair / its own device time
  cpu_baseline the reference's CPU brute force (oracle/_ref, else the port) on a bounded sample of the same pairs

Multi-GPU (torchrun, one rank per GPU): pairs are independent, so the pair list is sharded (2-D blocks of the pair matrix,
b200m_shard_pairs_2d: a rank uploads only the views its blocks touch) and there is NO collective on the data path;
torch.distributed is used for the barrier and the max-over-ranks reduction of the timings only.
--config 1 (default): weak scaling, ~4950 pairs per GPU.  --config 2 / 3 = BASELINE configs[2] / [3]: a FIXED list
(1000 x 8k SIFT vocabulary-tree style / 500 x 16k AKAZE-MLDB exhaustive) split over the ranks: strong scaling.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from alicevision_b200 import synth  # noqa: E402

IMAGES_FOR_GPUS = {1: 100, 2: 141, 4: 199, 8: 282}   # exhaustive pairs ~ 4950 * N


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="1", choices=["1", "2", "3"],
                    help="1 = BASELINE configs[1] (weak scaling over --gpus); 2 = configs[2]: 1000 x 8k SIFT, vocabulary-tree style list, strong "
                         "scaling; 3 = configs[3]: 500 x 16k AKAZE-MLDB exhaustive, Hamming path, strong scaling")
    ap.add_argument("--features", type=int, default=0, help="features per image (default: 8192, 16384 for --config 3)")
    ap.add_argument("--images", type=int, default=0, help="0 = the configuration's image count")
    ap.add_argument("--dtype", default="f32", choices=["f32", "u8", "bin"])
    ap.add_argument("--data", default="int", choices=["int", "real"], help="real = real-valued fp32 descriptors (not integer-valued)")
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="budget of the cpu_baseline sample")
    ap.add_argument("--tc-variant", type=int, default=4, choices=[1, 2, 3, 4], help="4 = CTA-pair tcgen05 kernel, half-norms folded into the GEMM (default); 2/3 = CTA pair with epilogue add (8/16 epilogue warps); 1 = single-CTA kernel")
    ap.add_argument("--pairs", default="", choices=["", "exhaustive", "voctree"],
                    help="voctree = synthetic vocabulary-tree style list, 50 neighbours per image (default for --config 2)")
    ap.add_argument("--sharding", default="2d", choices=["2d", "rows"], help="multi-rank split of the pair list: 2-D blocks (default) or by database image")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write what the last timed step returned to DIR/<name>.npy (float32 / float64, a seeded sample of the match lists)")
    a = ap.parse_args()
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs dumps the GPU path (--impl ours)")
    if a.config == "3":
        a.dtype = "bin"
    a.features = a.features or (16384 if a.config == "3" else 8192)
    a.pairs = a.pairs or ("voctree" if a.config == "2" else "exhaustive")
    return a


def n_images(args, world):
    if args.images:
        return args.images
    return {"1": IMAGES_FOR_GPUS.get(world, 100 * world), "2": 1000, "3": 500}[args.config]


def make_pairs(args, n_img):
    return synth.voctree_like_pairs(n_img, k=50) if args.pairs == "voctree" else synth.exhaustive_pairs(n_img)


def make_views(args, n_img, needed=None):
    """{image index: (descriptors, positions)} for the images in `needed` (all when None).  The default workload keeps round 1's
    sequential generator; the large fixed lists (--config 2 / 3) use the indexed one so that a rank builds only its own views."""
    if args.config == "1" and needed is None:
        if args.dtype == "bin":
            descs, xys = synth.mldb_images(n_img, args.features, seed=synth.SEED_DATA)
        else:
            descs, xys = synth.sift_images(n_img, args.features, np.float32 if args.dtype == "f32" else np.uint8, seed=synth.SEED_DATA, pool_factor=1.0)
            if args.data == "real":
                descs = synth.real_valued(descs)
        return {i: (descs[i], xys[i]) for i in range(n_img)}
    ids = range(n_img) if needed is None else sorted(needed)
    gen = synth.IndexedImages(args.features, "bin" if args.dtype == "bin" else ("f32" if args.dtype == "f32" else "u8"), seed=synth.SEED_DATA,
                              real=args.data == "real")
    return {i: gen(i) for i in ids}


def shard_pairs(pairs: np.ndarray, rank: int, world: int, how: str) -> np.ndarray:
    """This rank's shard.  2d: folded 2-D blocks of the pair matrix (b200m_shard_pairs_2d: the rank needs only part of the
    views); rows: database images dealt round-robin (b200m_shard_pairs, round 1).  Same host functions the single-process
    multi-GPU path uses."""
    if world == 1:
        return pairs
    from alicevision_b200 import matching
    s = matching.shard_pairs_2d(pairs, world) if how == "2d" else matching.shard_pairs(pairs, world)
    return pairs[s == rank]


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md clocks line)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.rows = []
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [x.strip() for x in line.split(",")]))

    def stop(self, t0: float, t1: float) -> dict:
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        rows = [r for t, r in self.rows if t0 <= t <= t1 and len(r) >= 9] or [r for _, r in self.rows if len(r) >= 9]
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        sm = sorted(float(r[1]) for r in rows)
        reasons = set()
        for r in rows:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(rows[0][2]), "power_w_max": max(float(r[3]) for r in rows),
                "samples": len(rows), "reasons": sorted(reasons)}


def physical_cores() -> int:
    """Physical cores this process may run on (SURVEY 8d: "all physical cores"); falls back to the affinity count."""
    allowed = os.sched_getaffinity(0)
    try:
        cores, cpu, phys = set(), None, None
        for line in open("/proc/cpuinfo"):
            k, _, v = line.partition(":")
            k = k.strip()
            if k == "processor":
                cpu, phys = int(v), None
            elif k == "physical id":
                phys = int(v)
            elif k == "core id" and cpu in allowed:
                cores.add((phys, int(v)))
        return len(cores) or len(allowed)
    except Exception:
        return len(allowed)


def cgroup_cpu_quota():
    """CPUs the container may actually USE (cgroup v2 cpu.max / v1 cfs quota), or None when unlimited.  The affinity mask of a GPU
    lease can list 64 cores while the quota allows far fewer: round 1's reference arm swung 4.4x between two such boxes."""
    try:
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max":
            return float(q) / float(p)
    except Exception:
        pass
    try:
        q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read()); p = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
        if q > 0:
            return q / p
    except Exception:
        pass
    return None


def host_cores() -> int:
    """Threads worth using: physical cores in the affinity mask, capped by the cgroup CPU quota."""
    n = physical_cores()
    q = cgroup_cpu_quota()
    return max(1, min(n, int(q + 0.5))) if q else n


def cores_info() -> dict:
    return {"affinity_cpus": len(os.sched_getaffinity(0)), "physical_cores": physical_cores(), "cgroup_cpu_quota": cgroup_cpu_quota(), "threads_used": host_cores()}


def cpu_baseline(views, pairs, hamming, budget_s):
    """The reference's CPU brute force (+ ratio test + de-duplication) on a bounded sample of the same pair list."""
    import oracle
    ora = oracle.best()
    ora.set_num_threads(host_cores())   # torchrun exports OMP_NUM_THREADS=1; the baseline gets every core this process may really use
    n = 0
    t0 = time.perf_counter()
    while n < len(pairs) and (time.perf_counter() - t0) < budget_s:
        i, j = int(pairs[n, 0]), int(pairs[n, 1])
        ora.regions_match(views[i][0], views[i][1], views[j][0], views[j][1], 0.8, hamming)
        n += 1
    dt = time.perf_counter() - t0
    return {"value": n / dt, "unit": "pairs/s", "cores": ora.num_threads(), "kind": "reference" if ora.kind == "ref" else "port", "host": cores_info(),
            "sample": f"{n} pairs of the same list (every k-th), {dt:.1f} s, ArrayMatcher_bruteForce + ratio test + de-duplication, "
                      f"{'g++ -O3 -msse2 -fopenmp on the reference headers' if ora.kind == 'ref' else 'C++ port of the reference'}"}


def cpu_baseline_cascade(views, pairs, budget_s):
    """The reference's CASCADE_HASHING_L2 matcher (matching/ArrayMatcher_cascadeHashing.hpp + CascadeHasher.hpp compiled from the
    reference tree into oracle/_ref) through the restated collection loop: one hashed database per image I, OpenMP over its J images
    (ImageCollectionMatcher_generic.cpp:39,68).  Whole database rows of the same pair list until the budget is used.  None when
    the compiled reference is not available (the port does not restate cascade hashing)."""
    import oracle
    if not oracle.available("ref"):
        return None
    ora = oracle.Oracle("ref")
    ora.set_num_threads(host_cores())
    firsts = np.unique(pairs[:, 0])
    ids = sorted(views)
    pos = {v: k for k, v in enumerate(ids)}
    descs = [views[v][0] for v in ids]; xys = [views[v][1] for v in ids]
    n = 0; matches = 0
    t0 = time.perf_counter()
    for f in firsts:
        row = pairs[pairs[:, 0] == f]
        local = np.array([[pos[int(a)], pos[int(b)]] for a, b in row], np.uint32)
        tot, _ = ora.collection_cascade(descs, xys, local, 0.8)
        n += len(row); matches += tot
        if time.perf_counter() - t0 > budget_s:
            break
    dt = time.perf_counter() - t0
    return {"value": n / dt, "unit": "pairs/s", "cores": ora.num_threads(), "kind": "reference",
            "sample": f"first {n} pairs (whole database rows) of the same list, {dt:.1f} s, ArrayMatcher_cascadeHashing + ratio test + de-duplication, database "
                      f"hashed once per image I, OpenMP over J as in ImageCollectionMatcher_generic; {matches} matches; g++ -O3 -msse2 -fopenmp on the "
                      "reference headers with plain-loop stand-ins for Eigen's MatrixXf/VectorXf (timing baseline, results unpinned)"}


def ncu_traffic(kernel_key: str):
    """DRAM bytes per launch of the dominant kernel from the committed `ncu --set full` capture (profiles/traffic.json), or None."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        return json.load(open(p)).get(kernel_key)
    except Exception:
        return None


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("bf16_tflops_sustained", 1449.7), "measured (MEASURED_PEAKS.json bf16_tflops_sustained: kernel timed inside a long step)"
    return 1400.0, "fallback (B200_PROFILING.md: ~1.4 PFLOP/s sustained)"


def burst_peak():
    """The burst (kernel-timed-alone) bf16 figure of MEASURED_PEAKS.json, reported next to `frac` because the sustained figure was taken at a
    1372 MHz median clock under random data and this kernel holds a higher clock: a `frac` above 1 is a statement about clocks, not about the pipe."""
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        return float(json.load(open(p)).get("bf16_tflops"))
    except Exception:
        return None


def workload_text(args, n_img, n_pairs):
    hamming = args.dtype == "bin"
    return (f"{n_img} synthetic images x {args.features} {'MLDB 64-byte' if hamming else 'SIFT 128-D ' + args.dtype + (' real-valued' if args.data == 'real' else '')} features, "
            f"{'vocabulary-tree style (50 neighbours/image)' if args.pairs == 'voctree' else 'exhaustive'} {int(n_pairs)} ordered pairs, "
            f"BRUTE_FORCE_{'HAMMING' if hamming else 'L2'}, ratio 0.8")


DUMP_SAMPLE_BYTES = 48 << 20     # the sampled match lists; the per-pair arrays add well under 1 MB at 4950 pairs


def dump_outputs(out_dir, pair_ids, offsets, matches, max_features):
    """What the timed path returned (pair ids, CSR offsets, match records i / j / ratio / dist) as DIR/<name>.npy in float64 /
    float32: the pair list and offsets, per-pair sums of ratio and dist over every match, and the complete match lists of a
    seeded sample of pairs.  The sample depends on the inputs only (pair count, features per view: at most one match per query
    feature), so two builds dump the same pairs, and it is sized to keep the files under 64 MB."""
    os.makedirs(out_dir, exist_ok=True)
    n = len(pair_ids)
    counts = np.diff(offsets)
    owner = np.repeat(np.arange(n), counts)
    k = min(n, max(1, DUMP_SAMPLE_BYTES // (24 * max(1, max_features))))
    sample = np.sort(np.random.default_rng(0).permutation(n)[:k])
    rows = np.concatenate([np.arange(offsets[p], offsets[p + 1]) for p in sample]) if k else np.zeros(0, np.int64)
    arrays = {"pair_ids": pair_ids.astype(np.float64), "offsets": offsets.astype(np.float64),
              "ratio_sum_per_pair": np.bincount(owner, weights=matches["ratio"], minlength=n),
              "dist_sum_per_pair": np.bincount(owner, weights=matches["dist"], minlength=n),
              "sample_pair_index": sample.astype(np.float64), "sample_offsets": np.concatenate([[0], np.cumsum(counts[sample])]).astype(np.float64),
              "sample_i": matches["i"][rows].astype(np.float64), "sample_j": matches["j"][rows].astype(np.float64),
              "sample_ratio": matches["ratio"][rows], "sample_dist": matches["dist"][rows]}
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), np.ascontiguousarray(a))


def pin_to_gpu_numa_node(local: int) -> str:
    """One rank per GPU on a two-socket host: keep this process (its pinned buffers, the engine's threads) on the GPU's NUMA node."""
    try:
        import torch
        bus = torch.cuda.get_device_properties(local).pci_bus_id if hasattr(torch.cuda.get_device_properties(local), "pci_bus_id") else None
        dom = torch.cuda.get_device_properties(local).pci_domain_id if bus is not None else 0
        if bus is None:
            return "unknown"
        dev = torch.cuda.get_device_properties(local).pci_device_id
        path = f"/sys/bus/pci/devices/{dom:04x}:{bus:02x}:{dev:02x}.0/numa_node"
        node = int(open(path).read())
        if node < 0:
            return "no numa node"
        cpus = set()
        for tok in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = tok.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if len(cpus) >= 2:
            os.sched_setaffinity(0, cpus)
            return f"node {node} ({len(cpus)} cpus)"
        return f"node {node} (not pinned)"
    except Exception as e:      # noqa: BLE001
        return f"not pinned ({type(e).__name__})"


def reference_arm(args, rank):
    """The reference's own CPU implementation on the box's host cores, rank 0 only: the SAME configuration as our arm at N=1 (same
    images, same pair list), every step a bounded sample of its pairs spread over the whole list."""
    if rank != 0:
        return
    hamming = args.dtype == "bin"
    n_img = n_images(args, 1)
    pairs = make_pairs(args, n_img)
    per_step_s = max(2.0, args.cpu_seconds / 2)
    # ~per_step_s of CPU work per step: the views of a sample are generated first, so bound the sample by what a step can match
    stride = max(1, len(pairs) // 256)
    sample_ids = sorted({int(v) for s in range(4) for v in pairs[s::stride * 4][:64].reshape(-1)}) if args.config != "1" else None
    views = make_views(args, n_img, sample_ids)
    per_step = []
    for s in range(args.warmup + args.steps):
        sub = pairs[s % 4::stride * 4][:64] if args.config != "1" else pairs[s % 4::4]
        sub = sub[np.random.default_rng(s).permutation(len(sub))] if args.config == "1" else sub     # spread over the list, not its first rows
        b = cpu_baseline(views, sub, hamming, per_step_s)
        if s >= args.warmup:
            per_step.append(b)
    v = float(np.mean([b["value"] for b in per_step])) if per_step else 0.0
    cb = dict(per_step[-1]) if per_step else {"kind": "port", "cores": 0, "sample": ""}
    cb["value"] = v
    out = {"impl": "reference", "metric": metric_name(args), "value": v, "unit": "pairs/s", "n_gpus": args.gpus, "steps": args.steps,
           "warmup": args.warmup, "ms_per_step": None, "higher_is_better": True, "scaling": "weak" if args.config == "1" else "strong", "vs_baseline": None,
           "dtype": "f32" if args.dtype == "f32" else args.dtype, "data": "synthetic",
           "config": {"workload": workload_text(args, n_img, len(pairs)), "sampled": "each step matches a bounded random sample of this list on the CPU"},
           "cpu_baseline": cb, "e2e": {"value": v, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    if not hamming and not args.no_cpu:       # the north star's second CPU baseline
        cc = cpu_baseline_cascade(views, pairs if args.config == "1" else pairs[::stride * 4][:64], max(2.0, args.cpu_seconds / 3))
        if cc:
            out["cpu_baseline_cascade_hashing"] = cc
    print(json.dumps(out))


def metric_name(args):
    hamming = args.dtype == "bin"
    return "image-pairs matched/sec (" + ("AKAZE-MLDB 64-byte, " if hamming else "SIFT 128-D, ") + f"{args.features} feat/img)"


def main():
    args = parse()
    rank = int(os.environ.get("RANK", 0)); world = int(os.environ.get("WORLD_SIZE", 1)); local = int(os.environ.get("LOCAL_RANK", 0))
    hamming = args.dtype == "bin"

    if args.impl == "reference":
        reference_arm(args, rank)
        return

    import torch
    import torch.distributed as dist
    from alicevision_b200 import EMatcherType, ImageCollectionMatcherB200, matching

    torch.cuda.set_device(local)
    numa = "single rank"
    if world > 1:
        # one engine process per GPU shares the host: stay on the GPU's NUMA node, split the cores between the ranks' pools and
        # keep fewer staging copies in flight per rank (profiles/r01d_multi_rank_host_settings.md)
        numa = pin_to_gpu_numa_node(local)
        # threads of this rank's staging / finishing pool: the CPUs it may use (after the pinning: one NUMA node) shared with the other
        # ranks on the same node, capped by the container's CPU quota split over all ranks
        sharing = max(1, world // 2) if numa.startswith("node") else world
        q = cgroup_cpu_quota()
        per_rank = min(len(os.sched_getaffinity(0)) // sharing, int(q // world) if q else 1 << 30)
        os.environ.setdefault("B200M_HOST_THREADS", str(max(6, min(32, per_rank))))
        os.environ.setdefault("B200M_UP_LAG", "6")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    n_img = n_images(args, world)
    pairs = make_pairs(args, n_img)
    mine = shard_pairs(pairs, rank, world, args.sharding)
    needed = sorted({int(v) for v in mine.reshape(-1)})
    views = make_views(args, n_img, needed if (args.config != "1") else None)
    my_views = {v: views[v] for v in needed}
    ctx = matching.Context(local)
    ctx.set_tc_variant(args.tc_variant)
    m = ImageCollectionMatcherB200(0.8, False, EMatcherType.BRUTE_FORCE_HAMMING_B200 if hamming else EMatcherType.BRUTE_FORCE_L2_B200, ctx)
    m.upload(my_views)

    # ---- value: descriptors resident in HBM; timed until the last match list has landed in pinned host memory ---------
    for _ in range(args.warmup):
        m.match_uploaded(mine, matching.STAGE_FULL)
    sampler = ClockSampler(local) if rank == 0 else None
    barrier()
    t0w = time.time()
    gpu_ms = 0.0; search_ms = 0.0; launches = 0; records = 0
    last = None
    for _ in range(args.steps):
        last = None                                   # a step's result is freed before the next step runs
        last = m.match_uploaded(mine, matching.STAGE_FULL)
        gpu_ms += ctx.last_gpu_ms(); search_ms += ctx.last_search_kernel_ms(); launches += ctx.last_launches(); records += ctx.last_records()
    barrier()
    t1w = time.time()
    clocks = sampler.stop(t0w, t1w) if sampler else None
    tc_pairs = ctx.last_tc_pairs(); errs = ctx.exactness_errors(); real_pairs = ctx.last_real_tc_pairs(); fb_rows = ctx.last_fallback_rows()
    if args.dump_outputs and last is not None:
        dump_outputs(args.dump_outputs if world == 1 else os.path.join(args.dump_outputs, f"rank{rank}"), *last,
                     max((len(d) for d, _ in my_views.values()), default=1))
    last = None

    # ---- e2e: host buffers -> upload -> match -> D2H -> finishing -> result arrays -------------------------------------
    e2e_s = 0.0; h2d = 0; d2h = 0; e2e_steps = 0
    if not args.no_e2e:
        m.clear(); m.Match(my_views, mine)            # warm-up of the full chain
        barrier()
        e2e_steps = max(1, min(args.steps, 3))
        te = time.perf_counter()
        for _ in range(e2e_steps):
            m.clear()
            res = m.Match(my_views, mine)
            n_matches = res.num_matches()             # offsets / matches arrays of the result are in host memory here
        barrier()
        e2e_s = (time.perf_counter() - te) / e2e_steps
        # bytes that cross PCIe: integer-valued fp32 descriptors are staged as uchar (1 byte per component); positions 8 B per feature
        esz = 1 if (args.dtype != "f32" or args.data == "int") else 4
        h2d = int(sum(d.shape[0] * d.shape[1] * esz + x.nbytes for d, x in my_views.values()))
        d2h = int(ctx.last_records() * 16 + len(mine) * 12)
        del res

    # ---- reduce over ranks (max time, total pairs) ------------------------------------------------------------------
    stats = torch.tensor([gpu_ms / args.steps, search_ms / args.steps, (t1w - t0w) * 1e3 / args.steps, e2e_s * 1e3], dtype=torch.float64, device="cuda")
    tot = torch.tensor([float(len(mine)), float(launches), float(records), float(errs), float(tc_pairs), float(h2d), float(d2h), float(len(needed)),
                        float(real_pairs), float(fb_rows)], dtype=torch.float64, device="cuda")
    mx = torch.tensor([float(len(mine)), float(len(needed))], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(stats, op=dist.ReduceOp.MAX)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
    ms_step, ms_search, ms_wall, ms_e2e = stats.tolist()
    n_pairs, launches, records, errs, tc_pairs, h2d, d2h, views_sum, real_pairs, fb_rows = tot.tolist()

    if rank == 0:
        M = args.features
        flop_pair = 2.0 * M * M * 128
        peak, peak_src = peaks()
        # the roofline kernel's rate on ONE GPU: the slowest rank's search-kernel time against the largest shard
        achieved = mx[0].item() * flop_pair / (ms_search * 1e-3) / 1e12 if not hamming else None
        out = {
            "metric": metric_name(args), "value": n_pairs / (ms_step * 1e-3), "unit": "pairs/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak" if args.config == "1" else "strong", "vs_baseline": None,
            "dtype": "u32-popcount" if hamming else ("f16 (fp16 operands, fp32 accumulate; exact on integer-valued SIFT)" if args.data == "int" else
                                                     "f32 results (fp16-rounded tensor-core filter + exact fp32 re-scoring)" if real_pairs > 0 else "f32 (real-valued descriptors, CUDA cores)"),
            "data": "synthetic",
            "config": {"workload": workload_text(args, n_img, n_pairs),
                       "pairs_per_gpu": n_pairs / world, "max_pairs_on_a_gpu": mx[0].item(), "views_per_gpu": views_sum / world, "max_views_on_a_gpu": mx[1].item(),
                       "sharding": ("2-D blocks of the pair matrix (b200m_shard_pairs_2d)" if args.sharding == "2d" else "pairs dealt round-robin by database image") + ", no collective on the data path",
                       "l2_policy": f"inputs larger than L2 ({mx[1].item() * M * (64 if hamming else 256) / 1e6:.0f} MB of resident descriptors per GPU vs 126 MB L2)",
                       "value_timing": "CUDA events: first enqueue of the step -> last match list landed in pinned host memory (b200m_match_pairs STAGE_FULL on resident views)",
                       "tensor_core_pairs": tc_pairs, "real_valued_tensor_core_pairs": real_pairs,
                       "fallback_rows_per_step": fb_rows, "fallback_rows_fraction_of_queries": (fb_rows / (real_pairs * M)) if real_pairs else 0.0,
                       "exactness_errors": errs, "wall_ms_per_step": ms_wall, "records_per_step": records / args.steps,
                       "host": cores_info(), "numa": numa},
            "clocks": clocks, "gpu_launches": int(launches),
            "e2e": {"value": (n_pairs / (ms_e2e * 1e-3)) if ms_e2e > 0 else None, "unit": "pairs/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "steps": e2e_steps,
                    "what": "b200m_clear_views + b200m_upload_views_async (every view the shard references, from pageable host memory; integer-valued fp32 staged as "
                            "uchar) + b200m_match_pairs(STAGE_FULL): H2D overlapped with the first pairs, kernels incl. device-side finishing, D2H, result assembly "
                            "in PairSet order; wall clock, max over ranks"},
        }
        if hamming:
            hb = mx[0].item() * 2.0 * M * 64 / (ms_search * 1e-3) / 1e9
            hp = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))).get("hbm_gbs", 6650.0) if os.path.exists(os.path.join(ROOT, "MEASURED_PEAKS.json")) else 6650.0
            tr = ncu_traffic("hamming_top2_kernel")
            out["roofline"] = {"bound": "hbm", "achieved": hb, "peak": hp, "unit": "GB/s", "frac": hb / hp, "traffic": tr["dram_bytes_per_launch"] if tr else None,
                               "traffic_note": tr["note"] if tr else None, "kernel": "hamming_top2_kernel", "kernel_ms_per_step": ms_search,
                               "note": "integer-ALU bound by construction (M^2 x (16 XOR + 22 LOP3 + 5 POPC) per pair vs 2*M*64 bytes); HBM fraction reported because the north star asks"}
        else:
            tr = (ncu_traffic("l2_top2_tc2_kernel") if tc_pairs > 0 else ncu_traffic("l2_top2_tc2_kernel_real") if real_pairs > 0 else None) if (args.tc_variant == 4 and M == 8192) else None
            kern = {1: "tc::l2_top2_tc_kernel", 2: "tc2::l2_top2_tc2_kernel<8,false> (cta_group::2)", 3: "tc2::l2_top2_tc2_kernel<16,false> (cta_group::2)",
                    4: "tc2::l2_top2_tc2_kernel<8,true> (cta_group::2, K=128+16)"}[args.tc_variant] if tc_pairs > 0 else (
                        "tc2::l2_top2_tc2_kernel<8,true,MODE_REAL> (cta_group::2, fp16-rounded filter GEMM, K=128+16) + exact re-scoring in the reference's fp32 order + exact_rows fallback"
                        if real_pairs > 0 else "exact_top2_kernel<float> (CUDA cores, reference summation order)")
            out["roofline"] = {"bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                               "traffic": tr["dram_bytes_per_launch"] if tr else None, "traffic_note": tr["note"] if tr else None,
                               "kernel": kern, "peak_source": peak_src, "flop_per_pair": flop_pair, "kernel_ms_per_step": ms_search,
                               "peak_burst": burst_peak(), "frac_of_burst_peak": (achieved / burst_peak()) if burst_peak() else None,
                               "ncu_tensor_pipe_pct": tr.get("tensor_pipe_pct") if tr else None}
        if not args.no_cpu and world == 1:      # contract: the CPU baseline is timed on rank 0 at N=1 only
            sub = pairs[np.random.default_rng(0).permutation(len(pairs))] if args.config == "1" else np.array([p for p in pairs if int(p[0]) in views and int(p[1]) in views], np.uint32)
            out["cpu_baseline"] = cpu_baseline(views, sub, hamming, args.cpu_seconds)
            if not hamming:                     # the north star also names the reference's cascade-hashing matcher (scalar descriptors only)
                cb = cpu_baseline_cascade(views, pairs, max(2.0, args.cpu_seconds / 3))
                if cb:
                    out["cpu_baseline_cascade_hashing"] = cb
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
