#!/usr/bin/env python
"""Benchmarks of the batched-search hot path on B200, one JSON line per run (contract: see the task statement).

  --config c3 (default)  BASELINE.json configs[2], the headline: Tree-AH 10M x 96 clustered unit vectors, K-means 2000
                         partitions, AsymmetricHasher 4-bit LUT16 with dims_per_block = 2 (S = 48), leaves_to_search =
                         64, reorder = 100, k = 10, DotProduct, 10k-query batches.
  --config c1 | c2       configs[0] / configs[1]: BruteForceSearcher SquaredL2 10k x 128 (1k queries) / DotProduct
                         1M x 128 (10k-query batch; --sq8 for the ScalarQuantized Int8 searcher).  Roofline = tensor.
  --config c4            configs[3]: Tree-X-Hybrid SquaredL2, 8192 partitions, 100M x 128 sharded by whole partitions
                         over the ranks (rows are generated per rank and exchanged to their owners), NCCL top-k merge,
                         leaves_to_search sweep, parity properties checked in the run.
  --config c5            configs[4]: Tree-AH over 1B x 96 PQ codes (24 B codes + u32 id per vector, no raw rows, no
                         reorder), K = 65,536, sharded over the ranks, leaves_to_search sweep (recall vs QPS).

A "step" = one search_batched pass of the hot path over one batch of --nq synthetic queries.
  value    queries/s with the query batch already resident in HBM (device pointers through the C ABI),
           timed with CUDA events over exactly --steps steps, max over ranks
  e2e      the same through the reference-facing host API: pinned host query buffer in, host results
           out, H2D/D2H copies inside the timed region
  roofline the dominant kernel of the step: algorithmic bytes (or flops) per launch / its device time measured live
           with CUDA events recorded around the kernel on its stream
  cpu_baseline  the CPU oracle (C++ restatement of the reference algorithm, all host threads) on a bounded
           sample of the same workload
--impl reference times that CPU arm alone (the reference crate is Rust and cannot be built here); it builds its index
with plain torch ops (oracle/ref_index.py) and never builds, loads or calls libscann_b200.so.
Multi-GPU (torchrun, one rank per GPU): the index is sharded by whole partitions (shard plan balanced on the probe
load of a calibration batch), every rank searches the whole batch on its shard with the two-phase protocol of
scann-rust_b200/distributed.py (token slices all-gathered, closest-leaf bounds all-reduced, local top-k all-gathered
and merged by a kernel); the dataset size is fixed, so scaling is "strong".
"""
import argparse
import importlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = {
    "c1": "queries/sec (BruteForce SquaredL2 10k x128, 1k-query batch, k=10)",
    "c2": "queries/sec (BruteForce DotProduct 1M x128, 10k-query batch, k=10)",
    "c3": "queries/sec @ recall@10>=0.95 (Tree-AH 10Mx96)",
    "c4": "queries/sec (Tree-X-Hybrid SquaredL2 100M x128, K=8192, sharded + NCCL merge)",
    "c5": "queries/sec (Tree-AH 1B x96 PQ codes 32 B/vector, K=65536, sharded, no reorder)",
}
DTYPE = {"c1": "bf16 ranking (tcgen05) + f32 exact re-score", "c2": "bf16 ranking (tcgen05) + f32 exact re-score",
         "c3": "u8 LUT / u32 accumulate, f32 reorder", "c4": "u8 LUT / u32 accumulate, f32 reorder",
         "c5": "u8 LUT / u32 accumulate"}
# per-config defaults of the size arguments (None on the command line = take these)
DEFAULTS = {
    "c1": dict(n=10_000, dim=128, nq=1_000, k=10),
    "c2": dict(n=1_000_000, dim=128, nq=10_000, k=10),
    "c3": dict(n=10_000_000, dim=96, partitions=2000, subspaces=48, leaves=64, reorder=100, k=10, nq=10_000,
               latent=8192, spread=0.5, decay=1.0, balance=3.0),
    "c4": dict(n=100_000_000, dim=128, partitions=8192, subspaces=64, leaves=64, reorder=100, k=10, nq=10_000,
               latent=16384, spread=0.5, decay=1.0, sweep="32,64,128", train_rows=1_000_000, kmeans_iters=15,
               balance=3.0),
    "c5": dict(n=1_000_000_000, dim=96, partitions=65536, subspaces=48, leaves=64, reorder=100, k=10, nq=10_000,
               latent=65536, spread=0.5, decay=1.0, sweep="16,32,64,128,256", train_rows=2_000_000, kmeans_iters=10,
               balance=3.0),
}


def parse():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=10)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--impl", default="ours", choices=["ours", "reference"])
    p.add_argument("--config", default="c3", choices=sorted(METRIC))
    p.add_argument("--rows", dest="n", type=int, default=None, help="same as --n (torchrun's own parser trips over --n)")
    for name, typ in [("n", int), ("dim", int), ("partitions", int), ("subspaces", int), ("leaves", int),
                      ("reorder", int), ("k", int), ("nq", int), ("latent", int), ("spread", float), ("decay", float),
                      ("train_rows", int), ("kmeans_iters", int), ("balance", float)]:
        p.add_argument("--" + name.replace("_", "-"), type=typ, default=None)
    p.add_argument("--sweep", default=None, help="c4/c5: comma list of leaves_to_search values (first JSON value = --leaves)")
    p.add_argument("--sq8", action="store_true", help="c2: ScalarQuantizedBruteForceSearcher (Int8) instead of f32")
    p.add_argument("--gt-queries", type=int, default=1000)
    p.add_argument("--cpu-queries", type=int, default=128)
    p.add_argument("--ref-queries", type=int, default=128)
    p.add_argument("--check-queries", type=int, default=256, help="multi-GPU self-check subsample (0 = off)")
    p.add_argument("--chunk-rows", type=int, default=1 << 20, help="c4/c5: rows generated per chunk")
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--shard", default="partition", choices=["partition", "rows"],
                   help="multi-GPU sharding: whole partitions per GPU (default) or rows round-robin inside partitions")
    p.add_argument("--emulate-shard", type=int, default=0,
                   help="single-GPU tuning aid: build and search only shard 0 of N (not a bench mode)")
    p.add_argument("--phase-times", action="store_true", help="multi-GPU: log the per-phase device times of the step")
    p.add_argument("--prefetch", action="store_true",
                   help="multi-GPU: prefetch the next batch's partition slice + token all-gather on a side stream "
                        "(distributed.TokenPrefetcher; measured: no gain at N=2, the persistent scan kernels leave no "
                        "SM for the side stream, the time moves into the result exchange)")
    p.add_argument("--split", action="store_true",
                   help="single-GPU tuning aid: use the two-phase search_begin/search_end path (no reduction)")
    p.add_argument("--sweep-leaves", default="", help="c3: comma list: print recall/QPS for each L (stderr) and exit")
    p.add_argument("--dump-outputs", metavar="DIR", default=None,
                   help="write the results of the last timed step as DIR/<name>.npy (ids and counts as float64, distances "
                        "as float32), so that two builds can be compared output for output")
    a = p.parse_args()
    if a.steps < 1:
        p.error("--steps must be at least 1")
    for k2, v in DEFAULTS[a.config].items():
        if getattr(a, k2, None) is None:
            setattr(a, k2, v)
    return a


def log(*a):
    print(*a, file=sys.stderr, flush=True)


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, ids, dists, counts):
    """Writes one search step's results ([nq, k] ids and distances, [nq] counts; numpy or torch) as <out_dir>/ids.npy,
    dists.npy and counts.npy.  Ids and counts are stored as float64, which holds every u32 exactly.  When the arrays
    exceed DUMP_LIMIT_BYTES, a fixed seeded sample of query rows is written instead, and rows.npy lists which."""
    arrs = {}
    for name, v, dt in (("ids", ids, np.float64), ("dists", dists, np.float32), ("counts", counts, np.float64)):
        v = v.cpu().numpy() if hasattr(v, "cpu") else np.asarray(v)
        if v.dtype == np.int32:  # device results: the same u32 values as the host API returns (padding = 0xFFFFFFFF)
            v = v.view(np.uint32)
        arrs[name] = v.astype(dt)
    nq = arrs["counts"].shape[0]
    row_bytes = sum(v.nbytes for v in arrs.values()) // max(nq, 1) + 8
    if nq * row_bytes > DUMP_LIMIT_BYTES:
        rows = np.sort(np.random.default_rng(0).choice(nq, DUMP_LIMIT_BYTES // row_bytes, replace=False))
        arrs = {name: v[rows] for name, v in arrs.items()}
        arrs["rows"] = rows.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for name, v in arrs.items():
        np.save(os.path.join(out_dir, name + ".npy"), v)
    log(f"dumped {', '.join(f'{n}{list(v.shape)}' for n, v in arrs.items())} to {out_dir}")


def noise_sigma(torch, dim, decay, device):
    sig = torch.arange(1, dim + 1, device=device, dtype=torch.float32) ** (-decay)
    return sig / torch.sqrt((sig * sig).mean())


def make_points(torch, n, dim, lat, spread, decay, seed, device, chunk=2_000_000, normalize=True):
    """SURVEY §8d mixture: point = latent centre + spread * anisotropic N(0,1) noise (L2-normalised for C3/C5).
    The noise spectrum sigma_j ∝ j^-decay (rms 1) gives the data a realistic low local intrinsic dimension;
    with decay = 0 it is the isotropic mixture of SURVEY §8d."""
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    sig = noise_sigma(torch, dim, decay, device)
    out = torch.empty((n, dim), dtype=torch.float32, device=device)
    for s in range(0, n, chunk):
        m = min(chunk, n - s)
        which = torch.randint(0, lat.shape[0], (m,), generator=g, device=device)
        x = lat[which] + spread * torch.randn((m, dim), generator=g, device=device) * sig[None, :]
        out[s:s + m] = x / x.norm(dim=1, keepdim=True) if normalize else x
    return out


class ClockSampler:
    def __init__(self, index=0):
        self.index = index
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self._stop = threading.Event()
        self._t = None

    def _run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                f = [v.strip() for v in out.strip().split("\n")[0].split(",")]
                self.samples.append(float(f[0]))
                self.max_mhz = float(f[1])
                for nm, v in zip(names, f[2:]):
                    if v.lower().startswith("active"):
                        self.reasons.add(nm)
            except Exception:
                pass
            self._stop.wait(0.1)

    def start(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()

    def stop(self):
        self._stop.set()
        if self._t:
            self._t.join(timeout=6)
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


def load_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return {}


def scan_roofline(a, tcp, scan_ms_per_launch, scan_bytes, pairs, peaks, clocks, traffic=None, traffic_src=None):
    """roofline object of the dominant kernel of a Tree-AH step.
    Tensor-core scan (tcscan.cu) active: bound = tensor, achieved = 2 * (query, point) pairs * S * 16 integer operations of
    the one-hot contraction / the live CUDA-event time of tc_scan_kernel.  Otherwise the register-LUT kernel with the
    north-star's algorithmic-bytes equivalence against the measured HBM peak."""
    peak_gbs = float(peaks.get("hbm_gbs", 6650.0))
    hbm = {"algorithmic_bytes_per_step": scan_bytes, "scan_stage_ms_per_step": scan_ms_per_launch,
           "algorithmic_GBps": scan_bytes / (scan_ms_per_launch / 1e3) / 1e9 if scan_ms_per_launch > 0 else 0.0,
           "hbm_peak_GBps": peak_gbs, "pairs_per_step": pairs}
    hbm["frac_of_hbm_peak"] = hbm["algorithmic_GBps"] / peak_gbs
    if tcp and tcp["launches"] > 0 and tcp["scan_ms"] > 0:
        ms = tcp["scan_ms"] / tcp["launches"]
        ops = 2.0 * tcp["pair_points"] * a.subspaces * 16
        ach = ops / (ms / 1e3) / 1e12
        mhz = (clocks or {}).get("sm_mhz") or float(peaks.get("sm_max_mhz", 1965.0))
        # 8192 u8 MACs per clock per SM: one M128 x N128 x K32 tcgen05.mma.kind::i8 per 64 clocks, measured on this pool
        # with tools/tcscan_probe.cu (profiles/r2_tcscan_probe.md); x 148 SMs x the SM clock sampled during the run
        peak = 2.0 * 8192 * 148 * mhz * 1e6 / 1e12
        return {"bound": "tensor", "kernel": "tc_scan_kernel (tcgen05.mma kind::i8, one-hot LUT16 scan)", "achieved": ach,
                "peak": peak, "unit": "TFLOP/s", "frac": ach / peak, "traffic": traffic, "traffic_source": traffic_src,
                "ops_are": "u8 x u8 -> s32 multiply-adds x 2 of the useful (query, point, subspace, code) contraction; "
                           "padding columns and the threshold atom are not counted",
                "ms_per_launch": ms, "lut_build_ms_per_launch": tcp["lut_ms"] / tcp["launches"],
                "pair_points_per_launch": tcp["pair_points"],
                "peak_source": f"probe-measured 8192 MAC/clk/SM (tools/tcscan_probe.cu) x 148 SMs x {mhz:.0f} MHz sampled "
                               "in this run; MEASURED_PEAKS.json holds no int8 figure (2 x its bf16 burst = "
                               f"{2 * float(peaks.get('bf16_tflops', 0.0)):.0f})",
                "hbm_equivalence": hbm}
    return {"bound": "hbm", "kernel": "lut16_scan_kernel", "achieved": hbm["algorithmic_GBps"], "peak": peak_gbs,
            "unit": "GB/s", "frac": hbm["frac_of_hbm_peak"], "traffic": traffic, "traffic_source": traffic_src,
            "physical_frac": (traffic / (scan_ms_per_launch / 1e3) / 1e9 / peak_gbs) if traffic else None,
            "algorithmic_bytes_per_launch": scan_bytes, "ms_per_launch": scan_ms_per_launch, "pairs_per_launch": pairs,
            "peak_source": "MEASURED_PEAKS.json hbm_gbs (measured copy bandwidth)" if "hbm_gbs" in peaks else "fallback 6650 GB/s",
            "limiter": "ALU pipe (ncu: 70 % ALU, 22 % FMA, L2 hit 96 %): a leaf's codes are streamed once for up to 8 "
                       "queries, so the kernel is bound by the register-LUT lookups, not by DRAM; the HBM figure is the "
                       "north-star's algorithmic-bytes equivalence",
            "note": "achieved = algorithmic code bytes / live CUDA-event time of the scan stage"}


def c3_config(a, K, shard_world, shard):
    workload = (f"Tree-AH {a.n}x{a.dim} K={K} LUT16 S={a.subspaces} ds={a.dim // a.subspaces} L={a.leaves} "
                f"R={a.reorder} k={a.k} DotProduct, batch={a.nq} queries")
    return {"workload": workload, "n": a.n, "dim": a.dim, "partitions": K, "subspaces": a.subspaces,
            "leaves_to_search": a.leaves, "reorder": a.reorder, "k": a.k, "batch_queries": a.nq,
            "data_model": f"mixture of {a.latent} latent centres, spread {a.spread}, noise spectrum j^-{a.decay}, "
                          "L2-normalised; seeds db 42 / queries 123+ / train 7",
            "index_training": "in-library Lloyd k-means (scann_kmeans_fit / scann_pq_train), 1M-row sample, 20 iterations"
                              + (f", partitions balanced to <= {a.balance:g}x the mean leaf" if a.balance > 1 else ""),
            "l2_policy": "inputs larger than L2: 24 B/point codes of the probed leaves (7.7 MB/query, 240 MB index) "
                         "+ 3.84 GB raw rows; two alternating query batches",
            "parallelism": (f"index {shard}-sharded x{shard_world}; per batch: token slices all-gathered, closest-leaf "
                            "bounds all-reduced (MIN), local top-k all-gathered + merge kernel (NCCL)"
                            if shard_world > 1 else "single GPU")}


# ======================================================================================== reference arm (CPU oracle)
def reference_arm(a, emit):
    """The reference's own CPU implementation of the path (oracle/ C++ restatement: the crate is Rust and cannot be built
    in this image) with all host threads on a bounded sample.  The index is built with plain torch ops
    (oracle/ref_index.py); the product package is never imported, so libscann_b200.so is neither built nor loaded."""
    import torch

    import oracle
    from oracle import ref_index

    oracle.build()
    nthreads = oracle.num_threads()
    dev = torch.device("cuda", 0) if torch.cuda.is_available() else torch.device("cpu")
    steps = a.warmup + a.steps
    g = torch.Generator(device=dev)
    g.manual_seed(42)

    def finish(nq_step, times, config, sample):
        tt = times[a.warmup:]
        val = nq_step * len(tt) / sum(tt)
        emit({"impl": "reference", "metric": METRIC[a.config], "value": val, "unit": "queries/s", "n_gpus": a.gpus,
              "steps": a.steps, "warmup": a.warmup, "ms_per_step": 1e3 * sum(tt) / len(tt), "higher_is_better": True,
              "scaling": "strong", "vs_baseline": None, "dtype": DTYPE[a.config], "data": "synthetic", "config": config,
              "cpu_baseline": {"value": val, "unit": "queries/s", "cores": nthreads, "kind": "port", "sample": sample},
              "e2e": {"value": val, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
              "gpu_launches": 0})
        return 0

    if a.config in ("c1", "c2"):
        x = torch.randn((a.n, a.dim), generator=g, device=dev)
        g.manual_seed(123)
        q = torch.randn((a.nq, a.dim), generator=g, device=dev)
        hx, hq = x.cpu().numpy(), q.cpu().numpy()
        measure = oracle.SQL2 if a.config == "c1" else oracle.DOT
        nqs = a.nq if a.config == "c1" else min(a.ref_queries, a.nq)
        times = []
        for _ in range(steps):
            t = time.perf_counter()
            res = oracle.bf_search(hx, hq[:nqs], a.k, measure, nthreads=nthreads)
            times.append(time.perf_counter() - t)
        if a.dump_outputs:
            dump_outputs(a.dump_outputs, *res[1:4])
        cfg = bf_config(a)
        return finish(nqs, times, cfg, f"{nqs} queries per step against the full {a.n}x{a.dim} database; oracle/ C++ "
                                       "restatement of BruteForceSearcher::search_batched (one task per query)")

    # Tree-AH / Tree-X-Hybrid: C3 at full size; C4/C5 on a 1 % row subsample (SURVEY §8d)
    frac = 1.0 if a.config == "c3" else 0.01
    n = int(a.n * frac)
    normalize = a.config != "c4"
    lat = torch.randn((a.latent, a.dim), generator=g, device=dev)
    x = make_points(torch, n, a.dim, lat, a.spread, a.decay, 42, dev, normalize=normalize)
    q = make_points(torch, a.nq, a.dim, lat, a.spread, a.decay, 123, dev, normalize=normalize)
    t0 = time.time()
    K = a.partitions
    idx = ref_index.build_treeah(torch, x, K, a.subspaces, min(a.train_rows or 1_000_000, n), 20 if a.config == "c3" else 8,
                                 balance_ratio=a.balance)
    log(f"reference arm: torch index K={idx['centers'].shape[0]} over {n} rows in {time.time() - t0:.1f}s")
    hc, hcb = idx["centers"].cpu().numpy(), idx["codebook"].cpu().numpy()
    hoff = idx["off"].cpu().numpy().astype(np.uint64)
    hids = idx["ids"].cpu().numpy().astype(np.uint32)
    hpacked = idx["packed"].cpu().numpy()
    raw = None if a.config == "c5" else x.cpu().numpy()
    hq = q[:min(a.ref_queries, a.nq)].cpu().numpy()
    measure = {"c3": oracle.DOT, "c4": oracle.SQL2, "c5": oracle.SQL2}[a.config]
    times = []
    for _ in range(steps):
        t = time.perf_counter()
        res = oracle.treex_search(hc, hcb, hoff, hids, hpacked, raw, hq, min(a.leaves, hc.shape[0]), a.reorder, a.k,
                                  lut16=True, use_residuals=True, reorder_measure=measure, nthreads=nthreads)
        times.append(time.perf_counter() - t)
    if a.dump_outputs:
        dump_outputs(a.dump_outputs, *res[1:4])
    if a.config == "c3":
        cfg = c3_config(a, hc.shape[0], max(1, a.gpus), a.shard)
        sample = (f"{hq.shape[0]} queries per step of the same workload (index trained and encoded with plain torch ops, "
                  "oracle/ref_index.py); oracle/ C++ restatement of the reference algorithm (the Rust crate cannot be "
                  "built in this image), one task per query over all host threads")
    else:
        cfg = sharded_config(a, max(1, a.gpus))
        sample = (f"{hq.shape[0]} queries per step on a 1 % row subsample ({n} rows, K={hc.shape[0]}) of the workload; "
                  "oracle/ C++ restatement of the reference algorithm, one task per query over all host threads")
    return finish(hq.shape[0], times, cfg, sample)


# ======================================================================================== C1 / C2: brute force
def bf_config(a):
    name = "ScalarQuantizedBruteForceSearcher Int8" if a.sq8 else "BruteForceSearcher f32"
    measure = "SquaredL2" if a.config == "c1" else "DotProduct"
    return {"workload": f"{name} {measure} {a.n}x{a.dim} i.i.d. N(0,1), batch={a.nq} queries, k={a.k}", "n": a.n,
            "dim": a.dim, "k": a.k, "batch_queries": a.nq, "data_model": "i.i.d. N(0,1); seeds db 42 / queries 123+",
            "l2_policy": ("two alternating query batches; the database (%.0f MB) is read once per 4096-query chunk"
                          % (a.n * a.dim * (1 if a.sq8 else 4) / 1e6)) +
                         (" and is smaller than L2 at C1 (launch-latency regime)" if a.config == "c1" else ""),
            "parallelism": "single GPU"}


def bench_bf(a, emit, torch, pkg, dev, local_rank):
    M = pkg.DistanceMeasure
    g = torch.Generator(device=dev)
    g.manual_seed(42)
    x = torch.randn((a.n, a.dim), generator=g, device=dev)
    queries = []
    for b in range(2):
        g.manual_seed(123 + b)
        queries.append(torch.randn((a.nq, a.dim), generator=g, device=dev))
    measure = M.SquaredL2 if a.config == "c1" else M.DotProduct
    if a.sq8:
        codes, cal = pkg.scalar_quantize(x, local_rank)
        s = pkg.ScalarQuantizedBruteForceSearcher.from_quantized(codes, float(cal[2]), measure, local_rank)
    else:
        s = pkg.BruteForceSearcher(x, measure, local_rank)
    for w in range(max(a.warmup, 1)):
        ids, dists, cnt = s.search_batched(queries[w % 2], a.k)
    torch.cuda.synchronize()
    # parity property in the run: the f32 searcher's result equals an independent exact top-k (torch f32, ties aside)
    ng = min(256, a.nq)
    qs = queries[(max(a.warmup, 1) - 1) % 2][:ng]
    sc = (qs * qs).sum(1)[:, None] - 2.0 * qs @ x.t() + (x * x).sum(1)[None, :] if a.config == "c1" else -(qs @ x.t())
    want = torch.topk(sc, a.k, dim=1, largest=False).indices
    agree = float(np.mean([len(set(ids[i].tolist()) & set(want[i].tolist())) / a.k for i in range(ng)]))
    del sc
    sampler = ClockSampler(local_rank)
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for st in range(a.steps):
        last = s.search_batched(queries[st % 2], a.k)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    value = a.nq * a.steps / (ms / 1e3)
    hq = [torch.empty((a.nq, a.dim), dtype=torch.float32, pin_memory=True) for _ in range(2)]
    for b in range(2):
        hq[b].copy_(queries[b])
    hq_np = [t.numpy() for t in hq]
    s.search_batched(hq_np[0], a.k)
    t = time.perf_counter()
    for st in range(a.steps):
        s.search_batched(hq_np[st % 2], a.k)
    e2e = a.nq * a.steps / (time.perf_counter() - t)
    clocks = sampler.stop()
    peaks = load_peaks()
    peak_tf = float(peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops", 1500.0)))
    flops = 2.0 * a.nq * a.n * a.dim
    ach = flops / (ms / a.steps / 1e3) / 1e12
    tc, legacy = s.path_stats()
    out = {"metric": METRIC[a.config], "value": value, "unit": "queries/s", "n_gpus": 1, "steps": a.steps,
           "warmup": a.warmup, "ms_per_step": ms / a.steps, "higher_is_better": True, "scaling": "strong",
           "vs_baseline": None, "dtype": DTYPE[a.config], "data": "synthetic", "config": bf_config(a),
           "agreement_with_independent_exact_topk": agree,
           "e2e": {"value": e2e, "unit": "queries/s", "h2d_bytes_per_step": a.nq * a.dim * 4,
                   "d2h_bytes_per_step": a.nq * (a.k * 8 + 4)},
           # per 4096-query chunk: prep, sample GEMM, bound, filter GEMM, overflow flag, exact re-score; from 32768 rows on
           # the filter runs as prefix pass + tightened bound + pass over the rest
           "gpu_launches": int(a.steps * ((a.nq + 4095) // 4096) * (8 if a.n >= 32768 else 6)),
           "path_chunks": {"tcgen05": tc, "cuda_core": legacy},
           "roofline": {"bound": "tensor", "kernel": "tc_score_kernel (whole step: sample + filter + exact re-score)",
                        "achieved": ach, "peak": peak_tf, "unit": "TFLOP/s", "frac": ach / peak_tf, "traffic": None,
                        "algorithmic_flops_per_step": flops,
                        "peak_source": "MEASURED_PEAKS.json bf16_tflops_sustained (kernel timed inside a long step)"},
           "clocks": clocks}
    if not a.no_cpu_baseline:
        import oracle
        oracle.build()
        nthreads = oracle.num_threads()
        nqc = a.nq if a.config == "c1" else min(a.cpu_queries, a.nq)
        hx = x.cpu().numpy()
        t = time.perf_counter()
        oracle.bf_search(hx, hq_np[0][:nqc], a.k, oracle.SQL2 if a.config == "c1" else oracle.DOT, nthreads=nthreads)
        out["cpu_baseline"] = {"value": nqc / (time.perf_counter() - t), "unit": "queries/s", "cores": nthreads,
                               "kind": "port", "sample": f"{nqc} queries of the same batch against the full database; "
                               "oracle/ C++ restatement of BruteForceSearcher::search_batched"}
    if a.dump_outputs:
        dump_outputs(a.dump_outputs, *last)
    emit(out)
    return 0


# ======================================================================================== C4 / C5: sharded build
def sharded_config(a, world):
    if a.config == "c4":
        wl = (f"Tree-X-Hybrid SquaredL2 {a.n}x{a.dim} K={a.partitions} LUT16 S={a.subspaces} L={a.leaves} R={a.reorder} "
              f"k={a.k}, batch={a.nq} queries, rows sharded by whole partitions over {world} GPU(s)")
        l2 = "inputs larger than L2: %.1f GB of codes + %.1f GB of raw rows per GPU" % (
            a.n * a.subspaces / 2 / world / 1e9, a.n * a.dim * 4 / world / 1e9)
    else:
        wl = (f"Tree-AH {a.n}x{a.dim} PQ codes only ({a.subspaces // 2} B codes + u32 id per vector) K={a.partitions} "
              f"LUT16 S={a.subspaces} L={a.leaves} R={a.reorder} k={a.k} no reorder, batch={a.nq} queries, sharded by "
              f"whole partitions over {world} GPU(s)")
        l2 = "inputs larger than L2: %.1f GB of codes per GPU" % (a.n * a.subspaces / 2 / world / 1e9)
    return {"workload": wl, "n": a.n, "dim": a.dim, "partitions": a.partitions, "subspaces": a.subspaces,
            "leaves_to_search": a.leaves, "reorder": a.reorder, "k": a.k, "batch_queries": a.nq,
            "data_model": f"mixture of {a.latent} latent centres, spread {a.spread}, noise spectrum j^-{a.decay}"
                          + (", L2-normalised" if a.config == "c5" else "") +
                          f"; generated on the device per rank in chunks of {a.chunk_rows} rows (seed per chunk)",
            "index_training": f"in-library Lloyd k-means (scann_kmeans_fit / scann_pq_train) on the first {a.train_rows} rows, "
                              f"{a.kmeans_iters} iterations" +
                              (f", partitions balanced to <= {a.balance:g}x the mean leaf" if a.balance > 1 else ""),
            "l2_policy": l2 + "; two alternating query batches",
            "parallelism": (f"index partition-sharded x{world}; per batch: token slices all-gathered, closest-leaf bounds "
                            "all-reduced (MIN), local top-k all-gathered + merge kernel (NCCL)" if world > 1
                            else "single GPU")}


def gen_chunk(torch, lat, sig, c, rows, spread, normalize, dev):
    g = torch.Generator(device=dev)
    g.manual_seed(1_000_003 * (c + 1) + 42)
    which = torch.randint(0, lat.shape[0], (rows,), generator=g, device=dev)
    x = lat[which] + spread * torch.randn((rows, lat.shape[1]), generator=g, device=dev) * sig[None, :]
    return x / x.norm(dim=1, keepdim=True) if normalize else x


def exchange_rows(torch, dist, arr, send_counts, recv_counts):
    """all_to_all of rows of `arr` (already sorted by destination rank) with uneven splits."""
    out = torch.empty((int(sum(recv_counts)),) + tuple(arr.shape[1:]), dtype=arr.dtype, device=arr.device)
    dist.all_to_all_single(out, arr.contiguous(), output_split_sizes=[int(v) for v in recv_counts],
                           input_split_sizes=[int(v) for v in send_counts])
    return out


def lpt_owner(load_leaf, world):
    """leaves dealt heaviest-first to the least-loaded shard (greedy LPT); the same on every rank"""
    import heapq
    K = len(load_leaf)
    owner = np.zeros(K, np.int64)
    heap = [(0.0, g) for g in range(world)]
    heapq.heapify(heap)
    for leaf in np.argsort(-load_leaf, kind="stable"):
        ld, g = heapq.heappop(heap)
        owner[leaf] = g
        heapq.heappush(heap, (ld + float(load_leaf[leaf]), g))
    loads = np.zeros(world)
    np.add.at(loads, owner, load_leaf)
    return owner, loads


def bench_sharded(a, emit, torch, dist, pkg, dev, rank, world, local_rank):
    ix = pkg.indexing
    c4 = a.config == "c4"
    normalize = not c4
    M = pkg.DistanceMeasure
    t0 = time.time()
    K, S, D = a.partitions, a.subspaces, a.dim
    g = torch.Generator(device=dev)
    g.manual_seed(42)
    lat = torch.randn((a.latent, D), generator=g, device=dev)
    sig = noise_sigma(torch, D, a.decay, dev)
    nchunks = (a.n + a.chunk_rows - 1) // a.chunk_rows
    c_lo, c_hi = rank * nchunks // world, (rank + 1) * nchunks // world
    row0 = c_lo * a.chunk_rows
    row1 = min(a.n, c_hi * a.chunk_rows)
    n_loc = row1 - row0
    n_batches = 2
    queries = [make_points(torch, a.nq, D, lat, a.spread, a.decay, 123 + b, dev, normalize=normalize)
               for b in range(n_batches)]

    # ---- training on rank 0 (first rows of the dataset), broadcast
    if rank == 0:
        parts, got, c = [], 0, 0
        while got < min(a.train_rows, a.n):
            rows = min(a.chunk_rows, a.n - c * a.chunk_rows)
            parts.append(gen_chunk(torch, lat, sig, c, rows, a.spread, normalize, dev))
            got += rows
            c += 1
        sample = torch.cat(parts)[:a.train_rows].contiguous()
        del parts
        torch.backends.cuda.matmul.allow_tf32 = True   # index TRAINING only (k-means matmuls)
        centers = ix.kmeans(sample, K, a.kmeans_iters, 7, balance_ratio=a.balance)
        a_s = ix.assign_partitions(sample, centers, local_rank)
        codebook = ix.train_codebook(sample - centers[a_s.long()], S, 16, 20, 42)
        torch.backends.cuda.matmul.allow_tf32 = False  # the exact ground truth below is plain f32
        del sample, a_s
        log(f"[rank 0] trained K={centers.shape[0]} centres + {S}x16 codebook in {time.time() - t0:.1f}s")
    else:
        centers = torch.empty((min(K, a.train_rows), D), dtype=torch.float32, device=dev)
        codebook = torch.empty((S, 16, D // S), dtype=torch.float32, device=dev)
    if world > 1:
        dist.broadcast(centers, 0)
        dist.broadcast(codebook, 0)
    K = centers.shape[0]

    # ---- local rows: generate, assign (TreePartitioner::partition(x, 1)), encode, exact ground truth
    ng = min(a.gt_queries, a.nq)
    gq = queries[0][:ng]
    gq_n = (gq * gq).sum(1)
    part = pkg.TreePartitioner(centers, local_rank)
    bpp = (S + 1) // 2
    assign_loc = torch.empty((n_loc,), dtype=torch.int32, device=dev)
    packed_loc = torch.empty((n_loc, bpp), dtype=torch.uint8, device=dev)
    x_loc = torch.empty((n_loc, D), dtype=torch.float32, device=dev) if c4 else None
    gt_d = torch.full((ng, a.k), float("inf"), device=dev)
    gt_i = torch.full((ng, a.k), -1, dtype=torch.int64, device=dev)
    for c in range(c_lo, c_hi):
        s = c * a.chunk_rows - row0
        rows = min(a.chunk_rows, a.n - c * a.chunk_rows)
        x = gen_chunk(torch, lat, sig, c, rows, a.spread, normalize, dev)
        tok, _ = part.partition(x, 1)
        tok = tok[:, 0].contiguous()
        assign_loc[s:s + rows] = tok
        packed_loc[s:s + rows] = pkg.pq_encode(codebook, x, centers, tok, local_rank)
        if c4:
            x_loc[s:s + rows] = x
        dd = gq_n[:, None] - 2.0 * (gq @ x.t()) + (x * x).sum(1)[None, :]  # exact SqL2 (unit vectors: same order as Dot)
        d2, i2 = torch.topk(dd, a.k, dim=1, largest=False)
        md, mi = torch.cat([gt_d, d2], 1), torch.cat([gt_i, i2 + (row0 + s)], 1)
        gt_d, sel = torch.topk(md, a.k, dim=1, largest=False)
        gt_i = torch.gather(mi, 1, sel)
        del x, dd
    torch.cuda.synchronize()
    part.close()
    if world > 1:
        gd = [torch.empty_like(gt_d) for _ in range(world)]
        gi = [torch.empty_like(gt_i) for _ in range(world)]
        dist.all_gather(gd, gt_d)
        dist.all_gather(gi, gt_i)
        md, mi = torch.cat(gd, 1), torch.cat(gi, 1)
        gt_d, sel = torch.topk(md, a.k, dim=1, largest=False)
        gt_i = torch.gather(mi, 1, sel)
    want = gt_i.cpu().numpy()
    log(f"[rank {rank}] generated/assigned/encoded {n_loc} rows in {time.time() - t0:.1f}s")

    # ---- shard plan: whole partitions per GPU, balanced on the probe load of a calibration batch
    counts = torch.bincount(assign_loc.long(), minlength=K)
    if world > 1:
        dist.all_reduce(counts)
    ids_loc = torch.arange(row0, row1, dtype=torch.int32, device=dev)
    if world > 1:
        calib = make_points(torch, 10_000, D, lat, a.spread, a.decay, 999, dev, normalize=normalize)
        part = pkg.TreePartitioner(centers, local_rank)
        tok, _ = part.partition(calib, min(a.leaves, K))
        probes = torch.bincount(tok.long().flatten().clamp_(0, K - 1), minlength=K).cpu().numpy()
        part.close()
        load_leaf = (probes.astype(np.float64) + 1.0) * counts.cpu().numpy().astype(np.float64)
        owner_h, loads = lpt_owner(load_leaf, world)
        if rank == 0:
            log(f"shard plan: calibrated probe load max/mean = {loads.max() / loads.mean():.4f}")
        owner = torch.from_numpy(owner_h).to(dev)
        dest = owner[assign_loc.long()]
        perm = torch.argsort(dest, stable=True)
        send = torch.bincount(dest, minlength=world)
        recv = torch.empty_like(send)
        dist.all_to_all_single(recv, send)
        send_h, recv_h = send.cpu().tolist(), recv.cpu().tolist()
        assign_sh = exchange_rows(torch, dist, assign_loc[perm], send_h, recv_h)
        ids_sh = exchange_rows(torch, dist, ids_loc[perm], send_h, recv_h)
        packed_sh = exchange_rows(torch, dist, packed_loc[perm], send_h, recv_h)
        raw_sh = exchange_rows(torch, dist, x_loc[perm], send_h, recv_h) if c4 else None
        del dest, perm
    else:
        assign_sh, ids_sh, packed_sh, raw_sh = assign_loc, ids_loc, packed_loc, x_loc
    del packed_loc

    def leaf_sorted(assign_rows, ids_rows, packed_rows, raw_rows):
        order = torch.argsort(assign_rows.long(), stable=True)
        cnt = torch.bincount(assign_rows.long(), minlength=K)
        off = torch.zeros((K + 1,), dtype=torch.int64, device=dev)
        off[1:] = torch.cumsum(cnt, 0)
        return (packed_rows[order].contiguous(), ids_rows[order].contiguous(), off,
                raw_rows[order].contiguous() if raw_rows is not None else None, assign_rows[order].contiguous())

    packed, ids32, off, raw, leaf_of_row = leaf_sorted(assign_sh, ids_sh, packed_sh, raw_sh)
    del assign_sh, ids_sh, packed_sh, raw_sh
    torch.cuda.empty_cache()
    cfg = pkg.TreeXHybridConfig(num_partitions=K, partitions_to_search=a.leaves, use_residuals=True,
                                pre_reorder_multiplier=a.reorder / a.k, distance_measure=M.SquaredL2)
    searcher = pkg.TreeXHybridSearcher(cfg, local_rank).build_from_index(centers, codebook, packed, ids32, off, raw,
                                                                        raw_by_position=True, borrow_raw=True)
    sizes = (off[1:] - off[:-1])
    log(f"[rank {rank}] shard index rows={ids32.numel()} leaves owned={int((sizes > 0).sum())} "
        f"(leaf sizes mean/max {float(sizes[sizes > 0].float().mean()):.0f}/{int(sizes.max())}) in {time.time() - t0:.1f}s")
    R = a.reorder

    def step_device(qb, L):
        if world > 1:
            ids, dists, cnt = pkg.distributed.two_phase_search(searcher, qb, a.k, partitions_to_search=L, pre_reorder_k=R)
            return pkg.distributed.exchange_and_merge(ids, dists)
        return searcher.search_batched(qb, a.k, partitions_to_search=L, pre_reorder_k=R)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- parity properties on the merged result of batch 0 at the headline L
    L0 = min(a.leaves, K)
    ids, dists, cnt = step_device(queries[0], L0)
    torch.cuda.synchronize()
    checks = {}
    idl = ids.long()
    checks["sorted_and_full"] = bool((dists[:, 1:] >= dists[:, :-1]).all().item() and (cnt == a.k).all().item())
    tokens_all = torch.cat([searcher.partition_tokens(queries[0][s:s + 1024].contiguous(), L0)
                            for s in range(0, a.nq, 1024)]).long()
    mine = (idl >= row0) & (idl < row1)
    loc = (idl - row0).clamp_(0, n_loc - 1)
    leaf_of = assign_loc.long()[loc]                                        # leaf of every returned id (where mine)
    in_probed = (leaf_of[:, :, None] == tokens_all[:, None, :]).any(-1)
    bad_leaf = ((~in_probed) & mine).sum().double()
    covered = mine.sum().double()
    max_rel = torch.zeros((), dtype=torch.float64, device=dev)
    if c4:  # independently recomputed exact distances of the returned ids (f64 on the rows this rank generated)
        qd = queries[0].double()
        for q0 in range(0, a.nq, 2048):
            rows = x_loc[loc[q0:q0 + 2048]].double()                        # [m, k, D]
            ex = ((rows - qd[q0:q0 + 2048, None, :]) ** 2).sum(-1)
            rel = (ex - dists[q0:q0 + 2048].double()).abs() / ex.clamp(min=1e-12)
            max_rel = torch.maximum(max_rel, (rel * mine[q0:q0 + 2048]).max())
    if world > 1:
        dist.all_reduce(bad_leaf)
        dist.all_reduce(covered)
        dist.all_reduce(max_rel, op=dist.ReduceOp.MAX)
    checks["results_outside_probed_leaves"] = int(bad_leaf.item())
    checks["result_ids_checked"] = int(covered.item())
    checks["result_ids_total"] = int(a.nq * a.k)
    if c4:
        checks["max_rel_err_vs_recomputed_f64_distance"] = float(max_rel.item())
    del x_loc, loc, mine, leaf_of, in_probed
    torch.cuda.empty_cache()

    # ---- sharded result vs ONE index holding every row (rank 0), on a subsample of the batch
    nchk = min(a.check_queries, a.nq)
    if nchk > 0:
        if world > 1:
            n_sh = torch.tensor([ids32.numel()], dtype=torch.int64, device=dev)
            all_n = [torch.empty_like(n_sh) for _ in range(world)]
            dist.all_gather(all_n, n_sh)
            all_n = [int(v.item()) for v in all_n]
            send_h = [ids32.numel() if d == 0 else 0 for d in range(world)]
            recv_h = all_n if rank == 0 else [0] * world
            f_leaf = exchange_rows(torch, dist, leaf_of_row, send_h, recv_h)
            f_ids = exchange_rows(torch, dist, ids32, send_h, recv_h)
            f_packed = exchange_rows(torch, dist, packed, send_h, recv_h)
            f_raw = exchange_rows(torch, dist, raw, send_h, recv_h) if c4 else None
        else:
            f_leaf, f_ids, f_packed, f_raw = leaf_of_row, ids32, packed, raw
        if rank == 0:
            if world > 1:
                fp, fi, fo, fr, _ = leaf_sorted(f_leaf, f_ids, f_packed, f_raw)
                del f_leaf, f_ids, f_packed, f_raw
                full = pkg.TreeXHybridSearcher(cfg, local_rank).build_from_index(centers, codebook, fp, fi, fo, fr,
                                                                                 raw_by_position=True, borrow_raw=True)
            else:
                full = searcher
            si, sd, sc = full.search_batched(queries[0][:nchk].contiguous(), a.k, partitions_to_search=L0, pre_reorder_k=R)
            torch.cuda.synchronize()
            gi_, gd_ = ids[:nchk], dists[:nchk]
            # every shard's list contains the global top-R members that live on it, so the merged exact distances can
            # only be <= the single-index ones rank by rank (equal when nothing was gained)
            checks["single_index_queries"] = nchk
            checks["sharded_dist_le_single_index"] = bool((gd_ <= sd + 1e-6 * sd.abs() + 1e-12).all().item())
            checks["id_agreement_with_single_index"] = float(np.mean(
                [len(set(gi_[i].tolist()) & set(si[i].tolist())) / a.k for i in range(nchk)]))
            if not c4:  # C5: recompute the LUT16 approximate distance of the returned ids from the codes (torch f32)
                checks["max_rel_err_vs_recomputed_lut16_distance"] = recompute_lut16(
                    torch, queries[0][:64], si[:64], sd[:64], centers, codebook, fi if world > 1 else ids32,
                    fp if world > 1 else packed, fo if world > 1 else off, S)
            if world > 1:
                full.close()
                del full, fp, fi, fo, fr
        else:
            del f_leaf, f_ids, f_packed, f_raw
        torch.cuda.empty_cache()
        barrier()
    if rank == 0:
        log(f"checks: {checks}")

    # ---- timed sweep over leaves_to_search
    sweep_L = [int(v) for v in str(a.sweep).split(",") if v] if a.sweep else [a.leaves]
    if a.leaves not in sweep_L:
        sweep_L.append(a.leaves)
    hq = [torch.empty((a.nq, D), dtype=torch.float32, pin_memory=True) for _ in range(n_batches)]
    for b in range(n_batches):
        hq[b].copy_(queries[b])
    peaks = load_peaks()
    results = {}
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    for L in sweep_L:
        L = min(L, K)
        ids, _, _ = step_device(queries[0], L)
        rec, rec_r = None, None
        if rank == 0:
            got = ids[:ng].cpu().numpy()
            rec = float(np.mean([len(set(got[i]) & set(want[i])) / a.k for i in range(ng)]))
        if not c4:
            # codes only, no reorder: the returned order is the approximate one, so also report how many of the exact
            # top-k are among the R best approximate candidates (what a reorder stage would be handed), untimed
            if world > 1:
                li, ld, _ = pkg.distributed.two_phase_search(searcher, queries[0], R, partitions_to_search=L, pre_reorder_k=R)
                ri, _, _ = pkg.distributed.exchange_and_merge(li, ld)
            else:
                ri, _, _ = searcher.search_batched(queries[0], R, partitions_to_search=L, pre_reorder_k=R)
            if rank == 0:
                gr = ri[:ng].cpu().numpy()
                rec_r = float(np.mean([len(set(gr[i]) & set(want[i])) / a.k for i in range(ng)]))
        for w in range(a.warmup):
            step_device(queries[w % n_batches], L)
        barrier()
        searcher.set_profiling(True)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        for s in range(a.steps):
            last = step_device(queries[s % n_batches], L)
        e1.record()
        barrier()
        if L == L0:
            head_out = last
        ms = e0.elapsed_time(e1)
        tcp = searcher.tc_profile()
        prof, launches = searcher.get_profile()
        searcher.set_profiling(False)
        scan_bytes, pairs = searcher.last_scan_bytes()
        tm = torch.tensor([ms, float(scan_bytes), prof["scan"]], dtype=torch.float64, device=dev)
        tsum = tm.clone()
        if world > 1:
            dist.all_reduce(tm, op=dist.ReduceOp.MAX)
            dist.all_reduce(tsum)
        ms = float(tm[0].item())

        def step_host(b):
            mi, md, mc = step_device(hq[b].to(dev, non_blocking=True), L)
            return mi.cpu().numpy(), md.cpu().numpy()

        step_host(0)
        barrier()
        t = time.perf_counter()
        for s in range(a.steps):
            step_host(s % n_batches)
        barrier()
        te = torch.tensor([time.perf_counter() - t], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        scan_ms = prof["scan"] / a.steps
        results[L] = {
            "L": L, "recall_at_10_vs_exact": rec, "recall_10_in_top_R_candidates": rec_r, "queries_per_s": a.nq * a.steps / (ms / 1e3), "ms_per_step": ms / a.steps,
            "e2e_queries_per_s": a.nq * a.steps / float(te.item()),
            "scan_ms_rank0": scan_ms, "scan_bytes_rank0": scan_bytes, "scan_bytes_all_ranks": float(tsum[1].item()),
            "scan_GBps_algorithmic_rank0": scan_bytes / (scan_ms / 1e3) / 1e9 if scan_ms > 0 else 0.0,
            "stage_ms_rank0": {k2: v / a.steps for k2, v in prof.items()}, "launches_rank0": int(launches),
            "tc_profile_rank0": tcp, "pairs_rank0": pairs}
        if rank == 0:
            log(f"L={L}: recall@{a.k}={rec:.4f} (10 in top-R: {rec_r}) {results[L]['queries_per_s']:.0f} q/s ({ms / a.steps:.3f} ms/step), "
                f"scan {scan_ms:.3f} ms = {results[L]['scan_GBps_algorithmic_rank0']:.0f} GB/s algorithmic")
    clocks = sampler.stop() if rank == 0 else None
    if rank != 0:
        return 0
    head = results[min(a.leaves, K)]
    roofline = scan_roofline(a, head["tc_profile_rank0"], head["scan_ms_rank0"], head["scan_bytes_rank0"],
                             head["pairs_rank0"], peaks, clocks)
    roofline["kernel"] += " (rank 0's shard)"
    out = {"metric": METRIC[a.config], "value": head["queries_per_s"], "unit": "queries/s", "n_gpus": world,
           "steps": a.steps, "warmup": a.warmup, "ms_per_step": head["ms_per_step"], "higher_is_better": True,
           "scaling": "strong", "vs_baseline": None, "dtype": DTYPE[a.config], "data": "synthetic",
           "config": sharded_config(a, world), "recall_at_10": head["recall_at_10_vs_exact"],
           "e2e": {"value": head["e2e_queries_per_s"], "unit": "queries/s", "h2d_bytes_per_step": a.nq * D * 4,
                   "d2h_bytes_per_step": a.nq * (a.k * 8 + 4)},
           "gpu_launches": head["launches_rank0"] + (a.steps if world > 1 else 0),
           "roofline": roofline,
           "scan_path": dict(zip(("tensor_core_chunks", "register_lut_chunks"), searcher.path_stats())),
           "sweep": [results[L] for L in sorted(results)], "checks": checks, "clocks": clocks,
           "build_seconds": time.time() - t0}
    if a.dump_outputs:
        dump_outputs(a.dump_outputs, *head_out)
    emit(out)
    return 0


def recompute_lut16(torch, q, ids, dists, centers, codebook, index_ids, packed, off, S):
    """max relative error between returned approximate distances and a torch restatement of the residual LUT16 score
    (lut16.rs:151-173, lut16_simd.rs:39-141) of the same (query, id) pairs; C5's stand-in for 'recomputed distances'."""
    dev = q.device
    n = index_ids.numel()
    pos_of = torch.full((int(index_ids.max().item()) + 1,), -1, dtype=torch.int64, device=dev)
    pos_of[index_ids.long()] = torch.arange(n, device=dev)
    worst = 0.0
    ds = codebook.shape[2]
    for i in range(q.shape[0]):
        pos = pos_of[ids[i].long()]
        leaf = torch.searchsorted(off, pos, right=True) - 1
        for j in range(ids.shape[1]):
            res = (q[i] - centers[leaf[j]]).view(S, 1, ds)
            lut = ((res - codebook) ** 2).sum(-1)                              # [S, 16]
            mn, mx = lut.min(), lut.max()
            rng = mx - mn
            scale = 255.0 / rng if rng >= 1e-10 else torch.tensor(1.0, device=dev)
            ql = torch.floor((lut - mn) * scale + 0.5).clamp(0, 255)
            row = packed[pos[j]].long()
            codes = torch.stack([row & 15, row >> 4], 1).flatten()[:S]
            ssum = ql[torch.arange(S, device=dev), codes].sum()
            d = ssum * (1.0 / scale) + mn * S
            worst = max(worst, float((d - dists[i, j]).abs() / d.abs().clamp(min=1e-12)))
    return worst


# ======================================================================================== main
def main():
    a = parse()
    sys.dont_write_bytecode = True  # the benchmark writes nothing into the tree (it may be read-only)
    # keep stdout clean for the single JSON line: libraries (NCCL banner, …) write to fd 1
    json_fd = os.dup(1)
    os.dup2(2, 1)

    def emit(obj):
        os.write(json_fd, (json.dumps(obj) + "\n").encode())

    rank = int(os.environ.get("RANK", "0"))
    if a.impl == "reference":
        if rank != 0:
            return 0
        return reference_arm(a, emit)

    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        emit({"error": "no CUDA device; the product path has no CPU fallback"})
        return 1
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    pkg = importlib.import_module("scann-rust_b200")
    pkg.load()  # the library __graft_entry__.build() compiled; missing is an error, never a rebuild
    if a.config in ("c1", "c2"):
        if rank != 0:
            return 0
        return bench_bf(a, emit, torch, pkg, dev, local_rank)
    if a.config in ("c4", "c5"):
        return bench_sharded(a, emit, torch, dist, pkg, dev, rank, world, local_rank)
    return bench_c3(a, emit, torch, dist, pkg, dev, rank, world, local_rank)


def bench_c3(a, emit, torch, dist, pkg, dev, rank, world, local_rank):
    t0 = time.time()
    # ---------------- synthetic data + index (untimed) ----------------
    g = torch.Generator(device=dev)
    g.manual_seed(42)
    lat = torch.randn((a.latent, a.dim), generator=g, device=dev)
    x = make_points(torch, a.n, a.dim, lat, a.spread, a.decay, 42, dev)
    n_batches = 2
    queries = [make_points(torch, a.nq, a.dim, lat, a.spread, a.decay, 123 + b, dev) for b in range(n_batches)]
    log(f"[rank {rank}] data {a.n}x{a.dim} in {time.time() - t0:.1f}s")

    ix = pkg.indexing
    if rank == 0:
        gs = torch.Generator(device=dev)
        gs.manual_seed(7)
        ns = min(1_000_000, a.n)
        sample = x[torch.randperm(a.n, generator=gs, device=dev)[:ns]].contiguous() if ns < a.n else x
        centers = ix.kmeans(sample, a.partitions, 20, 7, balance_ratio=a.balance)
        a_s = ix.assign_partitions(sample, centers, local_rank)
        codebook = ix.train_codebook(sample - centers[a_s.long()], a.subspaces, 16, 20, 42)
        del sample, a_s
    else:
        centers = torch.empty((min(a.partitions, a.n), a.dim), dtype=torch.float32, device=dev)
        codebook = torch.empty((a.subspaces, 16, a.dim // a.subspaces), dtype=torch.float32, device=dev)
    if world > 1:
        dist.broadcast(centers, 0)
        dist.broadcast(codebook, 0)
    K = centers.shape[0]
    assign = ix.assign_partitions(x, centers, local_rank)
    shard_world = world
    shard_rank = rank
    if a.emulate_shard > 1 and world == 1:
        shard_world, shard_rank = a.emulate_shard, 0
    order_all = torch.argsort(assign.long(), stable=True)
    counts = torch.bincount(assign.long(), minlength=K)
    off_all = torch.zeros((K + 1,), dtype=torch.int64, device=dev)
    off_all[1:] = torch.cumsum(counts, 0)

    def build_shard(sw, sr):
        """rows of shard sr of sw (sw == 1: everything) -> (packed codes grouped by partition, ids, offsets)"""
        order, off = order_all, off_all
        if sw > 1:
            pos = torch.arange(a.n, device=dev, dtype=torch.int64)
            leaf_sorted = assign.long()[order]
            if a.shard == "rows":  # round-robin inside each partition (SURVEY §8e)
                keep = ((pos - off[leaf_sorted]) % sw) == sr
            else:
                # whole partitions per GPU, balanced by MEASURED probe load: a calibration batch of queries from the
                # same generator (its own seed, never timed) is partitioned, load(leaf) = probes x leaf size, and the
                # leaves are dealt heaviest-first to the least-loaded shard (greedy LPT).  Every rank computes the
                # same assignment.
                calib = make_points(torch, 10_000, a.dim, lat, a.spread, a.decay, 999, dev)
                part = pkg.TreePartitioner(centers, local_rank)
                tok, _ = part.partition(calib, min(a.leaves, K))
                probes = torch.bincount(tok.long().flatten().clamp_(0, K - 1), minlength=K).cpu().numpy()
                part.close()
                cnt_h = counts.cpu().numpy().astype(np.float64)
                owner_h, load = lpt_owner((probes.astype(np.float64) + 1.0) * cnt_h, sw)
                owner = torch.from_numpy(owner_h).to(dev)
                keep = owner[leaf_sorted] == sr
                if sr == 0:
                    log(f"shard plan: calibrated probe load max/mean = {load.max() / load.mean():.4f}")
            order = order[keep]
            cnt = torch.bincount(leaf_sorted[keep], minlength=K)
            off = torch.zeros((K + 1,), dtype=torch.int64, device=dev)
            off[1:] = torch.cumsum(cnt, 0)
        bpp = (a.subspaces + 1) // 2
        packed = torch.empty((order.numel(), bpp), dtype=torch.uint8, device=dev)
        for s0 in range(0, order.numel(), 1 << 21):
            idx = order[s0:s0 + (1 << 21)]
            packed[s0:s0 + (1 << 21)] = pkg.pq_encode(codebook, x[idx].contiguous(), centers, assign[idx].contiguous(),
                                                      local_rank)
        return packed, order.to(torch.int32).contiguous(), off

    packed, ids32, off = build_shard(shard_world, shard_rank)
    torch.cuda.synchronize()
    log(f"[rank {rank}] index K={K} S={a.subspaces} rows={ids32.numel()} in {time.time() - t0:.1f}s "
        f"(leaf sizes min/mean/max {int((off[1:] - off[:-1]).min())}/{ids32.numel() / K:.0f}/"
        f"{int((off[1:] - off[:-1]).max())})")
    config = c3_config(a, K, shard_world, a.shard)

    # ---------------- the CPU arm (oracle = C++ restatement of the reference algorithm) ----------------
    def cpu_arm(nq_cpu):
        import oracle
        oracle.build()
        nthreads = oracle.num_threads()
        hc, hcb = centers.cpu().numpy(), codebook.cpu().numpy()
        hoff, hids = off.cpu().numpy().astype(np.uint64), ids32.cpu().numpy().view(np.uint32)
        hpacked, hx = packed.cpu().numpy(), x.cpu().numpy()
        hq = queries[0][:nq_cpu].cpu().numpy()
        t = time.perf_counter()
        res = oracle.treex_search(hc, hcb, hoff, hids, hpacked, hx, hq, a.leaves, a.reorder, a.k, lut16=True,
                                  use_residuals=True, reorder_measure=oracle.DOT, nthreads=nthreads)
        return nq_cpu, nthreads, time.perf_counter() - t, res

    # ---------------- the GPU searcher ----------------
    cfg = pkg.TreeXHybridConfig(num_partitions=K, partitions_to_search=a.leaves, use_residuals=True,
                                pre_reorder_multiplier=a.reorder / a.k, distance_measure=pkg.DistanceMeasure.DotProduct)
    searcher = pkg.TreeXHybridSearcher(cfg, local_rank).build_from_index(centers, codebook, packed, ids32, off, x,
                                                                        borrow_raw=True)
    R = a.reorder
    xchg_events = []  # (start, end) CUDA events around the all-gather + merge of the timed steps

    # --prefetch: the partition slice + token all-gather of the NEXT batch run on a side stream while the current batch is
    # scanned (every step still does all of its own work: the tokens of step i+1 are computed during step i)
    prefetcher = pkg.distributed.TokenPrefetcher(searcher, centers, a.leaves) if world > 1 and a.prefetch else None

    def step_device(qb, timed=False, nxt=None):
        if world > 1:
            ids, dists, cnt = pkg.distributed.two_phase_search(searcher, qb, a.k, pre_reorder_k=R, prefetcher=prefetcher,
                                                               next_queries=nxt)
        elif a.split:
            ids, dists, cnt = searcher.search_end(searcher.search_begin(qb, a.k, pre_reorder_k=R))
        else:
            ids, dists, cnt = searcher.search_batched(qb, a.k, pre_reorder_k=R)
        if world > 1:
            if timed:
                ev = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
                ev[0].record()
            ids, dists, cnt = pkg.distributed.exchange_and_merge(ids, dists)
            if timed:
                ev[1].record()
                xchg_events.append(ev)
        return ids, dists, cnt

    # recall vs exact ground truth (own brute-force searcher, DotProduct)
    recall = None
    ng = min(a.gt_queries, a.nq)
    ids, dists, _ = step_device(queries[0])
    multi_check = None
    if rank == 0:
        bf = pkg.BruteForceSearcher(x, pkg.DistanceMeasure.DotProduct, local_rank)
        gt, _, _ = bf.search_batched(queries[0][:ng].contiguous(), a.k)
        torch.cuda.synchronize()
        got, want = ids[:ng].cpu().numpy(), gt.cpu().numpy()
        recall = float(np.mean([len(set(got[i]) & set(want[i])) / a.k for i in range(ng)]))
        bf.close()
        del bf
        torch.cuda.empty_cache()
        log(f"recall@{a.k} vs exact = {recall:.4f} ({ng} queries)")
        if world > 1 and a.check_queries > 0:
            # multi-GPU self-check: the merged N-rank result against ONE index holding every row, on a subsample
            nchk = min(a.check_queries, a.nq)
            pk1, id1, off1 = build_shard(1, 0)
            full = pkg.TreeXHybridSearcher(cfg, local_rank).build_from_index(centers, codebook, pk1, id1, off1, x,
                                                                             borrow_raw=True)
            si, sd, _ = full.search_batched(queries[0][:nchk].contiguous(), a.k, pre_reorder_k=R)
            torch.cuda.synchronize()
            multi_check = {
                "queries": nchk,
                "sharded_dist_le_single_index": bool((dists[:nchk] <= sd + 1e-6 * sd.abs() + 1e-12).all().item()),
                "id_agreement_with_single_index": float(np.mean(
                    [len(set(ids[i].tolist()) & set(si[i].tolist())) / a.k for i in range(nchk)]))}
            full.close()
            del full, pk1, id1, off1
            torch.cuda.empty_cache()
            log(f"multi-GPU self-check: {multi_check}")

    if a.sweep_leaves:
        for Ls in a.sweep_leaves.split(","):
            Lv = int(Ls)
            searcher.config.partitions_to_search = Lv
            i2, _, _ = step_device(queries[0])
            torch.cuda.synchronize()
            t = time.perf_counter()
            for _ in range(3):
                step_device(queries[1])
            torch.cuda.synchronize()
            dt = (time.perf_counter() - t) / 3
            if rank == 0:
                g2 = i2[:ng].cpu().numpy()
                r = float(np.mean([len(set(g2[i]) & set(want[i])) / a.k for i in range(ng)]))
                log(f"L={Lv}: recall@{a.k}={r:.4f} qps={a.nq / dt:.0f}")
        return 0

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------- timed: device-resident ----------------
    for w in range(a.warmup):
        step_device(queries[w % n_batches], nxt=queries[(w + 1) % n_batches] if w + 1 < a.warmup else queries[0])
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    searcher.set_profiling(True)
    if a.phase_times and world > 1:
        pkg.distributed._PHASE_MARKS = []
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for s in range(a.steps):
        last = step_device(queries[s % n_batches], timed=True, nxt=queries[(s + 1) % n_batches])
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    tcp = searcher.tc_profile()
    prof, launches = searcher.get_profile()
    searcher.set_profiling(False)
    if a.phase_times and world > 1:
        mk = pkg.distributed._PHASE_MARKS
        pkg.distributed._PHASE_MARKS = None
        per = len(mk) // a.steps
        names = ["partition slice", "all-gather tokens", "search_begin", "all-reduce tau", "search_end"]
        acc = [0.0] * (per - 1)
        for st in range(a.steps):
            for j in range(per - 1):
                acc[j] += mk[st * per + j].elapsed_time(mk[st * per + j + 1])
        log(f"[rank {rank}] phases: " + ", ".join(f"{nm} {v / a.steps:.3f}" for nm, v in zip(names, acc)))
    scan_bytes, pairs = searcher.last_scan_bytes()  # algorithmic bytes of one step (this rank's shard)
    xchg_ms = sum(e[0].elapsed_time(e[1]) for e in xchg_events) / max(1, len(xchg_events))
    log(f"[rank {rank}] {ms / a.steps:.3f} ms/step; all-gather+merge {xchg_ms:.3f}; stages " +
        ", ".join(f"{k2} {v / a.steps:.3f}" for k2, v in prof.items()) + f"; scan bytes {scan_bytes / 1e9:.1f} GB")
    tmax = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    ms = float(tmax.item())
    value = a.nq * a.steps / (ms / 1e3)

    # ---------------- timed: end to end through the host API ----------------
    hq = [torch.empty((a.nq, a.dim), dtype=torch.float32, pin_memory=True) for _ in range(n_batches)]
    for b in range(n_batches):
        hq[b].copy_(queries[b])
    hq_np = [t.numpy() for t in hq]

    def step_host(b):
        if world > 1:  # pinned host queries -> device -> split search + exchange -> host results
            mi, md, mc = step_device(hq[b].to(dev, non_blocking=True))
            return mi.cpu().numpy(), md.cpu().numpy()
        ids, dists, cnt = searcher.search_batched(hq_np[b], a.k, pre_reorder_k=R)
        return ids, dists

    for w in range(max(1, a.warmup)):
        step_host(w % n_batches)
    barrier()
    t = time.perf_counter()
    for s in range(a.steps):
        step_host(s % n_batches)
    barrier()
    e2e_s = time.perf_counter() - t
    te = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_val = a.nq * a.steps / float(te.item())
    clocks = sampler.stop() if rank == 0 else None

    if rank != 0:
        return 0

    peaks = load_peaks()
    scan_ms_per_launch = prof["scan"] / a.steps
    # physical DRAM traffic of one scan launch from the committed `ncu --set full` capture of this kernel at this
    # workload (profiles/scan_traffic.json names the capture); null when the capture is of another workload / kernel
    traffic, traffic_src = None, None
    tp = os.path.join(ROOT, "profiles", "scan_traffic.json")
    if os.path.exists(tp) and world == 1 and a.n == DEFAULTS["c3"]["n"] and a.nq == DEFAULTS["c3"]["nq"]:
        try:
            tj = json.load(open(tp))
            key = "tc_scan_kernel" if tcp["launches"] > 0 else "lut16_scan_kernel"
            if key in tj:
                traffic, traffic_src = tj[key].get("dram_bytes_per_launch"), tj[key].get("source")
        except Exception:
            pass
    roofline = scan_roofline(a, tcp, scan_ms_per_launch, scan_bytes, pairs, peaks, clocks, traffic, traffic_src)
    out = {
        "metric": METRIC["c3"], "value": value, "unit": "queries/s",
        "n_gpus": world, "steps": a.steps, "warmup": a.warmup, "ms_per_step": ms / a.steps, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": DTYPE["c3"],
        "data": "synthetic", "config": config, "recall_at_10": recall,
        "e2e": {"value": e2e_val, "unit": "queries/s", "h2d_bytes_per_step": a.nq * a.dim * 4,
                "d2h_bytes_per_step": a.nq * (a.k * 8 + 4)},
        "gpu_launches": int(launches) + (a.steps if world > 1 else 0),  # + merge_topk per step when sharded
        "roofline": roofline,
        "scan_path": dict(zip(("tensor_core_chunks", "register_lut_chunks"), searcher.path_stats())),
        "stage_ms_per_step": {k2: v / a.steps for k2, v in prof.items()},
        "multi_gpu_check": multi_check,
        "clocks": clocks,
    }
    if world == 1 and not a.no_cpu_baseline:
        nqc, nthreads, secs, _ = cpu_arm(a.cpu_queries)
        out["cpu_baseline"] = {"value": nqc / secs, "unit": "queries/s", "cores": nthreads, "kind": "port",
                               "sample": f"{nqc} queries of the same batch on the same index; oracle/ C++ restatement "
                                         "of the reference algorithm, one task per query over all host threads"}
    if a.dump_outputs:
        dump_outputs(a.dump_outputs, *last)
    emit(out)
    return 0


if __name__ == "__main__":
    rc = main()
    try:
        import torch.distributed as dist
        if dist.is_initialized():
            dist.destroy_process_group()
    except Exception:
        pass
    sys.exit(rc)
