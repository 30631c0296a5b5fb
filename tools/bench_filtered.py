"""Filtered Tree-AH search on the C3 index: one 10k-query batch, unfiltered and with restrict filters.

Variants (alternated inside one run, on the index and queries bench.py --config c3 builds from its seeds):
  none          plain scann_treeah_search
  shared50      one filter for the whole batch, 50 % of the ids kept
  shared10      one filter, 10 % kept
  distinct16    16 distinct filters at 50 %, assigned to queries at random
  distinct256   256 distinct filters at 50 %

Timed through the C ABI with device-resident queries, bitmaps and rows (the bitmaps are packed once, outside the timed
window): CUDA events around each step.  Reports ms per step (median over rounds), the path counters (chunks on the
tensor-core / register-LUT scan) and, from one untimed SCANN_TC_DEBUG call, how many queries the tensor-core pass flagged
back to the register-LUT kernel.  Prints the card name and power limit beside the numbers.

  python tools/bench_filtered.py [--n 10000000] [--nq 10000] [--steps 5] [--rounds 3] [--out results/filtered.json]
"""
import argparse
import ctypes as C
import importlib
import json
import os
import re
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402  (seeded data model of the C3 benchmark)


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def capture_stderr(fn):
    """runs fn() and returns what the library printed on fd 2 meanwhile"""
    sys.stderr.flush()
    saved = os.dup(2)
    with tempfile.TemporaryFile(mode="w+b") as f:
        os.dup2(f.fileno(), 2)
        try:
            fn()
        finally:
            os.dup2(saved, 2)
            os.close(saved)
        f.seek(0)
        return f.read().decode("utf-8", "replace")


def main():
    d = bench.DEFAULTS["c3"]
    p = argparse.ArgumentParser()
    p.add_argument("--n", type=int, default=d["n"])
    p.add_argument("--nq", type=int, default=d["nq"])
    p.add_argument("--steps", type=int, default=5)
    p.add_argument("--rounds", type=int, default=3)
    p.add_argument("--out", default=None)
    a = p.parse_args()
    import torch

    pkg = importlib.import_module("scann-rust_b200")
    capi = pkg.capi
    lib = capi.load()
    dev = torch.device("cuda", 0)
    t0 = time.time()
    # ---- bench.py's C3 data and index (same seeds and steps as bench_c3, single GPU)
    g = torch.Generator(device=dev)
    g.manual_seed(42)
    lat = torch.randn((d["latent"], d["dim"]), generator=g, device=dev)
    x = bench.make_points(torch, a.n, d["dim"], lat, d["spread"], d["decay"], 42, dev)
    q = bench.make_points(torch, a.nq, d["dim"], lat, d["spread"], d["decay"], 123, dev)
    ix = pkg.indexing
    gs = torch.Generator(device=dev)
    gs.manual_seed(7)
    ns = min(1_000_000, a.n)
    sample = x[torch.randperm(a.n, generator=gs, device=dev)[:ns]].contiguous() if ns < a.n else x
    centers = ix.kmeans(sample, d["partitions"], 20, 7, balance_ratio=d["balance"])
    a_s = ix.assign_partitions(sample, centers, 0)
    codebook = ix.train_codebook(sample - centers[a_s.long()], d["subspaces"], 16, 20, 42)
    del sample, a_s
    K = centers.shape[0]
    assign = ix.assign_partitions(x, centers, 0)
    order = torch.argsort(assign.long(), stable=True)
    off = torch.zeros((K + 1,), dtype=torch.int64, device=dev)
    off[1:] = torch.cumsum(torch.bincount(assign.long(), minlength=K), 0)
    bpp = (d["subspaces"] + 1) // 2
    packed = torch.empty((a.n, bpp), dtype=torch.uint8, device=dev)
    for s0 in range(0, a.n, 1 << 21):
        idx = order[s0:s0 + (1 << 21)]
        packed[s0:s0 + (1 << 21)] = pkg.pq_encode(codebook, x[idx].contiguous(), centers, assign[idx].contiguous(), 0)
    ids32 = order.to(torch.int32).contiguous()
    R, k, L = d["reorder"], d["k"], d["leaves"]
    cfg = pkg.TreeXHybridConfig(num_partitions=K, partitions_to_search=L, use_residuals=True,
                                pre_reorder_multiplier=R / k, distance_measure=pkg.DistanceMeasure.DotProduct)
    s = pkg.TreeXHybridSearcher(cfg, 0).build_from_index(centers, codebook, packed, ids32, off, x, borrow_raw=True)
    torch.cuda.synchronize()
    print(f"index {a.n}x{d['dim']} K={K} in {time.time() - t0:.1f}s", file=sys.stderr)

    # ---- filters: packed bitmaps [F][ceil(n/8)] and rows on the device
    gen = torch.Generator(device=dev)
    gen.manual_seed(2024)
    nb = (a.n + 7) // 8

    def bitmaps(F, keep):
        return torch.randint(0, 256, (F, nb), generator=gen, device=dev, dtype=torch.uint8) if keep == 0.5 else \
            torch.stack([torch.nn.functional.pad(torch.rand(a.n, generator=gen, device=dev) < keep,
                                                 (0, nb * 8 - a.n)).reshape(nb, 8).to(torch.uint8)
                         .mul(torch.tensor([1, 2, 4, 8, 16, 32, 64, 128], dtype=torch.uint8, device=dev))
                         .sum(-1, dtype=torch.uint8) for _ in range(F)])

    def rows(F):
        return torch.randint(0, F, (a.nq,), generator=gen, device=dev, dtype=torch.int32)

    variants = {"none": None, "shared50": (bitmaps(1, 0.5), torch.zeros(a.nq, dtype=torch.int32, device=dev)),
                "shared10": (bitmaps(1, 0.1), torch.zeros(a.nq, dtype=torch.int32, device=dev)),
                "distinct16": (bitmaps(16, 0.5), rows(16)), "distinct256": (bitmaps(256, 0.5), rows(256))}
    ids = torch.empty((a.nq, k), dtype=torch.int32, device=dev)
    dists = torch.empty((a.nq, k), dtype=torch.float32, device=dev)
    counts = torch.empty((a.nq,), dtype=torch.int32, device=dev)
    ptr = lambda t: C.c_void_p(t.data_ptr())  # noqa: E731
    stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)

    def step(name):
        v = variants[name]
        if v is None:
            st = lib.scann_treeah_search(s._h, ptr(q), a.nq, d["dim"], L, R, k, ptr(ids), ptr(dists), ptr(counts), None,
                                         None, None, capi.DEVICE, stream)
        else:
            bits, fq = v
            st = lib.scann_treeah_search_filtered(s._h, ptr(q), a.nq, d["dim"], L, R, k, ptr(bits), bits.shape[0], a.n,
                                                  ptr(fq), ptr(ids), ptr(dists), ptr(counts), None, None, None,
                                                  capi.DEVICE, stream)
        capi.check(st)

    res = {}
    for name in variants:  # warm-up and the path counters of one call per variant
        step(name)
        tc0, lut0 = s.path_stats()
        step(name)
        tc1, lut1 = s.path_stats()
        torch.cuda.synchronize()
        res[name] = {"path_stats_per_call": {"tensor_core_chunks": tc1 - tc0, "register_lut_chunks": lut1 - lut0},
                     "mean_count": float(counts.float().mean()), "ms": []}
    for _ in range(a.rounds):
        for name in variants:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(a.steps):
                step(name)
            e1.record()
            torch.cuda.synchronize()
            res[name]["ms"].append(e0.elapsed_time(e1) / a.steps)
    for name in variants:  # after the timing: one SCANN_TC_DEBUG call (synchronising) for the flagged queries
        os.environ["SCANN_TC_DEBUG"] = "1"
        text = capture_stderr(lambda: (step(name), torch.cuda.synchronize()))
        os.environ.pop("SCANN_TC_DEBUG")
        m = re.findall(r"flagged (\d+)", text)
        mean = re.findall(r"candidates/query mean ([\d.]+)", text)
        res[name]["flagged_queries"] = sum(int(v) for v in m) if m else 0
        res[name]["tc_candidates_per_query_mean"] = float(mean[0]) if mean else None
    gpu = card()
    for name, r in res.items():
        r["ms_per_step"] = float(np.median(r["ms"]))
        print(f"{name:12s} {r['ms_per_step']:8.3f} ms/step  rounds {['%.3f' % v for v in r['ms']]}  "
              f"path (tc, lut) = ({r['path_stats_per_call']['tensor_core_chunks']}, "
              f"{r['path_stats_per_call']['register_lut_chunks']})  flagged {r['flagged_queries']}  "
              f"mean count {r['mean_count']:.2f}   [{gpu}]")
    out = {"gpu": gpu, "n": a.n, "nq": a.nq, "K": int(K), "L": L, "R": R, "k": k, "steps": a.steps, "rounds": a.rounds,
           "variants": res}
    print(json.dumps(out))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
