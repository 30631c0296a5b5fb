"""Tree-X-Hybrid over byte codes with the f32 LookupTable (scann_treeah_create_lut_f32): time, recall and the scan's
shared-memory lookup rate, next to the LUT16 handle on the same centres.

Workloads (bench.py's seeded C3 data model, device-resident queries):
  a_c3_f32    C3 geometry: 10M x 96, K = 2000 balanced k-means centres, S = 48, C = 256, L = 64, R = 100, k = 10, 10k
              queries, Dot reorder
  a_c3_lut16  the same centres with the 16-code nibble index (what bench.py measures)
  b_s24_f32   S = 24 (ds = 4), C = 256 on the same data and centres
  c_hashed    the "hashed" shape: flat K = 1, 1M x 128, S = 8, C = 256, k = 10 (approximate distances, no reorder)

Index: centres from the library's balanced scann_kmeans_fit (as bench.py's C3 does); the C = 256 codebook from
scann_kmeans_fit run once per subspace slice (pointer + s*ds, stride dim, K = C) over residuals of a 200k-row sample;
codes from a torch argmin encode — plumbing only: the oracle-checked tests feed the same arrays to both sides.

Reports per workload: ms per step (CUDA events, median over rounds), queries/s, device time per stage of one step,
recall@10 against exact ground truth (BruteForceSearcher) on the first 1000 queries, and for the byte-code scan its
lookup rate: Σ over pairs of |leaf| * S (scann_treeah_last_scan_bytes) over the scan stage's time, next to the bound of
32 lookups/clk/SM x SMs x the maximum SM clock.  For (a) recall@10 is also given at R = 30 for both code formats.
Prints the card name, power limit and maximum SM clock beside the numbers.

  python tools/bench_treeah_f32lut.py [--n 10000000] [--nq 10000] [--steps 3] [--rounds 3] [--out results/f32lut.json]
"""
import argparse
import ctypes as C
import importlib
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import bench  # noqa: E402  (seeded data model of the C3 benchmark)
from bench_filtered import card  # noqa: E402


def codebook_256(torch, lib, capi, resid, S, C_, seed):
    """scann_kmeans_fit once per subspace slice of resid [m, dim] (stride dim) -> [S, C, ds]"""
    m, dim = resid.shape
    ds = dim // S
    cb = torch.empty((S, C_, ds), dtype=torch.float32, device=resid.device)
    for s in range(S):
        capi.check(lib.scann_kmeans_fit(resid.data_ptr() + 4 * s * ds, m, ds, dim, C_, 20, seed + s, 0.0,
                                        cb[s].data_ptr(), 0, capi.DEVICE))
    return cb


def encode(torch, x, centers, assign, cb, chunk=1 << 20):
    """argmin encode of x - centers[assign] against cb [S, C, ds] -> [n, S] u8 (centers None: no residual)"""
    S, C_, ds = cb.shape
    out = torch.empty((x.shape[0], S), dtype=torch.uint8, device=x.device)
    for i in range(0, x.shape[0], chunk):
        r = x[i:i + chunk]
        if centers is not None:
            r = r - centers[assign[i:i + chunk].long()]
        r = r.reshape(r.shape[0], S, ds)
        for s in range(S):
            out[i:i + chunk, s] = torch.cdist(r[:, s], cb[s]).argmin(1).to(torch.uint8)
    return out


def main():
    d = bench.DEFAULTS["c3"]
    p = argparse.ArgumentParser()
    p.add_argument("--n", type=int, default=d["n"])
    p.add_argument("--nq", type=int, default=d["nq"])
    p.add_argument("--n_flat", type=int, default=1_000_000)
    p.add_argument("--steps", type=int, default=3)
    p.add_argument("--rounds", type=int, default=3)
    p.add_argument("--out", default=None)
    a = p.parse_args()
    import torch

    pkg = importlib.import_module("scann-rust_b200")
    capi = pkg.capi
    lib = capi.load()
    dev = torch.device("cuda", 0)
    t0 = time.time()
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
    resid = (sample - centers[a_s.long()])[:200_000].contiguous()
    cb16 = ix.train_codebook(sample - centers[a_s.long()], d["subspaces"], 16, 20, 42)
    cb48 = codebook_256(torch, lib, capi, resid, 48, 256, 42)
    cb24 = codebook_256(torch, lib, capi, resid, 24, 256, 42)
    del sample, a_s, resid
    K = centers.shape[0]
    assign = ix.assign_partitions(x, centers, 0)
    order = torch.argsort(assign.long(), stable=True)
    off = torch.zeros((K + 1,), dtype=torch.int64, device=dev)
    off[1:] = torch.cumsum(torch.bincount(assign.long(), minlength=K), 0)
    xs, asg = x[order].contiguous(), assign[order].contiguous()
    packed = torch.empty((a.n, (d["subspaces"] + 1) // 2), dtype=torch.uint8, device=dev)
    for s0 in range(0, a.n, 1 << 21):
        packed[s0:s0 + (1 << 21)] = pkg.pq_encode(cb16, xs[s0:s0 + (1 << 21)], centers, asg[s0:s0 + (1 << 21)], 0)
    codes48 = encode(torch, xs, centers, asg, cb48)
    codes24 = encode(torch, xs, centers, asg, cb24)
    del xs, asg
    ids32 = order.to(torch.int32).contiguous()
    R0, k0, L0 = d["reorder"], d["k"], d["leaves"]
    cfg = pkg.TreeXHybridConfig(num_partitions=K, partitions_to_search=L0, use_residuals=True,
                                pre_reorder_multiplier=R0 / k0, distance_measure=pkg.DistanceMeasure.DotProduct)
    handles = {
        "a_c3_f32": pkg.TreeXHybridSearcher(cfg, 0).build_from_byte_codes(centers, cb48, codes48, ids32, off, x,
                                                                          borrow_raw=True),
        "a_c3_lut16": pkg.TreeXHybridSearcher(cfg, 0).build_from_index(centers, cb16, packed, ids32, off, x,
                                                                       borrow_raw=True),
        "b_s24_f32": pkg.TreeXHybridSearcher(cfg, 0).build_from_byte_codes(centers, cb24, codes24, ids32, off, x,
                                                                           borrow_raw=True),
    }
    del codes48, codes24, packed
    # (c) the "hashed" shape: flat, 1M x 128, S = 8, C = 256, no residuals
    gf = torch.Generator(device=dev)
    gf.manual_seed(11)
    latf = torch.randn((d["latent"], 128), generator=gf, device=dev)
    xf = bench.make_points(torch, a.n_flat, 128, latf, d["spread"], d["decay"], 43, dev)
    qf = bench.make_points(torch, a.nq, 128, latf, d["spread"], d["decay"], 124, dev)
    cbf = codebook_256(torch, lib, capi, xf[:200_000].contiguous(), 8, 256, 42)
    cfgf = pkg.TreeXHybridConfig(num_partitions=1, partitions_to_search=1, use_residuals=False,
                                 pre_reorder_multiplier=1.0, distance_measure=pkg.DistanceMeasure.SquaredL2)
    handles["c_hashed"] = pkg.TreeXHybridSearcher(cfgf, 0).build_from_byte_codes(
        torch.zeros((1, 128), device=dev), cbf, encode(torch, xf, None, None, cbf),
        torch.arange(a.n_flat, dtype=torch.int32, device=dev), torch.tensor([0, a.n_flat], device=dev), None)
    torch.cuda.synchronize()
    print(f"indexes built in {time.time() - t0:.1f}s", file=sys.stderr)

    work = {name: (q, L0, R0, k0, 96, S, x, pkg.DistanceMeasure.DotProduct)
            for name, S in (("a_c3_f32", 48), ("a_c3_lut16", 48), ("b_s24_f32", 24))}
    work["c_hashed"] = (qf, 1, k0, k0, 128, 8, xf, pkg.DistanceMeasure.SquaredL2)
    ptr = lambda t: C.c_void_p(t.data_ptr())  # noqa: E731
    stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    outs = {name: (torch.empty((a.nq, k0), dtype=torch.int32, device=dev),
                   torch.empty((a.nq, k0), dtype=torch.float32, device=dev),
                   torch.empty((a.nq,), dtype=torch.int32, device=dev)) for name in work}

    def step(name, R=None):
        qq, L, R0_, k, dim, _, _, _ = work[name]
        i, dd, c = outs[name]
        capi.check(lib.scann_treeah_search(handles[name]._h, ptr(qq), qq.shape[0], dim, L, R if R else R0_, k, ptr(i),
                                           ptr(dd), ptr(c), None, None, None, capi.DEVICE, stream))

    gts = {}

    def recall(name, R=None):
        qq, _, _, k, _, _, xx, measure = work[name]
        key = (xx.data_ptr(), int(measure))
        if key not in gts:  # exact ground truth of the first 1000 queries
            bf = pkg.BruteForceSearcher(xx, measure)
            gts[key] = bf.search_batched(qq[:1000], k)[0].cpu().numpy()
            bf.close()
        step(name, R)
        got = outs[name][0][:1000].cpu().numpy()
        gt = gts[key]
        return float(np.mean([len(set(got[j]) & set(gt[j])) / k for j in range(len(got))]))

    res = {name: {"ms": []} for name in work}
    for name in work:
        step(name)  # warm-up
        res[name]["recall@10"] = round(recall(name), 4)
        if name.startswith("a_"):
            res[name]["recall@10_R30"] = round(recall(name, 30), 4)
    torch.cuda.synchronize()
    for _ in range(a.rounds):
        for name in work:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(a.steps):
                step(name)
            e1.record()
            torch.cuda.synchronize()
            res[name]["ms"].append(e0.elapsed_time(e1) / a.steps)
    gpu = card()
    try:
        sm_mhz = float(gpu.split(",")[2].strip().split()[0])
    except (IndexError, ValueError):
        sm_mhz = float("nan")
    sms = torch.cuda.get_device_properties(dev).multi_processor_count
    bound = 32.0 * sms * sm_mhz * 1e6  # shared-memory lookups per second: 32 per clock per SM
    for name in work:  # after the timing: device milliseconds per stage of one step (profiling on)
        s = handles[name]
        s.set_profiling(True)
        step(name)
        stages, _ = s.get_profile()
        s.set_profiling(False)
        r = res[name]
        r["stage_ms"] = {k: round(v, 3) for k, v in stages.items()}
        r["ms_per_step"] = float(np.median(r["ms"]))
        r["queries_per_s"] = round(a.nq / r["ms_per_step"] * 1e3)
        r["path_stats"] = s.path_stats()
        if name.endswith("f32") or name == "c_hashed":
            lookups, pairs = s.last_scan_bytes()  # Σ pairs |leaf| * S: one table lookup per byte
            r["lookups"] = int(lookups)
            r["lookups_per_s"] = lookups / (stages["scan"] * 1e-3)
            r["share_of_lookup_bound"] = round(r["lookups_per_s"] / bound, 3)
        print(f"{name:11s} {r['ms_per_step']:9.3f} ms/step  {r['queries_per_s']:9d} q/s  recall@10 {r['recall@10']}"
              f"{'  R30 %.4f' % r['recall@10_R30'] if 'recall@10_R30' in r else ''}  stages {r['stage_ms']}"
              f"{'  lookups/s %.3g (%.1f%% of bound)' % (r['lookups_per_s'], 100 * r['share_of_lookup_bound']) if 'lookups' in r else ''}"
              f"   [{gpu}]")
    out = {"gpu": gpu, "sms": sms, "lookup_bound_per_s": bound, "n": a.n, "n_flat": a.n_flat, "nq": a.nq, "K": int(K),
           "steps": a.steps, "rounds": a.rounds, "workloads": res}
    print(json.dumps(out))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
