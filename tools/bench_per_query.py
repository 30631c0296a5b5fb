"""Per-query search parameters on the C3 index: one 10k-query batch whose queries ask for different k, pre-reorder R or
leaves to search, timed three ways.

Workloads (per-query values drawn at random, seeded):
  k3        k_q in {1, 10, 100}, R_q = 10 * k_q
  leaves4   L_q in {16, 32, 64, 128}, k = 10, R = 100
  k100      k_q uniform in 1..100, R_q = 10 * k_q (100 groups)

Ways, alternated inside one run on the index and queries bench.py --config c3 builds from its seeds:
  grouped    one scann_treeah_search per distinct (L_q, R_q, k_q), one after another (the queries of every group are
             gathered outside the timed window)
  per_query  one scann_treeah_search_with_params call with device-resident per-query arrays
  uniform    one scann_treeah_search at the batch maxima (what a caller pays to serve every query at the largest values)

Timed through the C ABI with device-resident queries: CUDA events around each step.  Reports ms per step (median over
rounds), the path counters (chunks on the tensor-core / register-LUT scan) and the device time per stage of one step,
and checks that grouped and per_query return the same rows bit for bit.  Prints the card name and power limit beside
the numbers.

  python tools/bench_per_query.py [--n 10000000] [--nq 10000] [--steps 3] [--rounds 3] [--out results/per_query.json]
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


def main():
    d = bench.DEFAULTS["c3"]
    p = argparse.ArgumentParser()
    p.add_argument("--n", type=int, default=d["n"])
    p.add_argument("--nq", type=int, default=d["nq"])
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
    R0, k0, L0 = d["reorder"], d["k"], d["leaves"]
    cfg = pkg.TreeXHybridConfig(num_partitions=K, partitions_to_search=L0, use_residuals=True,
                                pre_reorder_multiplier=R0 / k0, distance_measure=pkg.DistanceMeasure.DotProduct)
    s = pkg.TreeXHybridSearcher(cfg, 0).build_from_index(centers, codebook, packed, ids32, off, x, borrow_raw=True)
    torch.cuda.synchronize()
    print(f"index {a.n}x{d['dim']} K={K} in {time.time() - t0:.1f}s", file=sys.stderr)

    # ---- workloads: per-query (L, R, k) [nq, 3]
    rng = np.random.default_rng(2024)
    nq = a.nq
    k3 = rng.choice([1, 10, 100], nq)
    k100 = rng.integers(1, 101, nq)
    workloads = {
        "k3": np.stack([np.full(nq, L0), 10 * k3, k3], 1),
        "leaves4": np.stack([rng.choice([16, 32, 64, 128], nq), np.full(nq, R0), np.full(nq, k0)], 1),
        "k100": np.stack([np.full(nq, L0), 10 * k100, k100], 1),
    }
    ptr = lambda t: C.c_void_p(t.data_ptr())  # noqa: E731
    stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    dim = d["dim"]

    def out_bufs(m, k):
        return (torch.empty((m, k), dtype=torch.int32, device=dev), torch.empty((m, k), dtype=torch.float32, device=dev),
                torch.empty((m,), dtype=torch.int32, device=dev))

    plans = {}
    for name, prm in workloads.items():
        Lm, Rm, km = (int(v) for v in prm.max(0))
        keys, inv = np.unique(prm, axis=0, return_inverse=True)
        inv = inv.reshape(-1)
        groups = []
        for gi, (L, R, k) in enumerate(keys):
            sel = np.nonzero(inv == gi)[0]
            groups.append((int(L), int(R), int(k), sel, q[torch.from_numpy(sel).to(dev)].contiguous(),
                           out_bufs(len(sel), int(k))))
        arrs = [torch.from_numpy(prm[:, j].astype(np.int32)).to(dev) for j in range(3)]
        plans[name] = dict(max=(Lm, Rm, km), groups=groups, arrs=arrs, pq=out_bufs(nq, km), uni=out_bufs(nq, km))

    def step(name, way):
        pl = plans[name]
        Lm, Rm, km = pl["max"]
        if way == "grouped":
            for L, R, k, _, qg, (i, dd, c) in pl["groups"]:
                capi.check(lib.scann_treeah_search(s._h, ptr(qg), qg.shape[0], dim, L, R, k, ptr(i), ptr(dd), ptr(c),
                                                   None, None, None, capi.DEVICE, stream))
        elif way == "per_query":
            i, dd, c = pl["pq"]
            La, Ra, ka = pl["arrs"]
            capi.check(lib.scann_treeah_search_with_params(s._h, ptr(q), nq, dim, Lm, Rm, km, ptr(La), ptr(Ra), ptr(ka),
                                                           ptr(i), ptr(dd), ptr(c), None, None, None, capi.DEVICE,
                                                           stream))
        else:
            i, dd, c = pl["uni"]
            capi.check(lib.scann_treeah_search(s._h, ptr(q), nq, dim, Lm, Rm, km, ptr(i), ptr(dd), ptr(c), None, None,
                                               None, capi.DEVICE, stream))

    ways = ("grouped", "per_query", "uniform")
    res = {}
    for name in workloads:  # warm-up, the path counters of one step, and the identity check
        res[name] = {"groups": len(plans[name]["groups"]), "max_L_R_k": plans[name]["max"]}
        for way in ways:
            step(name, way)
            tc0, lut0 = s.path_stats()
            step(name, way)
            tc1, lut1 = s.path_stats()
            torch.cuda.synchronize()
            res[name][way] = {"path_stats_per_step": {"tensor_core_chunks": tc1 - tc0, "register_lut_chunks": lut1 - lut0},
                              "ms": []}
        pi, pd, pc = (t.cpu().numpy() for t in plans[name]["pq"])
        for L, R, k, sel, _, (i, dd, c) in plans[name]["groups"]:
            i, dd, c = i.cpu().numpy(), dd.cpu().numpy(), c.cpu().numpy()
            assert (pc[sel] == c).all() and (pi[sel, :k] == i).all(), f"{name}: ids differ in group {(L, R, k)}"
            assert (pd[sel, :k].view(np.uint32) == dd.view(np.uint32)).all(), f"{name}: dists differ in group {(L, R, k)}"
            assert (pi[sel, k:] == -1).all() and np.isinf(pd[sel, k:]).all(), f"{name}: padding of group {(L, R, k)}"
        res[name]["grouped_equals_per_query"] = True
    for _ in range(a.rounds):
        for name in workloads:
            for way in ways:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(a.steps):
                    step(name, way)
                e1.record()
                torch.cuda.synchronize()
                res[name][way]["ms"].append(e0.elapsed_time(e1) / a.steps)
    for name in workloads:  # after the timing: device milliseconds per stage of one step (profiling on)
        for way in ways:
            s.set_profiling(True)
            step(name, way)
            stages, _ = s.get_profile()
            s.set_profiling(False)
            res[name][way]["stage_ms"] = {k: round(v, 3) for k, v in stages.items()}
    gpu = card()
    for name, r in res.items():
        for way in ways:
            w = r[way]
            w["ms_per_step"] = float(np.median(w["ms"]))
            ps = w["path_stats_per_step"]
            print(f"{name:8s} {way:9s} {w['ms_per_step']:9.3f} ms/step  rounds {['%.3f' % v for v in w['ms']]}  "
                  f"path (tc, lut) = ({ps['tensor_core_chunks']}, {ps['register_lut_chunks']})  groups {r['groups']}  "
                  f"stages {w['stage_ms']}   [{gpu}]")
    out = {"gpu": gpu, "n": a.n, "nq": nq, "K": int(K), "steps": a.steps, "rounds": a.rounds, "workloads": res}
    print(json.dumps(out))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
