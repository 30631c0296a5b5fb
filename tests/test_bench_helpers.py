"""CPU tests of the bench harness pieces that run without a GPU: the shard plan, the torch-only index build of the
reference arm (oracle/ref_index.py) and the reference arm itself at a tiny size."""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_lpt_owner_balances_and_is_deterministic():
    sys.path.insert(0, ROOT)
    import bench

    rng = np.random.default_rng(0)
    load = rng.pareto(1.5, 4096) + 0.01
    owner, loads = bench.lpt_owner(load, 8)
    owner2, _ = bench.lpt_owner(load, 8)
    assert (owner == owner2).all() and owner.min() == 0 and owner.max() == 7
    assert np.allclose(loads, np.bincount(owner, weights=load, minlength=8))
    assert loads.max() / loads.mean() < 1.02 or loads.max() - loads.mean() <= load.max()


def test_ref_index_build_and_oracle_search(oracle):
    """the reference arm's torch-only index gives a searchable Tree-AH index (recall vs exact on clustered data)"""
    import torch

    from oracle import ref_index

    sys.path.insert(0, ROOT)
    import bench

    g = torch.Generator().manual_seed(1)
    lat = torch.randn((32, 32), generator=g)
    x = bench.make_points(torch, 20_000, 32, lat, 0.5, 1.0, 42, torch.device("cpu"))
    q = bench.make_points(torch, 64, 32, lat, 0.5, 1.0, 123, torch.device("cpu"))
    idx = ref_index.build_treeah(torch, x, 16, 16, 20_000, 5)
    off = idx["off"].numpy().astype(np.uint64)
    assert off[0] == 0 and off[-1] == 20_000 and (np.diff(off.astype(np.int64)) >= 0).all()
    assert sorted(idx["ids"].tolist()) == list(range(20_000))
    rc, ids, dists, counts = oracle.treex_search(idx["centers"].numpy(), idx["codebook"].numpy(), off,
                                                 idx["ids"].numpy().astype(np.uint32), idx["packed"].numpy(), x.numpy(),
                                                 q.numpy(), 8, 100, 10, lut16=True, use_residuals=True,
                                                 reorder_measure=oracle.DOT, nthreads=4)[:4]
    assert rc == 0 and (counts == 10).all()
    want = torch.topk(q @ x.t(), 10, dim=1).indices.numpy()
    rec = np.mean([len(set(ids[i].tolist()) & set(want[i].tolist())) / 10 for i in range(64)])
    assert rec > 0.8, rec


def test_reference_arm_runs_without_the_product_library():
    """bench.py --impl reference prints the contract's JSON line and never loads libscann_b200.so"""
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--n", "20000", "--partitions", "16",
           "--latent", "32", "--nq", "32", "--ref-queries", "16", "--steps", "1", "--warmup", "1", "--leaves", "8"]
    env = dict(os.environ, LD_DEBUG="files")
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=env)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["metric"].startswith("queries/sec @ recall@10>=0.95")
    assert line["cpu_baseline"]["kind"] == "port" and line["e2e"]["h2d_bytes_per_step"] == 0
    assert "libscann_b200" not in r.stderr and "libscann_oracle" in r.stderr


def test_dump_outputs_is_identical_run_to_run(tmp_path):
    """--dump-outputs writes the last timed step's results; with the same arguments two runs write the same arrays"""
    dumps = []
    for run in range(2):
        out = tmp_path / f"run{run}"
        cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--n", "20000", "--partitions",
               "16", "--latent", "32", "--nq", "32", "--ref-queries", "16", "--steps", "2", "--warmup", "1", "--leaves",
               "8", "--dump-outputs", str(out)]
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr[-2000:]
        dumps.append({p.name: np.load(p) for p in sorted(out.iterdir())})
    assert sorted(dumps[0]) == ["counts.npy", "dists.npy", "ids.npy"]
    ids, dists, counts = dumps[0]["ids.npy"], dumps[0]["dists.npy"], dumps[0]["counts.npy"]
    assert ids.shape == dists.shape == (16, 10) and counts.shape == (16,)
    assert ids.dtype == counts.dtype == np.float64 and dists.dtype == np.float32
    assert (counts == 10).all() and (np.diff(dists, axis=1) >= 0).all()
    for name, v in dumps[0].items():
        assert np.array_equal(v, dumps[1][name]), name


def test_dump_outputs_samples_rows_above_the_size_cap(tmp_path, monkeypatch):
    sys.path.insert(0, ROOT)
    import bench

    nq, k = 1000, 10
    ids = np.arange(nq * k, dtype=np.int32).reshape(nq, k)
    ids[0, -1] = -1  # device padding reads as the host API's 0xFFFFFFFF
    dists = np.arange(nq * k, dtype=np.float32).reshape(nq, k)
    counts = np.full(nq, k, np.uint32)
    bench.dump_outputs(str(tmp_path / "all"), ids, dists, counts)
    got = np.load(tmp_path / "all" / "ids.npy")
    assert got.shape == (nq, k) and got[0, -1] == 0xFFFFFFFF and not (tmp_path / "all" / "rows.npy").exists()
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 64 << 10)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), ids, dists, counts)
    rows = np.load(tmp_path / "a" / "rows.npy")
    assert np.array_equal(rows, np.load(tmp_path / "b" / "rows.npy"))  # a fixed sample
    assert 0 < len(rows) < nq and (np.diff(rows) > 0).all()
    total = sum(os.path.getsize(p) for p in (tmp_path / "a").iterdir())
    assert total <= (64 << 10) + 4 * 128  # + the .npy headers
    r = rows.astype(np.int64)
    assert np.array_equal(np.load(tmp_path / "a" / "dists.npy"), dists[r])
    assert np.array_equal(np.load(tmp_path / "a" / "ids.npy"), ids.view(np.uint32)[r].astype(np.float64))


def test_ann_benchmark_recall_kat_and_flags():
    """src/bin/ann_benchmark.rs:481-492 (recall_at_k_basic) and the CLI spellings (:22-33,63-73)"""
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import ann_benchmark as ab

    r = ab.average_recall_at_k([[1, 2, 3], [5, 7, 9]], [[1, 4, 3], [5, 6, 7]], 3)
    assert abs(r - 2.0 / 3.0) < 1e-6
    assert ab.average_recall_at_k([], [[1]], 3) == 0.0 and ab.average_recall_at_k([[1]], [[1]], 0) == 0.0
    a = ab.parse(["--algorithm", "treeah", "--distance", "dot_product", "--k", "5", "--num-blocks", "16"])
    assert (a.algorithm, a.distance, a.k, a.num_blocks, a.num_partitions, a.partitions_to_search) == \
        ("tree_ah", "dot_product", 5, 16, 100, 10)
    d = ab.parse([])
    assert (d.algorithm, d.distance, d.synthetic_train, d.synthetic_test, d.dim, d.seed) == \
        ("brute_force", "squared_l2", 10_000, 200, 64, 42)
    train = np.array([[0.0, 0.0], [1.0, 0.0], [0.0, 2.0]], np.float32)
    gt = ab.exact_ground_truth(train, np.array([[0.9, 0.1]], np.float32), 2)
    assert gt[0].tolist() == [1, 0]
