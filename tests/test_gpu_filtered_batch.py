"""Per-query restrict filters in one Tree-AH batch (scann_treeah_search_filtered): every query of the batch is restricted
to its own filter row, nothing is stored on the handle, and the tensor-core scan serves filtered searches.  Results must
match the oracle's search_with_filter query by query, and be bit-identical to the register-LUT path and to a
handle-wide filter on the same queries."""
import ctypes as C
import os
import subprocess
import threading

import numpy as np
import pytest
import torch

import helpers
from test_gpu_parity import _check_stages

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture()
def env_restore():
    keys = ("SCANN_SCAN_TC", "SCANN_TC_RANKS")
    old = {k: os.environ.get(k) for k in keys}
    yield
    for k, v in old.items():
        if v is None:
            os.environ.pop(k, None)
        else:
            os.environ[k] = v


def _searcher(pkg, idx, x, L):
    cfg = pkg.TreeXHybridConfig(num_partitions=len(idx["centers"]), partitions_to_search=L)
    return pkg.TreeXHybridSearcher(cfg).build_from_index(idx["centers"], idx["codebook"], idx["packed"], idx["ids"],
                                                         idx["part_offsets"], x)


def _rows(out, sel):
    ids, dists, counts, (ci, cd, cc) = out
    return ids[sel], dists[sel], counts[sel], (ci[sel], cd[sel], cc[sel])


def _assert_identical(a, b):
    (i0, d0, c0, (ci0, cd0, cc0)), (i1, d1, c1, (ci1, cd1, cc1)) = a, b
    assert (c0 == c1).all() and (cc0 == cc1).all()
    assert (cd0.view(np.uint32) == cd1.view(np.uint32)).all() and (ci0 == ci1).all()
    assert (d0.view(np.uint32) == d1.view(np.uint32)).all() and (i0 == i1).all()


@pytest.fixture(scope="module")
def small(oracle):
    n, dim, K, S, nq = 60_000, 32, 40, 16, 300
    x, _ = helpers.clustered(n, dim, 48, 0.35, 17)
    qs, _ = helpers.clustered(nq, dim, 48, 0.35, 17)
    qs = (qs + 0.05 * helpers.gaussian(nq, dim, 18)).astype(np.float32)
    idx = helpers.build_index(oracle, x, K, S)
    rng = np.random.default_rng(23)
    keep = [0.5, 0.02, 0.999, 0.0, 1.0]
    allowed = np.stack([rng.random(n) < f for f in keep])
    fq = rng.integers(0, len(keep), nq).astype(np.uint32)
    return x, qs, idx, allowed, fq


def test_filtered_batch_matches_oracle_per_filter(gpu_lib, oracle, small):
    x, qs, idx, allowed, fq = small
    L, R, k = 8, 60, 10
    s = _searcher(gpu_lib, idx, x, L)
    ids, dists, counts, (ci, cd, cc) = s.search_with_filter(qs, k, allowed, filter_of_query=fq, pre_reorder_k=R,
                                                            want_candidates=True)
    for f in range(len(allowed)):
        sel = np.nonzero(fq == f)[0]
        assert len(sel) > 0
        bits = np.packbits(allowed[f], bitorder="little")
        rc, oids, odists, ocounts, ocand, ocd, ocn = oracle.treex_search(
            idx["centers"], idx["codebook"], idx["part_offsets"], idx["ids"], idx["packed"], x, qs[sel], L, R, k,
            lut16=True, nthreads=8, want_candidates=True, allow=bits)
        assert rc == 0
        _check_stages(oracle, x, oracle.SQL2, qs[sel], k, (ids[sel], dists[sel], counts[sel], ci[sel], cd[sel], cc[sel]),
                      (oids, odists, ocounts, ocand, ocd, ocn))
        valid = ids[sel] != 0xFFFFFFFF
        assert allowed[f][ids[sel][valid]].all(), f"filter {f}: a filtered-out datapoint was returned"
    assert (counts[fq == 3] == 0).all() and (cc[fq == 3] == 0).all()  # the 0 % filter
    assert (counts[fq != 3] == k).all()


def test_filtered_batch_groups_equal_handle_filter_alone(gpu_lib, small, env_restore):
    """Each filter group's rows of the shared batch are what set_filter(f) + search_batched of the group alone gives
    on the register-LUT path."""
    x, qs, idx, allowed, fq = small
    L, R, k = 8, 60, 10
    s = _searcher(gpu_lib, idx, x, L)
    batch = s.search_with_filter(qs, k, allowed, filter_of_query=fq, pre_reorder_k=R, want_candidates=True)
    os.environ["SCANN_SCAN_TC"] = "0"
    for f in range(len(allowed)):
        sel = np.nonzero(fq == f)[0]
        s.set_filter(allowed[f])
        try:
            alone = s.search_batched(qs[sel], k, pre_reorder_k=R, want_candidates=True)
        finally:
            s.set_filter(None)
        _assert_identical(_rows(batch, sel), alone)


@pytest.fixture(scope="module")
def big(oracle):
    x, _ = helpers.clustered(200_000, 96, 64, 0.35, 31)
    q, _ = helpers.clustered(3000, 96, 64, 0.35, 31)
    q = (q + 0.03 * helpers.gaussian(3000, 96, 32)).astype(np.float32)
    idx = helpers.build_index(oracle, x, 16, 48)
    rng = np.random.default_rng(77)
    allowed = np.stack([rng.random(len(x)) < f for f in (0.5, 0.02, 0.9, 0.3)])
    fq = rng.integers(0, len(allowed), len(q)).astype(np.uint32)
    return x, q, idx, allowed, fq


@pytest.mark.parametrize("ranks", [1, 2, 4])
def test_filtered_batch_tensor_core_path(gpu_lib, big, env_restore, ranks):
    x, q, idx, allowed, fq = big
    s = _searcher(gpu_lib, idx, x, 6)
    out = {}
    for mode in ("0", "1"):
        os.environ["SCANN_SCAN_TC"] = mode
        os.environ["SCANN_TC_RANKS"] = str(ranks)
        out[mode] = s.search_with_filter(q, 10, allowed, filter_of_query=fq, pre_reorder_k=100, want_candidates=True)
    assert s.path_stats() == (1, 1)
    _assert_identical(out["0"], out["1"])
    ids, _, counts, _ = out["1"]
    for f in range(len(allowed)):
        sel = fq == f
        valid = ids[sel] != 0xFFFFFFFF
        assert allowed[f][ids[sel][valid]].all()


@pytest.mark.parametrize("ranks", [1, 2, 4])
def test_handle_filter_tensor_core_path(gpu_lib, big, env_restore, ranks):
    """The handle-wide filter (set_filter) now takes the tensor-core path too, with the same results."""
    x, q, idx, allowed, _ = big
    s = _searcher(gpu_lib, idx, x, 6)
    s.set_filter(allowed[1])  # 2 %: queries without a bound are flagged back to the register-LUT kernel
    try:
        out = {}
        for mode in ("0", "1"):
            os.environ["SCANN_SCAN_TC"] = mode
            os.environ["SCANN_TC_RANKS"] = str(ranks)
            out[mode] = s.search_batched(q, 10, pre_reorder_k=100, want_candidates=True)
    finally:
        s.set_filter(None)
    assert s.path_stats() == (1, 1)
    _assert_identical(out["0"], out["1"])


def test_handle_filter_split_search_tensor_core_path(gpu_lib, big, env_restore):
    x, q, idx, allowed, _ = big
    s = _searcher(gpu_lib, idx, x, 6)
    qd = torch.tensor(q).cuda()
    s.set_filter(allowed[0])
    try:
        os.environ["SCANN_SCAN_TC"] = "0"
        ids, dists, counts = s.search_batched(qd, 10, pre_reorder_k=100)
        os.environ["SCANN_SCAN_TC"] = "1"
        tau = s.search_begin(qd, 10, pre_reorder_k=100)
        ids2, dists2, counts2 = s.search_end(tau)
        torch.cuda.synchronize()
    finally:
        s.set_filter(None)
    assert s.path_stats() == (1, 1)
    assert (ids.cpu() == ids2.cpu()).all() and (counts.cpu() == counts2.cpu()).all()
    assert (dists.cpu().numpy().view(np.uint32) == dists2.cpu().numpy().view(np.uint32)).all()
    valid = ids.cpu().numpy().view(np.uint32) != 0xFFFFFFFF
    assert allowed[0][ids.cpu().numpy().view(np.uint32)[valid]].all()


def test_filtered_batch_host_and_device_chunks(gpu_lib):
    """<= 1 GiB of candidates per chunk -> 128 queries at L = 512, R = 2048: 300 queries make three chunks, each of
    which reads its slice of filter_of_query."""
    x, _ = helpers.clustered(60_000, 32, 64, 0.35, 9)
    q = (x[:300] + 0.01).astype(np.float32)
    cfg = gpu_lib.TreeXHybridConfig(num_partitions=600, partitions_to_search=512)
    cfg.hash_config.num_subspaces = 16
    s = gpu_lib.TreeXHybridSearcher(cfg).build(x, train_rows=0, kmeans_iters=4, seed=3)
    rng = np.random.default_rng(4)
    allowed = np.stack([rng.random(len(x)) < f for f in (0.5, 0.1, 0.9)])
    fq = rng.integers(0, 3, len(q)).astype(np.uint32)
    host = s.search_with_filter(q, 10, allowed, filter_of_query=fq, pre_reorder_k=2048, want_candidates=True)
    dev = s.search_with_filter(torch.tensor(q).cuda(), 10, torch.tensor(allowed).cuda(),
                               filter_of_query=torch.tensor(fq.astype(np.int32)).cuda(), pre_reorder_k=2048,
                               want_candidates=True)
    torch.cuda.synchronize()
    ids, dists, counts, (ci, cd, cc) = dev
    dev = (ids.cpu().numpy().view(np.uint32), dists.cpu().numpy(), counts.cpu().numpy().view(np.uint32),
           (ci.cpu().numpy().view(np.uint32), cd.cpu().numpy(), cc.cpu().numpy().view(np.uint32)))
    _assert_identical(host, dev)
    assert (host[2] == 10).all()
    for f in range(3):
        sel = fq == f
        assert allowed[f][host[0][sel]].all()


def test_filtered_errors_leave_handle_usable(gpu_lib, small):
    x, qs, idx, allowed, fq = small
    capi = gpu_lib.capi
    lib = capi.load()
    s = _searcher(gpu_lib, idx, x, 8)
    q = qs[:40]
    f = fq[:40]
    ref = s.search_with_filter(q, 10, allowed, filter_of_query=f, pre_reorder_k=60)

    def call(bits, F, fqa, qa=q):
        ids = np.empty((len(qa), 10), np.uint32)
        dists = np.empty((len(qa), 10), np.float32)
        counts = np.empty(len(qa), np.uint32)
        return lib.scann_treeah_search_filtered(s._h, capi.np_ptr(qa), len(qa), qa.shape[1], 8, 60, 10, bits, F,
                                                allowed.shape[1], fqa, capi.np_ptr(ids), capi.np_ptr(dists),
                                                capi.np_ptr(counts), None, None, None, capi.HOST, None)

    packed = np.ascontiguousarray(np.packbits(allowed, axis=1, bitorder="little"))
    fqa = np.ascontiguousarray(f)
    assert call(capi.np_ptr(packed), len(allowed), capi.np_ptr(fqa)) == capi.OK
    assert call(capi.np_ptr(packed), 0, capi.np_ptr(fqa)) == capi.INVALID_ARGUMENT
    assert call(None, len(allowed), capi.np_ptr(fqa)) == capi.INVALID_ARGUMENT
    assert call(capi.np_ptr(packed), len(allowed), None) == capi.INVALID_ARGUMENT
    bad = fqa.copy()
    bad[7] = len(allowed)
    assert call(capi.np_ptr(packed), len(allowed), capi.np_ptr(bad)) == capi.INVALID_ARGUMENT
    s.set_filter(allowed[0])
    assert call(capi.np_ptr(packed), len(allowed), capi.np_ptr(fqa)) == capi.FAILED_PRECONDITION
    s.set_filter(None)
    qd = torch.tensor(q).cuda()
    s.search_begin(qd, 10, pre_reorder_k=60)
    assert call(capi.np_ptr(packed), len(allowed), capi.np_ptr(fqa)) == capi.FAILED_PRECONDITION
    s.search_abort()
    # the device path does not check rows: an out-of-range row allows nothing, the other queries are unaffected
    bad_d = torch.tensor(bad.astype(np.int64)).cuda()
    ids, dists, counts = s.search_with_filter(qd, 10, torch.tensor(allowed).cuda(), filter_of_query=bad_d,
                                              pre_reorder_k=60)
    torch.cuda.synchronize()
    counts = counts.cpu().numpy()
    assert counts[7] == 0
    keep = np.arange(len(q)) != 7
    assert (counts[keep] == ref[2][keep]).all()
    assert (ids.cpu().numpy().view(np.uint32)[keep] == ref[0][keep]).all()
    with pytest.raises(gpu_lib.ScannError):
        s.search_with_filter(q, 10, allowed)  # 5 filters for 40 queries and no filter_of_query
    again = s.search_with_filter(q, 10, allowed, filter_of_query=f, pre_reorder_k=60)
    for a, b in zip(ref, again):
        assert (a.view(np.uint32) == b.view(np.uint32)).all()


def test_filtered_search_from_two_threads(gpu_lib, small):
    x, qs, idx, allowed, _ = small
    s = _searcher(gpu_lib, idx, x, 8)
    q = qs[:64]
    want = [s.search_with_filter(q, 10, allowed[t], pre_reorder_k=60) for t in (0, 1)]
    errors = []

    def run(t):
        try:
            for _ in range(20):
                got = s.search_with_filter(q, 10, allowed[t], pre_reorder_k=60)
                for a, b in zip(want[t], got):
                    if not (a.view(np.uint32) == b.view(np.uint32)).all():
                        errors.append(f"thread {t}: result differs from its single-threaded result")
                        return
        except Exception as e:  # noqa: BLE001 - reported below
            errors.append(repr(e))

    threads = [threading.Thread(target=run, args=(t,)) for t in (0, 1)]
    for th in threads:
        th.start()
    for th in threads:
        th.join()
    assert not errors, errors


def test_cpp_mirror_filtered_batch(gpu_lib):
    libdir = os.path.dirname(gpu_lib.build_lib.build())
    src = os.path.join(ROOT, "tests", "cpp", "test_hpp_filtered.cpp")
    exe = os.path.join(ROOT, "tests", "cpp", "test_hpp_filtered.bin")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-Wall", "-I", os.path.join(ROOT, "include"), src, "-o", exe,
                           "-L", libdir, "-lscann_b200", f"-Wl,-rpath,{libdir}"])
    out = subprocess.run([exe], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0, out.stdout + out.stderr
    assert "hpp filtered ok" in out.stdout
