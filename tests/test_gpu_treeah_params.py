"""Per-query parameters in one Tree-AH batch (scann_treeah_search_with_params): query q searches L_q partitions, keeps
R_q candidates before the reorder and returns k_q neighbours.  Row q must be bit for bit what scann_treeah_search of
query q alone with (L_q, R_q, k_q) returns, padded up to the batch maxima, on both scan paths."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
import torch

import helpers
from test_gpu_parity import _check_stages

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# (L_q, R_q, k_q) of the mixed batch: L_q = 1 is below the tensor-core class-A ranks, R_q = 512 is above the size of
# most leaves, k_q > R_q returns fewer than k_q neighbours, R_q = 0 returns nothing
GROUPS = [(1, 1, 1), (3, 7, 10), (16, 100, 10), (16, 512, 1), (3, 0, 10), (1, 512, 520), (16, 7, 1), (3, 100, 120),
          (16, 512, 10)]
L_MAX = 16


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


@pytest.fixture(scope="module")
def mixed(oracle):
    """60k points in 200 leaves (about 300 points each), 2000 queries: 160 queries per probed leaf at L = 16, so the
    default path choice takes the tensor-core scan."""
    n, dim, K, S, nq = 60_000, 32, 200, 16, 2000
    x, _ = helpers.clustered(n, dim, 48, 0.35, 41)
    qs, _ = helpers.clustered(nq, dim, 48, 0.35, 41)
    qs = (qs + 0.05 * helpers.gaussian(nq, dim, 42)).astype(np.float32)
    idx = helpers.build_index(oracle, x, K, S)
    group = np.random.default_rng(43).integers(0, len(GROUPS), nq)
    prm = np.array([GROUPS[g] for g in group], np.uint32)
    return x, qs, idx, group, prm


def _searcher(pkg, idx, x, L=L_MAX):
    cfg = pkg.TreeXHybridConfig(num_partitions=len(idx["centers"]), partitions_to_search=L)
    return pkg.TreeXHybridSearcher(cfg).build_from_index(idx["centers"], idx["codebook"], idx["packed"], idx["ids"],
                                                         idx["part_offsets"], x)


def _per_query(s, q, prm):
    return s.search_batched_per_query(q, prm[:, 2], prm[:, 1], prm[:, 0], want_candidates=True)


def _np(out):
    ids, dists, counts, (ci, cd, cc) = out
    f = (lambda t: t.cpu().numpy()) if torch.is_tensor(ids) else (lambda t: t)
    u = lambda t: f(t).view(np.uint32)  # noqa: E731
    return u(ids), f(dists), u(counts), (u(ci), f(cd), u(cc))


def _assert_identical(a, b):
    (i0, d0, c0, (ci0, cd0, cc0)), (i1, d1, c1, (ci1, cd1, cc1)) = _np(a), _np(b)
    assert (c0 == c1).all() and (cc0 == cc1).all()
    assert (cd0.view(np.uint32) == cd1.view(np.uint32)).all() and (ci0 == ci1).all()
    assert (d0.view(np.uint32) == d1.view(np.uint32)).all() and (i0 == i1).all()


def _group_rows(out, sel, R, k):
    """rows `sel` of a mixed result cut to (R, k) of their group; the cut-off part must be padding (R == 0 pads the
    distances with 0x7F7F7F7F, as a search with R == 0 does)"""
    ids, dists, counts, (ci, cd, cc) = _np(out)
    pad = np.float32(np.uint32(0x7F7F7F7F).view(np.float32)) if R == 0 else np.float32(np.inf)
    assert (ids[sel, k:] == 0xFFFFFFFF).all() and (dists[sel, k:] == pad).all()
    assert (ci[sel, R:] == 0xFFFFFFFF).all() and np.isinf(cd[sel, R:]).all()
    Rc = max(R, 1)
    return ids[sel, :k], dists[sel, :k], counts[sel], (ci[sel, :Rc], cd[sel, :Rc], cc[sel])


def test_mixed_batch_matches_oracle_per_group(gpu_lib, oracle, mixed):
    x, qs, idx, group, prm = mixed
    qs, group, prm = qs[:600], group[:600], prm[:600]
    s = _searcher(gpu_lib, idx, x)
    out = _per_query(s, qs, prm)
    for g, (L, R, k) in enumerate(GROUPS):
        sel = np.nonzero(group == g)[0]
        assert len(sel) > 0
        ids, dists, counts, (ci, cd, cc) = _group_rows(out, sel, R, k)
        if R == 0:
            assert (counts == 0).all() and (cc == 0).all()
            continue
        rc, oids, odists, ocounts, ocand, ocd, ocn = oracle.treex_search(
            idx["centers"], idx["codebook"], idx["part_offsets"], idx["ids"], idx["packed"], x, qs[sel], L, R, k,
            lut16=True, nthreads=8, want_candidates=True)
        assert rc == 0
        _check_stages(oracle, x, oracle.SQL2, qs[sel], k, (ids, dists, counts, ci, cd, cc),
                      (oids, odists, ocounts, ocand, ocd, ocn))


@pytest.mark.parametrize("mode,ranks", [("0", 2), ("1", 1), ("1", 2), ("1", 4)])
def test_groups_equal_separate_calls(gpu_lib, mixed, env_restore, mode, ranks):
    """Each group's rows of the mixed batch are what a search of the group alone returns (on the register-LUT path),
    candidate taps included, whichever path the mixed batch takes."""
    x, qs, idx, group, prm = mixed
    s = _searcher(gpu_lib, idx, x)
    os.environ["SCANN_SCAN_TC"] = mode
    os.environ["SCANN_TC_RANKS"] = str(ranks)
    out = _per_query(s, qs, prm)
    assert s.path_stats() == ((1, 0) if mode == "1" else (0, 1))
    os.environ["SCANN_SCAN_TC"] = "0"
    for g, (L, R, k) in enumerate(GROUPS):
        sel = np.nonzero(group == g)[0]
        alone = s.search_batched(qs[sel], k, partitions_to_search=L, pre_reorder_k=R, want_candidates=True)
        _assert_identical(_group_rows(out, sel, R, k), alone)


def test_default_path_choice_takes_tensor_cores(gpu_lib, mixed, env_restore):
    x, qs, idx, group, prm = mixed
    s = _searcher(gpu_lib, idx, x)
    os.environ.pop("SCANN_SCAN_TC", None)
    mixed_out = _per_query(s, qs, prm)
    assert s.path_stats() == (1, 0)
    os.environ["SCANN_SCAN_TC"] = "0"
    _assert_identical(mixed_out, _per_query(s, qs, prm))


@pytest.mark.parametrize("handle_filter", [False, True])
def test_uniform_and_null_arrays_equal_plain_search(gpu_lib, mixed, handle_filter):
    x, qs, idx, _, _ = mixed
    s = _searcher(gpu_lib, idx, x)
    nq, L, R, k = len(qs), 12, 100, 10
    if handle_filter:
        s.set_filter(np.random.default_rng(5).random(len(x)) < 0.3)
    try:
        plain = s.search_batched(qs, k, partitions_to_search=L, pre_reorder_k=R, want_candidates=True)
        plain_bytes = s.last_scan_bytes()
        full = s.search_batched_per_query(qs, np.full(nq, k), np.full(nq, R), np.full(nq, L), want_candidates=True)
        assert s.last_scan_bytes() == plain_bytes
        null = s.search_batched_per_query(qs, k, R, L, want_candidates=True)  # NULL arrays
        assert s.last_scan_bytes() == plain_bytes
        dev = s.search_batched_per_query(torch.tensor(qs).cuda(), torch.full((nq,), k).cuda(),
                                         torch.full((nq,), R).cuda(), torch.full((nq,), L).cuda(), want_candidates=True)
        torch.cuda.synchronize()
    finally:
        s.set_filter(None)
    for other in (full, null, dev):
        _assert_identical(plain, other)


def test_masked_ranks_are_not_scanned(gpu_lib, mixed):
    """last_scan_bytes of the mixed call (Σ over (query, leaf) pairs of leaf_size * ceil(S/2)) is the sum over the
    groups' own calls: the ranks beyond L_q and the queries with R_q = 0 are not scanned."""
    x, qs, idx, group, prm = mixed
    s = _searcher(gpu_lib, idx, x)
    _per_query(s, qs, prm)
    mixed_bytes, mixed_pairs = s.last_scan_bytes()
    tot_bytes = tot_pairs = 0
    for g, (L, R, k) in enumerate(GROUPS):
        s.search_batched(qs[group == g], k, partitions_to_search=L, pre_reorder_k=R)
        b, p = s.last_scan_bytes()
        tot_bytes += b
        tot_pairs += p
    assert (mixed_bytes, mixed_pairs) == (tot_bytes, tot_pairs)
    assert 0 < mixed_pairs < len(qs) * L_MAX


def test_host_and_device_chunks(gpu_lib):
    """<= 1 GiB of candidates per chunk -> 128 queries at L = 512, R = 2048: 300 queries make three chunks, each of
    which reads its slice of the per-query arrays."""
    x, _ = helpers.clustered(60_000, 32, 64, 0.35, 9)
    q = (x[:300] + 0.01).astype(np.float32)
    cfg = gpu_lib.TreeXHybridConfig(num_partitions=600, partitions_to_search=512)
    cfg.hash_config.num_subspaces = 16
    s = gpu_lib.TreeXHybridSearcher(cfg).build(x, train_rows=0, kmeans_iters=4, seed=3)
    rng = np.random.default_rng(4)
    Lq = rng.choice([1, 40, 512], len(q)).astype(np.int64)
    Rq = rng.choice([0, 10, 300, 2048], len(q)).astype(np.int64)
    kq = rng.choice([1, 10, 64], len(q)).astype(np.int64)
    Lq[0], Rq[0] = 512, 2048  # the maxima set the chunk size
    host = s.search_batched_per_query(q, kq, Rq, Lq, want_candidates=True)
    dev = s.search_batched_per_query(torch.tensor(q).cuda(), torch.tensor(kq).cuda(), torch.tensor(Rq).cuda(),
                                     torch.tensor(Lq).cuda(), want_candidates=True)
    torch.cuda.synchronize()
    _assert_identical(host, dev)
    assert (host[2][Rq == 0] == 0).all() and (host[2][Rq > 0] > 0).all()
    for i in (0, 150, 299):  # one query of every chunk against its own call
        alone = s.search_batched(q[i:i + 1], int(kq[i]), partitions_to_search=int(Lq[i]), pre_reorder_k=int(Rq[i]),
                                 want_candidates=True)
        row = _group_rows(host, np.array([i]), int(Rq[i]), int(kq[i]))
        _assert_identical(row, alone)


def test_errors_and_bad_values(gpu_lib, mixed):
    x, qs, idx, _, _ = mixed
    capi = gpu_lib.capi
    lib = capi.load()
    s = _searcher(gpu_lib, idx, x)
    q = np.ascontiguousarray(qs[:40])
    nq, L, R, k = len(q), 8, 60, 10
    rng = np.random.default_rng(8)
    good = [rng.integers(1, L + 1, nq).astype(np.uint32), rng.integers(0, R + 1, nq).astype(np.uint32),
            rng.integers(1, k + 1, nq).astype(np.uint32)]
    ref = s.search_batched_per_query(q, good[2], good[1], good[0])

    def call(arrs):
        ids = np.empty((nq, k), np.uint32)
        dists = np.empty((nq, k), np.float32)
        counts = np.empty(nq, np.uint32)
        return lib.scann_treeah_search_with_params(s._h, capi.np_ptr(q), nq, q.shape[1], L, R, k,
                                                   *[capi.np_ptr(a) for a in arrs], capi.np_ptr(ids),
                                                   capi.np_ptr(dists), capi.np_ptr(counts), None, None, None,
                                                   capi.HOST, None)

    assert call(good) == capi.OK
    for which, value in ((0, 0), (0, L + 1), (1, R + 1), (2, 0), (2, k + 1)):
        bad = [a.copy() for a in good]
        bad[which][7] = value
        assert call(bad) == capi.INVALID_ARGUMENT, (which, value)
        again = s.search_batched_per_query(q, good[2], good[1], good[0])
        for a, b in zip(ref, again):
            assert (a.view(np.uint32) == b.view(np.uint32)).all()
    # the device path does not check: a query with a value out of range returns nothing, the others are unaffected
    qd = torch.tensor(q).cuda()
    for which, value in ((0, 0), (0, L + 1), (1, R + 1), (2, 0), (2, k + 1)):
        arrs = [torch.tensor(a.astype(np.int32)).cuda() for a in good]
        arrs[which][7] = value
        ids = torch.empty((nq, k), dtype=torch.int32, device="cuda")
        dists = torch.empty((nq, k), dtype=torch.float32, device="cuda")
        counts = torch.empty((nq,), dtype=torch.int32, device="cuda")
        cids = torch.empty((nq, R), dtype=torch.int32, device="cuda")
        cd = torch.empty((nq, R), dtype=torch.float32, device="cuda")
        cc = torch.empty((nq,), dtype=torch.int32, device="cuda")
        p = lambda t: C.c_void_p(t.data_ptr())  # noqa: E731
        assert lib.scann_treeah_search_with_params(s._h, p(qd), nq, q.shape[1], L, R, k, *[p(a) for a in arrs],
                                                   p(ids), p(dists), p(counts), p(cids), p(cd), p(cc), capi.DEVICE,
                                                   None) == capi.OK
        torch.cuda.synchronize()
        ids, dists, counts = ids.cpu().numpy().view(np.uint32), dists.cpu().numpy(), counts.cpu().numpy()
        assert counts[7] == 0 and cc[7].item() == 0 and (ids[7] == 0xFFFFFFFF).all()
        keep = np.arange(nq) != 7
        assert (counts[keep] == ref[2][keep]).all() and (ids[keep] == ref[0][keep]).all()
        assert (dists[keep].view(np.uint32) == ref[1][keep].view(np.uint32)).all()
    s.search_begin(qd, 10, pre_reorder_k=60)
    assert call(good) == capi.FAILED_PRECONDITION
    s.search_abort()
    assert call(good) == capi.OK


def test_search_batched_with_params_is_one_call(gpu_lib, mixed, monkeypatch):
    """TreeXHybridSearcher.search_batched_with_params sends the whole batch in one C call and returns what the grouped
    path (one call per distinct parameter set) returns."""
    x, qs, idx, _, _ = mixed
    s = _searcher(gpu_lib, idx, x, L=8)
    q = qs[:300]
    rng = np.random.default_rng(12)
    SP = gpu_lib.SearchParameters
    params = [SP(num_neighbors=[None, 1, 5, 30][int(rng.integers(0, 4))],
                 pre_reordering_num_neighbors=[None, 7, 64][int(rng.integers(0, 3))]) for _ in range(len(q))]
    grouped = gpu_lib.searchers._Handle.search_batched_with_params(s, q, params)
    lib = gpu_lib.capi.load()
    calls = {"params": 0, "plain": 0}
    orig_p, orig_s = lib.scann_treeah_search_with_params, lib.scann_treeah_search

    def count(name, fn):
        def wrapped(*args):
            calls[name] += 1
            return fn(*args)
        return wrapped

    monkeypatch.setattr(lib, "scann_treeah_search_with_params", count("params", orig_p))
    monkeypatch.setattr(lib, "scann_treeah_search", count("plain", orig_s))
    one = s.search_batched_with_params(q, params)
    assert calls == {"params": 1, "plain": 0}
    assert one == grouped
    assert s.search_batched_with_params(q[:0], []) == []
    with pytest.raises(gpu_lib.ScannError):
        s.search_batched_with_params(q, params[:-1])


def test_cpp_mirror_params_batch(gpu_lib, tmp_path):
    libdir = os.path.dirname(gpu_lib.build_lib.build())
    src = os.path.join(ROOT, "tests", "cpp", "test_hpp_params.cpp")
    exe = str(tmp_path / "test_hpp_params.bin")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-Wall", "-I", os.path.join(ROOT, "include"), src, "-o", exe,
                           "-L", libdir, "-lscann_b200", f"-Wl,-rpath,{libdir}"])
    out = subprocess.run([exe], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0, out.stdout + out.stderr
    assert "hpp params ok" in out.stdout
