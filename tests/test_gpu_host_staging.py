"""Host-staged (numpy, SCANN_HOST) and device-resident (CUDA tensors, SCANN_DEVICE) calls of every query-batched entry
point give identical results on batches that span several query chunks: the host path copies each chunk's queries in
and its outputs back, the device path writes the caller's arrays in place.  Sizes are chosen from each entry point's
chunk rule (noted per test) so that the batch is cut into at least three chunks."""
import ctypes as C

import numpy as np
import pytest

import helpers

pytestmark = pytest.mark.gpu


def _host(a):
    """numpy copy of a result; integer and float arrays as their raw 32-bit patterns"""
    if type(a).__module__.startswith("torch"):
        a = a.cpu().numpy()
    return np.ascontiguousarray(a).view(np.uint32)


def _same(host_out, dev_out):
    if isinstance(host_out, tuple):
        assert len(host_out) == len(dev_out)
        for h, d in zip(host_out, dev_out):
            _same(h, d)
    else:
        assert np.array_equal(_host(host_out), _host(dev_out))


def _both(search, q, pick=lambda r: r):
    """search(q) with numpy and with CUDA-tensor queries; pick(result) of the two must be identical"""
    import torch
    dev = pick(search(torch.as_tensor(q).cuda()))
    torch.cuda.synchronize()
    host = pick(search(q))
    _same(host, dev)
    return host


# brute force, tensor-core path: 4096 queries per chunk
@pytest.mark.parametrize("measure", ["SquaredL2", "DotProduct"])
def test_bf_tensor_core_chunks(gpu_lib, oracle, measure):
    db = helpers.gaussian(20_000, 64, 42)
    q = helpers.gaussian(9000, 64, 123)
    om = {"SquaredL2": oracle.SQL2, "DotProduct": oracle.DOT}[measure]
    bf = gpu_lib.BruteForceSearcher(db, gpu_lib.DistanceMeasure[measure])
    ids, dists, counts = _both(lambda x: bf.search_batched(x, 10), q)
    assert bf.path_stats() == (6, 0)  # 3 chunks per call
    rc, oids, odists, ocounts = oracle.bf_search(db, q, 10, om, nthreads=8)
    assert (counts == ocounts).all()
    compared, mism = helpers.ids_equal_away_from_ties(ids, dists, oids, odists, counts)
    assert mism == 0 and compared > 0
    same = ids == oids
    assert same.mean() > 0.999 and (dists[same].view(np.uint32) == odists[same].view(np.uint32)).all()


# brute force, CUDA-core path: 1024 queries per chunk
def test_bf_cuda_core_chunks(gpu_lib, oracle, monkeypatch):
    monkeypatch.setenv("SCANN_BF_NO_TC", "1")
    db = helpers.gaussian(20_000, 128, 42)
    q = helpers.gaussian(3000, 128, 123)
    bf = gpu_lib.BruteForceSearcher(db)
    ids, dists, counts = _both(lambda x: bf.search_batched(x, 10), q)
    assert bf.path_stats() == (0, 6)
    rc, oids, odists, ocounts = oracle.bf_search(db, q, 10, oracle.SQL2, nthreads=8)
    assert (counts == ocounts).all() and (ids == oids).mean() > 0.999


# scalar-quantised brute force, tensor-core path: 4096 queries per chunk
def test_sq8_chunks(gpu_lib, oracle):
    db = helpers.gaussian(20_000, 64, 42)
    q = helpers.gaussian(9000, 64, 123)
    ocodes, ocal = oracle.sq8_quantize(db)
    s = gpu_lib.ScalarQuantizedBruteForceSearcher.from_quantized(ocodes, float(ocal[2]))
    ids, dists, counts = _both(lambda x: s.search_batched(x, 10), q)
    assert s.path_stats() == (6, 0)
    rc, oids, odists, ocounts = oracle.sq8_search(ocodes, float(ocal[2]), q, 10, oracle.SQL2, nthreads=8)
    assert (counts == ocounts).all()
    compared, mism = helpers.ids_equal_away_from_ties(ids, dists, oids, odists, counts)
    assert mism == 0
    same = ids == oids
    assert same.mean() > 0.995 and (dists[same].view(np.uint32) == odists[same].view(np.uint32)).all()


# radius search: 4096 queries per chunk
def test_bf_search_radius_chunks(gpu_lib, oracle):
    db = helpers.gaussian(30_000, 96, 42)
    q = helpers.gaussian(9000, 96, 123)
    radius = 110.0
    bf = gpu_lib.BruteForceSearcher(db)
    ids, dists, counts = _both(lambda x: bf.search_radius_batched(x, radius, max_results=1024), q)
    assert counts.sum() > 1000 and counts.max() > 1
    for i in range(0, len(q), 97):  # a sample of queries from every chunk
        oi, od = oracle.bf_search_radius(db, q[i], radius, oracle.SQL2)
        assert counts[i] == len(oi)
        assert (dists[i, :len(oi)].view(np.uint32) == od.view(np.uint32)).all()
        assert (ids[i, :len(oi)] == oi).all() or len(set(od.tolist())) < len(od)
    # a truncation in any chunk is reported after every chunk has been written, on both paths
    import torch
    for x in (q, torch.as_tensor(q).cuda()):
        with pytest.warns(UserWarning):
            t = bf.search_radius_batched(x, radius, max_results=1, allow_truncated=True)
        torch.cuda.synchronize()
        assert (_host(t[2]) == np.minimum(counts, 1)).all()


# partitioner: 2 GiB of centre scores per chunk -> 8192 queries at K = 65,536
def test_partitioner_chunks(gpu_lib, oracle):
    centers = helpers.gaussian(65_536, 16, 5)
    q = helpers.gaussian(20_000, 16, 6)
    part = gpu_lib.TreePartitioner(centers)
    tokens, dists = _both(lambda x: part.partition(x, 8), q)
    sel = np.r_[0:50, 8190:8200, 16380:16390, 19950:20000]
    otok, odist = oracle.partition(centers, q[sel], 8, nthreads=8)
    assert (tokens[sel] == otok).all() and (dists[sel].view(np.uint32) == odist.view(np.uint32)).all()


# leaf-scan facade: 256 MiB of centre scores per chunk -> 1024 queries at K = 65,536 (most leaves empty)
def test_leafscan_chunks(gpu_lib, oracle):
    x = helpers.gaussian(20_000, 16, 7)
    centers = helpers.gaussian(65_536, 16, 8)
    assign = gpu_lib.TreePartitioner(centers).partition(x, 1)[0][:, 0]
    order = np.argsort(assign, kind="stable").astype(np.uint32)
    off = np.concatenate([[0], np.cumsum(np.bincount(assign, minlength=len(centers)))]).astype(np.uint64)
    q = (x[:2500] + 0.05).astype(np.float32)
    s = gpu_lib.LeafScanSearcher(centers, order, off, x)
    ids, dists, counts = _both(lambda t: s.search_partitioned(t, 10, 4), q)
    rc, oids, odists, ocounts = oracle.scann_partitioned(centers, off, order, x, q, 4, 10, oracle.SQL2, nthreads=8)
    assert rc == 0 and (counts == ocounts).all()
    assert (ids == oids).all() and (dists.view(np.uint32) == odists.view(np.uint32)).all()


# Tree-AH: <= 1 GiB of candidates per chunk -> 128 queries at L = 512, R = 2048
def test_treeah_chunks(gpu_lib):
    x, _ = helpers.clustered(60_000, 32, 64, 0.35, 9)
    q = (x[:300] + 0.01).astype(np.float32)
    cfg = gpu_lib.TreeXHybridConfig(num_partitions=600, partitions_to_search=512)
    cfg.hash_config.num_subspaces = 16
    s = gpu_lib.TreeXHybridSearcher(cfg).build(x, train_rows=0, kmeans_iters=4, seed=3)
    ids, dists, counts, (ci, cd, cc) = _both(
        lambda t: s.search_batched(t, 10, pre_reorder_k=2048, want_candidates=True), q)
    assert (counts == 10).all() and (cc > 0).all()
    # without candidate outputs: the same results
    _same(_both(lambda t: s.search_batched(t, 10, pre_reorder_k=2048), q), (ids, dists, counts))
    # pre_reorder_k = 0 keeps nothing: empty results
    ids0, _, counts0, cc0 = _both(lambda t: s.search_batched(t, 10, pre_reorder_k=0, want_candidates=True), q,
                                  lambda r: (*r[:3], r[3][2]))  # no candidate lists are written
    assert (counts0 == 0).all() and (cc0 == 0).all() and (ids0 == 0xFFFFFFFF).all()


def _wide_deep_tree(dim, seed):
    """root with 1024 children (1023 leaves + the head of a 31-node chain): 32 levels x 1024 children per query of
    scratch = 256 KiB, so 1024 queries per chunk"""
    rng = np.random.default_rng(seed)
    n_chain, n_leaves = 31, 1023
    nn = 1 + n_chain + n_leaves
    centers = rng.standard_normal((nn, dim)).astype(np.float32)
    depth = np.concatenate([[0], np.arange(1, n_chain + 1), np.ones(n_leaves)]).astype(np.uint32)
    root_children = [1] + list(range(1 + n_chain, nn))
    chain_children = list(range(2, n_chain + 1))
    children = np.array(root_children + chain_children, np.uint32)
    child_count = np.zeros(nn, np.uint32)
    child_begin = np.zeros(nn, np.uint32)
    child_count[0] = len(root_children)
    for i in range(1, n_chain):
        child_begin[i] = len(root_children) + i - 1
        child_count[i] = 1
    return centers, depth, child_begin, child_count, children


def test_kmtree_search_leaves_chunks(gpu_lib, oracle):
    import torch
    t = _wide_deep_tree(8, 3)
    q = np.random.default_rng(4).standard_normal((3500, 8)).astype(np.float32)
    tree = gpu_lib.KMeansTree().build_from_arrays(*t)
    nodes, dists, depths, counts = _both(lambda x: tree.search_leaves(x, 6), q)
    on, od, odp, oc = oracle.kmtree_search_leaves(*t, q, 6)
    assert (counts == oc).all() and (nodes == on).all() and (depths == odp).all()
    assert (dists.view(np.uint32) == od.view(np.uint32)).all()
    # SCANN_HOST on an explicit stream, optional outputs not requested
    lib, capi = gpu_lib.capi.load(), gpu_lib.capi
    st = torch.cuda.Stream()
    n2 = np.empty_like(on)
    c2 = np.empty_like(oc)
    capi.check(lib.scann_kmtree_search_leaves(tree._h, capi.np_ptr(q), len(q), 8, 6, capi.np_ptr(n2), None, None,
                                              capi.np_ptr(c2), capi.HOST, C.c_void_p(st.cuda_stream)))
    assert (n2 == on).all() and (c2 == oc).all()
