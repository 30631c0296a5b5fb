"""Tree-AH search across the index geometries scann_treeah_create accepts (1 <= S <= 256, any ds = dim / S, with or
without residuals, R <= 2048), held to the stage-wise, tie-proof oracle checks of test_gpu_parity._check_stages.

  * the tensor-core scan for ds = 1, 2 (tc_lut_kernel<1>, <2>) and ds >= 3 (<0>), up to the tc_scan_supported limit;
  * the register-LUT scan for odd S, S % 4 != 0 (padded subspace groups, half-byte row tails) and S > 64 (uncached
    LUT build, up to 64 subspace groups, both sides of the IDP.2A limit S = 128), in dense and tiny batches;
  * the largest LUT16 sum (255 * S) under the accumulation mode of S, on both sides of the IDP.2A limit;
  * the in-leaf position bits at their limit (16 bits at S = 256) and beyond 2^17 points on the tensor-core path;
  * batches dense enough for 8 queries per work item where 8 queries' shared memory does not fit.

Every case asserts which scan answered (path_stats), so a fallback cannot pass for coverage."""
import os

import numpy as np
import pytest

import helpers
from test_gpu_parity import _check_stages

_ENV = ("SCANN_SCAN_TC", "SCANN_TC_RANKS")


@pytest.fixture()
def env_restore():
    old = {k: os.environ.get(k) for k in _ENV}
    yield
    for k, v in old.items():
        if v is None:
            os.environ.pop(k, None)
        else:
            os.environ[k] = v


def _searcher(pkg, idx, x, L, use_residuals=True, measure=None):
    kw = {} if measure is None else {"distance_measure": measure}
    cfg = pkg.TreeXHybridConfig(num_partitions=len(idx["centers"]), partitions_to_search=L,
                                use_residuals=use_residuals, **kw)
    return pkg.TreeXHybridSearcher(cfg).build_from_index(idx["centers"], idx["codebook"], idx["packed"], idx["ids"],
                                                         idx["part_offsets"], x)


def _search(s, q, k, R, L=None):
    ids, dists, counts, (ci, cd, cc) = s.search_batched(q, k, partitions_to_search=L, pre_reorder_k=R,
                                                        want_candidates=True)
    return ids, dists, counts, ci, cd, cc


def _oracle(oracle, idx, x, q, L, R, k, use_residuals=True, measure=None):
    om = oracle.SQL2 if measure is None else measure
    rc, *ora = oracle.treex_search(idx["centers"], idx["codebook"], idx["part_offsets"], idx["ids"], idx["packed"], x, q,
                                   L, R, k, lut16=True, use_residuals=use_residuals, reorder_measure=om, nthreads=8,
                                   want_candidates=True)
    assert rc == 0
    return tuple(ora)


def _assert_identical(a, b):
    (i0, d0, c0, ci0, cd0, cc0), (i1, d1, c1, ci1, cd1, cc1) = a, b
    assert (c0 == c1).all() and (cc0 == cc1).all()
    assert (cd0.view(np.uint32) == cd1.view(np.uint32)).all() and (ci0 == ci1).all()
    assert (d0.view(np.uint32) == d1.view(np.uint32)).all() and (i0 == i1).all()


def _clustered(oracle, n, dim, K, S, nq, seed, use_residuals=True):
    x, _ = helpers.clustered(n, dim, max(8, K), 0.35, seed)
    q, _ = helpers.clustered(nq, dim, max(8, K), 0.35, seed)
    q = (q + 0.05 * helpers.gaussian(nq, dim, seed + 1)).astype(np.float32)
    return x, q, helpers.build_index(oracle, x, K, S, use_residuals=use_residuals)


def _tc_supported(dim, S):
    # tc_scan_supported (csrc/tcscan.cu): tc_lut_kernel takes dim*32 + S*128 bytes of dynamic shared memory and sets no
    # attribute, so 48 KB is its limit
    return S % 16 == 0 and 16 <= S <= 64 and dim % S == 0 and dim * 32 + S * 128 <= 48 * 1024


# ----------------------------------------------------------------------------- tensor-core scan: every ds
@pytest.mark.gpu
@pytest.mark.parametrize("dim,S,resid,dot", [
    (16, 16, True, False),     # ds = 1: tc_lut_kernel<1>
    (64, 64, True, False),     # ds = 1, eight table steps
    (48, 16, True, False),     # ds = 3: tc_lut_kernel<0> (codewords through lut_entry)
    (160, 32, True, False),    # ds = 5
    (512, 64, True, False),    # ds = 8
    (1280, 64, True, False),   # ds = 20: exactly at the tc_scan_supported limit
    (16, 16, False, False),    # the same kernels without residuals: ds = 1, 2, 3
    (64, 32, False, False),
    (48, 16, False, False),
    (160, 32, True, True),     # DotProduct reorder
])
def test_tc_scan_every_ds(gpu_lib, oracle, env_restore, dim, S, resid, dot):
    """16 leaves, 64 queries x 4 leaves: 16 queries per probed leaf.  The tensor-core scan matches the oracle stage by
    stage and the register-LUT scan of the same handle bit for bit."""
    assert _tc_supported(dim, S)
    n = 20_000 if dim <= 512 else 12_000
    K, L, nq, R, k = 16, 4, 64, 50, 10
    measure = gpu_lib.DistanceMeasure.DotProduct if dot else gpu_lib.DistanceMeasure.SquaredL2
    x, q, idx = _clustered(oracle, n, dim, K, S, nq, seed=dim + S + (0 if resid else 1), use_residuals=resid)
    s = _searcher(gpu_lib, idx, x, L, use_residuals=resid, measure=measure)
    os.environ["SCANN_SCAN_TC"] = "1"
    tc = _search(s, q, k, R)
    assert s.path_stats() == (1, 0)
    ora = _oracle(oracle, idx, x, q, L, R, k, use_residuals=resid, measure=oracle.DOT if dot else oracle.SQL2)
    _check_stages(oracle, x, oracle.DOT if dot else oracle.SQL2, q, k, tc, ora)
    os.environ["SCANN_SCAN_TC"] = "0"
    lut = _search(s, q, k, R)
    assert s.path_stats() == (1, 1)
    _assert_identical(tc, lut)


@pytest.mark.gpu
def test_tc_scan_past_shared_memory_limit_uses_register_lut(gpu_lib, oracle, env_restore):
    """ds = 21, one dimension group past the limit: the handle never offers the tensor-core scan, even when forced."""
    dim, S, K, L, nq, R, k = 1344, 64, 16, 4, 64, 50, 10
    assert not _tc_supported(dim, S) and _tc_supported(dim - S, S)
    x, q, idx = _clustered(oracle, 12_000, dim, K, S, nq, seed=13)
    s = _searcher(gpu_lib, idx, x, L)
    os.environ["SCANN_SCAN_TC"] = "1"
    gpu = _search(s, q, k, R)
    assert s.path_stats() == (0, 1)
    _check_stages(oracle, x, oracle.SQL2, q, k, gpu, _oracle(oracle, idx, x, q, L, R, k))


# ----------------------------------------------------------------------------- register-LUT scan: every S
@pytest.mark.gpu
@pytest.mark.parametrize("S,ds", [
    (1, 3), (3, 2), (5, 1), (7, 3), (10, 2), (25, 1), (47, 2),  # odd S, S % 4 != 0: padded groups, half-byte tails
    (65, 1), (96, 2), (128, 1),                                 # uncached LUT build (S*16 > 1024), IDP.2A
    (129, 3), (200, 1), (256, 2),                               # S > 128: mode 2; S = 256: SG = 64, 16 position bits
])
def test_register_lut_every_subspace_count(gpu_lib, oracle, env_restore, S, ds):
    """Each geometry answers a dense batch (64 queries x 4 of 16 leaves: 8 queries per work item) and a 3-query batch
    (one query per work item)."""
    dim, K, L, R, k = S * ds, 16, 4, 40, 10
    x, q, idx = _clustered(oracle, 20_000, dim, K, S, 64, seed=S * 10 + ds)
    s = _searcher(gpu_lib, idx, x, L)
    os.environ["SCANN_SCAN_TC"] = "0"
    for qb in (q, q[:3]):
        gpu = _search(s, qb, k, R)
        _check_stages(oracle, x, oracle.SQL2, qb, k, gpu, _oracle(oracle, idx, x, qb, L, R, k))
    assert s.path_stats() == (0, 2)


# ----------------------------------------------------------------------------- the largest LUT16 sum
def _ceiling_index(oracle, S, seed):
    """ds = 1, no residuals.  Subspace s has codewords 0, 0.1, ..., 1.5 in a random code order, and every query is a
    constant vector v <= 0, so the largest table entry of every subspace is the code of codeword 1.5 and quantises to
    255.  Some points carry that code in every subspace: LUT16 sum 255 * S.  Leaves 0-2 hold random codes with every
    50th point at the ceiling; leaf 3 (centre 0, where the queries are) holds 200 ceiling points and 100 random ones."""
    rng = np.random.default_rng(seed)
    sizes = [6000, 6000, 6000, 300]
    K, n = len(sizes), sum(sizes)
    cb = np.empty((S, 16, 1), np.float32)
    top = np.empty(S, np.int64)
    for s in range(S):
        p = rng.permutation(16)
        cb[s, p, 0] = np.arange(16, dtype=np.float32) * np.float32(0.1)
        top[s] = p[15]
    codes = rng.integers(0, 16, (n, S)).astype(np.uint8)
    off = np.concatenate([[0], np.cumsum(sizes)]).astype(np.uint64)
    ceiling = np.zeros(n, bool)
    ceiling[:int(off[3]):50] = True
    ceiling[int(off[3]):int(off[3]) + 200] = True
    codes[ceiling] = top
    ids = rng.permutation(n).astype(np.uint32)  # row r of the index is datapoint ids[r]
    x = np.empty((n, S), np.float32)
    x[ids] = cb[np.arange(S)[None, :], codes, 0] + np.float32(0.01) * rng.standard_normal((n, S), dtype=np.float32)
    centers = np.stack([np.full(S, c, np.float32) for c in (3.0, 4.0, 5.0, 0.0)])
    idx = dict(centers=centers, codebook=cb, packed=oracle.pack4(codes), ids=ids, part_offsets=off)
    q = np.repeat(-np.linspace(0.0, 0.3, 48, dtype=np.float32)[:, None], S, 1)
    return idx, x, q, codes, ceiling


@pytest.mark.gpu
@pytest.mark.parametrize("S", [128, 129, 256])
def test_lut16_sum_ceiling_accumulation_mode_of_s(gpu_lib, oracle, env_restore, S):
    """S = 128: sum 32640, the largest the 15-bit IDP.2A fields (mode 3) hold; S = 129: the first S of mode 2;
    S = 256: sum 65280.  A wrapped sum would pull ceiling points into the candidates; leaf 3 searched alone (L = 1,
    R > its size) returns them with their distance."""
    idx, x, q, codes, ceiling = _ceiling_index(oracle, S, seed=S)
    for i in (0, len(q) - 1):  # the construction does what it says
        l8, _, _, _ = oracle.lut16_build(idx["codebook"], q[i])
        assert (l8.max(1) == 255).all() and (l8[np.arange(S), codes[ceiling][0]] == 255).all()
    sums = oracle.lut16_scan_u32(idx["packed"][ceiling], oracle.lut16_build(idx["codebook"], q[0])[0], S)
    assert (sums == 255 * S).all()
    k = 10
    s = _searcher(gpu_lib, idx, x, 4, use_residuals=False)
    os.environ["SCANN_SCAN_TC"] = "0"
    for L, R in ((4, 64), (1, 512)):
        ora = _oracle(oracle, idx, x, q, L, R, k, use_residuals=False)
        if L == 1:
            assert (ora[5] == 300).all()  # every point of leaf 3, the 200 ceiling points among them
        _check_stages(oracle, x, oracle.SQL2, q, k, _search(s, q, k, R, L=L), ora)
    assert s.path_stats() == (0, 2)


# ----------------------------------------------------------------------------- in-leaf position bits
@pytest.mark.gpu
def test_position_bits_at_the_s256_limit(gpu_lib, oracle, env_restore):
    """S = 256 leaves 16 bits of the scan key for the position in the leaf: a leaf of 65 535 points is accepted and
    its last points are found; a leaf of 65 536 points is refused at build."""
    S, nA, nB = 256, 65_535, 1_000
    n = nA + nB
    rng = np.random.default_rng(256)
    x = rng.standard_normal((n, S), dtype=np.float32)
    cb = np.sort(rng.standard_normal((S, 16), dtype=np.float32), 1)[:, :, None]
    packed = oracle.pack4(oracle.pq_encode(cb, x))
    centers = np.stack([x[:nA].mean(0), x[nA:].mean(0)]).astype(np.float32)
    idx = dict(centers=centers, codebook=cb, packed=packed, ids=np.arange(n, dtype=np.uint32),
               part_offsets=np.array([0, nA, n], np.uint64))
    targets = np.array([nA - 1, nA - 2, nA - 3, nA - 255, nA - 256, nA - 257, nA - 4096, 0])
    q = (x[targets] + np.float32(0.01) * rng.standard_normal((len(targets), S), dtype=np.float32)).astype(np.float32)
    L, R, k = 2, 100, 10
    s = _searcher(gpu_lib, idx, x, L, use_residuals=False)
    os.environ["SCANN_SCAN_TC"] = "0"
    gpu = _search(s, q, k, R)
    _check_stages(oracle, x, oracle.SQL2, q, k, gpu, _oracle(oracle, idx, x, q, L, R, k, use_residuals=False))
    assert (gpu[0][:, 0] == targets).all()
    assert s.path_stats() == (0, 1)
    bad = dict(idx, part_offsets=np.array([0, nA + 1, n], np.uint64))
    with pytest.raises(gpu_lib.ScannError) as e:
        _searcher(gpu_lib, bad, x, L, use_residuals=False)
    assert e.value.code == gpu_lib.capi.OUT_OF_RANGE


@pytest.mark.gpu
def test_tc_scan_positions_beyond_2_17(gpu_lib, oracle, env_restore):
    """S = 16 (20 position bits): the tensor-core scan finds points at positions above 2^17 of a 140 000-point leaf.
    The queries' closest leaf (class A, SCANN_TC_RANKS=1) is another one and holds enough points for a bound, so the
    large leaf is scanned on the tensor cores."""
    S, dim, big, na, nc = 16, 32, 140_000, 5_000, 2_000
    rng = np.random.default_rng(17)
    p0 = np.full(dim, 1.0, np.float32)
    x = np.concatenate([rng.standard_normal((big, dim), dtype=np.float32),
                        0.5 * p0 + rng.standard_normal((na, dim), dtype=np.float32),
                        -p0 + rng.standard_normal((nc, dim), dtype=np.float32)]).astype(np.float32)
    x[big - 64:big] = p0 + np.float32(0.3) * rng.standard_normal((64, dim), dtype=np.float32)
    sample = x[rng.choice(len(x), 20_000, replace=False)]
    cb = np.stack([helpers.np_kmeans(np.ascontiguousarray(sample[:, 2 * s:2 * s + 2]), 16, 8, 42 + s)
                   for s in range(S)]).astype(np.float32)
    n = len(x)
    idx = dict(centers=np.stack([np.zeros(dim, np.float32), p0, -p0]), codebook=cb,
               packed=oracle.pack4(oracle.pq_encode(cb, x)), ids=np.arange(n, dtype=np.uint32),
               part_offsets=np.array([0, big, big + na, n], np.uint64))
    targets = np.arange(big - 48, big)
    assert targets.min() >= 1 << 17
    q = (x[targets] + np.float32(0.01) * rng.standard_normal((len(targets), dim), dtype=np.float32)).astype(np.float32)
    L, R, k = 3, 50, 10
    s = _searcher(gpu_lib, idx, x, L, use_residuals=False)
    os.environ["SCANN_SCAN_TC"] = "1"
    os.environ["SCANN_TC_RANKS"] = "1"
    tc = _search(s, q, k, R)
    assert s.path_stats() == (1, 0)
    _check_stages(oracle, x, oracle.SQL2, q, k, tc, _oracle(oracle, idx, x, q, L, R, k, use_residuals=False))
    assert (tc[0][:, 0] == targets).all()
    os.environ["SCANN_SCAN_TC"] = "0"
    _assert_identical(tc, _search(s, q, k, R))


# ----------------------------------------------------------------------------- queries per work item vs shared memory
SMEM_MAX = 227 * 1024


def _scan_smem_bytes(G, S, dim, R, filt=False, NW=8):
    """Restates scan_list_cap and scan_smem_bytes (csrc/lut16_scan_kernel.cuh): the dynamic shared memory of a
    register-LUT scan CTA of NW warps serving G queries.  It must follow the kernel's shared-memory layout."""
    S4 = (S + 3) // 4 * 4
    cap = (NW * 256 + 2 * R + 31) // 32 * 32
    return G * S4 * 16 + ((G * dim + 3) & ~3) * 4 + G * cap * 4 + NW * 256 * 4 + G * (7 if filt else 6) * 4 + 16


def _largest_r(G, S, dim):
    fit = [R for R in range(2049) if _scan_smem_bytes(G, S, dim, R) <= SMEM_MAX]
    return max(fit) if fit else None


@pytest.mark.parametrize("dim,S,r8", [(96, 48, 2048), (128, 64, 2048), (256, 128, 2048), (384, 192, 1888),
                                      (768, 256, 1568), (1024, 256, 1440), (2048, 256, 928), (4096, 256, None)])
def test_scan_smem_restatement_limits(dim, S, r8):
    """The largest R whose 8-query scan CTA fits (None: not even R = 0); 4, 2 and 1 queries always fit R = 2048."""
    assert _largest_r(8, S, dim) == r8
    assert all(_largest_r(G, S, dim) == 2048 for G in (4, 2, 1))


@pytest.mark.gpu
@pytest.mark.parametrize("dim,R,n", [(768, 2048, 20_000), (4096, 10, 12_000)])
def test_dense_batch_where_eight_queries_do_not_fit(gpu_lib, oracle, env_restore, dim, R, n):
    """48 queries x 2 of 8 leaves would put 8 queries in a work item, whose shared memory exceeds 227 KB here.  The
    search takes smaller items and returns what the oracle returns, bit for bit what the same queries return one at a
    time."""
    import torch

    S, K, L, k = 256, 8, 2, 10
    assert _scan_smem_bytes(8, S, dim, R) > SMEM_MAX and _scan_smem_bytes(1, S, dim, R) <= SMEM_MAX
    x, q, idx = _clustered(oracle, n, dim, K, S, 48, seed=dim)
    s = _searcher(gpu_lib, idx, x, L)
    os.environ["SCANN_SCAN_TC"] = "0"
    batch = _search(s, q, k, R)
    _check_stages(oracle, x, oracle.SQL2, q, k, batch, _oracle(oracle, idx, x, q, L, R, k))
    one = [_search(s, q[i:i + 1], k, R) for i in range(len(q))]
    _assert_identical(batch, tuple(np.concatenate([o[j] for o in one]) for j in range(6)))
    nsearch = 1 + len(q)
    if dim == 768:
        tq = torch.tensor(q).cuda()
        tau = s.search_begin(tq, k, pre_reorder_k=R)
        ids, dists, counts = s.search_end(tau)
        torch.cuda.synchronize()
        assert (ids.cpu().numpy().view(np.uint32) == batch[0]).all() and (counts.cpu().numpy() == batch[2]).all()
        assert (dists.cpu().numpy().view(np.uint32) == batch[1].view(np.uint32)).all()
        nsearch += 1
    assert s.path_stats() == (0, nsearch)
