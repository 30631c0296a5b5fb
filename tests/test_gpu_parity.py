"""GPU parity tests: the CUDA path (through the C ABI) against the CPU oracle on identical seeded inputs.
Bit-exact for integer/byte/index work; float distances are compared bit-for-bit where the kernel restates
the reference's operation order (all returned distances do) — the stated tolerance is rel 1e-4 but the
tests assert equality unless noted.  Run with -m gpu on a B200."""
import threading

import numpy as np
import pytest

import helpers

pytestmark = pytest.mark.gpu


# ----------------------------------------------------------------------------- LUT16 table build
@pytest.mark.parametrize("S,ds,nq,resid", [(48, 2, 64, True), (8, 4, 17, False), (3, 1, 5, True), (64, 2, 33, True),
                                           (255, 1, 3, False), (256, 1, 2, True), (1, 7, 4, False)])
def test_lut16_build_bit_exact(gpu_lib, oracle, S, ds, nq, resid):
    rng = np.random.default_rng(S * 100 + ds)
    cb = rng.normal(0, 0.3, (S, 16, ds)).astype(np.float32)
    q = rng.normal(0, 1, (nq, S * ds)).astype(np.float32)
    cen = rng.normal(0, 1, (nq, S * ds)).astype(np.float32) if resid else None
    l8, bias, mult = gpu_lib.lut16_build(cb, q, cen)
    for i in range(nq):
        o8, ob, om, _ = oracle.lut16_build(cb, q[i], cen[i] if resid else None)
        assert (l8[i] == o8).all(), f"query {i}: u8 table differs"
        assert bias[i] == np.float32(ob) and mult[i] == np.float32(om)


def test_lut16_build_degenerate_range(gpu_lib, oracle):
    cb = np.zeros((4, 16, 2), np.float32)  # every entry identical -> range 0 -> scale 1, multiplier 1
    q = np.full((2, 8), 1.5, np.float32)
    l8, bias, mult = gpu_lib.lut16_build(cb, q)
    o8, ob, om, _ = oracle.lut16_build(cb, q[0])
    assert (l8[0] == o8).all() and (l8 == 0).all() and mult[0] == 1.0 and bias[0] == np.float32(ob)


def test_lut16_reference_kats_through_cabi(gpu_lib):
    # src/hashes/lut16.rs:339-366 from_query KAT → tables, then src/simd/tests.rs:237-264 batch KAT
    cb = np.zeros((2, 16, 2), np.float32)
    cb[0, :, 0] = np.arange(16)
    cb[1, :, 1] = np.arange(16)
    l8, bias, mult = gpu_lib.lut16_build(cb, np.array([[5.0, 0.0, 0.0, 5.0]], np.float32))
    assert l8[0, 0, 5] == 0 and l8[0, 1, 5] == 0 and bias[0] == 0.0
    lut = np.zeros((2, 16), np.uint8)
    lut[0] = np.arange(16)
    lut[1] = 15 - np.arange(16)
    sums = gpu_lib.lut16_scan(np.array([[0x00], [0x11], [0x0F], [0xF0]], np.uint8), 2, lut)
    assert list(sums) == [15, 15, 30, 0]


# ----------------------------------------------------------------------------- LUT16 integer scan
@pytest.mark.parametrize("S,n", [(48, 100_003), (1, 1000), (2, 257), (3, 4099), (64, 50_000), (255, 3000),
                                 (256, 2049), (47, 70_001)])
def test_lut16_scan_accumulators_bit_exact(gpu_lib, oracle, S, n):
    rng = np.random.default_rng(S + n)
    codes = rng.integers(0, 16, (n, S), dtype=np.uint8)
    packed = oracle.pack4(codes)
    lut8 = rng.integers(0, 256, (S, 16), dtype=np.uint8)
    if S >= 255:
        lut8[:] = 255  # worst case for the packed 16-bit accumulators
    want = oracle.lut16_scan_u32(packed, lut8, S)
    got = gpu_lib.lut16_scan(packed, S, lut8)
    assert (got == want).all()


@pytest.mark.parametrize("S", [48, 128, 129])
def test_lut16_scan_accumulation_mode_of_s(gpu_lib, oracle, S):
    # scan_block accumulates with IDP.2A (mode 3) for S <= 128 and with IMAD/ALU adds (mode 2) above; S = 128 with
    # all-255 tables is the largest sum the 15-bit IDP.2A fields must hold (32640), S = 129 is the first S of mode 2
    mode = 3 if S <= 128 else 2  # scan_acc_mode(S)
    rng = np.random.default_rng(S * 7 + mode)
    n = 10_007
    codes = rng.integers(0, 16, (n, S), dtype=np.uint8)
    packed = oracle.pack4(codes)
    lut8 = np.full((S, 16), 255, np.uint8) if S >= 128 else rng.integers(0, 256, (S, 16), dtype=np.uint8)
    assert (gpu_lib.lut16_scan(packed, S, lut8) == oracle.lut16_scan_u32(packed, lut8, S)).all()


def test_lut16_scan_1m_x_96(gpu_lib, oracle):
    # SURVEY §7.2 minimum slice: 1M x 96 synthetic codes, S = 48: all u32 accumulators bit-identical
    rng = np.random.default_rng(5)
    n, S = 1_000_000, 48
    packed = rng.integers(0, 256, (n, S // 2), dtype=np.uint8)
    lut8 = rng.integers(0, 256, (S, 16), dtype=np.uint8)
    assert (gpu_lib.lut16_scan(packed, S, lut8) == oracle.lut16_scan_u32(packed, lut8, S)).all()


# ----------------------------------------------------------------------------- PQ encode + pack
@pytest.mark.parametrize("S,ds,n", [(48, 2, 5000), (8, 4, 1000), (5, 3, 777)])
def test_pq_encode_matches_oracle(gpu_lib, oracle, S, ds, n):
    rng = np.random.default_rng(11)
    cb = rng.normal(0, 0.5, (S, 16, ds)).astype(np.float32)
    x = rng.normal(0, 1, (n, S * ds)).astype(np.float32)
    want = oracle.pack4(oracle.pq_encode(cb, x))
    assert (gpu_lib.pq_encode(cb, x) == want).all()


def test_pq_encode_residual_device(gpu_lib, oracle):
    import torch
    rng = np.random.default_rng(12)
    S, ds, n, K = 12, 2, 3000, 7
    cb = rng.normal(0, 0.5, (S, 16, ds)).astype(np.float32)
    x = rng.normal(0, 1, (n, S * ds)).astype(np.float32)
    cen = rng.normal(0, 1, (K, S * ds)).astype(np.float32)
    assign = rng.integers(0, K, n).astype(np.uint32)
    want = oracle.pack4(oracle.pq_encode_residual(cb, x, cen, assign))
    got = gpu_lib.pq_encode(torch.tensor(cb).cuda(), torch.tensor(x).cuda(), torch.tensor(cen).cuda(),
                            torch.tensor(assign.astype(np.int32)).cuda())
    assert (got.cpu().numpy() == want).all()


# ----------------------------------------------------------------------------- partition selection
@pytest.mark.parametrize("K,dim,nq,L", [(2000, 96, 300, 64), (10, 2, 9, 3), (100, 128, 50, 100), (7, 5, 4, 12),
                                        (4099, 33, 20, 1)])
def test_partition_bit_exact(gpu_lib, oracle, K, dim, nq, L):
    rng = np.random.default_rng(K + dim)
    centers = rng.normal(0, 1, (K, dim)).astype(np.float32)
    q = rng.normal(0, 1, (nq, dim)).astype(np.float32)
    part = gpu_lib.TreePartitioner(centers)
    tokens, dists = part.partition(q, L)
    otok, odist = oracle.partition(centers, q, L)
    assert (tokens == otok).all()
    assert (dists.view(np.uint32) == odist.view(np.uint32)).all()


def test_partition_ties_lower_id_first_and_device_path(gpu_lib, oracle):
    import torch
    centers = np.array([[1, 0], [0, 1], [5, 5], [0, -1], [1, 0]], np.float32)
    q = np.zeros((3, 2), np.float32)
    part = gpu_lib.TreePartitioner(centers)
    tokens, dists = part.partition(q, 4)
    assert list(tokens[0]) == [0, 1, 3, 4]
    t2, d2 = part.partition(torch.tensor(q).cuda(), 4)
    torch.cuda.synchronize()
    assert (t2.cpu().numpy().view(np.uint32) == tokens).all()


def test_partition_errors(gpu_lib):
    part = gpu_lib.TreePartitioner()
    with pytest.raises(gpu_lib.ScannError) as e:
        part.partition(np.zeros((1, 2), np.float32), 1)
    assert e.value.code == gpu_lib.capi.FAILED_PRECONDITION  # "Partitioner not built"
    part = gpu_lib.TreePartitioner(np.zeros((3, 4), np.float32))
    with pytest.raises(gpu_lib.ScannError) as e:
        part.partition(np.zeros((1, 2), np.float32), 1)
    assert e.value.code == gpu_lib.capi.INVALID_ARGUMENT


# ----------------------------------------------------------------------------- Tree-AH end to end
def _check_stages(oracle, x, om, qs, k, gpu, ora):
    """Stage-wise parity of one Tree-AH batch.  Exact ties of the integer LUT16 score are the only licence
    to differ (BASELINE.json: 'away from exact ties'), so the comparison is made tie-proof:
      (1) the sorted approximate candidate distances are tie-independent -> bit-identical;
      (2) candidate ids strictly below the cut-off value are the same set;
      (3) the oracle's reorder (tree_x_hybrid/mod.rs:342-364) applied to the GPU's own candidate list must
          reproduce the GPU's final ids and bit-identical exact distances.
    Returns the end-to-end recall vs the oracle over the valid results (informational + bounded by callers)."""
    ids, dists, counts, ci, cd, cc = gpu
    oids, odists, ocounts, ocand, ocand_d, ocand_n = ora
    nq = len(qs)
    assert (cc == ocand_n).all()
    assert (cd.view(np.uint32) == ocand_d.view(np.uint32)).all(), "approximate (LUT16) candidate distances differ"
    hit = tot = 0
    for qi in range(nq):
        c = int(cc[qi])
        if c:
            cut = cd[qi, c - 1]
            a = set(ci[qi, :c][cd[qi, :c] < cut].tolist())
            b = set(ocand[qi, :c][ocand_d[qi, :c] < cut].tolist())
            assert a == b, f"query {qi}: candidate sets differ away from the cut-off tie"
        eids, ed = oracle.reorder(x, om, qs[qi], ci[qi, :c], k)
        m = len(eids)
        assert m == counts[qi] == ocounts[qi]
        assert (dists[qi, :m].view(np.uint32) == ed.view(np.uint32)).all(), "exact reorder distances differ"
        assert (ids[qi, :m] == eids).all() or len(set(ed.tolist())) < m, "reorder order differs without a tie"
        assert (ids[qi, m:] == 0xFFFFFFFF).all() and np.isinf(dists[qi, m:]).all()
        hit += len(set(ids[qi, :m].tolist()) & set(oids[qi, :m].tolist()))
        tot += m
        same = ids[qi, :m] == oids[qi, :m]
        assert (dists[qi, :m][same].view(np.uint32) == odists[qi, :m][same].view(np.uint32)).all()
    return hit / max(tot, 1)


def _treeah_case(gpu_lib, oracle, n, dim, K, S, nq, L, R, k, measure, seed, device_path=False, use_residuals=True,
                 min_recall=0.999):
    x, _ = helpers.clustered(n, dim, max(8, K), 0.35, seed)
    qs, _ = helpers.clustered(nq, dim, max(8, K), 0.35, seed)  # same latent centres (same seed → same lat)
    qs = (qs + 0.05 * helpers.gaussian(nq, dim, seed + 1)).astype(np.float32)
    idx = helpers.build_index(oracle, x, K, S, use_residuals=use_residuals)
    om = {gpu_lib.DistanceMeasure.SquaredL2: oracle.SQL2, gpu_lib.DistanceMeasure.DotProduct: oracle.DOT}[measure]
    rc, oids, odists, ocounts, ocand, ocand_d, ocand_n = oracle.treex_search(
        idx["centers"], idx["codebook"], idx["part_offsets"], idx["ids"], idx["packed"], x, qs, L, R, k, lut16=True,
        use_residuals=use_residuals, reorder_measure=om, nthreads=8, want_candidates=True)
    assert rc == 0
    cfg = gpu_lib.TreeXHybridConfig(num_partitions=K, partitions_to_search=L, use_residuals=use_residuals,
                                    distance_measure=measure)
    s = gpu_lib.TreeXHybridSearcher(cfg)
    if device_path:
        import torch
        t = lambda a, dt=None: torch.tensor(a if dt is None else a.astype(dt)).cuda()
        s.build_from_index(t(idx["centers"]), t(idx["codebook"]), t(idx["packed"]), t(idx["ids"], np.int32),
                           t(idx["part_offsets"], np.int64), t(x))
        ids, dists, counts, (ci, cd, cc) = s.search_batched(t(qs), k, pre_reorder_k=R, want_candidates=True)
        torch.cuda.synchronize()
        ids, dists, counts = ids.cpu().numpy().view(np.uint32), dists.cpu().numpy(), counts.cpu().numpy()
        ci, cd, cc = ci.cpu().numpy().view(np.uint32), cd.cpu().numpy(), cc.cpu().numpy()
    else:
        s.build_from_index(idx["centers"], idx["codebook"], idx["packed"], idx["ids"], idx["part_offsets"], x)
        ids, dists, counts, (ci, cd, cc) = s.search_batched(qs, k, pre_reorder_k=R, want_candidates=True)
    rec = _check_stages(oracle, x, om, qs, k, (ids, dists, counts, ci, cd, cc),
                        (oids, odists, ocounts, ocand, ocand_d, ocand_n))
    assert rec >= min_recall, f"recall vs oracle {rec}"
    by, pairs = s.last_scan_bytes()
    sizes = np.diff(idx["part_offsets"].astype(np.int64))
    otok, _ = oracle.partition(idx["centers"], qs, min(L, K))
    assert pairs == int((sizes[otok] > 0).sum()) and by == int(sizes[otok].sum()) * ((S + 1) // 2)
    return s


def test_treeah_small_sql2(gpu_lib, oracle):
    # coarse PQ (S=8) + small R: the approximate cut-off tie is large, so end-to-end recall vs the oracle is
    # only loosely bounded here; the stage-wise checks inside _treeah_case are exact
    _treeah_case(gpu_lib, oracle, n=20_000, dim=32, K=32, S=8, nq=40, L=6, R=30, k=10,
                 measure=gpu_lib.DistanceMeasure.SquaredL2, seed=1, min_recall=0.9)


@pytest.mark.parametrize("nq", [1, 7, 64, 700])
def test_treeah_c3_shape_dot(gpu_lib, oracle, nq):
    # C3 geometry scaled down: D=96, S=48 (ds=2), 16 codes, Dot reorder, R=100, k=10.  nq sweeps the
    # queries-per-leaf group size G (1, 2, 4, 8 variants of the scan kernel).
    # End-to-end recall vs the oracle is bounded by the cut-off tie only (FastTopNeighbors keeps a
    # history-dependent subset of the tied points, top_k.rs:341-353): >= 0.998 here, stage checks exact.
    _treeah_case(gpu_lib, oracle, n=120_000, dim=96, K=60, S=48, nq=nq, L=16, R=100, k=10,
                 measure=gpu_lib.DistanceMeasure.DotProduct, seed=3, min_recall=0.998)


def test_treeah_c4_shape_sql2_tensor_core_partition(gpu_lib, oracle):
    # C4 geometry scaled down: D=128, S=64 (32 B/point), SqL2 reorder, K=300 (>= 256: the centroid scoring runs on
    # tcgen05 and the survivors are re-scored exactly), R=100, k=10.
    _treeah_case(gpu_lib, oracle, n=150_000, dim=128, K=300, S=64, nq=200, L=24, R=100, k=10,
                 measure=gpu_lib.DistanceMeasure.SquaredL2, seed=8, min_recall=0.995)


def test_treeah_device_pointers(gpu_lib, oracle):
    _treeah_case(gpu_lib, oracle, n=30_000, dim=64, K=20, S=16, nq=128, L=5, R=50, k=10,
                 measure=gpu_lib.DistanceMeasure.SquaredL2, seed=4, device_path=True, min_recall=0.97)


def test_treeah_ragged_partitions_and_large_R(gpu_lib, oracle):
    # tiny / empty partitions, L > K, R larger than many leaves, k > available
    rng = np.random.default_rng(9)
    n, dim, K, S = 3000, 16, 40, 4
    x = rng.normal(0, 1, (n, dim)).astype(np.float32)
    idx = helpers.build_index(oracle, x, K, S)
    # force two empty partitions by moving their centres far away (offsets stay consistent: rebuild)
    idx["centers"][3] = 1e3
    idx["centers"][17] = -1e3
    assign = oracle.partition(idx["centers"], x, 1)[0][:, 0].astype(np.uint32)
    order = np.argsort(assign, kind="stable").astype(np.uint32)
    idx["ids"] = order
    idx["part_offsets"] = np.concatenate([[0], np.cumsum(np.bincount(assign, minlength=K))]).astype(np.uint64)
    idx["packed"] = oracle.pack4(oracle.pq_encode_residual(idx["codebook"], x[order], idx["centers"], assign[order]))
    q = rng.normal(0, 1, (33, dim)).astype(np.float32)
    for (L, R, k) in [(50, 600, 10), (3, 2000, 25), (40, 5, 10), (1, 1, 1)]:
        rc, oids, odists, ocounts, ocand, ocd, ocn = oracle.treex_search(
            idx["centers"], idx["codebook"], idx["part_offsets"], idx["ids"], idx["packed"], x, q, L, R, k,
            lut16=True, want_candidates=True)
        s = gpu_lib.TreeXHybridSearcher(gpu_lib.TreeXHybridConfig(num_partitions=K, partitions_to_search=L))
        s.build_from_index(idx["centers"], idx["codebook"], idx["packed"], idx["ids"], idx["part_offsets"], x)
        ids, dists, counts, (ci, cd, cc) = s.search_batched(q, k, pre_reorder_k=R, want_candidates=True)
        rec = _check_stages(oracle, x, oracle.SQL2, q, k, (ids, dists, counts, ci, cd, cc),
                            (oids, odists, ocounts, ocand, ocd, ocn))
        assert rec >= 0.95, (L, R, k, rec)


def test_treeah_no_raw_returns_approximate(gpu_lib, oracle):
    rng = np.random.default_rng(10)
    x = rng.normal(0, 1, (5000, 24)).astype(np.float32)
    idx = helpers.build_index(oracle, x, 12, 12)
    q = rng.normal(0, 1, (20, 24)).astype(np.float32)
    rc, oids, odists, ocounts = oracle.treex_search(idx["centers"], idx["codebook"], idx["part_offsets"], idx["ids"],
                                                    idx["packed"], None, q, 4, 30, 10, lut16=True)
    s = gpu_lib.TreeXHybridSearcher(gpu_lib.TreeXHybridConfig(num_partitions=12, partitions_to_search=4))
    s.build_from_index(idx["centers"], idx["codebook"], idx["packed"], idx["ids"], idx["part_offsets"], None)
    ids, dists, counts = s.search_batched(q, 10, pre_reorder_k=30)
    assert (dists.view(np.uint32) == odists.view(np.uint32)).all()


def test_treeah_errors(gpu_lib, oracle):
    rng = np.random.default_rng(13)
    x = rng.normal(0, 1, (500, 8)).astype(np.float32)
    idx = helpers.build_index(oracle, x, 4, 4)
    s = gpu_lib.TreeXHybridSearcher()
    with pytest.raises(gpu_lib.ScannError) as e:
        s.search_batched(x[:1], 5)
    assert e.value.code == gpu_lib.capi.FAILED_PRECONDITION
    with pytest.raises(gpu_lib.ScannError) as e:  # D % S != 0 (codebook.rs:154-159)
        s.build_from_index(np.zeros((4, 9), np.float32), idx["codebook"], idx["packed"], idx["ids"], idx["part_offsets"])
    assert e.value.code == gpu_lib.capi.INVALID_ARGUMENT
    s.build_from_index(idx["centers"], idx["codebook"], idx["packed"], idx["ids"], idx["part_offsets"], x)
    with pytest.raises(gpu_lib.ScannError) as e:  # "Query dimensionality mismatch"
        s.search_batched(np.zeros((1, 5), np.float32), 5)
    assert e.value.code == gpu_lib.capi.INVALID_ARGUMENT
    ids, dists, counts = s.search_batched(np.zeros((0, 8), np.float32), 5)
    assert ids.shape[0] == 0  # empty batch → Ok(vec![])


def test_flat_asymmetric_hasher(gpu_lib, oracle):
    rng = np.random.default_rng(14)
    n, dim, S = 20_000, 32, 16
    x = rng.normal(0, 1, (n, dim)).astype(np.float32)
    idx = helpers.build_index(oracle, x, 1, S, use_residuals=False)
    cb = idx["codebook"]
    packed = oracle.pack4(oracle.pq_encode(cb, x))
    q = rng.normal(0, 1, (50, dim)).astype(np.float32)
    ah = gpu_lib.AsymmetricHasher().build_from_index(cb, packed, x)
    ids, dists, counts = ah.search_batched(q, 10)
    rc, oids, odists, ocounts = oracle.ah_search(cb, packed, q, 10, lut16=True)
    assert (np.sort(dists, 1).view(np.uint32) == np.sort(odists, 1).view(np.uint32)).all()
    ids2, d2, c2 = ah.search_with_reordering(q, 10, 100)
    rc, oids2, od2, oc2 = oracle.ah_search(cb, packed, q, 10, lut16=True, raw=x, pre_k=100)
    assert helpers.recall(ids2, oids2, 10) >= 0.99


# ----------------------------------------------------------------------------- brute force (f32)
def test_bf_reference_kats(gpu_lib):
    ds5 = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0], [0, 0, 1], [1, 1, 1]], np.float32)
    bf = gpu_lib.BruteForceSearcher(ds5, gpu_lib.DistanceMeasure.SquaredL2)
    r = bf.search([0, 0, 0], 3)                       # searcher.rs:280-291
    assert len(r) == 3 and r[0][0] == 0 and abs(r[0][1]) < 1e-6
    r = bf.search([0.5, 0.5, 0.5], 5)                 # :293-306
    assert len(r) == 5 and all(r[i][1] >= r[i - 1][1] for i in range(1, 5))
    ids, dists, counts = bf.search_batched(np.array([[0, 0, 0], [1, 1, 1]], np.float32), 2)  # :340-354
    assert list(counts) == [2, 2] and ids[1, 0] == 4
    assert len(bf.search([0, 0, 0], 50)) == 5         # k clamped to n (:91)
    with pytest.raises(gpu_lib.ScannError) as e:      # :367-376
        bf.search([1.0, 2.0], 5)
    assert e.value.code == gpu_lib.capi.INVALID_ARGUMENT
    dot = gpu_lib.BruteForceSearcher(np.array([[1, 0], [0, 1], [1, 1]], np.float32), gpu_lib.DistanceMeasure.DotProduct)
    r = dot.search([1.0, 0.0], 3)                     # :308-325
    assert [d for _, d in r] == [-1.0, -1.0, 0.0] and r[2][0] == 1


def test_bf_empty_dataset_and_empty_batch(gpu_lib):
    bf = gpu_lib.BruteForceSearcher(np.zeros((0, 3), np.float32), gpu_lib.DistanceMeasure.SquaredL2, dim=3)
    assert bf.search([1.0, 2.0, 3.0], 5) == []        # searcher.rs:356-365
    bf2 = gpu_lib.BruteForceSearcher(np.ones((4, 3), np.float32))
    ids, dists, counts = bf2.search_batched(np.zeros((0, 3), np.float32), 5)
    assert ids.shape[0] == 0


@pytest.mark.parametrize("measure", ["SquaredL2", "DotProduct", "L2"])
@pytest.mark.parametrize("n,dim,nq,k", [(10_000, 128, 1000, 10), (3001, 100, 77, 25), (500, 3, 40, 7)])
def test_bf_matches_oracle(gpu_lib, oracle, measure, n, dim, nq, k):
    db = helpers.gaussian(n, dim, 42)
    q = helpers.gaussian(nq, dim, 123)
    m = gpu_lib.DistanceMeasure[measure]
    om = {"SquaredL2": oracle.SQL2, "DotProduct": oracle.DOT, "L2": oracle.L2}[measure]
    bf = gpu_lib.BruteForceSearcher(db, m)
    ids, dists, counts = bf.search_batched(q, k)
    rc, oids, odists, ocounts = oracle.bf_search(db, q, k, om, nthreads=8)
    assert (counts == ocounts).all()
    compared, mism = helpers.ids_equal_away_from_ties(ids, dists, oids, odists, counts)
    assert mism == 0 and compared > 0
    same = ids == oids
    assert same.mean() > 0.999
    # returned distances are re-scored in the reference's AVX2 order: bit-identical
    assert (dists[same].view(np.uint32) == odists[same].view(np.uint32)).all()
    assert np.allclose(dists, odists, rtol=1e-4, atol=0)


def test_bf_stress_recall_verification_property(gpu_lib, oracle):
    # tests/stress_tests.rs:325-363 through the GPU path
    db = np.random.default_rng(42).random((1000, 32), dtype=np.float32)
    q = np.random.default_rng(123).random((1, 32), dtype=np.float32)
    ids, dists, counts = gpu_lib.BruteForceSearcher(db).search_batched(q, 10)
    alld = np.array([oracle.pair_distance(oracle.SQL2, q[0], db[i]) for i in range(1000)], np.float32)
    order = np.argsort(alld, kind="stable")
    assert list(ids[0]) == list(order[:10]) and np.abs(dists[0] - alld[order[:10]]).max() < 1e-5


def test_bf_strided_dataset_and_device_queries(gpu_lib, oracle):
    import torch
    db = np.zeros((300, 16), np.float32)  # DenseDataset stride rule: dim 3 → stride 16
    db[:, :3] = helpers.gaussian(300, 3, 1)
    q = helpers.gaussian(20, 3, 2)
    bf = gpu_lib.BruteForceSearcher(db, gpu_lib.DistanceMeasure.SquaredL2, dim=3)
    ids, dists, counts = bf.search_batched(torch.tensor(q).cuda(), 5)
    torch.cuda.synchronize()
    rc, oids, odists, oc = oracle.bf_search(db, q, 5, oracle.SQL2, dim=3)
    assert (ids.cpu().numpy().view(np.uint32) == oids).all()
    assert (dists.cpu().numpy().view(np.uint32) == odists.view(np.uint32)).all()


def test_bf_concurrent_queries(gpu_lib, oracle):
    # tests/stress_tests.rs:256-297: 4 threads share one searcher
    db = helpers.gaussian(5000, 64, 7)
    bf = gpu_lib.BruteForceSearcher(db)
    qs = [helpers.gaussian(50, 64, 100 + t) for t in range(4)]
    out = [None] * 4

    def work(t):
        out[t] = bf.search_batched(qs[t], 10)

    th = [threading.Thread(target=work, args=(t,)) for t in range(4)]
    [t.start() for t in th]
    [t.join() for t in th]
    for t in range(4):
        rc, oids, odists, oc = oracle.bf_search(db, qs[t], 10, oracle.SQL2, nthreads=4)
        assert (out[t][0] == oids).all()


# ----------------------------------------------------------------------------- scalar-quantised brute force
def test_sq8_quantizer_matches_oracle(gpu_lib, oracle):
    db = helpers.gaussian(20_000, 64, 42)
    codes, cal = gpu_lib.scalar_quantize(db)
    ocodes, ocal = oracle.sq8_quantize(db)
    # the f64 Σ/Σ² are reduced in parallel: calibration may differ by an ulp (DESIGN.md), codes then differ
    # only at rounding boundaries
    assert np.allclose(cal, ocal, rtol=1e-6)
    assert (codes != ocodes).mean() < 1e-4
    if (cal == ocal).all():
        assert (codes == ocodes).all()


def test_sq8_reference_kats(gpu_lib):
    db = np.array([[0, 0, 0], [10, 0, 0], [0, 10, 0], [0, 0, 10], [10, 10, 10]], np.float32)
    s = gpu_lib.ScalarQuantizedBruteForceSearcher(db, gpu_lib.ScalarQuantizedConfig.squared_l2())
    r = s.search([0, 0, 0], 3)                        # scalar_quantized.rs:424-435
    assert len(r) == 3 and r[0][0] == 0
    db2 = np.array([[1, 2, 3], [4, 5, 6], [7, 8, 9], [1.1, 2.1, 3.1], [10, 0, 0]], np.float32)
    s2 = gpu_lib.ScalarQuantizedBruteForceSearcher(db2)
    f = gpu_lib.BruteForceSearcher(db2)
    assert s2.search([1, 2, 3], 3)[0][0] == f.search([1, 2, 3], 3)[0][0]  # :485-513


@pytest.mark.parametrize("measure", ["SquaredL2", "DotProduct"])
@pytest.mark.parametrize("n,dim,nq,k", [(20_000, 128, 300, 10), (1000, 20, 33, 5)])
def test_sq8_search_matches_oracle(gpu_lib, oracle, measure, n, dim, nq, k):
    db = helpers.gaussian(n, dim, 42)
    q = helpers.gaussian(nq, dim, 123)
    ocodes, ocal = oracle.sq8_quantize(db)  # identical int8 codes into both paths (incl. the wrap quirk)
    m = gpu_lib.DistanceMeasure[measure]
    om = {"SquaredL2": oracle.SQL2, "DotProduct": oracle.DOT}[measure]
    s = gpu_lib.ScalarQuantizedBruteForceSearcher.from_quantized(ocodes, float(ocal[2]), m)
    ids, dists, counts = s.search_batched(q, k)
    rc, oids, odists, ocounts = oracle.sq8_search(ocodes, float(ocal[2]), q, k, om, nthreads=8)
    assert (counts == ocounts).all()
    compared, mism = helpers.ids_equal_away_from_ties(ids, dists, oids, odists, counts)
    assert mism == 0
    same = ids == oids
    assert same.mean() > 0.995
    assert (dists[same].view(np.uint32) == odists[same].view(np.uint32)).all()


# ----------------------------------------------------------------------------- multi-GPU merge kernel
def test_merge_topk(gpu_lib):
    rng = np.random.default_rng(3)
    parts, nq, k = 8, 50, 10
    d = np.sort(rng.random((parts, nq, k), dtype=np.float32), axis=2)
    ids = rng.permutation(parts * nq * k).astype(np.uint32).reshape(parts, nq, k)
    ids[3, :, 7:] = 0xFFFFFFFF  # a short shard
    d[3, :, 7:] = np.inf
    oi, od, oc = gpu_lib.merge_topk(ids, d)
    for q in range(nq):
        cand = [(d[p, q, j], ids[p, q, j]) for p in range(parts) for j in range(k) if ids[p, q, j] != 0xFFFFFFFF]
        cand.sort()
        assert [c[1] for c in cand[:k]] == list(oi[q]) and oc[q] == k


# ----------------------------------------------------------------------------- façade
def test_scann_builder_brute_force_and_tree_ah(gpu_lib, oracle):
    x, _ = helpers.clustered(20_000, 32, 64, 0.3, 5)
    q = x[:64] + 0.01
    sc = gpu_lib.ScannBuilder().num_neighbors(5).distance_measure(gpu_lib.DistanceMeasure.SquaredL2).brute_force() \
        .build(x)
    assert sc.search_mode == gpu_lib.SearchMode.BruteForce and sc.config.num_neighbors == 5
    ids, dists, counts = sc.search_batched(q)
    assert ids.shape == (64, 5) and (ids[:, 0] == np.arange(64)).all()
    ta = gpu_lib.ScannBuilder().num_neighbors(10).tree(32, 8).hash(16).reorder(100).build(x)
    assert ta.search_mode == gpu_lib.SearchMode.TreeAH
    tids, td, tc = ta.search_batched(q, 10)
    rc, gt, _, _ = oracle.bf_search(x, q, 10, oracle.SQL2, nthreads=8)
    assert helpers.recall(tids, gt, 10) > 0.8
    with pytest.raises(gpu_lib.ScannError):
        gpu_lib.Scann.brute_force(np.zeros((0, 4), np.float32))  # "Dataset cannot be empty"


# ----------------------------------------------------------------------------- restrict filter in the scan
@pytest.mark.parametrize("keep_frac,nq", [(0.5, 64), (0.02, 200), (0.999, 9)])
def test_treeah_search_with_filter(gpu_lib, oracle, keep_frac, nq):
    # TreeXHybridSearcher::search_with_filter (tree_x_hybrid/mod.rs:245-250, 327-332): filtered-out points are skipped
    # before the per-leaf top-R, so sparse filters make leaves contribute fewer than R candidates.
    n, dim, K, S, L, R, k = 60_000, 32, 40, 16, 8, 60, 10
    x, _ = helpers.clustered(n, dim, 48, 0.35, 17)
    qs, _ = helpers.clustered(nq, dim, 48, 0.35, 17)
    qs = (qs + 0.05 * helpers.gaussian(nq, dim, 18)).astype(np.float32)
    idx = helpers.build_index(oracle, x, K, S)
    allowed = np.random.default_rng(5).random(n) < keep_frac
    bits = np.packbits(allowed, bitorder="little")
    rc, oids, odists, ocounts, ocand, ocd, ocn = oracle.treex_search(
        idx["centers"], idx["codebook"], idx["part_offsets"], idx["ids"], idx["packed"], x, qs, L, R, k, lut16=True,
        nthreads=8, want_candidates=True, allow=bits)
    s = gpu_lib.TreeXHybridSearcher(gpu_lib.TreeXHybridConfig(num_partitions=K, partitions_to_search=L))
    s.build_from_index(idx["centers"], idx["codebook"], idx["packed"], idx["ids"], idx["part_offsets"], x)
    ids, dists, counts, (ci, cd, cc) = s.search_with_filter(qs, k, allowed, pre_reorder_k=R, want_candidates=True)
    valid = ids != 0xFFFFFFFF
    assert allowed[ids[valid]].all(), "a filtered-out datapoint was returned"
    rec = _check_stages(oracle, x, oracle.SQL2, qs, k, (ids, dists, counts, ci, cd, cc),
                        (oids, odists, ocounts, ocand, ocd, ocn))
    assert rec >= 0.99, rec
    # the filter is cleared afterwards: the plain search is the unfiltered one again
    ids2, _, _ = s.search_batched(qs, k, pre_reorder_k=R)
    rc, pids, _, _ = oracle.treex_search(idx["centers"], idx["codebook"], idx["part_offsets"], idx["ids"], idx["packed"],
                                         x, qs, L, R, k, lut16=True, nthreads=8)
    assert helpers.recall(ids2, pids, k) >= 0.99


def test_search_batched_with_params_on_gpu(gpu_lib, oracle):
    # Searcher::search_batched_with_params: per-query k, grouped into GPU batches, answers in query order
    db = helpers.gaussian(2000, 16, 3)
    q = helpers.gaussian(6, 16, 4)
    P = gpu_lib.SearchParameters
    ks = [3, 7, 3, 1, 7, 5]
    out = gpu_lib.BruteForceSearcher(db).search_batched_with_params(q, [P().with_num_neighbors(k) for k in ks])
    for i, k in enumerate(ks):
        rc, oi, od, oc = oracle.bf_search(db, q[i:i + 1], k, oracle.SQL2)
        assert [p[0] for p in out[i]] == list(oi[0]) and len(out[i]) == k
