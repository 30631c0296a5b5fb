"""Class A of the tensor-core Tree-AH search: the T closest leaves of every query are scanned in full by the
register-LUT kernel, and the R-th approx distance of the union of a query's class-A lists (union_bound_kernel, treeah.cu)
bounds the tensor-core pass.  Whatever T (SCANN_TC_RANKS), the ids, distances and candidate lists must be bit-identical
to the register-LUT path (SCANN_SCAN_TC=0)."""
import os

import numpy as np
import pytest
import torch

import helpers

pytestmark = pytest.mark.gpu


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


def _searcher(pkg, idx, x, L, measure=None):
    kw = {} if measure is None else {"distance_measure": measure}
    cfg = pkg.TreeXHybridConfig(num_partitions=len(idx["centers"]), partitions_to_search=L, **kw)
    return pkg.TreeXHybridSearcher(cfg).build_from_index(idx["centers"], idx["codebook"], idx["packed"], idx["ids"],
                                                         idx["part_offsets"], x)


def _both_paths(s, q, k, R, ranks):
    out = {}
    for mode in ("0", "1"):
        os.environ["SCANN_SCAN_TC"] = mode
        os.environ["SCANN_TC_RANKS"] = str(ranks)
        out[mode] = s.search_batched(q, k, pre_reorder_k=R, want_candidates=True)
    return out["0"], out["1"]


def _assert_identical(a, b):
    (i0, d0, c0, (ci0, cd0, cc0)), (i1, d1, c1, (ci1, cd1, cc1)) = a, b
    assert (c0 == c1).all() and (cc0 == cc1).all()
    assert (cd0.view(np.uint32) == cd1.view(np.uint32)).all() and (ci0 == ci1).all()
    assert (d0.view(np.uint32) == d1.view(np.uint32)).all() and (i0 == i1).all()


@pytest.mark.parametrize("ranks", [1, 2, 4])
def test_classa_same_results_as_register_lut_kernel(gpu_lib, oracle, env_restore, ranks):
    """16 leaves, 3000 queries: every leaf is class A for several hundred queries."""
    x, _ = helpers.clustered(200_000, 96, 64, 0.35, 31)
    q, _ = helpers.clustered(3000, 96, 64, 0.35, 31)
    q = (q + 0.03 * helpers.gaussian(3000, 96, 32)).astype(np.float32)
    idx = helpers.build_index(oracle, x, 16, 48)
    s = _searcher(gpu_lib, idx, x, 6)
    a, b = _both_paths(s, q, 10, 100, ranks)
    tc, lut = s.path_stats()
    assert tc == 1 and lut == 1, (tc, lut)
    _assert_identical(a, b)


@pytest.mark.parametrize("ranks", [1, 2, 4])
def test_classa_small_leaves_and_short_unions(gpu_lib, oracle, env_restore, ranks):
    """Leaves smaller than one 128-point tile and smaller than R: a query whose class-A lists hold fewer than R points
    together gets no bound from them, is flagged and re-done by the register-LUT kernel."""
    rng = np.random.default_rng(9)
    dim, S, K = 32, 16, 8
    base = rng.normal(0, 1, (K, dim)).astype(np.float32) * 4
    sizes = [3000, 40, 2500, 12, 100, 2000, 127, 1500]
    x = np.concatenate([base[c] + 0.3 * rng.normal(0, 1, (m, dim)).astype(np.float32) for c, m in enumerate(sizes)])
    x = x.astype(np.float32)
    idx = helpers.build_index(oracle, x, K, S)
    q = np.concatenate([base[c][None] + 0.05 * rng.normal(0, 1, (60, dim)) for c in range(K)]).astype(np.float32)
    s = _searcher(gpu_lib, idx, x, 4)
    a, b = _both_paths(s, q, 10, 60, ranks)
    tc, lut = s.path_stats()
    assert tc == 1 and lut == 1, (tc, lut)
    _assert_identical(a, b)


def test_classa_two_phase_search(gpu_lib, oracle, env_restore):
    """search_begin runs class A and returns the union bounds; search_end gives what the register-LUT path gives, with
    the bounds as returned and with no bounds at all."""
    x, _ = helpers.clustered(120_000, 32, 64, 0.35, 41)
    idx = helpers.build_index(oracle, x, 24, 16)
    s = _searcher(gpu_lib, idx, x, 6)
    q = torch.tensor(x[:2000] + 0.01).cuda()
    os.environ["SCANN_SCAN_TC"] = "0"
    ids, dists, counts = s.search_batched(q, 10, pre_reorder_k=80)
    os.environ["SCANN_SCAN_TC"] = "1"
    for ranks in (1, 3):
        os.environ["SCANN_TC_RANKS"] = str(ranks)
        tau = s.search_begin(q, 10, pre_reorder_k=80)
        assert bool(torch.isfinite(tau).all())
        for t in (tau, None):
            if t is None:
                s.search_begin(q, 10, pre_reorder_k=80)
            ids2, dists2, counts2 = s.search_end(t)
            torch.cuda.synchronize()
            assert (ids.cpu() == ids2.cpu()).all() and (counts.cpu() == counts2.cpu()).all()
            assert (dists.cpu().numpy().view(np.uint32) == dists2.cpu().numpy().view(np.uint32)).all()
    tc, lut = s.path_stats()
    assert tc == 4 and lut == 1, (tc, lut)
