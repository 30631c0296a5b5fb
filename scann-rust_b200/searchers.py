"""Host-side mirror of the reference crate's searcher API over the C ABI (include/scann_b200.h).

Same names, argument meaning and error behaviour as the Rust types they mirror, so the parity tests read
like the reference's own tests:

  BruteForceSearcher                 src/brute_force/searcher.rs:34-208
  ScalarQuantizedBruteForceSearcher  src/brute_force/scalar_quantized.rs:99-326
  TreePartitioner (query side)       src/partitioning/tree_partitioner.rs:37-229
  AsymmetricHasher (LUT16 path)      src/hashes/hasher.rs:97-238
  TreeXHybridSearcher                src/tree_x_hybrid/mod.rs:114-294
  Scann / ScannBuilder               src/scann.rs:60-137,175-303,364-432

Inputs may be numpy arrays (host path: the library copies H2D/D2H and synchronises) or torch CUDA tensors
(device path: pointers are passed through, work is enqueued on torch's current stream, results are torch
tensors).  torch is only plumbing here (device memory + streams).
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field
from enum import IntEnum
from typing import Optional

import numpy as np

from . import capi
from .capi import ScannError


class DistanceMeasure(IntEnum):
    """The measures the hot path dispatches to SIMD kernels (src/distance_measures/mod.rs:32-66)."""
    SquaredL2 = capi.SQL2
    L2 = capi.L2
    DotProduct = capi.DOT


def _is_torch(x) -> bool:
    return type(x).__module__.startswith("torch")


def _torch():
    import torch
    return torch


def _stream_ptr(device_index: int):
    torch = _torch()
    return C.c_void_p(torch.cuda.current_stream(device_index).cuda_stream)


class _Batch:
    """Normalises a query batch to a contiguous f32 [nq, dim] buffer and remembers where it lives."""

    def __init__(self, queries, device_index: int):
        self.device = _is_torch(queries) and queries.is_cuda
        if _is_torch(queries):
            torch = _torch()
            q = queries.to(torch.float32).contiguous()
            if q.dim() == 1:
                q = q[None, :]
            self.arr = q
            self.nq, self.dim = int(q.shape[0]), int(q.shape[1]) if q.dim() == 2 else 0
            if self.device:
                self.ptr = C.c_void_p(q.data_ptr())
                self.memspace = capi.DEVICE
                self.stream = _stream_ptr(q.device.index if q.device.index is not None else device_index)
            else:
                self.np = q.numpy()
                self.ptr = capi.np_ptr(self.np)
                self.memspace = capi.HOST
                self.stream = None
        else:
            if isinstance(queries, (list, tuple)) and len(queries) > 0 and len({len(r) for r in queries}) > 1:
                raise ScannError(capi.INVALID_ARGUMENT, "ragged query batch: dimensionalities differ")
            q = capi.as_f32(queries)
            if q.ndim == 1:
                q = q[None, :] if q.size else q.reshape(0, 0)
            self.arr = q
            self.nq, self.dim = int(q.shape[0]), int(q.shape[1])
            self.ptr = capi.np_ptr(q)
            self.memspace = capi.HOST
            self.stream = None

    def outputs(self, k: int, extra_R: int = 0):
        if self.device:
            torch = _torch()
            dev = self.arr.device
            # one buffer [2, nq, k]: ids block + distances block, so a sharded deployment exchanges results with a
            # single all-gather (distributed.all_gather_packed)
            packed = torch.empty((2, self.nq, k), dtype=torch.int32, device=dev)
            ids, dists = packed[0], packed[1].view(torch.float32)
            counts = torch.empty((self.nq,), dtype=torch.int32, device=dev)
            return ids, dists, counts, C.c_void_p(ids.data_ptr()), C.c_void_p(dists.data_ptr()), \
                C.c_void_p(counts.data_ptr())
        ids = np.empty((self.nq, k), np.uint32)
        dists = np.empty((self.nq, k), np.float32)
        counts = np.zeros((self.nq,), np.uint32)
        return ids, dists, counts, capi.np_ptr(ids), capi.np_ptr(dists), capi.np_ptr(counts)


def _dataset_ptr(x, dtype):
    """(pointer, memspace, keepalive, n, dim) of a 2-D dataset given as numpy or torch (CPU/CUDA)."""
    if _is_torch(x):
        torch = _torch()
        tdt = {np.float32: torch.float32, np.int8: torch.int8, np.uint8: torch.uint8, np.uint32: torch.int32,
               np.uint64: torch.int64}[dtype]
        t = x.to(tdt).contiguous() if x.dtype != tdt else x.contiguous()
        if t.is_cuda:
            # the library reads index arrays on its own stream: whatever produced them must be done
            torch.cuda.current_stream(t.device).synchronize()
            return C.c_void_p(t.data_ptr()), capi.DEVICE, t
        a = t.numpy()
        return capi.np_ptr(a), capi.HOST, a
    a = np.ascontiguousarray(x, dtype=dtype)
    return capi.np_ptr(a), capi.HOST, a


def results_to_lists(ids, dists, counts):
    """ids/dists/counts → Vec<Vec<(u32, f32)>> shape (the reference's NNResultsVector per query)."""
    if _is_torch(ids):
        ids, dists, counts = ids.cpu().numpy().view(np.uint32), dists.cpu().numpy(), counts.cpu().numpy()
    return [[(int(ids[i, j]), float(dists[i, j])) for j in range(int(counts[i]))] for i in range(ids.shape[0])]


@dataclass
class SearchParameters:
    """SearchParameters (src/searcher.rs:23-77), the fields the GPU path reads."""
    num_neighbors: Optional[int] = None
    pre_reordering_num_neighbors: Optional[int] = None

    def with_num_neighbors(self, k: int):
        self.num_neighbors = int(k)
        return self

    def with_pre_reordering_neighbors(self, n: int):
        self.pre_reordering_num_neighbors = int(n)
        return self


class _Handle:
    _destroy = None

    def __init__(self):
        self._h = C.c_void_p(None)

    def search_batched_with_params(self, queries, params, default_k: int = 10):
        """Searcher::search_batched_with_params (src/searcher.rs:164-169): one SearchParameters per query.  Queries
        that share their parameters go to the GPU as one batch; the result is one [(index, distance)] list per query,
        in query order.  queries.len() != params.len() → InvalidArgument (brute_force/searcher.rs:233-237)."""
        q = queries if _is_torch(queries) else np.asarray(queries, np.float32)
        if len(q) != len(params):
            raise ScannError(capi.INVALID_ARGUMENT, "Number of queries must match number of parameter sets")
        groups = {}
        for i, p in enumerate(params):
            key = (p.num_neighbors if p.num_neighbors is not None else default_k, p.pre_reordering_num_neighbors)
            groups.setdefault(key, []).append(i)
        out = [None] * len(params)
        for (k, pre), idxs in groups.items():
            sub = q[idxs]
            kw = {"pre_reorder_k": pre} if pre is not None and "pre_reorder_k" in self.search_batched.__code__.co_varnames \
                else {}
            ids, dists, counts = self.search_batched(sub, k, **kw)[:3]
            for j, lst in zip(idxs, results_to_lists(ids, dists, counts)):
                out[j] = lst
        return out

    def close(self):
        if self._h and self._h.value:
            getattr(capi.load(), self._destroy)(self._h)
            self._h = C.c_void_p(None)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class BruteForceSearcher(_Handle):
    """BruteForceSearcher<f32> (src/brute_force/searcher.rs:18-209)."""
    _destroy = "scann_bf_destroy"

    def __init__(self, dataset, distance_measure=DistanceMeasure.SquaredL2, device: int = 0, dim: Optional[int] = None):
        super().__init__()
        capi.require_gpu()
        ptr, ms, self._keep = _dataset_ptr(dataset, np.float32)
        shape = tuple(dataset.shape)
        n = int(shape[0])
        stride = int(shape[1]) if len(shape) > 1 else 0
        self.dimensionality = int(dim) if dim is not None else stride
        self.size = n
        self.distance_measure = DistanceMeasure(distance_measure)
        self.device = device
        capi.check(capi.load().scann_bf_create(ptr, n, self.dimensionality, stride, int(self.distance_measure), device,
                                               ms, C.byref(self._h)))
        self._keep = None

    def search_batched(self, queries, k: int):
        """search_batched (searcher.rs:170-208): returns (ids [nq,k], dists [nq,k], counts [nq])."""
        b = _Batch(queries, self.device)
        ids, dists, counts, pi, pd, pc = b.outputs(k)
        if b.nq == 0:
            return ids, dists, counts
        capi.check(capi.load().scann_bf_search(self._h, b.ptr, b.nq, b.dim, k, pi, pd, pc, b.memspace, b.stream))
        return ids, dists, counts

    def search(self, query, k: int):
        """search (searcher.rs:77-93) → [(index, distance)] sorted by distance."""
        ids, dists, counts = self.search_batched(np.asarray(query, np.float32)[None, :], k)
        return results_to_lists(ids, dists, counts)[0]

    def search_radius_batched(self, queries, radius: float, max_results: int = 1024, allow_truncated: bool = False):
        """search_radius (searcher.rs:142-167) for a batch → (ids [nq, max_results], dists, counts).  When more than
        max_results rows lie inside the radius for some query the library still writes every query's nearest
        max_results rows and reports RESOURCE_EXHAUSTED: raised here unless allow_truncated (then a warning)."""
        b = _Batch(queries, self.device)
        ids, dists, counts, pi, pd, pc = b.outputs(max_results)
        if b.nq:
            st = capi.load().scann_bf_search_radius(self._h, b.ptr, b.nq, b.dim, float(radius), max_results, pi, pd, pc,
                                                    b.memspace, b.stream)
            if st == capi.RESOURCE_EXHAUSTED and allow_truncated:
                import warnings
                warnings.warn("search_radius: results truncated to max_results for some query")
            else:
                capi.check(st)
        return ids, dists, counts

    def search_radius(self, query, radius: float, max_results: int = 1024):
        ids, dists, counts = self.search_radius_batched(np.asarray(query, np.float32)[None, :], radius, max_results)
        return results_to_lists(ids, dists, counts)[0]

    def path_stats(self):
        """(query chunks answered by the tcgen05 ranking path, by the CUDA-core path) since construction."""
        a, b = C.c_uint64(0), C.c_uint64(0)
        capi.check(capi.load().scann_bf_path_stats(self._h, C.byref(a), C.byref(b)))
        return a.value, b.value


@dataclass
class ScalarQuantizedConfig:
    """ScalarQuantizedConfig (scalar_quantized.rs:25-76); only the distance measure reaches the GPU path."""
    distance_measure: DistanceMeasure = DistanceMeasure.SquaredL2

    @staticmethod
    def squared_l2():
        return ScalarQuantizedConfig(DistanceMeasure.SquaredL2)

    @staticmethod
    def dot_product():
        return ScalarQuantizedConfig(DistanceMeasure.DotProduct)


def scalar_quantize(dataset, device: int = 0):
    """QuantizedDataset::from_dataset (src/quantization/scalar.rs:195-226) on the GPU.
    Returns (codes i8 [n, dim], cal4 = [min, max, scale, inv_scale])."""
    capi.require_gpu()
    if _is_torch(dataset) and dataset.is_cuda:
        torch = _torch()
        x = dataset.to(torch.float32).contiguous()
        n, dim = x.shape
        if n == 0:
            raise ScannError(capi.INVALID_ARGUMENT, "Cannot quantize empty dataset")
        codes = torch.empty((n, dim), dtype=torch.int8, device=x.device)
        cal = torch.empty(4, dtype=torch.float32, device=x.device)
        capi.check(capi.load().scann_sq8_quantize(C.c_void_p(x.data_ptr()), n, dim, dim, C.c_void_p(codes.data_ptr()),
                                                  C.c_void_p(cal.data_ptr()), device, capi.DEVICE))
        return codes, cal.cpu().numpy()
    x = capi.as_f32(dataset)
    n, dim = x.shape if x.ndim == 2 else (0, 0)
    if n == 0:
        raise ScannError(capi.INVALID_ARGUMENT, "Cannot quantize empty dataset")
    codes = np.empty((n, dim), np.int8)
    cal = np.empty(4, np.float32)
    capi.check(capi.load().scann_sq8_quantize(capi.np_ptr(x), n, dim, dim, capi.np_ptr(codes), capi.np_ptr(cal), device,
                                              capi.HOST))
    return codes, cal


class ScalarQuantizedBruteForceSearcher(_Handle):
    """ScalarQuantizedBruteForceSearcher (src/brute_force/scalar_quantized.rs:82-348)."""
    _destroy = "scann_sq8_destroy"

    def __init__(self, dataset, config: ScalarQuantizedConfig = ScalarQuantizedConfig(), device: int = 0):
        """new(&dataset, config) (:99-113): quantises the float dataset, then builds the searcher."""
        super().__init__()
        codes, cal = scalar_quantize(dataset, device)
        self._init_from(codes, float(cal[2]), config.distance_measure, device)
        self.calibration = cal

    @classmethod
    def from_quantized(cls, codes, scale: float, distance_measure=DistanceMeasure.SquaredL2, device: int = 0):
        """from_quantized (:116-129)."""
        self = cls.__new__(cls)
        _Handle.__init__(self)
        capi.require_gpu()
        self._init_from(codes, scale, distance_measure, device)
        self.calibration = None
        return self

    def _init_from(self, codes, scale, distance_measure, device):
        ptr, ms, keep = _dataset_ptr(codes, np.int8)
        n, dim = int(codes.shape[0]), int(codes.shape[1]) if len(codes.shape) > 1 else 0
        self.size, self.dimensionality, self.scale = n, dim, float(scale)
        self.distance_measure = DistanceMeasure(distance_measure)
        self.device = device
        capi.check(capi.load().scann_sq8_create(ptr, n, dim, C.c_float(scale), int(self.distance_measure), device, ms,
                                                C.byref(self._h)))

    def search_batched(self, queries, k: int):
        b = _Batch(queries, self.device)
        ids, dists, counts, pi, pd, pc = b.outputs(k)
        if b.nq == 0:
            return ids, dists, counts
        capi.check(capi.load().scann_sq8_search(self._h, b.ptr, b.nq, b.dim, k, pi, pd, pc, b.memspace, b.stream))
        return ids, dists, counts

    def search(self, query, k: int):
        ids, dists, counts = self.search_batched(np.asarray(query, np.float32)[None, :], k)
        return results_to_lists(ids, dists, counts)[0]

    def path_stats(self):
        """(query chunks answered by the tcgen05 ranking path, by the CUDA-core path) since construction."""
        a, b = C.c_uint64(0), C.c_uint64(0)
        capi.check(capi.load().scann_sq8_path_stats(self._h, C.byref(a), C.byref(b)))
        return a.value, b.value


class TreePartitioner(_Handle):
    """Query side of TreePartitioner (src/partitioning/tree_partitioner.rs:148-229) over given centres."""
    _destroy = "scann_part_destroy"

    def __init__(self, centers=None, device: int = 0):
        super().__init__()
        self.device = device
        self.num_partitions = 0
        if centers is not None:
            self.build_from_centers(centers)

    def build_from_centers(self, centers):
        capi.require_gpu()
        ptr, ms, keep = _dataset_ptr(centers, np.float32)
        K, dim = int(centers.shape[0]), int(centers.shape[1])
        capi.check(capi.load().scann_part_create(ptr, K, dim, self.device, ms, C.byref(self._h)))
        self.num_partitions, self.dimensionality = K, dim

    def partition(self, queries, num_partitions: int):
        """Partitioner::partition (:196-229) for a batch → (tokens [nq, L], distances [nq, L])."""
        if not (self._h and self._h.value):
            raise ScannError(capi.FAILED_PRECONDITION, "Partitioner not built")
        b = _Batch(queries, self.device)
        L = int(num_partitions)
        if b.device:
            torch = _torch()
            tokens = torch.empty((b.nq, L), dtype=torch.int32, device=b.arr.device)
            dists = torch.empty((b.nq, L), dtype=torch.float32, device=b.arr.device)
            pt, pd = C.c_void_p(tokens.data_ptr()), C.c_void_p(dists.data_ptr())
        else:
            tokens = np.empty((b.nq, L), np.uint32)
            dists = np.empty((b.nq, L), np.float32)
            pt, pd = capi.np_ptr(tokens), capi.np_ptr(dists)
        if b.nq and L:
            capi.check(capi.load().scann_part_select(self._h, b.ptr, b.nq, b.dim, L, pt, pd, b.memspace, b.stream))
        return tokens, dists


@dataclass
class KMeansTreeConfig:
    """KMeansTreeConfig (src/trees/kmeans_tree.rs:17-56); distance is SquaredL2 (search_leaves hard-wires it, :358-366)."""
    num_children: int = 100
    max_depth: int = 1
    min_leaf_size: int = 1
    kmeans_max_iterations: int = 20
    seed: Optional[int] = None


class KMeansTree(_Handle):
    """KMeansTree (src/trees/kmeans_tree.rs:154-395): hierarchical k-means partitioning.  Nodes are numbered in
    preorder; ``search_leaves`` returns leaf NODE ids (``export()`` maps them to datapoint indices)."""
    _destroy = "scann_kmtree_destroy"

    def __init__(self, config: KMeansTreeConfig = KMeansTreeConfig(), device: int = 0):
        super().__init__()
        self.config = config
        self.device = device

    def build(self, dataset):
        capi.require_gpu()
        if dataset is None or int(dataset.shape[0]) == 0:
            raise ScannError(capi.INVALID_ARGUMENT, "Cannot build tree from empty dataset")
        p_x, space, keep = _dataset_ptr(dataset, np.float32)
        n, dim = int(dataset.shape[0]), int(dataset.shape[1])
        c = self.config
        self.close()
        capi.check(capi.load().scann_kmtree_build(p_x, n, dim, dim, int(c.num_children), int(c.max_depth),
                                                  int(c.min_leaf_size), int(c.kmeans_max_iterations),
                                                  int(c.seed if c.seed is not None else 42), self.device, space,
                                                  C.byref(self._h)))
        del keep
        return self

    def build_from_arrays(self, centers, depth, child_begin, child_count, children):
        """a tree built elsewhere (flattened in preorder, see include/scann_b200.h)"""
        capi.require_gpu()
        centers = capi.as_f32(centers)
        u32 = lambda a: np.ascontiguousarray(a, np.uint32)
        depth, child_begin, child_count, children = u32(depth), u32(child_begin), u32(child_count), u32(children)
        self.close()
        capi.check(capi.load().scann_kmtree_create(capi.np_ptr(centers), capi.np_ptr(depth), capi.np_ptr(child_begin),
                                                   capi.np_ptr(child_count), capi.np_ptr(children) if len(children) else None,
                                                   len(depth), len(children), centers.shape[1], self.device,
                                                   C.byref(self._h)))
        return self

    def info(self):
        v = [C.c_size_t(0) for _ in range(5)]
        capi.check(capi.load().scann_kmtree_info(self._h, *[C.byref(a) for a in v]))
        return dict(zip(("num_nodes", "num_leaves", "num_child_entries", "num_points", "dim"), (a.value for a in v)))

    def num_leaves(self) -> int:
        return self.info()["num_leaves"] if self._h else 0

    def size(self) -> int:
        return self.info()["num_points"] if self._h else 0

    def export(self):
        i = self.info()
        out = {
            "centers": np.empty((i["num_nodes"], i["dim"]), np.float32), "depth": np.empty(i["num_nodes"], np.uint32),
            "child_begin": np.empty(i["num_nodes"], np.uint32), "child_count": np.empty(i["num_nodes"], np.uint32),
            "children": np.empty(i["num_child_entries"], np.uint32), "leaf_begin": np.zeros(i["num_nodes"], np.uint32),
            "leaf_count": np.zeros(i["num_nodes"], np.uint32), "leaf_points": np.empty(i["num_points"], np.uint32),
        }
        capi.check(capi.load().scann_kmtree_export(self._h, *[capi.np_ptr(out[k]) for k in (
            "centers", "depth", "child_begin", "child_count", "children", "leaf_begin", "leaf_count", "leaf_points")]))
        return out

    def search_leaves(self, queries, k: int):
        """KMeansTree::search_leaves (:302-319) for a batch → (leaf node ids [nq,k], dists, depths, counts)"""
        if not self._h:
            raise ScannError(capi.FAILED_PRECONDITION, "Tree not built")
        b = _Batch(queries, self.device)
        kk = max(int(k), 1)
        if b.memspace == capi.DEVICE:
            torch = _torch()
            dev = queries.device
            nodes = torch.empty((b.nq, kk), dtype=torch.int32, device=dev)
            dists = torch.empty((b.nq, kk), dtype=torch.float32, device=dev)
            depths = torch.empty((b.nq, kk), dtype=torch.int32, device=dev)
            counts = torch.empty((b.nq,), dtype=torch.int32, device=dev)
            ptrs = [C.c_void_p(t.data_ptr()) for t in (nodes, dists, depths, counts)]
        else:
            nodes = np.empty((b.nq, kk), np.uint32)
            dists = np.empty((b.nq, kk), np.float32)
            depths = np.empty((b.nq, kk), np.uint32)
            counts = np.empty((b.nq,), np.uint32)
            ptrs = [capi.np_ptr(a) for a in (nodes, dists, depths, counts)]
        capi.check(capi.load().scann_kmtree_search_leaves(self._h, b.ptr, b.nq, b.dim, int(k), *ptrs, b.memspace, b.stream))
        return nodes[:, :k], dists[:, :k], depths[:, :k], counts


@dataclass
class AsymmetricHasherConfig:
    """AsymmetricHasherConfig (src/hashes/hasher.rs:19-69); the GPU path is the 16-code LUT16 variant."""
    num_codes: int = 16
    num_subspaces: int = 8
    seed: Optional[int] = None


@dataclass
class TreeXHybridConfig:
    """TreeXHybridConfig (src/tree_x_hybrid/mod.rs:23-78).  `distance_measure` is the reorder measure —
    the reference hard-wires SquaredL2 (:124); SURVEY §5 adds the setter config C3 needs."""
    num_partitions: int = 100
    partitions_to_search: int = 10
    hash_config: AsymmetricHasherConfig = field(default_factory=AsymmetricHasherConfig)
    use_residuals: bool = True
    pre_reorder_multiplier: float = 3.0
    distance_measure: DistanceMeasure = DistanceMeasure.SquaredL2

    def pre_reorder_k(self, k: int) -> int:
        # (k as f32 * self.config.pre_reorder_multiplier) as usize  (tree_x_hybrid/mod.rs:263)
        v = np.float32(k) * np.float32(self.pre_reorder_multiplier)
        return max(int(v), 0)


def _filter_table(allowed, filter_of_query, b: "_Batch"):
    """Packs per-query restrict filters for scann_treeah_search_filtered where the batch `b` lives → (bitmap pointer,
    num_filters, num_ids, filter_of_query pointer, arrays to keep alive for the call)."""
    nq = b.nq
    if len(allowed.shape) not in (1, 2):
        raise ScannError(capi.INVALID_ARGUMENT, "allowed must be [num_ids] or [num_filters, num_ids]")
    one = len(allowed.shape) == 1
    F = 1 if one else int(allowed.shape[0])
    num_ids = int(allowed.shape[-1])
    if filter_of_query is None:
        if not one and F != nq:
            raise ScannError(capi.INVALID_ARGUMENT,
                             f"filter_of_query is needed: {F} filters for {nq} queries")
        filter_of_query = np.zeros(nq, np.uint32) if one else np.arange(nq, dtype=np.uint32)
    if int(filter_of_query.shape[0]) != nq or len(filter_of_query.shape) != 1:
        raise ScannError(capi.INVALID_ARGUMENT, f"filter_of_query must hold one row index per query ({nq})")
    if b.device:
        torch = _torch()
        dev = b.arr.device
        m = (allowed if _is_torch(allowed) else torch.from_numpy(np.asarray(allowed))).to(dev).reshape(F, num_ids)
        m = m.to(torch.bool)
        pad = (-num_ids) % 8
        if pad:
            m = torch.nn.functional.pad(m, (0, pad))
        shifts = torch.arange(8, device=dev, dtype=torch.uint8)
        bits = (m.reshape(F, -1, 8).to(torch.uint8) << shifts).sum(-1, dtype=torch.uint8).contiguous()
        fq = filter_of_query if _is_torch(filter_of_query) else torch.from_numpy(np.asarray(filter_of_query))
        fq = fq.to(device=dev, dtype=torch.int64).to(torch.int32).contiguous()  # u32 bit patterns
        return C.c_void_p(bits.data_ptr()), F, num_ids, C.c_void_p(fq.data_ptr()), (bits, fq)
    m = allowed.cpu().numpy() if _is_torch(allowed) else np.asarray(allowed)
    bits = np.ascontiguousarray(np.packbits(m.reshape(F, num_ids).astype(bool), axis=1, bitorder="little"))
    fq = filter_of_query.cpu().numpy() if _is_torch(filter_of_query) else np.asarray(filter_of_query)
    fq = np.ascontiguousarray(fq.astype(np.int64).astype(np.uint32))
    return capi.np_ptr(bits), F, num_ids, capi.np_ptr(fq), (bits, fq)


class TreeXHybridSearcher(_Handle):
    """TreeXHybridSearcher (src/tree_x_hybrid/mod.rs:93-380) with the LUT16 scan.

    ``build_from_index`` takes the arrays ``build`` (:131-209) leaves behind: centres, the residual codebook
    [S,16,ds], PackedCodes4Bit rows grouped by partition, their datapoint ids, partition offsets and the
    raw dataset.  (Index training is an index-build concern — see ``indexing.py``.)"""
    _destroy = "scann_treeah_destroy"

    def __init__(self, config: TreeXHybridConfig = TreeXHybridConfig(), device: int = 0):
        super().__init__()
        self.config = config
        self.device = device
        self.num_datapoints = 0
        self.dimensionality = 0

    def build_from_index(self, centers, codebook, packed, ids, part_offsets, raw=None, raw_by_position: bool = False,
                         borrow_raw: bool = False):
        """raw_by_position: raw holds one row per index row in the order of packed/ids (a shard keeps its own rows, ids
        stay global); borrow_raw: CUDA tensors only — raw is not copied, this object keeps the tensor alive."""
        capi.require_gpu()
        if packed.shape[0] == 0:
            raise ScannError(capi.INVALID_ARGUMENT, "Cannot build from empty dataset")
        K, dim = int(centers.shape[0]), int(centers.shape[1])
        S = int(codebook.shape[0])
        if int(codebook.shape[1]) != 16:
            raise ScannError(capi.UNIMPLEMENTED, "the GPU AH path is LUT16: num_codes must be 16")
        if dim % S != 0:
            raise ScannError(capi.INVALID_ARGUMENT,
                             f"Dimensionality {dim} must be divisible by num_subspaces {S}")
        n = int(packed.shape[0])
        p_c, ms_c, k1 = _dataset_ptr(centers, np.float32)
        p_cb, ms_cb, k2 = _dataset_ptr(codebook, np.float32)
        p_pk, ms_pk, k3 = _dataset_ptr(packed, np.uint8)
        p_id, ms_id, k4 = _dataset_ptr(ids, np.uint32)
        p_off, ms_off, k5 = _dataset_ptr(part_offsets, np.uint64)
        spaces = {ms_c, ms_cb, ms_pk, ms_id, ms_off}
        p_raw, num_raw, stride = None, 0, 0
        if raw is not None:
            p_raw, ms_raw, k6 = _dataset_ptr(raw, np.float32)
            num_raw, stride = int(raw.shape[0]), int(raw.shape[1])
            spaces.add(ms_raw)
        if len(spaces) != 1:
            raise ScannError(capi.INVALID_ARGUMENT, "index arrays must all be host or all be device resident")
        self.close()
        space = spaces.pop()
        flags = (capi.TREEAH_RAW_BY_POSITION if raw_by_position and raw is not None else 0) | \
                (capi.TREEAH_BORROW_RAW if borrow_raw and raw is not None and space == capi.DEVICE else 0)
        self._raw_keep = k6 if flags & capi.TREEAH_BORROW_RAW else None
        capi.check(capi.load().scann_treeah_create_ex(p_c, K, dim, p_cb, S, p_pk, p_id, p_off, n, p_raw, num_raw, stride,
                                                      int(self.config.use_residuals),
                                                      int(self.config.distance_measure), flags, self.device, space,
                                                      C.byref(self._h)))
        self.num_datapoints, self.dimensionality, self.num_partitions, self.num_subspaces = n, dim, K, S
        return self

    def build(self, dataset, train_rows: int = 1_000_000, kmeans_iters: int = 20, seed: int = 7, keep_raw: bool = True):
        """TreeXHybridSearcher::build (:131-209) inside the library (scann_treeah_build, csrc/build_index.cu): k-means
        partition centres, residual LUT16 codebook, exact assignment / encode / packing.  dataset: numpy or torch
        (CPU/CUDA) [n, dim] f32."""
        capi.require_gpu()
        if dataset is None or int(dataset.shape[0]) == 0:
            raise ScannError(capi.INVALID_ARGUMENT, "Cannot build from empty dataset")
        p_x, space, keep = _dataset_ptr(dataset, np.float32)
        n, dim = int(dataset.shape[0]), int(dataset.shape[1])
        S = int(self.config.hash_config.num_subspaces)
        self.close()
        capi.check(capi.load().scann_treeah_build(p_x, n, dim, dim, int(self.config.num_partitions), S, int(train_rows),
                                                  int(kmeans_iters), int(seed), int(self.config.use_residuals),
                                                  int(self.config.distance_measure), int(keep_raw), self.device, space,
                                                  C.byref(self._h)))
        del keep
        self.num_datapoints, self.dimensionality, self.num_subspaces = n, dim, S
        self.num_partitions = min(int(self.config.num_partitions), n if train_rows <= 0 else min(n, int(train_rows)))
        return self

    def search_batched(self, queries, k: int, partitions_to_search: Optional[int] = None,
                       pre_reorder_k: Optional[int] = None, want_candidates: bool = False):
        return self._search(queries, k, partitions_to_search, pre_reorder_k, want_candidates)

    def search_batched_per_query(self, queries, k, pre_reorder_k=None, partitions_to_search=None,
                                 want_candidates: bool = False):
        """search_batched with per-query parameters in one GPU call (scann_treeah_search_with_params).  `k`,
        `pre_reorder_k` and `partitions_to_search` are each an int or one value per query (numpy, or torch on the
        device path).  pre_reorder_k None: config.pre_reorder_k(k_q) for every query; partitions_to_search None: the
        config's.  Row q is bit for bit what search_batched returns for query q alone with its own values.  The
        outputs have the row length of the largest k (the candidates: of the largest pre_reorder_k), padded beyond
        counts[q] with id 0xFFFFFFFF and distance +inf.  A per-query torch array is reduced to its maximum on the
        host, which synchronises with its stream."""
        return self._search(queries, k, partitions_to_search, pre_reorder_k, want_candidates, per_query=True)

    def search_batched_with_params(self, queries, params, default_k: int = 10):
        """Searcher::search_batched_with_params (src/searcher.rs:164-169): one SearchParameters per query, the whole
        batch in one GPU call.  k_q = num_neighbors (default_k when unset); R_q = pre_reordering_num_neighbors
        (config.pre_reorder_k(k_q) when unset).  The result is one [(index, distance)] list per query, in query order.
        queries.len() != params.len() → InvalidArgument (brute_force/searcher.rs:233-237)."""
        q = queries if _is_torch(queries) else np.asarray(queries, np.float32)
        if len(q) != len(params):
            raise ScannError(capi.INVALID_ARGUMENT, "Number of queries must match number of parameter sets")
        if len(params) == 0:
            return []
        ks = [p.num_neighbors if p.num_neighbors is not None else default_k for p in params]
        rs = [p.pre_reordering_num_neighbors if p.pre_reordering_num_neighbors is not None
              else self.config.pre_reorder_k(kq) for p, kq in zip(params, ks)]
        ids, dists, counts = self.search_batched_per_query(q, np.array(ks, np.int64), np.array(rs, np.int64))
        return results_to_lists(ids, dists, counts)

    def _query_params(self, b: "_Batch", k, partitions_to_search, pre_reorder_k):
        """(batch maximum, per-query u32 array where the batch lives or None) for k, L and R."""
        torch = _torch() if b.device else None

        def per_query(v, name):
            if _is_torch(v) and v.dim() == 0 or not _is_torch(v) and np.ndim(v) == 0:
                return v, None
            if b.device:
                a = (v if _is_torch(v) else torch.from_numpy(np.asarray(v))).to(device=b.arr.device, dtype=torch.int64)
            else:
                a = np.asarray(v.cpu().numpy() if _is_torch(v) else v).astype(np.int64)
            if tuple(a.shape) != (b.nq,):
                raise ScannError(capi.INVALID_ARGUMENT, f"{name} must hold one value per query ({b.nq})")
            return None, a

        def finish(v, a):
            if a is None:
                return int(v), None
            mx = max(int(a.max()), 0) if b.nq else 0
            return mx, (a.to(torch.int32).contiguous() if b.device else np.ascontiguousarray(a.astype(np.uint32)))

        k, ka = per_query(k, "k")
        L, La = per_query(partitions_to_search if partitions_to_search is not None
                          else self.config.partitions_to_search, "partitions_to_search")
        if pre_reorder_k is not None:
            R, Ra = per_query(pre_reorder_k, "pre_reorder_k")
        elif ka is None:
            R, Ra = self.config.pre_reorder_k(int(k)), None
        else:  # (k as f32 * multiplier) as usize, per query
            mult = np.float32(self.config.pre_reorder_multiplier)
            R, Ra = None, ((ka.to(torch.float32) * float(mult)).to(torch.int64).clamp(min=0) if b.device
                           else np.maximum((ka.astype(np.float32) * mult).astype(np.int64), 0))
        return finish(k, ka), finish(L, La), finish(R, Ra)

    def _search(self, queries, k, partitions_to_search, pre_reorder_k, want_candidates, allowed=None,
                filter_of_query=None, per_query=False):
        if not (self._h and self._h.value):
            raise ScannError(capi.FAILED_PRECONDITION, "searcher not built")
        b = _Batch(queries, self.device)
        if per_query:
            (k, ka), (L, La), (R, Ra) = self._query_params(b, k, partitions_to_search, pre_reorder_k)
        else:
            L = int(partitions_to_search if partitions_to_search is not None else self.config.partitions_to_search)
            R = int(pre_reorder_k if pre_reorder_k is not None else self.config.pre_reorder_k(k))
        ids, dists, counts, pi, pd, pc = b.outputs(k)
        cand = None
        pci = pcd = pcc = None
        if want_candidates:
            if b.device:
                torch = _torch()
                ci = torch.empty((b.nq, max(R, 1)), dtype=torch.int32, device=b.arr.device)
                cd = torch.empty((b.nq, max(R, 1)), dtype=torch.float32, device=b.arr.device)
                cc = torch.zeros((b.nq,), dtype=torch.int32, device=b.arr.device)
                pci, pcd, pcc = C.c_void_p(ci.data_ptr()), C.c_void_p(cd.data_ptr()), C.c_void_p(cc.data_ptr())
            else:
                ci = np.full((b.nq, max(R, 1)), 0xFFFFFFFF, np.uint32)
                cd = np.full((b.nq, max(R, 1)), np.inf, np.float32)
                cc = np.zeros((b.nq,), np.uint32)
                pci, pcd, pcc = capi.np_ptr(ci), capi.np_ptr(cd), capi.np_ptr(cc)
            cand = (ci, cd, cc)
        if b.nq and per_query:
            ptrs = [None if a is None else C.c_void_p(a.data_ptr()) if b.device else capi.np_ptr(a)
                    for a in (La, Ra, ka)]
            capi.check(capi.load().scann_treeah_search_with_params(self._h, b.ptr, b.nq, b.dim, L, R, k, *ptrs, pi, pd,
                                                                   pc, pci, pcd, pcc, b.memspace, b.stream))
        elif b.nq and allowed is None:
            capi.check(capi.load().scann_treeah_search(self._h, b.ptr, b.nq, b.dim, L, R, k, pi, pd, pc, pci, pcd, pcc,
                                                       b.memspace, b.stream))
        elif b.nq:
            bits, F, num_ids, fq, keep = _filter_table(allowed, filter_of_query, b)
            capi.check(capi.load().scann_treeah_search_filtered(self._h, b.ptr, b.nq, b.dim, L, R, k, bits, F, num_ids,
                                                                fq, pi, pd, pc, pci, pcd, pcc, b.memspace, b.stream))
            del keep
        if want_candidates:
            return ids, dists, counts, cand
        return ids, dists, counts

    def search(self, query, k: int):
        """search (:240-242) → [(index, distance)]"""
        ids, dists, counts = self.search_batched(np.asarray(query, np.float32)[None, :], k)
        return results_to_lists(ids, dists, counts)[0]

    def set_filter(self, allowed=None):
        """RestrictFilter for the following searches (scann_treeah_set_filter): `allowed` = boolean mask over datapoint
        ids (numpy or torch, True = may be returned) or None to clear."""
        if allowed is None:
            capi.check(capi.load().scann_treeah_set_filter(self._h, None, 0, capi.HOST))
            return
        m = allowed.cpu().numpy() if _is_torch(allowed) else np.asarray(allowed)
        bits = np.packbits(m.astype(bool), bitorder="little")
        capi.check(capi.load().scann_treeah_set_filter(self._h, capi.np_ptr(bits), int(m.size), capi.HOST))

    def search_with_filter(self, queries, k: int, allowed=None, filter_of_query=None,
                           partitions_to_search: Optional[int] = None, pre_reorder_k: Optional[int] = None,
                           want_candidates: bool = False):
        """search_with_filter (tree_x_hybrid/mod.rs:245-294): search_batched restricted to the allowed datapoints, with
        filters that belong to this call only (scann_treeah_search_filtered; safe to call from several threads).

        `allowed`: boolean mask over datapoint ids (True = may be returned), numpy or torch.  1-D [num_ids]: one filter
        for the whole batch.  2-D [F, num_ids]: F filters, query q uses row filter_of_query[q] (length nq; may be
        omitted when F == nq: query q uses row q).  None: the plain search.  CUDA queries take the device path and
        the masks are packed on the device.  Refused while a handle-wide filter (set_filter) is set."""
        if allowed is None:
            if filter_of_query is not None:
                raise ScannError(capi.INVALID_ARGUMENT, "filter_of_query without allowed")
            return self.search_batched(queries, k, partitions_to_search, pre_reorder_k, want_candidates)
        return self._search(queries, k, partitions_to_search, pre_reorder_k, want_candidates, allowed, filter_of_query)

    def partition_tokens(self, queries, partitions_to_search: Optional[int] = None):
        """The partition stage alone (scann_treeah_partition) for a slice of a batch: torch CUDA queries [m, dim] →
        tokens [m, L] int32 CUDA tensor."""
        b = _Batch(queries, self.device)
        torch = _torch()
        L = int(partitions_to_search if partitions_to_search is not None else self.config.partitions_to_search)
        tok = torch.empty((b.nq, L), dtype=torch.int32, device=b.arr.device)
        if b.nq:
            capi.check(capi.load().scann_treeah_partition(self._h, b.ptr, b.nq, b.dim, L, C.c_void_p(tok.data_ptr()),
                                                          b.stream))
        return tok

    def search_begin(self, queries, k: int, partitions_to_search: Optional[int] = None,
                     pre_reorder_k: Optional[int] = None, tokens=None):
        """First half of the split search for a sharded index (scann_treeah_search_begin): torch CUDA queries →
        tau [nq] f32 CUDA tensor, the bounds proved by every query's closest leaf on this shard (+inf when it lives
        elsewhere).  Min-reduce tau over the shards and pass it to search_end()."""
        if not (self._h and self._h.value):
            raise ScannError(capi.FAILED_PRECONDITION, "searcher not built")
        b = _Batch(queries, self.device)
        if not b.device or b.nq == 0:
            raise ScannError(capi.INVALID_ARGUMENT, "the split search takes a non-empty batch of CUDA queries")
        torch = _torch()
        L = int(partitions_to_search if partitions_to_search is not None else self.config.partitions_to_search)
        R = int(pre_reorder_k if pre_reorder_k is not None else self.config.pre_reorder_k(k))
        tau = torch.empty((b.nq,), dtype=torch.float32, device=b.arr.device)
        ptok = None
        if tokens is not None:
            tokens = tokens.contiguous()
            assert tuple(tokens.shape) == (b.nq, L) and tokens.dtype == torch.int32 and tokens.is_cuda
            ptok = C.c_void_p(tokens.data_ptr())
        capi.check(capi.load().scann_treeah_search_begin(self._h, b.ptr, b.nq, b.dim, L, R, k, ptok,
                                                         C.c_void_p(tau.data_ptr()), b.stream))
        self._split = (b, k, tokens)  # keeps the query and token tensors alive until search_end
        return tau

    def search_end(self, tau=None):
        """Second half (scann_treeah_search_end) → (ids, dists, counts) torch CUDA tensors."""
        b, k, _tokens = self._split
        ids, dists, counts, pi, pd, pc = b.outputs(k)
        pt = C.c_void_p(tau.data_ptr()) if tau is not None else None
        try:
            capi.check(capi.load().scann_treeah_search_end(self._h, pt, pi, pd, pc, b.stream))
        finally:
            self._split = None
        return ids, dists, counts

    def search_abort(self):
        """Gives the handle back after a search_begin whose search_end will not be called (scann_treeah_search_abort)."""
        if self._h and self._h.value:
            capi.check(capi.load().scann_treeah_search_abort(self._h))
        self._split = None

    def set_profiling(self, enable: bool):
        capi.check(capi.load().scann_treeah_set_profiling(self._h, int(enable)))

    def get_profile(self):
        """→ ({'partition','worklist','scan','merge'} device milliseconds since the last call, kernel launches)"""
        ms = (C.c_double * 4)()
        n = C.c_uint64(0)
        capi.check(capi.load().scann_treeah_get_profile(self._h, ms, C.byref(n)))
        return dict(zip(("partition", "worklist", "scan", "merge"), [float(v) for v in ms])), int(n.value)

    def path_stats(self):
        """(query chunks scanned by the tensor-core LUT16 kernel, by the register-LUT kernel) since construction."""
        a, b = C.c_uint64(0), C.c_uint64(0)
        capi.check(capi.load().scann_treeah_path_stats(self._h, C.byref(a), C.byref(b)))
        return a.value, b.value

    def tc_profile(self):
        """→ {'lut_ms', 'scan_ms', 'launches', 'pair_points'} of the tensor-core scan while profiling is on (call before
        get_profile, which resets)."""
        a, b, n, pp = C.c_double(0), C.c_double(0), C.c_uint64(0), C.c_uint64(0)
        capi.check(capi.load().scann_treeah_tc_profile(self._h, C.byref(a), C.byref(b), C.byref(n), C.byref(pp)))
        return {"lut_ms": a.value, "scan_ms": b.value, "launches": int(n.value), "pair_points": int(pp.value)}

    def last_scan_bytes(self):
        by, pr = C.c_uint64(0), C.c_uint64(0)
        capi.check(capi.load().scann_treeah_last_scan_bytes(self._h, C.byref(by), C.byref(pr)))
        return int(by.value), int(pr.value)


class AsymmetricHasher(TreeXHybridSearcher):
    """Flat AsymmetricHasher (src/hashes/hasher.rs:75-259) on the LUT16 path: one partition holding every
    point, no residuals.  search = approximate LUT16 distances; search_with_reordering re-ranks
    `pre_reorder_k` candidates by exact SquaredL2 (hard-coded in the reference, hasher.rs:208)."""

    def __init__(self, config: AsymmetricHasherConfig = AsymmetricHasherConfig(num_codes=16), device: int = 0):
        super().__init__(TreeXHybridConfig(num_partitions=1, partitions_to_search=1, hash_config=config,
                                           use_residuals=False, distance_measure=DistanceMeasure.SquaredL2), device)
        self._with_raw = None

    def build_from_index(self, codebook, packed, raw=None):
        n = int(packed.shape[0])
        dim = int(codebook.shape[0]) * int(codebook.shape[2])
        centers = np.zeros((1, dim), np.float32)
        ids = np.arange(n, dtype=np.uint32)
        off = np.array([0, n], np.uint64)
        self._raw = raw
        self._args = (centers, codebook, packed, ids, off)
        self._have = None
        return self

    def _ensure(self, with_raw: bool):
        if self._have is not with_raw:
            centers, cb, packed, ids, off = self._args
            if with_raw and self._raw is None:
                raise ScannError(capi.FAILED_PRECONDITION, "Dataset not stored")
            TreeXHybridSearcher.build_from_index(self, centers, cb, packed, ids, off, self._raw if with_raw else None)
            self._have = with_raw

    # pre_reordering_num_neighbors means something else here (search vs search_with_reordering): queries that share
    # their parameters go to the GPU as one batch
    search_batched_with_params = _Handle.search_batched_with_params

    def search_batched(self, queries, k: int):
        self._ensure(False)
        return TreeXHybridSearcher.search_batched(self, queries, k, 1, k)

    def search_with_reordering(self, queries, k: int, pre_reorder_k: int):
        self._ensure(True)
        return TreeXHybridSearcher.search_batched(self, queries, k, 1, pre_reorder_k)


class LeafScanSearcher(_Handle):
    """The Scann façade's tree modes that score every member of the probed leaves (src/scann.rs:215-294) over
    prebuilt index arrays (include/scann_b200.h scann_ivf_*):
      search_partitioned ← Scann::search_partitioned: exact distances inside the L closest leaves;
      search_tree_ah     ← Scann::search_tree_ah ("variant B"): one f32 LookupTable of the query over byte codes
                           indexed by datapoint id; K = 1 is the scoring of AsymmetricHasher::search.
    `reorder` re-scores the k results exactly (ReorderingHelper::reorder as Scann::search_impl applies it)."""
    _destroy = "scann_ivf_destroy"

    def __init__(self, centers, ids, part_offsets, dataset=None, codebook=None, codes_by_id=None, device: int = 0):
        super().__init__()
        capi.require_gpu()
        self.device = device
        on_gpu = any(_is_torch(a) and a.is_cuda for a in (centers, ids, part_offsets, dataset, codebook, codes_by_id)
                     if a is not None)

        def conv(a, dtype):
            if a is None:
                return None, None
            if on_gpu:
                torch = _torch()
                tdt = {np.float32: torch.float32, np.uint8: torch.uint8, np.uint32: torch.int32, np.uint64: torch.int64}[dtype]
                t = a if _is_torch(a) else torch.as_tensor(np.ascontiguousarray(a).view(
                    {np.uint32: np.int32, np.uint64: np.int64}.get(dtype, dtype)))
                t = t.to(device=f"cuda:{device}", dtype=tdt).contiguous()
                return C.c_void_p(t.data_ptr()), t
            arr = np.ascontiguousarray(a.cpu().numpy() if _is_torch(a) else a, dtype=dtype)
            return capi.np_ptr(arr), arr

        K, dim = int(centers.shape[0]), int(centers.shape[1])
        n = int(ids.shape[0])
        pc, k1 = conv(centers, np.float32)
        pi, k2 = conv(ids, np.uint32)
        po, k3 = conv(part_offsets, np.uint64)
        pr, k4 = conv(dataset, np.float32)
        pcb, k5 = conv(codebook, np.float32)
        pcd, k6 = conv(codes_by_id, np.uint8)
        num_raw = int(dataset.shape[0]) if dataset is not None else (int(codes_by_id.shape[0]) if codes_by_id is not None else 0)
        stride = int(dataset.shape[1]) if dataset is not None else dim
        S = int(codebook.shape[0]) if codebook is not None else 0
        Cc = int(codebook.shape[1]) if codebook is not None else 0
        if on_gpu:
            _torch().cuda.current_stream(device).synchronize()
        self.dimensionality, self.num_partitions, self.size = dim, K, n
        capi.check(capi.load().scann_ivf_create(pc, K, dim, pi, po, n, pr, num_raw, stride, pcb, S, Cc, pcd, device,
                                                capi.DEVICE if on_gpu else capi.HOST, C.byref(self._h)))

    def _search(self, mode, queries, k, L, measure, reorder):
        b = _Batch(queries, self.device)
        ids, dists, counts, pi, pd, pc = b.outputs(k)
        if b.nq:
            capi.check(capi.load().scann_ivf_search(self._h, mode, b.ptr, b.nq, b.dim, int(L), int(k), int(measure),
                                                    -1 if reorder is None else int(reorder), pi, pd, pc, b.memspace,
                                                    b.stream))
        return ids, dists, counts

    def search_partitioned(self, queries, k: int, partitions_to_search: int,
                           distance_measure=DistanceMeasure.SquaredL2, reorder=None):
        return self._search(0, queries, k, partitions_to_search, DistanceMeasure(distance_measure), reorder)

    def search_tree_ah(self, queries, k: int, partitions_to_search: int, reorder=None):
        return self._search(1, queries, k, partitions_to_search, DistanceMeasure.SquaredL2, reorder)

    def search_with_reordering(self, queries, k: int, pre_reorder_k: int, partitions_to_search: int = 1):
        """AsymmetricHasher::search_with_reordering (hashes/hasher.rs:188-229) on a K = 1 index: the pre_reorder_k
        best by the f32 LUT, exact SqL2 (hard-wired, :208) re-rank, first k."""
        ids, dists, counts = self._search(1, queries, max(int(pre_reorder_k), 1), partitions_to_search,
                                          DistanceMeasure.SquaredL2, DistanceMeasure.SquaredL2)
        if _is_torch(counts):
            return ids[:, :k].contiguous(), dists[:, :k].contiguous(), counts.clamp(max=k)
        return np.ascontiguousarray(ids[:, :k]), np.ascontiguousarray(dists[:, :k]), np.minimum(counts, k)


def merge_topk(ids_parts, dists_parts, device: int = 0):
    """k-way merge of per-shard results [parts, nq, k] by (distance, id) (SURVEY §8e)."""
    capi.require_gpu()
    if _is_torch(ids_parts) and ids_parts.is_cuda:
        torch = _torch()
        parts, nq, k = ids_parts.shape
        ii = ids_parts.contiguous()
        dd = dists_parts.to(torch.float32).contiguous()
        oi = torch.empty((nq, k), dtype=torch.int32, device=ii.device)
        od = torch.empty((nq, k), dtype=torch.float32, device=ii.device)
        oc = torch.empty((nq,), dtype=torch.int32, device=ii.device)
        capi.check(capi.load().scann_merge_topk(C.c_void_p(ii.data_ptr()), C.c_void_p(dd.data_ptr()), parts, nq, k,
                                                C.c_void_p(oi.data_ptr()), C.c_void_p(od.data_ptr()),
                                                C.c_void_p(oc.data_ptr()), ii.device.index or 0, capi.DEVICE,
                                                _stream_ptr(ii.device.index or 0)))
        return oi, od, oc
    ii = np.ascontiguousarray(ids_parts, np.uint32)
    dd = capi.as_f32(dists_parts)
    parts, nq, k = ii.shape
    oi, od, oc = np.empty((nq, k), np.uint32), np.empty((nq, k), np.float32), np.zeros(nq, np.uint32)
    capi.check(capi.load().scann_merge_topk(capi.np_ptr(ii), capi.np_ptr(dd), parts, nq, k, capi.np_ptr(oi),
                                            capi.np_ptr(od), capi.np_ptr(oc), device, capi.HOST, None))
    return oi, od, oc


def merge_topk_packed(gathered, device: int = 0):
    """merge_topk over ONE gathered CUDA buffer [parts, 2, nq, k] int32 (ids block + distance bits block per part)."""
    capi.require_gpu()
    torch = _torch()
    parts, two, nq, k = gathered.shape
    assert two == 2 and gathered.is_cuda and gathered.dtype == torch.int32 and gathered.is_contiguous()
    oi = torch.empty((nq, k), dtype=torch.int32, device=gathered.device)
    od = torch.empty((nq, k), dtype=torch.float32, device=gathered.device)
    oc = torch.empty((nq,), dtype=torch.int32, device=gathered.device)
    dev = gathered.device.index or 0
    capi.check(capi.load().scann_merge_topk_packed(C.c_void_p(gathered.data_ptr()), parts, nq, k,
                                                   C.c_void_p(oi.data_ptr()), C.c_void_p(od.data_ptr()),
                                                   C.c_void_p(oc.data_ptr()), dev, _stream_ptr(dev)))
    return oi, od, oc


# ----------------------------------------------------------------------------------------- taps
def lut16_build(codebook, queries, centroids=None, device: int = 0):
    """Parity tap → (lut8 [nq, S, 16] u8, bias [nq], mult [nq])."""
    capi.require_gpu()
    cb, q = capi.as_f32(codebook), capi.as_f32(queries)
    S, ncodes, ds = cb.shape
    assert ncodes == 16
    nq = q.shape[0]
    cen = capi.as_f32(centroids) if centroids is not None else None
    lut8 = np.empty((nq, S, 16), np.uint8)
    bias, mult = np.empty(nq, np.float32), np.empty(nq, np.float32)
    capi.check(capi.load().scann_lut16_build(capi.np_ptr(cb), S, ds, capi.np_ptr(q), nq, capi.np_ptr(cen),
                                             capi.np_ptr(lut8), capi.np_ptr(bias), capi.np_ptr(mult), device, capi.HOST))
    return lut8, bias, mult


def lut16_scan(packed, S: int, lut8, device: int = 0):
    """Parity tap → u32 sums [n] of one u8 table over PackedCodes4Bit rows."""
    capi.require_gpu()
    pk = np.ascontiguousarray(packed, np.uint8)
    l8 = np.ascontiguousarray(lut8, np.uint8)
    n = pk.shape[0]
    sums = np.empty(n, np.uint32)
    capi.check(capi.load().scann_lut16_scan(capi.np_ptr(pk), n, S, capi.np_ptr(l8), capi.np_ptr(sums), device, capi.HOST))
    return sums


def tc_scores(queries, rows, scale: float = 1.0, want_norm: bool = True, thr=None, cap: int = 0, device: int = 0):
    """Parity tap of the tcgen05 ranking contraction (csrc/tc_gemm.cu): v = hx - bf16(q)·bf16(x).
    rows f32 or int8 [n, dim]; → dense [nq, n] f32, or with thr [nq]: (cand [nq, cap] u64 = score key << 32 | row, counts [nq])."""
    capi.require_gpu()
    q = capi.as_f32(queries)
    i8 = np.asarray(rows).dtype == np.int8
    r = np.ascontiguousarray(rows, np.int8 if i8 else np.float32)
    nq, dim = q.shape
    n, stride = r.shape
    if thr is None:
        dense = np.empty((nq, n), np.float32)
        capi.check(capi.load().scann_tc_scores(capi.np_ptr(q), nq, dim, capi.np_ptr(r), int(i8), n, stride, scale,
                                               int(want_norm), None, capi.np_ptr(dense), None, 0, None, device))
        return dense
    t = capi.as_f32(thr)
    cand = np.zeros((nq, cap), np.uint64)
    cnt = np.zeros(nq, np.uint32)
    capi.check(capi.load().scann_tc_scores(capi.np_ptr(q), nq, dim, capi.np_ptr(r), int(i8), n, stride, scale,
                                           int(want_norm), capi.np_ptr(t), None, capi.np_ptr(cand), cap,
                                           capi.np_ptr(cnt), device))
    return cand, cnt


def pq_encode(codebook, x, centers=None, assign=None, device: int = 0):
    """Codebook::encode (+ residual) + PackedCodes4Bit::from_codes → packed [n, ceil(S/2)] u8.
    numpy inputs (no residual) or torch CUDA tensors (residual allowed)."""
    capi.require_gpu()
    S, ncodes, ds = (int(v) for v in codebook.shape)
    assert ncodes == 16
    bpp = (S + 1) // 2
    if _is_torch(x) and x.is_cuda:
        torch = _torch()
        xx = x.to(torch.float32).contiguous()
        cb = codebook.to(torch.float32).contiguous()
        n, stride = xx.shape
        out = torch.empty((n, bpp), dtype=torch.uint8, device=xx.device)
        pc = pa = None
        if centers is not None:
            cc = centers.to(torch.float32).contiguous()
            aa = assign.to(torch.int32).contiguous()
            pc, pa = C.c_void_p(cc.data_ptr()), C.c_void_p(aa.data_ptr())
        capi.check(capi.load().scann_pq_encode(C.c_void_p(cb.data_ptr()), S, ds, C.c_void_p(xx.data_ptr()), n, stride,
                                               pc, pa, C.c_void_p(out.data_ptr()), xx.device.index or 0, capi.DEVICE))
        return out
    cb, xx = capi.as_f32(codebook), capi.as_f32(x)
    n, stride = xx.shape
    if centers is not None:
        # residual on the host side of the boundary is plain f32 subtraction (tree_x_hybrid/mod.rs:181-185)
        xx = (xx - capi.as_f32(centers)[np.asarray(assign, np.int64)]).astype(np.float32)
    out = np.empty((n, bpp), np.uint8)
    capi.check(capi.load().scann_pq_encode(capi.np_ptr(cb), S, ds, capi.np_ptr(xx), n, stride, None, None,
                                           capi.np_ptr(out), device, capi.HOST))
    return out
