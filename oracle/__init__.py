"""ORACLE — TEST INFRASTRUCTURE ONLY.

ctypes loader for ``oracle/libscann_oracle.so`` (the C++ CPU restatement of the reference's hot path,
see ``scann_oracle.cpp``).  Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s
``cpu_baseline`` / ``--impl reference`` legs may import this package.  The product package
(``scann-rust_b200``) never does.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "libscann_oracle.so")

SQL2, L2, DOT = 0, 1, 2
OK, INVALID_ARGUMENT, FAILED_PRECONDITION = 0, 3, 9


def build(force: bool = False) -> str:
    import fcntl

    src = os.path.join(_HERE, "scann_oracle.cpp")

    def stale():
        return force or not os.path.exists(_LIB_PATH) or os.path.getmtime(_LIB_PATH) < os.path.getmtime(src)

    if not stale():  # up to date: touch nothing, so a built tree can be used read-only
        return _LIB_PATH
    with open(os.path.join(_HERE, ".build.lock"), "w") as lock:  # ranks of one torchrun serialise here
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            if stale():
                subprocess.check_call(["make", "-C", _HERE, "-B", "libscann_oracle.so"], stdout=subprocess.DEVNULL)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)
    return _LIB_PATH


_lib = None


def lib():
    global _lib
    if _lib is None:
        build()
        _lib = C.CDLL(_LIB_PATH)
        _lib.orc_pair_distance.restype = C.c_float
        _lib.orc_scalar_sqdist.restype = C.c_float
        _lib.orc_dense_stride.restype = C.c_size_t
        _lib.orc_topk_run.restype = C.c_uint32
        _lib.orc_ftn_run.restype = C.c_uint32
        _lib.orc_bf_search_radius.restype = C.c_size_t
        _lib.orc_sq8_quantize_value.restype = C.c_int8
        _lib.orc_sq8_dequantize_value.restype = C.c_float
        _lib.orc_lut16_distance_single.restype = C.c_float
        _lib.orc_reorder.restype = C.c_uint32
    return _lib


def _f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


def _p(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def _sz(x):
    return C.c_size_t(int(x))


def num_threads() -> int:
    return int(lib().orc_num_threads())


def dense_stride(dim: int, elem_size: int = 4) -> int:
    return int(lib().orc_dense_stride(_sz(dim), _sz(elem_size)))


# ----------------------------------------------------------------------------- distances
def one_to_many(q, db, measure, stride=None):
    q, db = _f32(q), _f32(db)
    n = db.shape[0]
    stride = db.shape[1] if stride is None else stride
    out = np.empty(n, np.float32)
    fn = lib().orc_one_to_many_dot if measure == DOT else lib().orc_one_to_many_sql2
    fn(_p(q), _sz(q.shape[0]), _p(db), _sz(stride), _sz(n), _p(out))
    if measure == L2:
        out = np.sqrt(out)
    return out


def one_to_many_flat(q, flat, stride, n, measure):
    q, flat = _f32(q), _f32(flat)
    out = np.empty(n, np.float32)
    fn = lib().orc_one_to_many_dot if measure == DOT else lib().orc_one_to_many_sql2
    fn(_p(q), _sz(q.shape[0]), _p(flat), _sz(stride), _sz(n), _p(out))
    return out


def one_to_many_i8(q, db_i8, inv_mul, measure):
    q = _f32(q)
    db = np.ascontiguousarray(db_i8, dtype=np.int8)
    n, dim = db.shape
    out = np.empty(n, np.float32)
    fn = lib().orc_one_to_many_i8_dot if measure == DOT else lib().orc_one_to_many_i8_sql2
    fn(_p(q), _sz(q.shape[0]), _p(db), C.c_float(inv_mul), _sz(dim), _sz(n), _p(out))
    return out


def pair_distance(measure, a, b):
    a, b = _f32(a), _f32(b)
    return float(lib().orc_pair_distance(C.c_int(measure), _p(a), _p(b), _sz(a.shape[0])))


def scalar_sqdist(a, b):
    a, b = _f32(a), _f32(b)
    return float(lib().orc_scalar_sqdist(_p(a), _p(b), _sz(a.shape[0])))


# ----------------------------------------------------------------------------- top-k trackers
def topk_run(k, ids, dists):
    ids = np.ascontiguousarray(ids, np.uint32)
    dists = _f32(dists)
    n = len(ids)
    oi, od = np.empty(max(k, 1), np.uint32), np.empty(max(k, 1), np.float32)
    acc = np.empty(max(n, 1), np.uint8)
    m = lib().orc_topk_run(_sz(k), _p(ids), _p(dists), _sz(n), _p(oi), _p(od), _p(acc))
    return oi[:m].copy(), od[:m].copy(), acc[:n].astype(bool)


def ftn_run(cap, ids, dists, batch_mode=False):
    ids = np.ascontiguousarray(ids, np.uint32)
    dists = _f32(dists)
    oi, od = np.empty(max(cap, 1), np.uint32), np.empty(max(cap, 1), np.float32)
    m = lib().orc_ftn_run(_sz(cap), _p(ids), _p(dists), _sz(len(ids)), C.c_int(int(batch_mode)), _p(oi), _p(od))
    return oi[:m].copy(), od[:m].copy()


# ----------------------------------------------------------------------------- brute force
def _alloc_out(nq, k):
    return (np.full((nq, max(k, 1)), 0xFFFFFFFF, np.uint32)[:, :k].copy(),
            np.full((nq, max(k, 1)), np.inf, np.float32)[:, :k].copy(), np.zeros(nq, np.uint32))


def bf_search(db, q, k, measure, nthreads=1, dim=None):
    """db: [n, stride] (rows may be padded: pass dim < stride)."""
    db, q = _f32(db), _f32(q)
    n, stride = db.shape
    dim = stride if dim is None else dim
    nq, qdim = q.shape
    ids, dists, counts = _alloc_out(nq, k)
    rc = lib().orc_bf_search(_p(db), _sz(n), _sz(dim), _sz(stride), C.c_int(measure), _p(q), _sz(nq), _sz(qdim),
                             _sz(k), _p(ids), _p(dists), _p(counts), C.c_int(nthreads))
    return rc, ids, dists, counts


def bf_search_radius(db, q, radius, measure):
    db, q = _f32(db), _f32(q)
    n, dim = db.shape
    ids, dists = np.empty(max(n, 1), np.uint32), np.empty(max(n, 1), np.float32)
    m = lib().orc_bf_search_radius(_p(db), _sz(n), _sz(dim), _sz(dim), C.c_int(measure), _p(q), C.c_float(radius),
                                   _p(ids), _p(dists), _sz(n))
    return ids[:m].copy(), dists[:m].copy()


# ----------------------------------------------------------------------------- scalar quantisation
def sq8_stats(db):
    db = _f32(db)
    out = np.empty(4, np.float32)
    lib().orc_sq8_stats(_p(db), _sz(db.shape[0]), _sz(db.shape[1]), _sz(db.shape[1]), _p(out))
    return out


def sq8_calibrate(stats4, num_std_devs=3.0, bits=8):
    stats4 = _f32(stats4)
    out = np.empty(4, np.float32)
    lib().orc_sq8_calibrate(_p(stats4), C.c_float(num_std_devs), C.c_int(bits), _p(out))
    return out  # min, max, scale, inv_scale


def sq8_quantize_value(v, cal4, bits=8):
    cal4 = _f32(cal4)
    return int(lib().orc_sq8_quantize_value(C.c_float(v), _p(cal4), C.c_int(bits)))


def sq8_dequantize_value(qv, cal4):
    cal4 = _f32(cal4)
    return float(lib().orc_sq8_dequantize_value(C.c_int8(qv), _p(cal4)))


def sq8_quantize(db):
    db = _f32(db)
    n, dim = db.shape
    out = np.empty((n, dim), np.int8)
    cal = np.empty(4, np.float32)
    lib().orc_sq8_quantize(_p(db), _sz(n), _sz(dim), _sz(dim), _p(out), _p(cal))
    return out, cal


def sq8_search(db_i8, scale, q, k, measure, nthreads=1):
    db = np.ascontiguousarray(db_i8, np.int8)
    q = _f32(q)
    n, dim = db.shape
    nq, qdim = q.shape
    ids, dists, counts = _alloc_out(nq, k)
    rc = lib().orc_sq8_search(_p(db), _sz(n), _sz(dim), C.c_float(scale), C.c_int(measure), _p(q), _sz(nq),
                              _sz(qdim), _sz(k), _p(ids), _p(dists), _p(counts), C.c_int(nthreads))
    return rc, ids, dists, counts


# ----------------------------------------------------------------------------- partitioning / PQ
def partition(centers, q, L, nthreads=1):
    centers, q = _f32(centers), _f32(q)
    K, dim = centers.shape
    nq = q.shape[0]
    tokens = np.empty((nq, L), np.uint32)
    dists = np.empty((nq, L), np.float32)
    lib().orc_partition(_p(centers), _sz(K), _sz(dim), _p(q), _sz(nq), _sz(L), _p(tokens), _p(dists),
                        C.c_int(nthreads))
    return tokens, dists


def kmtree_search_leaves(centers, depth, child_begin, child_count, children, q, k):
    """KMeansTree::search_leaves over a flattened tree → (leaf node ids [nq,k], dists, depths, counts)"""
    centers, q = _f32(centers), _f32(q)
    u32 = lambda a: np.ascontiguousarray(a, np.uint32)
    depth, child_begin, child_count, children = u32(depth), u32(child_begin), u32(child_count), u32(children)
    nq, dim = q.shape
    nodes = np.empty((nq, k), np.uint32)
    dists = np.empty((nq, k), np.float32)
    depths = np.empty((nq, k), np.uint32)
    counts = np.empty((nq,), np.uint32)
    lib().orc_kmtree_search_leaves(_p(centers), _p(depth), _p(child_begin), _p(child_count), _p(children), _sz(dim),
                                   _p(q), _sz(nq), _sz(k), _p(nodes), _p(dists), _p(depths), _p(counts))
    return nodes, dists, depths, counts


def pq_encode(cb, x):
    """cb: [S, C, ds] f32; x: [n, S*ds] → codes [n, S] u8"""
    cb, x = _f32(cb), _f32(x)
    S, Cc, ds = cb.shape
    n = x.shape[0]
    codes = np.empty((n, S), np.uint8)
    lib().orc_pq_encode(_p(cb), _sz(S), _sz(Cc), _sz(ds), _p(x), _sz(n), _sz(x.shape[1]), _p(codes))
    return codes


def pq_encode_residual(cb, x, centers, assign):
    cb, x, centers = _f32(cb), _f32(x), _f32(centers)
    assign = np.ascontiguousarray(assign, np.uint32)
    S, Cc, ds = cb.shape
    n = x.shape[0]
    codes = np.empty((n, S), np.uint8)
    lib().orc_pq_encode_residual(_p(cb), _sz(S), _sz(Cc), _sz(ds), _p(x), _sz(n), _sz(x.shape[1]), _p(centers),
                                 _p(assign), _p(codes))
    return codes


def pack4(codes):
    codes = np.ascontiguousarray(codes, np.uint8)
    n, S = codes.shape
    out = np.empty((n, (S + 1) // 2), np.uint8)
    lib().orc_pack4(_p(codes), _sz(n), _sz(S), _p(out))
    return out


def unpack4(packed, S):
    packed = np.ascontiguousarray(packed, np.uint8)
    n = packed.shape[0]
    out = np.empty((n, S), np.uint8)
    lib().orc_unpack4(_p(packed), _sz(n), _sz(S), _p(out))
    return out


def lut_f32(cb, q):
    cb, q = _f32(cb), _f32(q)
    S, Cc, ds = cb.shape
    out = np.empty((S, Cc), np.float32)
    lib().orc_lut_f32(_p(cb), _sz(S), _sz(Cc), _sz(ds), _p(q), _p(out))
    return out


def lut_f32_scan(lut, codes):
    lut = _f32(lut)
    codes = np.ascontiguousarray(codes, np.uint8)
    S, Cc = lut.shape
    n = codes.shape[0]
    out = np.empty(n, np.float32)
    lib().orc_lut_f32_scan(_p(lut), _sz(S), _sz(Cc), _p(codes), _sz(n), _p(out))
    return out


def lut16_quantize(lutf):
    lutf = _f32(lutf)
    S = lutf.shape[0]
    l8 = np.empty((S, 16), np.uint8)
    bias, mult = C.c_float(), C.c_float()
    lib().orc_lut16_quantize(_p(lutf), _sz(S), _p(l8), C.byref(bias), C.byref(mult))
    return l8, bias.value, mult.value


def lut16_build(cb, q, centroid=None):
    """cb [S,16,ds]; returns (lut8 [S,16] u8, bias, mult, lutf [S,16] f32)"""
    cb, q = _f32(cb), _f32(q)
    cen = _f32(centroid) if centroid is not None else None
    S, Cc, ds = cb.shape
    assert Cc == 16
    l8 = np.empty((S, 16), np.uint8)
    lf = np.empty((S, 16), np.float32)
    bias, mult = C.c_float(), C.c_float()
    lib().orc_lut16_build(_p(cb), _sz(S), _sz(ds), _p(q), _p(cen), _p(l8), C.byref(bias), C.byref(mult), _p(lf))
    return l8, bias.value, mult.value, lf


def lut16_scan_u32(packed, lut8, S):
    packed = np.ascontiguousarray(packed, np.uint8)
    lut8 = np.ascontiguousarray(lut8, np.uint8)
    n = packed.shape[0]
    out = np.empty(n, np.uint32)
    lib().orc_lut16_scan_u32(_p(packed), _p(lut8), _sz(S), _sz(n), _p(out))
    return out


def lut16_scan_f32(packed, lut8, S, n=None):
    packed = np.ascontiguousarray(packed, np.uint8)
    lut8 = np.ascontiguousarray(lut8, np.uint8)
    n = packed.shape[0] if n is None else n
    out = np.empty(n, np.float32)
    lib().orc_lut16_scan_f32(_p(packed), _p(lut8), _sz(S), _sz(n), _p(out))
    return out


def lut16_distances(packed, lut8, S, bias, mult, n=None):
    packed = np.ascontiguousarray(packed, np.uint8)
    lut8 = np.ascontiguousarray(lut8, np.uint8)
    n = packed.shape[0] if n is None else n
    out = np.empty(n, np.float32)
    lib().orc_lut16_distances(_p(packed), _p(lut8), _sz(S), _sz(n), C.c_float(bias), C.c_float(mult), _p(out))
    return out


def lut16_distance_single(codes, lut8, bias, mult):
    codes = np.ascontiguousarray(codes, np.uint8)
    lut8 = np.ascontiguousarray(lut8, np.uint8)
    S = lut8.shape[0]
    return float(lib().orc_lut16_distance_single(_p(codes), _p(lut8), _sz(S), C.c_float(bias), C.c_float(mult)))


# ----------------------------------------------------------------------------- searchers
def ah_search(cb, codes, q, k, lut16=False, raw=None, pre_k=0, nthreads=1):
    cb, q = _f32(cb), _f32(q)
    codes = np.ascontiguousarray(codes, np.uint8)
    rawc = _f32(raw) if raw is not None else None
    S, Cc, ds = cb.shape
    n = codes.shape[0]
    nq, qdim = q.shape
    ids, dists, counts = _alloc_out(nq, k)
    rc = lib().orc_ah_search(_p(cb), _sz(S), _sz(Cc), _sz(ds), _p(codes), _sz(n), C.c_int(int(lut16)), _p(rawc),
                             _sz(rawc.shape[1] if rawc is not None else 0), _p(q), _sz(nq), _sz(qdim), _sz(k),
                             _sz(pre_k), _p(ids), _p(dists), _p(counts), C.c_int(nthreads))
    return rc, ids, dists, counts


def treex_search(centers, cb, part_off, part_ids, codes, raw, q, L, R, k, lut16=True, use_residuals=True,
                 reorder_measure=SQL2, nthreads=1, want_candidates=False, allow=None):
    """allow: optional RestrictFilter as a packed bitmap over datapoint ids (np.packbits(mask, bitorder='little'))
    → TreeXHybridSearcher::search_with_filter (tree_x_hybrid/mod.rs:245-250)."""
    centers, cb, q = _f32(centers), _f32(cb), _f32(q)
    allow_arr = None
    if allow is not None:
        allow_arr = np.ascontiguousarray(allow, np.uint8)
        lib().orc_set_filter(_p(allow_arr), _sz(allow_arr.size * 8))
    rawc = _f32(raw) if raw is not None else None
    part_off = np.ascontiguousarray(part_off, np.uint64)
    part_ids = np.ascontiguousarray(part_ids, np.uint32)
    codes = np.ascontiguousarray(codes, np.uint8)
    K, dim = centers.shape
    S, Cc, ds = cb.shape
    nq, qdim = q.shape
    ids, dists, counts = _alloc_out(nq, k)
    cand = np.empty((nq, max(R, 1)), np.uint32) if want_candidates else None
    cand_d = np.empty((nq, max(R, 1)), np.float32) if want_candidates else None
    cand_n = np.zeros(nq, np.uint32) if want_candidates else None
    rc = lib().orc_treex_search(_p(centers), _sz(K), _sz(dim), _p(cb), _sz(S), _sz(Cc), _sz(ds), _p(part_off),
                                _p(part_ids), _p(codes), C.c_int(int(lut16)), _p(rawc),
                                _sz(rawc.shape[1] if rawc is not None else 0), C.c_int(int(use_residuals)),
                                C.c_int(reorder_measure), _p(q), _sz(nq), _sz(qdim), _sz(L), _sz(R), _sz(k),
                                _p(ids), _p(dists), _p(counts), _p(cand), _p(cand_d), _p(cand_n),
                                C.c_int(nthreads))
    if allow is not None:
        lib().orc_set_filter(None, _sz(0))
    if want_candidates:
        return rc, ids, dists, counts, cand, cand_d, cand_n
    return rc, ids, dists, counts


def scann_partitioned(centers, part_off, part_ids, raw, q, L, k, measure, nthreads=1):
    centers, raw, q = _f32(centers), _f32(raw), _f32(q)
    part_off = np.ascontiguousarray(part_off, np.uint64)
    part_ids = np.ascontiguousarray(part_ids, np.uint32)
    K, dim = centers.shape
    nq = q.shape[0]
    ids, dists, counts = _alloc_out(nq, k)
    rc = lib().orc_scann_partitioned(_p(centers), _sz(K), _sz(dim), _p(part_off), _p(part_ids), _p(raw),
                                     _sz(raw.shape[1]), C.c_int(measure), _p(q), _sz(nq), _sz(L), _sz(k), _p(ids),
                                     _p(dists), _p(counts), C.c_int(nthreads))
    return rc, ids, dists, counts


def scann_tree_ah(centers, part_off, part_ids, cb, codes_by_id, raw, q, L, k, reorder_measure=-1, nthreads=1):
    centers, cb, q = _f32(centers), _f32(cb), _f32(q)
    rawc = _f32(raw) if raw is not None else None
    part_off = np.ascontiguousarray(part_off, np.uint64)
    part_ids = np.ascontiguousarray(part_ids, np.uint32)
    codes_by_id = np.ascontiguousarray(codes_by_id, np.uint8)
    K, dim = centers.shape
    S, Cc, ds = cb.shape
    nq = q.shape[0]
    ids, dists, counts = _alloc_out(nq, k)
    rc = lib().orc_scann_tree_ah(_p(centers), _sz(K), _sz(dim), _p(part_off), _p(part_ids), _p(cb), _sz(S), _sz(Cc),
                                 _sz(ds), _p(codes_by_id), _p(rawc), _sz(rawc.shape[1] if rawc is not None else 0),
                                 C.c_int(reorder_measure), _p(q), _sz(nq), _sz(L), _sz(k), _p(ids), _p(dists),
                                 _p(counts), C.c_int(nthreads))
    return rc, ids, dists, counts


def reorder(raw, measure, q, cand, k):
    raw, q = _f32(raw), _f32(q)
    cand = np.ascontiguousarray(cand, np.uint32)
    ids, dists = np.empty(max(k, 1), np.uint32), np.empty(max(k, 1), np.float32)
    m = lib().orc_reorder(_p(raw), _sz(raw.shape[1]), _sz(q.shape[0]), C.c_int(measure), _p(q), _p(cand),
                          _sz(len(cand)), _sz(k), _p(ids), _p(dists))
    return ids[:m].copy(), dists[:m].copy()
