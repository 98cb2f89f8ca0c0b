"""TEST INFRASTRUCTURE — ctypes bindings for the two CPU checkers.

* ``Oracle``    : oracle/liboracle.so, our C restatement (hnsw_oracle.c); travels to the GPU box.
* ``Reference`` : oracle/_ref/libleann_ref.so, the reference's own HNSW.cpp / HNSW_search.cpp
                  compiled from /root/reference behind ref_harness.cpp; built in the dev container,
                  the prebuilt .so travels (git-ignored, not gpurun-ignored).
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
DIST_CB = C.CFUNCTYPE(None, C.c_void_p, C.POINTER(C.c_float), C.c_int64, C.POINTER(C.c_int64), C.POINTER(C.c_float))


def build(ref: bool = True) -> None:
    """liboracle.so, and oracle/_ref/ where the original LEANN's sources can be read: at the Makefile's REF, or at
    $LEANN_REFERENCE when that is set."""
    subprocess.run(["make", "-s", "-C", str(HERE), "all"], check=True)
    src = [f"REF={os.environ['LEANN_REFERENCE']}"] if os.environ.get("LEANN_REFERENCE") else []
    if ref and subprocess.run(["make", "-s", "-C", str(HERE), "have-ref", *src], capture_output=True).returncode == 0:
        subprocess.run(["make", "-s", "-j8", "-C", str(HERE), "ref", *src], check=True)


def _p(a, t):
    return a.ctypes.data_as(C.POINTER(t))


class _LboGraph(C.Structure):
    _fields_ = [("ntotal", C.c_int64), ("d", C.c_int), ("metric_ip", C.c_int),
                ("levels", C.POINTER(C.c_int32)), ("level_ptr", C.POINTER(C.c_uint64)),
                ("node_offsets", C.POINTER(C.c_uint64)), ("nbrs", C.POINTER(C.c_int32)),
                ("entry_point", C.c_int), ("max_level", C.c_int), ("vectors", C.POINTER(C.c_float))]


class _LboPq(C.Structure):
    _fields_ = [("ndims", C.c_int), ("n_chunks", C.c_int), ("tables_tr", C.POINTER(C.c_float)), ("centroid", C.POINTER(C.c_float)),
                ("chunk_offsets", C.POINTER(C.c_uint32)), ("codes", C.POINTER(C.c_uint8))]


def _wrap_cb(fn, d):
    """fn(q: np.ndarray[d], ids: np.ndarray[int64]) -> np.ndarray[float32]"""
    if fn is None:
        return C.cast(None, DIST_CB)

    def tramp(ctx, qp, n, idp, outp):
        q = np.ctypeslib.as_array(qp, shape=(d,))
        ids = np.ctypeslib.as_array(idp, shape=(n,))
        out = np.ctypeslib.as_array(outp, shape=(n,))
        out[:] = np.asarray(fn(q.copy(), ids.copy()), np.float32)

    return DIST_CB(tramp)


class Oracle:
    """C restatement of HNSW::search over a CSR graph (see hnsw_oracle.c)."""

    def __init__(self, graph, vectors=None):
        so = HERE / "liboracle.so"
        if not so.exists():
            build(ref=False)
        self.lib = C.CDLL(str(so))
        self.lib.lbo_search.restype = C.c_int
        self.lib.lbo_canon_ip.restype = C.c_float
        self.lib.lbo_canon_l2.restype = C.c_float
        self.lib.lbo_mmh_new.restype = C.c_void_p
        self.g = graph
        self._keep = dict(
            levels=np.ascontiguousarray(graph.levels, np.int32),
            level_ptr=np.ascontiguousarray(graph.level_ptr, np.uint64),
            node_offsets=np.ascontiguousarray(graph.node_offsets, np.uint64),
            nbrs=np.ascontiguousarray(graph.neighbors, np.int32),
        )
        self.vectors = None if vectors is None else np.ascontiguousarray(vectors, np.float32)
        k = self._keep
        self.cg = _LboGraph(graph.ntotal, graph.d, 1 if graph.metric_type == 0 else 0,
                            _p(k["levels"], C.c_int32), _p(k["level_ptr"], C.c_uint64),
                            _p(k["node_offsets"], C.c_uint64), _p(k["nbrs"], C.c_int32),
                            graph.entry_point, graph.max_level,
                            _p(self.vectors, C.c_float) if self.vectors is not None else None)

    def set_pq(self, pq, codes):
        """PQ pruning data (HNSW::load_pq_pruning_data, impl/HNSW_search.cpp:253-297): pq = diskann_format.PQTable
        (pivots [256, ndims], centroid, chunk_offsets), codes [ntotal, n_chunks] uint8."""
        self._pq_keep = dict(tables_tr=np.ascontiguousarray(np.asarray(pq.pivots, np.float32).T),  # [ndims, 256]
                             centroid=np.ascontiguousarray(pq.centroid, np.float32).reshape(-1),
                             chunk_offsets=np.ascontiguousarray(pq.chunk_offsets, np.uint32).reshape(-1),
                             codes=np.ascontiguousarray(codes, np.uint8))
        k = self._pq_keep
        self.cpq = _LboPq(int(pq.ndims), int(pq.n_chunks), _p(k["tables_tr"], C.c_float), _p(k["centroid"], C.c_float),
                          _p(k["chunk_offsets"], C.c_uint32), _p(k["codes"], C.c_uint8))

    def search(self, q, k, ef=64, beam=1, batch_size=0, check_rel=True, dist_fn=None, nthreads=1, prune_ratio=0.0,
               local_prune=False, send_ratio=0.0):
        q = np.ascontiguousarray(q, np.float32)
        nq = q.shape[0]
        D = np.empty((nq, k), np.float32)
        I = np.empty((nq, k), np.int64)
        ndis = np.zeros(nq, np.int64)
        nhops = np.zeros(nq, np.int64)
        cb = _wrap_cb(dist_fn, self.g.d)
        cpq = getattr(self, "cpq", None)
        rc = self.lib.lbo_search_pq(C.byref(self.cg), C.c_int64(nq), _p(q, C.c_float), int(k), int(ef), int(beam),
                                    int(batch_size), int(bool(check_rel)), _p(D, C.c_float), _p(I, C.c_int64),
                                    _p(ndis, C.c_int64), _p(nhops, C.c_int64), cb, None, int(nthreads),
                                    C.byref(cpq) if cpq is not None else None, C.c_float(prune_ratio), int(bool(local_prune)),
                                    C.c_float(send_ratio))
        if rc != 0:
            raise RuntimeError("lbo_search failed (no vectors and no callback?)")
        return D, I, ndis, nhops


def have_reference() -> bool:
    return (HERE / "_ref" / "libleann_ref.so").exists()


class Reference:
    """The compiled reference traversal (faiss fork HNSW.cpp / HNSW_search.cpp)."""

    def __init__(self, d, M=32, metric_ip=True):
        so = HERE / "_ref" / "libleann_ref.so"
        if not so.exists():
            raise FileNotFoundError(f"{so} missing: run `make -C oracle ref` in the dev container")
        lib = self.lib = C.CDLL(str(so))
        for name in ("ref_new", "ref_from_csr", "ref_mmh_new"):
            getattr(lib, name).restype = C.c_void_p
        for name in ("ref_neighbors", "ref_offsets", "ref_levels", "ref_cum", "ref_probas"):
            getattr(lib, name).restype = C.c_void_p
        lib.ref_ntotal.restype = C.c_int64
        lib.ref_neighbors_size.restype = C.c_int64
        self.d, self.M, self.metric_ip = d, M, metric_ip
        self.h = C.c_void_p(lib.ref_new(d, M, int(metric_ip)))
        self._keep = []

    @classmethod
    def from_csr(cls, graph, vectors=None, M=32):
        self = cls.__new__(cls)
        cls.__init__(self, graph.d, M, graph.metric_type == 0)
        self.lib.ref_free(self.h)
        lv = np.ascontiguousarray(graph.levels, np.int32)
        lp = np.ascontiguousarray(graph.level_ptr, np.uint64)
        no = np.ascontiguousarray(graph.node_offsets, np.uint64)
        nb = np.ascontiguousarray(graph.neighbors, np.int32)
        self.h = C.c_void_p(self.lib.ref_from_csr(graph.d, M, int(graph.metric_type == 0), C.c_int64(graph.ntotal),
                                                  _p(lv, C.c_int32), C.c_int64(len(lp)), _p(lp, C.c_uint64),
                                                  _p(no, C.c_uint64), C.c_int64(len(nb)), _p(nb, C.c_int32),
                                                  int(graph.entry_point), int(graph.max_level)))
        if vectors is not None:
            self.set_vectors(vectors)
        return self

    def set_vectors(self, x):
        x = np.ascontiguousarray(x, np.float32)
        self._keep.append(x)
        self.lib.ref_set_vectors(self.h, _p(x, C.c_float))

    def build(self, x, ef_construction=200, nthreads=1):
        x = np.ascontiguousarray(x, np.float32)
        self._keep.append(x)
        self.lib.ref_build(self.h, C.c_int64(x.shape[0]), _p(x, C.c_float), int(ef_construction), int(nthreads))

    def export(self):
        """Non-compact arrays (levels, offsets, neighbors padded with -1, ...) of the built graph."""
        lib, h = self.lib, self.h
        n = lib.ref_ntotal(h)
        nn = lib.ref_neighbors_size(h)

        def arr(ptr, count, dt):
            return np.ctypeslib.as_array(C.cast(ptr, C.POINTER(dt)), shape=(count,)).copy()

        return dict(
            ntotal=n, d=self.d, metric_ip=self.metric_ip,
            levels=arr(lib.ref_levels(h), n, C.c_int32),
            offsets=arr(lib.ref_offsets(h), n + 1, C.c_uint64),
            neighbors=arr(lib.ref_neighbors(h), nn, C.c_int32),
            cum=arr(lib.ref_cum(h), lib.ref_n_cum(h), C.c_int32),
            probas=arr(lib.ref_probas(h), lib.ref_n_probas(h), C.c_double),
            entry_point=lib.ref_entry_point(h), max_level=lib.ref_max_level(h),
            ef_construction=lib.ref_ef_construction(h), ef_search=lib.ref_ef_search(h),
        )

    def load_pq(self, pivots_path, compressed_path):
        """HNSW::load_pq_pruning_data (impl/HNSW_search.cpp:253-297) on DiskANN-format PQ files."""
        if self.lib.ref_load_pq(self.h, str(pivots_path).encode(), str(compressed_path).encode()) != 0:
            raise RuntimeError("reference load_pq_pruning_data failed")

    def search(self, q, k, ef=64, beam=1, batch_size=0, check_rel=True, dist_fn=None, nthreads=1, prune_ratio=0.0,
               local_prune=False, send_ratio=0.0):
        q = np.ascontiguousarray(q, np.float32)
        nq = q.shape[0]
        D = np.empty((nq, k), np.float32)
        I = np.empty((nq, k), np.int64)
        ndis = np.zeros(nq, np.int64)
        nhops = np.zeros(nq, np.int64)
        cb = _wrap_cb(dist_fn, self.d)
        rc = self.lib.ref_search_pq(self.h, C.c_int64(nq), _p(q, C.c_float), C.c_int64(k), int(ef), int(beam),
                                    int(batch_size), int(bool(check_rel)), C.c_float(prune_ratio), int(bool(local_prune)),
                                    C.c_float(send_ratio), _p(D, C.c_float), _p(I, C.c_int64),
                                    _p(ndis, C.c_int64), _p(nhops, C.c_int64), cb, None, int(nthreads))
        if rc != 0:
            raise RuntimeError("ref_search failed")
        return D, I, ndis, nhops

    def __del__(self):
        try:
            self.lib.ref_free(self.h)
        except Exception:
            pass


def export_to_csr(ex: dict):
    """Turn Reference.export() arrays (faiss non-compact layout: impl/HNSW.h:183-192) into a
    CSRGraph, dropping the -1 padding exactly as convert_to_csr.py:488-546 does."""
    from leann_b200.csr import CSRGraph

    n = ex["ntotal"]
    levels, offsets, nbrs, cum = ex["levels"], ex["offsets"].astype(np.int64), ex["neighbors"], ex["cum"]
    node_offsets = np.zeros(n + 1, np.uint64)
    node_offsets[1:] = np.cumsum(levels.astype(np.int64) + 1)
    level_ptr = np.zeros(int(node_offsets[-1]), np.uint64)
    out = []
    pos = 0
    for i in range(n):
        base = int(node_offsets[i])
        for l in range(int(levels[i])):
            level_ptr[base + l] = pos
            seg = nbrs[offsets[i] + cum[l]: offsets[i] + cum[l + 1]]
            seg = seg[seg >= 0]
            out.append(seg)
            pos += len(seg)
        level_ptr[base + int(levels[i])] = pos
    neighbors = np.concatenate(out).astype(np.int32) if out else np.zeros(0, np.int32)
    return CSRGraph(d=ex["d"], ntotal=n, metric_type=0 if ex["metric_ip"] else 1, levels=levels.astype(np.int32),
                    level_ptr=level_ptr, node_offsets=node_offsets, neighbors=neighbors,
                    entry_point=ex["entry_point"], max_level=ex["max_level"],
                    ef_construction=ex["ef_construction"], ef_search=ex["ef_search"],
                    assign_probas=ex["probas"], cum_nneighbor_per_level=ex["cum"])
