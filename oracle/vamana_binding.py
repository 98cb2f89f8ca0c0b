"""TEST INFRASTRUCTURE — ctypes bindings for the DiskANN/Vamana checkers.

* ``VamanaOracle``     : oracle/liboracle.so (vamana_oracle.c), the C restatement of the reference's
                         PQFlashIndex::cached_beam_search as LEANN drives it; travels to the GPU box.
* ``DiskannFlash``     : oracle/_ref/libleann_ref_diskann_flash.so, the reference's own PQFlashIndex::load +
                         cached_beam_search compiled from /root/reference (diskann_flash_harness.cpp: in-process file
                         reader and embedding fetch); the checker that PINS the search loop.
* ``DiskannPrimitives``: oracle/_ref/libleann_ref_diskann.so, the reference's own NeighborPriorityQueue and
                         FixedChunkPQTable compiled from /root/reference (diskann_ref_harness.cpp); prebuilt in the
                         dev container, the .so travels.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from .binding import HERE, _p, build

DEFERRED_FETCH, SKIP_SEARCH_REORDER = 1, 2
METRICS = {"l2": 0, "mips": 1, "cosine": 2}


class _VoIndex(C.Structure):
    _fields_ = [("n", C.c_int64), ("data_dim", C.c_int), ("metric", C.c_int), ("R", C.c_int),
                ("nbrs", C.POINTER(C.c_int32)), ("deg", C.POINTER(C.c_uint32)),
                ("medoids", C.POINTER(C.c_uint32)), ("n_medoids", C.c_int),
                ("centroid_data", C.POINTER(C.c_float)),
                ("n_chunks", C.c_int), ("pivots", C.POINTER(C.c_float)), ("centroid", C.POINTER(C.c_float)),
                ("chunk_offsets", C.POINTER(C.c_uint32)), ("codes", C.POINTER(C.c_uint8)),
                ("max_base_norm", C.c_float)]


def _lib():
    so = HERE / "liboracle.so"
    if not so.exists():
        build(ref=False)
    lib = C.CDLL(str(so))
    if not hasattr(lib, "vo_search_batch"):
        build(ref=False)
        lib = C.CDLL(str(so))
    lib.vo_npq_new.restype = C.c_void_p
    lib.vo_npq_size.restype = C.c_size_t
    lib.vo_pq_tables_tr.restype = C.POINTER(C.c_float)
    return lib


class VamanaOracle:
    def __init__(self, graph, pq, codes, metric: str, max_base_norm: float = 0.0, medoids=None, centroid_data=None):
        """graph: diskann_format.VamanaGraph; pq: diskann_format.PQTable; codes [n, n_chunks] uint8."""
        self.lib = _lib()
        self.metric = metric.lower()
        self.k = dict(
            nbrs=np.ascontiguousarray(graph.nbrs, np.int32),
            deg=np.ascontiguousarray(graph.degrees(), np.uint32),
            medoids=np.ascontiguousarray([graph.medoid] if medoids is None else medoids, np.uint32),
            pivots=np.ascontiguousarray(pq.pivots, np.float32),
            centroid=np.ascontiguousarray(pq.centroid, np.float32),
            chunk_offsets=np.ascontiguousarray(pq.chunk_offsets, np.uint32),
            codes=np.ascontiguousarray(codes, np.uint8),
        )
        self.centroid_data = None if centroid_data is None else np.ascontiguousarray(centroid_data, np.float32)
        k = self.k
        self.data_dim = pq.ndims
        self.cx = _VoIndex(graph.n, pq.ndims, METRICS[self.metric], graph.R, _p(k["nbrs"], C.c_int32), _p(k["deg"], C.c_uint32),
                           _p(k["medoids"], C.c_uint32), len(k["medoids"]),
                           _p(self.centroid_data, C.c_float) if self.centroid_data is not None else None,
                           pq.n_chunks, _p(k["pivots"], C.c_float), _p(k["centroid"], C.c_float),
                           _p(k["chunk_offsets"], C.c_uint32), _p(k["codes"], C.c_uint8), max_base_norm)

    @property
    def raw_dim(self) -> int:
        return self.data_dim - 1 if self.metric == "mips" else self.data_dim

    def search(self, q, k, L=64, beam_width=1, coords=None, emb=None, skip_search_reorder=False, io_limit=0xFFFFFFFF,
               cap_full=None, nthreads=1):
        """emb given -> deferred fetch (recompute_embeddings=True); else coords (stored node coordinates)."""
        q = np.ascontiguousarray(q, np.float32)
        nq, dim = q.shape
        assert dim == self.raw_dim, (dim, self.raw_dim)
        flags = (DEFERRED_FETCH if emb is not None else 0) | (SKIP_SEARCH_REORDER if skip_search_reorder else 0)
        cap_full = cap_full or (8 * L + 64)
        I = np.empty((nq, k), np.int64)
        D = np.empty((nq, k), np.float32)
        full_ids = np.zeros((nq, cap_full), np.uint32)
        full_d = np.zeros((nq, cap_full), np.float32)
        n_full = np.zeros(nq, np.int32)
        stats = np.zeros((nq, 3), np.int64)
        co = None if coords is None else np.ascontiguousarray(coords, np.float32)
        em = None if emb is None else np.ascontiguousarray(emb, np.float32)
        rc = self.lib.vo_search_batch(C.byref(self.cx), C.c_int64(nq), _p(q, C.c_float), dim, k, L, beam_width,
                                      C.c_uint32(io_limit), flags,
                                      _p(co, C.c_float) if co is not None else None,
                                      _p(em, C.c_float) if em is not None else None,
                                      _p(I, C.c_int64), _p(D, C.c_float), _p(full_ids, C.c_uint32), _p(full_d, C.c_float),
                                      cap_full, _p(n_full, C.c_int32), _p(stats, C.c_int64), nthreads)
        if rc:
            raise RuntimeError("vamana oracle: expansion list overflow")
        return D, I, dict(full_ids=full_ids, full_dists=full_d, n_full=n_full, cmps=stats[:, 0], n_ios=stats[:, 1],
                          n_hops=stats[:, 2])

    def prepare_query(self, q):
        """(aligned_query_T [data_dim], |q|) as cached_beam_search forms them (pq_flash_index.cpp:1819-1848)."""
        q = np.ascontiguousarray(q, np.float32)
        aq = np.zeros(self.data_dim, np.float32)
        nrm = C.c_float(0)
        self.lib.vo_prepare_query(C.byref(self.cx), _p(q, C.c_float), _p(aq, C.c_float), C.byref(nrm))
        return aq, nrm.value

    # primitive hooks (pinned against DiskannPrimitives)
    def lut(self, qvec_prepared):
        """qvec_prepared [data_dim] (already normalised / extended) -> (centred query, LUT [n_chunks, 256])."""
        qv = np.ascontiguousarray(qvec_prepared, np.float32).copy()
        tr = self.lib.vo_pq_tables_tr(C.byref(self.cx))
        self.lib.vo_pq_preprocess_query(C.byref(self.cx), _p(qv, C.c_float))
        lut = np.empty((self.cx.n_chunks, 256), np.float32)
        self.lib.vo_pq_populate_chunk_distances(C.byref(self.cx), tr, _p(qv, C.c_float), _p(lut, C.c_float))
        return qv, lut

    def pq_dists(self, lut, ids):
        ids = np.ascontiguousarray(ids, np.int64)
        scratch = np.ascontiguousarray(self.k["codes"][ids])
        out = np.empty(len(ids), np.float32)
        self.lib.vo_pq_dist_lookup(_p(scratch, C.c_uint8), C.c_size_t(len(ids)), C.c_size_t(self.cx.n_chunks),
                                   _p(np.ascontiguousarray(lut, np.float32), C.c_float), _p(out, C.c_float))
        return out


class OracleQueue:
    """vo_npq_* hooks: the restated NeighborPriorityQueue."""

    def __init__(self, capacity):
        self.lib = _lib()
        self.q = C.c_void_p(self.lib.vo_npq_new(C.c_size_t(capacity)))

    def insert(self, i, d):
        self.lib.vo_npq_insert(self.q, C.c_uint32(i), C.c_float(d))

    def closest_unexpanded(self):
        i, d = C.c_uint32(), C.c_float()
        self.lib.vo_npq_closest_unexpanded(self.q, C.byref(i), C.byref(d))
        return i.value, d.value

    def has_unexpanded(self):
        return bool(self.lib.vo_npq_has_unexpanded(self.q))

    def items(self):
        out = []
        for j in range(self.lib.vo_npq_size(self.q)):
            i, d, e = C.c_uint32(), C.c_float(), C.c_int()
            self.lib.vo_npq_get(self.q, C.c_size_t(j), C.byref(i), C.byref(d), C.byref(e))
            out.append((i.value, d.value, e.value))
        return out


def have_diskann_reference() -> bool:
    return (HERE / "_ref" / "libleann_ref_diskann.so").exists()


class DiskannPrimitives:
    """The reference's own queue and PQ table (compiled from /root/reference)."""

    def __init__(self):
        self.lib = C.CDLL(str(HERE / "_ref" / "libleann_ref_diskann.so"))
        self.lib.dref_npq_new.restype = C.c_void_p
        self.lib.dref_npq_size.restype = C.c_size_t
        self.lib.dref_pq_load.restype = C.c_void_p
        self.lib.dref_pq_num_chunks.restype = C.c_uint32

    class Queue:
        def __init__(self, lib, capacity):
            self.lib = lib
            self.q = C.c_void_p(lib.dref_npq_new(C.c_size_t(capacity)))

        def insert(self, i, d):
            self.lib.dref_npq_insert(self.q, C.c_uint32(i), C.c_float(d))

        def closest_unexpanded(self):
            i, d = C.c_uint32(), C.c_float()
            self.lib.dref_npq_closest_unexpanded(self.q, C.byref(i), C.byref(d))
            return i.value, d.value

        def has_unexpanded(self):
            return bool(self.lib.dref_npq_has_unexpanded(self.q))

        def items(self):
            out = []
            for j in range(self.lib.dref_npq_size(self.q)):
                i, d, e = C.c_uint32(), C.c_float(), C.c_int()
                self.lib.dref_npq_get(self.q, C.c_size_t(j), C.byref(i), C.byref(d), C.byref(e))
                out.append((i.value, d.value, e.value))
            return out

        def __del__(self):
            try:
                self.lib.dref_npq_free(self.q)
            except Exception:
                pass

    def queue(self, capacity):
        return DiskannPrimitives.Queue(self.lib, capacity)

    def pq_load(self, pivots_path: str, n_chunks: int):
        h = self.lib.dref_pq_load(str(pivots_path).encode(), C.c_size_t(n_chunks))
        if not h:
            raise RuntimeError("reference load_pq_centroid_bin failed")
        return C.c_void_p(h)

    def pq_num_chunks(self, table) -> int:
        return int(self.lib.dref_pq_num_chunks(table))

    def lut(self, table, qvec_prepared, n_chunks):
        qv = np.ascontiguousarray(qvec_prepared, np.float32).copy()
        self.lib.dref_pq_preprocess_query(table, _p(qv, C.c_float))
        lut = np.empty((n_chunks, 256), np.float32)
        self.lib.dref_pq_populate_chunk_distances(table, _p(qv, C.c_float), _p(lut, C.c_float))
        return qv, lut

    class QueryTable:
        """preprocess_query + populate_chunk_distances for one query, then pq_dist_lookup against that table."""

        def __init__(self, prims, table, qvec_prepared, n_chunks):
            self.prims = prims
            _, self.lut = prims.lut(table, qvec_prepared, n_chunks)

        def dists(self, ids, codes):
            return self.prims.pq_dists(self.lut, ids, codes)

    def query_table(self, table, qvec_prepared, n_chunks):
        return DiskannPrimitives.QueryTable(self, table, qvec_prepared, n_chunks)

    def pq_dists(self, lut, ids, codes):
        ids = np.ascontiguousarray(ids, np.uint32)
        codes = np.ascontiguousarray(codes, np.uint8)
        n_chunks = codes.shape[1]
        scratch = np.empty((len(ids), n_chunks), np.uint8)
        out = np.empty(len(ids), np.float32)
        self.lib.dref_pq_lookup(_p(ids, C.c_uint32), C.c_uint64(len(ids)), _p(codes, C.c_uint8), C.c_uint64(n_chunks),
                                _p(np.ascontiguousarray(lut, np.float32), C.c_float), _p(scratch, C.c_uint8), _p(out, C.c_float))
        return out


def have_diskann_flash() -> bool:
    return (HERE / "_ref" / "libleann_ref_diskann_flash.so").exists()


class DiskannFlash:
    """The reference's compiled PQFlashIndex (load + cached_beam_search) over index files on disk.  Arguments follow
    StaticDiskIndex (python/src/static_disk_index.cpp:15-48, 88-118): index prefix, pq prefix, partition prefix."""

    def __init__(self, index_prefix: str, metric: str, partition_prefix: str = "", pq_prefix: str | None = None, nthreads: int = 1):
        self.lib = C.CDLL(str(HERE / "_ref" / "libleann_ref_diskann_flash.so"))
        self.lib.dflash_open.restype = C.c_void_p
        h = self.lib.dflash_open(str(index_prefix).encode(), str(pq_prefix or index_prefix).encode(), str(partition_prefix).encode(),
                                 METRICS[metric.lower()], nthreads)
        if not h:
            raise RuntimeError(f"reference PQFlashIndex::load failed for {index_prefix}")
        self.h = C.c_void_p(h)
        self._emb = None

    def set_embeddings(self, emb):
        """The table the in-process embedding server answers fetch_embeddings_zmq from."""
        self._emb = np.ascontiguousarray(emb, np.float32)
        self.lib.dflash_set_embeddings(_p(self._emb, C.c_float), C.c_int64(self._emb.shape[0]), int(self._emb.shape[1]))

    def search(self, q, k, L=64, beam_width=1, deferred_fetch=False, skip_search_reorder=False, io_limit=0xFFFFFFFF):
        q = np.ascontiguousarray(q, np.float32)
        nq, dim = q.shape
        ids = np.zeros((nq, k), np.uint64)
        D = np.zeros((nq, k), np.float32)
        cmps, hops, ios = (np.zeros(nq, np.uint32) for _ in range(3))
        if deferred_fetch and self._emb is not None:  # the table is process-global: re-point it at this instance's
            self.lib.dflash_set_embeddings(_p(self._emb, C.c_float), C.c_int64(self._emb.shape[0]), int(self._emb.shape[1]))
        rc = self.lib.dflash_search(self.h, _p(q, C.c_float), C.c_int64(nq), dim, C.c_int64(k), C.c_int64(L), C.c_int64(beam_width),
                                    int(deferred_fetch), int(skip_search_reorder), C.c_uint32(io_limit), _p(ids, C.c_uint64),
                                    _p(D, C.c_float), _p(cmps, C.c_uint32), _p(hops, C.c_uint32), _p(ios, C.c_uint32))
        if rc:
            raise RuntimeError("reference cached_beam_search failed")
        return D, ids.astype(np.int64), dict(n_cmps=cmps.astype(np.int64), n_hops=hops.astype(np.int64), n_ios=ios.astype(np.int64))

    def __del__(self):
        try:
            self.lib.dflash_close(self.h)
        except Exception:
            pass
