"""CPU suite for the DiskANN/Vamana row: file formats, and the C restatement's primitives pinned against the
reference's own code (oracle/_ref/libleann_ref_diskann.so = DiskANN's neighbor.h + pq.cpp, and
oracle/_ref/libleann_ref_diskann_flash.so = its PQFlashIndex search loop; their outputs replayed from
tests/golden/reference_replay/, see helpers.ReferenceReplay)."""
from __future__ import annotations

import numpy as np
import pytest

from leann_b200 import diskann_format as dfmt
from leann_b200.vamana_build import build_diskann_index, build_vamana_graph
from helpers import reference  # noqa: F401  (fixture)
from oracle.vamana_binding import DiskannFlash, DiskannPrimitives, OracleQueue, VamanaOracle, have_diskann_flash

needs_flash = pytest.mark.skipif(not have_diskann_flash(), reason="compiled PQFlashIndex (oracle/_ref/libleann_ref_diskann_flash.so) not present")


def unit_rows(n, d, seed, clusters=12):
    rng = np.random.default_rng(seed)
    cen = rng.standard_normal((clusters, d)).astype(np.float32)
    x = cen[rng.integers(0, clusters, n)] + 0.45 * rng.standard_normal((n, d)).astype(np.float32)
    return x


@pytest.fixture(scope="module")
def small_index(tmp_path_factory):
    d = tmp_path_factory.mktemp("da")
    emb = unit_rows(1500, 48, 1)
    emb *= np.random.default_rng(2).uniform(0.5, 1.5, (len(emb), 1)).astype(np.float32)  # MIPS: norms matter
    prefix, g, coords, pq, codes, max_norm = build_diskann_index(d, "t", emb, metric="mips", R=16, n_chunks=12, device="cpu")
    return dict(prefix=prefix, g=g, coords=coords, pq=pq, codes=codes, max_norm=max_norm, emb=emb)


def test_file_formats_round_trip(small_index, tmp_path):
    s = small_index
    pq2 = dfmt.read_pq_pivots(s["prefix"] + "_pq_pivots.bin")
    assert np.array_equal(pq2.pivots, s["pq"].pivots) and np.array_equal(pq2.centroid, s["pq"].centroid)
    assert np.array_equal(pq2.chunk_offsets, s["pq"].chunk_offsets)
    assert np.array_equal(dfmt.read_bin(s["prefix"] + "_pq_compressed.bin", np.uint8), s["codes"])
    coords, g2 = dfmt.read_disk_index(s["prefix"] + "_disk.index")
    assert np.array_equal(coords, s["coords"]) and np.array_equal(g2.nbrs, s["g"].nbrs) and g2.medoid == s["g"].medoid
    assert dfmt.read_bin(s["prefix"] + "_disk.index_medoids.bin", np.uint32)[0, 0] == s["g"].medoid
    assert dfmt.read_bin(s["prefix"] + "_disk.index_max_base_norm.bin", np.float32)[0, 0] == np.float32(s["max_norm"])
    files = dfmt.index_files(s["prefix"])
    assert files["_partition.bin"] and files["_disk_graph.index"]
    # multi-sector nodes (max_node_len > 4096) and several nodes per sector both round-trip
    big = np.random.default_rng(0).standard_normal((7, 1100)).astype(np.float32)
    gb = dfmt.VamanaGraph(np.array([[1, 2, -1], [0, -1, -1], [3, 4, 5], [6, -1, -1], [0, 1, 2], [2, -1, -1], [5, 4, -1]], np.int32), 3)
    dfmt.write_disk_index(tmp_path / "big_disk.index", big, gb)
    c2, g3 = dfmt.read_disk_index(tmp_path / "big_disk.index")
    assert np.array_equal(c2, big) and np.array_equal(g3.nbrs, gb.nbrs)


def test_prepare_base_matches_the_searchers_preprocessing(small_index):
    """coords written at build time == preprocess_fetched_embeddings applied to the raw embedding (within fp32 noise)."""
    s = small_index
    o = VamanaOracle(s["g"], s["pq"], s["codes"], "mips", s["max_norm"])
    import ctypes as C
    out = np.empty(o.data_dim, np.float32)
    for i in (0, 7, 1499):
        e = np.ascontiguousarray(s["emb"][i])
        o.lib.vo_preprocess_embedding(C.byref(o.cx), e.ctypes.data_as(C.POINTER(C.c_float)), e.shape[0],
                                      out.ctypes.data_as(C.POINTER(C.c_float)))
        assert np.abs(out - s["coords"][i]).max() < 1e-6
    assert abs(np.linalg.norm(s["coords"], axis=1).max() - 1.0) < 1e-5


def test_queue_restatement_matches_reference_queue(reference):
    """Random insert / closest_unexpanded streams incl. distance ties, duplicate ids and a full queue."""
    ref = reference.proxy(DiskannPrimitives)
    rng = np.random.default_rng(5)
    for cap in (1, 4, 17, 64):
        a, b = ref.queue(cap), OracleQueue(cap)
        for step in range(600):
            if rng.random() < 0.75 or not a.has_unexpanded():
                i = int(rng.integers(0, 40))
                d = float(np.float32(rng.integers(0, 12)) / 4) if rng.random() < 0.7 else float(np.float32(rng.random()))
                a.insert(i, d); b.insert(i, d)
            else:
                assert a.closest_unexpanded() == b.closest_unexpanded()
            assert a.has_unexpanded() == b.has_unexpanded()
            if step % 37 == 0:
                assert a.items() == b.items()
        assert a.items() == b.items()


@pytest.mark.parametrize("metric", ["mips", "l2"])
def test_pq_restatement_matches_reference_pq_bit_for_bit(tmp_path, metric, reference):
    emb = unit_rows(900, 41, 3)  # 41 (+1) dims over 9 chunks: uneven chunk widths
    prefix, g, coords, pq, codes, max_norm = build_diskann_index(tmp_path, "p", emb, metric=metric, R=8, n_chunks=9, device="cpu")
    ref = reference.proxy(DiskannPrimitives)
    table = ref.pq_load(prefix + "_pq_pivots.bin", pq.n_chunks)
    assert ref.pq_num_chunks(table) == pq.n_chunks
    o = VamanaOracle(g, pq, codes, metric, max_norm)
    rng = np.random.default_rng(9)
    for _ in range(5):
        q = rng.standard_normal(pq.ndims).astype(np.float32)
        qa, la = ref.lut(table, q, pq.n_chunks)
        qb, lb = o.lut(q)
        assert np.array_equal(qa, qb) and np.array_equal(la, lb)
        ids = rng.integers(0, len(emb), 50)
        assert np.array_equal(ref.pq_dists(la, ids, codes), o.pq_dists(lb, ids))


@pytest.mark.parametrize("metric", ["mips", "l2", "cosine"])
def test_oracle_search_finds_true_neighbours(tmp_path, metric):
    emb = unit_rows(3000, 32, 11)
    if metric == "mips":
        emb *= np.random.default_rng(1).uniform(0.7, 1.3, (len(emb), 1)).astype(np.float32)
    prefix, g, coords, pq, codes, max_norm = build_diskann_index(tmp_path, "s", emb, metric=metric, R=24, n_chunks=16, device="cpu")
    q = unit_rows(40, 32, 12)
    o = VamanaOracle(g, pq, codes, metric, max_norm)
    D, I, info = o.search(q, 10, L=256, beam_width=2, coords=coords)
    if metric == "mips":
        gt = np.argsort(-(q @ emb.T), axis=1)[:, :10]
    elif metric == "cosine":
        en = emb / np.linalg.norm(emb, axis=1, keepdims=True)
        gt = np.argsort(-(q @ en.T), axis=1)[:, :10]
    else:
        gt = np.argsort(((q[:, None, :] - emb[None]) ** 2).sum(2), axis=1)[:, :10]
    rec = np.mean([len(set(I[i]) & set(gt[i])) / 10 for i in range(len(q))])
    assert rec > 0.85, rec  # low-contrast clusters: 0.64 at L=64, 0.9+ at L=256 (graph-limited, not PQ-limited)
    # distances follow the reference's output convention (pq_flash_index.cpp:2861-2883)
    if metric == "mips":   # -(L2 in the extended space) rescaled by max_base_norm * |q|: descending
        assert np.all(np.diff(D, axis=1) <= 0)
    else:
        assert np.all(np.diff(D, axis=1) >= 0)
    if metric == "l2":
        exact = ((q[:, None, :] - emb[I]) ** 2).sum(2)
        assert np.abs(exact - D).max() < 1e-3
    # the deferred-fetch path over the raw embeddings ranks the same candidates
    D2, I2, info2 = o.search(q, 10, L=256, beam_width=2, emb=emb)
    assert np.array_equal(info["full_ids"], info2["full_ids"])  # traversal is PQ-only: identical expansions
    assert np.mean(I == I2) > 0.98 and np.abs(D - D2).max() < 1e-3 * max(1.0, np.abs(D).max())
    assert info["n_full"].min() >= 10 and (info["n_ios"] == info["n_full"]).all()


@pytest.mark.parametrize("metric", ["mips", "l2"])
def test_reference_pq_reads_the_committed_fixture(golden_dir, metric, reference):
    """The reference's own load_pq_centroid_bin / populate_chunk_distances / pq_dist_lookup on the committed files."""
    from helpers import load_vamana_golden
    G = load_vamana_golden(golden_dir, metric)
    ref = reference.proxy(DiskannPrimitives)
    table = ref.pq_load(G["prefix"] + "_pq_pivots.bin", G["pq"].n_chunks)
    o = VamanaOracle(G["g"], G["pq"], G["codes"], metric, G["max_norm"])
    q = np.zeros(G["pq"].ndims, np.float32)
    q[: G["q"].shape[1]] = G["q"][0]
    qa, la = ref.lut(table, q, G["pq"].n_chunks)
    qb, lb = o.lut(q)
    assert np.array_equal(la, lb)
    ids = np.arange(0, 1200, 7)
    assert np.array_equal(ref.pq_dists(la, ids, G["codes"]), o.pq_dists(lb, ids))


@pytest.mark.parametrize("metric", ["mips", "l2"])
def test_oracle_reproduces_committed_goldens(golden_dir, metric):
    from helpers import VAMANA_GOLDEN_CASES, load_vamana_golden
    G = load_vamana_golden(golden_dir, metric)
    o = VamanaOracle(G["g"], G["pq"], G["codes"], metric, G["max_norm"])
    for L, beam, k in VAMANA_GOLDEN_CASES:
        for mode, kw in (("stored", dict(coords=G["coords"])), ("deferred", dict(emb=G["emb"])), ("pq", dict(skip_search_reorder=True))):
            D, I, info = o.search(G["q"], k, L=L, beam_width=beam, **kw)
            key = f"{metric}_L{L}_b{beam}_k{k}_{mode}"
            assert np.array_equal(I, G["exp"][key + "_I"]) and np.array_equal(D, G["exp"][key + "_D"]), key
            assert np.array_equal(info["n_full"], G["exp"][key + "_nfull"]) and np.array_equal(info["cmps"], G["exp"][key + "_cmps"])
            w = G["exp"][key + "_full"].shape[1]
            assert np.array_equal(info["full_ids"][:, :w], G["exp"][key + "_full"]), key


def _beam_search_with_reference_primitives(ref, table, G, q, L, beam, k, io_limit=2 ** 32 - 1, metric="l2", scale=None):
    """Second, independent transcription of the loop of PQFlashIndex::cached_beam_search (pq_flash_index.cpp:2110-2211,
    2419-2612, 2761, 2861-2883; L2 metric, skip_search_reorder) driving the REFERENCE's compiled queue and PQ table, so the
    only non-reference code involved is this loop."""
    g, codes, n_chunks = G["g"], G["codes"], G["pq"].n_chunks
    qt = ref.query_table(table, q, n_chunks)                  # preprocess_query + populate_chunk_distances
    retset = ref.queue(L)
    visited = set()
    med = g.medoid
    retset.insert(med, float(qt.dists([med], codes)[0]))
    visited.add(med)
    full, cmps, hops, ios = [], 0, 0, 0
    while retset.has_unexpanded() and ios < io_limit:
        frontier = []
        while retset.has_unexpanded() and len(frontier) < beam:
            frontier.append(retset.closest_unexpanded())
        if frontier:
            hops += 1
        ios += len(frontier)
        for node, d in frontier:
            full.append((d, node))
            nb = g.nbrs[node]
            nb = nb[nb >= 0]
            dists = qt.dists(nb, codes)
            for m, i in enumerate(nb.tolist()):
                if i not in visited:
                    visited.add(i)
                    cmps += 1
                    retset.insert(i, float(dists[m]))
    order = sorted(full)                                      # Neighbor::operator< : (distance, id)
    ids = [i for _, i in order[:k]] + [-1] * max(0, k - len(order))
    ds = np.array([d for d, _ in order[:k]], np.float32)
    if metric == "mips":                                      # :2873-2881
        ds = -ds
        if scale is not None:
            ds = ds * np.float32(scale)
    ds = np.concatenate([ds, np.full(max(0, k - len(order)), np.finfo(np.float32).max, np.float32)])
    return np.array(ids), ds, [i for _, i in full], cmps, hops


def test_search_loop_agrees_with_a_second_transcription_over_reference_primitives(golden_dir, reference):
    from helpers import load_vamana_golden
    G = load_vamana_golden(golden_dir, "l2")
    ref = reference.proxy(DiskannPrimitives)
    table = ref.pq_load(G["prefix"] + "_pq_pivots.bin", G["pq"].n_chunks)
    o = VamanaOracle(G["g"], G["pq"], G["codes"], "l2", 0.0)
    for L, beam, k, io_limit in [(64, 1, 10, 2 ** 32 - 1), (16, 4, 10, 2 ** 32 - 1), (8, 3, 20, 2 ** 32 - 1), (32, 2, 5, 9)]:
        D, I, info = o.search(G["q"], k, L=L, beam_width=beam, skip_search_reorder=True, io_limit=io_limit)
        for qi in range(len(G["q"])):
            ids, ds, full, cmps, hops = _beam_search_with_reference_primitives(ref, table, G, G["q"][qi], L, beam, k, io_limit)
            n = info["n_full"][qi]
            assert info["full_ids"][qi, :n].tolist() == full, (L, beam, qi)
            assert (info["cmps"][qi], info["n_hops"][qi]) == (cmps, hops)
            assert np.array_equal(I[qi], ids) and np.array_equal(D[qi], ds)


def test_search_loop_second_transcription_mips_with_query_normalisation(golden_dir, reference):
    """Same cross-check for the MIPS index: the query is normalised / extended by the oracle's vo_prepare_query, everything
    after that (centring, table, queue, distances) is the reference's compiled code."""
    from helpers import load_vamana_golden
    G = load_vamana_golden(golden_dir, "mips")
    ref = reference.proxy(DiskannPrimitives)
    table = ref.pq_load(G["prefix"] + "_pq_pivots.bin", G["pq"].n_chunks)
    o = VamanaOracle(G["g"], G["pq"], G["codes"], "mips", G["max_norm"])
    for L, beam, k in [(64, 1, 10), (16, 4, 10)]:
        D, I, info = o.search(G["q"], k, L=L, beam_width=beam, skip_search_reorder=True)
        for qi in range(len(G["q"])):
            aq, nrm = o.prepare_query(G["q"][qi])
            assert abs(nrm - np.linalg.norm(G["q"][qi])) < 1e-5 and aq[-1] == 0 and abs(np.linalg.norm(aq) - 1) < 1e-6
            scale = np.float32(G["max_norm"]) * np.float32(nrm)
            ids, ds, full, cmps, hops = _beam_search_with_reference_primitives(ref, table, G, aq, L, beam, k, metric="mips", scale=scale)
            n = info["n_full"][qi]
            assert info["full_ids"][qi, :n].tolist() == full and (info["cmps"][qi], info["n_hops"][qi]) == (cmps, hops)
            assert np.array_equal(I[qi], ids) and np.array_equal(D[qi], ds)


def test_vamana_builder_degree_and_connectivity():
    x = unit_rows(2000, 24, 4)
    g = build_vamana_graph(x, R=16, device="cpu")
    deg = g.degrees()
    assert deg.max() <= 16 and deg.min() >= 1 and g.nbrs.shape == (2000, 16)
    assert ((g.nbrs >= 0).cumsum(1)[:, -1] == deg).all() and (g.nbrs[np.arange(2000), np.maximum(deg - 1, 0)] >= 0).all()
    seen = np.zeros(2000, bool); seen[g.medoid] = True; frontier = [g.medoid]
    while frontier:
        nxt = g.nbrs[frontier].ravel(); nxt = np.unique(nxt[nxt >= 0]); nxt = nxt[~seen[nxt]]
        seen[nxt] = True; frontier = list(nxt)
    assert seen.mean() > 0.99


# ---------------------------------------------------------------------------------------------------------------------
# The search loop, PINNED: oracle/vamana_oracle.c against the reference's own PQFlashIndex::cached_beam_search
# (pq_flash_index.cpp:1779-2906, compiled from /root/reference into oracle/_ref/libleann_ref_diskann_flash.so).
def _expanded_degree_sum(g, full_ids, n_full):
    deg = g.degrees().astype(np.int64)
    return np.array([deg[full_ids[i, : n_full[i]]].sum() for i in range(len(n_full))], np.int64)


def _check_against_reference(o, G, q, k, L, beam, kw, rD, rI, rs, tag):
    D, I, info = o.search(q, k, L=L, beam_width=beam, **kw)
    # slots beyond the number of expanded nodes: the reference leaves whatever its scratch vector held (it copies k entries
    # of full_retset regardless, :2861-2872); the restatement and the C ABI define them as (-1, FLT_MAX)
    filled = np.arange(k)[None, :] < info["n_full"][:, None]
    assert np.array_equal(I[filled], rI[filled]), tag                        # identical ids, position by position
    assert (I[~filled] == -1).all(), tag
    assert np.abs(D[filled] - rD[filled]).max() <= 2e-5 * max(1.0, float(np.abs(rD[filled]).max())), (tag, float(np.abs(D - rD)[filled].max()))
    assert np.array_equal(info["n_hops"], rs["n_hops"]) and np.array_equal(info["n_full"], rs["n_ios"]), tag
    # QueryStats.n_cmps counts every PQ-scored neighbour of an expanded node plus every first visit (:2578, :2599);
    # the oracle's cmps is the local counter of first visits (:2596)
    assert np.array_equal(info["cmps"] + _expanded_degree_sum(G["g"], info["full_ids"], info["n_full"]), rs["n_cmps"]), tag


@pytest.mark.parametrize("metric", ["mips", "l2"])
def test_oracle_matches_the_committed_outputs_of_the_compiled_reference(golden_dir, metric):
    """Runs everywhere (no compiled reference needed): the *_ref* arrays of vamana_small_expected.npz were produced by the
    reference's compiled cached_beam_search over the committed index files (tests/golden/make_vamana_golden.py)."""
    from helpers import VAMANA_GOLDEN_CASES, load_vamana_golden
    G = load_vamana_golden(golden_dir, metric)
    o = VamanaOracle(G["g"], G["pq"], G["codes"], metric, G["max_norm"])
    for L, beam, k in VAMANA_GOLDEN_CASES:
        for mode, kw in (("stored", dict(coords=G["coords"])), ("deferred", dict(emb=G["emb"])), ("pq", dict(skip_search_reorder=True))):
            key = f"{metric}_L{L}_b{beam}_k{k}_{mode}"
            rs = dict(n_cmps=G["exp"][key + "_refcmps"], n_hops=G["exp"][key + "_refhops"], n_ios=G["exp"][key + "_refios"])
            _check_against_reference(o, G, G["q"], k, L, beam, kw, G["exp"][key + "_refD"], G["exp"][key + "_refI"], rs, key)


@needs_flash
@pytest.mark.parametrize("metric", ["mips", "l2"])
def test_compiled_reference_reproduces_its_committed_outputs(golden_dir, metric):
    from helpers import VAMANA_GOLDEN_CASES, load_vamana_golden
    G = load_vamana_golden(golden_dir, metric)
    for part in ("", G["prefix"]):
        ref = DiskannFlash(G["prefix"], metric, partition_prefix=part)
        ref.set_embeddings(G["emb"])
        for L, beam, k in VAMANA_GOLDEN_CASES:
            for mode in ("deferred", "pq") + (("stored",) if not part else ()):
                key = f"{metric}_L{L}_b{beam}_k{k}_{mode}"
                D, I, st = ref.search(G["q"], k, L=L, beam_width=beam, deferred_fetch=(mode == "deferred"), skip_search_reorder=(mode == "pq"))
                assert np.array_equal(I, G["exp"][key + "_refI"]) and np.array_equal(D, G["exp"][key + "_refD"]), key
                assert np.array_equal(st["n_cmps"], G["exp"][key + "_refcmps"]) and np.array_equal(st["n_hops"], G["exp"][key + "_refhops"])


@pytest.mark.parametrize("metric,R,n_chunks,dim", [("l2", 16, 12, 48), ("mips", 24, 10, 40), ("cosine", 12, 8, 32), ("mips", 32, 17, 51)])
def test_compiled_reference_search_loop_pins_the_oracle_on_fresh_indexes(tmp_path, metric, R, n_chunks, dim, reference):
    """Fresh random indexes (both file layouts), beam widths 1..8, tiny and huge L, io_limit: the restatement follows the
    compiled reference expansion for expansion (hops, I/Os, comparison counts) and returns the same ids."""
    emb = unit_rows(2500, dim, 11 + R)
    emb *= np.random.default_rng(5).uniform(0.6, 1.4, (len(emb), 1)).astype(np.float32)
    prefix, g, coords, pq, codes, max_norm = build_diskann_index(tmp_path, "f", emb, metric=metric, R=R, n_chunks=n_chunks,
                                                                 partition=True, keep_disk_index=True, device="cpu")
    G = dict(g=g)
    q = unit_rows(16, dim, 99)
    o = VamanaOracle(g, pq, codes, metric, max_norm)
    for part in ("", prefix):
        ref = reference.proxy(DiskannFlash, prefix, metric, partition_prefix=part)
        ref.set_embeddings(emb)
        for L, beam, k, io_limit in ((64, 1, 10, 2 ** 32 - 1), (10, 2, 10, 2 ** 32 - 1), (150, 4, 20, 2 ** 32 - 1), (64, 8, 5, 2 ** 32 - 1),
                                     (64, 2, 10, 7), (32, 1, 3, 1)):
            for mode, kw in (("deferred", dict(emb=emb)), ("pq", dict(skip_search_reorder=True))) + \
                            ((("stored", dict(coords=coords)),) if not part else ()):
                rD, rI, rs = ref.search(q, k, L=L, beam_width=beam, deferred_fetch=(mode == "deferred"),
                                        skip_search_reorder=(mode == "pq"), io_limit=io_limit)
                _check_against_reference(o, G, q, k, L, beam, dict(kw, io_limit=io_limit), rD, rI, rs,
                                         f"{metric} R{R} L{L} b{beam} k{k} io{io_limit} {mode} {'partition' if part else 'standard'}")
