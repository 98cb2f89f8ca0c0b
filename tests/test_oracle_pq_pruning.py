"""PQ-guided pruning of the HNSW search (SURVEY 8f row 3; faiss/impl/HNSW_search.cpp:442-465, 645-750 + impl/pq.cpp):
the C restatement (oracle/hnsw_oracle.c) against the reference's own compiled code (oracle/_ref/libleann_ref.so with
HNSW::load_pq_pruning_data reading DiskANN-format PQ files; its outputs replayed from tests/golden/reference_replay/) — ids,
distances, ndis, nhops identical for the three selection strategies (global / local / proportional), beams, batch mode and
both metrics."""
import numpy as np
import pytest

from leann_b200.graph_build import build_hnsw_graph
from leann_b200.vamana_build import build_diskann_index
from helpers import reference  # noqa: F401  (fixture)
from oracle.binding import Oracle, Reference

PRUNE_CASES = [  # (prune_ratio, local_prune, send_ratio, ef, beam, batch, check_rel, k)
    (0.5, False, 0.0, 32, 1, 0, True, 10), (0.8, False, 0.0, 64, 1, 0, True, 10), (0.3, False, 0.0, 24, 4, 0, True, 5),
    (0.5, True, 0.0, 32, 1, 0, True, 10), (0.0, True, 0.0, 32, 2, 0, True, 10), (0.7, True, 0.0, 48, 3, 0, False, 10),
    (0.5, False, 1.0, 32, 1, 0, True, 10), (0.25, False, 2.5, 64, 2, 0, True, 20), (0.0, False, 1.0, 16, 1, 0, True, 10),
    (0.5, False, 0.0, 32, 1, 24, True, 10), (0.6, True, 0.0, 32, 1, 40, True, 10),
]


def make_world(tmp_path, metric, n=4000, d=32, n_chunks=16, seed=0):
    rng = np.random.default_rng(seed)
    cen = rng.standard_normal((24, d)).astype(np.float32)
    x = cen[rng.integers(0, 24, n)] + 0.5 * rng.standard_normal((n, d)).astype(np.float32)
    x /= np.linalg.norm(x, axis=1, keepdims=True)
    q = x[:24] + 0.15 * rng.standard_normal((24, d)).astype(np.float32)
    q /= np.linalg.norm(q, axis=1, keepdims=True)
    g = build_hnsw_graph(x, M=8, metric=metric, device="cpu")
    # the pruning tables are DiskANN PQ files over the MIPS-extended base (d + 1 coordinates): the reference appends a zero
    # to the query and normalises it before the table look-up (HNSW_search.cpp:447-456)
    prefix, _, _, pq, codes, _ = build_diskann_index(tmp_path, f"pq_{metric}", x, metric="mips", R=8, n_chunks=n_chunks, device="cpu")
    return dict(x=x, q=q, g=g, pq=pq, codes=codes, prefix=prefix)


@pytest.mark.parametrize("metric", ["mips", "l2"])
def test_pq_pruning_restatement_matches_the_compiled_reference(tmp_path, metric, reference):
    W = make_world(tmp_path, metric)
    ref = reference.proxy(Reference.from_csr, W["g"], W["x"], M=8)
    ref.load_pq(W["prefix"] + "_pq_pivots.bin", W["prefix"] + "_pq_compressed.bin")
    o = Oracle(W["g"], W["x"])
    o.set_pq(W["pq"], W["codes"])
    base = ref.search(W["q"], 10, ef=32)
    saved = 0
    for pr, lp, sr, ef, beam, bs, cr, k in PRUNE_CASES:
        a = ref.search(W["q"], k, ef=ef, beam=beam, batch_size=bs, check_rel=cr, prune_ratio=pr, local_prune=lp, send_ratio=sr)
        b = o.search(W["q"], k, ef=ef, beam=beam, batch_size=bs, check_rel=cr, prune_ratio=pr, local_prune=lp, send_ratio=sr)
        for name, u, v in zip(("D", "I", "ndis", "nhops"), a, b):
            assert np.array_equal(u, v), (metric, pr, lp, sr, ef, beam, bs, cr, k, name)
        saved += int(a[2].sum() < ref.search(W["q"], k, ef=ef, beam=beam, batch_size=bs, check_rel=cr)[2].sum())
    assert saved >= 6  # pruning does cut the number of exact distance computations
    # with PQ data loaded but no pruning requested the default branch runs (perform_pq_pruning false, :442-445)
    for u, v in zip(base, o.search(W["q"], 10, ef=32)):
        assert np.array_equal(u, v)


def test_pq_lookup_table_matches_the_reference_bit_for_bit(tmp_path, reference):
    """lbo_pq_lut / lbo_pq_dist against a search that is driven entirely by the table: with local pruning at ratio ~0 nothing
    is selected unless ... instead compare through ndis of many ratios: covered above; here: odd chunk widths and a PQ
    whose dimension is not d + 1 aligned."""
    W = make_world(tmp_path, "mips", n=1500, d=20, n_chunks=7, seed=3)
    ref = reference.proxy(Reference.from_csr, W["g"], W["x"], M=8)
    ref.load_pq(W["prefix"] + "_pq_pivots.bin", W["prefix"] + "_pq_compressed.bin")
    o = Oracle(W["g"], W["x"])
    o.set_pq(W["pq"], W["codes"])
    for pr in (0.1, 0.45, 0.9):
        for kw in (dict(), dict(local_prune=True), dict(send_ratio=1.0)):
            a = ref.search(W["q"], 10, ef=40, prune_ratio=pr, **kw)
            b = o.search(W["q"], 10, ef=40, prune_ratio=pr, **kw)
            for u, v in zip(a, b):
                assert np.array_equal(u, v), (pr, kw)
