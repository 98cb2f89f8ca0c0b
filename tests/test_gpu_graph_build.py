"""GPU graph construction (SURVEY 8f row 1; csrc/graph_build.cu + leann_b200/graph_build.py): the insertion-as-search
builder against (a) a plain restatement of the reference's neighbour-selection heuristic, (b) brute force, and (c) the
exact batch builder, searched with the product's own (parity-checked) stored-vector traversal."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

from helpers import reference  # noqa: E402,F401  (fixture)


def clustered(n, d, n_clusters, seed, spread=0.35):
    rng = np.random.default_rng(seed)
    c = rng.normal(size=(n_clusters, d)).astype(np.float32)
    x = c[rng.integers(0, n_clusters, n)] + spread * rng.normal(size=(n, d)).astype(np.float32)
    return x / np.linalg.norm(x, axis=1, keepdims=True)


def shrink_reference(pd, dn, cand, keep):
    """HNSW::shrink_neighbor_list (faiss/impl/HNSW.cpp:426-468) on one sorted candidate row."""
    kept = []
    for j, c in enumerate(cand):
        if c < 0:
            break
        if all(not (pd[j, i] < dn[j]) for i in kept):
            kept.append(j)
            if len(kept) >= keep:
                break
    return [int(cand[j]) for j in kept]


def test_select_kernel_is_the_reference_heuristic():
    from leann_b200 import capi

    rng = np.random.default_rng(0)
    b, K, keep = 300, 48, 12
    pd = rng.random((b, K, K)).astype(np.float32)
    pd = (pd + pd.transpose(0, 2, 1)) / 2
    dn = np.sort(rng.random((b, K)).astype(np.float32) * 0.8, axis=1)
    cand = np.stack([rng.permutation(10_000)[:K] for _ in range(b)]).astype(np.int32)
    nvalid = rng.integers(1, K + 1, b)
    for r in range(b):
        cand[r, nvalid[r]:] = -1
    for as_f32 in (True, False):
        p = torch.from_numpy(pd).cuda()
        p = p if as_f32 else p.half()
        pref = p.float().cpu().numpy()
        oi = torch.empty((b, keep), dtype=torch.int32, device="cuda")
        od = torch.empty((b, keep), dtype=torch.float32, device="cuda")
        d_dn, d_cand = torch.from_numpy(dn).cuda(), torch.from_numpy(cand).cuda()  # keep the device copies alive across the call
        capi.build_select(p.data_ptr(), as_f32, d_dn.data_ptr(), d_cand.data_ptr(), b, K, keep, oi.data_ptr(), od.data_ptr())
        torch.cuda.synchronize()
        got = oi.cpu().numpy()
        for r in range(b):
            want = shrink_reference(pref[r], dn[r], cand[r], keep)
            assert got[r, :len(want)].tolist() == want and (got[r, len(want):] == -1).all()
        # fill: rejected candidates, nearest first, top the list up to the floor
        capi.build_select(p.data_ptr(), as_f32, d_dn.data_ptr(), d_cand.data_ptr(), b, K, keep, oi.data_ptr(), od.data_ptr(), fill=8)
        torch.cuda.synchronize()
        got = oi.cpu().numpy()
        for r in range(b):
            want = shrink_reference(pref[r], dn[r], cand[r], keep)
            rest = [int(c) for c in cand[r] if c >= 0 and int(c) not in want]
            want = want + rest[: max(0, 8 - len(want))]
            assert got[r, :len(want)].tolist() == want and (got[r, len(want):] == -1).all()


def _device_graph(g, M, dev):
    from leann_b200.graph_build import upper_level_arrays
    from leann_b200.graph_refine import level0_padded, upper_levels

    adj0 = torch.from_numpy(level0_padded(g, 2 * M)[:, :2 * M].astype(np.int32)).to(dev)
    up_row, up_adj = upper_level_arrays(g.levels, upper_levels(g, M), M, dev)
    return adj0.contiguous(), up_row, up_adj


def test_insert_search_finds_the_nearest_neighbours():
    from leann_b200 import capi
    from leann_b200.graph_build import build_hnsw_graph

    n, d, M, ef = 20000, 64, 16, 96
    x = clustered(n, d, 200, 1)
    g = build_hnsw_graph(x, M=M, metric="mips", device="cuda")
    adj0, up_row, up_adj = _device_graph(g, M, "cuda")
    xs = torch.from_numpy(x).cuda().half().contiguous()
    pts = torch.arange(0, 2048, dtype=torch.int32, device="cuda")
    oi = torch.empty((pts.numel(), ef), dtype=torch.int32, device="cuda")
    od = torch.empty((pts.numel(), ef), dtype=torch.float32, device="cuda")
    wb = capi.build_workspace_bytes(ef, 2 * M)
    ws = torch.empty(wb, dtype=torch.uint8, device="cuda")
    for metric_ip in (True, False):
        capi.build_insert_search(xs.data_ptr(), n, d, metric_ip, adj0.data_ptr(), 2 * M, up_row.data_ptr(), up_adj.data_ptr(), M,
                                 g.entry_point, g.max_level, pts.data_ptr(), pts.numel(), ef, oi.data_ptr(), od.data_ptr(),
                                 ws.data_ptr(), wb)
        torch.cuda.synchronize()
        ids, dist = oi.cpu().numpy(), od.cpu().numpy()
        xh = xs.float()
        ip = xh[:2048] @ xh.T
        ref = -ip if metric_ip else (2 - 2 * ip)  # unit vectors
        ref[torch.arange(2048), torch.arange(2048)] = float("inf")
        top = torch.topk(ref, 10, dim=1, largest=False)
        # sorted ascending, no self, no repeats, distances are the true ones
        assert (np.diff(dist, axis=1)[ids[:, 1:] >= 0] >= 0).all()
        assert not (ids == np.arange(2048)[:, None]).any()
        for r in range(0, 2048, 97):
            row = ids[r][ids[r] >= 0]
            assert len(set(row.tolist())) == len(row)
            np.testing.assert_allclose(dist[r][: len(row)], ref[r, torch.from_numpy(row).long().cuda()].cpu().numpy(), atol=2e-3)
        rec = np.mean([len(set(a.tolist()) & set(b.tolist())) / 10 for a, b in zip(ids[:, :10], top.indices.cpu().numpy())])
        assert rec > 0.9, rec


def _recall_with_product_search(g, x, q, gt, tmp_path, name):
    from leann_b200 import capi, csr

    f = tmp_path / f"{name}.index"
    csr.write_compact_index(str(f), g)
    idx = capi.Index(str(f), 0)
    idx.set_vectors(x)
    _, I = idx.search(q, 10, capi.make_params(64, recompute=False))
    idx.close()
    return float(np.mean([len(set(a.tolist()) & set(b.tolist())) / 10 for a, b in zip(I, gt)]))


def test_incremental_builder_matches_the_exact_builder(tmp_path):
    from leann_b200.graph_build import build_hnsw_graph, build_hnsw_graph_incremental
    from leann_b200.graph_refine import level0_padded

    n, d, M = 60000, 64, 16
    x = clustered(n, d, 600, 2)
    q = clustered(512, d, 600, 2)  # same cluster centres (same seed), fresh noise is not needed for a recall comparison
    q = x[:512] + 0.05 * np.random.default_rng(3).normal(size=(512, d)).astype(np.float32)
    q /= np.linalg.norm(q, axis=1, keepdims=True)
    gt = np.argsort(-(q @ x.T), axis=1)[:, :10]
    g_exact = build_hnsw_graph(x, M=M, metric="mips", device="cuda")
    g_inc = build_hnsw_graph_incremental(x, M=M, metric="mips", device="cuda", ef_construction=100, growth=0.25, min_seed=4000)
    # structural invariants of an HNSW graph in the reference's format
    assert g_inc.ntotal == n and np.array_equal(g_inc.levels, g_exact.levels) and g_inc.entry_point == g_exact.entry_point
    l0 = level0_padded(g_inc, 2 * M)
    assert l0.shape[1] == 2 * M  # never more than 2M links on level 0
    deg = (l0 >= 0).sum(1)
    assert deg.min() >= 1 and l0.max() < n
    assert not (l0 == np.arange(n)[:, None]).any()
    srt = np.sort(l0, axis=1)
    assert not ((srt[:, 1:] == srt[:, :-1]) & (srt[:, 1:] >= 0)).any()
    r_exact = _recall_with_product_search(g_exact, x, q, gt, tmp_path, "exact")
    r_inc = _recall_with_product_search(g_inc, x, q, gt, tmp_path, "inc")
    print(f"recall@10 ef=64: exact builder {r_exact:.3f}, insertion builder {r_inc:.3f}, mean degree {deg.mean():.1f}")
    assert r_inc > r_exact - 0.03 and r_inc > 0.9


def builder_points(n, d):
    x = clustered(n, d, 1000, 5)
    q = x[:1000] + 0.05 * np.random.default_rng(6).normal(size=(1000, d)).astype(np.float32)
    return x, q / np.linalg.norm(q, axis=1, keepdims=True)


def reference_builder_recall(n, d, M, efc):
    """recall@10 at efSearch 64 of the graph that the reference's own HNSW::add_with_locks (compiled, oracle/_ref) builds over
    builder_points(n, d), searched with the C restatement of the traversal (ids bit-identical to the product's stored-vector
    search, see test_gpu_search.py), and the graph's links per node."""
    from oracle.binding import Oracle, Reference, export_to_csr

    x, q = builder_points(n, d)
    ref = Reference(x.shape[1], M, True)
    ref.build(x, ef_construction=efc, nthreads=32)
    g = export_to_csr(ref.export())
    _, I, _, _ = Oracle(g, x).search(q, 10, ef=64, nthreads=32)
    gt = np.argsort(-(q @ x.T), axis=1)[:, :10]
    return float(np.mean([len(set(a.tolist()) & set(b.tolist())) / 10 for a, b in zip(I, gt)])), g.neighbors.size / len(x)


def test_incremental_builder_against_the_reference_builder(tmp_path, reference):
    """Same points, same levels' distribution, same M / efConstruction: the graph from the GPU insertion builder, searched
    with the product's stored-vector traversal at efSearch 64, and the graph from the reference's own HNSW::add_with_locks
    (its recall replayed from tests/golden/reference_replay/, see reference_builder_recall).  Construction is order- and
    thread-dependent in the reference too, so the comparison is on what the graph is for: recall, and the work a search
    does on it."""
    from leann_b200.graph_build import build_hnsw_graph_incremental

    n, d, M, efc = 100_000, 64, 16, 100
    x, q = builder_points(n, d)
    gt = torch.topk(torch.from_numpy(q).cuda() @ torch.from_numpy(x).cuda().T, 10, dim=1).indices.cpu().numpy()
    r_ref, links_ref = reference.proxy(reference_builder_recall, n, d, M, efc)
    g_inc = build_hnsw_graph_incremental(x, M=M, metric="mips", device="cuda", ef_construction=efc)
    r_inc = _recall_with_product_search(g_inc, x, q, gt, tmp_path, "inc")
    print(f"recall@10 ef=64: reference builder {r_ref:.3f} ({links_ref:.1f} links/node), "
          f"GPU insertion builder {r_inc:.3f} ({g_inc.neighbors.size / n:.1f} links/node)")
    assert r_inc > r_ref - 0.02
