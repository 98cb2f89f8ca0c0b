"""Driver for the ncu capture of the two traversal kernels (no encoder in the profiled launches):
  hnsw_step_kernel      stored-vector HNSW search (recompute_embeddings=False), persistent
  vamana_search_kernel  DiskANN PQ beam search (skip_search_reorder, no deferred fetch), persistent
usage: traversal_profile.py [chunks] [queries]"""
import sys, tempfile, time
from pathlib import Path
import numpy as np, torch
sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
from leann_b200 import capi, csr, synth, build
from leann_b200.graph_build import build_hnsw_graph
from leann_b200.vamana_build import build_diskann_index
from leann_b200.tooling import stub_graph, recall_at_k
if build.needs_build(): build.build()
N = int(sys.argv[1]) if len(sys.argv) > 1 else 400_000
NQ = int(sys.argv[2]) if len(sys.argv) > 2 else 8192
preset = synth.MINILM_L6
blob = synth.pack_weights(preset, synth.synthetic_weights(preset, 0))
tm, corpus = synth.make_corpus(N, preset.vocab_size, seed=1234, max_len=preset.max_pos)
queries = synth.make_queries(tm, NQ, seed=4321)
work = Path(tempfile.mkdtemp())
csr.write_compact_index(str(work / "stub.index"), stub_graph(N, 384))
enc = capi.Index(str(work / "stub.index"), 0)
enc.set_passages(corpus.tokens, corpus.offsets); enc.set_encoder(preset.config(), blob)
E = torch.empty((N, 384), dtype=torch.float32, device="cuda")
enc.encode_range_device(0, N, E.data_ptr())
Q = enc.encode_tokens(queries.tokens, queries.offsets); enc.close()
gt = torch.topk(torch.from_numpy(Q).cuda() @ E.T, 10, dim=1).indices.cpu().numpy()
g = build_hnsw_graph(E, M=32, metric="mips")
csr.write_compact_index(str(work / "g.index"), g)
idx = capi.Index(str(work / "g.index"), 0); idx.set_vectors_device(E.data_ptr())
for _ in range(2):
    D, I = idx.search(Q, 10, capi.make_params(64, recompute=False))
st = idx.last_stats
deg = g.neighbors.size / N
byts = st.nhops * (32 + 4 * deg + deg / 8) + (st.ndis + NQ) * (384 * 4 + 8)
print(f"hnsw stored: {NQ/(st.gpu_ms/1e3):.0f} q/s, recall {recall_at_k(I, gt):.3f}, algorithmic {byts/1e6:.1f} MB per launch -> {byts/(st.gpu_ms/1e3)/1e9:.0f} GB/s", flush=True)
idx.close()
prefix, vg, coords, pq, codes, mx = build_diskann_index(work, "da", E.cpu().numpy(), metric="mips", R=32, partition=True, keep_disk_index=False)
da = capi.DiskannIndex(prefix, "mips", prefix, 0)
for _ in range(2):
    D, I = da.search(Q, 10, capi.make_diskann_params(64, 1, recompute_embeddings=False, skip_search_reorder=True))
st = da.last_stats
byts = st.n_requested * (4 * 32 + 4) + st.ndis * pq.n_chunks
print(f"vamana pq-only: {NQ/(st.gpu_ms/1e3):.0f} q/s, recall(pq order) {recall_at_k(I, gt):.3f}, {st.n_requested/NQ:.0f} expansions, {st.ndis/NQ:.0f} PQ comparisons per query, "
      f"{pq.n_chunks} B codes; algorithmic {byts/1e6:.1f} MB per launch -> {byts/(st.gpu_ms/1e3)/1e9:.0f} GB/s", flush=True)
