#!/usr/bin/env python
"""Benchmark of the selective-recompute HNSW search path (BASELINE.json metric:
QPS @ recall@10, 10 M x 384 d, MiniLM-L6, efSearch ("beam") = 64).

    python bench.py --gpus N --steps K --warmup W                    # this repo (one rank per GPU under torchrun)
    python bench.py --impl reference --gpus N --steps K --warmup W   # the reference's CPU path, rank 0 only

One "step" = one Searcher.search() call of the plugin backend over one batch of synthetic queries per GPU
(recompute mode: traversal + encoder forward for every hop's new nodes + scoring, k=10, ef=64), HOST query
buffer in, HOST labels/distances out.  Both numbers come from the same K steps: `e2e` is the wall clock of
the calls (host<->device copies inside), `value` is the device time of the search inside them
(lb2_search_stats.gpu_ms: CUDA events on the launching stream, queries already in HBM).

Set-up (untimed, synthetic, seeded) is built ONCE per box and cached on disk ($LB2_CACHE, default
/tmp/lb2_cache/<config key>): topic-structured token corpus -> passage embeddings with the GPU encoder ->
HNSW graph by GPU insertion-as-search (leann_b200/graph_build.py + csrc/graph_build.cu) written in the
reference's CSR .index format -> query pool + exact ground truth.  Rank 0 (or the reference arm, whichever
runs first) builds it; every other process waits for the DONE marker and maps the files.
Prints ONE JSON line (rank 0).
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

METRIC = "QPS @ recall@10 (HNSW selective recompute, all-MiniLM-L6-v2 384d, efSearch=64, k=10)"
WORLD_VERSION = "w4"  # bump when the corpus generator / graph builder changes what a cached world holds
K = 10
DUMP_QUERIES = 1024  # queries per step per GPU of a --dump-outputs run without --queries


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--chunks", type=int, default=int(os.environ.get("LB2_BENCH_CHUNKS", 10_000_000)))
    ap.add_argument("--queries", type=int, default=int(os.environ.get("LB2_BENCH_QUERIES", 0)),
                    help="queries per step per GPU; 0 = sized from --budget-s after a calibration call "
                         f"({DUMP_QUERIES} with --dump-outputs, so that the inputs do not depend on a timing)")
    ap.add_argument("--budget-s", type=float, default=float(os.environ.get("LB2_BENCH_BUDGET_S", 300)),
                    help="wall budget of the warm-up + timed steps (sizes --queries when that is 0)")
    ap.add_argument("--ref-budget-s", type=float, default=float(os.environ.get("LB2_BENCH_REF_BUDGET_S", 300)),
                    help="reference arm: serial CPU queries are timed until this much wall time is used")
    ap.add_argument("--ef", type=int, default=64)
    ap.add_argument("--beam", type=int, default=1)
    ap.add_argument("--efc", type=int, default=int(os.environ.get("LB2_BENCH_EFC", 200)), help="efConstruction of the graph build")
    ap.add_argument("--sweeps", type=int, default=int(os.environ.get("LB2_BENCH_SWEEPS", 0)), help="graph build: repair sweeps")
    ap.add_argument("--ems", action="store_true", help="degree-pruned graph (configs[4] variant): top 2 %% of nodes by in-degree keep "
                    "2M level-0 links, the others 6-7 (graph_refine.prune_degrees = the reference's ems policy); not the headline")
    ap.add_argument("--pool", type=int, default=65536, help="size of the query pool (with exact ground truth)")
    ap.add_argument("--slots", type=int, default=int(os.environ.get("LB2_SLOTS", 1024)))
    ap.add_argument("--per-pass", type=int, default=int(os.environ.get("LB2_PER_PASS", 0)))
    ap.add_argument("--cache", default=os.environ.get("LB2_CACHE", "/tmp/lb2_cache"))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--extras", action="store_true", help="call-scope de-duplication and stored-vector (traversal-only) side measurements")
    ap.add_argument("--diskann", action="store_true", help="extra: the DiskANN/Vamana path over the same corpus")
    ap.add_argument("--rebuild", action="store_true", help="ignore a cached world")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one returned to the "
                    "caller as DIR/labels.npy (float64 passage ids, -1 = none) and DIR/distances.npy (float32), [queries, k]")
    return ap.parse_args()


def log(*a):
    if int(os.environ.get("RANK", 0)) == 0:
        print("[bench]", *a, file=sys.stderr, flush=True)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, gpu_index: int):
        self.rows = []
        self.proc = None
        self.gpu = gpu_index

    def start(self):
        q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", str(self.gpu)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm = [float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 9:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------ world
def world_dir(args) -> Path:
    from leann_b200 import synth

    cfg = {"v": WORLD_VERSION, "chunks": args.chunks, "model": synth.MINILM_L6.name, "M": 32, "efc": args.efc,
           "sweeps": args.sweeps, "pool": args.pool}
    if getattr(args, "ems", False):
        cfg["ems"] = "top2pct_in_degree_keep_2M_else_6_7"
    key = json.dumps(cfg, sort_keys=True)
    return Path(args.cache) / f"c{args.chunks}_{hashlib.sha1(key.encode()).hexdigest()[:12]}"


def exact_ground_truth(Q: np.ndarray, E, k: int = K, block: int = 2048):
    """Exact top-k by inner product over all passages (benchmarks/run_evaluation.py:358-367 with k=10): fp16 tensor-core
    scores shortlist 1 024 candidates per query (16 groups of 64 columns by group maximum — the top-k lie in the k best
    groups), which are re-scored in fp32."""
    import torch

    dev = E.device
    n, d = E.shape
    G = 64
    npad = (n + G - 1) // G * G
    Eh = torch.zeros((npad, d), dtype=torch.float16, device=dev)
    Eh[:n] = E
    out = np.empty((Q.shape[0], k), np.int64)
    Qt = torch.from_numpy(np.ascontiguousarray(Q)).to(dev)
    block = max(64, min(block, (24 << 30) // (2 * npad)))
    for b0 in range(0, Qt.shape[0], block):
        q = Qt[b0:b0 + block]
        s = q.half() @ Eh.T
        if npad > n:
            s[:, n:] = float("-inf")
        gm = s.view(q.shape[0], npad // G, G).amax(2)
        del s
        ng = min(16, gm.shape[1])
        grp = torch.topk(gm, ng, dim=1).indices                                    # [b, 16]
        cand = (grp[:, :, None] * G + torch.arange(G, device=dev)[None, None, :]).reshape(q.shape[0], -1).clamp(max=n - 1)
        sc = torch.bmm(E[cand], q.unsqueeze(2)).squeeze(2)                          # fp32 re-score
        # a clamped (out-of-range) column repeats id n-1: keep one copy
        srt, o = torch.sort(cand, dim=1)
        dup = torch.zeros_like(srt, dtype=torch.bool)
        dup[:, 1:] = srt[:, 1:] == srt[:, :-1]
        sc = torch.gather(sc, 1, o).masked_fill(dup, float("-inf"))
        top = torch.topk(sc, k, dim=1).indices
        out[b0:b0 + block] = torch.gather(srt, 1, top).cpu().numpy()
    return out


def build_world(args, wd: Path, device: int):
    """Untimed set-up on one GPU; writes the index directory + query pool + ground truth into `wd`."""
    import torch
    from leann_b200 import capi, csr, synth
    from leann_b200.graph_build import build_hnsw_graph, build_hnsw_graph_incremental
    from leann_b200.tooling import stub_graph, write_leann_index

    torch.cuda.set_device(device)
    wd.mkdir(parents=True, exist_ok=True)
    preset = synth.MINILM_L6
    info = {"chunks": args.chunks, "version": WORLD_VERSION}
    t0 = time.time()
    weights = synth.synthetic_weights(preset, 0)
    blob = synth.pack_weights(preset, weights)
    tm, corpus, queries = synth.make_bench_corpus(args.chunks, preset.vocab_size, preset.max_pos, f"cuda:{device}", args.pool)
    info["corpus_s"] = time.time() - t0
    log(f"corpus: {corpus.n} chunks, {corpus.tokens.size/1e6:.1f} M tokens, {tm.n_topics} topics ({info['corpus_s']:.1f}s)")
    # 1. passage embeddings with the GPU encoder (stub graph: the encoder needs an open index handle)
    stub = wd / "stub.index"
    csr.write_compact_index(str(stub), stub_graph(corpus.n, preset.hidden))
    enc = capi.Index(str(stub), device)
    enc.set_passages(corpus.tokens, corpus.offsets)
    enc.set_encoder(preset.config(), blob)
    E = torch.empty((corpus.n, preset.hidden), dtype=torch.float32, device=f"cuda:{device}")
    torch.cuda.synchronize()
    t1 = time.time()
    enc.encode_range_device(0, corpus.n, E.data_ptr())
    torch.cuda.synchronize()
    t_embed = time.time() - t1
    lens = np.minimum(np.diff(corpus.offsets.astype(np.int64)), preset.max_pos)
    embed_flops = float(sum(preset.flops_per_chunk(int(L)) * c for L, c in zip(*np.unique(lens, return_counts=True))))
    info.update(embed_s=t_embed, embed_tflops=embed_flops / t_embed / 1e12, mean_len=float(lens.mean()))
    log(f"embedded corpus in {t_embed:.1f}s = {info['embed_tflops']:.0f} TFLOP/s algorithmic (encoder only)")
    Q = enc.encode_tokens(queries.tokens, queries.offsets)
    enc.close()
    stub.unlink()
    # 2. graph in the reference's CSR format
    t2 = time.time()
    if corpus.n >= 50_000:
        g = build_hnsw_graph_incremental(E, M=32, metric="mips", device=f"cuda:{device}", ef_construction=args.efc,
                                         sweeps=args.sweeps, verbose=bool(os.environ.get("LB2_BENCH_VERBOSE")))
        info["graph_builder"] = f"gpu insertion-as-search, efConstruction={args.efc}, sweeps={args.sweeps}"
    else:
        g = build_hnsw_graph(E, M=32, metric="mips", device=f"cuda:{device}")
        info["graph_builder"] = "exact batch builder (small corpus)"
    if getattr(args, "ems", False):
        from leann_b200.graph_refine import prune_degrees
        full_edges = int(g.neighbors.size)
        g, _ = prune_degrees(E, g, M=32, device=f"cuda:{device}")
        info["graph_builder"] += f" + high-degree-preserving pruning (top 2 % keep 64 links, others 6-7; {full_edges} -> {int(g.neighbors.size)} edges)"
    torch.cuda.synchronize()
    info.update(graph_s=time.time() - t2, edges=int(g.neighbors.size), max_level=int(g.max_level))
    log(f"graph: {g.neighbors.size/1e6:.1f} M edges, max_level {g.max_level} ({info['graph_s']:.1f}s)")
    write_leann_index(wd, "bench", g, preset, corpus)
    # 3. exact ground truth over the same embeddings
    t3 = time.time()
    gt = exact_ground_truth(Q, E)
    info["gt_s"] = time.time() - t3
    np.save(wd / "Q.npy", Q)
    np.save(wd / "gt.npy", gt)
    if args.extras or os.environ.get("LB2_BENCH_KEEP_E"):
        np.save(wd / "E.npy", E.cpu().numpy())
    info["total_s"] = time.time() - t0
    (wd / "world.json").write_text(json.dumps(info))
    (wd / "DONE").write_text("ok")
    log(f"world built in {info['total_s']:.0f}s -> {wd}")
    del E
    torch.cuda.empty_cache()


def ensure_world(args, builder: bool, device: int) -> Path:
    wd = world_dir(args)
    done = wd / "DONE"
    if args.rebuild and builder and done.exists():
        done.unlink()
    if not done.exists():
        if builder:
            build_world(args, wd, device)
        else:
            t0 = time.time()
            while not done.exists():
                if time.time() - t0 > 1500:
                    raise RuntimeError(f"timed out waiting for rank 0 to build {wd}")
                time.sleep(1.0)
    return wd


def library_rendezvous(build, rank: int, world: int, cache: str, timeout_s: float = 900.0):
    """Rank 0 (re)builds libleann_b200.so when its sources are newer; under torchrun the other ranks must not dlopen a
    half-linked file, so they wait for a marker that rank 0 writes once the library is in place (one marker per launch:
    the ranks of a launch share MASTER_PORT and their parent, the elastic agent)."""
    if world == 1:
        if build.needs_build():
            build.build()
        return
    marker = Path(cache) / f".lib_ready_{os.environ.get('MASTER_PORT', '0')}_{os.getppid()}"
    if rank == 0:
        if build.needs_build():
            build.build()
        marker.parent.mkdir(parents=True, exist_ok=True)
        marker.write_text(str(time.time()))
    else:
        t0 = time.time()
        while not marker.exists():
            if time.time() - t0 > timeout_s:
                raise RuntimeError(f"timed out waiting for rank 0 to provide the library ({marker})")
            time.sleep(0.2)


def load_world(wd: Path):
    from leann_b200 import synth

    info = json.loads((wd / "world.json").read_text())
    return dict(dir=wd, index_path=wd / "bench.leann", Q=np.load(wd / "Q.npy", mmap_mode="r"), gt=np.load(wd / "gt.npy"),
                info=info, preset=synth.MINILM_L6)


def synth_corpus_params():
    from leann_b200 import synth
    return synth.BENCH_CORPUS


def workload_string(args, W, nq, extra=""):
    c = synth_corpus_params()
    return (f"{args.chunks} synthetic chunks (mean {W['info']['mean_len']:.0f} tokens; topic model: {c['topic_size']} chunks/topic, "
            f"{c['p_topic']:.2f}/{c['p_super']:.2f} topic/super-topic token share), all-MiniLM-L6-v2 384d architecture with "
            f"seeded synthetic weights, HNSW M=32 recompute ({W['info'].get('graph_builder', '?')}), efSearch={args.ef}, "
            f"beam_width={args.beam}, k={K}, {nq} queries/step/GPU{extra}")


# ------------------------------------------------------------------------------------------------ this repo's arm
def run_b200(args):
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    os.environ.setdefault("LB2_PROFILE_GEMM", "1")
    from leann_b200 import backend, build
    from leann_b200.tooling import recall_at_k

    library_rendezvous(build, rank, world, args.cache)
    wd = ensure_world(args, builder=(rank == 0), device=local)  # file-system rendezvous BEFORE the process group exists
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    W = load_world(wd)
    t_open = time.time()
    searcher = backend.B200HnswBackend.searcher(str(W["index_path"]), device=local, slots=args.slots,
                                                passages_per_pass=args.per_pass or None, shard_queries=(world > 1))
    port = searcher._ensure_server_running(str(W["index_path"]) + ".meta.json", 5557)
    log(f"index open + passages + encoder attached in {time.time()-t_open:.1f}s")
    P, d = W["Q"].shape
    dev = torch.device("cuda", local)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def call(q_host):
        return searcher.search(q_host, K, zmq_port=port, complexity=args.ef, beam_width=args.beam, recompute_embeddings=True)

    # ---- size the step from the wall budget: one calibration call of 256 queries per GPU
    Qpool = np.ascontiguousarray(W["Q"])
    nq = args.queries
    if nq <= 0 and args.dump_outputs:
        nq = min(DUMP_QUERIES, P // world)
    if nq <= 0:
        ncal = 256
        qc = Qpool[np.arange(world * ncal) % P]
        barrier()
        t0 = time.perf_counter()
        call(qc)
        dt = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        qps_cal = ncal / float(dt.item())
        nq = int(qps_cal * args.budget_s / max(1, args.steps + args.warmup)) // 64 * 64
        nq = max(64, min(2048, nq, P // world))
        log(f"calibration: {ncal} queries/GPU in {float(dt.item()):.2f}s -> {nq} queries/step/GPU for a {args.budget_s:.0f}s budget")
    gq = world * nq  # global batch of a step
    pinned = torch.empty((gq, d), dtype=torch.float32).pin_memory()

    def batch_ids(step):
        return (step * gq + np.arange(gq)) % P

    agg = dict(gpu_ms=0.0, encoder_ms=0.0, gemm_ms=0.0, gemm_flops=0.0, attention_ms=0.0, norm_ms=0.0, launches=0, ndis=0, nhops=0,
               n_recomputed=0, n_requested=0, n_tokens=0, steps=0, passes=0)
    for s in range(args.warmup):
        pinned.copy_(torch.from_numpy(Qpool[batch_ids(s)]))
        flush.fill_(s & 0xFF)
        call(pinned.numpy())
    clocks = ClockSampler(local)
    recalls = []
    barrier()
    clocks.start()
    t_begin = time.perf_counter()
    t_calls = 0.0
    for s in range(args.warmup, args.warmup + args.steps):
        ids = batch_ids(s)
        pinned.copy_(torch.from_numpy(Qpool[ids]))   # host-side staging of the step's input (pinned)
        flush.fill_(s & 0xFF)                        # L2 flush between timed iterations
        torch.cuda.synchronize()
        tc = time.perf_counter()
        out = call(pinned.numpy())                   # H2D + search (+ NCCL gather) + D2H
        t_calls += time.perf_counter() - tc
        st = searcher.last_stats
        for key in ("gpu_ms", "encoder_ms", "gemm_ms", "gemm_flops", "attention_ms", "norm_ms", "ndis", "nhops", "n_recomputed",
                    "n_requested", "n_tokens"):
            agg[key] += st[key]
        agg["launches"] += st["n_kernel_launches"]
        agg["steps"] += st["n_steps"]
        agg["passes"] += st["n_encoder_passes"]
        I = np.array([[int(x) for x in row] for row in out["labels"]], np.int64)
        recalls.append(recall_at_k(I, W["gt"][ids]))
    barrier()
    t_wall = time.perf_counter() - t_begin
    clk = clocks.stop()
    if args.dump_outputs and rank == 0 and args.steps > 0:
        dump_outputs(Path(args.dump_outputs), out)
    red = torch.tensor([agg["gpu_ms"] / 1e3, t_calls, t_wall], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(red, op=dist.ReduceOp.MAX)
    t_dev, t_e2e, t_wall = (float(v) for v in red.tolist())
    total_q = gq * args.steps
    value = total_q / t_dev
    e2e_value = total_q / t_e2e

    extras = {}
    if args.extras and rank == 0:
        extras = run_extras(args, W, searcher, local, flush)
    diskann = None
    if args.diskann and rank == 0:
        try:
            diskann = diskann_extra(W, args, local, flush, K)
        except Exception as e:
            diskann = {"error": repr(e)}

    out = None
    if rank == 0:
        peaks = {}
        try:
            peaks = json.loads((ROOT / "MEASURED_PEAKS.json").read_text())
        except Exception:
            pass
        peak = peaks.get("bf16_tflops_sustained") or peaks.get("bf16_tflops") or 1590.0
        peak_src = "measured (MEASURED_PEAKS.json bf16_tflops_sustained, cuBLAS bf16 sustained)" if peaks else "fallback 1590"
        gemm_tf = agg["gemm_flops"] / (agg["gemm_ms"] / 1e3) / 1e12 if agg["gemm_ms"] > 0 else None
        traffic, tr_ratio, tr_name = None, float("nan"), "none"
        try:  # DRAM bytes per GEMM launch = algorithmic bytes x the dram/algorithmic ratio of the committed ncu --set full capture
            tr_file = ROOT / "profiles" / "r02_gemm_traffic.json"
            if not tr_file.exists():
                tr_file = ROOT / "profiles" / "r01_final_gemm_traffic.json"
            tr = json.loads(tr_file.read_text())
            p_ = W["preset"]
            h, f = p_.hidden, p_.ffn
            bytes_tok_layer = 2 * ((h + 3 * h) + (3 * h) + (h + f) + (f + 2 * h))
            n_gemm = agg["passes"] * 4 * p_.layers
            if n_gemm > 0:
                traffic = agg["n_tokens"] * p_.layers * bytes_tok_layer * tr["dram_over_algorithmic"] / n_gemm
            tr_ratio, tr_name = tr["dram_over_algorithmic"], "profiles/" + tr_file.name
        except Exception:
            pass
        nqs = nq * args.steps  # this rank's queries (stats are per rank)
        mean_len = agg["n_tokens"] / max(1, agg["n_recomputed"])
        enc_flops = agg["n_recomputed"] * W["preset"].flops_per_chunk(int(round(mean_len)))
        out = {
            "metric": METRIC, "value": value, "unit": "queries/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": t_dev / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f16 (fp32 accumulate; fp32 scoring)", "data": "synthetic",
            "config": {"workload": workload_string(args, W, nq),
                       "l2": "256 MiB flush buffer written between timed steps; working set (graph+passages) > L2",
                       "queries": f"pool of {P} distinct queries with exact ground truth, consecutive slices per step and rank",
                       "parallelism": f"queries sharded over {world} GPU(s), graph/passages/encoder replicated, one NCCL all_gather of results"},
            "recall_at_10": float(np.mean(recalls)),
            "e2e": {"value": e2e_value, "unit": "queries/s", "h2d_bytes_per_step": gq * d * 4, "d2h_bytes_per_step": gq * K * 12,
                    "api": "B200HnswSearcher.search (the LEANN plugin call): pinned host queries in, host labels + distances out",
                    "wall_s_timed_region": t_wall},
            "gpu_launches": int(agg["launches"]),
            "clocks": clk,
            "roofline": {"bound": "tensor", "kernel": "tcgen05 GEMMs of the encoder: gemm_f16_ws_kernel (QKV, FFN-up) + gemm_f16_ln_pair_kernel (out-proj / FFN-down fused with residual + LayerNorm)",
                         "achieved": gemm_tf, "peak": peak,
                         "unit": "TFLOP/s", "frac": (gemm_tf / peak) if gemm_tf else None, "traffic": traffic,
                         "traffic_note": f"bytes per launch (average launch of the timed region); dram bytes = {tr_ratio:.2f} x algorithmic in the ncu capture ({tr_name})",
                         "peak_source": peak_src,
                         "share_of_step": agg["gemm_ms"] / agg["gpu_ms"] if agg["gpu_ms"] else None},
            "detail": {"ndis_per_query": agg["ndis"] / nqs, "nhops_per_query": agg["nhops"] / nqs,
                       "recomputed_per_query": agg["n_recomputed"] / nqs,
                       "dedup_saving": 1 - agg["n_recomputed"] / max(1, agg["n_requested"]),
                       "tokens_per_query": agg["n_tokens"] / nqs,
                       "traversal_steps_per_call": agg["steps"] / args.steps,
                       "encoder_share": agg["encoder_ms"] / agg["gpu_ms"] if agg["gpu_ms"] else None,
                       "attention_share": agg["attention_ms"] / agg["gpu_ms"] if agg["gpu_ms"] else None,
                       "layernorm_share": agg["norm_ms"] / agg["gpu_ms"] if agg["gpu_ms"] else None,
                       "encoder_algorithmic_tflops": enc_flops / (agg["encoder_ms"] / 1e3) / 1e12 if agg["encoder_ms"] else None,
                       "world": W["info"], **extras, "diskann": diskann},
        }
        parity = reference_arm_parity(W, call, Qpool) if world == 1 else None
        if not args.no_cpu_baseline and world == 1:
            cb = cpu_reference(W, args, n_max=1, budget_s=1e9)
            D_g = call(np.ascontiguousarray(Qpool[:len(cb["I"])]))
            inline = compare_results(np.array([[int(x) for x in r] for r in D_g["labels"]], np.int64), np.asarray(D_g["distances"]),
                                     cb["I"], cb["D"])
            inline["source"] = "cpu_baseline leg of this run (reference traversal + fp32 BertModel on the host)"
            parity = parity or inline
            if parity is not inline:
                parity["inline"] = inline
            out["cpu_baseline"] = {k_: cb[k_] for k_ in ("value", "unit", "cores", "kind", "sample", "recall_at_10", "seconds")}
        if parity:
            out["parity"] = parity
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if out is not None:
        emit(REAL_STDOUT, out)


def dump_outputs(d: Path, out):
    """The last timed step's result, as the caller received it (all ranks' queries: the results are gathered)."""
    d.mkdir(parents=True, exist_ok=True)
    np.save(d / "labels.npy", np.array([[int(x) for x in row] for row in out["labels"]], np.float64))
    np.save(d / "distances.npy", np.asarray(out["distances"], np.float32))
    log(f"outputs of the last timed step written to {d}")


def compare_results(I_gpu, D_gpu, I_ref, D_ref):
    """Top-k agreement of the GPU path with the CPU reference path on the same queries."""
    n = len(I_ref)
    overlap, ident, max_dd = [], 0, 0.0
    for a, da, b, db in zip(I_gpu[:n], D_gpu[:n], I_ref, D_ref):
        sa, sb = set(int(x) for x in a if x >= 0), set(int(x) for x in b if x >= 0)
        overlap.append(len(sa & sb) / max(1, len(sb)))
        ident += int(sa == sb)
        pos = {int(x): j for j, x in enumerate(b)}
        for j, x in enumerate(a):
            if int(x) in pos:
                max_dd = max(max_dd, abs(float(da[j]) - float(db[pos[int(x)]])))
    return {"queries": n, "topk_overlap": float(np.mean(overlap)), "identical_id_sets": ident, "max_abs_dD": max_dd}


def reference_arm_parity(W, call, Qpool):
    """If the reference arm ran on this box before (same cached world), compare the ids it found for the queries it
    timed with what the GPU path returns for the same queries."""
    f = W["dir"] / "ref_results.npz"
    if not f.exists():
        return None
    try:
        r = np.load(f)
        qi = r["query_index"]
        out = call(np.ascontiguousarray(Qpool[qi]))
        I = np.array([[int(x) for x in row] for row in out["labels"]], np.int64)
        res = compare_results(I, np.asarray(out["distances"]), r["I"], r["D"])
        res["source"] = "ids/distances written by `bench.py --impl reference` on this box (same cached world, same query vectors)"
        return res
    except Exception as e:
        return {"error": repr(e)}


def run_extras(args, W, searcher, local, flush):
    """Side measurements (not the headline): call-scope de-duplication; the traversal kernel alone on stored vectors."""
    import torch
    from leann_b200 import capi
    from leann_b200.tooling import recall_at_k

    idx = searcher._index
    dev = f"cuda:{local}"
    nq = 1024
    dq = torch.from_numpy(np.ascontiguousarray(W["Q"][:nq])).to(dev)
    dD = torch.empty((nq, K), dtype=torch.float32, device=dev)
    dI = torch.empty((nq, K), dtype=torch.int64, device=dev)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    params = capi.make_params(args.ef, args.beam, 0, True, recompute=True)
    res = {}
    try:
        idx.set_option("dedup_scope", 1)
        idx.search_device(dq.data_ptr(), nq, K, dD.data_ptr(), dI.data_ptr(), params)
        flush.fill_(1)
        torch.cuda.synchronize()
        ev0.record()
        idx.search_device(dq.data_ptr(), nq, K, dD.data_ptr(), dI.data_ptr(), params)
        ev1.record()
        torch.cuda.synchronize()
        res["call_scope_dedup"] = {"value": nq / (ev0.elapsed_time(ev1) / 1e3), "unit": "queries/s per GPU",
                                   "recomputed_per_query": idx.last_stats.n_recomputed / nq,
                                   "recall_at_10": recall_at_k(dI.cpu().numpy(), W["gt"][:nq]),
                                   "note": "embeddings reused across the hops of one call (dedup_scope=1); identical results; "
                                           "depends on how much the batch's queries overlap"}
        idx.set_option("dedup_scope", 0)
    except Exception as e:
        res["call_scope_dedup"] = {"error": str(e)}
    try:
        ef = W["dir"] / "E.npy"
        if not ef.exists():
            raise RuntimeError("no cached embeddings (build the world with --extras)")
        E = torch.from_numpy(np.load(ef)).to(dev)
        idx.set_vectors_device(E.data_ptr())
        idx.configure(148 * 32, 0)
        nst = min(len(W["Q"]), 8192)
        dqs = torch.from_numpy(np.ascontiguousarray(W["Q"][:nst])).to(dev)
        dDs = torch.empty((nst, K), dtype=torch.float32, device=dev)
        dIs = torch.empty((nst, K), dtype=torch.int64, device=dev)
        ps = capi.make_params(args.ef, args.beam, 0, True, recompute=False)
        idx.search_device(dqs.data_ptr(), nst, K, dDs.data_ptr(), dIs.data_ptr(), ps)
        flush.fill_(2)
        torch.cuda.synchronize()
        ev0.record()
        idx.search_device(dqs.data_ptr(), nst, K, dDs.data_ptr(), dIs.data_ptr(), ps)
        ev1.record()
        torch.cuda.synchronize()
        sec = ev0.elapsed_time(ev1) / 1e3
        sst = idx.last_stats
        deg = W["info"]["edges"] / args.chunks
        byts = sst.nhops * (32 + 4 * deg + deg / 8) + (sst.ndis + nst) * (W["preset"].hidden * 4 + 8)
        hbm_peak = (json.loads((ROOT / "MEASURED_PEAKS.json").read_text()).get("hbm_gbs") if (ROOT / "MEASURED_PEAKS.json").exists() else None) or 6650.0
        res["stored_vector_mode"] = {"queries": nst, "value": nst / sec, "unit": "queries/s", "ms": sec * 1e3,
                                     "recall_at_10": recall_at_k(dIs.cpu().numpy(), W["gt"][:nst]),
                                     "roofline": {"bound": "hbm", "kernel": "hnsw_step_kernel (persistent)", "achieved": byts / sec / 1e9,
                                                  "peak": hbm_peak, "unit": "GB/s", "frac": byts / sec / 1e9 / hbm_peak}}
        # id-level parity at bench scale: 64 queries, stored vectors, against the compiled reference traversal
        try:
            from oracle.binding import Reference, have_reference
            from leann_b200 import csr

            if have_reference():
                g = csr.read_compact_index(str(W["dir"] / "bench.index"))
                Eh = np.load(ef, mmap_mode="r")
                rD, rI, rnd, rnh = Reference.from_csr(g, Eh, M=32).search(np.ascontiguousarray(W["Q"][:64]), K, ef=args.ef, beam=args.beam, nthreads=16)
                gnd, gnh = idx.last_query_stats(nst)
                gI, gD = dIs[:64].cpu().numpy(), dDs[:64].cpu().numpy()
                res["stored_vector_parity"] = {"queries": 64, "ids_identical": bool(np.array_equal(gI, rI)),
                                               "distances_identical": bool(np.array_equal(gD, rD)),
                                               "ndis_identical": bool(np.array_equal(gnd[:64], rnd)),
                                               "nhops_identical": bool(np.array_equal(gnh[:64], rnh))}
        except Exception as e:
            res["stored_vector_parity"] = {"error": repr(e)}
    except Exception as e:
        res["stored_vector_mode"] = {"error": str(e)}
    return res


def diskann_extra(W, args, local, flush, k):
    """DiskANN backend in recompute mode (diskann_backend.py:440-447): PQ-only Vamana traversal, then ONE deferred
    re-rank of the expanded nodes from freshly encoded passages.  Index built by the torch tooling in the reference's
    partition layout (what is_recompute=True leaves on disk).  Needs the cached embeddings (--extras at world build)."""
    import torch
    from leann_b200 import capi, synth
    from leann_b200.tooling import recall_at_k
    from leann_b200.vamana_build import build_diskann_index

    t0 = time.time()
    E = np.load(W["dir"] / "E.npy")
    prefix, g, coords, pq, codes, max_norm = build_diskann_index(W["dir"], "bench_da", E, metric="mips", R=32,
                                                                 partition=True, keep_disk_index=False, device=f"cuda:{local}")
    t_build = time.time() - t0
    log(f"diskann index: R=32, {pq.n_chunks} PQ bytes/vector, mean degree {g.degrees().mean():.1f} ({t_build:.1f}s)")
    del coords
    idx = capi.DiskannIndex(prefix, "mips", prefix, local)
    idx.set_passages(np.load(W["dir"] / "bench.leann.tokens.npy", mmap_mode="r"), np.load(W["dir"] / "bench.leann.tokoffsets.npy"))
    preset = W["preset"]
    idx.set_encoder(preset.config(), synth.pack_weights(preset, synth.synthetic_weights(preset, 0)))
    if args.per_pass:
        idx.configure(0, args.per_pass)
    nq = min(len(W["Q"]), 4096)
    dq = torch.from_numpy(np.ascontiguousarray(W["Q"][:nq])).to(f"cuda:{local}")
    dD = torch.empty((nq, k), dtype=torch.float32, device=f"cuda:{local}")
    dI = torch.empty((nq, k), dtype=torch.int64, device=f"cuda:{local}")
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    res = {"build_s": t_build, "graph_degree": 32, "pq_bytes_per_vector": pq.n_chunks, "queries": nq}
    hbm_peak = (json.loads((ROOT / "MEASURED_PEAKS.json").read_text()).get("hbm_gbs") if (ROOT / "MEASURED_PEAKS.json").exists() else None) or 6650.0
    for name, p in (("recompute", capi.make_diskann_params(args.ef, max(1, args.beam), recompute_embeddings=True)),
                    ("recompute_L128", capi.make_diskann_params(2 * args.ef, max(1, args.beam), recompute_embeddings=True)),
                    ("pq_traversal_only", capi.make_diskann_params(args.ef, max(1, args.beam), recompute_embeddings=False, skip_search_reorder=True))):
        idx.search_device(dq.data_ptr(), nq, k, dD.data_ptr(), dI.data_ptr(), p)
        flush.fill_(3)
        torch.cuda.synchronize()
        ev0.record()
        idx.search_device(dq.data_ptr(), nq, k, dD.data_ptr(), dI.data_ptr(), p)
        ev1.record()
        torch.cuda.synchronize()
        sec = ev0.elapsed_time(ev1) / 1e3
        st = idx.last_stats
        r = {"value": nq / sec, "unit": "queries/s", "ms": sec * 1e3, "recall_at_10": recall_at_k(dI.cpu().numpy(), W["gt"][:nq]),
             "expansions_per_query": st.n_requested / nq, "pq_comparisons_per_query": st.ndis / nq,
             "recomputed_per_query": st.n_recomputed / nq, "encoder_share": st.encoder_ms / st.gpu_ms if st.gpu_ms else None}
        if name == "pq_traversal_only":
            byts = st.n_requested * (4 * 32 + 4) + st.ndis * pq.n_chunks
            r["roofline"] = {"bound": "hbm", "kernel": "vamana_search_kernel (persistent)", "achieved": byts / sec / 1e9, "peak": hbm_peak,
                             "unit": "GB/s", "frac": byts / sec / 1e9 / hbm_peak}
        res[name] = r
    idx.close()
    return res


# ------------------------------------------------------------------------------------------------ the reference's CPU path
def cpu_reference(W, args, n_max: int, budget_s: float):
    """The reference's own CPU path on this box's host cores: the faiss-fork traversal compiled from
    /root/reference (oracle/_ref, prebuilt) — or the C restatement when that library is absent — with
    distances_batch served by a torch-CPU fp32 BertModel forward + numpy scoring, exactly the
    embedding server's distance branch (hnsw_embedding_server.py:147-211), queries one at a time like
    the single REP loop.  Times queries 0, 1, ... of the pool until n_max are done or budget_s is used."""
    import torch
    from oracle.binding import Oracle, Reference, have_reference
    from oracle.encoder_oracle import EncoderOracle
    from leann_b200 import csr, synth
    from leann_b200.tooling import recall_at_k

    ncpu = os.cpu_count() or 1
    preset = W["preset"]
    tokens = np.load(W["dir"] / "bench.leann.tokens.npy", mmap_mode="r")
    offsets = np.load(W["dir"] / "bench.leann.tokoffsets.npy")
    eo = EncoderOracle(preset, synth.synthetic_weights(preset, 0))
    # The reference caps torch at min(8, cores) (embedding_compute.py:150).  A hop's batch is ~20 short
    # sequences, so more threads do not always help: calibrate on one hop-sized batch and keep the fastest.
    probe_ids = list(range(24))
    best, cores = None, 1
    for th in sorted({min(8, ncpu), min(16, ncpu), min(32, ncpu), min(64, ncpu)}):
        torch.set_num_threads(th)
        eo.encode_store(tokens, offsets, probe_ids, 64)
        t0 = time.perf_counter()
        eo.encode_store(tokens, offsets, probe_ids, 64)
        dt = time.perf_counter() - t0
        if best is None or dt < best:
            best, cores = dt, th
    torch.set_num_threads(cores)
    fn = eo.distance_fn(tokens, offsets, True, batch_size=64)
    kind = "reference" if have_reference() else "port"
    g = csr.read_compact_index(str(W["dir"] / "bench.index"))
    trav = Reference.from_csr(g, None, M=32) if kind == "reference" else Oracle(g)
    Ds, Is, nd = [], [], []
    t_all = 0.0
    for i in range(n_max):
        q = np.ascontiguousarray(W["Q"][i:i + 1])
        t0 = time.perf_counter()
        D, I, ndis, nhops = trav.search(q, K, ef=args.ef, beam=args.beam, dist_fn=fn, nthreads=1)
        t_all += time.perf_counter() - t0
        Ds.append(D[0]); Is.append(I[0]); nd.append(int(ndis[0]))
        if t_all >= budget_s:
            break
    n = len(Is)
    I, D = np.stack(Is), np.stack(Ds)
    return {"value": n / t_all, "unit": "queries/s", "cores": cores, "kind": kind,
            "sample": f"{n} queries of the same workload, serial (single embedding server), torch intra-op "
                      f"threads={cores} of {ncpu} host cores (fastest of 8/16/32/64 on a hop-sized batch), "
                      f"{float(np.mean(nd)):.0f} recomputes/query",
            "recall_at_10": recall_at_k(I, W["gt"][:n]), "seconds": t_all, "n": n, "I": I, "D": D, "ndis": np.asarray(nd)}


def run_reference(args):
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    import torch
    wd = world_dir(args)
    if not (wd / "DONE").exists() and not torch.cuda.is_available():
        emit(REAL_STDOUT, {"impl": "reference", "unavailable": "set-up (corpus embedding + graph) needs the GPU encoder; no GPU here"})
        return
    from leann_b200 import build
    if build.needs_build():
        build.build()
    wd = ensure_world(args, builder=True, device=0)
    W = load_world(wd)
    t0 = time.perf_counter()
    res = cpu_reference(W, args, n_max=max(1, args.steps), budget_s=args.ref_budget_s)
    np.savez(wd / "ref_results.npz", query_index=np.arange(res["n"]), I=res["I"], D=res["D"], ndis=res["ndis"])
    out = {"impl": "reference", "metric": METRIC, "value": res["value"], "unit": "queries/s", "n_gpus": args.gpus,
           "steps": args.steps, "warmup": args.warmup, "steps_timed": res["n"], "ms_per_step": res["seconds"] / res["n"] * 1e3,
           "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32 (CPU)", "data": "synthetic",
           "config": {"workload": workload_string(args, W, 1, extra=" — reference arm: one serial CPU query per step, "
                                                  f"{res['n']} of {args.steps} steps timed inside a {args.ref_budget_s:.0f}s wall budget; "
                                                  "warm-up = the encoder thread-count calibration batches")},
           "recall_at_10": res["recall_at_10"],
           "cpu_baseline": {k_: res[k_] for k_ in ("value", "unit", "cores", "kind", "sample")},
           "e2e": {"value": res["value"], "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "wall_s": time.perf_counter() - t0}
    emit(REAL_STDOUT, out)


def _claim_stdout():
    """Libraries (NCCL's version banner, nvcc chatter of an on-demand build) write to fd 1; the contract is ONE JSON
    line on stdout.  Point fd 1 at stderr for the whole run and keep the real stdout for the final line."""
    sys.stdout.flush()
    real = os.dup(1)
    os.dup2(2, 1)
    return real


def emit(real_fd, obj):
    os.write(real_fd, (json.dumps(obj) + "\n").encode())


if __name__ == "__main__":
    a = parse()
    REAL_STDOUT = _claim_stdout()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_b200(a)
