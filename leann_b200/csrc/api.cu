// C ABI (include/leann_b200.h) and the host-side driver of the search pipeline:
//   K1 traversal step  ->  hop work list (unique nodes, packed token offsets)
//                      ->  recompute stage (encoder.cu / gemm_tcgen05.cu) in passes of P passages
//                      ->  next K1 step scores the fresh embeddings and folds them into the beams.
// Ids, embeddings and distances never leave the GPU; per hop the host reads back three counters
// (unique passages, packed tokens, finished queries) to size the next launches.
#include <float.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <cmath>
#include <string>
#include <vector>

#include "../../include/leann_b200.h"
#include "common.cuh"
#include "index_io.h"
#include "traverse.cuh"
#include "vamana.cuh"
#include "vamana_io.h"

namespace lb2 {

static thread_local std::string g_err;

void set_error(const char* fmt, ...) {
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    g_err = buf;
}

namespace {

struct HopCtrl {  // written by gather_bounds_kernel into mapped pinned memory
    int n_unique;
    int n_done;
    long long n_tokens;
    int n_chunks;
    int pad;
};

__global__ void gather_bounds_kernel(const unsigned long long* claim, const int* n_done, const int* seq_start,
                                     int per_pass, HopCtrl* ctrl, int* bounds, int max_chunks) {
    const unsigned long long c = *claim;
    const int nu = static_cast<int>(c >> 40);
    const long long nt = static_cast<long long>(c & ((1ull << 40) - 1));
    const int nch = (nu + per_pass - 1) / per_pass;
    for (int i = threadIdx.x; i <= nch && i <= max_chunks; i += blockDim.x)
        bounds[i] = (i == nch) ? static_cast<int>(nt) : seq_start[i * per_pass];
    if (threadIdx.x == 0) {
        ctrl->n_unique = nu;
        ctrl->n_tokens = nt;
        ctrl->n_done = *n_done;
        ctrl->n_chunks = nch;
    }
}

__global__ void fill_empty_results_kernel(float* D, int64_t* I, int64_t n, float v) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i < n) { D[i] = v; I[i] = -1; }
}

template <class T>
bool dev_alloc(T** p, size_t n) {
    if (*p) { cudaFree(*p); *p = nullptr; }
    if (n == 0) n = 1;
    cudaError_t e = cudaMalloc(reinterpret_cast<void**>(p), n * sizeof(T));
    if (e != cudaSuccess) {
        set_error("cudaMalloc of %zu bytes failed: %s", n * sizeof(T), cudaGetErrorString(e));
        *p = nullptr;
        return false;
    }
    return true;
}
template <class T>
void dev_free(T** p) {
    if (*p) cudaFree(*p);
    *p = nullptr;
}

struct EventPool {
    std::vector<cudaEvent_t> ev;
    size_t used = 0;
    double total_ms = 0;
    cudaEvent_t get() {
        if (used == ev.size()) {
            cudaEvent_t e;
            cudaEventCreate(&e);
            ev.push_back(e);
        }
        return ev[used++];
    }
    void drain() {  // caller has synchronised the stream
        for (size_t i = 0; i + 1 < used; i += 2) {
            float ms = 0;
            if (cudaEventElapsedTime(&ms, ev[i], ev[i + 1]) == cudaSuccess) total_ms += ms;
        }
        used = 0;
    }
    void destroy() {
        for (auto e : ev) cudaEventDestroy(e);
        ev.clear();
        used = 0;
    }
};

}  // namespace
}  // namespace lb2

using namespace lb2;

struct lb2_index {
    int device = 0;
    int num_sms = 148;
    cudaStream_t stream = 0;  // legacy default stream: orders with the caller's default-stream work
    // graph
    DevGraph g;
    uint64_t* d_node_offsets = nullptr;
    uint64_t* d_level_ptr = nullptr;
    int32_t* d_nbrs = nullptr;
    int64_t n_edges = 0;
    // scoring sources
    float* d_vectors = nullptr;
    uint16_t* d_tokens = nullptr;
    uint64_t* d_tok_off = nullptr;
    std::vector<uint64_t> h_tok_off;
    int max_token = 0;  // largest token id of the attached store (checked against the encoder's vocabulary)
    // PQ-guided pruning data (lb2_load_pq_pruning)
    PqDev pq;
    float* dpq_tables_tr = nullptr; float* dpq_centroid = nullptr; uint32_t* dpq_chunk_offsets = nullptr; uint8_t* dpq_codes = nullptr;
    int pq_cap = 16384;        // PQ candidates a query may accumulate (global / proportional strategies)
    int alloc_pq_S = 0, alloc_pq_cap = 0, alloc_pq_chunks = 0, alloc_pq_dims = 0;
    Encoder enc;
    // tunables
    int cfg_slots = 0;
    int per_pass = 4096;
    int dedup_call_scope = 0;  // 0: de-duplicate recomputes per hop (default), 1: per search call
    // traversal state
    TravState st{};
    TravParams alloc_p{};
    int alloc_S = 0;
    int64_t alloc_nq = 0;
    bool alloc_recompute = false;
    int cap_unique = 0;
    int64_t cap_E_rows = 0;
    float* d_E = nullptr;
    HopCtrl* h_ctrl = nullptr;  // pinned + mapped
    int* h_bounds = nullptr;    // pinned + mapped
    int max_chunks = 0;
    uint32_t epoch = 0;
    // host-pointer convenience buffers
    float* d_q = nullptr; float* d_D = nullptr; int64_t* d_I = nullptr;
    int64_t cap_q = 0, cap_out = 0;
    long long* d_qndis = nullptr; long long* d_qnhops = nullptr;
    int64_t cap_qstats = 0, last_nq = 0;
    // encode scratch
    int* d_enc_node = nullptr; int* d_enc_start = nullptr; float* d_enc_out = nullptr;
    int64_t cap_enc = 0;
    bool profile_gemm = false;
    EventPool ev_total, ev_enc;
    // ---- DiskANN / Vamana handle (lb2_diskann_open)
    bool is_vamana = false;
    DevVamana vam;
    bool vam_partitioned = false;
    int64_t vam_edges = 0;
    int32_t* dv_nbrs = nullptr; uint8_t* dv_codes = nullptr; float* dv_tables_tr = nullptr; float* dv_centroid = nullptr;
    uint32_t* dv_chunk_offsets = nullptr; uint32_t* dv_medoids = nullptr; float* dv_centroid_data = nullptr; float* dv_coords = nullptr;
    VamanaWork vw{};           // buffers of the current wave (grow-only)
    int64_t vcap_q = 0;        // queries aq/qrot/qnorm/lut/full_*/n_full are sized for
    int vcap_full = 0, vcap_slots = 0;
    int64_t vcap_uniq = 0;     // uniq_node / seq_start entries
    int64_t vcap_E = 0;        // rows of d_vE
    float* d_vE = nullptr;
    bool vis_dirty = false;
    int64_t v_last_wave = 0;
};

namespace lb2 {
// encoder.cu calls these around its launches; they record CUDA events only when profiling is on
static EventPool g_prof_pool[PROF_NCAT];
static bool g_prof_on = false;
double g_gemm_flops = 0;
void prof_begin(cudaStream_t s, int cat) { if (g_prof_on) cudaEventRecord(g_prof_pool[cat].get(), s); }
void prof_end(cudaStream_t s, int cat, double flops) {
    if (g_prof_on) { cudaEventRecord(g_prof_pool[cat].get(), s); if (cat == PROF_GEMM) g_gemm_flops += flops; }
}
}  // namespace lb2

namespace {

bool use_device(const lb2_index* idx) {
    cudaError_t e = cudaSetDevice(idx->device);
    if (e != cudaSuccess) {
        set_error("cudaSetDevice(%d): %s", idx->device, cudaGetErrorString(e));
        return false;
    }
    return true;
}

void free_state(lb2_index* x) {
    TravState& s = x->st;
    dev_free(&s.phase); dev_free(&s.qid); dev_free(&s.level); dev_free(&s.nearest); dev_free(&s.prev_nearest);
    dev_free(&s.d_nearest); dev_free(&s.hk); dev_free(&s.hnvalid); dev_free(&s.nstep); dev_free(&s.pend_beam);
    dev_free(&s.n_req); dev_free(&s.ndis); dev_free(&s.nhops); dev_free(&s.heap_ids); dev_free(&s.heap_dis);
    dev_free(&s.res_ids); dev_free(&s.res_dis); dev_free(&s.req_ids); dev_free(&s.visited);
    dev_free(&s.next_query); dev_free(&s.n_done); dev_free(&s.stamp); dev_free(&s.slot_of[0]); dev_free(&s.slot_of[1]);
    dev_free(&s.claim); dev_free(&s.uniq_node); dev_free(&s.seq_start);
    dev_free(&s.pq_lut); dev_free(&s.pq_qprep); dev_free(&s.pq_qd); dev_free(&s.pq_qid); dev_free(&s.pq_qn); dev_free(&s.pq_qhead);
    dev_free(&s.error);
    x->alloc_pq_S = 0;
    dev_free(&x->d_E);
    if (x->h_ctrl) cudaFreeHost(x->h_ctrl);
    if (x->h_bounds) cudaFreeHost(x->h_bounds);
    x->h_ctrl = nullptr; x->h_bounds = nullptr;
    x->alloc_S = 0;
    x->cap_unique = 0;
    x->cap_E_rows = 0;
}

bool ensure_state(lb2_index* x, int S, const TravParams& p, bool recompute) {
    const TravParams& a = x->alloc_p;
    const int64_t need_rows = !recompute ? 0 : (x->dedup_call_scope ? std::max<int64_t>(x->g.ntotal, (int64_t)S * p.cap_req) : (int64_t)S * p.cap_req);
    // strides depend on S / hcap / k / cap_req: reallocate on any change (calls with stable params reuse)
    const bool pq_ok = !p.pq_mode || (x->alloc_pq_S == S && x->alloc_pq_cap == x->pq_cap && x->alloc_pq_chunks == x->pq.n_chunks &&
                                      x->alloc_pq_dims == x->pq.ndims);
    if (x->alloc_S == S && a.hcap == p.hcap && a.k == p.k && a.cap_req == p.cap_req && (!recompute || x->alloc_recompute) &&
        x->cap_E_rows >= need_rows && pq_ok)
        return true;
    free_state(x);
    TravState& s = x->st;
    s = TravState{};
    s.S = S;
    const size_t Ss = (size_t)S;
    const int64_t N = x->g.ntotal;
    s.vis_words = ((N + 31) / 32 + 3) & ~int64_t(3);
    bool ok = dev_alloc(&s.phase, Ss) && dev_alloc(&s.qid, Ss) && dev_alloc(&s.level, Ss) && dev_alloc(&s.nearest, Ss) &&
              dev_alloc(&s.prev_nearest, Ss) && dev_alloc(&s.d_nearest, Ss) && dev_alloc(&s.hk, Ss) &&
              dev_alloc(&s.hnvalid, Ss) && dev_alloc(&s.nstep, Ss) && dev_alloc(&s.pend_beam, Ss) &&
              dev_alloc(&s.n_req, Ss) && dev_alloc(&s.ndis, Ss) && dev_alloc(&s.nhops, Ss) &&
              dev_alloc(&s.heap_ids, Ss * p.hcap) && dev_alloc(&s.heap_dis, Ss * p.hcap) &&
              dev_alloc(&s.res_ids, Ss * p.k) && dev_alloc(&s.res_dis, Ss * p.k) &&
              dev_alloc(&s.req_ids, Ss * p.cap_req) && dev_alloc(&s.visited, Ss * (size_t)s.vis_words) &&
              dev_alloc(&s.next_query, 1) && dev_alloc(&s.n_done, 1);
    ok = ok && dev_alloc(&s.error, 1);
    if (ok && p.pq_mode) {
        ok = dev_alloc(&s.pq_lut, Ss * (size_t)x->pq.n_chunks * 256) && dev_alloc(&s.pq_qprep, Ss * (size_t)x->pq.ndims) &&
             dev_alloc(&s.pq_qd, Ss * (size_t)x->pq_cap) && dev_alloc(&s.pq_qid, Ss * (size_t)x->pq_cap) &&
             dev_alloc(&s.pq_qn, Ss) && dev_alloc(&s.pq_qhead, Ss);
        if (ok) { x->alloc_pq_S = S; x->alloc_pq_cap = x->pq_cap; x->alloc_pq_chunks = x->pq.n_chunks; x->alloc_pq_dims = x->pq.ndims; }
    }
    if (!ok) { free_state(x); return false; }
    s.pq_cap = x->pq_cap;
    if (cudaMemsetAsync(s.visited, 0, Ss * (size_t)s.vis_words * 4, x->stream) != cudaSuccess) {
        set_error("memset(visited) failed");
        free_state(x);
        return false;
    }
    if (recompute) {
        x->cap_unique = S * p.cap_req;
        x->max_chunks = (x->cap_unique + x->per_pass - 1) / x->per_pass + 1;
        ok = dev_alloc(&s.stamp, (size_t)N) && dev_alloc(&s.slot_of[0], (size_t)N) && dev_alloc(&s.slot_of[1], (size_t)N) &&
             dev_alloc(&s.claim, 1) && dev_alloc(&s.uniq_node, (size_t)x->cap_unique) &&
             dev_alloc(&s.seq_start, (size_t)x->cap_unique) && dev_alloc(&x->d_E, (size_t)need_rows * x->g.d);
        x->cap_E_rows = ok ? need_rows : 0;
        if (ok && cudaMemsetAsync(s.stamp, 0, (size_t)N * 4, x->stream) != cudaSuccess) ok = false;
        if (ok && cudaHostAlloc(reinterpret_cast<void**>(&x->h_ctrl), sizeof(HopCtrl), cudaHostAllocMapped) != cudaSuccess) ok = false;
        if (ok && cudaHostAlloc(reinterpret_cast<void**>(&x->h_bounds), sizeof(int) * (x->max_chunks + 2), cudaHostAllocMapped) != cudaSuccess) ok = false;
        if (!ok) {
            if (g_err.empty()) set_error("allocating the recompute work lists failed");
            free_state(x);
            return false;
        }
        x->epoch = 0;
    }
    x->alloc_S = S;
    x->alloc_p = p;
    x->alloc_recompute = recompute;
    return true;
}

int max_token(const uint16_t* t, uint64_t n) {
    uint16_t m = 0;
    for (uint64_t i = 0; i < n; i++) m = t[i] > m ? t[i] : m;
    return m;
}

int next_pow2(int v) {
    int p = 1;
    while (p < v) p <<= 1;
    return p;
}

// embed, work list, pool + per layer: 4 GEMMs, attention, and 2 LayerNorm kernels unless they ride in the GEMM epilogues
int encoder_kernels_per_pass(const Encoder& e) {
    return 3 + e.cfg.layers * (encoder_fuses_ln(e.cfg) ? 5 : 7);
}

int search_impl(lb2_index* x, int64_t nq, const float* d_q, int64_t k, float* d_D, int64_t* d_I,
                const lb2_search_params* prm, lb2_search_stats* stats) {
    lb2_search_params P;
    if (prm) P = *prm; else lb2_default_params(&P);
    if (x->is_vamana) { set_error("this handle is a DiskANN index: use lb2_diskann_search"); return LB2_ERR_STATE; }
    if (nq < 0 || k <= 0 || k > 4096) { set_error("bad nq/k (nq=%lld k=%lld)", (long long)nq, (long long)k); return LB2_ERR_ARG; }
    if (P.efSearch <= 0 || P.efSearch > 16384) { set_error("efSearch out of range: %d", P.efSearch); return LB2_ERR_ARG; }
    if (P.pq_pruning_ratio < 0.f || P.pq_pruning_ratio > 1.f) { set_error("pq_pruning_ratio must lie in [0, 1]"); return LB2_ERR_ARG; }
    const bool recompute = P.recompute != 0;
    if (recompute && (!x->d_tokens || !x->enc.loaded)) {
        set_error("recompute search needs lb2_set_passages() and lb2_set_encoder() first");
        return LB2_ERR_STATE;
    }
    if (!recompute && !x->d_vectors) {
        set_error("recompute=0 needs stored vectors (lb2_set_vectors or an index with flat storage)");
        return LB2_ERR_STATE;
    }
    if (recompute && x->enc.cfg.hidden != x->g.d) {
        set_error("encoder hidden size %d != index dimension %d", x->enc.cfg.hidden, x->g.d);
        return LB2_ERR_STATE;
    }
    if (stats) memset(stats, 0, sizeof(*stats));
    if (nq == 0) return LB2_OK;
    cudaStream_t st = x->stream;
    if (x->cap_qstats < nq) {
        if (!dev_alloc(&x->d_qndis, (size_t)nq) || !dev_alloc(&x->d_qnhops, (size_t)nq)) return LB2_ERR_CUDA;
        x->cap_qstats = nq;
    }
    x->last_nq = nq;
    cudaMemsetAsync(x->d_qndis, 0, nq * sizeof(long long), st);
    cudaMemsetAsync(x->d_qnhops, 0, nq * sizeof(long long), st);
    if (x->g.ntotal == 0 || x->g.entry_point < 0) {  // HNSW.cpp:1088-1090: untouched (heapified) results
        const int64_t n = nq * k;
        fill_empty_results_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(d_D, d_I, n, x->g.metric_ip ? -FLT_MAX : FLT_MAX);
        if (cudaStreamSynchronize(st) != cudaSuccess) { set_error("fill failed"); return LB2_ERR_CUDA; }
        return LB2_OK;
    }

    TravParams tp;
    tp.ef = P.efSearch;
    tp.k = (int)k;
    tp.hcap = std::max(tp.ef, tp.k);
    tp.beam = std::max(1, P.beam_size);
    tp.batch_size = std::max(0, P.batch_size);
    tp.check_rel = P.check_relative_distance != 0;
    const int deg0 = std::max(1, x->g.maxdeg0);
    // PQ-guided pruning: like the reference, only when PQ data was loaded AND the parameters ask for it
    // (perform_pq_pruning, HNSW_search.cpp:442-445); otherwise the three knobs are ignored
    tp.pq_ratio = 1.0f - P.pq_pruning_ratio;
    tp.pq_mode = 0;
    if (x->dpq_codes && (tp.pq_ratio < 1.f || P.local_prune || P.send_neigh_times_ratio != 0.f))
        tp.pq_mode = P.local_prune ? 2 : (P.send_neigh_times_ratio > 1e-6f ? 3 : 1);
    // unvisited neighbours one hop can gather.  Batch mode pops until total_neighbors >= batch_size, and with pruning each
    // pop only counts pq_select_ratio of its neighbours (:567-568): up to batch_size / ratio (+ one row), never more than
    // every candidate's row
    int64_t gather = (int64_t)tp.beam * deg0;
    if (tp.batch_size > 0) {
        const int64_t all_rows = (int64_t)tp.hcap * deg0;
        gather = tp.batch_size;
        if (tp.pq_mode && tp.pq_ratio < 1.f)  // every pop also truncates its contribution to an int: up to one lost per pop
            gather = tp.pq_ratio > 0.f ? (int64_t)std::min<double>(std::ceil((tp.batch_size + tp.hcap) / (double)tp.pq_ratio) + 1, (double)all_rows) : all_rows;
        gather = std::min(gather, all_rows) + deg0;
    }
    tp.cap_new = (int)std::max<int64_t>(std::max(1, x->g.maxdeg_up), gather);
    tp.p2 = next_pow2(tp.cap_new);
    // a hop selects at most (new neighbours) + (growth of the examined share of the queue) + 1 nodes: <= 2 cap_new + 2
    tp.cap_req = tp.pq_mode ? 2 * tp.cap_new + 2 : tp.cap_new;

    int S;
    if (x->cfg_slots > 0) S = x->cfg_slots;
    else S = recompute ? 2048 : x->num_sms * 32;
    // visited bitsets: keep them under ~16 GB
    const int64_t vis_bytes = (((x->g.ntotal + 31) / 32 + 3) & ~int64_t(3)) * 4;
    S = (int)std::min<int64_t>(S, std::max<int64_t>(64, (16ll << 30) / std::max<int64_t>(vis_bytes, 1)));
    S = (int)std::min<int64_t>(S, nq);
    S = std::max(S, 1);
    if (!ensure_state(x, S, tp, recompute)) return LB2_ERR_CUDA;
    if (recompute && !encoder_reserve(&x->enc, (int64_t)x->per_pass * x->enc.cfg.max_pos, x->per_pass)) return LB2_ERR_CUDA;

    TravState& s = x->st;
    s.queries = d_q; s.nq = nq; s.outD = d_D; s.outI = d_I; s.out_ndis = x->d_qndis; s.out_nhops = x->d_qnhops;
    s.recompute = recompute ? 1 : 0;
    s.vectors = x->d_vectors; s.E = x->d_E; s.tok_off = x->d_tok_off; s.max_pos = x->enc.cfg.max_pos;
    s.pq = x->pq;
    cudaMemsetAsync(s.error, 0, sizeof(int), st);

    x->ev_total.total_ms = 0; x->ev_enc.total_ms = 0;
    for (auto& pl : g_prof_pool) pl.total_ms = 0;
    g_gemm_flops = 0;
    g_prof_on = x->profile_gemm;
    cudaEventRecord(x->ev_total.get(), st);
    if (!launch_init_slots(st, s)) return LB2_ERR_CUDA;
    long long launches = 1, steps = 0, n_recomputed = 0, n_tokens = 0, n_passes = 0;

    if (!recompute) {
        s.epoch = 1;
        if (!launch_step(st, x->g, tp, s, 1 << 30, x->num_sms)) return LB2_ERR_CUDA;
        launches++; steps++;
    } else {
        s.call_scope = x->dedup_call_scope;
        const uint32_t call_epoch = x->epoch + 1;  // > every stamp written so far
        int64_t rows_this_call = 0;
        for (;;) {
            x->epoch++;
            s.epoch = x->epoch;
            s.stamp_value = s.call_scope ? call_epoch : s.epoch;
            s.row_base_hop = s.call_scope ? (int)rows_this_call : 0;
            cudaMemsetAsync(s.claim, 0, sizeof(unsigned long long), st);
            if (!launch_step(st, x->g, tp, s, 1, x->num_sms)) return LB2_ERR_CUDA;
            gather_bounds_kernel<<<1, 64, 0, st>>>(s.claim, s.n_done, s.seq_start, x->per_pass, x->h_ctrl, x->h_bounds, x->max_chunks);
            launches += 2; steps++;
            cudaError_t e = cudaStreamSynchronize(st);
            if (e != cudaSuccess) { set_error("traversal step failed: %s", cudaGetErrorString(e)); return LB2_ERR_CUDA; }
            const HopCtrl c = *x->h_ctrl;
            if (c.n_done >= nq) break;  // every query has written its results
            if (c.n_unique == 0) {
                // call scope: every node requested in this hop already has its embedding; hop scope: cannot happen
                if (!s.call_scope) { set_error("internal: traversal stalled (%d of %lld queries done)", c.n_done, (long long)nq); return LB2_ERR_CUDA; }
                continue;
            }
            if (c.n_unique > x->cap_unique || s.row_base_hop + (int64_t)c.n_unique > x->cap_E_rows) {
                set_error("internal: hop work list overflow");
                return LB2_ERR_CUDA;
            }
            n_recomputed += c.n_unique;
            n_tokens += c.n_tokens;
            cudaEventRecord(x->ev_enc.get(), st);
            for (int ch = 0; ch < c.n_chunks; ch++) {
                const int first = ch * x->per_pass;
                const int n_seq = std::min(x->per_pass, c.n_unique - first);
                const int row_base = x->h_bounds[ch];
                const int n_tok = x->h_bounds[ch + 1] - row_base;
                if (!encoder_forward(&x->enc, st, x->d_tokens, x->d_tok_off, s.uniq_node + first, s.seq_start + first,
                                     row_base, n_seq, n_tok, x->d_E + ((size_t)s.row_base_hop + first) * x->g.d))
                    return LB2_ERR_CUDA;
                launches += encoder_kernels_per_pass(x->enc);
                n_passes++;
            }
            cudaEventRecord(x->ev_enc.get(), st);
            rows_this_call += c.n_unique;
            if (x->ev_enc.used > 4000 || g_prof_pool[PROF_GEMM].used > 8000) {
                cudaStreamSynchronize(st);
                x->ev_enc.drain();
                for (auto& pl : g_prof_pool) pl.drain();
            }
        }
    }
    cudaEventRecord(x->ev_total.get(), st);
    cudaError_t e = cudaStreamSynchronize(st);
    g_prof_on = false;
    if (e != cudaSuccess) { set_error("search failed: %s", cudaGetErrorString(e)); return LB2_ERR_CUDA; }
    int kerr = 0;
    cudaMemcpy(&kerr, s.error, sizeof(int), cudaMemcpyDeviceToHost);
    if (kerr == 4) {
        set_error("batch_size with PQ pruning gathered more neighbours in one hop than this build reserves shared memory for");
        return LB2_ERR_STATE;
    }
    if (kerr == 3) {  // the reference's fetch raises on NaN embeddings (HNSW_zmq.cpp:383-400)
        set_error("a passage embedding or stored vector contains NaN");
        return LB2_ERR_STATE;
    }
    if (kerr) {
        set_error("PQ-guided pruning: a query exceeded %d PQ candidates (raise it with lb2_set_option(\"pq_queue_cap\"))", x->pq_cap);
        return LB2_ERR_STATE;
    }
    int done = 0;
    cudaMemcpy(&done, s.n_done, sizeof(int), cudaMemcpyDeviceToHost);
    if (done != nq) { set_error("internal: %d of %lld queries finished", done, (long long)nq); return LB2_ERR_CUDA; }
    x->ev_total.drain(); x->ev_enc.drain();
    for (auto& pl : g_prof_pool) pl.drain();
    if (stats) {
        std::vector<long long> a((size_t)nq), b((size_t)nq);
        cudaMemcpy(a.data(), x->d_qndis, nq * sizeof(long long), cudaMemcpyDeviceToHost);
        cudaMemcpy(b.data(), x->d_qnhops, nq * sizeof(long long), cudaMemcpyDeviceToHost);
        for (int64_t i = 0; i < nq; i++) { stats->ndis += a[i]; stats->nhops += b[i]; }
        stats->n_requested = stats->ndis + nq;
        stats->n_recomputed = n_recomputed;
        stats->n_tokens = n_tokens;
        stats->n_steps = steps;
        stats->n_kernel_launches = launches;
        stats->gpu_ms = x->ev_total.total_ms;
        stats->encoder_ms = x->ev_enc.total_ms;
        stats->gemm_ms = g_prof_pool[PROF_GEMM].total_ms;
        stats->gemm_flops = g_gemm_flops;
        stats->attention_ms = g_prof_pool[PROF_ATTN].total_ms;
        stats->norm_ms = g_prof_pool[PROF_NORM].total_ms;
        stats->n_encoder_passes = n_passes;
    }
    return LB2_OK;
}

bool ensure_enc_scratch(lb2_index* x, int64_t n) {
    if (x->cap_enc >= n) return true;
    if (!dev_alloc(&x->d_enc_node, (size_t)n) || !dev_alloc(&x->d_enc_start, (size_t)n) ||
        !dev_alloc(&x->d_enc_out, (size_t)n * x->enc.cfg.hidden)) { x->cap_enc = 0; return false; }
    x->cap_enc = n;
    return true;
}

// encode passages `nodes` (host, ids into the given token store) in passes; out is host or device
int encode_impl(lb2_index* x, const uint16_t* d_tok, const uint64_t* d_off, const uint64_t* h_off, int64_t n,
                const int* h_nodes /* null = first..first+n */, int64_t first, float* out, bool out_is_device) {
    if (!x->enc.loaded) { set_error("no encoder loaded"); return LB2_ERR_STATE; }
    const int H = x->enc.cfg.hidden, maxp = x->enc.cfg.max_pos;
    const int pp = x->per_pass;
    if (!encoder_reserve(&x->enc, (int64_t)pp * maxp, pp)) return LB2_ERR_CUDA;
    if (!ensure_enc_scratch(x, pp)) return LB2_ERR_CUDA;
    std::vector<int> nodes(pp), starts(pp);
    for (int64_t base = 0; base < n; base += pp) {
        const int m = (int)std::min<int64_t>(pp, n - base);
        long long tok = 0;
        for (int i = 0; i < m; i++) {
            const int64_t node = h_nodes ? h_nodes[base + i] : first + base + i;
            nodes[i] = (int)node;
            starts[i] = (int)tok;
            const uint64_t len = h_off[node + 1] - h_off[node];
            tok += (long long)std::min<uint64_t>(len, (uint64_t)maxp);
        }
        cudaMemcpyAsync(x->d_enc_node, nodes.data(), m * sizeof(int), cudaMemcpyHostToDevice, x->stream);
        cudaMemcpyAsync(x->d_enc_start, starts.data(), m * sizeof(int), cudaMemcpyHostToDevice, x->stream);
        float* dst = out_is_device ? out + (size_t)base * H : x->d_enc_out;
        if (!encoder_forward(&x->enc, x->stream, d_tok, d_off, x->d_enc_node, x->d_enc_start, 0, m, (int)tok, dst))
            return LB2_ERR_CUDA;
        if (!out_is_device)
            cudaMemcpyAsync(out + (size_t)base * H, x->d_enc_out, (size_t)m * H * 4, cudaMemcpyDeviceToHost, x->stream);
        cudaError_t e = cudaStreamSynchronize(x->stream);  // nodes/starts are reused by the next pass
        if (e != cudaSuccess) { set_error("encode failed: %s", cudaGetErrorString(e)); return LB2_ERR_CUDA; }
    }
    return LB2_OK;
}

// ------------------------------------------------------------------------------------------------ DiskANN / Vamana
void free_vamana(lb2_index* x) {
    dev_free(&x->dv_nbrs); dev_free(&x->dv_codes); dev_free(&x->dv_tables_tr); dev_free(&x->dv_centroid);
    dev_free(&x->dv_chunk_offsets); dev_free(&x->dv_medoids); dev_free(&x->dv_centroid_data); dev_free(&x->dv_coords);
    VamanaWork& w = x->vw;
    dev_free(&w.aq); dev_free(&w.qnorm); dev_free(&w.qrot); dev_free(&w.lut); dev_free(&w.visited); dev_free(&w.full_ids);
    dev_free(&w.full_dist); dev_free(&w.n_full); dev_free(&w.next_query); dev_free(&w.error_flag); dev_free(&w.stamp);
    dev_free(&w.slot_of); dev_free(&w.claim); dev_free(&w.uniq_node); dev_free(&w.seq_start);
    dev_free(&x->d_vE);
    x->vcap_q = 0; x->vcap_full = 0; x->vcap_slots = 0; x->vcap_uniq = 0; x->vcap_E = 0;
}

template <class T>
bool upload(T** dst, const std::vector<T>& src) {
    if (src.empty()) return true;
    if (!dev_alloc(dst, src.size())) return false;
    if (cudaMemcpy(*dst, src.data(), src.size() * sizeof(T), cudaMemcpyHostToDevice) != cudaSuccess) {
        set_error("uploading the index failed");
        return false;
    }
    return true;
}

constexpr int64_t VAM_WAVE = 4096;  // queries per wave: bounds the per-query tables (LUT = n_chunks KB per query)

bool ensure_vamana_work(lb2_index* x, int64_t wave, int L, int beam, int cap_full, bool deferred) {
    VamanaWork& w = x->vw;
    const DevVamana& v = x->vam;
    if (x->vcap_q < wave || x->vcap_full < cap_full) {
        const size_t q = (size_t)std::max(wave, x->vcap_q), cf = (size_t)std::max(cap_full, x->vcap_full);
        if (!dev_alloc(&w.aq, q * v.data_dim) || !dev_alloc(&w.qrot, q * v.data_dim) || !dev_alloc(&w.qnorm, q) ||
            !dev_alloc(&w.lut, q * v.n_chunks * 256) || !dev_alloc(&w.full_ids, q * cf) || !dev_alloc(&w.full_dist, q * cf) ||
            !dev_alloc(&w.n_full, q))
            return false;
        x->vcap_q = (int64_t)q; x->vcap_full = (int)cf;
    }
    if (!w.next_query && (!dev_alloc(&w.next_query, 1) || !dev_alloc(&w.error_flag, 1) || !dev_alloc(&w.claim, 1))) return false;
    w.L = L; w.beam = beam; w.cap_full = x->vcap_full;
    vamana_plan(v, w, x->num_sms);
    const int slots = w.slots;
    w.vis_words = ((v.n + 31) / 32 + 3) & ~int64_t(3);
    if (x->vcap_slots < slots) {
        if (!dev_alloc(&w.visited, (size_t)slots * (size_t)w.vis_words)) return false;
        x->vcap_slots = slots;
        x->vis_dirty = true;
    }
    w.slots = slots;
    if (x->vis_dirty) {
        if (cudaMemsetAsync(w.visited, 0, (size_t)x->vcap_slots * (size_t)w.vis_words * 4, x->stream) != cudaSuccess) { set_error("memset(visited) failed"); return false; }
        x->vis_dirty = false;
    }
    if (deferred) {
        if (!w.stamp) {
            if (!dev_alloc(&w.stamp, (size_t)v.n) || !dev_alloc(&w.slot_of, (size_t)v.n)) return false;
            if (cudaMemsetAsync(w.stamp, 0, (size_t)v.n * 4, x->stream) != cudaSuccess) { set_error("memset(stamp) failed"); return false; }
            x->epoch = 0;
        }
        const int64_t need = wave * (int64_t)x->vcap_full;
        if (x->vcap_uniq < need) {
            if (!dev_alloc(&w.uniq_node, (size_t)need) || !dev_alloc(&w.seq_start, (size_t)need)) return false;
            x->vcap_uniq = need;
        }
        const int need_chunks = (int)(need / x->per_pass) + 2;
        if (!x->h_ctrl || x->max_chunks < need_chunks) {
            if (x->h_ctrl) cudaFreeHost(x->h_ctrl);
            if (x->h_bounds) cudaFreeHost(x->h_bounds);
            x->h_ctrl = nullptr; x->h_bounds = nullptr;
            x->max_chunks = need_chunks;
            if (cudaHostAlloc(reinterpret_cast<void**>(&x->h_ctrl), sizeof(HopCtrl), cudaHostAllocMapped) != cudaSuccess ||
                cudaHostAlloc(reinterpret_cast<void**>(&x->h_bounds), sizeof(int) * (x->max_chunks + 2), cudaHostAllocMapped) != cudaSuccess) {
                set_error("pinned control block allocation failed");
                return false;
            }
        }
    }
    return true;
}

int diskann_search_impl(lb2_index* x, int64_t nq, const float* d_q, int64_t k, float* d_D, int64_t* d_I,
                        const lb2_diskann_params* prm, lb2_search_stats* stats) {
    if (!x->is_vamana) { set_error("this handle is an HNSW index: use lb2_search"); return LB2_ERR_STATE; }
    lb2_diskann_params P;
    if (prm) P = *prm; else lb2_diskann_default_params(&P);
    if (nq < 0 || k <= 0 || k > 4096) { set_error("bad nq/k (nq=%lld k=%lld)", (long long)nq, (long long)k); return LB2_ERR_ARG; }
    if (P.complexity <= 0 || P.complexity > 16384) { set_error("complexity out of range: %d", P.complexity); return LB2_ERR_ARG; }
    if (P.beam_width <= 0 || P.beam_width > 512) { set_error("beam_width out of range: %d", P.beam_width); return LB2_ERR_ARG; }
    if (P.recompute_neighbors) {
        set_error("recompute_neighbors=1 (per-hop neighbour recompute inside DiskANN) is not implemented; LEANN never sets it");
        return LB2_ERR_UNSUPPORTED;
    }
    const DevVamana& v = x->vam;
    const bool deferred = P.deferred_fetch != 0, skip = P.skip_search_reorder != 0;
    if (deferred && (!x->d_tokens || !x->enc.loaded)) {
        set_error("deferred fetch (recompute_embeddings) needs lb2_set_passages() and lb2_set_encoder() first");
        return LB2_ERR_STATE;
    }
    if (deferred && x->enc.cfg.hidden != v.raw_dim) {
        set_error("encoder hidden size %d != index dimension %d", x->enc.cfg.hidden, v.raw_dim);
        return LB2_ERR_STATE;
    }
    if (!deferred && !skip && !v.coords) {
        set_error("recompute_embeddings=False needs the full-precision coordinates of <prefix>_disk.index (not read in partition mode)");
        return LB2_ERR_STATE;
    }
    if (stats) memset(stats, 0, sizeof(*stats));
    if (nq == 0) return LB2_OK;
    cudaStream_t st = x->stream;
    if (x->cap_qstats < nq) {
        if (!dev_alloc(&x->d_qndis, (size_t)nq) || !dev_alloc(&x->d_qnhops, (size_t)nq)) return LB2_ERR_CUDA;
        x->cap_qstats = nq;
    }
    x->last_nq = nq;
    const int L = P.complexity, beam = P.beam_width;
    const int cap_full = 4 * L + 2 * beam + 64;
    const int64_t wave = std::min<int64_t>(nq, VAM_WAVE);
    if (!ensure_vamana_work(x, wave, L, beam, cap_full, deferred)) return LB2_ERR_CUDA;
    if (deferred && !encoder_reserve(&x->enc, (int64_t)x->per_pass * x->enc.cfg.max_pos, x->per_pass)) return LB2_ERR_CUDA;

    x->ev_total.total_ms = 0; x->ev_enc.total_ms = 0;
    for (auto& pl : g_prof_pool) pl.total_ms = 0;
    g_gemm_flops = 0;
    g_prof_on = x->profile_gemm;
    cudaEventRecord(x->ev_total.get(), st);
    long long launches = 0, n_recomputed = 0, n_tokens = 0, n_waves = 0, n_requested = 0;
    VamanaWork& w = x->vw;
    for (int64_t q0 = 0; q0 < nq; q0 += wave) {
        const int64_t wq = std::min(wave, nq - q0);
        w.nq = wq; w.k = (int)k; w.flags = (deferred ? VAM_DEFERRED_FETCH : 0) | (skip ? VAM_SKIP_SEARCH_REORDER : 0);
        w.io_limit = P.io_limit ? P.io_limit : 0xffffffffu;
        w.queries = d_q + q0 * v.raw_dim;
        w.cmps = x->d_qndis + q0; w.hops = x->d_qnhops + q0;
        w.outD = d_D + q0 * k; w.outI = d_I + q0 * k;
        w.tok_off = x->d_tok_off; w.max_pos = x->enc.cfg.max_pos;
        cudaMemsetAsync(w.error_flag, 0, sizeof(int), st);
        if (!vamana_launch_prepare(st, v, w) || !vamana_launch_search(st, v, w, x->num_sms)) return LB2_ERR_CUDA;
        launches += 3 + (wq + 65534) / 65535 - 1;
        n_waves++;
        if (deferred) {
            x->epoch++;
            w.call_epoch = x->epoch;
            cudaMemsetAsync(w.claim, 0, sizeof(unsigned long long), st);
            if (!vamana_launch_collect(st, v, w)) return LB2_ERR_CUDA;
            gather_bounds_kernel<<<1, 64, 0, st>>>(w.claim, w.error_flag, w.seq_start, x->per_pass, x->h_ctrl, x->h_bounds, x->max_chunks);
            launches += 2;
            cudaError_t e = cudaStreamSynchronize(st);
            if (e != cudaSuccess) { set_error("vamana traversal failed: %s", cudaGetErrorString(e)); x->vis_dirty = true; return LB2_ERR_CUDA; }
            const HopCtrl c = *x->h_ctrl;
            if (c.n_done != 0) { set_error("a query expanded more than %d nodes (complexity %d)", cap_full, L); x->vis_dirty = true; return LB2_ERR_CUDA; }
            if (c.n_unique > x->vcap_uniq) { set_error("internal: vamana work list overflow"); return LB2_ERR_CUDA; }
            if (x->vcap_E < c.n_unique) {
                if (!dev_alloc(&x->d_vE, (size_t)c.n_unique * v.raw_dim)) { x->vcap_E = 0; return LB2_ERR_CUDA; }
                x->vcap_E = c.n_unique;
            }
            n_recomputed += c.n_unique;
            n_tokens += c.n_tokens;
            cudaEventRecord(x->ev_enc.get(), st);
            for (int ch = 0; ch < c.n_chunks; ch++) {
                const int first = ch * x->per_pass;
                const int n_seq = std::min(x->per_pass, c.n_unique - first);
                const int row_base = x->h_bounds[ch];
                const int n_tok = x->h_bounds[ch + 1] - row_base;
                if (!encoder_forward(&x->enc, st, x->d_tokens, x->d_tok_off, w.uniq_node + first, w.seq_start + first, row_base,
                                     n_seq, n_tok, x->d_vE + (size_t)first * v.raw_dim))
                    return LB2_ERR_CUDA;
                launches += encoder_kernels_per_pass(x->enc);
            }
            cudaEventRecord(x->ev_enc.get(), st);
            w.E = x->d_vE;
        }
        if (!vamana_launch_rerank(st, v, w)) return LB2_ERR_CUDA;
        launches++;
        x->v_last_wave = wq;
        if (stats && (nq > wave)) {  // several waves reuse n_full: read it before the next wave overwrites it
            std::vector<int> nf((size_t)wq);
            cudaMemcpyAsync(nf.data(), w.n_full, wq * sizeof(int), cudaMemcpyDeviceToHost, st);
            cudaStreamSynchronize(st);
            for (int64_t i = 0; i < wq; i++) n_requested += nf[i];
        }
    }
    cudaEventRecord(x->ev_total.get(), st);
    cudaError_t e = cudaStreamSynchronize(st);
    g_prof_on = false;
    if (e != cudaSuccess) { set_error("diskann search failed: %s", cudaGetErrorString(e)); x->vis_dirty = true; return LB2_ERR_CUDA; }
    int err_flag = 0;
    cudaMemcpy(&err_flag, w.error_flag, sizeof(int), cudaMemcpyDeviceToHost);
    if (err_flag) { set_error("a query expanded more than %d nodes (complexity %d)", cap_full, L); x->vis_dirty = true; return LB2_ERR_CUDA; }
    x->ev_total.drain(); x->ev_enc.drain();
    for (auto& pl : g_prof_pool) pl.drain();
    if (stats) {
        std::vector<long long> a((size_t)nq), b((size_t)nq);
        cudaMemcpy(a.data(), x->d_qndis, nq * sizeof(long long), cudaMemcpyDeviceToHost);
        cudaMemcpy(b.data(), x->d_qnhops, nq * sizeof(long long), cudaMemcpyDeviceToHost);
        for (int64_t i = 0; i < nq; i++) { stats->ndis += a[i]; stats->nhops += b[i]; }
        if (nq <= wave) {
            std::vector<int> nf((size_t)nq);
            cudaMemcpy(nf.data(), w.n_full, nq * sizeof(int), cudaMemcpyDeviceToHost);
            for (int64_t i = 0; i < nq; i++) n_requested += nf[i];
        }
        stats->n_requested = n_requested;
        stats->n_recomputed = n_recomputed;
        stats->n_tokens = n_tokens;
        stats->n_steps = n_waves;
        stats->n_kernel_launches = launches;
        stats->gpu_ms = x->ev_total.total_ms;
        stats->encoder_ms = x->ev_enc.total_ms;
        stats->gemm_ms = g_prof_pool[PROF_GEMM].total_ms;
        stats->gemm_flops = g_gemm_flops;
        stats->attention_ms = g_prof_pool[PROF_ATTN].total_ms;
        stats->norm_ms = g_prof_pool[PROF_NORM].total_ms;
    }
    return LB2_OK;
}

}  // namespace

// =============================================================================================
extern "C" {

const char* lb2_last_error(void) { return g_err.c_str(); }
int lb2_version(void) { return 100; }

void lb2_default_params(lb2_search_params* p) {
    p->efSearch = 64; p->beam_size = 1; p->batch_size = 0; p->check_relative_distance = 1;
    p->pq_pruning_ratio = 0.f; p->local_prune = 0; p->send_neigh_times_ratio = 0.f; p->recompute = 1;
}

static lb2_index* open_impl(const char* index_path, int device);

lb2_index* lb2_open(const char* index_path, int device) {
    try {
        return open_impl(index_path, device);
    } catch (const std::exception& e) {  // e.g. bad_alloc on a corrupt element count
        set_error("%s: malformed index (%s)", index_path ? index_path : "(null)", e.what());
    } catch (...) {
        set_error("%s: malformed index", index_path ? index_path : "(null)");
    }
    return nullptr;
}

static lb2_index* open_impl(const char* index_path, int device) {
    if (!index_path) { set_error("index_path is null"); return nullptr; }
    // the file is parsed and validated first (host work), so a malformed index is reported as such on any machine
    HostIndex h;
    std::string err;
    if (!read_compact_index(index_path, &h, &err)) { set_error("%s: %s", index_path, err.c_str()); return nullptr; }
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        set_error("no CUDA device available: libleann_b200 has no CPU path");
        return nullptr;
    }
    if (device < 0 || device >= ndev) { set_error("device %d out of range (%d devices)", device, ndev); return nullptr; }
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess || prop.major != 10) {
        set_error("device %d is sm_%d%d; this library is built for sm_100a (B200) only", device, prop.major, prop.minor);
        return nullptr;
    }
    lb2_index* x = new lb2_index();
    x->device = device;
    if (!use_device(x)) { delete x; return nullptr; }
    x->num_sms = prop.multiProcessorCount;
    x->profile_gemm = getenv("LB2_PROFILE_GEMM") && atoi(getenv("LB2_PROFILE_GEMM")) != 0;
    DevGraph& g = x->g;
    g.ntotal = h.ntotal; g.d = h.d; g.metric_ip = (h.metric_type == 0); g.entry_point = h.entry_point; g.max_level = h.max_level;
    x->n_edges = (int64_t)h.neighbors.size();
    for (int64_t i = 0; i < h.ntotal; i++) {
        const uint64_t ps = h.node_offsets[i], pe = h.node_offsets[i + 1];
        for (uint64_t p = ps; p + 1 < pe; p++) {
            const int deg = (int)(h.level_ptr[p + 1] - h.level_ptr[p]);
            if (p == ps) g.maxdeg0 = std::max(g.maxdeg0, deg); else g.maxdeg_up = std::max(g.maxdeg_up, deg);
        }
    }
    bool ok = dev_alloc(&x->d_node_offsets, h.node_offsets.size()) && dev_alloc(&x->d_level_ptr, h.level_ptr.size()) &&
              dev_alloc(&x->d_nbrs, h.neighbors.size());
    if (ok) {
        ok = cudaMemcpy(x->d_node_offsets, h.node_offsets.data(), h.node_offsets.size() * 8, cudaMemcpyHostToDevice) == cudaSuccess &&
             cudaMemcpy(x->d_level_ptr, h.level_ptr.data(), h.level_ptr.size() * 8, cudaMemcpyHostToDevice) == cudaSuccess &&
             cudaMemcpy(x->d_nbrs, h.neighbors.data(), h.neighbors.size() * 4, cudaMemcpyHostToDevice) == cudaSuccess;
        if (!ok) set_error("uploading the graph failed");
    }
    if (ok && !h.vectors.empty()) {
        ok = dev_alloc(&x->d_vectors, h.vectors.size()) &&
             cudaMemcpy(x->d_vectors, h.vectors.data(), h.vectors.size() * 4, cudaMemcpyHostToDevice) == cudaSuccess;
    }
    if (!ok) { lb2_close(x); return nullptr; }
    g.node_offsets = x->d_node_offsets; g.level_ptr = x->d_level_ptr; g.nbrs = x->d_nbrs;
    return x;
}

void lb2_close(lb2_index* x) {
    if (!x) return;
    cudaSetDevice(x->device);
    cudaDeviceSynchronize();
    free_state(x);
    encoder_free(&x->enc);
    dev_free(&x->d_node_offsets); dev_free(&x->d_level_ptr); dev_free(&x->d_nbrs);
    dev_free(&x->d_vectors); dev_free(&x->d_tokens); dev_free(&x->d_tok_off);
    dev_free(&x->dpq_tables_tr); dev_free(&x->dpq_centroid); dev_free(&x->dpq_chunk_offsets); dev_free(&x->dpq_codes);
    dev_free(&x->d_q); dev_free(&x->d_D); dev_free(&x->d_I); dev_free(&x->d_qndis); dev_free(&x->d_qnhops);
    dev_free(&x->d_enc_node); dev_free(&x->d_enc_start); dev_free(&x->d_enc_out);
    free_vamana(x);
    x->ev_total.destroy(); x->ev_enc.destroy();
    delete x;
}

int lb2_info(const lb2_index* x, lb2_index_info* o) {
    if (!x || !o) { set_error("null argument"); return LB2_ERR_ARG; }
    o->ntotal = x->g.ntotal; o->d = x->g.d; o->metric_type = x->g.metric_ip ? 0 : 1;
    o->entry_point = x->g.entry_point; o->max_level = x->g.max_level; o->n_edges = x->n_edges;
    o->max_degree_level0 = x->g.maxdeg0; o->max_degree_upper = x->g.maxdeg_up;
    o->has_vectors = x->d_vectors != nullptr; o->has_passages = x->d_tokens != nullptr; o->has_encoder = x->enc.loaded;
    o->device = x->device;
    return LB2_OK;
}

int lb2_set_vectors(lb2_index* x, const float* v) {
    if (!x || !v) { set_error("null argument"); return LB2_ERR_ARG; }
    if (!use_device(x)) return LB2_ERR_CUDA;
    const size_t n = (size_t)x->g.ntotal * x->g.d;
    if (!dev_alloc(&x->d_vectors, n)) return LB2_ERR_CUDA;
    if (cudaMemcpy(x->d_vectors, v, n * 4, cudaMemcpyHostToDevice) != cudaSuccess) { set_error("vector upload failed"); return LB2_ERR_CUDA; }
    return LB2_OK;
}

int lb2_set_vectors_device(lb2_index* x, const float* d_v) {
    if (!x || !d_v) { set_error("null argument"); return LB2_ERR_ARG; }
    if (!use_device(x)) return LB2_ERR_CUDA;
    const size_t n = (size_t)x->g.ntotal * x->g.d;
    if (!dev_alloc(&x->d_vectors, n)) return LB2_ERR_CUDA;
    if (cudaMemcpy(x->d_vectors, d_v, n * 4, cudaMemcpyDeviceToDevice) != cudaSuccess) { set_error("vector copy failed"); return LB2_ERR_CUDA; }
    return LB2_OK;
}

int lb2_set_passages(lb2_index* x, const uint16_t* tokens, const uint64_t* offsets) {
    if (!x || !tokens || !offsets) { set_error("null argument"); return LB2_ERR_ARG; }
    if (!use_device(x)) return LB2_ERR_CUDA;
    const int64_t N = x->g.ntotal;
    for (int64_t i = 0; i < N; i++)
        if (offsets[i + 1] <= offsets[i]) {  // the reference's tokenizer always emits [CLS] .. [SEP]: no empty passages
            set_error("passage %lld is empty or its offsets are not monotone", (long long)i);
            return LB2_ERR_ARG;
        }
    const uint64_t total = offsets[N] - offsets[0];
    if (offsets[0] != 0) { set_error("passage offsets must start at 0"); return LB2_ERR_ARG; }
    const int max_tok = max_token(tokens, total);
    if (x->enc.loaded && max_tok >= x->enc.cfg.vocab_size) {
        set_error("passage store holds token id %d but the encoder's vocabulary has %d entries", max_tok, x->enc.cfg.vocab_size);
        return LB2_ERR_ARG;
    }
    if (!dev_alloc(&x->d_tokens, (size_t)total + 8) || !dev_alloc(&x->d_tok_off, (size_t)N + 1)) return LB2_ERR_CUDA;
    if (cudaMemcpy(x->d_tokens, tokens, total * 2, cudaMemcpyHostToDevice) != cudaSuccess ||
        cudaMemcpy(x->d_tok_off, offsets, (N + 1) * 8, cudaMemcpyHostToDevice) != cudaSuccess) {
        set_error("passage upload failed");
        return LB2_ERR_CUDA;
    }
    x->h_tok_off.assign(offsets, offsets + N + 1);
    x->max_token = max_tok;
    return LB2_OK;
}

int lb2_load_pq_pruning(lb2_index* x, const char* pq_pivots_path, const char* pq_compressed_path) {
    if (!x || !pq_pivots_path || !pq_compressed_path) { set_error("null argument"); return LB2_ERR_ARG; }
    if (x->is_vamana) { set_error("this handle is a DiskANN index"); return LB2_ERR_STATE; }
    PqHost h;
    std::string err;
    try {
        if (!read_pq_files(pq_pivots_path, pq_compressed_path, &h, &err)) { set_error("%s", err.c_str()); return LB2_ERR_IO; }
    } catch (const std::exception& e) {
        set_error("%s: malformed PQ file (%s)", pq_pivots_path, e.what());
        return LB2_ERR_IO;
    }
    if (h.n != x->g.ntotal) { set_error("PQ codes cover %lld vectors, the index has %lld", (long long)h.n, (long long)x->g.ntotal); return LB2_ERR_ARG; }
    // the reference copies ndims - 1 query coordinates and appends a zero (HNSW_search.cpp:451-456)
    if (h.ndims < 2 || h.ndims - 1 > x->g.d) { set_error("PQ dimension %d does not fit queries of dimension %d", h.ndims, x->g.d); return LB2_ERR_ARG; }
    if (!use_device(x)) return LB2_ERR_CUDA;
    if (!upload(&x->dpq_tables_tr, h.tables_tr) || !upload(&x->dpq_centroid, h.centroid) || !upload(&x->dpq_chunk_offsets, h.chunk_offsets) ||
        !upload(&x->dpq_codes, h.codes))
        return LB2_ERR_CUDA;
    x->pq.tables_tr = x->dpq_tables_tr; x->pq.centroid = x->dpq_centroid; x->pq.chunk_offsets = x->dpq_chunk_offsets;
    x->pq.codes = x->dpq_codes; x->pq.ndims = h.ndims; x->pq.n_chunks = h.n_chunks;
    return LB2_OK;
}

size_t lb2_encoder_weight_count(const lb2_encoder_config* c) {
    if (!c) return 0;
    EncoderConfig e{c->vocab_size, c->hidden, c->layers, c->heads, c->ffn, c->max_pos, c->type_vocab, c->ln_eps, c->pooling, c->normalize};
    return encoder_weight_floats(e);
}

int lb2_set_encoder(lb2_index* x, const lb2_encoder_config* c, const float* w, size_t n) {
    if (!x || !c || !w) { set_error("null argument"); return LB2_ERR_ARG; }
    if (!use_device(x)) return LB2_ERR_CUDA;
    EncoderConfig e{c->vocab_size, c->hidden, c->layers, c->heads, c->ffn, c->max_pos, c->type_vocab, c->ln_eps, c->pooling, c->normalize};
    if (x->d_tokens && x->max_token >= c->vocab_size) {  // the embedding kernel indexes word_emb unchecked
        set_error("attached passages hold token id %d but the encoder's vocabulary has %d entries", x->max_token, c->vocab_size);
        return LB2_ERR_ARG;
    }
    if (!encoder_load(&x->enc, e, w, n)) return LB2_ERR_ARG;
    x->enc.num_sms = x->num_sms;
    return LB2_OK;
}

int lb2_configure(lb2_index* x, int32_t slots, int32_t per_pass) {
    if (!x) { set_error("null argument"); return LB2_ERR_ARG; }
    if (slots > 0) x->cfg_slots = slots;
    if (per_pass > 0 && per_pass != x->per_pass) {
        x->per_pass = per_pass;
        if (use_device(x)) { free_state(x); x->alloc_p = TravParams{}; }
        dev_free(&x->d_enc_node); dev_free(&x->d_enc_start); dev_free(&x->d_enc_out);
        x->cap_enc = 0;
    }
    return LB2_OK;
}

int lb2_set_option(lb2_index* x, const char* key, int64_t value) {
    if (!x || !key) { set_error("null argument"); return LB2_ERR_ARG; }
    if (!strcmp(key, "slots")) return lb2_configure(x, (int32_t)value, 0);
    if (!strcmp(key, "passages_per_pass")) return lb2_configure(x, 0, (int32_t)value);
    if (!strcmp(key, "dedup_scope")) {  // 0 = per hop, 1 = per search call
        if (value != 0 && value != 1) { set_error("dedup_scope must be 0 (hop) or 1 (call)"); return LB2_ERR_ARG; }
        x->dedup_call_scope = (int)value;
        return LB2_OK;
    }
    if (!strcmp(key, "profile")) { x->profile_gemm = value != 0; return LB2_OK; }
    if (!strcmp(key, "pq_queue_cap")) {
        if (value < 256 || value > (1 << 22)) { set_error("pq_queue_cap must lie in [256, 4194304]"); return LB2_ERR_ARG; }
        x->pq_cap = (int)value;
        return LB2_OK;
    }
    set_error("unknown option '%s'", key);
    return LB2_ERR_ARG;
}

int lb2_search_device(lb2_index* x, int64_t nq, const float* d_q, int64_t k, float* d_D, int64_t* d_I,
                      const lb2_search_params* p, lb2_search_stats* s) {
    if (!x || (nq > 0 && (!d_q || !d_D || !d_I))) { set_error("null argument"); return LB2_ERR_ARG; }
    if (!use_device(x)) return LB2_ERR_CUDA;
    return search_impl(x, nq, d_q, k, d_D, d_I, p, s);
}

int lb2_search(lb2_index* x, int64_t nq, const float* q, int64_t k, float* D, int64_t* I, const lb2_search_params* p,
               lb2_search_stats* s) {
    if (!x || (nq > 0 && (!q || !D || !I))) { set_error("null argument"); return LB2_ERR_ARG; }
    if (k <= 0) { set_error("k must be positive"); return LB2_ERR_ARG; }
    if (!use_device(x)) return LB2_ERR_CUDA;
    if (nq == 0) return LB2_OK;
    if (x->cap_q < nq) { if (!dev_alloc(&x->d_q, (size_t)nq * x->g.d)) return LB2_ERR_CUDA; x->cap_q = nq; }
    if (x->cap_out < nq * k) {
        if (!dev_alloc(&x->d_D, (size_t)(nq * k)) || !dev_alloc(&x->d_I, (size_t)(nq * k))) return LB2_ERR_CUDA;
        x->cap_out = nq * k;
    }
    if (cudaMemcpyAsync(x->d_q, q, (size_t)nq * x->g.d * 4, cudaMemcpyHostToDevice, x->stream) != cudaSuccess) {
        set_error("query upload failed"); return LB2_ERR_CUDA;
    }
    const int rc = search_impl(x, nq, x->d_q, k, x->d_D, x->d_I, p, s);
    if (rc != LB2_OK) return rc;
    if (cudaMemcpyAsync(D, x->d_D, (size_t)(nq * k) * 4, cudaMemcpyDeviceToHost, x->stream) != cudaSuccess ||
        cudaMemcpyAsync(I, x->d_I, (size_t)(nq * k) * 8, cudaMemcpyDeviceToHost, x->stream) != cudaSuccess ||
        cudaStreamSynchronize(x->stream) != cudaSuccess) {
        set_error("result download failed"); return LB2_ERR_CUDA;
    }
    return LB2_OK;
}

int lb2_last_query_stats(lb2_index* x, int64_t nq, int64_t* ndis, int64_t* nhops) {
    if (!x || nq != x->last_nq) { set_error("no stats for %lld queries", (long long)nq); return LB2_ERR_ARG; }
    if (!use_device(x)) return LB2_ERR_CUDA;
    static_assert(sizeof(long long) == sizeof(int64_t), "");
    if (ndis) cudaMemcpy(ndis, x->d_qndis, nq * 8, cudaMemcpyDeviceToHost);
    if (nhops) cudaMemcpy(nhops, x->d_qnhops, nq * 8, cudaMemcpyDeviceToHost);
    return LB2_OK;
}

int lb2_encode_ids(lb2_index* x, int64_t n, const int64_t* ids, float* out) {
    if (!x || (n > 0 && (!ids || !out))) { set_error("null argument"); return LB2_ERR_ARG; }
    if (!x->d_tokens) { set_error("no passages attached"); return LB2_ERR_STATE; }
    if (!use_device(x)) return LB2_ERR_CUDA;
    std::vector<int> nodes((size_t)n);
    for (int64_t i = 0; i < n; i++) {
        if (ids[i] < 0 || ids[i] >= x->g.ntotal) { set_error("passage id %lld out of range", (long long)ids[i]); return LB2_ERR_ARG; }
        nodes[i] = (int)ids[i];
    }
    return encode_impl(x, x->d_tokens, x->d_tok_off, x->h_tok_off.data(), n, nodes.data(), 0, out, false);
}

int lb2_encode_range_device(lb2_index* x, int64_t first, int64_t n, float* d_out) {
    if (!x || (n > 0 && !d_out)) { set_error("null argument"); return LB2_ERR_ARG; }
    if (!x->d_tokens) { set_error("no passages attached"); return LB2_ERR_STATE; }
    if (first < 0 || first + n > x->g.ntotal) { set_error("range out of bounds"); return LB2_ERR_ARG; }
    if (!use_device(x)) return LB2_ERR_CUDA;
    return encode_impl(x, x->d_tokens, x->d_tok_off, x->h_tok_off.data(), n, nullptr, first, d_out, true);
}

int lb2_encode_tokens(lb2_index* x, int64_t n, const uint16_t* tokens, const uint64_t* offsets, float* out) {
    if (!x || (n > 0 && (!tokens || !offsets || !out))) { set_error("null argument"); return LB2_ERR_ARG; }
    if (!use_device(x)) return LB2_ERR_CUDA;
    if (n == 0) return LB2_OK;
    if (offsets[0] != 0) { set_error("offsets must start at 0"); return LB2_ERR_ARG; }
    for (int64_t i = 0; i < n; i++)
        if (offsets[i + 1] <= offsets[i]) { set_error("sequence %lld is empty or its offsets are not monotone", (long long)i); return LB2_ERR_ARG; }
    if (x->enc.loaded && max_token(tokens, offsets[n]) >= x->enc.cfg.vocab_size) {
        set_error("token id out of range for a vocabulary of %d entries", x->enc.cfg.vocab_size);
        return LB2_ERR_ARG;
    }
    uint16_t* dt = nullptr;
    uint64_t* doff = nullptr;
    const uint64_t total = offsets[n];
    if (!dev_alloc(&dt, (size_t)total + 8) || !dev_alloc(&doff, (size_t)n + 1)) { dev_free(&dt); dev_free(&doff); return LB2_ERR_CUDA; }
    cudaMemcpy(dt, tokens, total * 2, cudaMemcpyHostToDevice);
    cudaMemcpy(doff, offsets, (n + 1) * 8, cudaMemcpyHostToDevice);
    const int rc = encode_impl(x, dt, doff, offsets, n, nullptr, 0, out, false);
    dev_free(&dt); dev_free(&doff);
    return rc;
}

// ---------------------------------------------------------------- DiskANN / Vamana entry points
void lb2_diskann_default_params(lb2_diskann_params* p) {
    memset(p, 0, sizeof(*p));
    p->complexity = 64; p->beam_width = 1; p->deferred_fetch = 1; p->global_pruning = 1;
}

static lb2_index* diskann_open_impl(const char* index_prefix, const char* partition_prefix, int metric, int device);

lb2_index* lb2_diskann_open(const char* index_prefix, const char* partition_prefix, int metric, int device) {
    try {
        return diskann_open_impl(index_prefix, partition_prefix, metric, device);
    } catch (const std::exception& e) {
        set_error("%s: malformed index (%s)", index_prefix ? index_prefix : "(null)", e.what());
    } catch (...) {
        set_error("%s: malformed index", index_prefix ? index_prefix : "(null)");
    }
    return nullptr;
}

static lb2_index* diskann_open_impl(const char* index_prefix, const char* partition_prefix, int metric, int device) {
    if (!index_prefix) { set_error("index_prefix is null"); return nullptr; }
    VamanaHost h;
    std::string err;
    if (!read_diskann_index(index_prefix, partition_prefix, metric, &h, &err)) { set_error("%s", err.c_str()); return nullptr; }
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        set_error("no CUDA device available: libleann_b200 has no CPU path");
        return nullptr;
    }
    if (device < 0 || device >= ndev) { set_error("device %d out of range (%d devices)", device, ndev); return nullptr; }
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess || prop.major != 10) {
        set_error("device %d is sm_%d%d; this library is built for sm_100a (B200) only", device, prop.major, prop.minor);
        return nullptr;
    }
    lb2_index* x = new lb2_index();
    x->device = device;
    if (!use_device(x)) { delete x; return nullptr; }
    x->num_sms = prop.multiProcessorCount;
    x->profile_gemm = getenv("LB2_PROFILE_GEMM") && atoi(getenv("LB2_PROFILE_GEMM")) != 0;
    x->is_vamana = true;
    x->vam_partitioned = h.partitioned;
    x->vam_edges = h.n_edges;
    bool ok = upload(&x->dv_nbrs, h.nbrs) && upload(&x->dv_codes, h.codes) && upload(&x->dv_tables_tr, h.tables_tr) &&
              upload(&x->dv_centroid, h.centroid) && upload(&x->dv_chunk_offsets, h.chunk_offsets) && upload(&x->dv_medoids, h.medoids) &&
              upload(&x->dv_centroid_data, h.centroid_data) && upload(&x->dv_coords, h.coords);
    if (!ok) { lb2_close(x); return nullptr; }
    DevVamana& v = x->vam;
    v.n = h.n; v.data_dim = h.data_dim; v.raw_dim = metric == LB2_METRIC_MIPS ? h.data_dim - 1 : h.data_dim;
    v.metric = metric; v.R = h.R; v.n_chunks = h.n_chunks; v.n_medoids = (int)h.medoids.size();
    v.nbrs = x->dv_nbrs; v.codes = x->dv_codes; v.tables_tr = x->dv_tables_tr; v.centroid = x->dv_centroid;
    v.chunk_offsets = x->dv_chunk_offsets; v.medoids = x->dv_medoids; v.centroid_data = x->dv_centroid_data; v.coords = x->dv_coords;
    v.max_base_norm = h.max_base_norm;
    // the shared passage / encoder entry points size themselves from these
    x->g.ntotal = h.n; x->g.d = v.raw_dim; x->g.metric_ip = metric != LB2_METRIC_L2; x->g.entry_point = (int)h.medoids[0];
    x->n_edges = h.n_edges;
    return x;
}

int lb2_diskann_info(const lb2_index* x, lb2_diskann_info_t* o) {
    if (!x || !o) { set_error("null argument"); return LB2_ERR_ARG; }
    if (!x->is_vamana) { set_error("not a DiskANN handle"); return LB2_ERR_STATE; }
    const DevVamana& v = x->vam;
    o->npts = v.n; o->dim = v.raw_dim; o->data_dim = v.data_dim; o->n_chunks = v.n_chunks; o->max_degree = v.R; o->metric = v.metric;
    o->n_medoids = v.n_medoids; o->partitioned = x->vam_partitioned; o->has_coords = v.coords != nullptr;
    o->max_base_norm = v.max_base_norm; o->pad = 0; o->n_edges = x->vam_edges;
    return LB2_OK;
}

int lb2_diskann_search_device(lb2_index* x, int64_t nq, const float* d_q, int64_t k, float* d_D, int64_t* d_I,
                              const lb2_diskann_params* p, lb2_search_stats* s) {
    if (!x || (nq > 0 && (!d_q || !d_D || !d_I))) { set_error("null argument"); return LB2_ERR_ARG; }
    if (!use_device(x)) return LB2_ERR_CUDA;
    return diskann_search_impl(x, nq, d_q, k, d_D, d_I, p, s);
}

int lb2_diskann_search(lb2_index* x, int64_t nq, const float* q, int64_t k, float* D, int64_t* I, const lb2_diskann_params* p,
                       lb2_search_stats* s) {
    if (!x || (nq > 0 && (!q || !D || !I))) { set_error("null argument"); return LB2_ERR_ARG; }
    if (k <= 0) { set_error("k must be positive"); return LB2_ERR_ARG; }
    if (!x->is_vamana) { set_error("this handle is an HNSW index: use lb2_search"); return LB2_ERR_STATE; }
    if (!use_device(x)) return LB2_ERR_CUDA;
    if (nq == 0) return LB2_OK;
    if (x->cap_q < nq) { if (!dev_alloc(&x->d_q, (size_t)nq * x->g.d)) return LB2_ERR_CUDA; x->cap_q = nq; }
    if (x->cap_out < nq * k) {
        if (!dev_alloc(&x->d_D, (size_t)(nq * k)) || !dev_alloc(&x->d_I, (size_t)(nq * k))) return LB2_ERR_CUDA;
        x->cap_out = nq * k;
    }
    if (cudaMemcpyAsync(x->d_q, q, (size_t)nq * x->g.d * 4, cudaMemcpyHostToDevice, x->stream) != cudaSuccess) {
        set_error("query upload failed"); return LB2_ERR_CUDA;
    }
    const int rc = diskann_search_impl(x, nq, x->d_q, k, x->d_D, x->d_I, p, s);
    if (rc != LB2_OK) return rc;
    if (cudaMemcpyAsync(D, x->d_D, (size_t)(nq * k) * 4, cudaMemcpyDeviceToHost, x->stream) != cudaSuccess ||
        cudaMemcpyAsync(I, x->d_I, (size_t)(nq * k) * 8, cudaMemcpyDeviceToHost, x->stream) != cudaSuccess ||
        cudaStreamSynchronize(x->stream) != cudaSuccess) {
        set_error("result download failed"); return LB2_ERR_CUDA;
    }
    return LB2_OK;
}

int lb2_diskann_last_expansions(lb2_index* x, int64_t nq, int32_t cap, uint32_t* ids, int32_t* n_full) {
    if (!x || !ids || !n_full || cap <= 0) { set_error("null argument"); return LB2_ERR_ARG; }
    if (!x->is_vamana || nq != x->last_nq || nq > x->v_last_wave) { set_error("no expansion lists for %lld queries", (long long)nq); return LB2_ERR_ARG; }
    if (!use_device(x)) return LB2_ERR_CUDA;
    const VamanaWork& w = x->vw;
    std::vector<int> nf((size_t)nq);
    std::vector<uint32_t> all((size_t)nq * w.cap_full);
    if (cudaMemcpy(nf.data(), w.n_full, nq * sizeof(int), cudaMemcpyDeviceToHost) != cudaSuccess ||
        cudaMemcpy(all.data(), w.full_ids, all.size() * 4, cudaMemcpyDeviceToHost) != cudaSuccess) { set_error("download failed"); return LB2_ERR_CUDA; }
    for (int64_t q = 0; q < nq; q++) {
        n_full[q] = nf[q];
        for (int j = 0; j < cap; j++) ids[q * cap + j] = j < nf[q] && j < w.cap_full ? all[(size_t)q * w.cap_full + j] : 0xffffffffu;
    }
    return LB2_OK;
}

// ---------------------------------------------------------------- unit-test hooks
int lb2_test_gemm_f16(const void* dA, const void* dW, const float* dbias, const void* dres, void* dC, int M, int N,
                      int K, int epi) {
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (!gemm_f16(0, (const __half*)dA, nullptr, (const __half*)dW, dbias, (const __half*)dres, (__half*)dC, M, N, K, epi, sms))
        return LB2_ERR_CUDA;
    cudaError_t e = cudaDeviceSynchronize();
    if (e != cudaSuccess) { set_error("gemm: %s", cudaGetErrorString(e)); return LB2_ERR_CUDA; }
    return LB2_OK;
}

int lb2_test_gemm_grouped_f16(const void* dA, const void* dW, const float* dbias, void* dC, int M, int N, int K, int c_group) {
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (!gemm_f16(0, (const __half*)dA, nullptr, (const __half*)dW, dbias, nullptr, (__half*)dC, M, N, K, EPI_BIAS, sms, c_group))
        return LB2_ERR_CUDA;
    cudaError_t e = cudaDeviceSynchronize();
    if (e != cudaSuccess) { set_error("gemm: %s", cudaGetErrorString(e)); return LB2_ERR_CUDA; }
    return LB2_OK;
}

int lb2_test_gemm_res_ln_f16(const void* dA, const void* dW, const float* dbias, const void* dres, const float* dgamma,
                             const float* dbeta, float eps, void* dC, int M, int N, int K) {
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const bool ok = gemm_f16_res_ln(0, (const __half*)dA, nullptr, (const __half*)dW, dbias, (const __half*)dres, dgamma, dbeta, eps,
                                    (__half*)dC, M, N, K, sms);
    cudaError_t e = cudaDeviceSynchronize();
    if (!ok) return LB2_ERR_ARG;
    if (e != cudaSuccess) { set_error("gemm_res_ln: %s", cudaGetErrorString(e)); return LB2_ERR_CUDA; }
    return LB2_OK;
}

int lb2_test_layernorm_f16(const void* din, const float* dg, const float* db, void* dout, int rows, int hidden, float eps) {
    if (!launch_layernorm(0, (const __half*)din, dg, db, (__half*)dout, rows, hidden, eps)) return LB2_ERR_CUDA;
    cudaError_t e = cudaDeviceSynchronize();
    if (e != cudaSuccess) { set_error("layernorm: %s", cudaGetErrorString(e)); return LB2_ERR_CUDA; }
    return LB2_OK;
}

int lb2_test_attention_f16(const void* dqkv, const int32_t* d_seq_start, const int32_t* d_seq_len, int n_seq, int n_tokens,
                           int hidden, int heads, int max_len, void* dctx) {
    static int* items = nullptr;  // scratch of the hook: grows, never shrinks
    static int cap = 0;
    if (n_seq > cap) {
        if (!dev_alloc(&items, (size_t)n_seq * 8 + 1)) { cap = 0; return LB2_ERR_CUDA; }
        cap = n_seq;
    }
    const bool ok = launch_attention(0, (const __half*)dqkv, d_seq_start, d_seq_len, items, items + (size_t)cap * 8, 0, max_len,
                                     n_seq, n_tokens, hidden, heads, (__half*)dctx, true);
    cudaError_t e = cudaDeviceSynchronize();
    if (!ok) return LB2_ERR_CUDA;
    if (e != cudaSuccess) { set_error("attention: %s", cudaGetErrorString(e)); return LB2_ERR_CUDA; }
    return LB2_OK;
}

}  // extern "C"
