// DiskANN/Vamana query path on the GPU: what PQFlashIndex::cached_beam_search does per query
// (DiskANN/src/pq_flash_index.cpp:1779-2906) as LEANN's DiskannSearcher drives it
// (diskann_backend.py:383-472: recompute_neighbors=false, so the traversal scores with PQ distances only and
// the expanded nodes are re-ranked once at the end — from freshly encoded passages when recompute is on).
// All citations below are under /root/reference/packages/leann-backend-diskann/third_party/DiskANN/.
//
//   vamana_prepare_kernel   query normalisation / MIPS extension (:1819-1848) + centring (src/pq.cpp:180-198)
//   vamana_lut_kernel       populate_chunk_distances (src/pq.cpp:201-219): 256 x n_chunks table per query
//   vamana_search_kernel    persistent, one warp per in-flight query: NeighborPriorityQueue in shared memory
//                           (include/neighbor.h:39-152), beam selection (:2180-2211), adjacency row read,
//                           visited bitset in HBM, PQ distance lookups (src/pq.cpp:302-340), ordered inserts
//   vamana_collect_kernel   de-duplicates the expanded nodes of all queries into the encoder's work list
//   vamana_rerank_kernel    preprocess_fetched_embeddings (:1723-1777) + full-precision distance + sort + output
//                           rescale (:2761, 2861-2883)
//
// Arithmetic that decides ids is bit-identical to the CPU checker (the C restatement pinned to the reference's compiled
// pq.cpp / neighbor.h): PQ table entries are fused
// multiply-adds in dimension order (what the reference's -mfma build executes), PQ distances are plain
// fp32 sums in chunk order, full-precision distances use the canonical lane-strided order of oracle/canon_dist.h.
#include "vamana.cuh"

#include <algorithm>
#include <cfloat>

namespace lb2 {

namespace {

constexpr unsigned FULL = 0xffffffffu;
constexpr uint32_t EXPANDED = 0x80000000u;

// ------------------------------------------------------------------------------------------------ query preparation
// one block per query; thread 0 accumulates |q|^2 in index order with fma (as the reference's build does)
__global__ void vamana_prepare_kernel(DevVamana v, VamanaWork w) {
    const int64_t q = blockIdx.x;
    const float* src = w.queries + q * v.raw_dim;
    float* aq = w.aq + q * v.data_dim;
    float* qrot = w.qrot + q * v.data_dim;
    __shared__ float s_norm;
    const int D = v.data_dim;
    if (v.metric == VAM_MIPS || v.metric == VAM_COSINE) {
        const int inherent = v.metric == VAM_COSINE ? D : D - 1;
        if (threadIdx.x == 0) {
            float nrm = 0.f;
            for (int i = 0; i < inherent; i++) nrm = __fmaf_rn(src[i], src[i], nrm);
            s_norm = __fsqrt_rn(nrm);
            w.qnorm[q] = s_norm;
        }
        __syncthreads();
        for (int i = threadIdx.x; i < D; i += blockDim.x) {
            const float a = i < inherent ? __fdiv_rn(src[i], s_norm) : 0.f;
            aq[i] = a;
            qrot[i] = __fsub_rn(a, v.centroid[i]);
        }
    } else {
        if (threadIdx.x == 0) w.qnorm[q] = 0.f;
        for (int i = threadIdx.x; i < D; i += blockDim.x) {
            aq[i] = src[i];
            qrot[i] = __fsub_rn(src[i], v.centroid[i]);
        }
    }
}

// grid (n_chunks, nq), 256 threads: one table entry per thread
__global__ void vamana_lut_kernel(DevVamana v, VamanaWork w) {
    const int chunk = blockIdx.x;
    const int64_t q = blockIdx.y;
    const float* qrot = w.qrot + q * v.data_dim;
    float acc = 0.f;
    for (uint32_t j = v.chunk_offsets[chunk]; j < v.chunk_offsets[chunk + 1]; j++) {
        const float diff = __fsub_rn(v.tables_tr[(size_t)j * 256 + threadIdx.x], qrot[j]);
        acc = __fmaf_rn(diff, diff, acc);
    }
    w.lut[(q * v.n_chunks + chunk) * 256 + threadIdx.x] = acc;
}

// ------------------------------------------------------------------------------------------------ traversal
struct Queue {  // NeighborPriorityQueue of one warp: ids (bit 31 = expanded) and distances, L + 1 slots each
    uint32_t* ids;
    float* dist;
    int size, cap, cur;
};

__device__ __forceinline__ bool nbr_less(uint32_t ia, float da, uint32_t ib, float db) {
    return da < db || (da == db && ia < ib);
}

// include/neighbor.h:56-97; every lane calls with the same arguments
__device__ void queue_insert(Queue& q, uint32_t id, float d, int lane) {
    if (q.size == q.cap && nbr_less(q.ids[q.size - 1] & ~EXPANDED, q.dist[q.size - 1], id, d)) return;
    int lo = 0, hi = q.size;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        const uint32_t mi = q.ids[mid] & ~EXPANDED;
        if (nbr_less(id, d, mi, q.dist[mid])) hi = mid;
        else if (mi == id) return;
        else lo = mid + 1;
    }
    for (int base = q.size; base > lo; base -= 32) {  // memmove [lo, size) up by one, top chunk first
        const int i = base - 1 - lane;
        uint32_t vi = 0; float vd = 0.f;
        const bool ok = i >= lo;
        if (ok) { vi = q.ids[i]; vd = q.dist[i]; }
        __syncwarp();
        if (ok) { q.ids[i + 1] = vi; q.dist[i + 1] = vd; }
        __syncwarp();
    }
    if (lane == 0) { q.ids[lo] = id; q.dist[lo] = d; }
    __syncwarp();
    if (q.size < q.cap) q.size++;
    if (lo < q.cur) q.cur = lo;
}

// include/neighbor.h:99-108
__device__ void queue_closest_unexpanded(Queue& q, uint32_t* id, float* d, int lane) {
    const int pre = q.cur;
    *id = q.ids[pre] & ~EXPANDED;
    *d = q.dist[pre];
    __syncwarp();
    if (lane == 0) q.ids[pre] |= EXPANDED;
    __syncwarp();
    while (q.cur < q.size && (q.ids[q.cur] & EXPANDED)) q.cur++;
}

// PQ distance of one node: sum over chunks, in chunk order, of lut[chunk][code]  (src/pq.cpp:324-340)
__device__ __forceinline__ float pq_distance(const uint8_t* __restrict__ cp, const float* __restrict__ lut, int n_chunks) {
    float acc = 0.f;
    int c = 0;
    while (c < n_chunks && (reinterpret_cast<uintptr_t>(cp + c) & 3)) {
        acc = __fadd_rn(acc, __ldg(lut + c * 256 + cp[c]));
        c++;
    }
    for (; c + 4 <= n_chunks; c += 4) {
        const uint32_t wv = __ldg(reinterpret_cast<const uint32_t*>(cp + c));
        acc = __fadd_rn(acc, __ldg(lut + (c + 0) * 256 + (wv & 255u)));
        acc = __fadd_rn(acc, __ldg(lut + (c + 1) * 256 + ((wv >> 8) & 255u)));
        acc = __fadd_rn(acc, __ldg(lut + (c + 2) * 256 + ((wv >> 16) & 255u)));
        acc = __fadd_rn(acc, __ldg(lut + (c + 3) * 256 + (wv >> 24)));
    }
    for (; c < n_chunks; c++) acc = __fadd_rn(acc, __ldg(lut + c * 256 + cp[c]));
    return acc;
}

__device__ __forceinline__ float canon_l2(const float* __restrict__ a, const float* __restrict__ b, int d, int lane) {
    float acc = 0.f;
    for (int j = lane; j < d; j += 32) {
        const float t = __fsub_rn(a[j], __ldg(b + j));
        acc = __fmaf_rn(t, t, acc);
    }
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) acc += __shfl_xor_sync(FULL, acc, o);
    return acc;
}

__global__ void __launch_bounds__(256) vamana_search_kernel(DevVamana v, VamanaWork w, int warps_per_block) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int per_warp_words = 2 * (w.L + 1) + 2 * w.beam;
    uint32_t* base = reinterpret_cast<uint32_t*>(smem_raw) + (size_t)warp * per_warp_words;
    Queue q;
    q.ids = base;
    q.dist = reinterpret_cast<float*>(base + (w.L + 1));
    uint32_t* frontier = base + 2 * (w.L + 1);
    float* frontier_d = reinterpret_cast<float*>(frontier + w.beam);
    const int slot = blockIdx.x * warps_per_block + warp;
    uint32_t* vis = w.visited + (size_t)slot * w.vis_words;
    const int R = v.R;

    for (;;) {
        int qi = 0;
        if (lane == 0) qi = atomicAdd(w.next_query, 1);
        qi = __shfl_sync(FULL, qi, 0);
        if (qi >= w.nq) break;
        const float* lut = w.lut + (size_t)qi * v.n_chunks * 256;
        const float* aq = w.aq + (size_t)qi * v.data_dim;
        uint32_t* full_ids = w.full_ids + (size_t)qi * w.cap_full;
        float* full_dist = w.full_dist + (size_t)qi * w.cap_full;
        q.size = 0; q.cap = w.L; q.cur = 0;
        int n_full = 0;
        bool overflow = false;
        long long cmps = 0, hops = 0;
        uint32_t num_ios = 0;

        // medoid seed (:2117-2158)
        uint32_t best_medoid = 0;
        float best_dist = FLT_MAX;
        for (int m = 0; m < v.n_medoids; m++) {
            const float cur = v.centroid_data ? canon_l2(aq, v.centroid_data + (size_t)m * v.data_dim, v.data_dim, lane) : 0.f;
            if (cur < best_dist) { best_medoid = v.medoids[m]; best_dist = cur; }
        }
        {
            const float d0 = pq_distance(v.codes + (size_t)best_medoid * v.n_chunks, lut, v.n_chunks);
            queue_insert(q, best_medoid, d0, lane);
            if (lane == 0) atomicOr(&vis[best_medoid >> 5], 1u << (best_medoid & 31));
        }

        while (q.cur < q.size && num_ios < w.io_limit) {  // :2180
            int nf = 0;
            while (q.cur < q.size && nf < w.beam) {       // :2190-2211 (num_seen == frontier size: no node cache)
                uint32_t id; float d;
                queue_closest_unexpanded(q, &id, &d, lane);
                if (lane == 0) { frontier[nf] = id; frontier_d[nf] = d; }
                nf++;
            }
            __syncwarp();
            if (nf > 0) hops++;
            num_ios += (uint32_t)nf;
            for (int f = 0; f < nf; f++) {                // :2419-2612 with batch_recompute == false
                const uint32_t node = frontier[f];
                if (n_full < w.cap_full) {
                    if (lane == 0) {
                        full_ids[n_full] = node;
                        full_dist[n_full] = frontier_d[f];  // PQ distance; replaced by the re-rank unless skip_search_reorder
                    }
                    n_full++;
                } else {
                    overflow = true;
                }
                const int32_t* row = v.nbrs + (size_t)node * R;
                for (int b0 = 0; b0 < R; b0 += 32) {
                    const int m = b0 + lane;
                    const int32_t nb = m < R ? __ldg(row + m) : -1;
                    bool is_new = false;
                    float pd = 0.f;
                    if (nb >= 0) {
                        const uint32_t bit = 1u << (nb & 31);
                        is_new = (atomicOr(&vis[nb >> 5], bit) & bit) == 0;  // visited.insert(id).second
                        if (is_new) pd = pq_distance(v.codes + (size_t)nb * v.n_chunks, lut, v.n_chunks);
                    }
                    unsigned todo = __ballot_sync(FULL, is_new);
                    cmps += __popc(todo);
                    while (todo) {  // retset.insert in neighbour order
                        const int src = __ffs(todo) - 1;
                        todo &= todo - 1;
                        const uint32_t id = (uint32_t)__shfl_sync(FULL, nb, src);
                        const float d = __shfl_sync(FULL, pd, src);
                        queue_insert(q, id, d, lane);
                    }
                    if (__ballot_sync(FULL, nb < 0)) break;  // rows are degree-prefix packed
                }
            }
        }

        // un-mark everything this query marked: the neighbours of its expanded nodes + the medoid
        if (lane == 0) atomicAnd(&vis[best_medoid >> 5], ~(1u << (best_medoid & 31)));
        for (int i = 0; i < n_full; i++) {
            const int32_t* row = v.nbrs + (size_t)full_ids[i] * R;
            for (int m = lane; m < R; m += 32) {
                const int32_t nb = __ldg(row + m);
                if (nb >= 0) atomicAnd(&vis[nb >> 5], ~(1u << (nb & 31)));
            }
        }
        if (lane == 0) {
            w.n_full[qi] = n_full;
            w.cmps[qi] = cmps;
            w.hops[qi] = hops;
            if (overflow) atomicExch(w.error_flag, 1);
        }
        __syncwarp();
    }
}

// ------------------------------------------------------------------------------------------------ deferred fetch work list
// one thread per (query, expansion): the first to stamp a node claims a row of E and its packed token range
__global__ void vamana_collect_kernel(DevVamana v, VamanaWork w) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    const int64_t qi = i / w.cap_full;
    const int j = (int)(i % w.cap_full);
    if (qi >= w.nq || j >= w.n_full[qi]) return;
    const uint32_t node = w.full_ids[qi * w.cap_full + j];
    if (atomicExch(&w.stamp[node], w.call_epoch) == w.call_epoch) return;
    const uint64_t len64 = w.tok_off[node + 1] - w.tok_off[node];
    const unsigned long long len = len64 < (uint64_t)w.max_pos ? len64 : (unsigned long long)w.max_pos;
    const unsigned long long c = atomicAdd(w.claim, (1ull << 40) | len);
    const int row = (int)(c >> 40);
    w.uniq_node[row] = (int)node;
    w.seq_start[row] = (int)(c & ((1ull << 40) - 1));
    w.slot_of[node] = row;
}

// ------------------------------------------------------------------------------------------------ re-rank + output
// one warp per query
__global__ void vamana_rerank_kernel(DevVamana v, VamanaWork w) {
    const int lane = threadIdx.x & 31;
    const int64_t qi = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    if (qi >= w.nq) return;
    const int n_full = w.n_full[qi];
    const uint32_t* ids = w.full_ids + qi * w.cap_full;
    float* dist = w.full_dist + qi * w.cap_full;
    const float* aq = w.aq + qi * v.data_dim;
    const int D = v.data_dim, d = v.raw_dim;
    const bool deferred = (w.flags & VAM_DEFERRED_FETCH) != 0, skip = (w.flags & VAM_SKIP_SEARCH_REORDER) != 0;
    if (deferred) {
        for (int i = 0; i < n_full; i++) {
            const float* e = w.E + (size_t)w.slot_of[ids[i]] * d;
            float acc = 0.f;
            if (v.metric == VAM_MIPS) {  // :1735-1755
                float ns = 0.f;
                for (int j = lane; j < d; j += 32) { const float x = __ldg(e + j); ns = __fmaf_rn(x, x, ns); }
#pragma unroll
                for (int o = 16; o >= 1; o >>= 1) ns += __shfl_xor_sync(FULL, ns, o);
                float res = __fsub_rn(1.f, __fdiv_rn(ns, __fmul_rn(v.max_base_norm, v.max_base_norm)));
                res = res <= 0.f ? 0.f : __fsqrt_rn(res);
                for (int j = lane; j < D; j += 32) {
                    const float t = j < d ? __fdiv_rn(__ldg(e + j), v.max_base_norm) : res;
                    const float df = __fsub_rn(aq[j], t);
                    acc = __fmaf_rn(df, df, acc);
                }
            } else if (v.metric == VAM_COSINE) {  // :1756-1772
                float ns = 0.f;
                for (int j = lane; j < d; j += 32) { const float x = __ldg(e + j); ns = __fmaf_rn(x, x, ns); }
#pragma unroll
                for (int o = 16; o >= 1; o >>= 1) ns += __shfl_xor_sync(FULL, ns, o);
                const float nrm = __fsqrt_rn(ns);
                for (int j = lane; j < D; j += 32) {
                    float t = j < d ? __ldg(e + j) : 0.f;
                    if (nrm > 0.f) t = __fdiv_rn(t, nrm);
                    const float df = __fsub_rn(aq[j], t);
                    acc = __fmaf_rn(df, df, acc);
                }
            } else {
                for (int j = lane; j < D; j += 32) {
                    const float df = __fsub_rn(aq[j], j < d ? __ldg(e + j) : 0.f);
                    acc = __fmaf_rn(df, df, acc);
                }
            }
#pragma unroll
            for (int o = 16; o >= 1; o >>= 1) acc += __shfl_xor_sync(FULL, acc, o);
            if (lane == 0) dist[i] = acc;
        }
    } else if (!skip) {
        for (int i = 0; i < n_full; i++) {
            const float dd = canon_l2(aq, v.coords + (size_t)ids[i] * D, D, lane);
            if (lane == 0) dist[i] = dd;
        }
    }
    __syncwarp();
    // std::sort(full_retset) (:2761) — only the first k matter: k rounds of arg-min on (distance, id)
    const float scale = __fmul_rn(v.max_base_norm, w.qnorm[qi]);
    uint32_t last_id = 0; float last_d = -FLT_MAX; bool have_last = false;
    for (int r = 0; r < w.k; r++) {
        float bd = FLT_MAX; uint32_t bi = 0xffffffffu; bool found = false;
        for (int i = lane; i < n_full; i += 32) {
            const float di = dist[i]; const uint32_t ii = ids[i];
            // strictly after the previous pick in (distance, id) order; full_retset ids are unique
            if (have_last && !nbr_less(last_id, last_d, ii, di)) continue;
            if (!found || nbr_less(ii, di, bi, bd)) { bd = di; bi = ii; found = true; }
        }
#pragma unroll
        for (int o = 16; o >= 1; o >>= 1) {
            const float od = __shfl_xor_sync(FULL, bd, o);
            const uint32_t oi = __shfl_xor_sync(FULL, bi, o);
            const bool of = __shfl_xor_sync(FULL, found ? 1 : 0, o) != 0;
            if (of && (!found || nbr_less(oi, od, bi, bd))) { bd = od; bi = oi; found = true; }
        }
        if (lane == 0) {
            if (!found) {  // fewer expansions than k: the reference reads past the end of full_retset here
                w.outI[qi * w.k + r] = -1;
                w.outD[qi * w.k + r] = FLT_MAX;
            } else {
                float o = bd;
                if (v.metric == VAM_MIPS) {  // :2873-2881
                    o = -o;
                    if (v.max_base_norm != 0.f) o = __fmul_rn(o, scale);
                }
                w.outI[qi * w.k + r] = (int64_t)bi;
                w.outD[qi * w.k + r] = o;
            }
        }
        if (!found) { have_last = true; last_d = FLT_MAX; last_id = 0xffffffffu; }
        else { have_last = true; last_d = bd; last_id = bi; }
    }
}

size_t search_smem(const VamanaWork& w, int warps) { return (size_t)warps * (2 * (w.L + 1) + 2 * w.beam) * 4; }

int pick_warps(const VamanaWork& w) {
    int warps = 8;
    while (warps > 1 && search_smem(w, warps) > 200 * 1024) warps >>= 1;
    return warps;
}

}  // namespace

// Queries in flight = resident warps, one query per warp.  Every in-flight query streams its own n_chunks-KB distance
// table once per expansion; with every hardware slot occupied (5 920 queries x 154-268 KB) the tables thrash the L2 and
// ncu shows 65 GB of DRAM reads for 2.6 GB of algorithmic bytes (profiles/r01e_traversal_ncu.md).  Capping the
// in-flight tables to an L2-sized budget was measured and is SLOWER (1 M points, 154-byte codes: 64 MB -> 2.5e5 q/s,
// 128 MB -> 2.8e5, no cap -> 4.9e5; profiles/r01e_vamana_l2_budget_sweep.log): the kernel is bound by the latency of
// its dependent gathers, and thousands of warps hide it better than L2 hits do, so every slot is used.  DESIGN.md
// section 7 discusses the shared-memory-table variant.
void vamana_plan(const DevVamana& v, VamanaWork& w, int num_sms) {
    int warps = pick_warps(w);
    size_t smem = search_smem(w, warps);
    if (smem > 48 * 1024)
        cudaFuncSetAttribute(vamana_search_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    int blocks = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&blocks, vamana_search_kernel, warps * 32, smem) != cudaSuccess || blocks < 1)
        blocks = 1;
    const long long slots = (long long)num_sms * blocks * warps;
    w.warps = warps;
    w.slots = (int)slots;
}

bool vamana_launch_prepare(cudaStream_t s, const DevVamana& v, const VamanaWork& w) {
    if (w.nq == 0) return true;
    vamana_prepare_kernel<<<(unsigned)w.nq, 128, 0, s>>>(v, w);
    LB2_CUDA_OK(cudaGetLastError());
    for (int64_t q0 = 0; q0 < w.nq; q0 += 65535) {  // gridDim.y limit
        VamanaWork part = w;
        part.qrot = w.qrot + q0 * v.data_dim;
        part.lut = w.lut + q0 * v.n_chunks * 256;
        const unsigned ny = (unsigned)std::min<int64_t>(65535, w.nq - q0);
        vamana_lut_kernel<<<dim3((unsigned)v.n_chunks, ny), 256, 0, s>>>(v, part);
        LB2_CUDA_OK(cudaGetLastError());
    }
    return true;
}

bool vamana_launch_search(cudaStream_t s, const DevVamana& v, const VamanaWork& w, int num_sms) {
    if (w.nq == 0) return true;
    const int warps = w.warps;
    const size_t smem = search_smem(w, warps);
    if (smem > 227 * 1024) { set_error("complexity L=%d needs %zu bytes of shared memory per query", w.L, smem); return false; }
    if (smem > 48 * 1024)
        LB2_CUDA_OK(cudaFuncSetAttribute(vamana_search_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int blocks = w.slots / warps;
    (void)num_sms;
    LB2_CUDA_OK(cudaMemsetAsync(w.next_query, 0, sizeof(int), s));
    vamana_search_kernel<<<blocks, warps * 32, smem, s>>>(v, w, warps);
    LB2_CUDA_OK(cudaGetLastError());
    return true;
}

bool vamana_launch_collect(cudaStream_t s, const DevVamana& v, const VamanaWork& w) {
    const int64_t n = w.nq * w.cap_full;
    if (n == 0) return true;
    vamana_collect_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(v, w);
    LB2_CUDA_OK(cudaGetLastError());
    return true;
}

bool vamana_launch_rerank(cudaStream_t s, const DevVamana& v, const VamanaWork& w) {
    if (w.nq == 0) return true;
    vamana_rerank_kernel<<<(unsigned)((w.nq * 32 + 127) / 128), 128, 0, s>>>(v, w);
    LB2_CUDA_OK(cudaGetLastError());
    return true;
}

}  // namespace lb2
