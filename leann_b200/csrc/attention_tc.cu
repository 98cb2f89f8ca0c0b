// Recompute stage, self-attention on the 5th-generation tensor cores (head_dim 32, sequences <= 256 tokens:
// all-MiniLM-L6-v2).  softmax(Q K^T / sqrt(hd)) V per (passage, head), no padding keys — the arithmetic of
// BertSelfAttention inside SentenceTransformer.encode (leann-core/src/leann/embedding_compute.py:161, 231-239).
//
// One work item = (passage s, block of 128 query rows, head h).  Persistent CTAs, two per SM (256 TMEM columns
// each), 192 threads:
//   warp 4 lane 0 : TMA producer.  The head-major QKV activation [heads][tokens][q(32) | k(32) | v(32)] is read
//                   through two 3-D tensor maps: rows of (q | k) = 128 B into a SWIZZLE_128B tile (one load serves
//                   both MMA operands of S), rows of v = 64 B into a SWIZZLE_64B tile; 64-row boxes, 2-stage ring.
//   warp 5 lane 0 : MMA issuer.   S[128, Lp] = Q . K^T : two tcgen05.mma (K = 16 each), A = the query rows of the
//                   (q | k) tile, B = its key half (descriptor start + 64 B), both K-major SW128; N = Lp = L
//                   rounded up to 16 (<= 256).  Then O[128, 32] = P . V : Lp / 16 tcgen05.mma with A = P read from
//                   TENSOR MEMORY and B = the v tile as an MN-major operand (rows = keys, no transpose needed).
//   warps 0..3    : softmax, one thread per query row (tcgen05.ld 32x32b: TMEM lane = row, no shuffles): pass 1
//                   row maximum, pass 2 p = 2^((s - m) * scale * log2 e), row sum, fp16 P written back to TMEM
//                   IN PLACE over the columns of S already consumed (tcgen05.st), zeros for keys >= L.  After the
//                   P.V MMAs: O from TMEM -> * 1/sum -> fp16 -> ctx[token][h * 32 ..] (64 B per row).
// TMEM columns of a CTA: S = [0, Lp) fp32, P = [0, Lp / 2) packed fp16 (aliases S), two O accumulators [192, 224) and
// [224, 256) (alias the top S columns of passages longer than 192 keys only).  Barriers: full/empty (smem ring), s_ready,
// p_ready, o_ready[2], o_free[2].
// Bound: the softmax (MUFU ex2 + issue slots), not the tensor pipe — 4.L.h flops per token are 5 % of the layer.
#include <cuda_fp16.h>

#include "common.cuh"
#include "ptx.cuh"

namespace lb2 {

namespace {

constexpr int ATC_HD = 32;
constexpr int ATC_TM = 128;    // query rows per item
constexpr int ATC_MAXL = 256;  // keys per passage (TMEM columns of S)
constexpr int ATC_BOX = 64;    // rows per TMA box
constexpr int ATC_THREADS = 192;     // 4 softmax warps + TMA + MMA
constexpr int ATC_QK_BYTES = ATC_MAXL * 128;
constexpr int ATC_V_BYTES = ATC_MAXL * 64;
constexpr int ATC_STAGE_BYTES = ATC_QK_BYTES + ATC_V_BYTES;
constexpr int ATC_STAGES = 2;
constexpr int ATC_BAR_OFFSET = ATC_STAGES * ATC_STAGE_BYTES;
constexpr int ATC_SMEM = ATC_BAR_OFFSET + 256 + 1024;
constexpr int ATC_TMEM_COLS = 256;
constexpr int ATC_O_COL0 = 192;  // two O accumulators of 32 columns at the top of the allocation
constexpr int ATC_LONG = 192;    // an item whose S needs more columns than this overlaps them ("long" item)

__device__ __forceinline__ float ex2f(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ uint32_t pack2(float a, float b) {
    const __half2 h = __floats2half2_rn(a, b);
    return *reinterpret_cast<const uint32_t*>(&h);
}

// work list: one descriptor per (passage, 128-row query block): {first packed row of the passage, length, first query row
// q0, passage}.  One 16-byte load per work item in the kernel (no dependent items -> seq_len -> seq_start chain); a passage's
// blocks are adjacent.  The item's 128 MMA rows are the passage's rows [q0, q0 + 128); rows in [q0, L) are its output.
// First block: q0 = 0.  Second block (rows 128 .. L-1, usually only one or two warps' worth): q0 = 128, so a tail always
// sits in row quarter 0.  Spreading tails over the row quarters evens out the MUFU load of the SM sub-partitions but leaves
// the time unchanged (profiles/r02e_attention_rotation_ab.log): the kernel is bound by the per-item chain S -> softmax ->
// P.V of a CTA (a tail item costs a full item whatever its warps do), not by MUFU throughput per sub-partition.
__global__ void attention_tc_items_kernel(const int32_t* __restrict__ seq_start, const int32_t* __restrict__ seq_len, int n_seq,
                                          int row_base, int4* __restrict__ desc, int* __restrict__ count) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n_seq) return;
    const int L = seq_len[s];
    const int nb = (L + ATC_TM - 1) / ATC_TM;
    const int base = atomicAdd(count, nb);
    desc[base] = make_int4(seq_start[s] - row_base, L, 0, s);
    if (nb > 1) desc[base + 1] = make_int4(seq_start[s] - row_base, L, ATC_TM, s);
}

// Pipeline of one CTA over its items i = 0, 1, ... (two CTAs per SM interleave):
//   MMA warp     : S(0) | for i: wait P(i) -> P.V(i) into O[i & 1] -> S(i + 1) right behind it (the tensor pipe runs the
//                  MMAs in issue order, so S(i + 1) may overwrite the columns of P(i) without a barrier)
//   softmax warps: for i: wait S(i) -> softmax -> P(i) | read O(i - 1) out while P.V(i) and S(i + 1) execute
// so the chain per item is softmax -> P.V + S, and the O read-out, the TMA loads and the other CTA's softmax fill the gaps.
// A long item (S wider than 192 columns) would overwrite the O accumulators: both sides drain the pending read-outs first.
__global__ void __launch_bounds__(ATC_THREADS, 2)
attention_tc_kernel(const __grid_constant__ CUtensorMap tmap_qk, const __grid_constant__ CUtensorMap tmap_v,
                    const int4* __restrict__ desc, const int* __restrict__ n_items, int heads, int hidden,
                    __half* __restrict__ ctx) {
    extern __shared__ uint8_t att_smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(att_smem_raw) + 1023) & ~uintptr_t(1023));
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + ATC_BAR_OFFSET);
    uint64_t* empty_bar = full_bar + ATC_STAGES;
    uint64_t* s_ready = empty_bar + ATC_STAGES;
    uint64_t* p_ready = s_ready + 1;
    uint64_t* o_ready = p_ready + 1;  // [2]
    uint64_t* o_free = o_ready + 2;   // [2]
    uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(o_free + 2);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int total = *n_items * heads;
    const int n_it = total > static_cast<int>(blockIdx.x) ? (total - static_cast<int>(blockIdx.x) + static_cast<int>(gridDim.x) - 1) / static_cast<int>(gridDim.x) : 0;

    if (warp == 4 && lane == 0) {
        ptx::prefetch_tmap(&tmap_qk);
        ptx::prefetch_tmap(&tmap_v);
        for (int i = 0; i < ATC_STAGES; i++) {
            ptx::mbar_init(&full_bar[i], 1);
            ptx::mbar_init(&empty_bar[i], 1);
        }
        ptx::mbar_init(s_ready, 1);
        ptx::mbar_init(p_ready, 4);
        for (int i = 0; i < 2; i++) {
            ptx::mbar_init(&o_ready[i], 1);
            ptx::mbar_init(&o_free[i], 4);
        }
        ptx::fence_barrier_init();
    }
    if (warp == 5) {
        ptx::tmem_alloc(tmem_ptr, ATC_TMEM_COLS);
        ptx::tmem_relinquish();
    }
    ptx::tc_fence_before();
    __syncthreads();
    ptx::tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr;

    if (warp == 4) {
        // ===== TMA producer, whole warp + one elected issuer (the descriptor of the next item is fetched while this one's
        // loads are issued)
        int4 cur = n_it > 0 ? __ldg(&desc[blockIdx.x / heads]) : make_int4(0, 0, 0, 0);
        for (int it = 0; it < n_it; it++) {
            const int w = blockIdx.x + it * gridDim.x;
            const int4 nxt = it + 1 < n_it ? __ldg(&desc[(w + gridDim.x) / heads]) : cur;
            const int stage = it & 1;
            const uint32_t ph = (it >> 1) & 1;
            const int h = w % heads;
            const int L = cur.y;
            const int row0 = cur.x;
            const int nbox = (L + ATC_BOX - 1) / ATC_BOX;
            ptx::mbar_wait(&empty_bar[stage], ph ^ 1);
            uint8_t* qk = smem + stage * ATC_STAGE_BYTES;
            uint8_t* v = qk + ATC_QK_BYTES;
            if (ptx::elect_one()) {
                ptx::mbar_expect_tx(&full_bar[stage], nbox * ATC_BOX * (128 + 64));
                for (int b = 0; b < nbox; b++) {
                    ptx::tma_load_3d(qk + b * ATC_BOX * 128, &tmap_qk, &full_bar[stage], 0, row0 + b * ATC_BOX, h);
                    ptx::tma_load_3d(v + b * ATC_BOX * 64, &tmap_v, &full_bar[stage], 2 * ATC_HD, row0 + b * ATC_BOX, h);
                }
            }
            __syncwarp();
            cur = nxt;
        }
    } else if (warp == 5) {
        if (n_it > 0) {
            // ===== MMA issuer: the whole warp runs the loop, one elected lane issues (warp-uniform control flow keeps the
            // descriptors in uniform registers; under `if (lane == 0)` every tcgen05.mma sat in an ELECT / R2UR.BROADCAST
            // loop and the ten small MMAs of an item cost more to issue than to execute)
            auto issue_s = [&](int it, const int4& d) {
                const int Lp = (d.y + 15) & ~15;
                const uint32_t qk = ptx::smem_u32(smem + (it & 1) * ATC_STAGE_BYTES);
                const uint64_t a_desc = ptx::make_sw128_kmajor_desc(qk + d.z * 128);  // first query row q0 (0 or 128)
                const uint64_t b_desc = ptx::make_sw128_kmajor_desc(qk) + 4;  // the k half of the (q | k) rows: +64 B
                const uint32_t idesc_s = ptx::make_idesc_f16(ATC_TM, Lp);
                if (ptx::elect_one()) {
#pragma unroll
                    for (int k = 0; k < ATC_HD / 16; k++)
                        ptx::umma_f16(tmem_base, a_desc + 2 * k, b_desc + 2 * k, idesc_s, k != 0);
                    ptx::umma_commit(s_ready);
                }
                __syncwarp();
            };
            int4 cur = __ldg(&desc[blockIdx.x / heads]);
            int4 nxt = n_it > 1 ? __ldg(&desc[(blockIdx.x + gridDim.x) / heads]) : cur;
            ptx::mbar_wait(&full_bar[0], 0);
            ptx::tc_fence_after();
            issue_s(0, cur);
            for (int it = 0; it < n_it; it++) {
                const int stage = it & 1, b = it & 1;
                const int Lp = (cur.y + 15) & ~15;
                const int4 nn = it + 2 < n_it ? __ldg(&desc[(blockIdx.x + (it + 2) * gridDim.x) / heads]) : nxt;
                ptx::mbar_wait(p_ready, it & 1);
                ptx::mbar_wait(&o_free[b], ((it >> 1) & 1) ^ 1);  // the previous user of this O accumulator has been read out
                ptx::tc_fence_after();
                const uint32_t vb = ptx::smem_u32(smem + stage * ATC_STAGE_BYTES) + ATC_QK_BYTES;
                const uint32_t idesc_o = ptx::make_idesc_f16(ATC_TM, ATC_HD) | ptx::IDESC_B_MN_MAJOR;
                const uint32_t o_tmem = tmem_base + ATC_O_COL0 + 32 * b;
                if (ptx::elect_one()) {
                    for (int j = 0; j < Lp / 16; j++)  // 16 keys per MMA: 8 TMEM columns of P, 16 rows (1 KB) of V
                        ptx::umma_f16_ts(o_tmem, tmem_base + 8 * j, ptx::make_mn_major_desc(vb + j * 1024, 64), idesc_o, j != 0);
                    ptx::umma_commit(&o_ready[b]);
                    ptx::umma_commit(&empty_bar[stage]);
                }
                __syncwarp();
                if (it + 1 < n_it) {
                    ptx::mbar_wait(&full_bar[(it + 1) & 1], ((it + 1) >> 1) & 1);
                    if (((nxt.y + 15) & ~15) > ATC_LONG) {  // S(it + 1) covers the O accumulators: O(it) and O(it - 1) must be out
                        ptx::mbar_wait(&o_free[b], (it >> 1) & 1);
                        if (it >= 1) ptx::mbar_wait(&o_free[b ^ 1], ((it - 1) >> 1) & 1);
                    }
                    ptx::tc_fence_after();
                    issue_s(it + 1, nxt);
                }
                cur = nxt;
                nxt = nn;
            }
        }
    } else {
        // ===== softmax + output: thread = query row
        const float scale_log2 = rsqrtf(static_cast<float>(ATC_HD)) * 1.4426950408889634f;
        const uint32_t taddr = tmem_base + (static_cast<uint32_t>(warp * 32) << 16);
        float inv_sum[2] = {0.f, 0.f};
        long long out_off[2] = {-1, -1};  // element offset of this thread's output row, -1 = row beyond the passage
        int pend = 0;                     // first item whose O has not been read out yet

        auto readout = [&](int j) {
            const int b = j & 1;
            uint32_t o[32];
            ptx::mbar_wait(&o_ready[b], (j >> 1) & 1);
            ptx::tc_fence_after();
            ptx::tmem_ld_32x32(taddr + ATC_O_COL0 + 32 * b, o);
            ptx::tmem_ld_wait();
            ptx::tc_fence_before();
            __syncwarp();
            if (lane == 0) ptx::mbar_arrive(&o_free[b]);
            const long long off = b ? out_off[1] : out_off[0];
            if (off >= 0) {
                const float inv = b ? inv_sum[1] : inv_sum[0];
                uint4* dst = reinterpret_cast<uint4*>(ctx + off);
#pragma unroll
                for (int v4 = 0; v4 < 4; v4++) {
                    uint4 ov;
                    ov.x = pack2(__uint_as_float(o[8 * v4 + 0]) * inv, __uint_as_float(o[8 * v4 + 1]) * inv);
                    ov.y = pack2(__uint_as_float(o[8 * v4 + 2]) * inv, __uint_as_float(o[8 * v4 + 3]) * inv);
                    ov.z = pack2(__uint_as_float(o[8 * v4 + 4]) * inv, __uint_as_float(o[8 * v4 + 5]) * inv);
                    ov.w = pack2(__uint_as_float(o[8 * v4 + 6]) * inv, __uint_as_float(o[8 * v4 + 7]) * inv);
                    dst[v4] = ov;
                }
            }
        };

        int4 cur = n_it > 0 ? __ldg(&desc[blockIdx.x / heads]) : make_int4(0, 0, 0, 0);
        for (int it = 0; it < n_it; it++) {
            const int w = blockIdx.x + it * gridDim.x;
            const int4 nxt = it + 1 < n_it ? __ldg(&desc[(w + gridDim.x) / heads]) : cur;  // in flight during this item's softmax
            const int h = w % heads;
            const int q0 = cur.z;
            const int L = cur.y;
            const int q = q0 + threadIdx.x;
            // a warp whose 32 query rows all lie beyond the passage (short passages; the second query block) runs zero key
            // chunks: no exponentials, no P rows (its O rows are never stored) — only the barrier protocol
            const int nch = q0 + warp * 32 >= L ? 0 : (L + 31) >> 5;
            if (((L + 15) & ~15) > ATC_LONG)  // the MMA warp waits for these before it may issue S(it)
                while (pend < it) readout(pend++);
            ptx::mbar_wait(s_ready, it & 1);
            ptx::tc_fence_after();
            uint32_t ra[32], rb[32];
            // pass 1: row maximum over the L valid keys (TMEM loads one chunk ahead of the arithmetic)
            float m = -INFINITY;
            auto max_chunk = [&](int c, const uint32_t (&r)[32]) {
                if (c * 32 + 32 <= L) {
#pragma unroll
                    for (int j = 0; j < 32; j++) m = fmaxf(m, __uint_as_float(r[j]));
                } else {
#pragma unroll
                    for (int j = 0; j < 32; j++) m = (c * 32 + j < L) ? fmaxf(m, __uint_as_float(r[j])) : m;
                }
            };
            if (nch > 0) ptx::tmem_ld_32x32(taddr, ra);
            for (int c = 0; c < nch; c += 2) {
                ptx::tmem_ld_wait();
                if (c + 1 < nch) ptx::tmem_ld_32x32(taddr + (c + 1) * 32, rb);
                max_chunk(c, ra);
                if (c + 1 < nch) {
                    ptx::tmem_ld_wait();
                    if (c + 2 < nch) ptx::tmem_ld_32x32(taddr + (c + 2) * 32, ra);
                    max_chunk(c + 1, rb);
                }
            }
            // pass 2: probabilities (fp16, back into TMEM over the consumed S columns), row sum
            const float ms = m * scale_log2;
            float sum = 0.f;
            auto exp_chunk = [&](int c, const uint32_t (&r)[32]) {
                uint32_t pk[16];
                if (c * 32 + 32 <= L) {
#pragma unroll
                    for (int j = 0; j < 16; j++) {
                        const float p0 = ex2f(fmaf(__uint_as_float(r[2 * j]), scale_log2, -ms));
                        const float p1 = ex2f(fmaf(__uint_as_float(r[2 * j + 1]), scale_log2, -ms));
                        sum += p0 + p1;
                        pk[j] = pack2(p0, p1);
                    }
                } else {
#pragma unroll
                    for (int j = 0; j < 16; j++) {
                        float p0 = ex2f(fmaf(__uint_as_float(r[2 * j]), scale_log2, -ms));
                        float p1 = ex2f(fmaf(__uint_as_float(r[2 * j + 1]), scale_log2, -ms));
                        p0 = (c * 32 + 2 * j < L) ? p0 : 0.f;
                        p1 = (c * 32 + 2 * j + 1 < L) ? p1 : 0.f;
                        sum += p0 + p1;
                        pk[j] = pack2(p0, p1);
                    }
                }
                ptx::tmem_st_32x16(taddr + c * 16, pk);
            };
            if (nch > 0) ptx::tmem_ld_32x32(taddr, ra);
            for (int c = 0; c < nch; c += 2) {
                ptx::tmem_ld_wait();
                if (c + 1 < nch) ptx::tmem_ld_32x32(taddr + (c + 1) * 32, rb);
                exp_chunk(c, ra);
                if (c + 1 < nch) {
                    ptx::tmem_ld_wait();
                    if (c + 2 < nch) ptx::tmem_ld_32x32(taddr + (c + 2) * 32, ra);
                    exp_chunk(c + 1, rb);
                }
            }
            ptx::tmem_st_wait();
            ptx::tc_fence_before();
            __syncwarp();
            if (lane == 0) ptx::mbar_arrive(p_ready);
            const float inv = 1.0f / sum;
            const long long off = q < L ? static_cast<long long>(cur.x + q) * hidden + h * ATC_HD : -1;
            if (it & 1) { inv_sum[1] = inv; out_off[1] = off; } else { inv_sum[0] = inv; out_off[0] = off; }
            while (pend < it) readout(pend++);  // O(it - 1): its P.V was issued long ago; runs while P.V(it) and S(it + 1) execute
            cur = nxt;
        }
        while (pend < n_it) readout(pend++);
    }

    ptx::tc_fence_before();
    __syncthreads();
    if (warp == 5) {
        ptx::tc_fence_after();
        ptx::tmem_dealloc(tmem_base, ATC_TMEM_COLS);
    }
}

}  // namespace

bool attention_tc_supported(int hidden, int heads, int max_pos) { return hidden / heads == ATC_HD && max_pos <= ATC_MAXL; }

// qkv: head-major [heads][n_tokens][3 * 32] fp16; items: [n_seq * 2] work list + 1 counter behind it
bool launch_attention_tc(cudaStream_t s, const __half* qkv, const int32_t* seq_start, const int32_t* seq_len, int* items,
                         int* item_count, int row_base, int n_seq, int n_tokens, int hidden, int heads, __half* ctx,
                         bool build_items, int num_sms) {
    if (n_seq <= 0) return true;
    int4* desc = reinterpret_cast<int4*>(items);  // 2 descriptors per passage at most: fits the [n_seq * 8] int work-list buffer
    if (build_items) {  // once per encoder pass: the list is the same for every layer
        LB2_CUDA_OK(cudaMemsetAsync(item_count, 0, sizeof(int), s));
        attention_tc_items_kernel<<<(n_seq + 255) / 256, 256, 0, s>>>(seq_start, seq_len, n_seq, row_base, desc, item_count);
        LB2_CUDA_OK(cudaGetLastError());
    }
    CUtensorMap tm_qk, tm_v;
    if (!make_tmap_f16_3d(&tm_qk, qkv, 3 * ATC_HD, n_tokens, heads, 2 * ATC_HD, ATC_BOX) ||
        !make_tmap_f16_3d(&tm_v, qkv, 3 * ATC_HD, n_tokens, heads, ATC_HD, ATC_BOX))
        return false;
    static thread_local int attr_dev_mask[8] = {0};
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= 256 || !(attr_dev_mask[dev >> 5] & (1 << (dev & 31)))) {
        LB2_CUDA_OK(cudaFuncSetAttribute(attention_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, ATC_SMEM));
        if (dev >= 0 && dev < 256) attr_dev_mask[dev >> 5] |= 1 << (dev & 31);
    }
    // Four softmax warps: eight (two per row quarter) measured 3-8 % slower (profiles/r02c_attention_variants.log) — the item
    // time is set by the MUFU work of the two co-resident CTAs plus the softmax -> P.V -> S chain, not by latency hiding.
    attention_tc_kernel<<<2 * num_sms, ATC_THREADS, ATC_SMEM, s>>>(tm_qk, tm_v, desc, item_count, heads, hidden, ctx);
    LB2_CUDA_OK(cudaGetLastError());
    return true;
}

}  // namespace lb2
