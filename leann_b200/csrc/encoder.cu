// Recompute stage: BERT-family sentence encoder forward over a varlen-packed batch of
// passages, i.e. what the reference's embedding server does per hop
// (leann_backend_hnsw/hnsw_embedding_server.py:147-211 -> leann/embedding_compute.py:231-239,
// explicit equivalent :319-335: last_hidden_state -> masked mean pool; the model's own
// Normalize module L2-normalises).  fp16 weights/activations like the reference
// (embedding_compute.py:157-158), fp32 accumulation, fp32 LayerNorm / softmax / pooling.
//
// No padding: sequence i owns rows [seq_start[i]-row_base, +len_i) of the packed activation
// matrix.  Dense layers run on tcgen05 (gemm_tcgen05.cu); this file holds the memory-bound
// glue kernels and the attention kernel.
#include <math.h>
#include <string.h>

#include <vector>

#include "common.cuh"

namespace lb2 {

namespace {

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

__device__ __forceinline__ int passage_len(const uint64_t* tok_off, int node, int max_pos) {
    const int len = static_cast<int>(tok_off[node + 1] - tok_off[node]);
    return len < max_pos ? len : max_pos;  // tokenizer truncation=True (embedding_compute.py:164-168)
}

// ---------------------------------------------------------------------------------------
// embeddings: word + position + token_type(0) -> LayerNorm -> fp16   (BertEmbeddings)
// one block per sequence, one warp per token, VPL = hidden/32 values per lane
// ---------------------------------------------------------------------------------------
template <int VPL>
__global__ void __launch_bounds__(256)
embed_ln_kernel(const uint16_t* __restrict__ tok_store, const uint64_t* __restrict__ tok_off,
                const int32_t* __restrict__ seq_node, const int32_t* __restrict__ seq_start, int row_base,
                int max_pos, const __half* __restrict__ word_emb, const __half* __restrict__ pos_emb,
                const __half* __restrict__ type_emb, const float* __restrict__ g, const float* __restrict__ b,
                float eps, __half* __restrict__ x, int32_t* __restrict__ seq_len_out) {
    constexpr int H = VPL * 32;
    const int s = blockIdx.x;
    const int node = seq_node[s];
    const int len = passage_len(tok_off, node, max_pos);
    if (threadIdx.x == 0) seq_len_out[s] = len;  // attention / pooling read the length from here
    const uint16_t* toks = tok_store + tok_off[node];
    const int row0 = seq_start[s] - row_base;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarp = blockDim.x >> 5;
    for (int p = warp; p < len; p += nwarp) {
        const int tok = toks[p];
        float v[VPL];
        float sum = 0.f;
#pragma unroll
        for (int i = 0; i < VPL / 4; i++) {
            const int e = (i * 32 + lane) * 4;
            const uint2 w = *reinterpret_cast<const uint2*>(word_emb + static_cast<size_t>(tok) * H + e);
            const uint2 pp = *reinterpret_cast<const uint2*>(pos_emb + static_cast<size_t>(p) * H + e);
            const uint2 tt = *reinterpret_cast<const uint2*>(type_emb + e);
            const __half2* wh = reinterpret_cast<const __half2*>(&w);
            const __half2* ph = reinterpret_cast<const __half2*>(&pp);
            const __half2* th = reinterpret_cast<const __half2*>(&tt);
#pragma unroll
            for (int j = 0; j < 2; j++) {
                const float2 a = __half22float2(wh[j]), c = __half22float2(ph[j]), d = __half22float2(th[j]);
                v[i * 4 + 2 * j] = a.x + c.x + d.x;
                v[i * 4 + 2 * j + 1] = a.y + c.y + d.y;
                sum += v[i * 4 + 2 * j] + v[i * 4 + 2 * j + 1];
            }
        }
        const float mean = warp_sum(sum) * (1.0f / H);
        float sq = 0.f;
#pragma unroll
        for (int i = 0; i < VPL; i++) { const float d = v[i] - mean; sq += d * d; }
        const float rstd = rsqrtf(warp_sum(sq) * (1.0f / H) + eps);
        __half* out = x + static_cast<size_t>(row0 + p) * H;
#pragma unroll
        for (int i = 0; i < VPL / 4; i++) {
            const int e = (i * 32 + lane) * 4;
            const float4 gg = *reinterpret_cast<const float4*>(g + e);
            const float4 bb = *reinterpret_cast<const float4*>(b + e);
            uint2 o;
            __half2* oh = reinterpret_cast<__half2*>(&o);
            oh[0] = __floats2half2_rn((v[i * 4] - mean) * rstd * gg.x + bb.x, (v[i * 4 + 1] - mean) * rstd * gg.y + bb.y);
            oh[1] = __floats2half2_rn((v[i * 4 + 2] - mean) * rstd * gg.z + bb.z, (v[i * 4 + 3] - mean) * rstd * gg.w + bb.w);
            *reinterpret_cast<uint2*>(out + e) = o;
        }
    }
}

// ---------------------------------------------------------------------------------------
// LayerNorm over rows of a fp16 matrix (input already holds dense+bias+residual), one warp per row
// ---------------------------------------------------------------------------------------
template <int VPL>
__global__ void __launch_bounds__(256)
layernorm_kernel(const __half* __restrict__ in, const float* __restrict__ g, const float* __restrict__ b,
                 __half* __restrict__ out, int rows, float eps) {
    constexpr int H = VPL * 32;
    const int lane = threadIdx.x & 31;
    const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (row >= rows) return;
    const __half* ip = in + static_cast<size_t>(row) * H;
    float v[VPL];
    float sum = 0.f;
#pragma unroll
    for (int i = 0; i < VPL / 4; i++) {
        const int e = (i * 32 + lane) * 4;
        const uint2 w = *reinterpret_cast<const uint2*>(ip + e);
        const __half2* wh = reinterpret_cast<const __half2*>(&w);
        const float2 a = __half22float2(wh[0]), c = __half22float2(wh[1]);
        v[i * 4] = a.x; v[i * 4 + 1] = a.y; v[i * 4 + 2] = c.x; v[i * 4 + 3] = c.y;
        sum += a.x + a.y + c.x + c.y;
    }
    const float mean = warp_sum(sum) * (1.0f / H);
    float sq = 0.f;
#pragma unroll
    for (int i = 0; i < VPL; i++) { const float d = v[i] - mean; sq += d * d; }
    const float rstd = rsqrtf(warp_sum(sq) * (1.0f / H) + eps);
    __half* op = out + static_cast<size_t>(row) * H;
#pragma unroll
    for (int i = 0; i < VPL / 4; i++) {
        const int e = (i * 32 + lane) * 4;
        const float4 gg = *reinterpret_cast<const float4*>(g + e);
        const float4 bb = *reinterpret_cast<const float4*>(b + e);
        uint2 o;
        __half2* oh = reinterpret_cast<__half2*>(&o);
        oh[0] = __floats2half2_rn((v[i * 4] - mean) * rstd * gg.x + bb.x, (v[i * 4 + 1] - mean) * rstd * gg.y + bb.y);
        oh[1] = __floats2half2_rn((v[i * 4 + 2] - mean) * rstd * gg.z + bb.z, (v[i * 4 + 3] - mean) * rstd * gg.w + bb.w);
        *reinterpret_cast<uint2*>(op + e) = o;
    }
}

// ---------------------------------------------------------------------------------------
// Self-attention, one CTA per (sequence, head): softmax(Q K^T / sqrt(hd)) V, no padding keys.
// K and V of the head are staged once in shared memory (row-major, 16-byte copies); each warp owns
// 16-query tiles and walks the keys in blocks of 64 with an online softmax (fp32 statistics,
// ex2.approx), mma.sync m16n8k16 with ldmatrix / ldmatrix.trans operand fragments.
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ void mma_16816(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    asm volatile(
        "mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
        : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ uint32_t pack_h2(float a, float b) {
    const __half2 h = __floats2half2_rn(a, b);
    return *reinterpret_cast<const uint32_t*>(&h);
}

__device__ __forceinline__ void ldsm_x4(uint32_t (&r)[4], const void* smem_ptr) {
    const uint32_t a = static_cast<uint32_t>(__cvta_generic_to_shared(smem_ptr));
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(a));
}
__device__ __forceinline__ void ldsm_x4_trans(uint32_t (&r)[4], const void* smem_ptr) {
    const uint32_t a = static_cast<uint32_t>(__cvta_generic_to_shared(smem_ptr));
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(a));
}
__device__ __forceinline__ float fast_exp2(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc, int src_bytes) {
    const uint32_t d = static_cast<uint32_t>(__cvta_generic_to_shared(smem_dst));
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(d), "l"(gsrc), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// One CTA = (sequence, head, block of 64 query rows); 4 warps x 16 rows.  Keys/values stream through a
// double-buffered 64-key smem ring filled with cp.async (zero-fill past L), so the CTA's footprint is
// 20 KB whatever the sequence length and several CTAs per SM overlap each other's load latency.
// Input is HEAD-MAJOR: qkv[head][token][q(hd) | k(hd) | v(hd)], written that way by the QKV GEMM's
// grouped TMA store, so one (sequence, head) is a single contiguous run of L * 3hd halves: every DRAM
// line fetched is fully used (the token-major layout cost 2.7x the algorithmic DRAM reads, ncu).
// blockIdx.x walks a work list of (passage, query block) items in which a passage's blocks are adjacent, so
// the CTAs sharing a (sequence, head)'s keys are launched back to back; no CTA is launched for nothing.
// work list of the attention kernel for one encoder pass: one item per (passage, 64-row query block)
__global__ void attention_items_kernel(const int32_t* __restrict__ seq_len, int n_seq, int* __restrict__ items,
                                       int* __restrict__ count) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n_seq) return;
    const int nb = (seq_len[s] + 63) >> 6;
    const int base = atomicAdd(count, nb);
    for (int i = 0; i < nb; i++) items[base + i] = s * 8 + i;  // a passage's blocks stay adjacent: they share K/V in L2
}

template <int HD>
__global__ void __launch_bounds__(128, HD == 32 ? 8 : 4)
attention_kernel(const __half* __restrict__ qkv, const int32_t* __restrict__ seq_start,
                 const int32_t* __restrict__ seq_len, const int* __restrict__ items, const int* __restrict__ n_items,
                 int row_base, int n_tokens, int hidden, __half* __restrict__ ctx) {
    constexpr int P = HD + 8;  // row pitch in halves: 16-byte aligned rows, conflict-free ldmatrix
    __shared__ __align__(16) __half Ks[2][64 * P];
    __shared__ __align__(16) __half Vs[2][64 * P];
    if (static_cast<int>(blockIdx.x) >= *n_items) return;  // the grid is sized from a host-side upper bound
    const int item = items[blockIdx.x];
    const int s = item >> 3, h = blockIdx.y;
    const int L = seq_len[s];
    const int qblk0 = (item & 7) * 64;
    const int row0 = seq_start[s] - row_base;
    constexpr int ld = 3 * HD;
    const __half* qbase = qkv + (static_cast<size_t>(h) * n_tokens + row0) * ld;
    const __half* kbase = qbase + HD;
    const __half* vbase = qbase + 2 * HD;
    const int nkb = (L + 63) >> 6;

    auto prefetch = [&](int kb, int buf) {
        for (int idx = threadIdx.x; idx < 64 * (HD / 8); idx += 128) {
            const int kl = idx / (HD / 8), c8 = (idx % (HD / 8)) * 8;
            const int key = kb * 64 + kl;
            const int ok = key < L ? 16 : 0;           // src-size 0 -> the 16 bytes are zero-filled
            const size_t roff = static_cast<size_t>(key < L ? key : L - 1) * ld + c8;
            cp_async16(&Ks[buf][kl * P + c8], kbase + roff, ok);
            cp_async16(&Vs[buf][kl * P + c8], vbase + roff, ok);
        }
        cp_async_commit();
    };
    prefetch(0, 0);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int g = lane >> 2, t = lane & 3;
    const float scale_log2 = rsqrtf(static_cast<float>(HD)) * 1.4426950408889634f;
    const int lm_row = lane & 7, lm_mat = lane >> 3;
    const int q0 = qblk0 + warp * 16;
    const bool active = q0 < L;  // warp-uniform
    const int r0 = q0 + g, r1 = q0 + g + 8;

    // Q fragments (A operand) straight from global (64 B per row), in flight together with key block 0
    uint32_t qa[HD / 16][4];
#pragma unroll
    for (int ks = 0; ks < HD / 16; ks++) {
        const int c = ks * 16 + 2 * t;
        qa[ks][0] = (active && r0 < L) ? __ldg(reinterpret_cast<const uint32_t*>(qbase + static_cast<size_t>(r0) * ld + c)) : 0u;
        qa[ks][1] = (active && r1 < L) ? __ldg(reinterpret_cast<const uint32_t*>(qbase + static_cast<size_t>(r1) * ld + c)) : 0u;
        qa[ks][2] = (active && r0 < L) ? __ldg(reinterpret_cast<const uint32_t*>(qbase + static_cast<size_t>(r0) * ld + c + 8)) : 0u;
        qa[ks][3] = (active && r1 < L) ? __ldg(reinterpret_cast<const uint32_t*>(qbase + static_cast<size_t>(r1) * ld + c + 8)) : 0u;
    }
    float o[HD / 8][4];
#pragma unroll
    for (int i = 0; i < HD / 8; i++) { o[i][0] = o[i][1] = o[i][2] = o[i][3] = 0.f; }
    float m0 = -INFINITY, m1 = -INFINITY, l0 = 0.f, l1 = 0.f;

    for (int kb = 0; kb < nkb; kb++) {
        const int buf = kb & 1;
        if (kb + 1 < nkb) { prefetch(kb + 1, buf ^ 1); cp_async_wait<1>(); } else { cp_async_wait<0>(); }
        __syncthreads();
        if (active) {
            const __half* Kb = Ks[buf];
            const __half* Vb = Vs[buf];
#pragma unroll
            for (int hb = 0; hb < 2; hb++) {  // two halves of 32 keys keep the register footprint small
                const int key0 = kb * 64 + hb * 32;
                if (key0 >= L) break;  // wholly padded half (warp-uniform)
                float sc[4][4];
#pragma unroll
                for (int nt = 0; nt < 4; nt++) {
                    sc[nt][0] = sc[nt][1] = sc[nt][2] = sc[nt][3] = 0.f;
#pragma unroll
                    for (int kp = 0; kp < HD / 32; kp++) {
                        uint32_t b[4];
                        ldsm_x4(b, Kb + (hb * 32 + nt * 8 + lm_row) * P + kp * 32 + lm_mat * 8);
                        mma_16816(sc[nt], qa[2 * kp], b[0], b[1]);
                        mma_16816(sc[nt], qa[2 * kp + 1], b[2], b[3]);
                    }
                }
                float bm0 = -INFINITY, bm1 = -INFINITY;
#pragma unroll
                for (int nt = 0; nt < 4; nt++) {
                    const int key = key0 + nt * 8 + 2 * t;
                    if (key >= L) { sc[nt][0] = -INFINITY; sc[nt][2] = -INFINITY; }
                    if (key + 1 >= L) { sc[nt][1] = -INFINITY; sc[nt][3] = -INFINITY; }
                    bm0 = fmaxf(bm0, fmaxf(sc[nt][0], sc[nt][1]));
                    bm1 = fmaxf(bm1, fmaxf(sc[nt][2], sc[nt][3]));
                }
                bm0 = fmaxf(bm0, __shfl_xor_sync(0xffffffffu, bm0, 1));
                bm0 = fmaxf(bm0, __shfl_xor_sync(0xffffffffu, bm0, 2));
                bm1 = fmaxf(bm1, __shfl_xor_sync(0xffffffffu, bm1, 1));
                bm1 = fmaxf(bm1, __shfl_xor_sync(0xffffffffu, bm1, 2));
                const float nm0 = fmaxf(m0, bm0), nm1 = fmaxf(m1, bm1);  // finite: key0 < L is a valid key
                const float corr0 = fast_exp2((m0 - nm0) * scale_log2), corr1 = fast_exp2((m1 - nm1) * scale_log2);
                m0 = nm0; m1 = nm1;
                const float ms0 = m0 * scale_log2, ms1 = m1 * scale_log2;
                float rs0 = 0.f, rs1 = 0.f;
                uint32_t pa[2][4];
#pragma unroll
                for (int nt = 0; nt < 4; nt++) {
                    const float p0 = fast_exp2(fmaf(sc[nt][0], scale_log2, -ms0)), p1 = fast_exp2(fmaf(sc[nt][1], scale_log2, -ms0));
                    const float p2 = fast_exp2(fmaf(sc[nt][2], scale_log2, -ms1)), p3 = fast_exp2(fmaf(sc[nt][3], scale_log2, -ms1));
                    rs0 += p0 + p1; rs1 += p2 + p3;
                    const int kk = nt >> 1;
                    if ((nt & 1) == 0) { pa[kk][0] = pack_h2(p0, p1); pa[kk][1] = pack_h2(p2, p3); }
                    else               { pa[kk][2] = pack_h2(p0, p1); pa[kk][3] = pack_h2(p2, p3); }
                }
                l0 = l0 * corr0 + rs0; l1 = l1 * corr1 + rs1;
#pragma unroll
                for (int dt = 0; dt < HD / 8; dt++) { o[dt][0] *= corr0; o[dt][1] *= corr0; o[dt][2] *= corr1; o[dt][3] *= corr1; }
#pragma unroll
                for (int kk = 0; kk < 2; kk++) {
#pragma unroll
                    for (int dp = 0; dp < HD / 16; dp++) {
                        uint32_t b[4];
                        ldsm_x4_trans(b, Vb + (hb * 32 + kk * 16 + (lm_mat & 1) * 8 + lm_row) * P + (2 * dp + (lm_mat >> 1)) * 8);
                        mma_16816(o[2 * dp], pa[kk], b[0], b[1]);
                        mma_16816(o[2 * dp + 1], pa[kk], b[2], b[3]);
                    }
                }
            }
        }
        __syncthreads();  // everyone is done with `buf` before the next iteration's prefetch overwrites it
    }
    if (!active) return;
    l0 += __shfl_xor_sync(0xffffffffu, l0, 1); l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
    l1 += __shfl_xor_sync(0xffffffffu, l1, 1); l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
    const float inv0 = 1.0f / l0, inv1 = 1.0f / l1;
    __half* c0 = ctx + static_cast<size_t>(row0 + r0) * hidden + h * HD + 2 * t;
    __half* c1 = ctx + static_cast<size_t>(row0 + r1) * hidden + h * HD + 2 * t;
#pragma unroll
    for (int dt = 0; dt < HD / 8; dt++) {
        if (r0 < L) *reinterpret_cast<uint32_t*>(c0 + dt * 8) = pack_h2(o[dt][0] * inv0, o[dt][1] * inv0);
        if (r1 < L) *reinterpret_cast<uint32_t*>(c1 + dt * 8) = pack_h2(o[dt][2] * inv1, o[dt][3] * inv1);
    }
}

// ---------------------------------------------------------------------------------------
// pooling (+ L2 normalisation): one CTA of 128 threads per sequence, fp32 output
// ---------------------------------------------------------------------------------------
template <int EPT>  // elements per thread = hidden / 128
__global__ void __launch_bounds__(128)
pool_kernel(const __half* __restrict__ x, const int32_t* __restrict__ seq_start,
            const int32_t* __restrict__ seq_len, int row_base, int pooling, int normalize, float* __restrict__ out) {
    constexpr int H = EPT * 128;
    __shared__ float red[4];
    const int s = blockIdx.x;
    const int L = seq_len[s];
    const __half* xp = x + static_cast<size_t>(seq_start[s] - row_base) * H;
    float acc[EPT];
#pragma unroll
    for (int i = 0; i < EPT; i++) acc[i] = 0.f;
    const int n = pooling == 1 ? 1 : L;
    for (int p = 0; p < n; p++) {
#pragma unroll
        for (int i = 0; i < EPT; i++) acc[i] += __half2float(xp[static_cast<size_t>(p) * H + i * 128 + threadIdx.x]);
    }
    const float inv = 1.0f / static_cast<float>(n > 0 ? n : 1);
    float sq = 0.f;
#pragma unroll
    for (int i = 0; i < EPT; i++) { acc[i] *= inv; sq += acc[i] * acc[i]; }
    float scale = 1.0f;
    if (normalize) {
        sq = warp_sum(sq);
        if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = sq;
        __syncthreads();
        const float tot = red[0] + red[1] + red[2] + red[3];
        scale = 1.0f / fmaxf(sqrtf(tot), 1e-12f);  // torch.nn.functional.normalize eps
    }
#pragma unroll
    for (int i = 0; i < EPT; i++) out[static_cast<size_t>(s) * H + i * 128 + threadIdx.x] = acc[i] * scale;
}

size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

}  // namespace

// ---------------------------------------------------------------------------------------
// launch wrappers
// ---------------------------------------------------------------------------------------
bool launch_embed_ln(cudaStream_t s, const Encoder* enc, const uint16_t* tok_store, const uint64_t* tok_off,
                     const int32_t* seq_node, const int32_t* seq_start, int row_base, int n_seq, __half* x,
                     int32_t* seq_len_out) {
    if (n_seq <= 0) return true;
    const EncoderConfig& c = enc->cfg;
    if (c.hidden == 384)
        embed_ln_kernel<12><<<n_seq, 256, 0, s>>>(tok_store, tok_off, seq_node, seq_start, row_base, c.max_pos,
                                                   enc->word_emb, enc->pos_emb, enc->type_emb, enc->emb_ln_g,
                                                   enc->emb_ln_b, c.ln_eps, x, seq_len_out);
    else
        embed_ln_kernel<24><<<n_seq, 256, 0, s>>>(tok_store, tok_off, seq_node, seq_start, row_base, c.max_pos,
                                                   enc->word_emb, enc->pos_emb, enc->type_emb, enc->emb_ln_g,
                                                   enc->emb_ln_b, c.ln_eps, x, seq_len_out);
    LB2_CUDA_OK(cudaGetLastError());
    return true;
}

bool launch_layernorm(cudaStream_t s, const __half* in, const float* g, const float* b, __half* out, int rows,
                      int hidden, float eps) {
    if (rows <= 0) return true;
    const int grid = (rows + 7) / 8;
    if (hidden == 384)
        layernorm_kernel<12><<<grid, 256, 0, s>>>(in, g, b, out, rows, eps);
    else if (hidden == 768)
        layernorm_kernel<24><<<grid, 256, 0, s>>>(in, g, b, out, rows, eps);
    else {
        set_error("layernorm: unsupported hidden %d", hidden);
        return false;
    }
    LB2_CUDA_OK(cudaGetLastError());
    return true;
}

bool launch_attention(cudaStream_t s, const __half* qkv, const int32_t* seq_start, const int32_t* seq_len, int* items,
                      int* item_count, int row_base, int max_pos, int n_seq, int n_tokens, int hidden, int heads,
                      __half* ctx, bool build_items) {
    if (n_seq <= 0) return true;
    const int hd = hidden / heads;
    if (max_pos > 512) { set_error("attention: max_pos %d > 512", max_pos); return false; }
    // head_dim 32 and passages of at most 256 tokens (all-MiniLM-L6-v2): the tcgen05 kernel (attention_tc.cu).
    // Other shapes (bge-base: head_dim 64, up to 512 tokens) keep the mma.sync kernel below.
    if (attention_tc_supported(hidden, heads, max_pos)) {
        int dev = 0, sms = 148;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        return launch_attention_tc(s, qkv, seq_start, seq_len, items, item_count, row_base, n_seq, n_tokens, hidden, heads, ctx,
                                   build_items, sms);
    }
    if (build_items) {  // once per encoder pass: the list is the same for every layer
        LB2_CUDA_OK(cudaMemsetAsync(item_count, 0, sizeof(int), s));
        attention_items_kernel<<<(n_seq + 255) / 256, 256, 0, s>>>(seq_len, n_seq, items, item_count);
        LB2_CUDA_OK(cudaGetLastError());
    }
    // sum_s ceil(L_s / 64) <= n_tokens / 64 + n_seq
    dim3 grid(n_tokens / 64 + n_seq, heads);
    if (hd == 32)
        attention_kernel<32><<<grid, 128, 0, s>>>(qkv, seq_start, seq_len, items, item_count, row_base, n_tokens, hidden, ctx);
    else if (hd == 64)
        attention_kernel<64><<<grid, 128, 0, s>>>(qkv, seq_start, seq_len, items, item_count, row_base, n_tokens, hidden, ctx);
    else {
        set_error("attention: unsupported head_dim %d", hd);
        return false;
    }
    LB2_CUDA_OK(cudaGetLastError());
    return true;
}

bool launch_pool(cudaStream_t s, const __half* x, const int32_t* seq_start, const int32_t* seq_len, int row_base,
                 int n_seq, int hidden, int pooling, int normalize, float* out) {
    if (n_seq <= 0) return true;
    if (hidden == 384)
        pool_kernel<3><<<n_seq, 128, 0, s>>>(x, seq_start, seq_len, row_base, pooling, normalize, out);
    else if (hidden == 768)
        pool_kernel<6><<<n_seq, 128, 0, s>>>(x, seq_start, seq_len, row_base, pooling, normalize, out);
    else {
        set_error("pool: unsupported hidden %d", hidden);
        return false;
    }
    LB2_CUDA_OK(cudaGetLastError());
    return true;
}

// ---------------------------------------------------------------------------------------
// weights: one fp32 host blob (layout documented in include/leann_b200.h) -> fp16/fp32 device arena
// ---------------------------------------------------------------------------------------
size_t encoder_weight_floats(const EncoderConfig& c) {
    const size_t H = c.hidden, F = c.ffn;
    size_t n = (size_t)c.vocab_size * H + (size_t)c.max_pos * H + (size_t)c.type_vocab * H + 2 * H;
    n += (size_t)c.layers * (3 * H * H + 3 * H + H * H + H + 2 * H + F * H + F + H * F + H + 2 * H);
    return n;
}

bool encoder_load(Encoder* enc, const EncoderConfig& cfg, const float* w, size_t n_floats) {
    if (cfg.hidden != 384 && cfg.hidden != 768) { set_error("encoder: hidden must be 384 or 768 (got %d)", cfg.hidden); return false; }
    if (cfg.hidden % cfg.heads != 0 || (cfg.hidden / cfg.heads != 32 && cfg.hidden / cfg.heads != 64)) {
        set_error("encoder: head_dim must be 32 or 64"); return false;
    }
    if ((3 * cfg.hidden) % gemm_block_n() || cfg.ffn % gemm_block_n() || cfg.ffn % 64) {
        set_error("encoder: hidden/ffn must be multiples of %d", gemm_block_n()); return false;
    }
    if (cfg.vocab_size > 65536) { set_error("encoder: vocab_size %d exceeds the uint16 token store", cfg.vocab_size); return false; }
    if (n_floats != encoder_weight_floats(cfg)) {
        set_error("encoder: weight blob has %zu floats, config needs %zu", n_floats, encoder_weight_floats(cfg));
        return false;
    }
    encoder_free(enc);
    enc->cfg = cfg;
    const size_t H = cfg.hidden, F = cfg.ffn, Lr = cfg.layers;
    // pass 1: sizes
    size_t h16 = (size_t)cfg.vocab_size * H + (size_t)cfg.max_pos * H + (size_t)cfg.type_vocab * H + Lr * (3 * H * H + H * H + 2 * F * H);
    size_t f32 = 2 * H + Lr * (3 * H + H + 2 * H + F + H + 2 * H);
    size_t bytes = align_up(h16 * 2, 256) + f32 * 4 + 256 * (16 * Lr + 16);
    LB2_CUDA_OK(cudaMalloc(&enc->arena, bytes));
    std::vector<__half> hbuf;
    uint8_t* cur = static_cast<uint8_t*>(enc->arena);
    const float* src = w;
    auto put16 = [&](size_t n) -> __half* {
        hbuf.resize(n);
        for (size_t i = 0; i < n; i++) hbuf[i] = __float2half_rn(src[i]);
        __half* dst = reinterpret_cast<__half*>(cur);
        if (cudaMemcpy(dst, hbuf.data(), n * 2, cudaMemcpyHostToDevice) != cudaSuccess) return nullptr;
        cur += align_up(n * 2, 256);
        src += n;
        return dst;
    };
    auto put32 = [&](size_t n) -> float* {
        float* dst = reinterpret_cast<float*>(cur);
        if (cudaMemcpy(dst, src, n * 4, cudaMemcpyHostToDevice) != cudaSuccess) return nullptr;
        cur += align_up(n * 4, 256);
        src += n;
        return dst;
    };
    bool ok = true;
    ok &= (enc->word_emb = put16((size_t)cfg.vocab_size * H)) != nullptr;
    ok &= (enc->pos_emb = put16((size_t)cfg.max_pos * H)) != nullptr;
    ok &= (enc->type_emb = put16((size_t)cfg.type_vocab * H)) != nullptr;
    ok &= (enc->emb_ln_g = put32(H)) != nullptr;
    ok &= (enc->emb_ln_b = put32(H)) != nullptr;
    enc->layers = new LayerWeights[Lr];
    for (size_t l = 0; l < Lr && ok; l++) {
        LayerWeights& lw = enc->layers[l];
        {   // rows of [Wq; Wk; Wv] regrouped per head (q_h | k_h | v_h) so that the GEMM output is head-major
            const size_t hd = H / cfg.heads;
            std::vector<float> wp(3 * H * H), bp(3 * H);
            const float* bsrc = src + 3 * H * H;
            for (size_t h = 0; h < (size_t)cfg.heads; h++)
                for (size_t part = 0; part < 3; part++)
                    for (size_t j = 0; j < hd; j++) {
                        const size_t dst_row = h * 3 * hd + part * hd + j, src_row = part * H + h * hd + j;
                        memcpy(&wp[dst_row * H], src + src_row * H, H * sizeof(float));
                        bp[dst_row] = bsrc[src_row];
                    }
            const float* keep = src;
            src = wp.data();
            ok &= (lw.w_qkv = put16(3 * H * H)) != nullptr;
            src = bp.data();
            ok &= (lw.b_qkv = put32(3 * H)) != nullptr;
            src = keep + 3 * H * H + 3 * H;
        }
        ok &= (lw.w_o = put16(H * H)) != nullptr;
        ok &= (lw.b_o = put32(H)) != nullptr;
        ok &= (lw.ln1_g = put32(H)) != nullptr;
        ok &= (lw.ln1_b = put32(H)) != nullptr;
        ok &= (lw.w_1 = put16(F * H)) != nullptr;
        ok &= (lw.b_1 = put32(F)) != nullptr;
        ok &= (lw.w_2 = put16(H * F)) != nullptr;
        ok &= (lw.b_2 = put32(H)) != nullptr;
        ok &= (lw.ln2_g = put32(H)) != nullptr;
        ok &= (lw.ln2_b = put32(H)) != nullptr;
        if (!ok) break;
        const uint32_t bn = gemm_block_n();
        ok &= make_tmap_f16_2d(&lw.tm_qkv, lw.w_qkv, 3 * H, H, bn);
        ok &= make_tmap_f16_2d(&lw.tm_o, lw.w_o, H, H, bn);
        ok &= make_tmap_f16_2d(&lw.tm_1, lw.w_1, F, H, bn);
        ok &= make_tmap_f16_2d(&lw.tm_2, lw.w_2, H, F, bn);
    }
    if (!ok) {
        if (cur > static_cast<uint8_t*>(enc->arena) + bytes) set_error("encoder: arena overflow");
        encoder_free(enc);
        return false;
    }
    if (static_cast<size_t>(cur - static_cast<uint8_t*>(enc->arena)) > bytes) {
        set_error("encoder: arena overflow");
        encoder_free(enc);
        return false;
    }
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&enc->num_sms, cudaDevAttrMultiProcessorCount, dev);
    enc->loaded = true;
    return true;
}

void encoder_free(Encoder* enc) {
    if (enc->arena) cudaFree(enc->arena);
    enc->arena = nullptr;
    delete[] enc->layers;
    enc->layers = nullptr;
    for (__half** p : {&enc->x, &enc->y, &enc->qkv, &enc->ctx, &enc->ffn}) {
        if (*p) cudaFree(*p);
        *p = nullptr;
    }
    if (enc->seq_len) cudaFree(enc->seq_len);
    enc->seq_len = nullptr;
    if (enc->att_items) cudaFree(enc->att_items);
    enc->att_items = nullptr;
    enc->cap_tokens = enc->cap_seqs = 0;
    enc->loaded = false;
}

bool encoder_reserve(Encoder* enc, int64_t tokens, int64_t seqs) {
    if (seqs > enc->cap_seqs) {
        if (enc->seq_len) cudaFree(enc->seq_len);
        enc->seq_len = nullptr;
        enc->cap_seqs = 0;
        LB2_CUDA_OK(cudaMalloc(&enc->seq_len, static_cast<size_t>(seqs) * sizeof(int32_t)));
        if (enc->att_items) cudaFree(enc->att_items);
        enc->att_items = nullptr;
        LB2_CUDA_OK(cudaMalloc(&enc->att_items, (static_cast<size_t>(seqs) * 8 + 1) * sizeof(int)));  // [seqs * 8] items + count
        enc->cap_seqs = seqs;
    }
    if (tokens <= enc->cap_tokens) return true;
    for (__half** p : {&enc->x, &enc->y, &enc->qkv, &enc->ctx, &enc->ffn}) {
        if (*p) cudaFree(*p);
        *p = nullptr;
    }
    enc->cap_tokens = 0;
    const size_t H = enc->cfg.hidden, F = enc->cfg.ffn, T = static_cast<size_t>(tokens);
    LB2_CUDA_OK(cudaMalloc(&enc->x, T * H * 2));
    LB2_CUDA_OK(cudaMalloc(&enc->y, T * H * 2));
    LB2_CUDA_OK(cudaMalloc(&enc->qkv, T * 3 * H * 2));
    LB2_CUDA_OK(cudaMalloc(&enc->ctx, T * H * 2));
    LB2_CUDA_OK(cudaMalloc(&enc->ffn, T * F * 2));
    enc->cap_tokens = tokens;
    return true;
}

// hidden = 2 GEMM n-tiles (384): the residual projections carry their LayerNorm (gemm_f16_res_ln).  Other widths (bge-base,
// 768) run the residual GEMM and the separate bandwidth-bound LayerNorm kernel.
bool encoder_fuses_ln(const EncoderConfig& cfg) { return cfg.hidden == 2 * gemm_block_n(); }

bool encoder_forward(Encoder* enc, cudaStream_t st, const uint16_t* tok_store, const uint64_t* tok_off,
                     const int32_t* seq_node, const int32_t* seq_start, int row_base, int n_seq, int n_tokens,
                     float* out) {
    if (!enc->loaded) { set_error("encoder not loaded"); return false; }
    if (n_seq <= 0 || n_tokens <= 0) return true;
    if (n_tokens > enc->cap_tokens || n_seq > enc->cap_seqs) {
        set_error("encoder_forward: %d tokens / %d passages exceed the reserved %lld / %lld", n_tokens, n_seq,
                  (long long)enc->cap_tokens, (long long)enc->cap_seqs);
        return false;
    }
    const EncoderConfig& c = enc->cfg;
    const int H = c.hidden, F = c.ffn, T = n_tokens, sms = enc->num_sms;
    if (!launch_embed_ln(st, enc, tok_store, tok_off, seq_node, seq_start, row_base, n_seq, enc->x, enc->seq_len)) return false;
    auto gemm = [&](const __half* A, const CUtensorMap* tm, const __half* W, const float* bias, const __half* res,
                    __half* C, int N, int K, int epi, int c_group = 0) {
        prof_begin(st, PROF_GEMM);
        const bool ok = gemm_f16(st, A, tm, W, bias, res, C, T, N, K, epi, sms, c_group);
        prof_end(st, PROF_GEMM, 2.0 * T * (double)N * K);
        return ok;
    };
    const bool fused_ln = encoder_fuses_ln(c);
    for (int l = 0; l < c.layers; l++) {
        const LayerWeights& w = enc->layers[l];
        if (!gemm(enc->x, &w.tm_qkv, w.w_qkv, w.b_qkv, nullptr, enc->qkv, 3 * H, H, EPI_BIAS, 3 * (H / c.heads))) return false;
        prof_begin(st, PROF_ATTN);
        if (!launch_attention(st, enc->qkv, seq_start, enc->seq_len, enc->att_items, enc->att_items + enc->cap_seqs * 8,
                              row_base, c.max_pos, n_seq, T, H, c.heads, enc->ctx, l == 0))
            return false;
        prof_end(st, PROF_ATTN, 0);
        if (fused_ln) {
            // hidden 384: Linear + residual + LayerNorm in ONE kernel (gemm_f16_ln_kernel): x -> y -> x ping-pong, the
            // pre-norm activation never touches HBM
            prof_begin(st, PROF_GEMM);
            bool ok = gemm_f16_res_ln(st, enc->ctx, &w.tm_o, w.w_o, w.b_o, enc->x, w.ln1_g, w.ln1_b, c.ln_eps, enc->y, T, H, H, sms);
            prof_end(st, PROF_GEMM, 2.0 * T * (double)H * H);
            if (!ok) return false;
            if (!gemm(enc->y, &w.tm_1, w.w_1, w.b_1, nullptr, enc->ffn, F, H, EPI_BIAS_GELU)) return false;
            prof_begin(st, PROF_GEMM);
            ok = gemm_f16_res_ln(st, enc->ffn, &w.tm_2, w.w_2, w.b_2, enc->y, w.ln2_g, w.ln2_b, c.ln_eps, enc->x, T, H, F, sms);
            prof_end(st, PROF_GEMM, 2.0 * T * (double)H * F);
            if (!ok) return false;
            continue;
        }
        if (!gemm(enc->ctx, &w.tm_o, w.w_o, w.b_o, enc->x, enc->y, H, H, EPI_BIAS_RES)) return false;
        prof_begin(st, PROF_NORM);
        if (!launch_layernorm(st, enc->y, w.ln1_g, w.ln1_b, enc->x, T, H, c.ln_eps)) return false;
        prof_end(st, PROF_NORM, 0);
        if (!gemm(enc->x, &w.tm_1, w.w_1, w.b_1, nullptr, enc->ffn, F, H, EPI_BIAS_GELU)) return false;
        if (!gemm(enc->ffn, &w.tm_2, w.w_2, w.b_2, enc->x, enc->y, H, F, EPI_BIAS_RES)) return false;
        prof_begin(st, PROF_NORM);
        if (!launch_layernorm(st, enc->y, w.ln2_g, w.ln2_b, enc->x, T, H, c.ln_eps)) return false;
        prof_end(st, PROF_NORM, 0);
    }
    return launch_pool(st, enc->x, seq_start, enc->seq_len, row_base, n_seq, H, c.pooling, c.normalize, out);
}

}  // namespace lb2
