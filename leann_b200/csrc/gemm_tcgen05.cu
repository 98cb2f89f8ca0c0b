// Recompute stage, dense part: C[M,N] = epilogue(A[M,K] . W[N,K]^T + bias) on the
// 5th-generation tensor cores (tcgen05.mma, fp16 operands, fp32 accumulation in TMEM).
//
// This is the arithmetic the reference runs inside SentenceTransformer.encode
// (packages/leann-core/src/leann/embedding_compute.py:231-239; fp16 weights and
// activations, :157-158) for every hop's batch of neighbour chunks: the four
// nn.Linear layers of each BERT block (QKV, attention output, FFN up, FFN down).
//
// Kernel shape (one persistent CTA per SM, 384 threads, warp-specialised):
//   warp 0 lane 0 : TMA producer   (cp.async.bulk.tensor 2D, 128B swizzle, 4-stage ring)
//   warp 1 lane 0 : MMA issuer     (tcgen05.mma cta_group::1 kind::f16, M=128, N=192, K=16)
//   warp 2        : TMEM allocator (2 accumulator stages x 192 columns -> 512 columns)
//   warps 4..11   : epilogue       (tcgen05.ld 32x32b, register double-buffered -> bias / GELU /
//                                   residual -> fp16 -> swizzled smem box -> TMA store; residual tiles
//                                   arrive by TMA load); two warps per TMEM lane quarter
// Pipelines: smem full/empty mbarriers between TMA and MMA, TMEM full/empty mbarriers
// between MMA and epilogue, so the epilogue of tile i overlaps the MMAs of tile i+1.
// M is ragged (varlen-packed tokens): TMA zero-fills rows past M, stores are row-masked.
#include <cuda_fp16.h>

#include "common.cuh"
#include "ptx.cuh"

namespace lb2 {

namespace {

constexpr int BLOCK_M = 128;
constexpr int BLOCK_K = 64;  // 64 fp16 = 128 B = one swizzle span
constexpr int UMMA_K = 16;
constexpr int GEMM_THREADS = 384;  // 4 control warps + 8 epilogue warps
constexpr int EPI_WARPS = 8;

template <int BLOCK_N, int STAGES>
struct GemmSmem {
    static constexpr int A_BYTES = BLOCK_M * BLOCK_K * 2;
    static constexpr int B_BYTES = BLOCK_N * BLOCK_K * 2;
    static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
    // epilogue staging: per epilogue warp, one 32-row x 32-column fp16 box (2 KB, SWIZZLE_64B) per column chunk
    static constexpr int EPI_CHUNKS = BLOCK_N / 32 / 2;
    static constexpr int EPI_OFFSET = STAGES * STAGE_BYTES;
    static constexpr int EPI_BYTES = EPI_WARPS * EPI_CHUNKS * 2048;
    static constexpr int BAR_OFFSET = EPI_OFFSET + EPI_BYTES;
    static constexpr int TOTAL = BAR_OFFSET + (2 * STAGES + 4 + EPI_WARPS) * 8 + 16 + 1024 /*alignment slack*/;
};

// HF "gelu" (erf form: x * Phi(x)), the activation of all-MiniLM-L6-v2 / bge-base BERT blocks.
// The K=384 GEMMs leave ~12 issue slots per output element before the epilogue, not the tensor
// pipe, becomes the limiter, and erff() costs ~30.  Phi(x) = 0.5 (1 + tanh(x (c0 + c1 x^2 + c2 x^4)))
// with minimax-fitted coefficients reproduces erf-GELU to 2.5e-5 absolute / 4.5e-4 relative
// (|gelu| > 0.05) — below the fp16 rounding of the stored activation — in 7 FP ops + 1 MUFU.
__device__ __forceinline__ float gelu_fast(float x) {
    const float x2 = fminf(x * x, 64.0f);  // the fit is monotone up to |x| = 8, tanh saturated long before
    float p = fmaf(x2, -3.51516789e-04f, 3.70056460e-02f);
    p = fmaf(x2, p, 7.97507884e-01f);
    float t;
    asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(x * p));
    const float hx = 0.5f * x;
    return fmaf(hx, t, hx);
}

template <int BLOCK_N, int STAGES, int EPI>
__global__ void __launch_bounds__(GEMM_THREADS, 1)
gemm_f16_tn_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
                   const __grid_constant__ CUtensorMap tmap_c, const __grid_constant__ CUtensorMap tmap_r,
                   const float* __restrict__ bias, int M, int N, int K, int c_group) {
    using L = GemmSmem<BLOCK_N, STAGES>;
    constexpr int TMEM_COLS = (2 * BLOCK_N <= 32) ? 32 : (2 * BLOCK_N <= 64) ? 64 : (2 * BLOCK_N <= 128) ? 128
                            : (2 * BLOCK_N <= 256) ? 256 : 512;
    static_assert(2 * BLOCK_N <= 512, "two accumulator stages must fit TMEM");
    static_assert(BLOCK_N % 64 == 0 && BLOCK_N % 16 == 0 && BLOCK_N <= 256, "UMMA N constraint / two column halves");

    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + L::BAR_OFFSET);
    uint64_t* empty_bar = full_bar + STAGES;
    uint64_t* tmem_full = empty_bar + STAGES;
    uint64_t* tmem_empty = tmem_full + 2;
    uint64_t* res_bar = tmem_empty + 2;  // [EPI_WARPS] residual boxes landed
    uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(res_bar + EPI_WARPS);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int num_m = (M + BLOCK_M - 1) / BLOCK_M;
    const int num_n = N / BLOCK_N;
    const int num_k = K / BLOCK_K;
    const int num_tiles = num_m * num_n;

    if (warp == 0 && lane == 0) {
        ptx::prefetch_tmap(&tmap_a);
        ptx::prefetch_tmap(&tmap_b);
        ptx::prefetch_tmap(&tmap_c);
        if (EPI == EPI_BIAS_RES) ptx::prefetch_tmap(&tmap_r);
    }
    if (warp == 1 && lane == 0) {
        for (int i = 0; i < STAGES; i++) {
            ptx::mbar_init(&full_bar[i], 1);
            ptx::mbar_init(&empty_bar[i], 1);
        }
        for (int i = 0; i < 2; i++) {
            ptx::mbar_init(&tmem_full[i], 1);
            ptx::mbar_init(&tmem_empty[i], EPI_WARPS);  // one arrive per epilogue warp
        }
        for (int i = 0; i < EPI_WARPS; i++) ptx::mbar_init(&res_bar[i], 1);
        ptx::fence_barrier_init();
    }
    if (warp == 2) {
        ptx::tmem_alloc(tmem_ptr, TMEM_COLS);
        ptx::tmem_relinquish();
    }
    ptx::tc_fence_before();
    __syncthreads();
    ptx::tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr;

    if (warp == 0) {
        // ===== TMA producer (whole warp, one elected issuer) =====
        int stage = 0;
        uint32_t phase = 0;
        for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
            const int m_blk = tile / num_n, n_blk = tile % num_n;
            for (int kb = 0; kb < num_k; kb++) {
                ptx::mbar_wait(&empty_bar[stage], phase ^ 1);
                uint8_t* sa = smem + stage * L::STAGE_BYTES;
                uint8_t* sb = sa + L::A_BYTES;
                if (ptx::elect_one()) {
                    ptx::mbar_expect_tx(&full_bar[stage], L::STAGE_BYTES);
                    ptx::tma_load_2d(sa, &tmap_a, &full_bar[stage], kb * BLOCK_K, m_blk * BLOCK_M);
                    ptx::tma_load_2d(sb, &tmap_b, &full_bar[stage], kb * BLOCK_K, n_blk * BLOCK_N);
                }
                __syncwarp();
                if (++stage == STAGES) { stage = 0; phase ^= 1; }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer: the whole warp runs the loop (warp-uniform control flow keeps the descriptors in uniform
        // registers), one elected lane issues
        constexpr uint32_t idesc = ptx::make_idesc_f16(BLOCK_M, BLOCK_N);
        int stage = 0;
        uint32_t phase = 0;
        int it = 0;
        const uint32_t smem_base = ptx::smem_u32(smem);
        for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, it++) {
            const int as = it & 1;
            const uint32_t aphase = (it >> 1) & 1;
            ptx::mbar_wait(&tmem_empty[as], aphase ^ 1);
            ptx::tc_fence_after();
            const uint32_t d_tmem = tmem_base + as * BLOCK_N;
            for (int kb = 0; kb < num_k; kb++) {
                ptx::mbar_wait(&full_bar[stage], phase);
                ptx::tc_fence_after();
                const uint32_t sa = smem_base + stage * L::STAGE_BYTES;
                const uint64_t a_desc = ptx::make_sw128_kmajor_desc(sa);
                const uint64_t b_desc = ptx::make_sw128_kmajor_desc(sa + L::A_BYTES);
                if (ptx::elect_one()) {
#pragma unroll
                    for (int k = 0; k < BLOCK_K / UMMA_K; k++) {
                        // advance 16 fp16 = 32 B along K inside the 128B swizzle span: +2 in 16B units
                        ptx::umma_f16(d_tmem, a_desc + 2 * k, b_desc + 2 * k, idesc, (kb | k) != 0);
                    }
                    ptx::umma_commit(&empty_bar[stage]);  // smem slot reusable once these MMAs retire
                }
                __syncwarp();
                if (++stage == STAGES) { stage = 0; phase ^= 1; }
            }
            if (ptx::elect_one()) ptx::umma_commit(&tmem_full[as]);  // accumulator complete
            __syncwarp();
        }
    } else if (warp >= 4) {
        // ===== epilogue: 8 warps, two per TMEM lane quarter, each owning half of the tile's columns.
        // Per 32-column chunk: TMEM -> registers -> (+bias, GELU | +residual) -> fp16 -> this warp's
        // private 32x32 smem box (SWIZZLE_64B, conflict-free 16-byte stores) -> TMA store.  The
        // residual boxes of the tile are TMA-loaded into the same smem boxes before the accumulator
        // is ready and overwritten in place.  Rows past M are clipped / zero-filled by TMA.
        const int quarter = warp & 3;          // TMEM lanes [32*quarter, +32) are the ones this warp may read
        const int ew = warp - 4;
        const int half = ew >> 2;              // column half of the accumulator
        constexpr int NCH = L::EPI_CHUNKS;     // 32-column chunks per warp
        uint8_t* stage_buf = smem + L::EPI_OFFSET + ew * NCH * 2048;
        // swizzle-64B: the 16-byte chunk j of box row r lives at chunk j ^ ((r >> 1) & 3)
        const int swz = (lane >> 1) & 3;
        uint32_t res_phase = 0;
        int it = 0;
        for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, it++) {
            const int m_blk = tile / num_n, n_blk = tile % num_n;
            const int as = it & 1;
            const uint32_t aphase = (it >> 1) & 1;
            const int row0 = m_blk * BLOCK_M + quarter * 32;
            const int colbase = n_blk * BLOCK_N + half * NCH * 32;
            if (EPI == EPI_BIAS_RES) {
                if (lane == 0) {
                    ptx::bulk_wait_read<0>();  // previous tile's stores no longer read the boxes
                    ptx::mbar_expect_tx(&res_bar[ew], NCH * 2048);
#pragma unroll
                    for (int c = 0; c < NCH; c++)
                        ptx::tma_load_2d(stage_buf + c * 2048, &tmap_r, &res_bar[ew], colbase + c * 32, row0);
                }
            }
            ptx::mbar_wait(&tmem_full[as], aphase);
            ptx::tc_fence_after();
            const uint32_t taddr = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) + as * BLOCK_N + half * NCH * 32;
            uint32_t r[2][32];
            ptx::tmem_ld_32x32(taddr, r[0]);
            if (EPI == EPI_BIAS_RES) {
                ptx::mbar_wait(&res_bar[ew], res_phase);
                res_phase ^= 1;
            }
#pragma unroll
            for (int c = 0; c < NCH; c++) {
                ptx::tmem_ld_wait();
                if (c + 1 < NCH) ptx::tmem_ld_32x32(taddr + (c + 1) * 32, r[(c + 1) & 1]);  // overlaps the math below
                const uint32_t(&acc)[32] = r[c & 1];
                const int col0 = colbase + c * 32;
                uint8_t* box = stage_buf + c * 2048 + lane * 64;
                if (EPI != EPI_BIAS_RES) {
                    // the store issued from this box one tile ago must have finished reading it
                    if (lane == 0) ptx::bulk_wait_read<NCH - 1>();
                    __syncwarp();
                }
                const float4* bp = reinterpret_cast<const float4*>(bias + col0);
#pragma unroll
                for (int j4 = 0; j4 < 4; j4++) {  // 16-byte piece j4 of this thread's 64-byte row segment
                    uint4* slot = reinterpret_cast<uint4*>(box + ((j4 ^ swz) << 4));
                    float v[8];
#pragma unroll
                    for (int u = 0; u < 2; u++) {
                        const float4 b4 = __ldg(bp + 2 * j4 + u);  // warp-uniform address: one broadcast transaction
                        v[4 * u + 0] = __uint_as_float(acc[8 * j4 + 4 * u + 0]) + b4.x;
                        v[4 * u + 1] = __uint_as_float(acc[8 * j4 + 4 * u + 1]) + b4.y;
                        v[4 * u + 2] = __uint_as_float(acc[8 * j4 + 4 * u + 2]) + b4.z;
                        v[4 * u + 3] = __uint_as_float(acc[8 * j4 + 4 * u + 3]) + b4.w;
                    }
                    if (EPI == EPI_BIAS_GELU) {
#pragma unroll
                        for (int u = 0; u < 8; u++) v[u] = gelu_fast(v[u]);
                    }
                    if (EPI == EPI_BIAS_RES) {
                        const uint4 rv = *slot;
                        const __half2* rh = reinterpret_cast<const __half2*>(&rv);
#pragma unroll
                        for (int u = 0; u < 4; u++) {
                            const float2 rf = __half22float2(rh[u]);
                            v[2 * u] += rf.x;
                            v[2 * u + 1] += rf.y;
                        }
                    }
                    uint4 ov;
                    __half2* oh = reinterpret_cast<__half2*>(&ov);
#pragma unroll
                    for (int u = 0; u < 4; u++) oh[u] = __floats2half2_rn(v[2 * u], v[2 * u + 1]);
                    *slot = ov;
                }
                ptx::fence_async_smem();
                __syncwarp();
                if (lane == 0) {
                    if (c_group > 0)  // grouped (head-major) output [N / c_group][M][c_group]
                        ptx::tma_store_3d(&tmap_c, stage_buf + c * 2048, col0 % c_group, row0, col0 / c_group);
                    else
                        ptx::tma_store_2d(&tmap_c, stage_buf + c * 2048, col0, row0);
                    ptx::bulk_commit();
                }
            }
            ptx::tc_fence_before();
            __syncwarp();
            if (lane == 0) ptx::mbar_arrive(&tmem_empty[as]);
        }
        if (lane == 0) ptx::bulk_wait_all();
    }

    ptx::tc_fence_before();
    __syncthreads();
    if (warp == 2) {
        ptx::tc_fence_after();
        ptx::tmem_dealloc(tmem_base, TMEM_COLS);
    }
}


// ---------------------------------------------------------------------------------------------------------------------
// Weight-stationary variant for the K = 384 projections (QKV, FFN up).
//
// gemm_f16_tn_kernel refills shared memory with (128 + 192) rows x 128 B per 64-deep k-block, i.e. 40 KB per 384 tensor
// clocks = 106 B/clk per SM; ncu shows the tensor pipe active 50-55 % of the time on these shapes with HBM at 35-40 % —
// the L2 -> shared-memory fill rate, not HBM or the epilogue, is what the MMA warp waits for (cuBLAS lands on the same
// ~950 TFLOP/s).  With K = 384 a whole 192-row panel of W is only 144 KB: this kernel keeps it resident in shared memory
// and streams just the activations (16 KB per k-block = 43 B/clk).  The grid is (CTAs per panel) x (panels): CTA (i, p)
// computes panel p of the i-th contiguous slice of row blocks, so the N / 192 CTAs that need the same rows of A read them at
// the same time and all but the first read hit L2 (with 148 SMs and 6 or 8 panels, 144 CTAs run; a free-form split of the
// tile list would use all 148 but skew the readers of a row block by tens of tiles — hundreds of MB of L2 traffic apart).
// The kernel itself accepts any contiguous range of the panel-major tile list: a range that crosses a panel boundary
// drains the MMAs that read the old panel (b_empty) and reloads.  Epilogue as in gemm_f16_tn_kernel (bias / GELU -> fp16
// -> swizzled 32x32 box -> TMA store), one staging box per warp (reused per chunk: the box is free again long before the
// next chunk's arithmetic is done), bias panel in shared memory.
//
// How many k-blocks ahead of its loads the producer asks L2 for the activation rows (cp.async.bulk.prefetch.tensor).  The
// shared-memory ring only covers 4 k-blocks = ~1 500 tensor clocks of work, while a TMA load of rows that are not in L2 yet
// takes ~3 000 clocks under load (ncu: the MMA warp spent 42 % of its samples on the `full` barriers); the prefetch turns
// those loads into L2 hits without spending shared memory (12 k-blocks x 16 KB x 148 CTAs = 28 MB outstanding, L2 is 126 MB).
// Measured (profiles/r02c_gemm_prefetch_sweep.log): the weight-stationary kernel gains 3-4 % on the QKV shape with 6-12
// k-blocks, nothing on FFN-up; the streaming kernels (which also stream W) LOSE 10-30 % at K = 1536 — their prefetches
// compete with the loads they are meant to help — so only the weight-stationary kernel prefetches.
constexpr int WS_PF_TILES = 12;

template <int BLOCK_N, int NUM_K, int STAGES>
struct GemmWsSmem {
    static constexpr int A_BYTES = BLOCK_M * BLOCK_K * 2;       // one k-block of activations
    static constexpr int B_SLAB = BLOCK_N * BLOCK_K * 2;        // one k-block of the weight panel
    static constexpr int B_BYTES = NUM_K * B_SLAB;
    static constexpr int A_OFFSET = B_BYTES;
    static constexpr int EPI_OFFSET = A_OFFSET + STAGES * A_BYTES;
    static constexpr int EPI_BYTES = EPI_WARPS * 2048;
    static constexpr int BIAS_OFFSET = EPI_OFFSET + EPI_BYTES;
    static constexpr int BAR_OFFSET = BIAS_OFFSET + BLOCK_N * 4;
    static constexpr int TOTAL = BAR_OFFSET + (2 * STAGES + 6) * 8 + 16 + 1024 /*alignment slack*/;
};

template <int BLOCK_N, int NUM_K, int STAGES, int EPI>
__global__ void __launch_bounds__(GEMM_THREADS, 1)
gemm_f16_ws_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
                   const __grid_constant__ CUtensorMap tmap_c, const float* __restrict__ bias, int M, int N, int c_group,
                   int ctas_per_panel) {
    using L = GemmWsSmem<BLOCK_N, NUM_K, STAGES>;
    static_assert(L::TOTAL <= 232448, "shared memory budget");
    static_assert(EPI == EPI_BIAS || EPI == EPI_BIAS_GELU, "no residual variant");
    constexpr int TMEM_COLS = 512;
    static_assert(2 * BLOCK_N <= 512 && BLOCK_N % 64 == 0, "two accumulator stages must fit TMEM");

    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    float* bias_s = reinterpret_cast<float*>(smem + L::BIAS_OFFSET);
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + L::BAR_OFFSET);
    uint64_t* empty_bar = full_bar + STAGES;
    uint64_t* tmem_full = empty_bar + STAGES;
    uint64_t* tmem_empty = tmem_full + 2;
    uint64_t* b_full = tmem_empty + 2;
    uint64_t* b_empty = b_full + 1;
    uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(b_empty + 1);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int num_m = (M + BLOCK_M - 1) / BLOCK_M;
    const int num_n = N / BLOCK_N;
    // this CTA's contiguous range of the panel-major tile list (tile = panel * num_m + row block)
    int t_begin, t_end;
    if (ctas_per_panel > 0) {
        const int panel = blockIdx.x / ctas_per_panel, idx = blockIdx.x - panel * ctas_per_panel;
        t_begin = panel * num_m + static_cast<int>(static_cast<long long>(num_m) * idx / ctas_per_panel);
        t_end = panel * num_m + static_cast<int>(static_cast<long long>(num_m) * (idx + 1) / ctas_per_panel);
    } else {
        const long long num_tiles = static_cast<long long>(num_m) * num_n;
        t_begin = static_cast<int>(num_tiles * blockIdx.x / gridDim.x);
        t_end = static_cast<int>(num_tiles * (blockIdx.x + 1) / gridDim.x);
    }

    if (warp == 0 && lane == 0) {
        ptx::prefetch_tmap(&tmap_a);
        ptx::prefetch_tmap(&tmap_b);
        ptx::prefetch_tmap(&tmap_c);
    }
    if (warp == 1 && lane == 0) {
        for (int i = 0; i < STAGES; i++) {
            ptx::mbar_init(&full_bar[i], 1);
            ptx::mbar_init(&empty_bar[i], 1);
        }
        for (int i = 0; i < 2; i++) {
            ptx::mbar_init(&tmem_full[i], 1);
            ptx::mbar_init(&tmem_empty[i], EPI_WARPS);
        }
        ptx::mbar_init(b_full, 1);
        ptx::mbar_init(b_empty, 1);
        ptx::fence_barrier_init();
    }
    if (warp == 2) {
        ptx::tmem_alloc(tmem_ptr, TMEM_COLS);
        ptx::tmem_relinquish();
    }
    ptx::tc_fence_before();
    __syncthreads();
    ptx::tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr;

    if (warp == 0) {
        // ===== TMA producer (whole warp, one elected issuer): the weight panel when it changes, the activation k-blocks always
        int stage = 0;
        uint32_t phase = 0, bphase = 0;
        int cur_n = -1;
        for (int tile = t_begin; tile < t_end; tile++) {
            const int n_blk = tile / num_m, m_blk = tile - n_blk * num_m;
            if (n_blk != cur_n) {
                if (cur_n >= 0) {  // every MMA that reads the old panel has retired
                    ptx::mbar_wait(b_empty, bphase);
                    bphase ^= 1;
                }
                if (ptx::elect_one()) {
                    ptx::mbar_expect_tx(b_full, L::B_BYTES);
#pragma unroll
                    for (int kb = 0; kb < NUM_K; kb++)
                        ptx::tma_load_2d(smem + kb * L::B_SLAB, &tmap_b, b_full, kb * BLOCK_K, n_blk * BLOCK_N);
                }
                __syncwarp();
                cur_n = n_blk;
            }
            for (int kb = 0; kb < NUM_K; kb++) {
                // the A k-block this CTA loads WS_PF_TILES k-blocks from now: into L2 (only the CTAs of panel 0 ask — the
                // others read the same rows at the same time)
                const int pf_it = (kb + WS_PF_TILES) / NUM_K, pf_kb = (kb + WS_PF_TILES) - pf_it * NUM_K;
                const bool pf = n_blk == 0 && tile + pf_it < t_end;
                ptx::mbar_wait(&empty_bar[stage], phase ^ 1);
                if (ptx::elect_one()) {
                    if (pf) ptx::tma_prefetch_2d(&tmap_a, pf_kb * BLOCK_K, (m_blk + pf_it) * BLOCK_M);
                    ptx::mbar_expect_tx(&full_bar[stage], L::A_BYTES);
                    ptx::tma_load_2d(smem + L::A_OFFSET + stage * L::A_BYTES, &tmap_a, &full_bar[stage], kb * BLOCK_K,
                                     m_blk * BLOCK_M);
                }
                __syncwarp();
                if (++stage == STAGES) { stage = 0; phase ^= 1; }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer.  The WHOLE warp runs the loop and one elected lane issues: with warp-uniform control flow the
        // descriptors live in uniform registers; under `if (lane == 0)` the compiler wrapped every tcgen05.mma in an
        // ELECT / R2UR.BROADCAST / BRA.U.ANY loop and the issuing thread, not the tensor pipe, set the pace
        // (profiles/r02_gemm_ws_ncu.md).
        constexpr uint32_t idesc = ptx::make_idesc_f16(BLOCK_M, BLOCK_N);
        int stage = 0;
        uint32_t phase = 0, bphase = 0;
        int cur_n = -1;
        int it = 0;
        const uint32_t a_base = ptx::smem_u32(smem + L::A_OFFSET), b_base = ptx::smem_u32(smem);
        for (int tile = t_begin; tile < t_end; tile++, it++) {
            const int n_blk = tile / num_m;
            if (n_blk != cur_n) {
                ptx::mbar_wait(b_full, bphase);
                bphase ^= 1;
                cur_n = n_blk;
            }
            const int as = it & 1;
            ptx::mbar_wait(&tmem_empty[as], ((it >> 1) & 1) ^ 1);
            ptx::tc_fence_after();
            const uint32_t d_tmem = tmem_base + as * BLOCK_N;
#pragma unroll
            for (int kb = 0; kb < NUM_K; kb++) {
                ptx::mbar_wait(&full_bar[stage], phase);
                ptx::tc_fence_after();
                const uint64_t a_desc = ptx::make_sw128_kmajor_desc(a_base + stage * L::A_BYTES);
                const uint64_t b_desc = ptx::make_sw128_kmajor_desc(b_base + kb * L::B_SLAB);
                if (ptx::elect_one()) {
#pragma unroll
                    for (int k = 0; k < BLOCK_K / UMMA_K; k++)
                        ptx::umma_f16(d_tmem, a_desc + 2 * k, b_desc + 2 * k, idesc, (kb | k) != 0);
                    ptx::umma_commit(&empty_bar[stage]);
                }
                __syncwarp();
                if (++stage == STAGES) { stage = 0; phase ^= 1; }
            }
            const bool panel_ends = tile + 1 < t_end && (tile + 1) / num_m != n_blk;  // the panel may be replaced
            if (ptx::elect_one()) {
                ptx::umma_commit(&tmem_full[as]);
                if (panel_ends) ptx::umma_commit(b_empty);
            }
            __syncwarp();
        }
    } else if (warp >= 4) {
        // ===== epilogue: 8 warps, two per TMEM lane quarter, each owning half of the tile's columns
        const int quarter = warp & 3;
        const int ew = warp - 4;
        const int half = ew >> 2;
        constexpr int NCH = BLOCK_N / 32 / 2;
        uint8_t* box_base = smem + L::EPI_OFFSET + ew * 2048;
        const int swz = (lane >> 1) & 3;
        const int et = threadIdx.x - 128;  // 0..255 among the epilogue threads
        int cur_n = -1;
        int it = 0;
        for (int tile = t_begin; tile < t_end; tile++, it++) {
            const int n_blk = tile / num_m, m_blk = tile - n_blk * num_m;
            if (n_blk != cur_n) {  // new panel: its bias slice into shared memory (all epilogue warps are past the old one)
                asm volatile("bar.sync 1, 256;" ::: "memory");
                if (et < BLOCK_N) bias_s[et] = __ldg(bias + n_blk * BLOCK_N + et);
                asm volatile("bar.sync 1, 256;" ::: "memory");
                cur_n = n_blk;
            }
            const int as = it & 1;
            const int row0 = m_blk * BLOCK_M + quarter * 32;
            const int colbase = n_blk * BLOCK_N + half * NCH * 32;
            ptx::mbar_wait(&tmem_full[as], (it >> 1) & 1);
            ptx::tc_fence_after();
            const uint32_t taddr = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) + as * BLOCK_N + half * NCH * 32;
            uint32_t r[2][32];
            ptx::tmem_ld_32x32(taddr, r[0]);
#pragma unroll
            for (int c = 0; c < NCH; c++) {
                ptx::tmem_ld_wait();
                if (c + 1 < NCH) ptx::tmem_ld_32x32(taddr + (c + 1) * 32, r[(c + 1) & 1]);
                const uint32_t(&acc)[32] = r[c & 1];
                const int col0 = colbase + c * 32;
                const float4* bp = reinterpret_cast<const float4*>(bias_s + half * NCH * 32 + c * 32);
                uint4 ov[4];
#pragma unroll
                for (int j4 = 0; j4 < 4; j4++) {
                    float v[8];
#pragma unroll
                    for (int u = 0; u < 2; u++) {
                        const float4 b4 = bp[2 * j4 + u];  // warp-uniform address: broadcast
                        v[4 * u + 0] = __uint_as_float(acc[8 * j4 + 4 * u + 0]) + b4.x;
                        v[4 * u + 1] = __uint_as_float(acc[8 * j4 + 4 * u + 1]) + b4.y;
                        v[4 * u + 2] = __uint_as_float(acc[8 * j4 + 4 * u + 2]) + b4.z;
                        v[4 * u + 3] = __uint_as_float(acc[8 * j4 + 4 * u + 3]) + b4.w;
                    }
                    if (EPI == EPI_BIAS_GELU) {
#pragma unroll
                        for (int u = 0; u < 8; u++) v[u] = gelu_fast(v[u]);
                    }
                    __half2* oh = reinterpret_cast<__half2*>(&ov[j4]);
#pragma unroll
                    for (int u = 0; u < 4; u++) oh[u] = __floats2half2_rn(v[2 * u], v[2 * u + 1]);
                }
                uint8_t* box = box_base + lane * 64;
                // the store issued from this warp's box one chunk ago must have finished reading it
                if (lane == 0) ptx::bulk_wait_read<0>();
                __syncwarp();
#pragma unroll
                for (int j4 = 0; j4 < 4; j4++) *reinterpret_cast<uint4*>(box + ((j4 ^ swz) << 4)) = ov[j4];
                ptx::fence_async_smem();
                __syncwarp();
                if (lane == 0) {
                    if (c_group > 0)
                        ptx::tma_store_3d(&tmap_c, box_base, col0 % c_group, row0, col0 / c_group);
                    else
                        ptx::tma_store_2d(&tmap_c, box_base, col0, row0);
                    ptx::bulk_commit();
                }
            }
            ptx::tc_fence_before();
            __syncwarp();
            if (lane == 0) ptx::mbar_arrive(&tmem_empty[as]);
        }
        if (lane == 0) ptx::bulk_wait_all();
    }

    ptx::tc_fence_before();
    __syncthreads();
    if (warp == 2) {
        ptx::tc_fence_after();
        ptx::tmem_dealloc(tmem_base, TMEM_COLS);
    }
}


// ---------------------------------------------------------------------------------------------------------------------
// Residual projection with LayerNorm fused into the epilogue (hidden = 2 * BLOCK_N = 384 only):
//     x_out = LayerNorm(A . W^T + bias + residual) * gamma + beta
// i.e. the attention-output / FFN-down Linear, the residual add and BertSelfOutput / BertOutput's LayerNorm of one BERT
// block in one kernel: the pre-norm activation never goes to HBM (the separate LayerNorm kernel read and wrote 1.5 KB per
// token twice per layer).  A CTA owns WHOLE rows: it computes the two 192-column halves of a 128-row block back to back
// (two TMEM accumulator stages), the epilogue keeps both halves as fp16 in shared memory (the TMA-store staging boxes,
// 96 KB), accumulates per-row sum / sum of squares on the fp16-rounded values (the numerics of the unfused pipeline, which
// normalised the fp16 tensor), exchanges them between the two warps that share a row, normalises in place and stores.
// Same producer / MMA warps and mbarrier pipelines as gemm_f16_tn_kernel; 3 smem stages instead of 4 to make room.
template <int BLOCK_N, int STAGES, bool PAIR>
struct GemmLnSmem {
    static constexpr int A_BYTES = BLOCK_M * BLOCK_K * 2;
    static constexpr int B_BYTES = (PAIR ? BLOCK_N / 2 : BLOCK_N) * BLOCK_K * 2;  // a CTA pair splits the W rows of a panel
    static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
    static constexpr int EPI_CHUNKS = BLOCK_N / 32 / 2;            // 32-column chunks per warp and half
    static constexpr int TILE_BOX_BYTES = EPI_WARPS * EPI_CHUNKS * 2048;
    static constexpr int EPI_OFFSET = STAGES * STAGE_BYTES;
    static constexpr int EPI_BYTES = 2 * TILE_BOX_BYTES;           // both column halves of the row block
    static constexpr int STAT_OFFSET = EPI_OFFSET + EPI_BYTES;
    static constexpr int STAT_BYTES = EPI_WARPS * 32 * 8;
    static constexpr int BAR_OFFSET = STAT_OFFSET + STAT_BYTES;
    static constexpr int TOTAL = BAR_OFFSET + (2 * STAGES + 4 + 2 * EPI_WARPS) * 8 + 16 + 1024;
};

//
// PAIR = true: two CTAs of a cluster work as one (tcgen05 cta_group::2, M = 256): each owns one 128-row block and loads
// its own A tile plus HALF of the W rows of the panel (96 of 192); the MMA — issued by rank 0 only — reads both halves, each
// CTA accumulates its rows in its own tensor memory and runs its own epilogue.  The shared-memory fill per CTA drops from
// 40 KB to 28 KB per k-block (the MMA warp was waiting for it: tensor pipe 44-65 % active in the single-CTA kernels), and
// the ring gets its fourth stage back.  Barriers: every CTA's TMA completes on rank 0's `full` barrier; `empty` and
// `tmem_full` are multicast commits to both CTAs; all 16 epilogue warps of the pair arrive on rank 0's `tmem_empty`.
template <int BLOCK_N, int STAGES, bool PAIR>
__device__ __forceinline__ void
gemm_f16_ln_body(const CUtensorMap& tmap_a, const CUtensorMap& tmap_b, const CUtensorMap& tmap_c, const CUtensorMap& tmap_r,
                 const float* __restrict__ bias, const float* __restrict__ gamma, const float* __restrict__ beta, float eps,
                 int M, int K) {
    using L = GemmLnSmem<BLOCK_N, STAGES, PAIR>;
    const int rank = PAIR ? static_cast<int>(ptx::cluster_ctarank()) : 0;
    // row blocks are dealt to CTAs (pairs: to the pair, rank r takes the r-th of two consecutive ones; a block past the end
    // is computed on zero-filled rows and stored nowhere)
    const int blk_first = PAIR ? (blockIdx.x >> 1) * 2 + rank : blockIdx.x;
    const int blk_step = gridDim.x;
    constexpr int N = 2 * BLOCK_N;
    constexpr int TMEM_COLS = 512;
    static_assert(2 * BLOCK_N <= 512, "two accumulator stages must fit TMEM");
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + L::BAR_OFFSET);
    uint64_t* empty_bar = full_bar + STAGES;
    uint64_t* tmem_full = empty_bar + STAGES;
    uint64_t* tmem_empty = tmem_full + 2;
    uint64_t* res_bar = tmem_empty + 2;  // [2][EPI_WARPS] residual boxes of a half landed
    uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(res_bar + 2 * EPI_WARPS);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int num_m = (M + BLOCK_M - 1) / BLOCK_M;
    const int num_k = K / BLOCK_K;

    if (warp == 0 && lane == 0) {
        ptx::prefetch_tmap(&tmap_a);
        ptx::prefetch_tmap(&tmap_b);
        ptx::prefetch_tmap(&tmap_c);
        ptx::prefetch_tmap(&tmap_r);
    }
    if (warp == 1 && lane == 0) {
        for (int i = 0; i < STAGES; i++) {
            ptx::mbar_init(&full_bar[i], 1);
            ptx::mbar_init(&empty_bar[i], 1);
        }
        for (int i = 0; i < 2; i++) {
            ptx::mbar_init(&tmem_full[i], 1);
            ptx::mbar_init(&tmem_empty[i], PAIR ? 2 * EPI_WARPS : EPI_WARPS);
        }
        for (int i = 0; i < 2 * EPI_WARPS; i++) ptx::mbar_init(&res_bar[i], 1);
        ptx::fence_barrier_init();
    }
    if (warp == 2) {
        if (PAIR) {
            ptx::tmem_alloc_pair(tmem_ptr, TMEM_COLS);
            ptx::tmem_relinquish_pair();
        } else {
            ptx::tmem_alloc(tmem_ptr, TMEM_COLS);
            ptx::tmem_relinquish();
        }
    }
    ptx::tc_fence_before();
    if (PAIR) ptx::cluster_sync(); else __syncthreads();  // pair: the peer's barriers must be initialised before any remote arrive
    ptx::tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr;

    if (warp == 0) {
        // ===== TMA producer (whole warp, one elected issuer): row block m, column halves 0 and 1 back to back
        int stage = 0;
        uint32_t phase = 0;
        for (int m_blk = blk_first; m_blk < num_m + rank; m_blk += blk_step) {
            for (int n_blk = 0; n_blk < 2; n_blk++) {
                for (int kb = 0; kb < num_k; kb++) {
                    ptx::mbar_wait(&empty_bar[stage], phase ^ 1);
                    uint8_t* sa = smem + stage * L::STAGE_BYTES;
                    uint8_t* sb = sa + L::A_BYTES;
                    if (ptx::elect_one()) {
                        if (PAIR) {
                            // both CTAs' bytes complete on rank 0's barrier; rank 0 announces the total
                            if (rank == 0) ptx::mbar_expect_tx(&full_bar[stage], 2 * L::STAGE_BYTES);
                            ptx::tma_load_2d_pair(sa, &tmap_a, &full_bar[stage], kb * BLOCK_K, m_blk * BLOCK_M);
                            ptx::tma_load_2d_pair(sb, &tmap_b, &full_bar[stage], kb * BLOCK_K,
                                                  n_blk * BLOCK_N + rank * (BLOCK_N / 2));
                        } else {
                            ptx::mbar_expect_tx(&full_bar[stage], L::STAGE_BYTES);
                            ptx::tma_load_2d(sa, &tmap_a, &full_bar[stage], kb * BLOCK_K, m_blk * BLOCK_M);
                            ptx::tma_load_2d(sb, &tmap_b, &full_bar[stage], kb * BLOCK_K, n_blk * BLOCK_N);
                        }
                    }
                    __syncwarp();
                    if (++stage == STAGES) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        if (rank == 0) {  // ===== MMA issuer (rank 0 of a pair): half n accumulates in TMEM stage n; whole warp, one elected lane issues
            constexpr uint32_t idesc = ptx::make_idesc_f16(PAIR ? 2 * BLOCK_M : BLOCK_M, BLOCK_N);
            int stage = 0;
            uint32_t phase = 0;
            int it = 0;
            const uint32_t smem_base = ptx::smem_u32(smem);
            for (int m_blk = blk_first; m_blk < num_m; m_blk += blk_step, it++) {
                for (int as = 0; as < 2; as++) {
                    ptx::mbar_wait(&tmem_empty[as], (it & 1) ^ 1);
                    ptx::tc_fence_after();
                    const uint32_t d_tmem = tmem_base + as * BLOCK_N;
                    for (int kb = 0; kb < num_k; kb++) {
                        ptx::mbar_wait(&full_bar[stage], phase);
                        ptx::tc_fence_after();
                        const uint32_t sa = smem_base + stage * L::STAGE_BYTES;
                        const uint64_t a_desc = ptx::make_sw128_kmajor_desc(sa);
                        const uint64_t b_desc = ptx::make_sw128_kmajor_desc(sa + L::A_BYTES);
                        if (ptx::elect_one()) {
#pragma unroll
                            for (int k = 0; k < BLOCK_K / UMMA_K; k++) {
                                if (PAIR) ptx::umma_f16_pair(d_tmem, a_desc + 2 * k, b_desc + 2 * k, idesc, (kb | k) != 0);
                                else ptx::umma_f16(d_tmem, a_desc + 2 * k, b_desc + 2 * k, idesc, (kb | k) != 0);
                            }
                            if (PAIR) ptx::umma_commit_pair(&empty_bar[stage]); else ptx::umma_commit(&empty_bar[stage]);
                        }
                        __syncwarp();
                        if (++stage == STAGES) { stage = 0; phase ^= 1; }
                    }
                    if (ptx::elect_one()) {
                        if (PAIR) ptx::umma_commit_pair(&tmem_full[as]); else ptx::umma_commit(&tmem_full[as]);
                    }
                    __syncwarp();
                }
            }
        }
    } else if (warp >= 4) {
        // ===== epilogue: 8 warps; warp (quarter, half) owns rows [32 quarter, +32) and, in each column half of the row block,
        // the 96 columns [96 half, +96) as three 32-column chunks.  Thread = row.
        const int quarter = warp & 3;
        const int ew = warp - 4;
        const int half = ew >> 2;
        constexpr int NCH = L::EPI_CHUNKS;
        const int swz = (lane >> 1) & 3;
        float2* stat = reinterpret_cast<float2*>(smem + L::STAT_OFFSET);
        uint32_t res_phase = 0;
        int it = 0;
        for (int m_blk = blk_first; m_blk < num_m + rank; m_blk += blk_step, it++) {
            const int row0 = m_blk * BLOCK_M + quarter * 32;
            if (lane == 0) {
                ptx::bulk_wait_read<0>();  // the previous row block's stores no longer read the boxes
                for (int n_blk = 0; n_blk < 2; n_blk++) {
                    uint8_t* boxes = smem + L::EPI_OFFSET + n_blk * L::TILE_BOX_BYTES + ew * NCH * 2048;
                    ptx::mbar_expect_tx(&res_bar[n_blk * EPI_WARPS + ew], NCH * 2048);
#pragma unroll
                    for (int c = 0; c < NCH; c++)
                        ptx::tma_load_2d(boxes + c * 2048, &tmap_r, &res_bar[n_blk * EPI_WARPS + ew],
                                         n_blk * BLOCK_N + half * NCH * 32 + c * 32, row0);
                }
            }
            float sum = 0.f, sumsq = 0.f;
            // ---- pass 1: accumulator + bias + residual -> fp16 (kept in the boxes), row statistics
            for (int n_blk = 0; n_blk < 2; n_blk++) {
                uint8_t* boxes = smem + L::EPI_OFFSET + n_blk * L::TILE_BOX_BYTES + ew * NCH * 2048;
                const int colbase = n_blk * BLOCK_N + half * NCH * 32;
                ptx::mbar_wait(&tmem_full[n_blk], it & 1);
                ptx::tc_fence_after();
                const uint32_t taddr = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) + n_blk * BLOCK_N + half * NCH * 32;
                uint32_t r[2][32];
                ptx::tmem_ld_32x32(taddr, r[0]);
                ptx::mbar_wait(&res_bar[n_blk * EPI_WARPS + ew], res_phase);
#pragma unroll
                for (int c = 0; c < NCH; c++) {
                    ptx::tmem_ld_wait();
                    if (c + 1 < NCH) ptx::tmem_ld_32x32(taddr + (c + 1) * 32, r[(c + 1) & 1]);
                    const uint32_t(&acc)[32] = r[c & 1];
                    uint8_t* box = boxes + c * 2048 + lane * 64;
                    const float4* bp = reinterpret_cast<const float4*>(bias + colbase + c * 32);
#pragma unroll
                    for (int j4 = 0; j4 < 4; j4++) {
                        uint4* slot = reinterpret_cast<uint4*>(box + ((j4 ^ swz) << 4));
                        const uint4 rv = *slot;
                        const __half2* rh = reinterpret_cast<const __half2*>(&rv);
                        uint4 ov;
                        __half2* oh = reinterpret_cast<__half2*>(&ov);
#pragma unroll
                        for (int u = 0; u < 2; u++) {
                            const float4 b4 = __ldg(bp + 2 * j4 + u);
                            const float2 r0 = __half22float2(rh[2 * u]), r1 = __half22float2(rh[2 * u + 1]);
                            const __half2 h0 = __floats2half2_rn(__uint_as_float(acc[8 * j4 + 4 * u + 0]) + b4.x + r0.x,
                                                                 __uint_as_float(acc[8 * j4 + 4 * u + 1]) + b4.y + r0.y);
                            const __half2 h1 = __floats2half2_rn(__uint_as_float(acc[8 * j4 + 4 * u + 2]) + b4.z + r1.x,
                                                                 __uint_as_float(acc[8 * j4 + 4 * u + 3]) + b4.w + r1.y);
                            oh[2 * u] = h0; oh[2 * u + 1] = h1;
                            const float2 f0 = __half22float2(h0), f1 = __half22float2(h1);
                            sum += (f0.x + f0.y) + (f1.x + f1.y);
                            sumsq = fmaf(f0.x, f0.x, sumsq); sumsq = fmaf(f0.y, f0.y, sumsq);
                            sumsq = fmaf(f1.x, f1.x, sumsq); sumsq = fmaf(f1.y, f1.y, sumsq);
                        }
                        *slot = ov;
                    }
                }
                ptx::tc_fence_before();
                __syncwarp();
                if (lane == 0) {  // accumulator stage free for the next row block
                    if (PAIR) ptx::mbar_arrive_leader(&tmem_empty[n_blk]); else ptx::mbar_arrive(&tmem_empty[n_blk]);
                }
            }
            res_phase ^= 1;
            // ---- the two warps of a row quarter hold the two halves of each row's statistics
            stat[ew * 32 + lane] = make_float2(sum, sumsq);
            asm volatile("bar.sync 1, %0;" ::"n"(EPI_WARPS * 32) : "memory");
            const float2 other = stat[(ew ^ 4) * 32 + lane];
            const float mean = (sum + other.x) * (1.0f / N);
            const float var = fmaxf((sumsq + other.y) * (1.0f / N) - mean * mean, 0.f);
            const float rstd = rsqrtf(var + eps);
            asm volatile("bar.sync 1, %0;" ::"n"(EPI_WARPS * 32) : "memory");  // stat[] may be overwritten by the next row block
            // ---- pass 2: normalise in place, store
            for (int n_blk = 0; n_blk < 2; n_blk++) {
                uint8_t* boxes = smem + L::EPI_OFFSET + n_blk * L::TILE_BOX_BYTES + ew * NCH * 2048;
                const int colbase = n_blk * BLOCK_N + half * NCH * 32;
#pragma unroll
                for (int c = 0; c < NCH; c++) {
                    uint8_t* box = boxes + c * 2048 + lane * 64;
                    const float4* gp = reinterpret_cast<const float4*>(gamma + colbase + c * 32);
                    const float4* bp = reinterpret_cast<const float4*>(beta + colbase + c * 32);
#pragma unroll
                    for (int j4 = 0; j4 < 4; j4++) {
                        uint4* slot = reinterpret_cast<uint4*>(box + ((j4 ^ swz) << 4));
                        const uint4 rv = *slot;
                        const __half2* rh = reinterpret_cast<const __half2*>(&rv);
                        uint4 ov;
                        __half2* oh = reinterpret_cast<__half2*>(&ov);
#pragma unroll
                        for (int u = 0; u < 2; u++) {
                            const float4 g4 = __ldg(gp + 2 * j4 + u), b4 = __ldg(bp + 2 * j4 + u);
                            const float2 v0 = __half22float2(rh[2 * u]), v1 = __half22float2(rh[2 * u + 1]);
                            oh[2 * u] = __floats2half2_rn((v0.x - mean) * rstd * g4.x + b4.x, (v0.y - mean) * rstd * g4.y + b4.y);
                            oh[2 * u + 1] = __floats2half2_rn((v1.x - mean) * rstd * g4.z + b4.z, (v1.y - mean) * rstd * g4.w + b4.w);
                        }
                        *slot = ov;
                    }
                    ptx::fence_async_smem();
                    __syncwarp();
                    if (lane == 0) {
                        ptx::tma_store_2d(&tmap_c, boxes + c * 2048, colbase + c * 32, row0);
                        ptx::bulk_commit();
                    }
                }
            }
        }
        if (lane == 0) ptx::bulk_wait_all();
    }

    ptx::tc_fence_before();
    if (PAIR) ptx::cluster_sync(); else __syncthreads();
    if (warp == 2) {
        ptx::tc_fence_after();
        if (PAIR) ptx::tmem_dealloc_pair(tmem_base, TMEM_COLS); else ptx::tmem_dealloc(tmem_base, TMEM_COLS);
    }
}

template <int BLOCK_N, int STAGES>
__global__ void __launch_bounds__(GEMM_THREADS, 1)
gemm_f16_ln_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
                   const __grid_constant__ CUtensorMap tmap_c, const __grid_constant__ CUtensorMap tmap_r,
                   const float* __restrict__ bias, const float* __restrict__ gamma, const float* __restrict__ beta, float eps,
                   int M, int K) {
    gemm_f16_ln_body<BLOCK_N, STAGES, false>(tmap_a, tmap_b, tmap_c, tmap_r, bias, gamma, beta, eps, M, K);
}

template <int BLOCK_N, int STAGES>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(GEMM_THREADS, 1)
gemm_f16_ln_pair_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
                        const __grid_constant__ CUtensorMap tmap_c, const __grid_constant__ CUtensorMap tmap_r,
                        const float* __restrict__ bias, const float* __restrict__ gamma, const float* __restrict__ beta,
                        float eps, int M, int K) {
    gemm_f16_ln_body<BLOCK_N, STAGES, true>(tmap_a, tmap_b, tmap_c, tmap_r, bias, gamma, beta, eps, M, K);
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode_fn() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres);
        if (e != cudaSuccess || qres != cudaDriverEntryPointSuccess || !p) return nullptr;
        fn = reinterpret_cast<EncodeTiledFn>(p);
    }
    return fn;
}

}  // namespace

// Row-major [rows, cols] fp16 matrix, box = [box_rows, box_cols]; box_cols = 64 -> SWIZZLE_128B
// (MMA operand tiles), box_cols = 32 -> SWIZZLE_64B (epilogue boxes).
bool make_tmap_f16_2d(CUtensorMap* map, const void* ptr, uint64_t rows, uint64_t cols, uint32_t box_rows,
                      uint32_t box_cols) {
    EncodeTiledFn fn = get_encode_fn();
    if (!fn) {
        set_error("cuTensorMapEncodeTiled entry point unavailable");
        return false;
    }
    cuuint64_t dims[2] = {cols, rows};
    cuuint64_t strides[1] = {cols * 2};
    cuuint32_t box[2] = {box_cols, box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(ptr), dims, strides, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, box_cols == 32 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B,
                    CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_error("cuTensorMapEncodeTiled failed (%d) rows=%llu cols=%llu", (int)r, (unsigned long long)rows,
                  (unsigned long long)cols);
        return false;
    }
    return true;
}

// Group-major activation [groups][rows][row_elems] fp16 (the head-major QKV buffer), box = [1][box_rows][box_cols];
// box_cols = 64 -> SWIZZLE_128B, 32 -> SWIZZLE_64B (the inner box extent is exactly one swizzle span).
bool make_tmap_f16_3d(CUtensorMap* map, const void* ptr, uint64_t row_elems, uint64_t rows, uint64_t groups, uint32_t box_cols,
                      uint32_t box_rows) {
    EncodeTiledFn fn = get_encode_fn();
    if (!fn) {
        set_error("cuTensorMapEncodeTiled entry point unavailable");
        return false;
    }
    cuuint64_t dims[3] = {row_elems, rows, groups};
    cuuint64_t strides[2] = {row_elems * 2, rows * row_elems * 2};
    cuuint32_t box[3] = {box_cols, box_rows, 1};
    cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3, const_cast<void*>(ptr), dims, strides, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, box_cols == 32 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B,
                    CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_error("cuTensorMapEncodeTiled (3d) failed (%d) rows=%llu groups=%llu", (int)r, (unsigned long long)rows,
                  (unsigned long long)groups);
        return false;
    }
    return true;
}

// Output viewed as [groups][rows][group_cols] fp16 (group-major), box = [1][32 rows][32 cols], SWIZZLE_64B.
static bool make_tmap_f16_grouped(CUtensorMap* map, const void* ptr, uint64_t rows, uint64_t group_cols, uint64_t groups) {
    EncodeTiledFn fn = get_encode_fn();
    if (!fn) {
        set_error("cuTensorMapEncodeTiled entry point unavailable");
        return false;
    }
    cuuint64_t dims[3] = {group_cols, rows, groups};
    cuuint64_t strides[2] = {group_cols * 2, rows * group_cols * 2};
    cuuint32_t box[3] = {32, 32, 1};
    cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3, const_cast<void*>(ptr), dims, strides, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_error("cuTensorMapEncodeTiled (grouped) failed (%d) rows=%llu", (int)r, (unsigned long long)rows);
        return false;
    }
    return true;
}

constexpr int GEMM_BLOCK_N = 192;
constexpr int GEMM_STAGES = 4;

template <int EPI>
static cudaError_t launch_gemm(cudaStream_t stream, const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& tc,
                               const CUtensorMap& tr, const float* bias, int M, int N, int K, int c_group, int num_sms) {
    using L = GemmSmem<GEMM_BLOCK_N, GEMM_STAGES>;
    auto kern = gemm_f16_tn_kernel<GEMM_BLOCK_N, GEMM_STAGES, EPI>;
    static thread_local int attr_dev_mask[8] = {0};  // the opt-in is per device: remember which devices have it
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= 256 || !(attr_dev_mask[dev >> 5] & (1 << (dev & 31)))) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, L::TOTAL);
        if (e != cudaSuccess) return e;
        if (dev >= 0 && dev < 256) attr_dev_mask[dev >> 5] |= 1 << (dev & 31);
    }
    const int tiles = ((M + BLOCK_M - 1) / BLOCK_M) * (N / GEMM_BLOCK_N);
    const int grid = tiles < num_sms ? tiles : num_sms;
    kern<<<grid, GEMM_THREADS, L::TOTAL, stream>>>(ta, tb, tc, tr, bias, M, N, K, c_group);
    return cudaGetLastError();
}

// weight-stationary kernel for K = 384
constexpr int WS_NUM_K = 6;
constexpr int WS_STAGES = 4;

template <int EPI>
static cudaError_t launch_gemm_ws(cudaStream_t stream, const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& tc,
                                  const float* bias, int M, int N, int c_group, int num_sms) {
    using L = GemmWsSmem<GEMM_BLOCK_N, WS_NUM_K, WS_STAGES>;
    auto kern = gemm_f16_ws_kernel<GEMM_BLOCK_N, WS_NUM_K, WS_STAGES, EPI>;
    static thread_local int attr_dev_mask[8] = {0};
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= 256 || !(attr_dev_mask[dev >> 5] & (1 << (dev & 31)))) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, L::TOTAL);
        if (e != cudaSuccess) return e;
        if (dev >= 0 && dev < 256) attr_dev_mask[dev >> 5] |= 1 << (dev & 31);
    }
    const int num_m = (M + BLOCK_M - 1) / BLOCK_M, num_n = N / GEMM_BLOCK_N;
    int cpp = num_sms / num_n;  // CTAs per panel
    if (cpp > num_m) cpp = num_m;
    int grid = cpp * num_n;
    if (cpp == 0) {  // more panels than SMs: free-form split of the tile list
        const long long tiles = static_cast<long long>(num_m) * num_n;
        grid = tiles < num_sms ? static_cast<int>(tiles) : num_sms;
    }
    kern<<<grid, GEMM_THREADS, L::TOTAL, stream>>>(ta, tb, tc, bias, M, N, c_group, cpp);
    return cudaGetLastError();
}

// A [M,K] fp16 row-major, W [N,K] fp16 row-major (nn.Linear layout), C [M,N] fp16.
// c_group > 0: C is written group-major, [N / c_group][M][c_group] (the per-head q|k|v layout attention reads).
bool gemm_f16(cudaStream_t stream, const __half* A, const CUtensorMap* tmap_w, const __half* W, const float* bias,
              const __half* residual, __half* C, int M, int N, int K, int epi, int num_sms, int c_group) {
    if (M <= 0) return true;
    if (N % GEMM_BLOCK_N != 0 || K % BLOCK_K != 0) {
        set_error("gemm_f16: unsupported shape N=%d K=%d (need N%%192==0, K%%64==0)", N, K);
        return false;
    }
    if (epi == EPI_BIAS_RES && !residual) {
        set_error("gemm_f16: residual epilogue without a residual matrix");
        return false;
    }
    CUtensorMap ta, tb_local, tc, tr;
    if (!make_tmap_f16_2d(&ta, A, (uint64_t)M, (uint64_t)K, BLOCK_M, BLOCK_K)) return false;
    if (c_group > 0) {
        if (c_group % 32 != 0 || N % c_group != 0 || epi == EPI_BIAS_RES) {
            set_error("gemm_f16: bad grouped output (c_group=%d N=%d)", c_group, N);
            return false;
        }
        if (!make_tmap_f16_grouped(&tc, C, (uint64_t)M, (uint64_t)c_group, (uint64_t)(N / c_group))) return false;
    } else if (!make_tmap_f16_2d(&tc, C, (uint64_t)M, (uint64_t)N, 32, 32)) {
        return false;
    }
    if (!make_tmap_f16_2d(&tr, epi == EPI_BIAS_RES ? residual : C, (uint64_t)M, (uint64_t)N, 32, 32)) return false;
    if (!tmap_w) {
        if (!make_tmap_f16_2d(&tb_local, W, (uint64_t)N, (uint64_t)K, GEMM_BLOCK_N, BLOCK_K)) return false;
        tmap_w = &tb_local;
    }
    cudaError_t e;
    if (K == WS_NUM_K * BLOCK_K && epi != EPI_BIAS_RES) {
        e = epi == EPI_BIAS ? launch_gemm_ws<EPI_BIAS>(stream, ta, *tmap_w, tc, bias, M, N, c_group, num_sms)
                            : launch_gemm_ws<EPI_BIAS_GELU>(stream, ta, *tmap_w, tc, bias, M, N, c_group, num_sms);
        if (e != cudaSuccess) {
            set_error("gemm_f16 (weight-stationary) launch: %s", cudaGetErrorString(e));
            return false;
        }
        return true;
    }
    switch (epi) {
        case EPI_BIAS: e = launch_gemm<EPI_BIAS>(stream, ta, *tmap_w, tc, tr, bias, M, N, K, c_group, num_sms); break;
        case EPI_BIAS_GELU: e = launch_gemm<EPI_BIAS_GELU>(stream, ta, *tmap_w, tc, tr, bias, M, N, K, c_group, num_sms); break;
        case EPI_BIAS_RES: e = launch_gemm<EPI_BIAS_RES>(stream, ta, *tmap_w, tc, tr, bias, M, N, K, c_group, num_sms); break;
        default: set_error("gemm_f16: bad epilogue %d", epi); return false;
    }
    if (e != cudaSuccess) {
        set_error("gemm_f16 launch: %s", cudaGetErrorString(e));
        return false;
    }
    return true;
}

// x_out[M, 384] = LayerNorm(A[M, K] . W[384, K]^T + bias + residual) * gamma + beta: gemm_f16_ln_pair_kernel (CTA pairs)
// for two row blocks or more, gemm_f16_ln_kernel (one CTA) for a single row block
bool gemm_f16_res_ln(cudaStream_t stream, const __half* A, const CUtensorMap* tmap_w, const __half* W, const float* bias,
                     const __half* residual, const float* gamma, const float* beta, float eps, __half* C, int M, int N, int K,
                     int num_sms) {
    if (M <= 0) return true;
    if (N != 2 * GEMM_BLOCK_N || K % BLOCK_K != 0 || K <= 0 || !residual || !gamma || !beta) {
        set_error("gemm_f16_res_ln: unsupported shape M=%d N=%d K=%d (N must be %d)", M, N, K, 2 * GEMM_BLOCK_N);
        return false;
    }
    CUtensorMap ta, tb_local, tc, tr;
    if (!make_tmap_f16_2d(&ta, A, (uint64_t)M, (uint64_t)K, BLOCK_M, BLOCK_K)) return false;
    if (!make_tmap_f16_2d(&tc, C, (uint64_t)M, (uint64_t)N, 32, 32)) return false;
    if (!make_tmap_f16_2d(&tr, residual, (uint64_t)M, (uint64_t)N, 32, 32)) return false;
    const int num_m = (M + BLOCK_M - 1) / BLOCK_M;
    int dev = 0;
    cudaGetDevice(&dev);
    const bool dev_ok = dev >= 0 && dev < 256;
    if (num_m >= 2) {
        // CTA pairs (cta_group::2): each CTA loads half of the W rows of a panel -> its own tensor map (96-row boxes)
        constexpr int PAIR_STAGES = 4;
        using L = GemmLnSmem<GEMM_BLOCK_N, PAIR_STAGES, true>;
        if (!make_tmap_f16_2d(&tb_local, W, (uint64_t)N, (uint64_t)K, GEMM_BLOCK_N / 2, BLOCK_K)) return false;
        auto kern = gemm_f16_ln_pair_kernel<GEMM_BLOCK_N, PAIR_STAGES>;
        static thread_local int attr_dev_mask[8] = {0};
        static thread_local int max_clusters[256] = {0};
        if (!dev_ok || !(attr_dev_mask[dev >> 5] & (1 << (dev & 31)))) {
            cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, L::TOTAL);
            if (e != cudaSuccess) { set_error("gemm_f16_res_ln (pair): %s", cudaGetErrorString(e)); return false; }
            if (dev_ok) {
                attr_dev_mask[dev >> 5] |= 1 << (dev & 31);
                cudaLaunchConfig_t cfg = {};
                cfg.gridDim = dim3(num_sms & ~1);
                cfg.blockDim = dim3(GEMM_THREADS);
                cfg.dynamicSmemBytes = L::TOTAL;
                int n = 0;
                if (cudaOccupancyMaxActiveClusters(&n, kern, &cfg) == cudaSuccess && n > 0) max_clusters[dev] = n;
                else { cudaGetLastError(); max_clusters[dev] = num_sms / 2; }
            }
        }
        int pairs = dev_ok ? max_clusters[dev] : num_sms / 2;  // co-resident pairs: the kernel is persistent
        if (pairs > num_sms / 2) pairs = num_sms / 2;
        if (pairs > (num_m + 1) / 2) pairs = (num_m + 1) / 2;
        kern<<<2 * pairs, GEMM_THREADS, L::TOTAL, stream>>>(ta, tb_local, tc, tr, bias, gamma, beta, eps, M, K);
        cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) { set_error("gemm_f16_res_ln (pair) launch: %s", cudaGetErrorString(e)); return false; }
        return true;
    }
    constexpr int LN_STAGES = 3;
    using L = GemmLnSmem<GEMM_BLOCK_N, LN_STAGES, false>;
    if (!tmap_w) {
        if (!make_tmap_f16_2d(&tb_local, W, (uint64_t)N, (uint64_t)K, GEMM_BLOCK_N, BLOCK_K)) return false;
        tmap_w = &tb_local;
    }
    auto kern = gemm_f16_ln_kernel<GEMM_BLOCK_N, LN_STAGES>;
    static thread_local int attr_dev_mask[8] = {0};
    if (!dev_ok || !(attr_dev_mask[dev >> 5] & (1 << (dev & 31)))) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, L::TOTAL);
        if (e != cudaSuccess) { set_error("gemm_f16_res_ln: %s", cudaGetErrorString(e)); return false; }
        if (dev_ok) attr_dev_mask[dev >> 5] |= 1 << (dev & 31);
    }
    const int grid = num_m < num_sms ? num_m : num_sms;
    kern<<<grid, GEMM_THREADS, L::TOTAL, stream>>>(ta, *tmap_w, tc, tr, bias, gamma, beta, eps, M, K);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { set_error("gemm_f16_res_ln launch: %s", cudaGetErrorString(e)); return false; }
    return true;
}

int gemm_block_n() { return GEMM_BLOCK_N; }

}  // namespace lb2
