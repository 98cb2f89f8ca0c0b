// Internal declarations shared by the translation units of libleann_b200.so.
#pragma once
#include <cuda.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace lb2 {

// thread-local last-error string behind lb2_last_error()
void set_error(const char* fmt, ...);

#define LB2_CUDA_OK(expr)                                                              \
    do {                                                                               \
        cudaError_t _e = (expr);                                                       \
        if (_e != cudaSuccess) {                                                       \
            lb2::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
            return false;                                                              \
        }                                                                              \
    } while (0)

enum Epilogue { EPI_BIAS = 0, EPI_BIAS_GELU = 1, EPI_BIAS_RES = 2 };

// ---- gemm_tcgen05.cu
bool make_tmap_f16_2d(CUtensorMap* map, const void* ptr, uint64_t rows, uint64_t cols, uint32_t box_rows,
                      uint32_t box_cols = 64);
bool make_tmap_f16_3d(CUtensorMap* map, const void* ptr, uint64_t row_elems, uint64_t rows, uint64_t groups, uint32_t box_cols,
                      uint32_t box_rows);
bool gemm_f16(cudaStream_t stream, const __half* A, const CUtensorMap* tmap_w, const __half* W, const float* bias,
              const __half* residual, __half* C, int M, int N, int K, int epi, int num_sms, int c_group = 0);
bool gemm_f16_res_ln(cudaStream_t stream, const __half* A, const CUtensorMap* tmap_w, const __half* W, const float* bias,
                     const __half* residual, const float* gamma, const float* beta, float eps, __half* C, int M, int N, int K,
                     int num_sms);
int gemm_block_n();
// optional per-kernel-class timing with CUDA events (api.cu owns the pools; no-ops unless
// LB2_PROFILE_GEMM=1): category 0 = tcgen05 GEMMs, 1 = attention, 2 = LayerNorm / embed / pool
enum ProfCat { PROF_GEMM = 0, PROF_ATTN = 1, PROF_NORM = 2, PROF_NCAT = 3 };
void prof_begin(cudaStream_t s, int cat);
void prof_end(cudaStream_t s, int cat, double flops);

// ---- encoder.cu
struct EncoderConfig {
    int vocab_size, hidden, layers, heads, ffn, max_pos, type_vocab;
    float ln_eps;
    int pooling;    // 0 = masked mean (all-MiniLM-L6-v2), 1 = CLS (bge-base-en-v1.5)
    int normalize;  // 1 = L2-normalise the pooled vector (both models ship a Normalize module)
};

struct LayerWeights {
    __half* w_qkv;  // [3H, H]
    float* b_qkv;   // [3H]
    __half* w_o;    // [H, H]
    float* b_o;
    float *ln1_g, *ln1_b;
    __half* w_1;  // [F, H]
    float* b_1;
    __half* w_2;  // [H, F]
    float* b_2;
    float *ln2_g, *ln2_b;
    CUtensorMap tm_qkv, tm_o, tm_1, tm_2;
};

struct Encoder {
    EncoderConfig cfg{};
    bool loaded = false;
    __half *word_emb = nullptr, *pos_emb = nullptr, *type_emb = nullptr;
    float *emb_ln_g = nullptr, *emb_ln_b = nullptr;
    LayerWeights* layers = nullptr;  // host array of device pointers
    void* arena = nullptr;           // one device allocation holding every tensor above
    // workspaces, sized for `cap_tokens` packed tokens / `cap_seqs` sequences
    int64_t cap_tokens = 0, cap_seqs = 0;
    __half *x = nullptr, *y = nullptr, *qkv = nullptr, *ctx = nullptr, *ffn = nullptr;
    int32_t* seq_len = nullptr;  // [cap_seqs] truncated passage lengths of the current pass
    int* att_items = nullptr;    // [cap_seqs * 8 + 1] attention work list of the pass + its length
    int num_sms = 148;
};

size_t encoder_weight_floats(const EncoderConfig& cfg);
bool encoder_load(Encoder* enc, const EncoderConfig& cfg, const float* host_weights, size_t n_floats);
void encoder_free(Encoder* enc);
bool encoder_reserve(Encoder* enc, int64_t tokens, int64_t seqs);
// whether each layer's residual projections fuse their LayerNorm (5 kernels per layer instead of 7)
bool encoder_fuses_ln(const EncoderConfig& cfg);
// Encode n_seq passages.  Passage i is node seq_node[i] of the token store (tok_store / tok_off,
// device pointers); its rows in the packed activation matrix start at seq_start[i] - row_base;
// n_tokens = packed row count.  Writes pooled (+normalised) fp32 embeddings to out[n_seq, H].
bool encoder_forward(Encoder* enc, cudaStream_t stream, const uint16_t* tok_store, const uint64_t* tok_off,
                     const int32_t* seq_node, const int32_t* seq_start, int row_base, int n_seq, int n_tokens,
                     float* out);

// kernels exposed for the unit-test hooks in api.cu
bool launch_layernorm(cudaStream_t s, const __half* in, const float* g, const float* b, __half* out, int rows,
                      int hidden, float eps);
// qkv is head-major: [heads][n_tokens][3 * head_dim] (q | k | v per token)
bool launch_attention(cudaStream_t s, const __half* qkv, const int32_t* seq_start, const int32_t* seq_len, int* items,
                      int* item_count, int row_base, int max_pos, int n_seq, int n_tokens, int hidden, int heads,
                      __half* ctx, bool build_items);

// ---- attention_tc.cu: tcgen05 attention (head_dim 32, passages <= 256 tokens)
bool attention_tc_supported(int hidden, int heads, int max_pos);
bool launch_attention_tc(cudaStream_t s, const __half* qkv, const int32_t* seq_start, const int32_t* seq_len, int* items,
                         int* item_count, int row_base, int n_seq, int n_tokens, int hidden, int heads, __half* ctx,
                         bool build_items, int num_sms);

}  // namespace lb2
