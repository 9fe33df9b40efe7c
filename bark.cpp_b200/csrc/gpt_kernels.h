// Host-callable launchers of the GPT kernels (gpt_kernels.cu, decode_kernels.cu).
#pragma once
#include "model.h"

namespace bark {

enum EpiMode : int { EPI_STORE = 0, EPI_RESID = 1, EPI_GELU_ACT = 2, EPI_QKV = 3 };

struct MatmulEpilogue {
    int mode = EPI_STORE;
    float * out = nullptr; int ldo = 0;              // STORE / RESID target ([m][ldo]); QKV: q rows with ldo = E
    float * k_out = nullptr, * v_out = nullptr;      // QKV: K/V rows (KV cache slot of the first new position, or the fine model's buffers)
    // row-sharded fine pass (shard.cu): the same K/V rows are also stored into the other GPUs' buffers over NVLink (peer pointers),
    // so the all-gather of K and V is the mat-mul's own epilogue
    int n_peer = 0; float * k_peer[7] = {nullptr}, * v_peer[7] = {nullptr};
    void * act_out = nullptr; int act_wt = 0, act_Kp = 0;   // GELU_ACT: operand for the following mul_mat (act_Kp = its group stride)
    const __half * gelu_tab = nullptr;
};

void permute_to_li(const void * src_rowmajor, void * dst_li, int n_out, int K, WType t, cudaStream_t s);
void permute_to_gm(const void * src_rowmajor, void * dst_gm, int n_out, int o_pad, int K, WType t, cudaStream_t s);

void gpt_embed_causal(const GPTModel & m, const int32_t * d_tok, int N, int n_past, bool merge, float * x, cudaStream_t s);
void gpt_embed_fine(const GPTModel & m, const int32_t * d_ids, int nn, float * x, cudaStream_t s, int row0 = 0, int rows = 1024);   // rows [row0, row0 + rows) of the window

// `Kp` of the activation operands below is the GROUP STRIDE of the group-major layout (elements), not a row length
void layernorm_act(const float * x, int rows, int E, const float * g, const float * b, void * act, WType wt, int Kp,
                   unsigned * fallback_counter, cudaStream_t s);

void lane_matmul(const DMat & W, const void * act, int act_gs, int rows, const MatmulEpilogue & ep, cudaStream_t s, bool f32_containers = false);

void attention(const float * Q, const float * Kc, const float * Vc, int N, int n_kv, int n_past, int E, int H, bool causal,
               float * scores, void * act, WType wt, int Kp, cudaStream_t s);

// ---- q4_0 weights (q4_kernels.cu) ---------------------------------------------------------------------------------
void q4_split(const void * raw_blocks, size_t n_blocks, void * qs, void * scales, cudaStream_t s);
void q4_set_scratch(void * q8, void * q8_scales);      // int8 [rows][K] + f32 [rows][K/32] for the activation operand, owned by the context
void q4_matmul(const DMat & W, const void * act_f32, int ld_act, int rows, const MatmulEpilogue & ep, cudaStream_t s);

// ---- q4_1 / q5_0 / q5_1 / q8_0 weights (qx_kernels.cu) ---------------------------------------------------------------------------
bool   qx_supported(WType t);
size_t qx_block_bytes(WType t);
void   qx_split(const void * raw_blocks, size_t n_blocks, WType t, void * qs, void * qh, void * d, void * m, cudaStream_t s);
void   qx_set_scratch(void * q8, void * q8_scales, void * q8_sums);
void   qx_embed_causal(const GPTModel & m, const int32_t * d_tok, int N, int n_past, bool merge, float * x, cudaStream_t s);
void   qx_embed_fine(const GPTModel & m, const int32_t * d_ids, int nn, float * x, cudaStream_t s);
void   qx_matmul(const DMat & W, const void * act_f32, int ld_act, int rows, const MatmulEpilogue & ep, cudaStream_t s);

// ---- register-tiled multi-row kernels (gemm_kernels.cu) ------------------------------------------------------------
void lane_gemm_tiled(const DMat & W, const void * act, int act_gs, int rows, const MatmulEpilogue & ep, cudaStream_t s, bool f32_containers = false);
void expand_f16_to_f32(const void * src_f16, void * dst_f32, size_t n, cudaStream_t s);
void attention_tiled_scores(const float * Q, const float * Kc, int N, int n_kv, int n_past, int E, int H, float scale, bool causal, float * scores, cudaStream_t s);
void attention_tiled_pv(const float * scores, const float * Vc, int N, int n_kv, int E, int H, void * act, WType wt, int Kp, cudaStream_t s);

// ---- fast mode (fast_kernels.cu, BARK_B200_MODE=fast): tcgen05 GEMM + flash-style attention for the dense passes -------------------
enum { FEPI_F32 = 0, FEPI_RESID = 1, FEPI_GELU16 = 2, FEPI_F16 = 3, FEPI_QKV16 = 4 };
struct FastEpi {
    int mode = FEPI_F32;
    float * out32 = nullptr; __half * out16 = nullptr; int ldo = 0;      // row-major targets
    __half * vt = nullptr; int vt_ld = 0, v_col0 = 0;                    // QKV16: columns >= v_col0 are written transposed, vt[(n - v_col0) * vt_ld + m]
    const __half * gelu_tab = nullptr;
};
bool fast_gemm(const __half * A, int lda, const __half * W, int ldw, int M, int N, int K, const FastEpi & ep, int n_sm, cudaStream_t s);
bool fast_attention(const __half * qk, int ldq, int k_col0, const __half * vt, int n, int E, int H, __half * out, cudaStream_t s);
void fast_layernorm(const float * x, int rows, int E, const float * g, const float * b, __half * out, cudaStream_t s);

// ---- batched decode step (batch_kernels.cu; driven by batch.cu): B <= kBatchMax items, one new position each, all at the same n_past ----
constexpr int kBatchMax = 32;                        // one row tile (kBM) of lane_gemm_tiled_kernel: every mat-mul of a step is one row tile
struct RowIds { int32_t v[kBatchMax]; };             // one input id per row, passed by value
struct BatchKV { float * k[kBatchMax]; float * v[kBatchMax]; };   // per row: the item's K / V cache of the current layer, [block_size][E] f32
// x[b] = wte[tok[b]] + wpe[pos] for rows b < B (every weight type the loader accepts)
void gpt_embed_rows(const GPTModel & m, const RowIds & tok, int B, int pos, float * x, cudaStream_t s);
void qx_embed_rows(const GPTModel & m, const RowIds & tok, int B, int pos, float * x, cudaStream_t s);
// one layer's attention for B decode rows: appends each row's K / V slice (qkv [B][3E]) to its cache at n_past, then scores, soft_max
// and P.V over n_past + 1 keys in the reference's order; the result goes to the next mat-mul's operand (store_act)
void batch_decode_attention(const float * qkv, const BatchKV & kv, int B, int n_past, int E, int H, void * act, WType wt, int Kp,
                            unsigned * softmax_fallbacks, cudaStream_t s);

// ---- persistent decode step (decode_kernels.cu) -----------------------------------------------------------------
constexpr int kDecodeReplicas = 8;        // copies of each all-to-all exchange vector (gx, gq, gatt, gff): CTA c reads copy c % 8
struct DecodePhase { const void * w; int n_out, row_bytes, K, pad; const void * ws; };   // one streamed matrix: LI rows (f32 / f16), or q4_0 nibble words (16 B per block) with f16 block scales in ws
struct DecodeLayerVec { const float * ln_1_g, * ln_1_b, * ln_2_g, * ln_2_b; };
struct DecodeArgs {
    const DecodePhase * phases;          // [4L + 1]: per layer c_attn, c_proj, c_fc, mlp/c_proj; then lm_head
    const DecodeLayerVec * layer_vecs;   // [L]
    const void * wte; const float * wpe; const float * ln_f_g, * ln_f_b; const __half * gelu_tab;
    float * mem_k, * mem_v;              // f32 KV cache [L][block_size][E]
    // cross-CTA exchange vectors in L2: 8-byte {float value, u32 epoch} words
    unsigned long long * gx, * gq, * gk, * gv, * gatt, * gff, * gscores;
    float * logits;
    unsigned tag_base; unsigned * ln_fallbacks;
    unsigned long long * timing;         // optional [256][32] globaltimer stamps (debug, decode_kernels.cu tstamp)
    int E, H, L, block_size, n_past, token, lm_lo, lm_hi;
    const int32_t * token_ptr; int n_vocab_in;   // token_ptr != null: read the input token from device memory (written by sample_rows_kernel), clamped to the vocabulary
    double inv_E;                        // 1.0 / E (double), for the division-free LayerNorm decision
    // fused sampler (samp_n > 0): the CTA that finishes its lm_head rows last samples the token from logits [lm_lo, lm_lo + samp_n)
    // (sampling.cuh) — one launch per token instead of two
    int samp_n; float samp_temp; const double * samp_u; int32_t * samp_tok; int samp_tok_add; int32_t * samp_feed; float * samp_eos; int32_t * samp_flags; int samp_force;
    unsigned * done_counter;
    unsigned headstart[6];               // fixed head start (ns) before the first poll of each exchange: q, att (CTAs without a soft_max tile), x1, ff, x2, scores
    int kv_prefetch;                     // 1: every CTA asks the TMA engine to pull its slice of the NEXT layer's K / V rows into L2 (cp.async.bulk.prefetch.L2) one layer ahead
    unsigned * adapt;                    // [n_cta][8] adaptive head starts of the exchanges, carried from token to token (null: fixed knobs)
    int timing_tid; unsigned poll_ns, first_ns, att_ns;   // debug: stamping thread; back-off between polls of the tagged words; delay before the first poll of the residual exchanges (ns)
};
int  decode_tags_per_step(int n_layer);
void launch_decode_step(const DecodeArgs & args, WType wt, int n_sm, cudaStream_t s);
// the same token inside one 16-CTA cluster (DSMEM exchanges, no polling); see decode_kernels.cu
bool decode_cluster_supported(const DecodeArgs & args, WType wt, int max_row_bytes);
void launch_decode_cluster(const DecodeArgs & args, WType wt, cudaStream_t s);

}  // namespace bark
