// bark_context: everything one generation needs, owned by bark_load_model / bark_free.
// Host control plane in C++ (like the reference's bark.cpp:133-164), all tensors in HBM.
#pragma once
#include "../../include/bark.h"
#include "model.h"

#include <map>
#include <random>
#include <string>
#include <vector>

// row-sharded fine stage (shard.cu): this rank's IPC-exported buffer and the peers' mapped ones
struct ShardState {
    bool on = false; int rank = 0, world = 1;
    unsigned char * local = nullptr, * peer[8] = {nullptr};
    unsigned epoch = 0; unsigned * d_err = nullptr;
    unsigned long long nvlink_bytes = 0;             // bytes this rank stored into peer memory (K / V rows, sampled ids)
};

// batched generation on the context's GPU (batch.cu): per-item KV caches, step scratch, and the results of the last batch call
struct BatchItem { std::vector<int32_t> semantic, coarse, fine; std::vector<float> audio; };
struct BatchState {
    float * kv = nullptr; size_t slot_floats = 0; int slots = 0;   // one K + V cache region per item, sized for the larger causal model
    float * qkv = nullptr, * logits = nullptr;                      // step scratch: [32][3E] QKV rows, [32][n_out] logit rows
    double * h_u = nullptr, * d_u = nullptr;                        // sampling buffers of the batch (the single-prompt ones stay untouched)
    int32_t * h_tok = nullptr, * d_tok = nullptr, * h_flags = nullptr, * d_flags = nullptr;
    float * h_eos = nullptr, * d_eos = nullptr;
    long long n_sample_calls = 0;
    std::vector<BatchItem> items;                                   // results of the last successful bark_b200_generate_audio_batch
    int64_t stats[6] = {0, 0, 0, 0, 0, 0};                          // its semantic / coarse / fine / codec microseconds, batched steps, host replays
};

struct bark_context {
    int device = 0;
    cudaStream_t stream = nullptr;

    bark::GPTModel semantic, coarse, fine;
    bark::CodecModel codec;
    std::map<std::string, int32_t> token_to_id;      // WordPiece vocabulary (bark.cpp:664-690)

    __half * d_gelu_tab = nullptr;                   // 65536-entry table, ggml.c:3795-3810
    unsigned * d_ln_fallbacks = nullptr;             // [0] LayerNorm rows, [1] soft_max rows replayed sequentially
    unsigned tag_base = 0;                           // epoch counter of the decode kernel's tagged exchanges (advances 6*L per token)
    int n_sm = 0, n_sm_total = 0; bool use_decode_kernel = true;   // n_sm: CTAs of the persistent decode kernel (knob); n_sm_total: SMs of the device
    bool kv_reuse = true; unsigned long long n_kv_reused = 0;   // coarse windows start from the cached prefix (bark_api.cu run_coarse)
    // decode-kernel knobs (BARK_B200_DECODE_TIMING_TID / BARK_B200_POLL_NS / BARK_B200_POLL_FIRST_NS); defaults from the measured sweep
    // in profiles/r01_decode_knob_sweep.md: 40 ns back-off between polls, 500 ns head start for the two residual exchanges
    bool kv_prefetch = false;          // BARK_B200_KV_PREFETCH=1: bulk L2 prefetch of the next layer's K / V rows inside the decode step
    bool fuse_sampler = false; unsigned * d_done_counter = nullptr;  // BARK_B200_FUSE_SAMPLER=1: the decode kernel samples its own token (6411 instead of 8037 launches per clip; 233.3 vs 233.7 ms: neutral, so off)
    bool decode_cluster = false;                     // BARK_B200_DECODE=cluster: the decode step inside one 16-CTA cluster (decode_kernels.cu) where the model fits
    bool gemm_f32c = false;                          // BARK_B200_GEMM_F32C=1: multi-row passes of f16 models keep operands as f16 values in f32 containers
    bool adapt_on = false;                           // BARK_B200_ADAPT=1: self-tuning head starts instead of the fixed knobs below (measured worse, see decode_kernels.cu)
    unsigned headstart[6] = {0, 2000, 500, 400, 500, 0};   // BARK_B200_HEADSTART=q:att:x1:ff:x2:scores (ns): sleep before the first poll of each exchange
    int timing_tid = 0; unsigned poll_ns = 40, first_ns = 500, att_ns = 2000;   // att_ns (BARK_B200_POLL_ATT_NS): head start before CTAs without a soft_max tile poll for the attention output
    unsigned long long * d_timing = nullptr;         // optional phase timestamps of the decode kernel (BARK_B200_DECODE_TIMING=1)

    // BARK_B200_MODE=fast: the fine model's passes run on the tensor cores (fast_kernels.cu); not bit-identical to the reference
    bool fast_mode = false;
    __half * f_a16 = nullptr, * f_h16 = nullptr, * f_qk16 = nullptr, * f_vt16 = nullptr, * f_att16 = nullptr;   // [1024][E], [1024][4E], [1024][2E], [E][1024], [1024][E]

    ShardState shard;
    BatchState batch;

    bark::Workspace ws;
    void * d_q8_sums = nullptr;                       // experimental q4_1 / q5_1: q8_1 block sums s = f16(d * sum(q))
    void * d_q8 = nullptr, * d_q8_scales = nullptr;  // q4_0 models: q8_0 activation operand (int8 [rows][4E], f32 scales [rows][4E/32])
    const float * last_logits = nullptr;             // device logits of the latest gpt_eval / fine_eval
    double * d_u = nullptr, * h_u = nullptr;         // device sampling: uniforms, tokens, flags, eos probabilities (1024 rows)
    int32_t * d_stok = nullptr, * h_stok = nullptr, * d_sflags = nullptr, * h_sflags = nullptr;
    float * d_seos = nullptr, * h_seos = nullptr;
    int32_t * d_feed = nullptr;                      // token handed from sample_rows_kernel to the next decode step
    bool sample_on_device = true; long long n_sample_host_replays = 0;
    int debug_flag_every = 0; long long n_sample_calls = 0;   // BARK_B200_SAMPLE_FLAG_EVERY=k: force every k-th sample through the host replay (tests)
    float * h_logits = nullptr;                      // pinned, max(n_out) or 1024*fine_vocab
    int32_t * h_tok = nullptr;                       // pinned, 8*1024 ids

    // codec scratch
    float * c_buf[3] = {nullptr, nullptr, nullptr}; size_t c_cap = 0;   // ping-pong activations (floats)
    float * c_gi = nullptr;                                            // LSTM input projections
    float * c_hbuf = nullptr; unsigned * c_counter = nullptr;          // LSTM hidden-state exchange + grid barrier counter
    int32_t * d_codes = nullptr;

    std::mt19937 rng;                                // seeded once at load (bark.cpp:1179)

    std::vector<int32_t> tokens;                     // 513 prompt ids
    std::vector<int32_t> semantic_tokens;
    std::vector<int32_t> coarse_tokens;              // [T][2] flattened
    std::vector<int32_t> fine_tokens;                // [T][8] flattened
    std::vector<float> audio;

    bark_context_params params;
    bark_statistics stats{};

    std::vector<void *> device_allocs;               // everything cudaMalloc'ed for this context
};

namespace bark {

// loader.cu
bool load_model_file(const std::string & path, bark_context * ctx);
void * ctx_alloc(bark_context * ctx, size_t bytes);

// gpt_forward.cu — one evaluation of a causal model; mirrors bark_eval_encoder_internal (bark.cpp:1586-1643)
// logits [lm_lo, lm_hi) are computed and copied to logits_host + lm_lo (lm_hi <= 0: all of them)
// kv_k / kv_v: the [L][block_size][E] K / V cache to work on (null: the model's own, mem_k / mem_v)
bool gpt_eval(bark_context * ctx, GPTModel & m, const int32_t * tokens, int n, int * n_past, bool merge_ctx, float * logits_host, int lm_lo = 0, int lm_hi = 0,
              float * kv_k = nullptr, float * kv_v = nullptr);
void build_decode_tables(bark_context * ctx, GPTModel & m);
// one non-causal pass of the fine model; mirrors bark_eval_fine_encoder_internal (bark.cpp:1907-1959)
bool fine_eval(bark_context * ctx, const int32_t * in_buffer /*[8][1024]*/, int nn, float * logits_host /*[1024][n_out]*/);
bool fine_eval_shard(bark_context * ctx, const int32_t * in_buffer, int nn);                          // this rank's rows of one pass (shard.cu)
bool sample_shard(bark_context * ctx, int n, float temp, int32_t * out_all /*[1024]*/);
bool fine_eval_fast(bark_context * ctx, const int32_t * in_buffer, int nn, float * logits_host);      // tensor-core variant (fast mode)
// EnCodec decode; codes [8][T] on the host; result in ctx->audio
bool codec_decode(bark_context * ctx, const int32_t * codes, int T);

// sampling.cu / gpt_forward.cu / bark_api.cu
void sample_rows(const float * logits, int ld, int n, int rows, float temp, const double * d_u, int32_t * d_out_tok, int tok_add, int32_t * d_feed,
                 float * d_eos_p, int32_t * d_flags, int force_flag, cudaStream_t s);
// fs != null: the decode kernel also samples the token (fused sampler), leaving it in fs->d_tok / fs->d_feed
struct FusedSample { int n; float temp; const double * d_u; int32_t * d_tok; int tok_add; int32_t * d_feed; float * d_eos; int32_t * d_flags; int force; };
bool fused_sampler_available(const bark_context * ctx, const GPTModel & m, int samp_n);
bool gpt_decode_chained(bark_context * ctx, GPTModel & m, const int32_t * d_token, int * n_past, int lm_lo, int lm_hi, const FusedSample * fs = nullptr);
bool sample_device(bark_context * ctx, GPTModel & m, const float * d_logits, int ld, int n, int rows, float temp, int32_t * out_tok, float * out_eos);
struct SampleBufs { double * h_u, * d_u; int32_t * h_tok, * d_tok, * h_flags, * d_flags; float * h_eos, * d_eos; };   // pinned host / device, one entry per row
void sample_rows_sync(bark_context * ctx, const SampleBufs & b, const float * d_logits, int ld, int n, int rows, float temp, int tok_add, int force,
                      int32_t * out_tok, float * out_eos, long long * replays);
int32_t sample_token_given_u(const float * logits, int n, float temp, double u, float * eos_p);

int64_t now_us();

// bark_api.cu — stage pieces shared by the single-prompt stage loops and the batched ones (batch.cu)
void tokenize_input(bark_context * ctx, const std::string & text);                  // -> ctx->tokens (513 ids)
bool semantic_stop(const bark_context_params & P, int32_t tok, float eos_p);        // the semantic loop's stop test (bark.cpp:1675-1677)
struct CoarsePlan { float stc_ratio; int max_semantic_history, n_steps, n_windows; };
bool coarse_plan(const bark_context_params & P, size_t n_semantic, CoarsePlan * cp);     // false (with a message) when there is nothing to generate
// ids to evaluate for the coarse window that starts after the samples in `out`, with prefix reuse against the cache content kv_ids /
// kv_canon (updated for the window); *n_past = cached rows the evaluation starts from
std::vector<int32_t> coarse_window_input(const bark_context_params & P, const CoarsePlan & cp, const std::vector<int32_t> & sem, const std::vector<int32_t> & out,
                                         bool kv_reuse, std::vector<int32_t> & kv_ids, size_t & kv_canon, int * n_past);
int  coarse_lo(const bark_context_params & P, int step);                            // offset of coarse step `step`'s codebook window in the vocabulary
void coarse_codes(const bark_context_params & P, const std::vector<int32_t> & out, std::vector<int32_t> & codes);   // samples -> [T][2] codes
bool run_fine(bark_context * ctx);                                                  // ctx->coarse_tokens -> ctx->fine_tokens, drawing from ctx->rng
bool audio_params_supported(const bark_context_params & P);
bool fine_to_audio(bark_context * ctx);                                             // ctx->fine_tokens -> ctx->audio (EnCodec)

}  // namespace bark
