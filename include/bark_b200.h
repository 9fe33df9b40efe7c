/* bark_b200.h — additive C entry points of libbark_b200 (nothing here exists in the reference header).
 *
 * They expose, through the same C-ABI shared library, the per-call pieces the reference keeps file-static,
 * so that parity tests and the benchmark can drive and time one step of the hot path with HOST buffers:
 *
 *   bark_b200_gpt_eval ........ one causal GPT evaluation  == bark_eval_encoder_internal      (bark.cpp:1586-1643)
 *   bark_b200_fine_eval ....... one fine pass              == bark_eval_fine_encoder_internal (bark.cpp:1907-1959)
 *   bark_b200_encodec_decode .. codes -> waveform          == encodec_decompress_audio        (encodec.cpp/encodec.cpp:902-924)
 *   bark_b200_sample .......... gpt_sample on the context RNG                                 (bark.cpp:249-270)
 *   bark_b200_sample_rows ..... the same for `rows` logit rows, on the device sampler the stages use (host replay of rows it cannot decide)
 *   bark_b200_forward_* ....... extern "C" names for bark_forward_{text,coarse,fine}_encoder  (bark.cpp:1703,1865,2061)
 *   bark_b200_tokenize ........ bark_tokenize_input                                           (bark.cpp:622-662)
 *
 * plus device selection for one-context-per-GPU batching (SURVEY.md §8e): bark_context_params must keep the
 * reference layout, so the device is chosen by bark_b200_set_device() or the BARK_B200_DEVICE environment
 * variable before bark_load_model.
 */
#pragma once
#include "bark.h"

#ifdef __cplusplus
extern "C" {
#endif

BARK_API void bark_b200_set_device(int cuda_device);                       /* applies to subsequent bark_load_model calls */
BARK_API const char * bark_b200_version(void);

/* which: 0 semantic, 1 coarse.  Host pointers.  *n_past advances exactly like the reference (by 257 for the merged prompt). */
BARK_API int  bark_b200_gpt_eval(struct bark_context * ctx, int which, const int32_t * tokens, int n, int * n_past, int merge_ctx, float * logits_out);
/* in_buffer: [8][1024] ids; nn: codebook being predicted (2..7); logits_out: [1024][n_out_vocab] */
BARK_API int  bark_b200_fine_eval(struct bark_context * ctx, const int32_t * in_buffer, int nn, float * logits_out);
/* codes: [8][n_frames]; returns number of samples (320 * n_frames), copies min(n, out_cap) floats to out (may be NULL) */
BARK_API int  bark_b200_encodec_decode(struct bark_context * ctx, const int32_t * codes, int n_frames, float * out, int out_cap);
BARK_API int  bark_b200_sample(struct bark_context * ctx, int which, const float * logits, int n, float temp, float * eos_p);
BARK_API int  bark_b200_sample_rows(struct bark_context * ctx, const float * logits /*[rows][n], host*/, int n, int rows, float temp, int32_t * tokens_out,
                                     float * eos_p_out /*[rows] or NULL*/);   /* returns the number of rows replayed on the host, <0 on error */
BARK_API void bark_b200_reseed(struct bark_context * ctx, uint32_t seed);
BARK_API void bark_b200_tokenize(struct bark_context * ctx, const char * text, int32_t * out513);

BARK_API bool bark_b200_forward_text_encoder(struct bark_context * ctx, int n_threads);
BARK_API bool bark_b200_forward_coarse_encoder(struct bark_context * ctx, int n_threads);
BARK_API bool bark_b200_forward_fine_encoder(struct bark_context * ctx, int n_threads);

/* stage: 0 semantic [n], 1 coarse [T][2], 2 fine [T][8], 3 prompt [513].  Returns the element count. */
BARK_API int  bark_b200_get_tokens(struct bark_context * ctx, int stage, int32_t * out, int cap);
BARK_API void bark_b200_set_tokens(struct bark_context * ctx, int stage, const int32_t * in, int n);
/* per_model9: {predict_us, sample_us, n_sample} x {semantic, coarse, fine} */
BARK_API void bark_b200_get_stats(struct bark_context * ctx, struct bark_statistics * out, int64_t * per_model9);
BARK_API void bark_b200_get_hparams(struct bark_context * ctx, int which, int32_t * out10);
BARK_API unsigned long long bark_b200_kernel_launches(void);               /* kernels launched by this library so far */
BARK_API unsigned bark_b200_layernorm_fallbacks(struct bark_context * ctx); /* LayerNorm rows replayed sequentially (DESIGN.md) */

/* measurement hooks used by bench.py */
BARK_API void bark_b200_profile_enable(int on);                            /* CUDA-event timing of every kernel launch; clears previous records */
BARK_API int  bark_b200_profile_report(char * buf, int cap);               /* JSON {kernel: {launches, ms, work}}; returns bytes needed */
BARK_API void bark_b200_io_counters(unsigned long long * h2d_bytes, unsigned long long * d2h_bytes, int reset);
/* with BARK_B200_DECODE_TIMING=1 in the environment at load: %globaltimer stamps [256][32] of the last decode step (rows 0..L: the
 * stamping thread of CTA 0 per layer; rows 64 + cta: every CTA at layer 5; slot meaning in tools/decode_timing.py) */
BARK_API int  bark_b200_decode_timing(struct bark_context * ctx, unsigned long long * out, int n);
/* the decode kernel's self-tuned head starts before the first poll of each exchange, [n_cta][8] nanoseconds; which: 0 semantic, 1 coarse */
BARK_API int  bark_b200_decode_adapt(struct bark_context * ctx, int which, unsigned * out, int n);


/* ROW-SHARDED FINE STAGE (BASELINE configs[4]; csrc/shard.cu): one process per GPU; every rank loads the same file and the same coarse
 * tokens, evaluates rows [rank * 1024 / world, ...) of each fine pass, stores its K / V rows into the peers' buffers over NVLink from
 * the QKV mat-mul's epilogue, and ends with the full fine token array, bit-identical to the single-GPU run.
 *   1. bark_b200_shard_init(ctx, rank, world, handle64)   -> 64-byte CUDA IPC handle of this rank's exchange buffer
 *   2. (caller all-gathers the handles, e.g. torch.distributed)
 *   3. bark_b200_shard_connect(ctx, all_handles)           -> maps the peers' buffers; bark_b200_forward_fine_encoder is sharded from here on */
BARK_API int  bark_b200_shard_init(struct bark_context * ctx, int rank, int world, void * handle_out);
BARK_API int  bark_b200_shard_connect(struct bark_context * ctx, const void * all_handles);
BARK_API unsigned long long bark_b200_shard_nvlink_bytes(struct bark_context * ctx, int reset);

/* FAST MODE (BARK_B200_MODE=fast in the environment at load; opt-in, NOT bit-identical to the reference): the fine model's
 * 1024-row passes (bark.cpp:1416-1584) run as tcgen05 tensor-core GEMMs + flash-style attention (csrc/fast_kernels.cu).
 * The two kernel hooks below run on host buffers without a context, for the numerics tests:
 *   bark_b200_fast_gemm ....... C[M][N] (f32) = A[M][K] (f16 bits) * W[N][K]^T (f16 bits), K % 64 == 0
 *   bark_b200_fast_attention .. out[n][E] (f16 bits) = soft_max(Q K^T / 8) V per 64-wide head, non-causal, n % 256 == 0 */
BARK_API int  bark_b200_fast_mode(struct bark_context * ctx);              /* 1 if this context runs the fast fine passes */
BARK_API int  bark_b200_fast_gemm(const uint16_t * A, const uint16_t * W, float * C, int M, int N, int K);
BARK_API int  bark_b200_fast_attention(const uint16_t * q, const uint16_t * k, const uint16_t * v, uint16_t * out, int n, int E, int H);

/* BATCHED GENERATION on the context's GPU (csrc/batch.cu).  Item i's semantic / coarse / fine ids and waveform are bit-identical to
 * bark_load_model(same file, same params, seeds[i]) followed by ONE bark_generate_audio(texts[i]).  1 <= n <= 32.  The semantic and coarse
 * decode steps of all items run as one batched step; the fine and EnCodec stages run item by item.  The call leaves the context's
 * single-prompt state alone (RNG, token arrays, bark_get_audio_data, statistics) and reports no progress.  Returns false (message on
 * stderr) on bad arguments, a sharded context, unsupported audio parameters or too little device memory. */
BARK_API bool bark_b200_generate_audio_batch(struct bark_context * ctx, const char * const * texts, const uint32_t * seeds, int n);
BARK_API int  bark_b200_batch_audio(struct bark_context * ctx, int item, float * out, int cap);                 /* sample count, copies min(count, cap); -1 on a bad item */
BARK_API int  bark_b200_batch_tokens(struct bark_context * ctx, int item, int stage, int32_t * out, int cap);  /* stage as bark_b200_get_tokens (0, 1, 2) */
/* test hook: teacher-forced batched decode.  which: 0 semantic, 1 coarse.  Every item's `len` prompt ids are evaluated into the
 * item's own KV cache (n_past 0, no merge), then `steps` batched single-token steps with next[i][j]; logits_out [n][steps][n_out_vocab].
 * Returns 1, or 0 on failure. */
BARK_API int  bark_b200_batch_eval(struct bark_context * ctx, int which, int n, const int32_t * prompts /*[n][len]*/, int len,
                                   const int32_t * next /*[n][steps]*/, int steps, float * logits_out);
/* the last batch call: {semantic, coarse, fine, EnCodec} microseconds, batched decode steps, sampled rows replayed on the host */
BARK_API int  bark_b200_batch_stats(struct bark_context * ctx, int64_t * out6);

#ifdef __cplusplus
}
#endif
