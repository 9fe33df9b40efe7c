// Per-call orchestration of the GPT and EnCodec kernels: the device-side replacement of
// bark_eval_encoder_internal (bark.cpp:1586-1643), bark_eval_fine_encoder_internal (bark.cpp:1907-1959)
// and encodec_eval (encodec.cpp/encodec.cpp:819-847).  No graph is built or allocated per step: the
// workspace is sized once at load for the worst case (block_size rows).
#include "codec_kernels.h"
#include "context.h"
#include "gpt_kernels.h"

#include <algorithm>
#include <vector>
#include <time.h>

namespace bark {

int64_t now_us() {
    timespec ts; clock_gettime(CLOCK_MONOTONIC, &ts);
    return (int64_t) ts.tv_sec * 1000000 + ts.tv_nsec / 1000;
}


// transformer body shared by the causal and the fine model; x [N][E] is updated in place.
// K/V rows of this call go to k_dst/v_dst (KV-cache slot of position n_past, or the fine model's scratch),
// attention then reads n_kv rows starting at k_all/v_all.  Causal models: mem_k / mem_v is the [L][block_size][E] cache
// the call works on (the model's own, or one item's of a batch, batch.cu).
static void run_layers(bark_context * ctx, GPTModel & m, int N, int n_past, bool causal, float * mem_k = nullptr, float * mem_v = nullptr) {
    Workspace & ws = ctx->ws;
    cudaStream_t s = ctx->stream;
    const int E = m.n_embd, H = m.n_head;
    const bool q4 = is_quant(m.wtype);                       // quantised weights: f32 activation rows, quantised to q8 blocks in front of each mat-mul
    const bool c32 = ctx->gemm_f32c && m.wtype == W_F16 && N >= 16;      // f16 values in f32 containers (tiled mat-mul only)
    const int awt = q4 ? (int) W_Q4_0 : c32 ? W_F16R32 : (int) m.wtype;  // what the activation producers are told (store_act)
    const int kpE = q4 ? E : ws.max_rows * kGmGroup, kp4E = q4 ? 4 * E : kpE;      // group stride of the group-major activation operands; q4_0: f32 row stride
    if (q4) { q4_set_scratch(ctx->d_q8, ctx->d_q8_scales); qx_set_scratch(ctx->d_q8, ctx->d_q8_scales, ctx->d_q8_sums); }
    for (int il = 0; il < m.n_layer; il++) {
        const GPTLayer & L = m.layers[(size_t) il];
        layernorm_act(ws.x, N, E, L.ln_1_g, L.ln_1_b, ws.act, (WType) awt, kpE, ctx->d_ln_fallbacks, s);
        float * k_all, * v_all, * k_dst, * v_dst; int n_kv;
        if (causal) {
            k_all = mem_k + (size_t) il * m.block_size * E; v_all = mem_v + (size_t) il * m.block_size * E;
            k_dst = k_all + (size_t) n_past * E; v_dst = v_all + (size_t) n_past * E; n_kv = n_past + N;      // bark.cpp:1294-1300
        } else {
            k_all = k_dst = ws.kbuf; v_all = v_dst = ws.vbuf; n_kv = N;
        }
        MatmulEpilogue qkv; qkv.mode = EPI_QKV; qkv.out = ws.q; qkv.ldo = E; qkv.k_out = k_dst; qkv.v_out = v_dst;
        lane_matmul(L.c_attn, ws.act, kpE, N, qkv, s, c32);
        attention(ws.q, k_all, v_all, N, n_kv, n_past, E, H, causal, ws.scores, ws.act, (WType) awt, kpE, s);
        MatmulEpilogue res; res.mode = EPI_RESID; res.out = ws.x; res.ldo = E;
        lane_matmul(L.c_proj, ws.act, kpE, N, res, s, c32);                                                             // + inpL
        layernorm_act(ws.x, N, E, L.ln_2_g, L.ln_2_b, ws.act, (WType) awt, kpE, ctx->d_ln_fallbacks, s);
        MatmulEpilogue ge; ge.mode = EPI_GELU_ACT; ge.act_out = ws.act2; ge.act_wt = (int) awt; ge.act_Kp = kp4E; ge.gelu_tab = ctx->d_gelu_tab;
        lane_matmul(L.fc, ws.act, kpE, N, ge, s, c32);
        lane_matmul(L.proj, ws.act2, kp4E, N, res, s, c32);                                                               // + inpFF
    }
}

// Phase table + exchange buffers of the persistent decode kernel (decode_kernels.cu), once per causal model.
void build_decode_tables(bark_context * ctx, GPTModel & m) {
    const int L = m.n_layer, E = m.n_embd;
    // Fixed capacities of gpt_decode_step_kernel: shared-memory vectors of 1024 (x, q / probabilities) and 4096 (activation operand)
    // floats, 128 phase slots, one soft_max tile per CTA (H * head/16 tiles).  A model outside them steps
    // through the per-op kernels instead (same results, slower) — never through a kernel it would overrun.
    const int D = E / m.n_head;
    m.decode_ok = E <= 1024 && 4 * E <= 4096 && 4 * L + 1 <= 128 && m.block_size <= 1024 && m.n_head * (D / 16) <= ctx->n_sm;
    if (!m.decode_ok) {
        fprintf(stderr, "bark_b200: model (n_embd %d, n_layer %d, n_head %d, block_size %d) exceeds the persistent decode kernel's capacities; decoding with the per-op kernels\n", E, L, m.n_head, m.block_size);
        return;
    }
    const size_t es = m.wtype == W_F16 ? 2 : 4;
    const bool q4 = m.wtype == W_Q4_0;
    std::vector<DecodePhase> ph((size_t) 4 * L + 1);
    std::vector<DecodeLayerVec> lv((size_t) L);
    auto set = [&](DecodePhase & p, const DMat & d) {        // q4_0: 16 nibble bytes per 32-element block, block scales in a second array
        p.w = d.p; p.n_out = d.n_out; p.K = d.K; p.row_bytes = q4 ? d.K / 2 : (int)(d.Kp * es); p.pad = 0; p.ws = q4 ? d.scales : nullptr;
    };
    for (int l = 0; l < L; l++) {
        const GPTLayer & G = m.layers[(size_t) l];
        set(ph[(size_t) 4 * l], G.c_attn); set(ph[(size_t) 4 * l + 1], G.c_proj); set(ph[(size_t) 4 * l + 2], G.fc); set(ph[(size_t) 4 * l + 3], G.proj);
        lv[(size_t) l] = DecodeLayerVec{G.ln_1_g, G.ln_1_b, G.ln_2_g, G.ln_2_b};
    }
    set(ph[(size_t) 4 * L], m.lm_head[0]);
    m.d_phases = ctx_alloc(ctx, ph.size() * sizeof(DecodePhase));
    m.d_layer_vecs = ctx_alloc(ctx, lv.size() * sizeof(DecodeLayerVec));
    BARK_CUDA_CHECK(cudaMemcpy(m.d_phases, ph.data(), ph.size() * sizeof(DecodePhase), cudaMemcpyHostToDevice));
    BARK_CUDA_CHECK(cudaMemcpy(m.d_layer_vecs, lv.data(), lv.size() * sizeof(DecodeLayerVec), cudaMemcpyHostToDevice));
    auto tagged = [&](size_t n) { void * p = ctx_alloc(ctx, n * 8); BARK_CUDA_CHECK(cudaMemset(p, 0, n * 8)); return (unsigned long long *) p; };   // epoch 0 = never published
    const size_t R = kDecodeReplicas;                         // vectors every CTA gathers exist in R copies (decode_kernels.cu)
    m.gx = tagged(R * E); m.gq = tagged(R * E); m.gk = tagged((size_t) E); m.gv = tagged((size_t) E); m.gatt = tagged(R * E);
    m.gff = tagged(R * 4 * E); m.gscores = tagged((size_t) m.n_head * m.block_size);
    m.glogits = (float *) ctx_alloc(ctx, (size_t) m.n_out_vocab * 4);
    {   // adaptive head starts, [n_cta][8] (XT_* order: q, att, x1, ff, x2, scores): start from the measured fixed knobs
        std::vector<unsigned> init((size_t) ctx->n_sm_total * 8, 0u);
        for (int c = 0; c < ctx->n_sm_total; c++) { init[(size_t) c * 8 + 1] = ctx->att_ns; init[(size_t) c * 8 + 2] = ctx->first_ns; init[(size_t) c * 8 + 4] = ctx->first_ns; }
        m.d_adapt = (unsigned *) ctx_alloc(ctx, init.size() * 4);
        BARK_CUDA_CHECK(cudaMemcpy(m.d_adapt, init.data(), init.size() * 4, cudaMemcpyHostToDevice));
    }
}

// one decode token through the persistent kernel
static void decode_step(bark_context * ctx, GPTModel & m, int token, const int32_t * d_token, int n_past, int lm_lo, int lm_hi, const FusedSample * fs = nullptr) {
    // Epochs are 32-bit and must never repeat while a stale word could still carry the old value (~30 M tokens for 24 layers):
    // before the counter wraps, drain the stream, clear every exchange word (epoch 0 = never published) and start over.
    const unsigned step_tags = (unsigned) decode_tags_per_step(m.n_layer);
    if (ctx->tag_base + step_tags + 1u < ctx->tag_base) {
        BARK_CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
        for (GPTModel * g : {&ctx->semantic, &ctx->coarse}) {
            if (!g->decode_ok) continue;
            const size_t E8 = (size_t) g->n_embd * 8, R = kDecodeReplicas;
            BARK_CUDA_CHECK(cudaMemsetAsync(g->gx, 0, R * E8, ctx->stream)); BARK_CUDA_CHECK(cudaMemsetAsync(g->gq, 0, R * E8, ctx->stream));
            BARK_CUDA_CHECK(cudaMemsetAsync(g->gatt, 0, R * E8, ctx->stream)); BARK_CUDA_CHECK(cudaMemsetAsync(g->gff, 0, R * 4 * E8, ctx->stream));
            BARK_CUDA_CHECK(cudaMemsetAsync(g->gk, 0, E8, ctx->stream)); BARK_CUDA_CHECK(cudaMemsetAsync(g->gv, 0, E8, ctx->stream));
            BARK_CUDA_CHECK(cudaMemsetAsync(g->gscores, 0, (size_t) g->n_head * g->block_size * 8, ctx->stream));
        }
        ctx->tag_base = 0;
    }
    DecodeArgs a{};
    a.phases = (const DecodePhase *) m.d_phases; a.layer_vecs = (const DecodeLayerVec *) m.d_layer_vecs;
    a.wte = m.wte[0]; a.wpe = m.wpe; a.ln_f_g = m.ln_f_g; a.ln_f_b = m.ln_f_b; a.gelu_tab = ctx->d_gelu_tab;
    a.mem_k = m.mem_k; a.mem_v = m.mem_v;
    a.gx = m.gx; a.gq = m.gq; a.gk = m.gk; a.gv = m.gv; a.gatt = m.gatt; a.gff = m.gff; a.gscores = m.gscores; a.logits = m.glogits;
    a.tag_base = ctx->tag_base; a.ln_fallbacks = ctx->d_ln_fallbacks; a.timing = ctx->d_timing;
    a.E = m.n_embd; a.H = m.n_head; a.L = m.n_layer; a.block_size = m.block_size; a.n_past = n_past; a.token = token; a.lm_lo = lm_lo; a.lm_hi = lm_hi;
    a.token_ptr = d_token; a.n_vocab_in = m.n_in_vocab;
    a.inv_E = 1.0 / (double) m.n_embd;
    a.adapt = ctx->adapt_on ? m.d_adapt : nullptr;
    for (int i = 0; i < 6; i++) a.headstart[i] = ctx->headstart[i];
    if (fs) {
        a.samp_n = fs->n; a.samp_temp = fs->temp; a.samp_u = fs->d_u; a.samp_tok = fs->d_tok; a.samp_tok_add = fs->tok_add; a.samp_feed = fs->d_feed;
        a.samp_eos = fs->d_eos; a.samp_flags = fs->d_flags; a.samp_force = fs->force; a.done_counter = ctx->d_done_counter;
    }
    a.kv_prefetch = ctx->kv_prefetch ? 1 : 0;
    a.timing_tid = ctx->timing_tid; a.poll_ns = ctx->poll_ns; a.first_ns = ctx->first_ns; a.att_ns = ctx->att_ns;
    const double es = m.wtype == W_Q4_0 ? 18.0 / 32.0 : m.wtype == W_F16 ? 2.0 : 4.0;
    const double E = m.n_embd, L = m.n_layer;
    g_next_bytes = (12.0 * L * E * E + (double)(lm_hi - lm_lo) * E) * es + 2.0 * L * (double)(n_past + 1) * E * 4.0 + 2.0 * L * E * 4.0 + (double)(lm_hi - lm_lo) * 4.0;   // SURVEY §8d B_tok
    g_next_flops = 2.0 * (12.0 * L * E * E + (double)(lm_hi - lm_lo) * E) + 4.0 * L * (double)(n_past + 1) * E;
    int max_row_bytes = 0;
    for (const DMat * d : {&m.layers[0].c_attn, &m.layers[0].c_proj, &m.layers[0].fc, &m.layers[0].proj, &m.lm_head[0]}) max_row_bytes = std::max(max_row_bytes, (int)(d->Kp * (m.wtype == W_F16 ? 2 : 4)));   // (cluster kernel: f16 / f32 only)
    if (ctx->decode_cluster && decode_cluster_supported(a, m.wtype, max_row_bytes)) launch_decode_cluster(a, m.wtype, ctx->stream);
    else launch_decode_step(a, m.wtype, ctx->n_sm, ctx->stream);
    ctx->tag_base += (unsigned) decode_tags_per_step(m.n_layer);
}

bool gpt_eval(bark_context * ctx, GPTModel & m, const int32_t * tokens, int n, int * n_past, bool merge_ctx, float * logits_host, int lm_lo, int lm_hi,
              float * kv_k, float * kv_v) {
    if (!n_past) { fprintf(stderr, "%s: n_past is null\n", __func__); return false; }
    const int64_t t0 = now_us();
    Workspace & ws = ctx->ws;
    cudaStream_t s = ctx->stream;
    const int E = m.n_embd;
    int N = n;
    bool merge = false;
    if (lm_hi <= 0 || lm_hi > m.n_out_vocab || lm_lo < 0 || lm_lo >= lm_hi) { lm_lo = 0; lm_hi = m.n_out_vocab; }
    if (!tokens || n < 1 || n > 8 * 1024) { fprintf(stderr, "%s: bad token buffer (n = %d)\n", __func__, n); return false; }
    for (int i = 0; i < n; i++) if (tokens[i] < 0 || tokens[i] >= m.n_in_vocab) {      // the embedding gather is unchecked on the device
        fprintf(stderr, "%s: token id %d at position %d is outside the model's input vocabulary (%d)\n", __func__, tokens[i], i, m.n_in_vocab); return false;
    }
    const bool own_cache = !kv_k;                            // the persistent decode kernel works on the model's own cache only
    if (own_cache) { kv_k = m.mem_k; kv_v = m.mem_v; }
    if (*n_past > 0 && N == 1) {
        if (own_cache && ctx->use_decode_kernel && m.decode_ok && *n_past + 1 <= m.block_size) {
            decode_step(ctx, m, tokens[0], nullptr, *n_past, lm_lo, lm_hi);
            ctx->last_logits = m.glogits;
            if (logits_host) {
                const size_t nb = (size_t)(lm_hi - lm_lo) * sizeof(float);
                BARK_CUDA_CHECK(cudaMemcpyAsync(ctx->h_logits, m.glogits + lm_lo, nb, cudaMemcpyDeviceToHost, s)); g_d2h_bytes += nb;
                BARK_CUDA_CHECK(cudaStreamSynchronize(s));
                memcpy(logits_host + lm_lo, ctx->h_logits, nb);
            }
            *n_past += 1;
            m.t_predict_us += now_us() - t0;
            return true;
        }
    } else if (merge_ctx && *n_past == 0) {
        if (N != 513) { fprintf(stderr, "%s: merged prompt must hold 256+256+1 ids (got %d)\n", __func__, N); return false; }
        N = 257; merge = true;                                                                                  // bark.cpp:1230-1233
    }
    if (N < 1 || *n_past + N > m.block_size) { fprintf(stderr, "%s: context overflow (n_past %d + %d > %d)\n", __func__, *n_past, N, m.block_size); return false; }
    memcpy(ctx->h_tok, tokens, (size_t) n * sizeof(int32_t));
    BARK_CUDA_CHECK(cudaMemcpyAsync(ws.tok, ctx->h_tok, (size_t) n * sizeof(int32_t), cudaMemcpyHostToDevice, s)); g_h2d_bytes += (size_t) n * sizeof(int32_t);
    gpt_embed_causal(m, ws.tok, N, *n_past, merge, ws.x, s);
    run_layers(ctx, m, N, *n_past, true, kv_k, kv_v);
    // final norm + lm_head on the last position only (bark.cpp:1391-1405)
    const int kpE = is_quant(m.wtype) ? E : ws.max_rows * kGmGroup;
    layernorm_act(ws.x + (size_t)(N - 1) * E, 1, E, m.ln_f_g, m.ln_f_b, ws.act, is_quant(m.wtype) ? W_Q4_0 : m.wtype, kpE, ctx->d_ln_fallbacks, s);
    MatmulEpilogue st; st.mode = EPI_STORE; st.out = ws.logits; st.ldo = m.n_out_vocab;
    lane_matmul(m.lm_head[0], ws.act, kpE, 1, st, s);
    ctx->last_logits = ws.logits;
    if (logits_host) {
        BARK_CUDA_CHECK(cudaMemcpyAsync(ctx->h_logits, ws.logits, (size_t) m.n_out_vocab * sizeof(float), cudaMemcpyDeviceToHost, s)); g_d2h_bytes += (size_t) m.n_out_vocab * sizeof(float);
        BARK_CUDA_CHECK(cudaStreamSynchronize(s));
        memcpy(logits_host, ctx->h_logits, (size_t) m.n_out_vocab * sizeof(float));
    }
    *n_past += N;
    m.t_predict_us += now_us() - t0;
    return true;
}

// One decode step whose input token is read from device memory (the previous step's sample): nothing to wait for on the
// host, so a whole window of steps is enqueued back to back.
bool fused_sampler_available(const bark_context * ctx, const GPTModel & m, int samp_n) {
    return ctx->fuse_sampler && ctx->use_decode_kernel && m.decode_ok && !ctx->decode_cluster && (size_t) samp_n * 4 <= 64 * 1024;
}

bool gpt_decode_chained(bark_context * ctx, GPTModel & m, const int32_t * d_token, int * n_past, int lm_lo, int lm_hi, const FusedSample * fs) {
    if (!ctx->use_decode_kernel || !m.decode_ok || *n_past < 1) { fprintf(stderr, "%s: needs the persistent decode kernel and a filled KV cache\n", __func__); return false; }
    if (*n_past + 1 > m.block_size) { fprintf(stderr, "%s: context overflow (n_past %d + 1 > %d)\n", __func__, *n_past, m.block_size); return false; }
    if (lm_hi <= 0 || lm_hi > m.n_out_vocab || lm_lo < 0 || lm_lo >= lm_hi) { lm_lo = 0; lm_hi = m.n_out_vocab; }
    decode_step(ctx, m, 0, d_token, *n_past, lm_lo, lm_hi, fs);
    ctx->last_logits = m.glogits;
    *n_past += 1;
    return true;
}

bool fine_eval(bark_context * ctx, const int32_t * in_buffer, int nn, float * logits_host) {
    if (ctx->fast_mode) return fine_eval_fast(ctx, in_buffer, nn, logits_host);
    GPTModel & m = ctx->fine;
    if (nn < 1 || nn > 7) { fprintf(stderr, "%s: codebook index %d out of range\n", __func__, nn); return false; }
    const int64_t t0 = now_us();
    Workspace & ws = ctx->ws;
    cudaStream_t s = ctx->stream;
    const int E = m.n_embd, N = 1024;
    for (int i = 0; i < (nn + 1) * 1024; i++) if (in_buffer[i] < 0 || in_buffer[i] >= m.n_in_vocab) {
        fprintf(stderr, "%s: code %d (codebook %d, frame %d) is outside the fine model's input vocabulary (%d)\n", __func__, in_buffer[i], i / 1024, i % 1024, m.n_in_vocab); return false;
    }
    memcpy(ctx->h_tok, in_buffer, (size_t) 8 * 1024 * sizeof(int32_t));
    BARK_CUDA_CHECK(cudaMemcpyAsync(ws.tok, ctx->h_tok, (size_t) 8 * 1024 * sizeof(int32_t), cudaMemcpyHostToDevice, s)); g_h2d_bytes += (size_t) 8 * 1024 * sizeof(int32_t);
    gpt_embed_fine(m, ws.tok, nn, ws.x, s);
    run_layers(ctx, m, N, 0, false);
    const int kpE = is_quant(m.wtype) ? E : ws.max_rows * kGmGroup;
    const bool c32 = ctx->gemm_f32c && m.wtype == W_F16;
    layernorm_act(ws.x, N, E, m.ln_f_g, m.ln_f_b, ws.act, is_quant(m.wtype) ? W_Q4_0 : c32 ? (WType) W_F16R32 : m.wtype, kpE, ctx->d_ln_fallbacks, s);
    MatmulEpilogue st; st.mode = EPI_STORE; st.out = ws.logits; st.ldo = m.n_out_vocab;
    lane_matmul(m.lm_head[nn - 1], ws.act, kpE, N, st, s, c32);                                                           // n_codes_given = 1 (bark.cpp:61,1573)
    ctx->last_logits = ws.logits;
    if (logits_host) {
        const size_t nb = (size_t) N * m.n_out_vocab * sizeof(float);
        BARK_CUDA_CHECK(cudaMemcpyAsync(ctx->h_logits, ws.logits, nb, cudaMemcpyDeviceToHost, s)); g_d2h_bytes += nb;
        BARK_CUDA_CHECK(cudaStreamSynchronize(s));
        memcpy(logits_host, ctx->h_logits, nb);
    }
    m.t_predict_us += now_us() - t0;
    return true;
}

// FAST MODE: the same pass on the tensor cores (fast_kernels.cu): LayerNorm -> f16, tcgen05 GEMMs with fused epilogues, flash-style
// attention.  Same inputs / outputs as fine_eval; logits agree with the reference to f16-operand accuracy, not bit for bit.
bool fine_eval_fast(bark_context * ctx, const int32_t * in_buffer, int nn, float * logits_host) {
    GPTModel & m = ctx->fine;
    if (nn < 1 || nn > 7) { fprintf(stderr, "%s: codebook index %d out of range\n", __func__, nn); return false; }
    const int64_t t0 = now_us();
    Workspace & ws = ctx->ws;
    cudaStream_t s = ctx->stream;
    const int E = m.n_embd, H = m.n_head, N = 1024, n_sm = ctx->n_sm_total;
    for (int i = 0; i < (nn + 1) * 1024; i++) if (in_buffer[i] < 0 || in_buffer[i] >= m.n_in_vocab) {
        fprintf(stderr, "%s: code %d (codebook %d, frame %d) is outside the fine model's input vocabulary (%d)\n", __func__, in_buffer[i], i / 1024, i % 1024, m.n_in_vocab); return false;
    }
    memcpy(ctx->h_tok, in_buffer, (size_t) 8 * 1024 * sizeof(int32_t));
    BARK_CUDA_CHECK(cudaMemcpyAsync(ws.tok, ctx->h_tok, (size_t) 8 * 1024 * sizeof(int32_t), cudaMemcpyHostToDevice, s)); g_h2d_bytes += (size_t) 8 * 1024 * sizeof(int32_t);
    gpt_embed_fine(m, ws.tok, nn, ws.x, s);
    for (int il = 0; il < m.n_layer; il++) {
        const GPTLayer & L = m.layers[(size_t) il];
        fast_layernorm(ws.x, N, E, L.ln_1_g, L.ln_1_b, ctx->f_a16, s);
        FastEpi qkv; qkv.mode = FEPI_QKV16; qkv.out16 = ctx->f_qk16; qkv.ldo = 2 * E; qkv.vt = ctx->f_vt16; qkv.vt_ld = N; qkv.v_col0 = 2 * E;
        if (!fast_gemm(ctx->f_a16, E, (const __half *) L.c_attn.p_rm, E, N, 3 * E, E, qkv, n_sm, s)) return false;
        if (!fast_attention(ctx->f_qk16, 2 * E, E, ctx->f_vt16, N, E, H, ctx->f_att16, s)) return false;
        FastEpi res; res.mode = FEPI_RESID; res.out32 = ws.x; res.ldo = E;
        if (!fast_gemm(ctx->f_att16, E, (const __half *) L.c_proj.p_rm, E, N, E, E, res, n_sm, s)) return false;
        fast_layernorm(ws.x, N, E, L.ln_2_g, L.ln_2_b, ctx->f_a16, s);
        FastEpi ge; ge.mode = FEPI_GELU16; ge.out16 = ctx->f_h16; ge.ldo = 4 * E; ge.gelu_tab = ctx->d_gelu_tab;
        if (!fast_gemm(ctx->f_a16, E, (const __half *) L.fc.p_rm, E, N, 4 * E, E, ge, n_sm, s)) return false;
        if (!fast_gemm(ctx->f_h16, 4 * E, (const __half *) L.proj.p_rm, 4 * E, N, E, 4 * E, res, n_sm, s)) return false;
    }
    fast_layernorm(ws.x, N, E, m.ln_f_g, m.ln_f_b, ctx->f_a16, s);
    FastEpi st; st.mode = FEPI_F32; st.out32 = ws.logits; st.ldo = m.n_out_vocab;
    if (!fast_gemm(ctx->f_a16, E, (const __half *) m.lm_head[nn - 1].p_rm, E, N, m.n_out_vocab, E, st, n_sm, s)) return false;
    ctx->last_logits = ws.logits;
    if (logits_host) {
        const size_t nb = (size_t) N * m.n_out_vocab * sizeof(float);
        BARK_CUDA_CHECK(cudaMemcpyAsync(ctx->h_logits, ws.logits, nb, cudaMemcpyDeviceToHost, s)); g_d2h_bytes += nb;
        BARK_CUDA_CHECK(cudaStreamSynchronize(s));
        memcpy(logits_host, ctx->h_logits, nb);
    }
    m.t_predict_us += now_us() - t0;
    return true;
}

// Sample `rows` tokens from device-resident logits (sampling.cu); rows the kernel could not decide bit-safely are replayed
// on the host with the reference's exact arithmetic and the same uniform draw.  Leaves tokens (and optionally the
// probability of the last logit) in out_tok / out_eos.  The RNG stream advances exactly as gpt_sample would advance it.
bool sample_device(bark_context * ctx, GPTModel & m, const float * d_logits, int ld, int n, int rows, float temp, int32_t * out_tok, float * out_eos) {
    const int64_t t0 = now_us();
    if (rows < 1 || rows > 1024 || n < 2 || (size_t) n * 4 > 64 * 1024) { fprintf(stderr, "%s: unsupported shape (%d rows of %d)\n", __func__, rows, n); return false; }
    if (temp != 0.0f) for (int r = 0; r < rows; r++) ctx->h_u[r] = std::generate_canonical<double, 53>(ctx->rng);   // what discrete_distribution::operator() draws
    const int force = ctx->debug_flag_every > 0 && (ctx->n_sample_calls++ % ctx->debug_flag_every) == 0;
    const SampleBufs b{ctx->h_u, ctx->d_u, ctx->h_stok, ctx->d_stok, ctx->h_sflags, ctx->d_sflags, ctx->h_seos, ctx->d_seos};
    sample_rows_sync(ctx, b, d_logits, ld, n, rows, temp, 0, force, out_tok, out_eos, &ctx->n_sample_host_replays);
    m.t_sample_us += now_us() - t0;
    m.n_sample += rows;
    return true;
}

// sample_rows over `rows` rows whose uniforms are already in b.h_u, then one synchronisation and the host replay of flagged rows
void sample_rows_sync(bark_context * ctx, const SampleBufs & b, const float * d_logits, int ld, int n, int rows, float temp, int tok_add, int force,
                      int32_t * out_tok, float * out_eos, long long * replays) {
    cudaStream_t s = ctx->stream;
    if (temp != 0.0f) { BARK_CUDA_CHECK(cudaMemcpyAsync(b.d_u, b.h_u, (size_t) rows * sizeof(double), cudaMemcpyHostToDevice, s)); g_h2d_bytes += (size_t) rows * sizeof(double); }
    sample_rows(d_logits, ld, n, rows, temp, b.d_u, b.d_tok, 0, nullptr, b.d_eos, b.d_flags, force, s);
    BARK_CUDA_CHECK(cudaMemcpyAsync(b.h_tok, b.d_tok, (size_t) rows * 4, cudaMemcpyDeviceToHost, s));
    BARK_CUDA_CHECK(cudaMemcpyAsync(b.h_flags, b.d_flags, (size_t) rows * 4, cudaMemcpyDeviceToHost, s));
    BARK_CUDA_CHECK(cudaMemcpyAsync(b.h_eos, b.d_eos, (size_t) rows * 4, cudaMemcpyDeviceToHost, s)); g_d2h_bytes += (size_t) rows * 12;
    BARK_CUDA_CHECK(cudaStreamSynchronize(s));
    std::vector<float> row;
    for (int r = 0; r < rows; r++) {
        if (b.h_flags[r]) {
            row.resize((size_t) n);
            BARK_CUDA_CHECK(cudaMemcpy(row.data(), d_logits + (size_t) r * ld, (size_t) n * 4, cudaMemcpyDeviceToHost)); g_d2h_bytes += (size_t) n * 4;
            b.h_tok[r] = sample_token_given_u(row.data(), n, temp, b.h_u[r], &b.h_eos[r]);
            ++*replays;
        }
        out_tok[r] = tok_add + b.h_tok[r];
        if (out_eos) out_eos[r] = b.h_eos[r];
    }
}

bool codec_decode(bark_context * ctx, const int32_t * codes, int T) {
    if (T < 7) { fprintf(stderr, "%s: need at least 7 frames (reflect padding of the k=7 convolutions), got %d\n", __func__, T); return false; }
    CodecModel & cm = ctx->codec;
    cudaStream_t s = ctx->stream;
    static const int ratios[4] = {8, 5, 4, 2};
    for (size_t i = 0; i < (size_t) 8 * T; i++) if (codes[i] < 0 || codes[i] >= cm.n_bins) {
        fprintf(stderr, "%s: code %d (codebook %zu, frame %zu) is outside the codebooks (%d bins)\n", __func__, codes[i], i / T, i % T, cm.n_bins); return false;
    }
    const size_t need = (size_t) 10240 * T + 1024;             // largest activation: [64][160T] = [32][320T] = 10240*T floats
    if (need > ctx->c_cap) {
        // out of memory here is recoverable (a very long clip): report it and return false like the reference's failed encodec_eval
        auto grow = [&](void ** p, size_t bytes) { if (*p) { cudaFree(*p); *p = nullptr; } return cudaMalloc(p, bytes) == cudaSuccess; };
        ctx->c_cap = 0;
        bool ok = true;
        for (int i = 0; i < 3; i++) ok = ok && grow((void **) &ctx->c_buf[i], need * sizeof(float));
        ok = ok && grow((void **) &ctx->c_gi, (size_t) T * 2048 * sizeof(float)) && grow((void **) &ctx->d_codes, (size_t) 8 * T * sizeof(int32_t));
        if (!ok) { (void) cudaGetLastError(); fprintf(stderr, "%s: out of device memory for a %d-frame clip\n", __func__, T); return false; }
        if (!ctx->c_hbuf) { ctx->c_hbuf = (float *) ctx_alloc(ctx, 2 * 512 * sizeof(float)); ctx->c_counter = (unsigned *) ctx_alloc(ctx, sizeof(unsigned)); }
        ctx->c_cap = need;
    }
    float * a = ctx->c_buf[0], * b = ctx->c_buf[1], * c = ctx->c_buf[2];
    BARK_CUDA_CHECK(cudaMemcpyAsync(ctx->d_codes, codes, (size_t) 8 * T * sizeof(int32_t), cudaMemcpyHostToDevice, s)); g_h2d_bytes += (size_t) 8 * T * sizeof(int32_t);
    rvq_decode(cm, ctx->d_codes, T, a, s);                                                // [128][T]
    conv1d(a, cm.hidden_dim, T, cm.init, false, nullptr, b, s);                          // [512][T]
    int C = cm.init.cout;
    lstm_layer(b, C, T, cm.lstm_ih_w[0], cm.lstm_hh_w[0], cm.lstm_Kp, cm.lstm_ih_b[0], cm.lstm_hh_b[0], nullptr, ctx->c_gi, ctx->c_hbuf, ctx->c_counter, a, s);
    lstm_layer(a, C, T, cm.lstm_ih_w[1], cm.lstm_hh_w[1], cm.lstm_Kp, cm.lstm_ih_b[1], cm.lstm_hh_b[1], b /*skip (decoder.h:72)*/, ctx->c_gi, ctx->c_hbuf, ctx->c_counter, c, s);
    float * cur = c, * t1 = a, * t2 = b;
    int L = T;
    for (int i = 0; i < 4; i++) {
        convtr1d(cur, C, L, cm.blk[i].us, ratios[i], t1, s);          // ELU fused on the input; -> [C/2][L*r]
        C /= 2; L *= ratios[i];
        conv1d(t1, C, L, cm.blk[i].sc, false, nullptr, t2, s);        // shortcut on the raw up-sampled signal
        conv1d(t1, C, L, cm.blk[i].c1, true, nullptr, cur, s);        // ELU -> k3 -> [C/2][L]
        conv1d(cur, C / 2, L, cm.blk[i].c2, true, t2, t1, s);         // ELU -> k1, + shortcut
        std::swap(cur, t1);
    }
    conv1d(cur, C, L, cm.final_conv, true, nullptr, t1, s);           // ELU -> k7 -> [1][320 T]
    ctx->audio.resize((size_t) L);
    BARK_CUDA_CHECK(cudaMemcpyAsync(ctx->audio.data(), t1, (size_t) L * sizeof(float), cudaMemcpyDeviceToHost, s)); g_d2h_bytes += (size_t) L * sizeof(float);
    BARK_CUDA_CHECK(cudaStreamSynchronize(s));
    return true;
}

}  // namespace bark
