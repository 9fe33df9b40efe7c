// Batched generation: several prompts in one context on one GPU, every item bit-identical to its own single-prompt run.
//
// A decode step of bark-small streams ~188 MB of weights to produce one token and is bound by latency, not bandwidth
// (DESIGN.md §4.1, §7).  Decoding B prompts together reads those weights once per B tokens.  The batch runs stage by stage:
//   1. semantic for all items together,  2. coarse for all items together,  3. fine, one item at a time,  4. EnCodec, one item at a time
// (a fine pass already has 1024 rows and fills the GPU).  In stages 1-2:
//   * every item has its own KV cache region (one region serves both models: the semantic stage of all items ends before the coarse
//     stage starts) and its own std::mt19937(seed), consumed exactly as that item's single-prompt run consumes it;
//   * prefills (the 257-row merged semantic prompt, each coarse window's 60-91 rows after prefix reuse) run per item through
//     gpt_eval pointed at the item's cache; the decode steps of all still-active items run as ONE batched step (batch_step below:
//     the existing mat-mul kernels over B rows, which are bit-exact per row whatever the row count, plus batch_decode_attention);
//   * all items active at a step have the same n_past (the semantic prefill always leaves 257 positions, coarse window w always
//     has 257 + min(630, 60 w) prompt ids), so a step has one n_kv and per-item cache bases; items that stop drop out and the
//     batch is compacted.
// Sampling: sample_rows over the B logit rows, one uniform per row from that item's RNG, flagged rows replayed on the host; one host
// round trip per step.  The single-prompt state of the context (RNG, token arrays, audio, statistics, progress callback) is saved
// on entry and restored on exit.
#include "../../include/bark_b200.h"
#include "context.h"
#include "gpt_kernels.h"

#include <algorithm>
#include <cstring>
#include <numeric>

namespace bark {

namespace {

// What a batch call changes on the context that belongs to the single-prompt API; put back when the call ends, whatever happens.
struct SinglePromptState {
    bark_context * ctx;
    std::mt19937 rng; std::vector<int32_t> tokens, semantic, coarse, fine; std::vector<float> audio;
    bark_context_params params; bark_statistics stats;
    int64_t model[3][4];
    unsigned long long n_kv_reused; long long replays, calls; const float * last_logits;
    explicit SinglePromptState(bark_context * c)
        : ctx(c), rng(c->rng), tokens(c->tokens), semantic(c->semantic_tokens), coarse(c->coarse_tokens), fine(c->fine_tokens), audio(c->audio),
          params(c->params), stats(c->stats), n_kv_reused(c->n_kv_reused), replays(c->n_sample_host_replays), calls(c->n_sample_calls),
          last_logits(c->last_logits) {
        const GPTModel * m[3] = {&c->semantic, &c->coarse, &c->fine};
        for (int i = 0; i < 3; i++) { model[i][0] = m[i]->t_sample_us; model[i][1] = m[i]->t_predict_us; model[i][2] = m[i]->t_main_us; model[i][3] = m[i]->n_sample; }
        c->params.progress_callback = nullptr;                   // a batch call reports no progress
    }
    ~SinglePromptState() {
        bark_context * c = ctx;
        c->rng = rng; c->tokens.swap(tokens); c->semantic_tokens.swap(semantic); c->coarse_tokens.swap(coarse); c->fine_tokens.swap(fine); c->audio.swap(audio);
        c->params = params; c->stats = stats; c->n_kv_reused = n_kv_reused; c->n_sample_host_replays = replays; c->n_sample_calls = calls; c->last_logits = last_logits;
        GPTModel * m[3] = {&c->semantic, &c->coarse, &c->fine};
        for (int i = 0; i < 3; i++) { m[i]->t_sample_us = model[i][0]; m[i]->t_predict_us = model[i][1]; m[i]->t_main_us = model[i][2]; m[i]->n_sample = model[i][3]; }
    }
};

size_t slot_floats_needed(const bark_context * ctx) {
    size_t need = 0;
    for (const GPTModel * m : {&ctx->semantic, &ctx->coarse}) need = std::max(need, (size_t) 2 * m->n_layer * m->block_size * m->n_embd);
    return need;
}

// Scratch on the first call; per-item KV regions grown to n items.  Out of device memory is a reported failure, not an abort.
bool ensure_batch_memory(bark_context * ctx, int n) {
    BatchState & bs = ctx->batch;
    if (!bs.qkv) {
        const size_t E = (size_t) std::max(ctx->semantic.n_embd, ctx->coarse.n_embd), n_out = (size_t) std::max(ctx->semantic.n_out_vocab, ctx->coarse.n_out_vocab);
        bs.qkv = (float *) ctx_alloc(ctx, (size_t) kBatchMax * 3 * E * 4);
        bs.logits = (float *) ctx_alloc(ctx, (size_t) kBatchMax * n_out * 4);
        bs.d_u = (double *) ctx_alloc(ctx, kBatchMax * 8); bs.d_tok = (int32_t *) ctx_alloc(ctx, kBatchMax * 4);
        bs.d_flags = (int32_t *) ctx_alloc(ctx, kBatchMax * 4); bs.d_eos = (float *) ctx_alloc(ctx, kBatchMax * 4);
        BARK_CUDA_CHECK(cudaMemset(bs.d_u, 0, kBatchMax * 8));
        BARK_CUDA_CHECK(cudaMallocHost(&bs.h_u, kBatchMax * 8)); BARK_CUDA_CHECK(cudaMallocHost(&bs.h_tok, kBatchMax * 4));
        BARK_CUDA_CHECK(cudaMallocHost(&bs.h_flags, kBatchMax * 4)); BARK_CUDA_CHECK(cudaMallocHost(&bs.h_eos, kBatchMax * 4));
    }
    const size_t need = slot_floats_needed(ctx);
    if (n <= bs.slots && bs.slot_floats == need) return true;
    if (bs.kv) { BARK_CUDA_CHECK(cudaStreamSynchronize(ctx->stream)); cudaFree(bs.kv); bs.kv = nullptr; bs.slots = 0; }
    if (cudaMalloc(&bs.kv, (size_t) n * need * 4) != cudaSuccess) {
        (void) cudaGetLastError(); bs.kv = nullptr;
        fprintf(stderr, "bark_b200: out of device memory for %d per-item KV caches of %.1f MB\n", n, need * 4.0 / 1e6);
        return false;
    }
    bs.slots = n; bs.slot_floats = need;
    return true;
}

// item slot's region: the model's K cache [L][block_size][E], then its V cache
float * slot_k(bark_context * ctx, int slot) { return ctx->batch.kv + (size_t) slot * ctx->batch.slot_floats; }
float * slot_v(bark_context * ctx, const GPTModel & m, int slot) { return slot_k(ctx, slot) + (size_t) m.n_layer * m.block_size * m.n_embd; }

// One decode step for B rows: row b is item slot[b] with input id tok[b] at position n_past (the same for every row).
// Leaves the logits in batch.logits [B][n_out_vocab].
void batch_step(bark_context * ctx, GPTModel & m, const int * slot, const int32_t * tok, int B, int n_past) {
    Workspace & ws = ctx->ws;
    BatchState & bs = ctx->batch;
    cudaStream_t s = ctx->stream;
    const int E = m.n_embd, H = m.n_head;
    const bool q4 = is_quant(m.wtype);                        // quantised weights: f32 activation rows (as run_layers)
    const WType awt = q4 ? W_Q4_0 : m.wtype;
    const int kpE = q4 ? E : ws.max_rows * kGmGroup, kp4E = q4 ? 4 * E : kpE;
    if (q4) { q4_set_scratch(ctx->d_q8, ctx->d_q8_scales); qx_set_scratch(ctx->d_q8, ctx->d_q8_scales, ctx->d_q8_sums); }
    RowIds ids;
    for (int b = 0; b < B; b++) ids.v[b] = tok[b];
    gpt_embed_rows(m, ids, B, n_past, ws.x, s);
    const size_t layer = (size_t) m.block_size * E;
    unsigned * sm_fallbacks = ctx->d_ln_fallbacks ? ctx->d_ln_fallbacks + 1 : nullptr;
    for (int il = 0; il < m.n_layer; il++) {
        const GPTLayer & L = m.layers[(size_t) il];
        BatchKV kv;
        for (int b = 0; b < B; b++) { kv.k[b] = slot_k(ctx, slot[b]) + il * layer; kv.v[b] = slot_v(ctx, m, slot[b]) + il * layer; }
        layernorm_act(ws.x, B, E, L.ln_1_g, L.ln_1_b, ws.act, awt, kpE, ctx->d_ln_fallbacks, s);
        MatmulEpilogue qkv; qkv.mode = EPI_STORE; qkv.out = bs.qkv; qkv.ldo = 3 * E;
        lane_matmul(L.c_attn, ws.act, kpE, B, qkv, s);
        batch_decode_attention(bs.qkv, kv, B, n_past, E, H, ws.act, awt, kpE, sm_fallbacks, s);
        MatmulEpilogue res; res.mode = EPI_RESID; res.out = ws.x; res.ldo = E;
        lane_matmul(L.c_proj, ws.act, kpE, B, res, s);                                                        // + inpL
        layernorm_act(ws.x, B, E, L.ln_2_g, L.ln_2_b, ws.act, awt, kpE, ctx->d_ln_fallbacks, s);
        MatmulEpilogue ge; ge.mode = EPI_GELU_ACT; ge.act_out = ws.act2; ge.act_wt = (int) awt; ge.act_Kp = kp4E; ge.gelu_tab = ctx->d_gelu_tab;
        lane_matmul(L.fc, ws.act, kpE, B, ge, s);
        lane_matmul(L.proj, ws.act2, kp4E, B, res, s);                                                        // + inpFF
    }
    layernorm_act(ws.x, B, E, m.ln_f_g, m.ln_f_b, ws.act, awt, kpE, ctx->d_ln_fallbacks, s);
    MatmulEpilogue st; st.mode = EPI_STORE; st.out = bs.logits; st.ldo = m.n_out_vocab;
    lane_matmul(m.lm_head[0], ws.act, kpE, B, st, s);
    ctx->batch.stats[4]++;
}

// gpt_eval stages its ids in ONE pinned host buffer (ctx->h_tok) and copies them asynchronously: before the next item's prefill
// overwrites that buffer, the previous copy must have left it
bool prefill(bark_context * ctx, GPTModel & m, int slot, const int32_t * ids, int n, bool merge, int * n_past) {
    BARK_CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
    return gpt_eval(ctx, m, ids, n, n_past, merge, nullptr, 0, 0, slot_k(ctx, slot), slot_v(ctx, m, slot));
}

// prefill of one item into its own cache; its last-position logits go to row `row` of batch.logits
bool prefill_item(bark_context * ctx, GPTModel & m, int slot, const std::vector<int32_t> & ids, bool merge, int * n_past, int row) {
    if (!prefill(ctx, m, slot, ids.data(), (int) ids.size(), merge, n_past)) return false;
    const size_t nb = (size_t) m.n_out_vocab * 4;
    BARK_CUDA_CHECK(cudaMemcpyAsync(ctx->batch.logits + (size_t) row * m.n_out_vocab, ctx->ws.logits, nb, cudaMemcpyDeviceToDevice, ctx->stream));
    return true;
}

// one token for each of the B rows of batch.logits from logits [lo, lo + n); row b draws from rngs[b]
void sample_batch(bark_context * ctx, int ld, int lo, int n, int B, float temp, std::mt19937 * const * rngs, int32_t * tok, float * eos) {
    BatchState & bs = ctx->batch;
    if (temp != 0.0f) for (int b = 0; b < B; b++) bs.h_u[b] = std::generate_canonical<double, 53>(*rngs[b]);   // one draw per sample, as discrete_distribution makes
    const int force = ctx->debug_flag_every > 0 && (bs.n_sample_calls++ % ctx->debug_flag_every) == 0;
    const SampleBufs sb{bs.h_u, bs.d_u, bs.h_tok, bs.d_tok, bs.h_flags, bs.d_flags, bs.h_eos, bs.d_eos};
    long long replays = 0;
    sample_rows_sync(ctx, sb, bs.logits + lo, ld, n, B, temp, lo, force, tok, eos, &replays);
    bs.stats[5] += replays;
}

bool same_n_past(const std::vector<int> & n_past, const std::vector<int> & act) {
    for (int i : act) if (n_past[(size_t) i] != n_past[(size_t) act[0]]) {
        fprintf(stderr, "bark_b200: batched step with unequal positions (%d vs %d)\n", n_past[(size_t) i], n_past[(size_t) act[0]]); return false;
    }
    return true;
}

struct ItemState {
    std::mt19937 rng; std::vector<int32_t> prompt; BatchItem out;
    CoarsePlan cp{}; std::vector<int32_t> samples, kv_ids; size_t kv_canon = 0; int nw = 0;
};

// stage 1: semantic tokens of every item (run_semantic's loop, all items per step)
bool batch_semantic(bark_context * ctx, std::vector<ItemState> & it) {
    GPTModel & m = ctx->semantic;
    const bark_context_params & P = ctx->params;
    const int n = (int) it.size();
    std::vector<int> act((size_t) n), n_past((size_t) n, 0);
    std::iota(act.begin(), act.end(), 0);
    std::vector<int32_t> tok((size_t) n), last((size_t) n); std::vector<float> eos((size_t) n); std::vector<std::mt19937 *> rngs((size_t) n);
    for (int i = 0; i < n; i++) if (!prefill_item(ctx, m, i, it[(size_t) i].prompt, true, &n_past[(size_t) i], i)) return false;
    for (int j = 0; j < P.n_steps_text_encoder && !act.empty(); j++) {
        const int B = (int) act.size();
        if (!same_n_past(n_past, act)) return false;
        if (j > 0) {
            std::vector<int32_t> in((size_t) B);
            for (int b = 0; b < B; b++) in[(size_t) b] = last[(size_t) act[(size_t) b]];
            batch_step(ctx, m, act.data(), in.data(), B, n_past[(size_t) act[0]]);
            for (int i : act) n_past[(size_t) i]++;
        }
        for (int b = 0; b < B; b++) rngs[(size_t) b] = &it[(size_t) act[(size_t) b]].rng;
        sample_batch(ctx, m.n_out_vocab, 0, m.n_out_vocab, B, P.temp, rngs.data(), tok.data(), eos.data());   // over ALL n_out_vocab logits (quirk D.1)
        std::vector<int> keep;
        for (int b = 0; b < B; b++) {
            const int i = act[(size_t) b];
            if (semantic_stop(P, tok[(size_t) b], eos[(size_t) b])) continue;
            it[(size_t) i].out.semantic.push_back(tok[(size_t) b]);
            last[(size_t) i] = tok[(size_t) b];
            keep.push_back(i);
        }
        act.swap(keep);
    }
    return true;
}

// stage 2: coarse tokens of every item (run_coarse's windows, all items per step; an item leaves after its last window)
bool batch_coarse(bark_context * ctx, std::vector<ItemState> & it) {
    GPTModel & m = ctx->coarse;
    const bark_context_params & P = ctx->params;
    const int n = (int) it.size();
    int n_windows = 0;
    for (ItemState & s : it) { if (!coarse_plan(P, s.out.semantic.size(), &s.cp)) return false; n_windows = std::max(n_windows, s.cp.n_windows); }
    std::vector<int> n_past((size_t) n, 0);
    std::vector<int32_t> tok((size_t) n); std::vector<std::mt19937 *> rngs((size_t) n);
    for (int w = 0; w < n_windows; w++) {
        std::vector<int> act;
        for (int i = 0; i < n; i++) if (w < it[(size_t) i].cp.n_windows) act.push_back(i);
        for (size_t b = 0; b < act.size(); b++) {
            ItemState & s = it[(size_t) act[b]];
            const std::vector<int32_t> in_eval = coarse_window_input(P, s.cp, s.out.semantic, s.samples, ctx->kv_reuse, s.kv_ids, s.kv_canon, &n_past[(size_t) act[b]]);
            if (!prefill_item(ctx, m, act[b], in_eval, false, &n_past[(size_t) act[b]], (int) b)) return false;
            s.nw = std::min(P.sliding_window_size, s.cp.n_steps - (int) s.samples.size());
        }
        const int step0 = (int) it[(size_t) act[0]].samples.size();
        for (int j = 0; !act.empty(); j++) {
            const int B = (int) act.size();
            if (!same_n_past(n_past, act)) return false;
            if (j > 0) {
                std::vector<int32_t> in((size_t) B);
                for (int b = 0; b < B; b++) in[(size_t) b] = it[(size_t) act[(size_t) b]].samples.back();
                batch_step(ctx, m, act.data(), in.data(), B, n_past[(size_t) act[0]]);
                for (int i : act) n_past[(size_t) i]++;
            }
            for (int b = 0; b < B; b++) rngs[(size_t) b] = &it[(size_t) act[(size_t) b]].rng;
            // only logits [lo, lo + codebook_size) are looked at in this stage (bark.cpp:1829-1833)
            sample_batch(ctx, m.n_out_vocab, coarse_lo(P, step0 + j), P.codebook_size, B, P.temp, rngs.data(), tok.data(), nullptr);
            std::vector<int> keep;
            for (int b = 0; b < B; b++) {
                ItemState & s = it[(size_t) act[(size_t) b]];
                s.samples.push_back(tok[(size_t) b]);
                if (j + 1 < s.nw) { s.kv_ids.push_back(tok[(size_t) b]); keep.push_back(act[(size_t) b]); }     // the window's last sample is never evaluated
            }
            act.swap(keep);
        }
    }
    for (ItemState & s : it) coarse_codes(P, s.samples, s.out.coarse);
    return true;
}

bool check_batch_context(bark_context * ctx, const char * fn) {
    if (!ctx) { fprintf(stderr, "%s: invalid bark context\n", fn); return false; }
    if (ctx->shard.on) { fprintf(stderr, "%s: a context with a row-sharded fine stage cannot run batches\n", fn); return false; }
    for (const GPTModel * m : {&ctx->semantic, &ctx->coarse}) {
        const int D = m->n_embd / m->n_head;
        if (m->n_embd % m->n_head || D % 32 || D > 128 || m->block_size > 1024) {
            fprintf(stderr, "%s: model (n_embd %d, n_head %d, block_size %d) outside the batched decode step's shapes\n", fn, m->n_embd, m->n_head, m->block_size); return false;
        }
    }
    return true;
}

bool generate_batch(bark_context * ctx, const char * const * texts, const uint32_t * seeds, int n) {
    const char * fn = "bark_b200_generate_audio_batch";
    if (!check_batch_context(ctx, fn)) return false;
    if (n < 1 || n > kBatchMax) { fprintf(stderr, "%s: batch size %d outside 1..%d\n", fn, n, kBatchMax); return false; }
    if (!texts || !seeds) { fprintf(stderr, "%s: null prompt or seed array\n", fn); return false; }
    for (int i = 0; i < n; i++) if (!texts[i]) { fprintf(stderr, "%s: prompt %d is null\n", fn, i); return false; }
    const bark_context_params & P0 = ctx->params;
    if (!audio_params_supported(P0)) return false;
    if ((size_t) ctx->semantic.n_out_vocab * 4 > 64 * 1024 || P0.sliding_window_size > 1024 || P0.semantic_vocab_size + 2 * P0.codebook_size > ctx->coarse.n_out_vocab) {
        fprintf(stderr, "%s: vocabulary / window sizes outside the device sampler's range\n", fn); return false;
    }
    BARK_CUDA_CHECK(cudaSetDevice(ctx->device));
    ctx->batch.items.clear();
    if (!ensure_batch_memory(ctx, n)) return false;
    SinglePromptState saved(ctx);
    int64_t * st = ctx->batch.stats;
    std::fill(st, st + 6, 0);
    std::vector<ItemState> it((size_t) n);
    for (int i = 0; i < n; i++) {
        it[(size_t) i].rng = std::mt19937(seeds[i]);
        tokenize_input(ctx, texts[i]);
        it[(size_t) i].prompt = ctx->tokens;
    }
    int64_t t0 = now_us();
    if (!batch_semantic(ctx, it)) { fprintf(stderr, "%s: failed to forward text encoder\n", fn); return false; }
    st[0] = now_us() - t0; t0 = now_us();
    if (!batch_coarse(ctx, it)) { fprintf(stderr, "%s: failed to forward coarse encoder\n", fn); return false; }
    st[1] = now_us() - t0;
    for (ItemState & s : it) {                                 // fine and EnCodec: the single-prompt stages, on the item's tokens and RNG
        t0 = now_us();
        ctx->coarse_tokens = s.out.coarse;
        ctx->rng = s.rng;
        if (!run_fine(ctx)) { fprintf(stderr, "%s: failed to forward fine encoder\n", fn); return false; }
        s.out.fine = ctx->fine_tokens;
        st[2] += now_us() - t0; t0 = now_us();
        if (!fine_to_audio(ctx)) return false;
        s.out.audio = ctx->audio;
        st[3] += now_us() - t0;
    }
    for (ItemState & s : it) ctx->batch.items.push_back(std::move(s.out));
    return true;
}

// test hook: teacher-forced batched decode (see bark_b200.h)
int batch_eval(bark_context * ctx, int which, int n, const int32_t * prompts, int len, const int32_t * next, int steps, float * logits_out) {
    const char * fn = "bark_b200_batch_eval";
    if (!check_batch_context(ctx, fn)) return 0;
    if (which < 0 || which > 1 || n < 1 || n > kBatchMax || !prompts || len < 1 || steps < 0 || (steps > 0 && (!next || !logits_out))) {
        fprintf(stderr, "%s: bad arguments\n", fn); return 0;
    }
    GPTModel & m = which == 0 ? ctx->semantic : ctx->coarse;
    if (len + steps > m.block_size) { fprintf(stderr, "%s: %d + %d positions exceed the context (%d)\n", fn, len, steps, m.block_size); return 0; }
    for (int i = 0; i < n * steps; i++) if (next[i] < 0 || next[i] >= m.n_in_vocab) { fprintf(stderr, "%s: id %d outside the input vocabulary\n", fn, next[i]); return 0; }
    BARK_CUDA_CHECK(cudaSetDevice(ctx->device));
    if (!ensure_batch_memory(ctx, n)) return 0;
    SinglePromptState saved(ctx);
    for (int i = 0; i < n; i++) {
        int n_past = 0;
        if (!prefill(ctx, m, i, prompts + (size_t) i * len, len, false, &n_past)) return 0;
    }
    std::vector<int> slot((size_t) n); std::iota(slot.begin(), slot.end(), 0);
    std::vector<int32_t> in((size_t) n);
    std::vector<float> h((size_t) n * m.n_out_vocab);
    for (int j = 0; j < steps; j++) {
        for (int i = 0; i < n; i++) in[(size_t) i] = next[(size_t) i * steps + j];
        batch_step(ctx, m, slot.data(), in.data(), n, len + j);
        BARK_CUDA_CHECK(cudaMemcpyAsync(h.data(), ctx->batch.logits, h.size() * 4, cudaMemcpyDeviceToHost, ctx->stream));
        BARK_CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
        for (int i = 0; i < n; i++) memcpy(logits_out + ((size_t) i * steps + j) * m.n_out_vocab, h.data() + (size_t) i * m.n_out_vocab, (size_t) m.n_out_vocab * 4);
    }
    return 1;
}

const BatchItem * batch_item(bark_context * ctx, int item, const char * fn) {
    if (!ctx || item < 0 || item >= (int) ctx->batch.items.size()) {
        fprintf(stderr, "%s: no item %d in the last batch (%d items)\n", fn, item, ctx ? (int) ctx->batch.items.size() : 0); return nullptr;
    }
    return &ctx->batch.items[(size_t) item];
}

}  // namespace

}  // namespace bark

using namespace bark;

extern "C" bool bark_b200_generate_audio_batch(struct bark_context * ctx, const char * const * texts, const uint32_t * seeds, int n) {
    return guarded(false, [&] { return generate_batch(ctx, texts, seeds, n); });
}

extern "C" int bark_b200_batch_audio(struct bark_context * ctx, int item, float * out, int cap) {
    const BatchItem * b = batch_item(ctx, item, __func__);
    if (!b) return -1;
    if (out && cap > 0) memcpy(out, b->audio.data(), sizeof(float) * std::min(b->audio.size(), (size_t) cap));
    return (int) b->audio.size();
}

extern "C" int bark_b200_batch_tokens(struct bark_context * ctx, int item, int stage, int32_t * out, int cap) {
    const BatchItem * b = batch_item(ctx, item, __func__);
    if (!b) return -1;
    const std::vector<int32_t> * v = stage == 0 ? &b->semantic : stage == 1 ? &b->coarse : stage == 2 ? &b->fine : nullptr;
    if (!v) { fprintf(stderr, "%s: stage %d is not 0, 1 or 2\n", __func__, stage); return -1; }
    if (out && cap > 0) memcpy(out, v->data(), sizeof(int32_t) * std::min(v->size(), (size_t) cap));
    return (int) v->size();
}

extern "C" int bark_b200_batch_eval(struct bark_context * ctx, int which, int n, const int32_t * prompts, int len, const int32_t * next, int steps, float * logits_out) {
    return guarded(0, [&] { return batch_eval(ctx, which, n, prompts, len, next, steps, logits_out); });
}

extern "C" int bark_b200_batch_stats(struct bark_context * ctx, int64_t * out6) {
    if (!ctx || !out6) return 0;
    memcpy(out6, ctx->batch.stats, sizeof(ctx->batch.stats));
    return 1;
}
