// The bark.h C API (include/bark.h) and the host control plane behind it: tokenizer, the three
// stage loops, host sampling, statistics.  Semantics follow the reference's bark.cpp — including
// its quirks (SURVEY.md App. D) — because token parity depends on them; the code is new.
//
//   tokenizer ............ bark.cpp:480-662   (accent strip, [[:punct:]]|[[:alpha:]]+|[[:digit:]]+, greedy WordPiece)
//   sampling ............. bark.cpp:184-270   (+ libstdc++ std::discrete_distribution / std::mt19937)
//   semantic loop ........ bark.cpp:1645-1743
//   coarse loop .......... bark.cpp:1745-1905
//   fine loop ............ bark.cpp:1961-2104
//   generate / lifecycle . bark.cpp:1165-1184, 2125-2232, 2379-2407
#include "../../include/bark_b200.h"
#include "context.h"
#include "gpt_kernels.h"

#include <algorithm>
#include <cmath>
#include <cstring>

using namespace bark;

namespace {

thread_local int g_device_override = -1;   // bark_b200_set_device applies to the calling thread's next bark_load_model
bool quiet() { static const bool q = [] { const char * e = getenv("BARK_B200_QUIET"); return e && *e && *e != '0'; }(); return q; }

// ---------------------------------------------------------------------------------------------
// tokenizer
// ---------------------------------------------------------------------------------------------
inline bool is_alpha(unsigned char c) { return (c >= 'a' && c <= 'z') || (c >= 'A' && c <= 'Z'); }
inline bool is_digit(unsigned char c) { return c >= '0' && c <= '9'; }
inline bool is_punct(unsigned char c) { return c > 32 && c < 127 && !is_alpha(c) && !is_digit(c); }

// Latin-1 letters with diacritics (two-byte UTF-8, lead 0xC3) -> base ASCII letter; 0 if not mapped.
// Same 52 code points as the reference's table (bark.cpp:488-541).
char fold_accent(unsigned char second) {
    const unsigned cp = 0xC0u + (second - 0x80u);          // U+00C0 .. U+00FF
    const bool lower = cp >= 0xE0;
    const unsigned up = lower ? cp - 0x20 : cp;
    char base = 0;
    if (up >= 0xC0 && up <= 0xC5) base = 'A';
    else if (up == 0xC7) base = 'C';
    else if (up >= 0xC8 && up <= 0xCB) base = 'E';
    else if (up >= 0xCC && up <= 0xCF) base = 'I';
    else if (up == 0xD1) base = 'N';
    else if (up >= 0xD2 && up <= 0xD6) base = 'O';
    else if (up >= 0xD9 && up <= 0xDC) base = 'U';
    else if (up == 0xDD) base = 'Y';
    if (!base) return 0;
    return lower ? (char)(base + 32) : base;
}

std::string strip_accents_utf8(const std::string & in) {
    std::string out;
    for (size_t i = 0; i < in.size();) {
        const unsigned char c = (unsigned char) in[i];
        const unsigned hi = c >> 4;
        size_t len = hi < 12 ? 1 : hi < 14 ? 2 : hi == 14 ? 3 : 4;      // lead-byte length table, bark.cpp:480-484
        len = std::min(len, in.size() - i);
        char folded = 0;
        if (len == 2 && c == 0xC3) { const unsigned char d = (unsigned char) in[i + 1]; if (d >= 0x80 && d <= 0xBF) folded = fold_accent(d); }
        if (folded) out.push_back(folded); else out.append(in, i, len);
        i += len;
    }
    return out;
}

// bert_tokenize (bark.cpp:558-620)
void wordpiece(const std::map<std::string, int32_t> & vocab, const std::string & text, std::vector<int32_t> & out, int n_max_tokens) {
    const std::string s = strip_accents_utf8(text);
    out.clear();
    size_t i = 0;
    while (i < s.size()) {
        const unsigned char c = (unsigned char) s[i];
        size_t j = i;
        if (is_punct(c)) j = i + 1;
        else if (is_alpha(c)) { while (j < s.size() && is_alpha((unsigned char) s[j])) j++; }
        else if (is_digit(c)) { while (j < s.size() && is_digit((unsigned char) s[j])) j++; }
        else { i++; continue; }
        const std::string word = s.substr(i, j - i);
        i = j;
        size_t p = 0; bool cont = false;
        while (p < word.size()) {
            if ((int) out.size() >= n_max_tokens - 1) break;
            size_t e = word.size(); bool hit = false;
            for (; e > p; e--) {
                auto it = vocab.find((cont ? "##" : "") + word.substr(p, e - p));
                if (it != vocab.end()) { out.push_back(it->second); p = e; cont = true; hit = true; break; }
            }
            if (!hit) { fprintf(stderr, "%s: unknown token '%c'\n", "bert_tokenize", word[p]); cont = true; p++; }
        }
    }
}

}  // namespace

void bark::tokenize_input(bark_context * ctx, const std::string & text) {         // bark.cpp:622-662
    const bark_context_params & P = ctx->params;
    const int max_ctx = std::min(ctx->semantic.block_size, 256);
    std::vector<int32_t> pieces;
    wordpiece(ctx->token_to_id, text, pieces, max_ctx);
    std::vector<int32_t> t((size_t) max_ctx, 0);
    std::copy(pieces.begin(), pieces.end(), t.begin());
    for (auto & v : t) v += P.text_encoding_offset;                               // offset applied to every slot before padding (quirk D.4)
    for (size_t k = pieces.size(); k < t.size(); k++) t[k] = P.text_pad_token;
    t.insert(t.end(), 256, P.semantic_pad_token);                                 // empty semantic history
    t.push_back(P.semantic_infer_token);
    ctx->tokens = t;
    if (!quiet()) {
        printf("%s: prompt: '%s'\n", "bark_tokenize_input", text.c_str());
        printf("%s: number of tokens in prompt = %zu, first 8 tokens: ", "bark_tokenize_input", ctx->tokens.size());
        for (size_t k = 0; k < std::min<size_t>(8, ctx->tokens.size()); k++) printf("%d ", ctx->tokens[k]);
        printf("\n\n");
    }
}

namespace {

// ---------------------------------------------------------------------------------------------
// sampling (gpt_sample, bark.cpp:249-270)
// ---------------------------------------------------------------------------------------------
int32_t sample_token(bark_context * ctx, GPTModel & m, const float * logits, int n, float temp, float * eos_p) {
    const int64_t t0 = now_us();
    std::vector<float> p(logits, logits + n);
    const float div = temp == 0.0f ? 0.7f : temp;                                 // argmax path still divides by 0.7 (quirk D.3)
    for (float & v : p) v /= div;
    float mx = -INFINITY;
    for (float v : p) mx = std::max(mx, v);
    float sum = 0.0f;
    for (float & v : p) { v = (float) exp((double)(v - mx)); sum += v; }          // reference calls the double exp() on a float argument
    for (float & v : p) v /= sum;
    int32_t next = 0;
    if (temp == 0.0f) {
        float best = -INFINITY;
        for (int i = 0; i < n; i++) if (p[(size_t) i] > best) { best = p[(size_t) i]; next = i; }
    } else {
        std::discrete_distribution<int32_t> dist(p.begin(), p.end());
        next = dist(ctx->rng);
    }
    if (eos_p) *eos_p = p.back();                                                 // probability of the LAST logit (quirk D.2)
    m.t_sample_us += now_us() - t0;
    m.n_sample += 1;
    return next;
}

}  // namespace

// gpt_sample with the uniform draw already made: the reference's arithmetic end to end, discrete_distribution restated
// (bits/random.tcc: normalise in double, sequential partial sums, last one forced to 1.0, lower_bound of the draw).
// Only rows the device kernel flags as too close to call come here.
int32_t bark::sample_token_given_u(const float * logits, int n, float temp, double u, float * eos_p) {
    std::vector<float> p(logits, logits + n);
    const float div = temp == 0.0f ? 0.7f : temp;
    for (float & v : p) v /= div;
    float mx = -INFINITY;
    for (float v : p) mx = std::max(mx, v);
    float sum = 0.0f;
    for (float & v : p) { v = (float) exp((double)(v - mx)); sum += v; }
    for (float & v : p) v /= sum;
    if (eos_p) *eos_p = p.back();
    if (temp == 0.0f) {
        float best = -INFINITY; int32_t next = 0;
        for (int i = 0; i < n; i++) if (p[(size_t) i] > best) { best = p[(size_t) i]; next = i; }
        return next;
    }
    std::vector<double> cp(p.begin(), p.end());
    double tot = 0.0;
    for (double v : cp) tot += v;
    for (double & v : cp) v /= tot;
    for (size_t i = 1; i < cp.size(); i++) cp[i] += cp[i - 1];
    cp.back() = 1.0;
    return (int32_t)(std::lower_bound(cp.begin(), cp.end(), u) - cp.begin());
}

// ---------------------------------------------------------------------------------------------
// stage pieces shared by the single-prompt loops below and the batched ones (batch.cu)
// ---------------------------------------------------------------------------------------------
bool bark::semantic_stop(const bark_context_params & P, int32_t tok, float eos_p) {          // bark.cpp:1675-1677
    return tok == P.semantic_vocab_size || eos_p >= P.min_eos_p;
}

bool bark::coarse_plan(const bark_context_params & P, size_t n_semantic, CoarsePlan * cp) {
    cp->stc_ratio = P.coarse_rate_hz / P.semantic_rate_hz * P.n_coarse_codebooks;
    cp->max_semantic_history = (int) floorf(P.max_coarse_history / cp->stc_ratio);
    cp->n_steps = (int)(floorf(n_semantic * cp->stc_ratio / P.n_coarse_codebooks) * P.n_coarse_codebooks);
    if (cp->n_steps <= 0 || P.n_coarse_codebooks != 2) { fprintf(stderr, "%s: nothing to generate (%zu semantic tokens)\n", "run_coarse", n_semantic); return false; }
    cp->n_windows = (int) ceilf((float) cp->n_steps / P.sliding_window_size);
    return true;
}

std::vector<int32_t> bark::coarse_window_input(const bark_context_params & P, const CoarsePlan & cp, const std::vector<int32_t> & sem, const std::vector<int32_t> & out,
                                               bool kv_reuse, std::vector<int32_t> & kv_ids, size_t & kv_canon, int * n_past) {
    const int step = (int) out.size();
    const int semantic_idx = (int) roundf(step / cp.stc_ratio);
    // window input: semantic tokens from the history start TO THE END, cut/padded to 256 (quirk D.5), infer token, coarse history
    std::vector<int32_t> in(sem.begin() + std::max(semantic_idx - cp.max_semantic_history, 0), sem.end());
    in.resize(256, P.coarse_semantic_pad_token);
    in.push_back(P.coarse_infer_token);
    const size_t hist = std::min<size_t>((size_t) P.max_coarse_history, out.size());
    in.insert(in.end(), out.end() - (std::ptrdiff_t) hist, out.end());
    // Prefix reuse.  The reference re-evaluates the whole window prompt from n_past = 0 (bark.cpp:1795-1812).  Row p of
    // that evaluation depends on the ids at positions <= p and on the call's n_kv — but only through WHERE the summation
    // structure is cut: soft_max switches from the 8-wide polynomial to libm expf at column n_kv & ~7 and the P.V dot
    // from lane chains to the scalar leftovers at column n_kv & ~31 (ggml.c:2845-2888, 2144-2170).  For p < (n_kv & ~31)
    // every column beyond the cut is masked (an exact zero), so the row has ONE value whatever the call's n_kv:
    // "canonical".  Rows [0, n_kv & ~31) of every evaluation here are canonical (by induction over the layers), so a
    // window whose prompt starts with the ids the cache holds re-uses the canonical rows and evaluates the rest in one
    // call with the reference's own n_kv — bit-identical K/V rows and logits, 60-91 rows instead of 257-887.
    *n_past = 0;
    if (kv_reuse) {
        size_t common = 0;
        while (common < kv_ids.size() && common < in.size() && kv_ids[common] == in[common]) common++;
        *n_past = (int) std::min({common, kv_canon, in.size() & ~(size_t) 31, in.size() - 1});       // keep >= 1 id to evaluate
    }
    kv_canon = std::max((size_t) *n_past, in.size() & ~(size_t) 31);
    std::vector<int32_t> in_eval(in.begin() + *n_past, in.end());
    kv_ids = in;
    return in_eval;
}

int bark::coarse_lo(const bark_context_params & P, int step) {                                  // bark.cpp:1829-1833
    return P.semantic_vocab_size + ((step % P.n_coarse_codebooks == 0) ? 0 : 1) * P.codebook_size;
}

void bark::coarse_codes(const bark_context_params & P, const std::vector<int32_t> & out, std::vector<int32_t> & codes) {
    codes.resize(out.size());
    for (size_t i = 0; i + 1 < out.size(); i += 2) {
        codes[i] = out[i] - P.semantic_vocab_size;
        codes[i + 1] = out[i + 1] - P.semantic_vocab_size - P.codebook_size;
    }
}

bool bark::fine_to_audio(bark_context * ctx) {
    // [T][8] -> [8][T]: EnCodec wants one contiguous time series per codebook (bark.cpp:2151-2159)
    const int T = (int) ctx->fine_tokens.size() / 8;
    std::vector<int32_t> codes((size_t) 8 * T);
    for (int c = 0; c < 8; c++) for (int t = 0; t < T; t++) codes[(size_t) c * T + t] = ctx->fine_tokens[(size_t) t * 8 + c];
    if (!audio_params_supported(ctx->params)) return false;
    if (!codec_decode(ctx, codes.data(), T)) { printf("%s: Could not generate waveform from tokens with Encodec\n", "bark_generate_audio"); return false; }
    return true;
}

bool bark::audio_params_supported(const bark_context_params & P) {
    if (P.target_bandwidth != 6 || P.sample_rate != 24000) { fprintf(stderr, "%s: only target_bandwidth 6 / 24 kHz is implemented\n", "bark_generate_audio"); return false; }
    return true;
}

namespace {

void print_stage_stats(const GPTModel & m) {                                      // bark_print_statistics, bark.cpp:176-182
    if (quiet()) return;
    printf("\n\n");
    printf("%s:   sample time = %8.2f ms / %lld tokens\n", "bark_print_statistics", m.t_sample_us / 1000.0f, (long long) m.n_sample);
    printf("%s:  predict time = %8.2f ms / %.2f ms per token\n", "bark_print_statistics", m.t_predict_us / 1000.0f,
           m.n_sample ? m.t_predict_us / (double) m.n_sample / 1000.0 : 0.0);
    printf("%s:    total time = %8.2f ms\n", "bark_print_statistics", m.t_main_us / 1000.0f);
    printf("\n");
}

// ---------------------------------------------------------------------------------------------
// stage loops
// ---------------------------------------------------------------------------------------------
// Runs `n` consecutive sampling steps of one causal stream with the sampler on the device (sampling.cu).  Step 0 evaluates
// `first_in` (a prompt or the single token the host already knows); every later step reads its input token from device
// memory, where the previous step's sampler left it — so all n decode + sample launches are enqueued without a host round
// trip and there is one synchronisation at the end.  lo_of(j) is the offset of step j's logit window in the vocabulary
// (samp_n logits wide); tokens come back with that offset added.  A step the kernel flags as too close to call (see
// sampling.cu) is replayed on the host with the reference's arithmetic and the same uniform draw, and the chain restarts
// behind it; tokens and RNG state are identical to the step-by-step host path either way.
template <typename LoOf>
bool run_chain(bark_context * ctx, GPTModel & m, const std::vector<int32_t> & first_in, bool merge_ctx, int * n_past, int n, LoOf lo_of, int samp_n, float temp,
               int32_t * out_tok, float * out_eos) {
    if (n < 1 || n > 1024) return false;
    const int64_t t_begin = now_us();
    cudaStream_t s = ctx->stream;
    if (temp != 0.0f) {
        for (int j = 0; j < n; j++) ctx->h_u[j] = std::generate_canonical<double, 53>(ctx->rng);     // one draw per sample, as discrete_distribution::operator() makes
        BARK_CUDA_CHECK(cudaMemcpyAsync(ctx->d_u, ctx->h_u, (size_t) n * sizeof(double), cudaMemcpyHostToDevice, s)); bark::g_h2d_bytes += (size_t) n * sizeof(double);
    }
    const bool chain = ctx->use_decode_kernel && m.decode_ok;
    const bool fused = chain && fused_sampler_available(ctx, m, samp_n);
    std::vector<int> past_before((size_t) n);
    std::vector<int32_t> cur_in = first_in;
    std::vector<float> host_logits;
    int start = 0;
    while (start < n) {
        const int stop = chain ? n : start + 1;
        for (int j = start; j < stop; j++) {
            const int lo = lo_of(j);
            past_before[(size_t) j] = *n_past;
            if (j == start) { if (!gpt_eval(ctx, m, cur_in.data(), (int) cur_in.size(), n_past, merge_ctx && *n_past == 0, nullptr, lo, lo + samp_n)) return false; }
            const int force = ctx->debug_flag_every > 0 && (ctx->n_sample_calls++ % ctx->debug_flag_every) == 0;
            if (j > start && fused) {                         // decode + sample in ONE launch (the kernel's last CTA draws the token)
                const FusedSample fs{samp_n, temp, ctx->d_u + j, ctx->d_stok + j, lo, ctx->d_feed, ctx->d_seos + j, ctx->d_sflags + j, force};
                if (!gpt_decode_chained(ctx, m, ctx->d_feed, n_past, lo, lo + samp_n, &fs)) return false;
                continue;
            }
            if (j > start && !gpt_decode_chained(ctx, m, ctx->d_feed, n_past, lo, lo + samp_n)) return false;
            sample_rows(ctx->last_logits + lo, m.n_out_vocab, samp_n, 1, temp, ctx->d_u + j, ctx->d_stok + j, lo, ctx->d_feed, ctx->d_seos + j, ctx->d_sflags + j, force, s);
        }
        const size_t cnt = (size_t)(stop - start);
        BARK_CUDA_CHECK(cudaMemcpyAsync(ctx->h_stok + start, ctx->d_stok + start, cnt * 4, cudaMemcpyDeviceToHost, s));
        BARK_CUDA_CHECK(cudaMemcpyAsync(ctx->h_sflags + start, ctx->d_sflags + start, cnt * 4, cudaMemcpyDeviceToHost, s));
        BARK_CUDA_CHECK(cudaMemcpyAsync(ctx->h_seos + start, ctx->d_seos + start, cnt * 4, cudaMemcpyDeviceToHost, s)); bark::g_d2h_bytes += cnt * 12;
        BARK_CUDA_CHECK(cudaStreamSynchronize(s));
        int f = start;
        while (f < stop && !ctx->h_sflags[f]) f++;
        if (f == stop) { start = stop; if (start < n) cur_in.assign(1, ctx->h_stok[start - 1]); continue; }
        // step f must be decided on the host: re-evaluate it with its logits read back (steps before f stand)
        if (f > start) cur_in.assign(1, ctx->h_stok[f - 1]);
        *n_past = past_before[(size_t) f];
        const int lo = lo_of(f);
        host_logits.resize((size_t) m.n_out_vocab);
        if (!gpt_eval(ctx, m, cur_in.data(), (int) cur_in.size(), n_past, merge_ctx && *n_past == 0, host_logits.data(), lo, lo + samp_n)) return false;
        ctx->h_stok[f] = lo + sample_token_given_u(host_logits.data() + lo, samp_n, temp, ctx->h_u[f], &ctx->h_seos[f]);
        ctx->n_sample_host_replays++;
        start = f + 1;
        cur_in.assign(1, ctx->h_stok[f]);
    }
    for (int j = 0; j < n; j++) { out_tok[j] = ctx->h_stok[j]; if (out_eos) out_eos[j] = ctx->h_seos[j]; }
    m.n_sample += n;
    m.t_predict_us += now_us() - t_begin;      // evaluation and sampling overlap on the device: the split the reference prints does not exist here
    return true;
}

bool run_semantic(bark_context * ctx) {
    const int64_t t_start = now_us();
    GPTModel & m = ctx->semantic;
    const bark_context_params & P = ctx->params;
    std::vector<float> logits((size_t) m.n_out_vocab);
    std::vector<int32_t> input = ctx->tokens, output;
    int n_past = 0; float eos_p = 0.0f;
    const bool dev = ctx->sample_on_device && (size_t) m.n_out_vocab * 4 <= 64 * 1024;
    if (dev) {
        // batches of kBatch steps run ahead of the stop test; if the stop falls inside a batch, the RNG is wound back to
        // where the step-by-step loop would have left it and the surplus steps are dropped (their KV rows are never read)
        constexpr int kBatch = 64;
        std::vector<int32_t> tok(kBatch); std::vector<float> eos(kBatch);
        bool done = false;
        for (int i = 0; i < P.n_steps_text_encoder && !done; i += kBatch) {
            const int nb = std::min(kBatch, P.n_steps_text_encoder - i);
            const std::mt19937 saved = ctx->rng;
            if (!run_chain(ctx, m, input, true, &n_past, nb, [](int) { return 0; }, m.n_out_vocab, P.temp, tok.data(), eos.data())) { fprintf(stderr, "%s: Could not generate token\n", __func__); return false; }
            for (int j = 0; j < nb; j++) {
                if (P.progress_callback) P.progress_callback(ctx, SEMANTIC, 100 * (i + j + 1) / P.n_steps_text_encoder, P.progress_callback_user_data);
                if (semantic_stop(P, tok[(size_t) j], eos[(size_t) j])) {
                    if (P.temp != 0.0f) { ctx->rng = saved; for (int k = 0; k <= j; k++) (void) std::generate_canonical<double, 53>(ctx->rng); }
                    m.n_sample -= nb - (j + 1);
                    done = true; break;
                }
                output.push_back(tok[(size_t) j]);
            }
            if (!done && nb > 0) input.assign(1, tok[(size_t) nb - 1]);
        }
    } else
    for (int i = 0; i < P.n_steps_text_encoder; i++) {
        if (P.progress_callback) P.progress_callback(ctx, SEMANTIC, 100 * (i + 1) / P.n_steps_text_encoder, P.progress_callback_user_data);
        if (!gpt_eval(ctx, m, input.data(), (int) input.size(), &n_past, true, logits.data())) { fprintf(stderr, "%s: Could not generate token\n", __func__); return false; }
        // the reference samples over ALL n_out_vocab logits, not the 10001 "relevant" ones (quirk D.1)
        const int32_t next = sample_token(ctx, m, logits.data(), m.n_out_vocab, P.temp, &eos_p);
        if (semantic_stop(P, next, eos_p)) break;
        input.assign(1, next);
        output.push_back(next);
    }
    ctx->semantic_tokens = output;
    ctx->stats.n_sample_semantic = (int32_t) m.n_sample;
    m.t_main_us = now_us() - t_start;
    ctx->stats.t_semantic_us = m.t_main_us;
    print_stage_stats(m);
    return true;
}

bool run_coarse(bark_context * ctx) {
    const int64_t t_start = now_us();
    GPTModel & m = ctx->coarse;
    const bark_context_params & P = ctx->params;
    const std::vector<int32_t> & sem = ctx->semantic_tokens;
    std::vector<float> logits((size_t) m.n_out_vocab);
    CoarsePlan cp;
    if (!coarse_plan(P, sem.size(), &cp)) return false;
    const int n_steps = cp.n_steps;
    std::vector<int32_t> out; out.reserve((size_t) n_steps);
    const bool dev = ctx->sample_on_device && P.sliding_window_size <= 1024 && P.semantic_vocab_size + 2 * P.codebook_size <= m.n_out_vocab;
    int step = 0;
    std::vector<int32_t> kv_ids;                                                  // ids whose K/V rows the coarse cache holds, by position
    size_t kv_canon = 0;                                                          // leading rows of the cache known to be canonical (coarse_window_input)
    for (int w = 0; w < cp.n_windows; w++) {
        int n_past = 0;
        std::vector<int32_t> in_eval = coarse_window_input(P, cp, sem, out, ctx->kv_reuse, kv_ids, kv_canon, &n_past);
        ctx->n_kv_reused += (unsigned long long) n_past;
        if (dev) {
            // only logits [lo, lo + codebook_size) are ever looked at in this stage (bark.cpp:1829-1833): the window alternates with the codebook
            const int nw = std::min(P.sliding_window_size, n_steps - step), step0 = step;
            std::vector<int32_t> tok((size_t) nw);
            auto lo_of = [&](int j) { return coarse_lo(P, step0 + j); };
            if (!run_chain(ctx, m, in_eval, false, &n_past, nw, lo_of, P.codebook_size, P.temp, tok.data(), nullptr)) { fprintf(stderr, "%s: Could not generate token\n", __func__); return false; }
            for (int j = 0; j < nw; j++) {
                if (P.progress_callback) P.progress_callback(ctx, COARSE, 100 * (step + 1) / n_steps, P.progress_callback_user_data);
                out.push_back(tok[(size_t) j]); step++;
                if (j + 1 < nw) kv_ids.push_back(tok[(size_t) j]);      // the window's last sample is never evaluated
            }
            continue;
        }
        for (int j = 0; j < P.sliding_window_size && step < n_steps; j++) {
            if (P.progress_callback) P.progress_callback(ctx, COARSE, 100 * (step + 1) / n_steps, P.progress_callback_user_data);
            const int lo = coarse_lo(P, step);
            if (j > 0) kv_ids.push_back(in_eval[0]);
            if (!gpt_eval(ctx, m, in_eval.data(), (int) in_eval.size(), &n_past, false, logits.data(), lo, lo + P.codebook_size)) { fprintf(stderr, "%s: Could not generate token\n", __func__); return false; }
            const int32_t next = lo + sample_token(ctx, m, logits.data() + lo, P.codebook_size, P.temp, nullptr);
            in_eval.assign(1, next);
            out.push_back(next);
            step++;
        }
    }
    coarse_codes(P, out, ctx->coarse_tokens);
    ctx->stats.n_sample_coarse = (int32_t) m.n_sample;
    m.t_main_us = now_us() - t_start;
    ctx->stats.t_coarse_us = m.t_main_us;
    print_stage_stats(m);
    return true;
}

}  // namespace

bool bark::run_fine(bark_context * ctx) {
    const int64_t t_start = now_us();
    GPTModel & m = ctx->fine;
    const bark_context_params & P = ctx->params;
    const int n_coarse = P.n_coarse_codebooks, n_cb = P.n_fine_codebooks, cb_size = P.codebook_size;
    if (n_cb != 8 || n_coarse != 2 || cb_size != 1024) { fprintf(stderr, "%s: unsupported codebook configuration\n", __func__); return false; }
    const int T = (int) ctx->coarse_tokens.size() / 2;
    const int len = std::max(T, 1024);
    std::vector<int32_t> arr((size_t) len * 8, cb_size);                          // [len][8], padded with codebook_size (bark.cpp:1982-1996)
    for (int t = 0; t < T; t++) { arr[(size_t) t * 8] = ctx->coarse_tokens[(size_t) t * 2]; arr[(size_t) t * 8 + 1] = ctx->coarse_tokens[(size_t) t * 2 + 1]; }
    const int n_loops = std::max(0, (int) ceilf((len - 1024) / 512.f)) + 1;
    std::vector<float> logits((size_t) 1024 * m.n_out_vocab);
    std::vector<int32_t> buf((size_t) 8 * 1024), sampled(1024);
    const bool dev = ctx->sample_on_device;
    for (int n = 0; n < n_loops; n++) {
        const int start = std::min(n * 512, len - 1024), fill = std::min(n * 512, len - 512), rel = fill - start;
        for (int c = 0; c < 8; c++) for (int j = 0; j < 1024; j++) buf[(size_t) c * 1024 + j] = arr[(size_t)(start + j) * 8 + c];
        for (int nn = n_coarse; nn < n_cb; nn++) {
            if (P.progress_callback) P.progress_callback(ctx, FINE, 100 * (n * (n_cb - n_coarse) + (nn - n_coarse + 1)) / (n_loops * (n_cb - n_coarse)), P.progress_callback_user_data);
            if (ctx->shard.on) {                              // rows of the window split over the GPUs of the job (shard.cu)
                if (!fine_eval_shard(ctx, buf.data(), nn) || !sample_shard(ctx, cb_size, P.fine_temp, sampled.data())) { fprintf(stderr, "%s: Could not generate token\n", __func__); return false; }
            } else {
            if (!fine_eval(ctx, buf.data(), nn, dev ? nullptr : logits.data())) { fprintf(stderr, "%s: Could not generate token\n", __func__); return false; }
            if (dev && !sample_device(ctx, m, ctx->last_logits, m.n_out_vocab, cb_size, 1024, P.fine_temp, sampled.data(), nullptr)) return false;
            }
            for (int i = 0; i < 1024; i++) {
                const int32_t next = (dev || ctx->shard.on) ? sampled[(size_t) i] : sample_token(ctx, m, logits.data() + (size_t) i * m.n_out_vocab, cb_size, P.fine_temp, nullptr);
                // For clips <= 1024 frames (rel == 0) this is the reference's write (bark.cpp:2037).  For longer clips the
                // reference indexes buf[nn*1024 + rel + i] and runs off the buffer (SURVEY finding 5); there we keep the
                // original Bark semantics: every row is sampled (same RNG consumption) and rows >= rel are written in place.
                if (i >= rel) buf[(size_t) nn * 1024 + i] = next;
            }
        }
        for (int nn = n_coarse; nn < n_cb; nn++) for (int j = 0; j < 1024 - rel; j++) arr[(size_t)(fill + j) * 8 + nn] = buf[(size_t) nn * 1024 + rel + j];
    }
    ctx->fine_tokens.assign(arr.begin(), arr.begin() + (std::ptrdiff_t) T * 8);
    ctx->stats.n_sample_fine = (int32_t) m.n_sample;
    m.t_main_us = now_us() - t_start;
    ctx->stats.t_fine_us = m.t_main_us;
    print_stage_stats(m);
    return true;
}

namespace {

void alloc_workspace(bark_context * ctx) {
    int E = 0, H = 0; size_t kp_bytes = 0, n_logits = 0;
    for (GPTModel * m : {&ctx->semantic, &ctx->coarse, &ctx->fine}) {
        E = std::max(E, (int) m->n_embd); H = std::max(H, (int) m->n_head);
        const size_t es = (m->wtype == W_F16 && !ctx->gemm_f32c) ? 2 : 4;
        kp_bytes = std::max(kp_bytes, (size_t) li_padded_k(4 * m->n_embd, (int) es) * es);
    }
    n_logits = std::max<size_t>({(size_t) ctx->semantic.n_out_vocab, (size_t) ctx->coarse.n_out_vocab, (size_t) 1024 * ctx->fine.n_out_vocab});
    Workspace & ws = ctx->ws;
    const size_t R = 1024;
    ws.max_rows = (int) R; ws.E = E;
    ws.x    = (float *) ctx_alloc(ctx, R * E * 4);
    ws.act  = ctx_alloc(ctx, R * kp_bytes);
    ws.act2 = ctx_alloc(ctx, R * kp_bytes);
    ws.q    = (float *) ctx_alloc(ctx, R * E * 4);
    ws.kbuf = (float *) ctx_alloc(ctx, R * E * 4);
    ws.vbuf = (float *) ctx_alloc(ctx, R * E * 4);
    ws.scores = (float *) ctx_alloc(ctx, (size_t) H * R * R * 4);
    ws.logits = (float *) ctx_alloc(ctx, n_logits * 4);
    ws.tok  = (int32_t *) ctx_alloc(ctx, 8 * 1024 * 4);
    if (is_quant(ctx->semantic.wtype) || is_quant(ctx->coarse.wtype) || is_quant(ctx->fine.wtype)) {
        ctx->d_q8 = ctx_alloc(ctx, R * (size_t) 4 * E); ctx->d_q8_scales = ctx_alloc(ctx, R * (size_t)(4 * E / 32) * 4);
        ctx->d_q8_sums = ctx_alloc(ctx, R * (size_t)(4 * E / 32) * 4);
    }
    if (ctx->fast_mode) {
        const GPTModel & fm = ctx->fine;
        if (fm.wtype != W_F16 || fm.n_embd / fm.n_head != 64 || fm.n_embd % 64 != 0 || fm.n_embd > 1024) {
            fprintf(stderr, "bark_b200: BARK_B200_MODE=fast needs f16 fine-model weights with 64-wide heads; using the parity path\n");
            ctx->fast_mode = false;
        } else {
            const size_t FE = (size_t) fm.n_embd;
            ctx->f_a16 = (__half *) ctx_alloc(ctx, R * FE * 2); ctx->f_h16 = (__half *) ctx_alloc(ctx, R * 4 * FE * 2);
            ctx->f_qk16 = (__half *) ctx_alloc(ctx, R * 2 * FE * 2); ctx->f_vt16 = (__half *) ctx_alloc(ctx, FE * R * 2); ctx->f_att16 = (__half *) ctx_alloc(ctx, R * FE * 2);
        }
    }
    BARK_CUDA_CHECK(cudaMallocHost(&ctx->h_logits, n_logits * 4));
    BARK_CUDA_CHECK(cudaMallocHost(&ctx->h_tok, 8 * 1024 * 4));
    ctx->d_u = (double *) ctx_alloc(ctx, 1024 * 8); ctx->d_stok = (int32_t *) ctx_alloc(ctx, 1024 * 4);
    ctx->d_sflags = (int32_t *) ctx_alloc(ctx, 1024 * 4); ctx->d_seos = (float *) ctx_alloc(ctx, 1024 * 4);
    ctx->d_feed = (int32_t *) ctx_alloc(ctx, 64); BARK_CUDA_CHECK(cudaMemset(ctx->d_feed, 0, 64));
    ctx->d_done_counter = (unsigned *) ctx_alloc(ctx, 64); BARK_CUDA_CHECK(cudaMemset(ctx->d_done_counter, 0, 64));
    BARK_CUDA_CHECK(cudaMemset(ctx->d_u, 0, 1024 * 8));
    BARK_CUDA_CHECK(cudaMallocHost(&ctx->h_u, 1024 * 8)); BARK_CUDA_CHECK(cudaMallocHost(&ctx->h_stok, 1024 * 4));
    BARK_CUDA_CHECK(cudaMallocHost(&ctx->h_sflags, 1024 * 4)); BARK_CUDA_CHECK(cudaMallocHost(&ctx->h_seos, 1024 * 4));
}

}  // namespace

// ---------------------------------------------------------------------------------------------
// ggml.h shim
// ---------------------------------------------------------------------------------------------
extern "C" struct ggml_context * ggml_init(struct ggml_init_params) { static int token; return reinterpret_cast<struct ggml_context *>(&token); }   // nothing to initialise: f16 conversions are hardware instructions here
extern "C" void    ggml_free(struct ggml_context *) {}
extern "C" void    ggml_time_init(void) {}
extern "C" int64_t ggml_time_us(void) { return now_us(); }
extern "C" int64_t ggml_time_ms(void) { return now_us() / 1000; }

// ---------------------------------------------------------------------------------------------
// bark.h
// ---------------------------------------------------------------------------------------------
extern "C" struct bark_context_params bark_context_default_params(void) {
    bark_context_params p;
    memset(&p, 0, sizeof(p));
    p.verbosity = LOW;
    p.temp = 0.7f; p.fine_temp = 0.5f; p.min_eos_p = 0.2f;
    p.sliding_window_size = 60; p.max_coarse_history = 630;
    p.sample_rate = 24000; p.target_bandwidth = 6;
    p.cls_token_id = 101; p.sep_token_id = 102;
    p.n_steps_text_encoder = 768;
    p.text_pad_token = 129595; p.text_encoding_offset = 10048;
    p.semantic_rate_hz = 49.9f; p.semantic_pad_token = 10000; p.semantic_vocab_size = 10000; p.semantic_infer_token = 129599;
    p.coarse_rate_hz = 75.0f; p.coarse_infer_token = 12050; p.coarse_semantic_pad_token = 12048;
    p.n_coarse_codebooks = 2; p.n_fine_codebooks = 8; p.codebook_size = 1024;
    p.progress_callback = nullptr; p.progress_callback_user_data = nullptr;
    return p;
}

extern "C" void bark_b200_set_device(int device) { g_device_override = device; }

extern "C" struct bark_context * bark_load_model(const char * model_path, struct bark_context_params params, uint32_t seed) {
    const int64_t t0 = now_us();
    if (!model_path) { fprintf(stderr, "%s: null model path\n", __func__); return nullptr; }
    int n_dev = 0;
    if (cudaGetDeviceCount(&n_dev) != cudaSuccess || n_dev == 0) {
        fprintf(stderr, "%s: no CUDA device available — this library has no CPU path\n", __func__);
        return nullptr;
    }
    int dev = g_device_override;
    if (dev < 0) { const char * e = getenv("BARK_B200_DEVICE"); dev = e ? atoi(e) : 0; }
    if (dev < 0 || dev >= n_dev) { fprintf(stderr, "%s: CUDA device %d out of range (%d present)\n", __func__, dev, n_dev); return nullptr; }
    cudaDeviceProp prop;
    if (cudaSetDevice(dev) != cudaSuccess || cudaGetDeviceProperties(&prop, dev) != cudaSuccess) { fprintf(stderr, "%s: cannot use CUDA device %d: %s\n", __func__, dev, cudaGetErrorString(cudaGetLastError())); return nullptr; }
    if (prop.major != 10) {
        fprintf(stderr, "%s: device %d is sm_%d%d; this library is built for sm_100a (B200) only\n", __func__, dev, prop.major, prop.minor);
        return nullptr;
    }
    bark_context * ctx = new bark_context();
    ctx->device = dev;
    ctx->n_sm = ctx->n_sm_total = prop.multiProcessorCount;
    if (ctx->n_sm >= 132) ctx->n_sm = 128;                    // CTAs of the persistent decode step: 128 measured 1-2 % faster than 148 (fewer pollers per exchange; profiles/r02_decode_headstart_cta_sweep.txt)
    { const char * e = getenv("BARK_B200_MODE"); ctx->fast_mode = e && !strcmp(e, "fast"); }             // "fast": tensor-core fine passes (fast_kernels.cu), not bit-identical
    { const char * e = getenv("BARK_B200_DECODE_CTAS"); if (e && atoi(e) >= 64 && atoi(e) <= ctx->n_sm) ctx->n_sm = atoi(e); }   // experiment knob: CTAs of the persistent decode kernel
    { const char * e = getenv("BARK_B200_SAMPLE_FLAG_EVERY"); ctx->debug_flag_every = e ? atoi(e) : 0; }
    { const char * e = getenv("BARK_B200_SAMPLE"); ctx->sample_on_device = !(e && !strcmp(e, "host")); }      // "host": read logits back and sample on the CPU (A-B)
    { const char * e = getenv("BARK_B200_KV_REUSE"); ctx->kv_reuse = !(e && !strcmp(e, "0")); }              // "0": re-prefill every coarse window like the reference (A-B)
    { const char * e = getenv("BARK_B200_DECODE"); ctx->use_decode_kernel = !(e && !strcmp(e, "multi")); ctx->decode_cluster = e && !strcmp(e, "cluster"); }   // "multi": one kernel per op (debug / A-B)
    { const char * e = getenv("BARK_B200_DECODE_TIMING_TID"); if (e && atoi(e) >= 0 && atoi(e) < 512) ctx->timing_tid = atoi(e) & ~31; }
    { const char * e = getenv("BARK_B200_POLL_NS"); if (e && atoi(e) >= 0 && atoi(e) <= 100000) ctx->poll_ns = (unsigned) atoi(e); }
    { const char * e = getenv("BARK_B200_POLL_ATT_NS"); if (e && atoi(e) >= 0 && atoi(e) <= 100000) ctx->att_ns = (unsigned) atoi(e); }
    { const char * e = getenv("BARK_B200_POLL_FIRST_NS"); if (e && atoi(e) >= 0 && atoi(e) <= 100000) ctx->first_ns = (unsigned) atoi(e); }
    ctx->headstart[1] = ctx->att_ns; ctx->headstart[2] = ctx->headstart[4] = ctx->first_ns;
    { const char * e = getenv("BARK_B200_HEADSTART"); if (e) { unsigned v[6]; if (sscanf(e, "%u:%u:%u:%u:%u:%u", &v[0], &v[1], &v[2], &v[3], &v[4], &v[5]) == 6) for (int i = 0; i < 6; i++) ctx->headstart[i] = std::min(v[i], 100000u); } }
    { const char * e = getenv("BARK_B200_KV_PREFETCH"); ctx->kv_prefetch = e && !strcmp(e, "1"); }
    { const char * e = getenv("BARK_B200_FUSE_SAMPLER"); ctx->fuse_sampler = e && !strcmp(e, "1"); }        // "1": the decode kernel's last CTA samples the token (one launch per token); measured neutral end to end
    { const char * e = getenv("BARK_B200_GEMM_F32C"); ctx->gemm_f32c = e && !strcmp(e, "1"); }
    { const char * e = getenv("BARK_B200_ADAPT"); ctx->adapt_on = e && !strcmp(e, "1"); }                     // "1": self-tuning head starts (experiment; measured WORSE: the feedback is collective and runs away)
    ctx->params = params;
    const bool loaded = guarded(false, [&] {                  // a CUDA failure while loading (out of memory, ...) is a failed load, not an abort
    BARK_CUDA_CHECK(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
    if (!load_model_file(model_path, ctx)) return false;
    alloc_workspace(ctx);
    { const char * e = getenv("BARK_B200_TAG_BASE"); if (e) ctx->tag_base = (unsigned) strtoul(e, nullptr, 0); }      // tests: start the exchange epochs near the 32-bit wrap
    if (getenv("BARK_B200_DECODE_TIMING")) { ctx->d_timing = (unsigned long long *) ctx_alloc(ctx, 256 * 32 * 8); BARK_CUDA_CHECK(cudaMemset(ctx->d_timing, 0, 256 * 32 * 8)); }
    BARK_CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
    return true;
    });
    if (!loaded) {
        fprintf(stderr, "%s: failed to load model weights from '%s'\n", __func__, model_path);
        bark_free(ctx);
        return nullptr;
    }
    ctx->rng = std::mt19937(seed);
    ctx->stats.t_load_us = now_us() - t0;
    return ctx;
}

extern "C" void bark_reset_statistics(struct bark_context * ctx) {
    if (!ctx) return;
    const int64_t load = ctx->stats.t_load_us;
    memset(&ctx->stats, 0, sizeof(ctx->stats));
    ctx->stats.t_load_us = load;          // the reference zeroes the whole struct (bark.cpp:2403-2407) and so reports load time 0 after
                                          // the first generate; keeping it is the useful reading of "load time of the model"
}

extern "C" bool bark_b200_forward_text_encoder(struct bark_context * ctx, int) { return guarded(false, [&] { return ctx && run_semantic(ctx); }); }
extern "C" bool bark_b200_forward_coarse_encoder(struct bark_context * ctx, int) { return guarded(false, [&] { return ctx && run_coarse(ctx); }); }
extern "C" bool bark_b200_forward_fine_encoder(struct bark_context * ctx, int) { return guarded(false, [&] { return ctx && run_fine(ctx); }); }
// the reference also exports these three as C++ symbols without a header (bark.cpp:1703,1865,2061)
BARK_API bool bark_forward_text_encoder(struct bark_context * ctx, int n) { return bark_b200_forward_text_encoder(ctx, n); }
BARK_API bool bark_forward_coarse_encoder(struct bark_context * ctx, int n) { return bark_b200_forward_coarse_encoder(ctx, n); }
BARK_API bool bark_forward_fine_encoder(struct bark_context * ctx, int n) { return bark_b200_forward_fine_encoder(ctx, n); }

static bool bark_generate_audio_impl(struct bark_context * ctx, const char * text, int n_threads) {
    (void) n_threads;                      // CPU thread count of the reference's backend; nothing to size here
    if (!ctx) { fprintf(stderr, "%s: invalid bark context\n", __func__); return false; }
    if (!text) { fprintf(stderr, "%s: null prompt\n", __func__); return false; }
    bark_reset_statistics(ctx);
    const int64_t t0 = now_us();
    BARK_CUDA_CHECK(cudaSetDevice(ctx->device));
    tokenize_input(ctx, text);
    if (!run_semantic(ctx)) { fprintf(stderr, "%s: failed to forward text encoder\n", __func__); return false; }
    if (!run_coarse(ctx))   { fprintf(stderr, "%s: failed to forward coarse encoder\n", __func__); return false; }
    if (!run_fine(ctx))     { fprintf(stderr, "%s: failed to forward fine encoder\n", __func__); return false; }
    if (!fine_to_audio(ctx)) return false;
    ctx->stats.t_eval_us = now_us() - t0;
    return true;
}
extern "C" bool bark_generate_audio(struct bark_context * ctx, const char * text, int n_threads) { return guarded((bool) false, [&] { return bark_generate_audio_impl(ctx, text, n_threads); }); }

extern "C" float * bark_get_audio_data(struct bark_context * ctx) {
    if (!ctx) { fprintf(stderr, "%s: invalid bark context\n", __func__); return nullptr; }
    return ctx->audio.empty() ? nullptr : ctx->audio.data();
}
extern "C" int bark_get_audio_data_size(struct bark_context * ctx) {
    if (!ctx) { fprintf(stderr, "%s: invalid bark context\n", __func__); return 0; }
    return (int) ctx->audio.size();
}
extern "C" int64_t bark_get_load_time(struct bark_context * ctx) {
    if (!ctx) { fprintf(stderr, "%s: invalid bark context\n", __func__); return 0; }
    return ctx->stats.t_load_us;
}
extern "C" int64_t bark_get_eval_time(struct bark_context * ctx) {
    if (!ctx) { fprintf(stderr, "%s: invalid bark context\n", __func__); return 0; }
    return ctx->stats.t_eval_us;
}

extern "C" void bark_free(struct bark_context * ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    if (ctx->stream) cudaStreamSynchronize(ctx->stream);
    for (void * p : ctx->device_allocs) cudaFree(p);
    for (int p = 0; p < ctx->shard.world; p++) if (p != ctx->shard.rank && ctx->shard.peer[p]) cudaIpcCloseMemHandle(ctx->shard.peer[p]);
    if (ctx->shard.local) cudaFree(ctx->shard.local);
    for (int i = 0; i < 3; i++) if (ctx->c_buf[i]) cudaFree(ctx->c_buf[i]);
    if (ctx->c_gi) cudaFree(ctx->c_gi);
    if (ctx->d_codes) cudaFree(ctx->d_codes);
    if (ctx->h_logits) cudaFreeHost(ctx->h_logits);
    if (ctx->h_tok) cudaFreeHost(ctx->h_tok);
    if (ctx->h_u) cudaFreeHost(ctx->h_u);
    if (ctx->h_stok) cudaFreeHost(ctx->h_stok);
    if (ctx->h_sflags) cudaFreeHost(ctx->h_sflags);
    if (ctx->h_seos) cudaFreeHost(ctx->h_seos);
    if (ctx->batch.kv) cudaFree(ctx->batch.kv);
    for (void * p : {(void *) ctx->batch.h_u, (void *) ctx->batch.h_tok, (void *) ctx->batch.h_flags, (void *) ctx->batch.h_eos}) if (p) cudaFreeHost(p);
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
}

// ---------------------------------------------------------------------------------------------
// additive entry points (include/bark_b200.h): per-call hooks for parity tests and the benchmark
// ---------------------------------------------------------------------------------------------
static GPTModel * pick(bark_context * ctx, int which) { return which == 0 ? &ctx->semantic : which == 1 ? &ctx->coarse : which == 2 ? &ctx->fine : nullptr; }

static int bark_b200_gpt_eval_impl(struct bark_context * ctx, int which, const int32_t * tokens, int n, int * n_past, int merge_ctx, float * logits_out) {
    if (!ctx || which < 0 || which > 1 || !tokens || !logits_out) return 0;
    BARK_CUDA_CHECK(cudaSetDevice(ctx->device));
    return gpt_eval(ctx, *pick(ctx, which), tokens, n, n_past, merge_ctx != 0, logits_out) ? 1 : 0;
}
extern "C" int bark_b200_gpt_eval(struct bark_context * ctx, int which, const int32_t * tokens, int n, int * n_past, int merge_ctx, float * logits_out) { return guarded((int) 0, [&] { return bark_b200_gpt_eval_impl(ctx, which, tokens, n, n_past, merge_ctx, logits_out); }); }
static int bark_b200_fine_eval_impl(struct bark_context * ctx, const int32_t * in_buffer, int nn, float * logits_out) {
    if (!ctx || !in_buffer || !logits_out) return 0;
    BARK_CUDA_CHECK(cudaSetDevice(ctx->device));
    return fine_eval(ctx, in_buffer, nn, logits_out) ? 1 : 0;
}
extern "C" int bark_b200_fine_eval(struct bark_context * ctx, const int32_t * in_buffer, int nn, float * logits_out) { return guarded((int) 0, [&] { return bark_b200_fine_eval_impl(ctx, in_buffer, nn, logits_out); }); }
static int bark_b200_encodec_decode_impl(struct bark_context * ctx, const int32_t * codes, int n_frames, float * out, int out_cap) {
    if (!ctx || !codes) return -1;
    BARK_CUDA_CHECK(cudaSetDevice(ctx->device));
    if (!codec_decode(ctx, codes, n_frames)) return -1;
    const int n = (int) ctx->audio.size();
    if (out) memcpy(out, ctx->audio.data(), sizeof(float) * (size_t) std::min(n, out_cap));
    return n;
}
extern "C" int bark_b200_encodec_decode(struct bark_context * ctx, const int32_t * codes, int n_frames, float * out, int out_cap) { return guarded((int) -1, [&] { return bark_b200_encodec_decode_impl(ctx, codes, n_frames, out, out_cap); }); }
extern "C" int bark_b200_sample(struct bark_context * ctx, int which, const float * logits, int n, float temp, float * eos_p) {
    if (!ctx || !logits || n < 1) return -1;
    return sample_token(ctx, *pick(ctx, which < 0 || which > 2 ? 0 : which), logits, n, temp, eos_p);
}
static int bark_b200_sample_rows_impl(struct bark_context * ctx, const float * logits, int n, int rows, float temp, int32_t * tokens_out, float * eos_p_out) {
    if (!ctx || !logits || !tokens_out || rows < 1 || rows > 1024 || n < 2 || (size_t) n * 4 > 64 * 1024) return -1;
    const size_t cap = std::max<size_t>({(size_t) ctx->semantic.n_out_vocab, (size_t) ctx->coarse.n_out_vocab, (size_t) 1024 * ctx->fine.n_out_vocab});
    if ((size_t) rows * n > cap) return -1;
    BARK_CUDA_CHECK(cudaSetDevice(ctx->device));
    BARK_CUDA_CHECK(cudaMemcpyAsync(ctx->ws.logits, logits, (size_t) rows * n * 4, cudaMemcpyHostToDevice, ctx->stream));
    const long long before = ctx->n_sample_host_replays;
    if (!sample_device(ctx, ctx->fine, ctx->ws.logits, n, n, rows, temp, tokens_out, eos_p_out)) return -1;
    return (int)(ctx->n_sample_host_replays - before);
}
extern "C" int bark_b200_sample_rows(struct bark_context * ctx, const float * logits, int n, int rows, float temp, int32_t * tokens_out, float * eos_p_out) { return guarded((int) -1, [&] { return bark_b200_sample_rows_impl(ctx, logits, n, rows, temp, tokens_out, eos_p_out); }); }
extern "C" void bark_b200_reseed(struct bark_context * ctx, uint32_t seed) { if (ctx) ctx->rng = std::mt19937(seed); }
extern "C" void bark_b200_tokenize(struct bark_context * ctx, const char * text, int32_t * out513) {
    if (!ctx || !text || !out513) return;
    tokenize_input(ctx, text);
    memcpy(out513, ctx->tokens.data(), sizeof(int32_t) * 513);
}
extern "C" int bark_b200_get_tokens(struct bark_context * ctx, int stage, int32_t * out, int cap) {
    if (!ctx) return -1;
    const std::vector<int32_t> * v = stage == 0 ? &ctx->semantic_tokens : stage == 1 ? &ctx->coarse_tokens : stage == 2 ? &ctx->fine_tokens : stage == 3 ? &ctx->tokens : nullptr;
    if (!v) return -1;
    if (out) memcpy(out, v->data(), sizeof(int32_t) * std::min(v->size(), (size_t) std::max(cap, 0)));
    return (int) v->size();
}
extern "C" void bark_b200_set_tokens(struct bark_context * ctx, int stage, const int32_t * in, int n) {
    if (!ctx || !in || n < 0) return;
    if (stage == 0) ctx->semantic_tokens.assign(in, in + n); else if (stage == 1) ctx->coarse_tokens.assign(in, in + n); else if (stage == 3) ctx->tokens.assign(in, in + n);
}
extern "C" void bark_b200_get_stats(struct bark_context * ctx, struct bark_statistics * out, int64_t * per_model9) {
    if (!ctx) return;
    if (out) *out = ctx->stats;
    if (per_model9) { const GPTModel * m[3] = {&ctx->semantic, &ctx->coarse, &ctx->fine}; for (int i = 0; i < 3; i++) { per_model9[3 * i] = m[i]->t_predict_us; per_model9[3 * i + 1] = m[i]->t_sample_us; per_model9[3 * i + 2] = m[i]->n_sample; } }
}
extern "C" void bark_b200_get_hparams(struct bark_context * ctx, int which, int32_t * out10) {
    if (!ctx || !out10) return;
    const GPTModel * m = pick(ctx, which); if (!m) return;
    const int32_t v[10] = {m->n_layer, m->n_head, m->n_embd, m->block_size, m->bias, m->n_in_vocab, m->n_out_vocab, m->n_lm_heads, m->n_wtes, m->ftype};
    memcpy(out10, v, sizeof(v));
}
extern "C" unsigned long long bark_b200_kernel_launches(void) { return g_kernel_launches.load(); }
static unsigned bark_b200_layernorm_fallbacks_impl(struct bark_context * ctx) {
    if (!ctx) return 0;
    unsigned v = 0; BARK_CUDA_CHECK(cudaMemcpy(&v, ctx->d_ln_fallbacks, sizeof(v), cudaMemcpyDeviceToHost)); return v;
}
extern "C" unsigned bark_b200_layernorm_fallbacks(struct bark_context * ctx) { return guarded((unsigned) 0, [&] { return bark_b200_layernorm_fallbacks_impl(ctx); }); }
static int bark_b200_decode_timing_impl(struct bark_context * ctx, unsigned long long * out, int n) {
    if (!ctx || !ctx->d_timing || !out) return 0;
    BARK_CUDA_CHECK(cudaMemcpy(out, ctx->d_timing, sizeof(unsigned long long) * (size_t) std::min(n, 256 * 32), cudaMemcpyDeviceToHost));
    return std::min(n, 256 * 32);
}
extern "C" int bark_b200_decode_timing(struct bark_context * ctx, unsigned long long * out, int n) { return guarded((int) 0, [&] { return bark_b200_decode_timing_impl(ctx, out, n); }); }
// fast-mode kernels on host buffers (tests): C[M][N] = A[M][K] W[N][K]^T (f16 in, f32 out), and attention over [n][E] f16 q / k / v
static int bark_b200_fast_gemm_impl(const uint16_t * A, const uint16_t * W, float * C, int M, int N, int K) {
    if (!A || !W || !C || M < 1 || N < 1 || K < 64 || K % 64) return 0;
    __half * dA, * dW; float * dC; int dev = 0, n_sm = 0;
    BARK_CUDA_CHECK(cudaGetDevice(&dev)); BARK_CUDA_CHECK(cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev));
    BARK_CUDA_CHECK(cudaMalloc(&dA, (size_t) M * K * 2)); BARK_CUDA_CHECK(cudaMalloc(&dW, (size_t) N * K * 2)); BARK_CUDA_CHECK(cudaMalloc(&dC, (size_t) M * N * 4));
    BARK_CUDA_CHECK(cudaMemcpy(dA, A, (size_t) M * K * 2, cudaMemcpyHostToDevice)); BARK_CUDA_CHECK(cudaMemcpy(dW, W, (size_t) N * K * 2, cudaMemcpyHostToDevice));
    BARK_CUDA_CHECK(cudaMemset(dC, 0xff, (size_t) M * N * 4));
    FastEpi ep; ep.mode = FEPI_F32; ep.out32 = dC; ep.ldo = N;
    const bool ok = fast_gemm(dA, K, dW, K, M, N, K, ep, n_sm, 0);
    const cudaError_t e = cudaDeviceSynchronize();
    if (e != cudaSuccess) fprintf(stderr, "bark_b200_fast_gemm: %s\n", cudaGetErrorString(e));
    else BARK_CUDA_CHECK(cudaMemcpy(C, dC, (size_t) M * N * 4, cudaMemcpyDeviceToHost));
    cudaFree(dA); cudaFree(dW); cudaFree(dC);
    return ok && e == cudaSuccess;
}
extern "C" int bark_b200_fast_gemm(const uint16_t * A, const uint16_t * W, float * C, int M, int N, int K) { return guarded((int) 0, [&] { return bark_b200_fast_gemm_impl(A, W, C, M, N, K); }); }
static int bark_b200_fast_attention_impl(const uint16_t * q, const uint16_t * k, const uint16_t * v, uint16_t * out, int n, int E, int H) {
    if (!q || !k || !v || !out || n < 256 || n % 256 || E != H * 64) return 0;
    std::vector<uint16_t> qk((size_t) n * 2 * E), vt((size_t) E * n);
    for (int r = 0; r < n; r++) {
        memcpy(&qk[(size_t) r * 2 * E], q + (size_t) r * E, (size_t) E * 2); memcpy(&qk[(size_t) r * 2 * E + E], k + (size_t) r * E, (size_t) E * 2);
        for (int c = 0; c < E; c++) vt[(size_t) c * n + r] = v[(size_t) r * E + c];
    }
    __half * dqk, * dvt, * dout;
    BARK_CUDA_CHECK(cudaMalloc(&dqk, qk.size() * 2)); BARK_CUDA_CHECK(cudaMalloc(&dvt, vt.size() * 2)); BARK_CUDA_CHECK(cudaMalloc(&dout, (size_t) n * E * 2));
    BARK_CUDA_CHECK(cudaMemcpy(dqk, qk.data(), qk.size() * 2, cudaMemcpyHostToDevice)); BARK_CUDA_CHECK(cudaMemcpy(dvt, vt.data(), vt.size() * 2, cudaMemcpyHostToDevice));
    const bool ok = fast_attention(dqk, 2 * E, E, dvt, n, E, H, dout, 0);
    const cudaError_t e = cudaDeviceSynchronize();
    if (e != cudaSuccess) fprintf(stderr, "bark_b200_fast_attention: %s\n", cudaGetErrorString(e));
    else BARK_CUDA_CHECK(cudaMemcpy(out, dout, (size_t) n * E * 2, cudaMemcpyDeviceToHost));
    cudaFree(dqk); cudaFree(dvt); cudaFree(dout);
    return ok && e == cudaSuccess;
}
extern "C" int bark_b200_fast_attention(const uint16_t * q, const uint16_t * k, const uint16_t * v, uint16_t * out, int n, int E, int H) { return guarded((int) 0, [&] { return bark_b200_fast_attention_impl(q, k, v, out, n, E, H); }); }
// the decode kernel's self-tuned head starts, [n_cta][8] nanoseconds (decode_kernels.cu XT_* order); which: 0 semantic, 1 coarse
extern "C" int bark_b200_decode_adapt(struct bark_context * ctx, int which, unsigned * out, int n) {
    if (!ctx || !out || which < 0 || which > 1) return 0;
    return guarded(0, [&] {
        const GPTModel * m = pick(ctx, which);
        if (!m->d_adapt) return 0;
        const int cnt = std::min(n, ctx->n_sm_total * 8);
        BARK_CUDA_CHECK(cudaSetDevice(ctx->device));
        BARK_CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
        BARK_CUDA_CHECK(cudaMemcpy(out, m->d_adapt, (size_t) cnt * 4, cudaMemcpyDeviceToHost));
        return cnt;
    });
}
extern "C" int bark_b200_fast_mode(struct bark_context * ctx) { return ctx && ctx->fast_mode ? 1 : 0; }

extern "C" const char * bark_b200_version(void) { return "bark_b200 r2 (sm_100a; parity path + opt-in tcgen05 fast mode)"; }
