// ggml_weights.bin -> HBM.
//
// Reads the reference's file format unchanged (writer convert.py:293-350; readers bark.cpp:664-690
// vocab, bark.cpp:692-1078 GPT sections, bark.cpp:1080-1163 container, encodec.cpp/encodec.cpp:141-502
// codec section; layout in DESIGN.md "File format").  Differences in what happens to the bytes:
//   * 2-D GPT matrices are re-laid-out on the device into the lane-interleaved layout (common.cuh);
//   * token tables stay row-major (gather only); 1-D tensors and wpe are f32 as in the file;
//   * codec encoder tensors are validated and skipped (bark never runs the encoder, bark.cpp:2161);
//   * KV caches are f32 [n_layer][block_size][n_embd] in HBM, allocated for the two causal models
//     (bark.cpp:976-991).
// Error behaviour follows the reference: message on stderr, false/nullptr to the caller.
#include "context.h"
#include "codec_kernels.h"
#include "gpt_kernels.h"

#include <cmath>
#include <cstring>
#include <fstream>

namespace bark {

static const uint32_t kMagic = 0x67676d6c;   // GGML_FILE_MAGIC 'ggml'

void * ctx_alloc(bark_context * ctx, size_t bytes) {
    void * p = nullptr;
    BARK_CUDA_CHECK(cudaMalloc(&p, bytes ? bytes : 16));
    ctx->device_allocs.push_back(p);
    return p;
}

namespace {

template <typename T> bool rd(std::ifstream & f, T & v) { f.read(reinterpret_cast<char *>(&v), sizeof(T)); return (bool) f; }

size_t type_bytes(int ttype, size_t nel) {
    switch (ttype) {
        case W_F32: return nel * 4;
        case W_F16: return nel * 2;
        case W_Q4_0: return nel / 32 * 18;
        case W_Q4_1: case W_Q5_0: case W_Q5_1: case W_Q8_0: return nel / 32 * qx_block_bytes((WType) ttype);
        default: return 0;
    }
}

struct TensorHdr { int32_t n_dims = 0, ttype = 0; int32_t ne[3] = {1, 1, 1}; std::string name; size_t nel = 1; };

// returns 1 ok, 0 clean EOF (only legal in the codec section), -1 malformed
int read_hdr(std::ifstream & f, TensorHdr & h) {
    int32_t len = 0;
    if (!rd(f, h.n_dims)) return 0;
    if (!rd(f, len) || !rd(f, h.ttype)) return -1;
    if (h.n_dims < 1 || h.n_dims > 3 || len <= 0 || len > 512) return -1;
    h.ne[0] = h.ne[1] = h.ne[2] = 1; h.nel = 1;
    for (int i = 0; i < h.n_dims; i++) { if (!rd(f, h.ne[i]) || h.ne[i] <= 0) return -1; h.nel *= (size_t) h.ne[i]; }
    h.name.assign((size_t) len, '\0');
    f.read(&h.name[0], len);
    return f ? 1 : -1;
}

// raw bytes of one tensor -> freshly allocated device buffer (row-major, as in the file)
void * upload_raw(bark_context * ctx, std::ifstream & f, size_t bytes, std::vector<char> & host, bool keep) {
    host.resize(bytes);
    f.read(host.data(), (std::streamsize) bytes);
    if (!f) return nullptr;
    void * d = nullptr;
    if (keep) d = ctx_alloc(ctx, bytes); else BARK_CUDA_CHECK(cudaMalloc(&d, bytes));
    BARK_CUDA_CHECK(cudaMemcpyAsync(d, host.data(), bytes, cudaMemcpyHostToDevice, ctx->stream));
    BARK_CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
    return d;
}

struct Slot {              // where a named GPT tensor goes
    enum Kind { VEC, WPE, TABLE, MATRIX } kind;
    int ne0, ne1;
    float ** vec = nullptr; void ** table = nullptr; DMat * mat = nullptr;
    bool gm = false;        // MATRIX: also keep a group-major copy (operand of the multi-row tiled mat-mul)
};

bool load_gpt(bark_context * ctx, std::ifstream & f, GPTModel & m, const char * what) {
    if (!rd(f, m.n_layer) || !rd(f, m.n_head) || !rd(f, m.n_embd) || !rd(f, m.block_size) || !rd(f, m.bias) || !rd(f, m.n_in_vocab) ||
        !rd(f, m.n_out_vocab) || !rd(f, m.n_lm_heads) || !rd(f, m.n_wtes) || !rd(f, m.ftype)) return false;
    if (ctx->params.verbosity >= MEDIUM)
        printf("%s: %s model: n_layer=%d n_head=%d n_embd=%d block_size=%d bias=%d n_in_vocab=%d n_out_vocab=%d n_lm_heads=%d n_wtes=%d ftype=%d\n",
               __func__, what, m.n_layer, m.n_head, m.n_embd, m.block_size, m.bias, m.n_in_vocab, m.n_out_vocab, m.n_lm_heads, m.n_wtes, m.ftype);
    m.ftype %= 1000;                                                          // GGML_QNT_VERSION_FACTOR, bark.cpp:727
    // enum ggml_ftype -> enum ggml_type (ggml.c ggml_ftype_to_ggml_type): 0 f32, 1 f16, 2 q4_0 coincide; q4_1 3 -> 3, q8_0 7 -> 8, q5_0 8 -> 6, q5_1 9 -> 7
    int wt = -1;
    switch (m.ftype) { case 0: wt = W_F32; break; case 1: wt = W_F16; break; case 2: wt = W_Q4_0; break;
                       case 3: wt = W_Q4_1; break; case 7: wt = W_Q8_0; break; case 8: wt = W_Q5_0; break; case 9: wt = W_Q5_1; break; default: break; }
    if (wt < 0) {
        fprintf(stderr, "%s: unsupported weight type (ftype %d) in %s model: this build reads f32, f16, q4_0, q4_1, q5_0, q5_1 and q8_0 GPT weights\n", __func__, m.ftype, what);
        return false;
    }
    m.wtype = (WType) wt;
    const int E = m.n_embd;
    if (m.n_layer <= 0 || m.n_head <= 0 || E <= 0 || E > 1024 || E % 32 != 0 || E % m.n_head != 0 || (E / m.n_head) % 32 != 0 || (E / m.n_head) > 128 ||
        m.block_size <= 0 || m.block_size > 1024 || m.n_wtes < 1 || m.n_wtes > 8 || m.n_lm_heads < 1 || m.n_lm_heads > 8) {
        fprintf(stderr, "%s: unsupported %s model dimensions (need n_embd %% 32 == 0 and <= 1024, head size in {32,64,96,128}, block_size <= 1024)\n", __func__, what);
        return false;
    }
    const bool causal = (m.n_lm_heads == 1 && m.n_wtes == 1);
    if (causal && m.bias) { fprintf(stderr, "%s: %s model has bias=1; linear biases on the causal models are not supported\n", __func__, what); return false; }
    m.layers.assign((size_t) m.n_layer, GPTLayer());

    std::map<std::string, Slot> slots;                                        // same names as bark.cpp:885-938
    auto vec = [&](const std::string & n, float ** p, int len) { Slot s{Slot::VEC, len, 1}; s.vec = p; slots[n] = s; };
    auto mat = [&](const std::string & n, DMat * p, int K, int O, bool gm) { Slot s{Slot::MATRIX, K, O}; s.mat = p; s.gm = gm; slots[n] = s; };
    for (int i = 0; i < m.n_wtes; i++) { Slot s{Slot::TABLE, E, m.n_in_vocab}; s.table = &m.wte[i]; slots["model/wte/" + std::to_string(i)] = s; }
    for (int i = 0; i < m.n_lm_heads; i++) mat("model/lm_head/" + std::to_string(i), &m.lm_head[i], E, m.n_out_vocab, true);   // causal models: one row, or the 16-32 rows of a batched step (batch.cu)
    { Slot s{Slot::WPE, E, m.block_size}; s.vec = &m.wpe; slots["model/wpe"] = s; }
    vec("model/ln_f/g", &m.ln_f_g, E);
    if (m.bias) vec("model/ln_f/b", &m.ln_f_b, E);
    for (int l = 0; l < m.n_layer; l++) {
        const std::string p = "model/h" + std::to_string(l);
        GPTLayer & L = m.layers[(size_t) l];
        vec(p + "/ln_1/g", &L.ln_1_g, E); vec(p + "/ln_2/g", &L.ln_2_g, E);
        if (m.bias) { vec(p + "/ln_1/b", &L.ln_1_b, E); vec(p + "/ln_2/b", &L.ln_2_b, E); }
        mat(p + "/attn/c_attn/w", &L.c_attn, E, 3 * E, true); mat(p + "/attn/c_proj/w", &L.c_proj, E, E, true);
        mat(p + "/mlp/c_fc/w", &L.fc, E, 4 * E, true);        mat(p + "/mlp/c_proj/w", &L.proj, 4 * E, E, true);
    }

    int32_t n_tensors = 0;
    if (!rd(f, n_tensors) || n_tensors < 0) return false;
    std::vector<char> host;
    size_t total = 0;
    for (int i = 0; i < n_tensors; i++) {
        TensorHdr h;
        if (read_hdr(f, h) != 1 || h.n_dims > 2) { fprintf(stderr, "%s: malformed tensor record in %s model\n", __func__, what); return false; }
        auto it = slots.find(h.name);
        if (it == slots.end()) { fprintf(stderr, "%s: unknown tensor '%s' in model file\n", __func__, h.name.c_str()); return false; }
        const Slot & s = it->second;
        if (h.ne[0] != s.ne0 || h.ne[1] != s.ne1) {
            fprintf(stderr, "%s: tensor '%s' has wrong shape in model file: got [%d, %d], expected [%d, %d]\n", __func__, h.name.c_str(), h.ne[0], h.ne[1], s.ne0, s.ne1);
            return false;
        }
        const int want = (s.kind == Slot::VEC || s.kind == Slot::WPE) ? (int) W_F32 : (int) m.wtype;
        if (h.ttype != want) { fprintf(stderr, "%s: tensor '%s' has wrong type in model file: got %d, expected %d\n", __func__, h.name.c_str(), h.ttype, want); return false; }
        const size_t bytes = type_bytes(h.ttype, h.nel);
        total += bytes;
        if (s.kind == Slot::MATRIX) {
            void * raw = upload_raw(ctx, f, bytes, host, false);
            if (!raw) return false;
            DMat & d = *s.mat;
            if (qx_supported(m.wtype)) {                     // experimental types: qs / qh / d / m arrays (qx_kernels.cu)
                const size_t n_blocks = h.nel / 32;
                d.n_out = s.ne1; d.K = s.ne0; d.Kp = d.K; d.type = m.wtype;
                d.p = ctx_alloc(ctx, n_blocks * (m.wtype == W_Q8_0 ? 32 : 16)); d.scales = ctx_alloc(ctx, n_blocks * 2);
                d.mins = ctx_alloc(ctx, n_blocks * 2); d.qh = ctx_alloc(ctx, n_blocks * 4);
                qx_split(raw, n_blocks, m.wtype, d.p, d.qh, d.scales, d.mins, ctx->stream);
                BARK_CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
                BARK_CUDA_CHECK(cudaFree(raw));
                continue;
            }
            if (m.wtype == W_Q4_0) {                         // 18-byte blocks -> aligned nibble words + f16 scales (q4_kernels.cu)
                const size_t n_blocks = h.nel / 32;
                d.n_out = s.ne1; d.K = s.ne0; d.Kp = d.K; d.type = W_Q4_0;
                d.p = ctx_alloc(ctx, n_blocks * 16); d.scales = ctx_alloc(ctx, n_blocks * 2);
                q4_split(raw, n_blocks, d.p, d.scales, ctx->stream);
                BARK_CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
                BARK_CUDA_CHECK(cudaFree(raw));
                if (ctx->params.verbosity == HIGH) printf("%48s - [%5d, %5d], type = %d, %6.2f MB\n", h.name.c_str(), h.ne[0], h.ne[1], h.ttype, bytes / 1024.0 / 1024.0);
                continue;
            }
            d.n_out = s.ne1; d.K = s.ne0; d.type = m.wtype; d.Kp = li_padded_k(d.K, m.wtype == W_F16 ? 2 : 4);
            d.p = ctx_alloc(ctx, (size_t) d.n_out * d.Kp * (m.wtype == W_F16 ? 2 : 4));
            permute_to_li(raw, d.p, d.n_out, d.K, m.wtype, ctx->stream);
            if (s.gm) {                                  // second copy for the multi-row tiled mat-mul (group-major, rows padded to 16)
                d.o_pad = (d.n_out + 15) / 16 * 16;
                const size_t gm_bytes = (size_t) gm_groups(d.K) * d.o_pad * kGmGroup * (m.wtype == W_F16 ? 2 : 4);
                d.p_gm = ctx_alloc(ctx, gm_bytes);
                permute_to_gm(raw, d.p_gm, d.n_out, d.o_pad, d.K, m.wtype, ctx->stream);
                if (ctx->gemm_f32c && m.wtype == W_F16) {    // f16 values in f32 containers for the tiled mat-mul (no conversions in its inner loop)
                    const size_t n_el = gm_bytes / 2;
                    d.p_gm32 = ctx_alloc(ctx, n_el * 4);
                    expand_f16_to_f32(d.p_gm, d.p_gm32, n_el, ctx->stream);
                }
            }
            BARK_CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
            if (ctx->fast_mode && !causal && m.wtype == W_F16) { d.p_rm = raw; ctx->device_allocs.push_back(raw); }   // fast mode: the tensor cores read the file's own row-major layout
            else BARK_CUDA_CHECK(cudaFree(raw));
        } else {
            void * raw = upload_raw(ctx, f, bytes, host, true);
            if (!raw) return false;
            if (s.kind == Slot::TABLE) *s.table = raw; else *s.vec = (float *) raw;
        }
        if (ctx->params.verbosity == HIGH) printf("%48s - [%5d, %5d], type = %d, %6.2f MB\n", h.name.c_str(), h.ne[0], h.ne[1], h.ttype, bytes / 1024.0 / 1024.0);
    }
    // the reference does not notice missing tensors (bark.cpp:1007-1068); here they would be null device pointers, so check
    for (auto & kv : slots) {
        const Slot & s = kv.second;
        const bool present = s.kind == Slot::MATRIX ? s.mat->p != nullptr : s.kind == Slot::TABLE ? *s.table != nullptr : *s.vec != nullptr;
        if (!present) { fprintf(stderr, "%s: tensor '%s' missing from the %s model\n", __func__, kv.first.c_str(), what); return false; }
    }
    if (causal) {
        const size_t n = (size_t) m.n_layer * m.block_size * E;
        m.mem_k = (float *) ctx_alloc(ctx, n * 4); m.mem_v = (float *) ctx_alloc(ctx, n * 4);
        BARK_CUDA_CHECK(cudaMemsetAsync(m.mem_k, 0, n * 4, ctx->stream)); BARK_CUDA_CHECK(cudaMemsetAsync(m.mem_v, 0, n * 4, ctx->stream));
    }
    if (ctx->params.verbosity >= MEDIUM) printf("%s: %s model size = %8.2f MB\n", __func__, what, total / 1024.0 / 1024.0);
    return true;
}

bool load_codec(bark_context * ctx, std::ifstream & f, CodecModel & c) {
    uint32_t magic = 0; int32_t hp[9];
    if (!rd(f, magic) || magic != kMagic) { fprintf(stderr, "%s: invalid model file (bad magic)\n", __func__); return false; }
    for (int i = 0; i < 9; i++) if (!rd(f, hp[i])) return false;
    // in_channels, hidden_dim, n_filters, kernel_size, residual_kernel_size, n_bins, bandwidth, sr, ftype (encodec.cpp:156-165)
    c.hidden_dim = hp[1]; c.n_filters = hp[2]; c.kernel_size = hp[3]; c.res_kernel = hp[4]; c.n_bins = hp[5];
    const int ftype = hp[8] % 1000;
    if (hp[0] != 1 || c.hidden_dim != 128 || c.n_filters != 32 || c.kernel_size != 7 || c.res_kernel != 3) {
        fprintf(stderr, "%s: unsupported codec hyper-parameters (this build implements the 24 kHz EnCodec decoder)\n", __func__); return false;
    }
    if (ftype != W_F16) {   // an all-f32 codec cannot run in the reference either (ggml.c:14899 asserts an f16 kernel)
        fprintf(stderr, "%s: codec weights must be f16 (ftype %d)\n", __func__, ftype); return false;
    }
    struct CSlot { ConvW * cv = nullptr; bool is_w = false, transposed = false; __half ** hw = nullptr; float ** fb = nullptr; int ne[3]; };
    std::map<std::string, CSlot> slots;
    const int nf = c.n_filters, ks = c.kernel_size, rk = c.res_kernel;
    static const int ratios[4] = {8, 5, 4, 2};
    auto conv = [&](const std::string & base, ConvW * cv, int k, int cin, int cout, bool transposed) {
        cv->k = k; cv->cin = cin; cv->cout = cout;
        CSlot w; w.cv = cv; w.is_w = true; w.transposed = transposed; w.ne[0] = k; w.ne[1] = transposed ? cout : cin; w.ne[2] = transposed ? cin : cout; slots[base + ".weight"] = w;
        CSlot b; b.cv = cv; b.is_w = false; b.ne[0] = cout; b.ne[1] = 1; b.ne[2] = 1; slots[base + ".bias"] = b;
    };
    int mult = 16;
    conv("decoder.model.0.conv.conv", &c.init, ks, c.hidden_dim, mult * nf, false);
    for (int l = 0; l < 2; l++) {
        const int Hn = mult * nf;
        CSlot a; a.hw = &c.lstm_ih_w[l]; a.ne[0] = Hn; a.ne[1] = 4 * Hn; a.ne[2] = 1; slots["decoder.model.1.lstm.weight_ih_l" + std::to_string(l)] = a;
        CSlot b; b.hw = &c.lstm_hh_w[l]; b.ne[0] = Hn; b.ne[1] = 4 * Hn; b.ne[2] = 1; slots["decoder.model.1.lstm.weight_hh_l" + std::to_string(l)] = b;
        CSlot d; d.fb = &c.lstm_ih_b[l]; d.ne[0] = 4 * Hn; d.ne[1] = 1; d.ne[2] = 1; slots["decoder.model.1.lstm.bias_ih_l" + std::to_string(l)] = d;
        CSlot e; e.fb = &c.lstm_hh_b[l]; e.ne[0] = 4 * Hn; e.ne[1] = 1; e.ne[2] = 1; slots["decoder.model.1.lstm.bias_hh_l" + std::to_string(l)] = e;
    }
    for (int i = 0; i < 4; i++) {
        const int ch = mult * nf;
        const std::string up = "decoder.model." + std::to_string(3 * (i + 1)), rb = "decoder.model." + std::to_string(3 * (i + 1) + 1);
        conv(up + ".convtr.convtr", &c.blk[i].us, 2 * ratios[i], ch, ch / 2, true);
        conv(rb + ".block.1.conv.conv", &c.blk[i].c1, rk, ch / 2, ch / 4, false);
        conv(rb + ".block.3.conv.conv", &c.blk[i].c2, 1, ch / 4, ch / 2, false);
        conv(rb + ".shortcut.conv.conv", &c.blk[i].sc, 1, ch / 2, ch / 2, false);
        mult /= 2;
    }
    conv("decoder.model.15.conv.conv", &c.final_conv, ks, nf, 1, false);

    std::vector<char> host;
    size_t total = 0;
    for (;;) {
        TensorHdr h;
        const int r = read_hdr(f, h);
        if (r == 0) break;
        if (r < 0) { fprintf(stderr, "%s: malformed tensor record in codec section\n", __func__); return false; }
        const size_t bytes = type_bytes(h.ttype, h.nel);
        if (bytes == 0) { fprintf(stderr, "%s: tensor '%s' has unsupported type %d\n", __func__, h.name.c_str(), h.ttype); return false; }
        total += bytes;
        int q = -1;
        if (h.name.compare(0, 8, "encoder.") == 0) { f.seekg((std::streamoff) bytes, std::ios::cur); if (!f) return false; continue; }
        if (sscanf(h.name.c_str(), "quantizer.vq.layers.%d._codebook.embed", &q) == 1) {
            if (h.ttype != W_F32 || h.ne[0] != c.hidden_dim || h.ne[1] != c.n_bins) { fprintf(stderr, "%s: tensor '%s' has wrong shape/type\n", __func__, h.name.c_str()); return false; }
            if (q >= 0 && q < 8) { c.embed[q] = (float *) upload_raw(ctx, f, bytes, host, true); if (!c.embed[q]) return false; }
            else f.seekg((std::streamoff) bytes, std::ios::cur);      // bark uses codebooks 0..7 only (bandwidth 6, utils.h:22-30)
            continue;
        }
        auto it = slots.find(h.name);
        if (it == slots.end()) { fprintf(stderr, "%s: unknown tensor '%s' in model file\n", __func__, h.name.c_str()); return false; }
        CSlot & s = it->second;
        if (h.ne[0] != s.ne[0] || h.ne[1] != s.ne[1] || h.ne[2] != s.ne[2]) {
            fprintf(stderr, "%s: tensor '%s' has wrong shape in model file: got [%d, %d, %d], expected [%d, %d, %d]\n", __func__, h.name.c_str(),
                    h.ne[0], h.ne[1], h.ne[2], s.ne[0], s.ne[1], s.ne[2]);
            return false;
        }
        const bool is_weight = s.hw || (s.cv && s.is_w);
        if (h.ttype != (is_weight ? (int) W_F16 : (int) W_F32)) { fprintf(stderr, "%s: tensor '%s' has wrong type %d\n", __func__, h.name.c_str(), h.ttype); return false; }
        if (!is_weight) {
            void * d = upload_raw(ctx, f, bytes, host, true);
            if (!d) return false;
            if (s.fb) *s.fb = (float *) d; else s.cv->b = (float *) d;
            continue;
        }
        // f16 weights -> lane-interleaved rows (common.cuh) so every codec dot product streams like the GPT mat-muls
        __half * raw = (__half *) upload_raw(ctx, f, bytes, host, false);
        if (!raw) return false;
        int rows, K;
        __half * tmp = nullptr;
        const bool transposed = s.cv && s.transposed;
        if (s.hw) { rows = s.ne[1]; K = s.ne[0]; }
        else if (transposed) {                                               // stored [Cin][Cout][k] -> rows [Cout*k] x Cin
            rows = s.cv->cout * s.cv->k; K = s.cv->cin;
            BARK_CUDA_CHECK(cudaMalloc(&tmp, bytes));
            convtr_rows(raw, tmp, s.cv->cin, s.cv->cout, s.cv->k, ctx->stream);
        } else { rows = s.cv->cout; K = s.cv->cin * s.cv->k; }               // stored [Cout][Cin][k]: row o, column c*k + j (im2col order)
        if (K % 32 != 0 && (s.hw || transposed)) { fprintf(stderr, "%s: tensor '%s': contraction length %d is not a multiple of 32\n", __func__, h.name.c_str(), K); return false; }
        const int Kp = li_padded_k(K, 2);
        __half * li = (__half *) ctx_alloc(ctx, (size_t) rows * Kp * sizeof(__half));
        permute_to_li(tmp ? tmp : raw, li, rows, K, W_F16, ctx->stream);
        BARK_CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
        BARK_CUDA_CHECK(cudaFree(raw));
        if (tmp) BARK_CUDA_CHECK(cudaFree(tmp));
        if (s.hw) { *s.hw = li; c.lstm_Kp = Kp; } else { s.cv->w = li; s.cv->Kp = Kp; }
    }
    for (auto & kv : slots) {
        const CSlot & s = kv.second;
        const bool present = s.hw ? *s.hw != nullptr : s.fb ? *s.fb != nullptr : s.is_w ? s.cv->w != nullptr : s.cv->b != nullptr;
        if (!present) { fprintf(stderr, "%s: tensor '%s' missing from the codec section\n", __func__, kv.first.c_str()); return false; }
    }
    for (int q = 0; q < 8; q++) if (!c.embed[q]) { fprintf(stderr, "%s: codebook %d missing\n", __func__, q); return false; }
    if (ctx->params.verbosity >= MEDIUM) printf("%s: codec model size = %.2f MB\n", __func__, total / 1024.0 / 1024.0);
    return true;
}

}  // namespace

bool load_model_file(const std::string & path, bark_context * ctx) {
    std::ifstream f(path, std::ios::binary);
    if (!f) { fprintf(stderr, "%s: failed to open '%s'\n", __func__, path.c_str()); return false; }
    uint32_t magic = 0;
    if (!rd(f, magic) || magic != kMagic) { fprintf(stderr, "%s: invalid model file '%s' (bad magic)\n", __func__, path.c_str()); return false; }
    int32_t n_vocab = 0;
    if (!rd(f, n_vocab) || n_vocab < 0) { fprintf(stderr, "%s: failed to load vocab\n", __func__); return false; }
    std::string word;
    for (int i = 0; i < n_vocab; i++) {
        uint32_t len = 0;
        if (!rd(f, len) || len > (1u << 20)) { fprintf(stderr, "%s: failed to load vocab\n", __func__); return false; }
        word.assign(len, '\0');
        if (len) f.read(&word[0], len);
        ctx->token_to_id[word] = i;                                          // later duplicates win, like the reference's map assignment
    }
    if (!load_gpt(ctx, f, ctx->semantic, "text"))   { fprintf(stderr, "%s: invalid model file '%s' (bad text)\n", __func__, path.c_str()); return false; }
    if (!load_gpt(ctx, f, ctx->coarse, "coarse"))   { fprintf(stderr, "%s: invalid model file '%s' (bad coarse)\n", __func__, path.c_str()); return false; }
    if (!load_gpt(ctx, f, ctx->fine, "fine"))       { fprintf(stderr, "%s: invalid model file '%s' (bad fine)\n", __func__, path.c_str()); return false; }
    if (ctx->fine.n_wtes != 8 || ctx->fine.n_lm_heads != 7 || !ctx->fine.bias || ctx->fine.block_size != 1024) {
        fprintf(stderr, "%s: unexpected fine model layout (need 8 wtes, 7 lm_heads, LayerNorm biases, block_size 1024)\n", __func__); return false;
    }
    if (!load_codec(ctx, f, ctx->codec)) { fprintf(stderr, "%s: invalid model file '%s' (bad encodec)\n", __func__, path.c_str()); return false; }

    // GELU lookup table, built the way ggml_init does (ggml.c:3795-3810 with ggml_gelu_f32, ggml.c:2546) using the
    // host's tanhf.  The pinned reference build evaluates 1 + 0.044715*x*x as one fused multiply-add
    // (tests/test_oracle_vs_ref.py compares all 65536 entries against the reference's table).
    {
        std::vector<__half> tab(65536);
        const float A = 0.044715f, S = 0.79788456080286535587989211986876f;
        for (int i = 0; i < 65536; i++) {
            const __half hx = __ushort_as_half((unsigned short) i);
            const float x = __half2float(hx);
            const float inner = std::fmaf(A * x, x, 1.0f);
            const float g = (0.5f * x) * (1.0f + std::tanh((S * x) * inner));
            tab[(size_t) i] = __float2half_rn(g);
        }
        ctx->d_gelu_tab = (__half *) ctx_alloc(ctx, 65536 * sizeof(__half));
        BARK_CUDA_CHECK(cudaMemcpy(ctx->d_gelu_tab, tab.data(), 65536 * sizeof(__half), cudaMemcpyHostToDevice));
    }
    ctx->d_ln_fallbacks = (unsigned *) ctx_alloc(ctx, 4 * sizeof(unsigned));
    BARK_CUDA_CHECK(cudaMemset(ctx->d_ln_fallbacks, 0, 4 * sizeof(unsigned)));
    // f32, f16 and q4_0 models decode in the persistent kernel; the other quantised types step through the per-op kernels (decode_ok stays false)
    if (!is_quant(ctx->semantic.wtype) || ctx->semantic.wtype == W_Q4_0) build_decode_tables(ctx, ctx->semantic);
    if (!is_quant(ctx->coarse.wtype) || ctx->coarse.wtype == W_Q4_0) build_decode_tables(ctx, ctx->coarse);
    return true;
}

}  // namespace bark
