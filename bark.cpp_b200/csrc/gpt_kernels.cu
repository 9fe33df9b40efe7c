// GPT forward kernels, bit-exact ("parity") path.
//
// Replaces, for the B200, the ggml CPU kernels behind bark_build_gpt_graph (bark.cpp:1186-1414) and
// bark_build_fine_gpt_graph (bark.cpp:1416-1584): get_rows/add (ggml.c:13455, 9078), norm+mul+add
// (ggml.c:11964), mul_mat (ggml.c:12369, vec_dot_f16 2251 / vec_dot_f32 2144), scale, diag_mask_inf
// (13865), soft_max (13953) and gelu (2557).  All float arithmetic is issued with explicit IEEE
// intrinsics (__fmaf_rn, __fadd_rn, ...) so nvcc can neither contract nor reassociate it; the
// accumulation order is the reference's (see common.cuh "Lane order").
#include "gpt_kernels.h"
#include "epilogue.cuh"
#include "softmax_row.cuh"

#include <cstring>

namespace bark {

std::atomic<unsigned long long> g_kernel_launches{0};

// ------------------------------------------------------------------------------------------------
// weight re-layout: row-major [n_out][K] -> lane-interleaved [n_out][Kp]
// ------------------------------------------------------------------------------------------------
template <typename T>
__global__ void permute_to_li_kernel(const T * __restrict__ src, T * __restrict__ dst, int n_out, int K, int Kp) {
    constexpr int G = 16 / sizeof(T);
    const size_t total = (size_t) n_out * Kp;
    for (size_t i = (size_t) blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t) gridDim.x * blockDim.x) {
        const int o = (int)(i / Kp), j = (int)(i % Kp);
        // invert li_offset: j = ((c/G)*32 + v)*G + c%G
        const int e = j % G, gv = j / G, v = gv % 32, g = gv / 32;
        const int k = (g * G + e) * 32 + v;
        dst[i] = (k < K) ? src[(size_t) o * K + k] : T(0);
    }
}

void permute_to_li(const void * src, void * dst, int n_out, int K, WType t, cudaStream_t s) {
    if (t == W_F16) { const int Kp = li_padded_k(K, 2); BARK_LAUNCH(permute_to_li_kernel<__half>, 1184, 256, 0, s, (const __half *) src, (__half *) dst, n_out, K, Kp); }
    else            { const int Kp = li_padded_k(K, 4); BARK_LAUNCH(permute_to_li_kernel<float>, 1184, 256, 0, s, (const float *) src, (float *) dst, n_out, K, Kp); }
}

// row-major [n_out][K] -> group-major [groups][o_pad][128] (common.cuh); padding rows / columns are zero
template <typename T>
__global__ void permute_to_gm_kernel(const T * __restrict__ src, T * __restrict__ dst, int n_out, int o_pad, int K) {
    const size_t gs = (size_t) o_pad * kGmGroup, total = (size_t) gm_groups(K) * gs;
    for (size_t i = (size_t) blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t) gridDim.x * blockDim.x) {
        const int g = (int)(i / gs), r = (int)(i % gs), o = r / kGmGroup, w = r % kGmGroup, v = w >> 2, c = w & 3;
        const int k = g * kGmGroup + c * 32 + v;
        dst[i] = (o < n_out && k < K) ? src[(size_t) o * K + k] : T(0);
    }
}

void permute_to_gm(const void * src, void * dst, int n_out, int o_pad, int K, WType t, cudaStream_t s) {
    if (t == W_F16) BARK_LAUNCH(permute_to_gm_kernel<__half>, 1184, 256, 0, s, (const __half *) src, (__half *) dst, n_out, o_pad, K);
    else            BARK_LAUNCH(permute_to_gm_kernel<float>, 1184, 256, 0, s, (const float *) src, (float *) dst, n_out, o_pad, K);
}

// ------------------------------------------------------------------------------------------------
// embeddings
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float wte_value(const void * wte, int wt, int E, int row, int i) {
    if (wt == W_F16) return __half2float(((const __half *) wte)[(size_t) row * E + i]);
    if (wt == W_Q4_0) {                                      // dequantize_row_q4_0 (ggml-quants.c:1515-1533): (nibble - 8) * d on the file's 18-byte blocks
        const unsigned char * blk = (const unsigned char *) wte + ((size_t) row * (E >> 5) + (i >> 5)) * 18;
        const float d = __half2float(__ushort_as_half((unsigned short)(blk[0] | (blk[1] << 8))));
        const int j = i & 31, q = j < 16 ? (blk[2 + j] & 0x0f) : (blk[2 + j - 16] >> 4);
        return __fmul_rn((float)(q - 8), d);
    }
    return ((const float *) wte)[(size_t) row * E + i];
}

// causal models (bark.cpp:1224-1259): one block per position
__global__ void embed_causal_kernel(const void * __restrict__ wte, int wt, const float * __restrict__ wpe, const int32_t * __restrict__ tok,
                                    int N, int n_past, int merge, int E, float * __restrict__ x) {
    const int r = blockIdx.x;
    for (int i = threadIdx.x; i < E; i += blockDim.x) {
        float v;
        if (merge) {
            if (r < 256) v = __fadd_rn(wte_value(wte, wt, E, tok[r], i), wte_value(wte, wt, E, tok[256 + r], i));   // cat_emb = seq + ctx
            else         v = wte_value(wte, wt, E, tok[512], i);
        } else {
            v = wte_value(wte, wt, E, tok[r], i);
        }
        x[(size_t) r * E + i] = __fadd_rn(v, wpe[(size_t)(r + n_past) * E + i]);
    }
}

// fine model (bark.cpp:1454-1472): tok_emb starts as a zeroed leaf, then += wte[c][ids[c][r]] for c = 0..nn
struct FineTables { const void * wte[8]; };
__global__ void embed_fine_kernel(FineTables tabs, int wt, const float * __restrict__ wpe, const int32_t * __restrict__ ids /*[8][1024]*/,
                                  int nn, int E, float * __restrict__ x, int row0) {
    const int r = row0 + blockIdx.x;                        // x holds rows [row0, row0 + gridDim.x) of the window (row-sharded passes: shard.cu)
    for (int i = threadIdx.x; i < E; i += blockDim.x) {
        float v = 0.0f;
        for (int c = 0; c <= nn; c++) v = __fadd_rn(v, wte_value(tabs.wte[c], wt, E, ids[c * 1024 + r], i));
        x[(size_t) blockIdx.x * E + i] = __fadd_rn(v, wpe[(size_t) r * E + i]);
    }
}

// batched decode step (batch.cu): one block per row, every row at position pos
__global__ void embed_rows_kernel(const void * __restrict__ wte, int wt, const float * __restrict__ wpe, RowIds tok, int pos, int E, float * __restrict__ x) {
    const int r = blockIdx.x;
    for (int i = threadIdx.x; i < E; i += blockDim.x) x[(size_t) r * E + i] = __fadd_rn(wte_value(wte, wt, E, tok.v[r], i), wpe[(size_t) pos * E + i]);
}

void gpt_embed_causal(const GPTModel & m, const int32_t * d_tok, int N, int n_past, bool merge, float * x, cudaStream_t s) {
    if (qx_supported(m.wtype)) { qx_embed_causal(m, d_tok, N, n_past, merge, x, s); return; }
    BARK_LAUNCH(embed_causal_kernel, N, 256, 0, s, m.wte[0], (int) m.wtype, m.wpe, d_tok, N, n_past, merge ? 1 : 0, m.n_embd, x);
}
void gpt_embed_rows(const GPTModel & m, const RowIds & tok, int B, int pos, float * x, cudaStream_t s) {
    if (qx_supported(m.wtype)) { qx_embed_rows(m, tok, B, pos, x, s); return; }
    BARK_LAUNCH(embed_rows_kernel, B, 256, 0, s, m.wte[0], (int) m.wtype, m.wpe, tok, pos, m.n_embd, x);
}
void gpt_embed_fine(const GPTModel & m, const int32_t * d_ids, int nn, float * x, cudaStream_t s, int row0, int rows) {
    if (qx_supported(m.wtype)) { qx_embed_fine(m, d_ids, nn, x, s); return; }
    FineTables t; for (int i = 0; i < 8; i++) t.wte[i] = m.wte[i];
    BARK_LAUNCH(embed_fine_kernel, rows, 256, 0, s, t, (int) m.wtype, m.wpe, d_ids, nn, m.n_embd, x, row0);
}

// ------------------------------------------------------------------------------------------------
// LayerNorm (ggml.c:11964-12013) + gain (+ bias) -> activation operand.
// The reference sums the row SEQUENTIALLY in double.  A warp sums it as a tree and then PROVES the
// float it derives (mean, variance) cannot depend on the order: any two double summation orders of
// n terms differ by at most 2*n*2^-53*sum|x|, so if both ends of that interval round to the same
// float the sequential result rounds there too.  Otherwise (probability ~1e-6 per row) lane 0
// replays the sequential loop.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

__global__ void layernorm_act_kernel(const float * __restrict__ x, int rows, int E, const float * __restrict__ g, const float * __restrict__ b,
                                     void * __restrict__ act, int wt, int Kp, float eps, unsigned * __restrict__ fallback_counter) {
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (warp >= rows) return;
    const float * xr = x + (size_t) warp * E;
    const double slack = 2.0 * (double) E * 0x1p-53 * (1.0 + 1e-6);

    double s = 0.0, a = 0.0;
    for (int i = lane; i < E; i += 32) { const double v = (double) xr[i]; s += v; a += fabs(v); }
    s = warp_sum_d(s); a = warp_sum_d(a);
    double d = slack * a;
    float mean = __double2float_rn(__ddiv_rn(s, (double) E));
    if (__double2float_rn(__ddiv_rn(s - d, (double) E)) != __double2float_rn(__ddiv_rn(s + d, (double) E))) {
        double ss = 0.0;
        if (lane == 0) { for (int i = 0; i < E; i++) ss = __dadd_rn(ss, (double) xr[i]); if (fallback_counter) atomicAdd(fallback_counter, 1u); }
        ss = __shfl_sync(0xffffffffu, ss, 0);
        mean = __double2float_rn(__ddiv_rn(ss, (double) E));
    }

    double s2 = 0.0;
    for (int i = lane; i < E; i += 32) { const float v = __fsub_rn(xr[i], mean); s2 += (double) __fmul_rn(v, v); }
    s2 = warp_sum_d(s2);
    d = slack * s2;
    float variance = __double2float_rn(__ddiv_rn(s2, (double) E));
    if (__double2float_rn(__ddiv_rn(s2 - d, (double) E)) != __double2float_rn(__ddiv_rn(s2 + d, (double) E))) {
        double ss = 0.0;
        if (lane == 0) { for (int i = 0; i < E; i++) { const float v = __fsub_rn(xr[i], mean); ss = __dadd_rn(ss, (double) __fmul_rn(v, v)); } if (fallback_counter) atomicAdd(fallback_counter, 1u); }
        ss = __shfl_sync(0xffffffffu, ss, 0);
        variance = __double2float_rn(__ddiv_rn(ss, (double) E));
    }
    const float scale = __fdiv_rn(1.0f, __fsqrt_rn(__fadd_rn(variance, eps)));
    for (int i = lane; i < E; i += 32) {
        float y = __fmul_rn(__fsub_rn(xr[i], mean), scale);      // ggml_vec_scale_f32
        y = __fmul_rn(y, g[i]);                                    // ggml_mul
        if (b) y = __fadd_rn(y, b[i]);                             // ggml_add
        store_act(act, wt, Kp, warp, i, y);
    }
}

void layernorm_act(const float * x, int rows, int E, const float * g, const float * b, void * act, WType wt, int Kp, unsigned * fallback_counter, cudaStream_t s) {
    const int warps_per_block = 8;
    BARK_LAUNCH(layernorm_act_kernel, (rows + warps_per_block - 1) / warps_per_block, warps_per_block * 32, 0, s, x, rows, E, g, b, act, (int) wt, Kp, 1e-5f, fallback_counter);
}

// ------------------------------------------------------------------------------------------------
// mul_mat in lane order.  One warp owns one weight row o and MT activation rows: lane v walks its
// chain with fused multiply-adds, then the fixed tree.  Weights and activations are both in LI
// layout, so each chain group is one coalesced 16-byte load per lane.
// ------------------------------------------------------------------------------------------------
template <typename T> struct Quad;       // lane v's 4 elements of one row of one group of a group-major operand
template <> struct Quad<__half> {
    typedef uint2 V;
    __device__ static void unpack(const uint2 & u, float (&f)[4]) {
        const float2 a = __half22float2(*reinterpret_cast<const __half2 *>(&u.x)), b = __half22float2(*reinterpret_cast<const __half2 *>(&u.y));
        f[0] = a.x; f[1] = a.y; f[2] = b.x; f[3] = b.y;
    }
};
template <> struct Quad<float> {
    typedef uint4 V;
    __device__ static void unpack(const uint4 & u, float (&f)[4]) { f[0] = __uint_as_float(u.x); f[1] = __uint_as_float(u.y); f[2] = __uint_as_float(u.z); f[3] = __uint_as_float(u.w); }
};

// Few-row version (rows < 16: the 1-row lm_head of a prefill, tiny test shapes).  Weights in the row-major LI layout the
// decode kernel streams; activations in the group-major layout every producer writes.
template <typename T, int MT>
__global__ void __launch_bounds__(256) lane_matmul_kernel(const T * __restrict__ W, int K, int Kp, int O, const T * __restrict__ act, int act_gs, int M, MatmulEpilogue ep) {
    constexpr int G = 16 / sizeof(T), QPG = G / 4;             // quads (128-column groups of the activation) per weight group
    typedef typename Quad<T>::V QV;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int o = blockIdx.x * 8 + warp;
    const int m0 = blockIdx.y * MT;
    if (o >= O) return;
    const int nsteps = K >> 5;
    const int ngroups = (nsteps + G - 1) / G;
    const uint4 * wrow = reinterpret_cast<const uint4 *>(W + (size_t) o * Kp) + lane;
    const QV * arow[MT];
    int mvalid = 0;
#pragma unroll
    for (int mi = 0; mi < MT; mi++) { const int m = min(m0 + mi, M - 1); arow[mi] = reinterpret_cast<const QV *>(act + (size_t) m * kGmGroup) + lane; if (m0 + mi < M) mvalid = mi + 1; }
    const size_t qstride = (size_t) act_gs * sizeof(T) / sizeof(QV);      // one activation group, in QV words
    float acc[MT];
#pragma unroll
    for (int mi = 0; mi < MT; mi++) acc[mi] = 0.0f;
    for (int g = 0; g < ngroups; g++) {
        const int steps = min(G, nsteps - g * G);
        float w[G]; unpack16<T>(__ldg(wrow + g * 32), w);
#pragma unroll
        for (int mi = 0; mi < MT; mi++) {
#pragma unroll
            for (int qd = 0; qd < QPG; qd++) {
                if (qd * 4 < steps) {
                    float a[4]; Quad<T>::unpack(__ldg(arow[mi] + (size_t)(g * QPG + qd) * qstride), a);
#pragma unroll
                    for (int e = 0; e < 4; e++) if (qd * 4 + e < steps) acc[mi] = __fmaf_rn(w[qd * 4 + e], a[e], acc[mi]);
                }
            }
        }
    }
#pragma unroll
    for (int mi = 0; mi < MT; mi++) {
        const float r = lane_tree_reduce(acc[mi]);
        if (lane == 0 && mi < mvalid) matmul_epilogue(ep, m0 + mi, o, r);
    }
}

static bool use_tiled() { static const bool t = [] { const char * e = getenv("BARK_B200_GEMM"); return !(e && !strcmp(e, "simple")); }(); return t; }

__global__ void expand_f16_kernel(const __half * __restrict__ src, float * __restrict__ dst, size_t n) {
    for (size_t i = (size_t) blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t) gridDim.x * blockDim.x) dst[i] = __half2float(src[i]);
}
void expand_f16_to_f32(const void * src_f16, void * dst_f32, size_t n, cudaStream_t s) {
    BARK_LAUNCH(expand_f16_kernel, 1184, 256, 0, s, (const __half *) src_f16, (float *) dst_f32, n);
}

void lane_matmul(const DMat & W, const void * act, int act_gs, int rows, const MatmulEpilogue & ep, cudaStream_t s, bool f32_containers) {
    if (W.type == W_Q4_0) { q4_matmul(W, act, act_gs, rows, ep, s); return; }      // act_gs = f32 row stride for this type
    if (qx_supported(W.type)) { qx_matmul(W, act, act_gs, rows, ep, s); return; }
    const int gx = (W.n_out + 7) / 8;
    {   // roofline annotation: algorithmic HBM bytes (weights once + operands) and flops of this mat-mul
        const double es = W.type == W_F16 ? 2.0 : 4.0;
        g_next_bytes = (double) W.n_out * W.K * es + (double) rows * (W.K * es + W.n_out * 4.0);
        g_next_flops = 2.0 * rows * (double) W.n_out * W.K;
    }
    if (rows >= 16 && use_tiled() && (W.type == W_F16 || W.type == W_F32)) { lane_gemm_tiled(W, act, act_gs, rows, ep, s, f32_containers); return; }
    if (f32_containers) { fprintf(stderr, "bark_b200: f32-container operands need the tiled mat-mul (rows >= 16)\n"); throw std::runtime_error("unsupported configuration (see the message above)"); }
    if (W.type == W_F16) {
        if (rows == 1) BARK_LAUNCH((lane_matmul_kernel<__half, 1>), dim3(gx, 1), 256, 0, s, (const __half *) W.p, W.K, W.Kp, W.n_out, (const __half *) act, act_gs, rows, ep);
        else           BARK_LAUNCH((lane_matmul_kernel<__half, 8>), dim3(gx, (rows + 7) / 8), 256, 0, s, (const __half *) W.p, W.K, W.Kp, W.n_out, (const __half *) act, act_gs, rows, ep);
    } else if (W.type == W_F32) {
        if (rows == 1) BARK_LAUNCH((lane_matmul_kernel<float, 1>), dim3(gx, 1), 256, 0, s, (const float *) W.p, W.K, W.Kp, W.n_out, (const float *) act, act_gs, rows, ep);
        else           BARK_LAUNCH((lane_matmul_kernel<float, 8>), dim3(gx, (rows + 7) / 8), 256, 0, s, (const float *) W.p, W.K, W.Kp, W.n_out, (const float *) act, act_gs, rows, ep);
    } else {
        fprintf(stderr, "bark_b200: q4_0 mul_mat is not built in this revision\n"); throw std::runtime_error("unsupported configuration (see the message above)");
    }
}

// ------------------------------------------------------------------------------------------------
// attention (bark.cpp:1302-1339 / 1495-1530)
//   scores[h][q][k] = vec_dot_f32(D, K[k][h], Q[q][h]) * scale, masked to -inf for k > n_past + q
// ------------------------------------------------------------------------------------------------
template <int DSTEPS>
__global__ void attn_scores_kernel(const float * __restrict__ Q, const float * __restrict__ Kc, int N, int n_kv, int n_past, int E, int H,
                                   float scale, int causal, float * __restrict__ S) {
    const int D = DSTEPS * 32;
    const int lane = threadIdx.x & 31;
    const int wq = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);     // (h, q) pair
    if (wq >= H * N) return;
    const int h = wq / N, q = wq % N;
    float qv[DSTEPS];
#pragma unroll
    for (int c = 0; c < DSTEPS; c++) qv[c] = Q[(size_t) q * E + h * D + c * 32 + lane];
    float * srow = S + ((size_t) h * N + q) * n_kv;
    for (int k = 0; k < n_kv; k++) {
        const float * kr = Kc + (size_t) k * E + h * D;
        float acc = 0.0f;
#pragma unroll
        for (int c = 0; c < DSTEPS; c++) acc = __fmaf_rn(kr[c * 32 + lane], qv[c], acc);
        float r = lane_tree_reduce(acc);
        r = __fmul_rn(r, scale);                                              // ggml_scale_inplace
        if (causal && k > n_past + q) r = __int_as_float(0xff800000);         // ggml_diag_mask_inf
        if (lane == (k & 31)) srow[k] = r;
    }
}

// soft_max over one row (ggml.c:13953-14042 + ggml_vec_soft_max_f32 AVX2 branch ggml.c:2845-2888): in place, one warp per row
__global__ void attn_softmax_kernel(float * __restrict__ S, int rows, int n_kv) {
    const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (row >= rows) return;
    softmax_row_warp(S + (size_t) row * n_kv, n_kv, nullptr);
}

// KQV[q][h*D+d] = vec_dot_f32(n_kv, V^T[d][:], P[q][:]) (ggml.c:2144 incl. the compiled leftover handling,
// see oracle/bark_oracle.c orc_vec_dot_f32) -> activation operand for c_proj
__global__ void attn_pv_kernel(const float * __restrict__ S, const float * __restrict__ Vc, int N, int n_kv, int E, int H, int D,
                               void * __restrict__ act, int wt, int Kp) {
    const int d = threadIdx.x, q = blockIdx.x * blockDim.y + threadIdx.y, h = blockIdx.y;
    if (q >= N || d >= D) return;
    const float * p = S + ((size_t) h * N + q) * n_kv;
    const float * v = Vc + h * D + d;
    float acc[32];
#pragma unroll
    for (int l = 0; l < 32; l++) acc[l] = 0.0f;
    const int np = n_kv & ~31;
    for (int k0 = 0; k0 < np; k0 += 32) {
#pragma unroll
        for (int l = 0; l < 32; l++) acc[l] = __fmaf_rn(v[(size_t)(k0 + l) * E], p[k0 + l], acc[l]);
    }
    float sum = lane_tree_reduce_local(acc);
    int i = np, r = n_kv - np;
    while (r >= 8) { for (int l = 0; l < 8; l++) sum = __fadd_rn(sum, __fmul_rn(v[(size_t)(i + l) * E], p[i + l])); i += 8; r -= 8; }
    if (r >= 4)    { for (int l = 0; l < 4; l++) sum = __fadd_rn(sum, __fmul_rn(v[(size_t)(i + l) * E], p[i + l])); i += 4; r -= 4; }
    for (; r > 0; r--, i++) sum = __fmaf_rn(v[(size_t) i * E], p[i], sum);
    store_act(act, wt, Kp, q, h * D + d, sum);
}

void attention(const float * Q, const float * Kc, const float * Vc, int N, int n_kv, int n_past, int E, int H, bool causal,
               float * scores, void * act, WType wt, int Kp, cudaStream_t s) {
    const int D = E / H;
    const float scale = 1.0f / sqrtf((float) E / (float) H);                 // bark.cpp:1318
    const int rows = H * N;
    // (any N: for a single decode row the tiled kernels still spread the keys over ~130 CTAs, where the one-warp-per-(head, query)
    // kernels below walk all keys on 12 warps — 100 us + 77 us per layer in the per-op decode path of quantised models)
    if (use_tiled() && D % 32 == 0 && D <= 128) {
        g_next_bytes = 4.0 * ((double) n_kv * E + (double) N * E + (double) H * N * n_kv); g_next_flops = 2.0 * (double) N * n_kv * E;
        attention_tiled_scores(Q, Kc, N, n_kv, n_past, E, H, scale, causal, scores, s);
        g_next_bytes = 8.0 * (double) rows * n_kv;
        BARK_LAUNCH(attn_softmax_kernel, (rows + 7) / 8, 256, 0, s, scores, rows, n_kv);
        g_next_bytes = 4.0 * ((double) n_kv * E + (double) H * N * n_kv + (double) N * E); g_next_flops = 2.0 * (double) N * n_kv * E;
        attention_tiled_pv(scores, Vc, N, n_kv, E, H, act, wt, Kp, s);
        return;
    }
    g_next_bytes = 4.0 * ((double) n_kv * E + (double) N * E + (double) H * N * n_kv); g_next_flops = 2.0 * (double) N * n_kv * E;
    if (D == 64)       BARK_LAUNCH(attn_scores_kernel<2>, (rows + 7) / 8, 256, 0, s, Q, Kc, N, n_kv, n_past, E, H, scale, causal ? 1 : 0, scores);
    else if (D == 32)  BARK_LAUNCH(attn_scores_kernel<1>, (rows + 7) / 8, 256, 0, s, Q, Kc, N, n_kv, n_past, E, H, scale, causal ? 1 : 0, scores);
    else if (D == 96)  BARK_LAUNCH(attn_scores_kernel<3>, (rows + 7) / 8, 256, 0, s, Q, Kc, N, n_kv, n_past, E, H, scale, causal ? 1 : 0, scores);
    else if (D == 128) BARK_LAUNCH(attn_scores_kernel<4>, (rows + 7) / 8, 256, 0, s, Q, Kc, N, n_kv, n_past, E, H, scale, causal ? 1 : 0, scores);
    else { fprintf(stderr, "bark_b200: unsupported head size %d (need a multiple of 32, <= 128)\n", D); throw std::runtime_error("unsupported configuration (see the message above)"); }
    g_next_bytes = 8.0 * (double) rows * n_kv;
    BARK_LAUNCH(attn_softmax_kernel, (rows + 7) / 8, 256, 0, s, scores, rows, n_kv);
    const int qy = max(1, 256 / D);
    g_next_bytes = 4.0 * ((double) n_kv * E + (double) H * N * n_kv + (double) N * E); g_next_flops = 2.0 * (double) N * n_kv * E;
    BARK_LAUNCH(attn_pv_kernel, dim3((N + qy - 1) / qy, H), dim3(D, qy), 0, s, scores, Vc, N, n_kv, E, H, D, act, (int) wt, Kp);
}

}  // namespace bark
