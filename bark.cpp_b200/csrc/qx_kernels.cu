// q4_1, q5_0, q5_1 and q8_0 GPT weights (validated bit-exact against the oracle on a B200 in round 2) — the other
// types the reference's `quantize` tool writes.  Same scheme as q4_kernels.cu (eight lanes own the eight float accumulators of one
// output, one dp4a + one fma per 32-element block, hsum_float_8 as three xor-shuffles), with the per-type details of the pinned AVX2
// build (ggml-quants.c): q5 codes take their fifth bit from qh, q4_1 / q5_1 add `m_w * s_a` per block in ONE scalar fused chain
// (summs) where s_a = f16(d_a * sum(q_a)) comes from the q8_1 activation blocks, q8_0 weights are plain int8.  oracle/bark_oracle.c
// (vec_dot_q4_1_q8_1 ... vec_dot_q8_0_q8_0, pinned against the reference in tests/test_quantize.py) is the executable spec.
// Everything here is NEW code: the kernels the f32 / f16 / q4_0 paths run are not touched (their SASS is unchanged).
#include "epilogue.cuh"
#include "gpt_kernels.h"

namespace bark {

namespace {

__device__ __forceinline__ float f16_at(const unsigned char * p) { return __half2float(__ushort_as_half((unsigned short)(p[0] | (p[1] << 8)))); }
__device__ __forceinline__ uint32_t u32_at(const unsigned char * p) { return (uint32_t) p[0] | ((uint32_t) p[1] << 8) | ((uint32_t) p[2] << 16) | ((uint32_t) p[3] << 24); }
__host__ __device__ inline int block_bytes(int t) { return t == W_Q4_1 ? 20 : t == W_Q5_0 ? 22 : t == W_Q5_1 ? 24 : 34; }

// get_rows on the file's blocks: dequantize_row_q4_1 / q5_0 / q5_1 / q8_0 (ggml-quants.c:1542-1630); x*d + m is one fused multiply-add there
__device__ __forceinline__ float wte_value_q(const void * wte, int t, int E, int row, int i) {
    const int bb = block_bytes(t);
    const unsigned char * blk = (const unsigned char *) wte + ((size_t) row * (E >> 5) + (i >> 5)) * bb;
    const float d = f16_at(blk);
    const int j = i & 31;
    if (t == W_Q8_0) return __fmul_rn((float)(signed char) blk[2 + j], d);
    const unsigned char * qs = blk + (t == W_Q4_1 ? 4 : t == W_Q5_0 ? 6 : 8);
    int q = j < 16 ? (qs[j] & 0x0f) : (qs[j - 16] >> 4);
    if (t != W_Q4_1) q |= (int)((u32_at(blk + (t == W_Q5_0 ? 2 : 4)) >> j) & 1u) << 4;
    if (t == W_Q5_0) return __fmul_rn((float)(q - 16), d);
    return __fmaf_rn((float) q, d, f16_at(blk + 2));
}

__global__ void embed_causal_q_kernel(const void * __restrict__ wte, int wt, const float * __restrict__ wpe, const int32_t * __restrict__ tok,
                                      int N, int n_past, int merge, int E, float * __restrict__ x) {
    const int r = blockIdx.x;
    for (int i = threadIdx.x; i < E; i += blockDim.x) {
        float v;
        if (merge) {
            if (r < 256) v = __fadd_rn(wte_value_q(wte, wt, E, tok[r], i), wte_value_q(wte, wt, E, tok[256 + r], i));
            else         v = wte_value_q(wte, wt, E, tok[512], i);
        } else {
            v = wte_value_q(wte, wt, E, tok[r], i);
        }
        x[(size_t) r * E + i] = __fadd_rn(v, wpe[(size_t)(r + n_past) * E + i]);
    }
}
__global__ void embed_rows_q_kernel(const void * __restrict__ wte, int wt, const float * __restrict__ wpe, RowIds tok, int pos, int E, float * __restrict__ x) {
    const int r = blockIdx.x;
    for (int i = threadIdx.x; i < E; i += blockDim.x) x[(size_t) r * E + i] = __fadd_rn(wte_value_q(wte, wt, E, tok.v[r], i), wpe[(size_t) pos * E + i]);
}
struct FineTablesQ { const void * wte[8]; };
__global__ void embed_fine_q_kernel(FineTablesQ tabs, int wt, const float * __restrict__ wpe, const int32_t * __restrict__ ids, int nn, int E, float * __restrict__ x) {
    const int r = blockIdx.x;
    for (int i = threadIdx.x; i < E; i += blockDim.x) {
        float v = 0.0f;
        for (int c = 0; c <= nn; c++) v = __fadd_rn(v, wte_value_q(tabs.wte[c], wt, E, ids[c * 1024 + r], i));
        x[(size_t) r * E + i] = __fadd_rn(v, wpe[(size_t) r * E + i]);
    }
}

// file blocks -> aligned arrays: qs (16 B, or 32 B for q8_0), qh (u32, q5 only), d and m (f16)
__global__ void split_qx_kernel(const unsigned char * __restrict__ raw, size_t n_blocks, int t, unsigned char * __restrict__ qs, uint32_t * __restrict__ qh,
                                __half * __restrict__ d, __half * __restrict__ m) {
    const size_t b = (size_t) blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= n_blocks) return;
    const unsigned char * p = raw + b * block_bytes(t);
    d[b] = __ushort_as_half((unsigned short)(p[0] | (p[1] << 8)));
    if (t == W_Q4_1 || t == W_Q5_1) m[b] = __ushort_as_half((unsigned short)(p[2] | (p[3] << 8)));
    if (t == W_Q5_0) qh[b] = u32_at(p + 2);
    if (t == W_Q5_1) qh[b] = u32_at(p + 4);
    const unsigned char * src = p + (t == W_Q4_1 ? 4 : t == W_Q5_0 ? 6 : t == W_Q5_1 ? 8 : 2);
    const int nq = t == W_Q8_0 ? 32 : 16;
    for (int i = 0; i < nq; i++) qs[b * nq + i] = src[i];
}

// q8_0 / q8_1 activation blocks (quantize_row_q8_0 / q8_1, AVX2 branches): one warp per (row, block); s = f16(d * sum(q)) with the unrounded d
__global__ void quantize_q8x_kernel(const float * __restrict__ x, int ldx, int rows, int K, int8_t * __restrict__ q, float * __restrict__ d_out, float * __restrict__ s_out) {
    const int nb = K >> 5;
    const size_t w = ((size_t) blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (w >= (size_t) rows * nb) return;
    const int r = (int)(w / nb), b = (int)(w % nb);
    const float v = x[(size_t) r * ldx + b * 32 + lane];
    float amax = fabsf(v);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) amax = fmaxf(amax, __shfl_xor_sync(0xffffffffu, amax, o));
    const float d = __fdiv_rn(amax, 127.0f);
    const float id = amax != 0.0f ? __fdiv_rn(127.0f, amax) : 0.0f;
    const int qi = __float2int_rn(__fmul_rn(v, id));
    q[(size_t) r * K + b * 32 + lane] = (int8_t) qi;
    int sum = qi;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    if (lane == 0) {
        d_out[(size_t) r * nb + b] = __half2float(__float2half_rn(d));
        if (s_out) s_out[(size_t) r * nb + b] = __half2float(__float2half_rn(__fmul_rn(d, (float) sum)));
    }
}

constexpr int kQxMT = 8;

template <int QT>
__global__ void __launch_bounds__(256) qx_matmul_kernel(const unsigned char * __restrict__ qs, const uint32_t * __restrict__ qh, const __half * __restrict__ wd,
                                                        const __half * __restrict__ wm, int K, int O, const int8_t * __restrict__ aq, const float * __restrict__ ad,
                                                        const float * __restrict__ as, int M, MatmulEpilogue ep) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int l = lane & 7, grp = lane >> 3;
    const int o = (blockIdx.x * 8 + warp) * 4 + grp;
    const int m0 = blockIdx.y * kQxMT;
    const int nb = K >> 5;
    const int oc = min(o, O - 1);
    constexpr bool kHasMin = QT == W_Q4_1 || QT == W_Q5_1;
    float acc[kQxMT], summs[kQxMT];
#pragma unroll
    for (int mi = 0; mi < kQxMT; mi++) { acc[mi] = 0.0f; summs[mi] = 0.0f; }
    for (int b = 0; b < nb; b++) {
        const size_t wb = (size_t) oc * nb + b;
        int wi;
        if constexpr (QT == W_Q8_0) {
            wi = __ldg(reinterpret_cast<const int *>(qs + wb * 32) + l);
        } else {
            uint32_t w = __ldg(reinterpret_cast<const uint32_t *>(qs + wb * 16) + (l & 3));
            w = (l >= 4 ? (w >> 4) : w) & 0x0f0f0f0fu;
            if constexpr (QT == W_Q5_0 || QT == W_Q5_1) {
                const uint32_t bits = (__ldg(qh + wb) >> (4 * l)) & 0xfu;                  // element e <-> bit e; this lane's elements are 4l .. 4l+3
                w |= ((bits & 1u) << 4) | ((bits & 2u) << 11) | ((bits & 4u) << 18) | ((bits & 8u) << 25);
            }
            wi = QT == W_Q5_0 ? (int) __vsub4(w, 0x10101010u) : (int) w;                  // q5_0: code - 16; q4_1 / q5_1: unsigned codes <= 31 (fit a signed byte)
        }
        const float dw = __half2float(__ldg(wd + wb));
        const float mw = kHasMin ? __half2float(__ldg(wm + wb)) : 0.0f;
#pragma unroll
        for (int mi = 0; mi < kQxMT; mi++) {
            const int m = min(m0 + mi, M - 1);
            const int yi = __ldg(reinterpret_cast<const int *>(aq + (size_t) m * K + b * 32) + l);
            const float d = __fmul_rn(dw, __ldg(ad + (size_t) m * nb + b));
            acc[mi] = __fmaf_rn(d, (float) __dp4a(wi, yi, 0), acc[mi]);
            if constexpr (kHasMin) summs[mi] = __fmaf_rn(mw, __ldg(as + (size_t) m * nb + b), summs[mi]);   // summs += m * s: one fused chain per output (same in all 8 lanes)
        }
    }
#pragma unroll
    for (int mi = 0; mi < kQxMT; mi++) {
        float t = acc[mi];
        t = __fadd_rn(t, __shfl_xor_sync(0xffffffffu, t, 4));
        t = __fadd_rn(t, __shfl_xor_sync(0xffffffffu, t, 2));
        t = __fadd_rn(t, __shfl_xor_sync(0xffffffffu, t, 1));
        if constexpr (kHasMin) t = __fadd_rn(t, summs[mi]);                               // hsum_float_8(acc) + summs
        if (l == 0 && o < O && m0 + mi < M) matmul_epilogue(ep, m0 + mi, o, t);
    }
}

thread_local int8_t * g_qx_q8 = nullptr; thread_local float * g_qx_d = nullptr, * g_qx_s = nullptr;

}  // namespace

bool qx_supported(WType t) { return t == W_Q4_1 || t == W_Q5_0 || t == W_Q5_1 || t == W_Q8_0; }
size_t qx_block_bytes(WType t) { return (size_t) block_bytes((int) t); }

void qx_split(const void * raw_blocks, size_t n_blocks, WType t, void * qs, void * qh, void * d, void * m, cudaStream_t s) {
    BARK_LAUNCH(split_qx_kernel, (unsigned)((n_blocks + 255) / 256), 256, 0, s, (const unsigned char *) raw_blocks, n_blocks, (int) t, (unsigned char *) qs, (uint32_t *) qh,
                (__half *) d, (__half *) m);
}

void qx_set_scratch(void * q8, void * q8_scales, void * q8_sums) { g_qx_q8 = (int8_t *) q8; g_qx_d = (float *) q8_scales; g_qx_s = (float *) q8_sums; }

void qx_embed_causal(const GPTModel & m, const int32_t * d_tok, int N, int n_past, bool merge, float * x, cudaStream_t s) {
    BARK_LAUNCH(embed_causal_q_kernel, N, 256, 0, s, m.wte[0], (int) m.wtype, m.wpe, d_tok, N, n_past, merge ? 1 : 0, m.n_embd, x);
}
void qx_embed_rows(const GPTModel & m, const RowIds & tok, int B, int pos, float * x, cudaStream_t s) {
    BARK_LAUNCH(embed_rows_q_kernel, B, 256, 0, s, m.wte[0], (int) m.wtype, m.wpe, tok, pos, m.n_embd, x);
}
void qx_embed_fine(const GPTModel & m, const int32_t * d_ids, int nn, float * x, cudaStream_t s) {
    FineTablesQ t; for (int i = 0; i < 8; i++) t.wte[i] = m.wte[i];
    BARK_LAUNCH(embed_fine_q_kernel, 1024, 256, 0, s, t, (int) m.wtype, m.wpe, d_ids, nn, m.n_embd, x);
}

// act: f32 rows [rows][ld_act] as store_act(W_Q4_0) leaves them
void qx_matmul(const DMat & W, const void * act, int ld_act, int rows, const MatmulEpilogue & ep, cudaStream_t s) {
    if (!g_qx_q8 || !g_qx_d || !g_qx_s) { fprintf(stderr, "bark_b200: quantised-weight scratch buffers are not set\n"); throw std::runtime_error("unsupported configuration (see the message above)"); }
    const int nb = W.K / 32;
    const size_t warps = (size_t) rows * nb;
    const bool q81 = W.type == W_Q4_1 || W.type == W_Q5_1;
    BARK_LAUNCH(quantize_q8x_kernel, (unsigned)((warps * 32 + 255) / 256), 256, 0, s, (const float *) act, ld_act, rows, W.K, g_qx_q8, g_qx_d, q81 ? g_qx_s : nullptr);
    g_next_bytes = (double) W.n_out * nb * (double) block_bytes((int) W.type) + (double) rows * (W.K * 1.0 + nb * 8.0 + W.n_out * 4.0);
    g_next_flops = 2.0 * rows * (double) W.n_out * W.K;
    const dim3 grid((W.n_out + 31) / 32, (rows + kQxMT - 1) / kQxMT);
    const unsigned char * qs = (const unsigned char *) W.p; const uint32_t * qh = (const uint32_t *) W.qh; const __half * wd = (const __half *) W.scales, * wm = (const __half *) W.mins;
    switch (W.type) {
        case W_Q4_1: BARK_LAUNCH((qx_matmul_kernel<W_Q4_1>), grid, 256, 0, s, qs, qh, wd, wm, W.K, W.n_out, g_qx_q8, g_qx_d, g_qx_s, rows, ep); break;
        case W_Q5_0: BARK_LAUNCH((qx_matmul_kernel<W_Q5_0>), grid, 256, 0, s, qs, qh, wd, wm, W.K, W.n_out, g_qx_q8, g_qx_d, g_qx_s, rows, ep); break;
        case W_Q5_1: BARK_LAUNCH((qx_matmul_kernel<W_Q5_1>), grid, 256, 0, s, qs, qh, wd, wm, W.K, W.n_out, g_qx_q8, g_qx_d, g_qx_s, rows, ep); break;
        case W_Q8_0: BARK_LAUNCH((qx_matmul_kernel<W_Q8_0>), grid, 256, 0, s, qs, qh, wd, wm, W.K, W.n_out, g_qx_q8, g_qx_d, g_qx_s, rows, ep); break;
        default: fprintf(stderr, "bark_b200: unsupported quantised type %d\n", (int) W.type); throw std::runtime_error("unsupported configuration (see the message above)");
    }
}

}  // namespace bark
