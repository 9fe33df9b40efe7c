// soft_max over one attention row in the reference's order, run by ONE full warp (ggml.c:13953-14042 + the AVX2 branch of
// ggml_vec_soft_max_f32, ggml.c:2845-2888).  Shared by the per-op attention (gpt_kernels.cu attn_softmax_kernel) and the
// batched decode attention (batch_kernels.cu).  p: n_kv <= 1024 scores, in global or shared memory, replaced by the
// probabilities.  fallback_counter (may be null) counts the rows whose normaliser had to be replayed sequentially.
#pragma once
#include "common.cuh"

namespace bark {

__device__ __forceinline__ void softmax_row_warp(float * p, int n_kv, unsigned * fallback_counter) {
    const int lane = threadIdx.x & 31;
    float mx = __int_as_float(0xff800000);
    for (int i = lane; i < n_kv; i += 32) mx = fmaxf(mx, p[i]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    const int nchunks = n_kv >> 3;
    float csum[4] = {0.f, 0.f, 0.f, 0.f};                                    // chunk c is owned by lane c%32, slot c/32 (n_kv <= 1024)
#pragma unroll
    for (int slot = 0; slot < 4; slot++) {
        const int c = slot * 32 + lane;
        if (c < nchunks) {
            float v[8];
#pragma unroll
            for (int l = 0; l < 8; l++) { v[l] = ggml_v_expf_dev(__fsub_rn(p[c * 8 + l], mx)); }
#pragma unroll
            for (int l = 0; l < 8; l++) p[c * 8 + l] = v[l];
            const float t0 = __fadd_rn(v[4], v[0]), t1 = __fadd_rn(v[5], v[1]), t2 = __fadd_rn(v[6], v[2]), t3 = __fadd_rn(v[7], v[3]);
            csum[slot] = __fadd_rn(__fadd_rn(t0, t2), __fadd_rn(t1, t3));
        }
    }
    // The reference accumulates the chunk sums sequentially in double, then the tail (ggml.c:2845-2888).  All terms are positive, so a
    // tree sum S brackets the sequential one within +-2n*2^-53*S: if 1/sum rounds to the same float at both ends of the bracket the
    // order cannot matter (the persistent decode step decides the same way); otherwise replay the sequential chain (128 dependent
    // shuffle + add steps per row: it used to run for every row).
    for (int i = nchunks * 8; i < n_kv; i++) {                                // scalar tail through libm expf
        const float val = glibc_expf_dev(__fsub_rn(p[i], mx));
        if (lane == 0) p[i] = val;
    }
    __syncwarp();
    double tsum = 0.0;
#pragma unroll
    for (int slot = 0; slot < 4; slot++) tsum += (double) csum[slot];         // (zero where this lane owns no chunk)
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) tsum += __shfl_xor_sync(0xffffffffu, tsum, o);
    float sc;
    {
        const double dl = 2.0 * (double)(nchunks + 8) * 0x1p-53 * tsum * (1.0 + 1e-6);
        double lo = tsum - dl, hi = tsum + dl;
        for (int i = nchunks * 8; i < n_kv; i++) { const double tl = (double) p[i]; lo = __dadd_rn(lo, tl); hi = __dadd_rn(hi, tl); }
        const double mid = 0.5 * (lo + hi);
        double y = (double) __frcp_rn((float) mid);                          // 1/mid to ~2^-50: float seed + 2 Newton steps
        double e = __fma_rn(-mid, y, 1.0); y = __fma_rn(y, e, y);
        e = __fma_rn(-mid, y, 1.0);        y = __fma_rn(y, e, y);
        const double rw = (hi - lo) * y * 0.5 + 0x1p-48;
        sc = __double2float_rn(y * (1.0 - rw));
        if (sc != __double2float_rn(y * (1.0 + rw))) {                        // rare: the reference's own order
            double sum = 0.0;
#pragma unroll
            for (int slot = 0; slot < 4; slot++) {
                const int base = slot * 32;
                if (base < nchunks) {
                    const int cnt = min(32, nchunks - base);
                    for (int l = 0; l < cnt; l++) sum = __dadd_rn(sum, (double) __shfl_sync(0xffffffffu, csum[slot], l));
                }
            }
            for (int i = nchunks * 8; i < n_kv; i++) sum = __dadd_rn(sum, (double) p[i]);
            sc = __double2float_rn(__ddiv_rn(1.0, sum));
            if (fallback_counter && lane == 0) atomicAdd(fallback_counter, 1u);
        }
    }
    __syncwarp();
    for (int i = lane; i < n_kv; i += 32) p[i] = __fmul_rn(p[i], sc);
}

}  // namespace bark
