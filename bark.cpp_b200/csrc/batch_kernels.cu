// Batched decode attention: one launch per layer for B items x H heads of a batched decode step (batch.cu).
//
// Replaces, for B single-position rows that each have their OWN KV cache, the scores / soft_max / P.V sequence of the per-op path
// (gpt_kernels.cu attention) — with the same arithmetic in the same order, so every item's row is bit-identical to its
// single-prompt evaluation:
//   scores[k] = lane_tree_reduce(chain over D/32 steps, lane l owning elements l, l+32, ...) * scale     (attn_scores_kernel)
//   soft_max in the reference's order                                                                  (softmax_row.cuh)
//   out[d]    = 32 chains over keys k = l (mod 32) in increasing order, GGML_F32x8_REDUCE tree, then the compiled leftovers
//                                                                                                      (attn_pv_kernel)
// No mask: the only query is the last position.  One CTA per (item, head), 4*D threads.  K and V stream through shared memory
// in 32-key tiles (16-byte cp.async, a 64 KB ring of 512 / D tiles); the scores stay in shared memory.
#include "epilogue.cuh"
#include "gpt_kernels.h"
#include "softmax_row.cuh"

namespace bark {

namespace {

__device__ __forceinline__ void cp_async_16(void * dst_smem, const float * src) {
    const uint32_t dst = (uint32_t) __cvta_generic_to_shared(dst_smem);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

constexpr int kTile = 32;                                    // keys per staged tile = one step of every P.V chain
constexpr int kMaxKv = 1024;                                 // softmax_row_warp's capacity (block_size of every Bark model)

// rows [t*32, min(t*32 + 32, n_kv)) of one head's K or V slice -> tile [32][D]; the row of the new position comes straight from
// the QKV scratch (the same values the append stores), so nothing here waits for the append to land in the cache
template <int D, int NT>
__device__ __forceinline__ void load_tile(float * tile, const float * cache, const float * fresh, int t, int n_kv, int n_past, int E) {
    const int r0 = t * kTile, rows = min(kTile, n_kv - r0);
    for (int c = threadIdx.x; c < rows * (D / 4); c += NT) {
        const int r = c / (D / 4), j = (c % (D / 4)) * 4, k = r0 + r;
        cp_async_16(tile + r * D + j, (k == n_past ? fresh : cache + (size_t) k * E) + j);
    }
    cp_async_commit();
}

template <int DS> struct AttnShape {
    static constexpr int D = 32 * DS, NT = 128 * DS, NW = NT / 32, CPT = kTile / (NT / D);   // CPT = 8 chains of one column per thread
    static constexpr int NS = 512 / D;                       // tiles in flight (a 64 KB ring): two in flight hid too little latency
    static constexpr size_t smem = (size_t)(D + kMaxKv + NS * kTile * D) * sizeof(float);
};

// K tiles 0 .. ntiles-1, then V tiles 0 .. ntiles-1, stream through one NS-stage ring: the first V tiles arrive while the last scores
// are formed and the row is normalised.  Stage u lives in ring slot u % NS; one commit group per stage (empty past the end), so
// cp.async.wait_group NS-1 always means "stage u has landed".
template <int DS>
__global__ void __launch_bounds__(128 * DS) batch_decode_attention_kernel(const float * __restrict__ qkv, BatchKV kv, int n_past, int E, int H, float scale,
                                                                         void * __restrict__ act, int wt, int Kp, unsigned * __restrict__ fallbacks) {
    using S = AttnShape<DS>;
    constexpr int D = S::D, NT = S::NT, NW = S::NW, CPT = S::CPT, NS = S::NS;
    extern __shared__ __align__(16) float smem[];
    float * sq = smem, * sp = smem + D, * ring = smem + D + kMaxKv;
    const int b = blockIdx.x / H, h = blockIdx.x % H;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int n_kv = n_past + 1, ntiles = (n_kv + kTile - 1) / kTile, nstages = 2 * ntiles;
    const float * row = qkv + (size_t) b * 3 * E;
    const float * knew = row + E + h * D, * vnew = row + 2 * E + h * D;
    float * kc = kv.k[b] + h * D, * vc = kv.v[b] + h * D;

    // append this position's K / V head slice to the item's cache (vectorised), query slice to shared memory
    for (int i = tid; i < D / 4; i += NT) {
        const float4 k4 = reinterpret_cast<const float4 *>(knew)[i], v4 = reinterpret_cast<const float4 *>(vnew)[i];
        reinterpret_cast<float4 *>(kc + (size_t) n_past * E)[i] = k4;
        reinterpret_cast<float4 *>(vc + (size_t) n_past * E)[i] = v4;
        reinterpret_cast<float4 *>(sq)[i] = reinterpret_cast<const float4 *>(row + h * D)[i];
    }
    auto issue = [&](int u) {
        if (u < nstages) {
            if (u < ntiles) load_tile<D, NT>(ring + (u % NS) * kTile * D, kc, knew, u, n_kv, n_past, E);
            else            load_tile<D, NT>(ring + (u % NS) * kTile * D, vc, vnew, u - ntiles, n_kv, n_past, E);
        } else cp_async_commit();
    };
#pragma unroll 1
    for (int u = 0; u < NS - 1; u++) issue(u);

    const int d = tid % D, g = tid / D, np = n_kv & ~(kTile - 1), nfull = np / kTile;
    float acc[CPT];
#pragma unroll
    for (int j = 0; j < CPT; j++) acc[j] = 0.0f;
#pragma unroll 1
    for (int u = 0; u < nstages; u++) {
        issue(u + NS - 1);
        cp_async_wait<NS - 1>();
        __syncthreads();
        const float * tile = ring + (u % NS) * kTile * D;
        if (u < ntiles) {                                     // scores: warp w takes keys w, w + NW, ... of the tile
            const int rows = min(kTile, n_kv - u * kTile);
            for (int r = warp; r < rows; r += NW) {
                float a = 0.0f;
#pragma unroll
                for (int c = 0; c < DS; c++) a = __fmaf_rn(tile[r * D + c * 32 + lane], sq[c * 32 + lane], a);
                const float s = __fmul_rn(lane_tree_reduce(a), scale);           // ggml_scale_inplace
                if (lane == 0) sp[u * kTile + r] = s;
            }
        } else {
            const int t = u - ntiles;
            if (t == 0) {                                     // every score is in: normalise the row
                if (warp == 0) softmax_row_warp(sp, n_kv, fallbacks);
                __syncthreads();
            }
            if (t < nfull) {                                  // P.V: thread (d, g) runs chains l = g*8 .. g*8+7 of column d
#pragma unroll
                for (int j = 0; j < CPT; j++) { const int l = g * CPT + j; acc[j] = __fmaf_rn(tile[l * D + d], sp[t * kTile + l], acc[j]); }
            }
        }
        __syncthreads();
    }
    // the last (partial) V tile stays in its slot; the 32 chain partials of each column meet in the next one
    const float * tail = ring + ((nstages - 1) % NS) * kTile * D;
    float * part = ring + (nstages % NS) * kTile * D;
#pragma unroll
    for (int j = 0; j < CPT; j++) part[(g * CPT + j) * D + d] = acc[j];
    __syncthreads();
    if (tid < D) {
        float a[32];
#pragma unroll
        for (int l = 0; l < 32; l++) a[l] = part[l * D + tid];
        float sum = lane_tree_reduce_local(a);
        int i = np, r = n_kv - np;
        while (r >= 8) { for (int l = 0; l < 8; l++) sum = __fadd_rn(sum, __fmul_rn(tail[(i + l - np) * D + tid], sp[i + l])); i += 8; r -= 8; }
        if (r >= 4)    { for (int l = 0; l < 4; l++) sum = __fadd_rn(sum, __fmul_rn(tail[(i + l - np) * D + tid], sp[i + l])); i += 4; r -= 4; }
        for (; r > 0; r--, i++) sum = __fmaf_rn(tail[(i - np) * D + tid], sp[i], sum);
        store_act(act, wt, Kp, b, h * D + tid, sum);
    }
}

template <int DS>
void launch_attention(int grid, cudaStream_t s, const float * qkv, const BatchKV & kv, int n_past, int E, int H, float scale, void * act, WType wt, int Kp, unsigned * fb) {
    static std::atomic<unsigned long long> configured{0};
    if (first_use_on_this_device(configured))
        BARK_CUDA_CHECK(cudaFuncSetAttribute(batch_decode_attention_kernel<DS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) AttnShape<DS>::smem));
    BARK_LAUNCH(batch_decode_attention_kernel<DS>, grid, AttnShape<DS>::NT, AttnShape<DS>::smem, s, qkv, kv, n_past, E, H, scale, act, (int) wt, Kp, fb);
}

}  // namespace

void batch_decode_attention(const float * qkv, const BatchKV & kv, int B, int n_past, int E, int H, void * act, WType wt, int Kp,
                            unsigned * softmax_fallbacks, cudaStream_t s) {
    const int D = E / H, n_kv = n_past + 1;
    if (B < 1 || B > kBatchMax || E % H || D % 32 || D > 128 || n_kv > kMaxKv) {
        fprintf(stderr, "bark_b200: batched decode attention needs 1..%d rows, heads of 32/64/96/128 and <= %d keys (B %d, E %d, H %d, n_kv %d)\n",
                kBatchMax, kMaxKv, B, E, H, n_kv);
        throw std::runtime_error("unsupported configuration (see the message above)");
    }
    const float scale = 1.0f / sqrtf((float) E / (float) H);                 // bark.cpp:1318, as attention()
    g_next_bytes = (double) B * (2.0 * n_kv * E * 4.0 + 3.0 * E * 4.0 + 2.0 * E * 4.0 + E * 4.0);    // K / V rows read, QKV row, appended K / V, output
    g_next_flops = 4.0 * (double) B * n_kv * E;
    const int grid = B * H;
    switch (D / 32) {
        case 1: launch_attention<1>(grid, s, qkv, kv, n_past, E, H, scale, act, wt, Kp, softmax_fallbacks); break;
        case 2: launch_attention<2>(grid, s, qkv, kv, n_past, E, H, scale, act, wt, Kp, softmax_fallbacks); break;
        case 3: launch_attention<3>(grid, s, qkv, kv, n_past, E, H, scale, act, wt, Kp, softmax_fallbacks); break;
        default: launch_attention<4>(grid, s, qkv, kv, n_past, E, H, scale, act, wt, Kp, softmax_fallbacks); break;
    }
}

}  // namespace bark
