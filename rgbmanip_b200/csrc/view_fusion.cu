// Cross-view attention of the transformer variant (ADA/lib/fusion.py:11-82, ViewFusion(embed_dim = 32, num_heads = 4,
// depth = 4), used by StereoPoseNet_with_depth_baseline, ADA/lib/network_baseline.py:553,631-640) and the per-point depth MLP
// behind it (network_baseline.py:555-562,642).
//
// Tokens are the 1024 sampled pixels of each view, 32 channels.  One block of the reference is
//     x = MHA1(q = view 1, k = v = view 2) + view 1,      y = MHA2(q = view 2, k = v = view 1) + view 2
// both from the block's inputs.  One launch per block; a CTA owns (environment, direction, half of the queries): 512 threads, one
// query token each.  Per head the CTA projects K and V of all 1024 key tokens into shared memory (fp32, 64 KB), every thread
// projects its own query, and the 1024 x 8 dot products / softmax / weighted sum run out of registers with broadcast shared-memory
// reads (two passes over the keys: row maximum, then exp2 and accumulation; the 1 / sqrt(d_k) and log2(e) factors are folded into
// the query).  The four head outputs stay in registers, the output projection + bias + residual finish the token.  Everything
// is fp32 on the CUDA cores: d_k = 8 is half a tensor-core K step, and at 1.1 GFLOP per environment this stage is ~1 % of the
// network.  The last block writes the view-1 tokens as the bf16 hi/lo planes the pose MLP reads (columns 0..31 of xcat) and
// evaluates the depth MLP (32 -> 64 -> 32 -> 1, ReLU) in the same thread.
#include "stages.cuh"

namespace adp {

constexpr int VF_P = 1024, VF_C = 32, VF_H = 4, VF_DK = 8, VF_THREADS = 512;
constexpr int VF_LIN = VF_C * VF_C + VF_C;          // one nn.Linear(32, 32): weight [out][in] + bias
constexpr int VF_MHA = 4 * VF_LIN;                  // q, k, v, output projections (fusion.py:33)
constexpr int VF_DEPTH_W = 64 * 32 + 64 + 64 * 32 + 32 + 32 + 1;      // depth_head.0 [64][32], b, depth_head.2 TRANSPOSED [64][32], b, .4 [32], b

struct FusionArgs {
    const float* in[2];        // tokens of view 1 / view 2, [B,P,32] fp32 (ignored when feat != nullptr)
    const float* feat[2];      // block 0: feature maps [B,S*S,32] fp32 to gather the tokens from ...
    const int* choose[2];      // ... at these pixel indices [B,P]
    float* out[2];             // block outputs [B,P,32] fp32 (may be nullptr in the last block for view 1 when only planes are wanted)
    const uint8_t* valid;      // [B] or nullptr
    const float* w;            // this block's weights: [2 directions][VF_MHA]
    const float* depth_w;      // last block: VF_DEPTH_W floats, else nullptr
    float* depth;              // [B,P] (view 1), last block
    float* depth2;             // [B,P] (view 2) or nullptr
    bf16* xcat_hi; bf16* xcat_lo;      // [B,P,96] planes, columns 0..31 <- view-1 tokens, last block (nullptr = skip)
    int SS;                    // S * S
};

__device__ __forceinline__ const float* token_ptr(const FusionArgs& a, int view, int b, int t) {
    if (a.feat[view]) return a.feat[view] + ((size_t)b * a.SS + a.choose[view][(size_t)b * VF_P + t]) * VF_C;
    return a.in[view] + ((size_t)b * VF_P + t) * VF_C;
}

__device__ __forceinline__ void load_token(const float* p, float* x) {
#pragma unroll
    for (int q = 0; q < VF_C / 4; ++q) {
        const float4 v = __ldg(reinterpret_cast<const float4*>(p) + q);
        x[4 * q] = v.x; x[4 * q + 1] = v.y; x[4 * q + 2] = v.z; x[4 * q + 3] = v.w;
    }
}

// y[c] = W[row0 + c][:] . x + b[row0 + c], c < 8; W / b in shared memory (every thread reads the same address: broadcast)
__device__ __forceinline__ void project8(const float* __restrict__ lin, int row0, const float* x, float* y) {
#pragma unroll
    for (int c = 0; c < VF_DK; ++c) {
        const float4* wr = reinterpret_cast<const float4*>(lin + (row0 + c) * VF_C);
        float s = lin[VF_C * VF_C + row0 + c];
#pragma unroll
        for (int q = 0; q < VF_C / 4; ++q) {
            const float4 w = wr[q];
            s = fmaf(w.x, x[4 * q], s); s = fmaf(w.y, x[4 * q + 1], s); s = fmaf(w.z, x[4 * q + 2], s); s = fmaf(w.w, x[4 * q + 3], s);
        }
        y[c] = s;
    }
}

__global__ void __launch_bounds__(VF_THREADS, 2) view_fusion_kernel(FusionArgs a) {
    extern __shared__ __align__(16) float smem[];
    float* Ks = smem;                              // [P][8]
    float* Vs = smem + VF_P * VF_DK;               // [P][8]
    float* Wm = smem + 2 * VF_P * VF_DK;           // this direction's q, k, v, o projections
    const int b = blockIdx.x, dir = blockIdx.y, t = threadIdx.x;
    const int qi = blockIdx.z * VF_THREADS + t;
    const int qv = dir, kv = dir ^ 1;              // direction 0: view 1 queries view 2 (fusion1); 1: the other way (fusion2)
    const bool last = a.depth_w != nullptr;
    if (a.valid && !a.valid[b]) {                  // no estimate for this environment: defined zeros for everything downstream
        if (a.out[qv]) for (int c = 0; c < VF_C; ++c) a.out[qv][((size_t)b * VF_P + qi) * VF_C + c] = 0.f;
        if (last) {
            float* dp = dir == 0 ? a.depth : a.depth2;
            if (dp) dp[(size_t)b * VF_P + qi] = 0.f;
            if (dir == 0 && a.xcat_hi) {
                const float z[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
                for (int c8 = 0; c8 < VF_C; c8 += 8) st8_16(a.xcat_hi, a.xcat_lo, ((size_t)b * VF_P + qi) * 96 + c8, 0, z);
            }
        }
        return;
    }
    for (int i = t; i < VF_MHA; i += VF_THREADS) Wm[i] = a.w[(size_t)dir * VF_MHA + i];
    __syncthreads();
    const float* xq_p = token_ptr(a, qv, b, qi);
    float cat[VF_C];
    float x[VF_C];
    // exp(s / sqrt(d_k) - max) = exp2((s - max') * log2(e) / sqrt(d_k)): fold the factor into the query
    const float qscale = 1.4426950408889634f * 0.35355339059327379f;
#pragma unroll 1
    for (int h = 0; h < VF_H; ++h) {
        if (h) __syncthreads();                    // every thread is done with the previous head's K / V
#pragma unroll 1
        for (int j = t; j < VF_P; j += VF_THREADS) {
            load_token(token_ptr(a, kv, b, j), x);
            float y[VF_DK];
            project8(Wm + 1 * VF_LIN, h * VF_DK, x, y);
            reinterpret_cast<float4*>(Ks + j * VF_DK)[0] = make_float4(y[0], y[1], y[2], y[3]);
            reinterpret_cast<float4*>(Ks + j * VF_DK)[1] = make_float4(y[4], y[5], y[6], y[7]);
            project8(Wm + 2 * VF_LIN, h * VF_DK, x, y);
            reinterpret_cast<float4*>(Vs + j * VF_DK)[0] = make_float4(y[0], y[1], y[2], y[3]);
            reinterpret_cast<float4*>(Vs + j * VF_DK)[1] = make_float4(y[4], y[5], y[6], y[7]);
        }
        float q[VF_DK];
        load_token(xq_p, x);
        project8(Wm, h * VF_DK, x, q);
#pragma unroll
        for (int c = 0; c < VF_DK; ++c) q[c] *= qscale;
        __syncthreads();
        float m = -INFINITY;
#pragma unroll 4
        for (int j = 0; j < VF_P; ++j) {
            const float4 k0 = reinterpret_cast<const float4*>(Ks + j * VF_DK)[0], k1 = reinterpret_cast<const float4*>(Ks + j * VF_DK)[1];
            float s = q[0] * k0.x;
            s = fmaf(q[1], k0.y, s); s = fmaf(q[2], k0.z, s); s = fmaf(q[3], k0.w, s);
            s = fmaf(q[4], k1.x, s); s = fmaf(q[5], k1.y, s); s = fmaf(q[6], k1.z, s); s = fmaf(q[7], k1.w, s);
            m = fmaxf(m, s);
        }
        float l = 0.f, o[VF_DK];
#pragma unroll
        for (int c = 0; c < VF_DK; ++c) o[c] = 0.f;
#pragma unroll 4
        for (int j = 0; j < VF_P; ++j) {
            const float4 k0 = reinterpret_cast<const float4*>(Ks + j * VF_DK)[0], k1 = reinterpret_cast<const float4*>(Ks + j * VF_DK)[1];
            float s = q[0] * k0.x;
            s = fmaf(q[1], k0.y, s); s = fmaf(q[2], k0.z, s); s = fmaf(q[3], k0.w, s);
            s = fmaf(q[4], k1.x, s); s = fmaf(q[5], k1.y, s); s = fmaf(q[6], k1.z, s); s = fmaf(q[7], k1.w, s);
            const float p = exp2f(s - m);
            const float4 v0 = reinterpret_cast<const float4*>(Vs + j * VF_DK)[0], v1 = reinterpret_cast<const float4*>(Vs + j * VF_DK)[1];
            l += p;
            o[0] = fmaf(p, v0.x, o[0]); o[1] = fmaf(p, v0.y, o[1]); o[2] = fmaf(p, v0.z, o[2]); o[3] = fmaf(p, v0.w, o[3]);
            o[4] = fmaf(p, v1.x, o[4]); o[5] = fmaf(p, v1.y, o[5]); o[6] = fmaf(p, v1.z, o[6]); o[7] = fmaf(p, v1.w, o[7]);
        }
        const float inv = 1.0f / l;
#pragma unroll
        for (int c = 0; c < VF_DK; ++c) cat[h * VF_DK + c] = o[c] * inv;
    }
    // output projection + bias + residual (fusion.py:51,69-73)
    load_token(xq_p, x);
    float y[VF_C];
#pragma unroll
    for (int c0 = 0; c0 < VF_C; c0 += VF_DK) project8(Wm + 3 * VF_LIN, c0, cat, y + c0);
#pragma unroll
    for (int c = 0; c < VF_C; ++c) y[c] += x[c];
    if (a.out[qv]) {
        float4* op = reinterpret_cast<float4*>(a.out[qv] + ((size_t)b * VF_P + qi) * VF_C);
#pragma unroll
        for (int q4 = 0; q4 < VF_C / 4; ++q4) op[q4] = make_float4(y[4 * q4], y[4 * q4 + 1], y[4 * q4 + 2], y[4 * q4 + 3]);
    }
    if (!last) return;
    if (dir == 0 && a.xcat_hi) {
#pragma unroll
        for (int c8 = 0; c8 < VF_C; c8 += 8) st8_16(a.xcat_hi, a.xcat_lo, ((size_t)b * VF_P + qi) * 96 + c8, 0, y + c8);
    }
    float* dp = dir == 0 ? a.depth : a.depth2;
    if (!dp) return;
    // depth_head (network_baseline.py:555-562): 32 -> 64 -> 32 -> 1, ReLU after every layer; the hidden 64 are streamed
    const float* w0 = a.depth_w;
    const float* b0 = w0 + 64 * 32;
    const float* w1t = b0 + 64;                    // [64][32]: depth_head.2 transposed
    const float* b1 = w1t + 64 * 32;
    const float* w2 = b1 + 32;
    float h1[32];
#pragma unroll
    for (int c = 0; c < 32; ++c) h1[c] = __ldg(b1 + c);
#pragma unroll 2
    for (int i = 0; i < 64; ++i) {
        float s = __ldg(b0 + i);
#pragma unroll
        for (int q4 = 0; q4 < 8; ++q4) {
            const float4 w = __ldg(reinterpret_cast<const float4*>(w0 + i * 32) + q4);
            s = fmaf(w.x, y[4 * q4], s); s = fmaf(w.y, y[4 * q4 + 1], s); s = fmaf(w.z, y[4 * q4 + 2], s); s = fmaf(w.w, y[4 * q4 + 3], s);
        }
        s = fmaxf(s, 0.f);
#pragma unroll
        for (int q4 = 0; q4 < 8; ++q4) {
            const float4 w = __ldg(reinterpret_cast<const float4*>(w1t + i * 32) + q4);
            h1[4 * q4] = fmaf(w.x, s, h1[4 * q4]); h1[4 * q4 + 1] = fmaf(w.y, s, h1[4 * q4 + 1]);
            h1[4 * q4 + 2] = fmaf(w.z, s, h1[4 * q4 + 2]); h1[4 * q4 + 3] = fmaf(w.w, s, h1[4 * q4 + 3]);
        }
    }
    float d = __ldg(w2 + 32);
#pragma unroll
    for (int c = 0; c < 32; ++c) d = fmaf(__ldg(w2 + c), fmaxf(h1[c], 0.f), d);
    dp[(size_t)b * VF_P + qi] = fmaxf(d, 0.f);
}

// blocks: [4 blocks][2 directions][VF_MHA] floats; scratch: 4 x [B,P,32] fp32 (two ping-pong pairs)
int view_fusion_run(const float* feat1, const float* feat2, const int* choose1, const int* choose2, const uint8_t* valid,
                    const float* blocks, const float* depth_w, float* scratch, float* depth1, float* depth2, bf16* xcat_hi,
                    bf16* xcat_lo, float* fused1, float* fused2, int B, int S, int P, int n_blocks, cudaStream_t stream) {
    ADP_CHECK_ARG(P == VF_P, "1024 tokens per view");
    ADP_CHECK_ARG(n_blocks >= 1, "at least one attention block");
    if (B == 0) return ADP_OK;
    const int smem = (2 * VF_P * VF_DK + VF_MHA) * (int)sizeof(float);
    static bool attr[64] = {};
    int dev = 0;
    ADP_CUDA(cudaGetDevice(&dev));
    if (dev < 64 && !attr[dev]) {
        ADP_CUDA(cudaFuncSetAttribute(view_fusion_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        attr[dev] = true;
    }
    const size_t plane = (size_t)B * VF_P * VF_C;
    for (int blk = 0; blk < n_blocks; ++blk) {
        FusionArgs a = {};
        const bool first = blk == 0, last = blk == n_blocks - 1;
        for (int v = 0; v < 2; ++v) {
            a.feat[v] = first ? (v ? feat2 : feat1) : nullptr;
            a.choose[v] = first ? (v ? choose2 : choose1) : nullptr;
            a.in[v] = first ? nullptr : scratch + (size_t)(2 * ((blk + 1) & 1) + v) * plane;
            a.out[v] = last ? (v ? fused2 : fused1) : scratch + (size_t)(2 * (blk & 1) + v) * plane;
        }
        a.valid = valid;
        a.w = blocks + (size_t)blk * 2 * VF_MHA;
        a.depth_w = last ? depth_w : nullptr;
        a.depth = depth1; a.depth2 = depth2;
        a.xcat_hi = xcat_hi; a.xcat_lo = xcat_lo;
        a.SS = S * S;
        // the last block's view-2 direction feeds nothing but view2_depth / fused2: skipped unless the caller asks for them
        const int dirs = (last && !depth2 && !fused2) ? 1 : 2;
        view_fusion_kernel<<<dim3(B, dirs, VF_P / VF_THREADS), VF_THREADS, smem, stream>>>(a);
        ADP_CUDA(cudaGetLastError());
    }
    return ADP_OK;
}

}  // namespace adp
