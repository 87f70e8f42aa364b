// Decode of the sampled pixels of the reference view (ADA/lib/network_v5.py:432-465,486-499):
//   depth logits   = the `prob` 3x3x3 conv (8 -> 1) evaluated ONLY at the P sampled pixels x D depths
//   prob           = softmax over the D depths; depth = sum_d prob_d * depth_d                 (soft-argmax)
//   fused feature  = sum_d prob_d * (feat_ref + warp(feat_src, d))                              (depth-guided fusion)
//   NOCS           = tanh(nocs_head(instance_color(feat_ref at the pixel)))
//   pose feature   = pose_mlp1(cat(fused, nocs_pts_mlp(NOCS)))  -> per-env mean -> pose_mlp2 -> mean -> rotation head
// Kernels here: decode_gather (the gather / memory-bound part), colsum (deterministic per-env sums), pose_gbias, rot_head; the
// per-point MLPs are 1x1 convolutions on the tcgen05 conv kernel (engine.py: _build_decode_tc).
#include "stages.cuh"
#include "warp.cuh"

namespace adp {

constexpr int PB = 32;          // sampled pixels per block
constexpr int DEC_THREADS = 256;
constexpr int LDS = 260;        // padded row pitch (floats) of the activation ping-pong buffers, multiple of 4

struct DecodeArgs {
    const float* feat_ref;   // [B,S,S,32] fp32
    const float* feat_src;   // [B,S,S,32]
    const float* Mw;         // [B,12]
    const float* depths;     // [D]
    const bf16* x11;         // [B,D,S,S,8] last U-Net activation (conv0 + deconv11)
    const int* choose;       // [B,P]
    const uint8_t* valid;    // [B] or nullptr
    float* nocs;             // [B,P,3]
    float* depth;            // [B,P]
    float* pf1;              // [B,P,128] pose_mlp1 output
    float* gsum;             // [B,128]  sum over P of pf1 (zeroed by the caller)
    float* dbg_logits;       // [B,P,D] or nullptr
    float* dbg_fused;        // [B,P,32] or nullptr
    int B, S, D, P;
    int x11_f16;             // x11 holds IEEE half instead of bf16
    int x11_s2d;             // x11 is stored space-to-depth(2): [B,D/2,S/2,S/2,64], channel = (pz*4+py*2+px)*8 + c
    int regress;             // 0: stop after NOCS + depth (no pose heads: direct_regression = False)
};

// ------------------------------------------------------------------------------------------------
// decode, stage 1 (the gather-bound part): depth logits at the sampled pixels (the `prob` conv evaluated only there),
// softmax over depth + soft-argmax, depth-guided fused feature, and the reference feature at the pixel.  The per-point
// MLPs then run as 1x1 convolutions on the tcgen05 kernel (engine.py), so this kernel writes their inputs as bf16 hi/lo.
//   xfeat [B,P,32]  (instance_color input)           xcat [B,P,96] columns 0..31 = fused feature (pose_mlp1 input)
// ------------------------------------------------------------------------------------------------
// element offset of the 8 channels of voxel (dz, yy, xx) of x11
__device__ __forceinline__ size_t x11_offset(const DecodeArgs& a, int b, int dz, int yy, int xx) {
    if (a.x11_s2d) {
        const int S2 = a.S >> 1;
        return ((((size_t)b * (a.D >> 1) + (dz >> 1)) * S2 + (yy >> 1)) * S2 + (xx >> 1)) * 64 + (((dz & 1) * 4 + (yy & 1) * 2 + (xx & 1)) * 8);
    }
    return ((((size_t)b * a.D + dz) * a.S + yy) * a.S + xx) * 8;
}

struct GatherArgs {
    DecodeArgs a;
    bf16* xfeat_hi; bf16* xfeat_lo;
    bf16* xcat_hi;  bf16* xcat_lo;
};

__global__ void __launch_bounds__(DEC_THREADS)
decode_gather_kernel(const GatherArgs ga, const float* __restrict__ prob_w) {
    const DecodeArgs& a = ga.a;
    extern __shared__ float smf[];
    float* bufA = smf;                   // [PB][LDS] (only columns 0..31 used)
    float* bufB = smf + PB * LDS;
    float* s_logit = smf + 2 * PB * LDS;
    float* s_probw = s_logit + PB * 24;
    int* s_pix = reinterpret_cast<int*>(s_probw + 216);
    const int tid = threadIdx.x;
    const int b = blockIdx.y;
    const int p0 = blockIdx.x * PB;
    if (a.valid && !a.valid[b]) return;
    const int S = a.S, D = a.D;
    if (a.x11 != nullptr) for (int i = tid; i < 216; i += DEC_THREADS) s_probw[i] = prob_w[i];
    if (tid < PB) s_pix[tid] = a.choose[(size_t)b * a.P + p0 + tid];
    __syncthreads();
    if (a.x11 == nullptr) {
        // single-view mode (BASELINE configs[0..1]: backbone + NOCS of one frame, network_v5.py:432-444): only the reference
        // features at the sampled pixels are gathered; there is no volume, no depth and no fused feature
        const int r = tid >> 3, cq = tid & 7;
        const int pix = s_pix[r];
        const float4 fr = __ldg(reinterpret_cast<const float4*>(a.feat_ref + ((size_t)b * S * S + pix) * 32 + cq * 4));
        *reinterpret_cast<float4*>(bufA + r * LDS + cq * 4) = fr;
        __syncthreads();
        if ((tid & 7) < 4) {
            const int c8 = (tid & 7) * 8;
            st8_16(ga.xfeat_hi, ga.xfeat_lo, ((size_t)b * a.P + p0 + r) * 32 + c8, 0, bufA + r * LDS + c8);
        }
        return;
    }

    // ---- (a) depth logits at the sampled pixels: 3x3x3 conv over the 8-channel volume, zero padding.
    // One thread per (pixel, (ky, kx) column of the window) walks the depth axis once: every voxel of the 3 x 3 x (D + 2)
    // neighbourhood is loaded exactly once (16 bytes) and feeds the three depth taps that read it; the nine column partials of a
    // logit are then added in a fixed order (deterministic).
    float* s_part = bufA;                  // [PB][9][D] partial logits (the buffers are free until stage (c))
    for (int e = tid; e < PB * 9; e += DEC_THREADS) {
        const int r = e / 9, col = e - r * 9;
        const int ky = col / 3, kx = col - ky * 3;
        const int pix = s_pix[r];
        const int y = pix / S, x = pix - y * S;
        const int yy = y + ky - 1, xx = x + kx - 1;
        float* part = s_part + (r * 9 + col) * 24;
        if (yy < 0 || yy >= S || xx < 0 || xx >= S) {
            for (int d = 0; d < D; ++d) part[d] = 0.f;
            continue;
        }
        // w[kz][c] of this column
        float w0[8], w1[8], w2[8];
#pragma unroll
        for (int c = 0; c < 8; ++c) {
            w0[c] = s_probw[((0 * 3 + ky) * 3 + kx) * 8 + c];
            w1[c] = s_probw[((1 * 3 + ky) * 3 + kx) * 8 + c];
            w2[c] = s_probw[((2 * 3 + ky) * 3 + kx) * 8 + c];
        }
        float acc_prev = 0.f, acc_cur = 0.f;      // logits d-1 and d under construction while plane d is read
        for (int dz = 0; dz < D; ++dz) {
            const uint4 v = __ldg(reinterpret_cast<const uint4*>(a.x11 + x11_offset(a, b, dz, yy, xx)));
            const uint32_t u[4] = {v.x, v.y, v.z, v.w};
            float f[8];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                if (a.x11_f16) {
                    f[2 * q] = __half2float(__ushort_as_half((unsigned short)(u[q] & 0xffffu)));
                    f[2 * q + 1] = __half2float(__ushort_as_half((unsigned short)(u[q] >> 16)));
                } else {
                    f[2 * q] = __uint_as_float(u[q] << 16);
                    f[2 * q + 1] = __uint_as_float(u[q] & 0xffff0000u);
                }
            }
            float t0 = 0.f, t1 = 0.f, t2 = 0.f;   // plane dz is tap kz = 2 of logit dz-1, kz = 1 of logit dz, kz = 0 of logit dz+1
#pragma unroll
            for (int c = 0; c < 8; ++c) { t2 = fmaf(f[c], w2[c], t2); t1 = fmaf(f[c], w1[c], t1); t0 = fmaf(f[c], w0[c], t0); }
            if (dz >= 1) part[dz - 1] = acc_prev + t2;
            acc_prev = acc_cur + t1;
            acc_cur = t0;
        }
        part[D - 1] = acc_prev;
    }
    __syncthreads();
    for (int e = tid; e < PB * D; e += DEC_THREADS) {
        const int r = e / D, d = e - r * D;
        float acc = 0.f;
#pragma unroll
        for (int col = 0; col < 9; ++col) acc += s_part[(r * 9 + col) * 24 + d];
        s_logit[r * 24 + d] = acc;
        if (a.dbg_logits) a.dbg_logits[((size_t)b * a.P + p0 + r) * D + d] = acc;
    }
    __syncthreads();

    // ---- (b) softmax over depth + expectation: 8 lanes per pixel, shuffle reductions
    {
        const int r = tid >> 3, l = tid & 7;   // 32 pixels x 8 lanes
        float v[3], m = -INFINITY;
#pragma unroll
        for (int j = 0; j < 3; ++j) { v[j] = s_logit[r * 24 + l + 8 * j]; m = fmaxf(m, v[j]); }
        for (int o = 4; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
        float s = 0.f;
#pragma unroll
        for (int j = 0; j < 3; ++j) { v[j] = expf(v[j] - m); s += v[j]; }
        for (int o = 4; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        float dsum = 0.f;
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            const float pr = v[j] / s;
            s_logit[r * 24 + l + 8 * j] = pr;
            dsum = fmaf(pr, a.depths[l + 8 * j], dsum);
        }
        for (int o = 4; o > 0; o >>= 1) dsum += __shfl_xor_sync(0xffffffffu, dsum, o);
        if (l == 0) a.depth[(size_t)b * a.P + p0 + r] = dsum;
    }
    __syncthreads();

    // ---- (c) reference features at the pixel -> bufA[:, 0:32]; depth-guided fused features -> bufB[:, 0:32]
    {
        const int r = tid >> 3, cq = tid & 7;   // 4 channels per thread, 128-bit loads
        const int pix = s_pix[r];
        const int y = pix / S, x = pix - y * S;
        const float4 fr = __ldg(reinterpret_cast<const float4*>(a.feat_ref + (((size_t)b * S + y) * S + x) * 32 + cq * 4));
        *reinterpret_cast<float4*>(bufA + r * LDS + cq * 4) = fr;
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
        const float* src = a.feat_src + (size_t)b * S * S * 32 + cq * 4;
        for (int d = 0; d < D; ++d) {
            const float pr = s_logit[r * 24 + d];
            float ix, iy;
            warp_coords(a.Mw + 12 * b, (float)x, (float)y, a.depths[d], S, S, &ix, &iy);
            const Bilin bl = bilin_setup(ix, iy, S, S);
            float4 v = fr;
            if (bl.any) {
                const float wts[4] = {bl.w00, bl.w01, bl.w10, bl.w11};
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    if (wts[k] != 0.f) {
                        const float4 s4 = __ldg(reinterpret_cast<const float4*>(src + ((size_t)(bl.y0 + (k >> 1)) * S + bl.x0 + (k & 1)) * 32));
                        v.x = fmaf(wts[k], s4.x, v.x); v.y = fmaf(wts[k], s4.y, v.y);
                        v.z = fmaf(wts[k], s4.z, v.z); v.w = fmaf(wts[k], s4.w, v.w);
                    }
                }
            }
            acc.x = fmaf(pr, v.x, acc.x); acc.y = fmaf(pr, v.y, acc.y);
            acc.z = fmaf(pr, v.z, acc.z); acc.w = fmaf(pr, v.w, acc.w);
        }
        *reinterpret_cast<float4*>(bufB + r * LDS + cq * 4) = acc;
        if (a.dbg_fused) *reinterpret_cast<float4*>(a.dbg_fused + ((size_t)b * a.P + p0 + r) * 32 + cq * 4) = acc;
    }
    __syncthreads();

    // ---- write the MLP inputs as bf16 hi/lo
    {
        const int r = tid >> 3, c8 = (tid & 7) * 8;        // 32 pixels x 8 groups of 8 channels: groups 0-3 feat, 4-7 fused
        const size_t pt = (size_t)b * a.P + p0 + r;
        if (c8 < 32) st8_16(ga.xfeat_hi, ga.xfeat_lo, pt * 32 + c8, 0, bufA + r * LDS + c8);
        else st8_16(ga.xcat_hi, ga.xcat_lo, pt * 96 + (c8 - 32), 0, bufB + r * LDS + (c8 - 32));
    }
}

// column sums over the P points of an env: out[b, c] = sum_p x[b, p, c]   (hi + lo).  One block per (env, 64 columns): four row
// quarters are summed by four thread groups and combined in a fixed order -- no floating-point atomics, so an environment's
// result does not depend on what else is in the batch or on scheduling (shards reproduce the unsharded run bit for bit).
__global__ void __launch_bounds__(256)
colsum_kernel(const bf16* __restrict__ hi, const bf16* __restrict__ lo, const uint8_t* __restrict__ valid,
              float* __restrict__ out, int P, int C) {
    __shared__ float part[4][64];
    const int b = blockIdx.y;
    const int c = blockIdx.x * 64 + (threadIdx.x & 63), q = threadIdx.x >> 6;
    if (valid && !valid[b]) {
        if (q == 0 && c < C) out[(size_t)b * C + c] = 0.f;
        return;
    }
    float s = 0.f;
    if (c < C) {
        const int rows = (P + 3) / 4, r0 = q * rows, r1 = min(P, r0 + rows);
        float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;     // four independent chains (fixed association)
        int r = r0;
        for (; r + 3 < r1; r += 4) {
            s0 += ld_act(hi, lo, ((size_t)b * P + r) * C + c);
            s1 += ld_act(hi, lo, ((size_t)b * P + r + 1) * C + c);
            s2 += ld_act(hi, lo, ((size_t)b * P + r + 2) * C + c);
            s3 += ld_act(hi, lo, ((size_t)b * P + r + 3) * C + c);
        }
        for (; r < r1; ++r) s0 += ld_act(hi, lo, ((size_t)b * P + r) * C + c);
        s = (s0 + s1) + (s2 + s3);
    }
    part[q][threadIdx.x & 63] = s;
    __syncthreads();
    if (q == 0 && c < C) out[(size_t)b * C + c] = (part[0][threadIdx.x] + part[1][threadIdx.x]) + (part[2][threadIdx.x] + part[3][threadIdx.x]);
}

// per-env bias of pose_mlp2's first layer: gb[b, n] = bias[n] + sum_k W[128 + k][n] * (gsum[b, k] / P)   (network_v5.py:491-493)
__global__ void pose_gbias_kernel(const float* __restrict__ gsum, const float* __restrict__ q0_w, const float* __restrict__ q0_b,
                                  const uint8_t* __restrict__ valid, float* __restrict__ gb, int P) {
    __shared__ float gm[128];
    const int b = blockIdx.x, n = threadIdx.x;     // 256 threads
    if (valid && !valid[b]) return;
    if (n < 128) gm[n] = gsum[(size_t)b * 128 + n] / (float)P;
    __syncthreads();
    float acc = q0_b[n];
    for (int k = 0; k < 128; ++k) acc = fmaf(gm[k], __ldg(q0_w + (size_t)(128 + k) * 256 + n), acc);
    gb[(size_t)b * 256 + n] = acc;
}

// rotation head 256 -> 256 -> 128 -> 6 and the 6-D -> SO(3) map (ADA/lib/rotation_utils.py:4-27)
__global__ void __launch_bounds__(256)
rot_head_kernel(const float* __restrict__ psum, const uint8_t* __restrict__ valid, float* __restrict__ Rout, float* __restrict__ r6out,
                const adp_decode_weights w, int P) {
    __shared__ float v0[256], v1[256], v2[128], r6[6];
    const int b = blockIdx.x, tid = threadIdx.x;
    if (valid && !valid[b]) {
        if (tid < 9) Rout[9 * b + tid] = (tid % 4 == 0) ? 1.f : 0.f;
        return;
    }
    v0[tid] = psum[(size_t)b * 256 + tid] / (float)P;
    __syncthreads();
    {
        float acc = w.r0_b[tid];
        for (int k = 0; k < 256; ++k) acc = fmaf(v0[k], __ldg(w.r0_w + (size_t)k * 256 + tid), acc);
        v1[tid] = fmaxf(acc, 0.f);
    }
    __syncthreads();
    if (tid < 128) {
        float acc = w.r1_b[tid];
        for (int k = 0; k < 256; ++k) acc = fmaf(v1[k], __ldg(w.r1_w + (size_t)k * 128 + tid), acc);
        v2[tid] = fmaxf(acc, 0.f);
    }
    __syncthreads();
    if (tid < 6) {
        float acc = w.r2_b[tid];
        for (int k = 0; k < 128; ++k) acc = fmaf(v2[k], w.r2_w[k * 6 + tid], acc);
        r6[tid] = acc;
        if (r6out) r6out[6 * b + tid] = acc;
    }
    __syncthreads();
    if (tid == 0) {
        const float xr[3] = {r6[0], r6[1], r6[2]};
        float y[3] = {r6[3], r6[4], r6[5]};
        float n = fmaxf(sqrtf(y[0] * y[0] + y[1] * y[1] + y[2] * y[2]), 1e-8f);
        y[0] /= n; y[1] /= n; y[2] /= n;
        float z[3] = {xr[1] * y[2] - xr[2] * y[1], xr[2] * y[0] - xr[0] * y[2], xr[0] * y[1] - xr[1] * y[0]};
        n = fmaxf(sqrtf(z[0] * z[0] + z[1] * z[1] + z[2] * z[2]), 1e-8f);
        z[0] /= n; z[1] /= n; z[2] /= n;
        const float x[3] = {y[1] * z[2] - y[2] * z[1], y[2] * z[0] - y[0] * z[2], y[0] * z[1] - y[1] * z[0]};
        float* R = Rout + 9 * b;   // columns [x y z]
        R[0] = x[0]; R[1] = y[0]; R[2] = z[0];
        R[3] = x[1]; R[4] = y[1]; R[5] = z[1];
        R[6] = x[2]; R[7] = y[2]; R[8] = z[2];
    }
}

int decode_gather_run(const DecodeArgs& a, const float* prob_w, bf16* xfeat_hi, bf16* xfeat_lo, bf16* xcat_hi, bf16* xcat_lo,
                      cudaStream_t stream) {
    ADP_CHECK_ARG(a.D == 24 && a.P % PB == 0, "24 depth hypotheses, P multiple of 32");
    // row / column S-1 of an odd S would be read from s2d cell (S-1)/2, one past the end of a [B, D/2, S/2, S/2, 64] volume
    ADP_CHECK_ARG(!a.x11 || !a.x11_s2d || a.S % 2 == 0, "decode gather: the space-to-depth(2) x11 layout needs an even S");
    if (a.B == 0) return ADP_OK;
    const size_t smem1 = (size_t)(2 * PB * LDS + PB * 24 + 216) * sizeof(float) + PB * sizeof(int);
    static_assert(PB * 9 * 24 <= PB * LDS, "the partial-logit scratch fits the first activation buffer");
    static int attr[kMaxDevices];
    ADP_TRY(ensure_dyn_smem(decode_gather_kernel, (int)smem1, attr));
    GatherArgs ga;
    ga.a = a; ga.xfeat_hi = xfeat_hi; ga.xfeat_lo = xfeat_lo; ga.xcat_hi = xcat_hi; ga.xcat_lo = xcat_lo;
    decode_gather_kernel<<<dim3(a.P / PB, a.B), DEC_THREADS, smem1, stream>>>(ga, prob_w);
    ADP_CUDA(cudaGetLastError());
    return ADP_OK;
}

int colsum_run(const bf16* hi, const bf16* lo, const uint8_t* valid, float* out, int B, int P, int C, cudaStream_t stream) {
    if (B == 0) return ADP_OK;
    colsum_kernel<<<dim3((C + 63) / 64, B), 256, 0, stream>>>(hi, lo, valid, out, P, C);
    ADP_CUDA(cudaGetLastError());
    return ADP_OK;
}

int pose_gbias_run(const float* gsum, const float* q0_w, const float* q0_b, const uint8_t* valid, float* gb, int B, int P,
                   cudaStream_t stream) {
    if (B == 0) return ADP_OK;
    pose_gbias_kernel<<<B, 256, 0, stream>>>(gsum, q0_w, q0_b, valid, gb, P);
    ADP_CUDA(cudaGetLastError());
    return ADP_OK;
}

int rot_head_run(const float* psum, const uint8_t* valid, float* Rout, float* r6out, const adp_decode_weights* cw, int B, int P,
                 cudaStream_t stream) {
    if (B == 0) return ADP_OK;
    rot_head_kernel<<<B, 256, 0, stream>>>(psum, valid, Rout, r6out, *cw, P);
    ADP_CUDA(cudaGetLastError());
    return ADP_OK;
}

int decode_gather_c(const float* feat_ref, const float* feat_src, const float* Mw, const float* depths, const void* x11,
                    const int* choose, const uint8_t* valid, const float* prob_w, float* depth, void* xfeat_hi, void* xfeat_lo,
                    void* xcat_hi, void* xcat_lo, float* dbg_logits, float* dbg_fused, int B, int S, int D, int P, int x11_f16,
                    cudaStream_t stream) {
    DecodeArgs a{};
    a.feat_ref = feat_ref; a.feat_src = feat_src; a.Mw = Mw; a.depths = depths; a.x11 = reinterpret_cast<const bf16*>(x11);
    a.choose = choose; a.valid = valid; a.nocs = nullptr; a.depth = depth; a.pf1 = nullptr; a.gsum = nullptr;
    a.dbg_logits = dbg_logits; a.dbg_fused = dbg_fused; a.B = B; a.S = S; a.D = D; a.P = P; a.x11_f16 = x11_f16 & 1; a.x11_s2d = (x11_f16 >> 1) & 1; a.regress = 0;
    return decode_gather_run(a, prob_w, reinterpret_cast<bf16*>(xfeat_hi), reinterpret_cast<bf16*>(xfeat_lo),
                             reinterpret_cast<bf16*>(xcat_hi), reinterpret_cast<bf16*>(xcat_lo), stream);
}

}  // namespace adp
