// Memory-bound helpers of the PSPNet backbone (channels-last, hi(+lo) bf16 activations):
// 3x3/2 max-pool, pyramid pooling + 1x1 convs, pyramid concat fused with the first x2 bilinear upsample,
// plain x2 bilinear upsample (align_corners=True).  Reference: ADA/lib/pspnet.py:66-107,142-158.
#include "stages.cuh"

namespace adp {

// 8 consecutive channels (16 B per plane) <-> fp32 registers; f16 = 1: a single IEEE-half plane
__device__ __forceinline__ void ld8(const bf16* __restrict__ hi, const bf16* __restrict__ lo, size_t i, float* v, int f16) {
    const uint4 h = __ldg(reinterpret_cast<const uint4*>(hi + i));     // inputs are never written by these kernels
    const uint32_t hw[4] = {h.x, h.y, h.z, h.w};
    if (f16) {
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            v[2 * u] = __half2float(__ushort_as_half((unsigned short)(hw[u] & 0xffffu)));
            v[2 * u + 1] = __half2float(__ushort_as_half((unsigned short)(hw[u] >> 16)));
        }
        return;
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
        v[2 * u] = __uint_as_float(hw[u] << 16);
        v[2 * u + 1] = __uint_as_float(hw[u] & 0xffff0000u);
    }
    if (lo) {
        const uint4 l = __ldg(reinterpret_cast<const uint4*>(lo + i));
        const uint32_t lw[4] = {l.x, l.y, l.z, l.w};
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            v[2 * u] += __uint_as_float(lw[u] << 16);
            v[2 * u + 1] += __uint_as_float(lw[u] & 0xffff0000u);
        }
    }
}
__device__ __forceinline__ void st8(bf16* __restrict__ hi, bf16* __restrict__ lo, size_t i, const float* v, int f16) {
    st8_16(hi, lo, i, f16, v);
}

// ---------------------------------------------------------------------------------------------
// max-pool 3x3 stride 2 pad 1 (pspnet.py:39,69)
// ---------------------------------------------------------------------------------------------
__global__ void maxpool3x3s2_kernel(const bf16* __restrict__ in_hi, const bf16* __restrict__ in_lo, bf16* __restrict__ out_hi,
                                    bf16* __restrict__ out_lo, int B, int Hi, int Wi, int Ho, int Wo, int C, int f16) {
    const int C8 = C >> 3;
    const size_t total = (size_t)B * Ho * Wo * C8;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const int c = (int)(i % C8) * 8;
        size_t t = i / C8;
        const int ox = (int)(t % Wo); t /= Wo;
        const int oy = (int)(t % Ho);
        const int b = (int)(t / Ho);
        if (f16) {        // a single fp16 plane: the maximum is exact on packed halves (max.NaN.f16x2), no conversions
            __half2 hm[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) hm[j] = __half2half2(__ushort_as_half((unsigned short)0xfc00u));      // -inf
#pragma unroll
            for (int ky = 0; ky < 3; ++ky) {
                const int iy = oy * 2 - 1 + ky;
                if (iy < 0 || iy >= Hi) continue;
#pragma unroll
                for (int kx = 0; kx < 3; ++kx) {
                    const int ix = ox * 2 - 1 + kx;
                    if (ix < 0 || ix >= Wi) continue;
                    const uint4 u = __ldg(reinterpret_cast<const uint4*>(in_hi + (((size_t)b * Hi + iy) * Wi + ix) * C + c));
                    const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
                    for (int j = 0; j < 4; ++j) hm[j] = __hmax2_nan(hm[j], *reinterpret_cast<const __half2*>(&w[j]));
                }
            }
            uint4 o;
            o.x = *reinterpret_cast<const uint32_t*>(&hm[0]); o.y = *reinterpret_cast<const uint32_t*>(&hm[1]);
            o.z = *reinterpret_cast<const uint32_t*>(&hm[2]); o.w = *reinterpret_cast<const uint32_t*>(&hm[3]);
            *reinterpret_cast<uint4*>(out_hi + (((size_t)b * Ho + oy) * Wo + ox) * C + c) = o;
            continue;
        }
        float m[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) m[j] = -INFINITY;
#pragma unroll
        for (int ky = 0; ky < 3; ++ky) {
            const int iy = oy * 2 - 1 + ky;
            if (iy < 0 || iy >= Hi) continue;
#pragma unroll
            for (int kx = 0; kx < 3; ++kx) {
                const int ix = ox * 2 - 1 + kx;
                if (ix < 0 || ix >= Wi) continue;
                float v[8];
                ld8(in_hi, in_lo, (((size_t)b * Hi + iy) * Wi + ix) * C + c, v, f16);
#pragma unroll
                for (int j = 0; j < 8; ++j) m[j] = max_nan(m[j], v[j]);
            }
        }
        st8(out_hi, out_lo, (((size_t)b * Ho + oy) * Wo + ox) * C + c, m, f16);
    }
}

int maxpool3x3s2(const Act& in, const Act& out, int batch, cudaStream_t stream) {
    ADP_CHECK_ARG(in.C == out.C && out.H == (in.H + 1) / 2 && out.W == (in.W + 1) / 2 && in.C % 8 == 0 && in.f16 == out.f16, "maxpool shapes");
    size_t total = (size_t)batch * out.H * out.W * (out.C / 8);
    int grid = (int)((total + 255) / 256 < 148 * 16 ? (total + 255) / 256 : 148 * 16);
    if (grid == 0) return ADP_OK;
    maxpool3x3s2_kernel<<<grid, 256, 0, stream>>>(in.hi, in.lo, out.hi, out.lo, batch, in.H, in.W, out.H, out.W, in.C, in.f16);
    ADP_CUDA(cudaGetLastError());
    return ADP_OK;
}

// ---------------------------------------------------------------------------------------------
// pyramid pooling: adaptive average pools with bins (1,2,3,6) = 50 cells (pspnet.py:84-87)
// window of cell i along an axis of size S with b bins: [floor(i S / b), ceil((i+1) S / b))
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void psp_cell(int cell, int* bins, int* cy, int* cx) {
    // cells are ordered stage by stage: 1 + 4 + 9 + 36
    if (cell < 1) { *bins = 1; *cy = 0; *cx = 0; }
    else if (cell < 5) { *bins = 2; *cy = (cell - 1) / 2; *cx = (cell - 1) % 2; }
    else if (cell < 14) { *bins = 3; *cy = (cell - 5) / 3; *cx = (cell - 5) % 3; }
    else { *bins = 6; *cy = (cell - 14) / 6; *cx = (cell - 14) % 6; }
}

// one block per (cell, frame): 128-bit loads of 8 channels, the window rows split over blockDim.x / (C / 8) thread groups
__global__ void __launch_bounds__(256)
psp_pool_kernel(const bf16* __restrict__ in_hi, const bf16* __restrict__ in_lo, float* __restrict__ pooled,
                int H, int W, int C, int cs, int f16) {
    __shared__ float part[4][1024];
    const int b = blockIdx.y, cell = blockIdx.x;
    int bins, cy, cx;
    psp_cell(cell, &bins, &cy, &cx);
    const int y0 = (cy * H) / bins, y1 = ((cy + 1) * H + bins - 1) / bins;
    const int x0 = (cx * W) / bins, x1 = ((cx + 1) * W + bins - 1) / bins;
    const float inv = 1.f / (float)((y1 - y0) * (x1 - x0));
    const int groups = C >> 3;                       // 8-channel groups (<= 128)
    const int parts = blockDim.x / groups;           // row partitions (>= 1, <= 4 used)
    const int g = threadIdx.x % groups, pr = threadIdx.x / groups;
    float s[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    if (pr < parts && pr < 4) {
        const int np = parts < 4 ? parts : 4;
        for (int y = y0 + pr; y < y1; y += np)
            for (int x = x0; x < x1; ++x) {
                float v[8];
                ld8(in_hi, in_lo, (((size_t)b * H + y) * W + x) * cs + g * 8, v, f16);
#pragma unroll
                for (int j = 0; j < 8; ++j) s[j] += v[j];
            }
#pragma unroll
        for (int j = 0; j < 8; ++j) part[pr][g * 8 + j] = s[j];
    }
    __syncthreads();
    const int np = (parts < 4 ? parts : 4);
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
        float t = 0.f;
        for (int q = 0; q < np; ++q) t += part[q][c];
        pooled[((size_t)b * 50 + cell) * C + c] = t * inv;
    }
}

// 1x1 conv 512 -> 128 (no bias) + ReLU per stage; w: [4][Cin][128] fp32 (pspnet.py:88-90)
__global__ void psp_conv_kernel(const float* __restrict__ pooled, const float* __restrict__ w, float* __restrict__ priors,
                                int Cin) {
    extern __shared__ float sv[];
    const int b = blockIdx.y, cell = blockIdx.x;
    const int stage = cell < 1 ? 0 : cell < 5 ? 1 : cell < 14 ? 2 : 3;
    for (int c = threadIdx.x; c < Cin; c += blockDim.x) sv[c] = pooled[((size_t)b * 50 + cell) * Cin + c];
    __syncthreads();
    const int n = threadIdx.x;   // 128 threads
    const float* ws = w + (size_t)stage * Cin * 128;
    float acc = 0.f;
    for (int c = 0; c < Cin; ++c) acc = fmaf(sv[c], ws[(size_t)c * 128 + n], acc);
    priors[((size_t)b * 50 + cell) * 128 + n] = max_nan(acc, 0.f);
}

int psp_priors(const Act& feat, int feat_cs, const float* w, float* pooled, float* priors, int batch, cudaStream_t stream) {
    ADP_CHECK_ARG(feat.C <= 1024 && feat.C % 8 == 0 && 256 % (feat.C / 8) == 0, "psp channels");
    if (batch == 0) return ADP_OK;
    psp_pool_kernel<<<dim3(50, batch), 256, 0, stream>>>(feat.hi, feat.lo, pooled, feat.H, feat.W, feat.C, feat_cs > 0 ? feat_cs : feat.C, feat.f16);
    ADP_CUDA(cudaGetLastError());
    psp_conv_kernel<<<dim3(50, batch), 128, feat.C * sizeof(float), stream>>>(pooled, w, priors, feat.C);
    ADP_CUDA(cudaGetLastError());
    return ADP_OK;
}

// ---------------------------------------------------------------------------------------------
// concat(feat, upsampled priors) followed by the x2 bilinear upsample of up_1, in one pass:
// out[b, Y, X, :] for the (2H x 2W) grid, channels [0,C) from feat, [C + 128 s, C + 128 (s+1)) from stage s.
// Both interpolations use align_corners=True (pspnet.py:92-93,105).
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void lin_coord(int o, int in_size, int out_size, int* i0, int* i1, float* w1) {
    // align_corners=True: src = o * (in-1)/(out-1)
    const float scale = out_size > 1 ? (float)(in_size - 1) / (float)(out_size - 1) : 0.f;
    const float s = scale * (float)o;
    int a = (int)s;
    if (a > in_size - 1) a = in_size - 1;
    *i0 = a;
    *i1 = a + (a < in_size - 1 ? 1 : 0);
    *w1 = s - (float)a;
}

// ---------------------------------------------------------------------------------------------
// pyramid priors resized to the feature grid (pspnet.py:92-93, align_corners=True) and written into channels
// [coff, coff + 512) of the concat tensor out[b, y, x, :]; the 512 feature channels in front of them are written by the
// producing convolution itself (epilogue channel pitch), so the concat never exists as a separate pass.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
psp_fill_priors_kernel(const float* __restrict__ priors, bf16* __restrict__ out_hi, bf16* __restrict__ out_lo,
                       uint8_t* __restrict__ out_q8, int H, int W, int Ct, int coff, int f16) {
    __shared__ __align__(16) float spr[50 * 128];
    const int b = blockIdx.y, y = blockIdx.x;
    for (int i = threadIdx.x; i < 50 * 128 / 4; i += blockDim.x)
        reinterpret_cast<float4*>(spr)[i] = __ldg(reinterpret_cast<const float4*>(priors + (size_t)b * 50 * 128) + i);
    __syncthreads();
    for (int it = threadIdx.x; it < W * 64; it += blockDim.x) {
        const int x = it >> 6, c = (it & 63) * 8;                  // 512 prior channels = 64 groups of 8
        const int s = c >> 7, n0 = c & 127;
        const int bins = s == 0 ? 1 : s == 1 ? 2 : s == 2 ? 3 : 6;
        const int off = s == 0 ? 0 : s == 1 ? 1 : s == 2 ? 5 : 14;
        // one bilinear cell of the bins x bins prior map per (pixel, stage); 8 channels share its coordinates
        int y0, y1, x0, x1;
        float wy, wx;
        lin_coord(y, bins, H, &y0, &y1, &wy);
        lin_coord(x, bins, W, &x0, &x1, &wx);
        const float* pr = spr + off * 128 + n0;
        const float* p00 = pr + (y0 * bins + x0) * 128;
        const float* p01 = pr + (y0 * bins + x1) * 128;
        const float* p10 = pr + (y1 * bins + x0) * 128;
        const float* p11 = pr + (y1 * bins + x1) * 128;
        float o[8];
#pragma unroll
        for (int j = 0; j < 8; j += 4) {
            const float4 a = *reinterpret_cast<const float4*>(p00 + j), bq = *reinterpret_cast<const float4*>(p01 + j);
            const float4 cq = *reinterpret_cast<const float4*>(p10 + j), d = *reinterpret_cast<const float4*>(p11 + j);
            o[j + 0] = (1.f - wy) * ((1.f - wx) * a.x + wx * bq.x) + wy * ((1.f - wx) * cq.x + wx * d.x);
            o[j + 1] = (1.f - wy) * ((1.f - wx) * a.y + wx * bq.y) + wy * ((1.f - wx) * cq.y + wx * d.y);
            o[j + 2] = (1.f - wy) * ((1.f - wx) * a.z + wx * bq.z) + wy * ((1.f - wx) * cq.z + wx * d.z);
            o[j + 3] = (1.f - wy) * ((1.f - wx) * a.w + wx * bq.w) + wy * ((1.f - wx) * cq.w + wx * d.w);
        }
        const size_t oo = (((size_t)b * H + y) * W + x) * Ct + coff + c;
        st8(out_hi, out_lo, oo, o, f16);
        if (out_q8) *reinterpret_cast<uint2*>(out_q8 + oo) = pack8_q8(o);      // fp8 twin for the consumer's low-order pass
    }
}

int psp_fill_priors(const float* priors, const Act& out, int coff, int batch, cudaStream_t stream) {
    ADP_CHECK_ARG(coff % 8 == 0 && coff + 512 <= out.C, "psp prior channel range");
    if (batch == 0) return ADP_OK;
    psp_fill_priors_kernel<<<dim3(out.H, batch), 256, 0, stream>>>(priors, out.hi, out.lo, out.f16 ? out.q8 : nullptr, out.H, out.W, out.C,
                                                                   coff, out.f16);
    ADP_CUDA(cudaGetLastError());
    return ADP_OK;
}

// ---------------------------------------------------------------------------------------------
// x2 bilinear upsample, align_corners=True (pspnet.py:105).  One block = a 16 x 16 output tile of a 64-channel slab: the
// <= 10 x 10 input pixels it reads are staged in shared memory once (0.39 bytes read per byte written instead of up to 4
// through L1/L2), each thread then produces 8 channels of 8 output pixels with 128-bit stores.
// ---------------------------------------------------------------------------------------------
constexpr int UP_T = 16;        // output tile edge
constexpr int UP_IN = 10;       // input rows / columns a tile can touch
constexpr int UP_CS = 64;       // channels per slab (128 B per pixel)

__device__ __forceinline__ void up_unpack8(const uint4& u, float* v, bool f16) {
    const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        if (f16) {
            const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&w[q]));
            v[2 * q] = f.x; v[2 * q + 1] = f.y;
        } else {
            v[2 * q] = __uint_as_float(w[q] << 16); v[2 * q + 1] = __uint_as_float(w[q] & 0xffff0000u);
        }
    }
}

// SPLIT: activations are bf16 hi + lo planes (two raw tiles); otherwise one 16-bit plane (fp16 or bf16)
template <bool SPLIT>
__global__ void __launch_bounds__(256)
upsample2x_kernel(const bf16* __restrict__ in_hi, const bf16* __restrict__ in_lo, bf16* __restrict__ out_hi,
                  bf16* __restrict__ out_lo, uint8_t* __restrict__ out_q8, int H, int W, int C, int tiles_x, int f16) {
    __shared__ uint4 tile[(SPLIT ? 2 : 1) * UP_IN * UP_IN * (UP_CS / 8)];      // raw 16-bit values, 16 B per (pixel, 8 channels)
    constexpr int PLANE = UP_IN * UP_IN * (UP_CS / 8);
    const int Ho = 2 * H, Wo = 2 * W;
    const int tyi = blockIdx.x / tiles_x, txi = blockIdx.x - tyi * tiles_x;
    const int c0 = blockIdx.y * UP_CS, b = blockIdx.z;
    const int Y0 = tyi * UP_T, X0 = txi * UP_T;
    int iy0, ix0, dummy;
    float wdummy;
    lin_coord(Y0, H, Ho, &iy0, &dummy, &wdummy);
    lin_coord(X0, W, Wo, &ix0, &dummy, &wdummy);
    const size_t base = (size_t)b * H * W;
    for (int i = threadIdx.x; i < PLANE; i += 256) {
        const int g = i & 7, px = i >> 3;
        const int ly = px / UP_IN, lx = px - ly * UP_IN;
        const int y = min(iy0 + ly, H - 1), x = min(ix0 + lx, W - 1);
        const size_t off = (base + (size_t)y * W + x) * C + c0 + g * 8;
        tile[i] = __ldg(reinterpret_cast<const uint4*>(in_hi + off));
        if (SPLIT) tile[PLANE + i] = __ldg(reinterpret_cast<const uint4*>(in_lo + off));
    }
    __syncthreads();
    // thread -> (8-channel group g, output column X, output rows Y0 + r0, r0 + 2, ...): the x interpolation is hoisted
    const int g = threadIdx.x & 7;
    const int X = X0 + ((threadIdx.x >> 3) & (UP_T - 1));
    const int r0 = threadIdx.x >> 7;
    if (X >= Wo) return;
    int x0, x1;
    float wx;
    lin_coord(X, W, Wo, &x0, &x1, &wx);
    const int cx0 = (x0 - ix0) * 8 + g, cx1 = (x1 - ix0) * 8 + g;
    // fp16 plane: the x interpolation runs on the mixed-precision FMA (no conversions).  Its weights are k / (Wo - 1): the integer
    // numerators are exact fp16 multipliers, the denominator is folded into the y weights (see upconv_fold_row).
    const bool fast = !SPLIT && f16;
    const int n1x = __float2int_rn(wx * (float)(Wo - 1));
    const uint32_t xn0 = __half_as_ushort(__int2half_rn(Wo - 1 - n1x)), xn1 = __half_as_ushort(__int2half_rn(n1x));
    const float xs = 1.f / (float)(Wo - 1);
#pragma unroll 2
    for (int r = r0; r < UP_T; r += 2) {
        const int Y = Y0 + r;
        if (Y >= Ho) break;
        int y0, y1;
        float wy;
        lin_coord(Y, H, Ho, &y0, &y1, &wy);
        const int ry0 = (y0 - iy0) * UP_IN * 8, ry1 = (y1 - iy0) * UP_IN * 8;
        if (fast) {
            float t[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f}, u[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f}, o[8];
            fhfma8(tile[ry0 + cx0], xn0, t);
            fhfma8(tile[ry0 + cx1], xn1, t);
            fhfma8(tile[ry1 + cx0], xn0, u);
            fhfma8(tile[ry1 + cx1], xn1, u);
            const float w0 = (1.f - wy) * xs, w1 = wy * xs;
#pragma unroll
            for (int j = 0; j < 8; ++j) o[j] = fmaf(w1, u[j], w0 * t[j]);
            const size_t oo = (((size_t)b * Ho + Y) * Wo + X) * C + c0 + g * 8;
            st8(out_hi, out_lo, oo, o, f16);
            if (out_q8) *reinterpret_cast<uint2*>(out_q8 + oo) = pack8_q8(o);
            continue;
        }
        float a[8], bq[8], c[8], d[8], o[8];
        up_unpack8(tile[ry0 + cx0], a, !SPLIT && f16);
        up_unpack8(tile[ry0 + cx1], bq, !SPLIT && f16);
        up_unpack8(tile[ry1 + cx0], c, !SPLIT && f16);
        up_unpack8(tile[ry1 + cx1], d, !SPLIT && f16);
        if (SPLIT) {
            float t[8];
            up_unpack8(tile[PLANE + ry0 + cx0], t, false);
#pragma unroll
            for (int j = 0; j < 8; ++j) a[j] += t[j];
            up_unpack8(tile[PLANE + ry0 + cx1], t, false);
#pragma unroll
            for (int j = 0; j < 8; ++j) bq[j] += t[j];
            up_unpack8(tile[PLANE + ry1 + cx0], t, false);
#pragma unroll
            for (int j = 0; j < 8; ++j) c[j] += t[j];
            up_unpack8(tile[PLANE + ry1 + cx1], t, false);
#pragma unroll
            for (int j = 0; j < 8; ++j) d[j] += t[j];
        }
#pragma unroll
        for (int j = 0; j < 8; ++j)
            o[j] = (1.f - wy) * ((1.f - wx) * a[j] + wx * bq[j]) + wy * ((1.f - wx) * c[j] + wx * d[j]);
        const size_t oo = (((size_t)b * Ho + Y) * Wo + X) * C + c0 + g * 8;
        st8(out_hi, out_lo, oo, o, f16);
        if (out_q8) *reinterpret_cast<uint2*>(out_q8 + oo) = pack8_q8(o);      // fp8 twin for the consumer's low-order pass
    }
}

int upsample2x(const Act& in, const Act& out, int batch, cudaStream_t stream) {
    ADP_CHECK_ARG(out.C == in.C && out.H == 2 * in.H && out.W == 2 * in.W && in.C % UP_CS == 0 && in.f16 == out.f16, "upsample shapes");
    if (batch == 0) return ADP_OK;
    const int tiles_x = (out.W + UP_T - 1) / UP_T, tiles_y = (out.H + UP_T - 1) / UP_T;
    const dim3 grid(tiles_x * tiles_y, in.C / UP_CS, batch);
    if (in.lo && !in.f16) upsample2x_kernel<true><<<grid, 256, 0, stream>>>(in.hi, in.lo, out.hi, out.lo, nullptr, in.H, in.W, in.C, tiles_x, 0);
    else upsample2x_kernel<false><<<grid, 256, 0, stream>>>(in.hi, nullptr, out.hi, out.lo, out.f16 ? out.q8 : nullptr, in.H, in.W, in.C, tiles_x, in.f16);
    ADP_CUDA(cudaGetLastError());
    return ADP_OK;
}

// ---------------------------------------------------------------------------------------------
// PSPUpsample (pspnet.py:97-107) = bilinear x2 (align_corners=True) -> Conv2d 3x3 pad 1 -> PReLU, restructured.
// Interpolation and the conv's channel mixing are both linear and act on different axes, so
//     conv3x3(up(x))[Y,X] = bias + sum_{dy,dx} [ (Y+dy, X+dx) inside ] up(q_{dy,dx})[Y+dy, X+dx],      q_tap = W_tap x  (a 1x1 conv at LOW resolution)
// The nine q_tap come out of ONE tensor-core GEMM over the low-resolution map (N = 9 Cout, K = Cin: a quarter of the FLOPs of the
// 3x3 conv over the upsampled map, and the upsampled tensor never exists).  This kernel is the second half: per output pixel the
// 9 taps x 4 bilinear neighbours of q, + bias, PReLU.  A thread owns (output column X, 8 channels) and walks down a strip of
// output rows: per low-resolution row r it folds the horizontal part once, H_dy[r] = sum_{dx,j} wx_j(X+dx) q_{dy,dx}[r, x_j(X+dx)]
// (18 16-byte loads), keeps H of the three low-resolution rows a 3-row output window can touch in registers, and every output
// row is 27 FMAs per channel with coefficients that hold the vertical weights (zero where a tap falls outside the image:
// the conv's zero padding applies to the UPSAMPLED image).
// q: [B, h, w, 9 C] (channel = tap * C + c, tap = ky * 3 + kx), out: [B, 2h, 2w, C].
// ---------------------------------------------------------------------------------------------
// One low-resolution row of q, columns [col0, col0 + ncols), staged in shared memory: [col][9 C channels] 16-bit, column pitch padded
// by 16 bytes (9 C * 2 is a multiple of 128: without the pad the columns of different threads would share banks).
template <bool SPLIT, bool F16>
__device__ __forceinline__ void upconv_fold_row(const uint4* __restrict__ st_hi, const uint4* __restrict__ st_lo, int pitch16, int tap0, int C8,
                                                int cg, const int (&xo)[3][2], const float (&xw)[3][2], const uint32_t (&xn)[3][2], int f16,
                                                float* H) {
#pragma unroll
    for (int j = 0; j < 8; ++j) H[j] = 0.f;
    if (F16) {
        // fp16 plane: the mixed-precision FMA takes the stored halves as they are (no conversions: half the instructions of this
        // loop).  Its multiplier is fp16 too, so the weights are the integer numerators of k / (Wo - 1) (exact in fp16, exact
        // products, fp32 accumulation); the common denominator is folded into the vertical coefficients.
#pragma unroll
        for (int dx = 0; dx < 3; ++dx) {
#pragma unroll
            for (int j = 0; j < 2; ++j) fhfma8(st_hi[xo[dx][j] * pitch16 + (tap0 + dx) * C8 + cg], xn[dx][j], H);
        }
        return;
    }
#pragma unroll
    for (int dx = 0; dx < 3; ++dx) {
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            const int off = xo[dx][j] * pitch16 + (tap0 + dx) * C8 + cg;
            float v[8];
            up_unpack8(st_hi[off], v, !SPLIT && f16);
            if (SPLIT) {
                float t[8];
                up_unpack8(st_lo[off], t, false);
#pragma unroll
                for (int e = 0; e < 8; ++e) v[e] += t[e];
            }
            const float wgt = xw[dx][j];
#pragma unroll
            for (int e = 0; e < 8; ++e) H[e] = fmaf(wgt, v[e], H[e]);
        }
    }
}

__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gmem_src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

constexpr int UPB_MAX_STRIP = 64;      // output rows a block walks at most (shared-memory coefficient table)

// Block = 256 threads = (256 / (C/8)) consecutive output columns x C/8 channel groups; it walks a strip of output rows.  The q rows
// it needs come through a two-deep shared-memory ring filled with cp.async: every q element is fetched once per block (the
// direct version had each of them fetched by ~4 threads of different warps: 7 TB/s of L2 traffic, the kernel's bound).
template <bool SPLIT, bool F16>
__global__ void __launch_bounds__(256, 2)
upconv_blend_kernel(const bf16* __restrict__ q_hi, const bf16* __restrict__ q_lo, bf16* __restrict__ out_hi, bf16* __restrict__ out_lo,
                    uint8_t* __restrict__ out_q8, const float* __restrict__ bias, float slope, int h, int w, int C, int f16, int strip,
                    int ncols_max) {
    extern __shared__ uint4 upb_stage[];
    // per output row of the strip: 9 vertical coefficients [dy][window row] and the first low-resolution row of its window;
    // the rows are the same for every thread of the block, so they are worked out once
    __shared__ float s_cf[UPB_MAX_STRIP][9];
    __shared__ int s_rb[UPB_MAX_STRIP];
    const int C8 = C >> 3, Ho = 2 * h, Wo = 2 * w, C9 = 9 * C;
    const int Y0 = blockIdx.y * strip, Y1 = min(Y0 + strip, Ho);
    const int tid = threadIdx.x;
    for (int i = tid; i < (Y1 - Y0) * 3; i += 256) {
        const int yy = i / 3, dy = i - yy * 3, Y = Y0 + yy;
        int rb, y0, y1, dummy;
        float wy, wdummy;
        lin_coord(max(Y - 1, 0), h, Ho, &rb, &dummy, &wdummy);
        const int Yt = Y + dy - 1;
        const bool in = Yt >= 0 && Yt < Ho;
        lin_coord(in ? Yt : Y, h, Ho, &y0, &y1, &wy);
        const int k0 = y0 - rb, k1 = y1 - rb;          // k0 in {0, 1}, k1 in {k0, k0 + 1}: rows Y - 1 .. Y + 1 span < 1 low-resolution row
        // (fp16 plane: the horizontal fold works with integer numerators over Wo - 1, see upconv_fold_row)
        const float hs = (F16 && Wo > 1) ? 1.f / (float)(Wo - 1) : 1.f;
        for (int k = 0; k < 3; ++k) s_cf[yy][dy * 3 + k] = in ? hs * ((k == k0 ? 1.f - wy : 0.f) + (k == k1 ? wy : 0.f)) : 0.f;
        if (dy == 0) s_rb[yy] = rb;
    }
    __syncthreads();
    const int XB = 256 / C8;                            // output columns of this block
    const int Xb0 = blockIdx.x * XB;
    const int cg = tid % C8, X = Xb0 + tid / C8;
    const bool active = X < Wo;
    const int b = blockIdx.z;
    // low-resolution columns the block touches: taps of columns Xb0 - 1 .. Xb0 + XB
    int col0, col1, dummy;
    float wdummy;
    lin_coord(max(Xb0 - 1, 0), w, Wo, &col0, &dummy, &wdummy);
    lin_coord(min(Xb0 + XB, Wo - 1), w, Wo, &dummy, &col1, &wdummy);
    const int ncols = col1 - col0 + 1;                  // <= ncols_max = XB / 2 + 3
    const int pitch16 = 9 * C8 + 1;                     // column pitch in 16-byte units (+1: bank spread)
    const int plane16 = ncols_max * pitch16;
    const int buf16 = (SPLIT ? 2 : 1) * plane16;
    // horizontal taps of this thread's column: staged column index and weight of X - 1, X, X + 1 (weight 0 outside the image)
    int xo[3][2];
    float xw[3][2];
    uint32_t xn[3][2];
#pragma unroll
    for (int dx = 0; dx < 3; ++dx) {
        const int Xt = X + dx - 1;
        const bool in = active && Xt >= 0 && Xt < Wo;
        int x0, x1;
        float wx;
        lin_coord(in ? Xt : min(X, Wo - 1), w, Wo, &x0, &x1, &wx);
        xo[dx][0] = in ? x0 - col0 : 0; xo[dx][1] = in ? x1 - col0 : 0;
        xw[dx][0] = in ? 1.f - wx : 0.f; xw[dx][1] = in ? wx : 0.f;
        // wx = k / (Wo - 1) up to float rounding: the integer numerators as fp16 multipliers
        const int n1 = __float2int_rn(wx * (float)(Wo - 1));
        xn[dx][0] = in ? (uint32_t)__half_as_ushort(__int2half_rn(Wo - 1 - n1)) : 0u;
        xn[dx][1] = in ? (uint32_t)__half_as_ushort(__int2half_rn(n1)) : 0u;
    }
    float bv[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) bv[e] = __ldg(bias + cg * 8 + e);
    const int r_first = s_rb[0];
    const int n_rows = 3 + s_rb[Y1 - Y0 - 1] - r_first;          // low-resolution rows this block folds, in order
    const int per_col = 9 * C8;
    auto load_row = [&](int n) {                                   // row n of the sequence -> ring slot n & 1
        const int r = min(r_first + n, h - 1);
        uint4* dst = upb_stage + (n & 1) * buf16;
        const size_t src = (((size_t)b * h + r) * w + col0) * (size_t)C9;
        for (int i = tid; i < ncols * per_col; i += 256) {
            const int col = i / per_col, e = i - col * per_col;
            cp_async16(dst + col * pitch16 + e, q_hi + src + (size_t)col * C9 + e * 8);
            if (SPLIT) cp_async16(dst + plane16 + col * pitch16 + e, q_lo + src + (size_t)col * C9 + e * 8);
        }
        cp_async_commit();
    };
    float H[3][3][8];          // [dy][window row k = low-resolution row rb + k][channel]
    int n_done = 0;            // rows folded so far
    auto fold_next = [&](int k) {                                  // fold row n_done into window slot k (block-uniform call sequence)
        if (n_done + 1 < n_rows) load_row(n_done + 1); else cp_async_commit();
        cp_async_wait<1>();
        __syncthreads();
        const uint4* st = upb_stage + (n_done & 1) * buf16;
#pragma unroll
        for (int dy = 0; dy < 3; ++dy) upconv_fold_row<SPLIT, F16>(st, st + plane16, pitch16, dy * 3, C8, cg, xo, xw, xn, f16, H[dy][k]);
        __syncthreads();                                           // the slot may be refilled by the load issued in the next call
        ++n_done;
    };
    load_row(0);
    fold_next(0);
    fold_next(1);
    fold_next(2);
    int rb = r_first;
    size_t oo = (((size_t)b * Ho + Y0) * Wo + (active ? X : 0)) * C + cg * 8;
    const size_t ostep = (size_t)Wo * C;
    for (int yy = 0; yy < Y1 - Y0; ++yy, oo += ostep) {
        if (s_rb[yy] != rb) {        // the window moves down by one low-resolution row
            rb = s_rb[yy];
#pragma unroll
            for (int dy = 0; dy < 3; ++dy)
#pragma unroll
                for (int e = 0; e < 8; ++e) { H[dy][0][e] = H[dy][1][e]; H[dy][1][e] = H[dy][2][e]; }
            fold_next(2);
        }
        float acc[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) acc[e] = bv[e];
#pragma unroll
        for (int dy = 0; dy < 3; ++dy) {
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                const float cf = s_cf[yy][dy * 3 + k];
#pragma unroll
                for (int e = 0; e < 8; ++e) acc[e] = fmaf(cf, H[dy][k][e], acc[e]);
            }
        }
#pragma unroll
        for (int e = 0; e < 8; ++e) acc[e] = acc[e] >= 0.f ? acc[e] : slope * acc[e];
        if (active) {
            st8(out_hi, out_lo, oo, acc, f16);
            if (out_q8) *reinterpret_cast<uint2*>(out_q8 + oo) = pack8_q8(acc);
        }
    }
    cp_async_wait<0>();
}

int upconv_blend(const Act& q, const Act& out, const float* bias, float slope, int batch, cudaStream_t stream) {
    ADP_CHECK_ARG(q.C == 9 * out.C && out.H == 2 * q.H && out.W == 2 * q.W && out.C % 8 == 0 && q.f16 == out.f16, "upconv_blend shapes");
    ADP_CHECK_ARG((q.lo != nullptr) == (out.lo != nullptr) || q.f16, "upconv_blend: q and out must use the same plane format");
    const int C8 = out.C / 8;
    ADP_CHECK_ARG(256 % C8 == 0, "upconv_blend: C / 8 must divide 256");
    if (batch == 0) return ADP_OK;
    const int XB = 256 / C8;
    const int ncols_max = XB / 2 + 3;
    const bool split = q.lo && !q.f16;
    const int smem = 2 * (split ? 2 : 1) * ncols_max * (9 * C8 + 1) * 16;
    // strips of output rows: long enough to amortise the 3-row window fill, short enough to fill the GPU
    int strip = out.H < UPB_MAX_STRIP ? out.H : UPB_MAX_STRIP;
    const int xblocks = (out.W + XB - 1) / XB;
    while (strip > 8 && (size_t)batch * xblocks * ((out.H + strip - 1) / strip) < 4 * 148) strip = (strip + 1) / 2;
    const dim3 grid(xblocks, (out.H + strip - 1) / strip, batch);
    static int attr_s[kMaxDevices], attr_h[kMaxDevices], attr_f[kMaxDevices];
    if (split) {
        ADP_TRY(ensure_dyn_smem(upconv_blend_kernel<true, false>, smem, attr_s));
        upconv_blend_kernel<true, false><<<grid, 256, smem, stream>>>(q.hi, q.lo, out.hi, out.lo, nullptr, bias, slope, q.H, q.W, out.C, 0, strip, ncols_max);
    } else if (q.f16) {
        ADP_TRY(ensure_dyn_smem(upconv_blend_kernel<false, true>, smem, attr_f));
        upconv_blend_kernel<false, true><<<grid, 256, smem, stream>>>(q.hi, nullptr, out.hi, out.lo, out.q8, bias, slope, q.H, q.W, out.C, 1, strip,
                                                                      ncols_max);
    } else {
        ADP_TRY(ensure_dyn_smem(upconv_blend_kernel<false, false>, smem, attr_h));
        upconv_blend_kernel<false, false><<<grid, 256, smem, stream>>>(q.hi, nullptr, out.hi, out.lo, nullptr, bias, slope, q.H, q.W, out.C, 0, strip,
                                                                       ncols_max);
    }
    ADP_CUDA(cudaGetLastError());
    return ADP_OK;
}

// ---------------------------------------------------------------------------------------------
// fp32 crops [F,S,S,3] -> space-to-depth(2) [F,S/2,S/2,16]: channel (py*2+px)*3 + c, channels 12..15 zero
// ---------------------------------------------------------------------------------------------
__global__ void pack_s2d_kernel(const float* __restrict__ crops, bf16* __restrict__ out_hi, bf16* __restrict__ out_lo, int B, int S, int f16) {
    const int Hs = S / 2;
    const size_t total = (size_t)B * Hs * Hs * 2;     // two 8-channel halves per s2d pixel
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const int half = (int)(i & 1);
        size_t t = i >> 1;
        const int x = (int)(t % Hs); t /= Hs;
        const int y = (int)(t % Hs);
        const int b = (int)(t / Hs);
        float v[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int ch = half * 8 + j;
            float val = 0.f;
            if (ch < 12) {
                const int pp = ch / 3, c = ch - pp * 3;
                const int py = pp >> 1, px = pp & 1;
                val = crops[(((size_t)b * S + 2 * y + py) * S + 2 * x + px) * 3 + c];
            }
            v[j] = val;
        }
        st8(out_hi, out_lo, i * 8, v, f16);
    }
}

int pack_s2d(const float* crops, const Act& out, int batch, int S, cudaStream_t stream) {
    ADP_CHECK_ARG(out.C == 16 && out.H == S / 2 && out.W == S / 2 && S % 2 == 0, "s2d shapes");
    size_t total = (size_t)batch * out.H * out.W * 2;
    if (total == 0) return ADP_OK;
    int grid = (int)((total + 255) / 256 < 148 * 32 ? (total + 255) / 256 : 148 * 32);
    pack_s2d_kernel<<<grid, 256, 0, stream>>>(crops, out.hi, out.lo, batch, S, out.f16);
    ADP_CUDA(cudaGetLastError());
    return ADP_OK;
}

}  // namespace adp
