// Per-view preprocessing on device (ADA/interface_v5.py:58-170, ADA/lib/utils.py:10-38):
//   mask bounding box -> square crop window (multiple of 40, <= 440, shifted inside the frame)
//   -> bilinear crop resize to S x S (cv2 INTER_LINEAR semantics) + ImageNet normalisation
//   -> nearest mask resize (cv2 INTER_NEAREST index rule) -> exactly P sampled foreground indices
//   -> crop-adjusted intrinsics K'.
#include "stages.cuh"

namespace adp {

enum { DT_U8 = 0, DT_F32 = 1, DT_F64 = 2, DT_F16 = 3 };

__device__ __forceinline__ bool mask_on(const void* m, int dt, size_t i) {
    switch (dt) {
        case DT_U8: return reinterpret_cast<const uint8_t*>(m)[i] != 0;
        case DT_F32: return reinterpret_cast<const float*>(m)[i] != 0.f;
        default: return reinterpret_cast<const double*>(m)[i] != 0.0;
    }
}

// ---- 1. bounding box of the nonzero mask pixels: bbox[f] = {ymin, xmin, ymax, xmax}; init {H, W, -1, -1}
__global__ void mask_bbox_init_kernel(int* bbox, int F, int H, int W) {
    int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f < F) { bbox[4 * f] = H; bbox[4 * f + 1] = W; bbox[4 * f + 2] = -1; bbox[4 * f + 3] = -1; }
}

__global__ void mask_bbox_kernel(const void* __restrict__ mask, int dt, int* __restrict__ bbox, int H, int W) {
    const int f = blockIdx.y;
    const size_t base = (size_t)f * H * W;
    int ymin = H, xmin = W, ymax = -1, xmax = -1;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < H * W; i += gridDim.x * blockDim.x) {
        if (mask_on(mask, dt, base + i)) {
            const int y = i / W, x = i - y * W;
            ymin = min(ymin, y); ymax = max(ymax, y); xmin = min(xmin, x); xmax = max(xmax, x);
        }
    }
    for (int o = 16; o > 0; o >>= 1) {
        ymin = min(ymin, __shfl_xor_sync(0xffffffffu, ymin, o));
        xmin = min(xmin, __shfl_xor_sync(0xffffffffu, xmin, o));
        ymax = max(ymax, __shfl_xor_sync(0xffffffffu, ymax, o));
        xmax = max(xmax, __shfl_xor_sync(0xffffffffu, xmax, o));
    }
    if ((threadIdx.x & 31) == 0 && ymax >= 0) {
        atomicMin(&bbox[4 * f], ymin); atomicMin(&bbox[4 * f + 1], xmin);
        atomicMax(&bbox[4 * f + 2], ymax); atomicMax(&bbox[4 * f + 3], xmax);
    }
}

// ---- 2. crop window (utils.py:10-38) and K' (interface_v5.py:151-168).  win[f] = {rmin, rmax, cmin, cmax}; valid[f]
__global__ void window_kernel(const int* __restrict__ bbox, const double* __restrict__ K, int k_stride, int* __restrict__ win,
                              double* __restrict__ Kp, uint8_t* __restrict__ valid, int F, int H, int W, int S) {
    const int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= F) return;
    const int y1 = bbox[4 * f], x1 = bbox[4 * f + 1], y2 = bbox[4 * f + 2], x2 = bbox[4 * f + 3];
    if (y2 < 0) {
        valid[f] = 0;
        win[4 * f] = 0; win[4 * f + 1] = 40; win[4 * f + 2] = 0; win[4 * f + 3] = 40;
        if (Kp) for (int i = 0; i < 9; ++i) Kp[9 * f + i] = (i % 4 == 0) ? 1.0 : 0.0;
        return;
    }
    int ws = (max(y2 - y1, x2 - x1) / 40 + 1) * 40;
    ws = min(ws, 440);
    const int cy = (y1 + y2) / 2, cx = (x1 + x2) / 2;
    int rmin = cy - ws / 2, rmax = cy + ws / 2, cmin = cx - ws / 2, cmax = cx + ws / 2;
    if (rmin < 0) { rmax -= rmin; rmin = 0; }
    if (cmin < 0) { cmax -= cmin; cmin = 0; }
    if (rmax > H) { rmin -= rmax - H; rmax = H; }
    if (cmax > W) { cmin -= cmax - W; cmax = W; }
    win[4 * f] = rmin; win[4 * f + 1] = rmax; win[4 * f + 2] = cmin; win[4 * f + 3] = cmax;
    valid[f] = 1;
    if (!Kp) return;
    const double* k = K + (size_t)f * k_stride;
    const double ratio = (double)S / (double)(rmax - rmin);
    const double ccx = (double)(cmin + cmax) / 2, ccy = (double)(rmin + rmax) / 2;
    const double csx = (double)(cmax - cmin + 1), csy = (double)(rmax - rmin + 1);
    double* o = Kp + 9 * f;
    o[0] = k[0] * ratio; o[1] = 0; o[2] = (k[2] - (ccx - csx / 2)) * ratio;
    o[3] = 0; o[4] = k[4] * ratio; o[5] = (k[5] - (ccy - csy / 2)) * ratio;
    o[6] = 0; o[7] = 0; o[8] = 1;
}

// ---- 3. crop + bilinear resize + normalise -> fp32 NHWC3
// 8-bit frames: value / 255 in fp32, what torchvision's ToTensor (interface_v5.py:52,149) makes of a uint8 image.  The u8 path
// is defined as "the fp32 path on rgb.float() / 255" (bit for bit); the reference callers always pass floats in [0, 1].
struct U8AsF32 {};
template <typename S> struct rgb_math { typedef S type; };
template <> struct rgb_math<U8AsF32> { typedef float type; };
template <typename S>
__device__ __forceinline__ typename rgb_math<S>::type ld_rgb(const void* p, size_t i) { return reinterpret_cast<const S*>(p)[i]; }
template <>
__device__ __forceinline__ float ld_rgb<U8AsF32>(const void* p, size_t i) { return (float)reinterpret_cast<const uint8_t*>(p)[i] / 255.f; }

template <typename SRC>   // float or double: OpenCV interpolates in the source float type; U8AsF32: see above
__global__ void crop_resize_kernel(const void* __restrict__ rgb, const int* __restrict__ win, const uint8_t* __restrict__ valid,
                                   float* __restrict__ out, int H, int W, int S) {
    const int f = blockIdx.y;
    if (!valid[f]) {
        for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < S * S * 3; i += gridDim.x * blockDim.x)
            out[(size_t)f * S * S * 3 + i] = 0.f;
        return;
    }
    const int rmin = win[4 * f], rmax = win[4 * f + 1], cmin = win[4 * f + 2];
    const int ws = rmax - rmin;
    typedef typename rgb_math<SRC>::type T;
    const double scale = (double)ws / (double)S;
    const T mean[3] = {(T)0.485, (T)0.456, (T)0.406};
    const T stdv[3] = {(T)0.229, (T)0.224, (T)0.225};
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < S * S; i += gridDim.x * blockDim.x) {
        const int oy = i / S, ox = i - oy * S;
        double fy = ((double)oy + 0.5) * scale - 0.5, fx = ((double)ox + 0.5) * scale - 0.5;
        int y0 = (int)floor(fy), x0 = (int)floor(fx);
        T wy = (T)(fy - (double)y0), wx = (T)(fx - (double)x0);
        if (y0 < 0) { y0 = 0; wy = 0; }
        if (x0 < 0) { x0 = 0; wx = 0; }
        if (y0 >= ws - 1) { y0 = ws - 1; wy = 0; }
        if (x0 >= ws - 1) { x0 = ws - 1; wx = 0; }
        const int y1 = min(y0 + 1, ws - 1), x1 = min(x0 + 1, ws - 1);
        const size_t r0 = ((size_t)f * H + rmin + y0) * W + cmin, r1 = ((size_t)f * H + rmin + y1) * W + cmin;
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const T a = ld_rgb<SRC>(rgb, (r0 + x0) * 3 + c), b = ld_rgb<SRC>(rgb, (r0 + x1) * 3 + c);
            const T cc = ld_rgb<SRC>(rgb, (r1 + x0) * 3 + c), d = ld_rgb<SRC>(rgb, (r1 + x1) * 3 + c);
            const T top = a * ((T)1 - wx) + b * wx, bot = cc * ((T)1 - wx) + d * wx;   // horizontal pass first
            const T v = top * ((T)1 - wy) + bot * wy;
            out[((size_t)f * S * S + i) * 3 + c] = (float)((v - mean[c]) / stdv[c]);
        }
    }
}

// ---- 4. nearest mask resize + sampling of exactly P pixels (interface_v5.py:121-134)
__device__ __forceinline__ uint32_t mix32(uint32_t x) {
    x ^= x >> 16; x *= 0x7feb352du; x ^= x >> 15; x *= 0x846ca68bu; x ^= x >> 16;
    return x;
}

__device__ __forceinline__ int block_exclusive_scan(int v, int* warp_sums, int* total) {
    // blockDim.x == 1024
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    int x = v;
    for (int o = 1; o < 32; o <<= 1) {
        const int y = __shfl_up_sync(0xffffffffu, x, o);
        if (lane >= o) x += y;
    }
    if (lane == 31) warp_sums[w] = x;
    __syncthreads();
    if (w == 0) {
        int s = warp_sums[lane];
        for (int o = 1; o < 32; o <<= 1) {
            const int y = __shfl_up_sync(0xffffffffu, s, o);
            if (lane >= o) s += y;
        }
        warp_sums[lane] = s;
    }
    __syncthreads();
    const int base = w > 0 ? warp_sums[w - 1] : 0;
    *total = warp_sums[31];
    __syncthreads();
    return base + x - v;
}

// One CTA (1024 threads) per frame.  choose[f, P] ascending flat indices y*S + x.
// mode 0: device sampling (counter-based hash keyed by seed/frame/rank picks a uniform P-subset when more than P
//         foreground pixels exist -- same distribution as the reference's np.random.shuffle selector, different stream);
// mode 1: the caller supplies choose (exact replay of the reference RNG); only counts are produced.
__global__ void __launch_bounds__(1024)
choose_kernel(const void* __restrict__ mask, int dt, const int* __restrict__ win, uint8_t* __restrict__ valid,
              int* __restrict__ choose, int* __restrict__ counts, int H, int W, int S, int P, uint32_t seed, int mode,
              int frame_id0) {
    extern __shared__ int sm[];
    int* warp_sums = sm;                     // 32
    int* hist = sm + 32;                     // 256
    int* misc = sm + 32 + 256;               // 8
    uint8_t* flags = reinterpret_cast<uint8_t*>(sm + 32 + 256 + 8);   // S*S bytes
    const int f = blockIdx.x;
    const int tid = threadIdx.x;
    const int npix = S * S;
    if (!valid[f]) {
        if (tid == 0) counts[f] = 0;
        if (mode == 0) for (int i = tid; i < P; i += blockDim.x) choose[(size_t)f * P + i] = 0;
        return;
    }
    const int rmin = win[4 * f], rmax = win[4 * f + 1], cmin = win[4 * f + 2];
    const int ws = rmax - rmin;
    const double inv = 1.0 / ((double)S / (double)ws);   // OpenCV resizeNN: sx = floor(x * inv_scale), clamped
    for (int i = tid; i < npix; i += blockDim.x) {
        const int oy = i / S, ox = i - oy * S;
        const int sy = min((int)floor((double)oy * inv), ws - 1), sx = min((int)floor((double)ox * inv), ws - 1);
        flags[i] = mask_on(mask, dt, ((size_t)f * H + rmin + sy) * W + cmin + sx) ? 1 : 0;
    }
    __syncthreads();
    // per-thread contiguous segment so that ranks follow the row-major order
    const int per = (npix + blockDim.x - 1) / blockDim.x;
    const int lo = tid * per, hi = min(lo + per, npix);
    int cnt = 0;
    for (int i = lo; i < hi; ++i) cnt += flags[i];
    int n;
    const int rank0 = block_exclusive_scan(cnt, warp_sums, &n);
    if (tid == 0) counts[f] = n;
    if (n == 0) {
        if (tid == 0) valid[f] = 0;
        if (mode == 0) for (int i = tid; i < P; i += blockDim.x) choose[(size_t)f * P + i] = 0;
        return;
    }
    if (mode != 0) return;
    int* out = choose + (size_t)f * P;
    if (n <= P) {
        // np.pad(choose, (0, P - n), 'wrap')
        int r = rank0;
        for (int i = lo; i < hi; ++i)
            if (flags[i]) {
                for (int k = r; k < P; k += n) out[k] = i;
                ++r;
            }
        return;
    }
    // more than P candidates: keep the P smallest hash keys (ties resolved by rank), output in ascending index order
    // keyed by the caller's frame id (the global environment index), not by the position inside this launch: the drawn subset
    // of an environment does not depend on how the batch is chunked or sharded over GPUs
    const uint32_t salt = mix32(seed ^ (0x9e3779b9u * (uint32_t)(frame_id0 + f + 1)));
    uint32_t prefix = 0, pmask = 0;
    int need = P;   // how many still to take among keys matching the prefix
    for (int shift = 24; shift >= 0; shift -= 8) {
        for (int i = tid; i < 256; i += blockDim.x) hist[i] = 0;
        __syncthreads();
        int r = rank0;
        for (int i = lo; i < hi; ++i)
            if (flags[i]) {
                const uint32_t key = mix32(salt + (uint32_t)r * 0x85ebca6bu);
                if ((key & pmask) == prefix) atomicAdd(&hist[(key >> shift) & 255], 1);
                ++r;
            }
        __syncthreads();
        if (tid == 0) {
            int acc = 0, b = 0;
            for (; b < 256; ++b) {
                if (acc + hist[b] >= need) break;
                acc += hist[b];
            }
            misc[0] = b; misc[1] = need - acc;
        }
        __syncthreads();
        prefix |= (uint32_t)misc[0] << shift;
        pmask |= 0xffu << shift;
        need = misc[1];
        __syncthreads();
    }
    // keys < prefix are all taken; keys == prefix: the first `need` in rank order
    int sel = 0, eq = 0;
    {
        int r = rank0;
        for (int i = lo; i < hi; ++i)
            if (flags[i]) {
                const uint32_t key = mix32(salt + (uint32_t)r * 0x85ebca6bu);
                sel += key < prefix; eq += key == prefix;
                ++r;
            }
    }
    int tot_eq;
    const int eq0 = block_exclusive_scan(eq, warp_sums, &tot_eq);
    int take_eq = max(0, min(eq, need - eq0));
    int tot_sel;
    const int pos0 = block_exclusive_scan(sel + take_eq, warp_sums, &tot_sel);
    {
        int r = rank0, pos = pos0, e = eq0;
        for (int i = lo; i < hi; ++i)
            if (flags[i]) {
                const uint32_t key = mix32(salt + (uint32_t)r * 0x85ebca6bu);
                bool take = key < prefix;
                if (key == prefix) { take = e < need; ++e; }
                if (take && pos < P) out[pos++] = i;
                ++r;
            }
    }
}

// crop windows only (the first three kernels of preprocess_run): lets the host upload just the image rows a window covers
int mask_windows_run(const void* mask, int mask_dt, int F, int H, int W, int* bbox_ws, int* win, uint8_t* valid, cudaStream_t stream) {
    ADP_CHECK_ARG(mask_dt == DT_U8 || mask_dt == DT_F32 || mask_dt == DT_F64, "mask dtype must be u8, f32 or f64");
    ADP_CHECK_ARG(H >= 440 && W >= 440, "frames must be at least 440 x 440 (crop window of utils.py:get_bbox)");
    if (F == 0) return ADP_OK;
    mask_bbox_init_kernel<<<cdiv(F, 256), 256, 0, stream>>>(bbox_ws, F, H, W);
    mask_bbox_kernel<<<dim3(30, F), 256, 0, stream>>>(mask, mask_dt, bbox_ws, H, W);
    window_kernel<<<cdiv(F, 128), 128, 0, stream>>>(bbox_ws, nullptr, 0, win, nullptr, valid, F, H, W, 224);
    ADP_CUDA(cudaGetLastError());
    return ADP_OK;
}

int preprocess_run(const void* rgb, int rgb_dt, const void* mask, int mask_dt, const double* K, int k_stride, int F, int H, int W,
                   int S, int P, uint32_t seed, int choose_mode, int frame_id0, int* bbox_ws, int* win, double* Kp, uint8_t* valid,
                   float* crops, int* choose, int* counts, cudaStream_t stream) {
    ADP_CHECK_ARG(rgb_dt == DT_F32 || rgb_dt == DT_F64 || rgb_dt == DT_U8, "rgb dtype must be u8, f32 or f64");
    // the crop window is a square of up to 440 pixels shifted inside the frame (utils.py:10-38 hard-codes 480 x 640): a smaller
    // frame cannot hold it and the shifted window would start before the frame
    ADP_CHECK_ARG(H >= 440 && W >= 440, "frames must be at least 440 x 440 (crop window of utils.py:get_bbox)");
    ADP_CHECK_ARG(mask_dt == DT_U8 || mask_dt == DT_F32 || mask_dt == DT_F64, "mask dtype must be u8, f32 or f64");
    ADP_CHECK_ARG(S * S <= 65536 && P <= S * S, "sizes");
    if (F == 0) return ADP_OK;
    mask_bbox_init_kernel<<<cdiv(F, 256), 256, 0, stream>>>(bbox_ws, F, H, W);
    mask_bbox_kernel<<<dim3(30, F), 256, 0, stream>>>(mask, mask_dt, bbox_ws, H, W);
    window_kernel<<<cdiv(F, 128), 128, 0, stream>>>(bbox_ws, K, k_stride, win, Kp, valid, F, H, W, S);
    const size_t smem = (32 + 256 + 8) * sizeof(int) + (size_t)S * S;
    static int attr[kMaxDevices];
    ADP_TRY(ensure_dyn_smem(choose_kernel, 72 * 1024, attr));
    choose_kernel<<<F, 1024, smem, stream>>>(mask, mask_dt, win, valid, choose, counts, H, W, S, P, seed, choose_mode, frame_id0);
    if (rgb_dt == DT_U8)
        crop_resize_kernel<U8AsF32><<<dim3(49, F), 256, 0, stream>>>(rgb, win, valid, crops, H, W, S);
    else if (rgb_dt == DT_F32)
        crop_resize_kernel<float><<<dim3(49, F), 256, 0, stream>>>(rgb, win, valid, crops, H, W, S);
    else
        crop_resize_kernel<double><<<dim3(49, F), 256, 0, stream>>>(rgb, win, valid, crops, H, W, S);
    ADP_CUDA(cudaGetLastError());
    return ADP_OK;
}

}  // namespace adp
