// Plane-sweep volume: homography warp of the other view's feature map into the reference view for every
// depth hypothesis, fused with the reference features (ADA/lib/network_v5.py:378-416,429):
//   vol[b, d, y, x, :] = feat_ref[b, y, x, :] + bilinear(feat_src[b], u(d, y, x), v(d, y, x))
// The coordinate convention is reproduced as written: normalise with (W-1)/2, sample with
// align_corners=False, zeros padding.
#include "common.cuh"
#include "warp.cuh"

namespace adp {

// Tiled builder (fp16 features): one block = a 16 x 16 tile of reference pixels for VT_DG consecutive depth planes.
// The plane-sweep gather reads every source pixel ~4 times (once per bilinear footprint that covers it); done per voxel
// from global memory that is 256 B of L2 traffic per 64 B written, and the kernel is L2-bandwidth bound.  Here the
// source footprint of the tile at one depth (the bounding box of its 256 sample cells, found with a block min/max) is
// staged in shared memory once (cp.async, every copy in flight) and the four corners are read from there; the reference
// features are re-read per plane (L1 / L2 hits) rather than held in 16 registers.  A footprint larger than the staging
// buffer (strong rotation / scale between the views) falls back to the direct gather for that (tile, depth).
// The kernel was bound by instruction issue (529 warp instructions per voxel and plane, now 286), so the inner loop is kept
// lean: the bilinear blend runs on the mixed-precision
// FMA (fhfma8: the fp16 feature times the fp16-rounded bilinear weight, exact product, fp32 accumulation - the weight rounding
// of <= 2^-11 relative per corner sits below the fp16 storage rounding of the result), the per-voxel projection uses one
// reciprocal instead of four divisions (sample positions agree with the reference's expression to ~5e-5 px), and the footprint
// is staged row by row (no integer divisions).
constexpr int VT_T = 16;
constexpr int VT_DG = 8;
constexpr int VT_MAXPX = 480;                 // staged source pixels (x 64 B = 30 KB; + 16 KB of transpose buffers < 48 KB static)
constexpr int VT_PLANE = VT_MAXPX + 2;        // chunk planes 8 banks apart: the row-wise fill (lane -> chunk, pixel) is conflict-free

__device__ __forceinline__ void vt_unpack8(const uint4& u, float* v) {
    const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&w[q]));
        v[2 * q] = f.x; v[2 * q + 1] = f.y;
    }
}

__device__ __forceinline__ void vt_pack8(const float* v, int f16, uint4* o) {
    uint32_t w[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        if (f16) {
            const __half2 h = __floats2half2_rn(v[2 * q], v[2 * q + 1]);
            w[q] = *reinterpret_cast<const uint32_t*>(&h);
        } else {
            w[q] = (uint32_t)__bfloat16_as_ushort(__float2bfloat16_rn(v[2 * q])) | ((uint32_t)__bfloat16_as_ushort(__float2bfloat16_rn(v[2 * q + 1])) << 16);
        }
    }
    *o = make_uint4(w[0], w[1], w[2], w[3]);
}

// accumulate the four bilinear corners of one half (16 channels) of a voxel into v.  STAGED: corners come from the staged
// footprint (cidx[k] = clamped pixel index, so that a zero-weight corner multiplies finite data); otherwise from global memory.
template <bool STAGED>
__device__ __forceinline__ void vt_corners(const uint4 (*__restrict__ stage)[VT_PLANE], const __half* __restrict__ src, const int (&cidx)[4],
                                           const uint32_t (&wk)[4], int h, float* v) {
#pragma unroll
    for (int k = 0; k < 4; ++k) {
#pragma unroll
        for (int q = 0; q < 2; ++q) {
            uint4 u;
            if (STAGED) u = stage[2 * h + q][cidx[k]];
            else u = __ldg(reinterpret_cast<const uint4*>(src + (size_t)cidx[k] * 32) + 2 * h + q);
            fhfma8(u, wk[k], v + 8 * q);
        }
    }
}

__global__ void __launch_bounds__(256, 4)
build_volume_tile_kernel(const __half* __restrict__ f_ref, const __half* __restrict__ f_src, const float* __restrict__ Mw,
                         const float* __restrict__ depths, bf16* __restrict__ vol, int D, int H, int W, int tiles_x, int f16) {
    constexpr int C = 32;
    __shared__ uint4 stage[4][VT_PLANE];        // [16-byte channel chunk][pixel]: consecutive lanes -> consecutive words
    __shared__ uint4 obuf[8][32 * 4];           // per-warp output transpose: 32 voxels x 64 B
    __shared__ int s_box[2][4];                 // footprint box of the current depth plane, double-buffered by plane parity
    __shared__ unsigned char s_empty[VT_DG];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int tyi = blockIdx.x / tiles_x, txi = blockIdx.x - tyi * tiles_x;
    const int b = blockIdx.z, d0 = blockIdx.y * VT_DG;
    const int x = txi * VT_T + (tid & (VT_T - 1)), y = tyi * VT_T + (tid >> 4);
    const bool inb = x < W && y < H;
    const float* M = Mw + 12 * b;
    const __half* src = f_src + (size_t)b * H * W * C;
    // the reference features are re-read per plane (16 KB per tile: L1 / L2 hits) instead of living in 16 registers
    const uint4* rp = reinterpret_cast<const uint4*>(f_ref + (((size_t)b * H + min(y, H - 1)) * W + min(x, W - 1)) * C);
    if (tid < 8) s_box[tid >> 2][tid & 3] = (tid & 2) ? INT_MIN : INT_MAX;
    // Cheap emptiness test per depth plane: with positive projective depth at the four tile corners the tile maps to the convex
    // hull of its corner images, so if all four fall outside the source map on the same side no voxel of the tile samples
    // anything and the plane is the reference features bit for bit (one warp: 8 planes x 4 corners; 0.01 px safety margin).
    if (tid < 32) {
        const int dd = tid >> 2, c = tid & 3;
        const int cx = min(txi * VT_T + ((c & 1) ? VT_T - 1 : 0), W - 1), cy = min(tyi * VT_T + ((c & 2) ? VT_T - 1 : 0), H - 1);
        bool bad = true, left = false, right = false, top = false, bottom = false;
        if (d0 + dd < D) {
            const float dep = depths[d0 + dd];
            const float Z = (M[6] * (float)cx + M[7] * (float)cy + M[8]) * dep + M[11];
            float ix, iy;
            warp_coords(M, (float)cx, (float)cy, dep, W, H, &ix, &iy);
            bad = !(Z > 1e-6f) || !isfinite(ix) || !isfinite(iy);
            left = ix < -1.01f; right = ix > (float)W + 0.01f; top = iy < -1.01f; bottom = iy > (float)H + 0.01f;
        }
        unsigned int bits = (bad ? 1u : 0u) | (left ? 0u : 2u) | (right ? 0u : 4u) | (top ? 0u : 8u) | (bottom ? 0u : 16u);   // OR-reducible
        bits |= __shfl_xor_sync(0xffffffffu, bits, 1);
        bits |= __shfl_xor_sync(0xffffffffu, bits, 2);
        // bit 0 clear: every corner is in front of the camera; bit k clear (k = 1..4): every corner is outside on side k
        if (c == 0) s_empty[dd] = (!(bits & 1u) && ((bits & 30u) != 30u)) ? 1 : 0;
    }
    __syncthreads();
    // depth-independent part of the projection (warp.cuh)
    const float rx = M[0] * (float)x + M[1] * (float)y + M[2];
    const float ry = M[3] * (float)x + M[4] * (float)y + M[5];
    const float rz = M[6] * (float)x + M[7] * (float)y + M[8];
    // Output addressing, fixed over the depth loop.  A per-thread 64-byte row would make every store instruction touch 32 separate
    // lines (3.7 TB/s measured, against 6.9 TB/s for warp-contiguous stores: tools/micro/store_pattern.cu); the results pass the
    // warp's transpose buffer instead and store instruction k writes voxels 8 k .. 8 k + 7 of the warp x 64 B = 512 contiguous
    // bytes (a warp covers two tile rows of 16 voxels).
    uint4* ob = obuf[warp];
    const int vx0 = lane >> 2, oc = lane & 3;
    const int oy0 = tyi * VT_T + warp * 2, ox0 = txi * VT_T + vx0;
    uint4* op = reinterpret_cast<uint4*>(vol + ((((size_t)b * D + d0) * H + oy0) * W + ox0) * C) + oc;
    const size_t plane16 = (size_t)H * W * (C / 8), row16 = (size_t)W * (C / 8);
    const bool ok_x0 = ox0 < W, ok_x1 = ox0 + 8 < W, ok_y0 = oy0 < H, ok_y1 = oy0 + 1 < H;
    auto store_rows = [&](uint4* o) {            // obuf -> global (after a __syncwarp)
        const uint4 a0 = ob[vx0 * 4 + (oc ^ ((vx0 >> 1) & 3))], a1 = ob[(vx0 + 8) * 4 + (oc ^ ((vx0 >> 1) & 3))];
        const uint4 a2 = ob[(vx0 + 16) * 4 + (oc ^ ((vx0 >> 1) & 3))], a3 = ob[(vx0 + 24) * 4 + (oc ^ ((vx0 >> 1) & 3))];
        if (ok_y0 && ok_x0) o[0] = a0;
        if (ok_y0 && ok_x1) o[8 * (C / 8)] = a1;
        if (ok_y1 && ok_x0) o[row16] = a2;
        if (ok_y1 && ok_x1) o[row16 + 8 * (C / 8)] = a3;
    };
    const int osw = (lane >> 1) & 3;            // chunk swizzle of this lane's row in the transpose buffer
    // the same four (voxel, chunk) slots of the reference map: an empty plane is a plain copy with the store pattern's coalescing
    const uint4* rq = reinterpret_cast<const uint4*>(f_ref + (((size_t)b * H + min(oy0, H - 1)) * W + min(ox0, W - 1)) * C) + oc;
    for (int d = d0; d < d0 + VT_DG && d < D; ++d, op += plane16) {
        if (s_empty[d - d0] && f16) {       // uniform over the block
            if (ok_y0 && ok_x0) op[0] = __ldg(rq);
            if (ok_y0 && ok_x1) op[8 * (C / 8)] = __ldg(rq + 8 * (C / 8));
            if (ok_y1 && ok_x0) op[row16] = __ldg(rq + row16);
            if (ok_y1 && ok_x1) op[row16 + 8 * (C / 8)] = __ldg(rq + row16 + 8 * (C / 8));
            continue;
        }
        int* box = s_box[d & 1];
        Bilin bl;
        bl.any = false;
        if (inb) {
            float ix, iy;
            warp_coords_rcp(M, rx, ry, rz, depths[d], W, H, &ix, &iy);
            bl = bilin_setup(ix, iy, W, H);
        }
        {
            const unsigned int act = __ballot_sync(0xffffffffu, bl.any);
            if (bl.any) {
                const int xmn = __reduce_min_sync(act, bl.x0), ymn = __reduce_min_sync(act, bl.y0);
                const int xmx = __reduce_max_sync(act, bl.x0), ymx = __reduce_max_sync(act, bl.y0);
                if (lane == __ffs(act) - 1) {
                    atomicMin(&box[0], xmn); atomicMin(&box[1], ymn);
                    atomicMax(&box[2], xmx + 1); atomicMax(&box[3], ymx + 1);
                }
            }
        }
        __syncthreads();                         // A: the box is complete; the previous plane's readers of `stage` are done
        const bool some = box[2] >= box[0];                               // any thread of the tile samples inside the source map
        const int bx0 = some ? max(box[0], 0) : 0, by0 = some ? max(box[1], 0) : 0;
        const int bx1 = some ? min(box[2], W - 1) : -1, by1 = some ? min(box[3], H - 1) : -1;
        const int bw = bx1 - bx0 + 1, bh = by1 - by0 + 1;
        // Reset the other parity's box for plane d + 1 here, between A and B.  Its last readers (plane d - 1, between its own A
        // and B) are done before this plane's A, and its next writers (plane d + 1's atomics) start after this plane's B.  After B
        // the reset would be unordered against a faster warp's plane-(d + 1) atomics and could erase its extents.  A plane that
        // takes the empty shortcut above skips this reset, so the plane after it starts from the box of the plane two before:
        // a superset of its own box, which can only turn a staged plane into a fallback one, never drop a pixel.
        if (tid < 4) s_box[(d + 1) & 1][tid] = (tid & 2) ? INT_MIN : INT_MAX;
        const bool staged = bw > 0 && bh > 0 && bw * bh <= VT_MAXPX;       // uniform over the block
        if (staged) {           // a warp per footprint row (bw x 64 contiguous bytes, lane -> (pixel, 16-byte chunk)), every copy in flight at once;
                                // through L1: neighbouring planes and tiles re-read most of the footprint (.ca 1.51 ms, .cg 1.65 ms per chunk)
            const int rowq = bw * 4;
            for (int r = warp; r < bh; r += 8) {
                const uint4* g = reinterpret_cast<const uint4*>(src + ((size_t)(by0 + r) * W + bx0) * C);
                uint4* st = &stage[lane & 3][r * bw + (lane >> 2)];
                for (int i = lane; i < rowq; i += 32, st += 8) cp_async16_ca(st, g + i);
            }
            cp_async_wait_all();
        }
        __syncthreads();                         // B: the footprint is staged
        uint32_t wk[4];         // the weights as fp16 multipliers of the mixed-precision FMA (0 where a corner is outside)
        wk[0] = __half_as_ushort(__float2half_rn(bl.w00)); wk[1] = __half_as_ushort(__float2half_rn(bl.w01));
        wk[2] = __half_as_ushort(__float2half_rn(bl.w10)); wk[3] = __half_as_ushort(__float2half_rn(bl.w11));
        int cidx[4];
        if (staged) {
            const int i00 = (bl.y0 - by0) * bw + (bl.x0 - bx0), last = bw * bh - 1;
            cidx[0] = min(max(i00, 0), last); cidx[1] = min(max(i00 + 1, 0), last);
            cidx[2] = min(max(i00 + bw, 0), last); cidx[3] = min(max(i00 + bw + 1, 0), last);
        } else {
            const int xa = min(max(bl.x0, 0), W - 1), xb = min(max(bl.x0 + 1, 0), W - 1);
            const int ya = min(max(bl.y0, 0), H - 1), yb = min(max(bl.y0 + 1, 0), H - 1);
            cidx[0] = ya * W + xa; cidx[1] = ya * W + xb; cidx[2] = yb * W + xa; cidx[3] = yb * W + xb;
        }
#pragma unroll
        for (int h = 0; h < 2; ++h) {            // two halves of 16 channels: keeps the kernel under 64 registers
            float v[16];
            vt_unpack8(__ldg(rp + 2 * h), v);
            vt_unpack8(__ldg(rp + 2 * h + 1), v + 8);
            if (bl.any) {
                if (staged) vt_corners<true>(stage, src, cidx, wk, h, v);
                else vt_corners<false>(stage, src, cidx, wk, h, v);
            }
            // park the 16-bit result in the warp's transpose buffer (chunk index XOR-swizzled: conflict-free both ways)
#pragma unroll
            for (int q = 0; q < 2; ++q) {
                uint4 o;
                vt_pack8(v + 8 * q, f16, &o);
                ob[lane * 4 + ((2 * h + q) ^ osw)] = o;
            }
        }
        __syncwarp();
        store_rows(op);
        __syncwarp();
    }
}

int build_volume(const void* f_ref, const void* f_src, const float* Mw, const float* depths, bf16* vol, int B, int D, int H,
                 int W, int C, int f16, cudaStream_t stream) {
    ADP_CHECK_ARG(C == 32, "feature channels must be 32");
    if ((size_t)B * D * H * W == 0) return ADP_OK;
    const int tiles_x = cdiv(W, VT_T), tiles_y = cdiv(H, VT_T);
    build_volume_tile_kernel<<<dim3(tiles_x * tiles_y, cdiv(D, VT_DG), B), 256, 0, stream>>>(
        reinterpret_cast<const __half*>(f_ref), reinterpret_cast<const __half*>(f_src), Mw, depths, vol, D, H, W, tiles_x, f16);
    ADP_CUDA(cudaGetLastError());
    return ADP_OK;
}

// M = P_src * inv(P_ref) with P = [K' E[:3,:]; 0 0 0 1] (ADA/interface_v5.py:264-270, network_v5.py:389-392), in fp64.
// Mw[b] = {rot(9) row-major, trans(3)} as fp32.  Kp_* [B,9], E_* [B,16] row-major doubles.
__global__ void warp_matrices_kernel(const double* __restrict__ Kp_ref, const double* __restrict__ E_ref,
                                     const double* __restrict__ Kp_src, const double* __restrict__ E_src, float* __restrict__ Mw,
                                     const uint8_t* __restrict__ valid_ref, const uint8_t* __restrict__ valid_src,
                                     uint8_t* __restrict__ valid_env, int B) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    // an estimate needs both views (interface_v5.py:256-257)
    if (valid_env) valid_env[b] = (valid_ref ? valid_ref[b] : 1) && (valid_src ? valid_src[b] : 1);
    double Pr[16], Ps[16];
    for (int which = 0; which < 2; ++which) {
        const double* K = (which ? Kp_src : Kp_ref) + 9 * b;
        const double* E = (which ? E_src : E_ref) + 16 * b;
        double* P = which ? Ps : Pr;
        for (int r = 0; r < 3; ++r)
            for (int c = 0; c < 4; ++c) P[4 * r + c] = K[3 * r] * E[c] + K[3 * r + 1] * E[4 + c] + K[3 * r + 2] * E[8 + c];
        P[12] = 0; P[13] = 0; P[14] = 0; P[15] = 1;
    }
    // Gauss-Jordan inverse of P_ref
    double a[4][8];
    for (int r = 0; r < 4; ++r)
        for (int c = 0; c < 4; ++c) { a[r][c] = Pr[4 * r + c]; a[r][4 + c] = (r == c) ? 1.0 : 0.0; }
    for (int col = 0; col < 4; ++col) {
        int piv = col;
        double best = fabs(a[col][col]);
        for (int r = col + 1; r < 4; ++r) if (fabs(a[r][col]) > best) { best = fabs(a[r][col]); piv = r; }
        if (piv != col) for (int c = 0; c < 8; ++c) { double t = a[col][c]; a[col][c] = a[piv][c]; a[piv][c] = t; }
        const double d = 1.0 / a[col][col];
        for (int c = 0; c < 8; ++c) a[col][c] *= d;
        for (int r = 0; r < 4; ++r) if (r != col) {
            const double f = a[r][col];
            for (int c = 0; c < 8; ++c) a[r][c] -= f * a[col][c];
        }
    }
    float* out = Mw + 12 * b;
    for (int r = 0; r < 3; ++r) {
        for (int c = 0; c < 4; ++c) {
            double s = 0;
            for (int k = 0; k < 4; ++k) s += Ps[4 * r + k] * a[k][4 + c];
            if (c < 3) out[3 * r + c] = (float)s; else out[9 + r] = (float)s;
        }
    }
}

int warp_matrices(const double* Kp_ref, const double* E_ref, const double* Kp_src, const double* E_src, float* Mw,
                  const uint8_t* valid_ref, const uint8_t* valid_src, uint8_t* valid_env, int B, cudaStream_t stream) {
    if (B == 0) return ADP_OK;
    warp_matrices_kernel<<<cdiv(B, 64), 64, 0, stream>>>(Kp_ref, E_ref, Kp_src, E_src, Mw, valid_ref, valid_src, valid_env, B);
    ADP_CUDA(cudaGetLastError());
    return ADP_OK;
}

}  // namespace adp
