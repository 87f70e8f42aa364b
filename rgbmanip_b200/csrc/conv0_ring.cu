// conv0 of the cost-regularisation U-Net (ADA/lib/network_v5.py:263,283): 3x3x3, 32 -> 8 channels over the full
// [24, 224, 224] plane-sweep volume -- 68 % of the U-Net's FLOPs with only 8 output channels.
//
// A plain implicit GEMM (M = pixels, N = 8) re-reads the volume 27 times and leaves the MMA N dimension nearly empty.
// This kernel instead walks the depth axis sequentially and folds BOTH the depth taps and the row taps into N:
//
//   P[d'][y'][pixel, (kz, ky, co)] = sum_{kx,c} In[d', y', x+kx-1, c] * W[co, c, kz, ky, kx]          (N = 9 x 8 = 72 of 80)
//   out[d][y][pixel, co]           = sum_{kz,ky} P[d+kz-1][y+ky-1][pixel, (kz, ky, co)]
//
// One work unit = R = 4 image rows x one segment of 112 pixels (M = 128 rows of the UMMA tile) for all 24 depths.  For each
// input plane d' the rows y-1 .. y+R (with a one-pixel halo in x) are brought in by ONE TMA box in pixel-major
// 64-byte-swizzled K-major layout ([row][pixel][32 channels]); the swizzle is a function of the absolute shared-memory
// address, so the kx taps are plain pixel shifts of the descriptor start address (+64 B per pixel).  An MMA with N <= 64 is
// bound by the 128 B/clk shared-memory read of its A operand (4 KB per M128 x K16 instruction), not by the tensor pipe: with
// only kz in N (round 1: N = 24, 72 MMAs per plane step) the kernel sat at 93 % L1/TEX throughput.  With (kz, ky) in N every
// input row needs 3 (kx) x 2 (K steps) MMAs of N = 80 -- 36 per plane step, half the A bytes.  Each (plane, input row) product
// lands in one slot of a six-deep 80-column TMEM ring; the epilogue warps pull a slot out once, release it at once, and add its
// nine 8-column groups into three register accumulators per output row (output planes d'-1, d', d'+1), apply the folded
// BatchNorm + ReLU when a plane is complete and store 16 channels (8 real + 8 zero: conv1 needs Cin = 16 for the K = 16 MMA).
#include "common.cuh"
#include "ptx.cuh"

#include <cudaTypedefs.h>
#include <stdlib.h>

namespace adp {

constexpr int C0_THREADS = 320;              // warp 0: TMA, warp 1: MMA, warps 2-5 / 6-9: epilogue of output rows 0-1 / 2-3
constexpr int C0_SEG = 112;                 // pixels per unit (224 = 2 x 112)
constexpr int C0_R = 4;                                   // output rows per unit: rows y0-1 .. y0+R are loaded once for R outputs
constexpr int C0_PIXPITCH = 120;                          // pixels per slab row in smem (112 + halo, padded so that a row is a 128-byte multiple)
constexpr int C0_ROWPITCH = C0_PIXPITCH * 64;             // 7680 bytes: one slab row, 32 channels per pixel (a multiple of the 512-byte swizzle atom)
constexpr int C0_BOX_BYTES = (C0_R + 2) * C0_ROWPITCH;    // one depth plane of the unit = ONE TMA box
constexpr int C0_STAGE_BYTES = C0_BOX_BYTES + 1024;       // + slack: the M = 128 tile overhangs the last slab row by 10 pixels
constexpr int C0_STAGES = 4;
constexpr int C0_N = 80;                                  // MMA N: (kz, ky, co) = 72 columns, padded to a multiple of 16
constexpr int C0_W_BYTES = 3 * 4 * C0_N * 16;             // [kx][chunk][n = 80][8 ch] 16-bit
constexpr int C0_SLOTS = C0_R + 2;                        // TMEM ring over (plane, input row) items; column = slot * 80
constexpr int C0_SMEM = C0_STAGES * C0_STAGE_BYTES + C0_W_BYTES + 1024 + 256;

struct Conv0Params {
    int B, D, H, W;
    int f16;
    const uint16_t* w;        // packed weights, C0_W_BYTES
    const float* scale;       // [8] folded BatchNorm
    const float* shift;       // [8]
    uint16_t* out;            // [B, D, H, W, 16], or space-to-depth(2) [B, D/2, H/2, W/2, 64] (channel = parity * 8 + co)
    int out_s2d;
    int* err;
};

// A operand: K-major, 64-byte swizzle (rows of 64 B = 32 channels; one MMA consumes 32 B of each row), SBO = 8 rows.
__device__ __forceinline__ uint64_t make_desc_sw64(uint32_t addr) {
    return (uint64_t)((addr & 0x3FFFF) >> 4) | (1ull << 16) | ((uint64_t)(512 >> 4) << 32) | (1ull << 46) | (4ull << 61);
}
// B operand (weights): K-major, no swizzle: 8-row x 16-byte core matrices; LBO = byte distance between the two 16-byte K
// chunks of one MMA, SBO = byte distance between consecutive 8-row groups.
__device__ __forceinline__ uint64_t make_desc_noswz(uint32_t addr, uint32_t lbo, uint32_t sbo) {
    return (uint64_t)((addr & 0x3FFFF) >> 4) | ((uint64_t)(lbo >> 4) << 16) | ((uint64_t)(sbo >> 4) << 32) | (1ull << 46);
}

__device__ __forceinline__ void tmem_ld8(uint32_t taddr, uint32_t* r) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr));
}

__global__ void __launch_bounds__(C0_THREADS, 1)
conv0_ring_kernel(const __grid_constant__ CUtensorMap tmIn, const Conv0Params p, int batch) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint8_t* wsm = smem + C0_STAGES * C0_STAGE_BYTES;
    uint64_t* bars = reinterpret_cast<uint64_t*>(wsm + C0_W_BYTES);
    // bars: [0,S) full, [S,2S) empty, [2S,2S+SLOTS) tmem_full, [2S+SLOTS,2S+2 SLOTS) tmem_empty, then the TMEM base
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * C0_STAGES + 2 * C0_SLOTS);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t smem_base = ptx::smem_u32(smem);
    const uint32_t w_base = ptx::smem_u32(wsm);
    const uint32_t bar_base = ptx::smem_u32(bars);
    auto full_bar = [&](int s) { return bar_base + 8u * s; };
    auto empty_bar = [&](int s) { return bar_base + 8u * (C0_STAGES + s); };
    auto tfull_bar = [&](int s) { return bar_base + 8u * (2 * C0_STAGES + s); };
    auto tempty_bar = [&](int s) { return bar_base + 8u * (2 * C0_STAGES + C0_SLOTS + s); };

    // weights -> smem (generic proxy), made visible to the tensor core's async proxy by the fence below
    for (int i = threadIdx.x; i < C0_W_BYTES / 16; i += C0_THREADS)
        reinterpret_cast<uint4*>(wsm)[i] = __ldg(reinterpret_cast<const uint4*>(p.w) + i);
    // the overhang pixels (beyond the 114 loaded ones) are read by MMA rows >= 112 only; keep them finite
    for (int i = threadIdx.x; i < C0_STAGES * C0_STAGE_BYTES / 16; i += C0_THREADS)
        reinterpret_cast<uint4*>(smem)[i] = make_uint4(0, 0, 0, 0);
    ptx::fence_proxy_async();
    if (warp == 0 && lane == 0) {
        ptx::prefetch_tmap(&tmIn);
        for (int s = 0; s < C0_STAGES; ++s) { ptx::mbar_init(full_bar(s), 1); ptx::mbar_init(empty_bar(s), 1); }
        // slot == input row (C0_SLOTS items per plane); rows 2 and 3 feed output rows of both epilogue groups
        for (int s = 0; s < C0_SLOTS; ++s) { ptx::mbar_init(tfull_bar(s), 1); ptx::mbar_init(tempty_bar(s), (s == 2 || s == 3) ? 8 : 4); }
        ptx::fence_barrier_init();
    }
    if (warp == 1) {
        ptx::tmem_alloc(ptx::smem_u32(tmem_slot), 512);
        ptx::tmem_relinquish();
    }
    ptx::tc_fence_before();
    __syncthreads();
    ptx::tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    const int segs = p.W / C0_SEG;
    const int ygroups = p.H / C0_R;
    const int units = batch * ygroups * segs;
    const int D = p.D;

    if (warp == 0) {
        // ===================== TMA producer: one box per plane = (R + 2) rows x 120 pixels x 64 bytes =====================
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            for (int u = blockIdx.x; u < units; u += gridDim.x) {
                const int seg = u % segs, y = ((u / segs) % ygroups) * C0_R, b = u / (segs * ygroups);
                const int x0 = seg * C0_SEG - 1;
                for (int d = 0; d < D; ++d) {
                    ptx::mbar_wait(empty_bar(stage), phase ^ 1, p.err, 11);
                    const uint32_t sa = smem_base + stage * C0_STAGE_BYTES;
                    ptx::mbar_arrive_expect_tx(full_bar(stage), (uint32_t)C0_BOX_BYTES);
                    ptx::tma_load_5d(&tmIn, full_bar(stage), sa, 0, x0, y - 1, d, b);
                    if (++stage == C0_STAGES) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        // ===================== MMA issuer: per input row 3 kx taps x 2 K steps of N = 80 into the next ring slot =====================
        // warp-convergent: all lanes carry the same descriptors, the elected lane issues (see ptx::umma_bf16_elected)
        int stage = 0;
        uint32_t phase = 0;
        const uint32_t idesc = make_idesc_n(C0_N, p.f16);
        const uint32_t elected = ptx::elect_one();
        const uint32_t tbase = __shfl_sync(0xffffffffu, tmem_base, 0);
        int slot = 0;
        uint32_t sphase = 0;          // ring phase: flips every C0_SLOTS items
        for (int u = blockIdx.x; u < units; u += gridDim.x) {
            for (int d = 0; d < D; ++d) {
                ptx::mbar_wait(full_bar(stage), phase, p.err, 13);
                ptx::tc_fence_after();
                const uint32_t sa = smem_base + stage * C0_STAGE_BYTES;
                const uint64_t a0 = make_desc_sw64(sa);
                const uint64_t b0 = make_desc_noswz(w_base, C0_N * 16, 128);
#pragma unroll
                for (int r = 0; r < C0_R + 2; ++r) {
                    ptx::mbar_wait(tempty_bar(slot), sphase ^ 1, p.err, 12);
                    ptx::tc_fence_after();
                    const uint32_t tmem_d = tbase + (uint32_t)(slot * C0_N);
#pragma unroll
                    for (int kx = 0; kx < 3; ++kx)
#pragma unroll
                        for (int ks = 0; ks < 2; ++ks) {
                            // start-address field is (addr >> 4): constant offsets are plain adds (no carry out of the 14-bit field below 256 KB)
                            const uint64_t adesc = a0 + (uint64_t)((r * C0_ROWPITCH + kx * 64 + ks * 32) >> 4);
                            const uint64_t bdesc = b0 + (uint64_t)(((kx * 4 + 2 * ks) * C0_N * 16) >> 4);
                            ptx::umma_bf16_elected(tmem_d, adesc, bdesc, idesc, (kx | ks) ? 1u : 0u, elected);
                        }
                    ptx::umma_commit_elected(tfull_bar(slot), elected);
                    if (++slot == C0_SLOTS) { slot = 0; sphase ^= 1; }
                }
                ptx::umma_commit_elected(empty_bar(stage), elected);
                __syncwarp();
                if (++stage == C0_STAGES) { stage = 0; phase ^= 1; }
            }
        }
    } else {
        // ===================== epilogue: out[d][y] = sum_{kz,ky} P[d+kz-1][y+ky-1][(kz,ky)] =====================
        // Every (plane, input row) product is pulled out of TMEM as soon as it completes and its slot is released immediately.
        // Two groups of four warps: group g owns output rows 2g, 2g+1 of the unit (one warp per scheduler leaves every TMEM /
        // barrier latency exposed; the groups halve the work per warp).  Three accumulators per output row live in registers:
        // the output planes d'-1 (completed by plane d'), d' and d'+1.
        constexpr int RG = C0_R / 2;                // output rows per group
        const int grp = (warp - 2) >> 2;
        const int q = warp & 3;
        const int m = q * 32 + lane;
        const uint32_t lane_addr = tmem_base + ((uint32_t)(q * 32) << 16);
        float sc[8], sh[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) { sc[j] = p.scale[j]; sh[j] = p.shift[j]; }
        auto store_row = [&](const float* acc, int b, int d, int y, int x) {
            uint32_t o[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const float v0 = fmaxf(fmaf(acc[2 * j], sc[2 * j], sh[2 * j]), 0.f);
                const float v1 = fmaxf(fmaf(acc[2 * j + 1], sc[2 * j + 1], sh[2 * j + 1]), 0.f);
                if (p.f16)
                    o[j] = (uint32_t)__half_as_ushort(__float2half_rn(v0)) | ((uint32_t)__half_as_ushort(__float2half_rn(v1)) << 16);
                else
                    o[j] = (uint32_t)__bfloat16_as_ushort(__float2bfloat16_rn(v0)) |
                           ((uint32_t)__bfloat16_as_ushort(__float2bfloat16_rn(v1)) << 16);
            }
            if (p.out_s2d) {
                // only the 8 real channels, in the layout conv1 (stride 2) and conv11's skip connection read as stride-1 tensors
                const size_t vox = (((size_t)b * (D >> 1) + (d >> 1)) * (p.H >> 1) + (y >> 1)) * (p.W >> 1) + (x >> 1);
                *reinterpret_cast<uint4*>(p.out + vox * 64 + (((d & 1) * 4 + (y & 1) * 2 + (x & 1)) * 8)) = make_uint4(o[0], o[1], o[2], o[3]);
            } else {
                uint4* dst = reinterpret_cast<uint4*>(p.out + ((((size_t)b * D + d) * p.H + y) * p.W + x) * 16);
                dst[0] = make_uint4(o[0], o[1], o[2], o[3]);
                dst[1] = make_uint4(0, 0, 0, 0);
            }
        };
        uint32_t sphase = 0;          // slot == input row: one pass over the ring per plane
        for (int u = blockIdx.x; u < units; u += gridDim.x) {
            const int seg = u % segs, y0 = ((u / segs) % ygroups) * C0_R + grp * RG, b = u / (segs * ygroups);
            const int x = seg * C0_SEG + m;
            const bool valid = m < C0_SEG;
            float acc[3][RG][8];        // [0]: out[d'-1], [1]: out[d'], [2]: out[d'+1] while plane d' is being added
#pragma unroll
            for (int a = 0; a < 3; ++a)
#pragma unroll
                for (int r = 0; r < RG; ++r)
#pragma unroll
                    for (int j = 0; j < 8; ++j) acc[a][r][j] = 0.f;
            for (int d = 0; d < D; ++d, sphase ^= 1) {
#pragma unroll
                for (int rl = 0; rl < RG + 2; ++rl) {       // the group's input rows: unit rows grp * RG + rl  (= slot)
                    const int slot = grp * RG + rl;
                    ptx::mbar_wait(tfull_bar(slot), sphase, p.err, 14);
                    ptx::tc_fence_after();
                    // input row rl (group-local) feeds the group's output row rl - ky (ky = 0..2); the other column groups belong
                    // to the other group or to the units above / below and are not read
                    uint32_t rr[3][3][8];
#pragma unroll
                    for (int kz = 0; kz < 3; ++kz)
#pragma unroll
                        for (int ky = 0; ky < 3; ++ky)
                            if (rl - ky >= 0 && rl - ky < RG)
                                tmem_ld8(lane_addr + (uint32_t)(slot * C0_N + (kz * 3 + ky) * 8), rr[kz][ky]);
                    ptx::tmem_ld_wait();
                    ptx::tc_fence_before();
                    __syncwarp();
                    if (lane == 0) ptx::mbar_arrive(tempty_bar(slot));       // this warp is done with the slot
#pragma unroll
                    for (int kz = 0; kz < 3; ++kz)
#pragma unroll
                        for (int ky = 0; ky < 3; ++ky)
                            if (rl - ky >= 0 && rl - ky < RG) {
                                // plane d' contributes kz = 2 to out[d'-1], kz = 1 to out[d'], kz = 0 to out[d'+1]
#pragma unroll
                                for (int j = 0; j < 8; ++j) acc[2 - kz][rl - ky][j] += __uint_as_float(rr[kz][ky][j]);
                            }
                }
                // out[d-1] is complete; rotate the accumulators
#pragma unroll
                for (int r = 0; r < RG; ++r) {
                    if (d >= 1 && valid) store_row(acc[0][r], b, d - 1, y0 + r, x);
#pragma unroll
                    for (int j = 0; j < 8; ++j) { acc[0][r][j] = acc[1][r][j]; acc[1][r][j] = acc[2][r][j]; acc[2][r][j] = 0.f; }
                    if (d == D - 1 && valid) store_row(acc[0][r], b, d, y0 + r, x);
                }
            }
        }
    }
    ptx::tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        ptx::tc_fence_after();
        ptx::tmem_dealloc(tmem_base, 512);
    }
}

// ------------------------------------------------------------------------------------------------ host
struct Conv0Plan {
    CUtensorMap tmIn;
    Conv0Params p;
    int num_sms;
};

int tc_conv_init_driver();
extern PFN_cuTensorMapEncodeTiled_v12000 g_encode_shared;

Conv0Plan* conv0_alloc() { return new Conv0Plan(); }
void conv0_release(Conv0Plan* p) { delete p; }

int conv0_plan(Conv0Plan* pl, const Act& in, const uint16_t* w_packed, const float* scale, const float* shift, uint16_t* out,
               int flags, int num_sms) {
    const int planar = flags & 1;
    ADP_TRY(tc_conv_init_driver());
    ADP_CHECK_ARG(in.C == 32 && in.W % C0_SEG == 0 && in.D >= 2 && in.H % C0_R == 0,
                  "conv0 ring kernel: C = 32, W % 112 == 0, D >= 2, H % 4 == 0");
    // plane D-1 of an odd D would land at s2d depth (D-1)/2, one past the end of a [B, D/2, ...] output
    ADP_CHECK_ARG(!(flags & 2) || in.D % 2 == 0, "conv0 ring kernel: the space-to-depth(2) output layout needs an even D");
    cuuint64_t dims[5] = {(cuuint64_t)in.C, (cuuint64_t)in.W, (cuuint64_t)in.H, (cuuint64_t)in.D, (cuuint64_t)in.B};
    cuuint64_t strides[4] = {(cuuint64_t)in.C * 2, (cuuint64_t)in.W * in.C * 2, (cuuint64_t)in.H * in.W * in.C * 2,
                             (cuuint64_t)in.D * in.H * in.W * in.C * 2};
    cuuint32_t box[5] = {32, (cuuint32_t)C0_PIXPITCH, (cuuint32_t)(C0_R + 2), 1, 1};
    cuuint32_t estr[5] = {1, 1, 1, 1, 1};
    ADP_CHECK_ARG(!planar, "the depth-ring kernel reads the channels-last volume");
    const int rank = 5;
    CUresult r = g_encode_shared(&pl->tmIn, in.f16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, rank, in.hi, dims,
                                 strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B,
                                 CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_last_error("cuTensorMapEncodeTiled(conv0 volume) failed: %d", (int)r);
        return ADP_ERR_CUDA;
    }
    pl->p.B = in.B; pl->p.D = in.D; pl->p.H = in.H; pl->p.W = in.W; pl->p.f16 = in.f16;
    pl->p.w = w_packed; pl->p.scale = scale; pl->p.shift = shift; pl->p.out = out; pl->p.err = nullptr; pl->p.out_s2d = (flags >> 1) & 1;
    pl->num_sms = num_sms > 0 ? num_sms : 148;
    return ADP_OK;
}

int conv0_run(Conv0Plan* pl, int batch, int* err_flag, cudaStream_t stream) {
    ADP_CHECK_ARG(batch <= pl->p.B, "batch exceeds planned capacity");
    static int attr[kMaxDevices];
    ADP_TRY(ensure_dyn_smem(conv0_ring_kernel, C0_SMEM, attr));
    pl->p.err = err_flag;
    const int units = batch * (pl->p.H / C0_R) * (pl->p.W / C0_SEG);
    if (units == 0) return ADP_OK;
    const int slots = pl->num_sms;
    const int grid = units < slots ? units : slots;
    conv0_ring_kernel<<<grid, C0_THREADS, C0_SMEM, stream>>>(pl->tmIn, pl->p, batch);
    ADP_CUDA(cudaGetLastError());
    return ADP_OK;
}

}  // namespace adp
