// tcgen05 implicit-GEMM convolution -- see tc_conv.cuh for the scheme.
#include "tc_conv.cuh"
#include "ptx.cuh"

#include <cudaTypedefs.h>
#include <stdlib.h>

namespace adp {

// ------------------------------------------------------------------------------------------------
// descriptors
// ------------------------------------------------------------------------------------------------
// Shared-memory matrix descriptor, K-major operand whose rows are KC*2 bytes (= the swizzle span).
//   [0,14) start >> 4 | [16,30) LBO >> 4 (unused for swizzled K-major) | [32,46) SBO >> 4 (8-row group pitch)
//   [46,48) version = 1 (sm_100) | [49,52) base offset = 0 (tiles are 1024B aligned) | [61,64) layout type
template <int KC>
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t smem_addr) {
    constexpr uint64_t layout = (KC == 64) ? 2ull : (KC == 32) ? 4ull : 6ull;   // SWIZZLE_128B / 64B / 32B
    constexpr uint64_t sbo = (uint64_t)(8 * KC * 2) >> 4;
    return (uint64_t)((smem_addr & 0x3FFFF) >> 4) | (1ull << 16) | (sbo << 32) | (1ull << 46) | (layout << 61);
}
// Instruction descriptor for kind::f16: D = fp32, A = B = bf16, both K-major, M = 128, N = BN.
template <int BN>
__device__ __forceinline__ uint32_t make_idesc(int f16) {
    const uint32_t fmt = f16 ? 0u : 1u;   // F16 = 0, BF16 = 1
    return (1u << 4) | (fmt << 7) | (fmt << 10) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
}

// ------------------------------------------------------------------------------------------------
// kernel
// ------------------------------------------------------------------------------------------------
// Epilogue of one accumulator chunk: r[0..CH) fp32 accumulators of output pixel `pix`, channels [nbase, nbase + CH)
// FULL: the chunk is known to hold CH valid channels with 16-byte aligned per-channel vectors (the coalesced-store mode):
// scale / bias arrive as 128-bit broadcast loads and the per-element `j < nvalid` predicates disappear.  The epilogue of the
// small-K layers is instruction bound (ncu: the MMA warp waits on tmem_empty), so the issue slots matter.
template <int CH, bool FULL = false>
__device__ __forceinline__ void tc_epilogue_math(const TcConvParams& p, const uint32_t* r, size_t pix, int nbase, int b, float* v,
                                                 const float* res_pre = nullptr) {
                            const int nvalid = FULL ? CH : min(CH, p.Cout - nbase);
                            const size_t ro = pix * p.res_cs + nbase;
#pragma unroll
                            for (int j = 0; j < CH; ++j) v[j] = __uint_as_float(r[j]);
                            if (FULL) {
                                const float4* s4 = reinterpret_cast<const float4*>(p.scale + nbase);
                                const float4* b4 = reinterpret_cast<const float4*>(p.bias + (p.bias_per_batch ? (size_t)b * p.Cout : 0) + nbase);
                                if (p.scale && p.bias) {          // folded BatchNorm: one FFMA per channel
#pragma unroll
                                    for (int j = 0; j < CH; j += 4) {
                                        const float4 q = __ldg(s4 + (j >> 2)), t = __ldg(b4 + (j >> 2));
                                        v[j] = fmaf(v[j], q.x, t.x); v[j + 1] = fmaf(v[j + 1], q.y, t.y);
                                        v[j + 2] = fmaf(v[j + 2], q.z, t.z); v[j + 3] = fmaf(v[j + 3], q.w, t.w);
                                    }
                                } else if (p.scale) {
#pragma unroll
                                    for (int j = 0; j < CH; j += 4) {
                                        const float4 q = __ldg(s4 + (j >> 2));
                                        v[j] *= q.x; v[j + 1] *= q.y; v[j + 2] *= q.z; v[j + 3] *= q.w;
                                    }
                                } else if (p.bias) {
#pragma unroll
                                    for (int j = 0; j < CH; j += 4) {
                                        const float4 q = __ldg(b4 + (j >> 2));
                                        v[j] += q.x; v[j + 1] += q.y; v[j + 2] += q.z; v[j + 3] += q.w;
                                    }
                                }
                            } else {
                            if (p.scale) {
#pragma unroll
                                for (int j = 0; j < CH; ++j) if (j < nvalid) v[j] *= __ldg(p.scale + nbase + j);
                            }
                            if (p.bias) {
                                const float* bias = p.bias + (p.bias_per_batch ? (size_t)b * p.Cout : 0);
#pragma unroll
                                for (int j = 0; j < CH; ++j) if (j < nvalid) v[j] += __ldg(bias + nbase + j);
                            }
                            }
                            const bool vec_ok = ((p.Cout | p.res_cs | p.out_cs | p.out_coff) & 7) == 0;   // 128-bit accesses stay aligned
                            if (res_pre && !p.res_after_act) {
#pragma unroll
                                for (int j = 0; j < CH; ++j) v[j] += res_pre[j];
                            } else if (p.res_hi && !p.res_after_act) {
#pragma unroll
                                for (int j0 = 0; j0 < CH; j0 += 8) {
                                    if (vec_ok && j0 + 8 <= nvalid) {
                                        ld8_16(p.res_hi, ro + j0, p.f16, v + j0, true);
                                        if (p.res_lo && !p.f16) ld8_16(p.res_lo, ro + j0, 0, v + j0, true);
                                    } else {
#pragma unroll
                                        for (int j = j0; j < j0 + 8; ++j) if (j < nvalid) v[j] += ld_act16(p.res_hi, p.res_lo, ro + j, p.f16);
                                    }
                                }
                            }
                            if (p.act == 1) {
#pragma unroll
                                for (int j = 0; j < CH; ++j) v[j] = max_nan(v[j], 0.f);
                            } else if (p.act == 2) {
#pragma unroll
                                for (int j = 0; j < CH; ++j) v[j] = v[j] > 0.f ? v[j] : v[j] * p.prelu;
                            } else if (p.act == 3) {
#pragma unroll
                                for (int j = 0; j < CH; ++j) v[j] = tanhf(v[j]);
                            }
                            if (res_pre && p.res_after_act) {
#pragma unroll
                                for (int j = 0; j < CH; ++j) v[j] += res_pre[j];
                            } else if (p.res_hi && p.res_after_act) {
#pragma unroll
                                for (int j0 = 0; j0 < CH; j0 += 8) {
                                    if (vec_ok && j0 + 8 <= nvalid) {
                                        ld8_16(p.res_hi, ro + j0, p.f16, v + j0, true);
                                        if (p.res_lo && !p.f16) ld8_16(p.res_lo, ro + j0, 0, v + j0, true);
                                    } else {
#pragma unroll
                                        for (int j = j0; j < j0 + 8; ++j) if (j < nvalid) v[j] += ld_act16(p.res_hi, p.res_lo, ro + j, p.f16);
                                    }
                                }
                            }
                            if (p.check_finite) {
                                // range guard of the fp16 pipeline: an activation that left the half range upstream arrives here as
                                // inf / NaN (the last backbone layer sees every earlier one); the host reads err[1] after every call
                                bool bad = false;
#pragma unroll
                                for (int j = 0; j < CH; ++j) bad |= !(fabsf(v[j]) <= 3.0e38f);
                                if (bad && p.err) atomicOr(p.err + 1, 1);
                            }
}

// per-lane stores of one chunk (every lane writes its own pixel row): partial chunks, split hi + lo planes
template <int CH>
__device__ __forceinline__ void tc_epilogue_store_lane(const TcConvParams& p, const float* v, size_t pix, int nbase) {
                            const int nvalid = min(CH, p.Cout - nbase);
                            const size_t o = pix * p.Cout + nbase;
                            const size_t oh = pix * p.out_cs + p.out_coff + nbase;   // out_hi / out_lo may be a column range of a wider tensor
                            const bool vec_ok = ((p.Cout | p.res_cs | p.out_cs | p.out_coff) & 7) == 0;   // 128-bit accesses stay aligned
                            if (p.out_f32) {
                                if (nvalid == CH && (p.Cout & 3) == 0) {
#pragma unroll
                                    for (int j = 0; j < CH; j += 4)
                                        *reinterpret_cast<float4*>(p.out_f32 + o + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
                                } else {
#pragma unroll
                                    for (int j = 0; j < CH; ++j) if (j < nvalid) p.out_f32[o + j] = v[j];
                                }
                            }
                            if (p.out_h16) {
#pragma unroll
                                for (int j0 = 0; j0 < CH; j0 += 8) {
                                    if (vec_ok && j0 + 8 <= nvalid) st8_16(reinterpret_cast<bf16*>(p.out_h16), nullptr, o + j0, 1, v + j0);
                                    else {
#pragma unroll
                                        for (int j = j0; j < j0 + 8; ++j) if (j < nvalid) p.out_h16[o + j] = __float2half_rn(v[j]);
                                    }
                                }
                            }
                            if (p.out_hi) {
#pragma unroll
                                for (int j0 = 0; j0 < CH; j0 += 8) {
                                    if (vec_ok && j0 + 8 <= nvalid) {
                                        st8_16(p.out_hi, p.out_lo, oh + j0, p.f16, v + j0);
                                    } else {
#pragma unroll
                                        for (int j = j0; j < j0 + 8; ++j) if (j < nvalid) st_act16(p.out_hi, p.out_lo, oh + j, v[j], p.f16);
                                    }
                                }
                            }
}

// Warp-cooperative stores of one chunk.  A lane owns one pixel row, so per-lane 128-bit stores make every instruction touch
// 32 separate lines (2.2-3.7 TB/s measured, tools/micro/store_pattern.cu); here the rows go through a 2 KB per-warp transpose
// buffer (XOR-swizzled: conflict free both ways) and every store instruction writes whole 64-byte row pieces of 8 (16) rows.
// NP = 16-byte pieces per row in this call (4: 32 x 16-bit or 16 x fp32; 2: 16 x 16-bit).
template <int NP>
__device__ __forceinline__ void tc_store_rows(uint4* wbuf, int lane, const uint4* pieces, size_t pix, unsigned int validmask,
                                              uint8_t* base, size_t row_pitch_bytes, size_t col_off_bytes) {
    constexpr int SH = NP == 4 ? 1 : 2;            // swizzle source bits: lane >> SH
#pragma unroll
    for (int j = 0; j < NP; ++j) wbuf[lane * NP + (j ^ ((lane >> SH) & (NP - 1)))] = pieces[j];
    __syncwarp();
    constexpr int RPI = 32 / NP;                   // rows per store instruction
#pragma unroll
    for (int k = 0; k < NP; ++k) {
        const int row = RPI * k + lane / NP, piece = lane % NP;
        const uint4 val = wbuf[row * NP + (piece ^ ((row >> SH) & (NP - 1)))];
        const unsigned long long rp = __shfl_sync(0xffffffffu, (unsigned long long)pix, row);
        if ((validmask >> row) & 1u) *reinterpret_cast<uint4*>(base + (size_t)rp * row_pitch_bytes + col_off_bytes + piece * 16) = val;
    }
    __syncwarp();
}

// reverse direction: every load instruction reads whole row pieces of 8 (16) rows, each lane ends up with its own row.
// Two phases, so that the global loads can be issued early (before the accumulator is ready) and their latency overlaps
// the wait: issue = coalesced loads into registers, finish = transpose through the warp buffer.
template <int NP>
__device__ __forceinline__ void tc_load_rows_issue(int lane, uint4* regs, size_t pix, unsigned int validmask, const uint8_t* base,
                                                   size_t row_pitch_bytes, size_t col_off_bytes) {
    constexpr int RPI = 32 / NP;
#pragma unroll
    for (int k = 0; k < NP; ++k) {
        const int row = RPI * k + lane / NP, piece = lane % NP;
        const unsigned long long rp = __shfl_sync(0xffffffffu, (unsigned long long)pix, row);
        regs[k] = make_uint4(0, 0, 0, 0);
        if ((validmask >> row) & 1u) regs[k] = *reinterpret_cast<const uint4*>(base + (size_t)rp * row_pitch_bytes + col_off_bytes + piece * 16);
    }
}
template <int NP>
__device__ __forceinline__ void tc_load_rows_finish(uint4* wbuf, int lane, const uint4* regs, uint4* pieces) {
    constexpr int SH = NP == 4 ? 1 : 2;
    constexpr int RPI = 32 / NP;
#pragma unroll
    for (int k = 0; k < NP; ++k) {
        const int row = RPI * k + lane / NP, piece = lane % NP;
        wbuf[row * NP + (piece ^ ((row >> SH) & (NP - 1)))] = regs[k];
    }
    __syncwarp();
#pragma unroll
    for (int j = 0; j < NP; ++j) pieces[j] = wbuf[lane * NP + (j ^ ((lane >> SH) & (NP - 1)))];
    __syncwarp();
}

__device__ __forceinline__ void tc_unpack8(const uint4& u, int f16, float* v) {
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

// residual of one chunk for every lane's own row, fetched with coalesced row-piece loads
template <int CH>
__device__ __forceinline__ void tc_epilogue_res_issue(const TcConvParams& p, uint4* regs, size_t pix, int nbase, unsigned int validmask, int lane) {
    tc_load_rows_issue<CH / 8>(lane, regs, pix, validmask, reinterpret_cast<const uint8_t*>(p.res_hi), (size_t)p.res_cs * 2, (size_t)nbase * 2);
}
template <int CH>
__device__ __forceinline__ void tc_epilogue_res_finish(const TcConvParams& p, const uint4* regs, float* res, uint4* wbuf, int lane) {
    constexpr int NP16 = CH / 8;
    uint4 pc[NP16];
    tc_load_rows_finish<NP16>(wbuf, lane, regs, pc);
#pragma unroll
    for (int j = 0; j < NP16; ++j) tc_unpack8(pc[j], p.f16, res + 8 * j);
}

__device__ __forceinline__ uint4 tc_pack8(const float* v, int f16) {
    uint32_t w[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        if (f16) {
            const __half2 h = __floats2half2_rn(v[2 * q], v[2 * q + 1]);
            w[q] = *reinterpret_cast<const uint32_t*>(&h);
        } else {
            const __nv_bfloat162 h = __floats2bfloat162_rn(v[2 * q], v[2 * q + 1]);
            w[q] = *reinterpret_cast<const uint32_t*>(&h);
        }
    }
    return make_uint4(w[0], w[1], w[2], w[3]);
}

template <int CH>
__device__ __forceinline__ void tc_epilogue_store_warp(const TcConvParams& p, const float* v, size_t pix, int nbase, unsigned int validmask,
                                                       uint4* wbuf, int lane) {
    constexpr int NP16 = CH / 8;
    if (p.out_f32) {
#pragma unroll
        for (int h = 0; h < CH / 16; ++h) {
            uint4 pc[4];
#pragma unroll
            for (int j = 0; j < 4; ++j)
                pc[j] = make_uint4(__float_as_uint(v[16 * h + 4 * j]), __float_as_uint(v[16 * h + 4 * j + 1]),
                                   __float_as_uint(v[16 * h + 4 * j + 2]), __float_as_uint(v[16 * h + 4 * j + 3]));
            tc_store_rows<4>(wbuf, lane, pc, pix, validmask, reinterpret_cast<uint8_t*>(p.out_f32), (size_t)p.Cout * 4,
                             (size_t)(nbase + 16 * h) * 4);
        }
    }
    if (p.out_h16) {
        uint4 pc[NP16];
#pragma unroll
        for (int j = 0; j < NP16; ++j) pc[j] = tc_pack8(v + 8 * j, 1);
        tc_store_rows<NP16>(wbuf, lane, pc, pix, validmask, reinterpret_cast<uint8_t*>(p.out_h16), (size_t)p.Cout * 2, (size_t)nbase * 2);
    }
    if (p.out_hi) {
        uint4 pc[NP16];
#pragma unroll
        for (int j = 0; j < NP16; ++j) pc[j] = tc_pack8(v + 8 * j, p.f16);
        tc_store_rows<NP16>(wbuf, lane, pc, pix, validmask, reinterpret_cast<uint8_t*>(p.out_hi), (size_t)p.out_cs * 2,
                            (size_t)(p.out_coff + nbase) * 2);
        if (p.out_lo && !p.f16) {     // bf16 split precision: lo = bf16(v - hi), the same pitch and offset (the per-point MLPs)
#pragma unroll
            for (int j = 0; j < NP16; ++j) {
                const uint32_t hw[4] = {pc[j].x, pc[j].y, pc[j].z, pc[j].w};
                float l[8];
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    l[2 * q] = v[8 * j + 2 * q] - __uint_as_float(hw[q] << 16);
                    l[2 * q + 1] = v[8 * j + 2 * q + 1] - __uint_as_float(hw[q] & 0xffff0000u);
                }
                pc[j] = tc_pack8(l, 0);
            }
            tc_store_rows<NP16>(wbuf, lane, pc, pix, validmask, reinterpret_cast<uint8_t*>(p.out_lo), (size_t)p.out_cs * 2,
                                (size_t)(p.out_coff + nbase) * 2);
        }
    }
    if (CH == 32 && p.out_q8) {       // fp8 twin (value / 2, e4m3) for the low-order pass of the consuming layer: 32 bytes per row
        uint4 pc[2];
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            const uint2 a = pack8_q8(v + 16 * j), b = pack8_q8(v + 16 * j + 8);
            pc[j] = make_uint4(a.x, a.y, b.x, b.y);
        }
        tc_store_rows<2>(wbuf, lane, pc, pix, validmask, p.out_q8, (size_t)p.out_cs, (size_t)(p.out_coff + nbase));
    }
}

constexpr int kTcThreads = 192;   // warp 0: TMA producer, warp 1: MMA issuer + TMEM owner, warps 2-5: epilogue

// FUSED = 1: split-precision bf16x3 layers keep A_hi, A_lo, W_hi, W_lo of one (tap, K chunk) in the same stage and issue the
// three MMA groups (hi*hi, lo*hi, hi*lo) from it: 2x the bytes of a single pass instead of 3x.
// FUSED = 2: "fp16x2" -- one fp16 activation plane against fp16 hi + lo weights: stage = [A | W_hi | W_lo], two MMA groups.
// FUSED = 3: "fp16 + fp8 lo" (npass 4) -- the low-order term A W_lo only needs ~4 significant bits (W_lo <= 2^-12 |W|), so it runs
//            as an e4m3 x e4m3 MMA at twice the fp16 rate: first a sweep over K with [A8 | W8] stages (A8 = e4m3(A / 2), the
//            producer's fp8 twin; W8 = e4m3(W_lo 2^16); 128 channels per stage, K = 32 per MMA), then the fp16 sweep with
//            [A | W_hi] stages whose first MMA scales the accumulator by 2^-15 (scale-input-d).  1.5 MMA passes per
//            algorithmic FLOP instead of 2, same stage size (48 KB at BN = 256: 4 stages instead of 2).
template <int BN, int KC, int FUSED = 0>
struct TcCfg {
    static constexpr int A_BYTES = 128 * KC * 2;
    static constexpr int B_BYTES = BN * KC * 2;
    static constexpr int B_PAD = (B_BYTES + 1023) / 1024 * 1024;
    static_assert(FUSED != 3 || KC == 64, "the fp8 low-order sweep moves 128 one-byte channels per stage = the bytes of 64 fp16 channels");
    static constexpr int STAGE_BYTES = FUSED == 1 ? 2 * (A_BYTES + B_PAD) : FUSED == 2 ? (A_BYTES + 2 * B_PAD) : (A_BYTES + B_PAD);
    // small-N layers are latency bound per tile: fewer stages -> several CTAs per SM overlap their pipelines
    static constexpr int CTAS_PER_SM = FUSED ? ((BN <= 64 && FUSED != 3) ? 2 : 1) : (BN <= 16 && KC <= 32) ? 5 : BN <= 32 ? 3 : (BN <= 64 ? 2 : 1);
    static constexpr int EPI_BYTES = 4 * 2048;                  // per-epilogue-warp transpose buffers (coalesced stores)
    static constexpr int SMEM_BUDGET = (220 * 1024 - CTAS_PER_SM * (EPI_BYTES + 2048)) / CTAS_PER_SM;
    static constexpr int STAGES = (STAGE_BYTES * 6 <= SMEM_BUDGET) ? 6 : (SMEM_BUDGET / STAGE_BYTES);
    static constexpr int ACC_STRIDE = BN < 32 ? 32 : BN;   // TMEM columns per accumulator stage
    static constexpr int TMEM_COLS = (2 * ACC_STRIDE <= 64) ? 64 : (2 * ACC_STRIDE <= 128) ? 128 : (2 * ACC_STRIDE <= 256) ? 256 : 512;
    static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + EPI_BYTES + 1024 /*align slack*/ + 256 /*barriers*/;
};

template <int BN, int KC, int FUSED>
__global__ void __launch_bounds__(kTcThreads, TcCfg<BN, KC, FUSED>::CTAS_PER_SM)
tc_conv_kernel(const __grid_constant__ CUtensorMap tmA_hi, const __grid_constant__ CUtensorMap tmA_lo,
               const __grid_constant__ CUtensorMap tmW_hi, const __grid_constant__ CUtensorMap tmW_lo,
               const TcConvParams p, int batch) {
    using Cfg = TcCfg<BN, KC, FUSED>;
    constexpr int STAGES = Cfg::STAGES;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint4* epi_buf = reinterpret_cast<uint4*>(smem + STAGES * Cfg::STAGE_BYTES);
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + STAGES * Cfg::STAGE_BYTES + Cfg::EPI_BYTES);
    // bars[0..S) full, [S..2S) empty, [2S..2S+2) tmem_full, [2S+2..2S+4) tmem_empty, then the TMEM base address
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * STAGES + 4);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const uint32_t smem_base = ptx::smem_u32(smem);
    const uint32_t bar_base = ptx::smem_u32(bars);
    auto full_bar = [&](int s) { return bar_base + 8u * s; };
    auto empty_bar = [&](int s) { return bar_base + 8u * (STAGES + s); };
    auto tfull_bar = [&](int s) { return bar_base + 8u * (2 * STAGES + s); };
    auto tempty_bar = [&](int s) { return bar_base + 8u * (2 * STAGES + 2 + s); };

    if (warp == 0 && lane == 0) {
        ptx::prefetch_tmap(&tmA_hi);
        ptx::prefetch_tmap(&tmW_hi);
        if (p.npass > 1) {
            ptx::prefetch_tmap(&tmA_lo);
            ptx::prefetch_tmap(&tmW_lo);
        }
        for (int s = 0; s < STAGES; ++s) {
            ptx::mbar_init(full_bar(s), 1);
            ptx::mbar_init(empty_bar(s), 1);
        }
        for (int s = 0; s < 2; ++s) {
            ptx::mbar_init(tfull_bar(s), 1);
            ptx::mbar_init(tempty_bar(s), 4);   // one arrive per epilogue warp
        }
        ptx::fence_barrier_init();
    }
    if (warp == 1) {
        ptx::tmem_alloc(ptx::smem_u32(tmem_slot), Cfg::TMEM_COLS);
        ptx::tmem_relinquish();
    }
    ptx::tc_fence_before();
    __syncthreads();
    ptx::tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    const int taps = p.ntaps;
    const int npass_loop = FUSED ? 1 : p.npass;
    const int lo_iters = FUSED == 3 ? taps * (p.kchunks >> 1) : 0;      // fp8 sweep: 128 channels per stage
    const int k_iters = npass_loop * taps * p.kchunks + lo_iters;
    const int tiles_per_img = p.D * p.tiles_y * p.tiles_x * p.tiles_n;
    const int total_tiles = batch * tiles_per_img;
    const int rows_valid = p.TW * p.TH;

    if (warp == 0) {
        // ===================== TMA producer =====================
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            const uint32_t tx_bytes = (uint32_t)(FUSED == 1 ? 2 * (rows_valid * KC * 2 + Cfg::B_BYTES)
                                                 : FUSED == 2 ? (rows_valid * KC * 2 + 2 * Cfg::B_BYTES) : (rows_valid * KC * 2 + Cfg::B_BYTES));
            for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
                int t = tile;
                const int nt = t % p.tiles_n; t /= p.tiles_n;
                const int tx = t % p.tiles_x; t /= p.tiles_x;
                const int ty = t % p.tiles_y; t /= p.tiles_y;
                const int d = t % p.D;
                const int b = t / p.D;
                const int x0 = tx * p.TW, y0 = ty * p.TH, n0 = nt * BN;
                if (FUSED == 3) {      // low-order sweep first: [A8 | W8] stages from the fp8 twins (maps tmA_lo / tmW_lo)
                    for (int tap = 0; tap < taps; ++tap) {
                        const int cx = x0 * p.in_mul + p.tdx[tap], cy = y0 * p.in_mul + p.tdy[tap];
                        const int cz = d * p.in_mul + p.tdz[tap], wt = p.twt[tap];
                        for (int kc = 0; kc < (p.kchunks >> 1); ++kc) {
                            ptx::mbar_wait(empty_bar(stage), phase ^ 1, p.err, 1);
                            const uint32_t sa = smem_base + stage * Cfg::STAGE_BYTES;
                            ptx::mbar_arrive_expect_tx(full_bar(stage), tx_bytes);
                            ptx::tma_load_5d(&tmA_lo, full_bar(stage), sa, kc * 128, cx, cy, cz, b);
                            ptx::tma_load_3d(&tmW_lo, full_bar(stage), sa + Cfg::A_BYTES, kc * 128, n0, wt);
                            if (++stage == STAGES) { stage = 0; phase ^= 1; }
                        }
                    }
                }
                for (int pass = 0; pass < npass_loop; ++pass) {
                    // npass 3: (A_hi W_hi, A_lo W_hi, A_hi W_lo); npass 2: (A W_hi, A W_lo)
                    const CUtensorMap* mapA = (p.npass == 3 && pass == 1) ? &tmA_lo : &tmA_hi;
                    const CUtensorMap* mapW = (pass > 0 && pass == p.npass - 1) ? &tmW_lo : &tmW_hi;
                    for (int tap = 0; tap < taps; ++tap) {
                        const int cx = x0 * p.in_mul + p.tdx[tap], cy = y0 * p.in_mul + p.tdy[tap];
                        const int cz = d * p.in_mul + p.tdz[tap], wt = p.twt[tap];
                        for (int kc = 0; kc < p.kchunks; ++kc) {
                            ptx::mbar_wait(empty_bar(stage), phase ^ 1, p.err, 1);
                            const uint32_t sa = smem_base + stage * Cfg::STAGE_BYTES;
                            ptx::mbar_arrive_expect_tx(full_bar(stage), tx_bytes);
                            if (FUSED == 2) {   // [A | W_hi | W_lo]
                                ptx::tma_load_5d(&tmA_hi, full_bar(stage), sa, kc * KC, cx, cy, cz, b);
                                ptx::tma_load_3d(&tmW_hi, full_bar(stage), sa + Cfg::A_BYTES, kc * KC, n0, wt);
                                ptx::tma_load_3d(&tmW_lo, full_bar(stage), sa + Cfg::A_BYTES + Cfg::B_PAD, kc * KC, n0, wt);
                            } else if (FUSED == 1) {   // [A_hi | A_lo | W_hi | W_lo]
                                ptx::tma_load_5d(&tmA_hi, full_bar(stage), sa, kc * KC, cx, cy, cz, b);
                                ptx::tma_load_5d(&tmA_lo, full_bar(stage), sa + Cfg::A_BYTES, kc * KC, cx, cy, cz, b);
                                ptx::tma_load_3d(&tmW_hi, full_bar(stage), sa + 2 * Cfg::A_BYTES, kc * KC, n0, wt);
                                ptx::tma_load_3d(&tmW_lo, full_bar(stage), sa + 2 * Cfg::A_BYTES + Cfg::B_PAD, kc * KC, n0, wt);
                            } else {
                                ptx::tma_load_5d(mapA, full_bar(stage), sa, kc * KC, cx, cy, cz, b);
                                ptx::tma_load_3d(mapW, full_bar(stage), sa + Cfg::A_BYTES, kc * KC, n0, wt);
                            }
                            if (++stage == STAGES) { stage = 0; phase ^= 1; }
                        }
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ===================== MMA issuer =====================
        // warp-convergent: all lanes carry the same (uniform) descriptors and only the elected lane's tcgen05 instructions take
        // effect -- see ptx::umma_bf16_elected for why this is not written as `if (lane == 0)`
        int stage = 0;
        uint32_t phase = 0;
        int as = 0;
        uint32_t aphase = 0;
        const uint32_t idesc = make_idesc<BN>(p.f16);
        const uint32_t elected = ptx::elect_one();
        const uint32_t tbase = __shfl_sync(0xffffffffu, tmem_base, 0);
        for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
            ptx::mbar_wait(tempty_bar(as), aphase ^ 1, p.err, 2);
            ptx::tc_fence_after();
            const uint32_t tmem_d = tbase + (uint32_t)(as * Cfg::ACC_STRIDE);
            for (int it = 0; it < k_iters; ++it) {
                ptx::mbar_wait(full_bar(stage), phase, p.err, 3);
                ptx::tc_fence_after();
                const uint32_t sa = smem_base + stage * Cfg::STAGE_BYTES;
                if (FUSED == 2) {
                    const uint64_t ah = make_smem_desc<KC>(sa);
                    const uint64_t wh = make_smem_desc<KC>(sa + Cfg::A_BYTES);
                    const uint64_t wl = make_smem_desc<KC>(sa + Cfg::A_BYTES + Cfg::B_PAD);
#pragma unroll
                    for (int k = 0; k < KC / 16; ++k) {
                        // advance 16 elements = 32 bytes along K inside the swizzled row: +2 in the >>4 address field
                        ptx::umma_bf16_elected(tmem_d, ah + (uint64_t)(2 * k), wh + (uint64_t)(2 * k), idesc, (it > 0 || k > 0) ? 1u : 0u, elected);
                        ptx::umma_bf16_elected(tmem_d, ah + (uint64_t)(2 * k), wl + (uint64_t)(2 * k), idesc, 1u, elected);
                    }
                } else if (FUSED == 1) {
                    const uint64_t ah = make_smem_desc<KC>(sa), al = make_smem_desc<KC>(sa + Cfg::A_BYTES);
                    const uint64_t wh = make_smem_desc<KC>(sa + 2 * Cfg::A_BYTES);
                    const uint64_t wl = make_smem_desc<KC>(sa + 2 * Cfg::A_BYTES + Cfg::B_PAD);
#pragma unroll
                    for (int k = 0; k < KC / 16; ++k) {
                        ptx::umma_bf16_elected(tmem_d, ah + (uint64_t)(2 * k), wh + (uint64_t)(2 * k), idesc, (it > 0 || k > 0) ? 1u : 0u, elected);
                        ptx::umma_bf16_elected(tmem_d, al + (uint64_t)(2 * k), wh + (uint64_t)(2 * k), idesc, 1u, elected);
                        ptx::umma_bf16_elected(tmem_d, ah + (uint64_t)(2 * k), wl + (uint64_t)(2 * k), idesc, 1u, elected);
                    }
                } else if (FUSED == 3) {
                    const uint64_t adesc = make_smem_desc<KC>(sa);
                    const uint64_t bdesc = make_smem_desc<KC>(sa + Cfg::A_BYTES);
                    if (it < lo_iters) {            // e4m3 x e4m3, K = 32 (32 bytes of each 128-byte row) per MMA
#pragma unroll
                        for (int k = 0; k < 4; ++k)
                            ptx::umma_f8_elected(tmem_d, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idesc, (it > 0 || k > 0) ? 1u : 0u, elected);
                    } else if (it == lo_iters) {    // first fp16 step: the accumulator holds 2^15 x (A W_lo) -> scale it down while adding
                        ptx::umma_f16_scale15_elected(tmem_d, adesc, bdesc, idesc, elected);
#pragma unroll
                        for (int k = 1; k < 4; ++k)
                            ptx::umma_bf16_elected(tmem_d, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idesc, 1u, elected);
                    } else {
#pragma unroll
                        for (int k = 0; k < 4; ++k)
                            ptx::umma_bf16_elected(tmem_d, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idesc, 1u, elected);
                    }
                } else {
                    const uint64_t adesc = make_smem_desc<KC>(sa);
                    const uint64_t bdesc = make_smem_desc<KC>(sa + Cfg::A_BYTES);
#pragma unroll
                    for (int k = 0; k < KC / 16; ++k)
                        ptx::umma_bf16_elected(tmem_d, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idesc, (it > 0 || k > 0) ? 1u : 0u, elected);
                }
                ptx::umma_commit_elected(empty_bar(stage), elected);          // frees the smem slot when these MMAs retire
                if (it == k_iters - 1) ptx::umma_commit_elected(tfull_bar(as), elected);   // accumulator complete
                __syncwarp();
                if (++stage == STAGES) { stage = 0; phase ^= 1; }
            }
            if (++as == 2) { as = 0; aphase ^= 1; }
        }
    } else {
        // ===================== epilogue (4 warps, TMEM lane quarter = warp % 4) =====================
        const int q = warp & 3;
        const int m = q * 32 + lane;
        const int ty_l = m / p.TW, tx_l = m - ty_l * p.TW;
        int as = 0;
        uint32_t aphase = 0;
        constexpr int CH = (BN < 32) ? BN : 32;
        constexpr bool RES_PREFETCH = BN <= 64;          // residual of the whole tile fits in registers (<= 8 x 16 B per lane)
        const bool res_co = p.coalesce && p.res_hi && !p.res_lo && (p.res_cs & 7) == 0;
        uint4* wbuf = epi_buf + q * 128;
        for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
            int t = tile;
            const int nt = t % p.tiles_n; t /= p.tiles_n;
            const int tx = t % p.tiles_x; t /= p.tiles_x;
            const int ty = t % p.tiles_y; t /= p.tiles_y;
            const int d = t % p.D;
            const int b = t / p.D;
            const int x = tx * p.TW + tx_l, y = ty * p.TH + ty_l, n0 = nt * BN;
            const bool valid = (m < rows_valid) && (x < p.W) && (y < p.H);
            const size_t pix = (((size_t)b * p.oD + (d * p.out_mul + p.out_oz)) * p.oH + (y * p.out_mul + p.out_oy)) * p.oW +
                               (x * p.out_mul + p.out_ox);
            const unsigned int vmask = __ballot_sync(0xffffffffu, valid);
            uint4 res_regs[RES_PREFETCH ? BN / CH : 1][CH / 8];
            if (RES_PREFETCH && res_co) {      // residual loads in flight while the accumulator is still being produced
#pragma unroll
                for (int c = 0; c < BN / CH; ++c)
                    if (n0 + c * CH < p.Cout) tc_epilogue_res_issue<CH>(p, res_regs[c], pix, n0 + c * CH, vmask, lane);
            }
            ptx::mbar_wait(tfull_bar(as), aphase, p.err, 4);
            ptx::tc_fence_after();
#pragma unroll
            for (int c0 = 0; c0 < BN; c0 += CH) {
                uint32_t r[32];
                const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(as * Cfg::ACC_STRIDE + c0);
                ptx::tmem_ld16(taddr, r);
                if (CH == 32) ptx::tmem_ld16(taddr + 16, r + 16);
                ptx::tmem_ld_wait();
                const int nbase = n0 + c0;
                if (nbase < p.Cout) {       // Cout may be padded up to BN (e.g. 8 -> 16); uniform over the warp
                    float v[32];
                    if (p.coalesce) {
                        if (res_co) {
                            float res[CH];
                            if (!RES_PREFETCH) tc_epilogue_res_issue<CH>(p, res_regs[0], pix, nbase, vmask, lane);
                            tc_epilogue_res_finish<CH>(p, res_regs[RES_PREFETCH ? c0 / CH : 0], res, wbuf, lane);
                            if (valid) tc_epilogue_math<CH, true>(p, r, pix, nbase, b, v, res);
                        } else if (valid) {
                            tc_epilogue_math<CH, true>(p, r, pix, nbase, b, v);
                        }
                        tc_epilogue_store_warp<CH>(p, v, pix, nbase, vmask, wbuf, lane);
                    } else if (valid) {
                        tc_epilogue_math<CH>(p, r, pix, nbase, b, v);
                        tc_epilogue_store_lane<CH>(p, v, pix, nbase);
                    }
                }
            }
            ptx::tc_fence_before();
            __syncwarp();
            if (lane == 0) ptx::mbar_arrive(tempty_bar(as));
            if (++as == 2) { as = 0; aphase ^= 1; }
        }
    }

    ptx::tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        ptx::tc_fence_after();
        ptx::tmem_dealloc(tmem_base, Cfg::TMEM_COLS);
    }
}

// ------------------------------------------------------------------------------------------------
// Slab variant for small-channel 3-D convolutions (Cin = KC <= 64, Cout <= 64, one pass).
//
// The generic kernel above re-loads the shifted 128-pixel activation tile once per tap; with 16 or 32 channels a tile row
// is only 32-64 bytes and the TMA unit is bound by the NUMBER of rows it moves (27 taps x 128 rows per tile), not by bytes.
// Here a tile is 8 (x) x 16 (y) x 1 (z) output pixels and ONE box load brings the whole halo slab
// [SZ][SY][SX] pixels x KC channels (e.g. 3 x 18 x 10 = 540 rows for a 3x3x3 window) into swizzled K-major shared memory.
// The swizzle is a function of the absolute shared-memory address, so the A operand of tap (dz, dy, dx) is just the same
// slab read through a descriptor whose start address is shifted by ((dz SY + dy) SX + dx) rows and whose 8-row-group stride
// (SBO) is the slab's x pitch: 8 consecutive x pixels form one core-matrix group, consecutive y rows are SX rows apart.
// All tap weight tiles stay resident in shared memory.
// ------------------------------------------------------------------------------------------------
template <int KC>
__device__ __forceinline__ uint64_t make_slab_desc(uint32_t smem_addr, uint32_t sbo_bytes) {
    constexpr uint64_t layout = (KC == 64) ? 2ull : (KC == 32) ? 4ull : 6ull;   // SWIZZLE_128B / 64B / 32B
    return (uint64_t)((smem_addr & 0x3FFFF) >> 4) | (1ull << 16) | ((uint64_t)(sbo_bytes >> 4) << 32) | (1ull << 46) | (layout << 61);
}

template <int BN, int KC>
struct SlabCfg {
    static constexpr int W_SLOT = (BN * KC * 2 + 1023) / 1024 * 1024;
    static constexpr int ACC_STRIDE = BN < 32 ? 32 : BN;
    static constexpr int TMEM_COLS = (2 * ACC_STRIDE <= 64) ? 64 : (2 * ACC_STRIDE <= 128) ? 128 : 256;
    static constexpr int EPI_BYTES = 4 * 2048;
    static constexpr int TILE_BYTES = 128 * BN * 2;               // BULK epilogue: one residual / output tile (16-bit channels)
    static constexpr int BULK_BYTES = 3 * TILE_BYTES;             // two residual tiles + the output staging tile
    static constexpr int MAX_STAGES = 6;
};

// BULK (the full-resolution U-Net layer conv11: 64 fp16 channels out, 64-channel skip tensor, one 128-byte row per pixel): the
// epilogue moves no global memory through registers.  The residual tile (128 rows x 128 B) arrives by TMA into a buffer tied to
// the accumulator stage, issued by a second producer lane as soon as the epilogue has released that stage, and the result tile
// leaves through a 128-byte-swizzled staging buffer with one TMA store per epilogue warp (32 rows = a {64 ch, 8 x, 4 y} box).
// With per-lane loads the kernel sat at 2.6 TB/s on the latency of the residual loads at 8 epilogue warps per SM (ncu: long
// scoreboard 42 % of the stall samples, 18.75 % occupancy at 168 registers).
template <int BN, int KC, int CTAS, bool BULK = false>
__global__ void __launch_bounds__(kTcThreads, CTAS)
slab_conv_kernel(const __grid_constant__ CUtensorMap tmSlab, const __grid_constant__ CUtensorMap tmW, const __grid_constant__ CUtensorMap tmRes,
                 const __grid_constant__ CUtensorMap tmOut, const TcConvParams p, int batch) {
    using Cfg = SlabCfg<BN, KC>;
    const int STAGES = p.slab_stages;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    const int stage_bytes = (p.slab_bytes + 1023) & ~1023;
    uint8_t* wsm = smem + STAGES * stage_bytes;
    uint4* epi_buf = reinterpret_cast<uint4*>(wsm + p.ntaps * Cfg::W_SLOT);       // BULK: [residual tile x 2][output tile], 1 KB aligned
    uint64_t* bars = reinterpret_cast<uint64_t*>(reinterpret_cast<uint8_t*>(epi_buf) + (BULK ? Cfg::BULK_BYTES : Cfg::EPI_BYTES));
    // bars[0..S) full, [S..2S) empty, [2S..2S+2) tmem_full, [2S+2..2S+4) tmem_empty, [2S+4] weights, [2S+5..2S+7) residual full,
    // then the TMEM base address
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * Cfg::MAX_STAGES + 7);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const uint32_t smem_base = ptx::smem_u32(smem);
    const uint32_t w_base = ptx::smem_u32(wsm);
    const uint32_t bar_base = ptx::smem_u32(bars);
    auto full_bar = [&](int s) { return bar_base + 8u * s; };
    auto empty_bar = [&](int s) { return bar_base + 8u * (Cfg::MAX_STAGES + s); };
    auto tfull_bar = [&](int s) { return bar_base + 8u * (2 * Cfg::MAX_STAGES + s); };
    auto tempty_bar = [&](int s) { return bar_base + 8u * (2 * Cfg::MAX_STAGES + 2 + s); };
    const uint32_t w_bar = bar_base + 8u * (2 * Cfg::MAX_STAGES + 4);
    auto rfull_bar = [&](int s) { return bar_base + 8u * (2 * Cfg::MAX_STAGES + 5 + s); };
    const uint32_t res_base = ptx::smem_u32(epi_buf);                 // BULK: residual tile of accumulator stage s at + s * 16 KB
    const uint32_t obuf_base = res_base + 2u * Cfg::TILE_BYTES;       // BULK: output staging, 4 KB per epilogue warp

    if (warp == 0 && lane == 0) {
        ptx::prefetch_tmap(&tmSlab);
        ptx::prefetch_tmap(&tmW);
        if (BULK) {
            ptx::prefetch_tmap(&tmRes);
            ptx::prefetch_tmap(&tmOut);
            ptx::mbar_init(rfull_bar(0), 1);
            ptx::mbar_init(rfull_bar(1), 1);
        }
        for (int s = 0; s < STAGES; ++s) {
            ptx::mbar_init(full_bar(s), 1);
            ptx::mbar_init(empty_bar(s), 1);
        }
        for (int s = 0; s < 2; ++s) {
            ptx::mbar_init(tfull_bar(s), 1);
            ptx::mbar_init(tempty_bar(s), 4);
        }
        ptx::mbar_init(w_bar, 1);
        ptx::fence_barrier_init();
    }
    if (warp == 1) {
        ptx::tmem_alloc(ptx::smem_u32(tmem_slot), Cfg::TMEM_COLS);
        ptx::tmem_relinquish();
    }
    ptx::tc_fence_before();
    __syncthreads();
    ptx::tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    const int tiles_per_img = p.D * p.tiles_y * p.tiles_x;
    const int total_tiles = batch * tiles_per_img;

    if (warp == 0) {
        // ===================== TMA producer: resident weights once, then one halo slab per tile =====================
        if (lane == 0) {
            ptx::mbar_arrive_expect_tx(w_bar, (uint32_t)(p.ntaps * BN * KC * 2));
            for (int t = 0; t < p.ntaps; ++t) ptx::tma_load_3d(&tmW, w_bar, w_base + t * Cfg::W_SLOT, 0, 0, p.twt[t]);
            int stage = 0;
            uint32_t phase = 0;
            for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
                int t = tile;
                const int tx = t % p.tiles_x; t /= p.tiles_x;
                const int ty = t % p.tiles_y; t /= p.tiles_y;
                const int d = t % p.D;
                const int b = t / p.D;
                ptx::mbar_wait(empty_bar(stage), phase ^ 1, p.err, 31);
                ptx::mbar_arrive_expect_tx(full_bar(stage), (uint32_t)p.slab_bytes);
                ptx::tma_load_5d(&tmSlab, full_bar(stage), smem_base + stage * stage_bytes, 0, tx * p.TW + p.slox, ty * p.TH + p.sloy,
                                 d + p.sloz, b);
                if (++stage == STAGES) { stage = 0; phase ^= 1; }
            }
        } else if (BULK && lane == 1) {
            // second producer: the residual tile of a tile goes to the buffer of its accumulator stage once the epilogue has
            // released that stage (two tiles of residual in flight per CTA, independent of the slab ring)
            int as = 0;
            uint32_t aphase = 0;
            for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
                int t = tile;
                const int tx = t % p.tiles_x; t /= p.tiles_x;
                const int ty = t % p.tiles_y; t /= p.tiles_y;
                const int d = t % p.D;
                const int b = t / p.D;
                ptx::mbar_wait(tempty_bar(as), aphase ^ 1, p.err, 36);
                ptx::mbar_arrive_expect_tx(rfull_bar(as), (uint32_t)Cfg::TILE_BYTES);
                ptx::tma_load_5d(&tmRes, rfull_bar(as), res_base + (uint32_t)(as * Cfg::TILE_BYTES), 0, tx * p.TW, ty * p.TH, d, b);
                if (++as == 2) { as = 0; aphase ^= 1; }
            }
        }
    } else if (warp == 1) {
        // ===================== MMA issuer (warp-convergent, elected lane) =====================
        int stage = 0, as = 0;
        uint32_t phase = 0, aphase = 0;
        const uint32_t idesc = make_idesc<BN>(p.f16);
        const uint32_t elected = ptx::elect_one();
        const uint32_t tbase = __shfl_sync(0xffffffffu, tmem_base, 0);
        const uint32_t sbo = (uint32_t)(p.sSX * KC * 2);
        ptx::mbar_wait(w_bar, 0, p.err, 32);
        for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
            ptx::mbar_wait(tempty_bar(as), aphase ^ 1, p.err, 33);
            ptx::mbar_wait(full_bar(stage), phase, p.err, 34);
            ptx::tc_fence_after();
            const uint32_t tmem_d = tbase + (uint32_t)(as * Cfg::ACC_STRIDE);
            const uint32_t sa = smem_base + stage * stage_bytes;
            for (int t = 0; t < p.ntaps; ++t) {
                const int row = ((p.tdz[t] - p.sloz) * p.sSY + (p.tdy[t] - p.sloy)) * p.sSX + (p.tdx[t] - p.slox);
                const uint64_t adesc = make_slab_desc<KC>(sa + (uint32_t)(row * KC * 2), sbo);
                const uint64_t bdesc = make_smem_desc<KC>(w_base + t * Cfg::W_SLOT);
#pragma unroll
                for (int k = 0; k < KC / 16; ++k)
                    ptx::umma_bf16_elected(tmem_d, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idesc, (t > 0 || k > 0) ? 1u : 0u, elected);
            }
            ptx::umma_commit_elected(empty_bar(stage), elected);
            ptx::umma_commit_elected(tfull_bar(as), elected);
            __syncwarp();
            if (++stage == STAGES) { stage = 0; phase ^= 1; }
            if (++as == 2) { as = 0; aphase ^= 1; }
        }
    } else {
        // ===================== epilogue (same as the generic kernel; tile = TW 8 x TH 16) =====================
        const int q = warp & 3;
        const int m = q * 32 + lane;
        const int ty_l = m / p.TW, tx_l = m - ty_l * p.TW;
        int as = 0;
        uint32_t aphase = 0;
        constexpr int CH = (BN < 32) ? BN : 32;
        constexpr bool RES_PREFETCH = BN <= 64;          // residual of the whole tile fits in registers (<= 8 x 16 B per lane)
        const bool res_co = p.coalesce && p.res_hi && !p.res_lo && (p.res_cs & 7) == 0;
        uint4* wbuf = epi_buf + q * 128;
        if (BULK) {
            // a lane owns tile row m: 128 bytes at m * 128 of a 128-byte-swizzled tile (16-byte chunk c sits at c ^ (m & 7))
            const uint32_t rrow = (uint32_t)(m * 128), sw = (uint32_t)(m & 7);
            const uint32_t orow = obuf_base + rrow;
            for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
                int t = tile;
                const int tx = t % p.tiles_x; t /= p.tiles_x;
                const int ty = t % p.tiles_y; t /= p.tiles_y;
                const int d = t % p.D;
                const int b = t / p.D;
                ptx::mbar_wait(tfull_bar(as), aphase, p.err, 35);
                ptx::mbar_wait(rfull_bar(as), aphase, p.err, 37);
                ptx::tc_fence_after();
                if (lane == 0) ptx::bulk_wait_read0();         // the previous tile's store has read this warp's staging rows
                __syncwarp();
                const uint32_t rsrc = res_base + (uint32_t)(as * Cfg::TILE_BYTES) + rrow;
#pragma unroll
                for (int c0 = 0; c0 < BN; c0 += 32) {
                    uint32_t r[32];
                    const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(as * Cfg::ACC_STRIDE + c0);
                    ptx::tmem_ld16(taddr, r);
                    ptx::tmem_ld16(taddr + 16, r + 16);
                    float res[32], v[32];
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        uint4 u;
                        const uint32_t a = rsrc + ((((uint32_t)(c0 >> 3) + j) ^ sw) << 4);
                        asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(u.x), "=r"(u.y), "=r"(u.z), "=r"(u.w) : "r"(a));
                        tc_unpack8(u, 1, res + 8 * j);
                    }
                    ptx::tmem_ld_wait();
                    tc_epilogue_math<32, true>(p, r, 0, c0, b, v, res);
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const uint4 o = tc_pack8(v + 8 * j, 1);
                        const uint32_t a = orow + ((((uint32_t)(c0 >> 3) + j) ^ sw) << 4);
                        asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(a), "r"(o.x), "r"(o.y), "r"(o.z), "r"(o.w) : "memory");
                    }
                }
                // accumulator and residual stage are free again; the staged rows become visible to the TMA unit, one store per warp
                ptx::tc_fence_before();
                ptx::fence_proxy_async();
                __syncwarp();
                if (lane == 0) {
                    ptx::mbar_arrive(tempty_bar(as));
                    ptx::tma_store_5d(&tmOut, obuf_base + (uint32_t)(q * 4096), 0, tx * p.TW, ty * p.TH + 4 * q, d, b);
                    ptx::bulk_commit();
                }
                if (++as == 2) { as = 0; aphase ^= 1; }
            }
            if (lane == 0) ptx::bulk_wait0();
        } else
        for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
            int t = tile;
            const int tx = t % p.tiles_x; t /= p.tiles_x;
            const int ty = t % p.tiles_y; t /= p.tiles_y;
            const int d = t % p.D;
            const int b = t / p.D;
            const int x = tx * p.TW + tx_l, y = ty * p.TH + ty_l;
            const bool valid = (x < p.W) && (y < p.H);
            const size_t pix = (((size_t)b * p.oD + d) * p.oH + y) * p.oW + x;
            const int n0 = 0;
            const unsigned int vmask = __ballot_sync(0xffffffffu, valid);
            uint4 res_regs[RES_PREFETCH ? BN / CH : 1][CH / 8];
            if (RES_PREFETCH && res_co) {      // residual loads in flight while the accumulator is still being produced
#pragma unroll
                for (int c = 0; c < BN / CH; ++c)
                    if (n0 + c * CH < p.Cout) tc_epilogue_res_issue<CH>(p, res_regs[c], pix, n0 + c * CH, vmask, lane);
            }
            ptx::mbar_wait(tfull_bar(as), aphase, p.err, 35);
            ptx::tc_fence_after();
#pragma unroll
            for (int c0 = 0; c0 < BN; c0 += CH) {
                uint32_t r[32];
                const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(as * Cfg::ACC_STRIDE + c0);
                ptx::tmem_ld16(taddr, r);
                if (CH == 32) ptx::tmem_ld16(taddr + 16, r + 16);
                ptx::tmem_ld_wait();
                const int nbase = c0;
                if (nbase < p.Cout) {
                    float v[32];
                    if (p.coalesce) {
                        if (res_co) {
                            float res[CH];
                            if (!RES_PREFETCH) tc_epilogue_res_issue<CH>(p, res_regs[0], pix, nbase, vmask, lane);
                            tc_epilogue_res_finish<CH>(p, res_regs[RES_PREFETCH ? c0 / CH : 0], res, wbuf, lane);
                            if (valid) tc_epilogue_math<CH, true>(p, r, pix, nbase, b, v, res);
                        } else if (valid) {
                            tc_epilogue_math<CH, true>(p, r, pix, nbase, b, v);
                        }
                        tc_epilogue_store_warp<CH>(p, v, pix, nbase, vmask, wbuf, lane);
                    } else if (valid) {
                        tc_epilogue_math<CH>(p, r, pix, nbase, b, v);
                        tc_epilogue_store_lane<CH>(p, v, pix, nbase);
                    }
                }
            }
            ptx::tc_fence_before();
            __syncwarp();
            if (lane == 0) ptx::mbar_arrive(tempty_bar(as));
            if (++as == 2) { as = 0; aphase ^= 1; }
        }
    }
    ptx::tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        ptx::tc_fence_after();
        ptx::tmem_dealloc(tmem_base, Cfg::TMEM_COLS);
    }
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
static PFN_cuTensorMapEncodeTiled_v12000 g_encode = nullptr;
PFN_cuTensorMapEncodeTiled_v12000 g_encode_shared = nullptr;   // for the other tcgen05 translation units

int tc_conv_init_driver() {
    if (g_encode) return ADP_OK;
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    ADP_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
    if (qres != cudaDriverEntryPointSuccess || !fn) {
        set_last_error("cuTensorMapEncodeTiled not available from the driver (query result %d)", (int)qres);
        return ADP_ERR_CUDA;
    }
    g_encode = reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(fn);
    g_encode_shared = g_encode;
    return ADP_OK;
}

static CUtensorMapSwizzle swizzle_for(int KC) {
    return KC == 64 ? CU_TENSOR_MAP_SWIZZLE_128B : KC == 32 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B;
}

// esize 2: 16-bit plane (f16 selects half / bf16), KC channels per box; esize 1: the fp8 twin, 128 one-byte channels per box (the
// rows are 128 bytes either way -> SWIZZLE_128B)
static int encode_act_map(CUtensorMap* tm, const void* ptr, const Act& a, int KC, int TW, int TH, int in_mul, int f16, int esize = 2) {
    cuuint64_t dims[5] = {(cuuint64_t)a.C, (cuuint64_t)a.W, (cuuint64_t)a.H, (cuuint64_t)a.D, (cuuint64_t)a.B};
    cuuint64_t strides[4] = {(cuuint64_t)a.C * esize, (cuuint64_t)a.W * a.C * esize, (cuuint64_t)a.H * a.W * a.C * esize,
                             (cuuint64_t)a.D * a.H * a.W * a.C * esize};
    // with an element stride s the unit loads ceil(box / s) elements: a box of (T-1)*s+1 yields exactly T
    cuuint32_t box[5] = {(cuuint32_t)KC, (cuuint32_t)((TW - 1) * in_mul + 1), (cuuint32_t)((TH - 1) * in_mul + 1), 1, 1};
    cuuint32_t estr[5] = {1, (cuuint32_t)in_mul, (cuuint32_t)in_mul, (cuuint32_t)(a.D > 1 ? in_mul : 1), 1};
    const CUtensorMapDataType dt = esize == 1 ? CU_TENSOR_MAP_DATA_TYPE_UINT8 : f16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
    CUresult r = g_encode(tm, dt, 5, const_cast<void*>(ptr), dims, strides, box, estr,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, esize == 1 ? CU_TENSOR_MAP_SWIZZLE_128B : swizzle_for(KC), CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_last_error("cuTensorMapEncodeTiled(activation C=%d W=%d H=%d D=%d B=%d box=%dx%dx%d) failed: %d", a.C, a.W, a.H,
                       a.D, a.B, KC, TW, TH, (int)r);
        return ADP_ERR_CUDA;
    }
    return ADP_OK;
}

static int encode_w_map(CUtensorMap* tm, const void* ptr, int Cin, int CoutPad, int taps, int KC, int BN, int f16, int esize = 2) {
    cuuint64_t dims[3] = {(cuuint64_t)Cin, (cuuint64_t)CoutPad, (cuuint64_t)taps};
    cuuint64_t strides[2] = {(cuuint64_t)Cin * esize, (cuuint64_t)CoutPad * Cin * esize};
    cuuint32_t box[3] = {(cuuint32_t)KC, (cuuint32_t)BN, 1};
    cuuint32_t estr[3] = {1, 1, 1};
    const CUtensorMapDataType dt = esize == 1 ? CU_TENSOR_MAP_DATA_TYPE_UINT8 : f16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
    CUresult r = g_encode(tm, dt, 3, const_cast<void*>(ptr), dims, strides, box, estr,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, esize == 1 ? CU_TENSOR_MAP_SWIZZLE_128B : swizzle_for(KC), CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_last_error("cuTensorMapEncodeTiled(weights Cin=%d Cout=%d taps=%d box=%dx%d) failed: %d", Cin, CoutPad, taps, KC,
                       BN, (int)r);
        return ADP_ERR_CUDA;
    }
    return ADP_OK;
}

void tc_pick_tile(int H, int W, int* TW, int* TH) {
    // rectangle of <= 128 pixels; prefer exact divisors of the map so that no MMA rows are wasted
    int tw = W;
    if (W > 128) {
        tw = 128;
        for (int c = 128; c >= 8; --c) if (W % c == 0) { tw = c; break; }
    }
    int th = 128 / tw;
    if (th < 1) th = 1;
    if (th > H) th = H;
    // when W divides into a smaller power of two with an exact row fit, prefer it (224 -> 32x4, 112 -> 16x8)
    for (int c = 32; c >= 8; c >>= 1) {
        if (W % c == 0 && H % (128 / c) == 0) { tw = c; th = 128 / c; break; }
    }
    *TW = tw;
    *TH = th;
}

int tc_conv_plan(TcConvLayer* L, const Act& in, const bf16* w_hi, const bf16* w_lo, int Cout, int kd, int ks, int dil,
                 int npass, const TcGeom* geom, int f16) {
    ADP_TRY(tc_conv_init_driver());
    int KC = in.C % 64 == 0 ? 64 : in.C % 32 == 0 ? 32 : in.C % 16 == 0 ? 16 : 0;
    ADP_CHECK_ARG(KC != 0, "Cin must be a multiple of 16 for the tcgen05 path");
    ADP_CHECK_ARG(npass >= 1 && npass <= 4, "npass");
    ADP_CHECK_ARG(npass != 4 || (f16 && in.q8 && w_lo && in.C % 128 == 0),
                  "fp16 + fp8 low-order pass needs fp16 activations with an fp8 twin, packed e4m3 low-order weights and Cin % 128 == 0");
    ADP_CHECK_ARG(npass != 3 || (in.lo && w_lo && !f16), "bf16x3 needs bf16 lo planes of activations and weights");
    ADP_CHECK_ARG(npass != 2 || (w_lo && f16), "fp16x2 needs fp16 activations and a lo plane of the weights");
    int coutPad = (Cout + 15) / 16 * 16;
    int BN = coutPad % 256 == 0 ? 256 : coutPad % 128 == 0 ? 128 : coutPad % 64 == 0 ? 64 : coutPad % 32 == 0 ? 32 : 16;
    if (KC < 64 && BN > 64) BN = 64;
    TcConvParams& p = L->p;
    p = TcConvParams{};
    p.B = in.B;
    p.Cin = in.C; p.Cout = Cout; p.f16 = f16;
    int w_taps;
    if (geom) {
        ADP_CHECK_ARG(geom->ntaps >= 1 && geom->ntaps <= kTcMaxTaps, "tap count");
        p.D = geom->gD; p.H = geom->gH; p.W = geom->gW;
        p.ntaps = geom->ntaps;
        for (int t = 0; t < geom->ntaps; ++t) { p.tdz[t] = geom->dz[t]; p.tdy[t] = geom->dy[t]; p.tdx[t] = geom->dx[t]; p.twt[t] = geom->wt[t]; }
        p.in_mul = geom->in_mul; p.out_mul = geom->out_mul;
        p.out_oz = geom->out_oz; p.out_oy = geom->out_oy; p.out_ox = geom->out_ox;
        p.oD = geom->oD; p.oH = geom->oH; p.oW = geom->oW;
        w_taps = geom->w_taps;
    } else {
        p.D = in.D; p.H = in.H; p.W = in.W;
        p.ntaps = kd * ks * ks;
        ADP_CHECK_ARG(p.ntaps <= kTcMaxTaps, "tap count");
        for (int t = 0; t < p.ntaps; ++t) {
            const int kx = t % ks, ky = (t / ks) % ks, kz = t / (ks * ks);
            p.tdx[t] = (signed char)((kx - ks / 2) * dil); p.tdy[t] = (signed char)((ky - ks / 2) * dil);
            p.tdz[t] = (signed char)(kz - kd / 2); p.twt[t] = (signed char)t;
        }
        p.in_mul = 1; p.out_mul = 1; p.out_oz = p.out_oy = p.out_ox = 0;
        p.oD = in.D; p.oH = in.H; p.oW = in.W;
        w_taps = p.ntaps;
    }
    ADP_CHECK_ARG(p.in_mul == 1 || p.in_mul == 2, "in_mul");
    tc_pick_tile(p.H, p.W, &p.TW, &p.TH);
    p.tiles_x = cdiv(p.W, p.TW);
    p.tiles_y = cdiv(p.H, p.TH);
    p.tiles_n = coutPad / BN;
    p.kchunks = in.C / KC;
    p.npass = npass;
    L->BN = BN;
    L->KC = KC;
    ADP_CHECK_ARG(npass != 4 || BN == 256 || BN == 128, "the fp8 low-order pass needs a Cout tile of 128 or 256");
    // slab mode: single K chunk, single pass, small N, unit strides, a tap window of at most 3 planes x 4 x 4, 8 | W
    L->slab_ctas = 0;
    {
        int lo[3] = {127, 127, 127}, hi[3] = {-127, -127, -127};
        for (int t = 0; t < p.ntaps; ++t) {
            const int o[3] = {p.tdz[t], p.tdy[t], p.tdx[t]};
            for (int a = 0; a < 3; ++a) { lo[a] = o[a] < lo[a] ? o[a] : lo[a]; hi[a] = o[a] > hi[a] ? o[a] : hi[a]; }
        }
        const bool shape_ok = (BN == 16 && (KC == 16 || KC == 64)) || (BN == 64 && KC == 16) || (BN == 32 && KC == 32);
        // (2-D maps qualify too: the s2d stem runs here as 2 x 16 taps - hi and lo weight slabs of the same 4 x 4 window)
        if (p.kchunks == 1 && npass == 1 && coutPad == BN && shape_ok && p.in_mul == 1 && p.out_mul == 1 &&
            p.out_oz == 0 && p.out_oy == 0 && p.out_ox == 0 && p.W % 8 == 0 && p.ntaps >= 4 &&
            hi[0] - lo[0] <= 2 && hi[1] - lo[1] <= 3 && hi[2] - lo[2] <= 3) {
            p.TW = 8; p.TH = 16;
            p.tiles_x = cdiv(p.W, p.TW); p.tiles_y = cdiv(p.H, p.TH);
            p.sSX = 8 + hi[2] - lo[2]; p.sSY = 16 + hi[1] - lo[1]; p.sSZ = 1 + hi[0] - lo[0];
            p.sloz = lo[0]; p.sloy = lo[1]; p.slox = lo[2];
            p.slab_bytes = p.sSX * p.sSY * p.sSZ * KC * 2;
            const int stage_bytes = (p.slab_bytes + 1023) & ~1023;
            const int w_slot = (BN * KC * 2 + 1023) / 1024 * 1024;
            const int fixed = p.ntaps * w_slot + 8192 + 1024 + 512;
            // CTAs per SM; 32 -> 32 channels (conv4: 35 KB slabs + 54 KB of weights) runs one CTA per SM with more stages
            const int ctas = (BN == 32 && KC == 32) ? 1 : 2;
            int stages = (220 * 1024 / ctas - fixed) / stage_bytes;
            stages = stages > 6 ? 6 : stages;
            if (stages >= 2) {
                p.slab_stages = stages;
                L->slab_ctas = ctas;
                cuuint64_t dims[5] = {(cuuint64_t)in.C, (cuuint64_t)in.W, (cuuint64_t)in.H, (cuuint64_t)in.D, (cuuint64_t)in.B};
                cuuint64_t strides[4] = {(cuuint64_t)in.C * 2, (cuuint64_t)in.W * in.C * 2, (cuuint64_t)in.H * in.W * in.C * 2,
                                         (cuuint64_t)in.D * in.H * in.W * in.C * 2};
                cuuint32_t box[5] = {(cuuint32_t)KC, (cuuint32_t)p.sSX, (cuuint32_t)p.sSY, (cuuint32_t)p.sSZ, 1};
                cuuint32_t estr[5] = {1, 1, 1, 1, 1};
                CUresult r = g_encode(&L->tmSlab, f16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, in.hi, dims,
                                      strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle_for(KC), CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                                      CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
                if (r != CUDA_SUCCESS) {
                    set_last_error("cuTensorMapEncodeTiled(slab %dx%dx%d x %d) failed: %d", p.sSX, p.sSY, p.sSZ, KC, (int)r);
                    return ADP_ERR_CUDA;
                }
            } else {
                tc_pick_tile(p.H, p.W, &p.TW, &p.TH);
                p.tiles_x = cdiv(p.W, p.TW); p.tiles_y = cdiv(p.H, p.TH);
            }
        }
    }
    ADP_TRY(encode_act_map(&L->tmA_hi, in.hi, in, KC, p.TW, p.TH, p.in_mul, f16));
    ADP_TRY(encode_w_map(&L->tmW_hi, w_hi, in.C, coutPad, w_taps, KC, BN, f16));
    if (npass == 4) {        // the "lo" maps address the fp8 twins: 128 one-byte channels per box
        ADP_TRY(encode_act_map(&L->tmA_lo, in.q8, in, 128, p.TW, p.TH, p.in_mul, f16, 1));
        ADP_TRY(encode_w_map(&L->tmW_lo, w_lo, in.C, coutPad, w_taps, 128, BN, f16, 1));
    } else {
        ADP_TRY(encode_act_map(&L->tmA_lo, in.lo ? in.lo : in.hi, in, KC, p.TW, p.TH, p.in_mul, f16));
        ADP_TRY(encode_w_map(&L->tmW_lo, w_lo ? w_lo : w_hi, in.C, coutPad, w_taps, KC, BN, f16));
    }
    return ADP_OK;
}

// after the epilogue fields of L->p are set: the TMA epilogue where it applies, and its tensor maps
static int tc_conv_pick_bulk_epilogue(TcConvLayer* L) {
    TcConvParams& p = L->p;
    L->bulk_epi = false;
    const bool off = getenv("ADP_NO_BULK_EPI") != nullptr;        // read per plan: the A/B test builds one engine each way
    if (off || !L->slab_ctas || L->BN != 64 || L->KC != 16 || p.Cout != 64 || !p.f16 || !p.coalesce) return ADP_OK;
    if (!p.res_hi || p.res_lo || p.res_cs != 64 || !p.out_hi || p.out_lo || p.out_cs != 64 || p.out_coff != 0) return ADP_OK;
    if (p.out_f32 || p.out_h16 || p.out_q8 || p.bias_per_batch || p.TW != 8 || p.TH != 16) return ADP_OK;
    if (((uintptr_t)p.res_hi | (uintptr_t)p.out_hi) & 15) return ADP_OK;
    // shared memory: the residual / output tiles take the place of the transpose buffers; give up slab stages to stay at 2 CTAs per SM
    using Cfg = SlabCfg<64, 16>;
    const int stage_bytes = (p.slab_bytes + 1023) & ~1023;
    const int fixed = p.ntaps * Cfg::W_SLOT + Cfg::BULK_BYTES + 1024 + 512;
    int stages = p.slab_stages;
    while (stages >= 2 && stages * stage_bytes + fixed > 111 * 1024) --stages;
    if (stages < 2) return ADP_OK;
    cuuint64_t dims[5] = {64, (cuuint64_t)p.oW, (cuuint64_t)p.oH, (cuuint64_t)p.oD, (cuuint64_t)p.B};
    cuuint64_t strides[4] = {128, (cuuint64_t)p.oW * 128, (cuuint64_t)p.oH * p.oW * 128, (cuuint64_t)p.oD * p.oH * p.oW * 128};
    cuuint32_t estr[5] = {1, 1, 1, 1, 1};
    cuuint32_t box_r[5] = {64, 8, 16, 1, 1}, box_o[5] = {64, 8, 4, 1, 1};
    CUresult r = g_encode(&L->tmRes, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 5, const_cast<bf16*>(p.res_hi), dims, strides, box_r, estr,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r == CUDA_SUCCESS)
        r = g_encode(&L->tmOut, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 5, p.out_hi, dims, strides, box_o, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_last_error("cuTensorMapEncodeTiled(residual / output tiles %dx%dx%d) failed: %d", p.oW, p.oH, p.oD, (int)r);
        return ADP_ERR_CUDA;
    }
    p.slab_stages = stages;
    L->bulk_epi = true;
    return ADP_OK;
}

template <int BN, int KC, int FUSED = 0>
static int launch_impl(const TcConvLayer* L, int batch, int num_sms, cudaStream_t stream) {
    using Cfg = TcCfg<BN, KC, FUSED>;
    static int attr[kMaxDevices];
    ADP_TRY(ensure_dyn_smem(tc_conv_kernel<BN, KC, FUSED>, Cfg::SMEM_BYTES, attr));
    const TcConvParams& p = L->p;
    long long total = (long long)batch * p.D * p.tiles_y * p.tiles_x * p.tiles_n;
    const long long slots = (long long)num_sms * Cfg::CTAS_PER_SM;
    int grid = (int)(total < slots ? total : slots);
    if (grid <= 0) return ADP_OK;
    tc_conv_kernel<BN, KC, FUSED><<<grid, kTcThreads, Cfg::SMEM_BYTES, stream>>>(L->tmA_hi, L->tmA_lo, L->tmW_hi, L->tmW_lo, p, batch);
    ADP_CUDA(cudaGetLastError());
    return ADP_OK;
}

template <int BN, int KC, int CTAS, bool BULK = false>
static int launch_slab(const TcConvLayer* L, int batch, int num_sms, cudaStream_t stream) {
    using Cfg = SlabCfg<BN, KC>;
    const TcConvParams& p = L->p;
    const int stage_bytes = (p.slab_bytes + 1023) & ~1023;
    const int smem = p.slab_stages * stage_bytes + p.ntaps * Cfg::W_SLOT + (BULK ? Cfg::BULK_BYTES : Cfg::EPI_BYTES) + 1024 + 512;
    static int attr[kMaxDevices];
    ADP_TRY(ensure_dyn_smem(slab_conv_kernel<BN, KC, CTAS, BULK>, smem, attr));
    const long long total = (long long)batch * p.D * p.tiles_y * p.tiles_x;
    const long long slots = (long long)num_sms * CTAS;
    const int grid = (int)(total < slots ? total : slots);
    if (grid <= 0) return ADP_OK;
    slab_conv_kernel<BN, KC, CTAS, BULK><<<grid, kTcThreads, smem, stream>>>(L->tmSlab, L->tmW_hi, BULK ? L->tmRes : L->tmSlab,
                                                                             BULK ? L->tmOut : L->tmSlab, p, batch);
    ADP_CUDA(cudaGetLastError());
    return ADP_OK;
}

// Every kernel instance there is.  slab_ctas 0: the generic kernel; FUSED 0 = one pass, or the pass loop of split precision,
// 1 = bf16x3, 2 = fp16x2, 3 = fp16 + fp8 low-order pass.  slab_ctas > 0: the slab kernel (single pass) for that many CTAs per SM,
// bulk = TMA epilogue.
struct TcInstance {
    int slab_ctas;
    bool bulk;
    int fused, BN, KC;
    decltype(TcConvLayer::launch) launch;
};
static const TcInstance kTcInstances[] = {
    {0, false, 0, 256, 64, launch_impl<256, 64>},
    {0, false, 0, 128, 64, launch_impl<128, 64>},
    {0, false, 0, 64, 64, launch_impl<64, 64>},
    {0, false, 0, 32, 64, launch_impl<32, 64>},
    {0, false, 0, 16, 64, launch_impl<16, 64>},
    {0, false, 0, 64, 32, launch_impl<64, 32>},
    {0, false, 0, 32, 16, launch_impl<32, 16>},
    {0, false, 1, 256, 64, launch_impl<256, 64, 1>},
    {0, false, 1, 128, 64, launch_impl<128, 64, 1>},
    {0, false, 1, 64, 64, launch_impl<64, 64, 1>},
    {0, false, 1, 32, 64, launch_impl<32, 64, 1>},
    {0, false, 1, 64, 16, launch_impl<64, 16, 1>},
    {0, false, 2, 256, 64, launch_impl<256, 64, 2>},
    {0, false, 2, 128, 64, launch_impl<128, 64, 2>},
    {0, false, 2, 64, 64, launch_impl<64, 64, 2>},
    {0, false, 2, 32, 64, launch_impl<32, 64, 2>},
    {0, false, 3, 256, 64, launch_impl<256, 64, 3>},
    {0, false, 3, 128, 64, launch_impl<128, 64, 3>},
    {2, false, 0, 16, 16, launch_slab<16, 16, 2>},
    {2, false, 0, 16, 64, launch_slab<16, 64, 2>},
    {2, false, 0, 64, 16, launch_slab<64, 16, 2>},         // (3 CTAs per SM spill: 1.5 -> 1.9 ms)
    {2, true, 0, 64, 16, launch_slab<64, 16, 2, true>},
    {1, false, 0, 32, 32, launch_slab<32, 32, 1>},
};

static decltype(TcConvLayer::launch) find_instance(int slab_ctas, bool bulk, int fused, int BN, int KC) {
    for (const TcInstance& t : kTcInstances)
        if (t.slab_ctas == slab_ctas && t.bulk == bulk && t.fused == fused && t.BN == BN && t.KC == KC) return t.launch;
    return nullptr;
}

int tc_conv_finish_plan(TcConvLayer* L) {
    ADP_TRY(tc_conv_pick_bulk_epilogue(L));
    // split precision keeps its hi and lo operands in one pipeline stage where (BN, KC) has such an instance, and otherwise runs
    // the passes one after another through the FUSED = 0 kernel (the narrow per-point MLP layers)
    const int npass = L->p.npass;
    const int fused = npass == 2 ? 2 : npass == 3 ? 1 : npass == 4 ? 3 : 0;
    L->launch = find_instance(L->slab_ctas, L->bulk_epi, fused, L->BN, L->KC);
    if (!L->launch && (npass == 2 || npass == 3)) L->launch = find_instance(0, false, 0, L->BN, L->KC);
    if (!L->launch) {
        static const char* const mode[] = {"", "single pass", "fp16x2", "bf16x3", "fp16 + fp8 low-order pass"};
        set_last_error("no tcgen05 conv instantiation for BN=%d KC=%d (%s%s)", L->BN, L->KC, mode[npass],
                       L->slab_ctas ? ", slab kernel" : "");
        return ADP_ERR_ARG;
    }
    return ADP_OK;
}

int tc_conv_launch(const TcConvLayer* L, int batch, int num_sms, cudaStream_t stream) {
    ADP_CHECK_ARG(L->launch, "layer not planned");
    ADP_CHECK_ARG(batch <= L->p.B, "batch exceeds planned capacity");
    return L->launch(L, batch, num_sms, stream);
}

}  // namespace adp
