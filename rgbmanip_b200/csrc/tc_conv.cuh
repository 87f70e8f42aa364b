// tcgen05 / TMEM / TMA implicit-GEMM convolution for channels-last bf16 activations (sm_100a).
//
//   D[m, n] = sum_{tap, c} A[pixel(m) + offset(tap), c] * W[tap, n, c]
//
// m runs over a TH x TW rectangle of output pixels (<= 128 rows of the UMMA M=128 tile), n over BN output
// channels, the K loop over (pass, tap, 64-channel chunk).  Each K step is one TMA box load of the shifted
// activation rectangle (out-of-image coordinates are zero-filled by the TMA unit = the conv's zero padding)
// and one box load of the weight slab, both landing in 128B-swizzled K-major shared memory, followed by
// four tcgen05.mma (K = 16 each) accumulating into TMEM.  Stride-1 "same" convolutions only: 2-D with
// D == 1, or 3-D where the depth axis is one more tensor-map dimension.
//
// Split precision ("bf16x3"): activations and weights are stored as hi + lo bf16 pairs and the K loop runs
// three passes (A_hi W_hi, A_lo W_hi, A_hi W_lo) into the same fp32 accumulator, which restores ~16
// mantissa bits -- see DESIGN.md "precision policy".
#pragma once
#include "common.cuh"

namespace adp {

constexpr int kTcMaxTaps = 32;

struct TcConvParams {
    int B, D, H, W;          // tile-space extent: the grid the M tiles walk over (output grid for convs, input grid for
                             // the parity classes of a transposed conv); D == 1 for 2-D
    int Cin, Cout;
    // tap table: input coordinate = tile coordinate * in_mul + (dz, dy, dx); weight slab index wt
    int ntaps;
    signed char tdz[kTcMaxTaps], tdy[kTcMaxTaps], tdx[kTcMaxTaps], twt[kTcMaxTaps];
    int in_mul;              // 1, or 2 for stride-2 convs (TMA element stride 2)
    // output coordinate = tile coordinate * out_mul + (out_oz, out_oy, out_ox), inside an [oD, oH, oW] grid
    int out_mul, out_oz, out_oy, out_ox;
    int oD, oH, oW;
    int f16;                 // 0: bf16 operands/activations, 1: fp16
    int TW, TH;              // spatial tile; TW * TH <= 128
    int tiles_x, tiles_y, tiles_n;
    int kchunks;             // Cin / KC
    int npass;               // 1 = single pass, 2 = fp16x2 (A W_hi + A W_lo), 3 = bf16x3, 4 = fp16 + fp8 low-order pass
    // epilogue
    const float* bias;       // [Cout] or nullptr (BatchNorm shift is passed here too)
    const float* scale;      // [Cout] or nullptr (folded BatchNorm scale)
    float prelu;             // slope for act == 2
    int act;                 // 0 none, 1 relu, 2 prelu, 3 tanh
    int res_after_act;       // 0: act(acc + res)   1: act(acc) + res   (3-D U-Net skips)
    const bf16* res_hi;
    const bf16* res_lo;
    int res_cs;              // channel pitch of the residual tensor
    bf16* out_hi;
    bf16* out_lo;
    float* out_f32;
    uint8_t* out_q8;         // optional fp8 twin of out_hi (value / 2, e4m3; same channel pitch / offset): see Act::q8
    __half* out_h16;         // optional extra fp16 copy
    int out_cs, out_coff;    // channel pitch / first channel of out_hi, out_lo
    int bias_per_batch;      // bias is [B, Cout]
    // slab mode (small-channel 3-D convs, see slab_conv_kernel): halo slab extents / origin offset, bytes per stage
    int sSX, sSY, sSZ, slox, sloy, sloz, slab_bytes, slab_stages;
    int check_finite;        // OR bit 0 into err[1] when an output value is not finite (fp16 range guard on the feature map)
    int coalesce;            // epilogue stores go through the per-warp transpose buffers (full chunks, single 16-bit plane)
    int* err;                // device error flag (pipeline watchdog)
};

// Host side: build tensor maps + launch.  Returns ADP_OK or an error code (message via set_last_error).
struct TcConvLayer {
    CUtensorMap tmA_hi, tmA_lo, tmW_hi, tmW_lo;
    TcConvParams p;
    int BN;
    int KC;                  // channels per K step (64 -> SWIZZLE_128B, 32 -> 64B, 16 -> 32B)
    int slab_ctas = 0;       // > 0: slab mode (one halo slab per tile, taps by descriptor offsets, weights resident:
                             // slab_conv_kernel), with stages sized for this many CTAs per SM
    CUtensorMap tmSlab;
    bool bulk_epi = false;   // slab mode, 64 fp16 channels in and out with a 64-channel residual: residual tiles arrive by TMA, results
                             // leave by TMA store (tc_conv_finish_plan decides)
    CUtensorMap tmRes, tmOut;
    // the kernel instance of this layer, chosen by tc_conv_finish_plan; null until the plan is complete
    int (*launch)(const TcConvLayer* L, int batch, int num_sms, cudaStream_t stream) = nullptr;
    int instance = -1;       // its row in the instance table of tc_conv.cu (reported by tc_conv_plan_info)
};

int tc_conv_init_driver();
struct TcGeom {             // non-standard geometries (NULL = stride-1 "same" conv with a kd x ks x ks window)
    int ntaps;
    signed char dz[32], dy[32], dx[32], wt[32];
    int in_mul;
    int out_mul, out_oz, out_oy, out_ox;
    int gD, gH, gW;
    int oD, oH, oW;
    int w_taps;             // number of tap slabs in the packed weight tensor
};

int tc_conv_plan(TcConvLayer* L, const Act& in, const bf16* w_hi, const bf16* w_lo, int Cout, int kd, int ks,
                 int dil, int npass, const TcGeom* geom, int f16);
// after the epilogue fields of L->p are set: picks the TMA epilogue where it applies and the kernel instance; ADP_ERR_ARG when
// the library has no instance for the layer's tile, K step and pass mode
int tc_conv_finish_plan(TcConvLayer* L);
int tc_conv_launch(const TcConvLayer* L, int batch, int num_sms, cudaStream_t stream);
// the chosen instance and tiling of a planned layer: the 16 fields of adp_conv_tc_plan_info (include/adapose_b200.h)
int tc_conv_plan_info(const TcConvLayer* L, int32_t* info);

}  // namespace adp
