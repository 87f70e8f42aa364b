/* libadapose_b200.so -- C ABI of the B200-native AdaPose hot path.
 *
 * The reference (hyperplane-lab/RGBManip) is pure Python: it has no FFI for this path, the seam is the class
 * models/pose_estimator/AdaPose/interface_v5.py:37 `AdaPoseEstimator_v5`, whose `estimate()` (:213-227) loops
 * `predict()` (:229-374) over environments.  The entry points below are the device stages that replace the body
 * of that loop; the Python host mirror (rgbmanip_b200/estimator.py) binds them with ctypes and keeps the
 * reference's class/method surface.  INTEGRATION.md shows the binding a reference maintainer would add.
 *
 * Conventions: every function returns 0 on success and a negative code on failure (adp_last_error() holds the
 * message); pointers are raw CUDA device pointers unless named `host_*`; `stream` is a cudaStream_t passed as
 * void*; nothing allocates device memory except adp_conv_tc_plan (a small descriptor object on the host) and
 * nothing synchronises.  Activations are channels-last 16-bit planes: one IEEE-half plane (`f16 = 1`: the default "fp16x2"
 * backbone and the 3-D stage) or a bf16 `hi` plane plus an optional `lo` plane (value = hi + lo, "bf16x3" split precision);
 * fp32 tensors are plain channels-last.  `npass` of adp_conv_tc_plan selects the MMA passes per K step: 1 = A W,
 * 2 = A W_hi + A W_lo (fp16 activations, fp16 weights split in two planes), 3 = A_hi W_hi + A_lo W_hi + A_hi W_lo (bf16),
 * 4 = A W_hi in fp16 + the low-order term as an fp8 MMA at twice the rate: e4m3(A / 2) (the activation's q8 twin) x
 * e4m3(W_lo 2^16) (passed as w_lo, one byte per weight), joined through the MMA's 2^-15 accumulator scale.
 * No torch types appear.
 */
#ifndef ADAPOSE_B200_H
#define ADAPOSE_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ADP_ABI_VERSION 6

#if defined(__GNUC__)
#define ADP_API __attribute__((visibility("default")))
#else
#define ADP_API
#endif

/* dtype codes for host-facing image inputs */
#define ADP_DT_U8 0
#define ADP_DT_F32 1
#define ADP_DT_F64 2

/* activation codes of a convolution epilogue */
#define ADP_ACT_NONE 0
#define ADP_ACT_RELU 1
#define ADP_ACT_PRELU 2
#define ADP_ACT_TANH 3

typedef struct adp_act {      /* channels-last activation [B, D, H, W, C]; D == 1 for 2-D maps */
    void* hi;                 /* bf16 (or IEEE half when f16 != 0) */
    void* lo;                 /* bf16 or NULL */
    int32_t B, D, H, W, C;
    int32_t f16;              /* 1: 16-bit planes are IEEE half (3-D cost-regularisation stage), no lo plane */
    void* q8;                 /* optional fp8 (e4m3) twin of an f16 activation holding value / 2, or NULL: the A operand of the
                                 low-order pass of npass = 4 layers; written by the producing layer (adp_epilogue.out_q8) */
} adp_act;

typedef struct adp_tc_geom {  /* non-default geometry of a tcgen05 conv: explicit tap table and grid mapping */
    int32_t ntaps;            /* <= 32 */
    int8_t dz[32], dy[32], dx[32], wt[32];   /* input offset of each tap (after in_mul scaling) and its weight slab */
    int32_t in_mul;           /* input coord = tile coord * in_mul + offset: 2 for stride-2 convs */
    int32_t out_mul, out_oz, out_oy, out_ox; /* output coord = tile coord * out_mul + offset: 2 / parity for transposed convs */
    int32_t gD, gH, gW;       /* tile-space grid */
    int32_t oD, oH, oW;       /* output grid */
    int32_t w_taps;           /* tap slabs in the packed weights */
} adp_tc_geom;

typedef struct adp_epilogue { /* y = act(scale * acc + bias [+ res]) [+ res]  ->  out_hi/out_lo and/or out_f32 */
    const float* scale;       /* [Cout] or NULL : folded BatchNorm3d scale (network_v5.py:19,240) */
    const float* bias;        /* [Cout] or NULL : conv bias or folded BatchNorm shift */
    float prelu;              /* slope for ADP_ACT_PRELU (pspnet.py:100-103) */
    int32_t act;
    int32_t res_after_act;    /* 0: residual joins before the activation (pspnet.py:27-29); 1: after (network_v5.py:287-289) */
    const void* res_hi;       /* bf16 [.., Cout] or NULL */
    const void* res_lo;
    int32_t res_cstride;      /* channel pitch of the residual tensor (0 = Cout); lets a channel-padded tensor be the skip */
    void* out_hi;             /* bf16 or NULL */
    void* out_lo;
    float* out_f32;           /* fp32 or NULL */
    void* out_h16;            /* optional extra IEEE-half copy of the output (feature map for the volume builder) or NULL */
    int32_t out_cstride;      /* channel pitch of out_hi/out_lo (0 = Cout): lets a layer write a column range of a wider tensor */
    int32_t out_coff;         /* first channel of that range (torch.cat of network_v5.py:488 without a copy) */
    int32_t bias_per_batch;   /* 1: bias is [B, Cout] (the per-env global feature term of pose_mlp2, network_v5.py:491-493) */
    void* out_q8;             /* optional fp8 (e4m3) twin of out_hi holding value / 2 (same channel pitch / offset), or NULL: see adp_act.q8;
                                 needs fp16, Cout % 32 == 0 and out_cstride, out_coff multiples of 16 (else ADP_ERR_ARG at plan time) */
    int32_t check_finite;     /* 1: OR bit 0 into err_flag[1] when an output value is inf/NaN (fp16 range guard, set on the last backbone layer) */
} adp_epilogue;

typedef struct adp_decode_weights {   /* fp32, each matrix transposed to [K][N]; names follow the reference state_dict */
    const float *ic_w, *ic_b, *nh0_w, *nh0_b, *nh1_w, *nh1_b, *nh2_w, *nh2_b, *np0_w, *np0_b, *np1_w, *np1_b;
    const float *pm0_w, *pm0_b, *pm1_w, *pm1_b, *q0_w, *q0_b, *q1_w, *q1_b, *r0_w, *r0_b, *r1_w, *r1_b, *r2_w, *r2_b;
    const float* prob_w;      /* cost_regularization.prob.weight as [27][8] */
} adp_decode_weights;

typedef struct adp_conv_plan adp_conv_plan;   /* tcgen05 conv layer bound to fixed buffers (holds the TMA tensor maps) */

ADP_API int adp_abi_version(void);
ADP_API const char* adp_last_error(void);
/* number of kernels launched by this library since load (bench.py reports it as gpu_launches) */
ADP_API uint64_t adp_launch_count(void);
/* a captured CUDA graph replays kernels without passing through the entry points: the host adds the replayed launches */
ADP_API void adp_launch_count_add(uint64_t n);
ADP_API int adp_device_info(int device, int* num_sms, int* cc_major, int* cc_minor);

/* --- preprocessing: interface_v5.py:58-170 (prepare_model_input), utils.py:10-38 (get_bbox) ------------------
 * rgb [F,H,W,3] (f32|f64, or u8 = the f32 path on value / 255 like ToTensor; H, W >= 440), mask [F,H,W] (u8|f32|f64), K [F,3,3] f64 (k_stride doubles between frames; 0 = shared).
 * Outputs: win [F,4] = rmin,rmax,cmin,cmax; Kp [F,9] f64 crop intrinsics; valid [F]; crops [F,S,S,3] f32 normalised;
 * choose [F,P] i32 (written when choose_mode == 0, read-only when 1 = caller-supplied); counts [F] foreground pixels.
 * The device sampler (choose_mode 0) is a counter-based hash of (seed, frame_id0 + f, pixel rank): pass the global
 * environment index of frame 0 as frame_id0 and the subset drawn for an environment is independent of chunking / sharding. */
ADP_API int adp_preprocess(const void* rgb, int rgb_dtype, const void* mask, int mask_dtype, const double* K, int k_stride,
                   int F, int H, int W, int S, int P, uint32_t seed, int choose_mode, int frame_id0, int32_t* bbox_ws,
                   int32_t* win, double* Kp, uint8_t* valid, float* crops, int32_t* choose, int32_t* counts, void* stream);

/* Crop windows alone (the mask pass of adp_preprocess: utils.py:10-38): win [F,4] = rmin,rmax,cmin,cmax, valid [F].  The host
 * mirror uploads the masks first, reads the windows back and then uploads only the image rows a window covers (a 480 x 640 fp32
 * frame is 3.7 MB, the rows of a typical 160-pixel window 1.2 MB); adp_preprocess reads nothing outside the window. */
ADP_API int adp_mask_windows(const void* mask, int mask_dtype, int F, int H, int W, int32_t* bbox_ws, int32_t* win, uint8_t* valid,
                             void* stream);

/* --- backbone: pspnet.py:33-158 ------------------------------------------------------------------------------ */
ADP_API int adp_conv_tc_plan(adp_conv_plan** plan, const adp_act* in, const void* w_hi, const void* w_lo, int cout, int kd,
                     int ks, int dil, int npass, const adp_epilogue* ep, const adp_tc_geom* geom, int num_sms);
/* err_flag: int32[2] on the device -- [0] pipeline watchdog code (a stuck barrier traps the kernel instead of hanging the GPU),
 * [1] range flag (see adp_epilogue.check_finite).  The same two-word flag is passed to every *_run entry point. */
ADP_API int adp_conv_tc_run(adp_conv_plan* plan, int batch, int32_t* err_flag, void* stream);
/* The kernel instance a plan chose and its tiling, read-only (tests use it to tie each reference case to an instance).
 * info: int32[ADP_TC_PLAN_INFO_LEN] =
 *   [0] row of the instance table (tc_conv.cu kTcInstances)   [1] slab CTAs per SM (0: generic kernel)   [2] TMA epilogue
 *   [3] FUSED: 0 single pass or the split-precision pass loop, 1 bf16x3, 2 fp16x2, 3 fp16 + fp8 low-order pass
 *   [4] BN   [5] KC   [6] npass of the layer   [7] TW   [8] TH   [9] coalesced epilogue stores
 *   [10] tiles_x   [11] tiles_y   [12] tiles_n   [13] tile-grid depth (tiles per image = [10] [11] [12] [13])
 *   [14] K chunks   [15] taps */
#define ADP_TC_PLAN_INFO_LEN 16
ADP_API int adp_conv_tc_plan_info(const adp_conv_plan* plan, int32_t* info);
ADP_API void adp_conv_tc_free(adp_conv_plan* plan);
ADP_API int adp_maxpool3x3s2(const adp_act* in, const adp_act* out, int batch, void* stream);                 /* pspnet.py:39 */
/* feat_cstride: channel pitch of feat (0 = dense); the engine lets layer4's last conv write straight into the first 512
 * channels of the 1024-channel concat tensor, adp_psp_fill_priors writes the resized priors behind them (:92-94). */
ADP_API int adp_psp_priors(const adp_act* feat, int feat_cstride, const float* w, float* pooled, float* priors, int batch, void* stream); /* :84-90 */
ADP_API int adp_psp_fill_priors(const float* priors, const adp_act* out, int coff, int batch, void* stream);
ADP_API int adp_upsample2x(const adp_act* in, const adp_act* out, int batch, void* stream);                   /* pspnet.py:105 */
/* PSPUpsample (pspnet.py:97-107: bilinear x2, align_corners=True -> Conv2d 3x3 pad 1 -> PReLU), second half of its restructured
 * form: q [B,h,w,9*C] holds the nine per-tap 1x1 products W_tap x of the LOW-resolution input (channel = (ky*3+kx)*C + c, one
 * adp_conv_tc GEMM); this call blends them (9 taps x 4 bilinear neighbours, zero padding of the upsampled image), adds the bias and
 * applies the PReLU -> out [B,2h,2w,C].  Equal to conv(upsample(x)) up to fp32 summation order. */
ADP_API int adp_upconv_blend(const adp_act* q, const adp_act* out, const float* bias, float prelu_slope, int batch, void* stream);
/* fp32 crops [F,S,S,3] -> space-to-depth(2) activation [F,S/2,S/2,16] (channel = (py*2+px)*3 + c, 12 used): the 7x7/2
 * stem conv (pspnet.py:37) then is a 4x4 stride-1 conv over 16 channels and runs on the tcgen05 kernel. */
ADP_API int adp_pack_s2d(const float* crops, const adp_act* out, int batch, int S, void* stream);

/* conv0 of the cost-regularisation U-Net (network_v5.py:263,283) as a depth-ring tcgen05 kernel: vol [B,D,H,W,32] ->
 * out [B,D,H,W,16] (8 channels + 8 zero), folded BatchNorm + ReLU.  w: 16-bit [3 kx][4 chunks of 8 channels][80 n][8] with
 * n = (kz*3+ky)*8 + co (rows 72..79 zero): depth and row taps folded into the MMA's N (rgbmanip_b200.geometry.conv0_ring_weights).
 * flags: bit 0 must be 0 (reserved: planar volume layout); bit 1 (ADP_LAYOUT_S2D) = write the 8 real channels
 * space-to-depth(2): out [B,D/2,H/2,W/2,64] (D even, else ADP_ERR_ARG), channel = ((d&1)*4 + (y&1)*2 + (x&1))*8 + co.  In that
 * layout the stride-2 conv1 and the skip connection of the transposed conv11 (network_v5.py:265,278,283) read it as a stride-1
 * tensor. */
#define ADP_LAYOUT_F16 1
#define ADP_LAYOUT_S2D 2
typedef struct adp_conv0_plan adp_conv0_plan;
ADP_API int adp_conv0_plan_create(adp_conv0_plan** plan, const adp_act* vol, const void* w_packed, const float* scale,
                                  const float* shift, void* out, int flags, int num_sms);
ADP_API int adp_conv0_run(adp_conv0_plan* plan, int batch, int32_t* err_flag, void* stream);
ADP_API void adp_conv0_free(adp_conv0_plan* plan);

/* ConvTranspose3d(k3, s2, p1, op1) + folded BN + ReLU + skip (network_v5.py:217-258,274-278,287-289) with all 8 output
 * parity classes in one tcgen05 kernel.  in [B,D,H,W,Cin] (Cin 16|32, single 16-bit plane), w 16-bit [27][pad16(Cout)][Cin],
 * res [B,2D,2H,2W,res_cstride] or NULL, out [B,2D,2H,2W,Cout].  flags & ADP_LAYOUT_S2D: res and out are stored
 * space-to-depth(2), [B,D,H,W,8*Cout] with channel = parity*Cout + c (res_cstride ignored). */
typedef struct adp_tconv_plan adp_tconv_plan;
ADP_API int adp_tconv_plan_create(adp_tconv_plan** plan, const adp_act* in, const void* w, int cout, const float* scale,
                                  const float* bias, const void* res, int res_cstride, void* out, int flags, int num_sms);
ADP_API int adp_tconv_run(adp_tconv_plan* plan, int batch, int32_t* err_flag, void* stream);
ADP_API void adp_tconv_free(adp_tconv_plan* plan);

/* --- stereo volume: network_v5.py:378-416,429 ---------------------------------------------------------------- */
/* Mw[b] = {rot 3x3 row-major, trans 3} of P_src inv(P_ref), P = [K' E[:3,:]; 0 0 0 1] (interface_v5.py:264-270);
 * valid_env[b] = valid_ref[b] && valid_src[b] (an estimate needs both views, interface_v5.py:256-257). */
ADP_API int adp_warp_matrices(const double* Kp_ref, const double* E_ref, const double* Kp_src, const double* E_src,
                              float* Mw, const uint8_t* valid_ref, const uint8_t* valid_src, uint8_t* valid_env, int B,
                              void* stream);
/* feat_*: [B,H,W,32] IEEE half (the fp16 twin of the feature map written by the last backbone layer, adp_epilogue.out_h16).
 * vol: [B,D,H,W,32], IEEE half when f16 != 0 else bf16. */
ADP_API int adp_build_volume(const void* feat_ref, const void* feat_src, const float* Mw, const float* depths, void* vol,
                     int B, int D, int H, int W, int C, int f16, void* stream);

/* --- decode + heads: network_v5.py:432-465,486-499; rotation_utils.py:4-27 ----------------------------------- */
/* adp_decode_gather = the gather-bound part (depth logits at the sampled pixels = the `prob` conv evaluated only there,
 * softmax / soft-argmax, depth-guided fusion; network_v5.py:449-465) writing the MLP inputs as bf16 hi/lo
 * (xfeat [B,P,32], xcat [B,P,96] columns 0..31); the per-point MLPs (network_v5.py:432-444,486-493) then run as 1x1
 * convolutions through adp_conv_tc_*; adp_colsum = sum over points (fixed-order, no atomics), adp_pose_gbias = per-env bias of
 * pose_mlp2's first layer, adp_rot_head = rotation MLP + Ortho6d2Mat (rotation_utils.py:18-27).
 * x11_format: ADP_LAYOUT_F16 (IEEE half instead of bf16) | ADP_LAYOUT_S2D (x11 stored [B,D/2,S/2,S/2,64], S even, see
 * adp_conv0_plan_create).
 * x11 == NULL selects the single-view mode (backbone + NOCS of one frame, network_v5.py:432-444): only xfeat is written. */
ADP_API int adp_decode_gather(const float* feat_ref, const float* feat_src, const float* Mw, const float* depths, const void* x11,
                      const int32_t* choose, const uint8_t* valid, const float* prob_w, float* depth, void* xfeat_hi,
                      void* xfeat_lo, void* xcat_hi, void* xcat_lo, float* dbg_logits, float* dbg_fused, int B, int S, int D,
                      int P, int x11_format, void* stream);
ADP_API int adp_colsum(const void* hi, const void* lo, const uint8_t* valid, float* out, int B, int P, int C, void* stream);
ADP_API int adp_pose_gbias(const float* gsum, const float* q0_w, const float* q0_b, const uint8_t* valid, float* gb, int B,
                           int P, void* stream);
ADP_API int adp_rot_head(const float* psum, const uint8_t* valid, const adp_decode_weights* w, float* R, float* r6, int B,
                         int P, void* stream);

/* --- controller observation + actor forward (SURVEY 8(f)-2): rl_pose.py:173-187 (get_observation: [N, T*11] pose/bbox
 * history ++ one_hot(step, T), from the device-resident queues of the view ring) and algo/ppo/ppo/module.py:24-34,89-91
 * (act_inference: Linear/activation stack, torch weight layout [out][in]).  dims[0] = T*12, dims[nlayers] = action width;
 * weights / biases: host arrays of nlayers device pointers.  activation: the hidden activation of get_activation()
 * (module.py:110-126): ADP_ACTOR_ELU (rl.yaml), _SELU, _RELU (also "crelu"), _LRELU, _TANH, _SIGMOID.  obs_out [N, T*12] may be NULL. */
#define ADP_ACTOR_ELU 0
#define ADP_ACTOR_SELU 1
#define ADP_ACTOR_RELU 2
#define ADP_ACTOR_LRELU 3
#define ADP_ACTOR_TANH 4
#define ADP_ACTOR_SIGMOID 5
ADP_API int adp_actor_forward(const double* pose_queue, const double* bbox_queue, int T, int N, int step, int nlayers,
                              const int32_t* dims, const float* const* weights, const float* const* biases, int activation,
                              float* obs_out, float* act_out, void* stream);

/* --- pose fit + box: utils.py:40-119, interface_v5.py:318-321,354-374 ---------------------------------------- */
/* One 4-CTA thread-block cluster per environment; the exact-median radix select recomputes the pair ratios in every pass.
 * Points mode (pts_cam != NULL; branch C): the camera-frame points are given ([B,P,3], the first pts_count[b] valid, `nocs` in
 * the same order) instead of being back-projected from depth / choose / Kp; `scale` is the result of interest. */
ADP_API int adp_fit(const float* nocs, const float* depth, const int32_t* choose, const double* Kp, const float* R,
            const double* E, const uint8_t* valid, double* bbox, double* scale, double* trans, const float* pts_cam,
            const int32_t* pts_count, int B, int P, int S, void* stream);

/* --- pose fit, branch C, device part: utils.py:121-195 (depth_estimation_from_nocs_matches) -------------------------------
 * Per env: mutual nearest neighbours of the two views' NOCS maps (1024 x 1024, np.argmin tie rule), distance < 0.01, epipolar
 * filter |x1^T F x2| < 1 px (F from the UNCROPPED K and the two extrinsics, interface_v5.py:340-343), linear triangulation
 * (the DLT of cv2.triangulatePoints) and the transform into the view-1 camera frame.  Outputs: pts2d1 [B,P,2] (image
 * coordinates of every sampled view-1 pixel, interface_v5.py:136-145: the 2-D side of the PnP), pts_cam / nocs_m [B,P,3]
 * (matched points, compacted in ascending view-1 index), count [B], match_ids [B,P,2] (view-1 / view-2 index pairs; optional).
 * The median scale then comes from adp_fit in points mode; cv2.solvePnPRansac (align.py:104-115) stays a host call. */
ADP_API int adp_nocs_match(const float* nocs1, const float* nocs2, const int32_t* choose1, const int32_t* choose2,
                           const int32_t* win1, const int32_t* win2, const double* K, const double* E1, const double* E2,
                           const uint8_t* valid, int S, float* pts2d1, float* pts_cam, float* nocs_m, int32_t* count,
                           int32_t* match_ids, int B, int P, void* stream);

/* --- transformer variant: lib/fusion.py:11-82 (ViewFusion, 4 cross-view attention blocks, d = 32, 4 heads, 1024 tokens per view)
 * and the depth MLP of lib/network_baseline.py:555-562,631-643 (StereoPoseNet_with_depth_baseline; train.py:242-244) -----------
 * feat1/feat2 [B,S*S,32] fp32 channels-last feature maps, choose1/choose2 [B,P] sampled pixels (tokens = gathered features,
 * network_baseline.py:616-626).  blocks: [n_blocks][2 directions (fusion1, fusion2)][4 linears (q,k,v,out)][32*32 weight (out,in)
 * + 32 bias] fp32; depth_w: depth_head.0 weight [64][32], bias [64], depth_head.2 weight TRANSPOSED [64][32], bias [32],
 * depth_head.4 weight [32], bias [1].  scratch: 4 * B*P*32 floats.  Outputs: depth1 [B,P] (metres; required), depth2 / fused1 /
 * fused2 ([B,P,32] fp32 tokens after the last block) optional, xcat_hi/lo optional bf16 planes [B,P,96] whose columns 0..31 receive
 * the view-1 tokens (input of pose_mlp1).  Environments with valid[b] == 0 get zeros. */
ADP_API int adp_view_fusion(const float* feat1, const float* feat2, const int32_t* choose1, const int32_t* choose2,
                            const uint8_t* valid, const float* blocks, const float* depth_w, float* scratch, float* depth1,
                            float* depth2, void* xcat_hi, void* xcat_lo, float* fused1, float* fused2, int B, int S, int P,
                            int n_blocks, void* stream);

/* --- pose fit, branch B: align.py:44-102 (RANSAC + Umeyama), interface_v5.py:322-338 --------------------------
 * rand_idx: [B,128,5] sample indices (NULL = counter-based hash of `seed`); rot [B,9], trans [B,3], scale [B] optional. */
ADP_API int adp_fit_umeyama(const float* nocs, const float* depth, const int32_t* choose, const double* Kp, const double* E,
                    const uint8_t* valid, const int32_t* rand_idx, uint32_t seed, double* bbox, double* scale, double* rot,
                    double* trans, int B, int P, int S, void* stream);

#ifdef __cplusplus
}
#endif
#endif
