// Entry points of the stage translation units, called by the C ABI in api.cu.  Each defining .cu file includes this header, so
// the compiler checks every declaration against its definition.  The tcgen05 conv's entry points are in tc_conv.cuh.
#pragma once
#include "../../include/adapose_b200.h"
#include "common.cuh"

namespace adp {

// backbone_misc.cu
int maxpool3x3s2(const Act& in, const Act& out, int batch, cudaStream_t stream);
int psp_priors(const Act& feat, int feat_cs, const float* w, float* pooled, float* priors, int batch, cudaStream_t stream);
int psp_fill_priors(const float* priors, const Act& out, int coff, int batch, cudaStream_t stream);
int upsample2x(const Act& in, const Act& out, int batch, cudaStream_t stream);
int upconv_blend(const Act& q, const Act& out, const float* bias, float slope, int batch, cudaStream_t stream);
int pack_s2d(const float* crops, const Act& out, int batch, int S, cudaStream_t stream);

// preprocess.cu
int preprocess_run(const void* rgb, int rgb_dt, const void* mask, int mask_dt, const double* K, int k_stride, int F, int H, int W,
                   int S, int P, uint32_t seed, int choose_mode, int frame_id0, int* bbox_ws, int* win, double* Kp, uint8_t* valid,
                   float* crops, int* choose, int* counts, cudaStream_t stream);
int mask_windows_run(const void* mask, int mask_dt, int F, int H, int W, int* bbox_ws, int* win, uint8_t* valid, cudaStream_t stream);

// volume.cu
int build_volume(const void* f_ref, const void* f_src, const float* Mw, const float* depths, bf16* vol, int B, int D, int H,
                 int W, int C, int f16, cudaStream_t stream);
int warp_matrices(const double* Kp_ref, const double* E_ref, const double* Kp_src, const double* E_src, float* Mw,
                  const uint8_t* valid_ref, const uint8_t* valid_src, uint8_t* valid_env, int B, cudaStream_t stream);

// conv0_ring.cu: flags as in adp_conv0_plan_create
struct Conv0Plan;
Conv0Plan* conv0_alloc();
void conv0_release(Conv0Plan* p);
int conv0_plan(Conv0Plan* pl, const Act& in, const uint16_t* w_packed, const float* scale, const float* shift, uint16_t* out,
               int flags, int num_sms);
int conv0_run(Conv0Plan* pl, int batch, int* err_flag, cudaStream_t stream);

// tconv_fused.cu: flags as in adp_tconv_plan_create
struct TconvPlan;
TconvPlan* tconv_alloc();
void tconv_release(TconvPlan* p);
int tconv_plan(TconvPlan* pl, const Act& in, const bf16* w, int Cout, const float* scale, const float* bias, const bf16* res,
               int res_cs, bf16* out, int flags, int num_sms);
int tconv_run(TconvPlan* pl, int batch, int* err_flag, cudaStream_t stream);

// decode.cu
int decode_gather_c(const float* feat_ref, const float* feat_src, const float* Mw, const float* depths, const void* x11,
                    const int* choose, const uint8_t* valid, const float* prob_w, float* depth, void* xfeat_hi, void* xfeat_lo,
                    void* xcat_hi, void* xcat_lo, float* dbg_logits, float* dbg_fused, int B, int S, int D, int P, int x11_f16,
                    cudaStream_t stream);
int colsum_run(const bf16* hi, const bf16* lo, const uint8_t* valid, float* out, int B, int P, int C, cudaStream_t stream);
int pose_gbias_run(const float* gsum, const float* q0_w, const float* q0_b, const uint8_t* valid, float* gb, int B, int P,
                   cudaStream_t stream);
int rot_head_run(const float* psum, const uint8_t* valid, float* Rout, float* r6out, const adp_decode_weights* cw, int B, int P,
                 cudaStream_t stream);

// actor.cu
constexpr int ACT_MAXL = 8;         // layers of the actor MLP
struct ActorArgs {
    const double* pose;      // [T, N, 7]
    const double* bbox;      // [T, N, 4]
    int T, N, step;          // step = accumulate_steps - 1 (one-hot index)
    int nlayers;
    int activation;          // hidden activation, get_activation() of module.py:110-126: 0 elu, 1 selu, 2 relu/crelu, 3 lrelu, 4 tanh, 5 sigmoid
    int dims[ACT_MAXL + 1];  // dims[0] = T * 12
    const float* W[ACT_MAXL];   // torch layout [out][in]
    const float* b[ACT_MAXL];
    float* obs_out;          // [N, dims[0]] or nullptr
    float* act_out;          // [N, dims[nlayers]]
};
int actor_forward(const ActorArgs& a, cudaStream_t stream);

// fit.cu
int fit_run(const float* nocs, const float* depth, const int* choose, const double* Kp, const float* R, const double* E,
            const uint8_t* valid, double* bbox, double* scale_out, double* trans_out, const float* pts_cam, const int* pts_count,
            int B, int P, int S, cudaStream_t stream);

// fit_umeyama.cu
int fit_umeyama_run(const float* nocs, const float* depth, const int* choose, const double* Kp, const double* E, const uint8_t* valid,
                    const int* rand_idx, uint32_t seed, double* bbox, double* scale_out, double* rot_out, double* trans_out, int B,
                    int P, int S, cudaStream_t stream);

// nocs_match.cu
int nocs_match_run(const float* nocs1, const float* nocs2, const int* choose1, const int* choose2, const int* win1, const int* win2,
                   const double* K, const double* E1, const double* E2, const uint8_t* valid, int S, float* pts2d1, float* pts_cam,
                   float* nocs_m, int* count, int* match_ids, int B, int P, cudaStream_t stream);

// view_fusion.cu
int view_fusion_run(const float* feat1, const float* feat2, const int* choose1, const int* choose2, const uint8_t* valid,
                    const float* blocks, const float* depth_w, float* scratch, float* depth1, float* depth2, bf16* xcat_hi,
                    bf16* xcat_lo, float* fused1, float* fused2, int B, int S, int P, int n_blocks, cudaStream_t stream);

}  // namespace adp
