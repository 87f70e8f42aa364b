// extern "C" surface of libadapose_b200.so (see include/adapose_b200.h).
#include <stdarg.h>

#include <atomic>
#include <mutex>

#include "../../include/adapose_b200.h"
#include "common.cuh"
#include "tc_conv.cuh"

namespace adp {

static thread_local char g_err[1024] = "";
static std::atomic<uint64_t> g_launches{0};

void set_last_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

// implemented in the stage translation units
int maxpool3x3s2(const Act& in, const Act& out, int batch, cudaStream_t stream);
int psp_priors(const Act& feat, int feat_cs, const float* w, float* pooled, float* priors, int batch, cudaStream_t stream);
int psp_fill_priors(const float* priors, const Act& out, int coff, int batch, cudaStream_t stream);
int upsample2x(const Act& in, const Act& out, int batch, cudaStream_t stream);
int upconv_blend(const Act& q, const Act& out, const float* bias, float slope, int batch, cudaStream_t stream);
int pack_s2d(const float* crops, const Act& out, int batch, int S, cudaStream_t stream);
int preprocess_run(const void* rgb, int rgb_dt, const void* mask, int mask_dt, const double* K, int k_stride, int F, int H, int W,
                   int S, int P, uint32_t seed, int choose_mode, int frame_id0, int* bbox_ws, int* win, double* Kp, uint8_t* valid,
                   float* crops, int* choose, int* counts, cudaStream_t stream);
int mask_windows_run(const void* mask, int mask_dt, int F, int H, int W, int* bbox_ws, int* win, uint8_t* valid, cudaStream_t stream);
int build_volume(const void* f_ref, const void* f_src, const float* Mw, const float* depths, bf16* vol, int B, int D, int H,
                 int W, int C, int f16, cudaStream_t stream);
int warp_matrices(const double* Kp_ref, const double* E_ref, const double* Kp_src, const double* E_src, float* Mw,
                  const uint8_t* valid_ref, const uint8_t* valid_src, uint8_t* valid_env, int B, cudaStream_t stream);
int fit_run(const float* nocs, const float* depth, const int* choose, const double* Kp, const float* R, const double* E,
            const uint8_t* valid, double* bbox, double* scale_out, double* trans_out, const float* pts_cam, const int* pts_count,
            int B, int P, int S, cudaStream_t stream);
int nocs_match_run(const float* nocs1, const float* nocs2, const int* choose1, const int* choose2, const int* win1, const int* win2,
                   const double* K, const double* E1, const double* E2, const uint8_t* valid, int S, float* pts2d1, float* pts_cam,
                   float* nocs_m, int* count, int* match_ids, int B, int P, cudaStream_t stream);
int view_fusion_run(const float* feat1, const float* feat2, const int* choose1, const int* choose2, const uint8_t* valid,
                    const float* blocks, const float* depth_w, float* scratch, float* depth1, float* depth2, bf16* xcat_hi,
                    bf16* xcat_lo, float* fused1, float* fused2, int B, int S, int P, int n_blocks, cudaStream_t stream);

int fit_umeyama_run(const float* nocs, const float* depth, const int* choose, const double* Kp, const double* E, const uint8_t* valid,
                    const int* rand_idx, uint32_t seed, double* bbox, double* scale_out, double* rot_out, double* trans_out, int B,
                    int P, int S, cudaStream_t stream);
struct Conv0Plan;
Conv0Plan* conv0_alloc();
void conv0_release(Conv0Plan* p);
int conv0_plan(Conv0Plan* pl, const Act& in, const uint16_t* w_packed, const float* scale, const float* shift, uint16_t* out,
               int planar, int num_sms);
int conv0_run(Conv0Plan* pl, int batch, int* err_flag, cudaStream_t stream);

int decode_gather_c(const float* feat_ref, const float* feat_src, const float* Mw, const float* depths, const void* x11,
                    const int* choose, const uint8_t* valid, const float* prob_w, float* depth, void* xfeat_hi, void* xfeat_lo,
                    void* xcat_hi, void* xcat_lo, float* dbg_logits, float* dbg_fused, int B, int S, int D, int P, int x11_f16,
                    cudaStream_t stream);
int colsum_run(const bf16* hi, const bf16* lo, const uint8_t* valid, float* out, int B, int P, int C, cudaStream_t stream);
int pose_gbias_run(const float* gsum, const float* q0_w, const float* q0_b, const uint8_t* valid, float* gb, int B, int P,
                   cudaStream_t stream);
int rot_head_run(const float* psum, const uint8_t* valid, float* Rout, float* r6out, const adp_decode_weights* cw, int B, int P,
                 cudaStream_t stream);
constexpr int ACT_MAXL_API = 8;
struct ActorArgs {
    const double* pose; const double* bbox; int T, N, step; int nlayers; int activation; int dims[ACT_MAXL_API + 1];
    const float* W[ACT_MAXL_API]; const float* b[ACT_MAXL_API]; float* obs_out; float* act_out;
};
int actor_forward(const ActorArgs& a, cudaStream_t stream);
struct TconvPlan;
TconvPlan* tconv_alloc();
void tconv_release(TconvPlan* p);
int tconv_plan(TconvPlan* pl, const Act& in, const bf16* w, int Cout, const float* scale, const float* bias, const bf16* res,
               int res_cs, bf16* out, int flags, int num_sms);
int tconv_run(TconvPlan* pl, int batch, int* err_flag, cudaStream_t stream);

static Act to_act(const adp_act* a) {
    Act r;
    r.hi = reinterpret_cast<bf16*>(a->hi);
    r.lo = reinterpret_cast<bf16*>(a->lo);
    r.B = a->B; r.D = a->D; r.H = a->H; r.W = a->W; r.C = a->C; r.f16 = a->f16;
    r.q8 = reinterpret_cast<uint8_t*>(a->q8);
    return r;
}

}  // namespace adp

struct adp_conv_plan {
    adp::TcConvLayer layer;
    int num_sms;
};

using namespace adp;

extern "C" {

int adp_abi_version(void) { return ADP_ABI_VERSION; }
const char* adp_last_error(void) { return g_err; }
uint64_t adp_launch_count(void) { return g_launches.load(); }
void adp_launch_count_add(uint64_t n) { g_launches += n; }

int adp_device_info(int device, int* num_sms, int* cc_major, int* cc_minor) {
    cudaDeviceProp prop;
    ADP_CUDA(cudaGetDeviceProperties(&prop, device));
    if (num_sms) *num_sms = prop.multiProcessorCount;
    if (cc_major) *cc_major = prop.major;
    if (cc_minor) *cc_minor = prop.minor;
    return ADP_OK;
}

int adp_preprocess(const void* rgb, int rgb_dtype, const void* mask, int mask_dtype, const double* K, int k_stride, int F, int H,
                   int W, int S, int P, uint32_t seed, int choose_mode, int frame_id0, int32_t* bbox_ws, int32_t* win, double* Kp,
                   uint8_t* valid, float* crops, int32_t* choose, int32_t* counts, void* stream) {
    ADP_CHECK_ARG(rgb && mask && K && bbox_ws && win && Kp && valid && crops && choose && counts, "null pointer");
    g_launches += 5;
    return preprocess_run(rgb, rgb_dtype, mask, mask_dtype, K, k_stride, F, H, W, S, P, seed, choose_mode, frame_id0, bbox_ws, win, Kp,
                          valid, crops, choose, counts, (cudaStream_t)stream);
}

int adp_mask_windows(const void* mask, int mask_dtype, int F, int H, int W, int32_t* bbox_ws, int32_t* win, uint8_t* valid, void* stream) {
    ADP_CHECK_ARG(mask && bbox_ws && win && valid, "null pointer");
    g_launches += 3;
    return mask_windows_run(mask, mask_dtype, F, H, W, bbox_ws, win, valid, (cudaStream_t)stream);
}

int adp_conv_tc_plan(adp_conv_plan** plan, const adp_act* in, const void* w_hi, const void* w_lo, int cout, int kd, int ks,
                     int dil, int npass, const adp_epilogue* ep, const adp_tc_geom* geom, int num_sms) {
    ADP_CHECK_ARG(plan && in && w_hi && ep, "null pointer");
    ADP_CHECK_ARG(ep->out_hi || ep->out_f32, "epilogue has no output");
    adp_conv_plan* pl = new adp_conv_plan();
    TcGeom g;
    if (geom) {
        g.ntaps = geom->ntaps;
        for (int t = 0; t < 32; ++t) { g.dz[t] = geom->dz[t]; g.dy[t] = geom->dy[t]; g.dx[t] = geom->dx[t]; g.wt[t] = geom->wt[t]; }
        g.in_mul = geom->in_mul; g.out_mul = geom->out_mul; g.out_oz = geom->out_oz; g.out_oy = geom->out_oy; g.out_ox = geom->out_ox;
        g.gD = geom->gD; g.gH = geom->gH; g.gW = geom->gW; g.oD = geom->oD; g.oH = geom->oH; g.oW = geom->oW; g.w_taps = geom->w_taps;
    }
    int r = tc_conv_plan(&pl->layer, to_act(in), reinterpret_cast<const bf16*>(w_hi), reinterpret_cast<const bf16*>(w_lo), cout,
                         kd, ks, dil, npass, geom ? &g : nullptr, in->f16);
    if (r != ADP_OK) {
        delete pl;
        return r;
    }
    TcConvParams& p = pl->layer.p;
    p.bias = ep->bias; p.scale = ep->scale; p.prelu = ep->prelu; p.act = ep->act; p.res_after_act = ep->res_after_act;
    p.res_hi = reinterpret_cast<const bf16*>(ep->res_hi); p.res_lo = reinterpret_cast<const bf16*>(ep->res_lo);
    p.res_cs = ep->res_cstride ? ep->res_cstride : cout;
    p.out_hi = reinterpret_cast<bf16*>(ep->out_hi); p.out_lo = reinterpret_cast<bf16*>(ep->out_lo);
    p.out_f32 = ep->out_f32;
    p.out_h16 = reinterpret_cast<__half*>(ep->out_h16);
    p.out_q8 = reinterpret_cast<uint8_t*>(ep->out_q8);
    if (p.out_q8 && (pl->layer.BN < 32 || cout % 32 != 0 || ep->out_lo || !in->f16)) {
        set_last_error("out_q8 needs fp16 activations and Cout %% 32 == 0 (coalesced epilogue, 32-channel chunks)");
        delete pl;
        return ADP_ERR_ARG;
    }
    p.out_cs = ep->out_cstride ? ep->out_cstride : cout; p.out_coff = ep->out_coff; p.bias_per_batch = ep->bias_per_batch;
    p.check_finite = ep->check_finite;
    // coalesced epilogue stores need full accumulator chunks (bf16 hi + lo planes, fp32 / fp16 side outputs are fine)
    const int ch = pl->layer.BN < 32 ? pl->layer.BN : 32;
    p.coalesce = ((!ep->out_lo || !in->f16) && cout % ch == 0 && ((cout | p.out_cs | p.out_coff) & 7) == 0) ? 1 : 0;
    pl->num_sms = num_sms > 0 ? num_sms : 148;
    r = tc_conv_finish_plan(&pl->layer);
    if (r != ADP_OK) {
        delete pl;
        return r;
    }
    *plan = pl;
    return ADP_OK;
}

int adp_conv_tc_run(adp_conv_plan* plan, int batch, int32_t* err_flag, void* stream) {
    ADP_CHECK_ARG(plan, "null plan");
    plan->layer.p.err = err_flag;
    g_launches += 1;
    return tc_conv_launch(&plan->layer, batch, plan->num_sms, (cudaStream_t)stream);
}

void adp_conv_tc_free(adp_conv_plan* plan) { delete plan; }

int adp_maxpool3x3s2(const adp_act* in, const adp_act* out, int batch, void* stream) {
    ADP_CHECK_ARG(in && out, "null pointer");
    g_launches += 1;
    return maxpool3x3s2(to_act(in), to_act(out), batch, (cudaStream_t)stream);
}

int adp_psp_priors(const adp_act* feat, int feat_cstride, const float* w, float* pooled, float* priors, int batch, void* stream) {
    ADP_CHECK_ARG(feat && w && pooled && priors, "null pointer");
    g_launches += 2;
    return psp_priors(to_act(feat), feat_cstride, w, pooled, priors, batch, (cudaStream_t)stream);
}

int adp_psp_fill_priors(const float* priors, const adp_act* out, int coff, int batch, void* stream) {
    ADP_CHECK_ARG(priors && out, "null pointer");
    g_launches += 1;
    return psp_fill_priors(priors, to_act(out), coff, batch, (cudaStream_t)stream);
}

int adp_upsample2x(const adp_act* in, const adp_act* out, int batch, void* stream) {
    ADP_CHECK_ARG(in && out, "null pointer");
    g_launches += 1;
    return upsample2x(to_act(in), to_act(out), batch, (cudaStream_t)stream);
}

int adp_upconv_blend(const adp_act* q, const adp_act* out, const float* bias, float prelu_slope, int batch, void* stream) {
    ADP_CHECK_ARG(q && out && bias, "null pointer");
    g_launches += 1;
    return upconv_blend(to_act(q), to_act(out), bias, prelu_slope, batch, (cudaStream_t)stream);
}

int adp_conv0_plan_create(adp_conv0_plan** plan, const adp_act* vol, const void* w_packed, const float* scale, const float* shift,
                          void* out, int vol_planar, int num_sms) {
    ADP_CHECK_ARG(plan && vol && w_packed && scale && shift && out, "null pointer");
    Conv0Plan* pl = conv0_alloc();
    int r = conv0_plan(pl, to_act(vol), reinterpret_cast<const uint16_t*>(w_packed), scale, shift, reinterpret_cast<uint16_t*>(out),
                       vol_planar, num_sms);
    if (r != ADP_OK) {
        conv0_release(pl);
        return r;
    }
    *plan = reinterpret_cast<adp_conv0_plan*>(pl);
    return ADP_OK;
}

int adp_conv0_run(adp_conv0_plan* plan, int batch, int32_t* err_flag, void* stream) {
    ADP_CHECK_ARG(plan, "null plan");
    g_launches += 1;
    return conv0_run(reinterpret_cast<Conv0Plan*>(plan), batch, err_flag, (cudaStream_t)stream);
}

void adp_conv0_free(adp_conv0_plan* plan) { conv0_release(reinterpret_cast<Conv0Plan*>(plan)); }

int adp_tconv_plan_create(adp_tconv_plan** plan, const adp_act* in, const void* w, int cout, const float* scale, const float* bias,
                          const void* res, int res_cstride, void* out, int flags, int num_sms) {
    ADP_CHECK_ARG(plan && in && w && scale && bias && out, "null pointer");
    TconvPlan* pl = tconv_alloc();
    int r = tconv_plan(pl, to_act(in), reinterpret_cast<const bf16*>(w), cout, scale, bias, reinterpret_cast<const bf16*>(res),
                       res_cstride, reinterpret_cast<bf16*>(out), flags, num_sms);
    if (r != ADP_OK) {
        tconv_release(pl);
        return r;
    }
    *plan = reinterpret_cast<adp_tconv_plan*>(pl);
    return ADP_OK;
}

int adp_tconv_run(adp_tconv_plan* plan, int batch, int32_t* err_flag, void* stream) {
    ADP_CHECK_ARG(plan, "null plan");
    g_launches += 1;
    return tconv_run(reinterpret_cast<TconvPlan*>(plan), batch, err_flag, (cudaStream_t)stream);
}

void adp_tconv_free(adp_tconv_plan* plan) { tconv_release(reinterpret_cast<TconvPlan*>(plan)); }

int adp_pack_s2d(const float* crops, const adp_act* out, int batch, int S, void* stream) {
    ADP_CHECK_ARG(crops && out, "null pointer");
    g_launches += 1;
    return pack_s2d(crops, to_act(out), batch, S, (cudaStream_t)stream);
}

int adp_build_volume(const void* feat_ref, const void* feat_src, const float* Mw, const float* depths, void* vol, int B, int D,
                     int H, int W, int C, int f16, void* stream) {
    ADP_CHECK_ARG(feat_ref && feat_src && Mw && depths && vol, "null pointer");
    g_launches += 1;
    return build_volume(feat_ref, feat_src, Mw, depths, reinterpret_cast<bf16*>(vol), B, D, H, W, C, f16, (cudaStream_t)stream);
}

int adp_warp_matrices(const double* Kp_ref, const double* E_ref, const double* Kp_src, const double* E_src, float* Mw,
                      const uint8_t* valid_ref, const uint8_t* valid_src, uint8_t* valid_env, int B, void* stream) {
    ADP_CHECK_ARG(Kp_ref && E_ref && Kp_src && E_src && Mw, "null pointer");
    g_launches += 1;
    return warp_matrices(Kp_ref, E_ref, Kp_src, E_src, Mw, valid_ref, valid_src, valid_env, B, (cudaStream_t)stream);
}

int adp_decode_gather(const float* feat_ref, const float* feat_src, const float* Mw, const float* depths, const void* x11,
                      const int32_t* choose, const uint8_t* valid, const float* prob_w, float* depth, void* xfeat_hi, void* xfeat_lo,
                      void* xcat_hi, void* xcat_lo, float* dbg_logits, float* dbg_fused, int B, int S, int D, int P, int x11_f16,
                      void* stream) {
    ADP_CHECK_ARG(feat_ref && choose && xfeat_hi, "null pointer");
    ADP_CHECK_ARG(!x11 || (feat_src && Mw && depths && prob_w && depth && xcat_hi), "null pointer (stereo mode)");
    g_launches += 1;
    return decode_gather_c(feat_ref, feat_src, Mw, depths, x11, choose, valid, prob_w, depth, xfeat_hi, xfeat_lo, xcat_hi, xcat_lo,
                           dbg_logits, dbg_fused, B, S, D, P, x11_f16, (cudaStream_t)stream);
}

int adp_colsum(const void* hi, const void* lo, const uint8_t* valid, float* out, int B, int P, int C, void* stream) {
    ADP_CHECK_ARG(hi && out, "null pointer");
    g_launches += 1;
    return colsum_run(reinterpret_cast<const bf16*>(hi), reinterpret_cast<const bf16*>(lo), valid, out, B, P, C, (cudaStream_t)stream);
}

int adp_pose_gbias(const float* gsum, const float* q0_w, const float* q0_b, const uint8_t* valid, float* gb, int B, int P, void* stream) {
    ADP_CHECK_ARG(gsum && q0_w && q0_b && gb, "null pointer");
    g_launches += 1;
    return pose_gbias_run(gsum, q0_w, q0_b, valid, gb, B, P, (cudaStream_t)stream);
}

int adp_rot_head(const float* psum, const uint8_t* valid, const adp_decode_weights* w, float* R, float* r6, int B, int P, void* stream) {
    ADP_CHECK_ARG(psum && w && R, "null pointer");
    g_launches += 1;
    return rot_head_run(psum, valid, R, r6, w, B, P, (cudaStream_t)stream);
}

int adp_actor_forward(const double* pose_queue, const double* bbox_queue, int T, int N, int step, int nlayers, const int32_t* dims,
                      const float* const* weights, const float* const* biases, int activation, float* obs_out, float* act_out,
                      void* stream) {
    ADP_CHECK_ARG(pose_queue && bbox_queue && dims && weights && biases && act_out, "null pointer");
    ADP_CHECK_ARG(nlayers >= 1 && nlayers <= ACT_MAXL_API, "1..8 layers");
    ActorArgs a{};
    a.pose = pose_queue; a.bbox = bbox_queue; a.T = T; a.N = N; a.step = step; a.nlayers = nlayers; a.activation = activation;
    for (int l = 0; l <= nlayers; ++l) a.dims[l] = dims[l];
    for (int l = 0; l < nlayers; ++l) { a.W[l] = weights[l]; a.b[l] = biases[l]; }
    a.obs_out = obs_out; a.act_out = act_out;
    g_launches += 1;
    return actor_forward(a, (cudaStream_t)stream);
}

int adp_fit(const float* nocs, const float* depth, const int32_t* choose, const double* Kp, const float* R, const double* E,
            const uint8_t* valid, double* bbox, double* scale, double* trans, const float* pts_cam, const int32_t* pts_count, int B,
            int P, int S, void* stream) {
    ADP_CHECK_ARG(nocs && Kp && R && E && bbox && (pts_cam || (depth && choose)), "null pointer");
    g_launches += 1;
    return fit_run(nocs, depth, choose, Kp, R, E, valid, bbox, scale, trans, pts_cam, pts_count, B, P, S, (cudaStream_t)stream);
}

int adp_nocs_match(const float* nocs1, const float* nocs2, const int32_t* choose1, const int32_t* choose2, const int32_t* win1,
                   const int32_t* win2, const double* K, const double* E1, const double* E2, const uint8_t* valid, int S,
                   float* pts2d1, float* pts_cam, float* nocs_m, int32_t* count, int32_t* match_ids, int B, int P, void* stream) {
    ADP_CHECK_ARG(nocs1 && nocs2 && choose1 && choose2 && win1 && win2 && K && E1 && E2 && pts2d1 && pts_cam && nocs_m && count,
                  "null pointer");
    g_launches += 1;
    return nocs_match_run(nocs1, nocs2, choose1, choose2, win1, win2, K, E1, E2, valid, S, pts2d1, pts_cam, nocs_m, count, match_ids,
                          B, P, (cudaStream_t)stream);
}

int adp_view_fusion(const float* feat1, const float* feat2, const int32_t* choose1, const int32_t* choose2, const uint8_t* valid,
                    const float* blocks, const float* depth_w, float* scratch, float* depth1, float* depth2, void* xcat_hi,
                    void* xcat_lo, float* fused1, float* fused2, int B, int S, int P, int n_blocks, void* stream) {
    ADP_CHECK_ARG(feat1 && feat2 && choose1 && choose2 && blocks && depth_w && scratch && depth1, "null pointer");
    ADP_CHECK_ARG((xcat_hi == nullptr) == (xcat_lo == nullptr), "xcat planes come in pairs");
    g_launches += n_blocks;
    return view_fusion_run(feat1, feat2, choose1, choose2, valid, blocks, depth_w, scratch, depth1, depth2,
                           reinterpret_cast<bf16*>(xcat_hi), reinterpret_cast<bf16*>(xcat_lo), fused1, fused2, B, S, P, n_blocks,
                           (cudaStream_t)stream);
}

int adp_fit_umeyama(const float* nocs, const float* depth, const int32_t* choose, const double* Kp, const double* E,
                    const uint8_t* valid, const int32_t* rand_idx, uint32_t seed, double* bbox, double* scale, double* rot,
                    double* trans, int B, int P, int S, void* stream) {
    ADP_CHECK_ARG(nocs && depth && choose && Kp && E && bbox, "null pointer");
    g_launches += 1;
    return fit_umeyama_run(nocs, depth, choose, Kp, E, valid, rand_idx, seed, bbox, scale, rot, trans, B, P, S, (cudaStream_t)stream);
}

}  // extern "C"
