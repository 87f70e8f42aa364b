"""Helpers for the -m gpu parity tests: raw calls through the C ABI on torch-allocated device buffers."""
import ctypes as C

import numpy as np
import torch

from rgbmanip_b200 import _lib as L

DEV = "cuda:0"


def stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def split(x: torch.Tensor, with_lo=True):
    """fp32 channels-last tensor -> (hi, lo) bf16 device planes."""
    hi = x.to(torch.bfloat16)
    lo = (x - hi.float()).to(torch.bfloat16) if with_lo else None
    return hi.to(DEV).contiguous(), (lo.to(DEV).contiguous() if with_lo else None)


def act(hi, lo, B, D, H, W, Cn, f16=0, q8=None):
    return L.Act(L.ptr(hi), L.ptr(lo), B, D, H, W, Cn, f16, L.ptr(q8))


def to_e4m3(x):
    """fp32 -> e4m3 bytes (saturating), as a uint8 tensor; from_e4m3 is the inverse."""
    return x.clamp(-448.0, 448.0).to(torch.float8_e4m3fn).view(torch.uint8)


def from_e4m3(u):
    return u.view(torch.float8_e4m3fn).float()


def val(hi, lo):
    v = hi.float()
    return (v + lo.float()) if lo is not None else v


def to_cl(x):
    """NCHW / NCDHW -> channels-last contiguous."""
    if x.dim() == 4:
        return x.permute(0, 2, 3, 1).contiguous()
    return x.permute(0, 2, 3, 4, 1).contiguous()


def from_cl(x):
    if x.dim() == 4:
        return x.permute(0, 3, 1, 2).contiguous()
    return x.permute(0, 4, 1, 2, 3).contiguous()


def epilogue(out_hi=None, out_lo=None, out_f32=None, scale=None, bias=None, act_code=L.ACT_NONE, prelu=0.0, res_hi=None,
             res_lo=None, res_after_act=0, out_q8=None, *, res_cstride=0, out_h16=None, out_cstride=0, out_coff=0, bias_per_batch=0,
             check_finite=0):
    """Every field of adp_epilogue (include/adapose_b200.h); tensors may be None."""
    return L.Epilogue(L.ptr(scale), L.ptr(bias), float(prelu), act_code, res_after_act, L.ptr(res_hi), L.ptr(res_lo), res_cstride,
                      L.ptr(out_hi), L.ptr(out_lo), L.ptr(out_f32), L.ptr(out_h16), out_cstride, out_coff, bias_per_batch,
                      L.ptr(out_q8), check_finite)


def plan_info(plan):
    """adp_conv_tc_plan_info as a dict: the kernel instance a plan chose and its tiling."""
    info = (C.c_int32 * L.TC_PLAN_INFO_LEN)()
    L.check(L.load().adp_conv_tc_plan_info(plan, info), "plan_info")
    keys = ("row", "slab_ctas", "bulk", "fused", "BN", "KC", "npass", "TW", "TH", "coalesce", "tiles_x", "tiles_y", "tiles_n", "D",
            "kchunks", "ntaps")
    d = dict(zip(keys, list(info)))
    d["instance"] = (d["slab_ctas"], d["bulk"], d["fused"], d["BN"], d["KC"])
    return d


def rel_err(a, b):
    a, b = a.double().cpu(), b.double().cpu()
    return float((a - b).abs().max() / (b.abs().max() + 1e-30))


# ------------------------------------------------------------------------------------------------ per-element comparison
CANARY16, CANARY8 = 0x7E5A, 0x5A       # fill bits of output buffers: a 16-bit NaN / an fp8 byte no kernel computes here
CANARY32 = 0x7FC00000                   # the fp32 quiet NaN torch writes for float("nan")


def ulp(r, fmt):
    """One unit in the last place of `fmt` at |r| (normal range; the smallest normal's ulp below it)."""
    mant, emin = {"f16": (10, -14), "bf16": (7, -126)}[fmt]
    _, e = torch.frexp(r.abs())
    e = torch.where(r != 0, e - 1, torch.full_like(e, emin)).clamp_min(emin)
    return torch.pow(2.0, (e - mant).double())


def assert_close(got, ref, fmt, slack, what):
    """Per element: |got - ref| <= slack (+ one ulp of a 16-bit format at |ref|, or 2^-16 |ref| for a bf16 hi + lo pair).
    slack is a number or a tensor that broadcasts against ref.  Returns the largest error as a fraction of its bound."""
    got = got.double()
    err = (got - ref).abs()
    bound = torch.zeros_like(ref) + slack
    if fmt in ("f16", "bf16"):
        bound = bound + ulp(ref, fmt)
    elif fmt == "bf16x2":
        bound = bound + ref.abs() * 2.0 ** -16
    bad = ~(err <= bound)
    if bad.any():
        i = int(torch.nonzero(bad.reshape(-1))[0])
        raise AssertionError(f"{what}: {int(bad.sum())} of {bad.numel()} elements out of bound; first at index "
                             f"{tuple(np.unravel_index(i, tuple(ref.shape)))}: got {float(got.reshape(-1)[i])}, "
                             f"ref {float(ref.reshape(-1)[i])}, bound {float(bound.reshape(-1)[i])}")
    return float((err / bound).max())


def bits(t):
    """The raw bits of a tensor as an integer tensor of the same element size, on the CPU (NaN canaries compare equal)."""
    return t.view({1: torch.uint8, 2: torch.int16, 4: torch.int32}[t.element_size()]).cpu()


def canary16(shape, dt):
    return torch.full(shape, CANARY16, dtype=torch.int16, device=DEV).view(dt)


def canary32(shape):
    return torch.full(shape, CANARY32, dtype=torch.int32, device=DEV).view(torch.float32)


# ------------------------------------------------------------------------------------------------ thin runners of the
# cost-regularisation kernels: the caller owns every buffer (so it can pre-fill canaries); batch < the plan's B runs part of it
def _err_flag(err):
    return torch.zeros(2, dtype=torch.int32, device=DEV) if err is None else err


def conv0(vol, w_packed, scale, shift, out, *, flags=0, num_sms=148, batch=None, err=None):
    """adp_conv0_plan_create + adp_conv0_run.  vol: device [B,D,H,W,32] fp16 or bf16 (its dtype sets the format); w_packed:
    rgbmanip_b200.geometry.conv0_ring_weights in the same dtype; scale / shift: device fp32 [8]; out: [B,D,H,W,16] or, with
    flags = LAYOUT_S2D, [B,D/2,H/2,W/2,64].  The plan holds B = vol.shape[0] images and runs `batch` of them."""
    lib = L.load()
    B, D, H, W, Cn = vol.shape
    err = _err_flag(err)
    a = act(vol, None, B, D, H, W, Cn, int(vol.dtype == torch.float16))
    plan = C.c_void_p()
    L.check(lib.adp_conv0_plan_create(C.byref(plan), C.byref(a), L.ptr(w_packed), L.ptr(scale), L.ptr(shift), L.ptr(out), flags,
                                      num_sms), "conv0 plan")
    try:
        L.check(lib.adp_conv0_run(plan, B if batch is None else batch, L.ptr(err), stream()), "conv0 run")
        torch.cuda.synchronize()
    finally:
        lib.adp_conv0_free(plan)
    assert int(err[0].item()) == 0, f"watchdog code {int(err[0].item())}"
    return out


def tconv(x, w, cout, scale, bias, res, out, *, res_cstride=0, flags=0, num_sms=148, batch=None, err=None):
    """adp_tconv_plan_create + adp_tconv_run.  x: device [B,D,H,W,Cin] fp16 or bf16; w: [27, pad16(cout), Cin] in the same
    dtype; scale / bias: device fp32 [cout]; res: the skip tensor or None; out: [B,2D,2H,2W,cout] (or the s2d layout with
    flags = LAYOUT_S2D).  The plan holds B = x.shape[0] images and runs `batch` of them."""
    lib = L.load()
    B, D, H, W, Cn = x.shape
    err = _err_flag(err)
    a = act(x, None, B, D, H, W, Cn, int(x.dtype == torch.float16))
    plan = C.c_void_p()
    L.check(lib.adp_tconv_plan_create(C.byref(plan), C.byref(a), L.ptr(w), cout, L.ptr(scale), L.ptr(bias), L.ptr(res), res_cstride,
                                      L.ptr(out), flags, num_sms), "tconv plan")
    try:
        L.check(lib.adp_tconv_run(plan, B if batch is None else batch, L.ptr(err), stream()), "tconv run")
        torch.cuda.synchronize()
    finally:
        lib.adp_tconv_free(plan)
    assert int(err[0].item()) == 0, f"watchdog code {int(err[0].item())}"
    return out


def decode_gather(feat_ref, feat_src, Mw, depths, x11, choose, valid, prob_w, outs, *, batch, S, P, x11_format, D=24):
    """adp_decode_gather over `batch` environments.  outs: dict of the caller's device buffers depth, xfeat_hi, xfeat_lo,
    xcat_hi, xcat_lo, dbg_logits, dbg_fused (a missing key passes NULL).  x11 = None selects the single-view mode.  The kernel
    has no pipeline and takes no error flag."""
    lib = L.load()
    o = {k: L.ptr(outs.get(k)) for k in ("depth", "xfeat_hi", "xfeat_lo", "xcat_hi", "xcat_lo", "dbg_logits", "dbg_fused")}
    L.check(lib.adp_decode_gather(L.ptr(feat_ref), L.ptr(feat_src), L.ptr(Mw), L.ptr(depths), L.ptr(x11), L.ptr(choose), L.ptr(valid),
                                  L.ptr(prob_w), o["depth"], o["xfeat_hi"], o["xfeat_lo"], o["xcat_hi"], o["xcat_lo"], o["dbg_logits"],
                                  o["dbg_fused"], batch, S, D, P, x11_format, stream()), "decode_gather")
    torch.cuda.synchronize()
    return outs


def volume(feat_ref, feat_src, Mw, depths, out, *, batch=None):
    """adp_build_volume over `batch` environments (default out.shape[0]).  feat_ref / feat_src: device fp16 [>= batch, H, W, 32];
    Mw: device fp32 [>= batch, 12]; depths: device fp32 [D]; out: the caller's [>= batch, D, H, W, 32] buffer, fp16 or bf16
    (its dtype selects the output format)."""
    _, D, H, W, Cn = out.shape
    assert depths.numel() == D and out.dtype in (torch.float16, torch.bfloat16)
    L.check(L.load().adp_build_volume(L.ptr(feat_ref), L.ptr(feat_src), L.ptr(Mw), L.ptr(depths), L.ptr(out),
                                      out.shape[0] if batch is None else batch, D, H, W, Cn, int(out.dtype == torch.float16),
                                      stream()), "build_volume")
    torch.cuda.synchronize()
    return out


def tc_conv(x_cl, w, *, dil=1, npass=3, bias=None, scale=None, act_code=L.ACT_NONE, prelu=0.0, res_cl=None, res_after_act=0,
            batch=None, stride=1, transposed=False, f16=0, q8_out=None, geoms=None, cout=None, res_cstride=0, out_cstride=0,
            out_coff=0, bias_per_batch=0, check_finite=0, out_f32=None, out_hi=None, out_lo=None, out_h16=None, out_q8=None,
            num_sms=148, err=None, info_out=None, res_lo=None):
    """x_cl: fp32 [B,(D,)H,W,Cin] cpu; w: torch layout [Cout,Cin,(kd,)k,k] ([Cin,Cout,3,3,3] when transposed).
    Returns (fp32 output, 16-bit output as fp32), cpu, channels-last.

    The plan holds B = x_cl.shape[0] images; ``batch`` runs fewer.  ``geoms``: explicit tap tables (adp_tc_geom); w is then the
    packed fp32 [w_taps, Cout(Pad), Cin] tensor and ``cout`` the real output channel count.  ``out_f32`` / ``out_hi`` /
    ``out_lo`` / ``out_h16`` / ``out_q8``: device buffers the caller provides (pre-filled canaries stay where nothing is
    written), or False for no such output; None = the default (fresh fp32 NaN / 16-bit zero planes, no h16 / q8 copy).
    A returned value is None where there is no such output.  ``err``: the int32[2] device flag to pass (watchdog code must
    stay 0).  ``info_out``: a list that receives plan_info() of every plan.  ``res_lo=False``: a bf16 residual without lo plane."""
    from rgbmanip_b200 import geometry
    from rgbmanip_b200.engine import pack_tc_weights
    lib = L.load()
    three_d = x_cl.dim() == 5
    B = x_cl.shape[0]
    D = x_cl.shape[1] if three_d else 1
    H, Wd, Cin = x_cl.shape[-3], x_cl.shape[-2], x_cl.shape[-1]
    kd = w.shape[2] if (three_d and geoms is None) else 1
    ks = w.shape[-1] if geoms is None else 1
    if geoms is not None:
        Cout = cout
        wt = w.contiguous()
        g0 = geoms[0]
        oshape = (B, g0.oD, g0.oH, g0.oW, Cout) if three_d else (B, g0.oH, g0.oW, Cout)
    elif transposed:
        Cout = w.shape[1]
        wt = w.reshape(Cin, Cout, -1).permute(2, 1, 0).contiguous()
        geoms = geometry.transposed_classes(D, H, Wd)
        oshape = (B, 2 * D, 2 * H, 2 * Wd, Cout)
    else:
        Cout = w.shape[0]
        wt = w.reshape(Cout, Cin, -1).permute(2, 0, 1).contiguous()
        if stride == 2:
            geoms = [geometry.strided(three_d, D, H, Wd, ks, 2)]
            sp = ((D + 1) // 2, (H + 1) // 2, (Wd + 1) // 2) if three_d else ((H + 1) // 2, (Wd + 1) // 2)
            oshape = (B,) + sp + (Cout,)
        else:
            geoms = [None]
            oshape = tuple(x_cl.shape[:-1]) + (Cout,)
    cpad = (Cout + 15) // 16 * 16
    if wt.shape[1] < cpad:
        wt = torch.cat([wt, torch.zeros(wt.shape[0], cpad - wt.shape[1], Cin)], 1).contiguous()
    wh, wl = (t.to(DEV).contiguous() if t is not None else None for t in pack_tc_weights(wt, f16, npass))
    xq = None
    if f16:
        xh, xl = x_cl.to(torch.float16).to(DEV).contiguous(), None
        if npass == 4:      # the activation's e4m3(x / 2) twin for the fp8 low-order pass
            xq = to_e4m3(x_cl.to(torch.float16).float() * 0.5).to(DEV).contiguous()
        dt16 = torch.float16
    else:
        xh, xl = split(x_cl, npass == 3)
        dt16 = torch.bfloat16
    if out_f32 is None:
        out_f32 = torch.full(oshape, float("nan"), dtype=torch.float32, device=DEV)
    if out_hi is None:
        out_hi = torch.zeros(oshape, dtype=dt16, device=DEV)
    if out_lo is None:
        out_lo = torch.zeros(oshape, dtype=dt16, device=DEV) if not f16 else False
    out_f32, out_hi, out_lo = (t if t is not False else None for t in (out_f32, out_hi, out_lo))
    out_h16 = out_h16 if out_h16 is not False else None
    rh = rl = None
    if res_cl is not None:
        if f16:
            rh = res_cl.to(torch.float16).to(DEV).contiguous()
        else:
            rh, rl = split(res_cl, res_lo is not False)
    b_d = bias.to(DEV).contiguous() if bias is not None else None
    s_d = scale.to(DEV) if scale is not None else None
    if out_q8 is None or out_q8 is False:
        out_q8 = torch.zeros(oshape, dtype=torch.uint8, device=DEV) if q8_out is not None else None
    ep = epilogue(out_hi, out_lo, out_f32, s_d, b_d, act_code, prelu, rh, rl, res_after_act, out_q8=out_q8, res_cstride=res_cstride,
                  out_h16=out_h16, out_cstride=out_cstride, out_coff=out_coff, bias_per_batch=bias_per_batch, check_finite=check_finite)
    a = act(xh, xl, B, D, H, Wd, Cin, f16, xq)
    if err is None:
        err = torch.zeros(2, dtype=torch.int32, device=DEV)
    for g in geoms:
        plan = C.c_void_p()
        L.check(lib.adp_conv_tc_plan(C.byref(plan), C.byref(a), L.ptr(wh), L.ptr(wl), Cout, kd, ks, dil, npass, C.byref(ep),
                                     C.byref(g) if g is not None else None, num_sms), "plan")
        try:
            if info_out is not None:
                info_out.append(plan_info(plan))
            L.check(lib.adp_conv_tc_run(plan, B if batch is None else batch, L.ptr(err), stream()), "run")
            torch.cuda.synchronize()
        finally:
            lib.adp_conv_tc_free(plan)
    assert int(err[0].item()) == 0, f"watchdog code {int(err[0].item())}"
    if q8_out is not None:
        q8_out.append(from_e4m3(out_q8.cpu()) * 2.0)
    return (out_f32.cpu() if out_f32 is not None else None), (val(out_hi, out_lo).cpu() if out_hi is not None else None)
