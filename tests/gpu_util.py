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
             res_lo=None, res_after_act=0, out_q8=None):
    return L.Epilogue(L.ptr(scale), L.ptr(bias), float(prelu), act_code, res_after_act, L.ptr(res_hi), L.ptr(res_lo), 0,
                      L.ptr(out_hi), L.ptr(out_lo), L.ptr(out_f32), None, 0, 0, 0, L.ptr(out_q8), 0)


def rel_err(a, b):
    a, b = a.double().cpu(), b.double().cpu()
    return float((a - b).abs().max() / (b.abs().max() + 1e-30))


def tc_conv(x_cl, w, *, dil=1, npass=3, bias=None, scale=None, act_code=L.ACT_NONE, prelu=0.0, res_cl=None, res_after_act=0,
            batch=None, stride=1, transposed=False, f16=0, q8_out=None):
    """x_cl: fp32 [B,(D,)H,W,Cin] cpu; w: torch layout [Cout,Cin,(kd,)k,k] ([Cin,Cout,3,3,3] when transposed).
    Returns (fp32 output, 16-bit output as fp32), cpu, channels-last."""
    from rgbmanip_b200 import geometry
    from rgbmanip_b200.engine import pack_tc_weights
    lib = L.load()
    three_d = x_cl.dim() == 5
    B = x_cl.shape[0]
    D = x_cl.shape[1] if three_d else 1
    H, Wd, Cin = x_cl.shape[-3], x_cl.shape[-2], x_cl.shape[-1]
    kd = w.shape[2] if three_d else 1
    ks = w.shape[-1]
    if transposed:
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
    if cpad != Cout:
        wt = torch.cat([wt, torch.zeros(wt.shape[0], cpad - Cout, Cin)], 1).contiguous()
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
    out_f32 = torch.full(oshape, float("nan"), dtype=torch.float32, device=DEV)
    out_hi = torch.zeros(out_f32.shape, dtype=dt16, device=DEV)
    out_lo = torch.zeros_like(out_hi) if not f16 else None
    rh = rl = None
    if res_cl is not None:
        if f16:
            rh = res_cl.to(torch.float16).to(DEV).contiguous()
        else:
            rh, rl = split(res_cl, True)
    b_d = bias.to(DEV) if bias is not None else None
    s_d = scale.to(DEV) if scale is not None else None
    out_q8 = torch.zeros(out_f32.shape, dtype=torch.uint8, device=DEV) if q8_out is not None else None
    ep = epilogue(out_hi, out_lo, out_f32, s_d, b_d, act_code, prelu, rh, rl, res_after_act, out_q8=out_q8)
    a = act(xh, xl, B, D, H, Wd, Cin, f16, xq)
    err = torch.zeros(2, dtype=torch.int32, device=DEV)
    for g in geoms:
        plan = C.c_void_p()
        L.check(lib.adp_conv_tc_plan(C.byref(plan), C.byref(a), L.ptr(wh), L.ptr(wl), Cout, kd, ks, dil, npass, C.byref(ep),
                                     C.byref(g) if g is not None else None, 148), "plan")
        L.check(lib.adp_conv_tc_run(plan, B if batch is None else batch, L.ptr(err), stream()), "run")
        torch.cuda.synchronize()
        lib.adp_conv_tc_free(plan)
    assert int(err[0].item()) == 0, f"watchdog code {int(err[0].item())}"
    if q8_out is not None:
        q8_out.append(from_e4m3(out_q8.cpu()) * 2.0)
    return out_f32.cpu(), val(out_hi, out_lo).cpu()
