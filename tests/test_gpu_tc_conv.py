"""Every tcgen05 conv kernel instance the engine plans, and the epilogue options of its layers, against a float64 reference.

One reference case per instance of the table in csrc/tc_conv.cu that some engine configuration plans, at the channel counts,
kernel and geometry of an engine layer that runs on it (the spatial extent is reduced so that the CPU reference stays cheap) and
with that layer's epilogue.  Each case asserts the instance it lands on through adp_conv_tc_plan_info, and
test_engine_instances_have_reference_cases checks that no planned instance is left without a case.  The edge tests run the same
cases: one CTA against a full grid, a plan run below its capacity, channel-range outputs, ragged tiles, the TMA epilogue, the
per-image bias, the fp16 range guard and the fp8 twin's plan-time contract.

Reference: torch float64 on the CPU, evaluated over the tap table of the plan's geometry (the operation adp_conv_tc computes),
with the operands at their exact value in the kernel's format.  Bounds, per element:
  * one pass with exact operands leaves only the fp32 accumulation order: |got - ref| <= 1e-5 max|ref| (fp32 outputs); a 16-bit
    output adds its own rounding, at most one unit in the last place of the format at |ref| (half an ulp of the rounded value,
    which can sit one binade up);
  * split precision keeps the bounds derived in test_gpu_stages.py, relative to max|ref|: bf16x3 2e-4, fp16x2 2e-5, fp16 + fp8
    low-order pass 3e-5 and below 0.3 x the error of a single fp16 pass; a bf16 hi + lo output pair adds 2^-16 |ref| (hi rounds
    to 2^-8, lo to 2^-8 of the remainder);
  * everything that only moves the same arithmetic to another CTA, another batch size or another channel pitch is bit exact.
"""
import math
import zlib
from dataclasses import dataclass, field
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from gpu_util import CANARY8, CANARY16, assert_close, bits, canary16
from rgbmanip_b200 import _lib as L
from rgbmanip_b200 import geometry, weights

pytestmark = [pytest.mark.gpu, pytest.mark.filterwarnings("ignore")]


@pytest.fixture(scope="module")
def G():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    import importlib
    L.load()
    return importlib.import_module("gpu_util")


# (slab CTAs per SM, TMA epilogue, FUSED, BN, KC) -> a readable name
def inst_name(inst):
    slab, bulk, fused, bn, kc = inst
    if slab:
        return f"slab<{bn},{kc},{slab}{',bulk' if bulk else ''}>"
    return f"<{bn},{kc}{',' + str(fused) if fused else ''}>"


SPLIT_TOL = {2: 2e-5, 3: 2e-4, 4: 3e-5}       # npass -> bound relative to max|ref| (test_gpu_stages.py derives them)
ONE_PASS_TOL = 1e-5                           # fp32 accumulation order with exact operands


@dataclass
class Case:
    id: str
    layers: str             # the engine layer(s) the case stands for
    inst: tuple             # expected (slab CTAs, bulk, FUSED, BN, KC)
    npass: int
    f16: int
    x: tuple                # (B, D, H, W, Cin); D = 0: a 2-D map
    cout: int
    conv: tuple             # ("conv", ks, dil, stride) | ("tconv",) | ("stem",) | ("stem_split",) | ("s2d_strided",) | ("s2d_tconv",)
    outs: str               # outputs the layer writes: f32 hi lo h16 q8
    ep: dict = field(default_factory=dict)   # scale, bias, bias_per_batch, act, prelu, res, res_after_act, check_finite, cstride, coff
    ranges: tuple = ()      # extra (out_cstride, out_coff) for the channel-range test


R, P_, T = L.ACT_RELU, L.ACT_PRELU, L.ACT_TANH
CASES = [
    # ---- slab kernel
    Case("stem_fp16", "conv1 (stem: s2d 16 -> 64, 2 x 16 taps hi / lo), fp16x2 / fp16f8", (2, 0, 0, 64, 16), 1, 1, (3, 0, 40, 32, 16), 64,
         ("stem_split",), "hi", dict(act=R)),
    Case("unet_conv2", "cr.conv2 (3x3x3 16 -> 16)", (2, 0, 0, 16, 16), 1, 1, (3, 4, 24, 16, 16), 16, ("conv", 3, 1, 1), "hi",
         dict(scale=1, bias=1, act=R)),
    Case("unet_conv1", "cr.conv1 (s2d stride 2, 64 -> 16)", (2, 0, 0, 16, 64), 1, 1, (3, 3, 16, 16, 64), 16, ("s2d_strided",), "hi",
         dict(scale=1, bias=1, act=R)),
    Case("unet_conv4", "cr.conv4 (3x3x3 32 -> 32)", (1, 0, 0, 32, 32), 1, 1, (3, 3, 16, 16, 32), 32, ("conv", 3, 1, 1), "hi",
         dict(scale=1, bias=1, act=R)),
    Case("unet_conv11", "cr.conv11 (s2d transposed 16 -> 8 x 8, + conv0 skip after ReLU)", (2, 1, 0, 64, 16), 1, 1, (3, 3, 24, 16, 16),
         64, ("s2d_tconv",), "hi", dict(scale=1, bias=1, act=R, res=1, res_after_act=1)),
    Case("cout8_lane", "(Cout 8 padded to BN 16: per-lane stores)", (2, 0, 0, 16, 64), 1, 1, (3, 0, 16, 16, 64), 8, ("conv", 3, 1, 1), "hi",
         dict(bias=1, act=R), ranges=((24, 8),)),
    # ---- generic kernel, single pass
    Case("unet_conv3", "cr.conv3 (3x3x3 stride 2, 16 -> 32)", (0, 0, 0, 32, 16), 1, 1, (3, 4, 16, 16, 16), 32, ("conv", 3, 1, 2), "hi",
         dict(scale=1, bias=1, act=R)),
    Case("unet_conv5", "cr.conv5 (3x3x3 stride 2, 32 -> 64)", (0, 0, 0, 64, 32), 1, 1, (3, 6, 28, 28, 32), 64, ("conv", 3, 1, 2), "hi",
         dict(scale=1, bias=1, act=R)),
    Case("unet_conv6", "cr.conv6 (3x3x3 64 -> 64)", (0, 0, 0, 64, 64), 1, 1, (3, 3, 14, 14, 64), 64, ("conv", 3, 1, 1), "hi",
         dict(scale=1, bias=1, act=R)),
    Case("unet_conv7", "cr.conv7 (transposed 64 -> 32, 8 parity classes, + conv4 skip after ReLU)", (0, 0, 0, 32, 64), 1, 1,
         (3, 3, 8, 8, 64), 32, ("tconv",), "hi", dict(scale=1, bias=1, act=R, res=1, res_after_act=1)),
    Case("final_bf16", "final (1x1 64 -> 32, fp32 + fp16 copies, range guard), bf16", (0, 0, 0, 32, 64), 1, 0, (3, 0, 24, 24, 64), 32,
         ("conv", 1, 1, 1), "f32 h16", dict(bias=1, check_finite=1)),
    Case("layer4_bf16", "layer4.2.conv2 (3x3 dil 4, 512 -> 512, + residual, into the 1024-channel concat), bf16", (0, 0, 0, 256, 64), 1, 0,
         (3, 0, 12, 12, 512), 512, ("conv", 3, 4, 1), "hi", dict(act=R, res=1, cstride=1024, coff=0), ranges=((1024, 512),)),
    Case("layer2_down_bf16", "layer2.0.downsample (1x1 stride 2, 64 -> 128), bf16", (0, 0, 0, 128, 64), 1, 0, (3, 0, 28, 28, 64), 128,
         ("conv", 1, 1, 2), "hi", dict()),
    # ---- generic kernel, split precision through the pass loop (FUSED = 0, npass 3)
    Case("nocs_head4", "nocs_head.4 (64 -> 3, tanh, pitch-16 plane + dense fp32)", (0, 0, 0, 16, 64), 3, 0, (3, 0, 32, 32, 64), 3,
         ("conv", 1, 1, 1), "f32 hi lo", dict(bias=1, act=T, cstride=16, coff=0), ranges=((16, 5),)),
    Case("nocs_pts_mlp0", "nocs_pts_mlp.0 (16 -> 32)", (0, 0, 0, 32, 16), 3, 0, (3, 0, 32, 32, 16), 32, ("conv", 1, 1, 1), "f32 hi lo",
         dict(bias=1, act=R)),
    Case("nocs_pts_mlp2", "nocs_pts_mlp.2 (32 -> 64 into channels [32, 96) of xcat); instance_color.0", (0, 0, 0, 64, 32), 3, 0,
         (3, 0, 32, 32, 32), 64, ("conv", 1, 1, 1), "f32 hi lo", dict(bias=1, act=R, cstride=96, coff=32), ranges=((96, 32),)),
    Case("pose_mlp1_0", "pose_mlp1.0 (96 -> 128: two N tiles of 64)", (0, 0, 0, 64, 32), 3, 0, (3, 0, 32, 32, 96), 128, ("conv", 1, 1, 1),
         "f32 hi lo", dict(bias=1, act=R)),
    # ---- fused split precision
    Case("stem_bf16x3", "conv1 (stem: s2d 16 -> 64, 16 taps), bf16x3", (0, 0, 1, 64, 16), 3, 0, (3, 0, 32, 32, 16), 64, ("stem",), "f32 hi lo",
         dict(act=R)),
    Case("pose_mlp2_0", "pose_mlp2.0 (128 -> 256, per-env bias); layer3 / layer4, bf16x3", (0, 0, 1, 256, 64), 3, 0, (3, 0, 32, 32, 128),
         256, ("conv", 1, 1, 1), "f32 hi lo", dict(bias=1, bias_per_batch=1, act=R)),
    Case("nocs_head0", "nocs_head.0 (64 -> 128); layer2, bf16x3", (0, 0, 1, 128, 64), 3, 0, (3, 0, 32, 32, 64), 128, ("conv", 1, 1, 1),
         "f32 hi lo", dict(bias=1, act=R)),
    Case("nocs_head2", "nocs_head.2 (128 -> 64); layer1, up_2 / up_3, bf16x3", (0, 0, 1, 64, 64), 3, 0, (3, 0, 32, 32, 128), 64,
         ("conv", 1, 1, 1), "f32 hi lo", dict(bias=1, act=R)),
    Case("final_bf16x3", "final (1x1 64 -> 32, fp32 + fp16 copies, range guard), bf16x3", (0, 0, 1, 32, 64), 3, 0, (3, 0, 24, 24, 64), 32,
         ("conv", 1, 1, 1), "f32 h16", dict(bias=1, check_finite=1)),
    Case("up3_fp16x2", "up_3 (3x3 64 -> 64, bias + PReLU); layer1, up_2, fp16x2", (0, 0, 2, 64, 64), 2, 1, (3, 0, 18, 20, 64), 64,
         ("conv", 3, 1, 1), "f32 hi", dict(bias=1, act=P_, prelu=0.25)),
    Case("layer2_fp16x2", "layer2.0.conv1 (3x3 stride 2, 64 -> 128), fp16x2", (0, 0, 2, 128, 64), 2, 1, (3, 0, 28, 28, 64), 128,
         ("conv", 3, 1, 2), "f32 hi", dict(act=R)),
    Case("layer3_down_fp16x2", "layer3.0.downsample (1x1 128 -> 256), fp16x2", (0, 0, 2, 256, 64), 2, 1, (3, 0, 14, 14, 128), 256,
         ("conv", 1, 1, 1), "f32 hi", dict()),
    Case("final_fp16x2", "final (1x1 64 -> 32, fp32 + fp16 copies, range guard), fp16x2 / fp16f8", (0, 0, 2, 32, 64), 2, 1,
         (3, 0, 24, 24, 64), 32, ("conv", 1, 1, 1), "f32 h16", dict(bias=1, check_finite=1)),
    Case("layer2_fp8", "layer2.1.conv1 (3x3 128 -> 128, writes the fp8 twin), fp16f8", (0, 0, 3, 128, 64), 4, 1, (3, 0, 14, 14, 128), 128,
         ("conv", 3, 1, 1), "f32 hi q8", dict(act=R)),
    Case("layer4_fp8", "layer4.2.conv2 (3x3 dil 4, 512 -> 512, + residual, into the 1024-channel concat and its fp8 twin), fp16f8",
         (0, 0, 3, 256, 64), 4, 1, (3, 0, 12, 12, 512), 512, ("conv", 3, 4, 1), "f32 hi q8", dict(act=R, res=1, cstride=1024, coff=0),
         ranges=((1024, 512),)),
]
CASE_IDS = [c.id for c in CASES]
BY_ID = {c.id: c for c in CASES}


# ------------------------------------------------------------------------------------------------ inputs and reference
def _rng(case):
    return np.random.default_rng(zlib.crc32(case.id.encode()))


def _t(rng, *shape, scale=1.0):
    return torch.from_numpy((rng.standard_normal(shape) * scale).astype(np.float32))


def _exact(t, f16, split):
    """The value the kernel sees: IEEE half, bf16, or the bf16 hi + lo pair."""
    if f16:
        return t.half().double()
    hi = t.bfloat16()
    if not split:
        return hi.double()
    return hi.double() + (t - hi.float()).bfloat16().double()


def _plain_geom(D, H, W, kd, ks, dil):
    """The tap table adp_conv_tc_plan builds for a stride-1 'same' conv (geom = NULL)."""
    taps = []
    for t in range(kd * ks * ks):
        kx, ky, kz = t % ks, (t // ks) % ks, t // (ks * ks)
        taps.append(((kz - kd // 2), (ky - ks // 2) * dil, (kx - ks // 2) * dil, t))
    return SimpleNamespace(ntaps=len(taps), dz=[a[0] for a in taps], dy=[a[1] for a in taps], dx=[a[2] for a in taps],
                           wt=[a[3] for a in taps], in_mul=1, out_mul=1, out_oz=0, out_oy=0, out_ox=0, gD=D, gH=H, gW=W,
                           oD=D, oH=H, oW=W)


def build(case):
    """Seeded inputs of a case: what the helper is called with, and what the reference needs."""
    rng = _rng(case)
    B, D, H, W, Cin = case.x
    three_d = D > 0
    split = case.npass == 3
    single = case.npass == 1
    xs = (B, D, H, W, Cin) if three_d else (B, H, W, Cin)
    x = _t(rng, *xs)
    if case.npass == 4:
        x = x.relu()                             # the fp8 layers read post-ReLU activations
    if not split:                                 # make the activation exactly representable in its format
        x = x.half().float() if case.f16 else x.bfloat16().float()
    kind = case.conv[0]
    kw = dict(npass=case.npass, f16=case.f16)
    Dg = D if three_d else 1
    if kind == "conv":
        _, ks, dil, stride = case.conv
        kd = ks if three_d else 1
        w = _t(rng, case.cout, Cin, *((kd,) if three_d else ()), ks, ks, scale=math.sqrt(2.0 / (kd * ks * ks * Cin)))
        wt = w.reshape(case.cout, Cin, -1).permute(2, 0, 1).contiguous()
        if stride == 2:
            geoms = [geometry.strided(three_d, Dg, H, W, ks, 2)]
        else:
            geoms = [_plain_geom(Dg, H, W, kd, ks, dil)]
        kw.update(w=w, dil=dil, stride=stride)
    elif kind == "tconv":
        w = _t(rng, Cin, case.cout, 3, 3, 3, scale=math.sqrt(1.0 / (8 * Cin)))
        wt = w.reshape(Cin, case.cout, -1).permute(2, 1, 0).contiguous()
        geoms = geometry.transposed_classes(D, H, W)
        kw.update(w=w, transposed=True)
    else:
        if kind in ("stem", "stem_split"):
            w7 = _t(rng, 64, 3, 7, 7, scale=math.sqrt(2.0 / 147))
            wt = geometry.stem_s2d_weights(w7)
            if kind == "stem_split":                 # the fp16 stem: hi and lo weight slabs as 32 taps of one pass
                from rgbmanip_b200.engine import pack_tc_weights
                wt = torch.cat(pack_tc_weights(wt, 1, 2)).float()
                g = geometry.stem_s2d_split(2 * W)
            else:
                g = geometry.stem_s2d(2 * W)
            g.gH = g.oH = H                           # the stem grid is square in the engine; H != W here for a ragged slab
        elif kind == "s2d_strided":
            wt = geometry.strided_s2d_weights(_t(rng, case.cout, 8, 3, 3, 3, scale=math.sqrt(2.0 / 216)))
            g = geometry.strided_s2d(D, H, W)
        else:
            wt = geometry.transposed_s2d_weights(_t(rng, Cin, case.cout // 8, 3, 3, 3, scale=math.sqrt(1.0 / (8 * Cin))))
            g = geometry.transposed_s2d(D, H, W)
        geoms = [g]
        kw.update(w=wt, geoms=geoms, cout=case.cout)
    if single:
        wt = wt.half().float() if case.f16 else wt.bfloat16().float()
        if "w" in kw and kind in ("conv", "tconv"):
            kw["w"] = kw["w"].half().float() if case.f16 else kw["w"].bfloat16().float()
        elif "geoms" in kw:
            kw["w"] = wt
    g0 = geoms[0]
    oshape = (B, g0.oD, g0.oH, g0.oW, case.cout) if three_d else (B, g0.oH, g0.oW, case.cout)
    ep = case.ep
    ref_ep = {}
    rep = 8 if kind == "s2d_tconv" else 1             # the folded BatchNorm of conv11 repeats over the 8 output parities
    if ep.get("scale"):
        s = (_t(rng, case.cout // rep).abs() + 0.5).repeat(rep)
        kw["scale"] = s
        ref_ep["scale"] = s.double()
    if ep.get("bias"):
        b = _t(rng, B, case.cout) if ep.get("bias_per_batch") else _t(rng, case.cout // rep).repeat(rep)
        kw["bias"] = b
        kw["bias_per_batch"] = int(ep.get("bias_per_batch", 0))
        ref_ep["bias"] = b.double()
    if ep.get("res"):
        r = _t(rng, *oshape)
        kw["res_cl"] = r
        if not case.f16 and not split:
            kw["res_lo"] = False                      # a bf16 single-pass engine tensor has no lo plane
        ref_ep["res"] = _exact(r, case.f16, split)
    kw["act_code"] = ep.get("act", L.ACT_NONE)
    kw["prelu"] = ep.get("prelu", 0.0)
    kw["res_after_act"] = ep.get("res_after_act", 0)
    kw["check_finite"] = ep.get("check_finite", 0)
    if split:
        from rgbmanip_b200.engine import pack_tc_weights
        hi, lo = pack_tc_weights(wt, 0, 3)
        w_exact = hi.double() + lo.double()
    elif case.npass == 2:
        from rgbmanip_b200.engine import pack_tc_weights
        hi, lo = pack_tc_weights(wt, 1, 2)
        w_exact = hi.double() + lo.double()
    else:
        w_exact = wt.double()
    cpad = (case.cout + 15) // 16 * 16
    if w_exact.shape[1] < cpad:
        w_exact = torch.cat([w_exact, torch.zeros(w_exact.shape[0], cpad - w_exact.shape[1], Cin, dtype=torch.float64)], 1)
    return SimpleNamespace(x=x, kw=kw, geoms=geoms, oshape=oshape, x_exact=_exact(x, case.f16, split), w_exact=w_exact, wt=wt,
                           ref_ep=ref_ep, three_d=three_d)


def tap_conv(A, wt, geoms, oshape):
    """float64 [B, D, H, W, C] (D = 1 for 2-D) x packed [w_taps, N, C] over the tap tables -> [B, oD, oH, oW, N]."""
    B, D, H, W, Cn = A.shape
    P = 4
    ext = [max(n, 2 * g) + 2 * P for n, g in zip((D, H, W), (max(g.gD for g in geoms), max(g.gH for g in geoms),
                                                             max(g.gW for g in geoms)))]
    Ap = torch.zeros(B, *ext, Cn, dtype=torch.float64)
    Ap[:, P:P + D, P:P + H, P:P + W] = A
    out = torch.zeros(B, *oshape[1:4], wt.shape[1], dtype=torch.float64)
    for g in geoms:
        m, om = g.in_mul, g.out_mul
        acc = torch.zeros(B, g.gD, g.gH, g.gW, wt.shape[1], dtype=torch.float64)
        for t in range(g.ntaps):
            z0, y0, x0 = P + g.dz[t], P + g.dy[t], P + g.dx[t]
            acc += Ap[:, z0:z0 + m * g.gD:m, y0:y0 + m * g.gH:m, x0:x0 + m * g.gW:m] @ wt[g.wt[t]].t()
        out[:, g.out_oz:g.out_oz + om * g.gD:om, g.out_oy:g.out_oy + om * g.gH:om, g.out_ox:g.out_ox + om * g.gW:om] = acc
    return out


def reference(case, d, w_exact=None):
    """float64 output [B, (oD,) oH, oW, Cout] of the case's conv + epilogue."""
    A = d.x_exact if d.three_d else d.x_exact.unsqueeze(1)
    o5 = d.oshape if d.three_d else (d.oshape[0], 1) + d.oshape[1:]
    v = tap_conv(A, d.w_exact if w_exact is None else w_exact, d.geoms, o5)[..., :case.cout]
    if not d.three_d:
        v = v[:, 0]
    e = d.ref_ep
    bshape = (v.shape[0],) + (1,) * (v.dim() - 2) + (case.cout,)
    if "scale" in e:
        v = v * e["scale"]
    if "bias" in e:
        v = v + (e["bias"].reshape(bshape) if case.ep.get("bias_per_batch") else e["bias"])
    res = e.get("res")
    if res is not None and not case.ep.get("res_after_act"):
        v = v + res
    act = case.ep.get("act", L.ACT_NONE)
    if act == L.ACT_RELU:
        v = v.clamp_min(0)
    elif act == L.ACT_PRELU:
        v = torch.where(v > 0, v, v * case.ep["prelu"])
    elif act == L.ACT_TANH:
        v = torch.tanh(v)
    if res is not None and case.ep.get("res_after_act"):
        v = v + res
    return v


# ------------------------------------------------------------------------------------------------ running a case
def run(G, case, d, *, num_sms=148, batch=None, rng=None, x=None, err=None):
    """One adp_conv_tc run of the case into freshly canary-filled output buffers.  rng = (out_cstride, out_coff) overrides the
    layer's channel range ((0, 0) = dense).  Returns (buffers, plan infos, err flag)."""
    cs, coff = rng if rng is not None else (case.ep.get("cstride", 0), case.ep.get("coff", 0))
    wide = d.oshape[:-1] + ((cs or case.cout),)
    dt16 = torch.float16 if case.f16 else torch.bfloat16
    outs = case.outs.split()
    bufs = dict(out_f32=torch.full(d.oshape, float("nan"), device="cuda:0") if "f32" in outs else False,
                out_hi=canary16(wide, dt16) if "hi" in outs else False,
                out_lo=canary16(wide, dt16) if "lo" in outs else False,
                out_h16=canary16(d.oshape, torch.float16) if "h16" in outs else False,
                out_q8=torch.full(wide, CANARY8, dtype=torch.uint8, device="cuda:0") if "q8" in outs else False)
    info = []
    if err is None:
        err = torch.zeros(2, dtype=torch.int32, device="cuda:0")
    G.tc_conv(d.x if x is None else x, **d.kw, out_cstride=cs, out_coff=coff, num_sms=num_sms, batch=batch, err=err, info_out=info,
              **bufs)
    return {k: v for k, v in bufs.items() if v is not False}, info, err


_BUILT, _FULL = {}, {}


def built(case):
    if case.id not in _BUILT:
        _BUILT[case.id] = build(case)
    return _BUILT[case.id]


def full_run(G, case):
    """The case at 148 SMs over its whole planned batch (cached: the edge tests compare against it)."""
    if case.id not in _FULL:
        _FULL[case.id] = run(G, case, built(case))
    return _FULL[case.id]


# ------------------------------------------------------------------------------------------------ (a) instance coverage
ENGINE_CONFIGS = {"v5": dict(), "branch_b": dict(regress_pose=False), "branch_c": dict(regress_pose=False, use_depth=False),
                  "baseline": dict(arch="baseline")}


def engine_instances(G):
    """instance -> sorted list of "precision/config: layer" over every engine configuration (max_envs = 1)."""
    from rgbmanip_b200.engine import Engine
    table = {}
    sds = {cname: weights.init_state_dict(0, regress_pose=kw.get("regress_pose", True), arch=kw.get("arch", "v5"))
           for cname, kw in ENGINE_CONFIGS.items()}
    for prec in ("fp16f8", "fp16x2", "bf16x3", "bf16"):
        for cname, kw in ENGINE_CONFIGS.items():
            sd = sds[cname]
            eng = Engine(sd, device=G.DEV, max_envs=1, precision=prec, **kw)
            try:
                names = {}
                for nm, op in list(eng.backbone_ops) + list(getattr(eng, "cr_ops", [])) + list(eng.dec_ops):
                    for p in getattr(op, "plans", []):
                        names[p.value] = nm
                assert eng._plans
                for p in eng._plans:
                    info = G.plan_info(p)
                    loop = " (pass loop)" if info["fused"] == 0 and info["npass"] > 1 else ""
                    table.setdefault(info["instance"], set()).add(f"{names.get(p.value, '?')}{loop}")
            finally:
                eng.close()
    return {k: sorted(v) for k, v in table.items()}


def test_engine_instances_have_reference_cases(G):
    planned = engine_instances(G)
    reached = {}
    for case in CASES:
        for info in full_run(G, case)[1]:
            reached.setdefault(info["instance"], []).append(case.id)
    print("\ninstance -> engine layers (all precisions and configurations) | reference cases")
    for inst in sorted(planned, key=inst_name):
        print(f"  {inst_name(inst):22s} {', '.join(planned[inst])}  |  {', '.join(sorted(set(reached.get(inst, []))))}")
    missing = sorted(inst_name(i) for i in planned if i not in reached)
    assert not missing, f"planned instances without a reference case: {missing}"
    unplanned = sorted(inst_name(i) for i in reached if i not in planned)
    print("  reached by a case but planned by no engine configuration:", unplanned or "none")


# ------------------------------------------------------------------------------------------------ (b) reference table
@pytest.mark.parametrize("cid", CASE_IDS)
def test_instance_matches_fp64_reference(G, cid):
    case = BY_ID[cid]
    d = built(case)
    bufs, infos, err = full_run(G, case)
    assert {i["instance"] for i in infos} == {case.inst}, ([inst_name(i["instance"]) for i in infos], inst_name(case.inst))
    assert all(i["npass"] == case.npass for i in infos)
    assert err.tolist() == [0, 0]
    ref = reference(case, d)
    tol = ONE_PASS_TOL if case.npass == 1 else SPLIT_TOL[case.npass]
    slack = tol * float(ref.abs().max())
    fmt16 = "f16" if case.f16 else "bf16"
    cs, coff = case.ep.get("cstride", 0), case.ep.get("coff", 0)
    rng = slice(coff, coff + case.cout) if cs else slice(0, case.cout)
    worst = {}
    if "out_f32" in bufs:
        worst["f32"] = assert_close(bufs["out_f32"].cpu(), ref, "f32", slack, f"{cid} fp32")
    if "out_hi" in bufs:
        hi = bufs["out_hi"].cpu()[..., rng]
        worst["hi"] = assert_close(hi.float(), ref, fmt16, slack, f"{cid} hi")
        if "out_lo" in bufs:
            lo = bufs["out_lo"].cpu()[..., rng]
            worst["hi+lo"] = assert_close(hi.double() + lo.double(), ref, "bf16x2", slack, f"{cid} hi + lo")
        if cs:                                    # channels outside the layer's range keep their canary
            keep = torch.ones(cs, dtype=torch.bool)
            keep[rng] = False
            for k in ("out_hi", "out_lo", "out_q8"):
                if k in bufs:
                    b = bits(bufs[k])[..., keep]
                    assert (b == (CANARY8 if k == "out_q8" else CANARY16)).all(), k
    if "out_h16" in bufs:
        worst["h16"] = assert_close(bufs["out_h16"].cpu().float(), ref, "f16", slack, f"{cid} fp16 copy")
    if "out_q8" in bufs:                          # the fp8 twin: e4m3(value / 2), rounding ties aside (test_gpu_stages.py rule)
        got = G.from_e4m3(bufs["out_q8"].cpu()[..., rng].contiguous()) * 2.0
        want = G.from_e4m3(G.to_e4m3((ref * 0.5).float())) * 2.0
        assert float((got - want).abs().max()) <= 0.13 * float(want.abs().max())
        assert float(((got - want).abs() > 0).float().mean()) < 0.02
    if case.npass == 4:                           # the fp8 low-order term: well below a single fp16 pass (test_gpu_stages.py)
        one = reference(case, d, w_exact=d.wt.half().double())
        e = float((bufs["out_f32"].cpu().double() - ref).abs().max()) / float(ref.abs().max())
        e1 = float((one - ref).abs().max()) / float(ref.abs().max())
        print(f"{cid}: fp32 output error {e:.2e}, single fp16 pass {e1:.2e}")
        assert e < 0.3 * e1, (e, e1)
    print(f"{cid} on {inst_name(case.inst)}: largest error / bound " + ", ".join(f"{k} {v:.3f}" for k, v in worst.items()))


# ------------------------------------------------------------------------------------------------ (c) edges
@pytest.mark.parametrize("cid", CASE_IDS)
def test_one_cta_equals_full_grid(G, cid):
    """Each tile's arithmetic does not depend on the CTA that runs it: one SM's worth of CTAs walking every tile (many trips
    round the stage ring and both TMEM accumulator stages) writes the same bits as a full grid."""
    case = BY_ID[cid]
    full, _, _ = full_run(G, case)
    one, infos, err = run(G, case, built(case), num_sms=1)
    assert err.tolist() == [0, 0]
    for k in full:
        assert torch.equal(bits(one[k]), bits(full[k])), k


@pytest.mark.parametrize("cid", CASE_IDS)
def test_partial_batch(G, cid):
    """A plan for 3 images run on 2: image 2 keeps its canary bits, images 0-1 equal the full run bit for bit."""
    case = BY_ID[cid]
    full, _, _ = full_run(G, case)
    part, _, err = run(G, case, built(case), batch=2)
    assert err.tolist() == [0, 0]
    for k in full:
        assert torch.equal(bits(part[k])[:2], bits(full[k])[:2]), k
        canary = {"out_f32": 0x7FC00000, "out_q8": CANARY8}.get(k, CANARY16)
        assert (bits(part[k])[2] == canary).all(), k


def test_edge_shapes_are_covered(G):
    """The table exercises what the edge tests are about: several N tiles, an odd tile count, ragged tiles of the generic and
    the slab kernel and of the TMA epilogue, and both epilogue store paths."""
    infos = {c.id: full_run(G, c)[1] for c in CASES}
    flat = [(c, i) for c in CASES for i in infos[c.id]]
    tiles = lambda c, i: c.x[0] * i["D"] * i["tiles_y"] * i["tiles_x"] * i["tiles_n"]
    assert any(i["tiles_n"] > 1 for _, i in flat)
    assert any(tiles(c, i) % 2 == 1 for c, i in flat)
    assert any(i["slab_ctas"] == 0 and built(c).geoms[0].gH % i["TH"] for c, i in flat)
    assert any(i["slab_ctas"] and not i["bulk"] and built(c).geoms[0].gH % 16 for c, i in flat)
    assert any(i["bulk"] and built(c).geoms[0].gH % 16 for c, i in flat)
    assert any(i["coalesce"] for _, i in flat) and any(not i["coalesce"] for _, i in flat)


RANGE_CASES = [c.id for c in CASES if c.ranges]


@pytest.mark.parametrize("cid", RANGE_CASES)
def test_channel_range_output(G, cid):
    """out_cstride > Cout with out_coff > 0 on every 16-bit plane and the fp8 twin, on the coalesced and the per-lane store
    path: the range holds the dense run's bits, every channel outside it keeps its canary."""
    case = BY_ID[cid]
    d = built(case)
    dense, dinfo, _ = run(G, case, d, rng=(0, 0))
    for cs, coff in case.ranges:
        assert cs > case.cout and coff > 0
        wide, infos, err = run(G, case, d, rng=(cs, coff))
        assert err.tolist() == [0, 0]
        assert {i["coalesce"] for i in infos} == {i["coalesce"] for i in dinfo}
        keep = torch.ones(cs, dtype=torch.bool)
        keep[coff:coff + case.cout] = False
        for k in ("out_hi", "out_lo", "out_q8"):
            if k in wide:
                w = bits(wide[k])
                assert torch.equal(w[..., coff:coff + case.cout], bits(dense[k])), k
                assert (w[..., keep] == (CANARY8 if k == "out_q8" else CANARY16)).all(), k
        for k in ("out_f32", "out_h16"):          # dense side outputs do not move with the range
            if k in wide:
                assert torch.equal(bits(wide[k]), bits(dense[k])), k
    print(f"{cid}: coalesced store path {bool(dinfo[0]['coalesce'])}")


def test_per_lane_and_coalesced_ranges_are_both_covered(G):
    paths = {bool(run(G, BY_ID[cid], built(BY_ID[cid]), rng=BY_ID[cid].ranges[0])[1][0]["coalesce"]) for cid in RANGE_CASES}
    assert paths == {True, False}
    assert any("q8" in BY_ID[cid].outs for cid in RANGE_CASES) and any("lo" in BY_ID[cid].outs for cid in RANGE_CASES)


def test_tma_epilogue_ragged_tile_matches_per_lane_epilogue(G, monkeypatch):
    """conv11 on the slab kernel with the TMA epilogue at H2 = 24 (a ragged 16-row tile: the residual box load zero-fills and
    the result box store clips) against the coalesced per-lane epilogue (ADP_NO_BULK_EPI, read when the layer is planned):
    the same arithmetic per element, so the same bits; both agree with the fp64 reference through the reference test."""
    case = BY_ID["unet_conv11"]
    d = built(case)
    bulk, binfo, _ = full_run(G, case)
    monkeypatch.setenv("ADP_NO_BULK_EPI", "1")
    lane, linfo, err = run(G, case, d)
    assert err.tolist() == [0, 0]
    assert binfo[0]["bulk"] == 1 and linfo[0]["bulk"] == 0 and linfo[0]["slab_ctas"] == 2
    assert d.geoms[0].gH % 16 != 0
    assert torch.equal(bits(bulk["out_hi"]), bits(lane["out_hi"]))


FINITE_CASES = [c.id for c in CASES if c.ep.get("check_finite")]


@pytest.mark.parametrize("cid", FINITE_CASES)
def test_range_guard_flags_one_inf(G, cid):
    """check_finite: err[1] stays 0 on finite data (the reference run) and is set by a single inf in the input; err[0], the
    watchdog code, stays 0 throughout."""
    case = BY_ID[cid]
    d = built(case)
    assert full_run(G, case)[2].tolist() == [0, 0]
    x = d.x.clone()
    x[1, 5, 7, 3] = float("inf")
    _, _, err = run(G, case, d, x=x)
    assert err.tolist() == [0, 1]


def test_per_image_bias(G):
    """bias_per_batch: every image has its own bias row.  Reading image 0's row for all images would be an O(1) error, far
    outside the bound the reference test holds the output to."""
    case = BY_ID["pose_mlp2_0"]
    d = built(case)
    bufs = full_run(G, case)[0]
    got = bufs["out_f32"].cpu().double()
    ref = reference(case, d)
    wrong = reference(case, SimpleNamespace(**{**vars(d), "ref_ep": {**d.ref_ep, "bias": d.ref_ep["bias"][:1].expand(3, -1)}}))
    bound = SPLIT_TOL[3] * float(ref.abs().max())
    assert float((got - ref).abs().max()) <= bound
    for img in (1, 2):
        assert float((got[img] - wrong[img]).abs().max()) > 1000 * bound


# ------------------------------------------------------------------------------------------------ (d) the fp8 twin's contract
def test_fp8_twin_needs_coalesced_aligned_range(G):
    """out_q8 is only written by the coalesced epilogue, in 16-byte row pieces of one byte per channel.  A layer that would
    take the per-lane stores (out_coff 4) or misalign the pieces (out_coff 8) fails at plan time; at out_coff 16 the twin holds
    e4m3(out / 2) in the layer's range and the canary elsewhere."""
    rng = np.random.default_rng(88)
    B, H, W, Cin, Cout, cs = 2, 14, 14, 64, 64, 128
    x = torch.from_numpy(rng.standard_normal((B, H, W, Cin)).astype(np.float32)).relu().half().float()
    w = torch.from_numpy((rng.standard_normal((Cout, Cin, 3, 3)) * math.sqrt(2.0 / (9 * Cin))).astype(np.float32))
    for coff, why in ((4, "multiples of 16"), (8, "multiples of 16")):
        hi = torch.zeros((B, H, W, cs), dtype=torch.float16, device=G.DEV)
        q8 = torch.zeros((B, H, W, cs), dtype=torch.uint8, device=G.DEV)
        with pytest.raises(L.AdpError, match=r"out_q8 .*" + why):
            G.tc_conv(x, w, npass=2, f16=1, act_code=L.ACT_RELU, out_f32=False, out_hi=hi, out_q8=q8, out_cstride=cs, out_coff=coff)
    coff = 16
    hi = canary16((B, H, W, cs), torch.float16)
    q8 = torch.full((B, H, W, cs), CANARY8, dtype=torch.uint8, device=G.DEV)
    f32 = torch.full((B, H, W, Cout), float("nan"), device=G.DEV)
    G.tc_conv(x, w, npass=2, f16=1, act_code=L.ACT_RELU, out_f32=f32, out_hi=hi, out_q8=q8, out_cstride=cs, out_coff=coff)
    got = G.from_e4m3(q8.cpu()[..., coff:coff + Cout].contiguous()) * 2.0
    want = G.from_e4m3(G.to_e4m3(f32.cpu() * 0.5)) * 2.0
    assert float((got - want).abs().max()) <= 0.13 * float(want.abs().max())
    assert float(((got - want).abs() > 0).float().mean()) < 0.02      # a rounding tie here and there, otherwise identical
    keep = torch.ones(cs, dtype=torch.bool)
    keep[coff:coff + Cout] = False
    assert (q8.cpu()[..., keep] == CANARY8).all() and (bits(hi)[..., keep] == CANARY16).all()
