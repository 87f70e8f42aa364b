"""Stage-level parity on the B200: every CUDA stage, called through the C ABI, against the CPU oracle
(oracle/adapose_oracle.py, itself pinned to the reference by tests/test_oracle_golden.py) on the same seeded inputs.

Tolerances: integer/index work is bit exact; floating point stages state their bound next to the assert.  The
tensor-core convolution is checked in both precision modes: "bf16x3" (split precision, fp32-grade) and plain
"bf16" (one pass; bound = bf16 operand rounding)."""
import ctypes as C
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import adapose_oracle as O
from rgbmanip_b200 import _lib as L
from rgbmanip_b200 import synth, weights

pytestmark = [pytest.mark.gpu, pytest.mark.filterwarnings("ignore")]

@pytest.fixture(scope="module")
def G():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    import importlib
    L.load()
    return importlib.import_module("gpu_util")


def _rng(seed):
    return np.random.default_rng(seed)


def _t(rng, *shape, scale=1.0):
    return torch.from_numpy((rng.standard_normal(shape) * scale).astype(np.float32))


# ------------------------------------------------------------------------------------------------ convolutions
TC2D_CASES = [
    # (B, H, W, Cin, Cout, k, dil)
    (2, 28, 28, 64, 64, 3, 1),
    (1, 28, 28, 128, 256, 3, 2),
    (2, 28, 28, 256, 512, 3, 4),
    (1, 28, 28, 128, 256, 1, 1),
    (1, 56, 56, 64, 64, 3, 1),
    (1, 112, 112, 256, 64, 3, 1),
    (1, 224, 224, 64, 64, 3, 1),
    (1, 224, 224, 64, 32, 1, 1),
    (3, 20, 12, 64, 128, 3, 1),
    (2, 20, 24, 64, 64, 3, 1),          # 24 x 5 pixel tiles: 8 of the 128 MMA rows stay unused
]


@pytest.mark.parametrize("case", TC2D_CASES, ids=lambda c: "x".join(map(str, c)))
@pytest.mark.parametrize("npass", [3, 1])
def test_tc_conv2d_matches_oracle(G, case, npass):
    B, H, W, Cin, Cout, k, dil = case
    rng = _rng(hash(case) % 2**31)
    x = _t(rng, B, Cin, H, W)
    w = _t(rng, Cout, Cin, k, k, scale=math.sqrt(2.0 / (k * k * Cin)))
    bias = _t(rng, Cout)
    res = _t(rng, B, Cout, H, W)
    ref = F.relu(F.conv2d(x, w, bias, padding=dil * (k // 2), dilation=dil) + res)
    out32, out16 = G.tc_conv(G.to_cl(x), w, dil=dil, npass=npass, bias=bias, act_code=L.ACT_RELU, res_cl=G.to_cl(res))
    assert torch.isfinite(out32).all()
    e = G.rel_err(G.from_cl(out32), ref)
    # bf16x3 keeps ~16 mantissa bits of both operands; one bf16 pass keeps 8
    assert e < (2e-4 if npass == 3 else 2e-2), e
    assert G.rel_err(G.from_cl(out16), ref) < (2e-4 if npass == 3 else 2e-2)


@pytest.mark.parametrize("case", TC2D_CASES, ids=lambda c: "x".join(map(str, c)))
def test_tc_conv2d_fp16x2_matches_oracle(G, case):
    """fp16x2: one fp16 activation plane against fp16 hi + lo weights (two MMA passes).  The inputs are made exactly
    representable in fp16, so what is left is the weight split (~2^-22) and fp32 accumulation order."""
    B, H, W, Cin, Cout, k, dil = case
    rng = _rng(hash(case) % 2**31 + 1)
    x = _t(rng, B, Cin, H, W).half().float()
    w = _t(rng, Cout, Cin, k, k, scale=math.sqrt(2.0 / (k * k * Cin)))
    bias = _t(rng, Cout)
    res = _t(rng, B, Cout, H, W).half().float()
    ref = F.relu(F.conv2d(x.double(), w.double(), bias.double(), padding=dil * (k // 2), dilation=dil) + res.double()).float()
    out32, out16 = G.tc_conv(G.to_cl(x), w, dil=dil, npass=2, bias=bias, act_code=L.ACT_RELU, res_cl=G.to_cl(res), f16=1)
    assert torch.isfinite(out32).all()
    assert G.rel_err(G.from_cl(out32), ref) < 2e-5
    assert G.rel_err(G.from_cl(out16), ref) < 6e-4          # fp16 storage: 2^-11


FP8LO_CASES = [
    # (B, H, W, Cin, Cout, k, dil): the wide backbone layers (layer3, layer4, their 1x1 downsamples, up_1)
    (1, 28, 28, 128, 256, 3, 2),
    (2, 28, 28, 256, 512, 3, 4),
    (1, 28, 28, 128, 256, 1, 1),
    (3, 28, 28, 512, 512, 3, 4),
    (1, 56, 56, 1024, 256, 3, 1),
    (1, 20, 12, 128, 128, 3, 1),
]


@pytest.mark.parametrize("case", FP8LO_CASES, ids=lambda c: "x".join(map(str, c)))
def test_tc_conv2d_fp16_plus_fp8_low_order_pass(G, case):
    """npass 4 ("fp16f8"): A W_hi in fp16 + the low-order term e4m3(A / 2) x e4m3(W_lo 2^16) as an fp8 MMA sweep, joined by the
    2^-15 accumulator scale of the first fp16 MMA.  W_lo <= 2^-12 |W|, so its e4m3 rounding (2^-4) leaves ~2^-16 of the
    output: between fp16x2 (2^-22) and a single fp16 pass (2^-12).  A wrong scale would be off by orders of magnitude."""
    B, H, W, Cin, Cout, k, dil = case
    rng = _rng(hash(case) % 2**31 + 7)
    x = F.relu(_t(rng, B, Cin, H, W)).half().float()
    w = _t(rng, Cout, Cin, k, k, scale=math.sqrt(2.0 / (k * k * Cin)))
    bias = _t(rng, Cout)
    res = _t(rng, B, Cout, H, W).half().float()
    ref = F.relu(F.conv2d(x.double(), w.double(), bias.double(), padding=dil * (k // 2), dilation=dil) + res.double()).float()
    one_pass = F.relu(F.conv2d(x.double(), w.half().double(), bias.double(), padding=dil * (k // 2), dilation=dil) + res.double()).float()
    q8 = []
    out32, out16 = G.tc_conv(G.to_cl(x), w, dil=dil, npass=4, bias=bias, act_code=L.ACT_RELU, res_cl=G.to_cl(res), f16=1,
                             q8_out=q8 if Cout % 32 == 0 else None)
    assert torch.isfinite(out32).all()
    e, e1 = G.rel_err(G.from_cl(out32), ref), G.rel_err(one_pass, ref)
    print(f"fp16f8 rel err {e:.2e} (single fp16 pass would be {e1:.2e})")
    assert e < 3e-5 and e < 0.3 * e1, (e, e1)
    assert G.rel_err(G.from_cl(out16), ref) < 6e-4          # fp16 storage: 2^-11
    if q8:                                                    # the fp8 twin the next layer's low-order pass reads: value / 2 in e4m3
        got, want = q8[0], G.from_e4m3(G.to_e4m3(out32 * 0.5)) * 2.0
        assert float((got - want).abs().max()) <= 0.13 * float(want.abs().max())
        assert float(((got - want).abs() > 0).float().mean()) < 0.02     # a rounding tie here and there, otherwise identical


TC3D_CASES = [
    # (B, D, H, W, Cin, Cout)
    (1, 6, 28, 28, 64, 8),
    (1, 5, 56, 56, 16, 16),
    (2, 6, 28, 56, 32, 32),
    (1, 3, 28, 28, 64, 64),
    (1, 4, 224, 224, 64, 8),
]


@pytest.mark.parametrize("case", TC3D_CASES, ids=lambda c: "x".join(map(str, c)))
def test_tc_conv3d_matches_oracle(G, case):
    B, D, H, W, Cin, Cout = case
    rng = _rng(sum(case))
    x = _t(rng, B, Cin, D, H, W).bfloat16().float()       # the volume stage stores bf16: make the input exactly representable
    w = _t(rng, Cout, Cin, 3, 3, 3, scale=math.sqrt(1.0 / (27 * Cin)))
    scale, shift = _t(rng, Cout).abs() + 0.5, _t(rng, Cout)
    ref = F.relu(F.conv3d(x, w.bfloat16().float(), padding=1) * scale.view(1, -1, 1, 1, 1) + shift.view(1, -1, 1, 1, 1))
    out32, _ = G.tc_conv(G.to_cl(x), w, npass=1, bias=shift, scale=scale, act_code=L.ACT_RELU)
    assert torch.isfinite(out32).all()
    assert G.rel_err(G.from_cl(out32), ref) < 1e-4   # operands are exact bf16: only fp32 summation order differs


TC_GEOM_CASES = [
    # (dims, B, D, H, W, Cin, Cout, k, stride, transposed, f16)
    (2, 2, 1, 56, 56, 64, 128, 3, 2, False, 0),
    (2, 1, 1, 56, 56, 64, 128, 1, 2, False, 0),
    (3, 1, 12, 112, 112, 16, 32, 3, 2, False, 1),
    (3, 1, 6, 56, 56, 32, 64, 3, 2, False, 1),
    (3, 1, 6, 56, 56, 32, 64, 3, 2, False, 0),
    (3, 1, 3, 28, 28, 64, 32, 3, 2, True, 1),
    (3, 1, 6, 56, 56, 64, 16, 3, 2, True, 1),
    (3, 2, 4, 28, 28, 64, 8, 3, 2, True, 1),
    (3, 1, 4, 28, 28, 64, 8, 3, 2, True, 0),
    (3, 1, 5, 56, 56, 64, 8, 3, 1, False, 1),
]


@pytest.mark.parametrize("case", TC_GEOM_CASES, ids=lambda c: "x".join(map(str, c)))
def test_tc_conv_strided_transposed_fp16(G, case):
    """Stride-2 convs (TMA element stride), transposed convs (8 output-parity classes) and fp16 operands on tcgen05."""
    dims, B, D, H, W, Cin, Cout, k, stride, transposed, f16 = case
    rng = _rng(sum(int(v) for v in case) + 77)
    q = (lambda t: t.half().float()) if f16 else (lambda t: t.bfloat16().float())
    if dims == 2:
        x = q(_t(rng, B, Cin, H, W))
        w = q(_t(rng, Cout, Cin, k, k, scale=math.sqrt(1.0 / (k * k * Cin))))
        ref = F.conv2d(x, w, stride=stride, padding=k // 2)
        res = q(_t(rng, *ref.shape))
        ref = F.relu(ref) + res
    elif transposed:
        x = q(_t(rng, B, Cin, D, H, W))
        w = q(_t(rng, Cin, Cout, 3, 3, 3, scale=math.sqrt(1.0 / (8 * Cin))))
        ref = F.conv_transpose3d(x, w, stride=2, padding=1, output_padding=1)
        res = q(_t(rng, *ref.shape))
        ref = F.relu(ref) + res
    else:
        x = q(_t(rng, B, Cin, D, H, W))
        w = q(_t(rng, Cout, Cin, 3, 3, 3, scale=math.sqrt(1.0 / (27 * Cin))))
        ref = F.conv3d(x, w, stride=stride, padding=1)
        res = q(_t(rng, *ref.shape))
        ref = F.relu(ref) + res
    out32, out16 = G.tc_conv(G.to_cl(x), w, npass=1, act_code=L.ACT_RELU, res_cl=G.to_cl(res), res_after_act=1, stride=stride,
                             transposed=bool(transposed), f16=f16)
    assert out32.shape == G.to_cl(ref).shape
    assert torch.isfinite(out32).all()
    assert G.rel_err(G.from_cl(out32), ref) < 1e-4        # operands exactly representable: fp32 summation order only
    assert G.rel_err(G.from_cl(out16), ref) < (2e-3 if f16 else 1.2e-2)   # 16-bit output rounding


def test_tc_conv_plan_rejects_a_layer_without_kernel_instance(G):
    """A layer whose tile (BN x KC) and pass mode have no kernel instance fails when it is planned, not at its first launch:
    a stride-2 3-D conv from 32 to 8 channels needs BN 16 x KC 32 in a single pass, which no layer of the network uses."""
    from rgbmanip_b200 import geometry
    lib = L.load()
    B, D, H, W, Cin, Cout = 1, 4, 28, 28, 32, 8
    x = torch.zeros((B, D, H, W, Cin), dtype=torch.float16, device=G.DEV)
    w = torch.zeros((27, 16, Cin), dtype=torch.float16, device=G.DEV)
    out = torch.zeros((B, D // 2, H // 2, W // 2, Cout), dtype=torch.float16, device=G.DEV)
    ep = G.epilogue(out_hi=out)
    a = G.act(x, None, B, D, H, W, Cin, 1)
    plan = C.c_void_p()
    with pytest.raises(L.AdpError, match=r"BN=16 KC=32 \(single pass\)"):
        L.check(lib.adp_conv_tc_plan(C.byref(plan), C.byref(a), L.ptr(w), None, Cout, 3, 3, 1, 1, C.byref(ep),
                                     C.byref(geometry.strided(True, D, H, W, 3, 2)), 148), "plan")
    assert plan.value is None


@pytest.mark.parametrize("f16", [1, 0])
def test_conv0_depth_ring_kernel(G, f16):
    """conv0 (3x3x3, 32 -> 8) as the depth-ring tcgen05 kernel (csrc/conv0_ring.cu) against F.conv3d."""
    from rgbmanip_b200 import geometry
    lib = L.load()
    rng = _rng(31 + f16)
    B, D, H, W = 2, 8, 12, 224
    dt = torch.float16 if f16 else torch.bfloat16
    x = _t(rng, B, 32, D, H, W).to(dt).float()
    w = _t(rng, 8, 32, 3, 3, 3, scale=math.sqrt(1.0 / (27 * 32))).to(dt).float()
    scale, shift = _t(rng, 8).abs() + 0.5, _t(rng, 8)
    ref = F.relu(F.conv3d(x, w, padding=1) * scale.view(1, -1, 1, 1, 1) + shift.view(1, -1, 1, 1, 1))
    xd = G.to_cl(x).to(dt).to(G.DEV).contiguous()
    wd = geometry.conv0_ring_weights(w).to(dt).to(G.DEV).contiguous()
    sc = torch.cat([scale, torch.zeros(8)]).to(G.DEV)
    sh = torch.cat([shift, torch.zeros(8)]).to(G.DEV)
    out = torch.full((B, D, H, W, 16), float("nan"), dtype=dt, device=G.DEV)
    err = torch.zeros(2, dtype=torch.int32, device=G.DEV)
    plan = C.c_void_p()
    a = G.act(xd, None, B, D, H, W, 32, f16)
    L.check(lib.adp_conv0_plan_create(C.byref(plan), C.byref(a), L.ptr(wd), L.ptr(sc), L.ptr(sh), L.ptr(out), 0, 148), "plan")
    L.check(lib.adp_conv0_run(plan, B, L.ptr(err), G.stream()), "run")
    torch.cuda.synchronize()
    lib.adp_conv0_free(plan)
    assert int(err[0].item()) == 0
    got = out.float().cpu()
    assert torch.isfinite(got).all()
    assert float(got[..., 8:].abs().max()) == 0.0
    assert G.rel_err(G.from_cl(got[..., :8].contiguous()), ref) < (2e-3 if f16 else 1.2e-2)   # 16-bit output rounding
    # same launch writing the 8 real channels space-to-depth(2): bit-identical values, [B,D/2,H/2,W/2,64] layout
    out2 = torch.full((B, D // 2, H // 2, W // 2, 64), float("nan"), dtype=dt, device=G.DEV)
    L.check(lib.adp_conv0_plan_create(C.byref(plan), C.byref(a), L.ptr(wd), L.ptr(sc), L.ptr(sh), L.ptr(out2), L.LAYOUT_S2D, 148), "plan")
    L.check(lib.adp_conv0_run(plan, B, L.ptr(err), G.stream()), "run")
    torch.cuda.synchronize()
    lib.adp_conv0_free(plan)
    assert torch.equal(geometry.from_s2d(out2.float().cpu()), got[..., :8])


@pytest.mark.parametrize("case", [(2, 4, 28, 28, 16, 8, 1), (1, 3, 56, 56, 32, 16, 1), (1, 4, 28, 28, 16, 8, 0), (1, 5, 20, 12, 32, 16, 1)],
                         ids=lambda c: "x".join(map(str, c)))
def test_tconv_fused_kernel(G, case):
    """Transposed conv + BN + ReLU + skip with the 8 parity classes fused in one tcgen05 kernel (csrc/tconv_fused.cu)."""
    lib = L.load()
    B, D, H, W, Cin, Cout, f16 = case
    rng = _rng(sum(case) + 5)
    dt = torch.float16 if f16 else torch.bfloat16
    x = _t(rng, B, Cin, D, H, W).to(dt).float()
    w = _t(rng, Cin, Cout, 3, 3, 3, scale=math.sqrt(1.0 / (8 * Cin))).to(dt).float()
    scale, shift = _t(rng, Cout).abs() + 0.5, _t(rng, Cout)
    res_c = 16 if Cout == 8 else Cout                               # the conv0 skip tensor is channel padded
    res = _t(rng, B, res_c, 2 * D, 2 * H, 2 * W).to(dt).float()
    ref = F.relu(F.conv_transpose3d(x, w, stride=2, padding=1, output_padding=1) * scale.view(1, -1, 1, 1, 1)
                 + shift.view(1, -1, 1, 1, 1)) + res[:, :Cout]
    xd = G.to_cl(x).to(dt).to(G.DEV).contiguous()
    wt = w.reshape(Cin, Cout, 27).permute(2, 1, 0).contiguous()
    bn = 16 if Cout <= 16 else 32
    if bn != Cout:
        wt = torch.cat([wt, torch.zeros(27, bn - Cout, Cin)], 1).contiguous()
    wd = wt.to(dt).to(G.DEV).contiguous()
    rd = G.to_cl(res).to(dt).to(G.DEV).contiguous()
    out = torch.full((B, 2 * D, 2 * H, 2 * W, Cout), float("nan"), dtype=dt, device=G.DEV)
    err = torch.zeros(1, dtype=torch.int32, device=G.DEV)
    plan = C.c_void_p()
    a = G.act(xd, None, B, D, H, W, Cin, f16)
    sc, sh = scale.to(G.DEV), shift.to(G.DEV)
    L.check(lib.adp_tconv_plan_create(C.byref(plan), C.byref(a), L.ptr(wd), Cout, L.ptr(sc), L.ptr(sh), L.ptr(rd), res_c, L.ptr(out),
                                      0, 148), "plan")
    L.check(lib.adp_tconv_run(plan, B, L.ptr(err), G.stream()), "run")
    torch.cuda.synchronize()
    lib.adp_tconv_free(plan)
    assert int(err.item()) == 0
    got = out.float().cpu()
    assert torch.isfinite(got).all()
    assert G.rel_err(G.from_cl(got), ref) < (2e-3 if f16 else 1.2e-2)       # 16-bit output rounding
    if Cout != 8:
        return
    # space-to-depth(2) skip / output tensors (the level-0 layout of the engine): same values, [B,D,H,W,64]
    from rgbmanip_b200 import geometry
    rd2 = geometry.to_s2d(G.to_cl(res)[..., :Cout].contiguous()).to(dt).to(G.DEV).contiguous()
    out2 = torch.full((B, D, H, W, 8 * Cout), float("nan"), dtype=dt, device=G.DEV)
    L.check(lib.adp_tconv_plan_create(C.byref(plan), C.byref(a), L.ptr(wd), Cout, L.ptr(sc), L.ptr(sh), L.ptr(rd2), 0, L.ptr(out2),
                                      L.LAYOUT_S2D, 148), "plan")
    L.check(lib.adp_tconv_run(plan, B, L.ptr(err), G.stream()), "run")
    torch.cuda.synchronize()
    lib.adp_tconv_free(plan)
    assert int(err.item()) == 0
    assert torch.equal(geometry.from_s2d(out2.float().cpu()), got)


def test_level0_s2d_convs_on_generic_kernel(G):
    """conv1 (stride 2) reading and conv11 (transposed + skip) writing space-to-depth(2) tensors as stride-1 2x2x2-tap
    convolutions on the generic tcgen05 kernel (geometry.strided_s2d / transposed_s2d)."""
    from rgbmanip_b200 import geometry
    lib = L.load()
    rng = _rng(77)
    B, D2, H2, W2 = 1, 3, 16, 32
    dt = torch.float16

    def run(x_cl, wt, cout, geom, **ep_kw):
        xd = x_cl.to(dt).to(G.DEV).contiguous()
        wd = wt.to(dt).to(G.DEV).contiguous()
        out32 = torch.full((B, D2, H2, W2, cout), float("nan"), dtype=torch.float32, device=G.DEV)
        ep = G.epilogue(None, None, out32, **ep_kw)
        a = G.act(xd, None, B, D2, H2, W2, x_cl.shape[-1], 1)
        err = torch.zeros(1, dtype=torch.int32, device=G.DEV)
        plan = C.c_void_p()
        L.check(lib.adp_conv_tc_plan(C.byref(plan), C.byref(a), L.ptr(wd), None, cout, 1, 1, 1, 1, C.byref(ep), C.byref(geom), 148), "plan")
        L.check(lib.adp_conv_tc_run(plan, B, L.ptr(err), G.stream()), "run")
        torch.cuda.synchronize()
        lib.adp_conv_tc_free(plan)
        assert int(err.item()) == 0
        return out32.cpu()

    # conv1: Conv3d(8 -> 16, k3, s2, p1) on the s2d tensor
    x = _t(rng, B, 8, 2 * D2, 2 * H2, 2 * W2).half().float()
    w = _t(rng, 16, 8, 3, 3, 3, scale=0.1).half().float()
    ref = F.conv3d(x, w, stride=2, padding=1)
    got = run(geometry.to_s2d(G.to_cl(x)), geometry.strided_s2d_weights(w), 16, geometry.strided_s2d(D2, H2, W2))
    assert G.rel_err(G.from_cl(got), ref) < 1e-5
    # conv11: ConvTranspose3d(16 -> 8, k3, s2, p1, op1) + skip, output in s2d layout
    x = _t(rng, B, 16, D2, H2, W2).half().float()
    w = _t(rng, 16, 8, 3, 3, 3, scale=0.1).half().float()
    res = _t(rng, B, 8, 2 * D2, 2 * H2, 2 * W2).half().float()
    ref = F.relu(F.conv_transpose3d(x, w, stride=2, padding=1, output_padding=1)) + res
    rd = geometry.to_s2d(G.to_cl(res)).to(dt).to(G.DEV).contiguous()
    got = run(G.to_cl(x), geometry.transposed_s2d_weights(w), 64, geometry.transposed_s2d(D2, H2, W2),
              act_code=L.ACT_RELU, res_hi=rd, res_after_act=1)
    assert G.rel_err(G.from_cl(geometry.from_s2d(got)), ref) < 1e-5


# ------------------------------------------------------------------------------------------------ backbone helpers
def test_maxpool_psp_upsample(G):
    lib = L.load()
    rng = _rng(3)
    st = G.stream()
    # max-pool
    x = _t(rng, 2, 64, 30, 26)
    xh, xl = G.split(G.to_cl(x))
    oh = torch.zeros((2, 15, 13, 64), dtype=torch.bfloat16, device=G.DEV)
    ol = torch.zeros_like(oh)
    L.check(lib.adp_maxpool3x3s2(C.byref(G.act(xh, xl, 2, 1, 30, 26, 64)), C.byref(G.act(oh, ol, 2, 1, 15, 13, 64)), 2, st), "mp")
    ref = F.max_pool2d(G.from_cl(G.val(xh, xl).cpu()), 3, 2, 1)
    assert G.rel_err(G.from_cl(G.val(oh, ol).cpu()), ref) < 1e-5
    # pyramid pooling + concat + x2 upsample against the oracle's psp_module + interpolate
    sd = weights.init_state_dict(2)
    f = _t(rng, 2, 512, 28, 28).abs()
    fh, fl = G.split(G.to_cl(f))
    wpsp = torch.stack([torch.from_numpy(sd[f"img_extractor.psp.stages.{s}.1.weight"]).reshape(128, 512).t().contiguous()
                        for s in range(4)]).contiguous().to(G.DEV)
    pooled = torch.zeros((2, 50, 512), device=G.DEV)
    priors = torch.zeros((2, 50, 128), device=G.DEV)
    # the product path: the 512 feature channels sit in front of the concat tensor (written there by layer4's last conv through
    # the epilogue channel pitch), the priors are filled in behind them, then the whole tensor is upsampled
    ch = torch.zeros((2, 28, 28, 1024), dtype=torch.bfloat16, device=G.DEV)
    cl = torch.zeros_like(ch)
    ch[..., :512].copy_(fh); cl[..., :512].copy_(fl)
    fa = G.act(ch, cl, 2, 1, 28, 28, 512)
    ca = G.act(ch, cl, 2, 1, 28, 28, 1024)
    L.check(lib.adp_psp_priors(C.byref(fa), 1024, L.ptr(wpsp), L.ptr(pooled), L.ptr(priors), 2, st), "psp")
    L.check(lib.adp_psp_fill_priors(L.ptr(priors), C.byref(ca), 512, 2, st), "fill")
    uh = torch.zeros((2, 56, 56, 1024), dtype=torch.bfloat16, device=G.DEV)
    ul = torch.zeros_like(uh)
    L.check(lib.adp_upsample2x(C.byref(ca), C.byref(G.act(uh, ul, 2, 1, 56, 56, 1024)), 2, st), "cat")
    fin = G.from_cl(G.val(fh, fl).cpu())
    ref = F.interpolate(O.psp_module(sd, fin), scale_factor=2, mode="bilinear", align_corners=True)
    assert G.rel_err(G.from_cl(G.val(uh, ul).cpu()), ref) < 5e-5
    # plain x2 upsample
    y = _t(rng, 1, 64, 12, 20)
    yh, yl = G.split(G.to_cl(y))
    zh = torch.zeros((1, 24, 40, 64), dtype=torch.bfloat16, device=G.DEV)
    zl = torch.zeros_like(zh)
    L.check(lib.adp_upsample2x(C.byref(G.act(yh, yl, 1, 1, 12, 20, 64)), C.byref(G.act(zh, zl, 1, 1, 24, 40, 64)), 1, st), "up")
    ref = F.interpolate(G.from_cl(G.val(yh, yl).cpu()), scale_factor=2, mode="bilinear", align_corners=True)
    assert G.rel_err(G.from_cl(G.val(zh, zl).cpu()), ref) < 5e-5


@pytest.mark.parametrize("case", [(2, 12, 20, 32, 64, 1), (1, 28, 28, 64, 16, 1), (2, 7, 9, 64, 8, 0), (1, 5, 30, 16, 64, 0)],
                         ids=lambda c: "x".join(map(str, c)))
def test_upconv_restructured_matches_oracle(G, case):
    """PSPUpsample (pspnet.py:97-107) as per-tap 1x1 GEMM at low resolution (adp_conv_tc) + adp_upconv_blend against
    conv3x3(interpolate(x, 2, bilinear, align_corners=True)) + PReLU in torch fp32: fp16 planes and bf16 hi/lo planes, odd sizes,
    borders (the conv's zero padding applies to the upsampled image)."""
    lib = L.load()
    B, h, w, Cin, Cout, f16 = case
    rng = _rng(31)
    x = _t(rng, B, Cin, h, w)
    wgt = _t(rng, Cout, Cin, 3, 3, scale=1.0 / np.sqrt(9 * Cin))
    bias = _t(rng, Cout)
    slope = 0.25
    ref = F.prelu(F.conv2d(F.interpolate(x, scale_factor=2, mode="bilinear", align_corners=True), wgt, bias, padding=1),
                  torch.tensor([slope]))
    w1 = wgt.permute(2, 3, 0, 1).reshape(9 * Cout, Cin, 1, 1).contiguous()        # channel = (ky*3+kx)*Cout + co
    q32, _ = G.tc_conv(G.to_cl(x), w1, npass=2 if f16 else 3, f16=f16)
    dev = G.DEV
    if f16:
        qh, ql = q32.to(torch.float16).to(dev).contiguous(), None
        oh, ol = torch.zeros((B, 2 * h, 2 * w, Cout), dtype=torch.float16, device=dev), None
    else:
        qh, ql = G.split(q32)
        oh = torch.zeros((B, 2 * h, 2 * w, Cout), dtype=torch.bfloat16, device=dev)
        ol = torch.zeros_like(oh)
    bd = bias.to(dev)
    L.check(lib.adp_upconv_blend(C.byref(G.act(qh, ql, B, 1, h, w, 9 * Cout, f16)), C.byref(G.act(oh, ol, B, 1, 2 * h, 2 * w, Cout, f16)),
                                 L.ptr(bd), slope, B, G.stream()), "upconv_blend")
    torch.cuda.synchronize()
    got = G.from_cl(G.val(oh, ol).cpu())
    # fp16 planes: q and the result are rounded to 11 bits; bf16 hi/lo: 16 bits
    assert G.rel_err(got, ref) < (2e-3 if f16 else 1e-4), G.rel_err(got, ref)


def test_maxpool_psp_upsample_fp16_planes(G):
    """Same helpers on a single fp16 activation plane (the fp16x2 backbone)."""
    lib = L.load()
    rng = _rng(5)
    st = G.stream()
    h = lambda t: G.to_cl(t).to(torch.float16).to(G.DEV).contiguous()
    A = lambda t, *dims: G.act(t, None, *dims, 1)
    x = _t(rng, 2, 64, 30, 26)
    xh = h(x)
    oh = torch.zeros((2, 15, 13, 64), dtype=torch.float16, device=G.DEV)
    L.check(lib.adp_maxpool3x3s2(C.byref(A(xh, 2, 1, 30, 26, 64)), C.byref(A(oh, 2, 1, 15, 13, 64)), 2, st), "mp")
    ref = F.max_pool2d(G.from_cl(xh.float().cpu()), 3, 2, 1)
    assert G.rel_err(G.from_cl(oh.float().cpu()), ref) == 0.0
    sd = weights.init_state_dict(2)
    f = _t(rng, 2, 512, 28, 28).abs()
    fh = h(f)
    wpsp = torch.stack([torch.from_numpy(sd[f"img_extractor.psp.stages.{s}.1.weight"]).reshape(128, 512).t().contiguous()
                        for s in range(4)]).contiguous().to(G.DEV)
    pooled = torch.zeros((2, 50, 512), device=G.DEV)
    priors = torch.zeros((2, 50, 128), device=G.DEV)
    ch = torch.zeros((2, 28, 28, 1024), dtype=torch.float16, device=G.DEV)
    ch[..., :512].copy_(fh)
    fa, ca = A(ch, 2, 1, 28, 28, 512), A(ch, 2, 1, 28, 28, 1024)
    L.check(lib.adp_psp_priors(C.byref(fa), 1024, L.ptr(wpsp), L.ptr(pooled), L.ptr(priors), 2, st), "psp")
    L.check(lib.adp_psp_fill_priors(L.ptr(priors), C.byref(ca), 512, 2, st), "fill")
    uh = torch.zeros((2, 56, 56, 1024), dtype=torch.float16, device=G.DEV)
    uq = torch.zeros((2, 56, 56, 1024), dtype=torch.uint8, device=G.DEV)
    L.check(lib.adp_upsample2x(C.byref(ca), C.byref(G.act(uh, None, 2, 1, 56, 56, 1024, 1, uq)), 2, st), "cat")
    ref = F.interpolate(O.psp_module(sd, G.from_cl(fh.float().cpu())), scale_factor=2, mode="bilinear", align_corners=True)
    assert G.rel_err(G.from_cl(uh.float().cpu()), ref) < 6e-4
    # the fp8 twin the upsample writes for the fp16f8 low-order pass of up_1: e4m3(value / 2)
    want_q = G.from_e4m3(G.to_e4m3(G.to_cl(ref) * 0.5)) * 2.0
    got_q = G.from_e4m3(uq.cpu()) * 2.0
    assert float(((got_q - want_q).abs() > 0).float().mean()) < 0.02 and float((got_q - want_q).abs().max()) <= 0.13 * float(want_q.abs().max())
    y = _t(rng, 1, 64, 12, 20)
    yh = h(y)
    zh = torch.zeros((1, 24, 40, 64), dtype=torch.float16, device=G.DEV)
    L.check(lib.adp_upsample2x(C.byref(A(yh, 1, 1, 12, 20, 64)), C.byref(A(zh, 1, 1, 24, 40, 64)), 1, st), "up")
    ref = F.interpolate(G.from_cl(yh.float().cpu()), scale_factor=2, mode="bilinear", align_corners=True)
    assert G.rel_err(G.from_cl(zh.float().cpu()), ref) < 6e-4


# ------------------------------------------------------------------------------------------------ preprocess
def _preprocess(G, rgb, mask, K, choose=None, seed=0, frame_id0=0):
    lib = L.load()
    Fn = rgb.shape[0]
    dev = G.DEV
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    rgb_d, mask_d, K_d = t(rgb), t(mask), t(K.astype(np.float64))
    dt = {torch.float32: L.DT_F32, torch.float64: L.DT_F64, torch.bool: L.DT_U8, torch.uint8: L.DT_U8}
    H, W = rgb.shape[1], rgb.shape[2]
    out = dict(bbox=torch.zeros((Fn, 4), dtype=torch.int32, device=dev), win=torch.zeros((Fn, 4), dtype=torch.int32, device=dev),
               Kp=torch.zeros((Fn, 9), dtype=torch.float64, device=dev), valid=torch.zeros(Fn, dtype=torch.uint8, device=dev),
               crops=torch.zeros((Fn, 224, 224, 3), device=dev), choose=torch.zeros((Fn, 1024), dtype=torch.int32, device=dev),
               counts=torch.zeros(Fn, dtype=torch.int32, device=dev))
    mode = 0
    if choose is not None:
        out["choose"].copy_(torch.from_numpy(choose).to(torch.int32))
        mode = 1
    L.check(lib.adp_preprocess(L.ptr(rgb_d), dt[rgb_d.dtype], L.ptr(mask_d), dt[mask_d.dtype], L.ptr(K_d), 9, Fn, H, W, 224,
                               1024, seed, mode, frame_id0, L.ptr(out["bbox"]), L.ptr(out["win"]), L.ptr(out["Kp"]), L.ptr(out["valid"]),
                               L.ptr(out["crops"]), L.ptr(out["choose"]), L.ptr(out["counts"]), G.stream()), "preprocess")
    torch.cuda.synchronize()
    return {k: v.cpu().numpy() for k, v in out.items()}


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_preprocess_matches_oracle(G, dtype):
    batch = synth.make_batch(16, seed=5, dtype=dtype)
    mask = batch.mask1 if dtype == np.float32 else batch.mask1.astype(np.float64)
    got = _preprocess(G, batch.rgb1, mask, batch.K)
    n_checked = 0
    for e in range(16):
        ys, xs = np.nonzero(batch.mask1[e])
        if len(ys) == 0:
            assert got["valid"][e] == 0
            continue
        win = O.get_bbox(int(ys.min()), int(xs.min()), int(ys.max()), int(xs.max()))
        np.testing.assert_array_equal(got["win"][e], win)                         # integer work: bit exact
        np.random.seed(1)
        v, ch, _, Kp = O.prepare_model_input(batch.rgb1[e], batch.mask1[e], batch.K[e])
        nz = O.resize_nearest(batch.mask1[e][win[0]:win[1], win[2]:win[3]].astype(np.float32), 224).flatten().nonzero()[0]
        assert got["counts"][e] == len(nz)
        np.testing.assert_array_equal(got["Kp"][e].reshape(3, 3), Kp)
        np.testing.assert_allclose(got["crops"][e].transpose(2, 0, 1), v, rtol=0, atol=2e-5)
        c = got["choose"][e]
        if len(nz) <= 1024:
            np.testing.assert_array_equal(c, np.pad(nz, (0, 1024 - len(nz)), "wrap"))   # wrap padding: bit exact
        else:                                                                      # device sampling: a sorted 1024-subset
            assert len(np.unique(c)) == 1024 and (np.diff(c) > 0).all() and np.isin(c, nz).all()
        n_checked += 1
    assert n_checked >= 12


def test_preprocess_sampling_is_uniform_and_seeded(G):
    batch = synth.make_batch(4, seed=9, special=False)
    a = _preprocess(G, batch.rgb1, batch.mask1, batch.K, seed=1)["choose"]
    b = _preprocess(G, batch.rgb1, batch.mask1, batch.K, seed=1)["choose"]
    c = _preprocess(G, batch.rgb1, batch.mask1, batch.K, seed=2)["choose"]
    np.testing.assert_array_equal(a, b)
    assert (a != c).any()
    # the sampler is keyed by (seed, frame id): frames 2..3 launched on their own with frame_id0 = 2 draw the same subsets
    d = _preprocess(G, batch.rgb1[2:], batch.mask1[2:], batch.K[2:], seed=1, frame_id0=2)["choose"]
    np.testing.assert_array_equal(d, a[2:])
    # selection probability must not depend on the position: compare the mean rank of the picks with n/2
    win = None
    for e in range(4):
        ys, xs = np.nonzero(batch.mask1[e])
        win = O.get_bbox(int(ys.min()), int(xs.min()), int(ys.max()), int(xs.max()))
        nz = O.resize_nearest(batch.mask1[e][win[0]:win[1], win[2]:win[3]].astype(np.float32), 224).flatten().nonzero()[0]
        if len(nz) > 4096:
            ranks = np.searchsorted(nz, a[e])
            assert abs(ranks.mean() / len(nz) - 0.5) < 0.04


# ------------------------------------------------------------------------------------------------ volume / decode / fit
def _stereo_inputs(seed=0):
    batch = synth.make_batch(2, seed=seed, special=False)
    np.random.seed(seed)
    views = []
    for e in range(2):
        v1 = O.prepare_model_input(batch.rgb1[e], batch.mask1[e], batch.K[e])
        v2 = O.prepare_model_input(batch.rgb2[e], batch.mask2[e], batch.K[e])
        views.append((v1, v2))
    return batch, views


def test_warp_matrices_and_volume(G):
    lib = L.load()
    batch, views = _stereo_inputs(1)
    rng = _rng(4)
    dev = G.DEV
    f1 = _t(rng, 2, 32, 224, 224)
    f2 = _t(rng, 2, 32, 224, 224)
    Kp1 = torch.from_numpy(np.stack([v[0][3] for v in views]).reshape(2, 9)).to(dev)
    Kp2 = torch.from_numpy(np.stack([v[1][3] for v in views]).reshape(2, 9)).to(dev)
    E1 = torch.from_numpy(batch.E1.reshape(2, 16)).to(dev)
    E2 = torch.from_numpy(batch.E2.reshape(2, 16)).to(dev)
    Mw = torch.zeros((2, 12), device=dev)
    L.check(lib.adp_warp_matrices(L.ptr(Kp1), L.ptr(E1), L.ptr(Kp2), L.ptr(E2), L.ptr(Mw), None, None, None, 2, G.stream()), "wm")
    P1 = np.stack([O.projection(views[e][0][3], batch.E1[e]) for e in range(2)])
    P2 = np.stack([O.projection(views[e][1][3], batch.E2[e]) for e in range(2)])
    M = P2 @ np.linalg.inv(P1)
    want = np.concatenate([M[:, :3, :3].reshape(2, 9), M[:, :3, 3]], 1)
    np.testing.assert_allclose(Mw.cpu().numpy(), want, rtol=2e-6, atol=1e-6)
    depths = torch.from_numpy(O.depth_hypotheses()).to(dev)
    vol = torch.zeros((2, 24, 224, 224, 32), dtype=torch.float16, device=dev)
    f1, f2 = f1.half().float(), f2.half().float()            # the builder reads the fp16 twin of the feature map
    f1d, f2d = G.to_cl(f1).half().to(dev).contiguous(), G.to_cl(f2).half().to(dev).contiguous()
    L.check(lib.adp_build_volume(L.ptr(f1d), L.ptr(f2d), L.ptr(Mw), L.ptr(depths), L.ptr(vol), 2, 24, 224, 224, 32, 1, G.stream()), "vol")
    torch.cuda.synchronize()
    ref = f1[:, :, None] + O.homo_warping(f2, torch.from_numpy(P2).float(), torch.from_numpy(P1).float(),
                                          torch.from_numpy(O.depth_hypotheses())[None].repeat(2, 1))
    got = vol.float().cpu().permute(0, 4, 1, 2, 3)
    diff = (got - ref).abs()
    # fp16 storage (2^-11 relative) plus sample positions that agree to ~1e-4 px; a handful of voxels sit on a
    # bilinear cell boundary or the zero-padding edge where that flips a corner
    assert float(diff.mean()) < 6e-3
    assert float((diff > 0.05).float().mean()) < 2e-4


@pytest.mark.parametrize("case", ["shift", "rot40_scale1.3", "shrink0.6"])
def test_volume_tiled_fp16_features(G, case):
    """adp_build_volume on fp16 feature maps (the engine's path: shared-memory staged footprints, direct-gather fallback
    when the footprint of a tile exceeds the staging buffer) against grid_sample with the reference's coordinate convention
    (network_v5.py:389-413).  The warp is an affine map of the pixel grid, the same for every depth plane."""
    lib = L.load()
    rng = _rng(41)
    B, D, S = 2, 8, 224
    th, sc, tx, ty = {"shift": (0.0, 1.0, 3.3, -2.6), "rot40_scale1.3": (math.radians(40), 1.3, 60.0, -80.0),
                      "shrink0.6": (math.radians(-8), 0.6, 40.0, 50.0)}[case]
    A = np.array([[sc * math.cos(th), -sc * math.sin(th), tx], [sc * math.sin(th), sc * math.cos(th), ty], [0, 0, 1]], np.float32)
    Mw = torch.from_numpy(np.tile(np.concatenate([A.reshape(9), np.zeros(3, np.float32)]), (B, 1))).to(G.DEV)
    f1 = _t(rng, B, 32, S, S).half()
    f2 = _t(rng, B, 32, S, S).half()
    depths = torch.from_numpy(O.depth_hypotheses()[:D].copy()).to(G.DEV)
    vol = torch.zeros((B, D, S, S, 32), dtype=torch.float16, device=G.DEV)
    f1d, f2d = G.to_cl(f1).to(G.DEV).contiguous(), G.to_cl(f2).to(G.DEV).contiguous()
    L.check(lib.adp_build_volume(L.ptr(f1d), L.ptr(f2d), L.ptr(Mw), L.ptr(depths), L.ptr(vol), B, D, S, S, 32, 1, G.stream()), "vol")
    torch.cuda.synchronize()
    ys, xs = torch.meshgrid(torch.arange(S, dtype=torch.float32), torch.arange(S, dtype=torch.float32), indexing="ij")
    px = A[0, 0] * xs + A[0, 1] * ys + A[0, 2]
    py = A[1, 0] * xs + A[1, 1] * ys + A[1, 2]
    grid = torch.stack([px / ((S - 1) / 2) - 1, py / ((S - 1) / 2) - 1], -1)[None].repeat(B, 1, 1, 1)
    ref = f1.float() + F.grid_sample(f2.float(), grid, mode="bilinear", padding_mode="zeros", align_corners=False)
    got = vol.float().cpu().permute(0, 4, 1, 2, 3)
    for d in range(D):      # every depth plane sees the same warp
        diff = (got[:, :, d] - ref).abs()
        assert float(diff.max()) < 0.02 and float(diff.mean()) < 1e-3, (d, float(diff.max()), float(diff.mean()))   # fp16 storage of O(1..5) values


def test_conv11_tma_epilogue_is_bit_identical(G, monkeypatch):
    """conv11 on the slab kernel with the TMA epilogue (residual tiles by TMA load, results by TMA store through a swizzled
    staging tile) against the per-lane epilogue it replaces (ADP_NO_BULK_EPI): the same arithmetic per element, so the
    s2d output tensor must agree bit for bit, and with it every later stage."""
    from rgbmanip_b200.engine import Engine
    sd = weights.init_state_dict(0)
    batch, views = _stereo_inputs(3)
    outs = []
    for bulk in (True, False):
        if bulk:
            monkeypatch.delenv("ADP_NO_BULK_EPI", raising=False)
        else:
            monkeypatch.setenv("ADP_NO_BULK_EPI", "1")
        eng = Engine(sd, device=G.DEV, max_envs=2, debug=True)
        g = torch.Generator().manual_seed(5)
        feat = torch.randn((4, 224, 224, 32), generator=g) * 0.5
        eng.feat.copy_(feat)
        eng.feat16.copy_(eng.feat)
        eng.choose[:2].copy_(torch.from_numpy(np.stack([v[0][1] for v in views])).to(torch.int32))
        eng.Kp[:2].copy_(torch.from_numpy(np.stack([v[0][3] for v in views]).reshape(2, 9)))
        eng.Kp[2:4].copy_(torch.from_numpy(np.stack([v[1][3] for v in views]).reshape(2, 9)))
        eng.valid.fill_(1)
        eng.stereo(2, torch.from_numpy(batch.E1).to(G.DEV), torch.from_numpy(batch.E2).to(G.DEV))
        torch.cuda.synchronize()
        eng.check_error_flag()
        outs.append((eng.cr_taps["conv11"].value().cpu().clone(), eng.bbox.cpu().clone()))
        eng.close()
    assert float(outs[0][0].abs().max()) > 0
    assert torch.equal(outs[0][0], outs[1][0])
    assert torch.equal(outs[0][1], outs[1][1])


def _run_costreg_decode(G, sd, eng_kw):
    from rgbmanip_b200.engine import Engine
    eng = Engine(sd, device=G.DEV, max_envs=2, debug=True, **eng_kw)
    return eng


def test_costreg_and_decode_match_oracle(G):
    """Feed oracle feature maps into the device volume/cost-regularisation/decode stages."""
    from rgbmanip_b200.engine import Engine
    sd = weights.init_state_dict(0)
    batch, views = _stereo_inputs(2)
    eng = Engine(sd, device=G.DEV, max_envs=2, debug=True)
    dev = G.DEV
    with torch.no_grad():
        img1 = torch.from_numpy(np.stack([v[0][0] for v in views])).float()
        img2 = torch.from_numpy(np.stack([v[1][0] for v in views])).float()
        f1, f2 = O.pspnet(sd, img1), O.pspnet(sd, img2)
    eng.feat[:2].copy_(G.to_cl(f1))
    eng.feat[2:4].copy_(G.to_cl(f2))
    eng.feat16.copy_(eng.feat)           # the volume builder reads the fp16 twin written by the `final` conv
    ch1 = np.stack([v[0][1] for v in views])
    eng.choose[:2].copy_(torch.from_numpy(ch1).to(torch.int32))
    eng.Kp[:2].copy_(torch.from_numpy(np.stack([v[0][3] for v in views]).reshape(2, 9)))
    eng.Kp[2:4].copy_(torch.from_numpy(np.stack([v[1][3] for v in views]).reshape(2, 9)))
    eng.valid.fill_(1)
    E1 = torch.from_numpy(batch.E1).to(dev)
    E2 = torch.from_numpy(batch.E2).to(dev)
    eng.stereo(2, E1, E2)
    torch.cuda.synchronize()
    eng.check_error_flag()
    P1 = torch.from_numpy(np.stack([O.projection(views[e][0][3], batch.E1[e]) for e in range(2)])).float()
    P2 = torch.from_numpy(np.stack([O.projection(views[e][1][3], batch.E2[e]) for e in range(2)])).float()
    dv = torch.from_numpy(O.depth_hypotheses())[None].repeat(2, 1)
    tap = O.Taps(record=True)
    with torch.no_grad():
        fused = f1[:, :, None] + O.homo_warping(f2, P2, P1, dv)
        logits_vol = O.cost_reg_net(sd, fused, tap)
        ref = O.decode_view(sd, f1, fused, logits_vol, torch.from_numpy(ch1), dv, True, tap)
    # U-Net stages: bf16 storage of every activation -> a few 1e-3 of the activation scale
    for nm in ("conv0", "conv2", "conv4", "conv6", "conv7", "conv9", "conv11"):
        got = G.from_cl(eng.cr_taps[nm].value().cpu())
        want = tap.store[f"cr.{nm}"]
        if got.shape[1] != want.shape[1]:          # conv0's output carries 8 zero pad channels
            assert float(got[:, want.shape[1]:].abs().max()) == 0.0
            got = got[:, :want.shape[1]]
        assert G.rel_err(got, want) < 2e-2, nm
        assert float((got - want).abs().mean() / want.abs().mean()) < 4e-3, nm
    logits = eng.dbg_logits.cpu().permute(0, 2, 1)
    assert float((logits - tap.store["logits"]).abs().max()) < 0.08          # logits span ~ +-10
    np.testing.assert_allclose(eng.nocs.cpu().numpy(), ref["nocs"].numpy(), rtol=0, atol=2e-4)      # fp32 MLP (last layer gain 16) + tanhf
    assert float((eng.depth.cpu() - ref["depth"]).abs().max()) < 6e-3         # per-pixel depth, metres (bf16 U-Net)
    assert float((eng.depth.cpu() - ref["depth"]).abs().mean()) < 8e-4
    assert float((eng.dbg_fused.cpu().permute(0, 2, 1) - tap.store["fused_pts"]).abs().max()) < 2e-2
    Rg = eng.R.cpu().numpy().reshape(2, 3, 3)
    for e in range(2):
        assert O.rotation_angle_deg(Rg[e], ref["r"][e].numpy()) < 0.05        # degrees
    # fit on the device outputs vs the oracle's fit on the same numbers (fp32 vs fp64 arithmetic only)
    box = eng.bbox.cpu().numpy()
    for e in range(2):
        t, s = O.compute_scale_and_translation(eng.depth[e].cpu().numpy(), eng.nocs[e].cpu().numpy(), ch1[e], views[e][0][3], 224, Rg[e])
        assert abs(float(eng.scale[e]) - s) / s < 2e-6
        np.testing.assert_allclose(eng.trans[e].cpu().numpy(), t, rtol=0, atol=2e-6)
        want = O.box_from_fit(eng.nocs[e].cpu().numpy(), s, Rg[e], t, batch.E1[e])
        np.testing.assert_allclose(box[e], want, rtol=0, atol=5e-6)
    eng.close()


def test_fit_median_is_exact_and_sentinel(G):
    lib = L.load()
    dev = G.DEV
    rng = _rng(12)
    B, P = 4, 1024
    nocs = (rng.random((B, P, 3)).astype(np.float32) - 0.5)
    nocs[2] *= 0.001                                  # no pair passes |dn| > 0.01 -> NaN scale -> sentinel box
    depth = (0.8 + 0.05 * rng.standard_normal((B, P))).astype(np.float32)
    choose = np.stack([np.sort(rng.choice(224 * 224, P, replace=False)) for _ in range(B)]).astype(np.int32)
    Kp = np.tile(np.array([[800.0, 0, 100.5], [0, 800.0, 120.25], [0, 0, 1]]).reshape(1, 9), (B, 1))
    R = np.tile(np.eye(3, dtype=np.float32).reshape(1, 9), (B, 1))
    E = np.tile(np.eye(4).reshape(1, 16), (B, 1))
    E[1, 3] = 0.3
    valid = np.array([1, 1, 1, 0], np.uint8)
    t = lambda a: torch.from_numpy(a).to(dev)
    bbox = torch.zeros((B, 8, 3), dtype=torch.float64, device=dev)
    scale = torch.zeros(B, dtype=torch.float64, device=dev)
    trans = torch.zeros((B, 3), dtype=torch.float64, device=dev)
    args = [t(nocs), t(depth), t(choose), t(Kp), t(R), t(E), t(valid)]
    L.check(lib.adp_fit(*[L.ptr(a) for a in args], L.ptr(bbox), L.ptr(scale), L.ptr(trans), None, None, B, P, 224, G.stream()), "fit")
    torch.cuda.synchronize()
    for e in (0, 1):
        cam = O.back_project(depth[e], choose[e], Kp[e].reshape(3, 3))
        s = O.compute_scale(cam, nocs[e])
        assert abs(float(scale[e]) - s) / s < 1e-6     # exact order statistic; fp32 vs fp64 distance arithmetic
    np.testing.assert_array_equal(bbox[2].cpu().numpy(), O.DEFAULT_BBOX)
    np.testing.assert_array_equal(bbox[3].cpu().numpy(), O.DEFAULT_BBOX)


# ------------------------------------------------------------------------------------------------ backbone end to end
@pytest.mark.parametrize("precision,tol", [("fp16x2", 3e-3), ("bf16x3", 2e-3), ("bf16", 6e-2)])
def test_backbone_matches_oracle(G, precision, tol):
    from rgbmanip_b200.engine import Engine
    sd = weights.init_state_dict(0)
    rng = _rng(21)
    img = _t(rng, 2, 3, 224, 224)
    eng = Engine(sd, device=G.DEV, max_envs=1, precision=precision)
    eng.crops.copy_(G.to_cl(img))
    eng.run_backbone(2)
    torch.cuda.synchronize()
    eng.check_error_flag()
    tap = O.Taps(record=True)
    with torch.no_grad():
        ref = O.pspnet(sd, img, tap)
    errs = {}
    for nm, buf in eng.taps.items():
        key = nm if nm in tap.store else nm
        errs[nm] = G.rel_err(G.from_cl(buf.value(2).cpu()), tap.store[key])
    got = G.from_cl(eng.feat[:2].cpu())
    errs["feat"] = G.rel_err(got, ref)
    bad = {k: v for k, v in errs.items() if not v < tol}
    assert not bad, (bad, errs)
    kinds = [getattr(op, "kind", None) for _, op in eng.backbone_ops]
    assert kinds.count("tc") >= 40, kinds   # every backbone conv runs on the tcgen05 kernel (there is no other conv path)
    eng.close()


def test_fit_umeyama_ransac_matches_oracle(G):
    """Branch B (align.py:44-102): same 128 x 5 sample table on both sides -> same similarity transform and box."""
    lib = L.load()
    dev = G.DEV
    rng = _rng(44)
    B, P = 3, 1024
    nocs = (rng.random((B, P, 3)).astype(np.float32) - 0.5)
    Kp = np.tile(np.array([[400.0, 0, 112.0], [0, 400.0, 112.0], [0, 0, 1]]).reshape(1, 9), (B, 1))
    choose = np.zeros((B, P), np.int32)
    depth = np.zeros((B, P), np.float32)
    E = np.tile(np.eye(4).reshape(1, 16), (B, 1))
    E[1, 3] = 0.2
    for b in range(B):
        Rt = np.linalg.qr(rng.standard_normal((3, 3)))[0]
        if np.linalg.det(Rt) < 0:
            Rt[:, 0] *= -1
        cam = 0.2 * (Rt @ nocs[b].T.astype(np.float64)).T + np.array([0.02, -0.01, 0.8])
        px = np.clip(np.rint(400.0 * cam[:, 0] / cam[:, 2] + 112.0), 0, 223).astype(np.int32)    # the pixel the point lands on
        py = np.clip(np.rint(400.0 * cam[:, 1] / cam[:, 2] + 112.0), 0, 223).astype(np.int32)
        choose[b] = py * 224 + px
        depth[b] = (cam[:, 2] + 0.002 * rng.standard_normal(P)).astype(np.float32)
    depth[2, ::2] += 0.3                                                               # half the points are gross outliers
    depth[1, :] = rng.random(P).astype(np.float32) + 0.3                                # env 1: no consistent model at all
    ridx = rng.integers(0, P, size=(B, 128, 5)).astype(np.int32)
    t = lambda a: torch.from_numpy(a).to(dev)
    bbox = torch.zeros((B, 8, 3), dtype=torch.float64, device=dev)
    scale = torch.zeros(B, dtype=torch.float64, device=dev)
    rot = torch.zeros((B, 9), dtype=torch.float64, device=dev)
    trans = torch.zeros((B, 3), dtype=torch.float64, device=dev)
    args = [t(nocs), t(depth), t(choose), t(Kp), t(E), None, t(ridx)]
    L.check(lib.adp_fit_umeyama(*[L.ptr(a) for a in args], 0, L.ptr(bbox), L.ptr(scale), L.ptr(rot), L.ptr(trans), B, P, 224,
                                G.stream()), "fit_umeyama")
    torch.cuda.synchronize()
    for b in range(B):
        cam = O.back_project(depth[b], choose[b], Kp[b].reshape(3, 3))
        s, R, tr, _ = O.similarity_ransac(nocs[b], cam, rand_idx=ridx[b])
        if s is None:                                   # inlier ratio < 0.1 -> the reference returns None -> sentinel box
            np.testing.assert_array_equal(bbox[b].cpu().numpy(), O.DEFAULT_BBOX)
            continue
        assert abs(float(scale[b]) - s) / s < 1e-9
        np.testing.assert_allclose(rot[b].cpu().numpy().reshape(3, 3), R, atol=1e-9)
        np.testing.assert_allclose(trans[b].cpu().numpy(), tr, atol=1e-9)
        want = O.box_from_fit(nocs[b], s, R, tr, E[b].reshape(4, 4))
        np.testing.assert_allclose(bbox[b].cpu().numpy(), want, rtol=0, atol=1e-7)
