"""The hand-written cost-regularisation kernels besides adp_conv_tc against float64 references: the depth-ring conv0
(csrc/conv0_ring.cu), the fused transposed conv (csrc/tconv_fused.cu) and the decode gather (csrc/decode.cu).

Both tensor-core kernels are persistent: a CTA walks work units (conv0: 4 rows x 112 pixels through every depth plane; tconv:
one tile of input positions through its 8 shifted loads) and carries TMA ring stages, TMEM ring slots and (tconv) a
double-buffered TMEM accumulator from one unit to the next.  Every case therefore also runs at num_sms = 1, where one CTA
(conv0) or two (tconv: the grid is min(tiles, 2 num_sms)) walk every unit, and must write the bits of a full grid.

Reference: torch float64 on the CPU with the operands at their exact value in the kernel's format (16-bit volumes, weights and
skip tensors; fp32 scale / shift, prob_w, feature maps, Mw and depths).  Bounds, per element:
  * conv0 and tconv (fp32 accumulation, folded BatchNorm, ReLU, skip, one rounding to 16 bits): 1e-5 max|acc| |scale[c]| for
    the accumulation order (the convention of test_gpu_tc_conv.py) plus one ulp of the 16-bit output format at |ref|;
  * decode logits (the `prob` conv at the sampled pixels): 24 2^-24 sum|w x| (at most 24 fp32 roundings on the way, each below
    2^-24 of the sum of magnitudes);
  * decode depth: softmax and expectation in float64 from the kernel's own logits, 4e-6 m (a few fp32 ulps at 2.4 m);
  * decode fused features: float64 over the kernel's logits, sample coordinates in float64 from the fp32 Mw.  Bilinear sampling
    with zero padding is continuous and piecewise linear in the coordinate, so a coordinate error delta moves a sample by at most
    2 delta L, L = the largest difference between samples of the 4 x 4 neighbourhood (0 outside the image); delta = 2^-11 px.
    Plus the fp32 rounding of the 24-term sum: 2^-24 (|l - max l| + 40) |v| per term (the chain, the bilinear fmas, exp, sum and
    division of the softmax, and the rounding of the exponent l - max l itself);
  * the same arithmetic on another CTA, at another batch size or in another layout, and the bf16 hi / lo split of fp32 values,
    is bit exact.
"""
import math
import zlib
from dataclasses import dataclass
from types import SimpleNamespace

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from gpu_util import CANARY16, CANARY32, assert_close, bits, canary16, canary32
from rgbmanip_b200 import _lib as L
from rgbmanip_b200 import geometry

pytestmark = [pytest.mark.gpu, pytest.mark.filterwarnings("ignore")]

ACC_TOL = 1e-5           # fp32 accumulation order with exact operands, relative to max|acc|


@pytest.fixture(scope="module")
def G():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    import importlib
    L.load()
    return importlib.import_module("gpu_util")


def _rng(name):
    return np.random.default_rng(zlib.crc32(name.encode()))


def _t(rng, *shape, scale=1.0):
    return torch.from_numpy(rng.standard_normal(shape, dtype=np.float32) * np.float32(scale))


def _fmt(dt):
    return "f16" if dt == torch.float16 else "bf16"


# ================================================================================================ conv0 depth ring
def conv0_inputs(name, B, D, H, dt):
    rng = _rng(name)
    return SimpleNamespace(x=_t(rng, B, D, H, 224, 32).to(dt), w=_t(rng, 8, 32, 3, 3, 3, scale=math.sqrt(1.0 / 864)).to(dt),
                           scale=_t(rng, 8).abs() + 0.5, shift=_t(rng, 8) * 0.5, dt=dt)


def conv0_run(G, c, *, s2d=False, num_sms=148, batch=None, w=None):
    """One adp_conv0 run into a canary-filled output; w: torch-layout weights to pack instead of c.w.  Returns the output, cpu."""
    B, D, H, W, _ = c.x.shape
    if not hasattr(c, "xd"):
        c.xd = c.x.to(G.DEV).contiguous()
    out = canary16((B, D // 2, H // 2, W // 2, 64) if s2d else (B, D, H, W, 16), c.dt)
    wp = geometry.conv0_ring_weights((c.w if w is None else w).float()).to(c.dt).to(G.DEV).contiguous()
    G.conv0(c.xd, wp, c.scale.to(G.DEV), c.shift.to(G.DEV), out, flags=L.LAYOUT_S2D if s2d else 0, num_sms=num_sms, batch=batch)
    return out.cpu()


def conv0_acc(c, d0, d1, y0, y1):
    """float64 accumulators of output planes [d0, d1) and rows [y0, y1) (all columns), zero padded: [B, d1-d0, y1-y0, W, 8]."""
    D, H = c.x.shape[1], c.x.shape[2]
    zs, ze, ys, ye = max(d0 - 1, 0), min(d1 + 1, D), max(y0 - 1, 0), min(y1 + 1, H)
    sl = c.x[:, zs:ze, ys:ye].double().permute(0, 4, 1, 2, 3)
    sl = F.pad(sl, (1, 1, ys - (y0 - 1), (y1 + 1) - ye, zs - (d0 - 1), (d1 + 1) - ze))
    return F.conv3d(sl, c.w.double()).permute(0, 2, 3, 4, 1)


def conv0_check(c, got8, acc, what):
    """got8: the 8 real channels [B, d, y, W, 8] of a kernel output; acc: conv0_acc of the same region."""
    ref = (acc * c.scale.double() + c.shift.double()).clamp_min(0)
    slack = ACC_TOL * float(acc.abs().max()) * c.scale.double().abs()          # per channel, scaled by |scale[c]|
    return assert_close(got8, ref, _fmt(c.dt), slack, what)


C0_SMALL = {f"D{D}_{lay}_{_fmt(dt)}": (D, lay == "s2d", dt)
            for D in (2, 5, 6) for lay in ("plain", "s2d") for dt in (torch.float16, torch.bfloat16) if not (lay == "s2d" and D % 2)}
_C0 = {}


def c0_small(G, cid):
    """Inputs (B 2, H 8, W 224: 2 x 2 x 2 = 8 units), float64 accumulators and the 148-SM run of a small conv0 case (cached).
    The plain and the s2d case of one (D, dtype) share their inputs."""
    D, s2d, dt = C0_SMALL[cid]
    key = (D, dt)
    if key not in _C0:
        c = conv0_inputs(f"conv0_D{D}_{_fmt(dt)}", 2, D, 8, dt)
        _C0[key] = SimpleNamespace(c=c, acc=conv0_acc(c, 0, D, 0, 8), full={})
    e = _C0[key]
    if s2d not in e.full:
        e.full[s2d] = conv0_run(G, e.c, s2d=s2d)
    return e


@pytest.mark.parametrize("num_sms", [1, 3, 148], ids=lambda n: f"num_sms{n}")
@pytest.mark.parametrize("cid", list(C0_SMALL))
def test_conv0_multi_unit_matches_fp64(G, cid, num_sms):
    """8 units over 1, 3 or 8 CTAs (8, 3-3-2 or 1 units each).  D = 5 and 6 are not multiples of the 4-stage TMA ring, so the
    ring's stage and phase carry across unit boundaries at a different point in every unit."""
    D, s2d, dt = C0_SMALL[cid]
    e = c0_small(G, cid)
    got = conv0_run(G, e.c, s2d=s2d, num_sms=num_sms)
    if s2d:
        plain8 = geometry.from_s2d(got)
        assert torch.equal(bits(plain8), bits(c0_small(G, cid.replace("s2d", "plain")).full[False][..., :8].contiguous()))
    else:
        assert (bits(got[..., 8:]) == 0).all()                 # the 8 pad channels conv1 reads as K = 16 are exact zeros
        plain8 = got[..., :8]
    worst = conv0_check(e.c, plain8, e.acc, f"conv0 {cid} num_sms {num_sms}")
    assert torch.equal(bits(got), bits(e.full[s2d]))
    print(f"conv0 {cid} num_sms {num_sms}: largest error / bound {worst:.3f}")


def test_conv0_engine_geometry(G):
    """The engine's conv0: [24, 224, 224], fp16, s2d output, B 2 = 224 units.  The float64 reference covers every row of depth
    planes 0, 1, 12, 22, 23 and image rows 0-4, 110-113, 219-223 of every plane; one CTA and a full grid agree bit for bit on
    the whole tensor."""
    c = conv0_inputs("conv0_engine", 2, 24, 224, torch.float16)
    full = conv0_run(G, c, s2d=True)
    one = conv0_run(G, c, s2d=True, num_sms=1)
    assert torch.equal(bits(one), bits(full))
    got = geometry.from_s2d(full)
    worst = 0.0
    for d0, d1, y0, y1 in ((0, 2, 0, 224), (12, 13, 0, 224), (22, 24, 0, 224), (0, 24, 0, 5), (0, 24, 110, 114), (0, 24, 219, 224)):
        acc = conv0_acc(c, d0, d1, y0, y1)
        worst = max(worst, conv0_check(c, got[:, d0:d1, y0:y1], acc, f"conv0 planes [{d0},{d1}) rows [{y0},{y1})"))
    print(f"conv0 engine geometry: largest error / bound {worst:.3f}")


@pytest.mark.parametrize("s2d", [False, True], ids=["plain", "s2d"])
def test_conv0_partial_batch(G, s2d):
    """A plan for 3 images run on 2: image 2 keeps its canary bits, images 0-1 equal the full run bit for bit."""
    c = conv0_inputs("conv0_partial", 3, 6, 8, torch.bfloat16)
    full = conv0_run(G, c, s2d=s2d)
    part = conv0_run(G, c, s2d=s2d, batch=2)
    assert torch.equal(bits(part[:2]), bits(full[:2]))
    assert (bits(part[2]) == CANARY16).all()
    assert not (bits(full[2]) == CANARY16).any()


def test_conv0_s2d_rejects_odd_depth(G):
    """Plane D-1 of an odd D has no slot in a [B, D/2, ...] space-to-depth output: the plan fails and nothing is written (the
    buffer has room for that plane, so a plan that slipped through could not write outside it)."""
    c = conv0_inputs("conv0_odd", 1, 5, 4, torch.float16)
    out = canary16((1, 3, 2, 112, 64), c.dt)
    wp = geometry.conv0_ring_weights(c.w.float()).to(c.dt).to(G.DEV)
    with pytest.raises(L.AdpError, match="even D"):
        G.conv0(c.x.to(G.DEV), wp, c.scale.to(G.DEV), c.shift.to(G.DEV), out, flags=L.LAYOUT_S2D)
    assert (bits(out) == CANARY16).all()


# ================================================================================================ fused transposed conv
@dataclass
class Tc:
    id: str
    cin: int
    cout: int
    x: tuple                # (B, D, H, W) of the input
    dt: torch.dtype
    res_cs: int             # channel pitch of the skip tensor (ignored in the s2d layout)
    inst: tuple             # expected kernel instance (KC, BN)
    s2d: bool = False
    twin: str = ""          # the plain case whose inputs an s2d case shares (and whose output it must equal)


F16, BF16 = torch.float16, torch.bfloat16
TCONV_CASES = [
    # tiles = B x D x tiles_y x tiles_x of tc_pick_tile(H, W); the grid is min(tiles, 2 num_sms)
    Tc("conv9_32to16", 32, 16, (2, 6, 56, 56), F16, 16, (32, 16)),                 # the engine's conv9: 8 x 16 tiles, 336
    Tc("c16to8_skip16", 16, 8, (3, 4, 28, 28), F16, 16, (16, 16)),                  # conv0-style channel-padded skip, 84 tiles
    Tc("c16to8_s2d", 16, 8, (3, 4, 28, 28), F16, 0, (16, 16), s2d=True, twin="c16to8_skip16"),
    Tc("c16to24_bf16_ragged", 16, 24, (3, 3, 20, 12), BF16, 24, (16, 32)),           # 12 x 10 tiles (120 of 128 rows), 18 tiles
    Tc("c32to32", 32, 32, (3, 3, 28, 28), F16, 32, (32, 32)),                       # 28 x 4 tiles, 63
]
TC_BY_ID = {c.id: c for c in TCONV_CASES}
_TC = {}


def tconv_data(case):
    """Seeded inputs, float64 accumulators [B, 2D, 2H, 2W, Cout] and skip of a case (cached; an s2d case uses its twin's)."""
    src = TC_BY_ID[case.twin] if case.twin else case
    if src.id not in _TC:
        rng = _rng(src.id)
        B, D, H, W = src.x
        x = _t(rng, B, D, H, W, src.cin).to(src.dt)
        w = _t(rng, src.cin, src.cout, 3, 3, 3, scale=math.sqrt(1.0 / (8 * src.cin))).to(src.dt)
        res = _t(rng, B, 2 * D, 2 * H, 2 * W, src.res_cs).to(src.dt)
        acc = F.conv_transpose3d(x.double().permute(0, 4, 1, 2, 3), w.double(), stride=2, padding=1, output_padding=1)
        _TC[src.id] = SimpleNamespace(x=x, w=w, res=res, scale=_t(rng, src.cout).abs() + 0.5, bias=_t(rng, src.cout) * 0.5,
                                      acc=acc.permute(0, 2, 3, 4, 1).contiguous(), full={})
    return _TC[src.id]


def tconv_run(G, case, *, num_sms=148, batch=None, w=None, skip=True):
    """One adp_tconv run of a case into a canary-filled output, returned on the cpu in the plain layout [B, 2D, 2H, 2W, Cout] and
    as written.  w: torch-layout [Cin, Cout, 3, 3, 3] weights instead of the case's; skip=False passes res = NULL."""
    d = tconv_data(case)
    B, D, H, W = case.x
    bn = case.inst[1]
    wt = (d.w if w is None else w).float().reshape(case.cin, case.cout, 27).permute(2, 1, 0)
    wt = torch.cat([wt, torch.zeros(27, bn - case.cout, case.cin)], 1).to(case.dt).to(G.DEV).contiguous()
    res = None
    if skip:
        res = geometry.to_s2d(d.res[..., :case.cout].contiguous()) if case.s2d else d.res
        res = res.to(G.DEV).contiguous()
    out = canary16((B, D, H, W, 8 * case.cout) if case.s2d else (B, 2 * D, 2 * H, 2 * W, case.cout), case.dt)
    G.tconv(d.x.to(G.DEV).contiguous(), wt, case.cout, d.scale.to(G.DEV), d.bias.to(G.DEV), res, out,
            res_cstride=0 if case.s2d else case.res_cs, flags=L.LAYOUT_S2D if case.s2d else 0, num_sms=num_sms, batch=batch)
    raw = out.cpu()
    return (geometry.from_s2d(raw) if case.s2d else raw), raw


def tconv_check(case, got, what, skip=True):
    d = tconv_data(case)
    ref = (d.acc * d.scale.double() + d.bias.double()).clamp_min(0)
    if skip:
        ref = ref + d.res[..., :case.cout].double()                  # the skip joins after the ReLU (network_v5.py:287-289)
    slack = ACC_TOL * float(d.acc.abs().max()) * d.scale.double().abs()
    return assert_close(got, ref, _fmt(case.dt), slack, what)


def tconv_full(G, case):
    d = tconv_data(case)
    if case.id not in d.full:
        d.full[case.id] = tconv_run(G, case)
    return d.full[case.id]


@pytest.mark.parametrize("num_sms", [1, 148], ids=lambda n: f"num_sms{n}")
@pytest.mark.parametrize("cid", [c.id for c in TCONV_CASES])
def test_tconv_matches_fp64(G, cid, num_sms):
    """Every fused transposed-conv instance against the float64 reference.  At num_sms = 1 two CTAs walk every tile, through both
    TMEM accumulator sets; at 148 conv9's 336 tiles still give some CTAs two.  Both write the same bits."""
    case = TC_BY_ID[cid]
    assert case.inst == (case.cin, 16 if case.cout <= 16 else 32)      # tconv_plan: KC = Cin, BN = 16 if Cout <= 16 else 32
    got, raw = tconv_run(G, case, num_sms=num_sms)
    worst = tconv_check(case, got, f"tconv {cid} num_sms {num_sms}")
    assert torch.equal(bits(raw), bits(tconv_full(G, case)[1]))
    if case.twin:                                                       # s2d layout: the plain layout's bits, moved
        assert torch.equal(bits(got), bits(tconv_full(G, TC_BY_ID[case.twin])[0]))
    print(f"tconv {cid} (KC {case.inst[0]}, BN {case.inst[1]}) num_sms {num_sms}: largest error / bound {worst:.3f}")


def test_tconv_instances_covered():
    assert {c.inst for c in TCONV_CASES} == {(16, 16), (32, 16), (16, 32), (32, 32)}
    assert any(c.dt == BF16 for c in TCONV_CASES) and any(c.s2d for c in TCONV_CASES)


@pytest.mark.parametrize("cid", [c.id for c in TCONV_CASES])
def test_tconv_partial_batch(G, cid):
    """A plan for B images run on B - 1: the last image keeps its canary bits, the others equal the full run bit for bit."""
    case = TC_BY_ID[cid]
    B = case.x[0]
    full = tconv_full(G, case)[1]
    _, part = tconv_run(G, case, batch=B - 1)
    assert torch.equal(bits(part[:B - 1]), bits(full[:B - 1]))
    assert (bits(part[B - 1]) == CANARY16).all()
    assert not (bits(full[B - 1]) == CANARY16).any()


def test_tconv_without_skip(G):
    """res = NULL: the output is relu(scale acc + bias) alone."""
    case = TC_BY_ID["c32to32"]
    got, _ = tconv_run(G, case, skip=False)
    worst = tconv_check(case, got, "tconv c32to32 without skip", skip=False)
    print(f"tconv c32to32 without skip: largest error / bound {worst:.3f}")


# ================================================================================================ decode gather
X11_FORMATS = {"bf16": 0, "f16": L.LAYOUT_F16, "bf16_s2d": L.LAYOUT_S2D, "f16_s2d": L.LAYOUT_F16 | L.LAYOUT_S2D}
DEC_B, DEC_S, DEC_P, DEC_D = 3, 224, 1024, 24
DEC_VALID = (1, 0, 1)
DELTA = 2.0 ** -11           # px: bound on the kernel's fp32 sample coordinate error
DEPTH_TOL = 4e-6             # m
_DEC = {}


def _choose(rng, S, P):
    """P pixels: the four corners, 48 on each border row and column, the rest uniform; shuffled."""
    e = np.linspace(1, S - 2, 48).astype(np.int64)
    edge = [0, S - 1, (S - 1) * S, S * S - 1] + list(e) + list((S - 1) * S + e) + list(e * S) + list(e * S + S - 1)
    pix = np.concatenate([np.array(edge), rng.integers(0, S * S, P - len(edge))])
    return rng.permutation(pix).astype(np.int32)


def decode_data(G):
    """Seeded decode inputs (cached): random fp32 feature maps, Mw of real stereo geometry (adp_warp_matrices on synth scenes),
    the engine's 24 depths, an fp32 x11 rounded per format at run time, prob_w and the sampled pixels."""
    if "d" not in _DEC:
        from oracle import adapose_oracle as O
        from rgbmanip_b200 import synth
        B, S, P = DEC_B, DEC_S, DEC_P
        rng = _rng("decode")
        batch = synth.make_batch(B, seed=3, special=False)
        np.random.seed(3)
        kp1 = np.stack([O.prepare_model_input(batch.rgb1[e], batch.mask1[e], batch.K[e])[3] for e in range(B)])
        kp2 = np.stack([O.prepare_model_input(batch.rgb2[e], batch.mask2[e], batch.K[e])[3] for e in range(B)])
        # the camera buffers stay referenced until the kernel has run (L.ptr holds no reference; freed temporaries would alias)
        cams = [torch.from_numpy(np.ascontiguousarray(a).reshape(B, -1)).to(G.DEV) for a in (kp1, batch.E1, kp2, batch.E2)]
        Mw = torch.zeros((B, 12), device=G.DEV)
        L.check(L.load().adp_warp_matrices(*(L.ptr(t) for t in cams), L.ptr(Mw), None, None, None, B, G.stream()), "warp matrices")
        torch.cuda.synchronize()
        d = SimpleNamespace(feat_ref=_t(rng, B, S, S, 32), feat_src=_t(rng, B, S, S, 32), Mw=Mw.cpu(),
                            depths=torch.from_numpy(O.depth_hypotheses()), x11=_t(rng, B, DEC_D, S, S, 8),
                            prob_w=_t(rng, 27, 8, scale=0.25), choose=torch.from_numpy(np.stack([_choose(rng, S, P) for _ in range(B)])),
                            valid=torch.tensor(DEC_VALID, dtype=torch.uint8), runs={}, refs={})
        d.dev = {k: getattr(d, k).to(G.DEV).contiguous() for k in ("feat_ref", "feat_src", "Mw", "depths", "prob_w", "choose", "valid")}
        _DEC["d"] = d
    return _DEC["d"]


def decode_bufs(B, P):
    """Canary-filled outputs of adp_decode_gather."""
    return dict(depth=canary32((B, P)), xfeat_hi=canary16((B, P, 32), BF16), xfeat_lo=canary16((B, P, 32), BF16),
                xcat_hi=canary16((B, P, 96), BF16), xcat_lo=canary16((B, P, 96), BF16), dbg_logits=canary32((B, P, DEC_D)),
                dbg_fused=canary32((B, P, 32)))


def x11_dev(G, d, fmt, x11=None):
    """x11 on the device in format `fmt`: fp16 or bf16, plain [B, D, S, S, 8] or s2d [B, D/2, S/2, S/2, 64]."""
    code = X11_FORMATS[fmt]
    v = (d.x11 if x11 is None else x11).to(F16 if code & L.LAYOUT_F16 else BF16)
    return (geometry.to_s2d(v) if code & L.LAYOUT_S2D else v).to(G.DEV).contiguous()


def decode_run(G, d, fmt, *, batch=DEC_B, x11=None, prob_w=None):
    """One adp_decode_gather call in format `fmt` into canary-filled buffers; returns them on the cpu.  x11 / prob_w: inputs
    instead of the case's (fp32 x11 [B, D, S, S, 8] before rounding, prob_w [27, 8])."""
    bufs = decode_bufs(DEC_B, DEC_P)
    v = d.dev
    G.decode_gather(v["feat_ref"], v["feat_src"], v["Mw"], v["depths"], x11_dev(G, d, fmt, x11), v["choose"], v["valid"],
                    v["prob_w"] if prob_w is None else prob_w.to(G.DEV).contiguous(), bufs, batch=batch, S=DEC_S, P=DEC_P,
                    x11_format=X11_FORMATS[fmt])
    return {k: t.cpu() for k, t in bufs.items()}


def decode_full(G, d, fmt):
    if fmt not in d.runs:
        d.runs[fmt] = decode_run(G, d, fmt)
    return d.runs[fmt]


def logits_ref(d, b, x11_exact, prob_w):
    """float64 `prob` conv (3x3x3, 8 -> 1, zero padding in d, y and x) at env b's sampled pixels: (logits, sum|w x|), [P, D]."""
    S = DEC_S
    xp = F.pad(x11_exact[b], (0, 0, 1, 1, 1, 1, 1, 1))                     # [D + 2, S + 2, S + 2, 8]
    y, x = (d.choose[b] // S).long(), (d.choose[b] % S).long()
    nb = torch.stack([xp[:, y + ky, x + kx] for ky in range(3) for kx in range(3)], 2)       # [D + 2, P, 9, 8]
    win = nb.double().unfold(0, 3, 1)                                     # [D, P, 9, 8, kz]
    w = prob_w.double().reshape(3, 9, 8).permute(1, 2, 0)                 # [ky * 3 + kx, c, kz]
    return torch.einsum("dpjck,jck->pd", win, w), torch.einsum("dpjck,jck->pd", win.abs(), w.abs())


def fused_ref(d, b, logits):
    """float64 depth-guided fusion over the kernel's logits [P, D] of env b: (fused [P, 32], bound [P, 32], depth [P])."""
    S = DEC_S
    l = logits.double()
    p = torch.softmax(l, 1)                                                # [P, D]
    depth = (p * d.depths.double()).sum(1)
    M = d.Mw[b].double()
    y, x = (d.choose[b] // S).double(), (d.choose[b] % S).double()
    dep = d.depths.double()
    rx, ry, rz = (M[3 * i] * x + M[3 * i + 1] * y + M[3 * i + 2] for i in range(3))
    X, Y, Z = (r[:, None] * dep + M[9 + i] for i, r in enumerate((rx, ry, rz)))
    half = (S - 1) / 2.0
    ix = ((X / Z / half - 1 + 1) * S - 1) / 2
    iy = ((Y / Z / half - 1 + 1) * S - 1) / 2
    assert torch.isfinite(ix).all() and torch.isfinite(iy).all()
    x0, y0 = ix.floor(), iy.floor()
    ex, ey = (ix - x0)[..., None], (iy - y0)[..., None]
    off = torch.arange(-1, 3, dtype=torch.float64)
    xs = x0[..., None] + off                                               # [P, D, 4]
    ys = y0[..., None] + off
    inx, iny = (xs >= 0) & (xs < S), (ys >= 0) & (ys < S)
    xi, yi = xs.clamp(0, S - 1).long(), ys.clamp(0, S - 1).long()
    src = d.feat_src[b]
    nb = src[yi[..., :, None], xi[..., None, :]].double()                  # [P, D, 4 (y), 4 (x), 32]
    nb = nb * (iny[..., :, None] & inx[..., None, :])[..., None]
    Lr = nb.amax((2, 3)) - nb.amin((2, 3))                                 # [P, D, 32]
    c00, c01, c10, c11 = nb[:, :, 1, 1], nb[:, :, 1, 2], nb[:, :, 2, 1], nb[:, :, 2, 2]
    w00, w01, w10, w11 = (1 - ex) * (1 - ey), ex * (1 - ey), (1 - ex) * ey, ex * ey
    fr = d.feat_ref[b].reshape(S * S, 32)[d.choose[b].long()].double()[:, None]      # [P, 1, 32]
    v = fr + w00 * c00 + w01 * c01 + w10 * c10 + w11 * c11
    vabs = fr.abs() + w00 * c00.abs() + w01 * c01.abs() + w10 * c10.abs() + w11 * c11.abs()
    ulps = (l - l.amax(1, keepdim=True)).abs() + 40
    fused = (p[..., None] * v).sum(1)
    bound = (p[..., None] * (2 * DELTA * Lr + 2.0 ** -24 * ulps[..., None] * vabs)).sum(1)
    return fused, bound, depth


def split_bits(x):
    """bits of the bf16 hi / lo planes the kernel must write for fp32 values x (round to nearest even, as torch)."""
    hi = x.to(BF16)
    return bits(hi), bits((x - hi.float()).to(BF16))


def decode_check(G, d, fmt, out, x11=None, prob_w=None):
    """Every output of a decode run against the float64 reference; returns the largest error / bound ratio per quantity."""
    code = X11_FORMATS[fmt]
    x11_exact = (d.x11 if x11 is None else x11).to(F16 if code & L.LAYOUT_F16 else BF16).float()
    pw = d.prob_w if prob_w is None else prob_w
    worst = {"logits": 0.0, "depth": 0.0, "fused": 0.0}
    for b in range(DEC_B):
        if not DEC_VALID[b]:
            continue
        ref, mag = logits_ref(d, b, x11_exact, pw)
        got = out["dbg_logits"][b]
        worst["logits"] = max(worst["logits"], assert_close(got, ref, "f32", 24 * 2.0 ** -24 * mag, f"{fmt} env {b} logits"))
        fused, bound, depth = fused_ref(d, b, got)
        worst["depth"] = max(worst["depth"], assert_close(out["depth"][b], depth, "f32", DEPTH_TOL, f"{fmt} env {b} depth"))
        worst["fused"] = max(worst["fused"], assert_close(out["dbg_fused"][b], fused, "f32", bound, f"{fmt} env {b} fused"))
        # the MLP inputs: exact bf16 hi / lo splits of the fp32 values (feat_ref at the pixel; the kernel's fused feature)
        fr = d.feat_ref[b].reshape(DEC_S * DEC_S, 32)[d.choose[b].long()]
        hi, lo = split_bits(fr)
        assert torch.equal(bits(out["xfeat_hi"][b]), hi) and torch.equal(bits(out["xfeat_lo"][b]), lo)
        hi, lo = split_bits(out["dbg_fused"][b])
        assert torch.equal(bits(out["xcat_hi"][b][:, :32]), hi) and torch.equal(bits(out["xcat_lo"][b][:, :32]), lo)
        for k in ("xcat_hi", "xcat_lo"):                          # columns 32-95 belong to nocs_pts_mlp
            assert (bits(out[k][b][:, 32:]) == CANARY16).all(), k
    for b in range(DEC_B):
        if not DEC_VALID[b]:                                      # an invalid environment's outputs stay untouched
            for k, t in out.items():
                assert (bits(t[b]) == (CANARY32 if t.dtype == torch.float32 else CANARY16)).all(), (b, k)
    return worst


@pytest.mark.parametrize("fmt", list(X11_FORMATS))
def test_decode_gather_matches_fp64(G, fmt):
    """Logits, depth, fused features and the bf16 hi / lo MLP inputs of 3 environments (env 1 invalid) at 1024 pixels each,
    border rows and columns and the corners included.  The s2d layout of x11 gives the plain layout's bits."""
    d = decode_data(G)
    out = decode_full(G, d, fmt)
    if X11_FORMATS[fmt] & L.LAYOUT_S2D:
        plain = decode_full(G, d, fmt.replace("_s2d", ""))
        for k in out:
            assert torch.equal(bits(out[k]), bits(plain[k])), k
    worst = decode_check(G, d, fmt, out)
    print(f"decode {fmt}: largest error / bound " + ", ".join(f"{k} {v:.3f}" for k, v in worst.items()))


def test_decode_choose_covers_borders(G):
    d = decode_data(G)
    S = DEC_S
    for b in range(DEC_B):
        y, x = d.choose[b] // S, d.choose[b] % S
        for yy, xx in ((0, 0), (0, S - 1), (S - 1, 0), (S - 1, S - 1)):
            assert ((y == yy) & (x == xx)).any()
        assert ((y == 0) & (x > 0) & (x < S - 1)).any() and ((y == S - 1) & (x > 0) & (x < S - 1)).any()
        assert ((x == 0) & (y > 0) & (y < S - 1)).any() and ((x == S - 1) & (y > 0) & (y < S - 1)).any()


def test_decode_batch_independence(G):
    """Env 0 of a one-environment call equals env 0 of the three-environment call bit for bit; envs 1-2 keep their canaries."""
    d = decode_data(G)
    full = decode_full(G, d, "f16_s2d")
    one = decode_run(G, d, "f16_s2d", batch=1)
    for k in one:
        assert torch.equal(bits(one[k][0]), bits(full[k][0])), k
        assert (bits(one[k][1:]) == (CANARY32 if one[k].dtype == torch.float32 else CANARY16)).all(), k


def test_decode_single_view(G):
    """x11 = NULL: only xfeat is written (the hi / lo split of feat_ref at the pixel); xcat, depth and the debug buffers keep their
    canaries, and so does every output of the invalid environment."""
    d = decode_data(G)
    bufs = decode_bufs(DEC_B, DEC_P)
    v = d.dev
    G.decode_gather(v["feat_ref"], None, None, None, None, v["choose"], v["valid"], None, bufs, batch=DEC_B, S=DEC_S, P=DEC_P,
                    x11_format=0)
    out = {k: t.cpu() for k, t in bufs.items()}
    for b in range(DEC_B):
        for k, t in out.items():
            if DEC_VALID[b] and k in ("xfeat_hi", "xfeat_lo"):
                continue
            assert (bits(t[b]) == (CANARY32 if t.dtype == torch.float32 else CANARY16)).all(), (b, k)
        if DEC_VALID[b]:
            hi, lo = split_bits(d.feat_ref[b].reshape(DEC_S * DEC_S, 32)[d.choose[b].long()])
            assert torch.equal(bits(out["xfeat_hi"][b]), hi) and torch.equal(bits(out["xfeat_lo"][b]), lo)


def test_decode_s2d_rejects_odd_size(G):
    """Row and column S-1 of an odd S have no cell in an [B, D/2, S/2, S/2, 64] x11: the call fails before any launch (the
    buffers are those of S = 224, so a call that slipped through could not read outside them)."""
    d = decode_data(G)
    bufs = decode_bufs(DEC_B, DEC_P)
    v = d.dev
    choose = torch.zeros((1, 32), dtype=torch.int32, device=G.DEV)
    with pytest.raises(L.AdpError, match="even S"):
        G.decode_gather(v["feat_ref"], v["feat_src"], v["Mw"], v["depths"], x11_dev(G, d, "f16_s2d"), choose, v["valid"], v["prob_w"],
                        bufs, batch=1, S=DEC_S - 1, P=32, x11_format=X11_FORMATS["f16_s2d"])
    for k, t in bufs.items():
        assert (bits(t) == (CANARY32 if t.dtype == torch.float32 else CANARY16)).all(), k
