"""Device pipeline of the AdaPose hot path: weight packing, workspace, layer schedule.

Everything numerical runs in libadapose_b200.so (hand-written sm_100a CUDA) through the C ABI of
include/adapose_b200.h; torch is used for device memory, streams and host<->device copies only.

Stage map (reference lines relative to models/pose_estimator/AdaPose):
  preprocess   interface_v5.py:58-170          -> adp_preprocess
  backbone     lib/pspnet.py:33-158            -> adp_conv_tc_* (tcgen05) / adp_pack_s2d / adp_maxpool3x3s2 / adp_psp_priors /
                                                  adp_psp_fill_priors / adp_upconv_blend (up_1, up_2) / adp_upsample2x (up_3)
  volume       lib/network_v5.py:378-430       -> adp_warp_matrices, adp_build_volume
  cost reg.    lib/network_v5.py:260-291       -> adp_conv0_run (depth ring), adp_tconv_run (conv9), adp_conv_tc_* (everything else)
  decode       lib/network_v5.py:432-499       -> adp_decode_gather (the `prob` conv is evaluated at the sampled pixels only) +
                                                  per-point MLPs on adp_conv_tc_* + adp_colsum / adp_pose_gbias / adp_rot_head
  fit + box    lib/utils.py:40-119, lib/align.py, interface_v5.py:318-374 -> adp_fit / adp_fit_umeyama / adp_nocs_match
  transformer variant  lib/network_baseline.py:523-669, lib/fusion.py -> adp_view_fusion (arch="baseline")
"""
from __future__ import annotations

import ctypes as C
import threading
from dataclasses import dataclass

import numpy as np
import torch

from . import _lib as L
from . import geometry as G
from . import weights as W

IMG_SIZE = 224
N_PTS = 1024
N_DEPTH = 24
_CAPTURE_LOCK = threading.Lock()        # one CUDA-graph capture at a time per process


@dataclass
class ActBuf:
    hi: torch.Tensor
    lo: torch.Tensor | None
    B: int
    D: int
    H: int
    W: int
    Cn: int
    f16: int = 0
    s2d: bool = False        # level-0 U-Net tensor stored space-to-depth(2): logical [B, 2D, 2H, 2W, C/8]
    q8: torch.Tensor | None = None   # fp8 (e4m3) twin holding value / 2: A operand of the fp8 low-order pass of the consumer

    @property
    def c(self):
        return L.Act(L.ptr(self.hi), L.ptr(self.lo), self.B, self.D, self.H, self.W, self.Cn, self.f16, L.ptr(self.q8))

    def value(self, n=None):
        """fp32 torch view [B,(D,)H,W,C] (debug / tests)."""
        v = self.hi.float()
        if self.lo is not None:
            v = v + self.lo.float()
        if self.s2d:
            v = G.from_s2d(v)
        return v if n is None else v[:n]


def pack_tc_weights(wt: torch.Tensor, f16: int, npass: int):
    """fp32 [taps, CoutPad, Cin] weights -> the (hi, lo) planes adp_conv_tc_plan reads, on the host.  bf16: hi + lo split (lo for
    bf16x3 only); fp16: hi, plus the fp16 rounding residual as lo for fp16x2 (npass 2), or as e4m3(W_lo * 2^16) bytes for the fp8
    low-order pass (npass 4, see tc_conv.cu FUSED = 3).  lo is None for a single pass."""
    hi = wt.to(torch.float16 if f16 else torch.bfloat16)
    lo = wt - hi.float()
    if npass == 1:
        return hi, None
    if npass == 4:
        return hi, (lo * 65536.0).clamp(-448.0, 448.0).to(torch.float8_e4m3fn).view(torch.uint8)
    return hi, lo.to(hi.dtype)


class Engine:
    """One per device.  ``max_envs`` environments (2 x max_envs frames) are processed per chunk."""

    def __init__(self, state_dict, device="cuda:0", max_envs=16, precision="fp16f8", regress_pose=True, debug=False,
                 img_size=IMG_SIZE, n_pts=N_PTS, use_graph=True, use_depth=True, arch="v5"):
        if not torch.cuda.is_available():
            raise L.AdpError("no CUDA device: the AdaPose B200 path has no CPU fallback")
        if precision not in ("bf16", "bf16x3", "fp16x2", "fp16f8"):
            raise ValueError("precision must be 'fp16f8', 'fp16x2', 'bf16x3' or 'bf16'")
        self.lib = L.load()
        self.device = torch.device(device)
        self.E = int(max_envs)
        self.F = 2 * self.E
        self.S = int(img_size)
        self.P = int(n_pts)
        # backbone operand formats (DESIGN.md "precision policy"):
        #   fp16x2  one fp16 activation plane x (fp16 hi + lo) weights, 2 MMA passes
        #   bf16x3  (bf16 hi + lo) activations x (bf16 hi + lo) weights, 3 MMA passes
        #   bf16    single pass (fast, outside the parity tolerance)
        #   fp16f8  fp16x2, except that the wide layers (layer3, layer4, up_1: 81 % of the FLOPs) run the low-order term A W_lo
        #           as an e4m3 x e4m3 MMA at twice the rate (1.5 passes); W_lo <= 2^-12 |W| needs ~4 significant bits
        self.split = precision == "bf16x3"
        self.act_f16 = 1 if precision in ("fp16x2", "fp16f8") else 0
        self.fp8lo = precision == "fp16f8"
        self.npass = {"bf16": 1, "fp16x2": 2, "fp16f8": 2, "bf16x3": 3}[precision]
        self.precision = precision
        self.regress_pose = bool(regress_pose)
        # branch C (direct_regression = False, use_depth = False; interface_v5.py:339-349): NOCS of both views -> matching,
        # triangulation and median scale on the device, cv2 PnP on the host (estimator._pnp_tail); no volume / U-Net at all
        self.branch_c = (not self.regress_pose) and not bool(use_depth)
        # arch "baseline" = StereoPoseNet_with_depth_baseline (network_baseline.py:523-669): same backbone and NOCS head, 4 blocks of
        # cross-view attention + a depth MLP (csrc/view_fusion.cu) in place of the cost volume and its 3-D U-Net
        if arch not in ("v5", "baseline"):
            raise ValueError("arch must be 'v5' or 'baseline'")
        self.arch = arch
        self.need_volume = arch == "v5" and not self.branch_c
        if int(n_pts) != 1024 or int(img_size) % 224 != 0:
            raise ValueError("the device pipeline is built for n_pts = 1024 and img_size = 224 (every shipped adapose_* yaml)")
        self.use_graph = bool(use_graph) and not debug
        self._capture_stream = None
        self._graphs = {}           # chunk size -> (CUDAGraph, launches per replay)
        self._chunk_runs = {}       # chunk size -> eager runs so far (a size is captured on its second appearance)
        self._conv0_plans = []
        self._tconv_plans = []
        self.vol_f16 = 1            # the 3-D stage (volume, U-Net) stores IEEE half: BatchNorm keeps its activations O(10)
        self.debug = debug
        self._keep = []
        self._plans = []
        sms, maj, mnr = C.c_int(), C.c_int(), C.c_int()
        L.check(self.lib.adp_device_info(self.device.index or 0, C.byref(sms), C.byref(maj), C.byref(mnr)), "device_info")
        self.num_sms = sms.value
        self.cc = (maj.value, mnr.value)
        if self.cc[0] != 10:
            raise L.AdpError(f"device compute capability {self.cc} is not sm_100: this library ships sm_100a code only")
        sd = W.to_numpy_state_dict(state_dict)
        W.check_state_dict(sd, self.regress_pose, arch)
        self.sd = sd
        with torch.cuda.device(self.device):
            # [0] pipeline watchdog code, [1] fp16 range flag (set by the last backbone layer's epilogue on inf/NaN features)
            self.err_flag = torch.zeros(2, dtype=torch.int32, device=self.device)
            self._err_host = torch.zeros(2, dtype=torch.int32).pin_memory()
            self._err_event = None
            self._build_backbone()
            self._build_stereo()
            torch.cuda.synchronize()

    # ------------------------------------------------------------------ helpers
    def _dev(self, a, dtype=torch.float32):
        t = torch.as_tensor(np.ascontiguousarray(a)).to(dtype).to(self.device).contiguous()
        self._keep.append(t)
        return t

    def _act(self, B, H, Wd, Cn, D=1, split=None, f16=None, q8=False):
        if split is None and f16 is None:      # a backbone activation in the engine's precision
            f16 = self.act_f16
        f16 = int(f16 or 0)
        split = self.split if split is None else split
        shape = (B, D, H, Wd, Cn) if D > 1 else (B, H, Wd, Cn)
        dt = torch.float16 if f16 else torch.bfloat16
        hi = torch.zeros(shape, dtype=dt, device=self.device)
        lo = torch.zeros(shape, dtype=dt, device=self.device) if (split and not f16) else None
        buf = ActBuf(hi, lo, B, D, H, Wd, Cn, f16)
        if q8 and f16:
            buf.q8 = torch.zeros(shape, dtype=torch.uint8, device=self.device)
        self._keep.append(buf)   # layer plans hold raw pointers: the tensors must outlive them
        return buf

    @property
    def stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _epilogue(self, out: ActBuf | None, scale=None, bias=None, act=L.ACT_RELU, prelu=0.0, res: ActBuf | None = None,
                  res_after_act=0, out_f32=None, out_h16=None, out_cstride=0, out_coff=0, bias_per_batch=0, check_finite=0):
        return L.Epilogue(L.ptr(scale), L.ptr(bias), float(prelu), act, res_after_act,
                          L.ptr(res.hi) if res else None, L.ptr(res.lo) if (res and res.lo is not None) else None,
                          res.Cn if res else 0,
                          L.ptr(out.hi) if out else None, L.ptr(out.lo) if (out and out.lo is not None) else None,
                          L.ptr(out_f32), L.ptr(out_h16), out_cstride, out_coff, bias_per_batch,
                          L.ptr(out.q8) if (out is not None and out.q8 is not None) else None, check_finite)

    def _tc_plans(self, x: ActBuf, wt, cout, kd, ks, dil, npass, ep, geoms):
        """wt: fp32 [taps, CoutPad, Cin] packed weights -> callable(batch) launching one tcgen05 conv per geometry."""
        hi, lo = (t.to(self.device).contiguous() if t is not None else None for t in pack_tc_weights(wt, x.f16, npass))
        self._keep += [hi, lo]
        plans = []
        xa = x.c
        for g in geoms:
            plan = C.c_void_p()
            L.check(self.lib.adp_conv_tc_plan(C.byref(plan), C.byref(xa), L.ptr(hi), L.ptr(lo),
                                              cout, kd, ks, dil, npass, C.byref(ep), C.byref(g) if g is not None else None,
                                              self.num_sms), "conv_tc_plan")
            self._plans.append(plan)
            plans.append(plan)

        def run(batch, plans=plans):
            for plan in plans:
                L.check(self.lib.adp_conv_tc_run(plan, batch, L.ptr(self.err_flag), self.stream), "conv_tc_run")
        run.kind = "tc"
        return run

    def _with_fp8lo(self, npass, x: ActBuf, plain=True):
        """fp16f8: an fp16x2 conv (npass 2) runs its low-order term as the fp8 pass (npass 4) when x carries an fp8 twin, Cin is a
        multiple of 128 and the conv is plain (2-D, stride 1, not transposed)."""
        return 4 if (npass == 2 and self.fp8lo and plain and x.q8 is not None and x.Cn % 128 == 0) else npass

    def _conv(self, w_np, x: ActBuf, out: ActBuf | None, *, stride=1, dil=1, transposed=False, npass=None, **ep_kw):
        """Returns a callable(batch) running the convolution x -> out.  w_np: torch layout
        [Cout,Cin,(kd,)kh,kw] or, transposed, [Cin,Cout,kd,kh,kw]."""
        w = torch.as_tensor(np.ascontiguousarray(w_np)).float()
        three_d = w.dim() == 5
        if transposed:
            cin, cout = w.shape[0], w.shape[1]
            w_tcout_cin = w.reshape(cin, cout, -1).permute(2, 1, 0).contiguous()        # [taps, Cout, Cin]
        else:
            cout, cin = w.shape[0], w.shape[1]
            w_tcout_cin = w.reshape(cout, cin, -1).permute(2, 0, 1).contiguous()        # [taps, Cout, Cin]
        kd = w.shape[2] if three_d else 1
        ks = w.shape[-1]
        assert cin == x.Cn
        npass = self._with_fp8lo(self.npass if npass is None else npass, x, plain=not three_d and stride == 1 and not transposed)
        can_tc = (cin % 16 == 0 and ks in (1, 3) and (ks == w.shape[-2]) and stride in (1, 2)
                  and (npass == 1 or (npass in (2, 4) and x.f16) or (npass == 3 and x.lo is not None)))
        ep = self._epilogue(out, **ep_kw)
        if three_d:
            Do, Ho, Wo = (x.D * 2, x.H * 2, x.W * 2) if transposed else ((x.D + stride - 1) // stride,
                                                                        (x.H + stride - 1) // stride,
                                                                        (x.W + stride - 1) // stride)
        else:
            Do, Ho, Wo = 1, (x.H + stride - 1) // stride, (x.W + stride - 1) // stride
        if out is not None:
            assert (out.D, out.H, out.W, out.Cn) == (Do, Ho, Wo, cout), ((out.D, out.H, out.W, out.Cn), (Do, Ho, Wo, cout))
            assert out.f16 == x.f16
        if can_tc:
            cout_pad = (cout + 15) // 16 * 16
            wt = w_tcout_cin
            if cout_pad != cout:
                wt = torch.cat([wt, torch.zeros(wt.shape[0], cout_pad - cout, cin)], 1).contiguous()
            if transposed:
                geoms = G.transposed_classes(x.D, x.H, x.W)
            elif stride == 2:
                geoms = [G.strided(three_d, x.D, x.H, x.W, ks, 2)]
            else:
                geoms = [None]
            return self._tc_plans(x, wt, cout, kd, ks, dil, npass, ep, geoms)
        raise L.AdpError(f"no tcgen05 plan for this convolution (Cin {cin}, Cout {cout}, k {ks}, stride {stride}, npass {npass}): "
                         "the library has no CUDA-core fallback")

    # ------------------------------------------------------------------ backbone (pspnet.py)
    def _build_backbone(self):
        sd, F, S = self.sd, self.F, self.S
        ops = []
        p = "img_extractor.feats"
        self.crops = torch.zeros((F, S, S, 3), dtype=torch.float32, device=self.device)
        # conv1 7x7/2
        c1 = self._act(F, S // 2, S // 2, 64)
        w = torch.as_tensor(sd[f"{p}.conv1.weight"]).float()
        # stem on tensor cores: space-to-depth(2) repack of the crop, then a 4x4 stride-1 window over 16 channels
        s2d = self._act(F, S // 2, S // 2, 16)
        ops.append(("pack_s2d", lambda b, o=s2d: L.check(
            self.lib.adp_pack_s2d(L.ptr(self.crops), C.byref(o.c), b, S, self.stream), "pack_s2d")))
        wst = G.stem_s2d_weights(w)
        if s2d.f16 and self.npass == 2:
            # fp16 hi + lo weights as 2 x 16 taps of a single pass on the slab kernel (geometry.stem_s2d_split)
            ops.append(("conv1", self._tc_plans(s2d, torch.cat(pack_tc_weights(wst, 1, 2)).float(), 64, 1, 4, 1, 1,
                                                self._epilogue(c1, act=L.ACT_RELU), [G.stem_s2d_split(S)])))
        else:
            ops.append(("conv1", self._tc_plans(s2d, wst, 64, 1, 4, 1, self.npass,
                                                self._epilogue(c1, act=L.ACT_RELU), [G.stem_s2d(S)])))
        mp = self._act(F, S // 4, S // 4, 64)
        ops.append(("maxpool", lambda b, a=c1, o=mp: L.check(
            self.lib.adp_maxpool3x3s2(C.byref(a.c), C.byref(o.c), b, self.stream), "maxpool")))
        x = mp
        self.taps = {"conv1": c1, "maxpool": mp}
        # layer4's last conv writes straight into channels [0, 512) of the pyramid concat tensor (epilogue channel pitch 1024)
        cat = self._act(F, S // 8, S // 8, 1024, q8=self.fp8lo)
        for li, (planes, blocks, stride, dil) in enumerate(((64, 3, 1, 1), (128, 4, 2, 1), (256, 6, 1, 2), (512, 3, 1, 4)), 1):
            Hn = x.H // stride
            for bi in range(blocks):
                pre = f"{p}.layer{li}.{bi}"
                s_b = stride if bi == 0 else 1
                d_b = 1 if bi == 0 else dil
                # fp16f8: every activation that feeds a wide (layer3 / layer4) conv carries an fp8 twin written by its producer
                wide = self.fp8lo and li >= 2
                t = self._act(F, Hn, Hn, planes, q8=wide)
                ops.append((f"{pre}.conv1", self._conv(sd[f"{pre}.conv1.weight"], x, t, stride=s_b, dil=d_b, act=L.ACT_RELU)))
                res = x
                if f"{pre}.downsample.0.weight" in sd:
                    res = self._act(F, Hn, Hn, planes)
                    ops.append((f"{pre}.down", self._conv(sd[f"{pre}.downsample.0.weight"], x, res, stride=s_b, dil=1,
                                                          act=L.ACT_NONE)))
                last = li == 4 and bi == blocks - 1
                if last:
                    o = ActBuf(cat.hi[..., :planes], cat.lo[..., :planes] if cat.lo is not None else None, F, 1, Hn, Hn, planes, cat.f16,
                               q8=cat.q8)
                    ops.append((f"{pre}.conv2", self._conv(sd[f"{pre}.conv2.weight"], t, o, stride=1, dil=d_b, act=L.ACT_RELU,
                                                           res=res, out_cstride=1024)))
                else:
                    o = self._act(F, Hn, Hn, planes, q8=wide)
                    ops.append((f"{pre}.conv2", self._conv(sd[f"{pre}.conv2.weight"], t, o, stride=1, dil=d_b, act=L.ACT_RELU,
                                                           res=res)))
                self.taps[pre] = o
                x = o
        # pyramid pooling + concat + first upsample
        wpsp = torch.stack([torch.as_tensor(sd[f"img_extractor.psp.stages.{s}.1.weight"]).float().reshape(128, 512).t().contiguous()
                            for s in range(4)]).contiguous().to(self.device)          # [4][512][128]
        self._keep.append(wpsp)
        self.pooled = torch.zeros((F, 50, 512), dtype=torch.float32, device=self.device)
        self.priors = torch.zeros((F, 50, 128), dtype=torch.float32, device=self.device)
        l4 = x
        ops.append(("psp_priors", lambda b, a=l4: L.check(
            self.lib.adp_psp_priors(C.byref(a.c), 1024, L.ptr(wpsp), L.ptr(self.pooled), L.ptr(self.priors), b, self.stream), "psp")))
        ops.append(("psp_fill_priors", lambda b, o=cat: L.check(
            self.lib.adp_psp_fill_priors(L.ptr(self.priors), C.byref(o.c), 512, b, self.stream), "psp_fill")))
        # PSPUpsample x 3 (pspnet.py:97-107: bilinear x2 -> conv 3x3 -> PReLU).  Upsampling and channel mixing commute, so each
        # stage runs as ONE 1x1 GEMM over the LOW-resolution map producing the nine per-tap products (N = 9 Cout: a quarter of
        # the 3x3 conv's FLOPs over the upsampled map, which is never materialised), followed by adp_upconv_blend (9 taps x 4
        # bilinear neighbours + bias + PReLU).  Measured per 148 frames: up_1 2.94 -> 1.30 ms, up_2 1.30 -> 0.91 ms; up_3 (Cin = 64: the
        # nine products are 9x the input, 1.53 -> 3.09 ms) keeps the upsample + 3x3 conv form.
        restructured = ("up_1", "up_2")
        x = cat
        for nm, cout in (("up_1", 256), ("up_2", 64), ("up_3", 64)):
            bias = self._dev(sd[f"img_extractor.{nm}.conv.0.bias"])
            slope = float(np.asarray(sd[f"img_extractor.{nm}.conv.1.weight"]).reshape(-1)[0])
            wgt = torch.as_tensor(sd[f"img_extractor.{nm}.conv.0.weight"]).float()               # [Cout, Cin, 3, 3]
            o = self._act(F, 2 * x.H, 2 * x.W, cout)
            if nm in restructured:
                wt = wgt.permute(2, 3, 0, 1).reshape(1, 9 * cout, wgt.shape[1]).contiguous()      # [1][(ky*3+kx)*Cout + co][Cin]
                q = self._act(F, x.H, x.W, 9 * cout)
                npass = self._with_fp8lo(self.npass, x)
                gemm = self._tc_plans(x, wt, 9 * cout, 1, 1, 1, npass, self._epilogue(q, act=L.ACT_NONE), [None])
                ops.append((f"{nm}.taps", gemm))

                def blend(b, q=q, o=o, bias=bias, slope=slope):
                    L.check(self.lib.adp_upconv_blend(C.byref(q.c), C.byref(o.c), L.ptr(bias), slope, b, self.stream), "upconv_blend")
                blend.kind = "tc"         # completes the conv: timed with the tensor-core launches it belongs to
                ops.append((nm, blend))
            else:
                u = self._act(F, 2 * x.H, 2 * x.W, x.Cn, q8=self.fp8lo and nm == "up_1")
                ops.append((f"{nm}.upsample", lambda b, a=x, uu=u: L.check(
                    self.lib.adp_upsample2x(C.byref(a.c), C.byref(uu.c), b, self.stream), "upsample")))
                ops.append((nm, self._conv(wgt, u, o, bias=bias, act=L.ACT_PRELU, prelu=slope)))
            self.taps[nm] = o
            x = o
        self.feat = torch.zeros((F, S, S, 32), dtype=torch.float32, device=self.device)
        # fp16 twin of the feature map for the plane-sweep volume builder (the volume itself is fp16; halves its gather traffic)
        self.feat16 = torch.zeros((F, S, S, 32), dtype=torch.float16, device=self.device)
        fb = self._dev(sd["img_extractor.final.bias"])
        # the last layer sees every earlier one: an activation that left the fp16 range upstream arrives here as inf/NaN and
        # raises the range flag (err_flag[1]) that estimate() reads after every call
        ops.append(("final", self._conv(sd["img_extractor.final.weight"], x, None, bias=fb, act=L.ACT_NONE, out_f32=self.feat,
                                        out_h16=self.feat16, check_finite=1)))
        self.backbone_ops = ops

    def run_backbone(self, nframes):
        for _, op in self.backbone_ops:
            op(nframes)

    # ------------------------------------------------------------------ stereo head (network_v5.py)
    def _build_stereo(self):
        sd, E, S, D = self.sd, self.E, self.S, N_DEPTH
        dev = self.device
        self.depths = self._dev(np.arange(0.1, 0.1 * (D - 0.5) + 0.1, 0.1, dtype=np.float32))
        self.Mw = torch.zeros((E, 12), dtype=torch.float32, device=dev)
        self.valid_env = torch.zeros(E, dtype=torch.uint8, device=dev)
        self.E1buf = torch.zeros((E, 16), dtype=torch.float64, device=dev)
        self.E2buf = torch.zeros((E, 16), dtype=torch.float64, device=dev)
        if self.need_volume:
            self._build_cost_volume_stage()
        self._build_decode()

    def _build_cost_volume_stage(self):
        sd, E, S, D = self.sd, self.E, self.S, N_DEPTH
        self.vol = self._act(E, S, S, 32, D=D, split=False, f16=1)
        cr = "cost_regularization"

        def bn(name):
            sc, sh = W.fold_bn(sd, f"{cr}.{name}.bn")
            return self._dev(sc), self._dev(sh)

        ops = []
        dims = {0: (D, S), 1: (D // 2, S // 2), 2: (D // 4, S // 4), 3: (D // 8, S // 8)}

        def act3(level, Cn):
            d, s = dims[level]
            return self._act(E, s, s, Cn, D=d, split=False, f16=1)

        # The two full-resolution tensors (conv0 output, conv11 output) live in space-to-depth(2) layout [E, D/2, S/2, S/2, 64]
        # (channel = parity * 8 + c): conv1 (stride 2) and conv11 (transposed, + skip) become stride-1 2x2x2-tap convs.
        c0 = act3(1, 64); c0.s2d = True
        x11 = act3(1, 64); x11.s2d = True
        c1 = act3(1, 16); c2 = act3(1, 16); c3 = act3(2, 32); c4 = act3(2, 32)
        c5 = act3(3, 64); c6 = act3(3, 64); x7 = act3(2, 32); x9 = act3(1, 16)
        wcr = lambda nm: torch.as_tensor(sd[f"{cr}.{nm}.conv.weight"]).float()
        # conv0: depth-ring tcgen05 kernel (csrc/conv0_ring.cu), output written space-to-depth
        sc, sh = bn("conv0")
        w16 = G.conv0_ring_weights(wcr("conv0")).to(torch.float16).to(self.device).contiguous()
        self._keep.append(w16)
        plan = C.c_void_p()
        va = self.vol.c
        L.check(self.lib.adp_conv0_plan_create(C.byref(plan), C.byref(va), L.ptr(w16), L.ptr(sc), L.ptr(sh), L.ptr(c0.hi),
                                               L.LAYOUT_S2D, self.num_sms), "conv0_plan")
        self._conv0_plans.append(plan)

        def run0(batch, plan=plan):
            L.check(self.lib.adp_conv0_run(plan, batch, L.ptr(self.err_flag), self.stream), "conv0_run")
        run0.kind = "tc"
        ops.append(("cr.conv0", run0))
        # conv1 on the s2d tensor: a stride-1 2x2x2-tap conv over 64 channels
        sc, sh = bn("conv1")
        ops.append(("cr.conv1", self._tc_plans(c0, G.strided_s2d_weights(wcr("conv1")), 16, 1, 1, 1, 1,
                                               self._epilogue(c1, scale=sc, bias=sh, act=L.ACT_RELU), [G.strided_s2d(c0.D, c0.H, c0.W)])))
        for nm, xin, out, stride in (("conv2", c1, c2, 1), ("conv3", c2, c3, 2), ("conv4", c3, c4, 1), ("conv5", c4, c5, 2),
                                     ("conv6", c5, c6, 1)):
            sc, sh = bn(nm)
            ops.append((f"cr.{nm}", self._conv(wcr(nm).numpy(), xin, out, stride=stride, npass=1, scale=sc, bias=sh, act=L.ACT_RELU)))
        # conv7 (64 -> 32 at the coarsest level: 8 parity-class launches of the generic kernel) and conv9 (32 -> 16: the 8
        # parity classes fused in one kernel, csrc/tconv_fused.cu)
        sc, sh = bn("conv7")
        ops.append(("cr.conv7", self._conv(sd[f"{cr}.conv7.conv.weight"], c6, x7, stride=2, transposed=True, npass=1,
                                           scale=sc, bias=sh, act=L.ACT_RELU, res=c4, res_after_act=1)))
        for nm, xin, skip, out in (("conv9", x7, c2, x9),):
            sc, sh = bn(nm)
            wgt = wcr(nm)                                                              # [Cin, Cout, 3,3,3]
            cin, cout = wgt.shape[0], wgt.shape[1]
            bn_pad = 16 if cout <= 16 else 32
            wt = wgt.reshape(cin, cout, 27).permute(2, 1, 0).contiguous()              # [27, Cout, Cin]
            if bn_pad != cout:
                wt = torch.cat([wt, torch.zeros(27, bn_pad - cout, cin)], 1).contiguous()
            w16 = wt.to(torch.float16).to(self.device).contiguous()
            self._keep.append(w16)
            plan = C.c_void_p()
            xa = xin.c
            L.check(self.lib.adp_tconv_plan_create(C.byref(plan), C.byref(xa), L.ptr(w16), cout, L.ptr(sc), L.ptr(sh),
                                                   L.ptr(skip.hi), skip.Cn, L.ptr(out.hi), 0, self.num_sms), "tconv_plan")
            self._tconv_plans.append(plan)

            def runt(batch, plan=plan):
                L.check(self.lib.adp_tconv_run(plan, batch, L.ptr(self.err_flag), self.stream), "tconv_run")
            runt.kind = "tc"
            ops.append((f"cr.{nm}", runt))
        # conv11 (+ conv0 skip) writing the s2d layout: a stride-1 2x2x2-tap conv on the slab tcgen05 kernel
        sc, sh = bn("conv11")
        sc8, sh8 = self._dev(sc.cpu().repeat(8)), self._dev(sh.cpu().repeat(8))
        ep = self._epilogue(x11, scale=sc8, bias=sh8, act=L.ACT_RELU, res=c0, res_after_act=1)
        ops.append(("cr.conv11", self._tc_plans(x9, G.transposed_s2d_weights(wcr("conv11")), 64, 1, 1, 1, 1, ep,
                                                [G.transposed_s2d(x9.D, x9.H, x9.W)])))
        self.cr_ops = ops
        self.cr_taps = {"conv0": c0, "conv1": c1, "conv2": c2, "conv3": c3, "conv4": c4, "conv5": c5, "conv6": c6,
                        "conv7": x7, "conv9": x9, "conv11": x11}
        self.x11 = x11
        self.x11_format = L.LAYOUT_F16 | L.LAYOUT_S2D

    def _build_decode(self):
        sd, E, D, dev = self.sd, self.E, N_DEPTH, self.device
        cr = "cost_regularization"
        # decode weights, transposed to [K][N]
        def tw(name):
            w = torch.as_tensor(sd[name]).float()
            return self._dev(w.reshape(w.shape[0], -1).t().contiguous())
        dw = L.DecodeWeights()
        names = {"ic": "instance_color.0", "nh0": "nocs_head.0", "nh1": "nocs_head.2", "nh2": "nocs_head.4"}
        if self.regress_pose:
            names.update({"np0": "nocs_pts_mlp.0", "np1": "nocs_pts_mlp.2", "pm0": "pose_mlp1.0", "pm1": "pose_mlp1.2",
                          "q0": "pose_mlp2.0", "q1": "pose_mlp2.2", "r0": "rotation_estimator.0",
                          "r1": "rotation_estimator.2", "r2": "rotation_estimator.4"})
        for short, full in names.items():
            setattr(dw, f"{short}_w", L.ptr(tw(f"{full}.weight")))
            setattr(dw, f"{short}_b", L.ptr(self._dev(sd[f"{full}.bias"])))
        if self.need_volume:
            pw = torch.as_tensor(sd[f"{cr}.prob.weight"]).float()[0].permute(1, 2, 3, 0).contiguous()    # [kz,ky,kx,c]
            dw.prob_w = L.ptr(self._dev(pw.reshape(27, 8)))
        self.dw = dw
        P = self.P
        f32 = dict(dtype=torch.float32, device=dev)
        self.nocs = torch.zeros((self.F if self.branch_c else E, P, 3), **f32)
        self.depth = torch.zeros((E, P), **f32)
        self.gsum = torch.zeros((E, 128), **f32)
        self.psum = torch.zeros((E, 256), **f32)
        self.R = torch.zeros((E, 9), **f32)
        self.r6 = torch.zeros((E, 6), **f32)
        self.dbg_logits = torch.zeros((E, P, D), **f32) if self.debug else None
        self.dbg_fused = torch.zeros((E, P, 32), **f32) if self.debug else None
        # preprocess outputs (frames: [0,E) = view 1, [E,2E) = view 2)
        F = self.F
        self.bbox_ws = torch.zeros((F, 4), dtype=torch.int32, device=dev)
        self.win = torch.zeros((F, 4), dtype=torch.int32, device=dev)
        self.Kp = torch.zeros((F, 9), dtype=torch.float64, device=dev)
        self.valid = torch.zeros(F, dtype=torch.uint8, device=dev)
        self.choose = torch.zeros((F, P), dtype=torch.int32, device=dev)
        self.counts = torch.zeros(F, dtype=torch.int32, device=dev)
        self.bbox = torch.zeros((E, 8, 3), dtype=torch.float64, device=dev)
        self.scale = torch.zeros(E, dtype=torch.float64, device=dev)
        self.trans = torch.zeros((E, 3), dtype=torch.float64, device=dev)
        self.rot64 = torch.zeros((E, 9), dtype=torch.float64, device=dev)
        if self.branch_c:
            self.valid_f = torch.zeros(F, dtype=torch.uint8, device=dev)
            self.pts2d1 = torch.zeros((E, P, 2), **f32)
            self.pts_cam = torch.zeros((E, P, 3), **f32)
            self.nocs_m = torch.zeros((E, P, 3), **f32)
            self.match_count = torch.zeros(E, dtype=torch.int32, device=dev)
            self.match_ids = torch.zeros((E, P, 2), dtype=torch.int32, device=dev)
            self.R.copy_(torch.eye(3, device=dev).reshape(1, 9).expand(E, 9))
        elif self.arch == "baseline":
            # fusion.py:28-82 weights packed per block / direction / linear as [32 x 32 weight (out, in) | 32 bias]
            blocks = []
            for b in range(W.FUSION_DEPTH):
                for f in ("fusion1", "fusion2"):
                    for l in range(4):
                        nm = f"view_fusion.blocks.{b}.{f}.linears.{l}"
                        blocks += [np.asarray(sd[f"{nm}.weight"], np.float32).reshape(-1), np.asarray(sd[f"{nm}.bias"], np.float32)]
            self.fusion_w = self._dev(np.concatenate(blocks))
            g = lambda nm: np.asarray(sd[nm], np.float32)
            self.depth_w = self._dev(np.concatenate([g("depth_head.0.weight").reshape(64, 32).reshape(-1), g("depth_head.0.bias"),
                                                     g("depth_head.2.weight").reshape(32, 64).T.reshape(-1), g("depth_head.2.bias"),
                                                     g("depth_head.4.weight").reshape(-1), g("depth_head.4.bias")]))
            self.fusion_scratch = torch.zeros((4, E, P, 32), **f32)
            self.fused1 = torch.zeros((E, P, 32), **f32) if self.debug else None
            self.fused2 = torch.zeros((E, P, 32), **f32) if self.debug else None
            self.depth2 = torch.zeros((E, P), **f32) if self.debug else None
        self._build_decode_tc()

    def _build_decode_tc(self):
        """Per-point MLPs (network_v5.py:432-444,486-493) as 1x1 convolutions on the tcgen05 kernel: the P = 1024 sampled
        pixels of an env form a 32x32 "image", every layer is one split-precision (bf16x3) launch over all envs."""
        sd, P = self.sd, self.P
        assert P == 1024
        E = self.F if self.branch_c else self.E          # branch C decodes the frames of both views
        pt = lambda Cn: self._act(E, 32, 32, Cn, split=True)
        self.xfeat, self.xcat = pt(32), pt(96)
        h_ic, h_n0, h_n1, self.nocs16 = pt(64), pt(128), pt(64), pt(16)

        def fc(name, x, out, act=L.ACT_RELU, w=None, bias=None, **kw):
            w = torch.as_tensor(sd[f"{name}.weight"]).float().reshape(sd[f"{name}.weight"].shape[0], -1) if w is None else w
            cout, cin = w.shape
            if cin < x.Cn:      # nocs_pts_mlp.0 reads the 3 NOCS coordinates out of a 16-channel buffer
                w = torch.cat([w, torch.zeros(cout, x.Cn - cin)], 1)
            cout_pad = (cout + 15) // 16 * 16
            if cout_pad != cout:
                w = torch.cat([w, torch.zeros(cout_pad - cout, w.shape[1])], 0)
            bias = self._dev(sd[f"{name}.bias"]) if bias is None else bias
            ep = self._epilogue(out, bias=bias, act=act, **kw)
            return self._tc_plans(x, w[None].contiguous(), cout, 1, 1, 1, 3, ep, [None])

        ops = [("ic", fc("instance_color.0", self.xfeat, h_ic)),
               ("nh0", fc("nocs_head.0", h_ic, h_n0)),
               ("nh1", fc("nocs_head.2", h_n0, h_n1)),
               ("nh2", fc("nocs_head.4", h_n1, self.nocs16, act=L.ACT_TANH, out_f32=self.nocs, out_cstride=16))]
        if self.regress_pose:
            h_p0, h_m0, self.pf1b, h_q0, self.pf2b = pt(32), pt(128), pt(128), pt(256), pt(256)
            self.gbias = torch.zeros((E, 256), dtype=torch.float32, device=self.device)
            wq0 = torch.as_tensor(sd["pose_mlp2.0.weight"]).float().reshape(256, 256)
            ops += [("np0", fc("nocs_pts_mlp.0", self.nocs16, h_p0)),
                    ("np1", fc("nocs_pts_mlp.2", h_p0, self.xcat, out_cstride=96, out_coff=32)),
                    ("pm0", fc("pose_mlp1.0", self.xcat, h_m0)),
                    ("pm1", fc("pose_mlp1.2", h_m0, self.pf1b)),
                    ("gmean", lambda n: (
                        L.check(self.lib.adp_colsum(L.ptr(self.pf1b.hi), L.ptr(self.pf1b.lo), L.ptr(self.valid_env), L.ptr(self.gsum),
                                                    n, P, 128, self.stream), "colsum"),
                        L.check(self.lib.adp_pose_gbias(L.ptr(self.gsum), self.dw.q0_w, self.dw.q0_b, L.ptr(self.valid_env),
                                                        L.ptr(self.gbias), n, P, self.stream), "pose_gbias"))),
                    # pose_mlp2.0 on cat(pf, mean(pf)): the mean half of the product is the per-env bias computed above
                    ("q0", fc("pose_mlp2.0", self.pf1b, h_q0, w=wq0[:, :128].contiguous(), bias=self.gbias, bias_per_batch=1)),
                    ("q1", fc("pose_mlp2.2", h_q0, self.pf2b)),
                    ("rot", lambda n: (
                        L.check(self.lib.adp_colsum(L.ptr(self.pf2b.hi), L.ptr(self.pf2b.lo), L.ptr(self.valid_env), L.ptr(self.psum),
                                                    n, P, 256, self.stream), "colsum"),
                        L.check(self.lib.adp_rot_head(L.ptr(self.psum), L.ptr(self.valid_env), C.byref(self.dw), L.ptr(self.R),
                                                      L.ptr(self.r6), n, P, self.stream), "rot_head")))]
        self.dec_ops = ops

    # ------------------------------------------------------------------ stages
    @staticmethod
    def _dt(t, kinds):
        code = {torch.uint8: L.DT_U8, torch.bool: L.DT_U8, torch.float32: L.DT_F32, torch.float64: L.DT_F64}.get(t.dtype)
        if code is None or code not in kinds:
            raise TypeError(f"unsupported dtype {t.dtype}")
        return code

    def preprocess(self, view, rgb, mask, K, n, seed=0, choose=None, offset=None, frame_id0=0):
        """view 0/1; rgb [n,H,W,3] f32|f64|u8 (u8 = value / 255), mask [n,H,W] u8|bool|f32|f64, K [n,3,3] f64 -- device tensors.
        The frames land at [offset, offset + n) of the frame buffers (default: view * max_envs)."""
        E = self.E
        o = view * E if offset is None else offset
        assert rgb.is_cuda and mask.is_cuda and K.is_cuda and K.dtype == torch.float64
        assert rgb.is_contiguous() and mask.is_contiguous() and K.is_contiguous()
        if tuple(mask.shape) != tuple(rgb.shape[:3]) or rgb.shape[0] < n or rgb.shape[-1] != 3:
            raise ValueError(f"rgb {tuple(rgb.shape)} / mask {tuple(mask.shape)}: expected [n,H,W,3] and [n,H,W] with n >= {n}")
        H, Wd = rgb.shape[1], rgb.shape[2]
        mode = 0
        if choose is not None:
            self.choose[o:o + n].copy_(choose.to(torch.int32))
            mode = 1
        L.check(self.lib.adp_preprocess(
            L.ptr(rgb), self._dt(rgb, (L.DT_U8, L.DT_F32, L.DT_F64)), L.ptr(mask), self._dt(mask, (L.DT_U8, L.DT_F32, L.DT_F64)),
            L.ptr(K), 9, n, H, Wd, self.S, self.P, (seed * 2 + view) & 0xFFFFFFFF, mode, int(frame_id0),
            L.ptr(self.bbox_ws[o:]), L.ptr(self.win[o:]), L.ptr(self.Kp[o:]), L.ptr(self.valid[o:]), L.ptr(self.crops[o:]),
            L.ptr(self.choose[o:]), L.ptr(self.counts[o:]), self.stream), "preprocess")

    def stereo(self, n, E1, E2, mark=None, ransac_idx=None, seed=0, o2=None):
        """Frames [0,n) are view 1 and [E,E+n) view 2 of envs [0,n).  E1/E2 [n,4,4] f64 device tensors.
        ``mark(name)`` (optional) is called after each stage, e.g. to record CUDA events."""
        E, S, D, P = self.E, self.S, N_DEPTH, self.P
        if o2 is not None:
            E = o2          # view-2 frames start at frame o2 (partial chunks pack them right behind view 1)
        lib, st = self.lib, self.stream
        mark = mark or (lambda name: None)
        L.check(lib.adp_warp_matrices(L.ptr(self.Kp), L.ptr(E1), L.ptr(self.Kp[E:]), L.ptr(E2), L.ptr(self.Mw),
                                      L.ptr(self.valid), L.ptr(self.valid[E:]), L.ptr(self.valid_env), n, st), "warp_matrices")
        f1, f2 = self.feat, self.feat[E:]
        L.check(lib.adp_build_volume(L.ptr(self.feat16), L.ptr(self.feat16[E:]), L.ptr(self.Mw), L.ptr(self.depths),
                                     L.ptr(self.vol.hi), n, D, S, S, 32, 1, st), "build_volume")
        mark("volume")
        for name, op in self.cr_ops:
            op(n)
            mark(name)
        L.check(lib.adp_decode_gather(L.ptr(f1), L.ptr(f2), L.ptr(self.Mw), L.ptr(self.depths), L.ptr(self.x11.hi),
                                      L.ptr(self.choose), L.ptr(self.valid_env), self.dw.prob_w, L.ptr(self.depth),
                                      L.ptr(self.xfeat.hi), L.ptr(self.xfeat.lo), L.ptr(self.xcat.hi), L.ptr(self.xcat.lo),
                                      L.ptr(self.dbg_logits), L.ptr(self.dbg_fused), n, S, D, P, self.x11_format, st), "decode_gather")
        mark("decode_gather")
        for name, op in self.dec_ops:
            op(n)
        mark("decode")
        if self.regress_pose:
            L.check(lib.adp_fit(L.ptr(self.nocs), L.ptr(self.depth), L.ptr(self.choose), L.ptr(self.Kp), L.ptr(self.R), L.ptr(E1),
                                L.ptr(self.valid_env), L.ptr(self.bbox), L.ptr(self.scale), L.ptr(self.trans),
                                None, None, n, P, S, st), "fit")
        else:   # direct_regression = False, use_depth = True: RANSAC + Umeyama (interface_v5.py:322-338)
            L.check(lib.adp_fit_umeyama(L.ptr(self.nocs), L.ptr(self.depth), L.ptr(self.choose), L.ptr(self.Kp), L.ptr(E1),
                                        L.ptr(self.valid_env), L.ptr(ransac_idx), seed & 0xFFFFFFFF, L.ptr(self.bbox),
                                        L.ptr(self.scale), L.ptr(self.rot64), L.ptr(self.trans), n, P, S, st), "fit_umeyama")
        mark("fit")

    def single_view_nocs(self, rgb, mask, K, n, seed=0, choose=None, env0=0):
        """One view per environment (BASELINE configs[0..1]): preprocess -> backbone -> features at the sampled pixels ->
        instance_color -> nocs_head (network_v5.py:432-444; what the reference evaluates per view before any stereo term).
        n <= max_envs frames -> (self.nocs[:n] [n,P,3], self.choose[:n], self.valid[:n])."""
        assert n <= self.E
        self.preprocess(0, rgb, mask, K, n, seed, choose, frame_id0=env0)
        self.run_backbone(n)
        self.valid_env[:n].copy_(self.valid[:n])
        L.check(self.lib.adp_decode_gather(L.ptr(self.feat), None, None, None, None, L.ptr(self.choose), L.ptr(self.valid_env), None,
                                           None, L.ptr(self.xfeat.hi), L.ptr(self.xfeat.lo), None, None, None, None, n, self.S,
                                           N_DEPTH, self.P, 0, self.stream), "decode_gather(single view)")
        for _, op in self.dec_ops[:4]:          # instance_color, nocs_head x 3
            op(n)
        return self.nocs[:n], self.choose[:n], self.valid[:n]

    def run_chunk(self, K, rgb1, mask1, E1, rgb2, mask2, E2, seed=0, choose1=None, choose2=None, ransac_idx=None, env0=0):
        """Device tensors for n <= max_envs environments -> self.bbox[:n] ([n,8,3] f64, world frame).  ``env0``: global index
        of the chunk's first environment (keys the device pixel sampler, so a result does not depend on the chunking)."""
        n = K.shape[0]
        assert n <= self.E
        # view 2 sits right behind view 1 (frame n): a partial chunk runs the backbone on exactly 2 n frames
        self.preprocess(0, rgb1, mask1, K, n, seed, choose1, frame_id0=env0)
        self.preprocess(1, rgb2, mask2, K, n, seed, choose2, offset=n, frame_id0=env0)
        if self.use_graph and self.regress_pose and self.arch == "v5":
            # a chunk is ~95 launches from fixed buffers: replayed as one CUDA graph per chunk size (captured on the second
            # appearance of a size, after every kernel has run once and set its attributes).  estimate() splits a batch into
            # equal chunks, so a call sees at most two or three sizes.
            self.E1buf[:n].copy_(E1.reshape(n, 16))
            self.E2buf[:n].copy_(E2.reshape(n, 16))
            g = self._graphs.get(n)
            if g is None:
                runs = self._chunk_runs.get(n, 0) + 1
                self._chunk_runs[n] = runs
                if runs == 2 and len(self._graphs) < 8:
                    g = self._capture_graph(n)
            if g is not None:
                g[0].replay()
                self.lib.adp_launch_count_add(g[1])
                return self.bbox[:n]
            self.run_backbone(2 * n)
            self.stereo(n, self.E1buf, self.E2buf, o2=n)
            return self.bbox[:n]
        self.run_backbone(2 * n)
        if self.branch_c:
            return self.match_branch_c(n, K, E1, E2)
        if self.arch == "baseline":
            self.stereo_attention(n, E1, ransac_idx=ransac_idx, seed=seed, o2=n)
        else:
            self.stereo(n, E1, E2, ransac_idx=ransac_idx, seed=seed, o2=n)
        return self.bbox[:n]

    def stereo_attention(self, n, E1, ransac_idx=None, seed=0, o2=None):
        """The transformer variant behind the backbone (network_baseline.py:616-669): view-1 NOCS head, 4 cross-view attention
        blocks on the sampled point features of both views + depth MLP (adp_view_fusion), pose heads, fit.  Frames [0,n) are
        view 1, [o2,o2+n) view 2."""
        lib, st, P, S = self.lib, self.stream, self.P, self.S
        o2 = self.E if o2 is None else o2
        self.valid_env[:n].copy_(self.valid[:n] & self.valid[o2:o2 + n])
        L.check(lib.adp_decode_gather(L.ptr(self.feat), None, None, None, None, L.ptr(self.choose), L.ptr(self.valid_env), None,
                                      None, L.ptr(self.xfeat.hi), L.ptr(self.xfeat.lo), None, None, None, None, n, S,
                                      N_DEPTH, P, 0, st), "decode_gather(view 1)")
        for _, op in self.dec_ops[:4]:          # instance_color, nocs_head x 3
            op(n)
        L.check(lib.adp_view_fusion(L.ptr(self.feat), L.ptr(self.feat[o2:]), L.ptr(self.choose), L.ptr(self.choose[o2:]),
                                    L.ptr(self.valid_env), L.ptr(self.fusion_w), L.ptr(self.depth_w), L.ptr(self.fusion_scratch),
                                    L.ptr(self.depth), L.ptr(self.depth2), L.ptr(self.xcat.hi), L.ptr(self.xcat.lo),
                                    L.ptr(self.fused1), L.ptr(self.fused2), n, S, P, W.FUSION_DEPTH, st), "view_fusion")
        for _, op in self.dec_ops[4:]:          # nocs_pts_mlp, pose_mlp1 / 2, rotation head (regress_pose only)
            op(n)
        if self.regress_pose:
            L.check(lib.adp_fit(L.ptr(self.nocs), L.ptr(self.depth), L.ptr(self.choose), L.ptr(self.Kp), L.ptr(self.R), L.ptr(E1),
                                L.ptr(self.valid_env), L.ptr(self.bbox), L.ptr(self.scale), L.ptr(self.trans),
                                None, None, n, P, S, st), "fit")
        else:
            L.check(lib.adp_fit_umeyama(L.ptr(self.nocs), L.ptr(self.depth), L.ptr(self.choose), L.ptr(self.Kp), L.ptr(E1),
                                        L.ptr(self.valid_env), L.ptr(ransac_idx), seed & 0xFFFFFFFF, L.ptr(self.bbox),
                                        L.ptr(self.scale), L.ptr(self.rot64), L.ptr(self.trans), n, P, S, st), "fit_umeyama")

    def match_branch_c(self, n, K, E1, E2):
        """Frames [0,n) = view 1, [n,2n) = view 2 (features present).  -> dict of device tensors for the host PnP tail:
        nocs1 [n,P,3], pts2d1 [n,P,2], scale [n] (median scale of the triangulated matches), count [n], valid [n]."""
        lib, st, P, S = self.lib, self.stream, self.P, self.S
        self.valid_f[:2 * n].copy_(self.valid[:2 * n])
        L.check(lib.adp_decode_gather(L.ptr(self.feat), None, None, None, None, L.ptr(self.choose), L.ptr(self.valid_f), None,
                                      None, L.ptr(self.xfeat.hi), L.ptr(self.xfeat.lo), None, None, None, None, 2 * n, S,
                                      N_DEPTH, P, 0, st), "decode_gather(branch C)")
        for _, op in self.dec_ops[:4]:
            op(2 * n)
        self.valid_env[:n].copy_(self.valid[:n] & self.valid[n:2 * n])
        Kc = K.reshape(n, 9).contiguous()
        L.check(lib.adp_nocs_match(L.ptr(self.nocs), L.ptr(self.nocs[n:]), L.ptr(self.choose), L.ptr(self.choose[n:]), L.ptr(self.win),
                                   L.ptr(self.win[n:]), L.ptr(Kc), L.ptr(E1), L.ptr(E2), L.ptr(self.valid_env), S, L.ptr(self.pts2d1),
                                   L.ptr(self.pts_cam), L.ptr(self.nocs_m), L.ptr(self.match_count), L.ptr(self.match_ids), n, P, st),
                "nocs_match")
        L.check(lib.adp_fit(L.ptr(self.nocs_m), None, None, L.ptr(self.Kp), L.ptr(self.R), L.ptr(E1), L.ptr(self.valid_env),
                            L.ptr(self.bbox), L.ptr(self.scale), L.ptr(self.trans), L.ptr(self.pts_cam), L.ptr(self.match_count),
                            n, P, S, st), "fit(points mode)")
        return dict(nocs1=self.nocs[:n], pts2d1=self.pts2d1[:n], scale=self.scale[:n], count=self.match_count[:n],
                    valid=self.valid_env[:n], match_ids=self.match_ids[:n], pts_cam=self.pts_cam[:n])

    def _capture_graph(self, n):
        import warnings
        l0 = self.lib.adp_launch_count()
        try:
            g = torch.cuda.CUDAGraph()
            # thread-local capture mode: with one engine per GPU driven by one host thread each (single-process multi-GPU), the
            # other threads keep issuing copies / allocations on their own devices while this one captures
            # (and an explicit capture stream on THIS device: torch caches one process-wide default capture stream, created on
            # whichever device captured first, and would switch the current device to it)
            if self._capture_stream is None:
                self._capture_stream = torch.cuda.Stream(self.device)
            with _CAPTURE_LOCK, torch.cuda.graph(g, stream=self._capture_stream, capture_error_mode="thread_local"):
                self.run_backbone(2 * n)
                self.stereo(n, self.E1buf, self.E2buf, o2=n)
            launches = int(self.lib.adp_launch_count() - l0)
            self.lib.adp_launch_count_add(C.c_uint64(-launches & 0xFFFFFFFFFFFFFFFF))   # capture itself launched nothing
            self._graphs[n] = (g, launches)
            return self._graphs[n]
        except Exception as e:      # stay on the eager launch path (same kernels), say so once
            warnings.warn(f"CUDA graph capture of a chunk failed ({e}); launching eagerly")
            self.use_graph = False
            return None


    def post_error_flag(self):
        """Queue an asynchronous read of the device flags behind the work issued so far (no synchronisation)."""
        self._err_host.copy_(self.err_flag, non_blocking=True)
        self._err_event = torch.cuda.Event()
        self._err_event.record(torch.cuda.current_stream(self.device))

    def check_error_flag(self, wait=True):
        """Raise if the watchdog or the fp16 range guard fired.  ``wait=False`` only looks at a read posted earlier by
        :meth:`post_error_flag` that has already completed (the tensor-returning paths check one call late instead of
        synchronising)."""
        if self._err_event is None:
            if not wait:
                return
            self.post_error_flag()
        if not wait and not self._err_event.query():
            return
        self._err_event.synchronize()
        self._err_event = None
        code, rng = int(self._err_host[0]), int(self._err_host[1])
        if code or rng:
            self.err_flag.zero_()
        if code:
            raise L.AdpError(f"device pipeline watchdog tripped (code {code})")
        if rng:
            raise L.AdpError("non-finite backbone features: the activations of this checkpoint exceed the fp16 range; "
                             "construct the estimator with precision='bf16x3'")

    def close(self):
        self._graphs = {}            # the captured graphs reference the plans' parameter blocks
        for p in self._plans:
            self.lib.adp_conv_tc_free(p)
        self._plans = []
        for p in self._conv0_plans:
            self.lib.adp_conv0_free(p)
        self._conv0_plans = []
        for p in self._tconv_plans:
            self.lib.adp_tconv_free(p)
        self._tconv_plans = []

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
