"""The plane-sweep volume builder (csrc/volume.cu, build_volume_tile_kernel) per voxel against a float64 reference, and the
warp matrices that feed it (warp_matrices_kernel) against numpy float64.

    vol[b, d, y, x, :] = feat_ref[b, y, x, :] + bilinear(feat_src[b], ix(d, y, x), iy(d, y, x))

One block of the kernel is a 16 x 16 tile of reference pixels for 8 consecutive depth planes.  Per (tile, plane) it takes one of
three paths: the empty shortcut (fp16 output only: the four tile corners project outside the map on one side, with positive
depth, so the plane is a copy of feat_ref), the staged footprint (the bounding box of the tile's bilinear cells, <= 480 source
pixels, copied to shared memory) or the direct gather from global memory.  A CPU mirror of that decision (`census`) reports
which paths each case reaches; it runs without a GPU.

Reference: torch float64 (on the GPU for the large cases) over exactly what the kernel reads: the fp16 feature maps, the fp32
Mw and the fp32 depths.  Sample coordinates follow network_v5.py:389-413 as written (normalise with (W-1)/2, sample with
align_corners=False: ix = px W / (W-1) - 1/2), bilinear with zero padding.  Bound per voxel and channel, on top of one ulp of
the output format at |ref| (added by assert_close):
  * weight rounding: each bilinear weight is rounded to fp16 for the mixed-precision FMA: sum_k |c_k| (2^-11 w_k) (the fp16
    unit roundoff), plus 2^-25 per corner of the 4 x 4 neighbourhood for subnormal weights and 2^-9 delta max|c| for a corner the
    kernel picks on the other side of a cell edge (its weight is <= 2 delta);
  * accumulation: four fp32 roundings, 4 2^-24 (|feat_ref| + sum_k (w_k + 2 delta) |c_k|);
  * sample position: bilinear sampling with zero padding is continuous and piecewise linear in the coordinate, so a coordinate
    error delta moves a sample by at most 2 delta L, L = the per-channel range over the 4 x 4 neighbourhood (0 outside the map).
    delta = max(2^-11 px, a first-order model of the kernel's fp32 error): 6 roundings in each of X, Y, Z (relative to the sum
    of the magnitudes of their terms), rcp.approx (1 ulp), the product, and the normalisation chain, 2^-24 (8 (|ix| + 1) + W).
    Near Z = 0 the model grows without bound; a voxel whose delta exceeds DELTA_CAP is not compared, and their number is
    capped per case (MAX_EXCLUDED).
Exact bits:
  * a voxel that samples nothing in the reference (its coordinate beyond [-1, W] x [-1, H] by more than 2 delta, or not
    finite) is feat_ref: its bits for fp16 output, bf16(feat_ref) for bf16 output;
  * the same arithmetic in another block grouping (a sub-range of the depths, one environment alone) gives the same bits;
  * voxels outside the launch's [B, D, H, W, 32] keep their canary bits.
Warp matrices: per element one fp32 rounding of the numpy float64 P_src inv(P_ref) plus 1e-12 of the row's magnitude.
"""
import math
import zlib
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from gpu_util import CANARY16, assert_close, bits, canary16

pytestmark = [pytest.mark.filterwarnings("ignore")]
GPU = pytest.mark.gpu

VT_T, VT_DG, VT_MAXPX = 16, 8, 480          # tile edge, depth planes per block, staged pixels (csrc/volume.cu)
DELTA = 2.0 ** -11                          # px: the coordinate error bound of well-conditioned geometry
DELTA_CAP = 0.25                            # px: voxels with a larger modelled coordinate error are not compared
MAX_EXCLUDED = 64                           # per case, in pixels x planes
U = 2.0 ** -24
F16, BF16 = torch.float16, torch.bfloat16
REGIMES = ("empty", "staged", "fallback", "none", "ambiguous")


@pytest.fixture(scope="module")
def G():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    import importlib
    from rgbmanip_b200 import _lib as L
    L.load()
    return importlib.import_module("gpu_util")


def _rng(name):
    return np.random.default_rng(zlib.crc32(name.encode()))


# ================================================================================================ geometry of the cases
def affine(th_deg=0.0, sc=1.0, tx=0.0, ty=0.0, persp=(0.0, 0.0), trans=(0.0, 0.0, 0.0)):
    """Mw row (rot 3x3 row-major, trans 3) of px = (A (x, y, 1) dep + trans) / Z: a rotation by th, scale sc and shift (tx, ty)
    of the pixel grid, an optional perspective row and a depth-dependent translation."""
    c, s = sc * math.cos(math.radians(th_deg)), sc * math.sin(math.radians(th_deg))
    return [c, -s, tx, s, c, ty, persp[0], persp[1], 1.0, *trans]


def about(th_deg, sc, cx, cy, to_x, to_y, **kw):
    """affine() that maps reference point (cx, cy) to source point (to_x, to_y)."""
    c, s = sc * math.cos(math.radians(th_deg)), sc * math.sin(math.radians(th_deg))
    return affine(th_deg, sc, to_x - (c * cx - s * cy), to_y - (s * cx + c * cy), **kw)


def _px_target(i, n):
    """px of sample coordinate i in a map of n pixels (the inverse of i = px n / (n - 1) - 1/2)."""
    return (i + 0.5) * (n - 1) / n


def border_case():
    """Four environments translate the pixel grid by +-16 / dep along x or y (Mw[9] or Mw[10]), so that the depths below put
    a tile corner's image at ix (iy) = W (H) + {-0.01, +0.005, +0.02} (the left / top corner of tile column 2) and at
    -1.02, -1.005, -0.99 (the right / bottom corner of tile column 1), across the 0.01 px margin of the empty test."""
    S, a = 64, 16.0
    deps = [a / (_px_target(S + e, S) - 32) for e in (-0.01, 0.005, 0.02)]
    deps += [a / (31 - _px_target(-1 + e, S)) for e in (-0.02, -0.005, 0.01)]
    deps += [a / 5.0, a / 40.0]
    Mw = [affine(trans=(a, 0, 0)), affine(trans=(-a, 0, 0)), affine(trans=(0, a, 0)), affine(trans=(0, -a, 0))]
    return SimpleNamespace(name="borders", Mw=np.array(Mw, np.float32), depths=np.array(deps, np.float32), H=S, W=S)


def pole_case():
    """env 0: a 45-degree rotation with scale 3 that maps tile (0, 0)'s centre to (-3, -3): its four corner images lie outside
    the map, not all on one side, and its interior samples the map.  env 1: px = (-3 x dep + 80) / (x dep - 23.5),
    py = 10: Z changes sign at x = 23.5 / dep.  dep 1: Z crosses 0 between columns 23 and 24 (tile column 1, whose four corner
    images are all left of the map while its interior samples it); dep 47/32: Z = 0 exactly on column 16; dep 0.3: Z < 0
    everywhere; dep 4: the sign change inside tile column 0."""
    Mw = [about(45.0, 3.0, 7.5, 7.5, -3.0, -3.0), [-3.0, 0, 0, 10.0, 0, 0, 1.0, 0, 0, 80.0, -235.0, -23.5]]
    return SimpleNamespace(name="pole", Mw=np.array(Mw, np.float32), depths=np.array([1.0, 47 / 32, 0.3, 4.0, 2.0], np.float32),
                           H=64, W=64)


def footprint_case():
    """One launch over three environments at the engine size: a 40-degree rotation with scale 1.3 (interior tiles have ~900
    pixel footprints: the direct gather; border tiles clip to the map: staged), a strong shrink (0.35) and a translation by
    -2 + 48 / dep that moves part of the tile grid off the map (empty tiles beside staged ones in one plane)."""
    Mw = [about(40.0, 1.3, 111.5, 111.5, 111.5, 111.5, trans=(1.5, -1.0, 0.0)),
          about(-8.0, 0.35, 111.5, 111.5, 100.0, 120.0, persp=(1e-4, -5e-5)),
          affine(tx=-2.0, ty=3.0, trans=(48.0, 0.0, 0.0))]
    deps = np.array([0.1, 0.2, 0.3, 0.5, 0.8, 1.2, 1.7, 2.4, 0.45], np.float32)
    return SimpleNamespace(name="footprint", Mw=np.array(Mw, np.float32), depths=deps, H=224, W=224)


RAGGED = [(37, 50), (16, 17), (224, 200)]


def ragged_case(H, W, D):
    """Two environments with different, mildly projective Mw and depth-dependent translations; D of the engine's depths."""
    from oracle import adapose_oracle as O
    Mw = [about(5.0, 1.05, W / 2, H / 2, W / 2 + 2.3, H / 2 - 1.7, persp=(1e-4, 2e-4), trans=(0.4, -0.3, 0.002)),
          about(-12.0, 0.9, W / 2, H / 2, W / 2 - 3.1, H / 2 + 0.6, persp=(-2e-4, 1e-4), trans=(-0.2, 0.5, -0.001))]
    return SimpleNamespace(name=f"ragged_{H}x{W}_D{D}", Mw=np.array(Mw, np.float32), depths=O.depth_hypotheses()[:D].copy(),
                           H=H, W=W)


def engine_cameras(B=3, seed=5):
    """(Kp_ref, E_ref, Kp_src, E_src) float64 of B synth scenes through the oracle's crop (as the engine forms them)."""
    from oracle import adapose_oracle as O
    from rgbmanip_b200 import synth
    batch = synth.make_batch(B, seed=seed, special=False)
    np.random.seed(seed)
    kp1 = np.stack([O.prepare_model_input(batch.rgb1[e], batch.mask1[e], batch.K[e])[3] for e in range(B)])
    kp2 = np.stack([O.prepare_model_input(batch.rgb2[e], batch.mask2[e], batch.K[e])[3] for e in range(B)])
    return kp1, batch.E1.astype(np.float64), kp2, batch.E2.astype(np.float64)


def warp_ref(Kp_ref, E_ref, Kp_src, E_src):
    """float64 M = P_src inv(P_ref), P = [K' E[:3, :]; 0 0 0 1], as [B, 12] (rot row-major, trans)."""
    def P(K, E):
        p = np.tile(np.eye(4), (len(K), 1, 1))
        p[:, :3, :] = K @ E[:, :3, :]
        return p
    M = P(Kp_src, E_src) @ np.linalg.inv(P(Kp_ref, E_ref))
    return np.concatenate([M[:, :3, :3].reshape(-1, 9), M[:, :3, 3]], 1), M[:, :3, :]


def engine_case(Mw=None):
    """The engine's geometry: 3 synth scenes, 224 x 224, the 24 depth hypotheses.  Mw: the device's (adp_warp_matrices) or,
    without one, the float64 reference rounded to fp32."""
    from oracle import adapose_oracle as O
    if Mw is None:
        Mw = warp_ref(*engine_cameras())[0].astype(np.float32)
    return SimpleNamespace(name="engine", Mw=np.asarray(Mw, np.float32), depths=O.depth_hypotheses(), H=224, W=224)


# ================================================================================================ float64 reference
def coords(M, depths, H, W, dev="cpu"):
    """float64 sample coordinates (ix, iy) [D, H, W] of every reference pixel at every depth, Z, and delta: the coordinate error
    bound of the kernel's fp32 arithmetic (inf where the coordinate is not finite).  M: [12] fp32 values, depths: [D] fp32."""
    M = torch.as_tensor(np.asarray(M, np.float64), device=dev)
    dep = torch.as_tensor(np.asarray(depths, np.float64), device=dev)[:, None, None]
    y, x = torch.meshgrid(torch.arange(H, dtype=torch.float64, device=dev), torch.arange(W, dtype=torch.float64, device=dev),
                          indexing="ij")
    r = [M[3 * i] * x + M[3 * i + 1] * y + M[3 * i + 2] for i in range(3)]
    a = [(M[3 * i] * x).abs() + (M[3 * i + 1] * y).abs() + M[3 * i + 2].abs() for i in range(3)]
    X, Y, Z = (r[i] * dep + M[9 + i] for i in range(3))
    AX, AY, AZ = (a[i] * dep.abs() + M[9 + i].abs() for i in range(3))
    with np.errstate(all="ignore"):
        px, py = X / Z, Y / Z
        ix, iy = px * (W / (W - 1)) - 0.5, py * (H / (H - 1)) - 0.5
        ez = 6 * U * AZ / Z.abs()
        dx = (W / (W - 1)) * (6 * U * AX / Z.abs() + px.abs() * (ez + 3 * U)) + U * (8 * (ix.abs() + 1) + W)
        dy = (H / (H - 1)) * (6 * U * AY / Z.abs() + py.abs() * (ez + 3 * U)) + U * (8 * (iy.abs() + 1) + H)
    delta = torch.maximum(dx, dy).clamp_min(DELTA)
    delta = torch.where(torch.isfinite(ix) & torch.isfinite(iy), delta, torch.full_like(delta, math.inf))
    return ix, iy, Z, delta


def plane_ref(fr, fs, ix, iy, delta, H, W):
    """float64 reference of one plane: fr, fs [H, W, 32] (the fp16 values), ix, iy, delta [H, W].  Returns (ref, bound,
    nothing, excluded): nothing = samples no source pixel by a margin of 2 delta; excluded = delta > DELTA_CAP otherwise."""
    fin = torch.isfinite(ix) & torch.isfinite(iy)
    nothing = ~fin | (ix < -1 - 2 * delta) | (iy < -1 - 2 * delta) | (ix > W + 2 * delta) | (iy > H + 2 * delta)
    excluded = ~nothing & (delta > DELTA_CAP)
    ixc = torch.where(fin, ix, torch.full_like(ix, -8.0)).clamp(-8.0, W + 8.0)
    iyc = torch.where(fin, iy, torch.full_like(iy, -8.0)).clamp(-8.0, H + 8.0)
    x0, y0 = ixc.floor(), iyc.floor()
    ex, ey = (ixc - x0)[..., None], (iyc - y0)[..., None]
    off = torch.arange(-1, 3, dtype=torch.float64, device=ix.device)
    xs, ys = x0[..., None] + off, y0[..., None] + off                      # [H, W, 4]
    inx, iny = (xs >= 0) & (xs < W), (ys >= 0) & (ys < H)
    xi, yi = xs.clamp(0, W - 1).long(), ys.clamp(0, H - 1).long()
    nb = fs[yi[..., :, None], xi[..., None, :]]                            # [H, W, 4 (y), 4 (x), 32]
    nb = nb * (iny[..., :, None] & inx[..., None, :])[..., None]
    rng = nb.amax((2, 3)) - nb.amin((2, 3))
    mx = nb.abs().amax((2, 3))
    c = (nb[:, :, 1, 1], nb[:, :, 1, 2], nb[:, :, 2, 1], nb[:, :, 2, 2])
    w = ((1 - ex) * (1 - ey), ex * (1 - ey), (1 - ex) * ey, ex * ey)
    d = delta.clamp_max(DELTA_CAP)[..., None]
    ref = fr + sum(wk * ck for wk, ck in zip(w, c))
    bound = (sum(2.0 ** -11 * wk * ck.abs() for wk, ck in zip(w, c)) + (16 * 2.0 ** -25 + 2.0 ** -9 * d) * mx
             + 4 * U * (fr.abs() + sum((wk + 2 * d) * ck.abs() for wk, ck in zip(w, c))) + 2 * d * rng)
    bound = torch.where(excluded[..., None], torch.full_like(bound, math.inf), bound)
    return ref, bound, nothing, excluded


def as_out(x, dt):
    """The kernel's output format of fp32-exact values: fp16 as is, bf16 by round to nearest even."""
    return x.to(dt)


def check_volume(case, feats, vol, what, dev):
    """Every voxel of vol [B, D, H, W, 32] (device, fp16 or bf16) against the float64 reference.  feats: (feat_ref, feat_src)
    fp16 [B, H, W, 32] on `dev`.  Returns (largest error / bound, excluded voxel count, voxels that sample nothing)."""
    fmt = "f16" if vol.dtype == F16 else "bf16"
    B, D, H, W, _ = vol.shape
    worst, n_excl, n_nothing = 0.0, 0, 0
    for b in range(B):
        fr16, fs = feats[0][b], feats[1][b].double()
        fr = fr16.double()
        ix, iy, _, delta = coords(case.Mw[b], case.depths, H, W, dev)
        want_bits = as_out(fr16, vol.dtype).view(torch.int16)
        for d in range(D):
            ref, bound, nothing, excl = plane_ref(fr, fs, ix[d], iy[d], delta[d], H, W)
            got = vol[b, d]
            worst = max(worst, assert_close(got, ref, fmt, bound, f"{what} env {b} plane {d}"))
            g16 = got.view(torch.int16)
            same = (g16 == want_bits).all(-1)
            if not bool(same[nothing].all()):
                yx = torch.nonzero(nothing & ~same)[0].tolist()
                raise AssertionError(f"{what} env {b} plane {d}: voxel {yx} samples nothing but is not feat_ref "
                                     f"({int((nothing & ~same).sum())} such voxels)")
            n_excl += int(excl.sum())
            n_nothing += int(nothing.sum())
    assert n_excl <= MAX_EXCLUDED, f"{what}: {n_excl} voxels excluded near Z = 0"
    return worst, n_excl, n_nothing


# ================================================================================================ regime census (CPU)
def census(case, f16=True, margin=1e-3):
    """Mirror of the kernel's decision per (env, plane, tile) in float64: returns (codes [B, D, tiles_y, tiles_x] indexing
    REGIMES, extra counters).  A decision that the kernel's fp32 rounding could flip (within `margin` px of a threshold) is
    'ambiguous'; after one, the rest of that block's planes are too (the kernel's box carries over between planes).  The box
    is double-buffered by plane parity as in the kernel: an empty plane skips the reset, so the next plane's box also holds the
    plane two before."""
    H, W, D = case.H, case.W, len(case.depths)
    ty_n, tx_n = -(-H // VT_T), -(-W // VT_T)
    B = len(case.Mw)
    codes = np.zeros((B, D, ty_n, tx_n), np.int64)
    extra = {"one_side_but_z": 0, "outside_not_one_side": 0}
    pad = lambda a, fill: np.pad(a, ((0, 0), (0, ty_n * VT_T - H), (0, tx_n * VT_T - W)), constant_values=fill)
    tiles = lambda a: a.reshape(D, ty_n, VT_T, tx_n, VT_T)
    cx = np.minimum(np.arange(tx_n)[:, None] * VT_T + np.array([0, VT_T - 1]), W - 1)        # [tx, 2]
    cy = np.minimum(np.arange(ty_n)[:, None] * VT_T + np.array([0, VT_T - 1]), H - 1)
    for b in range(B):
        ix, iy, Z, _ = (t.numpy() for t in coords(case.Mw[b], case.depths, H, W))
        with np.errstate(invalid="ignore"):
            fin = np.isfinite(ix) & np.isfinite(iy)
            ixs, iys = np.where(fin, ix, -1e9), np.where(fin, iy, -1e9)
            # corners: [D, ty, 2, tx, 2]
            cix, ciy, cz = (a[:, cy[:, :, None, None], cx[None, None]] for a in (ixs, iys, Z))
            cfin = fin[:, cy[:, :, None, None], cx[None, None]]
            sides = []
            for m in (margin, -margin):          # m > 0: surely outside; m < 0: possibly outside
                s = np.stack([cix < -1.01 - m, cix > W + 0.01 + m, ciy < -1.01 - m, ciy > H + 0.01 + m], -1)
                sides.append(s.all((2, 4)).any(-1))                               # all four corners on one side: [D, ty, tx]
            zpos_sure = ((cz > 1e-6 + margin) & cfin).all((2, 4))
            zneg_maybe = ~((cz > 1e-6 - margin) & cfin).all((2, 4))
            empty_sure = sides[0] & zpos_sure
            empty_maybe = sides[1] & ~zneg_maybe if f16 else np.zeros_like(empty_sure)
            if not f16:
                empty_sure = np.zeros_like(empty_sure)
            out_all = (((cix < -1.01 - margin) | (cix > W + 0.01 + margin) | (ciy < -1.01 - margin)
                        | (ciy > H + 0.01 + margin)).all((2, 4)))
            # bilinear cells of the tile's pixels: the kernel's any / floor, bracketed by +-margin
            hi_any = fin & (ix >= -1 - margin) & (iy >= -1 - margin) & (ix <= W + margin) & (iy <= H + margin)
            lo_any = fin & (ix >= -1 + margin) & (iy >= -1 + margin) & (ix <= W - margin) & (iy <= H - margin)
            samples = tiles(pad(lo_any, False)).any((2, 4))                    # some pixel surely samples the map

            def red(v, sel, fn, fill):
                return fn(tiles(pad(np.where(sel, v, fill), fill)), axis=(2, 4))
            fxm, fxp = np.floor(ixs - margin), np.floor(ixs + margin)
            fym, fyp = np.floor(iys - margin), np.floor(iys + margin)
            big = 1e9
            outer = np.stack([red(fxm, hi_any, np.min, big), red(fym, hi_any, np.min, big),
                              red(fxp, hi_any, np.max, -big) + 1, red(fyp, hi_any, np.max, -big) + 1], -1)
            inner = np.stack([red(fxp, lo_any, np.min, big), red(fyp, lo_any, np.min, big),
                              red(fxm, lo_any, np.max, -big) + 1, red(fym, lo_any, np.max, -big) + 1], -1)
        extra["one_side_but_z"] += int((sides[0] & ~zpos_sure & samples).sum())
        extra["outside_not_one_side"] += int((out_all & ~sides[1] & samples).sum())

        def area(bx):
            x0, y0 = np.maximum(bx[..., 0], 0), np.maximum(bx[..., 1], 0)
            x1, y1 = np.minimum(bx[..., 2], W - 1), np.minimum(bx[..., 3], H - 1)
            ok = bx[..., 2] >= bx[..., 0]
            bw, bh = np.where(ok, x1 - x0 + 1, 0), np.where(ok, y1 - y0 + 1, 0)
            return np.where((bw > 0) & (bh > 0), bw * bh, 0)

        empty_box = np.array([big, big, -big, -big])
        for g0 in range(0, D, VT_DG):
            for ty in range(ty_n):
                for tx in range(tx_n):
                    box = {"o": [empty_box.copy(), empty_box.copy()], "i": [empty_box.copy(), empty_box.copy()]}
                    lost = False
                    for d in range(g0, min(g0 + VT_DG, D)):
                        if lost or (empty_maybe[d, ty, tx] and not empty_sure[d, ty, tx]):
                            codes[b, d, ty, tx], lost = REGIMES.index("ambiguous"), True
                            continue
                        if empty_sure[d, ty, tx]:
                            codes[b, d, ty, tx] = REGIMES.index("empty")
                            continue
                        p = d & 1
                        for k, src in (("o", outer), ("i", inner)):
                            bx = box[k][p]
                            bx[:2] = np.minimum(bx[:2], src[d, ty, tx, :2])
                            bx[2:] = np.maximum(bx[2:], src[d, ty, tx, 2:])
                        ao, ai = area(box["o"][p]), area(box["i"][p])
                        if ao == 0:
                            code = "none"
                        elif ai > VT_MAXPX:
                            code = "fallback"
                        elif ao <= VT_MAXPX and ai > 0:
                            code = "staged"
                        else:
                            code = "ambiguous"
                        codes[b, d, ty, tx] = REGIMES.index(code)
                        box["o"][p ^ 1], box["i"][p ^ 1] = empty_box.copy(), empty_box.copy()
    return codes, extra


def census_counts(codes):
    return {r: int((codes == i).sum()) for i, r in enumerate(REGIMES)}


def mixed_planes(codes, a, b):
    """Number of (env, plane) pairs with tiles in regime a and in regime b."""
    ia, ib = REGIMES.index(a), REGIMES.index(b)
    return int(((codes == ia).any((2, 3)) & (codes == ib).any((2, 3))).sum())


# What each case must reach (fp16 output).  Together: every regime, a launch with staged and fallback tiles, planes with staged
# and empty tiles, the Z guard and the not-on-one-side corner test.
EXPECT = {
    "engine": dict(staged=True),
    "footprint": dict(staged=True, fallback=True, empty=True, mixed=[("staged", "empty"), ("staged", "fallback")]),
    "borders": dict(staged=True, empty=True, none=True, mixed=[("staged", "empty")]),
    "pole": dict(staged=True, extra=("one_side_but_z", "outside_not_one_side")),
}


def _cpu_case(name):
    if name == "engine":
        return engine_case()
    return {"footprint": footprint_case, "borders": border_case, "pole": pole_case}[name]()


def assert_census(case, codes, extra):
    cnt = census_counts(codes)
    exp = EXPECT.get(case.name, {})
    for r in ("empty", "staged", "fallback", "none"):
        if exp.get(r):
            assert cnt[r] > 0, (case.name, r, cnt)
    for a, b in exp.get("mixed", []):
        assert mixed_planes(codes, a, b) > 0, (case.name, a, b, cnt)
    for k in exp.get("extra", ()):
        assert extra[k] > 0, (case.name, k, extra)
    return cnt


@pytest.mark.parametrize("name", list(EXPECT))
def test_regime_census(name):
    """The CPU mirror of the kernel's per-(tile, plane) path decision reaches what each case is built for."""
    case = _cpu_case(name)
    codes, extra = census(case)
    cnt = assert_census(case, codes, extra)
    print(f"census {name}: {cnt} {extra}")


def test_census_covers_every_regime():
    seen = set()
    for name in EXPECT:
        codes, _ = census(_cpu_case(name))
        seen |= {r for r, n in census_counts(codes).items() if n}
    assert {"empty", "staged", "fallback", "none"} <= seen


def test_census_bf16_output_never_shortcuts():
    codes, _ = census(border_case(), f16=False)
    assert census_counts(codes)["empty"] == 0


def test_reference_matches_oracle_homo_warping():
    """The float64 reference, evaluated in fp32-free form, against O.homo_warping (fp32, grid_sample) on a small projective
    case: this anchors the coordinate convention to the oracle."""
    from oracle import adapose_oracle as O
    case = ragged_case(37, 50, 5)
    rng = _rng("anchor")
    B, H, W = 2, case.H, case.W
    fs = torch.from_numpy(rng.standard_normal((B, H, W, 32), dtype=np.float32)).half().float()
    Mw = torch.from_numpy(case.Mw).double()
    proj = torch.eye(4, dtype=torch.float64).repeat(B, 1, 1)
    proj[:, :3, :3], proj[:, :3, 3] = Mw[:, :9].reshape(B, 3, 3), Mw[:, 9:]
    want = O.homo_warping(fs.permute(0, 3, 1, 2), proj.float(), torch.eye(4).repeat(B, 1, 1),
                          torch.from_numpy(case.depths)[None].repeat(B, 1)).permute(0, 2, 3, 4, 1)
    for b in range(B):
        ix, iy, _, delta = coords(case.Mw[b], case.depths, H, W)
        for d in range(len(case.depths)):
            ref, _, _, _ = plane_ref(torch.zeros(H, W, 32, dtype=torch.float64), fs[b].double(), ix[d], iy[d], delta[d], H, W)
            assert float((ref - want[b, d].double()).abs().max()) < 2e-3, (b, d)


# ================================================================================================ device runs
def dev_case(G, case, name=None, B=None):
    """Seeded fp16 feature maps and the device copies of a case's inputs."""
    rng = _rng(name or case.name)
    B = len(case.Mw) if B is None else B
    fr = torch.from_numpy(rng.standard_normal((B, case.H, case.W, 32), dtype=np.float32)).half().to(G.DEV)
    fs = torch.from_numpy(rng.standard_normal((B, case.H, case.W, 32), dtype=np.float32)).half().to(G.DEV)
    return SimpleNamespace(fr=fr, fs=fs, Mw=torch.from_numpy(case.Mw).to(G.DEV), depths=torch.from_numpy(case.depths).to(G.DEV))


def run(G, case, t, dt, *, extra_env=0, depths=None, Mw=None, fs=None):
    """One launch into a canary-filled [B + extra_env, D, H, W, 32] buffer of dtype dt; returns it (device)."""
    B = len(case.Mw)
    dep = t.depths if depths is None else depths
    out = canary16((B + extra_env, dep.numel(), case.H, case.W, 32), dt)
    G.volume(t.fr, t.fs if fs is None else fs, t.Mw if Mw is None else Mw, dep, out, batch=B)
    return out


_ENGINE = {}


def engine(G):
    """The engine case with the device's warp matrices, its inputs and fp16 run (cached)."""
    if "e" not in _ENGINE:
        cams = engine_cameras()
        Mw = warp_run(G, *cams, valid_env=False)[0].astype(np.float32)
        assert np.abs(Mw - warp_ref(*cams)[0]).max() < 1e-3              # three distinct real geometries, not aliased inputs
        case = engine_case(Mw)
        t = dev_case(G, case)
        _ENGINE["e"] = SimpleNamespace(case=case, t=t, f16=run(G, case, t, F16))
    return _ENGINE["e"]


def _report(what, worst, n_excl, n_nothing, cnt=None):
    print(f"volume {what}: largest error / bound {worst:.3f}, {n_nothing} voxels sample nothing, {n_excl} excluded"
          + (f"; census {cnt}" if cnt else ""))


@GPU
@pytest.mark.parametrize("dt", [F16, BF16], ids=["f16", "bf16"])
def test_volume_engine_geometry(G, dt):
    """B = 3 different real stereo geometries (adp_warp_matrices on synth scenes), the 24 depth hypotheses, S = 224: every
    voxel, fp16 and bf16 output."""
    e = engine(G)
    vol = e.f16 if dt == F16 else run(G, e.case, e.t, dt)
    codes, extra = census(e.case, f16=dt == F16)
    cnt = assert_census(e.case, codes, extra)
    worst, n_excl, n_nothing = check_volume(e.case, (e.t.fr, e.t.fs), vol, f"engine {dt}", G.DEV)
    _report(f"engine {dt}", worst, n_excl, n_nothing, cnt)


@GPU
@pytest.mark.parametrize("D", [1, 5, 13], ids=lambda d: f"D{d}")
@pytest.mark.parametrize("hw", RAGGED, ids=lambda s: f"{s[0]}x{s[1]}")
def test_volume_ragged(G, hw, D):
    """Partial tiles in x and y and partial depth groups, a different Mw per environment, and one extra environment allocated
    in a canary-filled output: every voxel of [B, D, H, W, 32] is written and checked, the extra environment keeps its bits."""
    case = ragged_case(*hw, D)
    t = dev_case(G, case)
    vol = run(G, case, t, F16, extra_env=1)
    assert (bits(vol[2]) == CANARY16).all()
    worst, n_excl, n_nothing = check_volume(case, (t.fr, t.fs), vol[:2], case.name, G.DEV)
    _report(case.name, worst, n_excl, n_nothing, census_counts(census(case)[0]))


@GPU
@pytest.mark.parametrize("dt", [F16, BF16], ids=["f16", "bf16"])
@pytest.mark.parametrize("name", ["footprint", "borders", "pole"])
def test_volume_regimes(G, name, dt):
    """The footprint regimes (staged and direct-gather tiles in one launch, staged and empty tiles in one plane) and the edges
    of the empty shortcut: corner images 0.005-0.02 px either side of its 0.01 px margin on all four borders, a tile with all
    corners outside but not on one side, tiles with Z <= 0 at some or all corners and Z crossing 0 inside a tile.  Every voxel;
    the bf16 output never takes the shortcut and must give bf16(feat_ref) wherever nothing is sampled."""
    case = _cpu_case(name)
    codes, extra = census(case, f16=dt == F16)
    cnt = assert_census(case, codes, extra) if dt == F16 else census_counts(codes)
    t = dev_case(G, case)
    vol = run(G, case, t, dt)
    worst, n_excl, n_nothing = check_volume(case, (t.fr, t.fs), vol, f"{name} {dt}", G.DEV)
    _report(f"{name} {dt}", worst, n_excl, n_nothing, cnt)


@GPU
def test_volume_depth_subrange_is_bit_identical(G):
    """depths[3:19] as a launch of its own: its planes fall into other blocks and parities (other box and staging decisions)
    and must equal planes 3..18 of the full launch bit for bit."""
    e = engine(G)
    sub = run(G, e.case, e.t, F16, depths=e.t.depths[3:19].contiguous())
    assert torch.equal(bits(sub), bits(e.f16[:, 3:19]))


@GPU
def test_volume_env_alone_is_bit_identical(G):
    """Each environment launched alone equals the same environment of the batch bit for bit."""
    e = engine(G)
    for b in range(len(e.case.Mw)):
        one = SimpleNamespace(fr=e.t.fr[b:b + 1], fs=e.t.fs[b:b + 1], Mw=e.t.Mw[b:b + 1], depths=e.t.depths)
        out = canary16((1, 24, 224, 224, 32), F16)
        G.volume(one.fr, one.fs, one.Mw, one.depths, out)
        assert torch.equal(bits(out[0]), bits(e.f16[b])), b


# ================================================================================================ adp_warp_matrices
def _rot(axis, deg):
    c, s = math.cos(math.radians(deg)), math.sin(math.radians(deg))
    i, j = [(1, 2), (2, 0), (0, 1)][axis]
    R = np.eye(3)
    R[i, i], R[i, j], R[j, i], R[j, j] = c, -s, s, c
    return R


def random_cameras(B, rng):
    """B random intrinsics (224-pixel crops) and extrinsics (rotations about all axes, translations of ~1 m)."""
    K = np.tile(np.eye(3), (B, 1, 1))
    K[:, 0, 0], K[:, 1, 1] = rng.uniform(150, 400, B), rng.uniform(150, 400, B)
    K[:, 0, 2], K[:, 1, 2] = rng.uniform(60, 160, B), rng.uniform(60, 160, B)
    E = np.tile(np.eye(4), (B, 1, 1))
    for b in range(B):
        E[b, :3, :3] = _rot(0, rng.uniform(-180, 180)) @ _rot(1, rng.uniform(-90, 90)) @ _rot(2, rng.uniform(-180, 180))
    E[:, :3, 3] = rng.uniform(-1, 1, (B, 3)) + np.array([0, 0, 1.5])
    return K, E


def warp_run(G, Kr, Er, Ks, Es, valid_ref=None, valid_src=None, valid_env=True):
    from rgbmanip_b200 import _lib as L
    B = len(Kr)
    # every device buffer stays referenced until the kernel has run: L.ptr holds no reference, and a freed block is handed to
    # the next allocation of the same size (four temporaries in one call would alias)
    cam = [torch.from_numpy(np.ascontiguousarray(a).reshape(B, -1)).to(G.DEV) for a in (Kr, Er, Ks, Es)]
    Mw = torch.full((B, 12), float("nan"), device=G.DEV)
    venv = torch.full((B,), 0xAA, dtype=torch.uint8, device=G.DEV) if valid_env else None
    vr = torch.tensor(valid_ref, dtype=torch.uint8, device=G.DEV) if valid_ref is not None else None
    vs = torch.tensor(valid_src, dtype=torch.uint8, device=G.DEV) if valid_src is not None else None
    L.check(L.load().adp_warp_matrices(*(L.ptr(t) for t in cam), L.ptr(Mw), L.ptr(vr), L.ptr(vs), L.ptr(venv), B, G.stream()),
            "warp matrices")
    torch.cuda.synchronize()
    return Mw.cpu().double().numpy(), (venv.cpu().numpy() if venv is not None else None)


def warp_check(got, Kr, Er, Ks, Es):
    want, M = warp_ref(Kr, Er, Ks, Es)
    row = np.abs(M).max(2)                                                  # [B, 3]
    rowmag = np.concatenate([np.repeat(row, 3, 1), row], 1)                 # rot entries of row r, then trans of row r
    bound = 2.0 ** -24 * np.abs(want) + 1e-12 * rowmag
    err = np.abs(got - want)
    assert (err <= bound).all(), (np.argwhere(~(err <= bound))[:4], got[~(err <= bound)][:4], want[~(err <= bound)][:4])
    return float((err / bound).max())


@GPU
def test_warp_matrices_three_blocks_and_pivoting(G):
    """B = 130 (three 64-thread blocks) random camera pairs, the engine's synth cameras, and env 0 with a 90-degree rotation
    about z in E_ref: P_ref's diagonal starts with an exact zero, so Gauss-Jordan must pivot."""
    rng = _rng("warp")
    Kr, Er = random_cameras(130, rng)
    Ks, Es = random_cameras(130, rng)
    Er[0, :3, :3] = [[0.0, -1.0, 0.0], [1.0, 0.0, 0.0], [0.0, 0.0, 1.0]]     # exact: cos(90 deg) in float64 is 6e-17, not 0
    Er[0, :3, 3] = [0.1, -0.2, 1.0]
    Kr[0, 0, 2] = Kr[0, 1, 2] = 0.0                      # K' R = [[0, -f, 0], [f, 0, 0], [0, 0, 1]]: a[0][0] = a[1][1] = 0
    ec = engine_cameras()
    Kr[1:4], Er[1:4], Ks[1:4], Es[1:4] = ec
    P0 = Kr[0] @ Er[0, :3, :]
    assert P0[0, 0] == 0.0 and P0[1, 1] == 0.0
    got, venv = warp_run(G, Kr, Er, Ks, Es)
    assert (venv == 1).all()
    worst = warp_check(got, Kr, Er, Ks, Es)
    print(f"warp matrices B 130: largest error / bound {worst:.3f}")


@GPU
def test_warp_matrices_valid_env(G):
    """valid_env = valid_ref && valid_src over all four combinations, with either pointer NULL meaning all valid; valid_env
    NULL writes nothing and still computes Mw."""
    rng = _rng("warp_valid")
    Kr, Er = random_cameras(8, rng)
    Ks, Es = random_cameras(8, rng)
    vr, vs = [0, 0, 1, 1, 0, 1, 1, 0], [0, 1, 0, 1, 1, 1, 0, 0]
    want = np.array(vr, np.uint8) & np.array(vs, np.uint8)
    for r, s, w in ((vr, vs, want), (None, vs, np.array(vs, np.uint8)), (vr, None, np.array(vr, np.uint8)),
                    (None, None, np.ones(8, np.uint8))):
        got, venv = warp_run(G, Kr, Er, Ks, Es, r, s)
        assert np.array_equal(venv, w), (r, s, venv)
        warp_check(got, Kr, Er, Ks, Es)
    got, venv = warp_run(G, Kr, Er, Ks, Es, vr, vs, valid_env=False)
    assert venv is None
    warp_check(got, Kr, Er, Ks, Es)
