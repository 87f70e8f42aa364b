"""Host-side tap tables / weight repacks (rgbmanip_b200/geometry.py) against torch convolutions, on CPU."""
import torch
import torch.nn.functional as F

from rgbmanip_b200 import geometry as G


def _run_taps(x_cl, wt, g):
    """Stride-1 multi-tap convolution with zero out-of-range reads, as the tcgen05 kernel evaluates a tap table."""
    B, D, H, W, _ = x_cl.shape
    out = torch.zeros(B, D, H, W, wt.shape[1], dtype=x_cl.dtype)
    xp = F.pad(x_cl, (0, 0, 2, 2, 2, 2, 2, 2))
    for i in range(g.ntaps):
        dz, dy, dx, t = g.dz[i], g.dy[i], g.dx[i], g.wt[i]
        out += xp[:, 2 + dz:2 + dz + D, 2 + dy:2 + dy + H, 2 + dx:2 + dx + W] @ wt[t].t()
    return out


def test_s2d_roundtrip():
    x = torch.randn(2, 4, 6, 8, 3)
    assert torch.equal(G.from_s2d(G.to_s2d(x)), x)
    assert G.to_s2d(x).shape == (2, 2, 3, 4, 24)


def test_stride2_conv_over_s2d_input():
    """network_v5.py:265 (conv1): Conv3d k3 s2 p1 == 2x2x2 stride-1 window over the space-to-depth(2) input."""
    torch.manual_seed(0)
    x = torch.randn(2, 8, 6, 8, 10, dtype=torch.float64)
    w = torch.randn(16, 8, 3, 3, 3, dtype=torch.float64)
    ref = F.conv3d(x, w, stride=2, padding=1)
    got = _run_taps(G.to_s2d(x.permute(0, 2, 3, 4, 1).contiguous()), G.strided_s2d_weights(w).double(), G.strided_s2d(3, 4, 5))
    assert float((got.permute(0, 4, 1, 2, 3) - ref).abs().max()) < 1e-5    # weights pass through fp32


def test_transposed_conv_to_s2d_output():
    """network_v5.py:278 (conv11): ConvTranspose3d k3 s2 p1 op1 == 2x2x2 stride-1 window producing 8 parities x Cout."""
    torch.manual_seed(1)
    x = torch.randn(2, 16, 3, 4, 5, dtype=torch.float64)
    w = torch.randn(16, 8, 3, 3, 3, dtype=torch.float64)
    ref = F.conv_transpose3d(x, w, stride=2, padding=1, output_padding=1)
    got = _run_taps(x.permute(0, 2, 3, 4, 1).contiguous(), G.transposed_s2d_weights(w).double(), G.transposed_s2d(3, 4, 5))
    assert float((G.from_s2d(got).permute(0, 4, 1, 2, 3) - ref).abs().max()) < 1e-5


def test_stem_s2d_weights_match_7x7_stride2():
    """pspnet.py:37: the 7x7/2 pad-3 stem == 4x4 stride-1 window over the s2d(2) image (adp_pack_s2d layout)."""
    torch.manual_seed(2)
    img = torch.randn(1, 3, 16, 16, dtype=torch.float64)
    w = torch.randn(64, 3, 7, 7, dtype=torch.float64)
    ref = F.conv2d(img, w, stride=2, padding=3)
    cl = img.permute(0, 2, 3, 1)
    s2d = torch.zeros(1, 1, 8, 8, 16, dtype=torch.float64)
    for py in range(2):
        for px in range(2):
            s2d[0, 0, :, :, (py * 2 + px) * 3:(py * 2 + px) * 3 + 3] = cl[0, py::2, px::2]
    got = _run_taps(s2d, G.stem_s2d_weights(w).double(), G.stem_s2d(16))
    assert float((got[0, 0].permute(2, 0, 1) - ref[0]).abs().max()) < 1e-5


def test_conv0_ring_weights_layout():
    """adp_conv0_run reads w[co, c, kz, ky, kx] at [kx][c // 8][(kz * 3 + ky) * 8 + co][c % 8]; rows 72..79 of N are zero."""
    w = torch.randn(8, 32, 3, 3, 3)
    p = G.conv0_ring_weights(w)
    assert p.shape == (3, 4, 80, 8)
    for co in range(8):
        for c in range(32):
            for kz in range(3):
                for ky in range(3):
                    for kx in range(3):
                        assert p[kx, c // 8, (kz * 3 + ky) * 8 + co, c % 8] == w[co, c, kz, ky, kx]
    assert (p[:, :, 72:] == 0).all()
