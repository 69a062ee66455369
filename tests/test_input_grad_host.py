"""The math of the stem's data gradient (svit_patch_embed_s2d_dgrad + svit_d2s_clip), checked on the CPU in fp64 before
any kernel runs: the transposed weight of ops.s2d_dgrad_weight applied as a stride-1 convolution over the output grid
into the cell grid, then depth-to-space and the crop to T / H / W, against torch.autograd.grad of F.conv3d."""
import pytest
import torch
import torch.nn.functional as F

from svit_b200.ops import s2d_conv_weight, s2d_dgrad_weight

KERNEL, STRIDE, PAD = (3, 7, 7), (2, 4, 4), (1, 3, 3)  # configs/ssv2.yaml PatchEmbed
GEOMS = [(2, 16, 224, 224), (3, 4, 32, 32), (5, 1, 224, 224), (1, 8, 312, 312), (2, 3, 30, 50)]


def _taps(k, s, p):
    lo = (-p) // s
    return lo, (k - 1 - p) // s - lo + 1


def _shift(x, dim, off, n_out):
    """y[c] = x[c + off] along `dim` for c < n_out, zero where c + off falls outside x."""
    shape = list(x.shape)
    shape[dim] = n_out
    y = x.new_zeros(shape)
    c0, c1 = max(0, -off), min(n_out, x.shape[dim] - off)
    if c1 > c0:
        y.narrow(dim, c0, c1 - c0).copy_(x.narrow(dim, c0 + off, c1 - c0))
    return y


def dclip_via_cells(dy, w, clip_shape):
    """dy [B, E, To, Ho, Wo] -> dclip [B, C, T, H, W]: what the dgrad kernel and svit_d2s_clip compute, in fp64."""
    B, C, T, H, W = clip_shape
    E = w.shape[0]
    st, sh, sw = STRIDE
    (lo_t, nt), (lo_h, nh), (lo_w, nw) = (_taps(k, s, p) for k, s, p in zip(KERNEL, STRIDE, PAD))
    lt, lh, lw = -lo_t - nt + 1, -lo_h - nh + 1, -lo_w - nw + 1
    Tc, Hc, Wc = -(-T // st), -(-H // sh), -(-W // sw)
    cell = C * st * sh * sw
    wt = s2d_dgrad_weight(w, STRIDE, PAD, torch.float64).reshape(cell, nt, nh, nw, E)
    rows = dy.permute(0, 2, 3, 4, 1)  # [B, To, Ho, Wo, E]
    dcells = torch.zeros(B, Tc, Hc, Wc, cell, dtype=torch.float64)
    for it in range(nt):
        a = _shift(rows, 1, lt + it, Tc)
        for ih in range(nh):
            b = _shift(a, 2, lh + ih, Hc)
            for iw in range(nw):
                dcells += _shift(b, 3, lw + iw, Wc) @ wt[:, it, ih, iw, :].T
    full = dcells.reshape(B, Tc, Hc, Wc, C, st, sh, sw).permute(0, 4, 1, 5, 2, 6, 3, 7)
    return full.reshape(B, C, Tc * st, Hc * sh, Wc * sw)[:, :, :T, :H, :W]


def test_tap_geometry_of_ssv2_stem():
    # lo = -1 and two taps per dimension, so the transposed convolution starts at lo' = 0
    for k, s, p in zip(KERNEL, STRIDE, PAD):
        lo, n = _taps(k, s, p)
        assert (lo, n, -lo - n + 1) == (-1, 2, 0)


def test_dgrad_weight_is_the_forward_weight_transposed_with_taps_reversed():
    g = torch.Generator().manual_seed(1)
    w = torch.randn(96, 3, *KERNEL, generator=g)
    fwd = s2d_conv_weight(w, STRIDE, PAD).reshape(96, 2, 2, 2, 96)
    bwd = s2d_dgrad_weight(w, STRIDE, PAD).reshape(96, 2, 2, 2, 96)
    assert bwd.dtype == torch.bfloat16
    assert torch.equal(bwd, fwd.flip(1, 2, 3).permute(4, 1, 2, 3, 0))


@pytest.mark.parametrize("geom", GEOMS, ids=lambda g: "x".join(map(str, g)))
def test_dclip_matches_conv3d_autograd_fp64(geom):
    B, T, H, W = geom
    if H >= 224:
        B = 1  # a one-sample slice keeps the fp64 reference conv3d fast on the CPU
    g = torch.Generator().manual_seed(sum(geom))
    w = torch.randn(96, 3, *KERNEL, generator=g, dtype=torch.float64) * 0.05
    clip = torch.randn(B, 3, T, H, W, generator=g, dtype=torch.float64, requires_grad=True)
    y = F.conv3d(clip, w, None, STRIDE, PAD)
    dy = torch.randn(y.shape, generator=g, dtype=torch.float64)
    (ref,) = torch.autograd.grad(y, clip, dy)
    got = dclip_via_cells(dy, w, clip.shape)
    assert got.shape == ref.shape
    assert (got - ref).abs().max().item() <= 1e-10 * ref.abs().max().item()
