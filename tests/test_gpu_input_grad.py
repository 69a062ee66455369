"""Gradients with respect to the input clip (run with -m gpu on the B200 box): the stem's data gradient at op level on
both paths (tcgen05 svit_patch_embed_s2d_dgrad + svit_d2s_clip; svit_gemm + svit_col2im3d), clip.grad of whole models
against the CPU oracle, frozen models (saliency), frame mode, and that a clip which does not require grad changes
nothing."""
import pytest
import torch
import torch.nn.functional as F

import svit_b200
from oracle import svit_oracle as O
from svit_b200 import _lib, ops
from svit_b200.config import block_specs, ssv2_cfg, state_shapes, tiny_cfg
from tests.conftest import max_rel_err
from tests.golden.recipe import synth_input, synth_state

pytestmark = pytest.mark.gpu
DEV = "cuda"
KERNEL, STRIDE, PAD = (3, 7, 7), (2, 4, 4), (1, 3, 3)
GEOMS = [(2, 16, 224, 224), (3, 4, 32, 32), (5, 1, 224, 224), (1, 8, 312, 312), (2, 3, 30, 50)]
INPUT_GRAD_CALLS = ("svit_patch_embed_s2d_dgrad", "svit_d2s_clip", "svit_col2im3d")


@pytest.fixture(autouse=True, scope="module")
def _need_cuda():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    assert _lib.lib().svit_abi_version() == 100
    yield
    ops.set_impl(gemm=ops.IMPL_AUTO, attn=ops.IMPL_AUTO)
    torch.cuda.synchronize()


def _seq_grad(dy, O_tot, dtype, seed):
    """dx [B, 1 + L + O_tot, E] whose patch rows are dy [B, E, To, Ho, Wo]; cls / object rows hold other values."""
    B, E = dy.shape[:2]
    g = torch.Generator().manual_seed(seed)
    dx = torch.randn(B, 1 + dy[0, 0].numel() + O_tot, E, generator=g)
    dx[:, 1:1 + dy[0, 0].numel()] = dy.flatten(2).transpose(1, 2).float()
    return dx.to(DEV, dtype)


def _reference(dy, w, clip_shape):
    """fp64 torch.autograd.grad of conv3d (on the GPU, for speed)."""
    clip = torch.zeros(clip_shape, dtype=torch.float64, device=DEV, requires_grad=True)
    y = F.conv3d(clip, w.to(DEV, torch.float64), None, STRIDE, PAD)
    assert y.shape == dy.shape
    return torch.autograd.grad(y, clip, dy.to(DEV, torch.float64))[0]


def _case(geom):
    B, T, H, W = geom
    g = torch.Generator().manual_seed(sum(geom))
    w = torch.randn(96, 3, *KERNEL, generator=g) * 0.05
    To, Ho, Wo = ((n + 2 * p - k) // s + 1 for n, k, s, p in zip((T, H, W), KERNEL, STRIDE, PAD))
    dy = torch.randn(B, 96, To, Ho, Wo, generator=g)
    return w, dy, (B, 3, T, H, W)


@pytest.mark.parametrize("geom", GEOMS, ids=lambda g: "x".join(map(str, g)))
def test_col2im_path_fp32(geom):
    w, dy, shape = _case(geom)
    ops.set_impl(gemm=ops.IMPL_SIMT)
    dx = _seq_grad(dy, 4 * shape[2], torch.float32, 1)
    got = ops.input_grad_col2im(dx, w.to(DEV), shape, torch.float32, KERNEL, STRIDE, PAD)
    ops.set_impl(gemm=ops.IMPL_AUTO)
    assert got.shape == shape and got.dtype == torch.float32
    assert max_rel_err(got, _reference(dy, w, shape)) <= 1e-5


@pytest.mark.parametrize("geom", GEOMS, ids=lambda g: "x".join(map(str, g)))
def test_tcgen05_path_bf16(geom):
    w, dy, shape = _case(geom)
    assert _lib.lib().svit_patch_embed_s2d_dgrad_supported(3, *KERNEL, *STRIDE, *PAD, 96)
    dx = _seq_grad(dy, 4 * shape[2], torch.bfloat16, 2)
    wd = w.to(DEV)
    got = ops.input_grad_s2d(dx, wd, shape, torch.float32, KERNEL, STRIDE, PAD)
    # the reference sees the same bf16-rounded gradient rows and weights
    ref = _reference(dy.bfloat16().double(), w.bfloat16().double(), shape)
    assert got.shape == shape and got.dtype == torch.float32
    assert (got.double() - ref).abs().max().item() <= 8e-3 * ref.abs().max().item()
    # a bf16 clip gets the same cell values (d2s moves bf16 values, it does not round again)
    got16 = ops.input_grad_s2d(dx, wd, shape, torch.bfloat16, KERNEL, STRIDE, PAD)
    assert got16.dtype == torch.bfloat16 and torch.equal(got16, got.bfloat16())
    # the dispatcher takes this path for bf16
    assert torch.equal(ops.patch_embed_input_grad(dx, wd, shape, torch.float32, KERNEL, STRIDE, PAD), got)


@pytest.mark.parametrize("geom", GEOMS, ids=lambda g: "x".join(map(str, g)))
def test_d2s_is_the_inverse_of_s2d(geom):
    B, T, H, W = geom
    st, sh, sw = STRIDE
    cells = synth_input(f"d2s{geom}", (B, -(-T // st), -(-H // sh), -(-W // sw), 3 * st * sh * sw), 3).to(DEV, torch.bfloat16)
    full = cells.reshape(*cells.shape[:4], 3, st, sh, sw).permute(0, 4, 1, 5, 2, 6, 3, 7)
    want = full.reshape(B, 3, cells.shape[1] * st, cells.shape[2] * sh, cells.shape[3] * sw)[:, :, :T, :H, :W]
    for dtype in (torch.float32, torch.bfloat16):
        got = ops.d2s_clip(cells, (B, 3, T, H, W), STRIDE, dtype)
        assert torch.equal(got, want.to(dtype))
    # and s2d_clip of that clip gives back the cells inside the clip (zero beyond it)
    back = ops.s2d_clip(want.contiguous(), STRIDE)
    mask = ops.s2d_clip(torch.ones(B, 3, T, H, W, device=DEV, dtype=torch.bfloat16), STRIDE)
    assert torch.equal(back, cells * mask)


# ------------------------------------------------------------------------------------------------ model level
def _tiny(dtype, golden):
    """The tiny SViT with the state of the reference gradients in tests/golden/svit_tiny.pt, in eval mode."""
    cfg = tiny_cfg()
    g = golden("svit_tiny.pt")["video"]
    params = synth_state(state_shapes(cfg), g["seed"], w_std=g["w_std"])
    m = svit_b200.SViT(cfg, compute_dtype=dtype)
    m.load_state_dict(params)
    return cfg, params, m.to(DEV).eval()


def _loss(extra):
    # the objective of the training-gradient parity tests: cross entropy + small box / contact terms
    logits = extra["logits"].float()
    tgt = torch.arange(logits.shape[0], device=logits.device) % logits.shape[1]
    return F.cross_entropy(logits, tgt) + 0.1 * extra["pred_bboxes"].float().square().mean() \
        + 0.1 * extra["pred_contact_state"].float().square().mean()


def _oracle_clip_grad(clip, params, cfg, device="cpu"):
    p = {k: v.to(device) for k, v in params.items()}
    x = clip.to(device).clone().requires_grad_(True)
    _loss(O.svit_forward(x, p, block_specs(cfg)[0], cfg)[1]).backward()
    return x.grad.cpu()


def _clip_grad(m, clip):
    x = clip.to(DEV).clone().requires_grad_(True)
    _loss(m([x])[1]).backward()
    return x.grad


def _stem_check(monkeypatch, m):
    """Records the sequence gradient that reaches the stem; check(g) then asserts that clip.grad is the transposed
    convolution of exactly that gradient (fp64 reference on the same bf16-rounded values, the op-level bound)."""
    seen = []
    orig = ops.patch_embed_input_grad

    def spy(dx, *args):
        seen.append(dx.detach().clone())
        return orig(dx, *args)

    monkeypatch.setattr(ops, "patch_embed_input_grad", spy)

    def check(g):
        dx = seen.pop()
        shape = g.shape if g.dim() == 5 else (g.shape[0], g.shape[1], 1, *g.shape[2:])
        w = m.patch_embed.proj.weight.detach()
        To, Ho, Wo = ((n + 2 * p - k) // s + 1 for n, k, s, p in zip(shape[2:], KERNEL, STRIDE, PAD))
        dy = dx[:, 1:1 + To * Ho * Wo].transpose(1, 2).reshape(shape[0], -1, To, Ho, Wo)
        ref = _reference(dy.double(), w.bfloat16().double(), shape)
        assert (g.reshape(shape).double() - ref).abs().max().item() <= 8e-3 * ref.abs().max().item()

    return check


def _norm_err(g, ref):
    g, ref = g.double().cpu(), ref.double().cpu()
    return ((g - ref).norm() / ref.norm()).item()


def test_tiny_fp32_clip_grad_matches_oracle(golden):
    ops.set_impl(gemm=ops.IMPL_SIMT, attn=ops.IMPL_SIMT)
    cfg, params, m = _tiny(torch.float32, golden)
    for clip in (synth_input("tiny.clip", (2, 3, 4, 32, 32), 5), synth_input("tiny.frames", (3, 3, 32, 32), 5)):
        g = _clip_grad(m, clip)
        assert g.shape == clip.shape and g.dtype == torch.float32  # frame mode [B, 3, H, W] too
        assert max_rel_err(g.cpu(), _oracle_clip_grad(clip, params, cfg)) <= 2e-3
    ops.set_impl(gemm=ops.IMPL_AUTO, attn=ops.IMPL_AUTO)


# Against the fp32 oracle the bf16 clip gradient carries the error of the whole bf16 backward above the stem (measured on
# B200: ||g - g_ref|| / ||g_ref|| 3.0e-2 to 3.4e-2 for the tiny model, video and frame mode, unfrozen and frozen; 8.2e-2 at
# the ssv2 geometry, cosine 0.9966 there).  What the stem itself adds is bounded separately and tightly by _stem_check.
BF16_TINY_TOL, BF16_FULL_TOL = 5e-2, 1e-1


def test_tiny_bf16_clip_grad_and_frozen_model(golden, monkeypatch):
    cfg, params, m = _tiny(torch.bfloat16, golden)
    stem = _stem_check(monkeypatch, m)
    for clip in (synth_input("tiny.clip", (2, 3, 4, 32, 32), 5), synth_input("tiny.frames", (3, 3, 32, 32), 5)):
        ref = _oracle_clip_grad(clip, params, cfg)
        m.zero_grad(set_to_none=True)
        g = _clip_grad(m, clip)
        assert g.shape == clip.shape
        stem(g)
        print(f"bf16 clip.grad {tuple(clip.shape)}: ||g - g_ref|| / ||g_ref|| = {_norm_err(g, ref):.2e}")
        assert _norm_err(g, ref) <= BF16_TINY_TOL
        # frozen: no parameter requires grad, the clip does (saliency / attribution)
        m.zero_grad(set_to_none=True)
        for p in m.parameters():
            p.requires_grad_(False)
        ops.profile_start()
        gf = _clip_grad(m, clip)
        names = set(ops.profile_stop()["detail"])
        for p in m.parameters():
            p.requires_grad_(True)
        assert all(p.grad is None for p in m.parameters())
        assert any(n.startswith("svit_patch_embed_s2d[") for n in names)  # implicit-GEMM forward
        assert not any(n.startswith("svit_im2col3d") for n in names)  # no im2col matrix
        assert any(n.startswith("svit_patch_embed_s2d_dgrad") for n in names)
        assert gf.shape == clip.shape
        stem(gf)
        assert _norm_err(gf, g) <= 3e-2
        assert _norm_err(gf, ref) <= BF16_TINY_TOL


def test_frozen_fp32_model_clip_grad(golden):
    # the fp32 parity mode has no implicit-GEMM forward: im2col + GEMM forward, col2im data gradient, no weight gradients
    ops.set_impl(gemm=ops.IMPL_SIMT, attn=ops.IMPL_SIMT)
    cfg, params, m = _tiny(torch.float32, golden)
    m.requires_grad_(False)
    clip = synth_input("tiny.clip", (2, 3, 4, 32, 32), 5)
    g = _clip_grad(m, clip)
    assert all(p.grad is None for p in m.parameters())
    assert max_rel_err(g.cpu(), _oracle_clip_grad(clip, params, cfg)) <= 2e-3
    ops.set_impl(gemm=ops.IMPL_AUTO, attn=ops.IMPL_AUTO)


def test_full_ssv2_bf16_clip_grad(golden, monkeypatch):
    cfg = ssv2_cfg()
    gf = golden("svit_full.pt")
    params = synth_state(state_shapes(cfg), gf["seed"], w_std=gf["w_std"])
    m = svit_b200.SViT(cfg, compute_dtype=torch.bfloat16)
    m.load_state_dict(params)
    m = m.to(DEV).eval()
    clip = synth_input("full.clip", (1, 3, 16, 224, 224), 6)
    stem = _stem_check(monkeypatch, m)
    g = _clip_grad(m, clip)
    stem(g)
    tf32 = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    try:
        ref = _oracle_clip_grad(clip, params, cfg, device=DEV)  # fp32 reference on the GPU (full geometry)
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = tf32
    cos = F.cosine_similarity(g.double().flatten().cpu(), ref.double().flatten(), dim=0).item()
    print(f"ssv2 bf16 clip.grad: ||g - g_ref|| / ||g_ref|| = {_norm_err(g, ref):.2e}, cosine {cos:.5f}")
    assert _norm_err(g, ref) <= BF16_FULL_TOL
    assert cos > 0.99


# ------------------------------------------------------------------------------------------------ nothing else changes
def test_clip_without_grad_runs_no_input_gradient_kernel(golden):
    cfg, params, m = _tiny(torch.bfloat16, golden)
    m.train()
    for mod in m.modules():
        if isinstance(mod, svit_b200.DropPath):
            mod.drop_prob = 0.0
    clip = synth_input("tiny.clip", (2, 3, 4, 32, 32), 5).to(DEV)
    counts = []
    for needs in (False, True):
        x = clip.clone().requires_grad_(needs)
        ops.profile_start()
        n0 = ops.launches()
        m([x])[0].float().square().sum().backward()
        counts.append(ops.launches() - n0)
        names = set(ops.profile_stop()["detail"])
        used = {c for c in INPUT_GRAD_CALLS if any(n.startswith(c) for n in names)}
        assert used == (set() if not needs else {"svit_patch_embed_s2d_dgrad", "svit_d2s_clip"})
        m.zero_grad(set_to_none=True)
    assert counts[1] == counts[0] + 2  # a training step with clip gradients adds exactly the two launches
