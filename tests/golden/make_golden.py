"""Generates tests/golden/*.pt by EXECUTING THE UNMODIFIED REFERENCE (build container only).

    python tests/golden/make_golden.py

Imports /root/reference through oracle/ref_loader.py (package-shell shim, SURVEY.md 8c),
runs the reference functions / modules on seeded synthetic inputs and stores inputs and
outputs.  The fixtures pin oracle/svit_oracle.py (tests/test_oracle_golden.py) and are the
ground truth of the GPU parity tests.  Weights come from tests/golden/recipe.py and are
regenerated, not stored, when they are large.
"""
import importlib.util
import os
import sys

import numpy as np
import torch
import torch.nn as nn

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from oracle import ref_loader  # noqa: E402
from svit_b200.config import ssv2_cfg, tiny_cfg  # noqa: E402
from tests.golden.recipe import synth_input, synth_state  # noqa: E402

torch.set_num_threads(8)
ns = ref_loader.load()
A = ns.attention
LN = lambda d: nn.LayerNorm(d, eps=1e-6)


def save(name, obj):
    path = os.path.join(HERE, name)
    torch.save(obj, path)
    print(f"{name}: {os.path.getsize(path) / 1024:.0f} KiB")


def load_state(mod, seed, **kw):
    sd = synth_state({k: v.shape for k, v in mod.state_dict().items()}, seed, **kw)
    mod.load_state_dict(sd)
    return sd


# ---------------------------------------------------------------- A4 index tables
def relpos_tables():
    pairs = [(56, 7), (28, 7), (28, 14), (14, 14), (14, 7), (7, 14), (7, 7), (8, 8), (8, 2), (4, 2),
             (4, 4), (2, 4), (1, 1), (78, 10), (39, 10), (39, 20), (20, 20), (20, 10), (10, 20), (10, 10),
             (16, 16), (5, 3), (3, 5), (13, 4), (9, 9)]
    out = {}
    for q, k in pairs:
        d = 2 * max(q, k) - 1
        # rows of the table are constant = row index / 96 so that q(=ones) . R[r] = r
        rel = (torch.arange(d, dtype=torch.float64)[:, None] / 96.0).expand(d, 96).contiguous()
        zero = torch.zeros_like(rel)
        attn = torch.zeros(1, 1, 1 + q * q + 1, 1 + k * k + 1, dtype=torch.float64)
        qq = torch.ones(1, 1, 1 + q * q + 1, 96, dtype=torch.float64)
        attn = A.cal_rel_pos_spatial(attn, qq, None, True, [1, q, q], [1, k, k], rel, zero)
        tab = attn[0, 0, 1:1 + q * q, 1:1 + k * k].reshape(q, q, k, k)[:, 0, :, 0]
        out[f"{q}_{k}"] = tab.round().long()
        # temporal variant goes through a different code path (attention.py:156-163)
        rel_t = rel
        attn = torch.zeros(1, 1, 1 + q + 1, 1 + k + 1, dtype=torch.float64)
        qq = torch.ones(1, 1, 1 + q + 1, 96, dtype=torch.float64)
        attn = A.cal_rel_pos_temporal(attn, qq, True, [q, 1, 1], [k, 1, 1], rel_t)
        tt = attn[0, 0, 1:1 + q, 1:1 + k].round().long()
        assert torch.equal(tt, out[f"{q}_{k}"]), (q, k)
    save("relpos_index.pt", out)


# ---------------------------------------------------------------- A1 attention_pool
def pool_cases():
    cases = []
    specs = [  # B, h, T, H, W, O, stride
        (2, 2, 2, 8, 8, 8, (1, 1, 1)), (1, 2, 2, 8, 8, 8, (1, 2, 2)), (2, 1, 2, 8, 8, 8, (1, 4, 4)),
        (1, 1, 2, 8, 8, 8, (1, 8, 8)), (1, 2, 3, 7, 7, 12, (1, 2, 2)), (1, 1, 1, 9, 9, 4, (1, 1, 1)),
        (1, 1, 2, 10, 10, 5, (1, 4, 4)), (1, 3, 4, 5, 6, 3, (1, 2, 2)),
    ]
    for i, (B, h, T, H, W, O, st) in enumerate(specs):
        conv = nn.Conv3d(96, 96, (3, 3, 3), stride=st, padding=(1, 1, 1), groups=96, bias=False)
        norm = LN(96)
        w = synth_input(f"pool{i}.w", conv.weight.shape, 1, 0.25)
        g = 1 + synth_input(f"pool{i}.g", (96,), 1, 0.2)
        b = synth_input(f"pool{i}.b", (96,), 1, 0.2)
        conv.weight.data.copy_(w); norm.weight.data.copy_(g); norm.bias.data.copy_(b)
        z = synth_input(f"pool{i}.z", (B, h, 1 + T * H * W + O, 96), 1).requires_grad_(True)
        out, thw = A.attention_pool(z, conv, [T, H, W], has_cls_embed=True, norm=norm)
        gy = synth_input(f"pool{i}.gy", out.shape, 1)
        out.backward(gy)
        cases.append(dict(B=B, h=h, thw=[T, H, W], O=O, stride=list(st), z=z.detach(), w=w, gamma=g, beta=b,
                          out=out.detach(), thw_out=thw, gy=gy, dz=z.grad.clone(), dw=conv.weight.grad.clone(),
                          dgamma=norm.weight.grad.clone(), dbeta=norm.bias.grad.clone()))
    # skip path: MaxPool3d, 3-D input, no norm
    skips = []
    for i, (B, C, T, H, W, O, st) in enumerate([(2, 192, 2, 8, 8, 8, (1, 2, 2)), (1, 96, 3, 7, 7, 4, (1, 2, 2)),
                                                (1, 96, 2, 6, 6, 4, (1, 1, 1))]):
        ks = [s + 1 if s > 1 else s for s in st]
        pool = nn.MaxPool3d(ks, st, [k // 2 for k in ks], ceil_mode=False)
        x = synth_input(f"skip{i}.x", (B, 1 + T * H * W + O, C), 1).requires_grad_(True)
        out, thw = A.attention_pool(x, pool, [T, H, W], has_cls_embed=True)
        gy = synth_input(f"skip{i}.gy", out.shape, 1)
        out.backward(gy)
        skips.append(dict(thw=[T, H, W], stride=list(st), x=x.detach(), out=out.detach(), thw_out=thw, gy=gy,
                          dx=x.grad.clone()))
    save("attention_pool.pt", dict(conv=cases, skip=skips))


# ---------------------------------------------------------------- A7 / A8 modules
def grads_of(mod):
    """Small gradients are stored whole; large ones as (norm, random projection) in fp64."""
    out = {}
    for k, p in mod.named_parameters():
        g = p.grad
        if g.numel() <= 20000:
            out[k] = g.clone()
        else:
            r = synth_input("proj:" + k, g.shape, 9).double()
            out[k] = dict(norm=g.double().norm(), proj=(g.double() * r).sum())
    return out


def msa_cases():
    out = []
    specs = [  # dim, dim_out, heads, input_size, stride_q, stride_kv, thw(run), B, O
        (96, 96, 1, [2, 8, 8], [1, 1, 1], [1, 4, 4], [2, 8, 8], 2, 8),
        (96, 192, 2, [2, 8, 8], [1, 2, 2], [1, 2, 2], [2, 8, 8], 1, 8),
        (192, 192, 2, [2, 4, 4], [1, 1, 1], [1, 2, 2], [2, 4, 4], 2, 8),
        (192, 384, 4, [4, 6, 6], [1, 2, 2], [1, 1, 1], [4, 6, 6], 1, 16),
        (96, 96, 1, [4, 8, 8], [1, 1, 1], [1, 2, 2], [1, 8, 8], 2, 4),     # frame mode: rel_pos_t 7 -> 1
        (96, 192, 2, [2, 6, 6], [1, 1, 1], [1, 2, 2], [2, 7, 7], 1, 8),     # runtime grid != ctor grid -> interp
        (96, 192, 2, [2, 9, 9], [1, 2, 2], [1, 4, 4], [2, 9, 9], 1, 8),    # odd grid, non-integer ratios
    ]
    for i, (dim, dout, nh, isz, sq, skv, thw, B, O) in enumerate(specs):
        m = A.MultiScaleAttention(dim, dout, input_size=isz, num_heads=nh, qkv_bias=True, kernel_q=[3, 3, 3],
                                  kernel_kv=[3, 3, 3], stride_q=sq, stride_kv=skv, norm_layer=LN,
                                  has_cls_embed=True, mode="conv", pool_first=False, rel_pos_spatial=True,
                                  rel_pos_temporal=True, rel_pos_zero_init=False, residual_pooling=True,
                                  separate_qkv=False)
        load_state(m, 100 + i, w_std=0.15)
        N = 1 + thw[0] * thw[1] * thw[2] + O
        x = synth_input(f"msa{i}.x", (B, N, dim), 2).requires_grad_(True)
        y, qshape = m(x, thw)
        gy = synth_input(f"msa{i}.gy", y.shape, 2)
        y.backward(gy)
        out.append(dict(dim=dim, dim_out=dout, num_heads=nh, input_size=isz, stride_q=sq, stride_kv=skv, thw=thw,
                        seed=100 + i, w_std=0.15, x=x.detach(), y=y.detach(), q_shape=list(qshape), gy=gy,
                        dx=x.grad.clone(), dparams=grads_of(m)))
    save("msa.pt", out)


def block_cases():
    out = []
    specs = [
        (96, 96, 1, [2, 8, 8], [1, 1, 1], [1, 4, 4], 2, 8),
        (96, 192, 2, [2, 8, 8], [1, 2, 2], [1, 2, 2], 2, 8),
        (192, 384, 4, [2, 6, 6], [1, 2, 2], [1, 1, 1], 1, 8),
        (384, 384, 4, [2, 3, 3], [1, 1, 1], [1, 1, 1], 2, 8),
    ]
    for i, (dim, dout, nh, isz, sq, skv, B, O) in enumerate(specs):
        m = A.MultiScaleBlock(dim=dim, dim_out=dout, num_heads=nh, input_size=isz, mlp_ratio=4.0, qkv_bias=True,
                              drop_rate=0.0, drop_path=0.0, norm_layer=LN, kernel_q=[3, 3, 3], kernel_kv=[3, 3, 3],
                              stride_q=sq, stride_kv=skv, mode="conv", has_cls_embed=True, pool_first=False,
                              rel_pos_spatial=True, rel_pos_temporal=True, rel_pos_zero_init=False,
                              residual_pooling=True, dim_mul_in_att=True, separate_qkv=False)
        load_state(m, 200 + i, w_std=0.08)
        N = 1 + isz[0] * isz[1] * isz[2] + O
        x = synth_input(f"blk{i}.x", (B, N, dim), 3).requires_grad_(True)
        y, thw2 = m(x, isz)
        gy = synth_input(f"blk{i}.gy", y.shape, 3)
        y.backward(gy)
        out.append(dict(dim=dim, dim_out=dout, num_heads=nh, input_size=isz, stride_q=sq, stride_kv=skv, seed=200 + i,
                        w_std=0.08, x=x.detach(), y=y.detach(), thw_out=list(thw2), gy=gy, dx=x.grad.clone(),
                        dparams=grads_of(m)))
    save("block.pt", out)


# ---------------------------------------------------------------- full models
def run_model(cfg, seed, clip, w_std, train_grads=False):
    m = ns.builder.SViT(cfg.clone())
    load_state(m, seed, w_std=w_std)
    m.eval()
    cap = {}
    hk = m.head.projection.register_forward_hook(lambda mod, i, o: cap.__setitem__("logits", o.detach().clone()))
    with torch.no_grad():
        probs, extra = m([clip])
    hk.remove()
    res = dict(seed=seed, w_std=w_std, probs=probs, logits=cap["logits"],
               obj_desc=extra["obj_desc"], pred_bboxes=extra["pred_bboxes"],
               pred_contact_state=extra["pred_contact_state"])
    if train_grads:
        # training-mode forward with stochastic parts disabled: DropPath -> identity, head dropout p=0
        m.train()
        for mod in m.modules():
            if isinstance(mod, ns.common.DropPath):
                mod.drop_prob = 0.0
            if isinstance(mod, nn.Dropout):
                mod.p = 0.0
        logits, extra = m([clip])
        tgt = torch.arange(clip.shape[0]) % logits.shape[1]
        loss = torch.nn.functional.cross_entropy(logits, tgt) + 0.1 * extra["pred_bboxes"].square().mean() \
            + 0.1 * extra["pred_contact_state"].square().mean()
        loss.backward()
        res["train_logits"] = logits.detach()
        res["loss"] = loss.detach()
        res["grad_norms"] = {k: p.grad.norm().double() for k, p in m.named_parameters()}
        keep = ["cls_token", "object_queries", "pos_embed_temporal", "blocks.0.attn.rel_pos_h", "blocks.1.attn.pool_q.weight",
                "blocks.1.attn.rel_pos_t", "blocks.3.norm1.weight", "blocks.2.attn.norm_k.bias", "patch_embed.proj.bias",
                "blocks.0.attn.qkv.bias", "head.projection.bias", "blocks.3.mlp.fc2.bias", "blocks.1.proj.bias"]
        res["grads"] = {k: dict(m.named_parameters())[k].grad.clone() for k in keep}
    return res


def model_cases():
    tc = tiny_cfg()
    clip = synth_input("tiny.clip", (2, 3, 4, 32, 32), 5)
    res = run_model(tc, 300, clip, 0.06, train_grads=True)
    # frame mode: 4-D input [B,3,H,W] (video_model_builder.py:317-318)
    frames = synth_input("tiny.frames", (3, 3, 32, 32), 5)
    res_f = run_model(tc, 300, frames, 0.06)
    save("svit_tiny.pt", dict(video=res, frames=res_f))

    fc = ssv2_cfg()
    clip = synth_input("full.clip", (1, 3, 16, 224, 224), 6)
    res = run_model(fc, 400, clip, 0.04)
    save("svit_full.pt", res)


# ---------------------------------------------------------------- training-mode parity with DropPath ON (SURVEY App. C)
def droppath_case():
    """Tiny SViT in train() with every DropPath at p = 0.5 and head dropout off.  The reference draws, in block order,
    two torch.rand((B, 1, 1)) masks per block with a DropPath (attention branch attention.py:565, MLP branch :570) from
    the global CPU generator: the test re-draws them with the same seed and injects them into the B200 modules."""
    tc = tiny_cfg()
    B = 4
    clip = synth_input("tiny.clip.dp", (B, 3, 4, 32, 32), 15)
    m = ns.builder.SViT(tc.clone())
    load_state(m, 300, w_std=0.06)
    m.train()
    n_dp = 0
    for mod in m.modules():
        if isinstance(mod, ns.common.DropPath):
            mod.drop_prob = 0.5
            n_dp += 1
        if isinstance(mod, nn.Dropout):
            mod.p = 0.0
    torch.manual_seed(777)
    logits, extra = m([clip])
    tgt = torch.arange(B) % logits.shape[1]
    loss = torch.nn.functional.cross_entropy(logits, tgt) + 0.1 * extra["pred_bboxes"].square().mean()
    loss.backward()
    torch.manual_seed(777)
    masks = [torch.rand((B, 1, 1)) for _ in range(2 * n_dp)]  # each DropPath module is applied twice per forward
    keep = ["cls_token", "blocks.0.attn.qkv.weight", "blocks.1.attn.pool_q.weight", "blocks.1.mlp.fc1.bias",
            "blocks.2.attn.rel_pos_h", "blocks.3.norm2.weight", "patch_embed.proj.bias", "head.projection.weight"]
    named = dict(m.named_parameters())
    save("svit_tiny_droppath.pt", dict(seed=300, w_std=0.06, rng_seed=777, drop_prob=0.5, n_droppath_modules=n_dp,
                                       rand=torch.stack(masks).reshape(2 * n_dp, B), logits=logits.detach(), loss=loss.detach(),
                                       grad_norms={k: p.grad.norm().double() for k, p in named.items()},
                                       grads={k: named[k].grad.clone() for k in keep}))


# ---------------------------------------------------------------- R4 integer box logic
def box_cases():
    rng = np.random.RandomState(1234)
    cases = []
    B = ns.box_ops
    for i in range(64):
        b = torch.from_numpy(rng.rand(1, 4, 4).astype(np.float32))
        b[..., 2:] = b[..., :2] + b[..., 2:] * 0.5
        if i % 5 == 1: b[0, 2] = 0
        if i % 7 == 2: b[0, 1] = 0
        if i % 11 == 3: b[0, 3] = 0; b[0, 2] = 0
        if i % 13 == 4: b[0, 0] = 0
        if i % 6 == 5: b[0, 2, :2] = b[0, 0, :2] + 0.01   # near contact
        if i % 9 == 6: b[0, 3, :2] = b[0, 0, :2] + 0.02; b[0, 2, :2] = b[0, 1, :2] - 0.03   # crossed
        out, cs = B.match_haog(b.clone())
        cases.append(dict(inp=b, out=out, contact=cs))
    zcases = []
    for i in range(16):
        b = torch.from_numpy(rng.rand(3, 4, 4).astype(np.float32))
        b[..., 2:] *= (0.12 if i % 2 else 1.0)
        zcases.append(dict(inp=b.clone(), out=B.zero_empty_boxes(b.clone(), mode="cxcywh")))
    save("boxes.pt", dict(match_haog=cases, zero_empty=zcases))


# ---------------------------------------------------------------- N2 losses (models/losses.py:50-168)
def loss_cases():
    """boxes_loss_ and VideoImageLoss._haog_loss / forward of the unmodified reference on seeded predictions:
    values and gradients w.r.t. the predictions, incl. the 'no valid target' branches and the 5-column soft-mask form."""
    import importlib
    import types
    L = importlib.import_module("slowfast.models.losses")
    rng = np.random.RandomState(77)
    cases = []
    for i in range(8):
        B_, T_, O_ = 2 + i % 2, 1 + (i % 3), 4
        pred = torch.from_numpy(rng.randn(B_, T_, O_, 5).astype(np.float32))
        pred[..., 1:] = torch.sigmoid(pred[..., 1:])                      # (cx, cy, w, h) in (0, 1)
        tar = torch.from_numpy(rng.rand(B_, T_, O_, 4).astype(np.float32)) * 0.5 + 0.2
        drop = torch.from_numpy(rng.rand(B_, T_, O_) < (1.1 if i == 3 else 0.35))  # case 3: no valid target at all
        tar[drop] = 0
        if i % 4 == 2:                                                       # 5-column target with a soft mask
            tar = torch.cat([torch.from_numpy(rng.rand(B_, T_, O_, 1).astype(np.float32)), tar], -1)
        p = pred.clone().requires_grad_(True)
        l1, bce, giou = L.boxes_loss_(p, tar)
        (l1 + 2 * bce + 3 * giou).backward()
        cases.append(dict(pred=pred, tar=tar, l1=l1.detach(), bce=bce.detach(), giou=giou.detach(), dpred=p.grad.clone()))
    haog = []
    cfg = ssv2_cfg()
    for i in range(4):
        B_ = 3
        pb = torch.from_numpy(rng.randn(B_, 1, 4, 5).astype(np.float32)); pb[..., 1:] = torch.sigmoid(pb[..., 1:])
        pc = torch.from_numpy(rng.randn(B_, 1, 2, 5).astype(np.float32))
        tb = torch.from_numpy(rng.rand(B_, 1, 4, 4).astype(np.float32)) * 0.5 + 0.2
        tb[torch.from_numpy(rng.rand(B_, 1, 4) < 0.3)] = 0
        cs = torch.from_numpy(rng.randint(-1, 5, (B_, 2)).astype(np.int64))
        if i == 2: cs[:] = -1                                               # no annotated hand at all
        stub = types.SimpleNamespace(ce_loss=nn.CrossEntropyLoss(reduction="mean"), cfg=cfg,
                                     get_default_val=lambda: torch.tensor(0., requires_grad=True))
        a, c = pb.clone().requires_grad_(True), pc.clone().requires_grad_(True)
        out = L.VideoImageLoss._haog_loss(stub, {"pred_bboxes": a, "pred_contact_state": c},
                                          {"haog_bboxes": tb, "contact_state": cs})
        sum(out.values()).backward()
        haog.append(dict(pred_bboxes=pb, pred_contact_state=pc, haog_bboxes=tb, contact_state=cs,
                         out={k: v.detach() for k, v in out.items()}, dboxes=a.grad.clone(),
                         dcontact=c.grad.clone() if c.grad is not None else torch.zeros_like(pc)))
    save("losses.pt", dict(boxes=cases, haog=haog))


# ---------------------------------------------------------------- N4 input side: crop / flip / normalise + boxes
def aug_cases():
    """The reference's own functions -- datasets/utils.py tensor_normalize, transform.py random_crop (crop_clip_boxes) and
    horizontal_flip with fixed draws, then the box post-processing of ssv2_frames.py:347-353 -- on uint8 frames and
    [N, 4] pixel boxes.  (NO_RAND_PARAMS is a module flag of transform.py: switched off at run time so that the crop
    offsets / flip draw can be passed in; the file itself is untouched.)"""
    import importlib
    ref_loader._shell("slowfast.datasets", os.path.join(ref_loader.REF_ROOT, "slowfast", "datasets"))
    TR = importlib.import_module("slowfast.datasets.transform")
    TR.NO_RAND_PARAMS = False
    spec = importlib.util.spec_from_file_location("ref_dutils_part", os.path.join(ref_loader.REF_ROOT, "slowfast", "datasets", "utils.py"))
    src = open(spec.origin).read()
    g = {"torch": torch}
    start = src.index("def tensor_normalize(")
    exec(src[start:src.index("\ndef ", start + 10)], g)   # tensor_normalize only (utils.py:287-303), verbatim
    tensor_normalize = g["tensor_normalize"]
    rng = np.random.RandomState(4242)
    mean, std = [0.45, 0.40, 0.35], [0.225, 0.25, 0.2]
    cases = []
    for i, (T, H, W, cs) in enumerate(((4, 40, 52, 32), (2, 36, 36, 36), (3, 48, 44, 24), (1, 33, 41, 28))):
        frames = torch.from_numpy(rng.randint(0, 256, (T, H, W, 3)).astype(np.uint8))
        xo = int(rng.randint(0, W - cs + 1)); yo = int(rng.randint(0, H - cs + 1))
        flip = bool(i % 2 == 0)
        boxes = rng.rand(12, 4).astype(np.float32) * np.array([W, H, W, H], np.float32) * 0.7
        boxes[:, 2:] = boxes[:, :2] + rng.rand(12, 2).astype(np.float32) * np.array([W, H], np.float32) * 0.6
        boxes[3] = 0                                           # an empty slot
        boxes[5, 2:] = boxes[5, :2] + 0.5                      # thinner than eps after normalisation
        x = tensor_normalize(frames, mean, std).permute(3, 0, 1, 2)          # C T H W
        rp = {"random_crop_x_offset": xo, "random_crop_y_offset": yo, "horizontal_flip": 0.25 if flip else 0.75}
        if H == cs and W == cs:
            xc, bc = x, TR.crop_clip_boxes(boxes, 0, 0, cs)    # random_crop returns the images alone in this case
        else:
            xc, bc = TR.random_crop(x, cs, boxes=boxes, rand_params=rp)
        xf, bf = TR.horizontal_flip(0.5, xc, boxes=bc, rand_params=rp)
        h, w = xf.shape[-2:]
        bb = bf.copy()
        bb[..., [0, 2]] = bb[..., [0, 2]] / w
        bb[..., [1, 3]] = bb[..., [1, 3]] / h
        bb = torch.from_numpy(np.clip(bb, 0, 1))
        bb = ns.box_ops.box_xyxy_to_cxcywh(bb)
        bb = ns.box_ops.zero_empty_boxes(bb, mode="cxcywh")
        cases.append(dict(frames=frames, boxes=torch.from_numpy(boxes), x_off=xo if not (H == cs and W == cs) else 0,
                          y_off=yo if not (H == cs and W == cs) else 0, flip=flip, crop=cs, mean=mean, std=std,
                          clip=xf.contiguous(), boxes_out=bb))
    save("aug.pt", cases)


# ---------------------------------------------------------------- N3 optimizer groups and learning-rate policy
def optim_cases():
    """models/optimizer.py of the unmodified reference: the weight-decay groups construct_optimizer builds for the tiny
    SViT (parameter names per weight decay), the optimizer's class and base lr, and get_epoch_lr on the ssv2.yaml cosine
    schedule without and with a 5-epoch warm-up.  The committed optim.pt was written by this function with
    svit_b200.optim standing in for construct_optimizer / get_epoch_lr, after tests/test_host_logic.py had matched the
    two bit for bit against the reference; neither has changed since."""
    import copy
    import importlib

    import svit_b200
    R = importlib.import_module("slowfast.models.optimizer")
    cfg = tiny_cfg()
    cfg.BN = type(cfg)({"WEIGHT_DECAY": 0.0}) if not hasattr(cfg, "BN") else cfg.BN
    model = svit_b200.SViT(cfg, compute_dtype=torch.float32)
    opt = R.construct_optimizer(model, cfg)
    names = {id(p): n for n, p in model.named_parameters()}
    groups = {float(g["weight_decay"]): sorted(names[id(p)] for p in g["params"]) for g in opt.param_groups}
    lr = []
    for warmup in (ssv2_cfg().SOLVER.WARMUP_EPOCHS, 5.0):
        c = ssv2_cfg()
        c.SOLVER.WARMUP_EPOCHS = warmup
        for e in (0.0, 0.37, 4.99, 5.0, 12.5, 49.999):
            lr.append(dict(warmup_epochs=warmup, epoch=e, out=copy.deepcopy(R.get_epoch_lr(e, c))))
    save("optim.pt", dict(wd_groups=groups, optimizer=type(opt).__name__, base_lr=opt.defaults["lr"], lr=lr))


if __name__ == "__main__":
    relpos_tables()
    pool_cases()
    msa_cases()
    block_cases()
    model_cases()
    droppath_case()
    aug_cases()
    box_cases()
    loss_cases()
    optim_cases()
