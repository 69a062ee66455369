"""torch.autograd glue over the C ABI (include/svit_b200.h).

PyTorch is used here for device memory, streams and the autograd tape only: every tensor-sized
computation is a call into libsvit_sm100.so.  Saved tensors are torch tensors; gradients of
parameters are produced in fp32 regardless of the activation dtype.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional, Sequence, Tuple

import torch

from . import _lib
from ._lib import BF16, F32, IMPL_AUTO, IMPL_SIMT, IMPL_TC, AttnArgs, GemmArgs, check

LN_EPS = 1e-6
HEAD_DIM = 96

_state = {"gemm_impl": IMPL_AUTO, "attn_impl": IMPL_AUTO, "launches": 0,
          # rel-pos gradient of the tensor-core attention backward in table-row space (A / B switch for measurements)
          "attn_tab_grad": os.environ.get("SVIT_ATTN_TAB_GRAD", "1") != "0"}


def set_impl(gemm: Optional[int] = None, attn: Optional[int] = None):
    """Select kernel families: IMPL_AUTO (tcgen05 for bf16 when supported), IMPL_SIMT, IMPL_TC."""
    if gemm is not None:
        _state["gemm_impl"] = gemm
    if attn is not None:
        _state["attn_impl"] = attn


def launches() -> int:
    """Number of C-ABI kernel-launching calls made so far (bench.py's gpu_launches)."""
    return _state["launches"]


def _dt(t: torch.Tensor) -> int:
    if t.dtype == torch.float32:
        return F32
    if t.dtype == torch.bfloat16:
        return BF16
    raise TypeError(f"svit_b200 supports float32 and bfloat16 activations, got {t.dtype}")


def _chk(t: torch.Tensor, name: str) -> torch.Tensor:
    if not t.is_cuda:
        raise RuntimeError(f"{name}: svit_b200 kernels are CUDA only (got a {t.device} tensor); there is no CPU path")
    return t


def _stream():
    # raw cudaStream_t of torch's current stream: torch.cuda.current_stream() costs ~5 us of Python per call
    # (device-index resolution through os.environ), the C accessors ~0.3 us -- there is one call per kernel launch
    return torch._C._cuda_getCurrentRawStream(torch._C._cuda_getDevice())


def _p(t: Optional[torch.Tensor]):
    return None if t is None else t.data_ptr()


def _f32(t: torch.Tensor) -> torch.Tensor:
    t = t.detach()
    return t if (t.dtype == torch.float32 and t.is_contiguous()) else t.float().contiguous()


_wcache = {}


def _cache_get(w, tag):
    ent = _wcache.get((id(w), tag))
    if ent is not None and ent[0]() is w and ent[1] == w._version and ent[2] == w.data_ptr():
        return ent[3]
    return None


def _cache_put(w, tag, value):
    import weakref

    key = (id(w), tag)
    _wcache[key] = (weakref.ref(w, lambda _r, k=key: _wcache.pop(k, None)), w._version, w.data_ptr(), value)
    return value


def cast_weight(w: torch.Tensor, dtype: torch.dtype) -> torch.Tensor:
    """Compute-dtype copy of a GEMM weight, cached per parameter object until it is modified
    (checked through param._version and data_ptr)."""
    if w.dtype == dtype and w.is_contiguous():
        return w.detach()
    c = _cache_get(w, dtype)
    if c is None:
        c = _cache_put(w, dtype, w.detach().to(dtype).contiguous())
    return c


_FAMILY = {"svit_gemm": "gemm", "svit_attn_fwd": "attention", "svit_attn_bwd": "attention_bwd",
           "svit_pool_ln_fwd": "pool_ln", "svit_pool_ln_fwd_save": "pool_ln", "svit_pool_ln_bwd": "pool_ln_bwd",
           "svit_pool_ln_bwd_saved": "pool_ln_bwd", "svit_layernorm_fwd": "layernorm", "svit_row_stats": "layernorm",
           "svit_layernorm_bwd": "layernorm_bwd", "svit_skip_maxpool_fwd": "skip_pool", "svit_skip_maxpool_fwd_idx": "skip_pool", "svit_im2col3d": "im2col", "svit_s2d_clip": "im2col",
           "svit_patch_embed_s2d": "gemm", "svit_mlp_fused": "gemm",
           "svit_patch_embed_s2d_dgrad": "gemm", "svit_d2s_clip": "im2col", "svit_col2im3d": "im2col"}
_prof = None


def profile_start():
    """Record a CUDA-event pair around every C-ABI call (bench.py's per-kernel breakdown; adds launch gaps,
    so it is only used in a separate instrumented pass, never in the timed region)."""
    global _prof
    _prof = []


def profile_stop(steps: int = 1):
    global _prof
    rec, _prof = _prof, None
    torch.cuda.synchronize()
    fam, detail = {}, {}
    for name, tag, e0, e1 in rec:
        ms = e0.elapsed_time(e1)
        f = fam.setdefault(_FAMILY.get(name, "misc"), {"ms_per_step": 0.0, "calls_per_step": 0.0})
        f["ms_per_step"] += ms / steps
        f["calls_per_step"] += 1.0 / steps
        d = detail.setdefault(f"{name}{tag or ''}", {"ms_per_step": 0.0, "calls_per_step": 0.0})
        d["ms_per_step"] += ms / steps
        d["calls_per_step"] += 1.0 / steps
    return {"families": fam, "detail": detail}


def _call(name, *args, tag=None):
    _state["launches"] += 1
    if _prof is not None:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        check(getattr(_lib.lib(), name)(*args), name)
        e1.record()
        _prof.append((name, tag, e0, e1))
        return
    check(getattr(_lib.lib(), name)(*args), name)


# --------------------------------------------------------------------------------------------
# GEMM
# --------------------------------------------------------------------------------------------
def gemm(A, B, out, M, N, K, lda, ldb, ldc, transA=0, transB=1, bias=None, residual=None, ldr=0,
         sample_scale=None, rows_per_sample=0, gelu_pre=None, ldg=0, pre_out=None, ldp=0, act=0,
         remap=(0, 0, 0), impl=None, batch=0, strideA=0, strideB=0, strideC=0, b_inner=0, strideB_inner=0,
         a_inner=0, strideA_inner=0, alpha=0.0, ln_stats=None, ln_colsum=None):
    a = GemmArgs()
    a.ln_stats, a.ln_colsum = _p(ln_stats), _p(ln_colsum)
    a.a_inner, a.strideA_inner, a.alpha = a_inner, strideA_inner, alpha
    a.batch, a.strideA, a.strideB, a.strideC, a.b_inner, a.strideB_inner = batch, strideA, strideB, strideC, b_inner, strideB_inner
    a.A, a.B, a.C = A.data_ptr(), B.data_ptr(), out.data_ptr()
    a.M, a.N, a.K, a.lda, a.ldb, a.ldc = M, N, K, lda, ldb, ldc
    a.transA, a.transB = transA, transB
    a.bias, a.residual, a.ldr = _p(bias), _p(residual), ldr
    a.sample_scale, a.rows_per_sample = _p(sample_scale), rows_per_sample
    a.gelu_pre, a.ldg, a.pre_out, a.ldp, a.act = _p(gelu_pre), ldg, _p(pre_out), ldp, act
    a.rows_in, a.rows_out, a.row_off = remap
    a.dtype, a.out_dtype = _dt(A), _dt(out)
    a.impl = _state["gemm_impl"] if impl is None else impl
    _call("svit_gemm", C.byref(a), _stream(), tag=f"[{M}x{N}x{K}]" if _prof is not None else None)
    return out


def _colsum(x2d: torch.Tensor, M, N) -> torch.Tensor:
    out = torch.zeros(N, dtype=torch.float32, device=x2d.device)
    _call("svit_colsum", x2d.data_ptr(), out.data_ptr(), M, N, N, _dt(x2d), _stream())
    return out


def _scale_rows(x: torch.Tensor, scale: torch.Tensor, rows_per_sample: int) -> torch.Tensor:
    y = torch.empty_like(x)
    Cn = x.shape[-1]
    _call("svit_scale_rows", x.data_ptr(), scale.data_ptr(), y.data_ptr(), x.numel() // Cn, Cn, rows_per_sample,
          _dt(x), _stream())
    return y


class _Linear(torch.autograd.Function):
    """y = residual + sample_scale * (x W^T + b)   (nn.Linear sites attention.py:345,462,561)."""

    @staticmethod
    def forward(ctx, x, weight, bias, residual, sample_scale):
        _chk(x, "linear")
        x = x.contiguous()
        K = x.shape[-1]
        N = weight.shape[0]
        M = x.numel() // K
        w = cast_weight(weight, x.dtype)
        out = torch.empty(*x.shape[:-1], N, dtype=x.dtype, device=x.device)
        rps = (M // sample_scale.numel()) if sample_scale is not None else 0
        res = residual.contiguous() if residual is not None else None
        gemm(x, w, out, M, N, K, K, K, N, 0, 1, bias=_f32(bias) if bias is not None else None, residual=res, ldr=N,
             sample_scale=sample_scale, rows_per_sample=rps)
        ctx.save_for_backward(x, weight, sample_scale)
        ctx.has_bias = bias is not None
        ctx.has_res = residual is not None
        ctx.rps = rps
        return out

    @staticmethod
    def backward(ctx, dy):
        x, weight, sample_scale = ctx.saved_tensors
        dy = dy.contiguous()
        K = x.shape[-1]
        N = weight.shape[0]
        M = x.numel() // K
        dres = dy if ctx.has_res else None
        g = _scale_rows(dy, sample_scale, ctx.rps) if sample_scale is not None else dy
        w = cast_weight(weight, x.dtype)
        dx = dw = db = None
        if ctx.needs_input_grad[0]:
            dx = torch.empty_like(x)
            gemm(g, w, dx, M, K, N, N, K, K, 0, 0)
        if ctx.needs_input_grad[1]:
            dw = torch.empty(N, K, dtype=torch.float32, device=x.device)
            gemm(g, x, dw, N, K, M, N, K, K, 1, 0)
        if ctx.has_bias and ctx.needs_input_grad[2]:
            db = _colsum(g, M, N)
        return dx, dw, db, dres, None


def linear(x, weight, bias=None, residual=None, sample_scale=None):
    return _Linear.apply(x, weight, bias, residual, sample_scale)


class _Mlp(torch.autograd.Function):
    """y = residual + sample_scale * fc2(gelu(fc1(x)))   (common.py:27-34, attention.py:567-570)."""

    @staticmethod
    def forward(ctx, x, w1, b1, w2, b2, residual, sample_scale, grad_mode):
        _chk(x, "mlp")
        x = x.contiguous()
        K = x.shape[-1]
        Hd = w1.shape[0]
        N = w2.shape[0]
        M = x.numel() // K
        need = grad_mode and any(ctx.needs_input_grad[:5])
        w1c, w2c = cast_weight(w1, x.dtype), cast_weight(w2, x.dtype)
        hid = torch.empty(*x.shape[:-1], Hd, dtype=x.dtype, device=x.device)
        pre = torch.empty_like(hid) if need else None
        gemm(x, w1c, hid, M, Hd, K, K, K, Hd, 0, 1, bias=_f32(b1), act=1, pre_out=pre, ldp=Hd)
        out = torch.empty(*x.shape[:-1], N, dtype=x.dtype, device=x.device)
        rps = (M // sample_scale.numel()) if sample_scale is not None else 0
        res = residual.contiguous() if residual is not None else None
        gemm(hid, w2c, out, M, N, Hd, Hd, Hd, N, 0, 1, bias=_f32(b2), residual=res, ldr=N, sample_scale=sample_scale,
             rows_per_sample=rps)
        if need:
            ctx.save_for_backward(x, w1, w2, pre, hid, sample_scale)
        ctx.has_res = residual is not None
        ctx.rps = rps
        return out

    @staticmethod
    def backward(ctx, dy):
        x, w1, w2, pre, hid, sample_scale = ctx.saved_tensors
        dy = dy.contiguous()
        K = x.shape[-1]
        Hd = w1.shape[0]
        N = w2.shape[0]
        M = x.numel() // K
        dres = dy if ctx.has_res else None
        g = _scale_rows(dy, sample_scale, ctx.rps) if sample_scale is not None else dy
        w1c, w2c = cast_weight(w1, x.dtype), cast_weight(w2, x.dtype)
        dw2 = torch.empty(N, Hd, dtype=torch.float32, device=x.device)
        gemm(g, hid, dw2, N, Hd, M, N, Hd, Hd, 1, 0)
        db2 = _colsum(g, M, N)
        dpre = torch.empty_like(pre)
        gemm(g, w2c, dpre, M, Hd, N, N, Hd, Hd, 0, 0, gelu_pre=pre, ldg=Hd)
        dw1 = torch.empty(Hd, K, dtype=torch.float32, device=x.device)
        gemm(dpre, x, dw1, Hd, K, M, Hd, K, K, 1, 0)
        db1 = _colsum(dpre, M, Hd)
        dx = torch.empty_like(x)
        gemm(dpre, w1c, dx, M, K, Hd, Hd, K, K, 0, 0)
        return dx, dw1, db1, dw2, db2, dres, None, None


_MLP_FUSED = {"enabled": os.environ.get("SVIT_MLP_FUSED", "1") != "0", "max_width": int(os.environ.get("SVIT_MLP_FUSED_MAXW", "192"))}


def mlp_fused_applicable(x, w1, w2, sample_scale=None) -> bool:
    """svit_mlp_fused: inference (no autograd, no DropPath scale), bf16, the tcgen05 path, a supported (C, H, N)."""
    if not _MLP_FUSED["enabled"] or torch.is_grad_enabled() or sample_scale is not None or x.dtype != torch.bfloat16:
        return False
    if _state["gemm_impl"] == IMPL_SIMT or not x.is_cuda or x.shape[-1] > _MLP_FUSED["max_width"]:
        return False
    M = x.numel() // x.shape[-1]
    return bool(_lib.lib().svit_mlp_fused_supported(M, x.shape[-1], w1.shape[0], w2.shape[0]))


def mlp_fused_has_ln(width: int) -> bool:
    """The LayerNorm prologue exists in the resident-weight kernel (width 96) only."""
    return width == 96


def mlp_fused(x, w1, b1, w2, b2, residual=None, ln=None):
    """out = residual + fc2(gelu(fc1(LN(x)))) in one kernel, the hidden activation never written to HBM (inference).
    ln = (gamma, beta, eps): x is the UN-normalised input, normalised on the fly; residual must then be x or None."""
    x = x.contiguous()
    K, Hd, N = x.shape[-1], w1.shape[0], w2.shape[0]
    M = x.numel() // K
    out = torch.empty(*x.shape[:-1], N, dtype=x.dtype, device=x.device)
    res = None
    if residual is not None:
        res = x if residual is x else residual.contiguous()
    g = bt = None
    eps = 0.0
    if ln is not None:
        g, bt, eps = _f32(ln[0]), _f32(ln[1]), float(ln[2])
        if res is not None and res.data_ptr() != x.data_ptr():
            raise ValueError("mlp_fused: with a LayerNorm prologue the residual must be the input itself")
    _call("svit_mlp_fused", x.data_ptr(), cast_weight(w1, x.dtype).data_ptr(), _f32(b1).data_ptr(),
          cast_weight(w2, x.dtype).data_ptr(), _f32(b2).data_ptr(), _p(res), out.data_ptr(), M, K, Hd, N, _p(g), _p(bt), eps,
          _stream(), tag=f"[{M}x{K}x{Hd}x{N}]" if _prof is not None else None)
    return out


def mlp(x, w1, b1, w2, b2, residual=None, sample_scale=None):
    if mlp_fused_applicable(x, w1, w2, sample_scale):
        return mlp_fused(x, w1, b1, w2, b2, residual)
    return _Mlp.apply(x, w1, b1, w2, b2, residual, sample_scale, torch.is_grad_enabled())


# --------------------------------------------------------------------------------------------
# LayerNorm
# --------------------------------------------------------------------------------------------
class _LayerNorm(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, gamma, beta, eps, grad_mode):
        _chk(x, "layer_norm")
        x = x.contiguous()
        Cn = x.shape[-1]
        rows = x.numel() // Cn
        need = grad_mode and any(ctx.needs_input_grad[:3])
        y = torch.empty_like(x)
        mean = torch.empty(rows, dtype=torch.float32, device=x.device) if need else None
        rstd = torch.empty(rows, dtype=torch.float32, device=x.device) if need else None
        g32 = _f32(gamma)
        _call("svit_layernorm_fwd", x.data_ptr(), g32.data_ptr(), _f32(beta).data_ptr(), y.data_ptr(), _p(mean),
              _p(rstd), rows, Cn, float(eps), _dt(x), _stream())
        if need:
            ctx.save_for_backward(x, g32, mean, rstd)
        return y

    @staticmethod
    def backward(ctx, dy):
        x, g32, mean, rstd = ctx.saved_tensors
        dy = dy.contiguous()
        Cn = x.shape[-1]
        rows = x.numel() // Cn
        dx = torch.empty_like(x)
        dgb = torch.zeros(2, Cn, dtype=torch.float32, device=x.device)  # one fill for both accumulators
        dg, db = dgb[0], dgb[1]
        _call("svit_layernorm_bwd", dy.data_ptr(), x.data_ptr(), g32.data_ptr(), mean.data_ptr(), rstd.data_ptr(),
              dx.data_ptr(), dg.data_ptr(), db.data_ptr(), rows, Cn, _dt(x), _stream())
        return dx, dg, db, None, None


def layer_norm(x, gamma, beta, eps=LN_EPS):
    return _LayerNorm.apply(x, gamma, beta, eps, torch.is_grad_enabled())


# LayerNorm folded into the consuming GEMM (inference; attention.py:558-561, 566-567):
#   LayerNorm(x) W^T + b = rstd * (x W'^T - mean * colsum(W')) + (b + W beta),   W' = W diag(gamma)
# The normalised activation never exists in HBM: one statistics pass reads x (svit_row_stats), the GEMM reads x
# itself and its epilogue applies the per-row correction.
# Measured on B200 (B = 64 forward): the 33 LayerNorm launches cost 1.54 ms, the statistics passes 0.88 ms, but the
# folded epilogues (two table values per column, one more FFMA2 per pair) add 0.64 ms to the qkv / fc1 GEMMs, which are
# epilogue-bound -- break-even, so the folded form is opt-in (SVIT_LN_FOLD=1) and the LayerNorm kernel stays the default.
_LN_FOLD = {"enabled": os.environ.get("SVIT_LN_FOLD", "0") == "1"}
_fold_cache = {}


def ln_fold_applicable(x: torch.Tensor, *weights) -> bool:
    """The folded form runs on the tcgen05 TMA-store GEMM only: bf16, no autograd, >= 128 rows, 8-aligned widths."""
    if not _LN_FOLD["enabled"] or torch.is_grad_enabled() or x.dtype != torch.bfloat16:
        return False
    if _state["gemm_impl"] == IMPL_SIMT or x.numel() // x.shape[-1] < 128 or x.shape[-1] % 8:
        return False
    return all(w.shape[0] % 8 == 0 for w in weights)


def row_stats(x: torch.Tensor, eps: float = LN_EPS) -> torch.Tensor:
    """[M, 2] fp32 (mean, rstd) of every row of x [.., C]."""
    _chk(x, "row_stats")
    x = x.contiguous()
    Cn = x.shape[-1]
    M = x.numel() // Cn
    stats = torch.empty(M, 2, dtype=torch.float32, device=x.device)
    _call("svit_row_stats", x.data_ptr(), stats.data_ptr(), M, Cn, float(eps), _dt(x), _stream())
    return stats


def folded_ln_weight(weight, bias, gamma, beta, dtype):
    """(W' [N, K] in `dtype`, table [N / 2, 4] fp32 = (c[2i], c[2i+1], b'[2i], b'[2i+1]) with c = the row sums of the
    ROUNDED W' and b' = bias + W beta), cached until any of the four parameters is modified."""
    tensors = (weight, bias, gamma, beta)
    key = (id(weight), id(gamma), dtype)
    sig = tuple((id(t), t._version, t.data_ptr()) if t is not None else None for t in tensors)
    ent = _fold_cache.get(key)
    if ent is not None and ent[0] == sig and all(r is None or r() is t for r, t in zip(ent[1], tensors)):
        return ent[2]
    import weakref

    w32, g32, b32 = weight.detach().float(), gamma.detach().float(), beta.detach().float()
    wf = (w32 * g32[None, :]).to(dtype).contiguous()
    colsum = wf.float().sum(dim=1).contiguous()
    bias2 = w32 @ b32
    if bias is not None:
        bias2 = bias2 + bias.detach().float()
    N = wf.shape[0]
    table = torch.cat([colsum.reshape(N // 2, 2), bias2.reshape(N // 2, 2)], dim=1).contiguous()
    refs = tuple(weakref.ref(t, lambda _r, k=key: _fold_cache.pop(k, None)) if t is not None else None for t in tensors)
    _fold_cache[key] = (sig, refs, (wf, table))
    return _fold_cache[key][2]


def linear_ln(x, stats, gamma, beta, weight, bias=None):
    """LayerNorm(x; gamma, beta) W^T + b with the statistics of `row_stats(x)`; inference only (no autograd)."""
    assert not torch.is_grad_enabled()
    x = x.contiguous()
    K = x.shape[-1]
    N = weight.shape[0]
    M = x.numel() // K
    wf, table = folded_ln_weight(weight, bias, gamma, beta, x.dtype)
    out = torch.empty(*x.shape[:-1], N, dtype=x.dtype, device=x.device)
    gemm(x, wf, out, M, N, K, K, K, N, 0, 1, ln_stats=stats, ln_colsum=table)
    return out


def mlp_ln(x, stats, gamma, beta, w1, b1, w2, b2, residual=None, sample_scale=None):
    """residual + sample_scale * fc2(gelu(fc1(LayerNorm(x))))  (common.py:27-34, attention.py:566-570); inference only."""
    assert not torch.is_grad_enabled()
    x = x.contiguous()
    K = x.shape[-1]
    Hd = w1.shape[0]
    N = w2.shape[0]
    M = x.numel() // K
    wf, table = folded_ln_weight(w1, b1, gamma, beta, x.dtype)
    hid = torch.empty(*x.shape[:-1], Hd, dtype=x.dtype, device=x.device)
    gemm(x, wf, hid, M, Hd, K, K, K, Hd, 0, 1, act=1, ln_stats=stats, ln_colsum=table)
    out = torch.empty(*x.shape[:-1], N, dtype=x.dtype, device=x.device)
    rps = (M // sample_scale.numel()) if sample_scale is not None else 0
    res = residual.contiguous() if residual is not None else None
    gemm(hid, cast_weight(w2, x.dtype), out, M, N, Hd, Hd, Hd, N, 0, 1, bias=_f32(b2), residual=res, ldr=N,
         sample_scale=sample_scale, rows_per_sample=rps)
    return out


# --------------------------------------------------------------------------------------------
# attention_pool (conv + LN) on the packed qkv tensor, and the max-pool skip path
# --------------------------------------------------------------------------------------------
_frac_cache = {}


def tap_fractions(stride_hw: int, device) -> torch.Tensor:
    """frac[tap] = (#outputs of conv3d(3x3x3 cube, k3, stride (1,s,s), pad 1) for which the tap is in bounds)
    / #outputs.  w_eff = conv_w . frac is the per-channel scale of an object token (attention.py:45-53)."""
    key = (stride_hw, str(device))
    if key not in _frac_cache:
        s = stride_hw
        n_t, n_hw = 3, (3 + 2 - 3) // s + 1
        frac = []
        for kt in range(3):
            ct = sum(1 for o in range(n_t) if 0 <= o - 1 + kt < 3)
            for kh in range(3):
                ch = sum(1 for o in range(n_hw) if 0 <= o * s - 1 + kh < 3)
                for kw in range(3):
                    cw = sum(1 for o in range(n_hw) if 0 <= o * s - 1 + kw < 3)
                    frac.append(ct * ch * cw / float(n_t * n_hw * n_hw))
        _frac_cache[key] = torch.tensor(frac, dtype=torch.float32, device=device)
    return _frac_cache[key]


def pooled_hw(n: int, s: int) -> int:
    return (n - 1) // s + 1


_side_streams = {}


def _branches(n: int):
    """n CUDA streams for independent kernel chains of one op (stream 0 = the current stream).  The q / k / v pooling
    kernels are small and latency-bound; running the three chains side by side fills the SMs that each kernel's tail
    leaves idle.  Fork / join are event waits, so the pattern is graph-capturable."""
    cur = torch.cuda.current_stream()
    key = (cur.device.index, n, cur.cuda_stream)  # per launching stream: concurrent forwards (graph lanes) do not share
    if key not in _side_streams:
        _side_streams[key] = [torch.cuda.Stream(device=cur.device) for _ in range(n - 1)]
    return [cur] + _side_streams[key]


class _Fork:
    """with _Fork(3) as f: for i in range(3): with f.branch(i): launch chain i   -> joined on exit."""

    def __init__(self, n):
        # per-kernel event timing (profile mode) needs the kernels one at a time
        self.streams = _branches(n) if (_state.get("multi_stream", True) and _prof is None) else None
        self.n = n

    def __enter__(self):
        if self.streams is not None:
            self.start = torch.cuda.Event()
            self.start.record(self.streams[0])
            self.done = []
        return self

    def branch(self, i):
        if self.streams is None or i == 0:
            return _NullCtx()
        return _Branch(self, i)

    def __exit__(self, *exc):
        if self.streams is not None:
            for ev in self.done:
                self.streams[0].wait_event(ev)
        return False


class _NullCtx:
    def __enter__(self):
        return self

    def __exit__(self, *exc):
        return False


class _Branch:
    def __init__(self, fork, i):
        self.fork, self.s = fork, fork.streams[i]
        self.ctx = torch.cuda.stream(self.s)

    def __enter__(self):
        self.s.wait_event(self.fork.start)
        self.ctx.__enter__()
        return self

    def __exit__(self, *exc):
        ev = torch.cuda.Event()
        ev.record(self.s)
        self.fork.done.append(ev)
        return self.ctx.__exit__(*exc)


class _QKVPool(torch.autograd.Function):
    """q, k, v = attention_pool(qkv[which], pool_which, thw, norm_which) for which in (q, k, v)
    (attention.py:368-388), reading the packed [B, N, 3, h, 96] GEMM output in place."""

    @staticmethod
    def forward(ctx, qkv, thw, O, stride_q, stride_kv, wq, gq, bq, wk, gk, bk, wv, gv, bv, grad_mode):
        _chk(qkv, "qkv_pool")
        qkv = qkv.contiguous()
        B, N, D3 = qkv.shape
        h = D3 // (3 * HEAD_DIM)
        T, H, W = thw
        outs = []
        params = ((wq, gq, bq, stride_q), (wk, gk, bk, stride_kv), (wv, gv, bv, stride_kv))
        saved = []
        prepared = []
        for which, (w, g, b, s) in enumerate(params):  # allocations and parameter casts stay on the current stream
            Ho, Wo = pooled_hw(H, s), pooled_hw(W, s)
            out = torch.empty(B, h, 1 + T * Ho * Wo + O, HEAD_DIM, dtype=qkv.dtype, device=qkv.device)
            prepared.append((out, _f32(w).reshape(HEAD_DIM, 27), _f32(g), _f32(b), tap_fractions(s, qkv.device), s))
        # training (bf16): the forward also writes the pre-LayerNorm rows, the backward reads them instead of recomputing
        # the convolution per output token (svit_pool_ln_fwd_save / svit_pool_ln_bwd_saved)
        save_pre = grad_mode and qkv.dtype == torch.bfloat16 and _state.get("pool_save_pre", True)
        pres = [torch.empty_like(p_[0]) if save_pre else None for p_ in prepared]
        with _Fork(3) as fork:
            for which, (out, w32, g32, b32, frac, s) in enumerate(prepared):
                with fork.branch(which):
                    src = qkv.data_ptr() + which * h * HEAD_DIM * qkv.element_size()
                    tag = f"[{'qkv'[which]} B{B} h{h} {T}x{H}x{W} s{s}]" if _prof is not None else None
                    if save_pre:
                        _call("svit_pool_ln_fwd_save", src, N * D3, D3, HEAD_DIM, w32.data_ptr(), frac.data_ptr(),
                              g32.data_ptr(), b32.data_ptr(), out.data_ptr(), pres[which].data_ptr(), B, h, T, H, W, O, s,
                              LN_EPS, _dt(qkv), _stream(), tag=tag)
                    else:
                        _call("svit_pool_ln_fwd", src, N * D3, D3, HEAD_DIM, w32.data_ptr(), frac.data_ptr(), g32.data_ptr(),
                              b32.data_ptr(), out.data_ptr(), B, h, T, H, W, O, s, LN_EPS, _dt(qkv), _stream(), tag=tag)
                outs.append(out)
                saved += [w32, g32]
        if save_pre:
            saved += pres
        ctx.save_pre = save_pre
        ctx.save_for_backward(qkv, *saved)
        ctx.geom = (B, N, h, T, H, W, O, stride_q, stride_kv)
        ctx.wshape = wq.shape
        return tuple(outs)

    @staticmethod
    def backward(ctx, dq, dk, dv):
        qkv, *saved = ctx.saved_tensors
        B, N, h, T, H, W, O, sq, skv = ctx.geom
        D3 = 3 * h * HEAD_DIM
        dqkv = torch.empty_like(qkv)
        grads = []
        acc = torch.zeros(3, HEAD_DIM * 29, dtype=torch.float32, device=qkv.device)  # dw | dgamma | dbeta x (q, k, v)
        douts = [d.contiguous() for d in (dq, dk, dv)]
        dpres = [torch.empty_like(d) for d in douts]  # allocated (and later freed) on the current stream
        fracs = [tap_fractions(s, qkv.device) for s in (sq, skv, skv)]
        with _Fork(3) as fork:
            for which, s in enumerate((sq, skv, skv)):
                w32, g32 = saved[2 * which], saved[2 * which + 1]
                dw, dg, db = acc[which, :HEAD_DIM * 27], acc[which, HEAD_DIM * 27:HEAD_DIM * 28], acc[which, HEAD_DIM * 28:]
                off = which * h * HEAD_DIM * qkv.element_size()
                with fork.branch(which):
                    if ctx.save_pre:
                        _call("svit_pool_ln_bwd_saved", qkv.data_ptr() + off, N * D3, D3, HEAD_DIM, w32.data_ptr(),
                              fracs[which].data_ptr(), g32.data_ptr(), douts[which].data_ptr(), saved[6 + which].data_ptr(),
                              dpres[which].data_ptr(), dqkv.data_ptr() + off, dw.data_ptr(), dg.data_ptr(), db.data_ptr(),
                              B, h, T, H, W, O, s, LN_EPS, _dt(qkv), _stream())
                    else:
                        _call("svit_pool_ln_bwd", qkv.data_ptr() + off, N * D3, D3, HEAD_DIM, w32.data_ptr(),
                              fracs[which].data_ptr(), g32.data_ptr(), douts[which].data_ptr(), dpres[which].data_ptr(),
                              dqkv.data_ptr() + off, dw.data_ptr(), dg.data_ptr(), db.data_ptr(), B, h, T, H, W, O, s,
                              LN_EPS, _dt(qkv), _stream())
                grads += [dw.reshape(ctx.wshape), dg, db]
        return (dqkv, None, None, None, None, *grads, None)


def qkv_pool(qkv, thw, O, stride_q, stride_kv, pq, nq, pk, nk, pv, nv):
    """pq/pk/pv: conv weights [96,1,3,3,3]; nq/nk/nv: (gamma, beta)."""
    return _QKVPool.apply(qkv, tuple(thw), O, stride_q, stride_kv, pq, nq[0], nq[1], pk, nk[0], nk[1], pv, nv[0], nv[1],
                          torch.is_grad_enabled())


class _SkipPool(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, thw, O, s):
        _chk(x, "skip_pool")
        x = x.contiguous()
        B, N, Cn = x.shape
        T, H, W = thw
        Ho, Wo = pooled_hw(H, s), pooled_hw(W, s)
        y = torch.empty(B, 1 + T * Ho * Wo + O, Cn, dtype=x.dtype, device=x.device)
        ctx.geom = (B, Cn, T, H, W, O, s)
        ctx.in_shape = x.shape
        if x.dtype == torch.bfloat16 and Cn % 8 == 0 and ctx.needs_input_grad[0]:
            # training: record the winning window position per output element (1 byte): the backward then needs neither
            # x nor a re-scan of the windows
            idx = torch.empty(y.shape, dtype=torch.uint8, device=x.device)
            _call("svit_skip_maxpool_fwd_idx", x.data_ptr(), y.data_ptr(), idx.data_ptr(), B, Cn, T, H, W, O, s, _dt(x),
                  _stream())
            ctx.save_for_backward(idx)
            ctx.by_index = True
            return y
        _call("svit_skip_maxpool_fwd", x.data_ptr(), y.data_ptr(), B, Cn, T, H, W, O, s, _dt(x), _stream())
        ctx.save_for_backward(x)
        ctx.by_index = False
        return y

    @staticmethod
    def backward(ctx, dy):
        (saved,) = ctx.saved_tensors
        B, Cn, T, H, W, O, s = ctx.geom
        dy = dy.contiguous()
        dx = torch.empty(ctx.in_shape, dtype=dy.dtype, device=dy.device)
        if ctx.by_index:
            _call("svit_skip_maxpool_bwd_idx", saved.data_ptr(), dy.data_ptr(), dx.data_ptr(), B, Cn, T, H, W, O, s, _dt(dy),
                  _stream())
        else:
            _call("svit_skip_maxpool_bwd", saved.data_ptr(), dy.data_ptr(), dx.data_ptr(), B, Cn, T, H, W, O, s, _dt(dy),
                  _stream())
        return dx, None, None, None


def skip_pool(x, thw, O, stride_hw):
    """attention_pool(x, MaxPool3d skip) (attention.py:562-564); identity for stride 1."""
    if stride_hw == 1:
        return x
    return _SkipPool.apply(x, tuple(thw), O, stride_hw)


# --------------------------------------------------------------------------------------------
# pooled attention core
# --------------------------------------------------------------------------------------------
def _attn_args(q, k, v, Rh, Rw, Rt, out, lse, q_thw, k_thw, O, scale):
    a = AttnArgs()
    a.q, a.k, a.v = q.data_ptr(), k.data_ptr(), v.data_ptr()
    if Rh is not None:  # None: tensor-core kernels only (un-gathered table + index tables)
        a.rel_h, a.rel_w, a.rel_t = Rh.data_ptr(), Rw.data_ptr(), Rt.data_ptr()
    a.out, a.lse = out.data_ptr(), _p(lse)
    a.B, a.h = q.shape[0], q.shape[1]
    a.qt, a.qh, a.qw = q_thw
    a.kt, a.kh, a.kw = k_thw
    a.O, a.scale, a.dtype, a.impl = O, scale, _dt(q), _state["attn_impl"]
    return a


def attention_tables_only(dtype, q_thw, k_thw, O, ntab) -> bool:
    """True where forward and backward of a bf16 attention run on the tensor-core kernels alone, with the rel-pos gradient
    in table-row space: the caller then need not build the gathered tables R[a, b, :] (attention.py:116-119) at all.
    Mirrors the conditions of svit_attn_bwd_tc (attn_bwd_tc.cu); a disagreement fails loudly there (SVIT_EINVAL)."""
    if dtype != torch.bfloat16 or _state["attn_impl"] == _lib.IMPL_SIMT or not _state["attn_tab_grad"]:
        return False
    ne = k_thw[0] + k_thw[1] + k_thw[2]
    Nk = 1 + k_thw[0] * k_thw[1] * k_thw[2] + O
    ntabp, Nkp = (ntab + 7) // 8 * 8, (Nk + 7) // 8 * 8
    return ne <= 64 and ntab >= 8 and ntabp <= min(Nkp, 512) and Nkp >= 2 * HEAD_DIM and Nk <= 32768


class _Attention(torch.autograd.Function):
    @staticmethod
    def forward(ctx, q, k, v, Rh, Rw, Rt, q_thw, k_thw, O, scale, tc_tables, grad_mode, tab=None):
        _chk(q, "attention")
        q, k, v = q.contiguous(), k.contiguous(), v.contiguous()
        if Rh is None:
            assert tc_tables is not None, "attention without gathered rel-pos tables needs the tensor-core tables"
        else:
            Rh, Rw, Rt = (r.to(q.dtype).contiguous() for r in (Rh, Rw, Rt))
        B, h, Nq, d = q.shape
        assert d == HEAD_DIM, "svit_b200 attention kernels are specialised for head_dim 96"
        need = grad_mode and any(ctx.needs_input_grad[:6])
        out = torch.empty(B, Nq, h * d, dtype=q.dtype, device=q.device)
        lse = torch.empty(B, h, Nq, dtype=torch.float32, device=q.device) if need else None
        a = _attn_args(q, k, v, Rh, Rw, Rt, out, lse, q_thw, k_thw, O, scale)
        if tc_tables is not None:
            tab, ntabs, ih, iw, it, kc = tc_tables[:6]
            a.rel_tab, a.idx_h, a.idx_w, a.idx_t, a.key_cols = (tab.data_ptr(), ih.data_ptr(), iw.data_ptr(),
                                                                it.data_ptr(), kc.data_ptr())
            a.ntab_h, a.ntab_w, a.ntab_t = ntabs
            sel = tc_tables[6] if len(tc_tables) > 6 else None
            if sel is not None:  # bias-in-MMA kernel (attn_tc3.cu)
                a.sel_tab, a.sel_cols = sel.data_ptr(), sel.shape[1]
        _call("svit_attn_fwd", C.byref(a), _stream(),
              tag=f"[B{B} h{h} Nq{Nq} Nk{k.shape[2]}]" if _prof is not None else None)
        if need:
            ctx.save_for_backward(q, k, v, Rh, Rw, Rt, out, lse)
        ctx.geom = (q_thw, k_thw, O, scale)
        ctx.tc_tables = tc_tables if need else None  # the backward gets its bias terms from q . T^T (one GEMM) + the index tables
        # `tab` = the concatenated un-gathered fp32 table WITH autograd history: the backward then returns the rel-pos
        # gradient in table-row space (two tcgen05 GEMMs) and nothing for the gathered tables
        ctx.tab_grad = (need and tab is not None and tc_tables is not None and ctx.needs_input_grad[12]
                        and _state.get("attn_tab_grad", True))
        return out

    @staticmethod
    def backward(ctx, dout):
        q, k, v, Rh, Rw, Rt, out, lse = ctx.saved_tensors
        q_thw, k_thw, O, scale = ctx.geom
        dout = dout.contiguous()
        B, h, Nq, d = q.shape
        Nk = k.shape[2]
        ne = k_thw[0] + k_thw[1] + k_thw[2]
        dev = q.device
        a = _attn_args(q, k, v, Rh, Rw, Rt, out, lse, q_thw, k_thw, O, scale)
        # bf16: the contractions run as batched tcgen05 GEMMs (attn_bwd_tc.cu); fp32 parity mode: CUDA-core kernels
        tc = q.dtype == torch.bfloat16 and _state["attn_impl"] != _lib.IMPL_SIMT and ne <= 64
        # tensor-core path: whole 16-column MMA steps (the fused S / dP kernel takes the bias terms as extra K columns)
        es = (ne + 15) // 16 * 16 if tc else ne
        dq, dk, dv = torch.empty_like(q), torch.empty_like(k), torch.empty_like(v)
        d_tab = None
        ntab = sum(ctx.tc_tables[1]) if ctx.tc_tables is not None else 0
        ntabp, Nkp = (ntab + 7) // 8 * 8, (Nk + 7) // 8 * 8
        if tc and ctx.tab_grad and ntab >= 8 and ntabp <= min(Nkp, 512) and Nkp >= 2 * d:
            # table-row space (attn_bwd_tc.cu: G scatter + two GEMMs); d_rel_h / d_rel_w / d_rel_t are not written
            d_tab = torch.empty(ntab, d, dtype=torch.float32, device=dev)
        dRh = dRw = dRt = None
        if d_tab is None:
            if Rh is None:
                raise RuntimeError("attention backward: no gathered rel-pos tables and no table-row-space path for this shape")
            dR = torch.zeros(Rh.numel() + Rw.numel() + Rt.numel(), dtype=torch.float32, device=dev)  # one fill
            dRh = dR[:Rh.numel()].view(Rh.shape)
            dRw = dR[Rh.numel():Rh.numel() + Rw.numel()].view(Rw.shape)
            dRt = dR[Rh.numel() + Rw.numel():].view(Rt.shape)
        ws_e = torch.empty(B, h, Nq, es, dtype=torch.float32, device=dev)
        ws_de = torch.empty(B, h, Nq, es, dtype=torch.float32, device=dev)
        ws_delta = torch.empty(B, h, Nq, dtype=torch.float32, device=dev)
        a.dout, a.dq, a.dk, a.dv = dout.data_ptr(), dq.data_ptr(), dk.data_ptr(), dv.data_ptr()
        if dRh is not None:
            a.d_rel_h, a.d_rel_w, a.d_rel_t = dRh.data_ptr(), dRw.data_ptr(), dRt.data_ptr()
        a.ws_e, a.ws_de, a.ws_delta = ws_e.data_ptr(), ws_de.data_ptr(), ws_delta.data_ptr()
        if tc:
            Nkp = (Nk + 7) // 8 * 8
            if Nk > 4096 or _state.get("attn_bwd_unfused"):  # beyond the fused S / dP / softmax kernel's key table: fp32 scratch for the unfused path
                ws_s = torch.empty(B, h, Nq, Nkp, dtype=torch.float32, device=dev)
                ws_dp = torch.empty(B, h, Nq, Nkp, dtype=torch.float32, device=dev)
                a.ws_s, a.ws_dp = ws_s.data_ptr(), ws_dp.data_ptr()
            ws_p = torch.empty(B, h, Nq, Nkp, dtype=torch.bfloat16, device=dev)
            ws_ds = torch.empty(B, h, Nq, Nkp, dtype=torch.bfloat16, device=dev)
            ws_dq = torch.empty(B, h, Nq, d, dtype=torch.float32, device=dev)
            sel = key_select_table_bwd(tuple(k_thw), O, es, dev)
            a.ws_p, a.ws_ds, a.ws_dq = ws_p.data_ptr(), ws_ds.data_ptr(), ws_dq.data_ptr()
            a.sel_bwd, a.nep = sel.data_ptr(), es
            if ctx.tc_tables is not None:
                tab, ntabs, ih, iw, it = ctx.tc_tables[:5]
                a.rel_tab, a.idx_h, a.idx_w, a.idx_t = tab.data_ptr(), ih.data_ptr(), iw.data_ptr(), it.data_ptr()
                a.ntab_h, a.ntab_w, a.ntab_t = ntabs
                if ntab > d and ntabp <= 512:  # E_tab = q . T^T does not fit the dQ scratch
                    ws_etab = torch.empty(B, h, Nq, ntabp, dtype=torch.float32, device=dev)
                    a.ws_etab = ws_etab.data_ptr()
                if d_tab is not None:
                    a.d_rel_tab = d_tab.data_ptr()
        _call("svit_attn_bwd", C.byref(a), _stream(),
              tag=f"[B{B} h{h} Nq{Nq} Nk{Nk}]" if _prof is not None else None)
        if d_tab is not None:
            return dq, dk, dv, None, None, None, None, None, None, None, None, None, d_tab
        return dq, dk, dv, dRh, dRw, dRt, None, None, None, None, None, None, None


_sel_bwd_cache = {}


def key_select_table_bwd(k_thw, O, nep, device) -> torch.Tensor:
    """0/1 matrix [Nk, nep] (bf16): row n = key n, ones in columns i'(n), kh + j'(n), kh + kw + t'(n) for patch
    keys, zero rows for cls / object keys.  dS @ Sel = the rel-pos bias gradient dE (attention.py:121-134, 175-181
    differentiated: the bias of key (t', i', j') is E_h[i'] + E_w[j'] + E_t[t'])."""
    key = (k_thw, O, nep, str(device))
    t = _sel_bwd_cache.get(key)
    if t is None:
        kt, kh, kw = k_thw
        Nk = 1 + kt * kh * kw + O
        sel = torch.zeros(Nk, nep, dtype=torch.float32)
        p = torch.arange(kt * kh * kw)
        rows = 1 + p
        sel[rows, (p // kw) % kh] = 1.0
        sel[rows, kh + p % kw] = 1.0
        sel[rows, kh + kw + p // (kw * kh)] = 1.0
        t = sel.to(device=device, dtype=torch.bfloat16)
        _sel_bwd_cache[key] = t
    return t


def attention(q, k, v, Rh, Rw, Rt, q_thw, k_thw, O, scale, tc_tables=None, tab=None):
    """softmax(scale q k^T + rel-pos bias) v + residual pooling -> [B, Nq, h*96] (attention.py:429-461).
    Rh/Rw/Rt: gathered tables (differentiable); tc_tables: (cat table bf16, [rows], idx_h, idx_w, idx_t, key codes)
    for the tcgen05 kernel, or None; tab: the concatenated fp32 table with autograd history (optional) -- where the
    tensor-core backward supports it, the rel-pos gradient arrives through `tab` instead of Rh / Rw / Rt."""
    return _Attention.apply(q, k, v, Rh, Rw, Rt, tuple(q_thw), tuple(k_thw), O, float(scale), tc_tables,
                            torch.is_grad_enabled(), tab)


# --------------------------------------------------------------------------------------------
# stem: patch embed + token assembly; final split
# --------------------------------------------------------------------------------------------
class _PatchEmbedTokens(torch.autograd.Function):
    """x[B, 1+L+Tx*O, C] = [cls | conv3d(clip) tokens | object queries + temporal embedding]
    (stem_helper.py:309-320; video_model_builder.py:326-330, 354-363)."""

    @staticmethod
    def forward(ctx, clip, w, b, cls, queries, pos_t, kernel, stride, padding, dtype):
        _chk(clip, "patch_embed")
        clip = clip.contiguous()
        B, Cin, T, H, W = clip.shape
        kt, kh, kw = kernel
        st, sh, sw = stride
        pt, ph, pw = padding
        To, Ho, Wo = (T + 2 * pt - kt) // st + 1, (H + 2 * ph - kh) // sh + 1, (W + 2 * pw - kw) // sw + 1
        L = To * Ho * Wo
        E = w.shape[0]
        K = Cin * kt * kh * kw
        Kpad = (K + 63) // 64 * 64
        Tx, O = T, queries.shape[1]
        Ntot = 1 + L + Tx * O
        cols = torch.empty(B * L, Kpad, dtype=dtype, device=clip.device)
        odt = F32 if dtype == torch.float32 else BF16
        _call("svit_im2col3d", clip.data_ptr(), cols.data_ptr(), B, Cin, T, H, W, kt, kh, kw, st, sh, sw, pt, ph, pw,
              Kpad, _dt(clip), odt, _stream())
        w2 = _padded_weight(w, K, Kpad, dtype)
        x = torch.empty(B, Ntot, E, dtype=dtype, device=clip.device)
        gemm(cols, w2, x, B * L, E, Kpad, Kpad, Kpad, E, 0, 1, bias=_f32(b), remap=(L, Ntot, 1))
        _call("svit_assemble_tokens_fwd", x.data_ptr(), _f32(cls).data_ptr(), _f32(queries).data_ptr(),
              _f32(pos_t).data_ptr(), B, L, Tx, O, E, odt, _stream())
        ctx.save_for_backward(cols if ctx.needs_input_grad[1] else None, w)
        ctx.geom = (B, L, Tx, O, E, K, Kpad, Ntot)
        ctx.shapes = (w.shape, cls.shape, queries.shape, pos_t.shape)
        ctx.conv = (clip.shape, clip.dtype, tuple(kernel), tuple(stride), tuple(padding))
        return x

    @staticmethod
    def backward(ctx, dx):
        cols, w = ctx.saved_tensors
        B, L, Tx, O, E, K, Kpad, Ntot = ctx.geom
        wshape, cshape, qshape, pshape = ctx.shapes
        need = ctx.needs_input_grad
        dx = dx.contiguous()
        dev = dx.device
        dclip = dw = db = dcls = dq = dp = None
        if need[0]:
            dclip = patch_embed_input_grad(dx, w, *ctx.conv)
        if need[1] or need[2]:
            # patch rows of dx as a strided [B*L, E] view are not contiguous across samples -> compact copy via gather GEMM
            dpatch = dx[:, 1:1 + L].reshape(B * L, E)  # torch view/copy glue (autograd tape only)
            if need[1]:
                dw = torch.empty(E, Kpad, dtype=torch.float32, device=dev)
                gemm(dpatch, cols, dw, E, Kpad, B * L, E, Kpad, Kpad, 1, 0)
                dw = dw[:, :K].reshape(wshape)
            if need[2]:
                db = _colsum(dpatch, B * L, E)
        if any(need[3:6]):
            dcls = torch.zeros(E, dtype=torch.float32, device=dev)
            dq = torch.zeros(O * E, dtype=torch.float32, device=dev)
            dp = torch.zeros(pshape[1] * E, dtype=torch.float32, device=dev)
            _call("svit_assemble_tokens_bwd", dx.data_ptr(), dcls.data_ptr(), dq.data_ptr(), dp.data_ptr(), B, L, Tx, O, E,
                  _dt(dx), _stream())
            dcls, dq, dp = dcls.reshape(cshape), dq.reshape(qshape), dp.reshape(pshape)
        return dclip, dw, db, dcls, dq, dp, None, None, None, None


class _PatchEmbedInputGrad(torch.autograd.Function):
    """The stem when only the clip needs a gradient (a frozen model: saliency, attribution, adversarial inputs): the
    bf16 implicit-GEMM forward of inference, no im2col matrix saved, and a backward that runs the data gradient alone."""

    @staticmethod
    def forward(ctx, clip, w, b, cls, queries, pos_t, kernel, stride, padding):
        x = _patch_embed_implicit(clip, w, b, cls, queries, pos_t, kernel, stride, padding, None, None)
        ctx.save_for_backward(w)
        ctx.conv = (clip.shape, clip.dtype, kernel, stride, padding)
        return x

    @staticmethod
    def backward(ctx, dx):
        (w,) = ctx.saved_tensors
        return (patch_embed_input_grad(dx.contiguous(), w, *ctx.conv),) + (None,) * 8


def _padded_weight(w, K, Kpad, dtype):
    tag = ("pad", Kpad, dtype)
    w2 = _cache_get(w, tag)
    if w2 is None:
        w2 = torch.zeros(w.shape[0], Kpad, dtype=dtype, device=w.device)
        w2[:, :K] = w.detach().reshape(w.shape[0], K).to(dtype)
        _cache_put(w, tag, w2)
    return w2


def _floor_div(a, b):
    return a // b  # Python floors towards -inf, which is what the tap arithmetic needs


def _s2d_taps(w, stride, padding, dtype=torch.float32):
    """[E, nt, nh, nw, C, st, sh, sw] in `dtype`: the conv weight scattered into the space-to-depth taps (s2d_conv_weight)."""
    E, Cin, kt, kh, kw = w.shape
    (st, sh, sw), (pt, ph, pw) = stride, padding
    lo = [_floor_div(-p_, s_) for p_, s_ in zip((pt, ph, pw), (st, sh, sw))]
    n = [_floor_div(k_ - 1 - p_, s_) - l_ + 1 for k_, p_, s_, l_ in zip((kt, kh, kw), (pt, ph, pw), (st, sh, sw), lo)]
    W2 = torch.zeros(E, n[0], n[1], n[2], Cin, st, sh, sw, dtype=dtype, device=w.device)
    wf = w.detach().to(dtype)
    for a in range(kt):
        it, tt = _floor_div(a - pt, st) - lo[0], (a - pt) % st
        for bb in range(kh):
            ih, hh = _floor_div(bb - ph, sh) - lo[1], (bb - ph) % sh
            for c in range(kw):
                iw, ww = _floor_div(c - pw, sw) - lo[2], (c - pw) % sw
                W2[:, it, ih, iw, :, tt, hh, ww] = wf[:, :, a, bb, c]
    return W2


def s2d_conv_weight(w, stride, padding):
    """Conv3d weight [E, C, kt, kh, kw] scattered into the space-to-depth taps of csrc/patch_embed_tc.cu:
    W2[E, ((it*nh + ih)*nw + iw) * cell + ((c*st + tt)*sh + hh)*sw + ww] = w[E, c, k_t, k_h, k_w] with
    k_t - pt = (lo_t + it)*st + tt (same for h, w); positions no kernel element maps to stay zero."""
    return _s2d_taps(w, stride, padding).reshape(w.shape[0], -1).to(torch.bfloat16).contiguous()


def s2d_dgrad_weight(w, stride, padding, dtype=torch.bfloat16):
    """Weight of the transposed stem convolution (svit_patch_embed_s2d_dgrad): [cell, ntaps * E] with
    W''[cell, ((it*nh + ih)*nw + iw) * E + e] = W2[e, tap (nt-1-it, nh-1-ih, nw-1-iw), cell] -- s2d_conv_weight transposed,
    tap order reversed in every dimension.  dtype float64 builds it exactly (the host-side check of the math)."""
    taps = _s2d_taps(w, stride, padding, torch.float64 if dtype == torch.float64 else torch.float32)
    E, nt, nh, nw = taps.shape[:4]
    taps = taps.reshape(E, nt, nh, nw, -1).flip(1, 2, 3)
    return taps.permute(4, 1, 2, 3, 0).reshape(taps.shape[4], -1).to(dtype).contiguous()


def s2d_clip(clip, stride, mean=None, std=None):
    """Space-to-depth cells of a clip for the implicit-GEMM patch embed: clip [B, C, T, H, W] (fp32 / bf16) or uint8 frames
    [B, T, H, W, C] (normalised on the fly) -> bf16 [B, ceil(T/st), ceil(H/sh), ceil(W/sw), C*st*sh*sw]."""
    _chk(clip, "s2d_clip")
    clip = clip.contiguous()
    st, sh, sw = stride
    if clip.dtype == torch.uint8:
        B, T, H, W, Cin = clip.shape
        kind = 2
        m, sd = list(mean) + [0.0] * 3, list(std) + [1.0] * 3
    else:
        B, Cin, T, H, W = clip.shape
        kind = _dt(clip)
        m, sd = [0.0] * 3, [1.0] * 3
    cells = torch.empty(B, -(-T // st), -(-H // sh), -(-W // sw), Cin * st * sh * sw, dtype=torch.bfloat16, device=clip.device)
    _call("svit_s2d_clip", clip.data_ptr(), cells.data_ptr(), B, Cin, T, H, W, st, sh, sw, kind, float(m[0]), float(m[1]),
          float(m[2]), float(sd[0]), float(sd[1]), float(sd[2]), _stream())
    return cells


def _patch_embed_implicit(clip, w, b, cls, queries, pos_t, kernel, stride, padding, mean, std):
    """Inference path: conv3d as an implicit GEMM over space-to-depth cells (no im2col matrix), then cls / object rows."""
    if clip.dtype == torch.uint8:
        B, T, H, W, Cin = clip.shape
    else:
        B, Cin, T, H, W = clip.shape
    kt, kh, kw = kernel
    st, sh, sw = stride
    pt, ph, pw = padding
    To, Ho, Wo = (T + 2 * pt - kt) // st + 1, (H + 2 * ph - kh) // sh + 1, (W + 2 * pw - kw) // sw + 1
    L = To * Ho * Wo
    E = w.shape[0]
    Tx, O = T, queries.shape[1]
    Ntot = 1 + L + Tx * O
    cells = s2d_clip(clip, stride, mean, std)
    tag = ("s2d", tuple(stride), tuple(padding))
    w2 = _cache_get(w, tag)
    if w2 is None:
        w2 = _cache_put(w, tag, s2d_conv_weight(w, stride, padding))
    x = torch.empty(B, Ntot, E, dtype=torch.bfloat16, device=clip.device)
    _call("svit_patch_embed_s2d", cells.data_ptr(), w2.data_ptr(), _f32(b).data_ptr(), x.data_ptr(), Ntot * E, 1, B, Cin, T, H, W,
          kt, kh, kw, st, sh, sw, pt, ph, pw, E, _stream(), tag=f"[B{B} {T}x{H}x{W}]" if _prof is not None else None)
    _call("svit_assemble_tokens_fwd", x.data_ptr(), _f32(cls).data_ptr(), _f32(queries).data_ptr(),
          _f32(pos_t).data_ptr(), B, L, Tx, O, E, BF16, _stream())
    return x


def d2s_clip(cells, clip_shape, stride, dtype):
    """Inverse of s2d_clip: bf16 cells [B, Tc, Hc, Wc, C*st*sh*sw] -> clip [B, C, T, H, W] in `dtype` (fp32 / bf16)."""
    _chk(cells, "d2s_clip")
    cells = cells.contiguous()
    B, Cin, T, H, W = clip_shape
    x = torch.empty(clip_shape, dtype=dtype, device=cells.device)
    _call("svit_d2s_clip", cells.data_ptr(), x.data_ptr(), B, Cin, T, H, W, *stride, _dt(x), _stream())
    return x


def patch_embed_input_grad(dx, w, clip_shape, clip_dtype, kernel, stride, padding):
    """Gradient of the stem with respect to the clip [B, C, T, H, W] (in clip_dtype) from the sequence gradient
    dx [B, 1 + L + Tx*O, E] (patch rows 1..L).  bf16 runs the transposed convolution on the tensor cores
    (input_grad_s2d); fp32, and a geometry that kernel does not cover, run input_grad_col2im."""
    Cin = clip_shape[1]
    if dx.dtype == torch.bfloat16 and _lib.lib().svit_patch_embed_s2d_dgrad_supported(Cin, *kernel, *stride, *padding,
                                                                                        w.shape[0]):
        return input_grad_s2d(dx, w, clip_shape, clip_dtype, kernel, stride, padding)
    return input_grad_col2im(dx, w, clip_shape, clip_dtype, kernel, stride, padding)


def input_grad_s2d(dx, w, clip_shape, clip_dtype, kernel, stride, padding):
    """bf16 dx: svit_patch_embed_s2d_dgrad reads the patch rows of dx in place (implicit GEMM over the cell grid, the
    weight s2d_dgrad_weight cached per parameter version), then svit_d2s_clip."""
    _chk(dx, "input_grad_s2d")
    B, Cin, T, H, W = clip_shape
    st, sh, sw = stride
    E, Ntot = w.shape[0], dx.shape[1]
    tag = ("s2d_dgrad", tuple(stride), tuple(padding))
    wt = _cache_get(w, tag)
    if wt is None:
        wt = _cache_put(w, tag, s2d_dgrad_weight(w, stride, padding).to(dx.device))
    dcells = torch.empty(B, -(-T // st), -(-H // sh), -(-W // sw), Cin * st * sh * sw, dtype=torch.bfloat16, device=dx.device)
    _call("svit_patch_embed_s2d_dgrad", dx.data_ptr(), Ntot * E, 1, wt.data_ptr(), dcells.data_ptr(), B, Cin, T, H, W,
          *kernel, *stride, *padding, E, _stream(), tag=f"[B{B} {T}x{H}x{W}]" if _prof is not None else None)
    return d2s_clip(dcells, clip_shape, stride, clip_dtype)


def input_grad_col2im(dx, w, clip_shape, clip_dtype, kernel, stride, padding):
    """dcols = dpatch . W on svit_gemm (fp32 output; CUDA cores in the fp32 parity mode), then the svit_col2im3d gather."""
    _chk(dx, "input_grad_col2im")
    B, Cin, T, H, W = clip_shape
    kt, kh, kw = kernel
    st, sh, sw = stride
    pt, ph, pw = padding
    E = w.shape[0]
    L = ((T + 2 * pt - kt) // st + 1) * ((H + 2 * ph - kh) // sh + 1) * ((W + 2 * pw - kw) // sw + 1)
    K = Cin * kt * kh * kw
    Kpad = (K + 63) // 64 * 64
    dpatch = dx[:, 1:1 + L].reshape(B * L, E)  # torch view/copy glue: the patch rows, compact
    dcols = torch.empty(B * L, Kpad, dtype=torch.float32, device=dx.device)
    gemm(dpatch, _padded_weight(w, K, Kpad, dx.dtype), dcols, B * L, Kpad, E, E, Kpad, Kpad, 0, 0)
    dclip = torch.empty(clip_shape, dtype=clip_dtype, device=dx.device)
    _call("svit_col2im3d", dcols.data_ptr(), dclip.data_ptr(), B, Cin, T, H, W, *kernel, *stride, *padding, Kpad, F32,
          _dt(dclip), _stream())
    return dclip


def patch_embed_tokens(clip, w, b, cls, queries, pos_t, kernel, stride, padding, dtype, mean=None, std=None):
    """[cls | conv3d(clip) patch tokens | object queries + temporal embedding].  clip: [B, C, T, H, W] (fp32 / bf16) or
    decoded uint8 frames [B, T, H, W, C].  Without autograd and in bf16 the stem is an implicit GEMM
    (csrc/patch_embed_tc.cu); with autograd (the weight gradient needs the im2col matrix) or in the fp32 parity mode it is
    svit_im2col3d + svit_gemm.  A clip that requires grad receives its gradient (patch_embed_input_grad); when no stem
    parameter needs one (a frozen model), bf16 keeps the implicit-GEMM forward and the backward runs the data gradient
    alone.  uint8 frames are not differentiable."""
    kernel, stride, padding = tuple(kernel), tuple(stride), tuple(padding)
    Cin = clip.shape[-1] if clip.dtype == torch.uint8 else clip.shape[1]
    needs_grad = torch.is_grad_enabled() and any(t.requires_grad for t in (w, b, cls, queries, pos_t))
    clip_grad = torch.is_grad_enabled() and clip.requires_grad
    implicit = (dtype == torch.bfloat16 and _state.get("implicit_patch_embed", True)
                and _lib.lib().svit_patch_embed_s2d_supported(Cin, *kernel, *stride, *padding, w.shape[0]))
    if implicit and not needs_grad:
        if clip_grad:
            return _PatchEmbedInputGrad.apply(clip, w, b, cls, queries, pos_t, kernel, stride, padding)
        return _patch_embed_implicit(clip, w, b, cls, queries, pos_t, kernel, stride, padding, mean, std)
    if clip.dtype == torch.uint8:
        clip = normalize_u8(clip, mean, std, torch.float32 if dtype == torch.float32 else torch.bfloat16)
    return _PatchEmbedTokens.apply(clip, w, b, cls, queries, pos_t, kernel, stride, padding, dtype)


class _GatherClsObj(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, O):
        _chk(x, "gather_cls_obj")
        x = x.contiguous()
        B, N, Cn = x.shape
        out = torch.empty(B, 1 + O, Cn, dtype=x.dtype, device=x.device)
        _call("svit_gather_cls_obj_fwd", x.data_ptr(), out.data_ptr(), B, N, O, Cn, _dt(x), _stream())
        ctx.geom = (B, N, O, Cn)
        return out

    @staticmethod
    def backward(ctx, dout):
        B, N, O, Cn = ctx.geom
        dout = dout.contiguous()
        dx = torch.empty(B, N, Cn, dtype=dout.dtype, device=dout.device)
        _call("svit_gather_cls_obj_bwd", dout.data_ptr(), dx.data_ptr(), B, N, O, Cn, _dt(dout), _stream())
        return dx, None


def gather_cls_obj(x, O):
    """[cls ; object tokens] of the final sequence (video_model_builder.py:377-384)."""
    return _GatherClsObj.apply(x, O)


# --------------------------------------------------------------------------------------------
# box-conditioned object tokens (inference path), integer box logic on device
# --------------------------------------------------------------------------------------------
class _RoITokens(torch.autograd.Function):
    """Per-frame box-conditioned object tokens (call site video_model_builder.py:385-392, 472-491; SURVEY R3).

    mode None      -> tokens [B, Tx*K, C]
    mode "replace" -> a copy of the sequence whose object rows 1 + T'H'W' + t*K + k hold the RoI tokens
    mode "add"     -> the same rows hold (learned object token + RoI token)
    Backward: the token gradients go to the arg-max bin's bilinear taps (svit_roi_tokens_bwd, fp32 atomics)."""

    @staticmethod
    def forward(ctx, x_tokens, boxes, thw, patch_stride_t, spatial_scale, out_size, mode):
        _chk(x_tokens, "roi_tokens")
        x_tokens = x_tokens.contiguous()
        B, N, Cn = x_tokens.shape
        Tf, Hf, Wf = thw
        L = Tf * Hf * Wf
        _, Tx, K, _ = boxes.shape
        bx = boxes.to(device=x_tokens.device, dtype=torch.float32).contiguous()
        need = ctx.needs_input_grad[0]
        argmax = torch.empty(B * Tx * K, Cn, dtype=torch.uint8, device=x_tokens.device) if need else None
        assign = torch.empty(B, Tx * K, 2, dtype=torch.int32, device=x_tokens.device)
        if mode is None:
            out = torch.empty(B, Tx * K, Cn, dtype=x_tokens.dtype, device=x_tokens.device)
            optr, obs, acc = out.data_ptr(), 0, 0
        else:
            if mode not in ("replace", "add"):
                raise ValueError(f"roi token scatter mode {mode!r}: expected 'replace' or 'add'")
            if N - 1 - L != Tx * K:
                raise ValueError(f"scattering {Tx}x{K} RoI tokens needs {Tx * K} object rows, the sequence has {N - 1 - L}")
            out = x_tokens.clone()
            optr, obs, acc = out.data_ptr() + (1 + L) * Cn * out.element_size(), N * Cn, int(mode == "add")
        _call("svit_roi_tokens_fwd", x_tokens.data_ptr(), N * Cn, bx.data_ptr(), optr, obs, _p(argmax), acc,
              assign.data_ptr(), B, Cn, Tf, Hf, Wf, Tx, K, patch_stride_t, float(spatial_scale), out_size, _dt(x_tokens),
              _stream())
        if need:
            ctx.save_for_backward(bx, argmax)
        ctx.geom = (B, N, Cn, Tf, Hf, Wf, Tx, K, patch_stride_t, float(spatial_scale), out_size, mode)
        ctx.mark_non_differentiable(assign)
        return out, assign

    @staticmethod
    def backward(ctx, dout, _dassign):
        bx, argmax = ctx.saved_tensors
        B, N, Cn, Tf, Hf, Wf, Tx, K, pst, scale, P, mode = ctx.geom
        L = Tf * Hf * Wf
        dout = dout.contiguous()
        dfeat = torch.zeros(B, L, Cn, dtype=torch.float32, device=dout.device)
        if mode is None:
            dptr, dbs = dout.data_ptr(), 0
        else:
            dptr, dbs = dout.data_ptr() + (1 + L) * Cn * dout.element_size(), N * Cn
        _call("svit_roi_tokens_bwd", dptr, dbs, argmax.data_ptr(), bx.data_ptr(), dfeat.data_ptr(), B, Cn, Tf, Hf, Wf, Tx, K,
              pst, scale, P, _dt(dout), _stream())
        if mode is None:
            dx = torch.zeros(B, N, Cn, dtype=dout.dtype, device=dout.device)
        else:
            dx = dout.clone()
            if mode == "replace":
                dx[:, 1 + L:].zero_()  # the learned object rows were overwritten
        dx[:, 1:1 + L] += dfeat.to(dx.dtype)  # [B, T'H'W', C] glue add (the atomics accumulate in fp32)
        return dx, None, None, None, None, None, None


def roi_tokens(x_tokens, thw, boxes, patch_stride_t=2, spatial_scale=1.0 / 16, out_size=7):
    """x_tokens [B, N, C] (token-major, patch rows 1..T'H'W'); boxes [B, Tx, K, 4] xyxy pixels.
    Returns (tokens [B, Tx*K, C], assign int32 [B, Tx*K, 2] = (batch, temporal slice)); differentiable in x_tokens."""
    return _RoITokens.apply(x_tokens, boxes, tuple(thw), patch_stride_t, spatial_scale, out_size, None)


def roi_scatter_tokens(x_tokens, thw, boxes, patch_stride_t=2, spatial_scale=1.0 / 16, out_size=7, mode="replace"):
    """The sequence with its object rows (index 1 + T'H'W' + t*K + k, SURVEY R3 / video_model_builder.py:354-363) replaced
    by -- or, mode="add", summed with -- the box-conditioned RoI tokens.  Returns (sequence [B, N, C], assign)."""
    return _RoITokens.apply(x_tokens, boxes, tuple(thw), patch_stride_t, spatial_scale, out_size, mode)


def roi_align_nhwc(feat_nhwc, rois, out_size, spatial_scale, sampling_ratio=0, aligned=True):
    _chk(feat_nhwc, "roi_align")
    feat_nhwc = feat_nhwc.contiguous()
    Nn, H, W, Cn = feat_nhwc.shape
    r = rois.to(device=feat_nhwc.device, dtype=torch.float32).contiguous()
    R = r.shape[0]
    out = torch.empty(R, out_size, out_size, Cn, dtype=feat_nhwc.dtype, device=feat_nhwc.device)
    _call("svit_roi_align_fwd", feat_nhwc.data_ptr(), r.data_ptr(), out.data_ptr(), Nn, Cn, H, W, R, out_size,
          float(spatial_scale), sampling_ratio, int(aligned), _dt(feat_nhwc), _stream())
    return out


def normalize_u8(frames: torch.Tensor, mean, std, dtype=torch.bfloat16) -> torch.Tensor:
    """uint8 frames [B, T, H, W, 3] -> normalised clip [B, 3, T, H, W] (datasets/utils.py:287-303 + the THWC -> CTHW
    permute of the loaders) in one streaming kernel; the uint8 tensor is what crosses PCIe."""
    if frames.dtype != torch.uint8 or frames.dim() != 5 or frames.shape[-1] != 3:
        raise ValueError("normalize_u8 expects uint8 [B, T, H, W, 3]")
    _chk(frames, "normalize_u8")
    frames = frames.contiguous()
    B, T, H, W, _ = frames.shape
    out = torch.empty(B, 3, T, H, W, dtype=dtype, device=frames.device)
    _call("svit_normalize_u8", frames.data_ptr(), out.data_ptr(), B, T, H, W, float(mean[0]), float(mean[1]), float(mean[2]),
          float(std[0]), float(std[1]), float(std[2]), _dt(out), _stream())
    return out


def match_haog_device(boxes):
    """boxes [n,4,4] fp32 CUDA (modified in place) -> contact [n,2] int64 (utils/box_ops.py:140-194)."""
    _chk(boxes, "match_haog")
    assert boxes.dtype == torch.float32 and boxes.is_contiguous()
    n = boxes.shape[0]
    contact = torch.empty(n, 2, dtype=torch.int64, device=boxes.device)
    _call("svit_match_haog", boxes.data_ptr(), contact.data_ptr(), n, _stream())
    return boxes, contact


def zero_empty_boxes_device(boxes, eps=0.05):
    _chk(boxes, "zero_empty_boxes")
    assert boxes.dtype == torch.float32 and boxes.is_contiguous()
    _call("svit_zero_empty_boxes", boxes.data_ptr(), boxes.numel() // 4, float(eps), _stream())
    return boxes


# --------------------------------------------------------------------------------------------
# head (inference) and HAOG losses (SURVEY 8f N2)
# --------------------------------------------------------------------------------------------
def head_forward(x, wp, bp, wb, bb, ws, bs, wc, bc, Tx, O, act_sigmoid=False, eval_mode=True, want_probs=True):
    """SViTHead.forward without autograd in one launch (video_model_builder.py:507-546).
    x [B, 1 + Tx*O, C].  Returns (logits, probs | None, obj_desc, pred_bboxes, pred_contact), all fp32."""
    _chk(x, "head_forward")
    x = x.contiguous()
    B, R, Cn = x.shape
    assert R == 1 + Tx * O
    NC = wp.shape[0]
    dev = x.device
    logits = torch.empty(B, NC, dtype=torch.float32, device=dev)
    probs = torch.empty(B, NC, dtype=torch.float32, device=dev) if want_probs else None
    obj = torch.empty(B, Tx, O, Cn, dtype=torch.float32, device=dev)
    boxes = torch.empty(B, Tx, O, 5, dtype=torch.float32, device=dev)
    contact = torch.empty(B, Tx, 2, 5, dtype=torch.float32, device=dev)
    ws_ = [_f32(t) for t in (wp, bp, wb, bb, ws, bs, wc, bc)]
    _call("svit_head_fwd", x.data_ptr(), *[t.data_ptr() for t in ws_], logits.data_ptr(), _p(probs), obj.data_ptr(),
          boxes.data_ptr(), contact.data_ptr(), B, Tx, O, Cn, NC, int(act_sigmoid), int(eval_mode), _dt(x), _stream())
    return logits, probs, obj, boxes, contact


class _HaogLoss(torch.autograd.Function):
    """(l1, bce, giou, contact ce) of VideoImageLoss._haog_loss (models/losses.py:50-92, 138-155) in one launch; the
    same launch produces the gradient of every term, so backward is four tiny scaled adds."""

    @staticmethod
    def forward(ctx, pred_bboxes, tar_boxes, pred_contact, tar_contact):
        _chk(pred_bboxes, "haog_loss")
        pb = pred_bboxes.detach().float().contiguous().reshape(-1, 5)
        tb = tar_boxes.detach().to(device=pb.device, dtype=torch.float32).contiguous()
        tcols = tb.shape[-1]
        tb = tb.reshape(-1, tcols)
        pc = pred_contact.detach().float().contiguous().reshape(-1, 5)
        tcn = tar_contact.detach().to(device=pb.device, dtype=torch.int64).contiguous().reshape(-1)
        N, M = pb.shape[0], pc.shape[0]
        out = torch.empty(4, dtype=torch.float32, device=pb.device)
        d_l1 = torch.empty(N, 4, dtype=torch.float32, device=pb.device)
        d_giou = torch.empty(N, 4, dtype=torch.float32, device=pb.device)
        d_bce = torch.empty(N, dtype=torch.float32, device=pb.device)
        d_ce = torch.empty(M, 5, dtype=torch.float32, device=pb.device)
        _call("svit_haog_loss", pb.data_ptr(), tb.data_ptr(), tcols, N, pc.data_ptr(), tcn.data_ptr(), M, out.data_ptr(),
              d_l1.data_ptr(), d_bce.data_ptr(), d_giou.data_ptr(), d_ce.data_ptr(), _stream())
        ctx.save_for_backward(d_l1, d_bce, d_giou, d_ce)
        ctx.shapes = (pred_bboxes.shape, pred_contact.shape, pred_bboxes.dtype, pred_contact.dtype)
        return out[0], out[1], out[2], out[3]

    @staticmethod
    def backward(ctx, g_l1, g_bce, g_giou, g_ce):
        d_l1, d_bce, d_giou, d_ce = ctx.saved_tensors
        bshape, cshape, bdt, cdt = ctx.shapes
        dboxes = torch.cat([(g_bce * d_bce).unsqueeze(-1), g_l1 * d_l1 + g_giou * d_giou], dim=-1)
        return dboxes.reshape(bshape).to(bdt), None, (g_ce * d_ce).reshape(cshape).to(cdt), None


def haog_loss(pred_bboxes, tar_boxes, pred_contact, tar_contact):
    """Returns (boxes_l1_loss, boxes_bce_loss, boxes_giou_loss, loss_contact_state) as device scalars."""
    return _HaogLoss.apply(pred_bboxes, tar_boxes, pred_contact, tar_contact)


# --------------------------------------------------------------------------------------------
# input side on the GPU (SURVEY 8f N4): crop + flip + normalise, boxes follow the frames
# --------------------------------------------------------------------------------------------
def _i32(v, n, device):
    t = torch.as_tensor(v, dtype=torch.int32)
    if t.dim() == 0:
        t = t.expand(n)
    return t.to(device).contiguous()


def crop_flip_normalize_u8(frames, x_off, y_off, flip, crop, mean, std, dtype=torch.bfloat16):
    """uint8 frames [B, T, H, W, 3] -> normalised clip [B, 3, T, crop, crop]: per-sample crop at (x_off[b], y_off[b])
    (transform.py:154-190), horizontal flip where flip[b] (transform.py:248-285), (x / 255 - mean) / std
    (datasets/utils.py:287-303), CTHW layout -- one streaming kernel; fp32 output bit-identical to the reference ops."""
    if frames.dtype != torch.uint8 or frames.dim() != 5 or frames.shape[-1] != 3:
        raise ValueError("crop_flip_normalize_u8 expects uint8 [B, T, H, W, 3]")
    _chk(frames, "crop_flip_normalize_u8")
    frames = frames.contiguous()
    B, T, H, W, _ = frames.shape
    ch, cw = (crop, crop) if isinstance(crop, int) else crop
    xo, yo = _i32(x_off, B, frames.device), _i32(y_off, B, frames.device)
    fl = _i32(flip, B, frames.device) if flip is not None else None
    if int(xo.max()) + cw > W or int(yo.max()) + ch > H or int(xo.min()) < 0 or int(yo.min()) < 0:
        raise ValueError("crop window leaves the frame")
    out = torch.empty(B, 3, T, ch, cw, dtype=dtype, device=frames.device)
    _call("svit_crop_flip_normalize_u8", frames.data_ptr(), out.data_ptr(), xo.data_ptr(), yo.data_ptr(), _p(fl), B, T, H, W,
          ch, cw, float(mean[0]), float(mean[1]), float(mean[2]), float(std[0]), float(std[1]), float(std[2]), _dt(out),
          _stream())
    return out


def boxes_crop_flip(boxes_xyxy, x_off, y_off, flip, crop, eps=0.05):
    """boxes [B, ..., 4] xyxy pixels of the un-cropped frames -> the loss's targets [B, ..., 4] cxcywh in [0, 1] for the
    cropped / flipped clip, boxes thinner than eps zeroed (transform.py:107-132, 248-285; ssv2_frames.py:347-353)."""
    _chk(boxes_xyxy, "boxes_crop_flip")
    b = boxes_xyxy.to(torch.float32).contiguous()
    B = b.shape[0]
    per = b[0].numel() // 4 if B else 0
    ch, cw = (crop, crop) if isinstance(crop, int) else crop
    xo, yo = _i32(x_off, B, b.device), _i32(y_off, B, b.device)
    fl = _i32(flip, B, b.device) if flip is not None else None
    out = torch.empty_like(b)
    _call("svit_boxes_crop_flip", b.data_ptr(), out.data_ptr(), xo.data_ptr(), yo.data_ptr(), _p(fl), B, per, ch, cw,
          float(eps), _stream())
    return out
