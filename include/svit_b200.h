/* svit_b200 -- C ABI of the B200 (sm_100a) kernels behind the SViT pooled-attention hot path.
 *
 * The reference (eladb3/SViT) is pure Python: its "FFI" for this path is the set of torch ops that
 * slowfast/models/attention.py, stem_helper.py, common.py and video_model_builder.py dispatch.  Each
 * entry point below replaces one of those op sites (cited per function); the Python host code in
 * svit_b200/ binds them with ctypes (see INTEGRATION.md for the stub a maintainer would add).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer owned by the caller (PyTorch allocates; the library allocates
 *     nothing persistent and keeps no state except cached TMA descriptors, freed by svit_destroy()).
 *   - `stream` is a cudaStream_t; calls are asynchronous, never synchronise, and are graph-capturable.
 *   - return value: 0 = ok, < 0 = argument error (SVIT_EINVAL -1, SVIT_ENOTSUP -2), > 0 = cudaError_t.
 *   - dtype: SVIT_F32 (0) or SVIT_BF16 (1) = storage type of activations; arithmetic is fp32 (SIMT path)
 *     or bf16 x bf16 -> fp32 (tcgen05 path).  Parameters (LN affine, conv taps, biases) are fp32.
 *   - token layout of every sequence: [cls | T*H*W patch tokens (t, h, w row-major) | O object tokens].
 *   - no CPU fallback exists.
 */
#ifndef SVIT_B200_H
#define SVIT_B200_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SVIT_DTYPE_F32 0
#define SVIT_DTYPE_BF16 1

/* Library / build identification: returns the compiled arch (100 for sm_100a). */
int svit_abi_version(void);
int svit_destroy(void);

/* ---- LayerNorm(C, eps) over tokens: attention.py:558,566 (norm1/norm2), video_model_builder.py:375 (norm).
 * mean/rstd ([rows], fp32) may be NULL in inference. */
int svit_layernorm_fwd(const void* x, const float* gamma, const float* beta, void* y, float* mean, float* rstd,
                       int64_t rows, int C, float eps, int dtype, void* stream);
/* dgamma/dbeta are accumulated into (+=). */
int svit_layernorm_bwd(const void* dy, const void* x, const float* gamma, const float* mean, const float* rstd,
                       void* dx, float* dgamma, float* dbeta, int64_t rows, int C, int dtype, void* stream);

/* ---- attention_pool with a Conv3d pool + LayerNorm: attention.py:13-65 (called at :368-388).
 * in: token (b, n) of head hd starts at in + b*in_batch_stride + n*in_tok_stride + hd*in_head_stride
 *     (element strides; lets the kernel read q/k/v slices of the packed qkv GEMM output in place).
 * conv_w [96*27] = pool.weight.reshape(96, 27); tap_frac [27] = fraction of the conv outputs of a 3x3x3
 * constant cube for which each tap is in bounds (host-computed geometry constant; w_eff = conv_w . tap_frac).
 * out [B, h, 1 + T*Ho*Wo + O, 96], Ho = (H-1)/stride_hw + 1. */
int svit_pool_ln_fwd(const void* in, int64_t in_batch_stride, int64_t in_tok_stride, int64_t in_head_stride,
                     const float* conv_w, const float* tap_frac, const float* gamma, const float* beta, void* out,
                     int B, int h, int T, int H, int W, int O, int stride_hw, float eps, int dtype, void* stream);
/* dpre: scratch shaped like `out`; dz written with the strides of `in`; dw[96*27], dgamma, dbeta += . */
int svit_pool_ln_bwd(const void* in, int64_t in_batch_stride, int64_t in_tok_stride, int64_t in_head_stride,
                     const float* conv_w, const float* tap_frac, const float* gamma, const void* dout, void* dpre,
                     void* dz, float* dw, float* dgamma, float* dbeta, int B, int h, int T, int H, int W, int O,
                     int stride_hw, float eps, int dtype, void* stream);
/* Training variants (bf16 only, else SVIT_ENOTSUP): the forward also writes the pre-LayerNorm rows to `pre` (shape of out)
 * and the backward reads them instead of recomputing the convolution per output token. */
int svit_pool_ln_fwd_save(const void* in, int64_t in_batch_stride, int64_t in_tok_stride, int64_t in_head_stride,
                          const float* conv_w, const float* tap_frac, const float* gamma, const float* beta, void* out,
                          void* pre, int B, int h, int T, int H, int W, int O, int stride_hw, float eps, int dtype,
                          void* stream);
int svit_pool_ln_bwd_saved(const void* in, int64_t in_batch_stride, int64_t in_tok_stride, int64_t in_head_stride,
                           const float* conv_w, const float* tap_frac, const float* gamma, const void* dout,
                           const void* pre, void* dpre, void* dz, float* dw, float* dgamma, float* dbeta, int B, int h,
                           int T, int H, int W, int O, int stride_hw, float eps, int dtype, void* stream);

/* ---- skip-path attention_pool with MaxPool3d k(1,3,3) s(1,s,s) p(0,1,1): attention.py:503-505,549-555,562-564.
 * x [B, 1+T*H*W+O, C] -> y [B, 1+T*Ho*Wo+O, C]; cls and object rows are copied. stride_hw must be >= 2. */
int svit_skip_maxpool_fwd(const void* x, void* y, int B, int C, int T, int H, int W, int O, int stride_hw, int dtype,
                          void* stream);
int svit_skip_maxpool_bwd(const void* x, const void* dy, void* dx, int B, int C, int T, int H, int W, int O,
                          int stride_hw, int dtype, void* stream);
/* Training variant (bf16, C % 8 == 0, else SVIT_ENOTSUP): the forward also records, per output element, which of the nine
 * window positions won (idx [B, 1+T*Ho*Wo+O, C] bytes, first maximum in ATen's scan order); the backward reads idx
 * instead of x and re-scanning the windows. */
int svit_skip_maxpool_fwd_idx(const void* x, void* y, void* idx, int B, int C, int T, int H, int W, int O, int stride_hw,
                              int dtype, void* stream);
int svit_skip_maxpool_bwd_idx(const void* idx, const void* dy, void* dx, int B, int C, int T, int H, int W, int O,
                              int stride_hw, int dtype, void* stream);

/* ---- GEMM with fused epilogue: nn.Linear sites attention.py:345 (qkv), :462 (proj), :561 (skip proj),
 * common.py:27-34 (fc1+GELU, fc2), stem_helper.py:317 (patch embed as im2col GEMM), and their gradients.
 *   C[M,N] = residual + sample_scale[row / rows_per_sample] * ( act(op(A).op(B) + bias) * gelu'(gelu_pre) )
 * Row-major storage.  transA=0: A is [M,K] (lda); 1: A is [K,M].  transB=1: B is [N,K] (nn.Linear weight); 0: [K,N].
 * Output row remap (rows_in > 0): row m -> (m / rows_in) * rows_out + row_off + m % rows_in (writes patch tokens
 * straight into rows 1..L of the [B, 1+L+O, C] sequence; residual uses the remapped row). */
typedef struct svit_gemm_args {
  const void* A;
  const void* B;
  void* C;
  int64_t M, N, K, lda, ldb, ldc;
  int32_t transA, transB;
  const float* bias;         /* [N] or NULL */
  const void* residual;      /* [*, N] (ldr), activation dtype, or NULL */
  int64_t ldr;
  const float* sample_scale; /* DropPath mask / keep_prob per sample, or NULL (common.py:46-59) */
  int64_t rows_per_sample;
  const void* gelu_pre;      /* multiply by gelu'(gelu_pre[m,n]) (ldg): backward through common.py:31 */
  int64_t ldg;
  void* pre_out;             /* store the pre-activation (after bias) for that backward (ldp), or NULL */
  int64_t ldp;
  int32_t act;               /* 0 none, 1 exact-erf GELU */
  int64_t rows_in, rows_out, row_off;
  int32_t dtype;             /* dtype of A, B, residual, gelu_pre, pre_out */
  int32_t out_dtype;         /* dtype of C */
  int32_t impl;              /* 0 auto (tcgen05 when bf16 and the shape qualifies), 1 CUDA cores, 2 tcgen05 */
  /* batched form (tcgen05 path only; batch <= 1 = plain GEMM): problem i uses A + i*strideA, C + i*strideC and
   * B + (i / b_inner)*strideB + (i % b_inner)*strideB_inner (two-level batch index, e.g. (sample, head) slices of a
   * [B, N, h, 96] tensor); strides in elements.  No epilogue extras except bias. */
  int64_t batch, strideA, strideB, strideC;
  int64_t b_inner, strideB_inner;
  /* same two-level split for A: A + (i / a_inner)*strideA + (i % a_inner)*strideA_inner when a_inner > 1 */
  int64_t a_inner, strideA_inner;
  float alpha;               /* accumulator scale applied before the bias; 0 is read as 1 (tcgen05 path only) */
  /* LayerNorm folded into the GEMM (inference; tcgen05 TMA-store kernel only, else SVIT_ENOTSUP; K-major B, no
   * residual / gelu_pre / sample_scale): A holds the UN-normalised rows x, B the weight scaled by gamma
   * (W' = W diag(gamma)), ln_stats [M, 2] = (mean, rstd) of every row (svit_row_stats), ln_colsum [N / 2][4] the
   * interleaved table (c[2i], c[2i+1], b'[2i], b'[2i+1]) with c[n] = sum_k W'[n, k] and b' = bias + W beta (`bias` itself
   * is ignored).  The epilogue computes rstd * (acc - mean * c[n]) + b'[n] = LayerNorm(x) W^T + bias
   * (attention.py:558-561, 566-567). */
  const float* ln_stats;
  const float* ln_colsum;
} svit_gemm_args;
int svit_gemm(const svit_gemm_args* args, void* stream);
/* stats[m] = (mean, 1 / sqrt(var + eps)) of row m of x [M, C] (fp32 pair per row): the LayerNorm statistics a folded
 * GEMM needs (half the traffic of a LayerNorm pass: the rows are read, nothing is written back) */
int svit_row_stats(const void* x, float* stats, int64_t M, int C, float eps, int dtype, void* stream);
/* Fused MLP (inference): out = residual + fc2(gelu(fc1(LN(x)))) with the hidden activation kept on chip (TMEM -> shared
 * memory), replacing the two svit_gemm calls of Mlp.forward (common.py:27-34), the residual add and -- optionally -- the
 * norm2 launch of MultiScaleBlock.forward (attention.py:566-570).  x [M, C], w1 [H, C], w2 [N, H], residual / out [M, N]:
 * bf16; b1 [H], b2 [N]: fp32; residual may be NULL; out must not alias x or residual.  ln_gamma / ln_beta [C] fp32 (both or neither): x is normalised on the
 * fly (LayerNorm over C, eps) and residual must then be x itself or NULL.  Supported:
 * (C, H, N) = (96, 384, 96), both weight matrices resident in shared memory; else SVIT_ENOTSUP. */
int svit_mlp_fused_supported(int64_t M, int C, int H, int N);
int svit_mlp_fused(const void* x, const void* w1, const float* b1, const void* w2, const float* b2, const void* residual,
                   void* out, int64_t M, int C, int H, int N, const float* ln_gamma, const float* ln_beta, float eps,
                   void* stream);
/* out[n] += sum_m x[m,n]  (bias gradients) */
int svit_colsum(const void* x, float* out, int64_t M, int N, int64_t ld, int dtype, void* stream);

/* ---- pooled attention core: attention.py:429-459 with cal_rel_pos_spatial (:84-137) and
 * cal_rel_pos_temporal (:140-183) fused into the score tile and the residual-pooling add (:455-459).
 *   S = scale * q k^T ; S[patch q, patch k] += q . (Rh[i,i'] + Rw[j,j'] + Rt[t,t']) (un-scaled q)
 *   out = softmax(S) v ; out[rows >= 1] += q
 * q [B,h,Nq,96], k/v [B,h,Nk,96]; rel_* are the GATHERED tables R[a, b, :] (activation dtype), built on the host
 * side with the reference's exact fp32 index expression; out [B, Nq, h, 96] (heads merged). lse [B,h,Nq] or NULL.
 * rel_* (and d_rel_*) may be NULL where only the tensor-core kernels run: the forward with rel_tab / idx_* present, the
 * backward with d_rel_tab; a call that would need them on a CUDA-core path returns SVIT_EINVAL. */
typedef struct svit_attn_args {
  const void* q;
  const void* k;
  const void* v;
  const void* rel_h; /* [qh, kh, 96] */
  const void* rel_w; /* [qw, kw, 96] */
  const void* rel_t; /* [qt, kt, 96] */
  void* out;
  float* lse;
  int32_t B, h, qt, qh, qw, kt, kh, kw, O;
  float scale;
  int32_t dtype;
  int32_t impl; /* 0 auto, 1 CUDA cores, 2 tcgen05 */
  /* backward only */
  const void* dout; /* [B, Nq, h, 96] */
  void* dq;         /* [B,h,Nq,96] */
  void* dk;         /* [B,h,Nk,96] */
  void* dv;
  float* d_rel_h;   /* fp32, same shapes as rel_*, accumulated into (+=) */
  float* d_rel_w;
  float* d_rel_t;
  float* ws_e;      /* scratch [B,h,Nq,kh+kw+kt] fp32: bias terms E */
  float* ws_de;     /* scratch [B,h,Nq,kh+kw+kt] fp32: dE */
  float* ws_delta;  /* scratch [B,h,Nq] fp32 */
  /* tcgen05 path only (may be NULL for impl 1): the un-gathered, interpolated tables and the integer
   * index tables of attention.py:100-119,156-163 so that q.R is one tensor-core product per query tile:
   * rel_tab [ntab_h + ntab_w + ntab_t, 96] = rows of get_rel_pos(rel_pos_h | rel_pos_w | rel_pos_t);
   * idx_h [qh,kh], idx_w [qw,kw], idx_t [qt,kt] int32 = dist.long(); key_cols [Nk rounded up to 64 (+64)] int32:
   * per key the packed E columns (i' | (kh+j')<<8 | (kh+kw+t')<<16), 0x00ffffff-style "zero slot" codes for
   * cls/object keys and bit 31 set for padding keys. */
  const void* rel_tab;
  const int32_t* idx_h;
  const int32_t* idx_w;
  const int32_t* idx_t;
  const int32_t* key_cols;
  int32_t ntab_h, ntab_w, ntab_t;
  /* bias-in-MMA kernel (attn_tc3.cu), optional: sel_tab [ceil(Nk/64)*64, sel_cols] in the activation dtype, row n =
   * key n: 1 in columns i'(n), kh + j'(n), kh + kw + t'(n) for patch keys, all zero for cls / object keys, and
   * -1e30 in the last column for padding keys (n >= Nk).  sel_cols must be 32 and kh + kw + kt <= 31. */
  const void* sel_tab;
  int32_t sel_cols;
  /* tensor-core backward (bf16, attn_bwd_tc.cu), optional: all six present -> the five contractions of the backward
   * run as batched tcgen05 GEMMs.  Nkp = Nk rounded up to 8; nep = kh+kw+kt rounded up to 8 (<= 64) -- to 16 for the
   * fused S / dP / softmax kernel (ws_s / ws_dp NULL), which takes the bias terms as extra K columns of its score
   * product and keeps them in the ws_e bytes as bf16 [B,h,Nq, hi (nep) | lo (nep)]; with these, ws_e and ws_de are
   * [B,h,Nq,nep].  sel_bwd [Nk, nep] (activation dtype): row n = key n with ones in columns i'(n), kh + j'(n),
   * kh + kw + t'(n) for patch keys, zero rows for cls / object keys.  rel_tab / idx_* / ntab_* (above), when present
   * and ntab_h + ntab_w + ntab_t <= 96, let the backward compute the bias terms as one GEMM q . rel_tab^T. */
  float* ws_s;      /* scratch fp32 [B,h,Nq,Nkp]: q k^T; ws_s / ws_dp may be NULL when Nk <= 4096 (fused kernel) */
  float* ws_dp;     /* scratch fp32 [B,h,Nq,Nkp]: dO v^T */
  void* ws_p;       /* scratch bf16 [B,h,Nq,Nkp]: softmax probabilities */
  void* ws_ds;      /* scratch bf16 [B,h,Nq,Nkp]: dS */
  float* ws_dq;     /* scratch fp32 [B,h,Nq,96] */
  const void* sel_bwd;
  int32_t nep;
  /* optional, tensor-core backward with rel_tab / idx_* present, ntab = ntab_h + ntab_w + ntab_t rounded up to 8 at most
   * min(Nkp, 512), Nkp >= 192 and (ntab <= 96 or ws_etab present), else SVIT_ENOTSUP: the
   * rel-pos gradient in TABLE space, fp32 [ntab_h + ntab_w + ntab_t, 96] (overwritten): row g = sum over query rows of
   * G[row, g] q[row] with G the scatter of dE into table-row space.  The table term of dq (G . rel_tab) and this
   * gradient (G^T . q) then run as two tcgen05 GEMMs and d_rel_h / d_rel_w / d_rel_t are NOT written (the caller maps
   * the table rows back through the index tables). */
  float* d_rel_tab;
  /* optional scratch, tensor-core backward: fp32 [B,h,Nq, ntab rounded up to 8] for E_tab = q . rel_tab^T when the
   * concatenated table has more than 96 rows (up to 96 rows the dQ scratch holds it) */
  float* ws_etab;
} svit_attn_args;
int svit_attn_fwd(const svit_attn_args* args, void* stream);
int svit_attn_bwd(const svit_attn_args* args, void* stream);

/* y[m,:] = x[m,:] * scale[m / rows_per_sample]: DropPath backward (common.py:46-59). */
int svit_scale_rows(const void* x, const float* scale, void* y, int64_t rows, int C, int64_t rows_per_sample, int dtype,
                    void* stream);

/* ---- token assembly: video_model_builder.py:326-330 (cls) and :354-363 (object tokens).
 * x [B, 1+L+Tx*O, C]: row 0 = cls; row 1+L+t*O+o = queries[o] + (Tx > 1 ? pos_t[t] : 0). Patch rows untouched. */
int svit_assemble_tokens_fwd(void* x, const float* cls, const float* queries, const float* pos_t, int B, int64_t L,
                             int Tx, int O, int C, int dtype, void* stream);
int svit_assemble_tokens_bwd(const void* dx, float* dcls, float* dqueries, float* dpos_t, int B, int64_t L, int Tx,
                             int O, int C, int dtype, void* stream);

/* ---- PatchEmbed im2col: stem_helper.py:309-320 (Conv3d k(3,7,7) s(2,4,4) p(1,3,3)) lowered to a GEMM.
 * cols [B*To*Ho*Wo, Kpad], column order (c, kt, kh, kw), zero padded to Kpad. */
int svit_im2col3d(const void* x, void* cols, int B, int Cin, int T, int H, int W, int kt, int kh, int kw, int st, int sh,
                  int sw, int pt, int ph, int pw, int Kpad, int in_dtype, int out_dtype, void* stream);
/* Its transpose, the stem's data gradient on the CUDA cores: x [B, Cin, T, H, W] (out_dtype, overwritten) = for every input
 * element the sum of the cols entries (in_dtype, same layout) of the <= ceil(kt/st) ceil(kh/sh) ceil(kw/sw) windows that
 * read it.  Deterministic (a fixed summation order, no atomics). */
int svit_col2im3d(const void* cols, void* x, int B, int Cin, int T, int H, int W, int kt, int kh, int kw, int st, int sh,
                  int sw, int pt, int ph, int pw, int Kpad, int in_dtype, int out_dtype, void* stream);

/* ---- PatchEmbed as an implicit GEMM (stem_helper.py:309-320; csrc/patch_embed_tc.cu): no im2col matrix.
 * svit_s2d_clip: the clip in space-to-depth cells, bf16 [B, ceil(T/st), ceil(H/sh), ceil(W/sw), C*st*sh*sw] with
 * cell index ((c*st + tt)*sh + hh)*sw + ww, zero beyond T/H/W.  in_kind: SVIT_F32 / SVIT_BF16 = clip [B, C, T, H, W];
 * 2 = uint8 frames [B, T, H, W, C] (C <= 3), normalised on the fly with mean / std (datasets/utils.py:287-303).
 * svit_patch_embed_s2d: out rows row_off + (t'*Ho + h')*Wo + w' of every sample (out_batch_stride elements apart, bf16,
 * E columns) = conv3d(clip) + bias; w2 [E, ntaps*cell] bf16 = the conv weight scattered into the cell taps
 * (tap-major, zero where a tap has no kernel element).  svit_patch_embed_s2d_supported tells whether a geometry fits. */
int svit_s2d_clip(const void* x, void* cells, int B, int C, int T, int H, int W, int st, int sh, int sw, int in_kind,
                  float mean0, float mean1, float mean2, float std0, float std1, float std2, void* stream);
int svit_patch_embed_s2d_supported(int C, int kt, int kh, int kw, int st, int sh, int sw, int pt, int ph, int pw, int E);
int svit_patch_embed_s2d(const void* cells, const void* w2, const float* bias, void* out, int64_t out_batch_stride,
                         int row_off, int B, int C, int T, int H, int W, int kt, int kh, int kw, int st, int sh, int sw,
                         int pt, int ph, int pw, int E, void* stream);
/* Gradients with respect to the clip.  svit_patch_embed_s2d_dgrad: the transposed stem convolution on the same tensor-core
 * kernel, dcells [B, ceil(T/st), ceil(H/sh), ceil(W/sw), C*st*sh*sw] bf16 (overwritten) from the patch rows of the bf16
 * sequence gradient, read in place (row row_off + (t'*Ho + h')*Wo + w' of sample b at dy + b*dy_batch_stride, E values).
 * w2t [C*st*sh*sw, ntaps*E] bf16 = the svit_patch_embed_s2d weight transposed with the tap order reversed in every
 * dimension: w2t[cell, ((it*nh + ih)*nw + iw)*E + e] = w2[e, (((nt-1-it)*nh + nh-1-ih)*nw + nw-1-iw)*cell + cell].
 * svit_patch_embed_s2d_dgrad_supported tells whether a geometry fits.  svit_d2s_clip: the inverse of svit_s2d_clip's cell
 * layout, cells (bf16) -> x [B, C, T, H, W] in out_dtype (SVIT_F32 / SVIT_BF16); cell values beyond T/H/W are dropped. */
int svit_patch_embed_s2d_dgrad_supported(int C, int kt, int kh, int kw, int st, int sh, int sw, int pt, int ph, int pw, int E);
int svit_patch_embed_s2d_dgrad(const void* dy, int64_t dy_batch_stride, int row_off, const void* w2t, void* dcells, int B,
                               int C, int T, int H, int W, int kt, int kh, int kw, int st, int sh, int sw, int pt, int ph,
                               int pw, int E, void* stream);
int svit_d2s_clip(const void* cells, void* x, int B, int C, int T, int H, int W, int st, int sh, int sw, int out_dtype,
                  void* stream);

/* ---- token split: video_model_builder.py:377-384. out [B, 1+O, C] = rows {0} U {N-O .. N-1} of x [B, N, C]. */
int svit_gather_cls_obj_fwd(const void* x, void* out, int B, int64_t N, int O, int C, int dtype, void* stream);
int svit_gather_cls_obj_bwd(const void* dout, void* dx, int B, int64_t N, int O, int C, int dtype, void* stream);

/* ---- box-conditioned object tokens: call site video_model_builder.py:385-392, 472-491 (RoIAlign 7x7,
 * spatial_scale 1/16, aligned, sampling_ratio 0 -> adaptive) applied per frame.
 * feat: token-major features; patch token (b, s, y, x) at feat + b*feat_batch_stride + (1 + (s*Hf + y)*Wf + x)*C.
 * boxes [B, Tx, K, 4] xyxy input pixels (fp32). token (b, t, k) = max over the P x P RoIAlign bins, written at
 * tokens + b*tokens_batch_stride + (t*K + k)*C (tokens_batch_stride 0 = dense [B, Tx*K, C]); pointing `tokens` at row
 * 1 + Tf*Hf*Wf of the token sequence with tokens_batch_stride = N*C scatters the RoI tokens to sequence rows
 * 1 + T'H'W' + t*K + k (SURVEY R3); accumulate != 0 adds to what is there.  argmax (optional) [B*Tx*K, C] uint8 = the
 * first maximal bin (what the backward needs).  Frame t reads temporal slice t / patch_stride_t (t when Tf == 1).
 * assign [B, Tx*K, 2] int32 = (b, slice).
 * Backward: dfeat [B, Tf*Hf*Wf, C] fp32 (+=, caller zero-fills): the gradient of every token spread over the bilinear taps
 * of the samples of its arg-max bin (fp32 atomics). */
int svit_roi_tokens_fwd(const void* feat, int64_t feat_batch_stride, const float* boxes, void* tokens,
                        int64_t tokens_batch_stride, uint8_t* argmax, int accumulate, int32_t* assign, int B, int C, int Tf,
                        int Hf, int Wf, int Tx, int K, int patch_stride_t, float spatial_scale, int P, int dtype,
                        void* stream);
int svit_roi_tokens_bwd(const void* dtokens, int64_t dtokens_batch_stride, const uint8_t* argmax, const float* boxes,
                        float* dfeat, int B, int C, int Tf, int Hf, int Wf, int Tx, int K, int patch_stride_t,
                        float spatial_scale, int P, int dtype, void* stream);
/* plain RoIAlign (torchvision semantics, aligned flag) on a channels-last map [N, H, W, C]; rois [R,5]; out [R,P,P,C] */
int svit_roi_align_fwd(const void* feat, const float* rois, void* out, int N, int C, int H, int W, int R, int P,
                       float spatial_scale, int sampling_ratio, int aligned, int dtype, void* stream);

/* ---- box -> slot integer logic on device (utils/box_ops.py:140-194 match_haog; :116-130 zero_empty_boxes).
 * boxes [n, 4, 4] fp32 in/out; contact [n, 2] int64 out. */
int svit_match_haog(float* boxes, int64_t* contact, int64_t n, void* stream);
int svit_zero_empty_boxes(float* boxes_cxcywh, int64_t n, float eps, void* stream);

/* ---- input side (SURVEY 8f N4): uint8 frames [B, T, H, W, 3] -> normalised [B, 3, T, H, W] (bf16 or fp32), the
 * arithmetic of datasets/utils.py:287-303 (x / 255 - mean) / std in fp32.  T*H*W must be a multiple of 16. */
int svit_normalize_u8(const void* frames, void* out, int B, int T, int H, int W, float mean0, float mean1, float mean2,
                      float std0, float std1, float std2, int out_dtype, void* stream);

/* ---- input side on the GPU (SURVEY 8f N4), beyond svit_normalize_u8: per-sample spatial crop (offsets x_off / y_off [B],
 * int32, device) + optional horizontal flip (flip [B] int32 or NULL) + colour normalisation + THWC -> CTHW, one pass
 * (datasets/transform.py:154-190, 248-285; datasets/utils.py:287-303); out [B, 3, T, crop_h, crop_w] fp32 / bf16.
 * svit_boxes_crop_flip moves the boxes with the frames and into the loss format: crop_clip_boxes, flip, / crop size,
 * clip [0, 1], xyxy -> cxcywh, zero boxes with w or h <= eps (transform.py:107-132; ssv2_frames.py:347-353;
 * utils/box_ops.py:32-36, 116-130); boxes [B, boxes_per_sample, 4] fp32 pixels -> [B, boxes_per_sample, 4]. */
int svit_crop_flip_normalize_u8(const void* frames, void* out, const int32_t* x_off, const int32_t* y_off,
                                const int32_t* flip, int B, int T, int H, int W, int crop_h, int crop_w, float mean0,
                                float mean1, float mean2, float std0, float std1, float std2, int out_dtype, void* stream);
int svit_boxes_crop_flip(const float* boxes_xyxy, float* out_cxcywh, const int32_t* x_off, const int32_t* y_off,
                         const int32_t* flip, int B, int64_t boxes_per_sample, int crop_h, int crop_w, float eps,
                         void* stream);

/* ---- head + losses (SURVEY 8f N2).
 * svit_head_fwd: SViTHead.forward without autograd (video_model_builder.py:507-546) in one launch.  x [B, 1 + Tx*O, C]
 * = [cls ; object tokens] (fp32 or bf16); weights fp32: projection [num_classes, C], boxes_mlp.0 [4, C], boxes_bce_mlp
 * [1, C], contact_mlp [5, C] and their biases.  Outputs fp32: logits [B, num_classes]; probs (optional; softmax, or
 * sigmoid when act_sigmoid) ; obj_desc [B, Tx, O, C]; pred_bboxes [B, Tx, O, 5] = (score | sigmoid(box)) with the score
 * passed through a sigmoid when eval_mode; pred_contact [B, Tx, 2, 5] (softmax when eval_mode) for object slots 0, 1.
 * svit_haog_loss: boxes_loss_ + contact-state cross entropy (models/losses.py:50-92, 138-155; utils/box_ops.py:41-77) as
 * masked means over paired boxes.  pred_bboxes [n_boxes, 5] = (score logit, cx, cy, w, h); target_boxes
 * [n_boxes, target_cols] (4: all-zero row = no box; 5: leading soft mask); pred_contact [n_contact, 5] logits,
 * target_contact [n_contact] int64 (-1 = ignore).  losses[4] = (l1, bce, giou, contact ce); d_l1 / d_giou [n_boxes, 4],
 * d_bce [n_boxes], d_ce [n_contact, 5] = the gradient of each term w.r.t. its prediction columns. */
int svit_head_fwd(const void* x, const float* w_proj, const float* b_proj, const float* w_box, const float* b_box,
                  const float* w_score, const float* b_score, const float* w_contact, const float* b_contact, float* logits,
                  float* probs, float* obj_desc, float* pred_bboxes, float* pred_contact, int B, int Tx, int O, int C,
                  int num_classes, int act_sigmoid, int eval_mode, int dtype, void* stream);
int svit_haog_loss(const float* pred_bboxes, const float* target_boxes, int target_cols, int64_t n_boxes,
                   const float* pred_contact, const int64_t* target_contact, int64_t n_contact, float* losses, float* d_l1,
                   float* d_bce, float* d_giou, float* d_ce, void* stream);

/* ---- fused optimizer step (SURVEY 8f N3): clip_grad_norm_ + torch.optim.AdamW over all parameter tensors
 * (tools/train_net.py:133-151, models/optimizer.py:89-104) in two launches.  `table` [ntensors] and the chunk map
 * (chunk c covers elements [chunk_start[c], chunk_start[c] + chunk) of tensor chunk_tensor[c]) live in device memory;
 * all tensors are fp32.  svit_grad_sqnorm writes sum(g^2) over every tensor to *out (zeroed first).  svit_adamw_step
 * applies, per element and in torch's operation order, g *= min(1, max_norm / (sqrt(*sqnorm) + 1e-6)) (skipped when
 * max_norm <= 0 or sqnorm is NULL), p *= 1 - lr * wd, m = lerp(m, g, 1 - beta1), v = beta2 v + (1 - beta2) g^2,
 * p -= lr / (1 - beta1^step) * m / (sqrt(v) / sqrt(1 - beta2^step) + eps). */
typedef struct svit_optim_tensor {
  void* param;
  const void* grad;
  void* exp_avg;
  void* exp_avg_sq;
  int64_t numel;
  float weight_decay;
  int32_t pad_;
} svit_optim_tensor;
int svit_grad_sqnorm(const svit_optim_tensor* table, const int32_t* chunk_tensor, const int64_t* chunk_start, int nchunks,
                     int chunk, float* out, void* stream);
int svit_adamw_step(const svit_optim_tensor* table, const int32_t* chunk_tensor, const int64_t* chunk_start, int nchunks,
                    int chunk, float lr, float beta1, float beta2, float eps, int step, float max_norm, const float* sqnorm,
                    void* stream);
/* Same update with the step-dependent scalars read from DEVICE memory: hyper = {lr, 1 - beta1^step, sqrt(1 - beta2^step)}.
 * Nothing step-dependent is baked into the launch, so a CUDA graph of the training step (svit_b200.GraphedTrainStep)
 * replays it; the caller refreshes `hyper` with a small H2D copy before each replay. */
int svit_adamw_step_dev(const svit_optim_tensor* table, const int32_t* chunk_tensor, const int64_t* chunk_start, int nchunks,
                        int chunk, const float* hyper, float beta1, float beta2, float eps, float max_norm,
                        const float* sqnorm, void* stream);

#ifdef __cplusplus
}
#endif
#endif
