// HBM-bound token kernels of the SViT hot path: LayerNorm, skip max-pool, token assembly
// (cls | patch | object tokens), im2col for the patch-embed GEMM, final token split.
// Each is one read + one write of the token tensor; all math in fp32.
#include "common.cuh"

// ------------------------------------------------------------------------------------------------
// LayerNorm over the channel dim (attention.py:558,566; video_model_builder.py:375), eps 1e-6.
// One warp per token row; lane l owns channels l, l+32, ... (coalesced 32-wide segments).
// ------------------------------------------------------------------------------------------------
#define LN_MAXV 24  // C <= 768

template <typename T>
__global__ void __launch_bounds__(256) layernorm_fwd_kernel(const T* __restrict__ x, const float* __restrict__ gamma,
                                                            const float* __restrict__ beta, T* __restrict__ y,
                                                            float* __restrict__ mean_out, float* __restrict__ rstd_out,
                                                            int64_t rows, int C, float eps) {
  const int lane = threadIdx.x & 31;
  const int nv = C >> 5;
  int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int64_t stride = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (; row < rows; row += stride) {
    const T* xr = x + row * C;
    float v[LN_MAXV];
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < LN_MAXV; ++i)
      if (i < nv) {
        v[i] = to_f(xr[lane + 32 * i]);
        s += v[i];
      }
    const float mean = warp_sum(s) / (float)C;
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < LN_MAXV; ++i)
      if (i < nv) {
        float d = v[i] - mean;
        q += d * d;
      }
    const float rstd = rsqrtf(warp_sum(q) / (float)C + eps);
    T* yr = y + row * C;
#pragma unroll
    for (int i = 0; i < LN_MAXV; ++i)
      if (i < nv) {
        int c = lane + 32 * i;
        yr[c] = from_f<T>((v[i] - mean) * rstd * gamma[c] + beta[c]);
      }
    if (lane == 0 && mean_out) {
      mean_out[row] = mean;
      rstd_out[row] = rstd;
    }
  }
}

// dx = rstd * (g*dy - mean(g*dy) - xhat * mean(g*dy*xhat)); dgamma += sum dy*xhat; dbeta += sum dy.
template <typename T>
__global__ void __launch_bounds__(256) layernorm_bwd_kernel(const T* __restrict__ dy, const T* __restrict__ x,
                                                            const float* __restrict__ gamma,
                                                            const float* __restrict__ mean_in,
                                                            const float* __restrict__ rstd_in, T* __restrict__ dx,
                                                            float* __restrict__ dgamma, float* __restrict__ dbeta,
                                                            int64_t rows, int C) {
  const int lane = threadIdx.x & 31;
  const int nv = C >> 5;
  float ag[LN_MAXV], ab[LN_MAXV];
#pragma unroll
  for (int i = 0; i < LN_MAXV; ++i) ag[i] = ab[i] = 0.f;
  int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int64_t stride = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (; row < rows; row += stride) {
    const float mean = mean_in[row], rstd = rstd_in[row];
    float xh[LN_MAXV], g[LN_MAXV];
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int i = 0; i < LN_MAXV; ++i)
      if (i < nv) {
        int c = lane + 32 * i;
        float d = to_f(dy[row * C + c]);
        xh[i] = (to_f(x[row * C + c]) - mean) * rstd;
        g[i] = d * gamma[c];
        s1 += g[i];
        s2 += g[i] * xh[i];
        ag[i] += d * xh[i];
        ab[i] += d;
      }
    s1 = warp_sum(s1) / (float)C;
    s2 = warp_sum(s2) / (float)C;
#pragma unroll
    for (int i = 0; i < LN_MAXV; ++i)
      if (i < nv) dx[row * C + lane + 32 * i] = from_f<T>(rstd * (g[i] - s1 - xh[i] * s2));
  }
  // block reduce the parameter gradients through shared memory, then one atomic per channel per CTA
  __shared__ float sg[LN_MAXV * 32], sb[LN_MAXV * 32];
  for (int i = threadIdx.x; i < C; i += blockDim.x) sg[i] = sb[i] = 0.f;
  __syncthreads();
#pragma unroll
  for (int i = 0; i < LN_MAXV; ++i)
    if (i < nv) {
      atomicAdd(&sg[lane + 32 * i], ag[i]);
      atomicAdd(&sb[lane + 32 * i], ab[i]);
    }
  __syncthreads();
  for (int i = threadIdx.x; i < C; i += blockDim.x) {
    atomicAdd(&dgamma[i], sg[i]);
    atomicAdd(&dbeta[i], sb[i]);
  }
}

// bf16, C % 8 == 0, C <= 256 * NV8: warp per row, lane owns the 8-channel units lane, lane + 32, ... (16-byte accesses).
template <int NV8>
__global__ void __launch_bounds__(256) layernorm_bwd_bf16x8_kernel(const bf16* __restrict__ dy, const bf16* __restrict__ x,
                                                                   const float* __restrict__ gamma,
                                                                   const float* __restrict__ mean_in,
                                                                   const float* __restrict__ rstd_in, bf16* __restrict__ dx,
                                                                   float* __restrict__ dgamma, float* __restrict__ dbeta,
                                                                   int64_t rows, int C) {
  __shared__ float sg[NV8 * 256], sb[NV8 * 256];
  const int lane = threadIdx.x & 31;
  const int n8 = C >> 3;
  float gm[NV8][8], ag[NV8][8], ab[NV8][8];
#pragma unroll
  for (int i = 0; i < NV8; ++i) {
    const int u = lane + 32 * i;
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      gm[i][e] = u < n8 ? gamma[u * 8 + e] : 0.f;
      ag[i][e] = ab[i][e] = 0.f;
    }
  }
  auto unpack = [](const uint4& v, float f[8]) {
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      f[2 * e] = __uint_as_float(w[e] << 16);
      f[2 * e + 1] = __uint_as_float(w[e] & 0xffff0000u);
    }
  };
  const float invC = 1.f / (float)C;
  int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int64_t stride = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (; row < rows; row += stride) {
    const float mean = mean_in[row], rstd = rstd_in[row];
    float xh[NV8][8], g[NV8][8];
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int i = 0; i < NV8; ++i) {
      const int u = lane + 32 * i;
      if (u < n8) {
        float d[8], xv[8];
        unpack(__ldg(reinterpret_cast<const uint4*>(dy + row * C + u * 8)), d);
        unpack(__ldg(reinterpret_cast<const uint4*>(x + row * C + u * 8)), xv);
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          xh[i][e] = (xv[e] - mean) * rstd;
          g[i][e] = d[e] * gm[i][e];
          s1 += g[i][e];
          s2 = fmaf(g[i][e], xh[i][e], s2);
          ag[i][e] = fmaf(d[e], xh[i][e], ag[i][e]);
          ab[i][e] += d[e];
        }
      }
    }
    s1 = warp_sum(s1) * invC;
    s2 = warp_sum(s2) * invC;
#pragma unroll
    for (int i = 0; i < NV8; ++i) {
      const int u = lane + 32 * i;
      if (u < n8) {
        __nv_bfloat162 h2[4];
#pragma unroll
        for (int e = 0; e < 4; ++e)
          h2[e] = __floats2bfloat162_rn(rstd * (g[i][2 * e] - s1 - xh[i][2 * e] * s2),
                                        rstd * (g[i][2 * e + 1] - s1 - xh[i][2 * e + 1] * s2));
        *reinterpret_cast<uint4*>(dx + row * C + u * 8) = *reinterpret_cast<uint4*>(h2);
      }
    }
  }
  for (int i = threadIdx.x; i < C; i += blockDim.x) sg[i] = sb[i] = 0.f;
  __syncthreads();
#pragma unroll
  for (int i = 0; i < NV8; ++i) {
    const int u = lane + 32 * i;
    if (u < n8) {
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        atomicAdd(&sg[u * 8 + e], ag[i][e]);
        atomicAdd(&sb[u * 8 + e], ab[i][e]);
      }
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < C; i += blockDim.x) {
    atomicAdd(&dgamma[i], sg[i]);
    atomicAdd(&dbeta[i], sb[i]);
  }
}

// ------------------------------------------------------------------------------------------------
// Skip-path pooling (attention.py:562-564): MaxPool3d k(1,3,3) s(1,2,2) p(0,1,1) on the patch tokens
// of a [B, N, C] sequence; cls row and object tail copied.  One thread per (token, channel).
// ------------------------------------------------------------------------------------------------
template <typename T>
__global__ void skip_maxpool_fwd_kernel(const T* __restrict__ x, T* __restrict__ y, int B, int C, int T_, int H, int W,
                                        int Ho, int Wo, int O, int s) {
  const int64_t Nin = 1 + (int64_t)T_ * H * W + O, Nout = 1 + (int64_t)T_ * Ho * Wo + O;
  const int64_t total = (int64_t)B * Nout * C;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    int c = (int)(i % C);
    int64_t r = i / C;
    int64_t tok = r % Nout;
    int b = (int)(r / Nout);
    const T* xb = x + (int64_t)b * Nin * C;
    float out;
    if (tok == 0) {
      out = to_f(xb[c]);
    } else if (tok > (int64_t)T_ * Ho * Wo) {
      out = to_f(xb[(tok - (int64_t)T_ * Ho * Wo + (int64_t)T_ * H * W) * C + c]);
    } else {
      int64_t p = tok - 1;
      int wo = (int)(p % Wo), ho = (int)((p / Wo) % Ho), t = (int)(p / ((int64_t)Wo * Ho));
      float m = -INFINITY;
      for (int dh = -1; dh <= 1; ++dh) {
        int hh = ho * s + dh;
        if (hh < 0 || hh >= H) continue;
        for (int dw = -1; dw <= 1; ++dw) {
          int ww = wo * s + dw;
          if (ww < 0 || ww >= W) continue;
          float v = to_f(xb[(1 + ((int64_t)t * H + hh) * W + ww) * C + c]);
          if (v > m || v != v) m = v;
        }
      }
      out = m;
    }
    y[i] = from_f<T>(out);
  }
}

// Backward: each output routes its gradient to the first maximal input of its window (strict >,
// scan order h then w, as ATen's max_pool3d does); windows overlap so inputs accumulate with atomics
// in fp32 scratch-free form: thread per INPUT element gathers from the <=4 windows that contain it.
template <typename T>
__global__ void skip_maxpool_bwd_kernel(const T* __restrict__ x, const T* __restrict__ dy, T* __restrict__ dx, int B,
                                        int C, int T_, int H, int W, int Ho, int Wo, int O, int s) {
  const int64_t Nin = 1 + (int64_t)T_ * H * W + O, Nout = 1 + (int64_t)T_ * Ho * Wo + O;
  const int64_t total = (int64_t)B * Nin * C;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    int c = (int)(i % C);
    int64_t r = i / C;
    int64_t tok = r % Nin;
    int b = (int)(r / Nin);
    const T* xb = x + (int64_t)b * Nin * C;
    const T* dyb = dy + (int64_t)b * Nout * C;
    float g = 0.f;
    if (tok == 0) {
      g = to_f(dyb[c]);
    } else if (tok > (int64_t)T_ * H * W) {
      g = to_f(dyb[(tok - (int64_t)T_ * H * W + (int64_t)T_ * Ho * Wo) * C + c]);
    } else {
      int64_t p = tok - 1;
      int w = (int)(p % W), h = (int)((p / W) % H), t = (int)(p / ((int64_t)W * H));
      // windows (ho, wo) with |ho*s - h| <= 1
      for (int ho = (h - 1 + s - 1) / s; ho * s <= h + 1 && ho < Ho; ++ho) {
        if (ho < 0) continue;
        for (int wo = (w - 1 + s - 1) / s; wo * s <= w + 1 && wo < Wo; ++wo) {
          if (wo < 0) continue;
          // find the argmax of this window
          float m = -INFINITY;
          int ah = -1, aw = -1;
          for (int dh = -1; dh <= 1; ++dh) {
            int hh = ho * s + dh;
            if (hh < 0 || hh >= H) continue;
            for (int dw = -1; dw <= 1; ++dw) {
              int ww = wo * s + dw;
              if (ww < 0 || ww >= W) continue;
              float v = to_f(xb[(1 + ((int64_t)t * H + hh) * W + ww) * C + c]);
              if (v > m || v != v) {
                m = v;
                ah = hh;
                aw = ww;
              }
            }
          }
          if (ah == h && aw == w) g += to_f(dyb[(1 + ((int64_t)t * Ho + ho) * Wo + wo) * C + c]);
        }
      }
    }
    dx[i] = from_f<T>(g);
  }
}

// bf16, C % 8 == 0: thread = 8 consecutive channels of one input token (16-byte accesses); same gather as above.
__global__ void __launch_bounds__(256) skip_maxpool_bwd_vec8_kernel(const bf16* __restrict__ x, const bf16* __restrict__ dy,
                                                                    bf16* __restrict__ dx, int B, int C, int T_, int H,
                                                                    int W, int Ho, int Wo, int O, int s) {
  const int C8 = C >> 3;
  const int64_t Nin = 1 + (int64_t)T_ * H * W + O, Nout = 1 + (int64_t)T_ * Ho * Wo + O;
  const int64_t total = (int64_t)B * Nin * C8;
  auto unpack = [](const uint4& v, float f[8]) {
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      f[2 * u] = __uint_as_float(w[u] << 16);
      f[2 * u + 1] = __uint_as_float(w[u] & 0xffff0000u);
    }
  };
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(i % C8) * 8;
    const int64_t r = i / C8;
    const int64_t tok = r % Nin;
    const int b = (int)(r / Nin);
    const bf16* xb = x + (int64_t)b * Nin * C + c;
    const bf16* dyb = dy + (int64_t)b * Nout * C + c;
    bf16* o = dx + r * C + c;
    if (tok == 0) {
      *reinterpret_cast<uint4*>(o) = __ldg(reinterpret_cast<const uint4*>(dyb));
      continue;
    }
    if (tok > (int64_t)T_ * H * W) {
      *reinterpret_cast<uint4*>(o) =
          __ldg(reinterpret_cast<const uint4*>(dyb + (tok - (int64_t)T_ * H * W + (int64_t)T_ * Ho * Wo) * C));
      continue;
    }
    const int64_t p = tok - 1;
    const int w = (int)(p % W), h = (int)((p / W) % H), t = (int)(p / ((int64_t)W * H));
    float g[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    for (int ho = (h - 1 + s - 1) / s; ho * s <= h + 1 && ho < Ho; ++ho) {
      if (ho < 0) continue;
      for (int wo = (w - 1 + s - 1) / s; wo * s <= w + 1 && wo < Wo; ++wo) {
        if (wo < 0) continue;
        // per channel: is (h, w) the first maximum of this window in ATen's scan order (h then w)?
        float m[8];
        bool mine[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) { m[u] = -INFINITY; mine[u] = false; }
#pragma unroll
        for (int dh = -1; dh <= 1; ++dh) {
          const int hh = ho * s + dh;
          if (hh < 0 || hh >= H) continue;
#pragma unroll
          for (int dw = -1; dw <= 1; ++dw) {
            const int ww = wo * s + dw;
            if (ww < 0 || ww >= W) continue;
            float v[8];
            unpack(__ldg(reinterpret_cast<const uint4*>(xb + (1 + ((int64_t)t * H + hh) * W + ww) * C)), v);
            const bool here = hh == h && ww == w;
#pragma unroll
            for (int u = 0; u < 8; ++u)
              if (v[u] > m[u] || v[u] != v[u]) { m[u] = v[u]; mine[u] = here; }
          }
        }
        float d[8];
        unpack(__ldg(reinterpret_cast<const uint4*>(dyb + (1 + ((int64_t)t * Ho + ho) * Wo + wo) * C)), d);
#pragma unroll
        for (int u = 0; u < 8; ++u) g[u] += mine[u] ? d[u] : 0.f;
      }
    }
    __nv_bfloat162 h2[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) h2[u] = __floats2bfloat162_rn(g[2 * u], g[2 * u + 1]);
    *reinterpret_cast<uint4*>(o) = *reinterpret_cast<uint4*>(h2);
  }
}

// ------------------------------------------------------------------------------------------------
// Token assembly (video_model_builder.py:326-363): x[b, 0] = cls; x[b, 1+L + t*O + o] = query[o] + pos_t[t]
// (no temporal term when Tx == 1).  Patch rows 1..L are written by the patch-embed GEMM epilogue.
// ------------------------------------------------------------------------------------------------
template <typename T>
__global__ void assemble_tokens_kernel(T* __restrict__ x, const float* __restrict__ cls, const float* __restrict__ queries,
                                       const float* __restrict__ pos_t, int B, int64_t L, int Tx, int O, int C) {
  const int64_t N = 1 + L + (int64_t)Tx * O;
  const int64_t per_b = (int64_t)(1 + Tx * O) * C;
  const int64_t total = (int64_t)B * per_b;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    int c = (int)(i % C);
    int64_t r = (i / C) % (1 + Tx * O);
    int b = (int)(i / per_b);
    float v;
    int64_t row;
    if (r == 0) {
      v = cls[c];
      row = 0;
    } else {
      int to = (int)(r - 1);
      int t = to / O, o = to % O;
      v = queries[o * C + c] + (Tx > 1 ? pos_t[t * C + c] : 0.f);
      row = 1 + L + to;
    }
    x[((int64_t)b * N + row) * C + c] = from_f<T>(v);
  }
}

// Backward of the assembly: dcls += sum_b dx[b,0]; dquery[o] += sum_{b,t} dx[b, 1+L+t*O+o]; dpos_t[t] += sum_{b,o}.
template <typename T>
__global__ void assemble_tokens_bwd_kernel(const T* __restrict__ dx, float* __restrict__ dcls, float* __restrict__ dq,
                                           float* __restrict__ dpos, int B, int64_t L, int Tx, int O, int C) {
  const int64_t N = 1 + L + (int64_t)Tx * O;
  // one thread per (row-kind r, c); loops over batch -> deterministic, no atomics
  const int64_t total = (int64_t)(1 + Tx * O) * C;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    int c = (int)(i % C);
    int64_t r = i / C;
    int64_t row = r == 0 ? 0 : 1 + L + (r - 1);
    float s = 0.f;
    for (int b = 0; b < B; ++b) s += to_f(dx[((int64_t)b * N + row) * C + c]);
    if (r == 0) {
      dcls[c] += s;
    } else {
      int to = (int)(r - 1);
      atomicAdd(&dq[(to % O) * C + c], s);
      if (Tx > 1) atomicAdd(&dpos[(to / O) * C + c], s);
    }
  }
}

// ------------------------------------------------------------------------------------------------
// im2col for PatchEmbed (stem_helper.py:309-320): clip [B,Cin,T,H,W] -> cols [B*To*Ho*Wo, Kpad] with
// column order (c, kt, kh, kw) matching weight.reshape(Cout, Cin*kt*kh*kw); zero padding outside.
// ------------------------------------------------------------------------------------------------
template <typename TI, typename TO>
__global__ void im2col3d_kernel(const TI* __restrict__ x, TO* __restrict__ cols, int B, int Cin, int T_, int H, int W,
                                int To, int Ho, int Wo, int kt, int kh, int kw, int st, int sh, int sw, int pt, int ph,
                                int pw, int Kpad) {
  const int K = Cin * kt * kh * kw;
  const int64_t total = (int64_t)B * To * Ho * Wo * Kpad;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    int k = (int)(i % Kpad);
    int64_t m = i / Kpad;
    float v = 0.f;
    if (k < K) {
      int dw = k % kw, dh = (k / kw) % kh, dt = (k / (kw * kh)) % kt, c = k / (kw * kh * kt);
      int wo = (int)(m % Wo), ho = (int)((m / Wo) % Ho), to = (int)((m / ((int64_t)Wo * Ho)) % To);
      int b = (int)(m / ((int64_t)Wo * Ho * To));
      int t = to * st - pt + dt, h = ho * sh - ph + dh, w = wo * sw - pw + dw;
      if (t >= 0 && t < T_ && h >= 0 && h < H && w >= 0 && w < W)
        v = to_f(x[((((int64_t)b * Cin + c) * T_ + t) * H + h) * W + w]);
    }
    cols[i] = from_f<TO>(v);
  }
}

// Transpose of im2col3d (the stem's data gradient on the CUDA cores): x[b, c, t, h, w] = the sum of cols[m, (c, dt, dh, dw)]
// over the kernel taps whose output position m = ((t + pt - dt) / st, (h + ph - dh) / sh, (w + pw - dw) / sw) is whole and
// in range.  One thread per input element sums its <= ceil(k / s)^3 windows in a fixed order: no atomics, deterministic.
template <typename TI, typename TO>
__global__ void col2im3d_kernel(const TI* __restrict__ cols, TO* __restrict__ x, int B, int Cin, int T_, int H, int W,
                                int To, int Ho, int Wo, int kt, int kh, int kw, int st, int sh, int sw, int pt, int ph,
                                int pw, int Kpad) {
  const int64_t total = (int64_t)B * Cin * T_ * H * W;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int w = (int)(i % W), h = (int)((i / W) % H), t = (int)((i / ((int64_t)W * H)) % T_);
    const int64_t bc = i / ((int64_t)W * H * T_);
    const int c = (int)(bc % Cin), b = (int)(bc / Cin);
    float acc = 0.f;
    for (int dt = (t + pt) % st; dt < kt; dt += st) {
      const int to = (t + pt - dt) / st;
      if (to >= To) continue;
      if (to < 0) break;
      for (int dh = (h + ph) % sh; dh < kh; dh += sh) {
        const int ho = (h + ph - dh) / sh;
        if (ho >= Ho) continue;
        if (ho < 0) break;
        for (int dw = (w + pw) % sw; dw < kw; dw += sw) {
          const int wo = (w + pw - dw) / sw;
          if (wo >= Wo) continue;
          if (wo < 0) break;
          const int64_t m = (((int64_t)b * To + to) * Ho + ho) * Wo + wo;
          acc += to_f(cols[m * Kpad + ((c * kt + dt) * kh + dh) * kw + dw]);
        }
      }
    }
    x[i] = from_f<TO>(acc);
  }
}

// Generic dtype conversion / strided row gather used by the token split (video_model_builder.py:377-384):
// out[b, j, :] = x[b, idx(j), :] for the rows {0} U {N-O..N-1}.
template <typename T>
__global__ void gather_cls_obj_kernel(const T* __restrict__ x, T* __restrict__ out, int B, int64_t N, int O, int C) {
  const int64_t total = (int64_t)B * (1 + O) * C;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    int c = (int)(i % C);
    int64_t j = (i / C) % (1 + O);
    int b = (int)(i / ((int64_t)(1 + O) * C));
    int64_t row = j == 0 ? 0 : N - O + (j - 1);
    out[i] = x[((int64_t)b * N + row) * C + c];
  }
}

template <typename T>
__global__ void scatter_cls_obj_bwd_kernel(const T* __restrict__ dout, T* __restrict__ dx, int B, int64_t N, int O, int C) {
  const int64_t total = (int64_t)B * N * C;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    int c = (int)(i % C);
    int64_t row = (i / C) % N;
    int b = (int)(i / (N * C));
    float v = 0.f;
    if (row == 0) v = to_f(dout[((int64_t)b * (1 + O)) * C + c]);
    else if (row >= N - O) v = to_f(dout[((int64_t)b * (1 + O) + 1 + (row - (N - O))) * C + c]);
    dx[i] = from_f<T>(v);
  }
}

// y[m, :] = x[m, :] * scale[m / rows_per_sample]   (DropPath backward, common.py:46-59)
template <typename T>
__global__ void scale_rows_kernel(const T* __restrict__ x, const float* __restrict__ scale, T* __restrict__ y,
                                  int64_t rows, int C, int64_t rows_per_sample) {
  const int64_t total = rows * C;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x)
    y[i] = from_f<T>(to_f(x[i]) * scale[(i / C) / rows_per_sample]);
}

// bf16, C % 8 == 0, 16-byte aligned: thread = 8 consecutive channels of one row (one index division per 16 bytes; the
// scalar kernel above spends two 64-bit divisions per 2-byte element)
__global__ void __launch_bounds__(256) scale_rows_bf16x8_kernel(const bf16* __restrict__ x, const float* __restrict__ scale,
                                                                bf16* __restrict__ y, int64_t units, int c8,
                                                                int64_t rows_per_sample) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < units; i += (int64_t)gridDim.x * blockDim.x) {
    const float sc = __ldg(scale + (i / c8) / rows_per_sample);
    const uint4 v = __ldg(reinterpret_cast<const uint4*>(x) + i);
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
    uint32_t o[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      __nv_bfloat162 h = __floats2bfloat162_rn(__uint_as_float(w[e] << 16) * sc, __uint_as_float(w[e] & 0xffff0000u) * sc);
      o[e] = *reinterpret_cast<uint32_t*>(&h);
    }
    reinterpret_cast<uint4*>(y)[i] = make_uint4(o[0], o[1], o[2], o[3]);
  }
}

static inline int grid_for(int64_t total, int threads) {
  int64_t g = ceil_div64(total, threads);
  int64_t cap = (int64_t)svit_num_sms() * 16;
  return (int)(g < cap ? (g > 0 ? g : 1) : cap);
}

// bf16 fast paths (stream_bf16.cu): return 1 when they handled the call, 0 when the shape is not covered
int svit_layernorm_fwd_bf16(const void* x, const float* gamma, const float* beta, void* y, float* mean, float* rstd,
                            int64_t rows, int C, float eps, cudaStream_t st);
int svit_im2col_rows(const void* x, void* cols, int B, int Cin, int T, int H, int W, int To, int Ho, int Wo, int kt, int kh,
                     int kw, int st_, int sh, int sw, int pt, int ph, int pw, int Kpad, int in_dtype, cudaStream_t st);
int svit_skip_maxpool_fwd_bf16(const void* x, void* y, int B, int C, int T, int H, int W, int Ho, int Wo, int O, int s,
                               cudaStream_t st);

extern "C" {

int svit_layernorm_fwd(const void* x, const float* gamma, const float* beta, void* y, float* mean, float* rstd,
                       int64_t rows, int C, float eps, int dtype, void* stream) {
  if (C % 32 != 0 || C > 32 * LN_MAXV || rows < 0) return SVIT_EINVAL;
  if (rows == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == SVIT_BF16) {
    int rc = svit_layernorm_fwd_bf16(x, gamma, beta, y, mean, rstd, rows, C, eps, st);
    if (rc == 1) return 0;
    if (rc >= 1000) return rc - 1000;
  }
  int grid = (int)(ceil_div64(rows, 8) < (int64_t)svit_num_sms() * 8 ? ceil_div64(rows, 8) : (int64_t)svit_num_sms() * 8);
  if (dtype == SVIT_F32)
    layernorm_fwd_kernel<float><<<grid, 256, 0, st>>>((const float*)x, gamma, beta, (float*)y, mean, rstd, rows, C, eps);
  else if (dtype == SVIT_BF16)
    layernorm_fwd_kernel<bf16><<<grid, 256, 0, st>>>((const bf16*)x, gamma, beta, (bf16*)y, mean, rstd, rows, C, eps);
  else
    return SVIT_EINVAL;
  SVIT_CHECK_LAUNCH();
  return 0;
}

int svit_layernorm_bwd(const void* dy, const void* x, const float* gamma, const float* mean, const float* rstd, void* dx,
                       float* dgamma, float* dbeta, int64_t rows, int C, int dtype, void* stream) {
  if (C % 32 != 0 || C > 32 * LN_MAXV || rows < 0) return SVIT_EINVAL;
  if (rows == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  int grid = (int)(ceil_div64(rows, 8) < (int64_t)svit_num_sms() * 2 ? ceil_div64(rows, 8) : (int64_t)svit_num_sms() * 2);
  if (dtype == SVIT_F32)
    layernorm_bwd_kernel<float><<<grid, 256, 0, st>>>((const float*)dy, (const float*)x, gamma, mean, rstd, (float*)dx,
                                                      dgamma, dbeta, rows, C);
  else if (dtype == SVIT_BF16 && C % 8 == 0 && C <= 768 &&
           ((reinterpret_cast<uintptr_t>(dy) | reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(dx)) & 15) == 0) {
    const bf16 *dyb = (const bf16*)dy, *xb = (const bf16*)x;
    if (C <= 256) layernorm_bwd_bf16x8_kernel<1><<<grid, 256, 0, st>>>(dyb, xb, gamma, mean, rstd, (bf16*)dx, dgamma, dbeta, rows, C);
    else if (C <= 512) layernorm_bwd_bf16x8_kernel<2><<<grid, 256, 0, st>>>(dyb, xb, gamma, mean, rstd, (bf16*)dx, dgamma, dbeta, rows, C);
    else layernorm_bwd_bf16x8_kernel<3><<<grid, 256, 0, st>>>(dyb, xb, gamma, mean, rstd, (bf16*)dx, dgamma, dbeta, rows, C);
  } else if (dtype == SVIT_BF16)
    layernorm_bwd_kernel<bf16><<<grid, 256, 0, st>>>((const bf16*)dy, (const bf16*)x, gamma, mean, rstd, (bf16*)dx,
                                                     dgamma, dbeta, rows, C);
  else
    return SVIT_EINVAL;
  SVIT_CHECK_LAUNCH();
  return 0;
}

int svit_skip_maxpool_fwd(const void* x, void* y, int B, int C, int T, int H, int W, int O, int stride_hw, int dtype,
                          void* stream) {
  if (stride_hw < 1 || B < 0 || O < 1) return SVIT_EINVAL;
  int Ho = (H - 1) / stride_hw + 1, Wo = (W - 1) / stride_hw + 1;
  if (stride_hw == 1) return SVIT_EINVAL;  // identity pool: caller aliases the tensor
  int64_t total = (int64_t)B * (1 + (int64_t)T * Ho * Wo + O) * C;
  if (total == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == SVIT_BF16) {
    int rc = svit_skip_maxpool_fwd_bf16(x, y, B, C, T, H, W, Ho, Wo, O, stride_hw, st);
    if (rc == 1) return 0;
    if (rc >= 1000) return rc - 1000;
  }
  if (dtype == SVIT_F32)
    skip_maxpool_fwd_kernel<float><<<grid_for(total, 256), 256, 0, st>>>((const float*)x, (float*)y, B, C, T, H, W, Ho, Wo, O, stride_hw);
  else if (dtype == SVIT_BF16)
    skip_maxpool_fwd_kernel<bf16><<<grid_for(total, 256), 256, 0, st>>>((const bf16*)x, (bf16*)y, B, C, T, H, W, Ho, Wo, O, stride_hw);
  else
    return SVIT_EINVAL;
  SVIT_CHECK_LAUNCH();
  return 0;
}

int svit_skip_maxpool_bwd(const void* x, const void* dy, void* dx, int B, int C, int T, int H, int W, int O,
                          int stride_hw, int dtype, void* stream) {
  if (stride_hw < 2 || B < 0 || O < 1) return SVIT_EINVAL;
  int Ho = (H - 1) / stride_hw + 1, Wo = (W - 1) / stride_hw + 1;
  int64_t total = (int64_t)B * (1 + (int64_t)T * H * W + O) * C;
  if (total == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == SVIT_F32)
    skip_maxpool_bwd_kernel<float><<<grid_for(total, 256), 256, 0, st>>>((const float*)x, (const float*)dy, (float*)dx, B, C, T, H, W, Ho, Wo, O, stride_hw);
  else if (dtype == SVIT_BF16 && C % 8 == 0 &&
           ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(dy) | reinterpret_cast<uintptr_t>(dx)) & 15) == 0)
    skip_maxpool_bwd_vec8_kernel<<<grid_for(total / 8, 256), 256, 0, st>>>((const bf16*)x, (const bf16*)dy, (bf16*)dx, B, C, T, H, W, Ho, Wo, O, stride_hw);
  else if (dtype == SVIT_BF16)
    skip_maxpool_bwd_kernel<bf16><<<grid_for(total, 256), 256, 0, st>>>((const bf16*)x, (const bf16*)dy, (bf16*)dx, B, C, T, H, W, Ho, Wo, O, stride_hw);
  else
    return SVIT_EINVAL;
  SVIT_CHECK_LAUNCH();
  return 0;
}

int svit_assemble_tokens_fwd(void* x, const float* cls, const float* queries, const float* pos_t, int B, int64_t L,
                             int Tx, int O, int C, int dtype, void* stream) {
  if (B < 0 || Tx < 1 || O < 1) return SVIT_EINVAL;
  int64_t total = (int64_t)B * (1 + Tx * O) * C;
  if (total == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == SVIT_F32)
    assemble_tokens_kernel<float><<<grid_for(total, 256), 256, 0, st>>>((float*)x, cls, queries, pos_t, B, L, Tx, O, C);
  else if (dtype == SVIT_BF16)
    assemble_tokens_kernel<bf16><<<grid_for(total, 256), 256, 0, st>>>((bf16*)x, cls, queries, pos_t, B, L, Tx, O, C);
  else
    return SVIT_EINVAL;
  SVIT_CHECK_LAUNCH();
  return 0;
}

int svit_assemble_tokens_bwd(const void* dx, float* dcls, float* dqueries, float* dpos_t, int B, int64_t L, int Tx,
                             int O, int C, int dtype, void* stream) {
  if (B < 0 || Tx < 1 || O < 1) return SVIT_EINVAL;
  int64_t total = (int64_t)(1 + Tx * O) * C;
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == SVIT_F32)
    assemble_tokens_bwd_kernel<float><<<grid_for(total, 128), 128, 0, st>>>((const float*)dx, dcls, dqueries, dpos_t, B, L, Tx, O, C);
  else if (dtype == SVIT_BF16)
    assemble_tokens_bwd_kernel<bf16><<<grid_for(total, 128), 128, 0, st>>>((const bf16*)dx, dcls, dqueries, dpos_t, B, L, Tx, O, C);
  else
    return SVIT_EINVAL;
  SVIT_CHECK_LAUNCH();
  return 0;
}

int svit_im2col3d(const void* x, void* cols, int B, int Cin, int T, int H, int W, int kt, int kh, int kw, int st_, int sh,
                  int sw, int pt, int ph, int pw, int Kpad, int in_dtype, int out_dtype, void* stream) {
  int To = (T + 2 * pt - kt) / st_ + 1, Ho = (H + 2 * ph - kh) / sh + 1, Wo = (W + 2 * pw - kw) / sw + 1;
  if (To < 1 || Ho < 1 || Wo < 1 || Kpad < Cin * kt * kh * kw) return SVIT_EINVAL;
  int64_t total = (int64_t)B * To * Ho * Wo * Kpad;
  if (total == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  if (out_dtype == SVIT_BF16) {
    int rc = svit_im2col_rows(x, cols, B, Cin, T, H, W, To, Ho, Wo, kt, kh, kw, st_, sh, sw, pt, ph, pw, Kpad, in_dtype, st);
    if (rc == 1) return 0;
    if (rc >= 1000) return rc - 1000;
  }
  int g = grid_for(total, 256);
#define IM2COL(TI, TO) im2col3d_kernel<TI, TO><<<g, 256, 0, st>>>((const TI*)x, (TO*)cols, B, Cin, T, H, W, To, Ho, Wo, kt, kh, kw, st_, sh, sw, pt, ph, pw, Kpad)
  if (in_dtype == SVIT_F32 && out_dtype == SVIT_F32) IM2COL(float, float);
  else if (in_dtype == SVIT_F32 && out_dtype == SVIT_BF16) IM2COL(float, bf16);
  else if (in_dtype == SVIT_BF16 && out_dtype == SVIT_BF16) IM2COL(bf16, bf16);
  else if (in_dtype == SVIT_BF16 && out_dtype == SVIT_F32) IM2COL(bf16, float);
  else return SVIT_EINVAL;
#undef IM2COL
  SVIT_CHECK_LAUNCH();
  return 0;
}

int svit_col2im3d(const void* cols, void* x, int B, int Cin, int T, int H, int W, int kt, int kh, int kw, int st_, int sh,
                  int sw, int pt, int ph, int pw, int Kpad, int in_dtype, int out_dtype, void* stream) {
  if (!cols || !x || B < 0 || Cin < 1 || T < 1 || H < 1 || W < 1 || st_ < 1 || sh < 1 || sw < 1 || pt < 0 || ph < 0 || pw < 0)
    return SVIT_EINVAL;
  int To = (T + 2 * pt - kt) / st_ + 1, Ho = (H + 2 * ph - kh) / sh + 1, Wo = (W + 2 * pw - kw) / sw + 1;
  if (To < 1 || Ho < 1 || Wo < 1 || Kpad < Cin * kt * kh * kw) return SVIT_EINVAL;
  int64_t total = (int64_t)B * Cin * T * H * W;
  if (total == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  int g = grid_for(total, 256);
#define COL2IM(TI, TO) col2im3d_kernel<TI, TO><<<g, 256, 0, st>>>((const TI*)cols, (TO*)x, B, Cin, T, H, W, To, Ho, Wo, kt, kh, kw, st_, sh, sw, pt, ph, pw, Kpad)
  if (in_dtype == SVIT_F32 && out_dtype == SVIT_F32) COL2IM(float, float);
  else if (in_dtype == SVIT_F32 && out_dtype == SVIT_BF16) COL2IM(float, bf16);
  else if (in_dtype == SVIT_BF16 && out_dtype == SVIT_BF16) COL2IM(bf16, bf16);
  else if (in_dtype == SVIT_BF16 && out_dtype == SVIT_F32) COL2IM(bf16, float);
  else return SVIT_EINVAL;
#undef COL2IM
  SVIT_CHECK_LAUNCH();
  return 0;
}

int svit_gather_cls_obj_fwd(const void* x, void* out, int B, int64_t N, int O, int C, int dtype, void* stream) {
  if (B < 0 || O < 0 || N < 1 + O) return SVIT_EINVAL;
  int64_t total = (int64_t)B * (1 + O) * C;
  if (total == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == SVIT_F32)
    gather_cls_obj_kernel<float><<<grid_for(total, 256), 256, 0, st>>>((const float*)x, (float*)out, B, N, O, C);
  else if (dtype == SVIT_BF16)
    gather_cls_obj_kernel<bf16><<<grid_for(total, 256), 256, 0, st>>>((const bf16*)x, (bf16*)out, B, N, O, C);
  else
    return SVIT_EINVAL;
  SVIT_CHECK_LAUNCH();
  return 0;
}

int svit_gather_cls_obj_bwd(const void* dout, void* dx, int B, int64_t N, int O, int C, int dtype, void* stream) {
  if (B < 0 || O < 0 || N < 1 + O) return SVIT_EINVAL;
  int64_t total = (int64_t)B * N * C;
  if (total == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == SVIT_F32)
    scatter_cls_obj_bwd_kernel<float><<<grid_for(total, 256), 256, 0, st>>>((const float*)dout, (float*)dx, B, N, O, C);
  else if (dtype == SVIT_BF16)
    scatter_cls_obj_bwd_kernel<bf16><<<grid_for(total, 256), 256, 0, st>>>((const bf16*)dout, (bf16*)dx, B, N, O, C);
  else
    return SVIT_EINVAL;
  SVIT_CHECK_LAUNCH();
  return 0;
}

int svit_scale_rows(const void* x, const float* scale, void* y, int64_t rows, int C, int64_t rows_per_sample, int dtype,
                    void* stream) {
  if (rows < 0 || rows_per_sample <= 0) return SVIT_EINVAL;
  if (rows == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == SVIT_F32)
    scale_rows_kernel<float><<<grid_for(rows * C, 256), 256, 0, st>>>((const float*)x, scale, (float*)y, rows, C, rows_per_sample);
  else if (dtype == SVIT_BF16 && C % 8 == 0 &&
           ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(y)) & 15) == 0)
    scale_rows_bf16x8_kernel<<<grid_for(rows * (C / 8), 256), 256, 0, st>>>((const bf16*)x, scale, (bf16*)y, rows * (C / 8), C / 8,
                                                                            rows_per_sample);
  else if (dtype == SVIT_BF16)
    scale_rows_kernel<bf16><<<grid_for(rows * C, 256), 256, 0, st>>>((const bf16*)x, scale, (bf16*)y, rows, C, rows_per_sample);
  else
    return SVIT_EINVAL;
  SVIT_CHECK_LAUNCH();
  return 0;
}

}  // extern "C"
