// PatchEmbed (Conv3d k(3,7,7) s(2,4,4) p(1,3,3) + flatten/transpose, slowfast/models/stem_helper.py:309-320) as an IMPLICIT
// GEMM on the 5th-generation tensor cores: no im2col matrix is ever written (round 1 materialised 1.44 GB of it per
// batch-64 step).
//
// Space-to-depth view.  The clip is held as cells X'[b, tc, hc, wc, (c, tt, hh, ww)] -- one cell = the stride-sized block
// st x sh x sw of all input channels (3 x 2 x 4 x 4 = 96 values for ssv2.yaml), written in that layout by the input
// kernels below (svit_s2d_from_u8 fuses it with the uint8 -> normalised conversion, so it costs no extra pass).  A strided
// convolution then is a stride-1 convolution over cells with ceil-sized taps: output (t', h', w') reads the cells
// (t' + dt, h' + dh, w' + dw), dt/dh/dw in {-1, 0} here, i.e. K = 8 taps x 96 values = 768 against the zero-padded weight
// matrix W'[E, tap, cell] (the 441 real taps scattered into it; 1.74x the MACs, all of them on the tensor pipe).
// Each tap of an output tile (R rows x Wo positions <= 128) is ONE shifted TMA box of the cell tensor -- the conv padding
// is the TMA out-of-bounds zero fill -- so the A operand never exists in global memory.
//
// Persistent CTAs, 1 per SM, 192 threads: warp 0 = TMA producer (3-stage ring, one tap per stage: cell/32 chunks of
// [rows x 32] bf16, 64-byte swizzle), warp 1 = tcgen05.mma issuer (M 128 x N E x K 16; W' resident in shared memory,
// 147 KB, loaded once per CTA), warps 2-5 = epilogue (thread = TMEM lane = output position: + bias -> bf16 -> the token
// row out[b, row_off + (t' Ho + h') Wo + w', :]); accumulators double-buffered in TMEM.
#include <cstdlib>

#include "tc_common.cuh"
#include "../../include/svit_b200.h"

namespace {

constexpr int PE_THREADS = 192;
constexpr int PE_STAGES = 3;
constexpr int PE_CHUNK_A = 8192;  // 128 rows x 64 B
constexpr int PE_MAX_E = 256;

struct PeParams {
  int B, Tc, Hc, Wc;        // cell grid
  int To, Ho, Wo;           // output grid
  int nt, nh, nw;           // taps per dimension
  int lo_t, lo_h, lo_w;     // first tap offset (cells) per dimension
  int chunks;               // cell values / 32
  int E;                    // output channels
  int R;                    // output rows (h') per tile
  int tiles_h;
  int64_t tiles;
  int64_t out_bs;           // elements between samples of `out`
  int row_off;              // first patch row of a sample (1: the cls token sits in row 0)
  const float* bias;
  bf16* out;
  int w_chunk_bytes;        // E x 64 B
  int uniq;                 // 0: one shifted TMA box per tap; 1: every cell once, taps = row-shifted descriptors
  int PW, PH;               // uniq: box extent in w / h (Wo + nw - 1, R + nh - 1)
  int chunk_a;              // bytes reserved per A chunk
};

// K-major, 64-byte swizzle (rows of 64 B, 8-row groups 512 B apart).  base_off = the descriptor's "matrix base offset"
// (bits 49-51): the phase of the swizzle pattern when the start address is not aligned to the pattern's repeat.
__device__ __forceinline__ uint64_t pe_desc_sw64(uint32_t smem_addr, uint32_t base_off = 0) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);
  d |= (uint64_t)(16 >> 4) << 16;
  d |= (uint64_t)(512 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)(base_off & 7) << 49;
  d |= (uint64_t)4 << 61;
  return d;
}

__device__ __forceinline__ uint32_t pe_pack2(float a, float b) {
  __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&v);
}

template <int E>
__global__ void __launch_bounds__(PE_THREADS, 1)
patch_embed_tc_kernel(const __grid_constant__ CUtensorMap tmap_x, const __grid_constant__ CUtensorMap tmap_w, PeParams p) {
  extern __shared__ unsigned char smem_raw[];
  unsigned char* smem = smem_raw + ((1024u - (tc::smem_u32(smem_raw) & 1023u)) & 1023u);
  const int ntaps = p.nt * p.nh * p.nw;
  const int w_bytes = ntaps * p.chunks * p.w_chunk_bytes;
  unsigned char* s_w = smem;                                        // [ntaps][chunks][E x 64 B]
  unsigned char* s_a = smem + ((w_bytes + 1023) & ~1023);           // [PE_STAGES][chunks][128 x 64 B]
  const int a_stage = p.chunks * p.chunk_a;
  const int n_stages = p.uniq ? 2 : PE_STAGES;
  uint64_t* bars = reinterpret_cast<uint64_t*>(s_a + n_stages * a_stage + 2048);  // 2 KB slack: shifted views read past a chunk
  uint64_t* full = bars;                    // [PE_STAGES]
  uint64_t* empty = bars + PE_STAGES;       // [PE_STAGES]
  uint64_t* tmem_full = bars + 2 * PE_STAGES;   // [2]
  uint64_t* tmem_empty = tmem_full + 2;         // [2]
  uint64_t* w_full = tmem_empty + 2;
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(w_full + 1);
  float* s_bias = reinterpret_cast<float*>(tmem_ptr + 4);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 0 && lane == 0) {
    tc::prefetch_tmap(&tmap_x);
    tc::prefetch_tmap(&tmap_w);
    for (int i = 0; i < PE_STAGES; ++i) {  // (uniq uses the first two of each)
      tc::mbar_init(&full[i], 1);
      tc::mbar_init(&empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      tc::mbar_init(&tmem_full[i], 1);
      tc::mbar_init(&tmem_empty[i], 4);  // one arrival per epilogue warp
    }
    tc::mbar_init(w_full, 1);
    tc::fence_barrier_init();
  }
  if (warp == 1) tc::tmem_alloc(tmem_ptr, 2 * (E <= 128 ? 128 : 256));
  for (int i = threadIdx.x; i < E; i += PE_THREADS) s_bias[i] = p.bias ? p.bias[i] : 0.f;
  tc::fence_before_sync();
  __syncthreads();
  tc::fence_after_sync();
  const uint32_t tmem_base = *tmem_ptr;
  constexpr int ACC_COLS = E <= 128 ? 128 : 256;

  if (warp == 0) {
    // =========================== TMA producer ===========================
    if (tc::elect_one()) {
      // the whole weight matrix, once
      tc::mbar_arrive_expect_tx(w_full, (uint32_t)w_bytes);
      for (int c = 0; c < ntaps * p.chunks; ++c)
        tc::tma_load_2d(s_w + c * p.w_chunk_bytes, &tmap_w, w_full, c * 32, 0);
      const uint32_t stage_bytes = (uint32_t)(p.chunks * (p.uniq ? p.PH * p.PW : p.R * p.Wo) * 64);
      int n = 0;  // ring position
      for (int64_t tile = blockIdx.x; tile < p.tiles; tile += gridDim.x) {
        const int hb = (int)(tile % p.tiles_h);
        const int64_t r = tile / p.tiles_h;
        const int to = (int)(r % p.To), b = (int)(r / p.To);
        if (p.uniq) {  // one stage = one temporal tap plane: every cell of the tile's halo box exactly once
          for (int it = 0; it < p.nt; ++it, ++n) {
            const int s = n & 1;
            tc::mbar_wait(&empty[s], ((n >> 1) & 1) ^ 1);
            tc::mbar_arrive_expect_tx(&full[s], stage_bytes);
            for (int c = 0; c < p.chunks; ++c)
              tc::tma_load_5d(s_a + s * a_stage + c * p.chunk_a, &tmap_x, &full[s], c * 32, p.lo_w, hb * p.R + p.lo_h,
                              to + p.lo_t + it, b);
          }
          continue;
        }
        for (int it = 0; it < p.nt; ++it)
          for (int ih = 0; ih < p.nh; ++ih)
            for (int iw = 0; iw < p.nw; ++iw, ++n) {
              const int s = n % PE_STAGES;
              tc::mbar_wait(&empty[s], ((n / PE_STAGES) & 1) ^ 1);
              tc::mbar_arrive_expect_tx(&full[s], stage_bytes);
              for (int c = 0; c < p.chunks; ++c)
                tc::tma_load_5d(s_a + s * a_stage + c * p.chunk_a, &tmap_x, &full[s], c * 32, p.lo_w + iw,
                                hb * p.R + p.lo_h + ih, to + p.lo_t + it, b);
            }
      }
    }
  } else if (warp == 1) {
    // =========================== MMA issuer ===========================
    if (tc::elect_one()) {
      constexpr uint32_t idesc = tc::idesc_bf16(128, E, 0, 0);
      tc::mbar_wait(w_full, 0);
      tc::fence_after_sync();
      const uint32_t sw = tc::smem_u32(s_w), sa = tc::smem_u32(s_a);
      int n = 0, lt = 0;
      for (int64_t tile = blockIdx.x; tile < p.tiles; tile += gridDim.x, ++lt) {
        const int as = lt & 1;
        tc::mbar_wait(&tmem_empty[as], ((lt >> 1) & 1) ^ 1);
        tc::fence_after_sync();
        const uint32_t d = tmem_base + as * ACC_COLS;
        if (p.uniq) {
          for (int it = 0; it < p.nt; ++it, ++n) {
            const int s = n & 1;
            tc::mbar_wait(&full[s], (n >> 1) & 1);
            tc::fence_after_sync();
            for (int ih = 0; ih < p.nh; ++ih)
              for (int iw = 0; iw < p.nw; ++iw) {
                const int tap = (it * p.nh + ih) * p.nw + iw;
                const uint32_t shift = (uint32_t)(ih * p.PW + iw) * 64u;  // the tap = the same cells, rows shifted
                for (int c = 0; c < p.chunks; ++c) {
                  const uint32_t a0 = sa + s * a_stage + c * p.chunk_a + shift;
                  const uint32_t b0 = sw + (tap * p.chunks + c) * p.w_chunk_bytes;
#pragma unroll
                  for (int k = 0; k < 2; ++k)
                    tc::umma_bf16_ss(d, pe_desc_sw64(a0 + k * 32), pe_desc_sw64(b0 + k * 32), idesc,
                                     (it | ih | iw | c | k) != 0 ? 1u : 0u);
                }
              }
            tc::umma_commit(&empty[s]);
          }
          tc::umma_commit(&tmem_full[as]);
          continue;
        }
        for (int tap = 0; tap < ntaps; ++tap, ++n) {
          const int s = n % PE_STAGES;
          tc::mbar_wait(&full[s], (n / PE_STAGES) & 1);
          tc::fence_after_sync();
          for (int c = 0; c < p.chunks; ++c) {
            const uint32_t a0 = sa + s * a_stage + c * p.chunk_a;
            const uint32_t b0 = sw + (tap * p.chunks + c) * p.w_chunk_bytes;
#pragma unroll
            for (int k = 0; k < 2; ++k)
              tc::umma_bf16_ss(d, pe_desc_sw64(a0 + k * 32), pe_desc_sw64(b0 + k * 32), idesc, (tap | c | k) != 0 ? 1u : 0u);
          }
          tc::umma_commit(&empty[s]);
        }
        tc::umma_commit(&tmem_full[as]);
      }
    }
  } else {
    // =========================== epilogue ===========================
    const int q = warp & 3;                 // TMEM lane quarter of this warp (warps 2..5 -> quarters 2, 3, 0, 1)
    const int i = q * 32 + lane;            // row of the tile = TMEM lane
    const uint32_t lane_addr = tmem_base + ((uint32_t)(q * 32) << 16);
    const int pitch = p.uniq ? p.PW : p.Wo;  // uniq: output (hrow, w) sits at row hrow * PW + w of the halo box
    const int hrow = i / pitch, w = i - hrow * pitch;
    int lt = 0;
    for (int64_t tile = blockIdx.x; tile < p.tiles; tile += gridDim.x, ++lt) {
      const int as = lt & 1;
      const int hb = (int)(tile % p.tiles_h);
      const int64_t r = tile / p.tiles_h;
      const int to = (int)(r % p.To), b = (int)(r / p.To);
      const int h = hb * p.R + hrow;
      const bool valid = hrow < p.R && h < p.Ho && w < p.Wo;
      tc::mbar_wait(&tmem_full[as], (lt >> 1) & 1);
      tc::fence_after_sync();
      bf16* dst = p.out + (int64_t)b * p.out_bs + ((int64_t)p.row_off + ((int64_t)to * p.Ho + h) * p.Wo + w) * E;
#pragma unroll
      for (int c0 = 0; c0 < E; c0 += 32) {
        float v[32];
        tc::tmem_ld32(lane_addr + as * ACC_COLS + c0, v);
        tc::tmem_ld_wait();
        if (valid) {
#pragma unroll
          for (int u = 0; u < 32; u += 8) {
            const uint4 o = {pe_pack2(v[u] + s_bias[c0 + u], v[u + 1] + s_bias[c0 + u + 1]),
                             pe_pack2(v[u + 2] + s_bias[c0 + u + 2], v[u + 3] + s_bias[c0 + u + 3]),
                             pe_pack2(v[u + 4] + s_bias[c0 + u + 4], v[u + 5] + s_bias[c0 + u + 5]),
                             pe_pack2(v[u + 6] + s_bias[c0 + u + 6], v[u + 7] + s_bias[c0 + u + 7])};
            *reinterpret_cast<uint4*>(dst + c0 + u) = o;
          }
        }
      }
      tc::fence_before_sync();
      __syncwarp();
      if (lane == 0) tc::mbar_arrive(&tmem_empty[as]);
    }
  }
  tc::fence_before_sync();
  __syncthreads();
  if (warp == 1) {
    tc::fence_after_sync();
    tc::tmem_dealloc(tmem_base, 2 * ACC_COLS);
  }
}

// ------------------------------------------------------------------------------------------------ space-to-depth input
// out[b, tc, hc, wc, ((c st + tt) sh + hh) sw + ww] = x[b, c, tc st + tt, hc sh + hh, wc sw + ww]   (0 beyond T / H / W)
struct S2dGeom {
  int B, C, T, H, W, st, sh, sw, Tc, Hc, Wc;
};

// uint8 frames [B, T, H, W, 3] -> normalised cells (datasets/utils.py:287-303 fused): thread = (b, t, h, wc): the sw
// pixels of a cell row are sw * C contiguous bytes
__global__ void __launch_bounds__(256) s2d_from_u8_kernel(const uint8_t* __restrict__ in, bf16* __restrict__ out, S2dGeom g,
                                                          float m0, float m1, float m2, float s0, float s1, float s2) {
  const float mean[3] = {m0, m1, m2}, sd[3] = {s0, s1, s2};
  const int64_t total = (int64_t)g.B * g.Tc * g.st * g.Hc * g.sh * g.Wc;
  const int cell = g.C * g.st * g.sh * g.sw;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int wc = (int)(i % g.Wc);
    int64_t r = i / g.Wc;
    const int h = (int)(r % (g.Hc * g.sh));
    r /= g.Hc * g.sh;
    const int t = (int)(r % (g.Tc * g.st));
    const int b = (int)(r / (g.Tc * g.st));
    const int tc_ = t / g.st, tt = t - tc_ * g.st, hc = h / g.sh, hh = h - hc * g.sh;
    bf16* dst = out + ((((int64_t)b * g.Tc + tc_) * g.Hc + hc) * g.Wc + wc) * cell;
    const bool row_ok = t < g.T && h < g.H;
    const uint8_t* src = in + ((((int64_t)b * g.T + t) * g.H + h) * g.W + (int64_t)wc * g.sw) * g.C;
    for (int c = 0; c < g.C; ++c) {
      bf16* d = dst + ((c * g.st + tt) * g.sh + hh) * g.sw;
      auto val = [&](int ww) {
        float v = 0.f;
        if (row_ok && wc * g.sw + ww < g.W)
          v = __fdiv_rn(__fsub_rn(__fdiv_rn((float)__ldg(src + ww * g.C + c), 255.0f), mean[c < 3 ? c : 2]), sd[c < 3 ? c : 2]);
        return v;
      };
      if (g.sw == 4) {  // one 8-byte store per channel (the cell row is 8-byte aligned)
        __nv_bfloat162 a = __floats2bfloat162_rn(val(0), val(1)), b2 = __floats2bfloat162_rn(val(2), val(3));
        *reinterpret_cast<uint2*>(d) = make_uint2(*reinterpret_cast<uint32_t*>(&a), *reinterpret_cast<uint32_t*>(&b2));
      } else {
        for (int ww = 0; ww < g.sw; ++ww) d[ww] = __float2bfloat16_rn(val(ww));
      }
    }
  }
}

// bf16 / fp32 clip [B, C, T, H, W] -> cells: thread = (b, c, t, h, wc), sw consecutive input values -> sw consecutive cell values
template <typename T>
__global__ void __launch_bounds__(256) s2d_from_clip_kernel(const T* __restrict__ in, bf16* __restrict__ out, S2dGeom g) {
  const int64_t total = (int64_t)g.B * g.C * g.Tc * g.st * g.Hc * g.sh * g.Wc;
  const int cell = g.C * g.st * g.sh * g.sw;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int wc = (int)(i % g.Wc);
    int64_t r = i / g.Wc;
    const int h = (int)(r % (g.Hc * g.sh));
    r /= g.Hc * g.sh;
    const int t = (int)(r % (g.Tc * g.st));
    r /= g.Tc * g.st;
    const int c = (int)(r % g.C);
    const int b = (int)(r / g.C);
    const int tc_ = t / g.st, tt = t - tc_ * g.st, hc = h / g.sh, hh = h - hc * g.sh;
    bf16* dst = out + ((((int64_t)b * g.Tc + tc_) * g.Hc + hc) * g.Wc + wc) * cell + ((c * g.st + tt) * g.sh + hh) * g.sw;
    const bool row_ok = t < g.T && h < g.H;
    const T* src = in + ((((int64_t)b * g.C + c) * g.T + t) * g.H + h) * g.W + (int64_t)wc * g.sw;
    if (g.sw == 4 && row_ok && wc * 4 + 3 < g.W) {
      __nv_bfloat162 a = __floats2bfloat162_rn(to_f(src[0]), to_f(src[1])), b2 = __floats2bfloat162_rn(to_f(src[2]), to_f(src[3]));
      *reinterpret_cast<uint2*>(dst) = make_uint2(*reinterpret_cast<uint32_t*>(&a), *reinterpret_cast<uint32_t*>(&b2));
    } else {
      for (int ww = 0; ww < g.sw; ++ww)
        dst[ww] = (row_ok && wc * g.sw + ww < g.W) ? __float2bfloat16_rn(to_f(src[ww])) : __float2bfloat16_rn(0.f);
    }
  }
}

// Fast path for sw == 4, W == 4 Wc, H == sh Hc, T == st Tc (ssv2.yaml): one CTA per row of cells (b, tc, hc).  The C st sh
// input rows that feed it are read with coalesced 8-byte (clip) / 12-byte (uint8 pixel quad) accesses into a shared-memory
// tile laid out like the output, which then leaves as one contiguous Wc x cell x 2-byte stream of 16-byte stores.
template <int KIND>  // 0: fp32 clip, 1: bf16 clip, 2: uint8 frames
__global__ void __launch_bounds__(256) s2d_rows_kernel(const void* __restrict__ in, bf16* __restrict__ out, S2dGeom g, float m0,
                                                       float m1, float m2, float s0, float s1, float s2) {
  extern __shared__ __align__(16) unsigned char s2d_smem[];
  bf16* tile = reinterpret_cast<bf16*>(s2d_smem);  // [Wc][cell]
  const int cell = g.C * g.st * g.sh * 4;
  const int hc = blockIdx.x % g.Hc, tc_ = (blockIdx.x / g.Hc) % g.Tc, b = blockIdx.x / (g.Hc * g.Tc);
  const int rows = g.C * g.st * g.sh;
  if (KIND == 2) {
    // (v / 255 - mean) / std has 256 possible results per channel: the CTA computes them once with the reference's exact
    // fp32 operation order (two IEEE divisions each) and every pixel is a table lookup -- bit-identical to computing it
    // per pixel, which spent 24 divisions per 12-byte pixel quad (0.53 ms per 64 clips against 0.20 ms from a bf16 clip)
    __shared__ uint16_t lut[3 * 256];
    for (int i = threadIdx.x; i < g.C * 256; i += blockDim.x) {
      const int c = i >> 8;
      const float mc = c == 0 ? m0 : (c == 1 ? m1 : m2), sc = c == 0 ? s0 : (c == 1 ? s1 : s2);
      const __nv_bfloat16 h = __float2bfloat16_rn(__fdiv_rn(__fsub_rn(__fdiv_rn((float)(i & 255), 255.0f), mc), sc));
      lut[i] = *reinterpret_cast<const uint16_t*>(&h);
    }
    __syncthreads();
    const uint8_t* src = reinterpret_cast<const uint8_t*>(in);
    for (int i = threadIdx.x; i < g.st * g.sh * g.Wc; i += blockDim.x) {
      const int wc = i % g.Wc, r = i / g.Wc;
      const int hh = r % g.sh, tt = r / g.sh;
      const uint32_t* px = reinterpret_cast<const uint32_t*>(
          src + ((((int64_t)b * g.T + tc_ * g.st + tt) * g.H + hc * g.sh + hh) * g.W + (int64_t)wc * 4) * g.C);
      uint8_t by[12];
      if (g.C == 3) {
        const uint32_t a = __ldg(px), bq = __ldg(px + 1), cq = __ldg(px + 2);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          by[k] = (a >> (8 * k)) & 255u;
          by[4 + k] = (bq >> (8 * k)) & 255u;
          by[8 + k] = (cq >> (8 * k)) & 255u;
        }
      } else {
        const uint8_t* pb = reinterpret_cast<const uint8_t*>(px);
        for (int k = 0; k < 4 * g.C; ++k) by[k] = __ldg(pb + k);
      }
      for (int c = 0; c < g.C; ++c) {
        const uint16_t* l = lut + c * 256;
        const uint32_t lo = (uint32_t)l[by[c]] | ((uint32_t)l[by[g.C + c]] << 16);
        const uint32_t hi = (uint32_t)l[by[2 * g.C + c]] | ((uint32_t)l[by[3 * g.C + c]] << 16);
        *reinterpret_cast<uint2*>(tile + wc * cell + ((c * g.st + tt) * g.sh + hh) * 4) = make_uint2(lo, hi);
      }
    }
  } else {
    // item = 8 consecutive input values of one of the C st sh input rows (two cells): 16-byte (bf16) / 2 x 16-byte (fp32)
    // loads, four items in flight per thread before the first shared-memory write (the kernel is latency-bound otherwise)
    const int half = g.Wc >> 1;  // Wc is even on this path
    const int n = rows * half;
    for (int base = threadIdx.x; base < n; base += 4 * blockDim.x) {
      uint4 v[4];
      int dsto[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int i = base + u * blockDim.x;
        dsto[u] = -1;
        if (i < n) {
          const int wp = i % half, r = i / half;  // r = (c st + tt) sh + hh
          const int hh = r % g.sh, tt = (r / g.sh) % g.st, c = r / (g.sh * g.st);
          const int64_t off = ((((int64_t)b * g.C + c) * g.T + tc_ * g.st + tt) * g.H + hc * g.sh + hh) * g.W + (int64_t)wp * 8;
          if (KIND == 1) {
            v[u] = __ldg(reinterpret_cast<const uint4*>(reinterpret_cast<const bf16*>(in) + off));
          } else {
            const float4 f0 = __ldg(reinterpret_cast<const float4*>(reinterpret_cast<const float*>(in) + off));
            const float4 f1 = __ldg(reinterpret_cast<const float4*>(reinterpret_cast<const float*>(in) + off + 4));
            __nv_bfloat162 a0 = __floats2bfloat162_rn(f0.x, f0.y), a1 = __floats2bfloat162_rn(f0.z, f0.w);
            __nv_bfloat162 a2 = __floats2bfloat162_rn(f1.x, f1.y), a3 = __floats2bfloat162_rn(f1.z, f1.w);
            v[u] = make_uint4(*reinterpret_cast<uint32_t*>(&a0), *reinterpret_cast<uint32_t*>(&a1),
                              *reinterpret_cast<uint32_t*>(&a2), *reinterpret_cast<uint32_t*>(&a3));
          }
          dsto[u] = (2 * wp) * cell + r * 4;
        }
      }
#pragma unroll
      for (int u = 0; u < 4; ++u)
        if (dsto[u] >= 0) {
          *reinterpret_cast<uint2*>(tile + dsto[u]) = make_uint2(v[u].x, v[u].y);
          *reinterpret_cast<uint2*>(tile + dsto[u] + cell) = make_uint2(v[u].z, v[u].w);
        }
    }
  }
  __syncthreads();
  uint4* dst = reinterpret_cast<uint4*>(out + (((int64_t)b * g.Tc + tc_) * g.Hc + hc) * g.Wc * cell);
  const uint4* st4 = reinterpret_cast<const uint4*>(tile);
  for (int i = threadIdx.x; i < g.Wc * cell / 8; i += blockDim.x) dst[i] = st4[i];
}

// Depth-to-space, the inverse of the cell layout (data gradient of svit_s2d_clip): x[b, c, t, h, w] = cells[b, t / st,
// h / sh, w / sw, ((c st + t % st) sh + h % sh) sw + w % sw] for t < T, h < H, w < W (the rest of a partial cell is
// dropped).  One CTA per row of cells (b, tc, hc): the row is read as one contiguous stream (into shared memory when it
// fits 48 KB), then written as C st sh output rows, coalesced along w.  vec: sw == 4, W == 4 Wc, 16-byte aligned rows --
// a thread moves one cell row (4 values).
template <typename T>
__global__ void __launch_bounds__(256) d2s_rows_kernel(const bf16* __restrict__ cells, T* __restrict__ x, S2dGeom g, int vec,
                                                       int staged) {
  extern __shared__ __align__(16) unsigned char d2s_smem[];
  const int cell = g.C * g.st * g.sh * g.sw;
  const int hc = blockIdx.x % g.Hc, tc_ = (blockIdx.x / g.Hc) % g.Tc, b = blockIdx.x / (g.Hc * g.Tc);
  const bf16* src = cells + (((int64_t)b * g.Tc + tc_) * g.Hc + hc) * g.Wc * cell;
  const bf16* rd = src;
  if (staged) {
    bf16* tile = reinterpret_cast<bf16*>(d2s_smem);  // [Wc][cell]
    const int n = g.Wc * cell;
    if (vec) {
      for (int i = threadIdx.x; i < n / 8; i += blockDim.x)
        reinterpret_cast<uint4*>(tile)[i] = __ldg(reinterpret_cast<const uint4*>(src) + i);
    } else {
      for (int i = threadIdx.x; i < n; i += blockDim.x) tile[i] = src[i];
    }
    __syncthreads();
    rd = tile;
  }
  const int rows = g.C * g.st * g.sh;  // r = (c st + tt) sh + hh
  if (vec) {
    for (int i = threadIdx.x; i < rows * g.Wc; i += blockDim.x) {
      const int wc = i % g.Wc, r = i / g.Wc;
      const int hh = r % g.sh, tt = (r / g.sh) % g.st, c = r / (g.sh * g.st);
      const int t = tc_ * g.st + tt, h = hc * g.sh + hh;
      if (t >= g.T || h >= g.H) continue;
      const uint2 v = *reinterpret_cast<const uint2*>(rd + wc * cell + r * 4);
      const float2 a = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&v.x));
      const float2 c2 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&v.y));
      T* d = x + ((((int64_t)b * g.C + c) * g.T + t) * g.H + h) * g.W + (int64_t)wc * 4;
      if constexpr (sizeof(T) == 4) {
        *reinterpret_cast<float4*>(d) = make_float4(a.x, a.y, c2.x, c2.y);
      } else {
        *reinterpret_cast<uint2*>(d) = v;
      }
    }
    return;
  }
  const int wmax = g.W;  // < Wc sw
  for (int i = threadIdx.x; i < rows * wmax; i += blockDim.x) {
    const int w = i % wmax, r = i / wmax;
    const int hh = r % g.sh, tt = (r / g.sh) % g.st, c = r / (g.sh * g.st);
    const int t = tc_ * g.st + tt, h = hc * g.sh + hh;
    if (t >= g.T || h >= g.H) continue;
    const int wc = w / g.sw;
    x[((((int64_t)b * g.C + c) * g.T + t) * g.H + h) * g.W + w] = from_f<T>(__bfloat162float(rd[wc * cell + r * g.sw + (w - wc * g.sw)]));
  }
}

}  // namespace

extern "C" {

int svit_s2d_clip(const void* x, void* cells, int B, int C, int T, int H, int W, int st, int sh, int sw, int in_kind,
                  float mean0, float mean1, float mean2, float std0, float std1, float std2, void* stream) {
  if (!x || !cells || B < 0 || C < 1 || T < 1 || H < 1 || W < 1 || st < 1 || sh < 1 || sw < 1) return SVIT_EINVAL;
  if (B == 0) return 0;
  S2dGeom g{B, C, T, H, W, st, sh, sw, (T + st - 1) / st, (H + sh - 1) / sh, (W + sw - 1) / sw};
  cudaStream_t s = (cudaStream_t)stream;
  const int cell = C * st * sh * sw;
  const bool aligned = (reinterpret_cast<uintptr_t>(x) & 15) == 0 && (reinterpret_cast<uintptr_t>(cells) & 15) == 0;
  if (sw == 4 && W == 4 * g.Wc && g.Wc % 2 == 0 && H == sh * g.Hc && T == st * g.Tc && cell % 8 == 0 && aligned &&
      (in_kind != 2 || C <= 3) &&
      (size_t)g.Wc * cell * 2 <= 48 * 1024 && (int64_t)B * g.Tc * g.Hc < (1ll << 31)) {
    const unsigned grid = (unsigned)((int64_t)B * g.Tc * g.Hc);
    const size_t sm = (size_t)g.Wc * cell * 2;
    if (in_kind == 2) s2d_rows_kernel<2><<<grid, 256, sm, s>>>(x, (bf16*)cells, g, mean0, mean1, mean2, std0, std1, std2);
    else if (in_kind == SVIT_BF16) s2d_rows_kernel<1><<<grid, 256, sm, s>>>(x, (bf16*)cells, g, 0, 0, 0, 1, 1, 1);
    else if (in_kind == SVIT_F32) s2d_rows_kernel<0><<<grid, 256, sm, s>>>(x, (bf16*)cells, g, 0, 0, 0, 1, 1, 1);
    else return SVIT_EINVAL;
    SVIT_CHECK_LAUNCH();
    return 0;
  }
  const int64_t rows = (int64_t)B * g.Tc * st * g.Hc * sh * g.Wc;
  const int64_t n = in_kind == 2 ? rows : rows * C;
  int64_t grid = (n + 255) / 256;
  const int64_t cap = (int64_t)svit_num_sms() * 32;
  if (grid > cap) grid = cap;
  if (in_kind == 2) {  // uint8 frames [B, T, H, W, C], C <= 3
    if (C > 3) return SVIT_ENOTSUP;
    s2d_from_u8_kernel<<<(unsigned)grid, 256, 0, s>>>((const uint8_t*)x, (bf16*)cells, g, mean0, mean1, mean2, std0, std1, std2);
  } else if (in_kind == SVIT_BF16) {
    s2d_from_clip_kernel<bf16><<<(unsigned)grid, 256, 0, s>>>((const bf16*)x, (bf16*)cells, g);
  } else if (in_kind == SVIT_F32) {
    s2d_from_clip_kernel<float><<<(unsigned)grid, 256, 0, s>>>((const float*)x, (bf16*)cells, g);
  } else {
    return SVIT_EINVAL;
  }
  SVIT_CHECK_LAUNCH();
  return 0;
}


int svit_d2s_clip(const void* cells, void* x, int B, int C, int T, int H, int W, int st, int sh, int sw, int out_dtype,
                  void* stream) {
  if (!cells || !x || B < 0 || C < 1 || T < 1 || H < 1 || W < 1 || st < 1 || sh < 1 || sw < 1) return SVIT_EINVAL;
  if (out_dtype != SVIT_F32 && out_dtype != SVIT_BF16) return SVIT_EINVAL;
  if (B == 0) return 0;
  S2dGeom g{B, C, T, H, W, st, sh, sw, (T + st - 1) / st, (H + sh - 1) / sh, (W + sw - 1) / sw};
  const int cell = C * st * sh * sw;
  if ((int64_t)B * g.Tc * g.Hc >= (1ll << 31) || (int64_t)g.Wc * cell >= (1ll << 31)) return SVIT_ENOTSUP;
  const bool aligned = (reinterpret_cast<uintptr_t>(x) & 15) == 0 && (reinterpret_cast<uintptr_t>(cells) & 15) == 0;
  const int vec = sw == 4 && W == 4 * g.Wc && ((int64_t)g.Wc * cell) % 8 == 0 && aligned;
  const size_t tile = (size_t)g.Wc * cell * 2;
  const int staged = tile <= 48 * 1024;
  const unsigned grid = (unsigned)((int64_t)B * g.Tc * g.Hc);
  cudaStream_t s = (cudaStream_t)stream;
  if (out_dtype == SVIT_F32)
    d2s_rows_kernel<float><<<grid, 256, staged ? tile : 0, s>>>((const bf16*)cells, (float*)x, g, vec, staged);
  else
    d2s_rows_kernel<bf16><<<grid, 256, staged ? tile : 0, s>>>((const bf16*)cells, (bf16*)x, g, vec, staged);
  SVIT_CHECK_LAUNCH();
  return 0;
}
}  // extern "C"

// First cell-tap offset (floor(-p / s)) and tap count of one dimension of a stride-s, padding-p, size-k convolution.
static void pe_taps(int k, int s, int pad, int* lo, int* n) {
  auto fl = [](int a, int b) { return a >= 0 ? a / b : -((-a + b - 1) / b); };
  *lo = fl(-pad, s);
  *n = fl(k - 1 - pad, s) - *lo + 1;
}

static int64_t pe_smem_bytes(int ntaps, int chunks, int n_cols, int stages, int chunk_a) {
  return (((int64_t)ntaps * chunks * n_cols * 64 + 1023) & ~(int64_t)1023) + (int64_t)stages * chunks * chunk_a + 2048 + 1024 +
         256 + PE_MAX_E * 4;
}

static bool pe_n_ok(int n) { return n == 32 || n == 64 || n == 96 || n == 128 || n == 192 || n == 256; }

// One stride-1 implicit-GEMM convolution over a channels-last 5-D input `in` (dims {K1, Wi, Hi, Ti, B} innermost first,
// byte strides of the outer four; K1 = p.chunks * 32 values per position) into rows row_off + (t Ho + h) Wo + w of
// every sample of p.out (p.E values each).  p carries the output grid (To, Ho, Wo), the taps (nt, nh, nw) and their
// first offsets (lo_*); w2 [p.E, ntaps * K1] bf16.  Used as the stem forward (in = cells, out = patch rows) and as its
// data gradient (in = the patch rows of the sequence gradient, out = cell gradients).
static int pe_launch(PeParams p, const void* in, const cuuint64_t in_dims[5], const cuuint64_t in_strides[4], const void* w2,
                     cudaStream_t s) {
  const int E = p.E;
  if (p.Wo < 1 || p.Wo > 128 || p.Ho < 1 || p.To < 1 || (E * 2) % 16) return SVIT_ENOTSUP;
  // SVIT_PE_MODE=0: one shifted TMA box per tap (every cell fetched up to 8 times from L2); 1 (default): every cell of the
  // tile's halo box once, the taps are row-shifted views of it -- the swizzle of a K-major tile is a function of the
  // absolute shared-memory address, so a descriptor whose start is shifted by whole rows (base offset 0) reads exactly the
  // rows TMA wrote (checked on B200: tests/test_gpu_parity.py::test_patch_embed_implicit_gemm; 412 -> 351 us at B = 64)
  static const int mode = []() { const char* e = getenv("SVIT_PE_MODE"); return e ? atoi(e) : 1; }();
  p.uniq = mode ? 1 : 0;
  p.PW = p.Wo + p.nw - 1;
  if (p.uniq && (p.PW > 128 || p.PW > 256)) p.uniq = 0;
  if (p.uniq) {
    p.R = (128 - p.Wo) / p.PW + 1;
  } else {
    p.R = 128 / p.Wo;
  }
  if (p.R > p.Ho) p.R = p.Ho;
  p.PH = p.R + p.nh - 1;
  p.chunk_a = p.uniq ? ((p.PH * p.PW * 64 + 1023) & ~1023) : PE_CHUNK_A;
  p.tiles_h = (p.Ho + p.R - 1) / p.R;
  p.tiles = (int64_t)p.B * p.To * p.tiles_h;
  p.w_chunk_bytes = E * 64;
  svit_tmap_encode_fn enc = svit_get_tmap_encode();
  if (!enc) return SVIT_ENOTSUP;
  CUtensorMap tx, tw;
  {
    cuuint64_t dims[5], strides[4];
    for (int i = 0; i < 5; ++i) dims[i] = in_dims[i];
    for (int i = 0; i < 4; ++i) strides[i] = in_strides[i];
    cuuint32_t box[5] = {32, (cuuint32_t)(p.uniq ? p.PW : p.Wo), (cuuint32_t)(p.uniq ? p.PH : p.R), 1, 1};
    cuuint32_t estr[5] = {1, 1, 1, 1, 1};
    if (enc(&tx, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, const_cast<void*>(in), dims, strides, box, estr,
            CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
      return SVIT_EINVAL;
    const int ktot = p.nt * p.nh * p.nw * p.chunks * 32;
    cuuint64_t wd[2] = {(cuuint64_t)ktot, (cuuint64_t)E};
    cuuint64_t ws[1] = {(cuuint64_t)ktot * 2};
    cuuint32_t wb[2] = {32, (cuuint32_t)E};
    cuuint32_t we[2] = {1, 1};
    if (enc(&tw, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(w2), wd, ws, wb, we, CU_TENSOR_MAP_INTERLEAVE_NONE,
            CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
      return SVIT_EINVAL;
  }
  const int ntaps = p.nt * p.nh * p.nw;
  const size_t smem = (size_t)pe_smem_bytes(ntaps, p.chunks, E, p.uniq ? 2 : PE_STAGES, p.chunk_a);
  if (smem > 227 * 1024) return SVIT_ENOTSUP;
  int64_t grid = svit_num_sms();
  if (grid > p.tiles) grid = p.tiles;
#define PE_LAUNCH(EV)                                                                                              \
  {                                                                                                                \
    auto kern = patch_embed_tc_kernel<EV>;                                                                         \
    static SvitDevOnce once;                                                                                       \
    if (once.need(smem)) {                                                                                         \
      SVIT_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));               \
      once.done(smem);                                                                                             \
    }                                                                                                              \
    kern<<<(unsigned)grid, PE_THREADS, smem, s>>>(tx, tw, p);                                                      \
  }
  switch (E) {
    case 32: PE_LAUNCH(32) break;
    case 64: PE_LAUNCH(64) break;
    case 96: PE_LAUNCH(96) break;
    case 128: PE_LAUNCH(128) break;
    case 192: PE_LAUNCH(192) break;
    case 256: PE_LAUNCH(256) break;
    default: return SVIT_ENOTSUP;
  }
#undef PE_LAUNCH
  SVIT_CHECK_LAUNCH();
  return 0;
}

extern "C" {

int svit_patch_embed_s2d_supported(int C, int kt, int kh, int kw, int st, int sh, int sw, int pt, int ph, int pw, int E) {
  const int cell = C * st * sh * sw;
  if (cell % 32 || cell > 256 || E % 16 || E < 16 || E > PE_MAX_E) return 0;
  int lo, nt, nh, nw;
  pe_taps(kt, st, pt, &lo, &nt);
  pe_taps(kh, sh, ph, &lo, &nh);
  pe_taps(kw, sw, pw, &lo, &nw);
  return pe_smem_bytes(nt * nh * nw, cell / 32, E, PE_STAGES, PE_CHUNK_A) <= 227 * 1024 && pe_n_ok(E);
}

// cells [B, Tc, Hc, Wc, cell] bf16 (svit_s2d_clip); w2 [E, ntaps * cell] bf16 (zero-padded taps, tap-major:
// ((it nh + ih) nw + iw) cell + inner); out rows row_off + (t' Ho + h') Wo + w' of every sample (out_batch_stride elements)
int svit_patch_embed_s2d(const void* cells, const void* w2, const float* bias, void* out, int64_t out_batch_stride,
                         int row_off, int B, int C, int T, int H, int W, int kt, int kh, int kw, int st, int sh, int sw,
                         int pt, int ph, int pw, int E, void* stream) {
  if (!cells || !w2 || !out || B < 0) return SVIT_EINVAL;
  if (!svit_patch_embed_s2d_supported(C, kt, kh, kw, st, sh, sw, pt, ph, pw, E)) return SVIT_ENOTSUP;
  if ((reinterpret_cast<uintptr_t>(cells) | reinterpret_cast<uintptr_t>(w2) | reinterpret_cast<uintptr_t>(out)) & 15)
    return SVIT_ENOTSUP;
  if (B == 0) return 0;
  PeParams p;
  const int cell = C * st * sh * sw;
  p.B = B; p.Tc = (T + st - 1) / st; p.Hc = (H + sh - 1) / sh; p.Wc = (W + sw - 1) / sw;
  p.To = (T + 2 * pt - kt) / st + 1; p.Ho = (H + 2 * ph - kh) / sh + 1; p.Wo = (W + 2 * pw - kw) / sw + 1;
  pe_taps(kt, st, pt, &p.lo_t, &p.nt);
  pe_taps(kh, sh, ph, &p.lo_h, &p.nh);
  pe_taps(kw, sw, pw, &p.lo_w, &p.nw);
  p.chunks = cell / 32;
  p.E = E;
  p.out_bs = out_batch_stride;
  p.row_off = row_off;
  p.bias = bias;
  p.out = (bf16*)out;
  const cuuint64_t dims[5] = {(cuuint64_t)cell, (cuuint64_t)p.Wc, (cuuint64_t)p.Hc, (cuuint64_t)p.Tc, (cuuint64_t)B};
  const cuuint64_t strides[4] = {(cuuint64_t)cell * 2, (cuuint64_t)p.Wc * cell * 2, (cuuint64_t)p.Hc * p.Wc * cell * 2,
                                 (cuuint64_t)p.Tc * p.Hc * p.Wc * cell * 2};
  return pe_launch(p, cells, dims, strides, w2, (cudaStream_t)stream);
}

// Data gradient of the stem: the same kernel with the roles swapped.  Cell c of a dimension is read by the outputs
// c - lo - i (i < n taps), so dcells[c] = sum_i' dY[c + lo' + i'] . W''_i' with lo' = -lo - n + 1 and W''_i' = W'_{n-1-i'}^T:
// a stride-1 convolution over the output grid (K = E values per position) into the cell grid (N = cell values per cell).
int svit_patch_embed_s2d_dgrad_supported(int C, int kt, int kh, int kw, int st, int sh, int sw, int pt, int ph, int pw, int E) {
  const int cell = C * st * sh * sw;
  if (E % 32 || E < 32 || E > PE_MAX_E || !pe_n_ok(cell)) return 0;
  int lo, nt, nh, nw;
  pe_taps(kt, st, pt, &lo, &nt);
  pe_taps(kh, sh, ph, &lo, &nh);
  pe_taps(kw, sw, pw, &lo, &nw);
  return pe_smem_bytes(nt * nh * nw, E / 32, cell, PE_STAGES, PE_CHUNK_A) <= 227 * 1024;
}

// dy: sequence gradient, bf16, sample b's patch row (t' Ho + h') Wo + w' at dy + b dy_batch_stride + (row_off + ...) E,
// read in place; w2t [cell, ntaps * E] bf16 (svit_b200.ops.s2d_dgrad_weight); dcells [B, Tc, Hc, Wc, cell] bf16.
int svit_patch_embed_s2d_dgrad(const void* dy, int64_t dy_batch_stride, int row_off, const void* w2t, void* dcells, int B,
                               int C, int T, int H, int W, int kt, int kh, int kw, int st, int sh, int sw, int pt, int ph,
                               int pw, int E, void* stream) {
  if (!dy || !w2t || !dcells || B < 0 || row_off < 0 || dy_batch_stride < 0) return SVIT_EINVAL;
  if (!svit_patch_embed_s2d_dgrad_supported(C, kt, kh, kw, st, sh, sw, pt, ph, pw, E)) return SVIT_ENOTSUP;
  const bf16* dy0 = (const bf16*)dy + (int64_t)row_off * E;
  if ((reinterpret_cast<uintptr_t>(dy0) | reinterpret_cast<uintptr_t>(w2t) | reinterpret_cast<uintptr_t>(dcells)) & 15 ||
      (dy_batch_stride * 2) % 16)
    return SVIT_ENOTSUP;
  if (B == 0) return 0;
  const int cell = C * st * sh * sw;
  const int To = (T + 2 * pt - kt) / st + 1, Ho = (H + 2 * ph - kh) / sh + 1, Wo = (W + 2 * pw - kw) / sw + 1;
  if (To < 1 || Ho < 1 || Wo < 1) return SVIT_EINVAL;
  if ((int64_t)To * Ho * Wo * E > dy_batch_stride && B > 1) return SVIT_EINVAL;
  PeParams p;
  p.B = B; p.Tc = (T + st - 1) / st; p.Hc = (H + sh - 1) / sh; p.Wc = (W + sw - 1) / sw;
  p.To = p.Tc; p.Ho = p.Hc; p.Wo = p.Wc;  // the output grid is the cell grid
  pe_taps(kt, st, pt, &p.lo_t, &p.nt);
  pe_taps(kh, sh, ph, &p.lo_h, &p.nh);
  pe_taps(kw, sw, pw, &p.lo_w, &p.nw);
  p.lo_t = -p.lo_t - p.nt + 1; p.lo_h = -p.lo_h - p.nh + 1; p.lo_w = -p.lo_w - p.nw + 1;
  p.chunks = E / 32;
  p.E = cell;
  p.out_bs = (int64_t)p.Tc * p.Hc * p.Wc * cell;
  p.row_off = 0;
  p.bias = nullptr;
  p.out = (bf16*)dcells;
  // dY positions outside the output grid are the TMA zero fill
  const cuuint64_t dims[5] = {(cuuint64_t)E, (cuuint64_t)Wo, (cuuint64_t)Ho, (cuuint64_t)To, (cuuint64_t)B};
  const cuuint64_t strides[4] = {(cuuint64_t)E * 2, (cuuint64_t)Wo * E * 2, (cuuint64_t)Ho * Wo * E * 2,
                                 (cuuint64_t)(B > 1 ? dy_batch_stride : (int64_t)To * Ho * Wo * E) * 2};
  return pe_launch(p, dy0, dims, strides, w2t, (cudaStream_t)stream);
}

}  // extern "C"
