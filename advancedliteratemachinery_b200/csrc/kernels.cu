// Non-GEMM kernels of the encoder path: patch im2col, gather + LayerNorm + operand split, Swin window
// attention core, row softmax.  All are HBM-/latency-bound: vectorised 16-byte accesses, one warp per row.
#include "alm_internal.h"
#include "mma.cuh"

namespace alm {

void count_launch(Ctx* c, int n) { c->launches += n; }

void check_launch(const char* what) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) throw AlmError{ALM_ERR_CUDA, std::string("launch of ") + what + ": " + cudaGetErrorString(e)};
}

namespace {

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

__device__ __forceinline__ void store_split4(bf16* hi, bf16* lo, long off, const float4& y) {
  uint32_t h01, l01, h23, l23;   // packed F2FP conversions (the scalar F2F.BF16 is an XU-pipe instruction)
  split_pack2_bf16(y.x, y.y, h01, l01);
  split_pack2_bf16(y.z, y.w, h23, l23);
  *reinterpret_cast<uint2*>(hi + off) = make_uint2(h01, h23);
  if (lo) *reinterpret_cast<uint2*>(lo + off) = make_uint2(l01, l23);
}

// ---------------------------------------------------------------------------------------------
// gather + LayerNorm + split.  One warp per output row; lane holds NV float4 (C = 128*NV, or CW < 128*NV with the
// tail lanes of the last float4 idle: CW = 192 is the ViT-tiny width of MGP-STR, mgp_str.py:207-216).
// ---------------------------------------------------------------------------------------------
template <int NV, int CW = NV * 128>
__global__ void __launch_bounds__(256)
gather_ln_kernel(const float* __restrict__ src, long lds, const int* __restrict__ map, int nsrc, int Cs, long rows,
                 const float* __restrict__ gamma, const float* __restrict__ beta, float eps, int zero_missing,
                 const float* __restrict__ add, long ld_add, float* __restrict__ out_f32, long ldo_f32,
                 bf16* __restrict__ out_hi, bf16* __restrict__ out_lo, long ldo_bf, bf16* __restrict__ out2_hi,
                 bf16* __restrict__ out2_lo, float* __restrict__ out2_f32) {
  const long r = static_cast<long>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (r >= rows) return;
  const int lane = threadIdx.x & 31;
  constexpr int C = CW;
  constexpr bool kFull = (CW == NV * 128);
  float4 v[NV];
  bool any = false;
#pragma unroll
  for (int j = 0; j < NV; ++j) {
    const int e = 4 * (lane + 32 * j);
    v[j] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (!kFull && e >= C) continue;
    const int s = e / Cs;
    const long sr = map ? map[r * nsrc + s] : r * nsrc + s;
    if (sr >= 0) {
      v[j] = *reinterpret_cast<const float4*>(src + sr * lds + (e - s * Cs));
      any = true;
    }
  }
  const bool dead = zero_missing && !__any_sync(0xffffffffu, any);
  if (gamma && !dead) {
    float s = 0.f;
#pragma unroll
    for (int j = 0; j < NV; ++j) s += (v[j].x + v[j].y) + (v[j].z + v[j].w);
    const float mean = warp_sum(s) * (1.0f / C);
    float q = 0.f;
#pragma unroll
    for (int j = 0; j < NV; ++j) {
      if (!kFull && 4 * (lane + 32 * j) >= C) continue;
      const float a = v[j].x - mean, b = v[j].y - mean, c = v[j].z - mean, d = v[j].w - mean;
      q += (a * a + b * b) + (c * c + d * d);
    }
    const float rstd = rsqrtf(warp_sum(q) * (1.0f / C) + eps);
#pragma unroll
    for (int j = 0; j < NV; ++j) {
      const int e = 4 * (lane + 32 * j);
      if (!kFull && e >= C) continue;
      const float4 g = *reinterpret_cast<const float4*>(gamma + e);
      const float4 b = *reinterpret_cast<const float4*>(beta + e);
      v[j].x = (v[j].x - mean) * rstd * g.x + b.x;
      v[j].y = (v[j].y - mean) * rstd * g.y + b.y;
      v[j].z = (v[j].z - mean) * rstd * g.z + b.z;
      v[j].w = (v[j].w - mean) * rstd * g.w + b.w;
    }
  }
#pragma unroll
  for (int j = 0; j < NV; ++j) {
    const int e = 4 * (lane + 32 * j);
    if (!kFull && e >= C) continue;
    if (out_f32) *reinterpret_cast<float4*>(out_f32 + r * ldo_f32 + e) = v[j];
    if (out_hi) store_split4(out_hi, out_lo, r * ldo_bf + e, v[j]);
    if (out2_hi || out2_f32) {
      float4 y = v[j];
      if (add) {
        const float4 a = *reinterpret_cast<const float4*>(add + r * ld_add + e);
        y.x += a.x; y.y += a.y; y.z += a.z; y.w += a.w;
      }
      if (out2_hi) store_split4(out2_hi, out2_lo, r * ldo_bf + e, y);
      if (out2_f32) *reinterpret_cast<float4*>(out2_f32 + r * ldo_f32 + e) = y;
    }
  }
}

// ---------------------------------------------------------------------------------------------
// 4x4 / stride-4 patch im2col of an NCHW fp32 image into a K-major [B*Hp*Wp, 64] split operand
// (k = c*16 + ky*4 + kx, columns 48..63 zero).  One thread per (patch, c, ky) -> one float4 of pixels.
// ---------------------------------------------------------------------------------------------
__global__ void im2col_patch4_kernel(const float* __restrict__ img, int B, int H, int W, int Hp, int Wp,
                                     bf16* __restrict__ hi, bf16* __restrict__ lo) {
  const long idx = static_cast<long>(blockIdx.x) * blockDim.x + threadIdx.x;
  const long total = static_cast<long>(B) * Hp * Wp * 16;
  if (idx >= total) return;
  const int q = static_cast<int>(idx & 15);
  const long patch = idx >> 4;
  float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
  if (q < 12) {
    const int c = q >> 2, ky = q & 3;
    const int pw = static_cast<int>(patch % Wp);
    const int ph = static_cast<int>((patch / Wp) % Hp);
    const int b = static_cast<int>(patch / (static_cast<long>(Wp) * Hp));
    const int y = 4 * ph + ky, x = 4 * pw;
    if (y < H) {
      const float* p = img + ((static_cast<long>(b) * 3 + c) * H + y) * W + x;
      if (x + 3 < W && (reinterpret_cast<uintptr_t>(p) & 15) == 0) {
        v = *reinterpret_cast<const float4*>(p);
      } else {
        if (x < W) v.x = p[0];
        if (x + 1 < W) v.y = p[1];
        if (x + 2 < W) v.z = p[2];
        if (x + 3 < W) v.w = p[3];
      }
    }
  }
  store_split4(hi, lo, patch * 64 + q * 4, v);
}

// ---------------------------------------------------------------------------------------------
// Swin W-MSA core (swin_transformer.py:127-148): one CTA per (window, head), thread i = query token i.
// scores = (q*scale) k^T + rel-pos bias + shift mask(-100) ; softmax ; P V.   fp32 FMA, K/V/bias in smem.
// ---------------------------------------------------------------------------------------------
constexpr int WT = 49;  // tokens per window
constexpr int HD = 32;  // head dim (all Swin-B stages)

__global__ void __launch_bounds__(64)
window_attention_kernel(const float* __restrict__ qkv, int C, int nWh, int nWw, int shift, int Hp, int Wp,
                        const float* __restrict__ bias_dense, bf16* __restrict__ out_hi, bf16* __restrict__ out_lo,
                        float* __restrict__ out_f32) {
  __shared__ __align__(16) float sk[WT][HD];
  __shared__ __align__(16) float sv[WT][HD];
  __shared__ float sbias[WT * WT];
  __shared__ int sreg[WT];
  const int win = blockIdx.x, h = blockIdx.y, t = threadIdx.x;
  const long row0 = static_cast<long>(win) * WT;
  const int ld = 3 * C;
  for (int i = t; i < WT * 8; i += 64) {
    const int r = i >> 3, c4 = (i & 7) * 4;
    const float* base = qkv + (row0 + r) * ld + h * HD + c4;
    *reinterpret_cast<float4*>(&sk[r][c4]) = *reinterpret_cast<const float4*>(base + C);
    *reinterpret_cast<float4*>(&sv[r][c4]) = *reinterpret_cast<const float4*>(base + 2 * C);
  }
  const float* bh = bias_dense + static_cast<long>(h) * WT * WT;
  for (int i = t; i < WT * WT; i += 64) sbias[i] = bh[i];
  if (t < WT) {
    int reg = 0;
    if (shift > 0) {
      const int wi = win % (nWh * nWw);
      const int hh = (wi / nWw) * 7 + t / 7, ww = (wi % nWw) * 7 + t % 7;
      const int rh = hh < Hp - 7 ? 0 : (hh < Hp - shift ? 1 : 2);
      const int rw = ww < Wp - 7 ? 0 : (ww < Wp - shift ? 1 : 2);
      reg = rh * 3 + rw;
    }
    sreg[t] = reg;
  }
  __syncthreads();
  if (t >= WT) return;

  float q[HD];
  {
    const float scale = 0.17677669529663687f;  // 32 ** -0.5
    const float4* qp = reinterpret_cast<const float4*>(qkv + (row0 + t) * ld + h * HD);
#pragma unroll
    for (int d = 0; d < HD / 4; ++d) {
      const float4 x = qp[d];
      q[4 * d] = x.x * scale; q[4 * d + 1] = x.y * scale; q[4 * d + 2] = x.z * scale; q[4 * d + 3] = x.w * scale;
    }
  }
  const int myreg = sreg[t];
  float s[WT];
  float m = -INFINITY;
#pragma unroll
  for (int j = 0; j < WT; ++j) {
    float a = 0.f;
#pragma unroll
    for (int d = 0; d < HD; d += 4) {
      const float4 kk = *reinterpret_cast<const float4*>(&sk[j][d]);
      a = fmaf(q[d], kk.x, a); a = fmaf(q[d + 1], kk.y, a); a = fmaf(q[d + 2], kk.z, a); a = fmaf(q[d + 3], kk.w, a);
    }
    a += sbias[t * WT + j];
    if (shift > 0 && sreg[j] != myreg) a += -100.0f;
    s[j] = a;
    m = fmaxf(m, a);
  }
  float sum = 0.f;
#pragma unroll
  for (int j = 0; j < WT; ++j) {
    s[j] = expf(s[j] - m);
    sum += s[j];
  }
  float o[HD];
#pragma unroll
  for (int d = 0; d < HD; ++d) o[d] = 0.f;
#pragma unroll
  for (int j = 0; j < WT; ++j) {
    const float pj = s[j] / sum;
#pragma unroll
    for (int d = 0; d < HD; d += 4) {
      const float4 vv = *reinterpret_cast<const float4*>(&sv[j][d]);
      o[d] = fmaf(pj, vv.x, o[d]); o[d + 1] = fmaf(pj, vv.y, o[d + 1]);
      o[d + 2] = fmaf(pj, vv.z, o[d + 2]); o[d + 3] = fmaf(pj, vv.w, o[d + 3]);
    }
  }
  const long ooff = (row0 + t) * C + h * HD;
#pragma unroll
  for (int d = 0; d < HD; d += 4) {
    const float4 y = make_float4(o[d], o[d + 1], o[d + 2], o[d + 3]);
    if (out_hi) store_split4(out_hi, out_lo, ooff + d, y);
    if (out_f32) *reinterpret_cast<float4*>(out_f32 + ooff + d) = y;
  }
}

// ---------------------------------------------------------------------------------------------
// Swin W-MSA core on the tensor cores: one CTA (4 warps) per (window, head); warp w owns query rows 16w..16w+15.
// Input is the qkv projection as split-bf16 planes straight from the GEMM epilogue (q already carries the
// 32^-0.5 scale: it is folded into the q rows of the qkv weight at load time), so staging is pure cp.async --
// no conversion, no transposition (P.V reads v [key][dim] through ldmatrix.trans).  Both products
// (S = q k^T, 64x64x32 ; O = P v, 64x32x64, padded from 49) run as mma.sync.m16n8k16 with the three-term split
// hi*hi + lo*hi + hi*lo accumulated in fp32 registers -- the same fp32-class scheme as the GEMM engine.
// Softmax stays in fp32 registers (quad shuffles).  These 49x49x32 tiles are too small for a tcgen05
// 128-row instruction (7 % of Swin FLOPs, SURVEY 8d), so the warp-level MMA is the right granularity.
// ---------------------------------------------------------------------------------------------
constexpr int WS_PITCH = 40;   // bf16 per staged row (32 + 8 pad -> conflict-free ldmatrix)
constexpr int WS_TILE = 64 * WS_PITCH;

__global__ void __launch_bounds__(128)
window_attention_split_kernel(const bf16* __restrict__ qkv_hi, const bf16* __restrict__ qkv_lo, int C, int nWh, int nWw,
                              int shift, int Hp, int Wp, const float* __restrict__ bias_dense, bf16* __restrict__ out_hi,
                              bf16* __restrict__ out_lo, float* __restrict__ out_f32) {
  __shared__ __align__(16) bf16 st[2][3][WS_TILE];  // [hi/lo][q,k,v][row][dim]
  __shared__ int sreg[64];
  const int win = blockIdx.x, h = blockIdx.y, tid = threadIdx.x;
  const int warp = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
  const long row0 = static_cast<long>(win) * WT;
  const long ld = 3L * C;
  // ---- stage q, k, v (rows >= 49 zero-filled): 64 rows x 4 x 16-byte chunks per tile and plane
#pragma unroll
  for (int i = tid; i < 3 * 256; i += 128) {
    const int which = i >> 8, rem = i & 255, r = rem >> 2, ch = (rem & 3) * 8;
    const bool ok = r < WT;
    const long src = (row0 + (ok ? r : 0)) * ld + which * C + h * HD + ch;
    cp_async16(&st[0][which][r * WS_PITCH + ch], qkv_hi + src, ok ? 16 : 0);
    cp_async16(&st[1][which][r * WS_PITCH + ch], qkv_lo + src, ok ? 16 : 0);
  }
  cp_async_commit();
  if (tid < 64) {
    int reg = 0;
    if (shift > 0 && tid < WT) {
      const int wi = win % (nWh * nWw);
      const int hh = (wi / nWw) * 7 + tid / 7, ww = (wi % nWw) * 7 + tid % 7;
      const int rh = hh < Hp - 7 ? 0 : (hh < Hp - shift ? 1 : 2);
      const int rw = ww < Wp - 7 ? 0 : (ww < Wp - shift ? 1 : 2);
      reg = rh * 3 + rw;
    }
    sreg[tid] = reg;
  }
  cp_async_wait<0>();
  __syncthreads();

  const int r_lo = warp * 16 + g, r_hi = r_lo + 8;  // the two query rows this lane holds
  const int lrow = lane & 7, lmat = lane >> 3;
  // ---- S = q k^T : A fragments of q (hi, lo) for both k-steps
  uint32_t aq[2][2][4];
#pragma unroll
  for (int p = 0; p < 2; ++p)
#pragma unroll
    for (int ks = 0; ks < 2; ++ks)
      ldmatrix_x4(aq[p][ks], &st[p][0][(warp * 16 + (lane & 15)) * WS_PITCH + ks * 16 + (lane >> 4) * 8]);
  float s[8][4];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    s[j][0] = s[j][1] = s[j][2] = s[j][3] = 0.f;
    uint32_t bh[4], bl[4];  // (ks0 b0, ks0 b1, ks1 b0, ks1 b1)
    ldmatrix_x4(bh, &st[0][1][(8 * j + lrow) * WS_PITCH + lmat * 8]);
    ldmatrix_x4(bl, &st[1][1][(8 * j + lrow) * WS_PITCH + lmat * 8]);
#pragma unroll
    for (int ks = 0; ks < 2; ++ks) {
      mma_bf16_16816(s[j], aq[0][ks], bh[2 * ks], bh[2 * ks + 1]);
      mma_bf16_16816(s[j], aq[1][ks], bh[2 * ks], bh[2 * ks + 1]);
      mma_bf16_16816(s[j], aq[0][ks], bl[2 * ks], bl[2 * ks + 1]);
    }
  }
  // ---- + relative-position bias + shift mask; exclude MMA padding columns; softmax per row (fp32)
  const float* bh_ = bias_dense + static_cast<long>(h) * WT * WT;
  const int reg_lo = sreg[min(r_lo, 63)], reg_hi = sreg[min(r_hi, 63)];
  float m_lo = -INFINITY, m_hi = -INFINITY;
#pragma unroll
  for (int j = 0; j < 8; ++j) {
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      const int col = 8 * j + 2 * t + e;
      if (col < WT) {
        const int rc = sreg[col];
        if (r_lo < WT) s[j][e] += __ldg(bh_ + r_lo * WT + col) + ((shift > 0 && rc != reg_lo) ? -100.0f : 0.0f);
        if (r_hi < WT) s[j][2 + e] += __ldg(bh_ + r_hi * WT + col) + ((shift > 0 && rc != reg_hi) ? -100.0f : 0.0f);
      } else {
        s[j][e] = -INFINITY;
        s[j][2 + e] = -INFINITY;
      }
      m_lo = fmaxf(m_lo, s[j][e]);
      m_hi = fmaxf(m_hi, s[j][2 + e]);
    }
  }
  m_lo = fmaxf(m_lo, __shfl_xor_sync(0xffffffffu, m_lo, 1)); m_lo = fmaxf(m_lo, __shfl_xor_sync(0xffffffffu, m_lo, 2));
  m_hi = fmaxf(m_hi, __shfl_xor_sync(0xffffffffu, m_hi, 1)); m_hi = fmaxf(m_hi, __shfl_xor_sync(0xffffffffu, m_hi, 2));
  float sum_lo = 0.f, sum_hi = 0.f;
#pragma unroll
  for (int j = 0; j < 8; ++j)
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      s[j][e] = expf(s[j][e] - m_lo);
      s[j][2 + e] = expf(s[j][2 + e] - m_hi);
      sum_lo += s[j][e];
      sum_hi += s[j][2 + e];
    }
  sum_lo += __shfl_xor_sync(0xffffffffu, sum_lo, 1); sum_lo += __shfl_xor_sync(0xffffffffu, sum_lo, 2);
  sum_hi += __shfl_xor_sync(0xffffffffu, sum_hi, 1); sum_hi += __shfl_xor_sync(0xffffffffu, sum_hi, 2);
  // ---- O = P v : P (normalised, split) becomes the A operand straight from the accumulator fragments;
  //      v [key][dim] is read through ldmatrix.trans: matrix i = (key half i&1, dim tile 2*np + (i>>1))
  float o[4][4];
#pragma unroll
  for (int n = 0; n < 4; ++n) o[n][0] = o[n][1] = o[n][2] = o[n][3] = 0.f;
#pragma unroll
  for (int kk = 0; kk < 4; ++kk) {
    uint32_t ph[4], pl[4];
    split_pack2(s[2 * kk][0] / sum_lo, s[2 * kk][1] / sum_lo, ph[0], pl[0]);
    split_pack2(s[2 * kk][2] / sum_hi, s[2 * kk][3] / sum_hi, ph[1], pl[1]);
    split_pack2(s[2 * kk + 1][0] / sum_lo, s[2 * kk + 1][1] / sum_lo, ph[2], pl[2]);
    split_pack2(s[2 * kk + 1][2] / sum_hi, s[2 * kk + 1][3] / sum_hi, ph[3], pl[3]);
#pragma unroll
    for (int np = 0; np < 2; ++np) {
      uint32_t vh[4], vl[4];  // (b0, b1) of dim tile 2np, (b0, b1) of dim tile 2np+1
      const int off = (16 * kk + (lmat & 1) * 8 + lrow) * WS_PITCH + (2 * np + (lmat >> 1)) * 8;
      ldmatrix_x4_trans(vh, &st[0][2][off]);
      ldmatrix_x4_trans(vl, &st[1][2][off]);
#pragma unroll
      for (int q = 0; q < 2; ++q) {
        mma_bf16_16816(o[2 * np + q], ph, vh[2 * q], vh[2 * q + 1]);
        mma_bf16_16816(o[2 * np + q], pl, vh[2 * q], vh[2 * q + 1]);
        mma_bf16_16816(o[2 * np + q], ph, vl[2 * q], vl[2 * q + 1]);
      }
    }
  }
  // ---- store: stage the 64x32 tile in smem (reusing the q tiles), then 16-byte row segments
  __syncthreads();
  float* so = reinterpret_cast<float*>(&st[0][0][0]);  // 64 x 36 floats = 9216 B <= 2 tiles (10240 B)
#pragma unroll
  for (int n = 0; n < 4; ++n) {
    *reinterpret_cast<float2*>(so + r_lo * 36 + 8 * n + 2 * t) = make_float2(o[n][0], o[n][1]);
    *reinterpret_cast<float2*>(so + r_hi * 36 + 8 * n + 2 * t) = make_float2(o[n][2], o[n][3]);
  }
  __syncthreads();
  for (int i = tid; i < WT * 8; i += 128) {
    const int r = i >> 3, c4 = (i & 7) * 4;
    const float4 y = *reinterpret_cast<const float4*>(so + r * 36 + c4);
    const long ooff = (row0 + r) * C + h * HD + c4;
    if (out_hi) store_split4(out_hi, out_lo, ooff, y);
    if (out_f32) *reinterpret_cast<float4*>(out_f32 + ooff) = y;
  }
}

// fp32 qkv -> split planes with the q columns scaled (only the op-level C entry point needs this: inside the
// encoder the qkv GEMM epilogue writes the planes directly)
__global__ void qkv_split_scale_kernel(const float* __restrict__ src, long rows, int C, float scale, bf16* __restrict__ hi,
                                       bf16* __restrict__ lo) {
  const long i = static_cast<long>(blockIdx.x) * blockDim.x + threadIdx.x;
  const int c4 = (3 * C) >> 2;
  if (i >= rows * c4) return;
  const long r = i / c4;
  const int e = static_cast<int>(i % c4) * 4;
  float4 v = *reinterpret_cast<const float4*>(src + r * 3 * C + e);
  if (e < C) { v.x *= scale; v.y *= scale; v.z *= scale; v.w *= scale; }
  store_split4(hi, lo, r * 3 * C + e, v);
}

// ---------------------------------------------------------------------------------------------
// fp32 -> split bf16 rows (C multiple of 4)
// ---------------------------------------------------------------------------------------------
__global__ void split_rows_kernel(const float* __restrict__ src, long lds, long rows, int C, bf16* __restrict__ hi,
                                  bf16* __restrict__ lo, long ldo) {
  const long i = static_cast<long>(blockIdx.x) * blockDim.x + threadIdx.x;
  const int c4 = C >> 2;
  if (i >= rows * c4) return;
  const long r = i / c4;
  const int e = static_cast<int>(i % c4) * 4;
  store_split4(hi, lo, r * ldo + e, *reinterpret_cast<const float4*>(src + r * lds + e));
}

// ---------------------------------------------------------------------------------------------
// row softmax over n columns with optional key-padding mask (1 = -inf).  One CTA (128 threads) per row,
// three passes over an L1/L2-resident row.  Output fp32 and/or split bf16 (columns n..ldo-1 untouched).
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128)
softmax_rows_kernel(const float* __restrict__ s, long lds, int n, const uint8_t* __restrict__ kpm, int rows_per_mask,
                    long mask_ld, float* __restrict__ out_f32, bf16* __restrict__ out_hi, bf16* __restrict__ out_lo,
                    long ldo) {
  __shared__ float red[4];
  const long r = blockIdx.x;
  const float* x = s + r * lds;
  const uint8_t* mk = kpm ? kpm + (r / rows_per_mask) * mask_ld : nullptr;
  const int t = threadIdx.x;
  float m = -INFINITY;
  for (int j = t; j < n; j += 128) {
    const float v = (mk && mk[j]) ? -INFINITY : x[j];
    m = fmaxf(m, v);
  }
  m = warp_max(m);
  if ((t & 31) == 0) red[t >> 5] = m;
  __syncthreads();
  m = fmaxf(fmaxf(red[0], red[1]), fmaxf(red[2], red[3]));
  __syncthreads();
  float sum = 0.f;
  for (int j = t; j < n; j += 128) {
    const float v = (mk && mk[j]) ? -INFINITY : x[j];
    sum += expf(v - m);
  }
  sum = warp_sum(sum);
  if ((t & 31) == 0) red[t >> 5] = sum;
  __syncthreads();
  sum = (red[0] + red[1]) + (red[2] + red[3]);
  for (int j = t; j < n; j += 128) {
    const float v = (mk && mk[j]) ? -INFINITY : x[j];
    const float p = expf(v - m) / sum;
    if (out_f32) out_f32[r * ldo + j] = p;
    if (out_hi) {
      bf16 h, l;
      split_bf16(p, h, l);
      out_hi[r * ldo + j] = h;
      if (out_lo) out_lo[r * ldo + j] = l;
    }
  }
}


// ---------------------------------------------------------------------------------------------
// Skinny fp32 linear for the point-loop decode (M <= 64 rows): out[m, n] = act(x[m,:].W[n,:] + b[n])
// (+ resid[m, n]).  One warp per output column streams its fp32 weight row once (coalesced float4) while the few
// activation rows come from L1; a tensor-core tile would be > 90 % padding here and the op is latency-bound anyway.
// Weights stay exact fp32, so this path is closer to the reference than the split-bf16 GEMM.
// ---------------------------------------------------------------------------------------------
// Optional fused pre-LayerNorm (ln_g != nullptr, K == 512 == the row width): the staged rows are the raw residual stream;
// every CTA normalises its private copy in shared memory (16 x 512 values: far cheaper than one more dependent launch in
// the latency-bound point loop) with exactly the arithmetic and summation order of gather_ln_kernel<4>, then adds the
// query position embedding `pos` for the output columns below pos_split (q | k of the packed self-attention projection;
// everything for the cross-attention query).
//
// The 64-row variant (up to 64 live sequences: several window prompts per page in the point loop) keeps every row's
// arithmetic of the 32-row one -- each lane still accumulates one row in the same lane-strided float4 order over K and the
// row is reduced by the same warp_sum -- so a row's result does not depend on how many rows share the launch.  Lane l
// writes rows l and l + 32.  Its K > 512 launches stage 256-float chunks (64 x 2 x 256 fp32 = 128 KB double-buffered,
// where 512-float chunks would need 256 KB): chunk c of 512 floats is chunks 2c, 2c + 1 of 256, so the per-lane order of
// the fused multiply-adds is unchanged.
template <int MR, int NW>  // MR = row capacity (8/16/32/64), NW = K / 128 float4 slices of the weight row per lane
__device__ __forceinline__ void
gemv_rows_body(const float* __restrict__ x, const float* __restrict__ x2, int n_split, long ldx,
                 const float* __restrict__ W, const float* __restrict__ bias, const float* __restrict__ resid, long ldr,
                 float* __restrict__ out, long ldo, int M, int N, int K, int act, const float* __restrict__ ln_g,
                 const float* __restrict__ ln_b, float ln_eps, const float* __restrict__ pos, int pos_split) {
  // activation rows, staged in K-chunks of <= 512 floats (double-buffered when K > 512): at most 64 KB for 16 rows,
  // so this kernel co-resides with the HBM-bound attention CTAs of the other in-flight decode streams
  extern __shared__ __align__(16) float sx[];
  constexpr int CW = (MR > 32 && NW > 4) ? 256 : 512;  // chunk width when K > 512 (floats)
  constexpr int SPC = CW / 128;             // float4 slices per lane of a full chunk
  constexpr int NC = (NW + SPC - 1) / SPC;  // chunks
  constexpr int NWC = NW < SPC ? NW : SPC;  // float4 slices per lane and chunk
  const int KC = NC == 1 ? K : CW;          // chunk width (floats)
  const int n = blockIdx.x * 4 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  const float* xin = (blockIdx.x * 4 < n_split) ? x : x2;  // columns [0, n_split) read x, the rest x2 (fused q|k|v)
  const uint32_t sbase = static_cast<uint32_t>(__cvta_generic_to_shared(sx));
  auto stage = [&](int chunk, int buf) {
    // NC is sized for K = 2048: when K = 1024 or 1536 the trailing chunks lie past column K (KC divides K, so a chunk
    // is either full or empty) -- they stage nothing, only commit their (empty) group so that the wait counts hold
    if (NC > 1 && chunk * KC >= K) {
      asm volatile("cp.async.commit_group;" ::: "memory");
      return;
    }
    const int k4 = KC >> 2;
    for (int i = threadIdx.x; i < M * k4; i += 128) {
      const int m = i / k4, c4 = i - m * k4;
      asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(sbase + static_cast<uint32_t>(((buf * M + m) * KC + c4 * 4) * 4)),
                   "l"(xin + m * ldx + chunk * KC + c4 * 4)
                   : "memory");
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
  };
  stage(0, 0);  // every 16-byte copy of the chunk is in flight at once: one memory round trip however many rows
  // the whole weight row of this column is requested up front (NW independent 16-byte loads per lane = one
  // round trip), overlapping the activation staging.  The 64-row kernel, whose 64 accumulators already take the
  // registers, requests each chunk's slices at the top of that chunk instead (same values, same order of use).
  constexpr bool PRELOAD = MR <= 32;
  float4 w[NW];
  if (!PRELOAD) {
  } else if (n < N) {
    const float* wrow = W + static_cast<long>(n) * K;
#pragma unroll
    for (int i = 0; i < NW; ++i) {
      const int k0 = (i * 32 + lane) * 4;
      w[i] = k0 < K ? *reinterpret_cast<const float4*>(wrow + k0) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
  } else {
#pragma unroll
    for (int i = 0; i < NW; ++i) w[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  float acc[MR];
#pragma unroll
  for (int m = 0; m < MR; ++m) acc[m] = 0.f;
#pragma unroll
  for (int c = 0; c < NC; ++c) {
    if (!PRELOAD) {
#pragma unroll
      for (int i = 0; i < NWC; ++i) {
        const int k0 = ((c * SPC + i) * 32 + lane) * 4;
        w[c * SPC + i] = (n < N && k0 < K) ? *reinterpret_cast<const float4*>(W + static_cast<long>(n) * K + k0)
                                           : make_float4(0.f, 0.f, 0.f, 0.f);
      }
    }
    if (c + 1 < NC) {
      stage(c + 1, (c + 1) & 1);
      asm volatile("cp.async.wait_group 1;" ::: "memory");
    } else {
      asm volatile("cp.async.wait_group 0;" ::: "memory");
    }
    __syncthreads();
    if (NC == 1 && ln_g != nullptr) {  // fused LayerNorm (+ pos) on the staged rows: warp w normalises rows w, w+4, ...
      const bool add_pos = pos != nullptr && blockIdx.x * 4 < pos_split;
      for (int m = threadIdx.x >> 5; m < M; m += 4) {
        float* row = sx + m * KC;
        float4 v[4];
        float s = 0.f;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          v[j] = *reinterpret_cast<const float4*>(row + 4 * (lane + 32 * j));
          s += (v[j].x + v[j].y) + (v[j].z + v[j].w);
        }
        const float mean = warp_sum(s) * (1.0f / 512);
        float q = 0.f;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float a = v[j].x - mean, b2 = v[j].y - mean, c2 = v[j].z - mean, d = v[j].w - mean;
          q += (a * a + b2 * b2) + (c2 * c2 + d * d);
        }
        const float rstd = rsqrtf(warp_sum(q) * (1.0f / 512) + ln_eps);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int e = 4 * (lane + 32 * j);
          const float4 g = *reinterpret_cast<const float4*>(ln_g + e);
          const float4 bb = *reinterpret_cast<const float4*>(ln_b + e);
          float4 y;
          y.x = (v[j].x - mean) * rstd * g.x + bb.x;
          y.y = (v[j].y - mean) * rstd * g.y + bb.y;
          y.z = (v[j].z - mean) * rstd * g.z + bb.z;
          y.w = (v[j].w - mean) * rstd * g.w + bb.w;
          if (add_pos) {
            const float4 pp = *reinterpret_cast<const float4*>(pos + e);
            y.x += pp.x; y.y += pp.y; y.z += pp.z; y.w += pp.w;
          }
          *reinterpret_cast<float4*>(row + e) = y;
        }
      }
      __syncthreads();
    }
    const float* xs = sx + static_cast<long>(c & 1) * M * KC;
#pragma unroll
    for (int m = 0; m < MR; ++m) {
      if (m < M) {
#pragma unroll
        for (int i = 0; i < NWC; ++i) {
          const int kk = (i * 32 + lane) * 4;
          if (c * KC + kk < K) {
            const float4 a = *reinterpret_cast<const float4*>(xs + m * KC + kk);
            const float4 ww = w[c * SPC + i];
            acc[m] = fmaf(a.x, ww.x, acc[m]); acc[m] = fmaf(a.y, ww.y, acc[m]);
            acc[m] = fmaf(a.z, ww.z, acc[m]); acc[m] = fmaf(a.w, ww.w, acc[m]);
          }
        }
      }
    }
    if (c + 2 < NC) __syncthreads();  // the buffer is refilled two chunks later
  }
  if (n >= N) return;
  constexpr int RPL = (MR + 31) / 32;  // rows written per lane
  float mine[RPL];
#pragma unroll
  for (int j = 0; j < RPL; ++j) mine[j] = 0.f;
#pragma unroll
  for (int m = 0; m < MR; ++m) {
    const float v = warp_sum(acc[m]);
    if (lane == (m & 31)) mine[m >> 5] = v;
  }
#pragma unroll
  for (int j = 0; j < RPL; ++j) {
    const int row = j * 32 + lane;
    if (row < M && row < MR) {
      float v = mine[j] + (bias ? bias[n] : 0.f);
      if (act == ACT_GELU) v = 0.5f * v * (1.0f + erff(v * 0.70710678118654752440f));
      else if (act == ACT_RELU) v = fmaxf(v, 0.f);
      if (resid) v += resid[row * ldr + n];
      out[row * ldo + n] = v;
    }
  }
}

#define ALM_GEMV_PARAMS                                                                                              \
  const float *__restrict__ x, const float *__restrict__ x2, int n_split, long ldx, const float *__restrict__ W,    \
      const float *__restrict__ bias, const float *__restrict__ resid, long ldr, float *__restrict__ out, long ldo,   \
      int M, int N, int K, int act, const float *__restrict__ ln_g, const float *__restrict__ ln_b, float ln_eps,     \
      const float *__restrict__ pos, int pos_split
#define ALM_GEMV_ARGS x, x2, n_split, ldx, W, bias, resid, ldr, out, ldo, M, N, K, act, ln_g, ln_b, ln_eps, pos, pos_split
template <int MR, int NW>  // up to 32 rows
__global__ void __launch_bounds__(128) gemv_rows_kernel(ALM_GEMV_PARAMS) {
  gemv_rows_body<MR, NW>(ALM_GEMV_ARGS);
}
template <int NW>  // 64 rows: one CTA per SM by its shared memory anyway, so the 64 accumulators may take the registers
__global__ void __launch_bounds__(128, 1) gemv_rows64_kernel(ALM_GEMV_PARAMS) {
  gemv_rows_body<64, NW>(ALM_GEMV_ARGS);
}
#undef ALM_GEMV_PARAMS
#undef ALM_GEMV_ARGS

}  // namespace

void gather_ln(Ctx* c, const float* src, long lds, const int* map, int nsrc, int Cs, long rows, const float* gamma,
               const float* beta, float eps, bool zero_missing, const float* add, long ld_add, float* out_f32,
               long ldo_f32, bf16* out_hi, bf16* out_lo, long ldo_bf, bf16* out2_hi, bf16* out2_lo, float* out2_f32) {
  if (c->skipped(4)) return;
  if (rows == 0) return;
  if (c->lo_unused) { out_lo = nullptr; out2_lo = nullptr; }  // single-pass bf16 ViT path: the lo planes are never read
  const int C = nsrc * Cs;
  ALM_REQUIRE((C % 128 == 0 || C == 192) && Cs % 4 == 0 && lds % 4 == 0, ALM_ERR_INVALID,
              "gather_ln: width must be a multiple of 128 (or 192)");
  const int nv = C == 192 ? 192 : C / 128;
  const int wpb = 8;
  dim3 grid(static_cast<unsigned>((rows + wpb - 1) / wpb)), block(wpb * 32);
#define ALM_GLN(NVV)                                                                                              \
  case NVV:                                                                                                       \
    ALM_PIN_CARVEOUT(gather_ln_kernel<NVV>);                                                                      \
    gather_ln_kernel<NVV><<<grid, block, 0, c->stream>>>(src, lds, map, nsrc, Cs, rows, gamma, beta, eps,         \
                                                         zero_missing ? 1 : 0, add, ld_add, out_f32, ldo_f32,     \
                                                         out_hi, out_lo, ldo_bf, out2_hi, out2_lo, out2_f32);     \
    break;
  switch (nv) {
    ALM_GLN(1) ALM_GLN(2) ALM_GLN(3) ALM_GLN(4) ALM_GLN(6) ALM_GLN(8) ALM_GLN(16)
    case 192: {
      auto k192 = gather_ln_kernel<2, 192>;
      ALM_PIN_CARVEOUT(k192);
      k192<<<grid, block, 0, c->stream>>>(src, lds, map, nsrc, Cs, rows, gamma, beta, eps, zero_missing ? 1 : 0, add,
                                          ld_add, out_f32, ldo_f32, out_hi, out_lo, ldo_bf, out2_hi, out2_lo, out2_f32);
      break;
    }
    default:
      throw AlmError{ALM_ERR_UNSUPPORTED, "gather_ln: unsupported width " + std::to_string(C)};
  }
#undef ALM_GLN
  count_launch(c);
  check_launch("gather_ln");
}

void im2col_patch4(Ctx* c, const float* img, int B, int H, int W, int Hp, int Wp, bf16* hi, bf16* lo) {
  const long total = static_cast<long>(B) * Hp * Wp * 16;
  im2col_patch4_kernel<<<static_cast<unsigned>((total + 255) / 256), 256, 0, c->stream>>>(img, B, H, W, Hp, Wp, hi, lo);
  count_launch(c);
  check_launch("im2col_patch4");
}

void window_attention_split(Ctx* c, const bf16* qkv_hi, const bf16* qkv_lo, int C, int heads, int nWh, int nWw, int B,
                            int shift, int Hp, int Wp, const float* bias_dense, bf16* out_hi, bf16* out_lo, float* out_f32) {
  ALM_REQUIRE(C == heads * HD, ALM_ERR_UNSUPPORTED, "window_attention: head_dim must be 32");
  if (c->wattn_impl == 2) {  // tcgen05 + TMA kernel (wattn_tc.cu)
    window_attention_tc(c, qkv_hi, qkv_lo, C, heads, nWh, nWw, B, shift, Hp, Wp, bias_dense, out_hi, out_lo, out_f32);
    return;
  }
  if (c->wattn_impl == 3 && heads % 2 == 0) {  // persistent TMA-fed mma.sync kernel over head pairs (wattn_ms.cu)
    window_attention_ms(c, qkv_hi, qkv_lo, C, heads, nWh, nWw, B, shift, Hp, Wp, bias_dense, out_hi, out_lo, out_f32);
    return;
  }
  dim3 grid(static_cast<unsigned>(B * nWh * nWw), heads);
  window_attention_split_kernel<<<grid, 128, 0, c->stream>>>(qkv_hi, qkv_lo, C, nWh, nWw, shift, Hp, Wp, bias_dense, out_hi,
                                                             out_lo, out_f32);
  count_launch(c);
  check_launch("window_attention_split");
}

// fp32 qkv (unscaled q) entry point of the op-level C API: wattn_impl 1 = fp32 SIMT kernel, 0 = the encoder's
// tensor-core kernel behind a split + scale pass
void window_attention(Ctx* c, const float* qkv, int C, int heads, int nWh, int nWw, int B, int shift, int Hp, int Wp,
                      const float* bias_dense, bf16* out_hi, bf16* out_lo, float* out_f32) {
  ALM_REQUIRE(C == heads * HD, ALM_ERR_UNSUPPORTED, "window_attention: head_dim must be 32");
  if (c->wattn_impl == 1) {
    dim3 grid(static_cast<unsigned>(B * nWh * nWw), heads);
    window_attention_kernel<<<grid, 64, 0, c->stream>>>(qkv, C, nWh, nWw, shift, Hp, Wp, bias_dense, out_hi, out_lo,
                                                        out_f32);
    count_launch(c);
    check_launch("window_attention");
    return;
  }
  const long rows = static_cast<long>(B) * nWh * nWw * WT;
  const size_t mk = c->ws.mark();
  bf16* hi = c->ws.get<bf16>(rows * 3 * C);
  bf16* lo = c->ws.get<bf16>(rows * 3 * C);
  const long total = rows * (3 * C / 4);
  qkv_split_scale_kernel<<<static_cast<unsigned>((total + 255) / 256), 256, 0, c->stream>>>(qkv, rows, C, WATTN_QSCALE, hi, lo);
  count_launch(c);
  check_launch("qkv_split_scale");
  window_attention_split(c, hi, lo, C, heads, nWh, nWw, B, shift, Hp, Wp, bias_dense, out_hi, out_lo, out_f32);
  c->ws.release(mk);  // stream-ordered: later allocations are only touched by later launches
}

void split_rows(Ctx* c, const float* src, long lds, long rows, int C, bf16* hi, bf16* lo, long ldo) {
  ALM_REQUIRE(C % 4 == 0 && lds % 4 == 0 && ldo % 4 == 0, ALM_ERR_INVALID, "split_rows: width must be a multiple of 4");
  const long total = rows * (C / 4);
  if (total == 0) return;
  split_rows_kernel<<<static_cast<unsigned>((total + 255) / 256), 256, 0, c->stream>>>(src, lds, rows, C, hi, lo, ldo);
  count_launch(c);
  check_launch("split_rows");
}

void softmax_rows(Ctx* c, const float* s, long lds, long rows, int n, const uint8_t* kpm, int rows_per_mask,
                  long mask_ld, float* out_f32, bf16* out_hi, bf16* out_lo, long ldo) {
  if (rows == 0) return;
  ALM_PIN_CARVEOUT(softmax_rows_kernel);
  softmax_rows_kernel<<<static_cast<unsigned>(rows), 128, 0, c->stream>>>(s, lds, n, kpm, rows_per_mask, mask_ld,
                                                                          out_f32, out_hi, out_lo, ldo);
  count_launch(c);
  check_launch("softmax_rows");
}

}  // namespace alm

namespace alm {
void gemv_rows(Ctx* c, const float* x, const float* x2, int n_split, long ldx, const float* W, const float* bias,
               const float* resid, long ldr, float* out, long ldo, int M, int N, int K, int act, const float* ln_g,
               const float* ln_b, float ln_eps, const float* pos, int pos_split) {
  if (c->skipped(2)) return;
  ALM_REQUIRE(ln_g == nullptr || (K == 512 && ln_b != nullptr), ALM_ERR_INVALID, "gemv_rows: fused LayerNorm needs K == 512");
  ALM_REQUIRE(M >= 1 && M <= 64 && K % 4 == 0 && ldx % 4 == 0 && K <= 2048 && n_split % 4 == 0 &&
                  (K <= 512 || K % 512 == 0),
              ALM_ERR_INVALID, "gemv_rows: M <= 64, K % 4 == 0, K <= 512 or a multiple of 512 up to 2048");
  const unsigned grid = static_cast<unsigned>((N + 3) / 4);
  // staged rows: one K-wide buffer, or two chunk buffers (512 floats; 256 for the 64-row kernel) when K > 512
  const size_t dyn = static_cast<size_t>(M) * (K <= 512 ? K : 2 * (M > 32 ? 256 : 512)) * sizeof(float);
#define ALM_GEMV_K(KERNEL)                                                                                         \
  do {                                                                                                             \
    static alm::DeviceOnce attr;                                                                                   \
    if (attr.need()) {                                                                                              \
      ALM_CHECK_CUDA(cudaFuncSetAttribute(KERNEL, cudaFuncAttributeMaxDynamicSharedMemorySize, 128 * 1024));       \
      alm::pin_carveout(KERNEL);                                                                                   \
      attr.mark();                                                                                                 \
    }                                                                                                              \
    KERNEL<<<grid, 128, dyn, c->stream>>>(x, x2 ? x2 : x, n_split, ldx, W, bias, resid, ldr, out, ldo, M, N, K, act, \
                                          ln_g, ln_b, ln_eps, pos, pos_split);                                     \
  } while (0)
#define ALM_GEMV(MRV, NWV) ALM_GEMV_K((gemv_rows_kernel<MRV, NWV>))
  const int nw = K <= 512 ? 4 : 16;
  if (M <= 8) { if (nw == 4) ALM_GEMV(8, 4); else ALM_GEMV(8, 16); }
  else if (M <= 16) { if (nw == 4) ALM_GEMV(16, 4); else ALM_GEMV(16, 16); }
  else if (M <= 32) { if (nw == 4) ALM_GEMV(32, 4); else ALM_GEMV(32, 16); }
  else { if (nw == 4) ALM_GEMV_K(gemv_rows64_kernel<4>); else ALM_GEMV_K(gemv_rows64_kernel<16>); }
#undef ALM_GEMV_K
#undef ALM_GEMV
  count_launch(c);
  check_launch("gemv_rows");
}
}  // namespace alm
