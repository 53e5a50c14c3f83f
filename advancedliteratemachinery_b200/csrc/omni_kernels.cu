// OmniParser-specific small kernels: window / merge / upsample index maps, FPN consumer-side assembly,
// sine position embedding, and the per-token decoder kernels (embedding, cached self-attention, vocabulary
// head selection).  All latency-/HBM-bound integer+fp32 work.
#include <algorithm>

#include "alm_internal.h"
#include "omni.h"
#include "ptx.cuh"

namespace alm {
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

// row r of the windowed tensor (b, wr, wc, ti, tj) -> pixel row of x[B, H*W] or -1 for a pad token.
// pad to x7 then roll(-shift) then 7x7 partition  (swin_transformer.py:213-229); the inverse mapping is the
// same table (window_reverse + roll(+shift) + crop, :235-245).
__global__ void window_map_kernel(int* map, int B, int H, int W, int nWh, int nWw, int shift) {
  const long r = static_cast<long>(blockIdx.x) * blockDim.x + threadIdx.x;
  const long total = static_cast<long>(B) * nWh * nWw * 49;
  if (r >= total) return;
  const int t = static_cast<int>(r % 49);
  const long w = r / 49;
  const int wc = static_cast<int>(w % nWw), wr = static_cast<int>((w / nWw) % nWh);
  const int b = static_cast<int>(w / (static_cast<long>(nWw) * nWh));
  const int Hp = nWh * 7, Wp = nWw * 7;
  const int sh = (wr * 7 + t / 7 + shift) % Hp, sw = (wc * 7 + t % 7 + shift) % Wp;
  map[r] = (sh < H && sw < W) ? static_cast<int>((static_cast<long>(b) * H + sh) * W + sw) : -1;
}

// PatchMerging gather (swin_transformer.py:279-291): out (b,i,j) <- rows (2i,2j),(2i+1,2j),(2i,2j+1),(2i+1,2j+1)
__global__ void merge_map_kernel(int* map, int B, int H, int W, int H2, int W2) {
  const long r = static_cast<long>(blockIdx.x) * blockDim.x + threadIdx.x;
  const long total = static_cast<long>(B) * H2 * W2;
  if (r >= total) return;
  const int j = static_cast<int>(r % W2), i = static_cast<int>((r / W2) % H2);
  const int b = static_cast<int>(r / (static_cast<long>(W2) * H2));
  const int dy[4] = {0, 1, 0, 1}, dx[4] = {0, 0, 1, 1};
#pragma unroll
  for (int s = 0; s < 4; ++s) {
    const int y = 2 * i + dy[s], x = 2 * j + dx[s];
    map[r * 4 + s] = (y < H && x < W) ? static_cast<int>((static_cast<long>(b) * H + y) * W + x) : -1;
  }
}

// F.interpolate(mode='nearest') source row for every destination pixel (fpn.py:24,28,32).
__global__ void nearest_map_kernel(int* map, int B, int Hd, int Wd, int Hs, int Ws) {
  const long r = static_cast<long>(blockIdx.x) * blockDim.x + threadIdx.x;
  const long total = static_cast<long>(B) * Hd * Wd;
  if (r >= total) return;
  const int x = static_cast<int>(r % Wd), y = static_cast<int>((r / Wd) % Hd);
  const int b = static_cast<int>(r / (static_cast<long>(Wd) * Hd));
  const float sy = static_cast<float>(Hs) / Hd, sx = static_cast<float>(Ws) / Wd;
  const int ys = min(static_cast<int>(floorf(y * sy)), Hs - 1), xs = min(static_cast<int>(floorf(x * sx)), Ws - 1);
  map[r] = static_cast<int>((static_cast<long>(b) * Hs + ys) * Ws + xs);
}

struct Bilin {
  int i0, i1;
  float l0, l1;
};
// F.interpolate(mode='bilinear', align_corners=False) source taps (ATen area_pixel_compute_source_index)
__device__ __forceinline__ Bilin bilin_tap(int dst, int in, int out) {
  const float scale = static_cast<float>(in) / out;
  float src = scale * (dst + 0.5f) - 0.5f;
  if (src < 0.f) src = 0.f;
  Bilin t;
  t.i0 = min(static_cast<int>(src), in - 1);
  t.i1 = t.i0 + (t.i0 < in - 1 ? 1 : 0);
  t.l1 = src - t.i0;
  t.l0 = 1.f - t.l1;
  return t;
}

// Build the input_proj operand: for each consumed pixel (y,x) = (2i,2j) of the stride-8 map, concatenate
// [bilinear(p2), p3, bilinear(p4), bilinear(p5)] (fpn.py:38-44 + the stride-2 sampling of omniparser.py:15).
// One warp per output pixel; lane handles 2 float4 of each 256-channel source.
__global__ void __launch_bounds__(256)
fpn_assemble_kernel(const float* __restrict__ p2, const float* __restrict__ p3, const float* __restrict__ p4,
                    const float* __restrict__ p5, int B, int H0, int W0, int H1, int W1, int H2, int W2, int H3,
                    int W3, int Ho, int Wo, bf16* __restrict__ hi, bf16* __restrict__ lo) {
  const long r = static_cast<long>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const long total = static_cast<long>(B) * Ho * Wo;
  if (r >= total) return;
  const int lane = threadIdx.x & 31;
  const int j = static_cast<int>(r % Wo), i = static_cast<int>((r / Wo) % Ho);
  const int b = static_cast<int>(r / (static_cast<long>(Wo) * Ho));
  const int y = 2 * i, x = 2 * j;  // position in the c3-sized (H1 x W1) map
  const float* srcs[4] = {p2, p3, p4, p5};
  const int Hs[4] = {H0, H1, H2, H3}, Ws[4] = {W0, W1, W2, W3};
#pragma unroll
  for (int s = 0; s < 4; ++s) {
    const float* base = srcs[s] + static_cast<long>(b) * Hs[s] * Ws[s] * 256;
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      const int ch = 4 * (lane + 32 * k);
      float4 v;
      if (s == 1) {
        v = *reinterpret_cast<const float4*>(base + (static_cast<long>(y) * W1 + x) * 256 + ch);
      } else {
        const Bilin ty = bilin_tap(y, Hs[s], H1), tx = bilin_tap(x, Ws[s], W1);
        const float4 a = *reinterpret_cast<const float4*>(base + (static_cast<long>(ty.i0) * Ws[s] + tx.i0) * 256 + ch);
        const float4 bq = *reinterpret_cast<const float4*>(base + (static_cast<long>(ty.i0) * Ws[s] + tx.i1) * 256 + ch);
        const float4 cq = *reinterpret_cast<const float4*>(base + (static_cast<long>(ty.i1) * Ws[s] + tx.i0) * 256 + ch);
        const float4 d = *reinterpret_cast<const float4*>(base + (static_cast<long>(ty.i1) * Ws[s] + tx.i1) * 256 + ch);
        v.x = ty.l0 * (tx.l0 * a.x + tx.l1 * bq.x) + ty.l1 * (tx.l0 * cq.x + tx.l1 * d.x);
        v.y = ty.l0 * (tx.l0 * a.y + tx.l1 * bq.y) + ty.l1 * (tx.l0 * cq.y + tx.l1 * d.y);
        v.z = ty.l0 * (tx.l0 * a.z + tx.l1 * bq.z) + ty.l1 * (tx.l0 * cq.z + tx.l1 * d.z);
        v.w = ty.l0 * (tx.l0 * a.w + tx.l1 * bq.w) + ty.l1 * (tx.l0 * cq.w + tx.l1 * d.w);
      }
      bf16 h0, l0, h1, l1, h2, l2, h3, l3;
      split_bf16(v.x, h0, l0); split_bf16(v.y, h1, l1); split_bf16(v.z, h2, l2); split_bf16(v.w, h3, l3);
      const long off = r * 1024 + s * 256 + ch;
      *reinterpret_cast<uint2*>(hi + off) = make_uint2(pack_bf16(h0, h1), pack_bf16(h2, h3));
      if (lo) *reinterpret_cast<uint2*>(lo + off) = make_uint2(pack_bf16(l0, l1), pack_bf16(l2, l3));
    }
  }
}

// Sine position embedding + key-padding mask at the memory resolution (position_embedding.py:24-44,
// swin_transformer.py:622).  Kernel 1 (one CTA per image): nearest-resized mask, cumulative sums, normalised
// y/x embeddings.  Kernel 2 (elementwise over B*h*w*512): sin / cos.   mask: u8 [B,H,W] or null.
__global__ void __launch_bounds__(256)
sine_embed_kernel(const uint8_t* __restrict__ mask, int H, int W, int h, int w, float* __restrict__ yemb,
                  float* __restrict__ xemb, uint8_t* __restrict__ kpm) {
  extern __shared__ float sm[];
  float* ye = sm;           // [h*w] cumsum over rows
  float* xe = sm + h * w;   // [h*w] cumsum over cols
  const int b = blockIdx.x, t = threadIdx.x;
  const uint8_t* mk = mask ? mask + static_cast<long>(b) * H * W : nullptr;
  const float sy = static_cast<float>(H) / h, sx = static_cast<float>(W) / w;
  for (int i = t; i < h * w; i += blockDim.x) {
    const int y = i / w, x = i % w;
    const int ys = min(static_cast<int>(floorf(y * sy)), H - 1), xs = min(static_cast<int>(floorf(x * sx)), W - 1);
    const uint8_t m = mk ? (mk[static_cast<long>(ys) * W + xs] != 0) : 0;
    kpm[static_cast<long>(b) * h * w + i] = m;
    ye[i] = m ? 0.f : 1.f;
    xe[i] = m ? 0.f : 1.f;
  }
  __syncthreads();
  for (int x = t; x < w; x += blockDim.x) {
    float acc = 0.f;
    for (int y = 0; y < h; ++y) { acc += ye[y * w + x]; ye[y * w + x] = acc; }
  }
  for (int y = t; y < h; y += blockDim.x) {
    float acc = 0.f;
    for (int x = 0; x < w; ++x) { acc += xe[y * w + x]; xe[y * w + x] = acc; }
  }
  __syncthreads();
  const float two_pi = 6.283185307179586f;
  for (int i = t; i < h * w; i += blockDim.x) {
    const int y = i / w, x = i % w;
    yemb[static_cast<long>(b) * h * w + i] = ye[i] / (ye[(h - 1) * w + x] + 1e-6f) * two_pi;
    xemb[static_cast<long>(b) * h * w + i] = xe[i] / (xe[y * w + (w - 1)] + 1e-6f) * two_pi;
  }
}
__global__ void sine_pos_kernel(const float* __restrict__ yemb, const float* __restrict__ xemb,
                                const float* __restrict__ dim_t, long npix, float* __restrict__ pos) {
  const long i = static_cast<long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= npix * 512) return;
  const int c = static_cast<int>(i & 511);
  const long px = i >> 9;
  const int cc = c & 255;
  const float a = (c < 256 ? yemb[px] : xemb[px]) / dim_t[cc];
  pos[i] = (cc & 1) ? cosf(a) : sinf(a);
}

// ----------------------------------------------------------------------------------------------- decoder
// x[s] = LN(word_emb[tok[s, t]] + pos_emb[t])   (transformer.py:313-325).  One warp per sequence, d = 512.
__global__ void __launch_bounds__(256)
embed_ln_kernel(const int* __restrict__ tokens, int tstride, const int* __restrict__ tptr, int S,
                const float* __restrict__ word_emb, const float* __restrict__ pos_emb, const float* __restrict__ gamma,
                const float* __restrict__ beta, float* __restrict__ x, float* __restrict__ qpos) {
  const int s = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (s >= S) return;
  const int lane = threadIdx.x & 31;
  const int t = *tptr;  // device-side position counter: the same captured graph serves every token
  if (s == 0) {         // query_pos of this step (transformer.py:328), read by every layer
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int e = 4 * (lane + 32 * j);
      *reinterpret_cast<float4*>(qpos + e) = *reinterpret_cast<const float4*>(pos_emb + static_cast<long>(t) * 512 + e);
    }
  }
  const int tok = tokens[static_cast<long>(s) * tstride + t];
  float4 v[4];
  float sum = 0.f;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int e = 4 * (lane + 32 * j);
    const float4 a = *reinterpret_cast<const float4*>(word_emb + static_cast<long>(tok) * 512 + e);
    const float4 p = *reinterpret_cast<const float4*>(pos_emb + static_cast<long>(t) * 512 + e);
    v[j] = make_float4(a.x + p.x, a.y + p.y, a.z + p.z, a.w + p.w);
    sum += (v[j].x + v[j].y) + (v[j].z + v[j].w);
  }
  const float mean = warp_sum(sum) * (1.f / 512);
  float q = 0.f;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const float a = v[j].x - mean, b = v[j].y - mean, c = v[j].z - mean, d = v[j].w - mean;
    q += (a * a + b * b) + (c * c + d * d);
  }
  const float rstd = rsqrtf(warp_sum(q) * (1.f / 512) + 1e-5f);
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int e = 4 * (lane + 32 * j);
    const float4 g = *reinterpret_cast<const float4*>(gamma + e);
    const float4 bb = *reinterpret_cast<const float4*>(beta + e);
    float4 y;
    y.x = (v[j].x - mean) * rstd * g.x + bb.x; y.y = (v[j].y - mean) * rstd * g.y + bb.y;
    y.z = (v[j].z - mean) * rstd * g.z + bb.z; y.w = (v[j].w - mean) * rstd * g.w + bb.w;
    *reinterpret_cast<float4*>(x + static_cast<long>(s) * 512 + e) = y;
  }
}

// Cached causal self-attention for ONE new position t (transformer.py:439-441 with tgt_mask):
// appends k,v (from the fused projections) to the caches and attends over positions 0..t.
// One warp per (sequence, head); head_dim 64; q is scaled by 1/8 first like nn.MultiheadAttention.
__global__ void __launch_bounds__(128)
self_attn_step_kernel(const float* __restrict__ qk, const float* __restrict__ vnew, float* __restrict__ kc,
                      float* __restrict__ vc, int S, const int* __restrict__ tptr, int Tmax, bf16* __restrict__ out_hi,
                      bf16* __restrict__ out_lo, float* __restrict__ out_f32, int ld_qk, int ld_v) {
  extern __shared__ float sp[];  // [4 warps][Tmax]
  const int t = *tptr;
  const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long g = static_cast<long>(blockIdx.x) * 4 + wid;
  if (g >= static_cast<long>(S) * 8) return;
  const int s = static_cast<int>(g >> 3), h = static_cast<int>(g & 7);
  float* p = sp + wid * Tmax;
  float* krow = kc + (static_cast<long>(s) * Tmax + t) * 512 + h * 64;
  float* vrow = vc + (static_cast<long>(s) * Tmax + t) * 512 + h * 64;
  const float* qrow = qk + static_cast<long>(s) * ld_qk + h * 64;
  // append
  krow[lane] = qrow[512 + lane]; krow[lane + 32] = qrow[512 + lane + 32];
  vrow[lane] = vnew[static_cast<long>(s) * ld_v + h * 64 + lane];
  vrow[lane + 32] = vnew[static_cast<long>(s) * ld_v + h * 64 + lane + 32];
  __syncwarp();
  float q[64];
#pragma unroll
  for (int d = 0; d < 64; d += 4) {
    const float4 a = *reinterpret_cast<const float4*>(qrow + d);
    q[d] = a.x * 0.125f; q[d + 1] = a.y * 0.125f; q[d + 2] = a.z * 0.125f; q[d + 3] = a.w * 0.125f;
  }
  float m = -INFINITY;
  for (int j = lane; j <= t; j += 32) {
    const float* kj = kc + (static_cast<long>(s) * Tmax + j) * 512 + h * 64;
    float a = 0.f;
#pragma unroll
    for (int d = 0; d < 64; d += 4) {
      const float4 kk = *reinterpret_cast<const float4*>(kj + d);
      a = fmaf(q[d], kk.x, a); a = fmaf(q[d + 1], kk.y, a); a = fmaf(q[d + 2], kk.z, a); a = fmaf(q[d + 3], kk.w, a);
    }
    p[j] = a;
    m = fmaxf(m, a);
  }
  m = warp_max(m);
  float sum = 0.f;
  for (int j = lane; j <= t; j += 32) {
    const float e = expf(p[j] - m);
    p[j] = e;
    sum += e;
  }
  sum = warp_sum(sum);
  __syncwarp();
  float o0 = 0.f, o1 = 0.f;
#pragma unroll 8
  for (int j = 0; j <= t; ++j) {
    const float pj = p[j] / sum;
    const float* vj = vc + (static_cast<long>(s) * Tmax + j) * 512 + h * 64;
    o0 = fmaf(pj, vj[lane], o0);
    o1 = fmaf(pj, vj[lane + 32], o1);
  }
  bf16 hh, ll;
  const long o = static_cast<long>(s) * 512 + h * 64;
  if (out_f32) { out_f32[o + lane] = o0; out_f32[o + lane + 32] = o1; }
  if (out_hi) {
    split_bf16(o0, hh, ll); out_hi[o + lane] = hh; if (out_lo) out_lo[o + lane] = ll;
    split_bf16(o1, hh, ll); out_hi[o + lane + 32] = hh; if (out_lo) out_lo[o + lane + 32] = ll;
  }
}

// Same step for FEW sequences (the pt loop: one per image): one CTA of 4 warps per (sequence, head) so that the
// t+1 cached positions are spread over 128 threads instead of one warp -- the step is pure latency.
__global__ void __launch_bounds__(128)
self_attn_step_wide_kernel(const float* __restrict__ qk, const float* __restrict__ vnew, float* __restrict__ kc,
                           float* __restrict__ vc, int S, const int* __restrict__ tptr, int Tmax, bf16* __restrict__ out_hi,
                           bf16* __restrict__ out_lo, float* __restrict__ out_f32, int ld_qk, int ld_v) {
  extern __shared__ __align__(16) float sw[];  // [Tmax] scores / probabilities, then [8][64] partial outputs
  __shared__ __align__(16) float sq[64];
  __shared__ float red[4];
  const int t = *tptr;
  const int tid = threadIdx.x, wid = tid >> 5, lane = tid & 31;
  const int s = blockIdx.x >> 3, h = blockIdx.x & 7;
  float* p = sw;
  float* part = sw + ((Tmax + 3) & ~3);
  const long cbase = static_cast<long>(s) * Tmax * 512 + h * 64;
  const float* qrow = qk + static_cast<long>(s) * ld_qk + h * 64;
  if (tid < 64) {  // append k, v of the new position; stage q / 8
    kc[cbase + static_cast<long>(t) * 512 + tid] = qrow[512 + tid];
    vc[cbase + static_cast<long>(t) * 512 + tid] = vnew[static_cast<long>(s) * ld_v + h * 64 + tid];
    sq[tid] = qrow[tid] * 0.125f;
  }
  __syncthreads();
  float m = -INFINITY;
  for (int j = tid; j <= t; j += 128) {
    const float* kj = kc + cbase + static_cast<long>(j) * 512;
    float a = 0.f;
#pragma unroll
    for (int d = 0; d < 64; d += 4) {
      const float4 kk = *reinterpret_cast<const float4*>(kj + d);
      const float4 qq = *reinterpret_cast<const float4*>(sq + d);
      a = fmaf(qq.x, kk.x, a); a = fmaf(qq.y, kk.y, a); a = fmaf(qq.z, kk.z, a); a = fmaf(qq.w, kk.w, a);
    }
    p[j] = a;
    m = fmaxf(m, a);
  }
  m = warp_max(m);
  if (lane == 0) red[wid] = m;
  __syncthreads();
  m = fmaxf(fmaxf(red[0], red[1]), fmaxf(red[2], red[3]));
  __syncthreads();
  float sum = 0.f;
  for (int j = tid; j <= t; j += 128) {
    const float e = expf(p[j] - m);
    p[j] = e;
    sum += e;
  }
  sum = warp_sum(sum);
  if (lane == 0) red[wid] = sum;
  __syncthreads();
  sum = (red[0] + red[1]) + (red[2] + red[3]);
  // P.V: 8 position groups x 16 threads (4 dims each); every V row is one coalesced 256-byte read
  const int jg = tid >> 4, dq = (tid & 15) * 4;
  float4 o = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 4
  for (int j = jg; j <= t; j += 8) {
    const float pj = p[j] / sum;
    const float4 v = *reinterpret_cast<const float4*>(vc + cbase + static_cast<long>(j) * 512 + dq);
    o.x = fmaf(pj, v.x, o.x); o.y = fmaf(pj, v.y, o.y); o.z = fmaf(pj, v.z, o.z); o.w = fmaf(pj, v.w, o.w);
  }
  *reinterpret_cast<float4*>(part + jg * 64 + dq) = o;
  __syncthreads();
  if (tid < 64) {
    float y = 0.f;
#pragma unroll
    for (int gidx = 0; gidx < 8; ++gidx) y += part[gidx * 64 + tid];
    const long oo = static_cast<long>(s) * 512 + h * 64 + tid;
    if (out_f32) out_f32[oo] = y;
    if (out_hi) {
      bf16 hh, ll;
      split_bf16(y, hh, ll);
      out_hi[oo] = hh;
      if (out_lo) out_lo[oo] = ll;
    }
  }
}

// Fused single-query cross-attention for the pt loop (one live sequence per image, transformer.py:444-447):
// scores = (q / 8) . K_c^T over the M memory tokens of the image, key-padding mask, softmax, P . V_c -- without
// materialising the [S*8, M] score / probability matrices.  K_c / V_c^T are the cached split-bf16 projections
// (hi + lo re-joined to fp32 on load, so the arithmetic is fp32 FMA).  HBM-bound: every (image, head) streams
// its 2 x M x 64 x 4 B of K and V exactly once per layer-step.
//   grid (nimg * 8, nsplit); split partials are merged by the last CTA of each (image, head) (self-resetting
//   counter), so a single launch suffices.
constexpr int XQ_THREADS = 256;

__device__ __forceinline__ void bf16x8_to_f32(const uint4& h, const uint4& l, float (&o)[8]) {
  const uint32_t hh[4] = {h.x, h.y, h.z, h.w}, ll[4] = {l.x, l.y, l.z, l.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    o[2 * i] = __uint_as_float(hh[i] << 16) + __uint_as_float(ll[i] << 16);
    o[2 * i + 1] = __uint_as_float(hh[i] & 0xffff0000u) + __uint_as_float(ll[i] & 0xffff0000u);
  }
}

__global__ void __launch_bounds__(XQ_THREADS)
cross_attn_q1_kernel(const float* __restrict__ q, const bf16* __restrict__ kc_hi, const bf16* __restrict__ kc_lo,
                     const bf16* __restrict__ vt_hi, const bf16* __restrict__ vt_lo, const uint8_t* __restrict__ kpm,
                     int M, int Mpad, int keys_per_split, float* __restrict__ partial, int* __restrict__ counters,
                     bf16* __restrict__ out_hi, bf16* __restrict__ out_lo, float* __restrict__ out_f32) {
  extern __shared__ float xs[];            // [keys_per_split] scores / probabilities
  __shared__ float sq[64];
  __shared__ float red[XQ_THREADS / 32];
  __shared__ float so[64];
  __shared__ int last_flag;
  const int pair = blockIdx.x, img = pair >> 3, h = pair & 7, split = blockIdx.y, nsplit = gridDim.y;
  const int t = threadIdx.x;
  const int k0 = split * keys_per_split, k1 = min(M, k0 + keys_per_split), nk = max(0, k1 - k0);
  if (t < 64) sq[t] = q[static_cast<long>(img) * 512 + h * 64 + t] * 0.125f;  // q scaled first (functional.py MHA)
  __syncthreads();
  // ---- scores: 8 lanes per key (8 dims = 16 B of hi + 16 B of lo each), 4 keys per warp instruction ->
  //      every K_c row is fetched as one coalesced 128-byte line per operand
  float lmax = -INFINITY;
  {
    const int lane = t & 31, wid = t >> 5, sub = lane & 7, kq = lane >> 3;
    float qd[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) qd[e] = sq[8 * sub + e];
    const long kbase = ((static_cast<long>(img) * 96 + h) * M + k0) * 64 + 8 * sub;  // K_c[img][dl(base)][h][key][64]
#pragma unroll 8
    for (int kb = wid * 4; kb < nk; kb += (XQ_THREADS / 32) * 4) {  // warp-uniform trip count (shuffles inside)
      const int kk = kb + kq;
      const bool live = kk < nk;
      float a = 0.f;
      if (live) {
        const uint4 vh = *reinterpret_cast<const uint4*>(kc_hi + kbase + static_cast<long>(kk) * 64);
        const uint4 vl = *reinterpret_cast<const uint4*>(kc_lo + kbase + static_cast<long>(kk) * 64);
        float kf[8];
        bf16x8_to_f32(vh, vl, kf);
#pragma unroll
        for (int e = 0; e < 8; ++e) a = fmaf(qd[e], kf[e], a);
      }
      a += __shfl_xor_sync(0xffffffffu, a, 1);
      a += __shfl_xor_sync(0xffffffffu, a, 2);
      a += __shfl_xor_sync(0xffffffffu, a, 4);
      if (live && sub == 0) {
        if (kpm && kpm[static_cast<long>(img) * M + k0 + kk]) a = -INFINITY;
        xs[kk] = a;
        lmax = fmaxf(lmax, a);
      }
    }
  }
  lmax = warp_max(lmax);
  if ((t & 31) == 0) red[t >> 5] = lmax;
  __syncthreads();
  float m = red[0];
#pragma unroll
  for (int i = 1; i < XQ_THREADS / 32; ++i) m = fmaxf(m, red[i]);
  __syncthreads();
  float lsum = 0.f;
  for (int kk = t; kk < nk; kk += XQ_THREADS) {
    const float e = (m == -INFINITY) ? 0.f : expf(xs[kk] - m);
    xs[kk] = e;
    lsum += e;
  }
  lsum = warp_sum(lsum);
  if ((t & 31) == 0) red[t >> 5] = lsum;
  __syncthreads();
  float l = 0.f;
#pragma unroll
  for (int i = 0; i < XQ_THREADS / 32; ++i) l += red[i];
  // ---- o[d] = sum_k p_k V[k][d] : warp w owns dims 8w..8w+7; lanes span 256 consecutive keys of a V^T row per
  //      step (coalesced 512-byte loads), probabilities come from shared memory; warp reduction per dim.
  {
    const int lane = t & 31, wid = t >> 5;
    const int nk8 = (nk + 7) >> 3;  // groups of 8 keys (p = 0 beyond nk)
    for (int kk = nk + t; kk < nk8 * 8; kk += XQ_THREADS) xs[kk] = 0.f;
    __syncthreads();
    float acc8[8];
#pragma unroll
    for (int dd = 0; dd < 8; ++dd) acc8[dd] = 0.f;
    const long vrow0 = (static_cast<long>(img) * 6144 + h * 64 + wid * 8) * Mpad + k0;
    for (int gidx = lane; gidx < nk8; gidx += 32) {
      // all 16 vector loads of this step (8 dims x hi/lo) are issued before any is consumed
      uint4 vh[8], vl[8];
#pragma unroll
      for (int dd = 0; dd < 8; ++dd) {
        vh[dd] = *reinterpret_cast<const uint4*>(vt_hi + vrow0 + static_cast<long>(dd) * Mpad + 8 * gidx);
        vl[dd] = *reinterpret_cast<const uint4*>(vt_lo + vrow0 + static_cast<long>(dd) * Mpad + 8 * gidx);
      }
      const float4 p0 = *reinterpret_cast<const float4*>(xs + 8 * gidx);
      const float4 p1 = *reinterpret_cast<const float4*>(xs + 8 * gidx + 4);
#pragma unroll
      for (int dd = 0; dd < 8; ++dd) {
        float vf[8];
        bf16x8_to_f32(vh[dd], vl[dd], vf);
        float a = acc8[dd];
        a = fmaf(p0.x, vf[0], a); a = fmaf(p0.y, vf[1], a); a = fmaf(p0.z, vf[2], a); a = fmaf(p0.w, vf[3], a);
        a = fmaf(p1.x, vf[4], a); a = fmaf(p1.y, vf[5], a); a = fmaf(p1.z, vf[6], a); a = fmaf(p1.w, vf[7], a);
        acc8[dd] = a;
      }
    }
#pragma unroll
    for (int dd = 0; dd < 8; ++dd) {
      const float a = warp_sum(acc8[dd]);
      if (lane == 0) so[wid * 8 + dd] = a;
    }
    __syncthreads();
  }
  const int d = t, part = (t < 64) ? 0 : 1;  // threads 0..63 publish one dim each
  const float acc = (t < 64) ? so[t] : 0.f;
  const long obase = static_cast<long>(img) * 512 + h * 64;
  if (nsplit == 1) {
    if (part == 0) {
      const float y = acc / l;
      if (out_f32) out_f32[obase + d] = y;
      if (out_hi) {
        bf16 hh, ll;
        split_bf16(y, hh, ll);
        out_hi[obase + d] = hh;
        if (out_lo) out_lo[obase + d] = ll;
      }
    }
    return;
  }
  // ---- multi-split: publish (m, l, o[64]); the last CTA of the pair merges
  float* my = partial + (static_cast<long>(pair) * nsplit + split) * 66;
  if (part == 0) my[2 + d] = acc;
  if (t == 0) { my[0] = m; my[1] = l; }
  __threadfence();
  __syncthreads();
  if (t == 0) last_flag = (atomicAdd(&counters[pair], 1) == nsplit - 1);
  __syncthreads();
  if (!last_flag) return;
  __threadfence();
  if (t < 64) {
    const float* base = partial + static_cast<long>(pair) * nsplit * 66;
    float mm = -INFINITY;
    for (int sidx = 0; sidx < nsplit; ++sidx) mm = fmaxf(mm, base[sidx * 66]);
    float ltot = 0.f, otot = 0.f;
    for (int sidx = 0; sidx < nsplit; ++sidx) {
      const float ms = base[sidx * 66];
      const float w = (ms == -INFINITY) ? 0.f : expf(ms - mm);
      ltot += w * base[sidx * 66 + 1];
      otot += w * base[sidx * 66 + 2 + t];
    }
    const float y = otot / ltot;
    if (out_f32) out_f32[obase + t] = y;
    if (out_hi) {
      bf16 hh, ll;
      split_bf16(y, hh, ll);
      out_hi[obase + t] = hh;
      if (out_lo) out_lo[obase + t] = ll;
    }
  }
  if (t == 0) counters[pair] = 0;  // ready for the next launch
}

// Softmax over the first `nsoft` logits, zero the disallowed classes, top-1 (transformer.py:108-125,
// 257-261, 273-280).  phase 0 = pt loop (mode alternates with the generated-token index), 1 = poly (bins),
// 2 = rec (chars num_bins..recog_pad + rec_eos).  One CTA per sequence.  Writes tokens[s, t+1] and (optionally)
// prob / EOS state.  The position t comes from the device-side counter so that the step can be graph-replayed.
__global__ void __launch_bounds__(256)
head_select_kernel(const float* __restrict__ logits, int V, int nsoft, int phase, HeadCfg cfg, int* __restrict__ tokens,
                   int tstride, const int* __restrict__ tptr, int n_prompt_m1, float* __restrict__ probs, int pstride,
                   int* __restrict__ finished, int* __restrict__ ntok) {
  __shared__ float redf[8];
  __shared__ int redi[8];
  const int s = blockIdx.x, t = threadIdx.x;
  const int pos_t = *tptr;
  const int gen_index = pos_t - n_prompt_m1;  // index of the token being generated
  const int tnext = pos_t + 1, pidx = gen_index;
  // pt: even step = coordinate or EOS, odd = coordinate (transformer.py:110-115); KIE adds a class slot (:117-123)
  int mode;
  if (phase == 0) mode = cfg.vie ? (gen_index % 3 == 0 ? 0 : (gen_index % 3 == 1 ? 1 : 3)) : (gen_index % 2 == 0 ? 0 : 1);
  else mode = phase;
  const float* x = logits + static_cast<long>(s) * V;
  float m = -INFINITY;
  for (int j = t; j < nsoft; j += 256) m = fmaxf(m, x[j]);
  m = warp_max(m);
  if ((t & 31) == 0) redf[t >> 5] = m;
  __syncthreads();
  m = redf[0];
#pragma unroll
  for (int i = 1; i < 8; ++i) m = fmaxf(m, redf[i]);
  __syncthreads();
  float sum = 0.f, best = -INFINITY;
  int bi = 0x7fffffff;
  for (int j = t; j < nsoft; j += 256) {
    const float v = x[j];
    sum += expf(v - m);
    bool ok;
    if (mode == 0) ok = j < cfg.num_bins || j == cfg.pt_eos;
    else if (mode == 1) ok = j < cfg.num_bins;
    else if (mode == 2) ok = (j >= cfg.num_bins && j <= cfg.recog_pad) || j == cfg.rec_eos;
    else ok = j >= V - cfg.vie;
    if (ok && v > best) { best = v; bi = j; }
  }
  sum = warp_sum(sum);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ob = __shfl_xor_sync(0xffffffffu, best, o);
    const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
    if (ob > best || (ob == best && oi < bi)) { best = ob; bi = oi; }
  }
  if ((t & 31) == 0) { redf[t >> 5] = sum; }
  __syncthreads();
  float tot = 0.f;
#pragma unroll
  for (int i = 0; i < 8; ++i) tot += redf[i];
  __syncthreads();
  if ((t & 31) == 0) { redf[t >> 5] = best; redi[t >> 5] = bi; }
  __syncthreads();
  if (t == 0) {
    for (int i = 1; i < 8; ++i)
      if (redf[i] > best || (redf[i] == best && redi[i] < bi)) { best = redf[i]; bi = redi[i]; }
    const float prob = expf(best - m) / tot;
    tokens[static_cast<long>(s) * tstride + tnext] = bi;
    if (probs) probs[static_cast<long>(s) * pstride + pidx] = prob;
    if (finished) {  // pt loop: per-sequence EOS bookkeeping (transformer.py:126-127; one window prompt each)
      if (!finished[s]) {
        if (bi == cfg.pt_eos) finished[s] = 1;
        else ntok[s] = gen_index + 1;
      }
    }
  }
}

// poly / rec prompts: [x, y, sos] per decoded point (transformer.py:252,268); dead slots get zeros.
__global__ void build_inst_prompts_kernel(const int* __restrict__ pt_tokens, int pt_stride, int n_prompt,
                                          const int* __restrict__ ntok, int B, int Ncap, int sos,
                                          int* __restrict__ tokens, int tstride) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * Ncap) return;
  const int b = i / Ncap, n = i % Ncap;
  const int ninst = ntok[b] / 2;
  int* row = tokens + static_cast<long>(i) * tstride;
  if (n < ninst) {
    row[0] = pt_tokens[static_cast<long>(b) * pt_stride + n_prompt + 2 * n];
    row[1] = pt_tokens[static_cast<long>(b) * pt_stride + n_prompt + 2 * n + 1];
  } else {
    row[0] = 0; row[1] = 0;
  }
  row[2] = sos;
}

__global__ void add_i32_kernel(int* p, int v) { *p += v; }

__global__ void fill_i32_kernel(int* p, long n, int v) {
  const long i = static_cast<long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i < n) p[i] = v;
}

}  // namespace

void window_map(Ctx* c, int* map, int B, int H, int W, int nWh, int nWw, int shift) {
  const long total = static_cast<long>(B) * nWh * nWw * 49;
  window_map_kernel<<<static_cast<unsigned>((total + 255) / 256), 256, 0, c->stream>>>(map, B, H, W, nWh, nWw, shift);
  count_launch(c); check_launch("window_map");
}
void merge_map(Ctx* c, int* map, int B, int H, int W, int H2, int W2) {
  const long total = static_cast<long>(B) * H2 * W2;
  merge_map_kernel<<<static_cast<unsigned>((total + 255) / 256), 256, 0, c->stream>>>(map, B, H, W, H2, W2);
  count_launch(c); check_launch("merge_map");
}
void nearest_map(Ctx* c, int* map, int B, int Hd, int Wd, int Hs, int Ws) {
  const long total = static_cast<long>(B) * Hd * Wd;
  nearest_map_kernel<<<static_cast<unsigned>((total + 255) / 256), 256, 0, c->stream>>>(map, B, Hd, Wd, Hs, Ws);
  count_launch(c); check_launch("nearest_map");
}
void fpn_assemble(Ctx* c, const float* p2, const float* p3, const float* p4, const float* p5, int B, const int* Hs,
                  const int* Ws, int Ho, int Wo, bf16* hi, bf16* lo) {
  const long total = static_cast<long>(B) * Ho * Wo;
  fpn_assemble_kernel<<<static_cast<unsigned>((total + 7) / 8), 256, 0, c->stream>>>(
      p2, p3, p4, p5, B, Hs[0], Ws[0], Hs[1], Ws[1], Hs[2], Ws[2], Hs[3], Ws[3], Ho, Wo, hi, lo);
  count_launch(c); check_launch("fpn_assemble");
}
void sine_pos(Ctx* c, const uint8_t* mask, int B, int H, int W, int h, int w, const float* dim_t, float* pos,
              uint8_t* kpm, float* scratch /* 2*B*h*w floats */) {
  const size_t sm = static_cast<size_t>(2) * h * w * sizeof(float);
  ALM_REQUIRE(sm <= 200 * 1024, ALM_ERR_UNSUPPORTED, "sine_pos: memory grid too large for shared memory");
  static DeviceOnce attr;
  if (attr.need()) {
    ALM_CHECK_CUDA(cudaFuncSetAttribute(sine_embed_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    attr.mark();
  }
  const long npix = static_cast<long>(B) * h * w;
  float* yemb = scratch;
  float* xemb = scratch + npix;
  sine_embed_kernel<<<B, 256, sm, c->stream>>>(mask, H, W, h, w, yemb, xemb, kpm);
  sine_pos_kernel<<<static_cast<unsigned>((npix * 512 + 255) / 256), 256, 0, c->stream>>>(yemb, xemb, dim_t, npix, pos);
  count_launch(c, 2); check_launch("sine_pos");
}
void embed_ln(Ctx* c, const int* tokens, int tstride, const int* tptr, int S, const float* word_emb,
              const float* pos_emb, const float* gamma, const float* beta, float* x, float* qpos) {
  ALM_PIN_CARVEOUT(embed_ln_kernel);
  embed_ln_kernel<<<(S + 7) / 8, 256, 0, c->stream>>>(tokens, tstride, tptr, S, word_emb, pos_emb, gamma, beta, x, qpos);
  count_launch(c); check_launch("embed_ln");
}
void self_attn_step(Ctx* c, const float* qk, const float* vnew, float* kc, float* vc, int S, const int* t, int Tmax,
                    bf16* out_hi, bf16* out_lo, float* out_f32, int ld_qk, int ld_v) {
  if (c->skipped(8)) return;
  const long groups = static_cast<long>(S) * 8;
  if (groups <= 4L * c->num_sms && c->sattn_wide) {  // few sequences: a whole CTA per (sequence, head)
    const size_t sm = (static_cast<size_t>((Tmax + 3) & ~3) + 8 * 64) * sizeof(float);
    ALM_PIN_CARVEOUT(self_attn_step_wide_kernel);
    self_attn_step_wide_kernel<<<static_cast<unsigned>(groups), 128, sm, c->stream>>>(qk, vnew, kc, vc, S, t, Tmax, out_hi,
                                                                                   out_lo, out_f32, ld_qk, ld_v);
    count_launch(c); check_launch("self_attn_step_wide");
    return;
  }
  const size_t sm = static_cast<size_t>(4) * Tmax * sizeof(float);
  ALM_PIN_CARVEOUT(self_attn_step_kernel);
  self_attn_step_kernel<<<static_cast<unsigned>((groups + 3) / 4), 128, sm, c->stream>>>(qk, vnew, kc, vc, S, t, Tmax,
                                                                                        out_hi, out_lo, out_f32, ld_qk, ld_v);
  count_launch(c); check_launch("self_attn_step");
}
void head_select(Ctx* c, const float* logits, int S, int V, int nsoft, int phase, const HeadCfg& cfg, int* tokens,
                 int tstride, const int* tptr, int n_prompt_m1, float* probs, int pstride, int* finished, int* ntok) {
  ALM_PIN_CARVEOUT(head_select_kernel);
  head_select_kernel<<<S, 256, 0, c->stream>>>(logits, V, nsoft, phase, cfg, tokens, tstride, tptr, n_prompt_m1, probs,
                                               pstride, finished, ntok);
  count_launch(c); check_launch("head_select");
}
void build_inst_prompts(Ctx* c, const int* pt_tokens, int pt_stride, int n_prompt, const int* ntok, int B, int Ncap,
                        int sos, int* tokens, int tstride) {
  build_inst_prompts_kernel<<<(B * Ncap + 255) / 256, 256, 0, c->stream>>>(pt_tokens, pt_stride, n_prompt, ntok, B,
                                                                           Ncap, sos, tokens, tstride);
  count_launch(c); check_launch("build_inst_prompts");
}
void cross_attn_q1(Ctx* c, const float* q, const bf16* kc_hi, const bf16* kc_lo, const bf16* vt_hi, const bf16* vt_lo,
                   const uint8_t* kpm, int nimg, int M, int Mpad, float* partial, int* counters, int nsplit,
                   bf16* out_hi, bf16* out_lo, float* out_f32) {
  if (c->skipped(1)) return;
  int kps = (M + nsplit - 1) / nsplit;
  kps = (kps + 7) & ~7;
  const size_t sm = static_cast<size_t>(kps) * sizeof(float);
  ALM_REQUIRE(sm <= 160 * 1024, ALM_ERR_UNSUPPORTED, "cross_attn_q1: split too long for shared memory");
  static DeviceOnce attr;
  if (attr.need()) {
    ALM_CHECK_CUDA(cudaFuncSetAttribute(cross_attn_q1_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024));
    pin_carveout(cross_attn_q1_kernel);
    attr.mark();
  }
  dim3 grid(nimg * 8, nsplit);
  cross_attn_q1_kernel<<<grid, XQ_THREADS, sm, c->stream>>>(q, kc_hi, kc_lo, vt_hi, vt_lo, kpm, M, Mpad, kps, partial,
                                                            counters, out_hi, out_lo, out_f32);
  count_launch(c); check_launch("cross_attn_q1");
}
int cross_attn_q1_splits(Ctx* c, int nimg, int M) {
  int ns = (6 * c->num_sms + nimg * 8 - 1) / (nimg * 8);  // ~6 resident CTAs per SM keep HBM busy across phases
  ns = std::max(1, std::min(ns, 16));
  while (ns > 1 && (M + ns - 1) / ns < 256) --ns;
  return ns;
}
void add_i32(Ctx* c, int* p, int v) {
  ALM_PIN_CARVEOUT(add_i32_kernel);
  add_i32_kernel<<<1, 1, 0, c->stream>>>(p, v);
  count_launch(c); check_launch("add_i32");
}
void fill_i32(Ctx* c, int* p, long n, int v) {
  if (n == 0) return;
  fill_i32_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, c->stream>>>(p, n, v);
  count_launch(c); check_launch("fill_i32");
}

}  // namespace alm
