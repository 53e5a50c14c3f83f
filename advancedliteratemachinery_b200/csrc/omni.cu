// OmniParser forward on the GPU: Swin-B encoder -> FPN -> input_proj -> three KV-cached point-conditioned
// decoders.  This file is the host-side graph (sequence of kernel launches on the context stream); the
// arithmetic lives in gemm.cu / kernels.cu / omni_kernels.cu.
//
// Reference being replaced (relative to /root/reference/OCR/OmniParser/):
//   model/omniparser.py:19-32, model/backbone/swin_transformer.py:597-625, model/fpn.py:21-45,
//   model/backbone/position_embedding.py:24-44, model/transformer.py:74-141,219-286.
#include <math.h>

#include <algorithm>

#include "omni.h"

namespace alm {

SplitW upload_split(Ctx* c, const float* w, int N, int K, int Kpad);

namespace {

const int kDepths[4] = {2, 2, 18, 2};
const int kHeads[4] = {4, 8, 16, 32};

LNW load_ln(Ctx* c, const std::map<std::string, HostTensor>& t, const std::string& p, int dim) {
  const HostTensor& g = need(t, p + ".weight");
  const HostTensor& b = need(t, p + ".bias");
  ALM_REQUIRE(static_cast<int>(g.numel()) == dim && static_cast<int>(b.numel()) == dim, ALM_ERR_INVALID,
              "LayerNorm shape mismatch at " + p);
  LNW l;
  l.g = upload_f32(c, g.f32.data(), dim);
  l.b = upload_f32(c, b.f32.data(), dim);
  return l;
}

Lin load_lin(Ctx* c, const std::map<std::string, HostTensor>& t, const std::string& p, int N, int K, bool bias = true,
             int Kpad = 0, bool keep_f32 = false) {
  const HostTensor& w = need(t, p + ".weight");
  ALM_REQUIRE(static_cast<long>(w.numel()) == static_cast<long>(N) * K, ALM_ERR_INVALID,
              "Linear weight shape mismatch at " + p);
  Lin l;
  l.w = upload_split(c, w.f32.data(), N, K, Kpad);
  if (keep_f32) l.wf = upload_f32(c, w.f32.data(), w.numel());
  if (bias) {
    const HostTensor& b = need(t, p + ".bias");
    ALM_REQUIRE(static_cast<int>(b.numel()) == N, ALM_ERR_INVALID, "Linear bias shape mismatch at " + p);
    l.b = upload_f32(c, b.f32.data(), N);
  }
  return l;
}

// Swin qkv projection with the attention scale folded into the q rows (swin_transformer.py:130 multiplies q by
// head_dim^-0.5 right after the projection): the GEMM epilogue then emits the operand planes of q*scale directly
Lin load_qkv_qscaled(Ctx* c, const std::map<std::string, HostTensor>& t, const std::string& p, int C) {
  const HostTensor& w = need(t, p + ".weight");
  const HostTensor& b = need(t, p + ".bias");
  ALM_REQUIRE(static_cast<long>(w.numel()) == 3L * C * C && static_cast<long>(b.numel()) == 3L * C, ALM_ERR_INVALID,
              "qkv shape mismatch at " + p);
  std::vector<float> ws(w.f32), bs(b.f32);
  for (size_t i = 0; i < static_cast<size_t>(C) * C; ++i) ws[i] *= WATTN_QSCALE;
  for (int i = 0; i < C; ++i) bs[i] *= WATTN_QSCALE;
  Lin l;
  l.w = upload_split(c, ws.data(), 3 * C, C, 0);
  l.b = upload_f32(c, bs.data(), bs.size());
  return l;
}

// rows [r0, r0+n) of a packed in_proj weight/bias
Lin load_inproj_rows(Ctx* c, const std::map<std::string, HostTensor>& t, const std::string& p, int r0, int n) {
  const HostTensor& w = need(t, p + ".in_proj_weight");
  const HostTensor& b = need(t, p + ".in_proj_bias");
  ALM_REQUIRE(w.numel() == size_t(1536) * 512 && b.numel() == 1536, ALM_ERR_INVALID, "in_proj shape mismatch at " + p);
  Lin l;
  l.w = upload_split(c, w.f32.data() + static_cast<size_t>(r0) * 512, n, 512, 0);
  l.wf = upload_f32(c, w.f32.data() + static_cast<size_t>(r0) * 512, static_cast<size_t>(n) * 512);
  l.b = upload_f32(c, b.f32.data() + r0, n);
  return l;
}

Operand act_op(const bf16* hi, const bf16* lo, long rows, int K, long ld) {
  Operand o;
  o.hi = hi; o.lo = lo; o.rows = static_cast<int>(rows); o.K = K; o.ld = ld;
  return o;
}

struct SplitBuf {
  bf16* hi = nullptr;
  bf16* lo = nullptr;
};
SplitBuf alloc_split(Ctx* c, size_t n) {
  SplitBuf s;
  s.hi = c->ws.get<bf16>(n);
  s.lo = c->ws.get<bf16>(n);
  return s;
}

void linear(Ctx* c, const SplitBuf& a, long rows, const Lin& l, int act, float* out_f32, SplitBuf* out_split,
            const float* resid = nullptr, const int* out_map = nullptr, const int* resid_map = nullptr, long ldr = 0) {
  Epilogue e;
  e.out_f32 = out_f32;
  if (out_split) { e.out_hi = out_split->hi; e.out_lo = out_split->lo; }
  e.ldo = l.w.N;
  e.bias = l.b;
  e.bias_mode = l.b ? BIAS_COL : BIAS_NONE;
  e.act = act;
  e.resid = resid;
  e.ldr = ldr ? ldr : l.w.N;
  e.out_map = out_map;
  e.resid_map = resid_map;
  gemm(c, act_op(a.hi, a.lo, rows, l.w.K, l.w.K), l.w.op(), e);
}

}  // namespace

// ================================================================================================ load
void omni_load(Ctx* c, int kind, const std::map<std::string, HostTensor>& t) {
  OmniModel* m = new OmniModel();
  const std::string bb = "backbone.0.";
  m->patch = load_lin(c, t, bb + "patch_embed.proj", 128, 48, true, 64);
  m->patch_norm = load_ln(c, t, bb + "patch_embed.norm", 128);
  // relative_position_index [49,49] (swin_transformer.py:98-109): recomputed, then cross-checked if present
  std::vector<int> rel_index(49 * 49);
  for (int i = 0; i < 49; ++i)
    for (int j = 0; j < 49; ++j)
      rel_index[i * 49 + j] = (i / 7 - j / 7 + 6) * 13 + (i % 7 - j % 7 + 6);
  for (int s = 0; s < 4; ++s) {
    const int C = 128 << s, heads = kHeads[s];
    m->stage[s].blocks.resize(kDepths[s]);
    for (int b = 0; b < kDepths[s]; ++b) {
      const std::string p = bb + "layers." + std::to_string(s) + ".blocks." + std::to_string(b) + ".";
      SwinBlockW& w = m->stage[s].blocks[b];
      w.n1 = load_ln(c, t, p + "norm1", C);
      w.n2 = load_ln(c, t, p + "norm2", C);
      w.qkv = load_qkv_qscaled(c, t, p + "attn.qkv", C);
      w.proj = load_lin(c, t, p + "attn.proj", C, C);
      w.fc1 = load_lin(c, t, p + "mlp.fc1", 4 * C, C);
      w.fc2 = load_lin(c, t, p + "mlp.fc2", C, 4 * C);
      const HostTensor& tab = need(t, p + "attn.relative_position_bias_table");
      ALM_REQUIRE(static_cast<int>(tab.numel()) == 169 * heads, ALM_ERR_INVALID, "bias table shape mismatch at " + p);
      auto it = t.find(p + "attn.relative_position_index");
      if (it != t.end() && !it->second.placeholder) {
        ALM_REQUIRE(it->second.numel() == 49 * 49, ALM_ERR_INVALID, "relative_position_index shape at " + p);
        for (int i = 0; i < 49 * 49; ++i)
          ALM_REQUIRE(static_cast<int>(it->second.f32[i]) == rel_index[i], ALM_ERR_INVALID,
                      "relative_position_index differs from the Swin definition at " + p);
      }
      std::vector<float> dense(static_cast<size_t>(heads) * 49 * 49);
      for (int h = 0; h < heads; ++h)
        for (int i = 0; i < 49 * 49; ++i) dense[static_cast<size_t>(h) * 2401 + i] = tab.f32[rel_index[i] * heads + h];
      w.bias_dense = upload_f32(c, dense.data(), dense.size());
    }
    m->stage[s].out_norm = load_ln(c, t, bb + "norm" + std::to_string(s), C);
    if (s < 3) {
      const std::string p = bb + "layers." + std::to_string(s) + ".downsample.";
      m->stage[s].merge_norm = load_ln(c, t, p + "norm", 4 * C);
      m->stage[s].merge_red = load_lin(c, t, p + "reduction", 2 * C, 4 * C, false).w;
    }
  }
  const int fpn_in[4] = {1024, 512, 256, 128};
  for (int i = 0; i < 4; ++i) m->fpn[i] = load_lin(c, t, "fpn.fpn_in." + std::to_string(i), 256, fpn_in[i], false).w;
  m->inproj = load_lin(c, t, "input_proj", 512, 1024);
  {
    std::vector<float> dt(256);
    for (int i = 0; i < 256; ++i) dt[i] = powf(10000.0f, (2.0f * static_cast<float>(i / 2)) / 256.0f);
    m->dim_t = upload_f32(c, dt.data(), 256);
  }
  // ---- decoder
  const std::string tr = "transformer.";
  const HostTensor& we = need(t, tr + "embedding.word_embeddings.weight");
  ALM_REQUIRE(we.shape.size() == 2 && we.shape[1] == 512, ALM_ERR_INVALID, "word_embeddings shape");
  m->V = static_cast<int>(we.shape[0]);
  m->vie = m->V - 1104;
  ALM_REQUIRE(m->vie >= 0, ALM_ERR_INVALID, "vocabulary smaller than the text-spotting layout (1104)");
  ALM_REQUIRE(kind != ALM_MODEL_OMNI_SPOT || m->vie == 0, ALM_ERR_INVALID, "text-spotting checkpoint must have V = 1104");
  m->word_emb = upload_f32(c, we.f32.data(), we.numel());
  const char* kinds[3] = {"pt", "poly", "rec"};
  for (int d = 0; d < 3; ++d) {
    const HostTensor& pe = need(t, tr + "embedding." + kinds[d] + "_position_embeddings.weight");
    ALM_REQUIRE(pe.numel() == size_t(1024) * 512, ALM_ERR_INVALID, "position embedding shape");
    m->pos_emb[d] = upload_f32(c, pe.f32.data(), pe.numel());
  }
  m->emb_norm = load_ln(c, t, tr + "embedding.LayerNorm", 512);
  std::vector<float> kw(size_t(12) * 512 * 512), kb(12 * 512), vw(size_t(12) * 512 * 512), vb(12 * 512);
  for (int d = 0; d < 3; ++d) {
    for (int l = 0; l < 4; ++l) {
      const std::string p = tr + kinds[d] + "_decoder.layers." + std::to_string(l) + ".";
      DecLayerW& w = m->dec[d][l];
      w.n1 = load_ln(c, t, p + "norm1", 512);
      w.n2 = load_ln(c, t, p + "norm2", 512);
      w.n3 = load_ln(c, t, p + "norm3", 512);
      {
        const HostTensor& ipw0 = need(t, p + "self_attn.in_proj_weight");
        const HostTensor& ipb0 = need(t, p + "self_attn.in_proj_bias");
        w.sa_qkv_f = upload_f32(c, ipw0.f32.data(), ipw0.numel());
        w.sa_qkv_b = upload_f32(c, ipb0.f32.data(), ipb0.numel());
      }
      w.sa_qk = load_inproj_rows(c, t, p + "self_attn", 0, 1024);
      w.sa_v = load_inproj_rows(c, t, p + "self_attn", 1024, 512);
      w.sa_out = load_lin(c, t, p + "self_attn.out_proj", 512, 512, true, 0, true);
      w.ca_q = load_inproj_rows(c, t, p + "multihead_attn", 0, 512);
      w.ca_out = load_lin(c, t, p + "multihead_attn.out_proj", 512, 512, true, 0, true);
      w.l1 = load_lin(c, t, p + "linear1", 2048, 512, true, 0, true);
      w.l2 = load_lin(c, t, p + "linear2", 512, 2048, true, 0, true);
      const HostTensor& ipw = need(t, p + "multihead_attn.in_proj_weight");
      const HostTensor& ipb = need(t, p + "multihead_attn.in_proj_bias");
      const size_t dl = static_cast<size_t>(d) * 4 + l;
      std::copy(ipw.f32.begin() + size_t(512) * 512, ipw.f32.begin() + size_t(1024) * 512, kw.begin() + dl * 512 * 512);
      std::copy(ipw.f32.begin() + size_t(1024) * 512, ipw.f32.begin() + size_t(1536) * 512, vw.begin() + dl * 512 * 512);
      std::copy(ipb.f32.begin() + 512, ipb.f32.begin() + 1024, kb.begin() + dl * 512);
      std::copy(ipb.f32.begin() + 1024, ipb.f32.begin() + 1536, vb.begin() + dl * 512);
    }
    m->dec_norm[d] = load_ln(c, t, tr + kinds[d] + "_decoder.norm", 512);
    const std::string hp = tr + kinds[d] + "_pred_layer.layers.";
    m->head[d][0] = load_lin(c, t, hp + "0", 512, 512, true, 0, true);
    m->head[d][1] = load_lin(c, t, hp + "1", 512, 512, true, 0, true);
    m->head[d][2] = load_lin(c, t, hp + "2", m->V, 512, true, 0, true);
  }
  m->ca_k_all.w = upload_split(c, kw.data(), 12 * 512, 512, 0);
  m->ca_k_all.b = upload_f32(c, kb.data(), kb.size());
  m->ca_v_all.w = upload_split(c, vw.data(), 12 * 512, 512, 0);
  m->ca_v_all.b = upload_f32(c, vb.data(), vb.size());
  delete c->omni;
  c->omni = m;
}

OmniModel* omni_share(const OmniModel* owner) {
  OmniModel* m = new OmniModel(*owner);  // weight pointers (the slabs are ref-counted by Ctx::wstore)
  m->step_graphs.clear();                // graphs, encode state and cache pointers belong to the owner's arena
  m->encoded = false;
  m->B = m->H = m->W = m->M = m->Mpad = m->mh = m->mw = 0;
  for (auto& f : m->feat) f = nullptr;
  m->memory = m->pos = nullptr;
  m->kpm = nullptr;
  m->kc_hi = m->kc_lo = m->vc_hi = m->vc_lo = m->vt_hi = m->vt_lo = nullptr;
  m->ws_mark = 0;
  return m;
}

// ================================================================================================ encode
void omni_encode(Ctx* c, const float* img, const uint8_t* mask, int B, int H, int W) {
  OmniModel* m = c->omni;
  ALM_REQUIRE(m != nullptr, ALM_ERR_STATE, "alm_omni_encode before alm_load_weights");
  ALM_REQUIRE(B > 0 && H >= 32 && W >= 32, ALM_ERR_INVALID, "image batch must be non-empty and at least 32x32");
  c->ensure_ws();
  Arena& ws = c->ws;
  ws.off = 0;
  m->encoded = false;
  struct CapGuard {
    Ctx* c;
    ~CapGuard() { c->gemm_grid_cap = 0; }
  } cap_guard{c};
  c->gemm_grid_cap = c->enc_grid_cap;
  if (!c->ev_t[0]) for (auto& e : c->ev_t) ALM_CHECK_CUDA(cudaEventCreate(&e));
  ALM_CHECK_CUDA(cudaEventRecord(c->ev_t[0], c->stream));
  m->B = B; m->H = H; m->W = W;
  int hs = (H + 3) / 4, wsz = (W + 3) / 4;
  for (int s = 0; s < 4; ++s) {
    m->Hs[s] = hs; m->Ws[s] = wsz;
    hs = (hs + 1) / 2; wsz = (wsz + 1) / 2;
  }
  m->mh = m->Hs[2]; m->mw = m->Ws[2];
  m->M = m->mh * m->mw;
  m->Mpad = (m->M + 7) & ~7;
  const long BM = static_cast<long>(B) * m->M;

  // ---- encode-persistent buffers
  for (int s = 0; s < 4; ++s) m->feat[s] = ws.get<float>(static_cast<size_t>(B) * m->Hs[s] * m->Ws[s] * (128 << s));
  m->memory = ws.get<float>(BM * 512);
  m->pos = ws.get<float>(BM * 512);
  m->kpm = ws.get<uint8_t>(BM);
  m->kc_hi = ws.get<bf16>(BM * 6144);
  m->kc_lo = ws.get<bf16>(BM * 6144);
  m->vc_hi = ws.get<bf16>(BM * 6144);
  m->vc_lo = ws.get<bf16>(BM * 6144);
  m->vt_hi = m->vt_lo = nullptr;
  if (c->xattn_impl == 1) {  // the unfused debug path multiplies P by a feature-major V_c^T
    m->vt_hi = ws.get<bf16>(static_cast<size_t>(B) * 6144 * m->Mpad);
    m->vt_lo = ws.get<bf16>(static_cast<size_t>(B) * 6144 * m->Mpad);
    // the GEMM writes columns 0..M-1 only; cross_attn_q1 multiplies the padding columns M..Mpad-1 by p = 0, which stays
    // 0 only if they hold finite values -- never whatever the arena held before
    ALM_CHECK_CUDA(cudaMemsetAsync(m->vt_hi, 0, static_cast<size_t>(B) * 6144 * m->Mpad * sizeof(bf16), c->stream));
    ALM_CHECK_CUDA(cudaMemsetAsync(m->vt_lo, 0, static_cast<size_t>(B) * 6144 * m->Mpad * sizeof(bf16), c->stream));
  }
  m->ws_mark = ws.mark();

  // ---- patch embed: im2col -> GEMM(+bias) -> LN   (swin_transformer.py:427-443)
  long rows = static_cast<long>(B) * m->Hs[0] * m->Ws[0];
  float* x = ws.get<float>(rows * 128);
  {
    const size_t mk = ws.mark();
    SplitBuf a = alloc_split(c, rows * 64);
    float* tmp = ws.get<float>(rows * 128);
    im2col_patch4(c, img, B, H, W, m->Hs[0], m->Ws[0], a.hi, a.lo);
    linear(c, a, rows, m->patch, ACT_NONE, tmp, nullptr);
    gather_ln(c, tmp, 128, nullptr, 1, 128, rows, m->patch_norm.g, m->patch_norm.b, 1e-5f, false, nullptr, 0, x, 128,
              nullptr, nullptr, 0, nullptr, nullptr);
    ws.release(mk);
    // x was allocated before mk, tmp/a are dead after the LN (stream-ordered)
  }

  SplitBuf feat_split[4];
  for (int s = 0; s < 4; ++s) {
    const int C = 128 << s, heads = kHeads[s];
    const int Hc = m->Hs[s], Wc = m->Ws[s];
    const int nWh = (Hc + 6) / 7, nWw = (Wc + 6) / 7;
    const long rowsP = static_cast<long>(B) * nWh * nWw * 49;
    rows = static_cast<long>(B) * Hc * Wc;
    const size_t stage_mark = ws.mark();
    int* map0 = ws.get<int>(rowsP);
    int* map1 = ws.get<int>(rowsP);
    window_map(c, map0, B, Hc, Wc, nWh, nWw, 0);
    window_map(c, map1, B, Hc, Wc, nWh, nWw, 3);
    SplitBuf lnw = alloc_split(c, std::max(rowsP, rows) * C);
    SplitBuf qkv = alloc_split(c, rowsP * 3 * C);
    SplitBuf att = alloc_split(c, rowsP * C);
    SplitBuf hid = alloc_split(c, rows * 4 * C);
    for (int b = 0; b < kDepths[s]; ++b) {
      const SwinBlockW& w = m->stage[s].blocks[b];
      const int shift = (b & 1) ? 3 : 0;
      const int* map = shift ? map1 : map0;
      // LN1 -> zero-pad -> roll -> window partition, as one gather (pad tokens stay live keys, F10)
      gather_ln(c, x, C, map, 1, C, rowsP, w.n1.g, w.n1.b, 1e-5f, true, nullptr, 0, nullptr, 0, lnw.hi, lnw.lo, C,
                nullptr, nullptr);
      linear(c, lnw, rowsP, w.qkv, ACT_NONE, nullptr, &qkv);
      window_attention_split(c, qkv.hi, qkv.lo, C, heads, nWh, nWw, B, shift, nWh * 7, nWw * 7, w.bias_dense, att.hi,
                             att.lo, nullptr);
      // proj + window reverse + un-roll + crop + residual, fused in the GEMM epilogue (scatter map)
      linear(c, att, rowsP, w.proj, ACT_NONE, x, nullptr, x, map, nullptr, C);
      gather_ln(c, x, C, nullptr, 1, C, rows, w.n2.g, w.n2.b, 1e-5f, false, nullptr, 0, nullptr, 0, lnw.hi, lnw.lo, C,
                nullptr, nullptr);
      linear(c, lnw, rows, w.fc1, ACT_GELU, nullptr, &hid);
      linear(c, hid, rows, w.fc2, ACT_NONE, x, nullptr, x, nullptr, nullptr, C);
    }
    ws.release(stage_mark);
    // per-stage output norm (swin_transformer.py:616-618): fp32 feature (API) + split operand (FPN)
    feat_split[s] = alloc_split(c, rows * C);
    gather_ln(c, x, C, nullptr, 1, C, rows, m->stage[s].out_norm.g, m->stage[s].out_norm.b, 1e-5f, false, nullptr, 0,
              m->feat[s], C, feat_split[s].hi, feat_split[s].lo, C, nullptr, nullptr);
    if (s < 3) {
      // PatchMerging: 2x2 gather-concat -> LN(4C) -> Linear 4C->2C (swin_transformer.py:269-296)
      const int H2 = m->Hs[s + 1], W2 = m->Ws[s + 1];
      const long rows2 = static_cast<long>(B) * H2 * W2;
      float* xn = ws.get<float>(rows2 * 2 * C);
      const size_t mk = ws.mark();
      int* mm = ws.get<int>(rows2 * 4);
      SplitBuf ma = alloc_split(c, rows2 * 4 * C);
      merge_map(c, mm, B, Hc, Wc, H2, W2);
      gather_ln(c, x, C, mm, 4, C, rows2, m->stage[s].merge_norm.g, m->stage[s].merge_norm.b, 1e-5f, false, nullptr, 0,
                nullptr, 0, ma.hi, ma.lo, 4 * C, nullptr, nullptr);
      Lin red;
      red.w = m->stage[s].merge_red;
      linear(c, ma, rows2, red, ACT_NONE, xn, nullptr);
      ws.release(mk);
      x = xn;
    }
  }

  // ---- FPN (fpn.py:21-45): p5, p4 = c4' + up(p5), p3, p2 at full resolution, fp32
  float* p[4];  // p[0]=p2 (stage 0 res) ... p[3]=p5
  for (int s = 0; s < 4; ++s) p[s] = ws.get<float>(static_cast<size_t>(B) * m->Hs[s] * m->Ws[s] * 256);
  for (int s = 3; s >= 0; --s) {
    rows = static_cast<long>(B) * m->Hs[s] * m->Ws[s];
    Lin l;
    l.w = m->fpn[3 - s];
    if (s == 3) {
      linear(c, feat_split[s], rows, l, ACT_NONE, p[s], nullptr);
    } else {
      const size_t mk = ws.mark();
      int* up = ws.get<int>(rows);
      nearest_map(c, up, B, m->Hs[s], m->Ws[s], m->Hs[s + 1], m->Ws[s + 1]);
      linear(c, feat_split[s], rows, l, ACT_NONE, p[s], nullptr, p[s + 1], nullptr, up, 256);
      ws.release(mk);  // map is consumed by the GEMM already enqueued; later allocations are stream-ordered after it
    }
  }
  // consumer-side assembly of the stride-2-sampled concat + input_proj (omniparser.py:15,31)
  SplitBuf cat = alloc_split(c, BM * 1024);
  fpn_assemble(c, p[0], p[1], p[2], p[3], B, m->Hs, m->Ws, m->mh, m->mw, cat.hi, cat.lo);
  linear(c, cat, BM, m->inproj, ACT_NONE, m->memory, nullptr);
  {
    float* scratch = ws.get<float>(static_cast<size_t>(2) * BM);
    sine_pos(c, mask, B, H, W, m->mh, m->mw, m->dim_t, m->pos, m->kpm, scratch);
  }
  // operands for the cross-attention K/V projections: memory and memory + pos
  SplitBuf mem = alloc_split(c, BM * 512), memp = alloc_split(c, BM * 512);
  gather_ln(c, m->memory, 512, nullptr, 1, 512, BM, nullptr, nullptr, 0.f, false, m->pos, 512, nullptr, 0, mem.hi,
            mem.lo, 512, memp.hi, memp.lo);
  {  // K_c[b][dl][h][m][64] = (memory + pos) Wk^T + bk for all 12 (decoder, layer) pairs: head-major so that the keys
     // of one (image, layer, head) are one contiguous 128-byte-row block (the per-token decode streams exactly that)
    Operand a = act_op(memp.hi, memp.lo, m->M, 512, 512);
    a.nb1 = B; a.bs1 = static_cast<long>(m->M) * 512;
    Operand w = m->ca_k_all.w.op();
    w.rows = 512; w.nb0 = 4 * c->kv_decoders; w.bs0 = static_cast<long>(512) * 512;  // (decoder, layer) slices, 8 heads wide
    Epilogue e;
    e.out_hi = m->kc_hi; e.out_lo = m->kc_lo; e.ldo = 64;
    e.obs0 = static_cast<long>(8) * m->M * 64; e.obs1 = static_cast<long>(96) * m->M * 64;
    e.col_group = 64; e.col_group_stride = static_cast<long>(m->M) * 64;  // head h = column / 64 -> its own [M, 64] block
    e.bias = m->ca_k_all.b; e.bias_mode = BIAS_COL; e.bias_bs0 = 512;
    gemm(c, a, w, e);
  }
  {  // V_c[b][dl][h][m][64] = memory Wv^T + bv, same head-major layout: a 64-key block of one (image, layer, head) is
     // one contiguous 8 KB run per plane, which is what the fused attention streams
    Operand a = act_op(mem.hi, mem.lo, m->M, 512, 512);
    a.nb1 = B; a.bs1 = static_cast<long>(m->M) * 512;
    Operand w = m->ca_v_all.w.op();
    w.rows = 512; w.nb0 = 4 * c->kv_decoders; w.bs0 = static_cast<long>(512) * 512;
    Epilogue e;
    e.out_hi = m->vc_hi; e.out_lo = m->vc_lo; e.ldo = 64;
    e.obs0 = static_cast<long>(8) * m->M * 64; e.obs1 = static_cast<long>(96) * m->M * 64;
    e.col_group = 64; e.col_group_stride = static_cast<long>(m->M) * 64;
    e.bias = m->ca_v_all.b; e.bias_mode = BIAS_COL; e.bias_bs0 = 512;
    gemm(c, a, w, e);
  }
  if (m->vt_hi) {  // V_c^T[b, dl*512 + f, m] = Wv memory^T + bv  (feature-major so that P.V is a K-major GEMM)
    Operand bop = act_op(mem.hi, mem.lo, m->M, 512, 512);
    bop.nb1 = B; bop.bs1 = static_cast<long>(m->M) * 512;
    Epilogue e;
    e.out_hi = m->vt_hi; e.out_lo = m->vt_lo; e.ldo = m->Mpad; e.obs1 = static_cast<long>(6144) * m->Mpad;
    e.bias = m->ca_v_all.b; e.bias_mode = BIAS_ROW;
    gemm(c, m->ca_v_all.w.op(), bop, e);
  }
  ws.release(m->ws_mark);
  m->encoded = true;
  m->kv_decoders = c->kv_decoders;
  ALM_CHECK_CUDA(cudaEventRecord(c->ev_t[1], c->stream));
  c->timing_valid[0] = true;
}

// ================================================================================================ decode
namespace {

struct DecodeBufs {
  int S = 0, Tmax = 0, Ncap = 0;
  float* x = nullptr;
  float* qpos = nullptr;  // [512] query_pos of the current step
  int* tpos = nullptr;    // device-side position counter (so one captured graph serves every token)
  SplitBuf ln, lnp, att, q, o, hid, h0, h1;
  float *qk = nullptr, *v = nullptr, *scores = nullptr, *logits = nullptr, *qf = nullptr;
  float* qkv = nullptr;  // skinny path: fused [S,1536] q|k|v
  float *lnf = nullptr, *lnpf = nullptr, *attf = nullptr, *of = nullptr, *hidf = nullptr, *h0f = nullptr, *h1f = nullptr;
  bool skinny = false;          // few live sequences: all-fp32 SIMT GEMV path instead of tensor-core tiles
  float* xq_partial = nullptr;  // fused single-query cross-attention: split partials + counters
  int* xq_counters = nullptr;
  int xq_splits = 1;
  int mq_grid = 1, mq_parts = 1;  // fused cross-attention: persistent grid size, partial slots per (image, head, query block)
  bool fused_xattn = false;
  bool tma_xattn = false;  // fused, TMA + mbarrier variant of the mma.sync kernel (xattn_impl 2)
  bool tc_xattn = false;   // fused, tcgen05 + TMA ring (xattn_impl 3)
  SplitBuf prob;
  float* kc[4] = {nullptr, nullptr, nullptr, nullptr};
  float* vc[4] = {nullptr, nullptr, nullptr, nullptr};
};

// pt_loop: the point loop, whose Ncap sequences per image are the window prompts of the image.  It takes the exact-fp32
// skinny path for at most 32 images and 64 rows (for one prompt per image: at most 32 images, as the other loops).
DecodeBufs alloc_decode(Ctx* c, OmniModel* m, int B, int Ncap, int Tmax, bool pt_loop = false) {
  DecodeBufs d;
  d.S = B * Ncap; d.Tmax = Tmax; d.Ncap = Ncap;
  const size_t S = d.S;
  d.x = c->ws.get<float>(S * 512);
  d.qpos = c->ws.get<float>(512);
  d.tpos = c->ws.get<int>(1);
  d.ln = alloc_split(c, S * 512);
  d.lnp = alloc_split(c, S * 512);
  d.att = alloc_split(c, S * 512);
  d.q = alloc_split(c, S * 512);
  d.o = alloc_split(c, S * 512);
  d.hid = alloc_split(c, S * 2048);
  d.h0 = alloc_split(c, S * 512);
  d.h1 = alloc_split(c, S * 512);
  d.qk = c->ws.get<float>(S * 1024);
  d.v = c->ws.get<float>(S * 512);
  d.qf = c->ws.get<float>(S * 512);
  // several queries per image in the skinny path need the fused cross-attention (the unfused debug path is one query)
  d.skinny = pt_loop ? (B <= 32 && d.S <= 64 && (Ncap == 1 || c->xattn_impl != 1)) : (Ncap == 1 && d.S <= 32);
  if (d.skinny) {
    d.lnf = c->ws.get<float>(S * 512); d.lnpf = c->ws.get<float>(S * 512); d.attf = c->ws.get<float>(S * 512);
    d.of = c->ws.get<float>(S * 512); d.hidf = c->ws.get<float>(S * 2048); d.h0f = c->ws.get<float>(S * 512);
    d.h1f = c->ws.get<float>(S * 512);
    d.qkv = c->ws.get<float>(S * 1536);
  }
  if (c->xattn_impl == 0 || c->xattn_impl == 2 || c->xattn_impl == 3) {
    int pairs = 0;
    d.fused_xattn = true;
    d.tma_xattn = c->xattn_impl == 2;
    // the tcgen05 kernel maps one query row to one thread: right for the 64-query polygon / recognition loops, wrong for
    // the point loop's single query per image (its 128 keys per block would be one lane's serial work) -- that keeps the
    // mma.sync 16-row kernel, which spreads the keys of a block over the warps
    d.tc_xattn = c->xattn_impl == 3 && Ncap > 16;
    if (d.tc_xattn) cross_attn_tc_plan(c, B, Ncap, m->M, &d.mq_grid, &d.mq_parts, &pairs);
    else if (d.tma_xattn) cross_attn_tma_plan(c, B, Ncap, m->M, &d.mq_grid, &d.mq_parts, &pairs);
    else cross_attn_mq_plan(c, B, Ncap, m->M, &d.mq_grid, &d.mq_parts, &pairs);
    d.xq_partial = c->ws.get<float>(cross_attn_mq_partial_floats(pairs, d.mq_parts));
    d.xq_counters = c->ws.get<int>(pairs);
    fill_i32(c, d.xq_counters, pairs, 0);
  } else if (Ncap == 1) {
    d.xq_splits = cross_attn_q1_splits(c, B, m->M);
    d.xq_partial = c->ws.get<float>(static_cast<size_t>(B) * 8 * d.xq_splits * 66);
    d.xq_counters = c->ws.get<int>(static_cast<size_t>(B) * 8);
    fill_i32(c, d.xq_counters, static_cast<long>(B) * 8, 0);
  } else {
    d.scores = c->ws.get<float>(S * 8 * m->Mpad);
    d.prob = alloc_split(c, S * 8 * m->Mpad);
  }
  d.logits = c->ws.get<float>(S * m->V);
  for (int l = 0; l < 4; ++l) {
    d.kc[l] = c->ws.get<float>(S * Tmax * 512);
    d.vc[l] = c->ws.get<float>(S * Tmax * 512);
  }
  return d;
}

// Fused cross-attention of `nimg` images x Ncap queries against decoder-layer dl of the cached K_c / V_c
void fused_xattn(Ctx* c, OmniModel* m, DecodeBufs& u, const bf16* q_hi, const bf16* q_lo, const float* q_f32, int img0, int nimg,
                 int Ncap, long dl, bf16* out_hi, bf16* out_lo, float* out_f32) {
  const int M = m->M;
  const uint8_t* kpm = m->kpm + static_cast<long>(img0) * M;
  if (u.tc_xattn) {
    cross_attn_tc(c, q_hi, q_lo, q_f32, nimg, Ncap, m->kc_hi, m->kc_lo, m->vc_hi, m->vc_lo, static_cast<long>(m->B) * 96,
                  static_cast<int>(img0 * 96 + dl * 8), kpm, M, u.mq_grid, u.mq_parts, u.xq_partial, u.xq_counters, out_hi, out_lo,
                  out_f32);
    return;
  }
  if (u.tma_xattn) {
    cross_attn_tma(c, q_hi, q_lo, q_f32, nimg, Ncap, m->kc_hi, m->kc_lo, m->vc_hi, m->vc_lo, static_cast<long>(m->B) * 96,
                   static_cast<int>(img0 * 96 + dl * 8), kpm, M, u.mq_grid, u.mq_parts, u.xq_partial, u.xq_counters, out_hi,
                   out_lo, out_f32);
    return;
  }
  const long koff = (static_cast<long>(img0) * 96 + dl * 8) * M * 64;
  cross_attn_mq(c, q_hi, q_lo, q_f32, nimg, Ncap, m->kc_hi + koff, m->kc_lo + koff, m->vc_hi + koff, m->vc_lo + koff, kpm, M,
                u.mq_grid, u.mq_parts, u.xq_partial, u.xq_counters, out_hi, out_lo, out_f32);
}

// One decoder pass over the token at position *u.tpos of every sequence (pre-norm layer, transformer.py:430-454,
// with self-attention K/V cached and the cross-attention K/V precomputed per image).
// img0: first image of the batch slice the S sequences belong to; nimg images x Ncap sequences each.
void decoder_step(Ctx* c, OmniModel* m, int d, DecodeBufs& u, const int* tokens, int tstride, int img0, int nimg,
                  bool want_logits) {
  const int S = u.S, Ncap = u.Ncap, M = m->M, Mpad = m->Mpad;
  embed_ln(c, tokens, tstride, u.tpos, S, m->word_emb, m->pos_emb[d], m->emb_norm.g, m->emb_norm.b, u.x, u.qpos);
  const float* qpos = u.qpos;
  if (u.skinny) {
    // At most 32 images and 64 live sequences (Ncap window prompts per image in the point loop, one otherwise): every
    // linear is a skinny fp32 GEMV (exact fp32 weights, one warp per output column), no operand splitting, no tensor-core
    // tile padding.  A row's arithmetic does not depend on how many rows share the launch.
    auto lin = [&](const float* x, int K, const Lin& w, int act, float* out, const float* resid) {
      gemv_rows(c, x, nullptr, 1 << 30, K, w.wf, w.b, resid, w.w.N, out, w.w.N, S, w.w.N, K, act);
    };
    c->skip_scope = true;  // (timing experiments: alm_set_option debug_skip drops kernel classes inside the layers)
    if (c->fuse_ln_gemv && u.fused_xattn) {
      // same arithmetic, 13 fewer dependent launches per token: every pre-LayerNorm (+ query position) is applied by the
      // GEMV that consumes it, on its own staged copy of the rows
      auto lnlin = [&](const LNW& n, const float* pos, int pos_split, const float* W_, const float* b_, int N_, int act,
                       float* out, long ldo) {
        gemv_rows(c, u.x, nullptr, 1 << 30, 512, W_, b_, nullptr, 0, out, ldo, S, N_, 512, act, n.g, n.b, 1e-5f, pos, pos_split);
      };
      for (int l = 0; l < 4; ++l) {
        const DecLayerW& w = m->dec[d][l];
        const long dl = static_cast<long>(d) * 4 + l;
        lnlin(w.n1, qpos, 1024, w.sa_qkv_f, w.sa_qkv_b, 1536, ACT_NONE, u.qkv, 1536);   // q | k from LN(x)+pos, v from LN(x)
        self_attn_step(c, u.qkv, u.qkv + 1024, u.kc[l], u.vc[l], S, u.tpos, u.Tmax, nullptr, nullptr, u.attf, 1536, 1536);
        lin(u.attf, 512, w.sa_out, ACT_NONE, u.x, u.x);
        lnlin(w.n2, qpos, 1 << 30, w.ca_q.wf, w.ca_q.b, 512, ACT_NONE, u.qf, 512);
        fused_xattn(c, m, u, nullptr, nullptr, u.qf, img0, nimg, Ncap, dl, nullptr, nullptr, u.of);
        lin(u.of, 512, w.ca_out, ACT_NONE, u.x, u.x);
        lnlin(w.n3, nullptr, 0, w.l1.wf, w.l1.b, 2048, ACT_RELU, u.hidf, 2048);
        lin(u.hidf, 2048, w.l2, ACT_NONE, u.x, u.x);
      }
      c->skip_scope = false;
      if (!want_logits) return;
      lnlin(m->dec_norm[d], nullptr, 0, m->head[d][0].wf, m->head[d][0].b, 512, ACT_RELU, u.h0f, 512);
      lin(u.h0f, 512, m->head[d][1], ACT_RELU, u.h1f, nullptr);
      lin(u.h1f, 512, m->head[d][2], ACT_NONE, u.logits, nullptr);
      return;
    }
    for (int l = 0; l < 4; ++l) {
      const DecLayerW& w = m->dec[d][l];
      const long dl = static_cast<long>(d) * 4 + l;
      gather_ln(c, u.x, 512, nullptr, 1, 512, S, w.n1.g, w.n1.b, 1e-5f, false, qpos, 0, u.lnf, 512, nullptr, nullptr, 512,
                nullptr, nullptr, u.lnpf);
      // q|k from LN(x)+pos and v from LN(x) in ONE launch: the fp32 in_proj rows are contiguous (q, k, v)
      gemv_rows(c, u.lnpf, u.lnf, 1024, 512, w.sa_qkv_f, w.sa_qkv_b, nullptr, 0, u.qkv, 1536, S, 1536, 512, ACT_NONE);
      self_attn_step(c, u.qkv, u.qkv + 1024, u.kc[l], u.vc[l], S, u.tpos, u.Tmax, nullptr, nullptr, u.attf, 1536, 1536);
      lin(u.attf, 512, w.sa_out, ACT_NONE, u.x, u.x);
      gather_ln(c, u.x, 512, nullptr, 1, 512, S, w.n2.g, w.n2.b, 1e-5f, false, qpos, 0, nullptr, 512, nullptr, nullptr, 512,
                nullptr, nullptr, u.lnpf);
      lin(u.lnpf, 512, w.ca_q, ACT_NONE, u.qf, nullptr);
      const long koff = (static_cast<long>(img0) * 96 + dl * 8) * M * 64;
      const long voff = (static_cast<long>(img0) * 6144 + dl * 512) * Mpad;
      if (u.fused_xattn)
        fused_xattn(c, m, u, nullptr, nullptr, u.qf, img0, nimg, Ncap, dl, nullptr, nullptr, u.of);
      else
        cross_attn_q1(c, u.qf, m->kc_hi + koff, m->kc_lo + koff, m->vt_hi + voff, m->vt_lo + voff,
                      m->kpm + static_cast<long>(img0) * M, nimg, M, Mpad, u.xq_partial, u.xq_counters, u.xq_splits, nullptr,
                      nullptr, u.of);
      lin(u.of, 512, w.ca_out, ACT_NONE, u.x, u.x);
      gather_ln(c, u.x, 512, nullptr, 1, 512, S, w.n3.g, w.n3.b, 1e-5f, false, nullptr, 0, u.lnf, 512, nullptr, nullptr, 512,
                nullptr, nullptr);
      lin(u.lnf, 512, w.l1, ACT_RELU, u.hidf, nullptr);
      lin(u.hidf, 2048, w.l2, ACT_NONE, u.x, u.x);
    }
    c->skip_scope = false;
    if (!want_logits) return;
    gather_ln(c, u.x, 512, nullptr, 1, 512, S, m->dec_norm[d].g, m->dec_norm[d].b, 1e-5f, false, nullptr, 0, u.lnf, 512,
              nullptr, nullptr, 512, nullptr, nullptr);
    lin(u.lnf, 512, m->head[d][0], ACT_RELU, u.h0f, nullptr);
    lin(u.h0f, 512, m->head[d][1], ACT_RELU, u.h1f, nullptr);
    lin(u.h1f, 512, m->head[d][2], ACT_NONE, u.logits, nullptr);
    return;
  }
  c->skip_scope = true;
  for (int l = 0; l < 4; ++l) {
    const DecLayerW& w = m->dec[d][l];
    const long dl = static_cast<long>(d) * 4 + l;
    // --- self attention
    gather_ln(c, u.x, 512, nullptr, 1, 512, S, w.n1.g, w.n1.b, 1e-5f, false, qpos, 0, nullptr, 0, u.ln.hi, u.ln.lo, 512,
              u.lnp.hi, u.lnp.lo);
    linear(c, u.lnp, S, w.sa_qk, ACT_NONE, u.qk, nullptr);
    linear(c, u.ln, S, w.sa_v, ACT_NONE, u.v, nullptr);
    self_attn_step(c, u.qk, u.v, u.kc[l], u.vc[l], S, u.tpos, u.Tmax, u.att.hi, u.att.lo);
    linear(c, u.att, S, w.sa_out, ACT_NONE, u.x, nullptr, u.x, nullptr, nullptr, 512);
    // --- cross attention against the per-image cached K / V^T
    gather_ln(c, u.x, 512, nullptr, 1, 512, S, w.n2.g, w.n2.b, 1e-5f, false, qpos, 0, nullptr, 0, nullptr, nullptr, 512,
              u.lnp.hi, u.lnp.lo);
    if (Ncap == 1) {
      // one query per image: fused scores + mask + softmax + P.V, K/V streamed once (HBM-bound)
      linear(c, u.lnp, S, w.ca_q, ACT_NONE, u.qf, nullptr);
      const long koff = (static_cast<long>(img0) * 96 + dl * 8) * M * 64;
      const long voff = (static_cast<long>(img0) * 6144 + dl * 512) * Mpad;
      if (u.fused_xattn)
        fused_xattn(c, m, u, nullptr, nullptr, u.qf, img0, nimg, 1, dl, u.o.hi, u.o.lo, nullptr);
      else
        cross_attn_q1(c, u.qf, m->kc_hi + koff, m->kc_lo + koff, m->vt_hi + voff, m->vt_lo + voff,
                      m->kpm + static_cast<long>(img0) * M, nimg, M, Mpad, u.xq_partial, u.xq_counters, u.xq_splits, u.o.hi,
                      u.o.lo);
    } else if (u.fused_xattn) {
      // Ncap queries per image: scores, mask, online softmax and P.V fused; K_c / V_c^T streamed once per layer-step
      linear(c, u.lnp, S, w.ca_q, ACT_NONE, nullptr, &u.q);
      fused_xattn(c, m, u, u.q.hi, u.q.lo, nullptr, img0, nimg, Ncap, dl, u.o.hi, u.o.lo, nullptr);
    } else {
      linear(c, u.lnp, S, w.ca_q, ACT_NONE, nullptr, &u.q);
      {
        Operand a = act_op(u.q.hi, u.q.lo, Ncap, 64, 512);
        a.nb0 = 8; a.bs0 = 64; a.nb1 = nimg; a.bs1 = static_cast<long>(Ncap) * 512;
        const long koff = (static_cast<long>(img0) * 96 + dl * 8) * M * 64;
        Operand k = act_op(m->kc_hi + koff, m->kc_lo + koff, M, 64, 64);
        k.nb0 = 8; k.bs0 = static_cast<long>(M) * 64; k.nb1 = nimg; k.bs1 = static_cast<long>(96) * M * 64;
        Epilogue e;
        e.out_f32 = u.scores; e.ldo = Mpad; e.obs0 = static_cast<long>(Ncap) * Mpad; e.obs1 = static_cast<long>(8) * Ncap * Mpad;
        e.alpha = 0.125f;  // == scaling q by 64^-0.5 before q k^T (exact: power of two)
        gemm(c, a, k, e);
      }
      softmax_rows(c, u.scores, Mpad, static_cast<long>(S) * 8, M, m->kpm + static_cast<long>(img0) * M, 8 * Ncap, M,
                   nullptr, u.prob.hi, u.prob.lo, Mpad);
      {
        Operand a = act_op(u.prob.hi, u.prob.lo, Ncap, M, Mpad);
        a.nb0 = 8; a.bs0 = static_cast<long>(Ncap) * Mpad; a.nb1 = nimg; a.bs1 = static_cast<long>(8) * Ncap * Mpad;
        const long voff = (static_cast<long>(img0) * 6144 + dl * 512) * Mpad;
        Operand v = act_op(m->vt_hi + voff, m->vt_lo + voff, 64, M, Mpad);
        v.nb0 = 8; v.bs0 = static_cast<long>(64) * Mpad; v.nb1 = nimg; v.bs1 = static_cast<long>(6144) * Mpad;
        Epilogue e;
        e.out_hi = u.o.hi; e.out_lo = u.o.lo; e.ldo = 512; e.obs0 = 64; e.obs1 = static_cast<long>(Ncap) * 512;
        gemm(c, a, v, e);
      }
    }
    linear(c, u.o, S, w.ca_out, ACT_NONE, u.x, nullptr, u.x, nullptr, nullptr, 512);
    // --- FFN
    gather_ln(c, u.x, 512, nullptr, 1, 512, S, w.n3.g, w.n3.b, 1e-5f, false, nullptr, 0, nullptr, 0, u.ln.hi, u.ln.lo,
              512, nullptr, nullptr);
    linear(c, u.ln, S, w.l1, ACT_RELU, nullptr, &u.hid);
    linear(c, u.hid, S, w.l2, ACT_NONE, u.x, nullptr, u.x, nullptr, nullptr, 512);
  }
  c->skip_scope = false;
  if (!want_logits) return;
  gather_ln(c, u.x, 512, nullptr, 1, 512, S, m->dec_norm[d].g, m->dec_norm[d].b, 1e-5f, false, nullptr, 0, nullptr, 0,
            u.ln.hi, u.ln.lo, 512, nullptr, nullptr);
  linear(c, u.ln, S, m->head[d][0], ACT_RELU, nullptr, &u.h0);
  linear(c, u.h0, S, m->head[d][1], ACT_RELU, nullptr, &u.h1);
  linear(c, u.h1, S, m->head[d][2], ACT_NONE, u.logits, nullptr);
}

// Sleep (do not spin) until everything enqueued on `s` has finished.  The decode loops wait for the GPU several
// times per batch and a serving process keeps several contexts (host threads) per GPU in flight: spinning threads
// would fight over the host cores (cgroup quotas are far below the visible CPU count on the GPU boxes).  The
// device-to-pageable-host copies that follow each wait would otherwise spin inside cudaMemcpyAsync.
void wait_stream(Ctx* c, cudaStream_t s) {
  if (!c->ev_block)
    ALM_CHECK_CUDA(cudaEventCreateWithFlags(&c->ev_block, cudaEventBlockingSync | cudaEventDisableTiming));
  ALM_CHECK_CUDA(cudaEventRecord(c->ev_block, s));
  ALM_CHECK_CUDA(cudaEventSynchronize(c->ev_block));
}

struct HeadArgs {
  bool on = false;
  HeadCfg cfg{};
  int* tokens = nullptr;
  int tstride = 0, n_prompt_m1 = 0;
  float* probs = nullptr;
  int pstride = 0;
  int* finished = nullptr;  // pt loop: per-sequence EOS state
  int* ntok = nullptr;
  int nsoft = 0;  // logits entering the softmax (V, or V - vie_categories for the KIE poly/rec loops)
};

// `n` consecutive token steps of decoder d.  The step (all ~62 launches + the counter increment) is captured once
// into a CUDA graph per distinct (shape, pointer) signature and replayed: the per-token host cost drops from
// ~62 launches to one cudaGraphLaunch.
void run_steps(Ctx* c, OmniModel* m, int d, DecodeBufs& u, const int* tokens, int tstride, int img0, int nimg, int n,
               const HeadArgs& h) {
  if (n <= 0) return;
  auto body = [&] {
    decoder_step(c, m, d, u, tokens, tstride, img0, nimg, h.on);
    if (h.on)
      head_select(c, u.logits, u.S, m->V, h.nsoft ? h.nsoft : m->V, d, h.cfg, h.tokens, h.tstride, u.tpos, h.n_prompt_m1, h.probs, h.pstride,
                  h.finished, h.ntok);
    add_i32(c, u.tpos, 1);
  };
  if (!c->use_graphs || c->profile_gemm || c->gemm_impl != 0) {
    for (int i = 0; i < n; ++i) body();
    return;
  }
  std::vector<long> key = {d, u.S, u.Ncap, u.skinny ? 1 : 0, u.Tmax, img0, nimg, m->M, h.on ? 1 : 0, c->nsplit,
                           reinterpret_cast<long>(u.x), reinterpret_cast<long>(tokens), tstride,
                           reinterpret_cast<long>(h.probs), reinterpret_cast<long>(h.finished), h.n_prompt_m1,
                           reinterpret_cast<long>(m->kc_hi), reinterpret_cast<long>(u.kc[3]), h.cfg.pt_eos, h.cfg.num_bins,
                           h.cfg.rec_eos, h.cfg.recog_pad, reinterpret_cast<long>(c->trace_buf), h.nsoft, h.cfg.vie, c->xattn_impl, c->gemm_grid_cap, c->debug_skip, c->xattn_ctas_per_sm, c->sattn_wide, c->xattn_wg, c->fuse_ln_gemv};
  auto it = m->step_graphs.find(key);
  if (it == m->step_graphs.end()) {
    if (m->step_graphs.size() > 64) {
      for (auto& kv : m->step_graphs) cudaGraphExecDestroy(kv.second.exec);
      m->step_graphs.clear();
    }
    const long before = c->launches;
    cudaGraph_t graph = nullptr;
    ALM_CHECK_CUDA(cudaStreamBeginCapture(c->stream, cudaStreamCaptureModeThreadLocal));
    try {
      body();
    } catch (...) {
      cudaStreamEndCapture(c->stream, &graph);
      if (graph) cudaGraphDestroy(graph);
      throw;
    }
    ALM_CHECK_CUDA(cudaStreamEndCapture(c->stream, &graph));
    OmniModel::StepGraph sg{nullptr, c->launches - before};
    c->launches = before;
    cudaError_t e = cudaGraphInstantiate(&sg.exec, graph, 0);
    cudaGraphDestroy(graph);
    if (e != cudaSuccess) throw AlmError{ALM_ERR_CUDA, std::string("cudaGraphInstantiate: ") + cudaGetErrorString(e)};
    it = m->step_graphs.emplace(key, sg).first;
  }
  for (int i = 0; i < n; ++i) ALM_CHECK_CUDA(cudaGraphLaunch(it->second.exec, c->stream));
  c->launches += it->second.launches * n;
}

}  // namespace

// Greedy decoding of every encoded image under R pt prompts each: B x R point sequences, sequence b * R + r being prompt r
// of image b.  Text spotting (transformer.py:234-286) and KIE (:143-217) share the pt loop and the batched poly / rec
// loops; they differ in the pt step pattern (x, y[, class]), in which decoded tokens form (x, y) instances and in the
// number of logits entering the poly / rec softmax.  Outputs are per sequence; the poly / rec loops run per image over the
// instances of all its prompts, concatenated in prompt order, so the K_c / V_c stream of an image serves every prompt.
void omni_decode_impl(Ctx* c, const int64_t* prompts, int R, int n_prompt, const alm_decode_cfg& cfg, bool kie,
                      int32_t* n_tok_out, int64_t* pt_tok_out, float* pt_prob_out, int32_t* n_inst, int32_t* inst_pos,
                      int64_t* pt, int64_t* poly, int64_t* rec, float* rec_prob, bool points_only = false) {
  OmniModel* m = c->omni;
  ALM_REQUIRE(m && m->encoded, ALM_ERR_STATE, "alm_omni_decode before alm_omni_encode");
  ALM_REQUIRE(c->xattn_impl != 1 || m->vt_hi, ALM_ERR_STATE, "xattn_impl 1 must be set before alm_omni_encode");
  ALM_REQUIRE(n_prompt >= 1 && n_prompt <= 16, ALM_ERR_INVALID, "pt prompt length");
  ALM_REQUIRE(R >= 1 && R <= 16, ALM_ERR_INVALID, "prompts per image must be 1..16");
  ALM_REQUIRE(cfg.pt_seq_length >= 1, ALM_ERR_INVALID, "pt_seq_length");
  // The reference default is --pt_seq_length 1024 (utils/parser.py:21) with a 5- or 7-token prompt: more steps than the
  // 1024-row position table (transformer.py:475) can serve.  It works because EOS ends the loop (:126) long before
  // step 1025 - n_prompt, where the embedding lookup (:312) would raise.  Same here: the loop is sized by the table,
  // and a sequence that is still alive when the table is exhausted is an error, as in the reference.
  const int pt_steps = std::min(cfg.pt_seq_length, 1025 - n_prompt);
  const bool pt_clamped = pt_steps < cfg.pt_seq_length;
  ALM_REQUIRE(cfg.vie_categories == m->vie, ALM_ERR_INVALID, "vie_categories does not match the loaded checkpoint");
  ALM_REQUIRE(kie == (m->vie > 0), ALM_ERR_INVALID, "use alm_omni_decode for text spotting and alm_omni_decode_kie for KIE");
  ALM_REQUIRE(m->kv_decoders == 3 || points_only, ALM_ERR_STATE,
              "the batch was encoded with kv_decoders < 3: only alm_omni_decode_points can run on it");
  ALM_REQUIRE(points_only || cfg.max_instances >= (pt_steps / 2), ALM_ERR_INVALID, "max_instances < pt_seq_length / 2");
  ALM_REQUIRE(points_only || cfg.poly_length == 32, ALM_ERR_UNSUPPORTED, "polygon length is fixed at 32 (transformer.py:254)");
  const int B = m->B;
  const int SP = B * R;  // point sequences
  Arena& ws = c->ws;
  ws.release(m->ws_mark);
  HeadCfg hc{cfg.num_bins, cfg.pt_eos, cfg.rec_eos, cfg.recog_pad, m->vie};
  c->timing_valid[1] = false;
  // The decode loops optionally run on internal high-priority streams (fork from / join to the caller's stream)
  struct DecodeScope {
    Ctx* c;
    cudaStream_t user;
    bool swapped;
    ~DecodeScope() {
      c->gemm_grid_cap = 0;
      if (swapped) {
        cudaStream_t hi = c->stream;
        c->stream = user;
        if (cudaEventRecord(c->ev_prio, hi) == cudaSuccess) cudaStreamWaitEvent(user, c->ev_prio, 0);
      }
    }
  } scope{c, c->stream, false};
  c->gemm_grid_cap = c->dec_grid_cap;
  if (c->decode_priority) {
    int least = 0, greatest = 0;
    ALM_CHECK_CUDA(cudaDeviceGetStreamPriorityRange(&least, &greatest));
    if (!c->stream_hi) {
      ALM_CHECK_CUDA(cudaStreamCreateWithPriority(&c->stream_hi, cudaStreamNonBlocking, greatest));
      ALM_CHECK_CUDA(cudaEventCreateWithFlags(&c->ev_prio, cudaEventDisableTiming));
    }
    if (!c->stream2) ALM_CHECK_CUDA(cudaStreamCreateWithPriority(&c->stream2, cudaStreamNonBlocking, greatest));
    ALM_CHECK_CUDA(cudaEventRecord(c->ev_prio, c->stream));
    ALM_CHECK_CUDA(cudaStreamWaitEvent(c->stream_hi, c->ev_prio, 0));
    c->stream = c->stream_hi;
    scope.swapped = true;
  }
  ALM_CHECK_CUDA(cudaEventRecord(c->ev_t[2], c->stream));

  // ------------------------------------------------------------------ pt loop (transformer.py:102-141)
  // One prompt length for all sequences: the single device position counter and query position serve every row.
  const int Tpt = n_prompt + pt_steps;
  int* pt_tok = ws.get<int>(static_cast<size_t>(SP) * Tpt);
  float* pt_prob = ws.get<float>(static_cast<size_t>(SP) * pt_steps);
  int* finished = ws.get<int>(SP);
  int* ntok = ws.get<int>(SP);
  {
    std::vector<int> h(static_cast<size_t>(SP) * Tpt, 0);
    for (int s = 0; s < SP; ++s)
      for (int i = 0; i < n_prompt; ++i)
        h[static_cast<size_t>(s) * Tpt + i] = static_cast<int>(prompts[static_cast<size_t>(s) * n_prompt + i]);
    ALM_CHECK_CUDA(cudaMemcpyAsync(pt_tok, h.data(), h.size() * sizeof(int), cudaMemcpyHostToDevice, c->stream));
    wait_stream(c, c->stream);  // h goes out of scope (this also waits for the encoder)
  }
  fill_i32(c, finished, SP, 0);
  fill_i32(c, ntok, SP, 0);
  const size_t after_pt_tokens = ws.mark();
  {
    DecodeBufs u = alloc_decode(c, m, B, R, Tpt - 1, true);
    fill_i32(c, u.tpos, 1, 0);
    HeadArgs off;
    run_steps(c, m, 0, u, pt_tok, Tpt, 0, B, n_prompt - 1, off);  // prompt tokens only fill the caches
    HeadArgs h;
    h.on = true; h.cfg = hc; h.tokens = pt_tok; h.tstride = Tpt; h.n_prompt_m1 = n_prompt - 1;
    h.probs = pt_prob; h.pstride = pt_steps;
    h.finished = finished; h.ntok = ntok;
    std::vector<int> fin(SP);
    bool all_done = false;
    for (int done = 0; done < pt_steps && !all_done;) {
      const int chunk = std::min(16, pt_steps - done);
      run_steps(c, m, 0, u, pt_tok, Tpt, 0, B, chunk, h);
      done += chunk;
      if (done < pt_steps || pt_clamped) {  // every sequence hit EOS?  (one small sync per 16 tokens)
        wait_stream(c, c->stream);
        ALM_CHECK_CUDA(cudaMemcpyAsync(fin.data(), finished, SP * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
        ALM_CHECK_CUDA(cudaStreamSynchronize(c->stream));
        all_done = std::all_of(fin.begin(), fin.end(), [](int v) { return v != 0; });
      }
    }
    ALM_REQUIRE(!pt_clamped || all_done, ALM_ERR_INVALID,
                "a point sequence produced no EOS within the 1024-row position table (the reference raises at "
                "transformer.py:312)");
  }
  ALM_CHECK_CUDA(cudaEventRecord(c->ev_t[3], c->stream));
  wait_stream(c, c->stream);
  std::vector<int> h_ntok(SP), h_tok(static_cast<size_t>(SP) * Tpt);
  std::vector<float> h_prob(static_cast<size_t>(SP) * pt_steps);
  ALM_CHECK_CUDA(cudaMemcpyAsync(h_ntok.data(), ntok, SP * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
  ALM_CHECK_CUDA(cudaMemcpyAsync(h_tok.data(), pt_tok, h_tok.size() * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
  ALM_CHECK_CUDA(cudaMemcpyAsync(h_prob.data(), pt_prob, h_prob.size() * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
  ALM_CHECK_CUDA(cudaStreamSynchronize(c->stream));
  const int maxI = cfg.max_instances;
  // which decoded tokens form (x, y) instances, per sequence
  std::vector<std::vector<int>> starts(SP);
  for (int s = 0; s < SP; ++s) {
    int len = h_ntok[s];
    if (len % 2) --len;  // transformer.py:138-139 (applied in both modes by the reference)
    const int* t = &h_tok[static_cast<size_t>(s) * Tpt + n_prompt];
    if (points_only) {  // the raw point sequence is the result (decode_pt_seq alone, transformer.py:102-141)
      n_tok_out[s] = len;
      for (int i = 0; i < len; ++i) {
        pt_tok_out[static_cast<size_t>(s) * cfg.pt_seq_length + i] = t[i];
        if (pt_prob_out) pt_prob_out[static_cast<size_t>(s) * cfg.pt_seq_length + i] = h_prob[static_cast<size_t>(s) * pt_steps + i];
      }
      continue;
    }
    if (!kie) {
      for (int i = 0; i + 1 < len; i += 2) starts[s].push_back(i);
    } else {
      for (int i = 0; i < len;) {  // the walk of decode_vie_pt_poly_rec_seq (transformer.py:148-215)
        if (t[i] < cfg.num_bins && i + 1 <= len - 1 && t[i + 1] < cfg.num_bins) { starts[s].push_back(i); i += 2; }
        else ++i;
      }
      if (n_tok_out) n_tok_out[s] = len;
      for (int i = 0; i < len; ++i) {
        pt_tok_out[static_cast<size_t>(s) * cfg.pt_seq_length + i] = t[i];
        pt_prob_out[static_cast<size_t>(s) * cfg.pt_seq_length + i] = h_prob[static_cast<size_t>(s) * pt_steps + i];
      }
    }
    n_inst[s] = static_cast<int>(starts[s].size());
    ALM_REQUIRE(n_inst[s] <= maxI, ALM_ERR_INVALID, "decoded more points than max_instances");
    for (int n = 0; n < n_inst[s]; ++n) {
      if (inst_pos) inst_pos[static_cast<size_t>(s) * maxI + n] = starts[s][n];
      if (pt) {
        pt[(static_cast<size_t>(s) * maxI + n) * 2] = t[starts[s][n]];
        pt[(static_cast<size_t>(s) * maxI + n) * 2 + 1] = t[starts[s][n] + 1];
      }
    }
  }
  if (points_only) {
    c->timing_valid[1] = true;
    ALM_CHECK_CUDA(cudaEventRecord(c->ev_t[4], c->stream));
    ws.release(m->ws_mark);
    return;
  }
  // the instances of image b: (sequence, instance) pairs of its prompts 0..R-1, in prompt order
  std::vector<std::vector<std::pair<int, int>>> inst(B);
  int Ncap = 0;
  for (int b = 0; b < B; ++b) {
    for (int r = 0; r < R; ++r)
      for (int n = 0; n < n_inst[b * R + r]; ++n) inst[b].emplace_back(b * R + r, n);
    Ncap = std::max(Ncap, static_cast<int>(inst[b].size()));
  }
  if (Ncap == 0) return;

  // ------------------------------------------------------------------ poly / rec loops (:249-284 ; :153-185 for KIE)
  // The two loops only depend on the decoded points, not on each other: they run concurrently on two streams
  // (their per-token kernels are far too small to fill 148 SMs one at a time).
  if (!c->stream2) ALM_CHECK_CUDA(cudaStreamCreateWithFlags(&c->stream2, cudaStreamNonBlocking));
  if (!c->ev_fork) {
    ALM_CHECK_CUDA(cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming));
    ALM_CHECK_CUDA(cudaEventCreateWithFlags(&c->ev_join, cudaEventDisableTiming));
  }
  cudaStream_t s0 = c->stream, s1 = c->decode_streams == 2 ? c->stream2 : c->stream;
  ws.release(after_pt_tokens);
  const int S = B * Ncap;
  int* toks[3] = {nullptr, nullptr, nullptr};
  float* prbs[3] = {nullptr, nullptr, nullptr};
  std::vector<int> h_prompt[3];
  for (int phase = 1; phase <= 2; ++phase) {  // [x, y, sos] per instance (transformer.py:252,268 ; :153,172); dead slots 0,0,sos
    const int T = 3 + (phase == 1 ? cfg.poly_length : cfg.rec_length);
    h_prompt[phase].assign(static_cast<size_t>(S) * T, 0);
    for (int b = 0; b < B; ++b)
      for (int n = 0; n < Ncap; ++n) {
        int* row = &h_prompt[phase][(static_cast<size_t>(b) * Ncap + n) * T];
        if (n < static_cast<int>(inst[b].size())) {
          const int sq = inst[b][n].first;
          const int* t = &h_tok[static_cast<size_t>(sq) * Tpt + n_prompt + starts[sq][inst[b][n].second]];
          row[0] = t[0]; row[1] = t[1];
        }
        row[2] = phase == 1 ? cfg.poly_sos : cfg.rec_sos;
      }
    toks[phase] = ws.get<int>(static_cast<size_t>(S) * T);
    prbs[phase] = ws.get<float>(static_cast<size_t>(S) * (T - 3));
    ALM_CHECK_CUDA(cudaMemcpyAsync(toks[phase], h_prompt[phase].data(), h_prompt[phase].size() * sizeof(int),
                                   cudaMemcpyHostToDevice, s0));
  }
  ALM_CHECK_CUDA(cudaEventRecord(c->ev_fork, s0));
  ALM_CHECK_CUDA(cudaStreamWaitEvent(s1, c->ev_fork, 0));
  try {
    for (int phase = 1; phase <= 2; ++phase) {
      c->stream = (phase == 1) ? s0 : s1;
      const int len = phase == 1 ? cfg.poly_length : cfg.rec_length;
      const int T = 3 + len;
      DecodeBufs u = alloc_decode(c, m, B, Ncap, T - 1);
      fill_i32(c, u.tpos, 1, 0);
      HeadArgs off;
      run_steps(c, m, phase, u, toks[phase], T, 0, B, 2, off);
      HeadArgs h;
      h.on = true; h.cfg = hc; h.tokens = toks[phase]; h.tstride = T; h.n_prompt_m1 = 2; h.probs = prbs[phase];
      h.pstride = len;
      h.nsoft = m->V - m->vie;  // logits[:, -1, :-vie_categories] (transformer.py:156,176)
      run_steps(c, m, phase, u, toks[phase], T, 0, B, len, h);
    }
  } catch (...) {
    c->stream = s0;
    cudaStreamSynchronize(s1);
    throw;
  }
  c->stream = s0;
  ALM_CHECK_CUDA(cudaEventRecord(c->ev_join, s1));
  ALM_CHECK_CUDA(cudaStreamWaitEvent(s0, c->ev_join, 0));
  ALM_CHECK_CUDA(cudaEventRecord(c->ev_t[4], s0));
  c->timing_valid[1] = true;
  wait_stream(c, c->stream);
  for (int phase = 1; phase <= 2; ++phase) {
    const int len = phase == 1 ? cfg.poly_length : cfg.rec_length;
    const int T = 3 + len;
    std::vector<int> hh(static_cast<size_t>(S) * T);
    std::vector<float> hp(static_cast<size_t>(S) * len);
    ALM_CHECK_CUDA(cudaMemcpyAsync(hh.data(), toks[phase], hh.size() * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    ALM_CHECK_CUDA(cudaMemcpyAsync(hp.data(), prbs[phase], hp.size() * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
    ALM_CHECK_CUDA(cudaStreamSynchronize(c->stream));
    for (int b = 0; b < B; ++b)
      for (int j = 0; j < static_cast<int>(inst[b].size()); ++j) {  // scattered back per (image, prompt)
        const size_t sq = static_cast<size_t>(b) * Ncap + j;
        const size_t dst = static_cast<size_t>(inst[b][j].first) * maxI + inst[b][j].second;
        for (int k = 0; k < len; ++k) {
          const size_t o = dst * len + k;
          if (phase == 1) poly[o] = hh[sq * T + 3 + k];
          else { rec[o] = hh[sq * T + 3 + k]; rec_prob[o] = hp[sq * len + k]; }
        }
      }
  }
  ws.release(m->ws_mark);
}

namespace {
// the single prompt of the classic entry points, broadcast to every encoded image
std::vector<int64_t> broadcast_prompt(Ctx* c, const int64_t* pt_prompt, int n_prompt) {
  ALM_REQUIRE(c->omni && c->omni->encoded, ALM_ERR_STATE, "alm_omni_decode before alm_omni_encode");
  ALM_REQUIRE(n_prompt >= 1 && n_prompt <= 16, ALM_ERR_INVALID, "pt prompt length");
  std::vector<int64_t> p(static_cast<size_t>(c->omni->B) * n_prompt);
  for (size_t i = 0; i < p.size(); ++i) p[i] = pt_prompt[i % n_prompt];
  return p;
}

// caller-supplied prompts [B][R][n_prompt] of the prompted entry points: every id is an embedding row
void check_prompts(Ctx* c, const int64_t* prompts, int R, int n_prompt) {
  OmniModel* m = c->omni;
  ALM_REQUIRE(m && m->encoded, ALM_ERR_STATE, "alm_omni_decode_prompted before alm_omni_encode");
  ALM_REQUIRE(m->vie == 0, ALM_ERR_UNSUPPORTED, "window-prompted decoding is text spotting only (not KIE checkpoints)");
  ALM_REQUIRE(R >= 1 && R <= 16, ALM_ERR_INVALID, "prompts per image must be 1..16");
  ALM_REQUIRE(n_prompt >= 1 && n_prompt <= 16, ALM_ERR_INVALID, "pt prompt length");
  const size_t n = static_cast<size_t>(m->B) * R * n_prompt;
  for (size_t i = 0; i < n; ++i)
    ALM_REQUIRE(prompts[i] >= 0 && prompts[i] < m->V, ALM_ERR_INVALID, "prompt token id out of range [0, V)");
}
}  // namespace

void omni_decode(Ctx* c, const int64_t* pt_prompt, int n_prompt, const alm_decode_cfg& cfg, int32_t* n_inst,
                 int64_t* pt, int64_t* poly, int64_t* rec, float* rec_prob) {
  const std::vector<int64_t> p = broadcast_prompt(c, pt_prompt, n_prompt);
  omni_decode_impl(c, p.data(), 1, n_prompt, cfg, false, nullptr, nullptr, nullptr, n_inst, nullptr, pt, poly, rec, rec_prob);
}

void omni_decode_kie(Ctx* c, const int64_t* pt_prompt, int n_prompt, const alm_decode_cfg& cfg, int32_t* n_tok,
                     int64_t* pt_tokens, float* pt_probs, int32_t* n_inst, int32_t* inst_pos, int64_t* poly,
                     int64_t* rec, float* rec_prob) {
  const std::vector<int64_t> p = broadcast_prompt(c, pt_prompt, n_prompt);
  omni_decode_impl(c, p.data(), 1, n_prompt, cfg, true, n_tok, pt_tokens, pt_probs, n_inst, inst_pos, nullptr, poly, rec,
                   rec_prob);
}

void omni_decode_points(Ctx* c, const int64_t* pt_prompt, int n_prompt, const alm_decode_cfg& cfg, int32_t* n_tok,
                        int64_t* pt_tokens, float* pt_probs) {
  const std::vector<int64_t> p = broadcast_prompt(c, pt_prompt, n_prompt);
  omni_decode_impl(c, p.data(), 1, n_prompt, cfg, c->omni->vie > 0, n_tok, pt_tokens, pt_probs, nullptr, nullptr,
                   nullptr, nullptr, nullptr, nullptr, true);
}

void omni_decode_prompted(Ctx* c, const int64_t* prompts, int R, int n_prompt, const alm_decode_cfg& cfg,
                          int32_t* n_inst, int64_t* pt, int64_t* poly, int64_t* rec, float* rec_prob) {
  check_prompts(c, prompts, R, n_prompt);
  omni_decode_impl(c, prompts, R, n_prompt, cfg, false, nullptr, nullptr, nullptr, n_inst, nullptr, pt, poly, rec, rec_prob);
}

void omni_decode_points_prompted(Ctx* c, const int64_t* prompts, int R, int n_prompt, const alm_decode_cfg& cfg,
                                 int32_t* n_tok, int64_t* pt_tokens, float* pt_probs) {
  check_prompts(c, prompts, R, n_prompt);
  omni_decode_impl(c, prompts, R, n_prompt, cfg, false, n_tok, pt_tokens, pt_probs, nullptr, nullptr, nullptr, nullptr,
                   nullptr, nullptr, true);
}

// Teacher-forced logits for one image: every position of every sequence (Transformer.decode, :74-100).
void omni_decode_logits(Ctx* c, int image, int kind, const int64_t* seq, int n_seq, int len, float* logits) {
  OmniModel* m = c->omni;
  ALM_REQUIRE(m && m->encoded, ALM_ERR_STATE, "alm_omni_decode_logits before alm_omni_encode");
  ALM_REQUIRE(c->xattn_impl != 1 || m->vt_hi, ALM_ERR_STATE, "xattn_impl 1 must be set before alm_omni_encode");
  ALM_REQUIRE(image >= 0 && image < m->B && kind >= 0 && kind < 3 && n_seq > 0 && len > 0 && len <= 1024,
              ALM_ERR_INVALID, "decode_logits arguments");
  ALM_REQUIRE(kind < m->kv_decoders, ALM_ERR_STATE, "the batch was encoded without this decoder's K/V cache (kv_decoders)");
  Arena& ws = c->ws;
  ws.release(m->ws_mark);
  std::vector<int> h(static_cast<size_t>(n_seq) * len);
  for (size_t i = 0; i < h.size(); ++i) {
    ALM_REQUIRE(seq[i] >= 0 && seq[i] < m->V, ALM_ERR_INVALID, "token id out of range");
    h[i] = static_cast<int>(seq[i]);
  }
  int* tok = ws.get<int>(h.size());
  ALM_CHECK_CUDA(cudaMemcpyAsync(tok, h.data(), h.size() * sizeof(int), cudaMemcpyHostToDevice, c->stream));
  DecodeBufs u = alloc_decode(c, m, 1, n_seq, len);
  fill_i32(c, u.tpos, 1, 0);
  for (int t = 0; t < len; ++t) {
    decoder_step(c, m, kind, u, tok, len, image, 1, true);
    add_i32(c, u.tpos, 1);
    // logits [n_seq, len, V] <- step t rows
    ALM_CHECK_CUDA(cudaMemcpy2DAsync(logits + static_cast<size_t>(t) * m->V, static_cast<size_t>(len) * m->V * sizeof(float),
                                     u.logits, static_cast<size_t>(m->V) * sizeof(float), static_cast<size_t>(m->V) * sizeof(float),
                                     n_seq, cudaMemcpyDeviceToHost, c->stream));
  }
  ALM_CHECK_CUDA(cudaStreamSynchronize(c->stream));
  ws.release(m->ws_mark);
}

}  // namespace alm
