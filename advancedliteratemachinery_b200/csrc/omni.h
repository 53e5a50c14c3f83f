// OmniParser model state (weights + per-batch encode/decode buffers) and kernel wrappers.
#pragma once
#include "alm_internal.h"

namespace alm {

struct HeadCfg {
  int num_bins, pt_eos, rec_eos, recog_pad, vie;
};

struct LNW {
  float* g = nullptr;
  float* b = nullptr;
};
struct Lin {
  SplitW w;
  float* b = nullptr;
  float* wf = nullptr;  // exact fp32 [N,K] copy (decoder weights only): the skinny M <= 64 decode path
};

struct SwinBlockW {
  LNW n1, n2;
  Lin qkv, proj, fc1, fc2;
  float* bias_dense = nullptr;  // [heads,49,49] = table[index]  (swin_transformer.py:133-135)
};
struct SwinStageW {
  std::vector<SwinBlockW> blocks;
  LNW out_norm;   // norm{s}
  LNW merge_norm;  // downsample.norm
  SplitW merge_red;
};
struct DecLayerW {
  LNW n1, n2, n3;
  Lin sa_qk;   // rows [0,1024) of self_attn.in_proj (q then k)
  Lin sa_v;    // rows [1024,1536)
  float* sa_qkv_f = nullptr;  // exact fp32 packed in_proj [1536,512] + bias [1536] (skinny decode path)
  float* sa_qkv_b = nullptr;
  Lin sa_out;
  Lin ca_q;    // rows [0,512) of multihead_attn.in_proj
  Lin ca_out;
  Lin l1, l2;
};

struct OmniModel {
  int V = 0;
  int vie = 0;
  Lin patch;
  LNW patch_norm;
  SwinStageW stage[4];
  SplitW fpn[4];  // fpn_in[0..3] : c5,c4,c3,c2
  Lin inproj;
  float* dim_t = nullptr;  // [256]
  // decoder
  float* word_emb = nullptr;
  float* pos_emb[3] = {nullptr, nullptr, nullptr};  // pt, poly, rec
  LNW emb_norm;
  DecLayerW dec[3][4];
  LNW dec_norm[3];
  Lin ca_k_all;  // [12*512, 512]  rows (d*4+l)*512..: cross-attn K projections of all decoder layers
  Lin ca_v_all;  // [12*512, 512]
  Lin head[3][3];

  // ---- state of the last alm_omni_encode -------------------------------------------------------
  bool encoded = false;
  int kv_decoders = 3;  // decoders whose K/V caches the last encode filled
  int B = 0, H = 0, W = 0;
  int Hs[4] = {0, 0, 0, 0}, Ws[4] = {0, 0, 0, 0};
  int mh = 0, mw = 0, M = 0, Mpad = 0;
  float* feat[4] = {nullptr, nullptr, nullptr, nullptr};  // LN'd stage outputs, NHWC fp32
  float* memory = nullptr;                                // [B*M,512]
  float* pos = nullptr;                                   // [B*M,512]
  uint8_t* kpm = nullptr;                                 // [B*M]
  bf16 *kc_hi = nullptr, *kc_lo = nullptr;                // [B, 12 (dec,layer), 8 heads, M, 64]
  bf16 *vc_hi = nullptr, *vc_lo = nullptr;                // [B, 12 (dec,layer), 8 heads, M, 64]
  bf16 *vt_hi = nullptr, *vt_lo = nullptr;                // [B, 6144, Mpad] (only for the unfused debug path, xattn_impl 1)
  size_t ws_mark = 0;                                     // arena offset after the encode-persistent buffers
  // captured decode-step graphs, keyed by everything that determines the launch sequence and its pointers
  struct StepGraph { cudaGraphExec_t exec; long launches; };
  std::map<std::vector<long>, StepGraph> step_graphs;
  ~OmniModel() {
    for (auto& kv : step_graphs) cudaGraphExecDestroy(kv.second.exec);
  }
};

void omni_load(Ctx* c, int kind, const std::map<std::string, HostTensor>& t);
// a second execution context over the same device weights: weight pointers copied, per-batch state fresh
OmniModel* omni_share(const OmniModel* owner);
void omni_encode(Ctx* c, const float* img_dev, const uint8_t* mask_dev, int B, int H, int W);
void omni_decode(Ctx* c, const int64_t* pt_prompt, int n_prompt, const alm_decode_cfg& cfg, int32_t* n_inst,
                 int64_t* pt, int64_t* poly, int64_t* rec, float* rec_prob);
void omni_decode_kie(Ctx* c, const int64_t* pt_prompt, int n_prompt, const alm_decode_cfg& cfg, int32_t* n_tok,
                     int64_t* pt_tokens, float* pt_probs, int32_t* n_inst, int32_t* inst_pos, int64_t* poly,
                     int64_t* rec, float* rec_prob);
void omni_decode_points(Ctx* c, const int64_t* pt_prompt, int n_prompt, const alm_decode_cfg& cfg, int32_t* n_tok,
                        int64_t* pt_tokens, float* pt_probs);
// R window prompts per image, prompts int64 [B][R][n_prompt] (text spotting): outputs per (image, prompt)
void omni_decode_prompted(Ctx* c, const int64_t* prompts, int R, int n_prompt, const alm_decode_cfg& cfg,
                          int32_t* n_inst, int64_t* pt, int64_t* poly, int64_t* rec, float* rec_prob);
void omni_decode_points_prompted(Ctx* c, const int64_t* prompts, int R, int n_prompt, const alm_decode_cfg& cfg,
                                 int32_t* n_tok, int64_t* pt_tokens, float* pt_probs);
void omni_decode_logits(Ctx* c, int image, int kind, const int64_t* seq, int n_seq, int len, float* logits);

// kernels (omni_kernels.cu)
void window_map(Ctx* c, int* map, int B, int H, int W, int nWh, int nWw, int shift);
void merge_map(Ctx* c, int* map, int B, int H, int W, int H2, int W2);
void nearest_map(Ctx* c, int* map, int B, int Hd, int Wd, int Hs, int Ws);
void fpn_assemble(Ctx* c, const float* p2, const float* p3, const float* p4, const float* p5, int B, const int* Hs,
                  const int* Ws, int Ho, int Wo, bf16* hi, bf16* lo);
void sine_pos(Ctx* c, const uint8_t* mask, int B, int H, int W, int h, int w, const float* dim_t, float* pos,
              uint8_t* kpm, float* scratch);
void embed_ln(Ctx* c, const int* tokens, int tstride, const int* tptr, int S, const float* word_emb,
              const float* pos_emb, const float* gamma, const float* beta, float* x, float* qpos);
void self_attn_step(Ctx* c, const float* qk, const float* vnew, float* kc, float* vc, int S, const int* tptr, int Tmax,
                    bf16* out_hi, bf16* out_lo, float* out_f32 = nullptr, int ld_qk = 1024, int ld_v = 512);
void head_select(Ctx* c, const float* logits, int S, int V, int nsoft, int phase, const HeadCfg& cfg, int* tokens,
                 int tstride, const int* tptr, int n_prompt_m1, float* probs, int pstride, int* finished, int* ntok);
void cross_attn_q1(Ctx* c, const float* q, const bf16* kc_hi, const bf16* kc_lo, const bf16* vt_hi, const bf16* vt_lo,
                   const uint8_t* kpm, int nimg, int M, int Mpad, float* partial, int* counters, int nsplit,
                   bf16* out_hi, bf16* out_lo, float* out_f32 = nullptr);
int cross_attn_q1_splits(Ctx* c, int nimg, int M);
// fused multi-query cross-attention (xattn.cu): Ncap query rows per image against the cached K_c / V_c^T
void cross_attn_mq_plan(Ctx* c, int nimg, int Ncap, int M, int* grid, int* max_parts, int* pairs);
size_t cross_attn_mq_partial_floats(int pairs, int max_parts);
void cross_attn_mq(Ctx* c, const bf16* q_hi, const bf16* q_lo, const float* q_f32, int nimg, int Ncap, const bf16* kc_hi,
                   const bf16* kc_lo, const bf16* vc_hi, const bf16* vc_lo, const uint8_t* kpm, int M,
                   int grid, int max_parts, float* partial, int* counters, bf16* out_hi, bf16* out_lo,
                   float* out_f32);
// experimental TMA + mbarrier variant (xattn_tma.cu, "xattn_impl" 2)
void cross_attn_tma_plan(Ctx* c, int nimg, int Ncap, int M, int* grid, int* max_parts, int* pairs);
void cross_attn_tma(Ctx* c, const bf16* q_hi, const bf16* q_lo, const float* q_f32, int nimg, int Ncap, const bf16* kc_hi,
                    const bf16* kc_lo, const bf16* vc_hi, const bf16* vc_lo, long slices, int z0, const uint8_t* kpm, int M,
                    int grid, int max_parts, float* partial, int* counters, bf16* out_hi, bf16* out_lo, float* out_f32);
// tcgen05 + TMA-ring variant (xattn_tc.cu, "xattn_impl" 3): 128-key blocks, S / P in tensor memory, one CTA per SM
void cross_attn_tc_plan(Ctx* c, int nimg, int Ncap, int M, int* grid, int* max_parts, int* pairs);
void cross_attn_tc(Ctx* c, const bf16* q_hi, const bf16* q_lo, const float* q_f32, int nimg, int Ncap, const bf16* kc_hi,
                   const bf16* kc_lo, const bf16* vc_hi, const bf16* vc_lo, long slices, int z0, const uint8_t* kpm, int M,
                   int grid, int max_parts, float* partial, int* counters, bf16* out_hi, bf16* out_lo, float* out_f32);
void add_i32(Ctx* c, int* p, int v);
void build_inst_prompts(Ctx* c, const int* pt_tokens, int pt_stride, int n_prompt, const int* ntok, int B, int Ncap,
                        int sos, int* tokens, int tstride);
void fill_i32(Ctx* c, int* p, long n, int v);

}  // namespace alm
