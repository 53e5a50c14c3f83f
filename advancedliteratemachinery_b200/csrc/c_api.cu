// extern "C" surface of libalm_ocr.so (include/alm_ocr.h).  Nothing throws across this boundary.
#include <string.h>

#include <algorithm>

#include "alm_internal.h"
#include "mgp.h"
#include "omni.h"
#include "pre.h"
#include "ptx.cuh"

using namespace alm;


struct alm_ctx {
  Ctx c;
  void* dev_in = nullptr;  // staging for host-resident inputs
  size_t dev_in_bytes = 0;
  void* dev_mask = nullptr;
  size_t dev_mask_bytes = 0;
};

namespace {

template <class F>
int guarded(alm_ctx* h, F&& f) {
  if (!h) return ALM_ERR_INVALID;
  try {
    cudaSetDevice(h->c.device);
    f();
    h->c.err.clear();
    return ALM_OK;
  } catch (const AlmError& e) {
    h->c.err = e.msg;
    return e.code;
  } catch (const std::exception& e) {
    h->c.err = std::string("exception: ") + e.what();
    return ALM_ERR_INVALID;
  } catch (...) {
    h->c.err = "unknown exception";
    return ALM_ERR_INVALID;
  }
}

bool is_device_ptr(const void* p) {
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
    cudaGetLastError();
    return false;
  }
  return a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged;
}

// returns a device pointer for `p` (host buffers are copied into the context's staging slab on the stream)
const void* stage_input(alm_ctx* h, const void* p, size_t bytes, void** slab, size_t* slab_bytes) {
  if (p == nullptr) return nullptr;
  if (is_device_ptr(p)) return p;
  if (*slab_bytes < bytes) {
    if (*slab) cudaFree(*slab);
    *slab = nullptr;
    *slab_bytes = 0;
    if (cudaMalloc(slab, bytes) != cudaSuccess) throw AlmError{ALM_ERR_OOM, "cudaMalloc of the input staging buffer failed"};
    *slab_bytes = bytes;
  }
  ALM_CHECK_CUDA(cudaMemcpyAsync(*slab, p, bytes, cudaMemcpyHostToDevice, h->c.stream));
  return *slab;
}

void d2h(Ctx* c, void* dst, const void* src, size_t bytes) {
  ALM_CHECK_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, c->stream));
}

float bf16_bits_to_f32(uint16_t v) {
  uint32_t u = static_cast<uint32_t>(v) << 16;
  float f;
  memcpy(&f, &u, 4);
  return f;
}
float f16_bits_to_f32(uint16_t v) {
  const uint32_t s = (v >> 15) & 1, e = (v >> 10) & 31, m = v & 1023;
  uint32_t u;
  if (e == 0) {
    if (m == 0) u = s << 31;
    else {
      int ee = -1;
      uint32_t mm = m;
      do { ++ee; mm <<= 1; } while ((mm & 1024) == 0);
      u = (s << 31) | ((127 - 15 - ee) << 23) | ((mm & 1023) << 13);
    }
  } else if (e == 31) u = (s << 31) | 0x7f800000u | (m << 13);
  else u = (s << 31) | ((e - 15 + 127) << 23) | (m << 13);
  float f;
  memcpy(&f, &u, 4);
  return f;
}

}  // namespace

extern "C" {

const char* alm_version(void) { return "alm_ocr 0.1 (sm_100a, tcgen05)"; }

int alm_init(int device, void* stream, alm_ctx** out) {
  if (!out) return ALM_ERR_INVALID;
  *out = nullptr;
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || device < 0 || device >= n) {
    cudaGetLastError();
    return ALM_ERR_CUDA;  // no CUDA device: the library has no CPU fallback
  }
  alm_ctx* h = new alm_ctx();
  h->c.device = device;
  int rc = guarded(h, [&] {
    ALM_CHECK_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    ALM_CHECK_CUDA(cudaGetDeviceProperties(&prop, device));
    ALM_REQUIRE(prop.major == 10, ALM_ERR_UNSUPPORTED,
                "libalm_ocr is built for sm_100a only; device is sm_" + std::to_string(prop.major) + std::to_string(prop.minor));
    h->c.num_sms = prop.multiProcessorCount;
    if (stream) h->c.stream = static_cast<cudaStream_t>(stream);
    else {
      ALM_CHECK_CUDA(cudaStreamCreateWithFlags(&h->c.stream, cudaStreamNonBlocking));
      h->c.own_stream = true;
    }
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult q;
    ALM_CHECK_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q));
    ALM_REQUIRE(fn != nullptr && q == cudaDriverEntryPointSuccess, ALM_ERR_CUDA, "cuTensorMapEncodeTiled not available");
    h->c.encode = reinterpret_cast<PFN_encodeTiled>(fn);
  });
  if (rc != ALM_OK) {
    delete h;
    return rc;
  }
  *out = h;
  return ALM_OK;
}

void alm_free(alm_ctx* h) {
  if (!h) return;
  cudaSetDevice(h->c.device);
  cudaStreamSynchronize(h->c.stream);
  delete h->c.omni;
  mgp_free(h->c.mgp);
  comm_release(&h->c);
  if (h->c.gather_buf) cudaFree(h->c.gather_buf);
  h->c.wstore.reset();  // frees the slabs when this was the last context using them
  if (h->c.ws.base) cudaFree(h->c.ws.base);
  if (h->dev_in) cudaFree(h->dev_in);
  if (h->dev_mask) cudaFree(h->dev_mask);
  if (h->c.stream2) cudaStreamDestroy(h->c.stream2);
  if (h->c.stream_hi) cudaStreamDestroy(h->c.stream_hi);
  if (h->c.ev_prio) cudaEventDestroy(h->c.ev_prio);
  if (h->c.ev_block) cudaEventDestroy(h->c.ev_block);
  if (h->c.ev_order) cudaEventDestroy(h->c.ev_order);
  if (h->c.ev_fork) { cudaEventDestroy(h->c.ev_fork); cudaEventDestroy(h->c.ev_join); }
  for (auto e : h->c.ev_t) if (e) cudaEventDestroy(e);
  if (h->c.own_stream) cudaStreamDestroy(h->c.stream);
  delete h;
}

const char* alm_last_error(const alm_ctx* h) { return h ? h->c.err.c_str() : "null context"; }

int alm_set_option(alm_ctx* h, const char* key, long value) {
  return guarded(h, [&] {
    const std::string k = key ? key : "";
    if (k == "nsplit") {
      ALM_REQUIRE(value == 1 || value == 3, ALM_ERR_INVALID, "nsplit must be 1 or 3");
      h->c.nsplit = static_cast<int>(value);
    } else if (k == "gemm_impl") {
      ALM_REQUIRE(value == 0 || value == 1, ALM_ERR_INVALID, "gemm_impl must be 0 or 1");
      h->c.gemm_impl = static_cast<int>(value);
    } else if (k == "trace_gemm") {
      if (h->c.trace_buf) { cudaFree(h->c.trace_buf); cudaFree(h->c.trace_idx); h->c.trace_buf = nullptr; h->c.trace_idx = nullptr; }
      h->c.trace_cap = static_cast<int>(value);
      if (value > 0) {
        ALM_CHECK_CUDA(cudaMalloc(&h->c.trace_buf, static_cast<size_t>(value) * 6 * sizeof(unsigned long long)));
        ALM_CHECK_CUDA(cudaMalloc(&h->c.trace_idx, sizeof(int)));
        ALM_CHECK_CUDA(cudaMemset(h->c.trace_idx, 0, sizeof(int)));
      }
    } else if (k == "trace_detail") {
      if (h->c.detail_buf) { cudaFree(h->c.detail_buf); h->c.detail_buf = nullptr; }
      if (value) {
        ALM_CHECK_CUDA(cudaMalloc(&h->c.detail_buf, 64 * 6 * sizeof(unsigned long long)));
        ALM_CHECK_CUDA(cudaMemset(h->c.detail_buf, 0, 64 * 6 * sizeof(unsigned long long)));
      }
    } else if (k == "xattn_impl") {
      ALM_REQUIRE(value >= 0 && value <= 3, ALM_ERR_INVALID, "xattn_impl must be 0..3");
      h->c.xattn_impl = static_cast<int>(value);
    } else if (k == "fuse_ln_gemv") {
      h->c.fuse_ln_gemv = value ? 1 : 0;
    } else if (k == "kv_decoders") {
      ALM_REQUIRE(value >= 1 && value <= 3, ALM_ERR_INVALID, "kv_decoders must be 1..3");
      h->c.kv_decoders = static_cast<int>(value);
    } else if (k == "attn_impl") {
      ALM_REQUIRE(value == 0 || value == 1, ALM_ERR_INVALID, "attn_impl must be 0 or 1");
      h->c.attn_impl = static_cast<int>(value);
    } else if (k == "wattn_impl") {
      ALM_REQUIRE(value >= 0 && value <= 3, ALM_ERR_INVALID, "wattn_impl must be 0 .. 3");
      h->c.wattn_impl = static_cast<int>(value);
    } else if (k == "enc_grid_cap") {
      h->c.enc_grid_cap = static_cast<int>(value);
    } else if (k == "dec_grid_cap") {
      h->c.dec_grid_cap = static_cast<int>(value);
    } else if (k == "xattn_ctas_per_sm") {
      ALM_REQUIRE(value >= 1 && value <= 3, ALM_ERR_INVALID, "xattn_ctas_per_sm must be 1..3");
      h->c.xattn_ctas_per_sm = static_cast<int>(value);
    } else if (k == "xattn_wg") {
      ALM_REQUIRE(value == 1 || value == 2, ALM_ERR_INVALID, "xattn_wg must be 1 or 2");
      h->c.xattn_wg = static_cast<int>(value);
    } else if (k == "sattn_wide") {
      h->c.sattn_wide = value ? 1 : 0;
    } else if (k == "debug_skip") {
      h->c.debug_skip = static_cast<int>(value);
    } else if (k == "decode_priority") {
      h->c.decode_priority = value ? 1 : 0;
    } else if (k == "small_grid_cap") {
      h->c.small_grid_cap = static_cast<int>(value);
    } else if (k == "gemm_plain_epilogue") {
      ALM_REQUIRE(value >= 0 && value <= 2, ALM_ERR_INVALID, "gemm_plain_epilogue must be 0, 1 or 2");
      h->c.gemm_plain_epilogue = static_cast<int>(value);
    } else if (k == "wide_tiles") {
      h->c.wide_tiles = value ? 1 : 0;
    } else if (k == "decode_streams") {
      ALM_REQUIRE(value == 1 || value == 2, ALM_ERR_INVALID, "decode_streams must be 1 or 2");
      h->c.decode_streams = static_cast<int>(value);
    } else if (k == "use_graphs") {
      h->c.use_graphs = value ? 1 : 0;
    } else if (k == "profile_gemm") {
      h->c.profile_gemm = value ? 1 : 0;
    } else if (k == "workspace_mb") {
      ALM_REQUIRE(value >= 64 && h->c.ws.base == nullptr, ALM_ERR_STATE, "workspace_mb must be set before first use");
      h->c.ws_bytes = static_cast<size_t>(value) << 20;
    } else {
      throw AlmError{ALM_ERR_INVALID, "unknown option " + k};
    }
  });
}

long alm_launch_count(alm_ctx* h, int reset) {
  if (!h) return -1;
  const long n = h->c.launches;
  if (reset) h->c.launches = 0;
  return n;
}

int alm_profile_read(alm_ctx* h, double* gemm_ms, double* gemm_flops, long* gemm_launches) {
  return guarded(h, [&] {
    ALM_CHECK_CUDA(cudaStreamSynchronize(h->c.stream));
    double ms = 0, fl = 0;
    for (auto& r : h->c.gemm_recs) {
      float t = 0;
      ALM_CHECK_CUDA(cudaEventElapsedTime(&t, r.a, r.b));
      ms += t;
      fl += r.flops;
      cudaEventDestroy(r.a);
      cudaEventDestroy(r.b);
    }
    if (gemm_ms) *gemm_ms = ms;
    if (gemm_flops) *gemm_flops = fl;
    if (gemm_launches) *gemm_launches = static_cast<long>(h->c.gemm_recs.size());
    h->c.gemm_recs.clear();
  });
}

int alm_trace_read(alm_ctx* h, unsigned long long* out, int max_records, int* n_records) {
  return guarded(h, [&] {
    ALM_REQUIRE(h->c.trace_buf && out && n_records, ALM_ERR_STATE, "trace_gemm is not enabled");
    ALM_CHECK_CUDA(cudaStreamSynchronize(h->c.stream));
    int n = 0;
    ALM_CHECK_CUDA(cudaMemcpy(&n, h->c.trace_idx, sizeof(int), cudaMemcpyDeviceToHost));
    n = std::min(n, std::min(h->c.trace_cap, max_records));
    ALM_CHECK_CUDA(cudaMemcpy(out, h->c.trace_buf, static_cast<size_t>(n) * 6 * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
    ALM_CHECK_CUDA(cudaMemset(h->c.trace_idx, 0, sizeof(int)));
    *n_records = n;
  });
}

int alm_bench_graph_floor(alm_ctx* h, int nodes, int iters, float* us_per_node) {
  // replay cost of a captured chain of `nodes` trivial dependent kernels: the per-kernel floor of the decode loop
  return guarded(h, [&] {
    ALM_REQUIRE(nodes > 0 && iters > 0 && us_per_node, ALM_ERR_INVALID, "alm_bench_graph_floor arguments");
    Ctx* c = &h->c;
    c->ensure_ws();
    ArenaScope arena_scope(c->ws);
    int* p = c->ws.get<int>(4);
    ALM_CHECK_CUDA(cudaMemsetAsync(p, 0, 16, c->stream));
    cudaGraph_t g = nullptr;
    cudaGraphExec_t ge = nullptr;
    ALM_CHECK_CUDA(cudaStreamBeginCapture(c->stream, cudaStreamCaptureModeThreadLocal));
    for (int i = 0; i < nodes; ++i) fill_i32(c, p, 1, i);
    ALM_CHECK_CUDA(cudaStreamEndCapture(c->stream, &g));
    ALM_CHECK_CUDA(cudaGraphInstantiate(&ge, g, 0));
    cudaGraphDestroy(g);
    for (int i = 0; i < 3; ++i) ALM_CHECK_CUDA(cudaGraphLaunch(ge, c->stream));
    cudaEvent_t e0, e1;
    ALM_CHECK_CUDA(cudaEventCreate(&e0));
    ALM_CHECK_CUDA(cudaEventCreate(&e1));
    ALM_CHECK_CUDA(cudaEventRecord(e0, c->stream));
    for (int i = 0; i < iters; ++i) ALM_CHECK_CUDA(cudaGraphLaunch(ge, c->stream));
    ALM_CHECK_CUDA(cudaEventRecord(e1, c->stream));
    ALM_CHECK_CUDA(cudaStreamSynchronize(c->stream));
    float ms = 0;
    ALM_CHECK_CUDA(cudaEventElapsedTime(&ms, e0, e1));
    *us_per_node = ms * 1e3f / (static_cast<float>(iters) * nodes);
    cudaEventDestroy(e0); cudaEventDestroy(e1); cudaGraphExecDestroy(ge);
  });
}

int alm_bench_gemm_ex(alm_ctx* h, int M, int N, int K, int batch, int split_out, int act, int iters,
                      float* ms_per_launch, unsigned long long* detail_out /* 64*6 or NULL */) {
  return guarded(h, [&] {
    ALM_REQUIRE(M > 0 && N > 0 && K > 0 && K % 8 == 0 && batch > 0 && iters > 0 && ms_per_launch, ALM_ERR_INVALID,
                "alm_bench_gemm_ex arguments");
    Ctx* c = &h->c;
    c->ensure_ws();
    ArenaScope arena_scope(c->ws);
    const size_t na = static_cast<size_t>(batch) * M * K, nb = static_cast<size_t>(batch) * N * K;
    const int ldo = (N + 7) & ~7;
    Operand a, b;
    bf16* ah = c->ws.get<bf16>(na); bf16* al = c->ws.get<bf16>(na);
    bf16* bh = c->ws.get<bf16>(nb); bf16* bl = c->ws.get<bf16>(nb);
    ALM_CHECK_CUDA(cudaMemsetAsync(ah, 0x3c, na * 2, c->stream)); ALM_CHECK_CUDA(cudaMemsetAsync(al, 0x30, na * 2, c->stream));
    ALM_CHECK_CUDA(cudaMemsetAsync(bh, 0x3c, nb * 2, c->stream)); ALM_CHECK_CUDA(cudaMemsetAsync(bl, 0x30, nb * 2, c->stream));
    a.hi = ah; a.lo = al; a.rows = M; a.K = K; a.ld = K; a.nb0 = batch; a.bs0 = static_cast<long>(M) * K;
    b.hi = bh; b.lo = bl; b.rows = N; b.K = K; b.ld = K; b.nb0 = batch; b.bs0 = static_cast<long>(N) * K;
    Epilogue e;
    const size_t no = static_cast<size_t>(batch) * M * ldo;
    if (split_out) { e.out_hi = c->ws.get<bf16>(no); e.out_lo = c->ws.get<bf16>(no); }
    else e.out_f32 = c->ws.get<float>(no);
    e.ldo = ldo; e.obs0 = static_cast<long>(M) * ldo; e.act = act;
    for (int i = 0; i < 3; ++i) gemm(c, a, b, e);
    cudaEvent_t e0, e1;
    ALM_CHECK_CUDA(cudaEventCreate(&e0));
    ALM_CHECK_CUDA(cudaEventCreate(&e1));
    ALM_CHECK_CUDA(cudaEventRecord(e0, c->stream));
    for (int i = 0; i < iters; ++i) gemm(c, a, b, e);
    ALM_CHECK_CUDA(cudaEventRecord(e1, c->stream));
    ALM_CHECK_CUDA(cudaStreamSynchronize(c->stream));
    float ms = 0;
    ALM_CHECK_CUDA(cudaEventElapsedTime(&ms, e0, e1));
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    *ms_per_launch = ms / iters;
    if (detail_out && c->detail_buf)
      ALM_CHECK_CUDA(cudaMemcpy(detail_out, c->detail_buf, 64 * 6 * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
  });
}

int alm_bench_gemm(alm_ctx* h, int M, int N, int K, int iters, float* ms_per_launch) {
  return guarded(h, [&] {
    ALM_REQUIRE(M > 0 && N > 0 && K > 0 && K % 8 == 0 && N % 8 == 0 && iters > 0 && ms_per_launch, ALM_ERR_INVALID,
                "alm_bench_gemm arguments");
    Ctx* c = &h->c;
    c->ensure_ws();
    ArenaScope arena_scope(c->ws);
    float* fa = c->ws.get<float>(static_cast<size_t>(M) * K);
    float* fb = c->ws.get<float>(static_cast<size_t>(N) * K);
    // any finite data does; reuse whatever the arena holds after clamping it through a split
    ALM_CHECK_CUDA(cudaMemsetAsync(fa, 0x3c, static_cast<size_t>(M) * K * 4, c->stream));
    ALM_CHECK_CUDA(cudaMemsetAsync(fb, 0x3c, static_cast<size_t>(N) * K * 4, c->stream));
    Operand a, b;
    bf16* ah = c->ws.get<bf16>(static_cast<size_t>(M) * K); bf16* al = c->ws.get<bf16>(static_cast<size_t>(M) * K);
    bf16* bh = c->ws.get<bf16>(static_cast<size_t>(N) * K); bf16* bl = c->ws.get<bf16>(static_cast<size_t>(N) * K);
    split_rows(c, fa, K, M, K, ah, al, K);
    split_rows(c, fb, K, N, K, bh, bl, K);
    a.hi = ah; a.lo = al; a.rows = M; a.K = K; a.ld = K;
    b.hi = bh; b.lo = bl; b.rows = N; b.K = K; b.ld = K;
    Epilogue e;
    e.out_f32 = c->ws.get<float>(static_cast<size_t>(M) * N);
    e.ldo = N;
    for (int i = 0; i < 3; ++i) gemm(c, a, b, e);
    cudaEvent_t e0, e1;
    ALM_CHECK_CUDA(cudaEventCreate(&e0));
    ALM_CHECK_CUDA(cudaEventCreate(&e1));
    ALM_CHECK_CUDA(cudaEventRecord(e0, c->stream));
    for (int i = 0; i < iters; ++i) gemm(c, a, b, e);
    ALM_CHECK_CUDA(cudaEventRecord(e1, c->stream));
    ALM_CHECK_CUDA(cudaStreamSynchronize(c->stream));
    float ms = 0;
    ALM_CHECK_CUDA(cudaEventElapsedTime(&ms, e0, e1));
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    *ms_per_launch = ms / iters;
  });
}

int alm_load_weights(alm_ctx* h, int model_kind, const alm_tensor_desc* tensors, int n) {
  return guarded(h, [&] {
    ALM_REQUIRE(tensors && n > 0, ALM_ERR_INVALID, "empty state dict");
    std::map<std::string, HostTensor> t;
    for (int i = 0; i < n; ++i) {
      const alm_tensor_desc& d = tensors[i];
      ALM_REQUIRE(d.name && d.ndim >= 0 && d.ndim <= 4, ALM_ERR_INVALID, "bad tensor descriptor");
      HostTensor ht;
      size_t numel = 1;
      for (int k = 0; k < d.ndim; ++k) {
        ht.shape.push_back(d.shape[k]);
        numel *= static_cast<size_t>(d.shape[k]);
      }
      ht.f32.resize(numel);
      if (d.data == nullptr) {  // shape-only placeholder (non-root ranks before alm_broadcast_weights)
        ht.placeholder = true;
        t.emplace(d.name, std::move(ht));
        continue;
      }
      switch (d.dtype) {
        case ALM_F32: memcpy(ht.f32.data(), d.data, numel * 4); break;
        case ALM_F16:
          for (size_t j = 0; j < numel; ++j) ht.f32[j] = f16_bits_to_f32(static_cast<const uint16_t*>(d.data)[j]);
          break;
        case ALM_BF16:
          for (size_t j = 0; j < numel; ++j) ht.f32[j] = bf16_bits_to_f32(static_cast<const uint16_t*>(d.data)[j]);
          break;
        case ALM_I64:
          for (size_t j = 0; j < numel; ++j) ht.f32[j] = static_cast<float>(static_cast<const int64_t*>(d.data)[j]);
          break;
        default: throw AlmError{ALM_ERR_INVALID, std::string("unknown dtype for ") + d.name};
      }
      t.emplace(d.name, std::move(ht));
    }
    if (model_kind == ALM_MODEL_OMNI_SPOT || model_kind == ALM_MODEL_OMNI_KIE) omni_load(&h->c, model_kind, t);
    else if (model_kind == ALM_MODEL_MGPSTR) mgp_load(&h->c, t);
    else throw AlmError{ALM_ERR_INVALID, "unknown model kind"};
    ALM_CHECK_CUDA(cudaDeviceSynchronize());
  });
}

int alm_synchronize(alm_ctx* h) {
  return guarded(h, [&] { ALM_CHECK_CUDA(cudaStreamSynchronize(h->c.stream)); });
}

// ------------------------------------------------------------------------------------------ sharing / streams / comm
int alm_share_weights(alm_ctx* h, alm_ctx* owner) {
  return guarded(h, [&] {
    ALM_REQUIRE(owner && owner != h, ALM_ERR_INVALID, "alm_share_weights: owner context");
    ALM_REQUIRE(owner->c.device == h->c.device, ALM_ERR_INVALID, "alm_share_weights: contexts are on different devices");
    ALM_REQUIRE(owner->c.wstore && (owner->c.omni || owner->c.mgp), ALM_ERR_STATE, "alm_share_weights: owner has no weights");
    delete h->c.omni;
    h->c.omni = nullptr;
    mgp_free(h->c.mgp);
    h->c.mgp = nullptr;
    h->c.wstore = owner->c.wstore;  // ref-counted: the slabs live until the last context using them is freed
    h->c.wbase = nullptr; h->c.wcap = 0; h->c.woff = 0;
    if (owner->c.omni) h->c.omni = omni_share(owner->c.omni);
    if (owner->c.mgp) h->c.mgp = mgp_share(owner->c.mgp);
  });
}

int alm_stream_wait(alm_ctx* h, void* producer_stream) {
  return guarded(h, [&] {
    Ctx* c = &h->c;
    if (!c->ev_order) ALM_CHECK_CUDA(cudaEventCreateWithFlags(&c->ev_order, cudaEventDisableTiming));
    ALM_CHECK_CUDA(cudaEventRecord(c->ev_order, static_cast<cudaStream_t>(producer_stream)));
    ALM_CHECK_CUDA(cudaStreamWaitEvent(c->stream, c->ev_order, 0));
  });
}

int alm_stream_release(alm_ctx* h, void* consumer_stream) {
  return guarded(h, [&] {
    Ctx* c = &h->c;
    if (!c->ev_order) ALM_CHECK_CUDA(cudaEventCreateWithFlags(&c->ev_order, cudaEventDisableTiming));
    ALM_CHECK_CUDA(cudaEventRecord(c->ev_order, c->stream));
    ALM_CHECK_CUDA(cudaStreamWaitEvent(static_cast<cudaStream_t>(consumer_stream), c->ev_order, 0));
  });
}

int alm_comm_unique_id(void* id128) {
  if (!id128) return ALM_ERR_INVALID;
  try {
    comm_unique_id(id128);
    return ALM_OK;
  } catch (const AlmError& e) {
    return e.code;
  } catch (...) {
    return ALM_ERR_INVALID;
  }
}

int alm_comm_init(alm_ctx* h, const void* id128, int rank, int world) {
  return guarded(h, [&] { comm_init(&h->c, id128, rank, world); });
}

int alm_comm_attach(alm_ctx* h, void* nccl_comm, int rank, int world) {
  return guarded(h, [&] { comm_attach(&h->c, nccl_comm, rank, world); });
}

int alm_broadcast_weights(alm_ctx* h, int root) {
  return guarded(h, [&] { comm_broadcast_weights(&h->c, root); });
}

int alm_gather_sequences(alm_ctx* h, const void* send, size_t bytes_per_rank, void* recv_host) {
  return guarded(h, [&] { comm_gather(&h->c, send, bytes_per_rank, recv_host); });
}

// ------------------------------------------------------------------------------------------ pre-processing
namespace {

// device copies of the caller's uint8 HWC images (host pointers are staged into the workspace on the stream)
std::vector<PreImage> stage_images(alm_ctx* h, const uint8_t* const* rgb, const int* heights, const int* widths, int n) {
  Ctx* c = &h->c;
  c->ensure_ws();
  std::vector<PreImage> imgs(static_cast<size_t>(n));
  for (int i = 0; i < n; ++i) {
    ALM_REQUIRE(rgb[i] && heights[i] > 0 && widths[i] > 0, ALM_ERR_INVALID, "image pointer / size");
    const size_t bytes = static_cast<size_t>(heights[i]) * widths[i] * 3;
    const uint8_t* d = rgb[i];
    if (!is_device_ptr(d)) {
      uint8_t* slot = c->ws.get<uint8_t>(bytes);
      ALM_CHECK_CUDA(cudaMemcpyAsync(slot, rgb[i], bytes, cudaMemcpyHostToDevice, c->stream));
      d = slot;
    }
    imgs[static_cast<size_t>(i)] = PreImage{d, heights[i], widths[i], 0, 0};
  }
  return imgs;
}

}  // namespace

int alm_pre_omni_plan(const int* heights, const int* widths, int n, int test_min_size, int test_max_size, int* sizes,
                      int* Hmax, int* Wmax) {
  if (!heights || !widths || n < 0 || test_min_size <= 0 || !sizes || !Hmax || !Wmax) return ALM_ERR_INVALID;
  int hm = 0, wm = 0;
  for (int i = 0; i < n; ++i) {
    if (heights[i] <= 0 || widths[i] <= 0) return ALM_ERR_INVALID;
    pre_omni_size(heights[i], widths[i], test_min_size, test_max_size, &sizes[2 * i], &sizes[2 * i + 1]);
    hm = std::max(hm, sizes[2 * i]);
    wm = std::max(wm, sizes[2 * i + 1]);
  }
  *Hmax = hm; *Wmax = wm;
  return ALM_OK;
}

int alm_pre_coeffs(int in_size, int out_size, int filter, int* ksize, int* bounds, int* coefs, size_t cap_ints) {
  try {
    return pre_coeffs(in_size, out_size, filter, ksize, bounds, coefs, cap_ints);
  } catch (...) {
    return ALM_ERR_INVALID;
  }
}

int alm_pre_omni_pages(alm_ctx* h, const uint8_t* const* rgb, const int* heights, const int* widths, int n,
                       int test_min_size, int test_max_size, float* tensors, uint8_t* mask) {
  return guarded(h, [&] {
    ALM_REQUIRE(rgb && heights && widths && n > 0 && test_min_size > 0 && tensors && mask, ALM_ERR_INVALID,
                "alm_pre_omni_pages arguments");
    ALM_REQUIRE(is_device_ptr(tensors) && is_device_ptr(mask), ALM_ERR_INVALID, "outputs must be device buffers");
    Ctx* c = &h->c;
    c->ensure_ws();
    ArenaScope arena_scope(c->ws);
    std::vector<PreImage> imgs = stage_images(h, rgb, heights, widths, n);
    int Hc = 0, Wc = 0;
    for (auto& im : imgs) {
      pre_omni_size(im.h, im.w, test_min_size, test_max_size, &im.oh, &im.ow);
      Hc = std::max(Hc, im.oh);
      Wc = std::max(Wc, im.ow);
    }
    pre_resize_batch(c, imgs, PRE_BILINEAR, true, tensors, Hc, Wc, mask);
  });
}

int alm_pre_mgp_crops(alm_ctx* h, const uint8_t* const* rgb, const int* heights, const int* widths, int n, int imgH,
                      int imgW, float* out) {
  return guarded(h, [&] {
    ALM_REQUIRE(rgb && heights && widths && n > 0 && imgH > 0 && imgW > 0 && out, ALM_ERR_INVALID,
                "alm_pre_mgp_crops arguments");
    ALM_REQUIRE(is_device_ptr(out), ALM_ERR_INVALID, "output must be a device buffer");
    Ctx* c = &h->c;
    c->ensure_ws();
    ArenaScope arena_scope(c->ws);
    std::vector<PreImage> imgs = stage_images(h, rgb, heights, widths, n);
    for (auto& im : imgs) { im.oh = imgH; im.ow = imgW; }
    pre_resize_batch(c, imgs, PRE_BICUBIC, false, out, imgH, imgW, nullptr);
  });
}

// ------------------------------------------------------------------------------------------ OmniParser
int alm_omni_encode(alm_ctx* h, const float* img, const uint8_t* mask, int B, int H, int W) {
  return guarded(h, [&] {
    ALM_REQUIRE(img != nullptr && B > 0 && H > 0 && W > 0, ALM_ERR_INVALID, "alm_omni_encode arguments");
    const size_t px = static_cast<size_t>(B) * H * W;
    const float* dimg = static_cast<const float*>(stage_input(h, img, px * 3 * sizeof(float), &h->dev_in, &h->dev_in_bytes));
    const uint8_t* dmask = static_cast<const uint8_t*>(stage_input(h, mask, px, &h->dev_mask, &h->dev_mask_bytes));
    omni_encode(&h->c, dimg, dmask, B, H, W);
  });
}

int alm_omni_memory_shape(alm_ctx* h, int* B, int* mh, int* mw) {
  return guarded(h, [&] {
    ALM_REQUIRE(h->c.omni && h->c.omni->encoded, ALM_ERR_STATE, "no encoded batch");
    if (B) *B = h->c.omni->B;
    if (mh) *mh = h->c.omni->mh;
    if (mw) *mw = h->c.omni->mw;
  });
}

int alm_omni_last_timing(alm_ctx* h, float* encode_ms, float* pt_ms, float* polyrec_ms) {
  return guarded(h, [&] {
    ALM_CHECK_CUDA(cudaStreamSynchronize(h->c.stream));
    float e = -1.f, p = -1.f, r = -1.f;
    if (h->c.timing_valid[0]) ALM_CHECK_CUDA(cudaEventElapsedTime(&e, h->c.ev_t[0], h->c.ev_t[1]));
    if (h->c.timing_valid[1]) {
      ALM_CHECK_CUDA(cudaEventElapsedTime(&p, h->c.ev_t[2], h->c.ev_t[3]));
      ALM_CHECK_CUDA(cudaEventElapsedTime(&r, h->c.ev_t[3], h->c.ev_t[4]));
    }
    if (encode_ms) *encode_ms = e;
    if (pt_ms) *pt_ms = p;
    if (polyrec_ms) *polyrec_ms = r;
  });
}

int alm_omni_vocab(alm_ctx* h) { return (h && h->c.omni) ? h->c.omni->V : ALM_ERR_STATE; }

int alm_omni_get_feature(alm_ctx* h, int level, float* out, size_t out_elems) {
  return guarded(h, [&] {
    OmniModel* m = h->c.omni;
    ALM_REQUIRE(m && m->encoded, ALM_ERR_STATE, "no encoded batch");
    ALM_REQUIRE(level >= 0 && level < 4 && out, ALM_ERR_INVALID, "feature level");
    const size_t n = static_cast<size_t>(m->B) * m->Hs[level] * m->Ws[level] * (128 << level);
    ALM_REQUIRE(out_elems == n, ALM_ERR_INVALID, "feature buffer size mismatch: expected " + std::to_string(n));
    d2h(&h->c, out, m->feat[level], n * sizeof(float));
    ALM_CHECK_CUDA(cudaStreamSynchronize(h->c.stream));
  });
}

int alm_omni_get_memory(alm_ctx* h, int which, float* out, size_t out_elems) {
  return guarded(h, [&] {
    OmniModel* m = h->c.omni;
    ALM_REQUIRE(m && m->encoded, ALM_ERR_STATE, "no encoded batch");
    const size_t n = static_cast<size_t>(m->B) * m->M * 512;
    ALM_REQUIRE(out && out_elems == n && (which == 0 || which == 1), ALM_ERR_INVALID, "memory buffer size mismatch");
    d2h(&h->c, out, which == 0 ? m->memory : m->pos, n * sizeof(float));
    ALM_CHECK_CUDA(cudaStreamSynchronize(h->c.stream));
  });
}

int alm_omni_decode(alm_ctx* h, const int64_t* pt_prompt, int n_prompt, const alm_decode_cfg* cfg, int32_t* n_inst,
                    int64_t* pt, int64_t* poly, int64_t* rec, float* rec_prob) {
  return guarded(h, [&] {
    ALM_REQUIRE(pt_prompt && cfg && n_inst && pt && poly && rec && rec_prob, ALM_ERR_INVALID, "null argument");
    omni_decode(&h->c, pt_prompt, n_prompt, *cfg, n_inst, pt, poly, rec, rec_prob);
  });
}

int alm_omni_decode_kie(alm_ctx* h, const int64_t* pt_prompt, int n_prompt, const alm_decode_cfg* cfg, int32_t* n_tok,
                        int64_t* pt_tokens, float* pt_probs, int32_t* n_inst, int32_t* inst_pos, int64_t* poly,
                        int64_t* rec, float* rec_prob) {
  return guarded(h, [&] {
    ALM_REQUIRE(pt_prompt && cfg && n_tok && pt_tokens && pt_probs && n_inst && inst_pos && poly && rec && rec_prob,
                ALM_ERR_INVALID, "null argument");
    omni_decode_kie(&h->c, pt_prompt, n_prompt, *cfg, n_tok, pt_tokens, pt_probs, n_inst, inst_pos, poly, rec, rec_prob);
  });
}

int alm_omni_decode_points(alm_ctx* h, const int64_t* pt_prompt, int n_prompt, const alm_decode_cfg* cfg, int32_t* n_tok,
                           int64_t* pt_tokens, float* pt_probs) {
  return guarded(h, [&] {
    ALM_REQUIRE(pt_prompt && cfg && n_tok && pt_tokens, ALM_ERR_INVALID, "null argument");
    omni_decode_points(&h->c, pt_prompt, n_prompt, *cfg, n_tok, pt_tokens, pt_probs);
  });
}

int alm_omni_decode_prompted(alm_ctx* h, const int64_t* prompts, int R, int n_prompt, const alm_decode_cfg* cfg,
                             int32_t* n_inst, int64_t* pt, int64_t* poly, int64_t* rec, float* rec_prob) {
  return guarded(h, [&] {
    ALM_REQUIRE(prompts && cfg && n_inst && pt && poly && rec && rec_prob, ALM_ERR_INVALID, "null argument");
    omni_decode_prompted(&h->c, prompts, R, n_prompt, *cfg, n_inst, pt, poly, rec, rec_prob);
  });
}

int alm_omni_decode_points_prompted(alm_ctx* h, const int64_t* prompts, int R, int n_prompt, const alm_decode_cfg* cfg,
                                    int32_t* n_tok, int64_t* pt_tokens, float* pt_probs) {
  return guarded(h, [&] {
    ALM_REQUIRE(prompts && cfg && n_tok && pt_tokens, ALM_ERR_INVALID, "null argument");
    omni_decode_points_prompted(&h->c, prompts, R, n_prompt, *cfg, n_tok, pt_tokens, pt_probs);
  });
}

int alm_omni_decode_logits(alm_ctx* h, int image, int kind, const int64_t* seq, int n_seq, int len, float* logits) {
  return guarded(h, [&] {
    ALM_REQUIRE(seq && logits, ALM_ERR_INVALID, "null argument");
    omni_decode_logits(&h->c, image, kind, seq, n_seq, len, logits);
  });
}

// ------------------------------------------------------------------------------------------ MGP-STR
int alm_mgpstr_forward(alm_ctx* h, const float* img, int B, float* attn, float* char_logits, float* bpe_logits,
                       float* wp_logits, int32_t* ids, float* prob) {
  return guarded(h, [&] {
    ALM_REQUIRE(img && B > 0, ALM_ERR_INVALID, "alm_mgpstr_forward arguments");
    const float* dimg = static_cast<const float*>(
        stage_input(h, img, static_cast<size_t>(B) * 3 * 32 * 128 * sizeof(float), &h->dev_in, &h->dev_in_bytes));
    mgp_forward(&h->c, dimg, B, attn, char_logits, bpe_logits, wp_logits, ids, prob);
  });
}

int alm_mgpstr_info(alm_ctx* h, int* dim, int* depth, int* heads, int* n_a3, int* vocab3) {
  return guarded(h, [&] {
    ALM_REQUIRE(h->c.mgp != nullptr, ALM_ERR_STATE, "alm_mgpstr_info before alm_load_weights");
    mgp_info(h->c.mgp, dim, depth, heads, n_a3, vocab3);
  });
}

// ------------------------------------------------------------------------------------------ unit ops
int alm_op_linear(alm_ctx* h, const float* A, const float* W, const float* bias, float* C, int M, int N, int K, int act,
                  int batch) {
  return guarded(h, [&] {
    ALM_REQUIRE(A && W && C && M > 0 && N > 0 && K > 0 && batch > 0, ALM_ERR_INVALID, "alm_op_linear arguments");
    ALM_REQUIRE(is_device_ptr(A) && is_device_ptr(W) && is_device_ptr(C), ALM_ERR_INVALID, "device pointers required");
    Ctx* c = &h->c;
    c->ensure_ws();
    ArenaScope arena_scope(c->ws);
    const int Kp = (K + 7) & ~7;
    bf16* ah = c->ws.get<bf16>(static_cast<size_t>(batch) * M * Kp);
    bf16* al = c->ws.get<bf16>(static_cast<size_t>(batch) * M * Kp);
    bf16* wh = c->ws.get<bf16>(static_cast<size_t>(batch) * N * Kp);
    bf16* wl = c->ws.get<bf16>(static_cast<size_t>(batch) * N * Kp);
    if (Kp != K) {
      ALM_CHECK_CUDA(cudaMemsetAsync(ah, 0, static_cast<size_t>(batch) * M * Kp * 2, c->stream));
      ALM_CHECK_CUDA(cudaMemsetAsync(al, 0, static_cast<size_t>(batch) * M * Kp * 2, c->stream));
      ALM_CHECK_CUDA(cudaMemsetAsync(wh, 0, static_cast<size_t>(batch) * N * Kp * 2, c->stream));
      ALM_CHECK_CUDA(cudaMemsetAsync(wl, 0, static_cast<size_t>(batch) * N * Kp * 2, c->stream));
    }
    ALM_REQUIRE(K % 4 == 0, ALM_ERR_UNSUPPORTED, "alm_op_linear: K must be a multiple of 4");
    split_rows(c, A, K, static_cast<long>(batch) * M, K, ah, al, Kp);
    split_rows(c, W, K, static_cast<long>(batch) * N, K, wh, wl, Kp);
    Operand a, b;
    a.hi = ah; a.lo = al; a.rows = M; a.K = K; a.ld = Kp; a.nb0 = batch; a.bs0 = static_cast<long>(M) * Kp;
    b.hi = wh; b.lo = wl; b.rows = N; b.K = K; b.ld = Kp; b.nb0 = batch; b.bs0 = static_cast<long>(N) * Kp;
    Epilogue e;
    e.out_f32 = C; e.ldo = N; e.obs0 = static_cast<long>(M) * N;
    e.bias = bias; e.bias_mode = bias ? BIAS_COL : BIAS_NONE; e.act = act;
    gemm(c, a, b, e);
    ALM_CHECK_CUDA(cudaStreamSynchronize(c->stream));
  });
}

int alm_op_attention(alm_ctx* h, const float* qkv, float* out, int B, int T, int H) {
  return guarded(h, [&] {
    ALM_REQUIRE(qkv && out && B > 0 && T > 0 && H > 0, ALM_ERR_INVALID, "alm_op_attention arguments");
    ALM_REQUIRE(is_device_ptr(qkv) && is_device_ptr(out), ALM_ERR_INVALID, "device pointers required");
    Ctx* c = &h->c;
    c->ensure_ws();
    ArenaScope arena_scope(c->ws);
    const long R = static_cast<long>(B) * T;
    const int D = H * 64;
    bf16* hi = c->ws.get<bf16>(static_cast<size_t>(R) * 3 * D);
    bf16* lo = c->ws.get<bf16>(static_cast<size_t>(R) * 3 * D);
    split_rows(c, qkv, 3 * D, R, 3 * D, hi, lo, 3 * D);
    attention_tc(c, hi, lo, 3L * D, B, T, H, nullptr, nullptr, out, D);
    ALM_CHECK_CUDA(cudaStreamSynchronize(c->stream));
  });
}

int alm_op_layernorm(alm_ctx* h, const float* x, const float* gamma, const float* beta, float eps, float* y, long rows,
                     int C) {
  return guarded(h, [&] {
    ALM_REQUIRE(x && gamma && beta && y && rows > 0, ALM_ERR_INVALID, "alm_op_layernorm arguments");
    gather_ln(&h->c, x, C, nullptr, 1, C, rows, gamma, beta, eps, false, nullptr, 0, y, C, nullptr, nullptr, 0, nullptr,
              nullptr);
    ALM_CHECK_CUDA(cudaStreamSynchronize(h->c.stream));
  });
}

int alm_op_window_attention(alm_ctx* h, const float* qkv, const float* bias_table, float* out, int B, int nWh, int nWw,
                            int C, int heads, int shift) {
  return guarded(h, [&] {
    ALM_REQUIRE(qkv && bias_table && out, ALM_ERR_INVALID, "alm_op_window_attention arguments");
    Ctx* c = &h->c;
    c->ensure_ws();
    ArenaScope arena_scope(c->ws);
    std::vector<float> tab(static_cast<size_t>(169) * heads), dense(static_cast<size_t>(heads) * 2401);
    ALM_CHECK_CUDA(cudaMemcpy(tab.data(), bias_table, tab.size() * 4, cudaMemcpyDeviceToHost));
    for (int hh = 0; hh < heads; ++hh)
      for (int i = 0; i < 49; ++i)
        for (int j = 0; j < 49; ++j)
          dense[static_cast<size_t>(hh) * 2401 + i * 49 + j] =
              tab[static_cast<size_t>((i / 7 - j / 7 + 6) * 13 + (i % 7 - j % 7 + 6)) * heads + hh];
    float* dd = c->ws.get<float>(dense.size());
    ALM_CHECK_CUDA(cudaMemcpyAsync(dd, dense.data(), dense.size() * 4, cudaMemcpyHostToDevice, c->stream));
    window_attention(c, qkv, C, heads, nWh, nWw, B, shift, nWh * 7, nWw * 7, dd, nullptr, nullptr, out);
    ALM_CHECK_CUDA(cudaStreamSynchronize(c->stream));
  });
}

int alm_op_gemv(alm_ctx* h, const float* x, const float* x2, int n_split, long ldx, const float* W, const float* bias,
                const float* resid, long ldr, float* out, long ldo, int M, int N, int K, int act, const float* ln_g,
                const float* ln_b, float ln_eps, const float* pos, int pos_split) {
  return guarded(h, [&] {
    ALM_REQUIRE(x && W && out && N > 0 && K > 0 && act >= 0 && act <= 2, ALM_ERR_INVALID, "alm_op_gemv arguments");
    ALM_REQUIRE(ldx >= K && ldo >= N && (resid == nullptr || ldr >= N), ALM_ERR_INVALID, "alm_op_gemv strides");
    gemv_rows(&h->c, x, x2, n_split, ldx, W, bias, resid, ldr, out, ldo, M, N, K, act, ln_g, ln_b, ln_eps, pos, pos_split);
    ALM_CHECK_CUDA(cudaStreamSynchronize(h->c.stream));
  });
}

int alm_op_self_attn_step(alm_ctx* h, const float* qk, int ld_qk, const float* vnew, int ld_v, float* kc, float* vc, int S,
                          int t, int Tmax, float* out_f32, uint16_t* out_hi, uint16_t* out_lo) {
  return guarded(h, [&] {
    ALM_REQUIRE(qk && vnew && kc && vc && (out_f32 || out_hi) && S > 0, ALM_ERR_INVALID, "alm_op_self_attn_step arguments");
    // the 1024-row position table bounds every decode loop; q / k rows are read as float4
    ALM_REQUIRE(Tmax >= 1 && Tmax <= 1024 && t >= 0 && t < Tmax, ALM_ERR_INVALID, "alm_op_self_attn_step: 0 <= t < Tmax <= 1024");
    ALM_REQUIRE(ld_qk >= 1024 && ld_qk % 4 == 0 && ld_v >= 512, ALM_ERR_INVALID, "alm_op_self_attn_step strides");
    Ctx* c = &h->c;
    c->ensure_ws();
    ArenaScope arena_scope(c->ws);
    int* tp = c->ws.get<int>(1);  // the kernels read the position from the device, as in a graph-replayed decode step
    ALM_CHECK_CUDA(cudaMemcpyAsync(tp, &t, sizeof(int), cudaMemcpyHostToDevice, c->stream));
    self_attn_step(c, qk, vnew, kc, vc, S, tp, Tmax, reinterpret_cast<bf16*>(out_hi), reinterpret_cast<bf16*>(out_lo),
                   out_f32, ld_qk, ld_v);
    ALM_CHECK_CUDA(cudaStreamSynchronize(c->stream));
  });
}

}  // extern "C"

namespace {

// [img][8][M][64] fp32 values of decoder-layer slot dl -> the feature-major V_c^T planes of the unfused path
// ([img*6144 + dl*512 + h*64 + d][Mpad]); vt_* point at the first row of the slot, padding columns M..Mpad-1 are zero
__global__ void op_vt_kernel(const float* __restrict__ v, int nimg, int M, int Mpad, bf16* __restrict__ vt_hi,
                             bf16* __restrict__ vt_lo) {
  const long i = static_cast<long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= static_cast<long>(nimg) * 512 * Mpad) return;
  const int m = static_cast<int>(i % Mpad), f = static_cast<int>((i / Mpad) % 512), img = static_cast<int>(i / (512L * Mpad));
  const float y = m < M ? v[((static_cast<long>(img) * 8 + (f >> 6)) * M + m) * 64 + (f & 63)] : 0.f;
  const long o = (static_cast<long>(img) * 6144 + f) * Mpad + m;
  split_bf16(y, vt_hi[o], vt_lo[o]);
}

__global__ void op_join_kernel(const bf16* __restrict__ hi, const bf16* __restrict__ lo, long n, float* __restrict__ out) {
  const long i = static_cast<long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i < n) out[i] = __bfloat162float(hi[i]) + __bfloat162float(lo[i]);
}

}  // namespace

extern "C" {

int alm_op_cross_attention(alm_ctx* h, const float* q, const float* k, const float* v, const uint8_t* kpm, int B, int img0,
                           int nimg, int Ncap, int M, int dl, int q_split, float* out) {
  return guarded(h, [&] {
    ALM_REQUIRE(q && k && v && out && B > 0 && nimg > 0 && img0 >= 0 && img0 + nimg <= B && Ncap > 0 && M > 0 && dl >= 0 &&
                    dl < 12 && (q_split == 0 || q_split == 1),
                ALM_ERR_INVALID, "alm_op_cross_attention arguments");
    Ctx* c = &h->c;
    const int impl = c->xattn_impl;
    ALM_REQUIRE(impl != 1 || (Ncap == 1 && q_split == 0), ALM_ERR_UNSUPPORTED,
                "alm_op_cross_attention: xattn_impl 1 runs the fused kernel for one fp32 query per image only");
    c->ensure_ws();
    ArenaScope arena_scope(c->ws);
    // the K / V cache of alm_omni_encode: split bf16 [B*96 (image, decoder-layer slot, head)][M][64] per plane (and the
    // feature-major V_c^T [B*6144][Mpad] for xattn_impl 1); every slice but (img0 .. img0+nimg-1, dl) holds NaN
    const long slice = static_cast<long>(M) * 64, plane = static_cast<long>(B) * 96 * slice;
    const int Mpad = (M + 7) & ~7;
    const int nan2 = 0x7fc07fc0;  // two bf16 quiet NaNs
    bf16* kv[4];
    for (auto& p : kv) {
      p = c->ws.get<bf16>(plane);
      fill_i32(c, reinterpret_cast<int*>(p), plane / 2, nan2);
    }
    for (int i = img0; i < img0 + nimg; ++i) {
      const long off = (static_cast<long>(i) * 96 + static_cast<long>(dl) * 8) * slice;
      split_rows(c, k + i * 8 * slice, 64, 8L * M, 64, kv[0] + off, kv[1] + off, 64);
      split_rows(c, v + i * 8 * slice, 64, 8L * M, 64, kv[2] + off, kv[3] + off, 64);
    }
    bf16 *vt_hi = nullptr, *vt_lo = nullptr;
    if (impl == 1) {
      const long vplane = static_cast<long>(B) * 6144 * Mpad;
      vt_hi = c->ws.get<bf16>(vplane);
      vt_lo = c->ws.get<bf16>(vplane);
      fill_i32(c, reinterpret_cast<int*>(vt_hi), vplane / 2, nan2);
      fill_i32(c, reinterpret_cast<int*>(vt_lo), vplane / 2, nan2);
      const long voff = (static_cast<long>(img0) * 6144 + static_cast<long>(dl) * 512) * Mpad;
      const long n = static_cast<long>(nimg) * 512 * Mpad;
      op_vt_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, c->stream>>>(v + img0 * 8 * slice, nimg, M, Mpad,
                                                                                  vt_hi + voff, vt_lo + voff);
      check_launch("op_vt");
    }
    const long rows = static_cast<long>(nimg) * Ncap;
    bf16 *q_hi = nullptr, *q_lo = nullptr;
    if (q_split) {
      q_hi = c->ws.get<bf16>(rows * 512);
      q_lo = c->ws.get<bf16>(rows * 512);
      split_rows(c, q, 512, rows, 512, q_hi, q_lo, 512);
    }
    const float* q_f32 = q_split ? nullptr : q;
    // the decode loops take fp32 output only from fp32 queries on the <= 16-query path; otherwise the split pair
    const bool f32_out = !q_split && Ncap <= 16;
    bf16 *o_hi = nullptr, *o_lo = nullptr;
    if (!f32_out) {
      o_hi = c->ws.get<bf16>(rows * 512);
      o_lo = c->ws.get<bf16>(rows * 512);
    }
    float* o_f32 = f32_out ? out : nullptr;
    const uint8_t* kpm_i = kpm ? kpm + static_cast<long>(img0) * M : nullptr;
    const long koff = (static_cast<long>(img0) * 96 + static_cast<long>(dl) * 8) * slice;
    int* counters = nullptr;
    int pairs = 0;
    if (impl == 1) {  // alloc_decode + decoder_step for one query per image
      const int ns = cross_attn_q1_splits(c, nimg, M);
      float* partial = c->ws.get<float>(static_cast<size_t>(nimg) * 8 * ns * 66);
      pairs = nimg * 8;
      counters = c->ws.get<int>(pairs);
      fill_i32(c, counters, pairs, 0);
      const long voff = (static_cast<long>(img0) * 6144 + static_cast<long>(dl) * 512) * Mpad;
      cross_attn_q1(c, q, kv[0] + koff, kv[1] + koff, vt_hi + voff, vt_lo + voff, kpm_i, nimg, M, Mpad, partial, counters,
                    ns, o_hi, o_lo, o_f32);
    } else {  // alloc_decode + fused_xattn
      int grid = 1, parts = 1;
      const bool tc = impl == 3 && Ncap > 16;
      if (tc) cross_attn_tc_plan(c, nimg, Ncap, M, &grid, &parts, &pairs);
      else if (impl == 2) cross_attn_tma_plan(c, nimg, Ncap, M, &grid, &parts, &pairs);
      else cross_attn_mq_plan(c, nimg, Ncap, M, &grid, &parts, &pairs);
      float* partial = c->ws.get<float>(cross_attn_mq_partial_floats(pairs, parts));
      counters = c->ws.get<int>(pairs);
      fill_i32(c, counters, pairs, 0);
      const int z0 = static_cast<int>(img0 * 96 + dl * 8);
      if (tc)
        cross_attn_tc(c, q_hi, q_lo, q_f32, nimg, Ncap, kv[0], kv[1], kv[2], kv[3], static_cast<long>(B) * 96, z0, kpm_i, M,
                      grid, parts, partial, counters, o_hi, o_lo, o_f32);
      else if (impl == 2)
        cross_attn_tma(c, q_hi, q_lo, q_f32, nimg, Ncap, kv[0], kv[1], kv[2], kv[3], static_cast<long>(B) * 96, z0, kpm_i, M,
                       grid, parts, partial, counters, o_hi, o_lo, o_f32);
      else
        cross_attn_mq(c, q_hi, q_lo, q_f32, nimg, Ncap, kv[0] + koff, kv[1] + koff, kv[2] + koff, kv[3] + koff, kpm_i, M, grid,
                      parts, partial, counters, o_hi, o_lo, o_f32);
    }
    if (!f32_out) {
      const long n = rows * 512;
      op_join_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, c->stream>>>(o_hi, o_lo, n, out);
      check_launch("op_join");
    }
    // the merge counters reset themselves for the next launch (a captured decode step replays without re-zeroing them)
    std::vector<int> cnt(pairs);
    ALM_CHECK_CUDA(cudaMemcpyAsync(cnt.data(), counters, pairs * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    ALM_CHECK_CUDA(cudaStreamSynchronize(c->stream));
    ALM_REQUIRE(std::all_of(cnt.begin(), cnt.end(), [](int x) { return x == 0; }), ALM_ERR_STATE,
                "alm_op_cross_attention: merge counters were not reset by the kernel");
  });
}

int alm_op_head_select(alm_ctx* h, const float* logits, int S, int V, int nsoft, int phase, const alm_decode_cfg* cfg, int t,
                       int n_prompt_m1, int32_t* tokens, int tstride, float* probs, int pstride, int32_t* finished,
                       int32_t* ntok) {
  return guarded(h, [&] {
    ALM_REQUIRE(logits && cfg && tokens && S > 0 && V > 0 && nsoft > 0 && nsoft <= V && phase >= 0 && phase <= 2,
                ALM_ERR_INVALID, "alm_op_head_select arguments");
    ALM_REQUIRE(t >= n_prompt_m1 && n_prompt_m1 >= 0 && t + 1 < tstride && (probs == nullptr || t - n_prompt_m1 < pstride),
                ALM_ERR_INVALID, "alm_op_head_select: position / strides");
    ALM_REQUIRE((finished == nullptr) == (ntok == nullptr), ALM_ERR_INVALID, "alm_op_head_select: finished and ntok go together");
    Ctx* c = &h->c;
    c->ensure_ws();
    ArenaScope arena_scope(c->ws);
    int* tp = c->ws.get<int>(1);
    ALM_CHECK_CUDA(cudaMemcpyAsync(tp, &t, sizeof(int), cudaMemcpyHostToDevice, c->stream));
    const HeadCfg hc{cfg->num_bins, cfg->pt_eos, cfg->rec_eos, cfg->recog_pad, cfg->vie_categories};  // as omni.cu maps it
    head_select(c, logits, S, V, nsoft, phase, hc, tokens, tstride, tp, n_prompt_m1, probs, pstride, finished, ntok);
    ALM_CHECK_CUDA(cudaStreamSynchronize(c->stream));
  });
}

}  // extern "C"
