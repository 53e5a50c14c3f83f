/*
 * libalm_ocr.so -- C-ABI of the B200-native OCR forward path.
 *
 * The reference (AlibabaResearch/AdvancedLiterateMachinery) has no FFI table; its boundary for this
 * path is two Python `nn.Module.forward` call sites plus two checkpoint layouts (SURVEY.md 8b):
 *
 *   OmniParser : `output = model(samples, seqs)`      OCR/OmniParser/engine/val.py:35
 *                (OmniParser.forward, OCR/OmniParser/model/omniparser.py:19-32)
 *   MGP-STR    : `model(image, is_eval=True)`         OCR/MGP-STR/demo.py:33, test_final.py:140
 *                (MGPSTR.forward, OCR/MGP-STR/modules/mgp_str.py:96-101)
 *   weights    : torch.load(path)['model']            OCR/OmniParser/utils/checkpointer.py:20,44-47
 *                bare state_dict 'module.mgp_str.*'   OCR/MGP-STR/test_final.py:348,356
 *
 * The only native-API precedent in the reference is the two-function iOS library
 * `init_ocr(path, threads)` / `ocr_recognize(data, w, h, c, flag)`
 * (OCR/LiteWeightOCR/.../Headers/LiteWeight_Mobile_OCR_Recognize.h:17-19); this header keeps that
 * shape: init -> load -> run -> free, plain pointers and sizes, no C++ or torch types.
 *
 * Conventions: every function returns 0 or a negative ALM_ERR_* code and never throws across the
 * ABI; `alm_last_error` gives the message.  One `alm_ctx` per GPU per thread (no internal locking).
 * All kernels are enqueued on the context's stream.  Inputs are caller-owned (host or device
 * pointers are both accepted: host buffers are staged through pinned memory inside the call);
 * outputs are written to caller-provided host buffers after a stream synchronise.
 */
#ifndef ALM_OCR_H_
#define ALM_OCR_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define ALM_API __attribute__((visibility("default")))
#else
#define ALM_API
#endif

#define ALM_OK 0
#define ALM_ERR_INVALID (-1)   /* bad argument / missing tensor / shape mismatch          */
#define ALM_ERR_CUDA (-2)      /* CUDA runtime or driver error (message has the call)      */
#define ALM_ERR_OOM (-3)       /* workspace arena or weight slab exhausted                 */
#define ALM_ERR_STATE (-4)     /* call order violated (e.g. decode before encode)          */
#define ALM_ERR_UNSUPPORTED (-5)

typedef struct alm_ctx alm_ctx;

/* model kinds for alm_load_weights */
#define ALM_MODEL_OMNI_SPOT 1 /* OmniParser text spotting (V = 1104)                         */
#define ALM_MODEL_OMNI_KIE 2  /* OmniParser KIE: V = 1104 + vie_categories (derived from V) */
#define ALM_MODEL_MGPSTR 3    /* MGP-STR (dim/depth/heads derived from the tensors)          */

/* element types of alm_tensor_desc.data */
#define ALM_F32 0
#define ALM_F16 1
#define ALM_BF16 2
#define ALM_I64 3

/* One state-dict entry.  `name` is the reference key verbatim
 * (e.g. "backbone.0.layers.2.blocks.5.attn.qkv.weight", "module.mgp_str.blocks.0.norm1.bias").
 * `data` is a HOST pointer (or NULL: shape-only placeholder, see alm_load_weights); the library converts and uploads,
 * the caller keeps ownership. */
typedef struct alm_tensor_desc {
  const char* name;
  const void* data;
  int dtype;
  int ndim;
  int64_t shape[4];
} alm_tensor_desc;

/* ---- lifecycle ---------------------------------------------------------------------------- */
/* device: CUDA ordinal.  stream: a cudaStream_t to enqueue on, or NULL for a private stream. */
ALM_API int alm_init(int device, void* stream, alm_ctx** out);
ALM_API void alm_free(alm_ctx* ctx);
ALM_API const char* alm_last_error(const alm_ctx* ctx); /* valid until the next call on ctx */
ALM_API const char* alm_version(void);

/* options: "nsplit" (3 = bf16x3 split operands, fp32-class results [default]; 1 = single-pass bf16),
 *          "gemm_impl" (0 = tcgen05 [default], 1 = SIMT debug kernel), "workspace_mb", "profile_gemm",
 *          "trace_gemm" (capacity; see alm_trace_read), "trace_detail" (see alm_bench_gemm_ex),
 *          "fuse_ln_gemv" (point loop: 1 = every pre-LayerNorm runs inside the GEMV that consumes it, 13 fewer dependent
 *          launches per token [default]; 0 = separate LayerNorm launches),
 *          "kv_decoders" (3 = alm_omni_encode fills the cross-attention K/V caches of the pt, poly and rec decoders
 *          [default]; 1 = only the point decoder's, for callers that run alm_omni_decode_points alone),
 *          "attn_impl" (ViT attention of MGP-STR: 0 = fused tcgen05 kernel, scores / probabilities in tensor memory
 *          [default]; 1 = score GEMM + softmax + P.V GEMM, the A/B reference),
 *          "wattn_impl" (0 = mma.sync window attention, one CTA per (window, head), 1 = fp32 SIMT debug kernel, 2 = tcgen05 kernel with
 *          TMA-staged window tiles, two windows per M = 128 tile, scores / probabilities in tensor memory, 3 = persistent
 *          mma.sync kernel fed by a TMA + mbarrier ring, one head pair per 128-byte row segment, bias in shared memory [default]),
 *          "small_grid_cap" (0 = off [default]; n = small GEMM launches use at most n CTAs so that concurrent
 *          streams / in-flight batches can share the GPU),
 *          "gemm_plain_epilogue" (2 = map-free GEMM launches use the slim epilogue specialisation and, when the only output is
 *          an unbatched split-bf16 matrix, its TMA-store form [default]; 1 = slim only; 0 = generic),
 *          "wide_tiles" (1 = 128x256 GEMM tiles for large problems [default], 0 = 128x128 only),
 *          "decode_streams" (2 = polygon and recognition loops overlap on two streams [default], 1 = serial),
 *          "use_graphs" (1 = replay captured CUDA graphs for the per-token decode steps [default], 0 = eager),
 *          "xattn_impl" (0 = fused flash-style decoder cross-attention [default]; 1 = unfused score GEMM + softmax +
 *          P.V GEMM / fp32 single-query kernel, the A/B reference -- must be set before alm_omni_encode; 2 = the mma.sync
 *          kernel with a TMA + mbarrier operand ring; 3 = tcgen05 kernel: 128-key TMA ring, scores / probabilities in
 *          tensor memory, running output in registers),
 *          "xattn_ctas_per_sm" (persistent grid of the fused cross-attention: 1..3 CTAs per SM, default 2),
 *          "sattn_wide" (1 = CTA per (sequence, head) self-attention step when few sequences are live [default]),
 *          "enc_grid_cap" / "dec_grid_cap" (0 = off [default]; n = GEMM launches of alm_omni_encode / of the decode
 *          loops use at most n CTAs), "decode_priority" (1 = decode loops run on internal high-priority streams;
 *          default 0) -- co-scheduling knobs for several contexts on one GPU,
 *          "debug_skip" (timing experiments only: bit mask of decoder-layer kernel classes NOT launched; results
 *          are garbage; default 0). */
ALM_API int alm_set_option(alm_ctx* ctx, const char* key, long value);
/* block until everything enqueued on the context's stream has finished */
ALM_API int alm_synchronize(alm_ctx* ctx);
/* kernels launched on this context since the last call with reset != 0 */
ALM_API long alm_launch_count(alm_ctx* ctx, int reset);

/* Per-GEMM device timing (measurement aid, off by default): after alm_set_option(ctx, "profile_gemm", 1) every
 * tensor-core GEMM launch is bracketed by CUDA events on the context stream.  alm_profile_read synchronises,
 * returns the summed kernel time (ms), the summed algorithmic FLOPs (2*M*N*K) and the launch count, and clears. */
ALM_API int alm_profile_read(alm_ctx* ctx, double* gemm_ms, double* gemm_flops, long* gemm_launches);
/* In-kernel GEMM timeline (measurement aid): after alm_set_option(ctx, "trace_gemm", capacity) CTA 0 of every
 * tcgen05 GEMM stamps %globaltimer at entry and exit.  Records are 6 x u64: start ns, end ns, M, N, K,
 * tiles*1000 + BLOCK_N.  Works inside graph replays.  Reading clears the buffer. */
ALM_API int alm_trace_read(alm_ctx* ctx, unsigned long long* out, int max_records, int* n_records);
/* Times `iters` back-to-back launches of one [M,K]x[N,K]^T GEMM (operands pre-split, resident) with CUDA events
 * on the context stream; ms_per_launch is the average kernel duration. */
ALM_API int alm_bench_gemm(alm_ctx* ctx, int M, int N, int K, int iters, float* ms_per_launch);
/* Replay cost (microseconds per node) of a captured chain of `nodes` trivial dependent kernels. */
ALM_API int alm_bench_graph_floor(alm_ctx* ctx, int nodes, int iters, float* us_per_node);
/* Same, batched, with a choice of epilogue (split_out: bf16 hi/lo output; act: 0/1/2).  With the "trace_detail" option
 * on, detail_out receives 64 x 6 u64 stamps of CTA 0's first tiles: TMA issue, MMA tile start, operands landed,
 * MMA committed, epilogue start, epilogue end (ns, %globaltimer). */
ALM_API int alm_bench_gemm_ex(alm_ctx* ctx, int M, int N, int K, int batch, int split_out, int act, int iters,
                              float* ms_per_launch, unsigned long long* detail_out);

/* Replaces reference `model.load_state_dict(torch.load(path)['model'])`
 * (OCR/OmniParser/utils/checkpointer.py:44-47; OCR/MGP-STR/test_final.py:353-356). */
ALM_API int alm_load_weights(alm_ctx* ctx, int model_kind, const alm_tensor_desc* tensors, int n);
/* A descriptor with data == NULL is a shape-only placeholder: the tensor is laid out (zeros) exactly as if it had been
 * loaded, and its values arrive later through alm_broadcast_weights -- what the non-root ranks of a multi-GPU job do. */

/* One model, many execution contexts: `ctx` (same device as `owner`) serves the weights already resident in `owner`
 * -- no copy, the device slabs are reference-counted and freed with the last context using them.  Per-batch state
 * (arena, K/V caches, captured graphs, stream) stays private to each context, so contexts can run concurrently from
 * different host threads.  Replaces the reference's one-module-per-process shape (OCR/OmniParser/model/__init__.py:7-19)
 * for serving several batches in flight per GPU. */
ALM_API int alm_share_weights(alm_ctx* ctx, alm_ctx* owner);

/* Stream ordering for device-resident inputs / outputs.  The context enqueues on its own stream (alm_init), which is
 * NOT ordered with the caller's streams: before passing device buffers written on `producer_stream` call
 * alm_stream_wait (the context's stream waits for everything enqueued on producer_stream so far); before reading
 * device outputs (alm_pre_*) on `consumer_stream` call alm_stream_release.  Host buffers need neither. */
ALM_API int alm_stream_wait(alm_ctx* ctx, void* producer_stream /* cudaStream_t */);
ALM_API int alm_stream_release(alm_ctx* ctx, void* consumer_stream /* cudaStream_t */);

/* ---- multi-GPU (SURVEY.md 8b/8e): pages shard across GPUs with no data-path collective ------- */
/* The reference has no inference collective (its NCCL use is DDP training, OCR/OmniParser/utils/dist.py:25,43-44);
 * a data-parallel serving job needs two: ONE broadcast of the weights at start-up and ONE gather of the decoded
 * sequences per batch.  NCCL is bound at run time (dlopen libnccl.so.2); ALM_ERR_UNSUPPORTED if it is absent.
 *   rank 0: alm_comm_unique_id(id) -> ship the 128 bytes to the other ranks by any means (file, socket, MPI, ...)
 *   all   : alm_comm_init(ctx, id, rank, world)        (or alm_comm_attach with a communicator the caller owns)
 *   all   : alm_load_weights (root: real tensors; others: shape-only placeholders), then alm_broadcast_weights(ctx, 0):
 *           the converted bf16 hi/lo planes and fp32 vectors travel once over NVLink straight into place
 *   batch : alm_gather_sequences(ctx, buf, bytes, recv): all-gather of one fixed-size packed buffer per rank
 *           (send: host or device; recv: host, world * bytes, rank-major, or NULL), on the context's stream.
 * With world == 1 (no communicator) broadcast is a no-op and gather a copy.
 * Several contexts of one process (each with its own communicator) must issue their collectives in ONE order that is the
 * same on every rank -- NCCL's rule for multiple communicators: a gather kernel spins on the device until its peers arrive,
 * and two ranks that start different contexts' gathers first can block each other for good.  Number the batches the same
 * way on every rank and issue gather(batch s) only after gather(batch s - 1) returned (dist.CollectiveOrder in the Python
 * adapter; a mutex + counter in a C host). */
ALM_API int alm_comm_unique_id(void* id128);
ALM_API int alm_comm_init(alm_ctx* ctx, const void* id128, int rank, int world);
ALM_API int alm_comm_attach(alm_ctx* ctx, void* nccl_comm /* ncclComm_t, caller-owned */, int rank, int world);
ALM_API int alm_broadcast_weights(alm_ctx* ctx, int root);
ALM_API int alm_gather_sequences(alm_ctx* ctx, const void* send, size_t bytes_per_rank, void* recv_host);

/* ---- OmniParser ---------------------------------------------------------------------------- */
/* Vocabulary / decode configuration: OCR/OmniParser/utils/parser.py:16-21,91-103. */
typedef struct alm_decode_cfg {
  int num_bins;       /* 1000 */
  int pt_eos, poly_eos, rec_eos, pt_sos, poly_sos, rec_sos, recog_pad;
  int pt_seq_length;  /* --pt_seq_length : max generated pt tokens                           */
  int rec_length;     /* --rec_length    : 25                                                */
  int poly_length;    /* 32 (transformer.py:254)                                             */
  int vie_categories; /* 0 for text spotting                                                 */
  int max_instances;  /* capacity of the per-image output buffers (>= pt_seq_length / 2)      */
} alm_decode_cfg;

/* Replaces `features, pos = self.backbone(samples)`, FPN and input_proj
 * (OCR/OmniParser/model/omniparser.py:20-31): Swin-B encoder -> FPN -> 1x1 stride-2 projection.
 * img  : f32 [B,3,H,W] normalised pixels (NestedTensor.tensors), host or device.
 * mask : u8  [B,H,W], 1 = padding (NestedTensor.mask), host or device, or NULL for all-valid.
 * The image memory ([B, M, 512], M = ceil(H/16)*ceil(W/16)) stays resident in the context. */
ALM_API int alm_omni_encode(alm_ctx* ctx, const float* img, const uint8_t* mask, int B, int H, int W);

/* Staged-parity readbacks (host buffers).
 * level 0..3 : LN'd Swin stage outputs, NHWC f32 [B, S_l, S_l', 128<<l]  (joiner.py:10-18)
 * which 0 = memory [B,M,512], 1 = sine position embedding [B,M,512]       (position_embedding.py:24-44) */
ALM_API int alm_omni_get_feature(alm_ctx* ctx, int level, float* out, size_t out_elems);
ALM_API int alm_omni_get_memory(alm_ctx* ctx, int which, float* out, size_t out_elems);
ALM_API int alm_omni_memory_shape(alm_ctx* ctx, int* B, int* h, int* w);

/* Replaces `self.transformer(self.input_proj(src), mask, pos, sequence)` in eval mode
 * (OCR/OmniParser/model/transformer.py:234-286): greedy point / polygon / recognition decoding for
 * every encoded image, each image keeping the reference's batch-1 semantics.
 * pt_prompt: int64 [n_prompt] (engine/val.py:25-28).  Outputs (host), per image b:
 *   n_inst[b]                         number of decoded points (0 <=> the reference returns None)
 *   pt  [b, max_inst, 2]   int64      transformer.py:134-141
 *   poly[b, max_inst, 32]  int64      transformer.py:265
 *   rec [b, max_inst, rec_length]     transformer.py:284
 *   rec_prob [b, max_inst, rec_length] f32   transformer.py:286 */
ALM_API int alm_omni_decode(alm_ctx* ctx, const int64_t* pt_prompt, int n_prompt, const alm_decode_cfg* cfg, int32_t* n_inst,
                    int64_t* pt, int64_t* poly, int64_t* rec, float* rec_prob);

/* The point loop alone: `decode_pt_seq` (transformer.py:102-141) for every encoded image -- the structure / layout
 * sequence decoders built on this model (the unreleased table-recognition head, OCR/OmniParser/README.md:85-101) run
 * exactly this loop for hundreds of tokens.  Outputs (host), per image b: n_tok[b] generated tokens (prompt stripped,
 * a trailing odd token dropped as in :138-139), pt_tokens[b, pt_seq_length] int64, pt_probs[b, pt_seq_length] f32
 * (may be NULL).  max_instances / poly_length of cfg are ignored. */
ALM_API int alm_omni_decode_points(alm_ctx* ctx, const int64_t* pt_prompt, int n_prompt, const alm_decode_cfg* cfg,
                                   int32_t* n_tok, int64_t* pt_tokens, float* pt_probs);

/* Window-prompted text spotting: R pt prompts per encoded image, decoded over ONE encode (the encoder, FPN and
 * cross-attention K/V of an image serve all its prompts).  A prompt is [x0, y0, x1, y1, char_lo, char_hi, pt_sos] (or
 * the 5-token form without the character window): a spatial window in bins and a character window in class ids, as the
 * model is trained (dataset/collate_fn.py:46-115).  Each (image b, prompt r) is exactly what alm_omni_decode returns
 * for that image under that prompt: every prompt ends at its own EOS, and the polygon / recognition loops of an image
 * take the points of all its prompts at once.  Tiling a page into R windows also lifts the 509-point cap of one point
 * sequence (the 1024-row position table) to R x 509.
 * prompts: int64 [B][R][n_prompt] (B = images of the last alm_omni_encode), 1 <= R <= 16, 1 <= n_prompt <= 16, every id
 * in [0, V).  Outputs (host), per (image b, prompt r), max_inst = cfg->max_instances per prompt:
 *   n_inst [B][R]; pt [B][R][max_inst][2]; poly [B][R][max_inst][32];
 *   rec / rec_prob [B][R][max_inst][rec_length]
 * Text-spotting checkpoints only: a KIE checkpoint returns ALM_ERR_UNSUPPORTED. */
ALM_API int alm_omni_decode_prompted(alm_ctx* ctx, const int64_t* prompts, int R, int n_prompt, const alm_decode_cfg* cfg,
                                     int32_t* n_inst, int64_t* pt, int64_t* poly, int64_t* rec, float* rec_prob);
/* The point loop alone under R prompts per image: n_tok [B][R], pt_tokens / pt_probs [B][R][pt_seq_length] (pt_probs may
 * be NULL), each (b, r) exactly what alm_omni_decode_points returns for that prompt. */
ALM_API int alm_omni_decode_points_prompted(alm_ctx* ctx, const int64_t* prompts, int R, int n_prompt,
                                            const alm_decode_cfg* cfg, int32_t* n_tok, int64_t* pt_tokens,
                                            float* pt_probs);

/* KIE variant (--infer_vie): replaces the eval branch with `decode_vie_pt_poly_rec_seq` (transformer.py:143-217,243-246).
 * The pt loop emits (x, y, class) triples (:117-123) with the class slot restricted to the last vie_categories
 * ids; every (x, y) pair found by the reference's walk (:148-210) gets a polygon and a transcription whose
 * softmax runs over the first V - vie_categories logits (:156,176).  Outputs (host), per image b:
 *   n_tok[b]; pt_tokens[b, pt_seq_length] int64 and pt_probs[b, pt_seq_length] f32 (prompt stripped, :132-141);
 *   n_inst[b]; inst_pos[b, max_inst] = index in pt_tokens where the pair starts;
 *   poly[b, max_inst, 32], rec[b, max_inst, rec_length], rec_prob[b, max_inst, rec_length].
 * The entity grouping / class names / rectangles (:163-169,190-215) are plain host post-processing over these. */
ALM_API int alm_omni_decode_kie(alm_ctx* ctx, const int64_t* pt_prompt, int n_prompt, const alm_decode_cfg* cfg,
                                int32_t* n_tok, int64_t* pt_tokens, float* pt_probs, int32_t* n_inst, int32_t* inst_pos,
                                int64_t* poly, int64_t* rec, float* rec_prob);

/* Teacher-forced logits: replaces `Transformer.decode(input_seq, memory, mask, pos_embed, input_type)`
 * (transformer.py:74-100) for image `image`: seq int64 [n_seq, len] -> logits f32 [n_seq, len, V].
 * kind: 0 = pt, 1 = poly, 2 = rec. */
ALM_API int alm_omni_decode_logits(alm_ctx* ctx, int image, int kind, const int64_t* seq, int n_seq, int len, float* logits);
ALM_API int alm_omni_vocab(alm_ctx* ctx);
/* Device time (CUDA events on the context stream) of the last alm_omni_encode and of the two halves of the last
 * decode: the point loop, and the polygon + recognition loops (incl. the host round trip between them); -1 = n/a. */
ALM_API int alm_omni_last_timing(alm_ctx* ctx, float* encode_ms, float* pt_ms, float* polyrec_ms);

/* ---- MGP-STR ------------------------------------------------------------------------------- */
/* Replaces `model(image, is_eval=True)` (OCR/MGP-STR/modules/mgp_str.py:96-101).
 * img: f32 [B,3,32,128] in [0,1].  Any output pointer may be NULL.  Host buffers:
 *   attn   [3][B,27,257] f32 (char, bpe, wp A^3 maps)
 *   char_logits [B,27,38], bpe_logits [B,27,50257], wp_logits [B,27,30522]  f32
 *   ids    [3][B,27] int32 top-1 ids, prob [3][B,27] f32 max softmax prob (demo.py:36-60).
 * The model variant comes from the checkpoint: tiny / small / base / large (embed 192 / 384 / 768 / 1024, 64-wide heads,
 * mgp_str.py:176-230) and the char-only CHAR-STR ablation (modules/char_str.py:43-81: one A^3 module, logits through
 * timm's `head`).  For CHAR-STR only the first plane of attn / ids / prob and char_logits are written; the class
 * counts of the heads (the widths of the logit buffers) are reported by alm_mgpstr_info. */
ALM_API int alm_mgpstr_info(alm_ctx* ctx, int* dim, int* depth, int* heads, int* n_a3, int* vocab3 /*[3]*/);
ALM_API int alm_mgpstr_forward(alm_ctx* ctx, const float* img, int B, float* attn, float* char_logits, float* bpe_logits,
                       float* wp_logits, int32_t* ids, float* prob);

/* ---- low-level ops (unit parity tests call these through the ABI; device pointers only) ------ */
/* C[M,N] f32 = A[M,K] f32 * W[N,K]^T f32 (+bias[N]) with act 0 none / 1 gelu(erf) / 2 relu; runs the same
 * operand split + tcgen05 kernel as the model graphs.  batch > 1: contiguous batches of A, W and C. */
ALM_API int alm_op_linear(alm_ctx* ctx, const float* A, const float* W, const float* bias, float* C, int M, int N, int K,
                  int act, int batch);
/* softmax((q k^T) * 64^-0.5) v for B sequences of T <= 272 tokens and H heads of width 64: qkv f32 [B*T, 3*H*64] (q | k | v
 * column blocks, head h at columns h*64 of its block: the layout of timm's packed qkv Linear), out f32 [B*T, H*64].
 * Runs the fused tcgen05 kernel of the ViT blocks (scores and probabilities stay in tensor memory). */
ALM_API int alm_op_attention(alm_ctx* ctx, const float* qkv, float* out, int B, int T, int H);
ALM_API int alm_op_layernorm(alm_ctx* ctx, const float* x, const float* gamma, const float* beta, float eps, float* y,
                     long rows, int C);
/* Swin W-MSA core on an already windowed qkv tensor [B*nWh*nWw*49, 3C] (swin_transformer.py:127-148). */
ALM_API int alm_op_window_attention(alm_ctx* ctx, const float* qkv, const float* bias_table /*[169,heads]*/, float* out,
                            int B, int nWh, int nWw, int C, int heads, int shift);

/* Kernels of the OmniParser decode step.  Every call synchronises before it returns. */
/* Skinny exact-fp32 linear of the decode loops (M <= 64 rows, K <= 512 or K in {1024, 1536, 2048}):
 *   out[m*ldo + n] = act(xin[m*ldx + 0..K) . W[n*K + 0..K) + bias[n]) (+ resid[m*ldr + n]),  act 0 none / 1 gelu / 2 relu
 * with xin = x for the columns n < n_split and x2 (NULL: x) for the rest.  ln_g / ln_b non-NULL (K == 512): the rows are
 * LayerNorm'd (eps ln_eps) first, and pos[0..512) is added to them for the columns n < pos_split.  bias / resid / pos may
 * be NULL; n_split, pos_split and every stride are multiples of 4. */
ALM_API int alm_op_gemv(alm_ctx* ctx, const float* x, const float* x2, int n_split, long ldx, const float* W, const float* bias,
                        const float* resid, long ldr, float* out, long ldo, int M, int N, int K, int act, const float* ln_g,
                        const float* ln_b, float ln_eps, const float* pos, int pos_split);
/* Cached self-attention step at position t (host int, 0 <= t < Tmax <= 1024) for S sequences x 8 heads of width 64:
 * appends k = qk[s*ld_qk + 512 .. 1024) and v = vnew[s*ld_v + 0 .. 512) as row t of kc / vc ([S][Tmax][512] fp32), then
 * out[s] = softmax((q / 8) . kc[s][0..t]^T) vc[s][0..t] with q = qk[s*ld_qk + 0 .. 512).  out_f32 [S][512] and the split
 * bf16 pair out_hi / out_lo (bits, [S][512]) may each be NULL.  The "sattn_wide" option picks the kernel as in the model. */
ALM_API int alm_op_self_attn_step(alm_ctx* ctx, const float* qk, int ld_qk, const float* vnew, int ld_v, float* kc, float* vc,
                                  int S, int t, int Tmax, float* out_f32, uint16_t* out_hi, uint16_t* out_lo);
/* Decoder cross-attention of nimg images x Ncap queries against decoder-layer slot dl (0..11) of a K/V cache of B
 * images: out[i*Ncap + n][h*64 + d] = softmax((q_n / 8) . K_{img0+i,h}^T, keys with kpm != 0 excluded) V_{img0+i,h}.
 * q f32 [nimg*Ncap][512]; k, v f32 [B][8][M][64] (images img0 .. img0+nimg-1 are read); kpm u8 [B][M] or NULL.  The call
 * lays the cache out as alm_omni_encode does, every slice it must not read filled with NaN, and runs the kernel the
 * "xattn_impl" option selects for this shape, as the decode loops do.  q_split 1: the queries are split to bf16 hi / lo
 * first (polygon / recognition loops).  out f32 [nimg*Ncap][512]. */
ALM_API int alm_op_cross_attention(alm_ctx* ctx, const float* q, const float* k, const float* v, const uint8_t* kpm, int B,
                                   int img0, int nimg, int Ncap, int M, int dl, int q_split, float* out);
/* Greedy head step of the decode loops at position t: for each of S rows of logits [S][V], the top-1 of the candidate
 * classes of `phase` (0 = point loop, whose mode follows the generated index t - n_prompt_m1; 1 = polygon; 2 =
 * recognition), its softmax probability over the first nsoft logits; writes tokens[s*tstride + t + 1] and
 * probs[s*pstride + t - n_prompt_m1] (probs may be NULL).  finished / ntok ([S] int32, both or neither): EOS bookkeeping
 * of the point loop. */
ALM_API int alm_op_head_select(alm_ctx* ctx, const float* logits, int S, int V, int nsoft, int phase, const alm_decode_cfg* cfg,
                               int t, int n_prompt_m1, int32_t* tokens, int tstride, float* probs, int pstride,
                               int32_t* finished, int32_t* ntok);

/* ---- test-time image pipeline on the GPU (SURVEY 8f rank 1) ----------------------------------- */
/* Replaces RandomResize([test_min_size], test_max_size) -> ToTensor -> Normalize -> nested_tensor_from_tensor_list
 * (OCR/OmniParser/dataset/__init__.py:109-113, dataset/transforms.py:249-298,312-322, utils/nested_tensor.py:37-54)
 * for a batch of decoded 8-bit RGB pages.  The resize is Pillow's two-pass 8-bit bilinear resampling, reproduced bit
 * for bit (integer kernels; weights computed like Pillow computes them); ToTensor / Normalize are the same float32
 * operations, so tensors and mask equal the reference's.
 * alm_pre_omni_plan (host only): resized (h, w) per page = get_size_with_aspect_ratio, and the batch canvas.
 * alm_pre_omni_pages: rgb[i] = host or device pointer to page i, [heights[i]][widths[i]][3] uint8.  Outputs are
 * DEVICE buffers sized from the plan: tensors f32 [n,3,Hmax,Wmax] (zero padded), mask u8 [n,Hmax,Wmax] (1 = pad);
 * they feed alm_omni_encode directly. */
ALM_API int alm_pre_omni_plan(const int* heights, const int* widths, int n, int test_min_size, int test_max_size,
                              int* sizes /*[n][2] resized h, w*/, int* Hmax, int* Wmax);
/* Introspection (host only): the 22-bit fixed-point weights of ONE resampling pass exactly as the kernels use them
 * (filter 0 = bilinear, 1 = bicubic): bounds [out_size][2] = (first source index, taps), coefs [out_size][*ksize].
 * Call with coefs == NULL to obtain *ksize first (returns ALM_ERR_INVALID after storing it). */
ALM_API int alm_pre_coeffs(int in_size, int out_size, int filter, int* ksize, int* bounds, int* coefs, size_t cap_ints);
ALM_API int alm_pre_omni_pages(alm_ctx* ctx, const uint8_t* const* rgb, const int* heights, const int* widths, int n,
                               int test_min_size, int test_max_size, float* tensors, uint8_t* mask);
/* Replaces `img.resize((imgW, imgH), Image.BICUBIC)` + ToTensor (OCR/MGP-STR/demo.py:126-132, dataset.py:459-461):
 * out = DEVICE f32 [n,3,imgH,imgW] in [0,1], the input of alm_mgpstr_forward. */
ALM_API int alm_pre_mgp_crops(alm_ctx* ctx, const uint8_t* const* rgb, const int* heights, const int* widths, int n,
                              int imgH, int imgW, float* out);

/* ---- post-processing (host only: no context, no GPU; SURVEY 8f rank 2) ------------------------ */
/* Sequences -> structured result, the step right after the forward.  Errors: negative ALM_ERR_*; the message of
 * the last failing call of the calling thread is returned by alm_post_last_error(). */
ALM_API const char* alm_post_last_error(void);

/* Replaces decode_pred_seq + decode_seq (OCR/OmniParser/engine/val.py:70-100, utils/misc.py:147-189) for ONE image:
 *   pt [2*n] / poly [32*n] / rec [n*rec_length] int64 ids and rec_prob [n*rec_length] f32 as returned by
 *   alm_omni_decode (one row of its outputs); chars = args.chars as UTF-8 (one code point per class id
 *   num_bins + i); orig_h / orig_w = target['orig_size'].
 * Outputs (caller buffers): pts [n,2] and polys [n,32] doubles holding the reference's float32 values
 * (id / num_bins * size, both steps rounded to f32 like the torch expressions), scores [n] doubles
 * (sum(p) / (len + 1e-5) in double), texts: n NUL-terminated UTF-8 strings at stride text_stride bytes. */
ALM_API int alm_post_omni_spotting(const int64_t* pt, const int64_t* poly, const int64_t* rec, const float* rec_prob, int n,
                                   int rec_length, int num_bins, int recog_pad_index, int rec_eos_index, const char* chars,
                                   long orig_h, long orig_w, double* pts, double* polys, double* scores, char* texts,
                                   size_t text_stride);
/* The same results as the JSON text `json.dumps(results, indent=4)` writes for this image (val.py:63-67; keys
 * image_id, pts, score, polys, rec; Python float repr; ensure_ascii escapes).  Writes at most cap bytes incl. NUL
 * and always stores the needed size (incl. NUL) in *needed; returns ALM_ERR_INVALID if cap is too small. */
ALM_API int alm_post_omni_json(const int64_t* pt, const int64_t* poly, const int64_t* rec, const float* rec_prob, int n,
                               int rec_length, int num_bins, int recog_pad_index, int rec_eos_index, const char* chars,
                               long orig_h, long orig_w, const char* image_id, char* json, size_t cap, size_t* needed);

/* KIE: the entity walk of decode_vie_pt_poly_rec_seq (OCR/OmniParser/model/transformer.py:148-215) over ONE image's
 * outputs of alm_omni_decode_kie (tokens / probs [n_tok], inst_pos [n_inst], poly [n_inst,32], rec [n_inst,rec_length]),
 * written as the JSON text `json.dump(output, f)` stores (engine/val.py:38-42):
 * [[text, class_name, prob, [[x0, y0, x1, y1], ...]], ...].  classes[i] names token id class_base + i
 * (class_base = padding_index + 1, transformer.py:54-61).  Size protocol as alm_post_omni_json. */
ALM_API int alm_post_omni_kie_json(const int64_t* tokens, const float* probs, int n_tok, const int32_t* inst_pos, int n_inst,
                                   const int64_t* poly, const int64_t* rec, int rec_length, int num_bins,
                                   int recog_pad_index, int rec_eos_index, const char* chars, const char* const* classes,
                                   int n_classes, int class_base, long orig_h, long orig_w, char* json, size_t cap,
                                   size_t* needed);

/* MGP-STR A^3 fusion (OCR/MGP-STR/test_final.py:176-240, demo.py:36-112, utils.py:52-87) for B crops.
 *   ids / prob: [3][B,T] int32 top-1 ids and f32 max-softmax probabilities of the char, bpe and wp heads INCLUDING
 *   position 0 (exactly what alm_mgpstr_forward returns; T = 27).
 *   tables: token strings per id, UTF-8 -- char: ['[GO]', '[s]'] + opt.character; bpe: the byte-decoded GPT-2 token
 *   strings; wp: the WordPiece tokens of bert-base-uncased.  (The reference obtains them from the HuggingFace
 *   tokenizers; they are data, passed in by the caller.)
 * Per crop and head: text (pruned at the end-of-sentence marker the way the reference prunes it -- string find of
 * '[s]' / '#' / '[SEP]', including its -1 quirk) and confidence = cumprod of the max-probs up to the EOS position
 * (first id 1 / 2 / 102 for char / bpe / wp; char uses the STRING index like the reference); fused = the head with
 * the largest confidence (strictly greater, in char, bpe, wp order; none if all are 0).
 * Outputs: texts [3][B] and fused [B] strings at stride text_stride; conf [3][B] f32; source [B] int32 (0 char, 1 bpe,
 * 2 wp, -1 none). */
ALM_API int alm_post_mgp_fuse(const int32_t* ids, const float* prob, int B, int T, const char* const* char_table, int n_char,
                              const char* const* bpe_table, int n_bpe, const char* const* wp_table, int n_wp, char* texts,
                              char* fused, size_t text_stride, float* conf, int32_t* source);

#ifdef __cplusplus
}
#endif
#endif /* ALM_OCR_H_ */
