/*
 * parseq_b200.h - C ABI of the B200-native PARSeq inference engine (libparseq_b200.so).
 *
 * The reference (baudm/parseq) has no FFI / plugin boundary for this path: it sits behind the Python
 * class strhub.models.parseq.system.PARSeq (system.py:33-88) wrapping the nn.Module
 * strhub.models.parseq.model.PARSeq (model.py:31-169).  Each entry point below states the reference
 * method it replaces.  All pointers are plain device or host pointers; no torch types cross this
 * boundary.  All functions return 0 on success and a negative parseq_status on failure;
 * parseq_last_error() returns a human-readable message for the calling thread's last failure.
 *
 * Threading / streams: an engine handle is NOT thread-safe (one handle per device and stream user).
 * All work is enqueued on the caller's stream; the only host synchronisation is inside
 * parseq_forward_host (which must return host-visible results) and parseq_finalize.
 */
#ifndef PARSEQ_B200_H_
#define PARSEQ_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct parseq_engine parseq_engine;
typedef void* parseq_stream_t;           /* cudaStream_t */

typedef enum parseq_status {
  PARSEQ_OK = 0,
  PARSEQ_ERR_INVALID_ARG = -1,
  PARSEQ_ERR_UNSUPPORTED = -2,           /* configuration outside what the kernels cover */
  PARSEQ_ERR_CUDA = -3,
  PARSEQ_ERR_STATE = -4,                 /* e.g. forward before finalize, missing weight */
  PARSEQ_ERR_NO_DEVICE = -5              /* no sm_100 device: there is NO CPU fallback */
} parseq_status;

/* Architecture hyper-parameters: the ctor arguments of model.PARSeq (model.py:33-49) /
 * system.PARSeq (system.py:35-60).  num_tokens = len(tokenizer) = charset + EOS + BOS + PAD. */
typedef struct parseq_config {
  int32_t img_h, img_w;                  /* img_size     */
  int32_t patch_h, patch_w;              /* patch_size   */
  int32_t embed_dim;
  int32_t enc_num_heads, enc_mlp_ratio, enc_depth;
  int32_t dec_num_heads, dec_mlp_ratio, dec_depth;   /* dec_depth must be 1 (all reference configs) */
  int32_t max_label_length;              /* 25 -> 26 decode positions */
  int32_t num_tokens;                    /* 97: EOS=0, chars 1..94, BOS=95, PAD=96 (data/utils.py:102-111) */
  int32_t max_batch;                     /* images per super-chunk / CUDA graph (workspace sizing); 0 = 512 */
  int32_t device;                        /* CUDA device ordinal */
  int32_t arch;                          /* 0: PARSeq (parseq/model.py); 1: ViTSTR (vitstr/model.py:14-28: the same ViT with
                                          * a class token and a per-token head; the dec_* fields are ignored) */
} parseq_config;

/* Replaces model.PARSeq.__init__ (model.py:33-71): allocates device weights + workspace.
 * arch = 1 replaces vitstr/system.py:50-59 (ViTSTR(VisionTransformer) ctor): state_dict keys are then those of the
 * timm ViT itself ("cls_token", "pos_embed" [1, T+1, D], "patch_embed.proj.*", "blocks.<i>.*", "norm.*", "head.*");
 * parseq_forward* ignore decode_ar / refine_iters and return vitstr/system.py:65-71: head(norm(x))[:, 1 : max_length+2]
 * as logits [N, num_steps, num_tokens-2]; parseq_encode returns forward_features [N, T+1, D]. */
int parseq_create(const parseq_config* cfg, parseq_engine** out);
void parseq_destroy(parseq_engine* e);

/* Replaces model.PARSeq.load_state_dict as used by strhub/models/utils.py:80-82: `key` is a
 * state_dict key of the inner model (e.g. "encoder.blocks.3.attn.qkv.weight",
 * "decoder.layers.0.cross_attn.in_proj_weight", "pos_queries"); `data` is a HOST pointer to `numel`
 * contiguous fp32 values in PyTorch layout.  GEMM weight matrices are rounded to bf16 on upload. */
int parseq_set_weight(parseq_engine* e, const char* key, const float* data, int64_t numel);
/* Number of state_dict keys the engine expects, and the i-th key / its element count. */
int parseq_num_weights(const parseq_engine* e);
const char* parseq_weight_key(const parseq_engine* e, int i, int64_t* numel);

/* Input-independent precomputation (content K/V table over (position, token), query projections
 * of pos_queries); must be called after all weights are set and after any weight update. */
int parseq_finalize(parseq_engine* e, parseq_stream_t stream);

/* Decode options of one forward call: model.PARSeq.forward(tokenizer, images, max_length)
 * (model.py:105-169) with the module attributes decode_ar / refine_iters (model.py:55-56). */
typedef struct parseq_forward_args {
  int32_t batch;                         /* N images */
  int32_t max_length;                    /* -1 = None ("testing": early-exit length reported in *steps) */
  int32_t decode_ar;                     /* 0 / 1 */
  int32_t refine_iters;
  /* Optional teacher forcing (debug / parity): device int32 [batch, num_steps]; AR step i feeds
   * forced_ids[:, i+1] instead of its own argmax.  NULL in production. */
  const int32_t* forced_ids;
  /* Optional: device int32 [refine_iters, batch, num_steps] contexts (BOS included) for the cloze passes. */
  const int32_t* forced_refine;
} parseq_forward_args;

/* Replaces system.PARSeq.forward -> model.PARSeq.forward (system.py:87-88, model.py:105-169).
 *   images : DEVICE fp32 [N,3,H,W] (NCHW, values as produced by T.Normalize(0.5,0.5))
 *   logits : DEVICE fp32 [N, num_steps, num_tokens-2], num_steps = min(max_length,25)+1 (26 if -1)
 *   ids    : DEVICE int32 [N, num_steps] argmax of `logits` (may be NULL)
 *   steps  : DEVICE int32 [1] (may be NULL): S = number of AR steps the reference would have run
 *            before its batch-wide early exit (model.py:144); == num_steps when max_length >= 0,
 *            when decode_ar == 0.  Only affects the returned SHAPE when refine_iters == 0. */
int parseq_forward(parseq_engine* e, const parseq_forward_args* args, const float* images,
                   float* logits, int32_t* ids, int32_t* steps, parseq_stream_t stream);

/* End-to-end variant with HOST buffers (pinned or pageable): H2D of images, forward, D2H of
 * logits / ids / steps, synchronised on return.  This is what bench.py times as `e2e`. */
int parseq_forward_host(parseq_engine* e, const parseq_forward_args* args, const float* images_host,
                        float* logits_host, int32_t* ids_host, int32_t* steps_host,
                        parseq_stream_t stream);

/* "Next" rows of the path (SURVEY.md section 8f).
 * Raw-crop input: images uint8 [N, H, W, 3] (HWC, as PIL / numpy hold them, already resized to img_size); the reference's
 * T.ToTensor() + T.Normalize(0.5, 0.5) (strhub/data/module.py:68-82) is folded into the patch gather.  Device / host
 * variants mirror parseq_forward / parseq_forward_host.  Crops of any size go through parseq_forward_crops below. */
int parseq_forward_u8(parseq_engine* e, const parseq_forward_args* args, const uint8_t* images_hwc,
                      float* logits, int32_t* ids, int32_t* steps, parseq_stream_t stream);
int parseq_forward_host_u8(parseq_engine* e, const parseq_forward_args* args, const uint8_t* images_hwc_host,
                           float* logits_host, int32_t* ids_host, int32_t* steps_host, parseq_stream_t stream);

/* Variable-size RGB uint8 crops: the reference's whole input transform (strhub/data/module.py:69-82, read.py)
 *   [img.rotate(rotation, expand=True)] -> T.Resize(img_size, BICUBIC) -> T.ToTensor() -> T.Normalize(0.5, 0.5)
 * on the GPU.  The resize is bit-exact with PIL's bicubic resampler (what torchvision's Resize runs on PIL images), so
 * the result is bit-identical to parseq_forward_u8 on the PIL-resized stack, for any batch.
 * A crop is `height` rows of 3 * `width` bytes (R, G, B per pixel), row i starting at byte offset + i * row_stride of
 * `pixels`; row_stride >= 3 * width, so a crop can be a view into a larger frame.  Each side is 1..4096 pixels; every
 * crop must lie inside [0, pixels_bytes).  Anything else returns PARSEQ_ERR_INVALID_ARG before any work is enqueued. */
typedef struct parseq_crop {
  int64_t offset;
  int32_t height, width, row_stride;
  int32_t reserved;                      /* 0 */
} parseq_crop;
typedef struct parseq_crops {
  int32_t count;                         /* == args->batch */
  const parseq_crop* desc;               /* HOST array [count]; may be reused as soon as the call returns */
  const uint8_t* pixels;                 /* packed RGB bytes: DEVICE for parseq_forward_crops, HOST for the _host variant */
  int64_t pixels_bytes;                  /* the host variant uploads all of [0, pixels_bytes) */
  int32_t rotation;                      /* 0, 90, 180, 270: counter-clockwise, expand=True (read.py / test.py --rotation) */
} parseq_crops;
int parseq_forward_crops(parseq_engine* e, const parseq_forward_args* args, const parseq_crops* crops, float* logits,
                         int32_t* ids, int32_t* steps, parseq_stream_t stream);
int parseq_forward_host_crops(parseq_engine* e, const parseq_forward_args* args, const parseq_crops* crops,
                              float* logits_host, int32_t* ids_host, int32_t* steps_host, parseq_stream_t stream);
/* The resize alone: out_hwc DEVICE uint8 [count, img_h, img_w, 3] (the input of parseq_forward_u8); crops->pixels is
 * DEVICE.  Needs no weights. */
int parseq_resize_crops(parseq_engine* e, const parseq_crops* crops, uint8_t* out_hwc, parseq_stream_t stream);
/* Fused post-processing of BaseSystem._eval_step (strhub/models/base.py:132-142) + Tokenizer._filter
 * (strhub/data/utils.py:120-129): DEVICE logits [N, num_steps, num_classes] -> ids [N, num_steps] (greedy), lengths [N]
 * (index of the first EOS, num_steps if none) and confidence [N] (product of the max softmax probabilities up to and
 * including the EOS position). */
int parseq_postprocess(const float* logits, int32_t batch, int32_t num_steps, int32_t num_classes, int32_t eos_id,
                       int32_t* ids, int32_t* lengths, float* confidence, parseq_stream_t stream);

/* Replaces model.PARSeq.encode (model.py:83-84): memory DEVICE fp32 [N, T, D]. */
int parseq_encode(parseq_engine* e, int32_t batch, const float* images, float* memory,
                  parseq_stream_t stream);

/* Replaces model.PARSeq.decode (strhub/models/parseq/model.py:86-103 -> modules.py:55-125, depth-1 decoder: query stream
 * only): tgt DEVICE int32 [N, J] context ids (tgt[:, 0] = BOS; token k >= 1 receives pos_queries[k-1], model.py:96-99),
 * memory DEVICE fp32 [N, T, D] (what parseq_encode returns), query DEVICE fp32 [N, NQ, D] or NULL (= pos_queries[:NQ],
 * model.py:100-101), query_mask DEVICE uint8 [NQ, J] or NULL (1 = key masked for that query: the bool `tgt_query_mask`),
 * padding_mask DEVICE uint8 [N, J] or NULL (`tgt_padding_mask`); out DEVICE fp32 [N, NQ, D] = Decoder output including
 * the final LayerNorm (modules.py:123-125).  1 <= J, NQ <= max_label_length + 1.  A query whose keys are all masked
 * yields NaN, as the reference's softmax does.  `tgt_mask` (content stream) has no effect at decoder depth 1. */
int parseq_decode(parseq_engine* e, int32_t batch, int32_t ctx_len, int32_t num_queries, const int32_t* tgt,
                  const float* memory, const float* query, const uint8_t* query_mask, const uint8_t* padding_mask,
                  float* out, parseq_stream_t stream);
/* Replaces model.PARSeq.head (model.py:63: nn.Linear(embed_dim, num_tokens - 2)): x DEVICE fp32 [rows, D] ->
 * logits DEVICE fp32 [rows, num_tokens - 2] (bf16 tensor-core operands, fp32 accumulate). */
int parseq_head(parseq_engine* e, int32_t rows, const float* x, float* logits, parseq_stream_t stream);
/* Replaces TokenEmbedding.forward (modules.py:175-176): out[i, :] = sqrt(D) * embedding[ids[i], :], DEVICE fp32 [n, D]. */
int parseq_text_embed(parseq_engine* e, int32_t n, const int32_t* ids, float* out, parseq_stream_t stream);

/* Introspection used by bench.py / tests. */
int64_t parseq_kernel_launches(const parseq_engine* e);      /* cumulative count of kernels launched */
/* Microbenchmark of the AR kernel's TMA ring (tests/bench_tma_stream.py): `ctas` CTAs in clusters of `cluster` stream `nboxes`
 * 16 KB boxes each from `buf` through `nslot` slots, no compute. */
int parseq_bench_tma_stream(void* buf, int64_t bytes, int cluster, int ctas, int nboxes, int nslot, int mode, void* sink,
                            parseq_stream_t stream);
/* Debug counters by name ("ar2_occupancy_mt2", "ar2_clusters_mt2", "ar_last_per", "ar_last_clusters", "sm_count"); -1 if unknown. */
int64_t parseq_debug_int(parseq_engine* e, const char* name);
/* Options: "max_batch" (images per super-chunk = one CUDA graph), "chunk" (images per encoder pass inside a
 * super-chunk), "dec_chunk" (images per decoder chain; the chains of a super-chunk run concurrently on their own
 * streams), "use_graph" (0/1), "pdl" (programmatic dependent launch, 0/1), "timing" (1: record a CUDA-event pair around every launch
 * for parseq_get_timing; 0: off + clear), "block_n" (engine-independent GEMM tile override, tests), "fuse_ln" (bit 0: the attention-projection GEMM, bit 1: the fc2 GEMM
 * also produces the LayerNorm that follows it, used when the batch fills the machine at least twice with 128-row tiles; bit 2:
 * for any batch; default 3; 0: separate LayerNorm kernels), "ar_kernel" (AR loop: 2 = cluster-owned persistent kernel,
 * default; 1 = grid-barrier persistent kernel; 0 = chain of separate kernels), "fuse_mlp" (1: fc1 + GELU + fc2 + residual +
 * LayerNorm of an encoder block in one kernel where fuse_ln bit 1 applies - bit-identical results, slower on B200, default 0),
 * "attn_impl", "cta_group" / "ln_cta_group" / "mlp_cta_group" (0 auto, 1 single CTA, 2 CTA pair: GEMM / fused GEMM+LayerNorm /
 * one-kernel MLP), "ln_split" (fused GEMM+LayerNorm: 0 auto = the column-split CTA-pair kernel for K >= 768, 1 never, 2 always),
 * "pair_pdl", "gemm_stages", "tma_epilogue" (kernel-variant switches for tests).  Options are PER HANDLE; with
 * e == NULL the launch options (block_n, attn_impl, pdl, tma_epilogue, gemm_stages, cta_group, ln_cta_group, mlp_cta_group,
 * ln_split, pair_pdl) set the process defaults that the stand-alone kernel
 * entry points below use and that handles created afterwards inherit. */
int parseq_set_option(parseq_engine* e, const char* name, int64_t value);
/* After a synchronised forward with "timing"=1: device milliseconds, algorithmic FLOPs and launch count of
 * category 0 encoder GEMM, 1 encoder attention, 2 LayerNorm, 3 decoder GEMM, 4 decoder attention, 5 other,
 * 6 encoder residual GEMM fused with LayerNorm, 7 persistent AR-loop kernel. */
int parseq_get_timing(parseq_engine* e, int category, double* ms, double* flops, int64_t* count);
/* Debug: after a forward with option "ar_prof"=1, copies the [32 steps][16 slots] globaltimer (ns) stamps that block 0 of
 * the persistent AR kernel recorded at its phase boundaries. */
int parseq_get_ar_profile(parseq_engine* e, uint64_t* out512);
const char* parseq_last_error(void);
const char* parseq_version(void);

/* Stand-alone kernel entry points (unit tests of the building blocks; all pointers DEVICE). */
/* C[M,N] = epilogue(A[M,K](bf16,row-major,lda) * W[N,K]^T(bf16,row-major,ldw) + bias) on tcgen05.
 * mode: 0 -> fp32 out (alpha*(acc+bias) [+ resid[row % resid_mod or row]]), 1 -> bf16 out,
 *       2 -> bf16 gelu(acc+bias). */
int parseq_gemm_bf16(const void* A, int64_t lda, const void* W, int64_t ldw, const float* bias,
                     int M, int N, int K, int mode, float alpha, const float* resid, int64_t ldr,
                     int resid_mod, void* out, int64_t ldo, parseq_stream_t stream);
/* Residual GEMM fused with the LayerNorm that follows it (timm Block: x = x + proj(attn) ; norm2(x) and
 * x = x + fc2(..) ; next norm1(x)):  x_inout[M, D] += A[M, K] * W[D, K]^T + bias (fp32, in place),
 * xn_bf16[M, D] = bf16(LayerNorm(x_inout; gamma, beta, eps)).  D in {192, 384}. */
int parseq_gemm_ln_bf16(const void* A, int64_t lda, const void* W, int64_t ldw, const float* bias,
                        int M, int D, int K, float* x_inout, const float* gamma, const float* beta,
                        float eps, void* xn_bf16, parseq_stream_t stream);
/* The whole MLP of a timm Block + the LayerNorm that follows (x = x + fc2(GELU(fc1(norm2(x)))) ; next norm1(x)) in one
 * kernel: x_inout[M, D] += GELU(xn[M, D] * W1[4D, D]^T + b1) * W2[D, 4D]^T + b2 (fp32, in place; the bf16 hidden activation
 * stays on the SM), xn_out_bf16[M, D] = bf16(LayerNorm(x_inout; gamma, beta, eps)); xn_out_bf16 may alias xn.  D in {192, 384}. */
int parseq_mlp_ln_bf16(const void* xn, const void* W1, const float* b1, const void* W2, const float* b2,
                       int M, int D, float* x_inout, const float* gamma, const float* beta, float eps,
                       void* xn_out_bf16, parseq_stream_t stream);
/* Same with cycle counters of CTA 0 (16 x uint64, device) for tests/prof_mlp_ln.py. */
int parseq_mlp_ln_bf16_prof(const void* xn, const void* W1, const float* b1, const void* W2, const float* b2,
                            int M, int D, float* x_inout, const float* gamma, const float* beta, float eps,
                            void* xn_out_bf16, unsigned long long* prof_dev, parseq_stream_t stream);
/* y = bf16(LayerNorm(x; gamma, beta, eps)), x fp32 [M, D]. */
int parseq_layernorm_bf16(const float* x, const float* gamma, const float* beta, float eps, int M,
                          int D, void* y_bf16, float* y_f32_or_null, parseq_stream_t stream);
/* out[B*T, D] = softmax(QK^T/sqrt(64)) V per (image, head) from packed qkv bf16 [B*T, 3D]. */
int parseq_enc_attention(const void* qkv_bf16, int B, int T, int D, int heads, void* out_bf16,
                         parseq_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* PARSEQ_B200_H_ */
