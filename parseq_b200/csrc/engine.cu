// libparseq_b200.so: host-side engine + C ABI (include/parseq_b200.h) of the B200-native PARSeq
// inference path.  Restates, as a fixed kernel schedule on one CUDA stream, what
// strhub/models/parseq/model.py:105-169 (PARSeq.forward: encode, AR loop, NAR, cloze refinement)
// does through nn.Module calls.  There is no CPU path: without an sm_100 device creation fails.
#include <cuda.h>
#include <cuda_runtime.h>

#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <string>
#include <vector>

#include "../../include/parseq_b200.h"
#include "gemm.cuh"
#include "kernels.cuh"
#include "dec_ar.cuh"
#include "dec_ar2.cuh"
#include "attn_tc.cuh"
#include "gemm_ln.cuh"
#include "gemm_ln2.cuh"
#include "mlp_ln.cuh"
#include "resize.cuh"

namespace {

thread_local std::string g_last_error;

int fail(int code, const std::string& msg) {
  g_last_error = msg;
  return code;
}
#define PQ_CUDA(expr)                                                                              \
  do {                                                                                             \
    cudaError_t _e = (expr);                                                                       \
    if (_e != cudaSuccess)                                                                         \
      return fail(PARSEQ_ERR_CUDA, std::string(#expr) + " -> " + cudaGetErrorString(_e));          \
  } while (0)
#define PQ_TRY(expr)                 \
  do {                               \
    int _r = (expr);                 \
    if (_r != PARSEQ_OK) return _r;  \
  } while (0)

// ---------------------------------------------------------------- driver entry point for TMA descriptors
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
PFN_encodeTiled g_encode = nullptr;

int load_driver_api() {
  if (g_encode != nullptr) return PARSEQ_OK;
  void* fn = nullptr;
  cudaDriverEntryPointQueryResult qres;
  cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres);
  if (e != cudaSuccess || fn == nullptr || qres != cudaDriverEntryPointSuccess)
    return fail(PARSEQ_ERR_CUDA, "cuTensorMapEncodeTiled not available from the driver");
  g_encode = reinterpret_cast<PFN_encodeTiled>(fn);
  return PARSEQ_OK;
}

// 2D tensor map: rows x cols (cols contiguous), row stride ld elements, box = box_rows x box_cols (box_cols * esize
// = 128 B), 128B swizzle.  esize 2 = bf16, 4 = fp32.
int make_tmap(CUtensorMap* tm, const void* ptr, int esize, long long rows, long long cols, long long ld, int box_cols,
              int box_rows) {
  PQ_TRY(load_driver_api());
  if ((reinterpret_cast<uintptr_t>(ptr) & 15u) != 0 || ((ld * esize) & 15) != 0)
    return fail(PARSEQ_ERR_INVALID_ARG, "GEMM operand must be 16-byte aligned with a 16-byte multiple row stride");
  cuuint64_t dims[2] = {static_cast<cuuint64_t>(cols), static_cast<cuuint64_t>(rows)};
  cuuint64_t strides[1] = {static_cast<cuuint64_t>(ld) * static_cast<cuuint64_t>(esize)};
  cuuint32_t box[2] = {static_cast<cuuint32_t>(box_cols), static_cast<cuuint32_t>(box_rows)};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = g_encode(tm, esize == 2 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2,
                        const_cast<void*>(ptr), dims, strides, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(PARSEQ_ERR_CUDA, "cuTensorMapEncodeTiled failed: " + std::to_string(int(r)));
  return PARSEQ_OK;
}

// 3D bf16 tensor map [d2][d1][d0] (d0 contiguous), strides in elements, box = box_d0 x box_d1 x 1, 128B swizzle:
// the decoder's cross K/V cache viewed as [image][key][2D] (keys past T read as zeros).
int make_tmap3d(CUtensorMap* tm, const void* ptr, long long d0, long long d1, long long d2, long long ld1, long long ld2,
                int box_d0, int box_d1) {
  PQ_TRY(load_driver_api());
  if ((reinterpret_cast<uintptr_t>(ptr) & 15u) != 0 || ((ld1 * 2) & 15) != 0 || ((ld2 * 2) & 15) != 0)
    return fail(PARSEQ_ERR_INVALID_ARG, "tensor map operand must be 16-byte aligned with 16-byte multiple strides");
  cuuint64_t dims[3] = {static_cast<cuuint64_t>(d0), static_cast<cuuint64_t>(d1), static_cast<cuuint64_t>(d2)};
  cuuint64_t strides[2] = {static_cast<cuuint64_t>(ld1) * 2u, static_cast<cuuint64_t>(ld2) * 2u};
  cuuint32_t box[3] = {static_cast<cuuint32_t>(box_d0), static_cast<cuuint32_t>(box_d1), 1u};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = g_encode(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(ptr), dims, strides, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(PARSEQ_ERR_CUDA, "cuTensorMapEncodeTiled(3d) failed: " + std::to_string(int(r)));
  return PARSEQ_OK;
}

uint16_t f32_to_bf16_rne(float f) {
  uint32_t u;
  std::memcpy(&u, &f, 4);
  if ((u & 0x7fffffffu) > 0x7f800000u) return static_cast<uint16_t>((u >> 16) | 0x40u);  // NaN
  u += 0x7fffu + ((u >> 16) & 1u);
  return static_cast<uint16_t>(u >> 16);
}

// Launch options.  Every engine handle owns one (parseq_set_option(handle, ...)); `g_default_opts` serves only the
// bare kernel exports (parseq_gemm_bf16 & co., unit tests) and parseq_set_option(NULL, ...).
struct LaunchOpts {
  int sm_count = 0;
  bool use_pdl = true;          // programmatic dependent launch on every kernel of the forward chain
  int block_n = 0;              // 0 = auto
  int cta_group = 0;            // 0 = auto, 1 / 2 = forced (tests)
  int ln_cta_group = 0;         // same for the fused GEMM + LayerNorm kernel
  int ln_split = 0;             // fused GEMM + LayerNorm: 2 = column-split CTA-pair kernel (gemm_ln2.cuh), 0 / 1 = gemm_ln.cuh
  int mlp_cta_group = 0;        // one-kernel MLP (mlp_ln.cuh): 0 = auto (pairs), 1 / 2 = forced
  bool pair_pdl = false;        // experiments: programmatic dependent launch also on CTA-pair (cluster) launches
  bool no_tma_epilogue = false; // tests: force the direct-store epilogue
  int gemm_stages = 0;          // experiments: cap the operand ring depth (0 = full)
  int attn_impl = 1;            // 1: tcgen05 kernel (attn_tc.cuh), 0: mma.sync kernel (kernels.cuh)
};
LaunchOpts g_default_opts;

int ensure_sm_count(LaunchOpts& o) {
  if (o.sm_count == 0) {
    int dev = 0;
    PQ_CUDA(cudaGetDevice(&dev));
    PQ_CUDA(cudaDeviceGetAttribute(&o.sm_count, cudaDevAttrMultiProcessorCount, dev));
  }
  return PARSEQ_OK;
}

// cudaLaunchKernelEx wrapper: optional PDL attribute (the kernels call griddepcontrol.{launch_dependents,wait}).
template <typename... KArgs, typename... Args>
int launch_k(const LaunchOpts& lo, void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = lo.use_pdl ? 1 : 0;
  PQ_CUDA(cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...));
  return PARSEQ_OK;
}

template <int BN, int CG>
int launch_gemm_cfg(const LaunchOpts& lo, const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& tc,
                    const pq::GemmParams& p, int tiles, cudaStream_t st) {
  auto kern = pq::gemm_bf16_tcgen05_kernel<BN, CG>;
  using Cfg = pq::GemmCfg<BN, CG>;
  static bool attr_set = false;
  if (!attr_set) {
    PQ_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmemBytes));
    attr_set = true;
  }
  const int max_groups = lo.sm_count / CG;
  const int groups = tiles < max_groups ? tiles : max_groups;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(static_cast<unsigned>(groups * CG));
  cfg.blockDim = dim3(pq::GEMM_THREADS);
  cfg.dynamicSmemBytes = Cfg::kSmemBytes;
  cfg.stream = st;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CG;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = (lo.use_pdl && (CG == 1 || lo.pair_pdl)) ? 2 : 1;
  PQ_CUDA(cudaLaunchKernelEx(&cfg, kern, ta, tb, tc, p));
  return PARSEQ_OK;
}

// instantiate + set the smem attribute of every configuration outside of any stream capture
template <int BN, int CG>
int warm_gemm_cfg() {
  return cudaFuncSetAttribute(pq::gemm_bf16_tcgen05_kernel<BN, CG>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                              pq::GemmCfg<BN, CG>::kSmemBytes) == cudaSuccess ? PARSEQ_OK
                                                                                : fail(PARSEQ_ERR_CUDA, "cudaFuncSetAttribute(gemm)");
}
size_t head_smem_bytes(int C, int D) {
  return ((static_cast<size_t>(C) * (D / 2 + 1) * 4 + 15) / 16) * 16 + static_cast<size_t>(pq::HEAD_ROWS) * D * 4 +
         4 * pq::HEAD_ROWS * 128 * 4 + pq::HEAD_ROWS * 128 * 4;
}
int ln_head_argmax_launch(const LaunchOpts& lo, const float* y, const float* g, const float* b, float eps, const __nv_bfloat16* Wh, const float* bh,
                          int M, int C, int D, float* logits, long long logits_ld, int* ids, int ids_ld, int nq, int dst_off,
                          const int* forced, int forced_ld, cudaStream_t st) {
  if (C > 128) return fail(PARSEQ_ERR_UNSUPPORTED, "head kernel covers at most 128 classes");
  const dim3 grid((M + pq::HEAD_ROWS - 1) / pq::HEAD_ROWS), block(384);
  const size_t sm = head_smem_bytes(C, D);
  switch (D) {
    case 192: return launch_k(lo, pq::dec_ln_head_argmax_kernel<192>, grid, block, sm, st, y, g, b, eps, Wh, bh, M, C, logits,
                              logits_ld, ids, ids_ld, nq, dst_off, forced, forced_ld);
    case 384: return launch_k(lo, pq::dec_ln_head_argmax_kernel<384>, grid, block, sm, st, y, g, b, eps, Wh, bh, M, C, logits,
                              logits_ld, ids, ids_ld, nq, dst_off, forced, forced_ld);
    case 768: return launch_k(lo, pq::dec_ln_head_argmax_kernel<768>, grid, block, sm, st, y, g, b, eps, Wh, bh, M, C, logits,
                              logits_ld, ids, ids_ld, nq, dst_off, forced, forced_ld);
    default: return fail(PARSEQ_ERR_UNSUPPORTED, "head kernel: embed_dim must be 192, 384 or 768");
  }
}

template <int D, int MT, int CS>
int ar2_attr() {
  PQ_CUDA(cudaFuncSetAttribute(pq::dec_ar2_kernel<D, MT, CS>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                               static_cast<int>(pq::dec_ar2_smem_bytes<D, MT, CS>())));
  if constexpr (MT == 1 && CS == 8 && D / 64 <= CS)      // head-split variant for tiny batches
    PQ_CUDA(cudaFuncSetAttribute(pq::dec_ar2_kernel<D, MT, CS, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 static_cast<int>(pq::dec_ar2_smem_bytes<D, MT, CS>())));
  return PARSEQ_OK;
}
int ar2_set_attributes() {
  PQ_TRY((ar2_attr<192, 1, 8>())); PQ_TRY((ar2_attr<192, 2, 8>())); PQ_TRY((ar2_attr<384, 1, 8>())); PQ_TRY((ar2_attr<384, 2, 8>()));
  PQ_TRY((ar2_attr<768, 1, 8>()));
  PQ_TRY((ar2_attr<192, 1, 6>())); PQ_TRY((ar2_attr<192, 2, 6>())); PQ_TRY((ar2_attr<384, 1, 6>())); PQ_TRY((ar2_attr<384, 2, 6>()));
  PQ_TRY((ar2_attr<768, 1, 6>()));
  return PARSEQ_OK;
}

int init_kernel_attributes() {
  PQ_CUDA(cudaFuncSetAttribute(pq::enc_attention_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, pq::ATC_SMEM_BYTES));
  PQ_CUDA(cudaFuncSetAttribute(pq::dec_ar_kernel<192, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(pq::dec_ar_smem_bytes<192>())));
  PQ_CUDA(cudaFuncSetAttribute(pq::dec_ar_kernel<192, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(pq::dec_ar_smem_bytes<192>())));
  PQ_CUDA(cudaFuncSetAttribute(pq::dec_ar_kernel<384, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(pq::dec_ar_smem_bytes<384>())));
  PQ_CUDA(cudaFuncSetAttribute(pq::dec_ar_kernel<384, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(pq::dec_ar_smem_bytes<384>())));
  PQ_CUDA(cudaFuncSetAttribute(pq::dec_ar_kernel<768, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(pq::dec_ar_smem_bytes<768>())));
  PQ_CUDA(cudaFuncSetAttribute(pq::dec_ar_kernel<768, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(pq::dec_ar_smem_bytes<768>())));
  PQ_TRY(ar2_set_attributes());
  PQ_CUDA(cudaFuncSetAttribute(pq::dec_ln_head_argmax_kernel<192>, cudaFuncAttributeMaxDynamicSharedMemorySize, 120 * 1024));
  PQ_CUDA(cudaFuncSetAttribute(pq::dec_ln_head_argmax_kernel<384>, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024));
  PQ_CUDA(cudaFuncSetAttribute(pq::dec_ln_head_argmax_kernel<768>, cudaFuncAttributeMaxDynamicSharedMemorySize, 226 * 1024));
  PQ_CUDA(cudaFuncSetAttribute(pq::gemm_ln_fused_kernel<192, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, pq::GemmLnCfg<192, 1>::kSmemBytes));
  PQ_CUDA(cudaFuncSetAttribute(pq::gemm_ln_fused_kernel<384, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, pq::GemmLnCfg<384, 1>::kSmemBytes));
  PQ_CUDA(cudaFuncSetAttribute(pq::gemm_ln_fused_kernel<192, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, pq::GemmLnCfg<192, 2>::kSmemBytes));
  PQ_CUDA(cudaFuncSetAttribute(pq::gemm_ln_fused_kernel<384, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, pq::GemmLnCfg<384, 2>::kSmemBytes));
  PQ_CUDA(cudaFuncSetAttribute(pq::gemm_ln_split_kernel<384>, cudaFuncAttributeMaxDynamicSharedMemorySize, pq::GemmLn2Cfg<384>::kSmemBytes));
  PQ_CUDA(cudaFuncSetAttribute(pq::mlp_ln_fused_kernel<192, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, pq::MlpLnCfg<192, 1>::kSmemBytes));
  PQ_CUDA(cudaFuncSetAttribute(pq::mlp_ln_fused_kernel<384, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, pq::MlpLnCfg<384, 1>::kSmemBytes));
  PQ_CUDA(cudaFuncSetAttribute(pq::mlp_ln_fused_kernel<192, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, pq::MlpLnCfg<192, 2>::kSmemBytes));
  PQ_CUDA(cudaFuncSetAttribute(pq::mlp_ln_fused_kernel<384, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, pq::MlpLnCfg<384, 2>::kSmemBytes));
  PQ_TRY((warm_gemm_cfg<64, 1>()));
  PQ_TRY((warm_gemm_cfg<128, 1>()));
  PQ_TRY((warm_gemm_cfg<192, 1>()));
  PQ_TRY((warm_gemm_cfg<256, 1>()));
  PQ_TRY((warm_gemm_cfg<128, 2>()));
  PQ_TRY((warm_gemm_cfg<192, 2>()));
  PQ_TRY((warm_gemm_cfg<256, 2>()));
  return PARSEQ_OK;
}

// blocked_rows > 0: `out` is a column-blocked bf16 buffer [N/64][blocked_rows][64] (ptx.cuh: blocked_off); ldo is ignored
int gemm_launch(LaunchOpts& lo, const void* A, long long lda, const void* W, long long ldw, const float* bias, int M, int N,
                int K, int mode, float alpha, const float* resid, long long ldr, int resid_mod, void* out, long long ldo,
                cudaStream_t st, long long blocked_rows = 0) {
  if (M <= 0 || N <= 0 || K <= 0) return fail(PARSEQ_ERR_INVALID_ARG, "gemm: empty problem");
  PQ_TRY(ensure_sm_count(lo));
  // Tile choice from tests/bench_gemm.py on B200 (profiles/r1_gemm_microbench*.txt): single-CTA 128 x 256 tiles win
  // for the wide projections (QKV 1152 -> 4.5 tiles, fc1 1536), 128 x 192 for N = 384 / 768 (no padded columns),
  // 128 x 128 for the small decoder GEMMs.
  // CTA pairs (cta_group::2: each CTA holds half of the W tile) win once the main loop is long enough to amortise the
  // pair's per-tile handshakes: measured (profiles/r2_gemm_cta_pair_sweep.txt) 0.81 - 0.98x the single-CTA time for
  // K >= 768 (D = 768 configs, unfused fc2), 1.05 - 1.21x for K = 384.  The accumulation order per output element is the
  // same, so the choice does not change a single bit of the result (test_cta_pair_rows_equal_single_cta_rows).
  int CG = (K >= 768 && M >= 1024) ? 2 : 1;
  if (lo.cta_group) CG = lo.cta_group;
  int BN;
  if (CG == 2) BN = (N % 256 == 0) ? 256 : (N % 192 == 0) ? 192 : 128;
  else BN = (N <= 64) ? 64 : (M < 1024) ? 128 : (N >= 1024) ? 256 : (N % 192 == 0) ? 192 : 128;
  if (lo.block_n) {
    BN = lo.block_n;
    if (CG == 2 && BN == 64) BN = 128;
  }
  CUtensorMap ta, tb, tc;
  PQ_TRY(make_tmap(&ta, A, 2, M, K, lda, pq::GEMM_BLOCK_K, pq::GEMM_BLOCK_M));
  PQ_TRY(make_tmap(&tb, W, 2, N, K, ldw, pq::GEMM_BLOCK_K, BN / CG));
  pq::GemmParams p;
  p.M = M; p.N = N; p.K = K; p.mode = mode; p.alpha = alpha; p.bias = bias;
  p.resid = resid; p.ldr = ldr; p.resid_mod = resid_mod; p.out = out; p.ldo = ldo;
  const int esz = (mode == pq::EPI_F32) ? 4 : 2;
  bool vec = ((reinterpret_cast<uintptr_t>(out) & 15u) == 0) && ((ldo * esz) % 16 == 0);
  if (resid != nullptr) vec = vec && ((reinterpret_cast<uintptr_t>(resid) & 15u) == 0) && ((ldr * 4) % 16 == 0);
  if (bias != nullptr) vec = vec && ((reinterpret_cast<uintptr_t>(bias) & 15u) == 0);
  p.vec_ok = vec ? 1 : 0;
  // asynchronous TMA epilogue whenever the output is TMA-addressable; residual only as in-place accumulate
  p.tma_out = 0;
  const bool out_ok = ((reinterpret_cast<uintptr_t>(out) & 15u) == 0) && ((ldo * esz) % 16 == 0) && !lo.no_tma_epilogue;
  if (out_ok) {
    if (mode != pq::EPI_F32) p.tma_out = 3;
    else if (resid == nullptr) p.tma_out = 1;
    else if (resid == out && ldr == ldo && resid_mod == 0) p.tma_out = 2;
  }
  if (blocked_rows > 0) {
    if (mode == pq::EPI_F32 || N % 64 != 0 || blocked_rows < M || (reinterpret_cast<uintptr_t>(out) & 15u) != 0)
      return fail(PARSEQ_ERR_INVALID_ARG, "gemm: blocked output needs a bf16 epilogue, N % 64 == 0 and rows >= M");
    p.tma_out = 4;
    PQ_TRY(make_tmap3d(&tc, out, 64, blocked_rows, N / 64, 64, 64 * blocked_rows, 64, 32));
  } else if (p.tma_out == 3) PQ_TRY(make_tmap(&tc, out, 2, M, N, ldo, 64, 32));
  else if (p.tma_out != 0) PQ_TRY(make_tmap(&tc, out, 4, M, N, ldo, 32, 32));
  else tc = ta;
  const int tile_m = pq::GEMM_BLOCK_M * CG;
  p.max_stages = lo.gemm_stages;
  p.num_m_tiles = (M + tile_m - 1) / tile_m;
  p.num_n_tiles = (N + BN - 1) / BN;
  const int tiles = p.num_m_tiles * p.num_n_tiles;
  if (CG == 2) {
    if (BN == 256) return launch_gemm_cfg<256, 2>(lo, ta, tb, tc, p, tiles, st);
    if (BN == 192) return launch_gemm_cfg<192, 2>(lo, ta, tb, tc, p, tiles, st);
    return launch_gemm_cfg<128, 2>(lo, ta, tb, tc, p, tiles, st);
  }
  if (BN == 256) return launch_gemm_cfg<256, 1>(lo, ta, tb, tc, p, tiles, st);
  if (BN == 192) return launch_gemm_cfg<192, 1>(lo, ta, tb, tc, p, tiles, st);
  if (BN == 64) return launch_gemm_cfg<64, 1>(lo, ta, tb, tc, p, tiles, st);
  return launch_gemm_cfg<128, 1>(lo, ta, tb, tc, p, tiles, st);
}

// x[M, D] += A[M, K] * W[D, K]^T + bias (fp32, in place); xn[M, D] = bf16(LayerNorm(x; gamma, beta, eps))   (gemm_ln.cuh)
bool gemm_ln_supported(int D) { return D == 192 || D == 384; }
template <int D, int CG>
int launch_gemm_ln(const LaunchOpts& lo, const void* A, long long lda, const void* W, long long ldw, const float* bias, int M, int K, float* x,
                   const float* gamma, const float* beta, float eps, void* xn, cudaStream_t st) {
  using Cfg = pq::GemmLnCfg<D, CG>;
  auto kern = pq::gemm_ln_fused_kernel<D, CG>;
  static bool attr_set = false;
  if (!attr_set) {
    PQ_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmemBytes));
    attr_set = true;
  }
  CUtensorMap ta, tb, tx, tn;
  PQ_TRY(make_tmap(&ta, A, 2, M, K, lda, pq::GEMM_BLOCK_K, pq::GEMM_BLOCK_M));
  PQ_TRY(make_tmap(&tb, W, 2, D, K, ldw, pq::GEMM_BLOCK_K, Cfg::kBRows));
  PQ_TRY(make_tmap(&tx, x, 4, M, D, D, 32, 32));
  PQ_TRY(make_tmap(&tn, xn, 2, M, D, D, 64, 32));
  pq::GemmLnParams p;
  p.M = M; p.K = K; p.bias = bias; p.gamma = gamma; p.beta = beta; p.eps = eps;
  const int tile_m = pq::GEMM_BLOCK_M * CG;
  p.num_m_tiles = (M + tile_m - 1) / tile_m;
  const int max_groups = lo.sm_count / CG;
  const int groups = p.num_m_tiles < max_groups ? p.num_m_tiles : max_groups;
  if constexpr (CG == 1) {
    return launch_k(lo, kern, dim3(groups), dim3(pq::GLN_THREADS), Cfg::kSmemBytes, st, ta, tb, tx, tn, p);
  } else {
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(static_cast<unsigned>(groups * CG));
    cfg.blockDim = dim3(pq::GLN_THREADS);
    cfg.dynamicSmemBytes = Cfg::kSmemBytes;
    cfg.stream = st;
    cudaLaunchAttribute attr[2];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = CG;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[1].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = (lo.use_pdl && lo.pair_pdl) ? 2 : 1;
    PQ_CUDA(cudaLaunchKernelEx(&cfg, kern, ta, tb, tx, tn, p));
    return PARSEQ_OK;
  }
}
// version 2 (gemm_ln2.cuh): the columns of a 128-row tile split over a CTA pair, double-buffered TMEM, statistics through DSMEM
int launch_gemm_ln_split(const LaunchOpts& lo, const void* A, long long lda, const void* W, long long ldw, const float* bias, int M, int K,
                         float* x, const float* gamma, const float* beta, float eps, void* xn, cudaStream_t st) {
  constexpr int D = 384;
  using Cfg = pq::GemmLn2Cfg<D>;
  auto kern = pq::gemm_ln_split_kernel<D>;
  static bool attr_set = false;
  if (!attr_set) {
    PQ_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmemBytes));
    attr_set = true;
  }
  CUtensorMap ta, tb, tx, tn;
  PQ_TRY(make_tmap(&ta, A, 2, M, K, lda, pq::GEMM_BLOCK_K, pq::GEMM_BLOCK_M));
  PQ_TRY(make_tmap(&tb, W, 2, D, K, ldw, pq::GEMM_BLOCK_K, Cfg::kN));
  PQ_TRY(make_tmap(&tx, x, 4, M, D, D, 32, 32));
  PQ_TRY(make_tmap(&tn, xn, 2, M, D, D, 64, 32));
  pq::GemmLnParams p;
  p.M = M; p.K = K; p.bias = bias; p.gamma = gamma; p.beta = beta; p.eps = eps;
  p.num_m_tiles = (M + pq::GEMM_BLOCK_M - 1) / pq::GEMM_BLOCK_M;
  const int max_groups = lo.sm_count / 2;
  const int groups = p.num_m_tiles < max_groups ? p.num_m_tiles : max_groups;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(static_cast<unsigned>(groups * 2));
  cfg.blockDim = dim3(pq::GLN_THREADS);
  cfg.dynamicSmemBytes = Cfg::kSmemBytes;
  cfg.stream = st;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = lo.use_pdl ? 2 : 1;
  PQ_CUDA(cudaLaunchKernelEx(&cfg, kern, ta, tb, tx, tn, p));
  return PARSEQ_OK;
}
int gemm_ln_launch(LaunchOpts& lo, const void* A, long long lda, const void* W, long long ldw, const float* bias, int M, int D,
                   int K, float* x, const float* gamma, const float* beta, float eps, void* xn, cudaStream_t st) {
  if (M <= 0 || K <= 0) return fail(PARSEQ_ERR_INVALID_ARG, "gemm_ln: empty problem");
  PQ_TRY(ensure_sm_count(lo));
  PQ_TRY(load_driver_api());
  // CTA pairs stage 30 % fewer operand bytes per row, bit-identical results - and no gain (profiles/r2_gemm_ln_cta_pair.txt:
  // fc2' 124.5 -> 123.7 us, proj' 64.8 -> 71.6 us): this kernel is not operand-ingest bound.  Opt-in ("ln_cta_group").
  // The column-split pair kernel (gemm_ln2.cuh) pays where the MMAs of a tile are long enough to be worth hiding under the
  // previous tile's epilogue: fc2 (K = 1536) 124.6 -> 110.7 us, attn.proj (K = 384) 64.8 -> 68.1 us
  // (profiles/r2_gemm_ln_split_pair.txt).  ln_split: 0 auto (K >= 768), 1 never, 2 always (D = 384).  Where the fused kernels are
  // used at all is decided by the caller from the batch regime (encode_chunk).
  if (D == 384 && (lo.ln_split == 2 || (lo.ln_split == 0 && K >= 768)))   // by K only: a row's bits must not depend on the batch
    return launch_gemm_ln_split(lo, A, lda, W, ldw, bias, M, K, x, gamma, beta, eps, xn, st);
  int CG = 1;
  if (lo.ln_cta_group) CG = lo.ln_cta_group;
  if (CG == 2) {
    if (D == 384) return launch_gemm_ln<384, 2>(lo, A, lda, W, ldw, bias, M, K, x, gamma, beta, eps, xn, st);
    if (D == 192) return launch_gemm_ln<192, 2>(lo, A, lda, W, ldw, bias, M, K, x, gamma, beta, eps, xn, st);
  }
  if (D == 384) return launch_gemm_ln<384, 1>(lo, A, lda, W, ldw, bias, M, K, x, gamma, beta, eps, xn, st);
  if (D == 192) return launch_gemm_ln<192, 1>(lo, A, lda, W, ldw, bias, M, K, x, gamma, beta, eps, xn, st);
  return fail(PARSEQ_ERR_UNSUPPORTED, "gemm_ln: embed_dim must be 192 or 384 (full rows in 512 TMEM columns)");
}

// x[M, D] += GELU(xn W1^T + b1) W2^T + b2 (fp32, in place); xn_out = bf16(LayerNorm(x; gamma, beta, eps))   (mlp_ln.cuh)
template <int D, int CG>
int launch_mlp_ln(const LaunchOpts& lo, const void* xn, const void* W1, const float* b1, const void* W2, const float* b2, int M,
                  float* x, const float* gamma, const float* beta, float eps, void* xn_out, cudaStream_t st, unsigned long long* prof) {
  using Cfg = pq::MlpLnCfg<D, CG>;
  auto kern = pq::mlp_ln_fused_kernel<D, CG>;
  static bool attr_set = false;
  if (!attr_set) {
    PQ_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmemBytes));
    attr_set = true;
  }
  CUtensorMap txn, tw1, tw2, tx, tn;
  PQ_TRY(make_tmap(&txn, xn, 2, M, D, D, pq::GEMM_BLOCK_K, pq::GEMM_BLOCK_M));
  PQ_TRY(make_tmap(&tw1, W1, 2, Cfg::kH, D, D, pq::GEMM_BLOCK_K, Cfg::kW1Rows));
  PQ_TRY(make_tmap(&tw2, W2, 2, D, Cfg::kH, Cfg::kH, pq::GEMM_BLOCK_K, Cfg::kW2Rows));
  PQ_TRY(make_tmap(&tx, x, 4, M, D, D, 32, 32));
  PQ_TRY(make_tmap(&tn, xn_out, 2, M, D, D, 64, 32));
  pq::MlpLnParams p;
  p.M = M; p.b1 = b1; p.b2 = b2; p.gamma = gamma; p.beta = beta; p.eps = eps; p.prof = prof;
  const int tile_m = pq::GEMM_BLOCK_M * CG;
  p.num_m_tiles = (M + tile_m - 1) / tile_m;
  const int max_groups = lo.sm_count / CG;
  const int groups = p.num_m_tiles < max_groups ? p.num_m_tiles : max_groups;
  if constexpr (CG == 1) {
    return launch_k(lo, kern, dim3(groups), dim3(pq::MLP_THREADS), Cfg::kSmemBytes, st, txn, tw1, tw2, tx, tn, p);
  } else {
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(static_cast<unsigned>(groups * CG));
    cfg.blockDim = dim3(pq::MLP_THREADS);
    cfg.dynamicSmemBytes = Cfg::kSmemBytes;
    cfg.stream = st;
    cudaLaunchAttribute attr[2];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = CG;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[1].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = (lo.use_pdl && lo.pair_pdl) ? 2 : 1;
    PQ_CUDA(cudaLaunchKernelEx(&cfg, kern, txn, tw1, tw2, tx, tn, p));
    return PARSEQ_OK;
  }
}
int mlp_ln_launch(LaunchOpts& lo, const void* xn, const void* W1, const float* b1, const void* W2, const float* b2, int M, int D,
                  float* x, const float* gamma, const float* beta, float eps, void* xn_out, cudaStream_t st,
                  unsigned long long* prof = nullptr) {
  if (M <= 0) return fail(PARSEQ_ERR_INVALID_ARG, "mlp_ln: empty problem");
  PQ_TRY(ensure_sm_count(lo));
  PQ_TRY(load_driver_api());
  // CTA pairs stage half of every weight box per CTA: the same ring covers twice as many k-steps (mlp_ln.cuh)
  const int CG = lo.mlp_cta_group ? lo.mlp_cta_group : 2;
  if (CG == 2) {
    if (D == 384) return launch_mlp_ln<384, 2>(lo, xn, W1, b1, W2, b2, M, x, gamma, beta, eps, xn_out, st, prof);
    if (D == 192) return launch_mlp_ln<192, 2>(lo, xn, W1, b1, W2, b2, M, x, gamma, beta, eps, xn_out, st, prof);
  }
  if (D == 384) return launch_mlp_ln<384, 1>(lo, xn, W1, b1, W2, b2, M, x, gamma, beta, eps, xn_out, st, prof);
  if (D == 192) return launch_mlp_ln<192, 1>(lo, xn, W1, b1, W2, b2, M, x, gamma, beta, eps, xn_out, st, prof);
  return fail(PARSEQ_ERR_UNSUPPORTED, "mlp_ln: embed_dim must be 192 or 384 (hidden width 4 * embed_dim)");
}

int layernorm_launch(const LaunchOpts& lo, const float* x, const float* g, const float* b, float eps, int M, int D, void* y, float* y32,
                     cudaStream_t st, const float* add = nullptr, int add_mod = 1, float* xw = nullptr) {
  const int rows_per_block = 8;
  const int grid = (M + rows_per_block - 1) / rows_per_block;
  __nv_bfloat16* yb = reinterpret_cast<__nv_bfloat16*>(y);
  switch (D) {
    case 192: return launch_k(lo, pq::layernorm_kernel<192>, dim3(grid), dim3(256), 0, st, x, g, b, eps, M, yb, y32, add, add_mod, xw);
    case 384: return launch_k(lo, pq::layernorm_kernel<384>, dim3(grid), dim3(256), 0, st, x, g, b, eps, M, yb, y32, add, add_mod, xw);
    case 768: return launch_k(lo, pq::layernorm_kernel<768>, dim3(grid), dim3(256), 0, st, x, g, b, eps, M, yb, y32, add, add_mod, xw);
    default: return fail(PARSEQ_ERR_UNSUPPORTED, "layernorm: embed_dim must be 192, 384 or 768");
  }
}

int enc_attention_launch(const LaunchOpts& lo, const void* qkv, int B, int T, int D, int heads, void* out, cudaStream_t st) {
  if (D != heads * pq::ATT_DH) return fail(PARSEQ_ERR_UNSUPPORTED, "encoder attention kernels cover head_dim=64");
  if (T != pq::ATT_T && lo.attn_impl == 1 && T <= 256) {   // general token count on tcgen05: 3D maps [image][token][channel]
    static bool attr_set2 = false;
    if (!attr_set2) {
      PQ_CUDA(cudaFuncSetAttribute(pq::enc_attention_tc2_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, pq::atc2_smem_bytes<1>()));
      PQ_CUDA(cudaFuncSetAttribute(pq::enc_attention_tc2_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, pq::atc2_smem_bytes<2>()));
      attr_set2 = true;
    }
    CUtensorMap tq, to;
    PQ_TRY(make_tmap3d(&tq, qkv, 3ll * D, T, B, 3ll * D, 3ll * D * T, 64, 128));
    PQ_TRY(make_tmap3d(&to, out, D, T, B, D, 1ll * D * T, 64, 32));
    const dim3 grid(static_cast<unsigned>(B * heads), static_cast<unsigned>((T + 127) / 128));
    if (T <= 128)
      return launch_k(lo, pq::enc_attention_tc2_kernel<1>, grid, dim3(pq::ATC_THREADS), pq::atc2_smem_bytes<1>(), st, tq, to, D, heads, T);
    return launch_k(lo, pq::enc_attention_tc2_kernel<2>, grid, dim3(pq::ATC_THREADS), pq::atc2_smem_bytes<2>(), st, tq, to, D, heads, T);
  }
  if (T != pq::ATT_T) {   // attn_impl = 0: masked two-pass mma.sync kernel (reference implementation of the unit tests)
    return launch_k(lo, pq::enc_attention_any_kernel, dim3(B * heads, (T + pq::ATT_T - 1) / pq::ATT_T), dim3(256), 0, st,
                    reinterpret_cast<const __nv_bfloat16*>(qkv), reinterpret_cast<__nv_bfloat16*>(out), T, D, heads);
  }
  if (lo.attn_impl == 1) {
    static bool attr_set = false;
    if (!attr_set) {
      PQ_CUDA(cudaFuncSetAttribute(pq::enc_attention_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, pq::ATC_SMEM_BYTES));
      attr_set = true;
    }
    CUtensorMap tq, to;
    PQ_TRY(make_tmap(&tq, qkv, 2, static_cast<long long>(B) * T, 3ll * D, 3ll * D, 64, 128));
    PQ_TRY(make_tmap(&to, out, 2, static_cast<long long>(B) * T, D, D, 64, 32));
    return launch_k(lo, pq::enc_attention_tc_kernel, dim3(B * heads), dim3(pq::ATC_THREADS), pq::ATC_SMEM_BYTES, st, tq, to, D, heads);
  }
  return launch_k(lo, pq::enc_attention_kernel, dim3(B * heads), dim3(256), 0, st,
                  reinterpret_cast<const __nv_bfloat16*>(qkv), reinterpret_cast<__nv_bfloat16*>(out), D, heads);
}

struct Slot {
  std::string key;   // internal name (PARSeq state_dict key)
  std::string pub;   // state_dict key of the served architecture (== key for PARSeq; ViTSTR drops the "encoder." prefix)
  long long numel;
  bool bf16;
  void* dev;
  bool set;
};

}  // namespace

struct parseq_engine {
  parseq_config cfg;
  int D, T, Kp, Me, Md, L, V, C, gh, gw, dh_dec;   // T: tokens per image in the encoder (patches + class token if any)
  int arch = 0, Tp = 0;                              // arch 1 = ViTSTR; Tp = gh * gw patches
  std::map<std::string, int> pub_index;
  float* vt_rows = nullptr;                          // ViTSTR tail: gathered token rows [chunk * L, D] fp32
  int chunk;
  std::vector<Slot> slots;
  std::map<std::string, int> index;
  bool finalized = false;
  bool broken = false;                               // workspace could not be (re)allocated: every forward fails
  LaunchOpts lo;                                     // per-handle launch options
  long long launches = 0;
  // optional per-category device timing (bench.py roofline pass; off on the throughput pass)
  bool timing = false;
  struct TimedLaunch { int cat; double flops; cudaEvent_t a, b; };
  std::vector<TimedLaunch> timed;
  std::vector<cudaEvent_t> event_pool;
  int cur_cat = 5;
  // derived tables
  __nv_bfloat16* kvtab = nullptr;   // [L*V, 2D]
  float* qs = nullptr;              // [L, D]
  // encoder workspace (one pipeline stage = `chunk` images; the encoder runs serialised on `main`)
  __nv_bfloat16 *a_pe = nullptr, *xn = nullptr, *qkv = nullptr, *att = nullptr, *hid = nullptr;
  float* x = nullptr;
  // per-stage decoder state: the decoder of stage s runs on its own stream while `main` encodes stage s+1
  __nv_bfloat16 *mem = nullptr, *ckv = nullptr;   // [max_batch*T, D] encoder output, [max_batch*T, 2D] cross K/V
  int dec_chunk = 128;              // images per decoder chain (each chain runs on its own stream)
  // persistent AR-loop kernel state (whole super-chunk)
  bool use_ar_kernel = true;
  int ar_impl = 2;                  // 2: cluster-owned kernel (dec_ar2.cuh), 1: grid-barrier kernel (dec_ar.cuh)
  pq::DecAr2Maps ar2_maps[2];       // TMA descriptors (decoder weights, K/V cache) for cluster size 8 [0] and 6 [1]
  bool ar2_maps_ok = false;
  int ar2_clusters[3][2] = {{0, 0}, {0, 0}, {0, 0}};   // max co-resident clusters, index [MT][cluster size 6 ? 1 : 0]
  int ar2_occ[3][2] = {{0, 0}, {0, 0}, {0, 0}};        // what cudaOccupancyMaxActiveClusters answered (debug)
  int ar_last_cs = 0;
  int ar_last_per = 0, ar_last_ncl = 0;
  int ar_cs = 0;                    // option "ar_cluster_size": 0 = auto, 6 / 8 = forced
  int ar_clusters_override = 0;     // option "ar_clusters": clusters the AR kernel spreads a batch over (0 = derived)
  int fuse_mlp = 0;                 // fc1 + GELU + fc2 + residual + LayerNorm in one kernel (mlp_ln.cuh) where fuse_ln bit 1 applies
  int fuse_ln = 3;                  // bit 0: attn.proj, bit 1: mlp.fc2 also produce the LayerNorm that follows (gemm_ln.cuh)
  __nv_bfloat16 *ar_sa = nullptr, *ar_ca = nullptr, *ar_hd = nullptr;
  float *ar_y = nullptr, *ar_qc = nullptr, *ar_part = nullptr;
  int* ar_ids = nullptr;
  unsigned int* ar_bar = nullptr;
  unsigned long long* ar_prof = nullptr;   // [32][16] phase time stamps of the AR kernel (debug option "ar_prof")
  bool ar_prof_on = false;
  cudaEvent_t ev_enc = nullptr;
  struct Stage {
    __nv_bfloat16 *sa = nullptr, *yn = nullptr, *ca = nullptr, *hd = nullptr;
    float *y = nullptr, *qc = nullptr;
    int *ids_ar = nullptr, *ids_ctx = nullptr;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev_enc = nullptr, ev_done = nullptr;
  };
  std::vector<Stage> stages;
  int max_batch = 512;              // images per graph / super-chunk = stages.size() * chunk
  cudaStream_t main = nullptr;      // engine-owned: user stream -> (event) -> main -> (event) -> user stream
  cudaStream_t copy = nullptr;      // host entry points: input upload in two halves, overlapped with the first half's encoder
  cudaEvent_t ev_c[3] = {nullptr, nullptr, nullptr};
  cudaEvent_t ev_in = nullptr, ev_out = nullptr;
  // static I/O buffers the CUDA graphs are captured on
  float* in_images = nullptr; float* out_logits = nullptr; int* out_ids = nullptr; int* out_steps = nullptr;
  uint8_t* in_images_u8 = nullptr;  // static input of the uint8 HWC entry points
  bool use_graph = true;
  struct GraphEntry { cudaGraphExec_t exec; long long kernels; };
  std::map<std::vector<int>, GraphEntry> graphs;
  // crop entry points (resize.cuh): the plan of the current call, built on the host and uploaded to engine-owned
  // buffers that grow on demand, plus the device staging copy of host pixels
  std::vector<pq::RzCrop> rz_hcrops;
  std::vector<pq::RzTask> rz_htasks;
  std::vector<long long> rz_first;  // [count + 1] index of the first task of each crop
  int rz_smem = 0;                  // dynamic shared memory of the plan's largest task
  int rz_rot = 0;                   // rotation of the plan
  pq::RzCrop* rz_crops = nullptr; long long rz_crops_cap = 0;
  pq::RzTask* rz_tasks = nullptr; long long rz_tasks_cap = 0;
  uint8_t* rz_stage = nullptr; long long rz_stage_cap = 0;

  void* w(const std::string& k) const { return slots[index.at(k)].dev; }
  const float* wf(const std::string& k) const { return reinterpret_cast<const float*>(w(k)); }
  const __nv_bfloat16* wb(const std::string& k) const { return reinterpret_cast<const __nv_bfloat16*>(w(k)); }
};

namespace {

void add_slot(parseq_engine* e, const std::string& key, long long numel, bool bf16) {
  std::string pub = key;
  if (e->arch == 1 && key.rfind("encoder.", 0) == 0) pub = key.substr(8);
  e->index[key] = static_cast<int>(e->slots.size());
  e->pub_index[pub] = static_cast<int>(e->slots.size());
  e->slots.push_back(Slot{key, pub, numel, bf16, nullptr, false});
}

template <typename Tp>
int dev_alloc(Tp** p, long long n) {
  PQ_CUDA(cudaMalloc(reinterpret_cast<void**>(p), static_cast<size_t>(n) * sizeof(Tp)));
  return PARSEQ_OK;
}

int alloc_workspace(parseq_engine* e) {
  const long long R = static_cast<long long>(e->chunk) * e->T;          // encoder rows per chunk
  const long long RB = static_cast<long long>(e->max_batch) * e->T;     // rows of a whole super-chunk
  const long long Rd = static_cast<long long>(e->dec_chunk) * e->L;     // decoder rows per chain
  const int D = e->D;
  PQ_TRY(dev_alloc(&e->a_pe, R * e->Kp));
  PQ_TRY(dev_alloc(&e->x, R * D));
  PQ_TRY(dev_alloc(&e->xn, R * D));
  PQ_TRY(dev_alloc(&e->qkv, R * 3 * D));
  PQ_TRY(dev_alloc(&e->att, R * D));
  PQ_TRY(dev_alloc(&e->hid, R * e->Me));
  PQ_TRY(dev_alloc(&e->mem, RB * D));
  PQ_TRY(dev_alloc(&e->ckv, RB * 2 * D));
  PQ_TRY(dev_alloc(&e->ar_sa, 1ll * e->max_batch * D));
  PQ_TRY(dev_alloc(&e->ar_ca, 1ll * e->max_batch * D));
  PQ_TRY(dev_alloc(&e->ar_hd, 1ll * e->max_batch * e->Md));
  PQ_TRY(dev_alloc(&e->ar_y, 1ll * e->max_batch * D));
  PQ_TRY(dev_alloc(&e->ar_qc, 1ll * e->max_batch * D));
  PQ_TRY(dev_alloc(&e->ar_part, 3ll * e->max_batch * D));
  PQ_TRY(dev_alloc(&e->ar_ids, 1ll * e->max_batch * 32));
  PQ_TRY(dev_alloc(&e->ar_bar, 64));
  PQ_TRY(dev_alloc(&e->ar_prof, 32 * 16));
  if (e->arch == 1) PQ_TRY(dev_alloc(&e->vt_rows, 1ll * e->chunk * e->L * D));
  PQ_CUDA(cudaEventCreateWithFlags(&e->ev_enc, cudaEventDisableTiming));
  const int n_stages = (e->max_batch + e->dec_chunk - 1) / e->dec_chunk;
  e->stages.resize(static_cast<size_t>(n_stages));
  for (auto& sg : e->stages) {
    PQ_TRY(dev_alloc(&sg.sa, Rd * D));
    PQ_TRY(dev_alloc(&sg.yn, Rd * D));
    PQ_TRY(dev_alloc(&sg.ca, Rd * D));
    PQ_TRY(dev_alloc(&sg.hd, Rd * e->Md));
    PQ_TRY(dev_alloc(&sg.y, Rd * D));
    PQ_TRY(dev_alloc(&sg.qc, Rd * D));
    PQ_TRY(dev_alloc(&sg.ids_ar, static_cast<long long>(e->dec_chunk) * 32));
    PQ_TRY(dev_alloc(&sg.ids_ctx, static_cast<long long>(e->dec_chunk) * 32));
    PQ_CUDA(cudaStreamCreateWithFlags(&sg.stream, cudaStreamNonBlocking));
    PQ_CUDA(cudaEventCreateWithFlags(&sg.ev_enc, cudaEventDisableTiming));
    PQ_CUDA(cudaEventCreateWithFlags(&sg.ev_done, cudaEventDisableTiming));
  }
  const long long NB = e->max_batch;
  PQ_TRY(dev_alloc(&e->in_images, NB * 3 * e->cfg.img_h * e->cfg.img_w));
  PQ_TRY(dev_alloc(&e->in_images_u8, NB * 3 * e->cfg.img_h * e->cfg.img_w));
  PQ_TRY(dev_alloc(&e->out_logits, NB * e->L * e->C));
  PQ_TRY(dev_alloc(&e->out_ids, NB * e->L));
  PQ_TRY(dev_alloc(&e->out_steps, 4));
  return PARSEQ_OK;
}

void drop_graphs(parseq_engine* e) {
  for (auto& kv : e->graphs) cudaGraphExecDestroy(kv.second.exec);
  e->graphs.clear();
}

void free_workspace(parseq_engine* e) {
  drop_graphs(e);
  e->ar2_maps_ok = false;           // holds the address of the K/V cache
  void* ptrs[] = {e->a_pe, e->x, e->xn, e->qkv, e->att, e->hid, e->mem, e->ckv, e->in_images, e->out_logits, e->out_ids,
                  e->out_steps, e->in_images_u8, e->ar_sa, e->ar_ca, e->ar_hd, e->ar_y, e->ar_qc, e->ar_part, e->ar_ids, e->ar_bar, e->ar_prof};
  e->ar_part = nullptr; e->ar_prof = nullptr; e->in_images_u8 = nullptr;
  if (e->vt_rows) { cudaFree(e->vt_rows); e->vt_rows = nullptr; }
  e->ar_sa = e->ar_ca = e->ar_hd = nullptr; e->ar_y = e->ar_qc = nullptr; e->ar_ids = nullptr; e->ar_bar = nullptr;
  for (void* p : ptrs)
    if (p) cudaFree(p);
  if (e->ev_enc) { cudaEventDestroy(e->ev_enc); e->ev_enc = nullptr; }
  e->a_pe = e->xn = e->qkv = e->att = e->hid = e->mem = e->ckv = nullptr;
  e->x = e->in_images = e->out_logits = nullptr;
  e->out_ids = e->out_steps = nullptr;
  for (auto& sg : e->stages) {
    void* q[] = {sg.sa, sg.yn, sg.ca, sg.hd, sg.y, sg.qc, sg.ids_ar, sg.ids_ctx};
    for (void* p : q)
      if (p) cudaFree(p);
    if (sg.stream) cudaStreamDestroy(sg.stream);
    if (sg.ev_enc) cudaEventDestroy(sg.ev_enc);
    if (sg.ev_done) cudaEventDestroy(sg.ev_done);
  }
  e->stages.clear();
}

// categories: 0 encoder GEMM, 1 encoder attention, 2 LayerNorm, 3 decoder GEMM, 4 decoder attention, 5 other
enum { CAT_ENC_GEMM = 0, CAT_ENC_ATTN = 1, CAT_LN = 2, CAT_DEC_GEMM = 3, CAT_DEC_ATTN = 4, CAT_MISC = 5, CAT_ENC_GEMM_LN = 6, CAT_DEC_AR = 7,
       CAT_COUNT = 8 };

cudaEvent_t pool_event(parseq_engine* e) {
  if (!e->event_pool.empty()) { cudaEvent_t ev = e->event_pool.back(); e->event_pool.pop_back(); return ev; }
  cudaEvent_t ev; cudaEventCreate(&ev); return ev;
}
struct TimedScope {   // records a CUDA-event pair around the launches issued in its lifetime
  parseq_engine* e; cudaStream_t st; int idx = -1;
  TimedScope(parseq_engine* e_, cudaStream_t st_, int cat, double flops) : e(e_), st(st_) {
    e->launches++;
    if (!e->timing) return;
    parseq_engine::TimedLaunch t{cat, flops, pool_event(e), pool_event(e)};
    cudaEventRecord(t.a, st);
    e->timed.push_back(t);
    idx = static_cast<int>(e->timed.size()) - 1;
  }
  ~TimedScope() { if (idx >= 0) cudaEventRecord(e->timed[idx].b, st); }
};

int gemm(parseq_engine* e, const void* A, long long lda, const void* W, long long ldw, const float* bias, int M, int N,
         int K, int mode, float alpha, const float* resid, long long ldr, int resid_mod, void* out, long long ldo,
         cudaStream_t st, long long blocked_rows = 0) {
  TimedScope ts(e, st, e->cur_cat == CAT_DEC_GEMM ? CAT_DEC_GEMM : CAT_ENC_GEMM, 2.0 * M * N * K);
  return gemm_launch(e->lo, A, lda, W, ldw, bias, M, N, K, mode, alpha, resid, ldr, resid_mod, out, ldo, st, blocked_rows);
}
// x += A W^T + b;  y = bf16(LayerNorm(x; <ln_prefix>))  in one kernel
int gemm_ln(parseq_engine* e, const void* A, long long lda, const std::string& lin, int M, int K, float* x,
            const std::string& ln_prefix, float eps, void* y, cudaStream_t st) {
  TimedScope ts(e, st, CAT_ENC_GEMM_LN, 2.0 * M * e->D * K);
  return gemm_ln_launch(e->lo, A, lda, e->w(lin + ".weight"), K, e->wf(lin + ".bias"), M, e->D, K, x, e->wf(ln_prefix + ".weight"),
                        e->wf(ln_prefix + ".bias"), eps, y, st);
}
// x += fc2(GELU(fc1(xn)));  y = bf16(LayerNorm(x; <ln_prefix>))  in one kernel (block prefix `blk`, e.g. "encoder.blocks.3.")
int mlp_ln(parseq_engine* e, const void* xn, const std::string& blk, int M, float* x, const std::string& ln_prefix, float eps,
           void* y, cudaStream_t st) {
  TimedScope ts(e, st, CAT_ENC_GEMM_LN, 4.0 * M * e->D * e->Me);
  return mlp_ln_launch(e->lo, xn, e->w(blk + "mlp.fc1.weight"), e->wf(blk + "mlp.fc1.bias"), e->w(blk + "mlp.fc2.weight"),
                       e->wf(blk + "mlp.fc2.bias"), M, e->D, x, e->wf(ln_prefix + ".weight"), e->wf(ln_prefix + ".bias"), eps, y, st);
}
int layernorm(parseq_engine* e, const float* x, const std::string& prefix, float eps, int M, void* y, float* y32,
              cudaStream_t st, const float* add = nullptr, int add_mod = 1, float* xw = nullptr) {
  TimedScope ts(e, st, CAT_LN, 0.0);
  return layernorm_launch(e->lo, x, e->wf(prefix + ".weight"), e->wf(prefix + ".bias"), eps, M, e->D, y, y32, st, add, add_mod, xw);
}

// ---------------------------------------------------------------- encoder (model.py:83-84 -> timm forward_features)
int encode_chunk(parseq_engine* e, const void* images_any, bool u8, int B, __nv_bfloat16* mem_out, float* memory32,
                 cudaStream_t st, bool final_norm = true, int regime_batch = 0) {
  // regime_batch: the batch whose size selects the kernel variants (a half batch encoded on its own, under the upload of
  // the other half, must run the kernels the whole batch would: rows stay bit-identical to the unsplit call)
  const int D = e->D, T = e->T, M = B * T;
  e->cur_cat = CAT_ENC_GEMM;
  {
    TimedScope ts(e, st, CAT_MISC, 0.0);
    if (u8) {
      const long long total = static_cast<long long>(B) * e->gh * e->gw * e->cfg.patch_h;
      const int grid = static_cast<int>((total + 255) / 256);
      PQ_TRY(launch_k(e->lo, pq::im2col_patch_u8_kernel, dim3(grid), dim3(256), 0, st, static_cast<const uint8_t*>(images_any), e->a_pe,
                      B, e->cfg.img_h, e->cfg.img_w, e->cfg.patch_h, e->cfg.patch_w, e->gh, e->gw));
    } else {
      const long long total = static_cast<long long>(B) * e->gh * e->gw * 3 * e->cfg.patch_h;
      const int grid = static_cast<int>((total + 255) / 256);
      PQ_TRY(launch_k(e->lo, pq::im2col_patch_kernel, dim3(grid), dim3(256), 0, st, static_cast<const float*>(images_any), e->a_pe, B,
                      e->cfg.img_h, e->cfg.img_w, e->cfg.patch_h, e->cfg.patch_w, e->gh, e->gw));
    }
  }
  if (e->arch == 0) {
    // x = patches * Wpe^T + bpe + pos_embed
    PQ_TRY(gemm(e, e->a_pe, e->Kp, e->w("encoder.patch_embed.proj.weight"), e->Kp,
                e->wf("encoder.patch_embed.proj.bias"), M, D, e->Kp, pq::EPI_F32, 1.0f, e->wf("encoder.pos_embed"), D, T,
                e->x, D, st));
  } else {
    // timm _pos_embed with a class token: x = cat(cls_token, patches * Wpe^T + bpe) + pos_embed[0..Tp]
    float* tmp = reinterpret_cast<float*>(e->hid);      // [B*Tp, D] fp32 fits the (still unused) [B*T, 4D] bf16 MLP buffer
    PQ_TRY(gemm(e, e->a_pe, e->Kp, e->w("encoder.patch_embed.proj.weight"), e->Kp,
                e->wf("encoder.patch_embed.proj.bias"), B * e->Tp, D, e->Kp, pq::EPI_F32, 1.0f,
                e->wf("encoder.pos_embed") + D, D, e->Tp, tmp, D, st));
    TimedScope ts(e, st, CAT_MISC, 0.0);
    const long long total = 1ll * M * (D / 4);
    const int grid = static_cast<int>(std::min<long long>((total + 255) / 256, 148ll * 16));
    PQ_TRY(launch_k(e->lo, pq::cls_assemble_kernel, dim3(grid), dim3(256), 0, st, reinterpret_cast<const float4*>(tmp),
                    reinterpret_cast<const float4*>(e->wf("encoder.cls_token")),
                    reinterpret_cast<const float4*>(e->wf("encoder.pos_embed")), reinterpret_cast<float4*>(e->x), B, e->Tp,
                    D / 4));
  }
  // With fuse_ln the two residual GEMMs of a block also emit the LayerNorm that consumes their result (norm2 after
  // attn.proj; the next block's norm1 - or the final encoder.norm - after mlp.fc2): the fp32 residual stream is read
  // and written once per GEMM instead of once more per LayerNorm.
  // The fused kernel owns whole 128-row tiles (one CTA per tile, both column halves in sequence): it pays off once
  // the tiles fill the machine about twice; below that the N-split GEMM + LayerNorm pair has the lower latency
  // (bs=1: 1.67 ms vs 1.93 ms p50).  "fuse_ln" bit 2 forces it for any M (tests).
  const int Mr = (regime_batch > B ? regime_batch : B) * T;
  const bool big = (Mr + pq::GEMM_BLOCK_M - 1) / pq::GEMM_BLOCK_M >= 2 * e->lo.sm_count || (e->fuse_ln & 4);
  const bool fuse_proj = (e->fuse_ln & 1) && gemm_ln_supported(D) && big;
  const bool fuse_fc2 = (e->fuse_ln & 2) && gemm_ln_supported(D) && big;
  const bool fuse_mlp = e->fuse_mlp && fuse_fc2 && e->Me == 4 * D;
  bool final_done = false;
  for (int i = 0; i < e->cfg.enc_depth; ++i) {
    const std::string p = "encoder.blocks." + std::to_string(i) + ".";
    const bool last = (i == e->cfg.enc_depth - 1);
    if (!(fuse_fc2 && i > 0)) PQ_TRY(layernorm(e, e->x, p + "norm1", 1e-6f, M, e->xn, nullptr, st));
    PQ_TRY(gemm(e, e->xn, D, e->w(p + "attn.qkv.weight"), D, e->wf(p + "attn.qkv.bias"), M, 3 * D, D, pq::EPI_BF16,
                1.0f, nullptr, 0, 0, e->qkv, 3 * D, st));
    {
      TimedScope ts(e, st, CAT_ENC_ATTN, 4.0 * B * T * T * D);
      PQ_TRY(enc_attention_launch(e->lo, e->qkv, B, T, D, e->cfg.enc_num_heads, e->att, st));
    }
    if (fuse_proj) {
      PQ_TRY(gemm_ln(e, e->att, D, p + "attn.proj", M, D, e->x, p + "norm2", 1e-6f, e->xn, st));
    } else {
      PQ_TRY(gemm(e, e->att, D, e->w(p + "attn.proj.weight"), D, e->wf(p + "attn.proj.bias"), M, D, D, pq::EPI_F32, 1.0f,
                  e->x, D, 0, e->x, D, st));
      PQ_TRY(layernorm(e, e->x, p + "norm2", 1e-6f, M, e->xn, nullptr, st));
    }
    if (fuse_mlp && (!last || (final_norm && memory32 == nullptr))) {
      // the whole MLP + the next LayerNorm in one kernel: the hidden activation never leaves the SM (mlp_ln.cuh)
      if (!last) {
        PQ_TRY(mlp_ln(e, e->xn, p, M, e->x, "encoder.blocks." + std::to_string(i + 1) + ".norm1", 1e-6f, e->xn, st));
      } else {
        PQ_TRY(mlp_ln(e, e->xn, p, M, e->x, "encoder.norm", 1e-6f, mem_out, st));
        final_done = true;
      }
      continue;
    }
    PQ_TRY(gemm(e, e->xn, D, e->w(p + "mlp.fc1.weight"), D, e->wf(p + "mlp.fc1.bias"), M, e->Me, D, pq::EPI_GELU_BF16,
                1.0f, nullptr, 0, 0, e->hid, e->Me, st));
    if (fuse_fc2 && !last) {
      PQ_TRY(gemm_ln(e, e->hid, e->Me, p + "mlp.fc2", M, e->Me, e->x, "encoder.blocks." + std::to_string(i + 1) + ".norm1",
                     1e-6f, e->xn, st));
    } else if (fuse_fc2 && final_norm && memory32 == nullptr) {
      PQ_TRY(gemm_ln(e, e->hid, e->Me, p + "mlp.fc2", M, e->Me, e->x, "encoder.norm", 1e-6f, mem_out, st));
      final_done = true;
    } else {
      PQ_TRY(gemm(e, e->hid, e->Me, e->w(p + "mlp.fc2.weight"), e->Me, e->wf(p + "mlp.fc2.bias"), M, D, e->Me,
                  pq::EPI_F32, 1.0f, e->x, D, 0, e->x, D, st));
    }
  }
  if (final_done) return PARSEQ_OK;
  if (final_norm) PQ_TRY(layernorm(e, e->x, "encoder.norm", 1e-6f, M, mem_out, memory32, st));
  return PARSEQ_OK;
}

// ---------------------------------------------------------------- ViTSTR tail (vitstr/model.py:19-28, vitstr/system.py:65-71)
// logits[b, j] = head(norm(x[b, 1 + j])), j < L = max_length + 1: the reference computes tokens [0, max_length + 2) and
// drops token 0 (the class token); norm and head are row-wise, so only the kept rows are gathered and computed.
int argmax_rows(parseq_engine* e, const float* logits, int L, int B, int nrows, int src0, int* ids, int ids_ld, int dst0,
                const int* forced, int forced_ld, cudaStream_t st);
int vitstr_tail(parseq_engine* e, int B, int L, float* logits, int* ids_out, cudaStream_t st) {
  const int D = e->D, M = B * L;
  {
    TimedScope ts(e, st, CAT_MISC, 0.0);
    const long long total = 1ll * M * (D / 4);
    const int grid = static_cast<int>(std::min<long long>((total + 255) / 256, 148ll * 16));
    PQ_TRY(launch_k(e->lo, pq::gather_token_rows_kernel, dim3(grid), dim3(256), 0, st, reinterpret_cast<const float4*>(e->x),
                    reinterpret_cast<float4*>(e->vt_rows), B, e->T, 1, L, D / 4));
  }
  PQ_TRY(layernorm(e, e->vt_rows, "encoder.norm", 1e-6f, M, e->xn, nullptr, st));
  PQ_TRY(gemm(e, e->xn, D, e->w("head.weight"), D, e->wf("head.bias"), M, e->C, D, pq::EPI_F32, 1.0f, nullptr, 0, 0, logits,
              e->C, st));
  if (ids_out != nullptr) PQ_TRY(argmax_rows(e, logits, L, B, L, 0, ids_out, L, 0, nullptr, 0, st));
  return PARSEQ_OK;
}

// ---------------------------------------------------------------- one Decoder call (model.py:86-103, modules.py:55-125)
// rows are (b, qi), qi in [0,nq); query position q0+qi; context ids[b, 0..nkeys-1].
// Tail: LayerNorm(decoder.norm) + head + (optionally) greedy argmax -> ids_dst[b*32 + dst_off + qi] in one kernel.
// Caller-supplied pieces of PARSeq.decode (model.py:86-103) that the inference loops never use: explicit query rows,
// explicit masks, decoder output instead of logits.
struct DecodeExtras {
  const float* query = nullptr;          // [B*nq, D] fp32 raw queries (residual base); null -> pos_queries[q0 + qi]
  const unsigned char* qmask = nullptr;  // [nq, nkeys], 1 = masked
  const unsigned char* pmask = nullptr;  // [B, nkeys], 1 = masked
  float* out_norm = nullptr;             // [B*nq, D] fp32: decoder.norm(y) is the result (no head)
};
int decode_pass(parseq_engine* e, parseq_engine::Stage& sg, int b_first, int B, int nq, int q0, int nkeys,
                int mode, const int* ids, float* logits_out, long long logits_ld, int* ids_dst, int dst_off,
                const int* forced, int forced_ld, cudaStream_t st, const DecodeExtras* ex = nullptr) {
  const int D = e->D, M = B * nq;
  const std::string Ly = "decoder.layers.0.";
  const float qscale = 1.0f / std::sqrt(static_cast<float>(e->dh_dec));
  const __nv_bfloat16* Wc = e->wb(Ly + "cross_attn.in_proj_weight");
  const float* bc = e->wf(Ly + "cross_attn.in_proj_bias");
  e->cur_cat = CAT_DEC_GEMM;
  const float* qself = e->qs;            // [L, D] table of W_q LN_q(pos_queries), pre-scaled
  const unsigned char *qmask = nullptr, *pmask = nullptr;
  if (ex != nullptr && ex->query != nullptr) {
    // custom queries: q = scale * (W_q LN_q(query) + b_q), one row per (image, query)
    PQ_TRY(layernorm(e, ex->query, Ly + "norm_q", 1e-5f, M, sg.yn, nullptr, st));
    PQ_TRY(gemm(e, sg.yn, D, e->w(Ly + "self_attn.in_proj_weight"), D, e->wf(Ly + "self_attn.in_proj_bias"), M, D, D,
                pq::EPI_F32, qscale, nullptr, 0, 0, sg.qc, D, st));
    qself = sg.qc;
    mode = 2;
  }
  if (ex != nullptr && (ex->qmask != nullptr || ex->pmask != nullptr)) {
    if (mode != 2) {                     // masks with the default queries: expand the table rows (tiny) so mode 2 applies
      const int n4 = nq * D / 4;
      PQ_TRY(launch_k(e->lo, pq::bcast_rows_kernel, dim3(static_cast<unsigned>(std::min((B * n4 + 255) / 256, 148 * 8))), dim3(256), 0, st,
                      reinterpret_cast<const float4*>(e->qs + static_cast<long long>(q0) * D), reinterpret_cast<float4*>(sg.qc), n4, B));
      e->launches++;
      qself = sg.qc;
      mode = 2;
    }
    qmask = ex->qmask; pmask = ex->pmask;
  }
  {
    TimedScope ts(e, st, CAT_DEC_ATTN, 4.0 * M * nkeys * D);
    const int qsplit = (nq >= 8) ? 4 : 1;
    PQ_TRY(launch_k(e->lo, pq::dec_self_attn2_kernel, dim3(B * qsplit), dim3(D < 384 ? D : 384), 0, st, qself,
                    static_cast<const __nv_bfloat16*>(e->kvtab), ids, 32, e->V, D, nq, q0, nkeys, mode, /*eos*/ 0, sg.sa,
                    qsplit, qmask, pmask));
  }
  // y = query + out_proj(sa): the GEMM stores out_proj(sa) with its TMA epilogue, the LayerNorm kernel adds the query
  // residual (broadcast pos_queries[q0 + qi], or the caller's rows), writes y back and emits norm1(y)
  const bool own_q = ex != nullptr && ex->query != nullptr;
  const float* resid = own_q ? ex->query : e->wf("pos_queries") + static_cast<long long>(q0) * D;
  PQ_TRY(gemm(e, sg.sa, D, e->w(Ly + "self_attn.out_proj.weight"), D, e->wf(Ly + "self_attn.out_proj.bias"), M, D, D,
              pq::EPI_F32, 1.0f, nullptr, 0, 0, sg.y, D, st));
  PQ_TRY(layernorm(e, sg.y, Ly + "norm1", 1e-5f, M, sg.yn, nullptr, st, resid, own_q ? M : nq, sg.y));
  PQ_TRY(gemm(e, sg.yn, D, Wc, D, bc, M, D, D, pq::EPI_F32, qscale, nullptr, 0, 0, sg.qc, D, st));
  {
    TimedScope ts(e, st, CAT_DEC_ATTN, 4.0 * M * e->T * D);
    const long long kv_rows = 1ll * e->max_batch * e->T;
    if (e->T <= 128)
      PQ_TRY(launch_k(e->lo, pq::dec_cross_attn3_kernel<4>, dim3(B * e->cfg.dec_num_heads), dim3(128), 0, st,
                      static_cast<const float*>(sg.qc), static_cast<const __nv_bfloat16*>(e->ckv), kv_rows, b_first, e->T, D,
                      e->cfg.dec_num_heads, nq, sg.ca));
    else
      PQ_TRY(launch_k(e->lo, pq::dec_cross_attn3_kernel<8>, dim3(B * e->cfg.dec_num_heads), dim3(128), 0, st,
                      static_cast<const float*>(sg.qc), static_cast<const __nv_bfloat16*>(e->ckv), kv_rows, b_first, e->T, D,
                      e->cfg.dec_num_heads, nq, sg.ca));
  }
  PQ_TRY(gemm(e, sg.ca, D, e->w(Ly + "cross_attn.out_proj.weight"), D, e->wf(Ly + "cross_attn.out_proj.bias"), M, D, D,
              pq::EPI_F32, 1.0f, sg.y, D, 0, sg.y, D, st));
  PQ_TRY(layernorm(e, sg.y, Ly + "norm2", 1e-5f, M, sg.yn, nullptr, st));
  PQ_TRY(gemm(e, sg.yn, D, e->w(Ly + "linear1.weight"), D, e->wf(Ly + "linear1.bias"), M, e->Md, D, pq::EPI_GELU_BF16,
              1.0f, nullptr, 0, 0, sg.hd, e->Md, st));
  PQ_TRY(gemm(e, sg.hd, e->Md, e->w(Ly + "linear2.weight"), e->Md, e->wf(Ly + "linear2.bias"), M, D, e->Md, pq::EPI_F32,
              1.0f, sg.y, D, 0, sg.y, D, st));
  if (ex != nullptr && ex->out_norm != nullptr) {
    // PARSeq.decode returns the decoder output: final LayerNorm only (modules.py:123-125)
    PQ_TRY(layernorm(e, sg.y, "decoder.norm", 1e-5f, M, sg.yn, ex->out_norm, st));
  } else if (nq > 1 && ids_dst == nullptr) {
    // multi-query passes (refine / NAR): LayerNorm kernel + tcgen05 GEMM for the head (weights read once per tile).
    // Chosen by pass type, not by batch size, so that a row's result does not depend on the batch it is computed in.
    PQ_TRY(layernorm(e, sg.y, "decoder.norm", 1e-5f, M, sg.yn, nullptr, st));
    PQ_TRY(gemm(e, sg.yn, D, e->w("head.weight"), D, e->wf("head.bias"), M, e->C, D, pq::EPI_F32, 1.0f, nullptr, 0, 0,
                logits_out, logits_ld, st));
  } else {
    TimedScope ts(e, st, CAT_DEC_GEMM, 2.0 * M * e->C * D);
    PQ_TRY(ln_head_argmax_launch(e->lo, sg.y, e->wf("decoder.norm.weight"), e->wf("decoder.norm.bias"), 1e-5f, e->wb("head.weight"),
                                 e->wf("head.bias"), M, e->C, D, logits_out, logits_ld, ids_dst, 32, nq, dst_off, forced,
                                 forced_ld, st));
  }
  return PARSEQ_OK;
}

int argmax_rows(parseq_engine* e, const float* logits, int L, int B, int nrows, int src0, int* ids, int ids_ld, int dst0,
                const int* forced, int forced_ld, cudaStream_t st) {
  const int warps = B * nrows;
  if (warps <= 0) return PARSEQ_OK;
  TimedScope ts(e, st, CAT_MISC, 0.0);
  return launch_k(e->lo, pq::argmax_rows_kernel, dim3((warps + 7) / 8), dim3(256), 0, st, logits, L, e->C, B, nrows, src0, ids, ids_ld,
                  dst0, forced, forced_ld);
}

// Decoder chain of one group of B <= dec_chunk images (their cross K/V is at `ckv`): AR loop / NAR pass, cloze
// refinement, final argmax.  model.py:113-169.
int decode_stage(parseq_engine* e, parseq_engine::Stage& sg, int b_first, const parseq_forward_args* a, int b0,
                 int B, int L, float* logits, int* ids_out, int* steps, cudaStream_t st, bool ar_done) {
  // b_first: index of the group's first image inside the super-chunk (row of the K/V cache); b0: inside the caller's batch
  const int C = e->C;
  const int bos = e->V - 2, pad = e->V - 1;
  const bool testing = a->max_length < 0;
  const long long LC = static_cast<long long>(L) * C;
  if (a->decode_ar && ar_done) {
    // the AR loop of the whole super-chunk already ran in the persistent kernel (ar_decode)
  } else if (a->decode_ar) {
    PQ_TRY(launch_k(e->lo, pq::fill_ids_kernel, dim3((B * 32 + 255) / 256), dim3(256), 0, st, sg.ids_ar, B, 32, bos, pad));
    e->launches++;
    const int* forced = a->forced_ids ? a->forced_ids + static_cast<long long>(b0) * L : nullptr;
    for (int i = 0; i < L; ++i) {
      // step i: context ids[:, :i+1], query position i; the fused tail writes ids[:, i+1] = argmax (model.py:142)
      PQ_TRY(decode_pass(e, sg, b_first, B, 1, i, i + 1, 0, sg.ids_ar, logits + static_cast<long long>(i) * C, LC,
                         (i + 1 < L) ? sg.ids_ar : nullptr, i + 1, forced, L, st));
    }
    if (testing && steps != nullptr) {
      PQ_TRY(launch_k(e->lo, pq::ar_steps_kernel, dim3(1), dim3(256), 0, st, static_cast<const int*>(sg.ids_ar), 32, B, L, 0, steps));
      e->launches++;
    }
  } else {
    PQ_TRY(launch_k(e->lo, pq::fill_ids_kernel, dim3((B * 32 + 255) / 256), dim3(256), 0, st, sg.ids_ctx, B, 32, bos, pad));
    e->launches++;
    PQ_TRY(decode_pass(e, sg, b_first, B, L, 0, 1, 0, sg.ids_ctx, logits, C, nullptr, 0, nullptr, 0, st));
  }
  for (int it = 0; it < a->refine_iters; ++it) {
    PQ_TRY(launch_k(e->lo, pq::fill_ids_kernel, dim3((B * 32 + 255) / 256), dim3(256), 0, st, sg.ids_ctx, B, 32, bos, pad));
    e->launches++;
    const int* forced = a->forced_refine
                            ? a->forced_refine + (static_cast<long long>(it) * a->batch + b0) * L
                            : nullptr;
    // ctx = [BOS, argmax(logits[:, :L-1])]  (model.py:161)
    PQ_TRY(argmax_rows(e, logits, L, B, L - 1, 0, sg.ids_ctx, 32, 1, forced, L, st));
    PQ_TRY(decode_pass(e, sg, b_first, B, L, 0, L, 1, sg.ids_ctx, logits, C, nullptr, 0, nullptr, 0, st));
  }
  if (ids_out != nullptr) PQ_TRY(argmax_rows(e, logits, L, B, L, 0, ids_out, L, 0, nullptr, 0, st));
  return PARSEQ_OK;
}


// ---- cluster-owned AR kernel (dec_ar2.cuh) ----
bool ar2_supported(const parseq_engine* e) {
  return e->arch == 0 && e->cfg.dec_mlp_ratio == 4 && e->C <= 96 && e->T <= 256 && e->dh_dec == 32;
}
// weight descriptors: once per weight set (parseq_finalize); K/V cache descriptor: once per workspace
int ar2_build_maps(parseq_engine* e) {
  const int D = e->D;
  const std::string Ly = "decoder.layers.0.";
  for (int ci = 0; ci < 2; ++ci) {
    const int cs = ci == 0 ? 8 : 6;
    pq::DecAr2Maps& m = e->ar2_maps[ci];
    const int DS = D / cs, MS = e->Md / cs;
    const int NC1 = (MS % 128 == 0) ? 128 : 96, NC2 = (D % 128 == 0) ? 128 : 96;
    PQ_TRY(make_tmap(&m.wo_s, e->w(Ly + "self_attn.out_proj.weight"), 2, D, D, D, 64, DS));
    PQ_TRY(make_tmap(&m.wq_c, e->w(Ly + "cross_attn.in_proj_weight"), 2, D, D, D, 64, DS));
    PQ_TRY(make_tmap(&m.wo_c, e->w(Ly + "cross_attn.out_proj.weight"), 2, D, D, D, 64, DS));
    PQ_TRY(make_tmap(&m.w1, e->w(Ly + "linear1.weight"), 2, e->Md, D, D, 64, NC1));
    PQ_TRY(make_tmap(&m.w2, e->w(Ly + "linear2.weight"), 2, D, e->Md, e->Md, 64, NC2));
    PQ_TRY(make_tmap(&m.wh, e->w("head.weight"), 2, e->C, D, D, 64, 96));
    const int tbox = e->T <= 64 ? 64 : 128;
    const long long kv_rows = 1ll * e->max_batch * e->T;     // column-blocked cache [2D/64][kv_rows][64]
    PQ_TRY(make_tmap3d(&m.ckv, e->ckv, 64, kv_rows, 2 * D / 64, 64, 64 * kv_rows, 64, tbox));
  }
  e->ar2_maps_ok = true;
  return PARSEQ_OK;
}
template <int D, int MT, int CS>
void ar2_config(parseq_engine* e, cudaLaunchConfig_t& cfg, cudaLaunchAttribute* attr, int ncl, cudaStream_t st) {
  cfg = cudaLaunchConfig_t{};
  cfg.gridDim = dim3(static_cast<unsigned>(ncl * CS));
  cfg.blockDim = dim3(pq::A2_LAUNCH_THREADS);
  cfg.dynamicSmemBytes = pq::dec_ar2_smem_bytes<D, MT, CS>();
  cfg.stream = st;
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CS;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
}
template <int D, int MT, int CS>
int ar2_launch(parseq_engine* e, const pq::DecAr2Params& p, int ncl, cudaStream_t st) {
  cudaLaunchConfig_t cfg;
  cudaLaunchAttribute attr[1];
  ar2_config<D, MT, CS>(e, cfg, attr, ncl, st);
  e->ar_last_per = p.per; e->ar_last_ncl = ncl; e->ar_last_cs = CS;
  if constexpr (MT == 1 && CS == 8 && D / 64 <= CS) {
    // so few images per cluster that (images x head pairs) fit its CTAs: every CTA takes one (image, head pair) of the
    // cross-attention instead of whole images (bs = 1: 9 -> 2.5 us per step; same bits per head)
    if (p.per * (D / 64) <= CS) {
      PQ_CUDA(cudaLaunchKernelEx(&cfg, pq::dec_ar2_kernel<D, MT, CS, true>, e->ar2_maps[0], p));
      return PARSEQ_OK;
    }
  }
  PQ_CUDA(cudaLaunchKernelEx(&cfg, pq::dec_ar2_kernel<D, MT, CS>, e->ar2_maps[CS == 6 ? 1 : 0], p));
  return PARSEQ_OK;
}
// Clusters of this instantiation that can be co-resident.  A cluster lives inside one GPC; on the B200s of this pool the
// occupancy query answers 15 for 8-CTA clusters (measured: 15 clusters run in 1.89 ms, 16 in 3.72 ms = two waves), so
// 512 images do not fit one wave of 32-row clusters of 8; clusters of 6 pack more SMs (23 x 6 = 138).
template <int D, int MT, int CS>
int ar2_max_clusters(parseq_engine* e) {
  int& cache = e->ar2_clusters[MT][CS == 6 ? 1 : 0];
  if (cache > 0) return cache;
  cudaLaunchConfig_t cfg;
  cudaLaunchAttribute attr[1];
  ar2_config<D, MT, CS>(e, cfg, attr, e->lo.sm_count / CS, nullptr);
  int n = 0;
  if (cudaOccupancyMaxActiveClusters(&n, pq::dec_ar2_kernel<D, MT, CS>, &cfg) != cudaSuccess || n <= 0) {
    cudaGetLastError();
    n = (CS == 8) ? (e->lo.sm_count / 10) : 1;   // unknown: a conservative guess for 8, "do not use" for 6
  }
  e->ar2_occ[MT][CS == 6 ? 1 : 0] = n;
  if (e->ar_clusters_override > 0) n = e->ar_clusters_override;
  cache = n;
  return n;
}
// Spread the batch over the co-resident clusters.  Candidates in order of per-step cost: clusters of 8 with one m16 row
// tile, clusters of 8 with two, clusters of 6 (a third more weight bytes per CTA and step); the first that holds the
// batch in ONE wave wins (the loop is latency-bound: a second wave doubles its time), else the fewest waves.
template <int D>
int ar2_dispatch(parseq_engine* e, pq::DecAr2Params& p, cudaStream_t st) {
  constexpr bool kHas2 = (D != 768);            // two m16 tiles of D = 768 rows do not fit shared memory
  struct Cand { int mt, cs, maxc, rows; };
  Cand c[4];
  int nc = 0;
  const bool allow6 = e->ar_cs != 8, allow8 = e->ar_cs != 6;
  if (allow8) c[nc++] = Cand{1, 8, ar2_max_clusters<D, 1, 8>(e), 16};
  if constexpr (kHas2) { if (allow8) c[nc++] = Cand{2, 8, ar2_max_clusters<D, 2, 8>(e), 32}; }
  if (allow6) c[nc++] = Cand{1, 6, ar2_max_clusters<D, 1, 6>(e), 16};
  if constexpr (kHas2) { if (allow6) c[nc++] = Cand{2, 6, ar2_max_clusters<D, 2, 6>(e), 32}; }
  int best = -1, best_waves = 1 << 30;
  for (int i = 0; i < nc; ++i) {
    const int need = (p.B + c[i].rows - 1) / c[i].rows;             // clusters at full rows
    const int waves = (need + c[i].maxc - 1) / c[i].maxc;
    if (waves < best_waves) { best = i; best_waves = waves; }
  }
  const Cand& k = c[best];
  int per = (p.B + k.maxc * best_waves - 1) / (k.maxc * best_waves);   // even spread over the clusters of all waves
  if (per > k.rows) per = k.rows;
  if (per < 1) per = 1;
  p.per = per;
  const int ncl = (p.B + per - 1) / per;
  if (k.cs == 8) {
    if (k.mt == 1) return ar2_launch<D, 1, 8>(e, p, ncl, st);
    if constexpr (kHas2) return ar2_launch<D, 2, 8>(e, p, ncl, st);
  } else {
    if (k.mt == 1) return ar2_launch<D, 1, 6>(e, p, ncl, st);
    if constexpr (kHas2) return ar2_launch<D, 2, 6>(e, p, ncl, st);
  }
  return fail(PARSEQ_ERR_STATE, "dec_ar2: no launch configuration");
}

// The whole AR loop (model.py:119-147) of B images in one persistent launch (csrc/dec_ar.cuh).
int ar_decode(parseq_engine* e, const parseq_forward_args* a, int b0, int B, int L, float* logits, int* steps, cudaStream_t st) {
  const int D = e->D;
  const std::string Ly = "decoder.layers.0.";
  const bool testing = a->max_length < 0;
  PQ_TRY(launch_k(e->lo, pq::fill_ids_kernel, dim3((B * 32 + 255) / 256), dim3(256), 0, st, e->ar_ids, B, 32, e->V - 2, e->V - 1));
  e->launches++;
  if (e->ar_impl == 2 && ar2_supported(e)) {
    if (!e->ar2_maps_ok) PQ_TRY(ar2_build_maps(e));
    pq::DecAr2Params q;
    q.B = B; q.L = L; q.V = e->V; q.C = e->C; q.T = e->T; q.per = 0;
    q.tbox = e->T <= 64 ? 64 : 128; q.tb = (e->T + 127) / 128;
    q.qscale = 1.0f / std::sqrt(static_cast<float>(e->dh_dec));
    q.qs = e->qs; q.kvtab = e->kvtab; q.posq = e->wf("pos_queries");
    q.bo_s = e->wf(Ly + "self_attn.out_proj.bias"); q.bq_c = e->wf(Ly + "cross_attn.in_proj_bias");
    q.bo_c = e->wf(Ly + "cross_attn.out_proj.bias"); q.b1 = e->wf(Ly + "linear1.bias"); q.b2 = e->wf(Ly + "linear2.bias");
    q.bh = e->wf("head.bias");
    q.g1 = e->wf(Ly + "norm1.weight"); q.be1 = e->wf(Ly + "norm1.bias");
    q.g2 = e->wf(Ly + "norm2.weight"); q.be2 = e->wf(Ly + "norm2.bias");
    q.g3 = e->wf("decoder.norm.weight"); q.be3 = e->wf("decoder.norm.bias");
    q.ids = e->ar_ids; q.ids_ld = 32; q.logits = logits;
    q.forced = a->forced_ids ? a->forced_ids + static_cast<long long>(b0) * L : nullptr;
    q.forced_ld = L;
    q.prof = e->ar_prof_on ? e->ar_prof : nullptr;
    {
      const double macs = static_cast<double>(B) * L * (3.0 * D * D + 2.0 * D * e->Md + 1.0 * e->C * D + 2.0 * e->T * D);
      TimedScope ts(e, st, CAT_DEC_AR, 2.0 * macs);
      switch (D) {
        case 192: PQ_TRY(ar2_dispatch<192>(e, q, st)); break;
        case 384: PQ_TRY(ar2_dispatch<384>(e, q, st)); break;
        case 768: PQ_TRY(ar2_dispatch<768>(e, q, st)); break;
        default: return fail(PARSEQ_ERR_UNSUPPORTED, "dec_ar2: embed_dim must be 192, 384 or 768");
      }
    }
    if (testing && steps != nullptr) {
      PQ_TRY(launch_k(e->lo, pq::ar_steps_kernel, dim3(1), dim3(256), 0, st, static_cast<const int*>(e->ar_ids), 32, B, L, 0, steps));
      e->launches++;
    }
    return PARSEQ_OK;
  }
  PQ_CUDA(cudaMemsetAsync(e->ar_bar, 0, 64, st));
  pq::DecArParams p;
  p.B = B; p.L = L; p.Md = e->Md; p.V = e->V; p.C = e->C; p.T = e->T; p.heads = e->cfg.dec_num_heads;
  p.qscale = 1.0f / std::sqrt(static_cast<float>(e->dh_dec));
  p.qs = e->qs; p.kvtab = e->kvtab; p.posq = e->wf("pos_queries");
  p.Wo_s = e->wb(Ly + "self_attn.out_proj.weight"); p.bo_s = e->wf(Ly + "self_attn.out_proj.bias");
  p.Wq_c = e->wb(Ly + "cross_attn.in_proj_weight"); p.bq_c = e->wf(Ly + "cross_attn.in_proj_bias");
  p.Wo_c = e->wb(Ly + "cross_attn.out_proj.weight"); p.bo_c = e->wf(Ly + "cross_attn.out_proj.bias");
  p.W1 = e->wb(Ly + "linear1.weight"); p.b1 = e->wf(Ly + "linear1.bias");
  p.W2 = e->wb(Ly + "linear2.weight"); p.b2 = e->wf(Ly + "linear2.bias");
  p.Wh = e->wb("head.weight"); p.bh = e->wf("head.bias");
  p.g1 = e->wf(Ly + "norm1.weight"); p.be1 = e->wf(Ly + "norm1.bias");
  p.g2 = e->wf(Ly + "norm2.weight"); p.be2 = e->wf(Ly + "norm2.bias");
  p.g3 = e->wf("decoder.norm.weight"); p.be3 = e->wf("decoder.norm.bias");
  p.ckv = e->ckv; p.kv_rows = 1ll * e->max_batch * e->T; p.ids = e->ar_ids; p.ids_ld = 32;
  p.sa = e->ar_sa; p.ca = e->ar_ca; p.hd = e->ar_hd; p.y = e->ar_y; p.qc = e->ar_qc; p.part = e->ar_part;
  p.logits = logits;
  p.forced = a->forced_ids ? a->forced_ids + static_cast<long long>(b0) * L : nullptr;
  p.forced_ld = L;
  p.bar = e->ar_bar;
  p.prof = e->ar_prof_on ? e->ar_prof : nullptr;
  {
    // per image and step: 3 D^2 (self out, cross q, cross out) + 2 D Md (MLP) + C D (head) + attention dots
    const double macs = static_cast<double>(B) * L * (3.0 * D * D + 2.0 * D * e->Md + 1.0 * e->C * D + 2.0 * e->T * D);
    TimedScope ts(e, st, CAT_DEC_AR, 2.0 * macs);
    const dim3 grid(static_cast<unsigned>(e->lo.sm_count)), block(pq::DEC_THREADS);
    switch (D) {
      case 192:
        if (e->T <= 128) PQ_TRY(launch_k(e->lo, pq::dec_ar_kernel<192, 1>, grid, block, pq::dec_ar_smem_bytes<192>(), st, p));
        else PQ_TRY(launch_k(e->lo, pq::dec_ar_kernel<192, 2>, grid, block, pq::dec_ar_smem_bytes<192>(), st, p));
        break;
      case 384:
        if (e->T <= 128) PQ_TRY(launch_k(e->lo, pq::dec_ar_kernel<384, 1>, grid, block, pq::dec_ar_smem_bytes<384>(), st, p));
        else PQ_TRY(launch_k(e->lo, pq::dec_ar_kernel<384, 2>, grid, block, pq::dec_ar_smem_bytes<384>(), st, p));
        break;
      case 768:
        if (e->T <= 128) PQ_TRY(launch_k(e->lo, pq::dec_ar_kernel<768, 1>, grid, block, pq::dec_ar_smem_bytes<768>(), st, p));
        else PQ_TRY(launch_k(e->lo, pq::dec_ar_kernel<768, 2>, grid, block, pq::dec_ar_smem_bytes<768>(), st, p));
        break;
      default: return fail(PARSEQ_ERR_UNSUPPORTED, "dec_ar: embed_dim must be 192, 384 or 768");
    }
  }
  if (testing && steps != nullptr) {
    PQ_TRY(launch_k(e->lo, pq::ar_steps_kernel, dim3(1), dim3(256), 0, st, static_cast<const int*>(e->ar_ids), 32, B, L, 0, steps));
    e->launches++;
  }
  return PARSEQ_OK;
}

// One super-chunk (B <= max_batch images): `main` encodes everything (in `chunk`-image pieces) and projects the cross
// K/V of the whole super-chunk; then the decoder - a latency-bound chain of small kernels - runs as ceil(B/dec_chunk)
// independent chains on their own streams, concurrently (event fork/join, capturable into a CUDA graph).
// part 0: the whole super-chunk.  part 1 / 2 (host entry points, PARSeq only): the encoder of images [0, split) alone /
// the encoder of images [split, B) and everything after it - two graphs, so that the second half of the input is still
// uploading while the first half is being encoded.
int forward_super(parseq_engine* e, const parseq_forward_args* a, int b0, int B, int L, const void* images, bool u8,
                  float* logits, int* ids_out, int* steps, int part = 0, int split = 0) {
  const long long img_sz = 3ll * e->cfg.img_h * e->cfg.img_w * (u8 ? 1 : 4);   // bytes per image
  const int D = e->D, T = e->T;
  if (part == 1)
    return encode_chunk(e, images, u8, split, e->mem, nullptr, e->main, true, B);
  if (e->arch == 1) {               // ViTSTR: encoder blocks, then norm + head on the kept token rows of each chunk
    for (int o = 0; o < B; o += e->chunk) {
      const int Bs = (B - o < e->chunk) ? (B - o) : e->chunk;
      PQ_TRY(encode_chunk(e, static_cast<const char*>(images) + o * img_sz, u8, Bs, nullptr, nullptr, e->main, false));
      PQ_TRY(vitstr_tail(e, Bs, L, logits + 1ll * o * L * e->C, ids_out ? ids_out + 1ll * o * L : nullptr, e->main));
    }
    return PARSEQ_OK;
  }
  if (part == 2) {
    PQ_TRY(encode_chunk(e, static_cast<const char*>(images) + split * img_sz, u8, B - split, e->mem + 1ll * split * T * D, nullptr,
                        e->main, true, B));
  } else {
    for (int o = 0; o < B; o += e->chunk) {
      const int Bs = (B - o < e->chunk) ? (B - o) : e->chunk;
      // kernel regime (fused GEMM + LayerNorm or not) from the super-chunk, so that it does not depend on `chunk`
      PQ_TRY(encode_chunk(e, static_cast<const char*>(images) + o * img_sz, u8, Bs, e->mem + 1ll * o * T * D, nullptr, e->main,
                          true, B));
    }
  }
  // cross-attention K/V of the image memory, once per image (the reference recomputes it in every decode call)
  e->cur_cat = CAT_DEC_GEMM;
  {
    const std::string Ly = "decoder.layers.0.";
    const __nv_bfloat16* Wkv = e->wb(Ly + "cross_attn.in_proj_weight") + static_cast<long long>(D) * D;
    const float* bkv = e->wf(Ly + "cross_attn.in_proj_bias") + D;
    // stored column-blocked [2D/64][max_batch * T][64]: an image's K (V) panel of 64 channels is one contiguous T x 128 B
    // run - what a TMA box of the AR kernel and a head of the refine-pass attention read
    PQ_TRY(gemm(e, e->mem, D, Wkv, D, bkv, B * T, 2 * D, D, pq::EPI_BF16, 1.0f, nullptr, 0, 0, e->ckv, 2 * D, e->main,
                1ll * e->max_batch * T));
  }
  const bool ar_done = a->decode_ar && e->use_ar_kernel;
  if (ar_done) {
    PQ_TRY(ar_decode(e, a, b0, B, L, logits, steps, e->main));
    if (a->refine_iters == 0) {      // nothing left for the chains but the final argmax
      if (ids_out != nullptr) PQ_TRY(argmax_rows(e, logits, L, B, L, 0, ids_out, L, 0, nullptr, 0, e->main));
      return PARSEQ_OK;
    }
  }
  const int n = (B + e->dec_chunk - 1) / e->dec_chunk;
  const bool fork = (n > 1) && !e->timing;      // timing mode: everything on `main` (isolated kernel times)
  if (fork) PQ_CUDA(cudaEventRecord(e->ev_enc, e->main));
  for (int s = 0; s < n; ++s) {
    parseq_engine::Stage& sg = e->stages[static_cast<size_t>(s)];
    const int o = s * e->dec_chunk;
    const int Bs = (B - o < e->dec_chunk) ? (B - o) : e->dec_chunk;
    cudaStream_t ds = fork ? sg.stream : e->main;
    if (fork) PQ_CUDA(cudaStreamWaitEvent(ds, e->ev_enc, 0));
    PQ_TRY(decode_stage(e, sg, o, a, b0 + o, Bs, L, logits + 1ll * o * L * e->C,
                        ids_out ? ids_out + 1ll * o * L : nullptr, steps, ds, ar_done));
    if (fork) PQ_CUDA(cudaEventRecord(sg.ev_done, ds));
  }
  if (fork)
    for (int s = 0; s < n; ++s) PQ_CUDA(cudaStreamWaitEvent(e->main, e->stages[static_cast<size_t>(s)].ev_done, 0));
  return PARSEQ_OK;
}

int num_steps_of(const parseq_engine* e, int max_length) {
  const int ml = (max_length < 0) ? e->cfg.max_label_length
                                  : (max_length < e->cfg.max_label_length ? max_length : e->cfg.max_label_length);
  return ml + 1;
}

// Replays (capturing on first use) the CUDA graph of one super-chunk of Bc images on the static I/O buffers.
int run_graph(parseq_engine* e, const parseq_forward_args* a, int Bc, int L, bool u8, int part = 0, int split = 0) {
  std::vector<int> key = {Bc, L, a->max_length < 0 ? 1 : 0, a->decode_ar ? 1 : 0, a->refine_iters, u8 ? 1 : 0, part, split};
  auto it = e->graphs.find(key);
  if (it == e->graphs.end()) {
    parseq_forward_args aa = *a;
    aa.batch = Bc;
    aa.forced_ids = nullptr;
    aa.forced_refine = nullptr;
    const long long before = e->launches;
    PQ_CUDA(cudaStreamBeginCapture(e->main, cudaStreamCaptureModeThreadLocal));
    int r = forward_super(e, &aa, 0, Bc, L, u8 ? static_cast<const void*>(e->in_images_u8) : static_cast<const void*>(e->in_images),
                          u8, e->out_logits, e->out_ids, e->out_steps, part, split);
    cudaGraph_t g = nullptr;
    cudaError_t ce = cudaStreamEndCapture(e->main, &g);
    if (r != PARSEQ_OK) { if (g) cudaGraphDestroy(g); return r; }
    if (ce != cudaSuccess) return fail(PARSEQ_ERR_CUDA, std::string("graph capture: ") + cudaGetErrorString(ce));
    cudaGraphExec_t exec = nullptr;
    ce = cudaGraphInstantiate(&exec, g, 0);
    cudaGraphDestroy(g);
    if (ce != cudaSuccess) return fail(PARSEQ_ERR_CUDA, std::string("graph instantiate: ") + cudaGetErrorString(ce));
    parseq_engine::GraphEntry ge{exec, e->launches - before};
    e->launches = before;
    it = e->graphs.emplace(key, ge).first;
  }
  PQ_CUDA(cudaGraphLaunch(it->second.exec, e->main));
  e->launches += it->second.kernels;
  return PARSEQ_OK;
}

// ---------------------------------------------------------------- variable-size crops (resize.cuh)
constexpr int RZ_MAX_SIDE = 4096;
constexpr int RZ_BAND = 8;                      // output rows per task at most
constexpr int RZ_SMEM_BUDGET = 48 * 1024;       // per-task shared memory the planner aims for (several CTAs per SM)

// shared memory of a task (the layout of resize_bicubic_u8_kernel)
long long rz_task_bytes(int ny, int nx, int nr, int wcols, int kh, int kv) {
  return 4ll * (2 * ny + 2 * nx + 1ll * ny * kv + 1ll * nx * kh) + 3ll * nr * wcols;
}

// Host copy of the kernel's first-tap / tap-count arithmetic (precompute_coeffs), used to size the row windows.
void rz_bounds(int in_size, int out_size, std::vector<int>& xmin, std::vector<int>& cnt) {
  xmin.resize(static_cast<size_t>(out_size));
  cnt.resize(static_cast<size_t>(out_size));
  if (in_size == out_size) {
    for (int i = 0; i < out_size; ++i) { xmin[i] = i; cnt[i] = 1; }
    return;
  }
  const double scale = static_cast<double>(in_size) / out_size;
  const double support = 2.0 * (scale < 1.0 ? 1.0 : scale);
  for (int xx = 0; xx < out_size; ++xx) {
    const double center = (xx + 0.5) * scale;
    int lo = static_cast<int>(center - support + 0.5);
    if (lo < 0) lo = 0;
    int hi = static_cast<int>(center + support + 0.5);
    if (hi > in_size) hi = in_size;
    xmin[xx] = lo;
    cnt[xx] = hi - lo;
  }
}

// Validates every crop, then splits each into tasks: (band of <= RZ_BAND output rows) x (tile of output columns) whose
// shared memory fits RZ_SMEM_BUDGET where possible and the device limit always.  Changes nothing on failure.
int rz_plan(parseq_engine* e, const parseq_crops* cr) {
  if (cr == nullptr) return fail(PARSEQ_ERR_INVALID_ARG, "null crops");
  if (cr->count < 0) return fail(PARSEQ_ERR_INVALID_ARG, "negative crop count");
  if (cr->count > 0 && (cr->desc == nullptr || cr->pixels == nullptr))
    return fail(PARSEQ_ERR_INVALID_ARG, "crops: null desc / pixels");
  if (cr->rotation != 0 && cr->rotation != 90 && cr->rotation != 180 && cr->rotation != 270)
    return fail(PARSEQ_ERR_INVALID_ARG, "crops: rotation must be 0, 90, 180 or 270, got " + std::to_string(cr->rotation));
  if (cr->pixels_bytes < 0) return fail(PARSEQ_ERR_INVALID_ARG, "crops: negative pixels_bytes");
  for (int i = 0; i < cr->count; ++i) {
    const parseq_crop& d = cr->desc[i];
    const std::string at = "crop " + std::to_string(i) + ": ";
    if (d.height < 1 || d.width < 1 || d.height > RZ_MAX_SIDE || d.width > RZ_MAX_SIDE)
      return fail(PARSEQ_ERR_INVALID_ARG, at + "size " + std::to_string(d.height) + "x" + std::to_string(d.width) +
                                              " outside 1..4096");
    if (d.row_stride < 3 * d.width) return fail(PARSEQ_ERR_INVALID_ARG, at + "row_stride < 3 * width");
    if (d.offset < 0 || d.offset + 1ll * (d.height - 1) * d.row_stride + 3ll * d.width > cr->pixels_bytes)
      return fail(PARSEQ_ERR_INVALID_ARG, at + "extends outside [0, pixels_bytes)");
  }
  int optin = 0, dev = 0;
  PQ_CUDA(cudaGetDevice(&dev));
  PQ_CUDA(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
  const int H = e->cfg.img_h, W = e->cfg.img_w;
  std::vector<pq::RzCrop> crops;
  std::vector<pq::RzTask> tasks;
  std::vector<long long> first;
  crops.reserve(static_cast<size_t>(cr->count));
  first.reserve(static_cast<size_t>(cr->count) + 1);
  long long smem = 0;
  std::vector<int> vmin, vcnt;
  for (int i = 0; i < cr->count; ++i) {
    const parseq_crop& d = cr->desc[i];
    const bool turn = cr->rotation == 90 || cr->rotation == 270;
    pq::RzCrop c{d.offset, d.height, d.width, d.row_stride, turn ? d.width : d.height, turn ? d.height : d.width, 0};
    c.vfirst = (c.hr > 100 * c.wr && H < c.hr) ? 1 : 0;    // PIL Image.resize: very tall images shrink height first
    const int kh = c.wr != W ? pq::rz_ksize(c.wr, W) : 0, kv = c.hr != H ? pq::rz_ksize(c.hr, H) : 0;
    rz_bounds(c.hr, H, vmin, vcnt);
    // window rows of output rows [y0, y1) and their width in pixels for a tile of nx columns
    auto rows = [&](int y0, int y1) { return c.vfirst ? (y1 - y0) : (vmin[y1 - 1] + vcnt[y1 - 1] - vmin[y0]); };
    auto bytes = [&](int y0, int y1, int nx) {
      return rz_task_bytes(y1 - y0, nx, rows(y0, y1), c.vfirst ? c.wr : nx, kh, kv);
    };
    int max_rows = 0;
    for (int y = 0; y < H; ++y) max_rows = std::max(max_rows, rows(y, y + 1));
    auto one_row = [&](int nx) {
      return rz_task_bytes(1, nx, c.vfirst ? 1 : max_rows, c.vfirst ? c.wr : nx, kh, kv);
    };
    const long long budget = std::max<long long>(RZ_SMEM_BUDGET, one_row(1));
    if (budget > optin) return fail(PARSEQ_ERR_UNSUPPORTED, "crop " + std::to_string(i) + ": resize does not fit shared memory");
    int tiles = 1;
    while (one_row((W + tiles - 1) / tiles) > budget) ++tiles;
    const int nx = (W + tiles - 1) / tiles;
    first.push_back(static_cast<long long>(tasks.size()));
    for (int y0 = 0; y0 < H;) {
      int y1 = y0 + 1;
      while (y1 < H && y1 - y0 < RZ_BAND && bytes(y0, y1 + 1, nx) <= budget) ++y1;
      for (int x0 = 0; x0 < W; x0 += nx) {
        const int n = std::min(nx, W - x0);
        tasks.push_back(pq::RzTask{i, y0, y1 - y0, x0, n, c.vfirst ? 0 : vmin[y0], rows(y0, y1)});
        smem = std::max(smem, bytes(y0, y1, n));
      }
      y0 = y1;
    }
    crops.push_back(c);
  }
  first.push_back(static_cast<long long>(tasks.size()));
  e->rz_hcrops.swap(crops);
  e->rz_htasks.swap(tasks);
  e->rz_first.swap(first);
  e->rz_smem = static_cast<int>((smem + 15) & ~15ll);
  e->rz_rot = cr->rotation;
  return PARSEQ_OK;
}

// Grows an engine-owned device buffer to hold n elements; on failure the old buffer is kept.
template <typename Tp>
int rz_reserve(parseq_engine* e, Tp** buf, long long* cap, long long n) {
  if (n <= *cap) return PARSEQ_OK;
  Tp* p = nullptr;
  PQ_TRY(dev_alloc(&p, n));
  PQ_CUDA(cudaStreamSynchronize(e->main));       // the old buffer may still be read by enqueued work
  if (*buf) cudaFree(*buf);
  *buf = p;
  *cap = n;
  return PARSEQ_OK;
}

// Validates and plans the crops, then uploads the plan (and, for host pixels, the pixels) on `main`.
// Returns the device address of the pixels through *pixels_dev.
int rz_prepare(parseq_engine* e, const parseq_crops* cr, bool host, const uint8_t** pixels_dev) {
  PQ_TRY(rz_plan(e, cr));
  PQ_TRY(rz_reserve(e, &e->rz_crops, &e->rz_crops_cap, std::max<long long>(1, cr->count)));
  PQ_TRY(rz_reserve(e, &e->rz_tasks, &e->rz_tasks_cap, std::max<long long>(1, static_cast<long long>(e->rz_htasks.size()))));
  if (host) PQ_TRY(rz_reserve(e, &e->rz_stage, &e->rz_stage_cap, std::max<long long>(16, cr->pixels_bytes)));
  PQ_CUDA(cudaMemcpyAsync(e->rz_crops, e->rz_hcrops.data(), e->rz_hcrops.size() * sizeof(pq::RzCrop), cudaMemcpyHostToDevice,
                          e->main));
  PQ_CUDA(cudaMemcpyAsync(e->rz_tasks, e->rz_htasks.data(), e->rz_htasks.size() * sizeof(pq::RzTask), cudaMemcpyHostToDevice,
                          e->main));
  if (host && cr->pixels_bytes > 0)
    PQ_CUDA(cudaMemcpyAsync(e->rz_stage, cr->pixels, static_cast<size_t>(cr->pixels_bytes), cudaMemcpyHostToDevice, e->main));
  *pixels_dev = host ? e->rz_stage : cr->pixels;
  return PARSEQ_OK;
}

// Resizes planned crops [b0, b0 + B) into out [B, img_h, img_w, 3].
int rz_launch(parseq_engine* e, const uint8_t* pixels, int b0, int B, uint8_t* out, cudaStream_t st) {
  static int smem_attr = 0;
  if (e->rz_smem > smem_attr) {
    PQ_CUDA(cudaFuncSetAttribute(pq::resize_bicubic_u8_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, e->rz_smem));
    smem_attr = e->rz_smem;
  }
  const long long t0 = e->rz_first[static_cast<size_t>(b0)], t1 = e->rz_first[static_cast<size_t>(b0 + B)];
  if (t1 == t0) return PARSEQ_OK;
  TimedScope ts(e, st, CAT_MISC, 0.0);
  return launch_k(e->lo, pq::resize_bicubic_u8_kernel, dim3(static_cast<unsigned>(t1 - t0)), dim3(pq::RZ_THREADS),
                  static_cast<size_t>(e->rz_smem), st, pixels, static_cast<const pq::RzCrop*>(e->rz_crops),
                  static_cast<const pq::RzTask*>(e->rz_tasks + t0), b0, out, e->cfg.img_h, e->cfg.img_w, e->rz_rot);
}

// Common driver of parseq_forward / parseq_forward_host. `host` selects H2D/D2H vs D2D staging copies.
// crop_pixels != NULL (crop entry points, plan uploaded by rz_prepare): each super-chunk is resized into the uint8 input
// buffer instead of copied there, then runs exactly as parseq_forward_u8 would.
int forward_impl(parseq_engine* e, const parseq_forward_args* a, const void* images_any, float* logits, int32_t* ids,
                 int32_t* steps, cudaStream_t user, bool host, bool u8 = false, const uint8_t* crop_pixels = nullptr) {
  const int L = num_steps_of(e, a->max_length);
  const bool testing = a->max_length < 0;
  const long long img_sz = 3ll * e->cfg.img_h * e->cfg.img_w * (u8 ? 1 : 4);   // bytes per image
  const char* images = static_cast<const char*>(images_any);
  void* in_static = u8 ? static_cast<void*>(e->in_images_u8) : static_cast<void*>(e->in_images);
  const bool eager = !e->use_graph || e->timing || a->forced_ids != nullptr || a->forced_refine != nullptr;
  const cudaMemcpyKind kin = host ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice;
  const cudaMemcpyKind kout = host ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice;
  // user stream -> main
  PQ_CUDA(cudaEventRecord(e->ev_in, user));
  PQ_CUDA(cudaStreamWaitEvent(e->main, e->ev_in, 0));
  PQ_TRY(launch_k(e->lo, pq::set_int_kernel, dim3(1), dim3(32), 0, e->main, e->out_steps,
                  (testing && a->decode_ar && e->arch == 0) ? 0 : L));
  e->launches++;
  for (int b0 = 0; b0 < a->batch; b0 += e->max_batch) {
    const int Bc = (a->batch - b0 < e->max_batch) ? (a->batch - b0) : e->max_batch;
    if (eager && !host && crop_pixels == nullptr) {
      PQ_TRY(forward_super(e, a, b0, Bc, L, images + b0 * img_sz, u8, logits + 1ll * b0 * L * e->C,
                           ids ? ids + 1ll * b0 * L : nullptr, e->out_steps));
      continue;
    }
    if (host && !eager && e->arch == 0 && Bc >= 256 && e->chunk >= Bc && crop_pixels == nullptr) {
      // upload in two halves on the copy stream; the encoder of the first half (its own graph) runs under the second upload
      const int split = ((Bc / 2 + 7) / 8) * 8;
      PQ_CUDA(cudaEventRecord(e->ev_c[2], e->main));                       // previous work on `main` (and the caller's stream)
      PQ_CUDA(cudaStreamWaitEvent(e->copy, e->ev_c[2], 0));
      PQ_CUDA(cudaMemcpyAsync(in_static, images + b0 * img_sz, static_cast<size_t>(split * img_sz), kin, e->copy));
      PQ_CUDA(cudaEventRecord(e->ev_c[0], e->copy));
      PQ_CUDA(cudaMemcpyAsync(static_cast<char*>(in_static) + split * img_sz, images + (b0 + split) * img_sz,
                              static_cast<size_t>((Bc - split) * img_sz), kin, e->copy));
      PQ_CUDA(cudaEventRecord(e->ev_c[1], e->copy));
      PQ_CUDA(cudaStreamWaitEvent(e->main, e->ev_c[0], 0));
      PQ_TRY(run_graph(e, a, Bc, L, u8, 1, split));
      PQ_CUDA(cudaStreamWaitEvent(e->main, e->ev_c[1], 0));
      PQ_TRY(run_graph(e, a, Bc, L, u8, 2, split));
      PQ_CUDA(cudaMemcpyAsync(logits + 1ll * b0 * L * e->C, e->out_logits, static_cast<size_t>(1ll * Bc * L * e->C) * 4, kout,
                              e->main));
      if (ids) PQ_CUDA(cudaMemcpyAsync(ids + 1ll * b0 * L, e->out_ids, static_cast<size_t>(1ll * Bc * L) * 4, kout, e->main));
      continue;
    }
    if (crop_pixels != nullptr)
      PQ_TRY(rz_launch(e, crop_pixels, b0, Bc, e->in_images_u8, e->main));
    else
      PQ_CUDA(cudaMemcpyAsync(in_static, images + b0 * img_sz, static_cast<size_t>(Bc * img_sz), kin, e->main));
    if (eager) {
      PQ_TRY(forward_super(e, a, b0, Bc, L, in_static, u8, e->out_logits, e->out_ids, e->out_steps));
    } else {
      PQ_TRY(run_graph(e, a, Bc, L, u8));
    }
    PQ_CUDA(cudaMemcpyAsync(logits + 1ll * b0 * L * e->C, e->out_logits, static_cast<size_t>(1ll * Bc * L * e->C) * 4, kout,
                            e->main));
    if (ids) PQ_CUDA(cudaMemcpyAsync(ids + 1ll * b0 * L, e->out_ids, static_cast<size_t>(1ll * Bc * L) * 4, kout, e->main));
  }
  if (steps) PQ_CUDA(cudaMemcpyAsync(steps, e->out_steps, 4, kout, e->main));
  // main -> user stream
  PQ_CUDA(cudaEventRecord(e->ev_out, e->main));
  PQ_CUDA(cudaStreamWaitEvent(user, e->ev_out, 0));
  return PARSEQ_OK;
}

}  // namespace

// =============================================================================== C ABI
extern "C" {

const char* parseq_last_error(void) { return g_last_error.c_str(); }
const char* parseq_version(void) { return "parseq_b200 0.1 (sm_100a, tcgen05/TMA)"; }

int parseq_create(const parseq_config* cfg, parseq_engine** out) {
  if (cfg == nullptr || out == nullptr) return fail(PARSEQ_ERR_INVALID_ARG, "null argument");
  *out = nullptr;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
    return fail(PARSEQ_ERR_NO_DEVICE, "no CUDA device: parseq_b200 has no CPU fallback");
  if (cfg->device < 0 || cfg->device >= ndev) return fail(PARSEQ_ERR_INVALID_ARG, "bad device ordinal");
  PQ_CUDA(cudaSetDevice(cfg->device));
  cudaDeviceProp prop;
  PQ_CUDA(cudaGetDeviceProperties(&prop, cfg->device));
  if (prop.major != 10)
    return fail(PARSEQ_ERR_NO_DEVICE, std::string("device is sm_") + std::to_string(prop.major * 10 + prop.minor) +
                                          ", the kernels are sm_100a (B200) only");
  const int sm_count = prop.multiProcessorCount;
  PQ_TRY(init_kernel_attributes());
  PQ_TRY(load_driver_api());
  if (cfg->arch != 0 && cfg->arch != 1) return fail(PARSEQ_ERR_INVALID_ARG, "arch: 0 (PARSeq) or 1 (ViTSTR)");
  const bool vitstr = cfg->arch == 1;
  if (!vitstr && cfg->dec_depth != 1) return fail(PARSEQ_ERR_UNSUPPORTED, "dec_depth must be 1");
  if (cfg->img_h % cfg->patch_h || cfg->img_w % cfg->patch_w) return fail(PARSEQ_ERR_INVALID_ARG, "img/patch mismatch");
  const int D = cfg->embed_dim;
  if (D != 192 && D != 384 && D != 768) return fail(PARSEQ_ERR_UNSUPPORTED, "embed_dim must be 192, 384 or 768");
  if (D != cfg->enc_num_heads * 64) return fail(PARSEQ_ERR_UNSUPPORTED, "encoder head_dim must be 64");
  if (!vitstr && D != cfg->dec_num_heads * 32) return fail(PARSEQ_ERR_UNSUPPORTED, "decoder head_dim must be 32");
  if (cfg->max_label_length + 1 > 32) return fail(PARSEQ_ERR_UNSUPPORTED, "max_label_length must be <= 31");
  if (cfg->max_label_length < 0) return fail(PARSEQ_ERR_INVALID_ARG, "negative max_label_length");
  // the head tiles of the decoder kernels hold one row of logits in 128 columns (charset_train of <= 126 characters;
  // the reference's largest, 94_full, has 94)
  if (cfg->num_tokens < 4 || cfg->num_tokens - 2 > 128)
    return fail(PARSEQ_ERR_UNSUPPORTED, "num_tokens must be in [4, 130] (at most 128 head classes)");
  if (cfg->enc_mlp_ratio < 1 || cfg->enc_depth < 1) return fail(PARSEQ_ERR_INVALID_ARG, "enc_mlp_ratio / enc_depth");
  // decoder MLP: 128-wide linear1 tiles and a 3-way split-K of linear2 in 64-element k-blocks
  if (!vitstr && (cfg->dec_mlp_ratio < 1 || (D * cfg->dec_mlp_ratio) % 384 != 0))
    return fail(PARSEQ_ERR_UNSUPPORTED, "embed_dim * dec_mlp_ratio must be a multiple of 384");
  auto* e = new parseq_engine();
  e->cfg = *cfg;
  e->lo = g_default_opts;         // process defaults (parseq_set_option(NULL, ...)) seed a new handle
  e->lo.sm_count = sm_count;
  if (vitstr) {                     // no decoder: neutral values keep the (unused) decoder workspace sizes sane
    e->cfg.dec_num_heads = D / 32;
    e->cfg.dec_mlp_ratio = 1;
    e->cfg.dec_depth = 0;
  }
  cfg = &e->cfg;
  e->arch = cfg->arch;
  e->D = D;
  e->gh = cfg->img_h / cfg->patch_h;
  e->gw = cfg->img_w / cfg->patch_w;
  e->Tp = e->gh * e->gw;
  e->T = e->Tp + (vitstr ? 1 : 0);   // class token (timm VisionTransformer default, kept by vitstr/model.py)
  e->Kp = 3 * cfg->patch_h * cfg->patch_w;
  e->Me = D * cfg->enc_mlp_ratio;
  e->Md = D * cfg->dec_mlp_ratio;
  e->L = cfg->max_label_length + 1;
  e->V = cfg->num_tokens;
  e->C = cfg->num_tokens - 2;
  e->dh_dec = D / cfg->dec_num_heads;
  e->max_batch = cfg->max_batch > 0 ? cfg->max_batch : 512;
  // One pipeline stage per super-chunk by default: measured on B200 the decoder chain is latency-bound and the
  // encoder GEMMs occupy every SM, so splitting into stages only shrinks the GEMMs ("chunk" option re-enables it).
  e->chunk = e->max_batch;
  e->dec_chunk = e->max_batch < 128 ? e->max_batch : 128;
  if (e->T > 256) {
    delete e;
    return fail(PARSEQ_ERR_UNSUPPORTED, "at most 256 image tokens (img_size / patch_size) are supported");
  }
  if (vitstr && e->Tp < e->L) {     // vitstr/model.py:21 slices max_length + 2 tokens out of the T + 1 available
    delete e;
    return fail(PARSEQ_ERR_UNSUPPORTED, "ViTSTR needs at least max_label_length + 1 patches");
  }
  if ((e->Kp * 2) % 16 != 0) { delete e; return fail(PARSEQ_ERR_UNSUPPORTED, "patch dim must be a multiple of 8"); }
  // ---- weight slots: state_dict keys of strhub.models.parseq.model.PARSeq ----
  // ---- (arch 1: keys of vitstr.model.ViTSTR = timm VisionTransformer; the public names drop "encoder.") ----
  if (vitstr) add_slot(e, "encoder.cls_token", D, false);
  add_slot(e, "encoder.pos_embed", 1ll * e->T * D, false);
  add_slot(e, "encoder.patch_embed.proj.weight", 1ll * D * e->Kp, true);
  add_slot(e, "encoder.patch_embed.proj.bias", D, false);
  for (int i = 0; i < cfg->enc_depth; ++i) {
    const std::string p = "encoder.blocks." + std::to_string(i) + ".";
    add_slot(e, p + "norm1.weight", D, false);
    add_slot(e, p + "norm1.bias", D, false);
    add_slot(e, p + "attn.qkv.weight", 3ll * D * D, true);
    add_slot(e, p + "attn.qkv.bias", 3 * D, false);
    add_slot(e, p + "attn.proj.weight", 1ll * D * D, true);
    add_slot(e, p + "attn.proj.bias", D, false);
    add_slot(e, p + "norm2.weight", D, false);
    add_slot(e, p + "norm2.bias", D, false);
    add_slot(e, p + "mlp.fc1.weight", 1ll * e->Me * D, true);
    add_slot(e, p + "mlp.fc1.bias", e->Me, false);
    add_slot(e, p + "mlp.fc2.weight", 1ll * D * e->Me, true);
    add_slot(e, p + "mlp.fc2.bias", D, false);
  }
  add_slot(e, "encoder.norm.weight", D, false);
  add_slot(e, "encoder.norm.bias", D, false);
  const std::string Ly = "decoder.layers.0.";
  if (!vitstr) {
    for (const char* att : {"self_attn", "cross_attn"}) {
      add_slot(e, Ly + att + ".in_proj_weight", 3ll * D * D, true);
      add_slot(e, Ly + att + ".in_proj_bias", 3 * D, false);
      add_slot(e, Ly + att + ".out_proj.weight", 1ll * D * D, true);
      add_slot(e, Ly + att + ".out_proj.bias", D, false);
    }
    add_slot(e, Ly + "linear1.weight", 1ll * e->Md * D, true);
    add_slot(e, Ly + "linear1.bias", e->Md, false);
    add_slot(e, Ly + "linear2.weight", 1ll * D * e->Md, true);
    add_slot(e, Ly + "linear2.bias", D, false);
    for (const char* n : {"norm1", "norm2", "norm_q", "norm_c"}) {
      add_slot(e, Ly + n + ".weight", D, false);
      add_slot(e, Ly + n + ".bias", D, false);
    }
    add_slot(e, "decoder.norm.weight", D, false);
    add_slot(e, "decoder.norm.bias", D, false);
  }
  add_slot(e, "head.weight", 1ll * e->C * D, true);
  add_slot(e, "head.bias", e->C, false);
  if (!vitstr) {
    add_slot(e, "text_embed.embedding.weight", 1ll * e->V * D, false);
    add_slot(e, "pos_queries", 1ll * e->L * D, false);
  }
  for (auto& s : e->slots) {
    // +64 elements of slack: head.bias (95 floats) is read with float4 only when in range, but keep
    // every buffer 16-byte padded
    const size_t bytes = static_cast<size_t>(s.numel + 64) * (s.bf16 ? 2 : 4);
    if (cudaMalloc(&s.dev, bytes) != cudaSuccess) { parseq_destroy(e); return fail(PARSEQ_ERR_CUDA, "cudaMalloc weights"); }
    cudaMemset(s.dev, 0, bytes);
  }
  int r = dev_alloc(&e->kvtab, 1ll * e->L * e->V * 2 * D);
  if (r == PARSEQ_OK) r = dev_alloc(&e->qs, 1ll * e->L * D);
  if (r == PARSEQ_OK) r = alloc_workspace(e);
  if (r == PARSEQ_OK && cudaStreamCreateWithFlags(&e->main, cudaStreamNonBlocking) != cudaSuccess) r = fail(PARSEQ_ERR_CUDA, "stream");
  if (r == PARSEQ_OK && cudaStreamCreateWithFlags(&e->copy, cudaStreamNonBlocking) != cudaSuccess) r = fail(PARSEQ_ERR_CUDA, "stream");
  for (int i = 0; i < 3 && r == PARSEQ_OK; ++i)
    if (cudaEventCreateWithFlags(&e->ev_c[i], cudaEventDisableTiming) != cudaSuccess) r = fail(PARSEQ_ERR_CUDA, "event");
  if (r == PARSEQ_OK && (cudaEventCreateWithFlags(&e->ev_in, cudaEventDisableTiming) != cudaSuccess ||
                         cudaEventCreateWithFlags(&e->ev_out, cudaEventDisableTiming) != cudaSuccess))
    r = fail(PARSEQ_ERR_CUDA, "event");
  if (r != PARSEQ_OK) { parseq_destroy(e); return r; }
  *out = e;
  return PARSEQ_OK;
}

void parseq_destroy(parseq_engine* e) {
  if (e == nullptr) return;
  cudaSetDevice(e->cfg.device);
  cudaDeviceSynchronize();
  for (auto& s : e->slots)
    if (s.dev) cudaFree(s.dev);
  if (e->kvtab) cudaFree(e->kvtab);
  if (e->qs) cudaFree(e->qs);
  free_workspace(e);
  for (void* p : {static_cast<void*>(e->rz_crops), static_cast<void*>(e->rz_tasks), static_cast<void*>(e->rz_stage)})
    if (p) cudaFree(p);
  if (e->main) cudaStreamDestroy(e->main);
  if (e->copy) cudaStreamDestroy(e->copy);
  for (auto ev : e->ev_c) if (ev) cudaEventDestroy(ev);
  if (e->ev_in) cudaEventDestroy(e->ev_in);
  if (e->ev_out) cudaEventDestroy(e->ev_out);
  for (auto& t : e->timed) { cudaEventDestroy(t.a); cudaEventDestroy(t.b); }
  for (auto ev : e->event_pool) cudaEventDestroy(ev);
  delete e;
}

int parseq_num_weights(const parseq_engine* e) { return e ? static_cast<int>(e->slots.size()) : 0; }
const char* parseq_weight_key(const parseq_engine* e, int i, int64_t* numel) {
  if (e == nullptr || i < 0 || i >= static_cast<int>(e->slots.size())) return nullptr;
  if (numel) *numel = e->slots[i].numel;
  return e->slots[i].pub.c_str();
}

int parseq_set_weight(parseq_engine* e, const char* key, const float* data, int64_t numel) {
  if (e == nullptr || key == nullptr || data == nullptr) return fail(PARSEQ_ERR_INVALID_ARG, "null argument");
  auto it = e->pub_index.find(key);
  if (it == e->pub_index.end()) return fail(PARSEQ_ERR_INVALID_ARG, std::string("unexpected state_dict key: ") + key);
  Slot& s = e->slots[it->second];
  if (numel != s.numel)
    return fail(PARSEQ_ERR_INVALID_ARG, std::string("size mismatch for ") + key + ": got " + std::to_string(numel) +
                                            ", expected " + std::to_string(s.numel));
  PQ_CUDA(cudaSetDevice(e->cfg.device));
  if (s.bf16) {
    std::vector<uint16_t> tmp(static_cast<size_t>(numel));
    for (int64_t i = 0; i < numel; ++i) tmp[static_cast<size_t>(i)] = f32_to_bf16_rne(data[i]);
    PQ_CUDA(cudaMemcpy(s.dev, tmp.data(), tmp.size() * 2, cudaMemcpyHostToDevice));
  } else {
    PQ_CUDA(cudaMemcpy(s.dev, data, static_cast<size_t>(numel) * 4, cudaMemcpyHostToDevice));
  }
  s.set = true;
  e->finalized = false;
  return PARSEQ_OK;
}

int parseq_finalize(parseq_engine* e, parseq_stream_t stream) {
  if (e == nullptr) return fail(PARSEQ_ERR_INVALID_ARG, "null engine");
  for (auto& s : e->slots)
    if (!s.set) return fail(PARSEQ_ERR_STATE, "weight not set: " + s.pub);
  PQ_CUDA(cudaSetDevice(e->cfg.device));
  if (e->arch == 1) {               // ViTSTR has no input-independent tables
    e->finalized = true;
    return PARSEQ_OK;
  }
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const int D = e->D, L = e->L, V = e->V;
  const std::string Ly = "decoder.layers.0.";
  const long long rows = 1ll * L * V;
  float* ctx = nullptr;
  __nv_bfloat16* ctxn = nullptr;
  __nv_bfloat16* qn = nullptr;
  int r = dev_alloc(&ctx, rows * D);
  if (r == PARSEQ_OK) r = dev_alloc(&ctxn, rows * D);
  if (r == PARSEQ_OK) r = dev_alloc(&qn, 1ll * L * D);
  if (r != PARSEQ_OK) { cudaFree(ctx); cudaFree(ctxn); cudaFree(qn); return r; }
  pq::build_ctx_rows_kernel<<<1024, 256, 0, st>>>(e->wf("text_embed.embedding.weight"), e->wf("pos_queries"), ctx, L, V, D,
                                                  std::sqrt(static_cast<float>(D)));
  if (cudaGetLastError() != cudaSuccess) r = fail(PARSEQ_ERR_CUDA, "build_ctx_rows_kernel launch");
  if (r == PARSEQ_OK) r = layernorm_launch(e->lo, ctx, e->wf(Ly + "norm_c.weight"), e->wf(Ly + "norm_c.bias"), 1e-5f, static_cast<int>(rows), D,
                           ctxn, nullptr, st);
  // content K/V for every (position, token): rows D..3D-1 of self_attn.in_proj (enc-dec packed projection)
  if (r == PARSEQ_OK)
    r = gemm_launch(e->lo, ctxn, D, e->wb(Ly + "self_attn.in_proj_weight") + 1ll * D * D, D,
                    e->wf(Ly + "self_attn.in_proj_bias") + D, static_cast<int>(rows), 2 * D, D, pq::EPI_BF16, 1.0f, nullptr,
                    0, 0, e->kvtab, 2 * D, st);
  // query projections of the (input independent) position queries, pre-scaled by 1/sqrt(head_dim)
  if (r == PARSEQ_OK)
    r = layernorm_launch(e->lo, e->wf("pos_queries"), e->wf(Ly + "norm_q.weight"), e->wf(Ly + "norm_q.bias"), 1e-5f, L, D, qn,
                         nullptr, st);
  if (r == PARSEQ_OK)
    r = gemm_launch(e->lo, qn, D, e->wb(Ly + "self_attn.in_proj_weight"), D, e->wf(Ly + "self_attn.in_proj_bias"), L, D, D,
                    pq::EPI_F32, 1.0f / std::sqrt(static_cast<float>(e->dh_dec)), nullptr, 0, 0, e->qs, D, st);
  cudaError_t ce = cudaStreamSynchronize(st);
  cudaFree(ctx);
  cudaFree(ctxn);
  cudaFree(qn);
  if (r != PARSEQ_OK) return r;
  if (ce != cudaSuccess) return fail(PARSEQ_ERR_CUDA, std::string("finalize: ") + cudaGetErrorString(ce));
  e->ar2_maps_ok = false;
  if (ar2_supported(e)) PQ_TRY(ar2_build_maps(e));
  e->finalized = true;
  return PARSEQ_OK;
}

int parseq_forward(parseq_engine* e, const parseq_forward_args* a, const float* images, float* logits, int32_t* ids,
                   int32_t* steps, parseq_stream_t stream) {
  if (e == nullptr || a == nullptr || images == nullptr || logits == nullptr)
    return fail(PARSEQ_ERR_INVALID_ARG, "null argument");
  if (e->broken) return fail(PARSEQ_ERR_STATE, "engine workspace is gone (a failed resize): destroy the handle");
  if (!e->finalized) return fail(PARSEQ_ERR_STATE, "parseq_finalize has not been called after the last weight update");
  if (a->batch < 0 || a->refine_iters < 0) return fail(PARSEQ_ERR_INVALID_ARG, "negative batch / refine_iters");
  if (a->batch == 0) return PARSEQ_OK;
  PQ_CUDA(cudaSetDevice(e->cfg.device));
  return forward_impl(e, a, images, logits, ids, steps, reinterpret_cast<cudaStream_t>(stream), false);
}

int parseq_forward_host(parseq_engine* e, const parseq_forward_args* a, const float* images_host, float* logits_host,
                        int32_t* ids_host, int32_t* steps_host, parseq_stream_t stream) {
  if (e == nullptr || a == nullptr || images_host == nullptr || logits_host == nullptr)
    return fail(PARSEQ_ERR_INVALID_ARG, "null argument");
  if (e->broken) return fail(PARSEQ_ERR_STATE, "engine workspace is gone (a failed resize): destroy the handle");
  if (!e->finalized) return fail(PARSEQ_ERR_STATE, "parseq_finalize has not been called after the last weight update");
  if (a->batch < 0 || a->refine_iters < 0) return fail(PARSEQ_ERR_INVALID_ARG, "negative batch / refine_iters");
  if (a->batch == 0) return PARSEQ_OK;
  if (a->forced_ids != nullptr || a->forced_refine != nullptr)
    return fail(PARSEQ_ERR_INVALID_ARG, "teacher forcing is a device-pointer API (parseq_forward)");
  PQ_CUDA(cudaSetDevice(e->cfg.device));
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  PQ_TRY(forward_impl(e, a, images_host, logits_host, ids_host, steps_host, st, true));
  PQ_CUDA(cudaStreamSynchronize(e->main));
  return PARSEQ_OK;
}

int parseq_forward_u8(parseq_engine* e, const parseq_forward_args* a, const uint8_t* images_hwc, float* logits, int32_t* ids,
                      int32_t* steps, parseq_stream_t stream) {
  if (e == nullptr || a == nullptr || images_hwc == nullptr || logits == nullptr)
    return fail(PARSEQ_ERR_INVALID_ARG, "null argument");
  if (e->broken) return fail(PARSEQ_ERR_STATE, "engine workspace is gone (a failed resize): destroy the handle");
  if (!e->finalized) return fail(PARSEQ_ERR_STATE, "parseq_finalize has not been called after the last weight update");
  if (a->batch < 0 || a->refine_iters < 0) return fail(PARSEQ_ERR_INVALID_ARG, "negative batch / refine_iters");
  if (a->batch == 0) return PARSEQ_OK;
  PQ_CUDA(cudaSetDevice(e->cfg.device));
  return forward_impl(e, a, images_hwc, logits, ids, steps, reinterpret_cast<cudaStream_t>(stream), false, true);
}

int parseq_forward_host_u8(parseq_engine* e, const parseq_forward_args* a, const uint8_t* images_hwc_host, float* logits_host,
                           int32_t* ids_host, int32_t* steps_host, parseq_stream_t stream) {
  if (e == nullptr || a == nullptr || images_hwc_host == nullptr || logits_host == nullptr)
    return fail(PARSEQ_ERR_INVALID_ARG, "null argument");
  if (e->broken) return fail(PARSEQ_ERR_STATE, "engine workspace is gone (a failed resize): destroy the handle");
  if (!e->finalized) return fail(PARSEQ_ERR_STATE, "parseq_finalize has not been called after the last weight update");
  if (a->batch < 0 || a->refine_iters < 0) return fail(PARSEQ_ERR_INVALID_ARG, "negative batch / refine_iters");
  if (a->batch == 0) return PARSEQ_OK;
  if (a->forced_ids != nullptr || a->forced_refine != nullptr)
    return fail(PARSEQ_ERR_INVALID_ARG, "teacher forcing is a device-pointer API (parseq_forward)");
  PQ_CUDA(cudaSetDevice(e->cfg.device));
  PQ_TRY(forward_impl(e, a, images_hwc_host, logits_host, ids_host, steps_host, reinterpret_cast<cudaStream_t>(stream), true, true));
  PQ_CUDA(cudaStreamSynchronize(e->main));
  return PARSEQ_OK;
}

int parseq_forward_crops(parseq_engine* e, const parseq_forward_args* a, const parseq_crops* crops, float* logits, int32_t* ids,
                         int32_t* steps, parseq_stream_t stream) {
  if (e == nullptr || a == nullptr || crops == nullptr || logits == nullptr)
    return fail(PARSEQ_ERR_INVALID_ARG, "null argument");
  if (e->broken) return fail(PARSEQ_ERR_STATE, "engine workspace is gone (a failed resize): destroy the handle");
  if (!e->finalized) return fail(PARSEQ_ERR_STATE, "parseq_finalize has not been called after the last weight update");
  if (a->batch < 0 || a->refine_iters < 0) return fail(PARSEQ_ERR_INVALID_ARG, "negative batch / refine_iters");
  if (crops->count != a->batch) return fail(PARSEQ_ERR_INVALID_ARG, "crops->count != args->batch");
  PQ_CUDA(cudaSetDevice(e->cfg.device));
  const uint8_t* px = nullptr;
  PQ_TRY(rz_prepare(e, crops, false, &px));
  if (a->batch == 0) return PARSEQ_OK;
  return forward_impl(e, a, nullptr, logits, ids, steps, reinterpret_cast<cudaStream_t>(stream), false, true, px);
}

int parseq_forward_host_crops(parseq_engine* e, const parseq_forward_args* a, const parseq_crops* crops, float* logits_host,
                              int32_t* ids_host, int32_t* steps_host, parseq_stream_t stream) {
  if (e == nullptr || a == nullptr || crops == nullptr || logits_host == nullptr)
    return fail(PARSEQ_ERR_INVALID_ARG, "null argument");
  if (e->broken) return fail(PARSEQ_ERR_STATE, "engine workspace is gone (a failed resize): destroy the handle");
  if (!e->finalized) return fail(PARSEQ_ERR_STATE, "parseq_finalize has not been called after the last weight update");
  if (a->batch < 0 || a->refine_iters < 0) return fail(PARSEQ_ERR_INVALID_ARG, "negative batch / refine_iters");
  if (crops->count != a->batch) return fail(PARSEQ_ERR_INVALID_ARG, "crops->count != args->batch");
  if (a->forced_ids != nullptr || a->forced_refine != nullptr)
    return fail(PARSEQ_ERR_INVALID_ARG, "teacher forcing is a device-pointer API (parseq_forward)");
  PQ_CUDA(cudaSetDevice(e->cfg.device));
  const uint8_t* px = nullptr;
  PQ_TRY(rz_prepare(e, crops, true, &px));
  if (a->batch == 0) return PARSEQ_OK;
  PQ_TRY(forward_impl(e, a, nullptr, logits_host, ids_host, steps_host, reinterpret_cast<cudaStream_t>(stream), true, true, px));
  PQ_CUDA(cudaStreamSynchronize(e->main));
  return PARSEQ_OK;
}

int parseq_resize_crops(parseq_engine* e, const parseq_crops* crops, uint8_t* out_hwc, parseq_stream_t stream) {
  if (e == nullptr || crops == nullptr || out_hwc == nullptr) return fail(PARSEQ_ERR_INVALID_ARG, "null argument");
  PQ_CUDA(cudaSetDevice(e->cfg.device));
  const uint8_t* px = nullptr;
  PQ_TRY(rz_prepare(e, crops, false, &px));
  if (crops->count == 0) return PARSEQ_OK;
  cudaStream_t user = reinterpret_cast<cudaStream_t>(stream);
  PQ_CUDA(cudaEventRecord(e->ev_in, user));
  PQ_CUDA(cudaStreamWaitEvent(e->main, e->ev_in, 0));
  PQ_TRY(rz_launch(e, px, 0, crops->count, out_hwc, e->main));
  PQ_CUDA(cudaEventRecord(e->ev_out, e->main));
  PQ_CUDA(cudaStreamWaitEvent(user, e->ev_out, 0));
  return PARSEQ_OK;
}

int parseq_postprocess(const float* logits, int32_t batch, int32_t num_steps, int32_t num_classes, int32_t eos_id, int32_t* ids,
                       int32_t* lengths, float* confidence, parseq_stream_t stream) {
  if (logits == nullptr || ids == nullptr || lengths == nullptr || confidence == nullptr)
    return fail(PARSEQ_ERR_INVALID_ARG, "null argument");
  if (batch <= 0) return batch == 0 ? PARSEQ_OK : fail(PARSEQ_ERR_INVALID_ARG, "negative batch");
  pq::postprocess_kernel<<<(batch + 7) / 8, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(logits, batch, num_steps, num_classes,
                                                                                              eos_id, ids, lengths, confidence);
  PQ_CUDA(cudaGetLastError());
  return PARSEQ_OK;
}

int parseq_encode(parseq_engine* e, int32_t batch, const float* images, float* memory, parseq_stream_t stream) {
  if (e == nullptr || images == nullptr || memory == nullptr) return fail(PARSEQ_ERR_INVALID_ARG, "null argument");
  if (e->broken) return fail(PARSEQ_ERR_STATE, "engine workspace is gone (a failed resize): destroy the handle");
  if (!e->finalized) return fail(PARSEQ_ERR_STATE, "parseq_finalize has not been called");
  PQ_CUDA(cudaSetDevice(e->cfg.device));
  cudaStream_t user = reinterpret_cast<cudaStream_t>(stream);
  PQ_CUDA(cudaEventRecord(e->ev_in, user));
  PQ_CUDA(cudaStreamWaitEvent(e->main, e->ev_in, 0));
  const long long img_sz = 3ll * e->cfg.img_h * e->cfg.img_w;
  for (int b0 = 0; b0 < batch; b0 += e->chunk) {
    const int B = (batch - b0 < e->chunk) ? (batch - b0) : e->chunk;
    PQ_TRY(encode_chunk(e, images + b0 * img_sz, false, B, e->mem, memory + 1ll * b0 * e->T * e->D, e->main));
  }
  PQ_CUDA(cudaEventRecord(e->ev_out, e->main));
  PQ_CUDA(cudaStreamWaitEvent(user, e->ev_out, 0));
  return PARSEQ_OK;
}

int parseq_decode(parseq_engine* e, int32_t batch, int32_t ctx_len, int32_t num_queries, const int32_t* tgt, const float* memory,
                  const float* query, const uint8_t* query_mask, const uint8_t* padding_mask, float* out,
                  parseq_stream_t stream) {
  if (e == nullptr || tgt == nullptr || memory == nullptr || out == nullptr) return fail(PARSEQ_ERR_INVALID_ARG, "null argument");
  if (e->broken) return fail(PARSEQ_ERR_STATE, "engine workspace is gone (a failed resize): destroy the handle");
  if (!e->finalized) return fail(PARSEQ_ERR_STATE, "parseq_finalize has not been called");
  if (e->arch != 0) return fail(PARSEQ_ERR_UNSUPPORTED, "decode: PARSeq only");
  if (batch < 0 || ctx_len < 1 || ctx_len > e->L || num_queries < 1 || num_queries > e->L)
    return fail(PARSEQ_ERR_INVALID_ARG, "decode: 1 <= context length, queries <= max_label_length + 1");
  if (batch == 0) return PARSEQ_OK;
  PQ_CUDA(cudaSetDevice(e->cfg.device));
  cudaStream_t user = reinterpret_cast<cudaStream_t>(stream);
  PQ_CUDA(cudaEventRecord(e->ev_in, user));
  PQ_CUDA(cudaStreamWaitEvent(e->main, e->ev_in, 0));
  const int D = e->D, T = e->T, J = ctx_len, NQ = num_queries;
  const std::string Ly = "decoder.layers.0.";
  const __nv_bfloat16* Wkv = e->wb(Ly + "cross_attn.in_proj_weight") + static_cast<long long>(D) * D;
  const float* bkv = e->wf(Ly + "cross_attn.in_proj_bias") + D;
  parseq_engine::Stage& sg = e->stages[0];
  cudaStream_t st = e->main;
  for (int b0 = 0; b0 < batch; b0 += e->dec_chunk) {
    const int Bc = (batch - b0 < e->dec_chunk) ? (batch - b0) : e->dec_chunk;
    // memory (fp32, caller's) -> bf16 operand -> cross K/V cache rows [0, Bc * T)
    const long long n4 = 1ll * Bc * T * D / 4;
    pq::f32_to_bf16_kernel<<<static_cast<unsigned>(std::min<long long>((n4 + 255) / 256, 148ll * 8)), 256, 0, st>>>(
        reinterpret_cast<const float4*>(memory + 1ll * b0 * T * D), reinterpret_cast<uint2*>(e->mem), n4);
    PQ_CUDA(cudaGetLastError());
    e->cur_cat = CAT_DEC_GEMM;
    PQ_TRY(gemm(e, e->mem, D, Wkv, D, bkv, Bc * T, 2 * D, D, pq::EPI_BF16, 1.0f, nullptr, 0, 0, e->ckv, 2 * D, st,
                1ll * e->max_batch * T));
    pq::copy_ids_kernel<<<(Bc * 32 + 255) / 256, 256, 0, st>>>(tgt + 1ll * b0 * J, J, sg.ids_ctx, Bc);
    PQ_CUDA(cudaGetLastError());
    e->launches += 2;
    DecodeExtras ex;
    ex.query = query ? query + 1ll * b0 * NQ * D : nullptr;
    ex.qmask = query_mask;
    ex.pmask = padding_mask ? padding_mask + 1ll * b0 * J : nullptr;
    ex.out_norm = out + 1ll * b0 * NQ * D;
    PQ_TRY(decode_pass(e, sg, 0, Bc, NQ, 0, J, 0, sg.ids_ctx, nullptr, 0, nullptr, 0, nullptr, 0, st, &ex));
  }
  PQ_CUDA(cudaEventRecord(e->ev_out, e->main));
  PQ_CUDA(cudaStreamWaitEvent(user, e->ev_out, 0));
  return PARSEQ_OK;
}

int parseq_head(parseq_engine* e, int32_t rows, const float* x, float* logits, parseq_stream_t stream) {
  if (e == nullptr || x == nullptr || logits == nullptr) return fail(PARSEQ_ERR_INVALID_ARG, "null argument");
  if (e->broken || !e->finalized) return fail(PARSEQ_ERR_STATE, "engine not ready");
  if (rows <= 0) return rows == 0 ? PARSEQ_OK : fail(PARSEQ_ERR_INVALID_ARG, "negative rows");
  PQ_CUDA(cudaSetDevice(e->cfg.device));
  cudaStream_t user = reinterpret_cast<cudaStream_t>(stream);
  PQ_CUDA(cudaEventRecord(e->ev_in, user));
  PQ_CUDA(cudaStreamWaitEvent(e->main, e->ev_in, 0));
  const int D = e->D;
  const int cap = e->dec_chunk * e->L;                 // rows of the bf16 staging buffer of a decoder chain
  parseq_engine::Stage& sg = e->stages[0];
  for (int r0 = 0; r0 < rows; r0 += cap) {
    const int n = (rows - r0 < cap) ? (rows - r0) : cap;
    const long long n4 = 1ll * n * D / 4;
    pq::f32_to_bf16_kernel<<<static_cast<unsigned>(std::min<long long>((n4 + 255) / 256, 148ll * 8)), 256, 0, e->main>>>(
        reinterpret_cast<const float4*>(x + 1ll * r0 * D), reinterpret_cast<uint2*>(sg.yn), n4);
    PQ_CUDA(cudaGetLastError());
    e->launches++;
    e->cur_cat = CAT_DEC_GEMM;
    PQ_TRY(gemm(e, sg.yn, D, e->w("head.weight"), D, e->wf("head.bias"), n, e->C, D, pq::EPI_F32, 1.0f, nullptr, 0, 0,
                logits + 1ll * r0 * e->C, e->C, e->main));
  }
  PQ_CUDA(cudaEventRecord(e->ev_out, e->main));
  PQ_CUDA(cudaStreamWaitEvent(user, e->ev_out, 0));
  return PARSEQ_OK;
}

int parseq_text_embed(parseq_engine* e, int32_t n, const int32_t* ids, float* out, parseq_stream_t stream) {
  if (e == nullptr || ids == nullptr || out == nullptr) return fail(PARSEQ_ERR_INVALID_ARG, "null argument");
  if (e->arch != 0) return fail(PARSEQ_ERR_UNSUPPORTED, "text_embed: PARSeq only");
  if (n <= 0) return n == 0 ? PARSEQ_OK : fail(PARSEQ_ERR_INVALID_ARG, "negative count");
  if (!e->slots[e->index.at("text_embed.embedding.weight")].set) return fail(PARSEQ_ERR_STATE, "weights not set");
  PQ_CUDA(cudaSetDevice(e->cfg.device));
  const long long total = 1ll * n * e->D;
  pq::text_embed_kernel<<<static_cast<unsigned>(std::min<long long>((total + 255) / 256, 148ll * 8)), 256, 0,
                          reinterpret_cast<cudaStream_t>(stream)>>>(ids, e->wf("text_embed.embedding.weight"), out, n, e->D, e->V,
                                                                    std::sqrt(static_cast<float>(e->D)));
  PQ_CUDA(cudaGetLastError());
  return PARSEQ_OK;
}

int parseq_bench_tma_stream(void* buf, int64_t bytes, int cluster, int ctas, int nboxes, int nslot, int mode, void* sink,
                            parseq_stream_t stream) {
  if (buf == nullptr || sink == nullptr || cluster < 1 || cluster > 8 || ctas % cluster != 0 || nslot < 1 || nslot > 12)
    return fail(PARSEQ_ERR_INVALID_ARG, "bench_tma_stream: bad arguments");
  const long long rows_total = 8192;                         // rows per 64-column block
  const int blocks = static_cast<int>(bytes / (rows_total * 128));
  if (blocks < 1) return fail(PARSEQ_ERR_INVALID_ARG, "bench_tma_stream: buffer too small");
  CUtensorMap map;
  PQ_TRY(make_tmap3d(&map, buf, 64, rows_total, blocks, 64, 64 * rows_total, 64, 128));
  const int smem = 12 * pq::A2_SLOT + 1024 + 256;
  PQ_CUDA(cudaFuncSetAttribute(pq::tma_stream_bench_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(static_cast<unsigned>(ctas));
  cfg.blockDim = dim3(pq::A2_THREADS + 32);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = reinterpret_cast<cudaStream_t>(stream);
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = static_cast<unsigned>(cluster);
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = cluster > 1 ? 1 : 0;
  PQ_CUDA(cudaLaunchKernelEx(&cfg, pq::tma_stream_bench_kernel, map, nboxes, nslot, static_cast<int>(rows_total / 128), blocks, mode,
                             static_cast<unsigned int*>(sink)));
  return PARSEQ_OK;
}

int64_t parseq_debug_int(parseq_engine* e, const char* name) {
  if (e == nullptr || name == nullptr) return -1;
  const std::string n(name);
  if (n == "ar2_occupancy_mt1_cs8") return e->ar2_occ[1][0];
  if (n == "ar2_occupancy_mt2_cs8") return e->ar2_occ[2][0];
  if (n == "ar2_occupancy_mt1_cs6") return e->ar2_occ[1][1];
  if (n == "ar2_occupancy_mt2_cs6") return e->ar2_occ[2][1];
  if (n == "ar_last_cluster_size") return e->ar_last_cs;
  if (n == "ar_last_per") return e->ar_last_per;
  if (n == "ar_last_clusters") return e->ar_last_ncl;
  if (n == "sm_count") return e->lo.sm_count;
  return -1;
}
int64_t parseq_kernel_launches(const parseq_engine* e) { return e ? e->launches : 0; }

int parseq_set_option(parseq_engine* e, const char* name, int64_t value) {
  if (name == nullptr) return fail(PARSEQ_ERR_INVALID_ARG, "null option");
  const std::string n(name);
  // launch options: per handle; with a NULL handle they set the process defaults used by the bare kernel exports
  // (parseq_gemm_bf16 & co.) and inherited by handles created afterwards
  LaunchOpts& lo = e ? e->lo : g_default_opts;
  if (n == "block_n") {
    if (value != 0 && value != 64 && value != 128 && value != 192 && value != 256)
      return fail(PARSEQ_ERR_INVALID_ARG, "block_n: 0/64/128/192/256");
    lo.block_n = static_cast<int>(value);
    if (e) drop_graphs(e);
    return PARSEQ_OK;
  }
  if (n == "attn_impl") { lo.attn_impl = value != 0 ? 1 : 0; if (e) drop_graphs(e); return PARSEQ_OK; }
  if (n == "pdl") { lo.use_pdl = value != 0; if (e) drop_graphs(e); return PARSEQ_OK; }
  if (n == "tma_epilogue") { lo.no_tma_epilogue = (value == 0); if (e) drop_graphs(e); return PARSEQ_OK; }
  if (n == "gemm_stages") { lo.gemm_stages = value > 0 ? static_cast<int>(value) : 0; if (e) drop_graphs(e); return PARSEQ_OK; }
  if (n == "cta_group") {
    if (value < 0 || value > 2) return fail(PARSEQ_ERR_INVALID_ARG, "cta_group: 0 (auto) / 1 / 2");
    lo.cta_group = static_cast<int>(value);
    if (e) drop_graphs(e);
    return PARSEQ_OK;
  }
  if (n == "ln_cta_group") {
    if (value < 0 || value > 2) return fail(PARSEQ_ERR_INVALID_ARG, "ln_cta_group: 0 (auto) / 1 / 2");
    lo.ln_cta_group = static_cast<int>(value);
    if (e) drop_graphs(e);
    return PARSEQ_OK;
  }
  if (n == "ln_split") {
    if (value < 0 || value > 2) return fail(PARSEQ_ERR_INVALID_ARG, "ln_split: 0 (auto) / 1 (off) / 2 (on)");
    lo.ln_split = static_cast<int>(value);
    if (e) drop_graphs(e);
    return PARSEQ_OK;
  }
  if (n == "mlp_cta_group") {
    if (value < 0 || value > 2) return fail(PARSEQ_ERR_INVALID_ARG, "mlp_cta_group: 0 (auto) / 1 / 2");
    lo.mlp_cta_group = static_cast<int>(value);
    if (e) drop_graphs(e);
    return PARSEQ_OK;
  }
  if (n == "pair_pdl") { lo.pair_pdl = value != 0; if (e) drop_graphs(e); return PARSEQ_OK; }
  if (n == "fuse_mlp") {
    if (e == nullptr) return fail(PARSEQ_ERR_INVALID_ARG, "null engine");
    e->fuse_mlp = value != 0 ? 1 : 0;
    drop_graphs(e);
    return PARSEQ_OK;
  }
  if (n == "fuse_ln") {
    if (e == nullptr) return fail(PARSEQ_ERR_INVALID_ARG, "null engine");
    e->fuse_ln = static_cast<int>(value) & 7;
    drop_graphs(e);
    return PARSEQ_OK;
  }
  if (e == nullptr) return fail(PARSEQ_ERR_INVALID_ARG, "null engine");
  if (n == "timing") {
    e->timing = value != 0;
    for (auto& t : e->timed) { e->event_pool.push_back(t.a); e->event_pool.push_back(t.b); }
    e->timed.clear();
    return PARSEQ_OK;
  }
  if (n == "use_graph") { e->use_graph = value != 0; return PARSEQ_OK; }
  if (n == "ar_prof") { e->ar_prof_on = value != 0; drop_graphs(e); return PARSEQ_OK; }
  if (n == "ar_clusters") {
    if (value < 0 || value > 1024) return fail(PARSEQ_ERR_INVALID_ARG, "ar_clusters out of range");
    e->ar_clusters_override = static_cast<int>(value);
    for (auto& r : e->ar2_clusters) r[0] = r[1] = 0;
    drop_graphs(e);
    return PARSEQ_OK;
  }
  if (n == "ar_cluster_size") {
    if (value != 0 && value != 6 && value != 8) return fail(PARSEQ_ERR_INVALID_ARG, "ar_cluster_size: 0 (auto) / 6 / 8");
    e->ar_cs = static_cast<int>(value);
    drop_graphs(e);
    return PARSEQ_OK;
  }
  if (n == "ar_kernel") {           // 0: AR loop as separate kernels, 1: grid-barrier kernel (dec_ar.cuh), 2: cluster kernel
    if (value < 0 || value > 2) return fail(PARSEQ_ERR_INVALID_ARG, "ar_kernel: 0 / 1 / 2");
    e->use_ar_kernel = value != 0;
    e->ar_impl = value == 1 ? 1 : 2;
    drop_graphs(e);
    return PARSEQ_OK;
  }
  if (n == "chunk" || n == "max_batch" || n == "dec_chunk") {
    if (value <= 0 || value > 8192) return fail(PARSEQ_ERR_INVALID_ARG, "chunk / max_batch / dec_chunk out of range");
    // validate the new sizes BEFORE touching the workspace
    int chunk = e->chunk, dec_chunk = e->dec_chunk, max_batch = e->max_batch;
    if (n == "chunk") chunk = static_cast<int>(value);
    else if (n == "dec_chunk") dec_chunk = static_cast<int>(value);
    else { max_batch = static_cast<int>(value); chunk = max_batch; }
    if (chunk > max_batch) chunk = max_batch;
    if (dec_chunk > max_batch) dec_chunk = max_batch;
    if ((max_batch + dec_chunk - 1) / dec_chunk > 64) return fail(PARSEQ_ERR_INVALID_ARG, "too many decoder chains");
    PQ_CUDA(cudaSetDevice(e->cfg.device));
    PQ_CUDA(cudaDeviceSynchronize());
    const int old_chunk = e->chunk, old_dec = e->dec_chunk, old_max = e->max_batch;
    free_workspace(e);
    e->chunk = chunk; e->dec_chunk = dec_chunk; e->max_batch = max_batch;
    int r = alloc_workspace(e);
    if (r != PARSEQ_OK) {            // out of memory: back to the sizes that worked
      const std::string why = g_last_error;
      free_workspace(e);
      e->chunk = old_chunk; e->dec_chunk = old_dec; e->max_batch = old_max;
      if (alloc_workspace(e) != PARSEQ_OK) { e->finalized = false; free_workspace(e); e->broken = true; }
      return fail(r, why);
    }
    return PARSEQ_OK;
  }
  return fail(PARSEQ_ERR_INVALID_ARG, "unknown option: " + n);
}

int parseq_get_ar_profile(parseq_engine* e, uint64_t* out512) {
  if (e == nullptr || out512 == nullptr) return fail(PARSEQ_ERR_INVALID_ARG, "null argument");
  PQ_CUDA(cudaMemcpy(out512, e->ar_prof, 32 * 16 * 8, cudaMemcpyDeviceToHost));
  return PARSEQ_OK;
}

int parseq_get_timing(parseq_engine* e, int category, double* ms, double* flops, int64_t* count) {
  if (e == nullptr || category < 0 || category >= CAT_COUNT) return fail(PARSEQ_ERR_INVALID_ARG, "bad timing query");
  double tms = 0.0, tf = 0.0;
  int64_t n = 0;
  for (auto& t : e->timed) {
    if (t.cat != category) continue;
    float dt = 0.f;
    cudaError_t ce = cudaEventElapsedTime(&dt, t.a, t.b);
    if (ce != cudaSuccess) return fail(PARSEQ_ERR_CUDA, std::string("timing readback: ") + cudaGetErrorString(ce));
    tms += dt; tf += t.flops; ++n;
  }
  if (ms) *ms = tms;
  if (flops) *flops = tf;
  if (count) *count = n;
  return PARSEQ_OK;
}

int parseq_gemm_bf16(const void* A, int64_t lda, const void* W, int64_t ldw, const float* bias, int M, int N, int K,
                     int mode, float alpha, const float* resid, int64_t ldr, int resid_mod, void* out, int64_t ldo,
                     parseq_stream_t stream) {
  if (mode < 0 || mode > 2) return fail(PARSEQ_ERR_INVALID_ARG, "bad epilogue mode");
  return gemm_launch(g_default_opts, A, lda, W, ldw, bias, M, N, K, mode, alpha, resid, ldr, resid_mod, out, ldo,
                     reinterpret_cast<cudaStream_t>(stream));
}
int parseq_gemm_ln_bf16(const void* A, int64_t lda, const void* W, int64_t ldw, const float* bias, int M, int D, int K,
                         float* x_inout, const float* gamma, const float* beta, float eps, void* xn_bf16,
                         parseq_stream_t stream) {
  return gemm_ln_launch(g_default_opts, A, lda, W, ldw, bias, M, D, K, x_inout, gamma, beta, eps, xn_bf16, reinterpret_cast<cudaStream_t>(stream));
}
int parseq_mlp_ln_bf16(const void* xn, const void* W1, const float* b1, const void* W2, const float* b2, int M, int D,
                       float* x_inout, const float* gamma, const float* beta, float eps, void* xn_out_bf16, parseq_stream_t stream) {
  return mlp_ln_launch(g_default_opts, xn, W1, b1, W2, b2, M, D, x_inout, gamma, beta, eps, xn_out_bf16,
                       reinterpret_cast<cudaStream_t>(stream));
}
// same, with 16 cycle counters of CTA 0 written to `prof_dev` (tests/prof_mlp_ln.py; see mlp_ln.cuh for the slots)
int parseq_mlp_ln_bf16_prof(const void* xn, const void* W1, const float* b1, const void* W2, const float* b2, int M, int D,
                            float* x_inout, const float* gamma, const float* beta, float eps, void* xn_out_bf16,
                            unsigned long long* prof_dev, parseq_stream_t stream) {
  return mlp_ln_launch(g_default_opts, xn, W1, b1, W2, b2, M, D, x_inout, gamma, beta, eps, xn_out_bf16,
                       reinterpret_cast<cudaStream_t>(stream), prof_dev);
}
int parseq_layernorm_bf16(const float* x, const float* gamma, const float* beta, float eps, int M, int D, void* y_bf16,
                          float* y_f32_or_null, parseq_stream_t stream) {
  return layernorm_launch(g_default_opts, x, gamma, beta, eps, M, D, y_bf16, y_f32_or_null, reinterpret_cast<cudaStream_t>(stream));
}
int parseq_enc_attention(const void* qkv_bf16, int B, int T, int D, int heads, void* out_bf16, parseq_stream_t stream) {
  PQ_TRY(ensure_sm_count(g_default_opts));
  return enc_attention_launch(g_default_opts, qkv_bf16, B, T, D, heads, out_bf16, reinterpret_cast<cudaStream_t>(stream));
}

}  // extern "C"
