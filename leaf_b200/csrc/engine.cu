// C ABI of the LEAF attack engine (include/leaf_b200.h). Host-side orchestration only: every computation is
// a CUDA kernel launched from here (k1_tokenize.cuh, gemm_sm100.cuh, tower_kernels.cuh). No CPU compute path.
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <map>
#include <string>
#include <tuple>
#include <vector>

#include "../../include/leaf_b200.h"
#include "gemm2_sm100.cuh"
#include "gemm_sm100.cuh"
#include "k1_tables_host.h"
#include "constrain_kernel.cuh"
#include "k1_tokenize.cuh"
#include "tower_kernels.cuh"
#include "attention2.cuh"
#include "train_kernels.cuh"

using namespace leaf;

static thread_local std::string g_err;

static int fail(int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  g_err = buf;
  return code;
}

#define CK(expr)                                                                                       \
  do {                                                                                                 \
    cudaError_t _e = (expr);                                                                           \
    if (_e != cudaSuccess) return fail(LEAF_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), \
                                       __FILE__, __LINE__);                                            \
  } while (0)

typedef CUresult (*encode_tiled_fn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

struct LayerW {
  __nv_bfloat16 *qkv_w = nullptr, *out_w = nullptr, *fc1_w = nullptr, *fc2_w = nullptr;   // engine-owned bf16 copies
  float* qkv_b_own = nullptr;                                                              // HF layout only
  const float* qkv_b = nullptr;
};

struct TrainLayer {        // activations one layer keeps for the backward pass (K4)
  float *x_in = nullptr, *x_mid = nullptr;
  __nv_bfloat16 *h1 = nullptr, *qkv = nullptr, *o = nullptr, *h2 = nullptr, *u = nullptr, *g = nullptr;
};

struct TrainWs {
  int max_seqs = 0;
  long rows_cap = 0;
  int N = 0, M = 0, T = 0;            // sequences / packed rows / longest sequence of the saved forward
  bool have_forward = false;
  int64_t generation = 0;           // of the saved forward (leaf_forward_train counts up)
  std::vector<TrainLayer> L;
  float *x_out = nullptr, *dx = nullptr, *dtmp = nullptr, *scratch = nullptr;
  __nv_bfloat16 *pooled = nullptr, *d16 = nullptr, *dx16 = nullptr;
  float* ln_stats = nullptr;         // (mean, rstd) per row, from the LayerNorm backward's row kernel to its column kernel
  // deterministic mode only (leaf_set_deterministic): partial sums of the fixed-order reductions, their arrival counters (zero
  // between launches) and the embedding backward's row sort (row_tok | order | key, rows_cap each)
  float* det_ws = nullptr;
  int* det_cnt = nullptr;
  int* det_idx = nullptr;
  size_t det_ws_floats = 0, det_cnt_ints = 0;
  int *tok = nullptr, *cu = nullptr, *eos_row = nullptr, *total_rows = nullptr, *pfx = nullptr, *own_len = nullptr;
  int4* meta = nullptr;
  std::vector<void*> allocs;
};

struct leaf_engine {
  leaf_cfg_t cfg;
  int device = 0;
  int sm_count = 148;
  encode_tiled_fn encode_tiled = nullptr;
  // K1 tables
  bool bpe_loaded = false;
  bool hf_tokenizer = false;          // leaf_set_tokenizer_mode
  int max_caption_bytes = LEAF_MAX_CAPTION_BYTES;   // leaf_set_max_caption_bytes
  std::vector<void*> table_allocs;
  K1Tables tables{};
  // --constrain filter: hash sets of the word list and of Punkt abbreviation types
  CnTables cn{};
  bool words_loaded = false;
  int32_t* cn_count = nullptr;
  int cn_count_cap = 0;
  // weights
  bool bound = false;
  leaf_weight_ptrs_t wp{};
  std::vector<leaf_layer_ptrs_t> layer_ptrs;
  std::vector<LayerW> lw;
  __nv_bfloat16* proj_w = nullptr;    // [E, W] bf16
  __nv_bfloat16* proj_w_lo = nullptr; // [E, W] what proj_w's rounding dropped (split-precision final projection of leaf_encode)
  __nv_bfloat16* pooled_lo = nullptr; // [max_seqs, W] likewise for the ln_final output
  TrainWs tw;
  int64_t train_generation = 0;
  leaf_backward_hook_t bwd_hook = nullptr;   // host callback after each layer's gradients are enqueued (leaf_set_backward_hook)
  void* bwd_hook_user = nullptr;
  // workspace
  int max_seqs = 0;
  long rows_cap = 0;
  float* x = nullptr;                 // [rows_cap, W] fp32 residual stream
  __nv_bfloat16* h = nullptr;         // [rows_cap, W]  LN output / attention output
  __nv_bfloat16* big = nullptr;       // [rows_cap, 4W] qkv (3W) or MLP hidden (4W)
  __nv_bfloat16* dlt = nullptr;       // [rows_cap, W]  out-proj result of the current layer (added to x by fc2's epilogue)
  __nv_bfloat16* pooled = nullptr;    // [max_seqs, W]
  float* xc = nullptr;                // [max_seqs, W] fp32 residual rows of the pooled positions (final layer, compact)
  int* first_of = nullptr;            // [max_seqs] sequence whose rows stand for sequence i
  bool prune_last = true;             // final layer: out-proj + MLP on the pooled rows only
  int gemm_sm_budget = 0;             // > 0: the persistent GEMM grids use at most this many SMs (leaf_set_sm_budget)
  int pdl = 1;                        // launch the per-layer chain with programmatic dependent launch (LEAF_PDL=0 turns it off)
  bool deterministic = false;         // leaf_set_deterministic: fixed-order reductions in leaf_backward / leaf_sumsq
  float* det_sum_ws = nullptr;        // leaf_sumsq's per-block sums and arrival counter in deterministic mode
  int* det_sum_cnt = nullptr;
  int att_impl = 1;                   // 1 = register-fed attention_kernel (default: faster in situ), 2 = cp.async ring attention2_kernel (LEAF_ATTENTION_IMPL=2)
  int *cu = nullptr, *eos_row = nullptr, *total_rows = nullptr, *pfx = nullptr, *own_len = nullptr, *dup_of = nullptr, *need = nullptr;
  int4* meta = nullptr;
  // bookkeeping
  int64_t launches = 0;
  bool timing = false;
  struct Span { cudaEvent_t a, b; int cat; };
  std::vector<Span> spans;            // cat: 0 GEMM, 1 LayerNorm, 2 attention, 3 everything else of the encode
  double span_ms[10] = {0};        // 4 + epi: the GEMM launches of one epilogue kind (also counted in class 0);
  int span_n[10] = {0};            // 8: the residual GEMMs with K > N (fc2), counted in class 6 as well; 9: bf16 store, N == K (out-proj)
  std::vector<cudaEvent_t> event_pool;
  std::map<std::tuple<const void*, long, long, int>, CUtensorMap> tmaps;
};

extern "C" const char* leaf_last_error(void) { return g_err.c_str(); }
extern "C" const char* leaf_version(void) { return "leaf_b200 0.1 (sm_100a)"; }

static int make_tmap(leaf_engine* e, const void* ptr, long rows, long cols, int box_rows, CUtensorMap* out) {
  auto key = std::make_tuple(ptr, rows, cols, box_rows);
  auto it = e->tmaps.find(key);
  if (it != e->tmaps.end()) { *out = it->second; return LEAF_OK; }
  if (cols % 8 != 0) return fail(LEAF_ERR_INVALID, "GEMM K (%ld) must be a multiple of 8", cols);
  if (reinterpret_cast<uintptr_t>(ptr) & 15) return fail(LEAF_ERR_INVALID, "GEMM operand must be 16-byte aligned");
  cuuint64_t dims[2] = {static_cast<cuuint64_t>(cols), static_cast<cuuint64_t>(rows)};
  cuuint64_t strides[1] = {static_cast<cuuint64_t>(cols) * 2};
  cuuint32_t box[2] = {static_cast<cuuint32_t>(GEMM_BK), static_cast<cuuint32_t>(box_rows)};
  cuuint32_t estr[2] = {1, 1};
  CUtensorMap m;
  CUresult r = e->encode_tiled(&m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(ptr), dims, strides, box, estr,
                               CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                               CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(LEAF_ERR_CUDA, "cuTensorMapEncodeTiled failed (%d) rows=%ld cols=%ld", (int)r, rows, cols);
  if (e->tmaps.size() > 4096) e->tmaps.clear();
  e->tmaps[key] = m;
  *out = m;
  return LEAF_OK;
}

// operand stored [k_rows, mn_cols] row-major (MN-major): boxes of 64 MN elements (one 128-byte swizzle row) x 64 k
static int make_tmap_mn(leaf_engine* e, const void* ptr, long k_rows, long mn_cols, long pitch, CUtensorMap* out) {
  if (pitch <= 0) pitch = mn_cols;
  auto key = std::make_tuple(ptr, k_rows, mn_cols, -static_cast<int>(pitch));
  auto it = e->tmaps.find(key);
  if (it != e->tmaps.end()) { *out = it->second; return LEAF_OK; }
  if (mn_cols % 8 != 0 || pitch % 8 != 0) return fail(LEAF_ERR_INVALID, "MN-major operand width (%ld) and pitch (%ld) must be multiples of 8", mn_cols, pitch);
  if (reinterpret_cast<uintptr_t>(ptr) & 15) return fail(LEAF_ERR_INVALID, "GEMM operand must be 16-byte aligned");
  cuuint64_t dims[2] = {static_cast<cuuint64_t>(mn_cols), static_cast<cuuint64_t>(k_rows)};
  cuuint64_t strides[1] = {static_cast<cuuint64_t>(pitch) * 2};
  cuuint32_t box[2] = {64, 64};
  cuuint32_t estr[2] = {1, 1};
  CUtensorMap m;
  CUresult r = e->encode_tiled(&m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(ptr), dims, strides, box, estr,
                               CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                               CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(LEAF_ERR_CUDA, "cuTensorMapEncodeTiled (MN-major) failed (%d) rows=%ld cols=%ld", (int)r, k_rows, mn_cols);
  if (e->tmaps.size() > 4096) e->tmaps.clear();
  e->tmaps[key] = m;
  *out = m;
  return LEAF_OK;
}

static cudaEvent_t get_event(leaf_engine* e) {
  if (!e->event_pool.empty()) { cudaEvent_t ev = e->event_pool.back(); e->event_pool.pop_back(); return ev; }
  cudaEvent_t ev;
  cudaEventCreate(&ev);
  return ev;
}

// CUDA events on the launching stream around a group of launches (only while leaf_set_timing is on)
struct TimedSpan {
  leaf_engine* e; cudaStream_t st; cudaEvent_t a = nullptr, b = nullptr; int cat;
  TimedSpan(leaf_engine* e_, int cat_, cudaStream_t st_) : e(e_), st(st_), cat(cat_) {
    if (e->timing) { a = get_event(e); b = get_event(e); cudaEventRecord(a, st); }
  }
  ~TimedSpan() {
    if (a) { cudaEventRecord(b, st); e->spans.push_back({a, b, cat}); }
  }
};

// C[M,N] = A[M,K] . Bt[N,K]^T with the fused epilogue `epi`
static int launch_gemm(leaf_engine* e, const __nv_bfloat16* A, long a_rows, const __nv_bfloat16* Bt, const float* bias,
                       void* C, int ldc, int M, int N, int K, int epi, int act, const int* m_dev, cudaStream_t st,
                       const __nv_bfloat16* delta = nullptr, int mn_major = 0, long a_pitch = 0, const float* res = nullptr,
                       void* C2 = nullptr, bool allow_split_k = false) {
  if (M <= 0 || N <= 0 || K <= 0) return fail(LEAF_ERR_INVALID, "GEMM shape %dx%dx%d", M, N, K);
  if (N % 8 != 0) return fail(LEAF_ERR_INVALID, "GEMM N (%d) must be a multiple of 8", N);
  CUtensorMap ta, tb;
  int a_box = a_rows < 128 ? static_cast<int>(a_rows) : 128;
  int b_box = N < 128 ? N : 128;
  int rc;
  if (mn_major & GEMM_A_MN) {                  // A is [K, M] row-major
    if (M % 8 != 0) return fail(LEAF_ERR_INVALID, "MN-major GEMM M (%d) must be a multiple of 8", M);
    if ((rc = make_tmap_mn(e, A, K, M, a_pitch, &ta))) return rc;      // a_pitch: row pitch when A is a column block of a wider matrix
    a_box = 128;
  } else if ((rc = make_tmap(e, A, a_rows, K, a_box, &ta))) return rc;
  if (mn_major & GEMM_B_MN) {                  // Bt is [K, N] row-major
    if ((rc = make_tmap_mn(e, Bt, K, N, 0, &tb))) return rc;
    b_box = 128;
  } else if ((rc = make_tmap(e, Bt, N, K, b_box, &tb))) return rc;
  GemmParams p;
  p.mn_major = mn_major;
  p.res = res;
  p.C2 = C2;
  p.split_k = 1;
  p.ws = nullptr;
  p.cnt = nullptr;
  p.tx_bytes = static_cast<uint32_t>(a_box + b_box) * GEMM_BK * 2 * 2;       // both CTAs of the pair
  p.M = M; p.m_dev = m_dev; p.N = N; p.K = K; p.bias = bias; p.C = C; p.ldc = ldc; p.act = act; p.delta = delta;
  const int m_tiles = (M + GEMM2_BM - 1) / GEMM2_BM, n_tiles = (N + GEMM_BN - 1) / GEMM_BN;
  long tiles = static_cast<long>(m_tiles) * n_tiles;
  const int pairs_cap = ((e->gemm_sm_budget > 0 && e->gemm_sm_budget < e->sm_count) ? e->gemm_sm_budget : e->sm_count) / 2;
  // Deterministic mode: fc1's bias gradient and the split-K partial sums are added in a fixed order (gemm_sm100.cuh,
  // EPI_*_DET), and the split factor is chosen for the whole device, so that an SM budget cannot change the summation order.
  const bool det = e->deterministic && ((epi == EPI_BF16_ACTBWD && C2) || allow_split_k);
  const int split_pairs = det ? e->sm_count / 2 : pairs_cap;
  if (det) {
    if (!e->tw.det_ws) return fail(LEAF_ERR_STATE, "deterministic mode without its workspace (leaf_train_reserve)");
    p.ws = e->tw.det_ws;
    p.cnt = e->tw.det_cnt;
    if (epi == EPI_BF16_ACTBWD) {
      if (static_cast<size_t>((M + 31) / 32) * N > e->tw.det_ws_floats || static_cast<size_t>(n_tiles) * 4 > e->tw.det_cnt_ints)
        return fail(LEAF_ERR_STATE, "deterministic workspace too small for a %dx%d bias reduction", M, N);
      epi = EPI_BF16_ACTBWD_DET;
    }
  }
  if (allow_split_k && epi == EPI_F32_RESIDUAL && !bias && !delta && !res && !m_dev && tiles < split_pairs) {
    // C += A.B with few output tiles and a long contraction (the weight gradients: 16-64 tiles, K = packed rows): divide the
    // k-blocks over several work units so that the launch fills the 74 CTA pairs; cost model = waves x (k-blocks per part +
    // 3 for the epilogue and the pipeline ramp). Partial sums are added with red.global.add.v4.f32.
    const int kblocks = (K + GEMM_BK - 1) / GEMM_BK;
    long best = ((tiles + split_pairs - 1) / split_pairs) * (kblocks + 3);
    for (int s = 2; s <= 8 && s <= kblocks; ++s) {
      const int kpb = (kblocks + s - 1) / s;
      const int s_eff = (kblocks + kpb - 1) / kpb;              // every part non-empty
      if (det && tiles * s_eff > 2L * split_pairs) continue;    // the partial tiles' workspace holds two waves of units
      const long cost = ((tiles * s_eff + split_pairs - 1) / split_pairs) * (kpb + 3);
      if (cost < best) { best = cost; p.split_k = s_eff; }
    }
    if (det && p.split_k > 1 && (static_cast<size_t>(tiles) * p.split_k * GEMM2_BM * GEMM_BN > e->tw.det_ws_floats ||
                                 static_cast<size_t>(tiles) * 2 * EPI_WARPS > e->tw.det_cnt_ints))
      return fail(LEAF_ERR_STATE, "deterministic workspace too small for a %dx%d split-K product", M, N);
    tiles *= p.split_k;
    if (p.split_k > 1) epi = det ? EPI_F32_SPLITK_DET : EPI_F32_SPLITK;
  }
  TimedSpan span(e, (epi == EPI_F32_SPLITK || epi == EPI_F32_SPLITK_DET) ? 4 + EPI_F32_RESIDUAL :
                    (epi == EPI_BF16_ACTBWD || epi == EPI_BF16_ACTBWD_DET) ? 4 + EPI_F32 : (epi == EPI_F32_RESIDUAL && K > N) ? 8 : (epi == EPI_BF16 && K == N) ? 9 : 4 + epi, st);
  const int pairs = static_cast<int>(tiles < pairs_cap ? tiles : pairs_cap);
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(2 * pairs);
  cfg.blockDim = dim3(GEMM_THREADS);
  cfg.dynamicSmemBytes = GEMM2_SMEM_BYTES;
  cfg.stream = st;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;      // see pdl_wait() in gemm_sm100.cuh
  attr[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = e->pdl ? 2 : 1;
  switch (epi) {
    case EPI_BF16: CK(cudaLaunchKernelEx(&cfg, gemm2_bf16_tn_kernel<EPI_BF16>, ta, tb, p)); break;
    case EPI_BF16_ACT: CK(cudaLaunchKernelEx(&cfg, gemm2_bf16_tn_kernel<EPI_BF16_ACT>, ta, tb, p)); break;
    case EPI_F32_RESIDUAL: CK(cudaLaunchKernelEx(&cfg, gemm2_bf16_tn_kernel<EPI_F32_RESIDUAL>, ta, tb, p)); break;
    case EPI_F32: CK(cudaLaunchKernelEx(&cfg, gemm2_bf16_tn_kernel<EPI_F32>, ta, tb, p)); break;
    case EPI_F32_SPLITK: CK(cudaLaunchKernelEx(&cfg, gemm2_bf16_tn_kernel<EPI_F32_SPLITK>, ta, tb, p)); break;
    case EPI_BF16_ACTBWD: CK(cudaLaunchKernelEx(&cfg, gemm2_bf16_tn_kernel<EPI_BF16_ACTBWD>, ta, tb, p)); break;
    case EPI_F32_SPLITK_DET: CK(cudaLaunchKernelEx(&cfg, gemm2_bf16_tn_kernel<EPI_F32_SPLITK_DET>, ta, tb, p)); break;
    case EPI_BF16_ACTBWD_DET: CK(cudaLaunchKernelEx(&cfg, gemm2_bf16_tn_kernel<EPI_BF16_ACTBWD_DET>, ta, tb, p)); break;
    default: return fail(LEAF_ERR_INVALID, "unknown epilogue %d", epi);
  }
  e->launches++;
  CK(cudaGetLastError());
  return LEAF_OK;
}

extern "C" int leaf_create(const leaf_cfg_t* cfg, leaf_handle_t* out) {
  if (!cfg || !out) return fail(LEAF_ERR_INVALID, "null argument");
  if (cfg->width <= 0 || cfg->width % 128 != 0 || cfg->width > 2048)
    return fail(LEAF_ERR_INVALID, "width %d must be a multiple of 128 in (0, 2048]", cfg->width);
  if (cfg->heads <= 0 || cfg->width != cfg->heads * 64) return fail(LEAF_ERR_INVALID, "head_dim must be 64 (W=%d, H=%d)", cfg->width, cfg->heads);
  if (cfg->embed_dim <= 0 || cfg->embed_dim % 8 != 0) return fail(LEAF_ERR_INVALID, "embed_dim %d must be a multiple of 8", cfg->embed_dim);
  if (cfg->layers <= 0) return fail(LEAF_ERR_INVALID, "layers");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail(LEAF_ERR_CUDA, "no CUDA device: leaf_b200 has no CPU path");
  int dev = 0;
  CK(cudaGetDevice(&dev));
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, dev));
  if (prop.major != 10) return fail(LEAF_ERR_CUDA, "device %s is sm_%d%d; leaf_b200 is built for sm_100a only", prop.name, prop.major, prop.minor);
  leaf_engine* e = new leaf_engine();
  e->cfg = *cfg;
  e->device = dev;
  e->sm_count = prop.multiProcessorCount;
  void* fn = nullptr;
  cudaDriverEntryPointQueryResult qres;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) != cudaSuccess || !fn) {
    delete e;
    return fail(LEAF_ERR_CUDA, "cuTensorMapEncodeTiled not available from the driver");
  }
  e->encode_tiled = reinterpret_cast<encode_tiled_fn>(fn);
  CK(cudaFuncSetAttribute(gemm2_bf16_tn_kernel<EPI_BF16>, cudaFuncAttributeMaxDynamicSharedMemorySize, GEMM2_SMEM_BYTES));
  CK(cudaFuncSetAttribute(gemm2_bf16_tn_kernel<EPI_BF16_ACT>, cudaFuncAttributeMaxDynamicSharedMemorySize, GEMM2_SMEM_BYTES));
  CK(cudaFuncSetAttribute(gemm2_bf16_tn_kernel<EPI_F32_RESIDUAL>, cudaFuncAttributeMaxDynamicSharedMemorySize, GEMM2_SMEM_BYTES));
  CK(cudaFuncSetAttribute(gemm2_bf16_tn_kernel<EPI_F32>, cudaFuncAttributeMaxDynamicSharedMemorySize, GEMM2_SMEM_BYTES));
  CK(cudaFuncSetAttribute(gemm2_bf16_tn_kernel<EPI_F32_SPLITK>, cudaFuncAttributeMaxDynamicSharedMemorySize, GEMM2_SMEM_BYTES));
  CK(cudaFuncSetAttribute(gemm2_bf16_tn_kernel<EPI_BF16_ACTBWD>, cudaFuncAttributeMaxDynamicSharedMemorySize, GEMM2_SMEM_BYTES));
  CK(cudaFuncSetAttribute(gemm2_bf16_tn_kernel<EPI_F32_SPLITK_DET>, cudaFuncAttributeMaxDynamicSharedMemorySize, GEMM2_SMEM_BYTES));
  CK(cudaFuncSetAttribute(gemm2_bf16_tn_kernel<EPI_BF16_ACTBWD_DET>, cudaFuncAttributeMaxDynamicSharedMemorySize, GEMM2_SMEM_BYTES));
  CK(cudaFuncSetAttribute(embed_sort_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, LEAF_VOCAB * 4));
  CK(cudaFuncSetAttribute(topk_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  CK(cudaFuncSetAttribute(attention2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, AT2_SMEM_BYTES));
  CK(cudaFuncSetAttribute(attention2_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
  if (const char* ai = getenv("LEAF_ATTENTION_IMPL")) e->att_impl = atoi(ai) == 2 ? 2 : 1;
  if (const char* pd = getenv("LEAF_PDL")) e->pdl = atoi(pd) != 0;
  CK(cudaFuncSetAttribute(attention_bwd_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, attb_smem_bytes(LEAF_CTX)));
  CK(cudaFuncSetAttribute(attention_bwd_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, attb_smem_bytes(LEAF_CTX)));
  *out = e;
  return LEAF_OK;
}

static void free_workspace(leaf_engine* e) {
  cudaFree(e->x); cudaFree(e->h); cudaFree(e->big); cudaFree(e->pooled); cudaFree(e->pooled_lo); e->pooled_lo = nullptr; cudaFree(e->xc); cudaFree(e->first_of); cudaFree(e->dlt);
  e->xc = nullptr; e->first_of = nullptr; e->dlt = nullptr;
  cudaFree(e->cu); cudaFree(e->eos_row); cudaFree(e->total_rows); cudaFree(e->pfx); cudaFree(e->own_len); cudaFree(e->dup_of); cudaFree(e->need); cudaFree(e->meta);
  e->x = nullptr; e->h = nullptr; e->big = nullptr; e->pooled = nullptr;
  e->cu = e->eos_row = e->total_rows = e->pfx = e->own_len = e->dup_of = e->need = nullptr;
  e->meta = nullptr;
  e->max_seqs = 0; e->rows_cap = 0;
  e->tmaps.clear();
}

static void free_weights(leaf_engine* e) {
  for (auto& l : e->lw) {
    cudaFree(l.qkv_w); cudaFree(l.out_w); cudaFree(l.fc1_w); cudaFree(l.fc2_w); cudaFree(l.qkv_b_own);
  }
  e->lw.clear();
  cudaFree(e->proj_w); cudaFree(e->proj_w_lo);
  e->proj_w = e->proj_w_lo = nullptr;
  e->bound = false;
  e->tmaps.clear();
}

extern "C" int leaf_destroy(leaf_handle_t e) {
  if (!e) return LEAF_OK;
  cudaDeviceSynchronize();
  free_workspace(e);
  for (void* p : e->tw.allocs) cudaFree(p);
  e->tw = TrainWs();
  free_weights(e);
  for (void* p : e->table_allocs) cudaFree(p);
  cudaFree(e->cn_count);
  cudaFree(e->det_sum_ws);
  cudaFree(e->det_sum_cnt);
  for (auto& sp : e->spans) { cudaEventDestroy(sp.a); cudaEventDestroy(sp.b); }
  for (auto ev : e->event_pool) cudaEventDestroy(ev);
  delete e;
  return LEAF_OK;
}

template <typename Tp>
static int upload(leaf_engine* e, const Tp* host, size_t count, const Tp** dev_out) {
  void* d = nullptr;
  CK(cudaMalloc(&d, count * sizeof(Tp)));
  e->table_allocs.push_back(d);
  CK(cudaMemcpy(d, host, count * sizeof(Tp), cudaMemcpyHostToDevice));
  *dev_out = static_cast<const Tp*>(d);
  return LEAF_OK;
}

extern "C" int leaf_load_bpe(leaf_handle_t e, const uint32_t* merge_pairs_host, int32_t n_merges) {
  if (!e || !merge_pairs_host) return fail(LEAF_ERR_INVALID, "null argument");
  if (n_merges != LEAF_N_MERGES) return fail(LEAF_ERR_INVALID, "CLIP's BPE has %d merges, got %d", LEAF_N_MERGES, n_merges);
  if (e->bpe_loaded) return LEAF_OK;
  std::vector<uint64_t> tab = k1_build_merge_table(merge_pairs_host, n_merges);
  K1Tables T{};
  int rc;
  if ((rc = upload(e, k1host::k1_host_byte_id, 256, &T.byte_id))) return rc;
  if ((rc = upload(e, k1host::k1_host_class, K1_TABLE_CPS, &T.cls))) return rc;
  if ((rc = upload(e, k1host::k1_host_ws, K1_TABLE_CPS, &T.ws))) return rc;
  if ((rc = upload(e, k1host::k1_host_lower, K1_TABLE_CPS, &T.lower))) return rc;
  if ((rc = upload(e, k1host::k1_host_numref, 256, &T.numref))) return rc;
  if ((rc = upload(e, k1host::k1_host_ent_off, K1_N_ENTITIES, &T.ent_off))) return rc;
  if ((rc = upload(e, k1host::k1_host_ent_len, K1_N_ENTITIES, &T.ent_len))) return rc;
  if ((rc = upload(e, k1host::k1_host_ent_val, K1_N_ENTITIES, &T.ent_val))) return rc;
  if ((rc = upload(e, k1host::k1_host_ent_blob, K1_ENTITY_BLOB_BYTES, &T.ent_blob))) return rc;
  if ((rc = upload(e, tab.data(), tab.size(), &T.merge_tab))) return rc;
  T.n_ent = K1_N_ENTITIES;
  T.merge_bits = K1_MERGE_BITS;
  e->tables = T;
  e->bpe_loaded = true;
  return LEAF_OK;
}

static int cast_to(leaf_engine* e, const float* src, __nv_bfloat16* dst, size_t n, cudaStream_t st, int residual = 0) {
  if (n % 4 != 0) return fail(LEAF_ERR_INVALID, "weight size not a multiple of 4");
  size_t blocks = (n / 4 + 255) / 256;
  if (blocks > 4096) blocks = 4096;
  cast_bf16_kernel<<<static_cast<int>(blocks), 256, 0, st>>>(src, dst, n, residual);
  e->launches++;
  CK(cudaGetLastError());
  return LEAF_OK;
}

extern "C" int leaf_refresh_weights(leaf_handle_t e, void* stream) {
  if (!e || !e->bound) return fail(LEAF_ERR_STATE, "weights not bound");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const size_t W = e->cfg.width, E = e->cfg.embed_dim;
  int rc;
  for (int l = 0; l < e->cfg.layers; ++l) {
    const leaf_layer_ptrs_t& p = e->layer_ptrs[l];
    LayerW& w = e->lw[l];
    if (p.in_proj_w) {
      if ((rc = cast_to(e, p.in_proj_w, w.qkv_w, 3 * W * W, st))) return rc;
      w.qkv_b = p.in_proj_b;
    } else {
      if ((rc = cast_to(e, p.q_w, w.qkv_w, W * W, st))) return rc;
      if ((rc = cast_to(e, p.k_w, w.qkv_w + W * W, W * W, st))) return rc;
      if ((rc = cast_to(e, p.v_w, w.qkv_w + 2 * W * W, W * W, st))) return rc;
      copy_f32_kernel<<<8, 256, 0, st>>>(p.q_b, w.qkv_b_own, W);
      copy_f32_kernel<<<8, 256, 0, st>>>(p.k_b, w.qkv_b_own + W, W);
      copy_f32_kernel<<<8, 256, 0, st>>>(p.v_b, w.qkv_b_own + 2 * W, W);
      e->launches += 3;
      w.qkv_b = w.qkv_b_own;
    }
    if ((rc = cast_to(e, p.out_w, w.out_w, W * W, st))) return rc;
    if ((rc = cast_to(e, p.fc1_w, w.fc1_w, 4 * W * W, st))) return rc;
    if ((rc = cast_to(e, p.fc2_w, w.fc2_w, 4 * W * W, st))) return rc;
  }
  if (e->wp.projection_is_ew) {
    if ((rc = cast_to(e, e->wp.text_projection, e->proj_w, E * W, st))) return rc;
    if ((rc = cast_to(e, e->wp.text_projection, e->proj_w_lo, E * W, st, 1))) return rc;
  } else {
    dim3 grid(static_cast<unsigned>((E + 31) / 32), static_cast<unsigned>((W + 31) / 32));
    cast_bf16_transpose_kernel<<<grid, dim3(32, 8), 0, st>>>(e->wp.text_projection, e->proj_w, static_cast<int>(W), static_cast<int>(E));
    cast_bf16_transpose_kernel<<<grid, dim3(32, 8), 0, st>>>(e->wp.text_projection, e->proj_w_lo, static_cast<int>(W), static_cast<int>(E), 1);
    e->launches += 2;
  }
  CK(cudaGetLastError());
  return LEAF_OK;
}

extern "C" int leaf_bind_weights(leaf_handle_t e, const leaf_weight_ptrs_t* w, void* stream) {
  if (!e || !w || !w->layers) return fail(LEAF_ERR_INVALID, "null argument");
  if (!w->token_embedding || !w->positional_embedding || !w->lnf_w || !w->lnf_b || !w->text_projection)
    return fail(LEAF_ERR_INVALID, "missing tower parameter");
  const size_t W = e->cfg.width, E = e->cfg.embed_dim;
  for (int l = 0; l < e->cfg.layers; ++l) {
    const leaf_layer_ptrs_t& p = w->layers[l];
    const bool fused = p.in_proj_w && p.in_proj_b;
    const bool split = p.q_w && p.k_w && p.v_w && p.q_b && p.k_b && p.v_b;
    if (!(fused || split) || !p.ln1_w || !p.ln1_b || !p.out_w || !p.out_b || !p.ln2_w || !p.ln2_b || !p.fc1_w || !p.fc1_b ||
        !p.fc2_w || !p.fc2_b)
      return fail(LEAF_ERR_INVALID, "missing parameter in layer %d", l);
  }
  free_weights(e);
  e->wp = *w;
  e->layer_ptrs.assign(w->layers, w->layers + e->cfg.layers);
  e->wp.layers = e->layer_ptrs.data();
  e->lw.resize(e->cfg.layers);
  for (auto& l : e->lw) {
    CK(cudaMalloc(&l.qkv_w, 3 * W * W * 2));
    CK(cudaMalloc(&l.out_w, W * W * 2));
    CK(cudaMalloc(&l.fc1_w, 4 * W * W * 2));
    CK(cudaMalloc(&l.fc2_w, 4 * W * W * 2));
    CK(cudaMalloc(&l.qkv_b_own, 3 * W * 4));
  }
  CK(cudaMalloc(&e->proj_w, E * W * 2));
  CK(cudaMalloc(&e->proj_w_lo, E * W * 2));
  e->bound = true;
  return leaf_refresh_weights(e, stream);
}

extern "C" int leaf_reserve(leaf_handle_t e, int32_t max_seqs) {
  if (!e || max_seqs <= 0) return fail(LEAF_ERR_INVALID, "max_seqs");
  if (max_seqs <= e->max_seqs) return LEAF_OK;
  cudaDeviceSynchronize();
  free_workspace(e);
  const size_t W = e->cfg.width;
  const size_t rows = ((static_cast<size_t>(max_seqs) * LEAF_CTX + 127) / 128) * 128;
  CK(cudaMalloc(&e->x, rows * W * 4));
  CK(cudaMalloc(&e->h, rows * W * 2));
  CK(cudaMalloc(&e->big, rows * 4 * W * 2));
  CK(cudaMalloc(&e->dlt, rows * W * 2));
  CK(cudaMalloc(&e->pooled, (static_cast<size_t>(max_seqs) + 128) * W * 2));
  CK(cudaMalloc(&e->pooled_lo, (static_cast<size_t>(max_seqs) + 128) * W * 2));
  CK(cudaMalloc(&e->xc, (static_cast<size_t>(max_seqs) + 128) * W * 4));
  CK(cudaMalloc(&e->first_of, static_cast<size_t>(max_seqs) * 4));
  CK(cudaMalloc(&e->cu, (static_cast<size_t>(max_seqs) + 1) * 4));
  CK(cudaMalloc(&e->eos_row, static_cast<size_t>(max_seqs) * 4));
  CK(cudaMalloc(&e->pfx, static_cast<size_t>(max_seqs) * 4));
  CK(cudaMalloc(&e->own_len, static_cast<size_t>(max_seqs) * 4));
  CK(cudaMalloc(&e->dup_of, static_cast<size_t>(max_seqs) * 4));
  CK(cudaMalloc(&e->need, static_cast<size_t>(max_seqs) * 4));
  CK(cudaMalloc(&e->meta, static_cast<size_t>(max_seqs) * 16));
  CK(cudaMalloc(&e->total_rows, 4));
  CK(cudaMemset(e->total_rows, 0, 4));
  e->max_seqs = max_seqs;
  e->rows_cap = static_cast<long>(rows);
  return LEAF_OK;
}

extern "C" int leaf_expand_tokenize(leaf_handle_t e, const uint8_t* caps, const int32_t* cap_off, int32_t B, int32_t n,
                                    const int32_t* pos, const int32_t* chr, const int32_t* sel, const uint8_t* valid,
                                    int32_t* tok_out, int32_t* len_out, int32_t* base_out, int32_t* status_out, void* stream) {
  if (!e || !caps || !cap_off || !tok_out || !len_out) return fail(LEAF_ERR_INVALID, "null argument");
  if (!e->bpe_loaded) return fail(LEAF_ERR_STATE, "leaf_load_bpe has not been called");
  if (B <= 0 || n < 0) return fail(LEAF_ERR_INVALID, "B=%d n=%d", B, n);
  if (n > 0 && (!pos || !chr)) return fail(LEAF_ERR_INVALID, "pos/chr required when n > 0");
  K1Args a{caps, cap_off, B, n, pos, chr, sel, valid, tok_out, len_out, base_out, status_out, e->hf_tokenizer ? 1 : 0};
  const long R = static_cast<long>(B) * (n > 0 ? n : 1) + (n > 0 ? B : 0);
  if (e->max_caption_bytes > LEAF_MAX_CAPTION_BYTES) {        // long captions: one warp per CTA with 4 KB text buffers
    k1_expand_tokenize_kernel<K1_LONG_TEXT, 1><<<static_cast<int>(R), 32, 0, static_cast<cudaStream_t>(stream)>>>(e->tables, a);
  } else {
    const int grid = static_cast<int>((R + K1_WARPS_PER_CTA - 1) / K1_WARPS_PER_CTA);
    k1_expand_tokenize_kernel<K1_MAX_TEXT, K1_WARPS_PER_CTA><<<grid, K1_WARPS_PER_CTA * 32, 0, static_cast<cudaStream_t>(stream)>>>(e->tables, a);
  }
  e->launches++;
  CK(cudaGetLastError());
  return LEAF_OK;
}

// A launch that may start while the previous kernel of the stream drains (programmatic dependent launch): the kernel
// must call pdl_wait() before its first global access (gemm_sm100.cuh).
template <typename... KArgs, typename... Args>
static cudaError_t launch_pdl(const leaf_engine* e, void (*kernel)(KArgs...), dim3 grid, dim3 block, cudaStream_t st, Args... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = e->pdl ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

static int launch_layernorm(leaf_engine* e, const float* x, const int* rows_dev, int rows_max, const int* gather,
                            const float* g, const float* b, __nv_bfloat16* y, cudaStream_t st,
                            const __nv_bfloat16* delta = nullptr, __nv_bfloat16* y_lo = nullptr) {
  const int W = e->cfg.width;
  const int vpl = W / 128;
  TimedSpan span(e, 1, st);
  long warps = rows_max;
  int blocks = static_cast<int>((warps + 7) / 8);
  const int cap = e->sm_count * 8;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
#define LN_CASE(V) case V: CK(launch_pdl(e, layernorm_bf16_kernel<V>, dim3(blocks), dim3(256), st, x, rows_dev, rows_max, gather, W, g, b, e->cfg.ln_eps, y, delta, y_lo)); break;
  switch (vpl) {
    LN_CASE(1) LN_CASE(2) LN_CASE(3) LN_CASE(4) LN_CASE(5) LN_CASE(6) LN_CASE(7) LN_CASE(8)
    LN_CASE(9) LN_CASE(10) LN_CASE(11) LN_CASE(12) LN_CASE(13) LN_CASE(14) LN_CASE(15) LN_CASE(16)
    default: return fail(LEAF_ERR_INVALID, "unsupported width %d", W);
  }
#undef LN_CASE
  e->launches++;
  CK(cudaGetLastError());
  return LEAF_OK;
}

// causal attention over the packed rows (tower_kernels.cuh)
static int launch_attention(leaf_engine* e, const __nv_bfloat16* qkv, const int4* meta, int N, __nv_bfloat16* out, int last_only,
                            cudaStream_t st, long rows_cap_hint = 0) {
  if (rows_cap_hint <= 0) rows_cap_hint = static_cast<long>(N) * LEAF_CTX;      // no sequence has more than 77 rows
  const int H = e->cfg.heads, W = e->cfg.width;
  if (e->att_impl == 2 && static_cast<unsigned long long>(rows_cap_hint) * 3ull * W < (1ull << 32)) {
    const long ctas = (static_cast<long>(N) * H + AT2_WARPS - 1) / AT2_WARPS;
    const int grid2 = static_cast<int>(ctas < 2L * e->sm_count ? ctas : 2L * e->sm_count);     // persistent: 2 CTAs of 8 warps per SM
    attention2_kernel<<<grid2, AT2_WARPS * 32, AT2_SMEM_BYTES, st>>>(qkv, meta, N, H, W, out, last_only);
    e->launches++;
    CK(cudaGetLastError());
    return LEAF_OK;
  }
  const int grid = (N * H + ATT_WARPS - 1) / ATT_WARPS;
  CK(launch_pdl(e, attention_kernel, dim3(grid), dim3(ATT_WARPS * 32), st, qkv, meta, N, H, W, out, last_only));
  e->launches++;
  CK(cudaGetLastError());
  return LEAF_OK;
}

extern "C" int leaf_encode(leaf_handle_t e, const int32_t* tok, const int32_t* len, const int32_t* base, int32_t N,
                           int32_t dedup_rows, int32_t dedup_group, int32_t trim_providers, int32_t normalize, float* feat_out,
                           void* stream) {
  if (!e || !tok || !len || !feat_out) return fail(LEAF_ERR_INVALID, "null argument");
  if (!e->bound) return fail(LEAF_ERR_STATE, "weights not bound");
  if (N <= 0) return fail(LEAF_ERR_INVALID, "N=%d", N);
  if (N > e->max_seqs) return fail(LEAF_ERR_STATE, "workspace reserved for %d rows, need %d (leaf_reserve)", e->max_seqs, N);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int W = e->cfg.width, E = e->cfg.embed_dim;
  const int rows_max = static_cast<int>(static_cast<long>(N) * LEAF_CTX);
  int rc;
  const int* dup = nullptr;
  {
  TimedSpan span(e, 3, st);
  if (dedup_group > 1 && dedup_rows > 0) {
    if (dedup_rows > N || dedup_rows % dedup_group != 0) return fail(LEAF_ERR_INVALID, "dedup_rows=%d dedup_group=%d N=%d", dedup_rows, dedup_group, N);
    dedup_kernel<<<(N + 7) / 8, 256, 0, st>>>(tok, len, dedup_rows, dedup_group, N, e->dup_of);
    e->launches++;
    dup = e->dup_of;
  }
  const bool trim = trim_providers && base && dedup_rows > 0 && dedup_rows < N;
  if (trim) CK(cudaMemsetAsync(e->need, 0, static_cast<size_t>(N) * 4, st));
  prefix_kernel<<<(N + 7) / 8, 256, 0, st>>>(tok, len, base, dup, N, e->pfx, e->own_len, trim ? e->need : nullptr);
  if (trim) {
    trim_providers_kernel<<<(N - dedup_rows + 255) / 256, 256, 0, st>>>(base, e->need, dedup_rows, N, e->own_len);
    e->launches++;
  }
  scan_lengths_kernel<<<1, 1024, 0, st>>>(e->own_len, N, e->cu, e->total_rows);
  meta_kernel<<<(N + 255) / 256, 256, 0, st>>>(e->cu, e->pfx, base, dup, N, e->meta, e->eos_row, e->first_of);
  embed_kernel<<<N, 256, 0, st>>>(tok, e->meta, N, W, e->wp.token_embedding, e->wp.positional_embedding, e->x);
  e->launches += 4;
  }
  CK(cudaGetLastError());
  for (int l = 0; l < e->cfg.layers; ++l) {
    const leaf_layer_ptrs_t& p = e->layer_ptrs[l];
    const LayerW& w = e->lw[l];
    if ((rc = launch_layernorm(e, e->x, e->total_rows, rows_max, nullptr, p.ln1_w, p.ln1_b, e->h, st))) return rc;
    if ((rc = launch_gemm(e, e->h, e->rows_cap, w.qkv_w, w.qkv_b, e->big, 3 * W, rows_max, 3 * W, W, EPI_BF16, 0, e->total_rows, st))) return rc;
    // Final layer: only the pooled EOS position of a sequence is read after it (transformer.py:661), so everything past
    // the key/value projection runs on ONE row per sequence: attention writes the EOS query's output to h[seq], the
    // residual rows are compacted into xc, and out-proj / LayerNorm / MLP see N rows instead of the packed row count.
    const bool last = e->prune_last && l == e->cfg.layers - 1;
    const __nv_bfloat16* dl = e->dlt;
    {
      TimedSpan span(e, 2, st);
      if ((rc = launch_attention(e, e->big, e->meta, N, e->h, last ? 1 : 0, st))) return rc;
    }
    // The attention branch's out-proj result stays OUT of the fp32 residual stream for now: it is stored as a bf16
    // delta (2 B per element, no read), LayerNorm normalises x + delta on the fly, and fc2's epilogue writes
    // x + delta + mlp back in one read-modify-write. A separate x += out-proj pass made the K = W out-proj GEMM the one
    // launch whose epilogue (8 B of fp32 residual traffic per 2 KFLOP) outran L2/HBM: 379 us against 230 us with a bf16
    // store at 130 k rows (tools/ab_gemm.py, profiles/r38_gemm_ab.log). 16-bit Linear outputs are what the reference's
    // own autocast path produces; the fp32 stream itself is untouched.
    if (last) {
      {
        TimedSpan span(e, 3, st);
        gather_rows_f32_kernel<<<(N + 7) / 8, 256, 0, st>>>(e->x, e->eos_row, N, W, e->xc);
        e->launches++;
      }
      if ((rc = launch_gemm(e, e->h, e->rows_cap, w.out_w, p.out_b, e->dlt, W, N, W, W, EPI_BF16, 0, nullptr, st))) return rc;
      if ((rc = launch_layernorm(e, e->xc, nullptr, N, nullptr, p.ln2_w, p.ln2_b, e->h, st, dl))) return rc;
      if ((rc = launch_gemm(e, e->h, e->rows_cap, w.fc1_w, p.fc1_b, e->big, 4 * W, N, 4 * W, W, EPI_BF16_ACT, e->cfg.activation, nullptr, st))) return rc;
      if ((rc = launch_gemm(e, e->big, e->rows_cap, w.fc2_w, p.fc2_b, e->xc, W, N, W, 4 * W, EPI_F32_RESIDUAL, 0, nullptr, st, dl))) return rc;
      break;
    }
    if ((rc = launch_gemm(e, e->h, e->rows_cap, w.out_w, p.out_b, e->dlt, W, rows_max, W, W, EPI_BF16, 0, e->total_rows, st))) return rc;
    if ((rc = launch_layernorm(e, e->x, e->total_rows, rows_max, nullptr, p.ln2_w, p.ln2_b, e->h, st, dl))) return rc;
    if ((rc = launch_gemm(e, e->h, e->rows_cap, w.fc1_w, p.fc1_b, e->big, 4 * W, rows_max, 4 * W, W, EPI_BF16_ACT, e->cfg.activation, e->total_rows, st))) return rc;
    if ((rc = launch_gemm(e, e->big, e->rows_cap, w.fc2_w, p.fc2_b, e->x, W, rows_max, W, 4 * W, EPI_F32_RESIDUAL, 0, e->total_rows, st, dl))) return rc;
  }
  // ln_final and the projection in split precision: both operands carry what their bf16 rounding dropped as a second bf16
  // matrix (pooled = hi + lo, P = hi + lo; feat = hi.hi + lo.hi + hi.lo, fp32 accumulate: error 2^-17 instead of 2^-9). One row
  // per sequence and 2 W E FLOP each: 0.1 ms per step, and it removes ~15 % of the TextFARE-loss error against the fp32
  // reference (tests/tools/exp_final_stage_precision.py: the last stage's rounding alone is worth 1.2-1.9e-3 of loss rel. error).
  if (e->prune_last) rc = launch_layernorm(e, e->xc, nullptr, N, e->first_of, e->wp.lnf_w, e->wp.lnf_b, e->pooled, st, nullptr, e->pooled_lo);
  else rc = launch_layernorm(e, e->x, nullptr, N, e->eos_row, e->wp.lnf_w, e->wp.lnf_b, e->pooled, st, nullptr, e->pooled_lo);
  if (rc) return rc;
  if ((rc = launch_gemm(e, e->pooled, e->max_seqs + 128, e->proj_w, nullptr, feat_out, E, N, E, W, EPI_F32, 0, nullptr, st))) return rc;
  if ((rc = launch_gemm(e, e->pooled_lo, e->max_seqs + 128, e->proj_w, nullptr, feat_out, E, N, E, W, EPI_F32_RESIDUAL, 0, nullptr, st))) return rc;
  if ((rc = launch_gemm(e, e->pooled, e->max_seqs + 128, e->proj_w_lo, nullptr, feat_out, E, N, E, W, EPI_F32_RESIDUAL, 0, nullptr, st))) return rc;
  if (normalize) {
    l2_normalize_kernel<<<(N + 7) / 8, 256, 0, st>>>(feat_out, N, E);
    e->launches++;
  }
  CK(cudaGetLastError());
  return LEAF_OK;
}

extern "C" int leaf_score(leaf_handle_t e, const float* feat, const float* anchor, int32_t B, int32_t n, int32_t objective,
                          float* loss_out, int32_t* best_out, float* best_feat_out, void* stream) {
  if (!e || !feat || !anchor || !best_out) return fail(LEAF_ERR_INVALID, "null argument");
  if (B <= 0 || n <= 0 || objective < 0 || objective > 3) return fail(LEAF_ERR_INVALID, "B=%d n=%d objective=%d", B, n, objective);
  if (e->cfg.embed_dim % 4 != 0) return fail(LEAF_ERR_INVALID, "embed_dim");
  if (static_cast<size_t>(n) * 4 > 48 * 1024) return fail(LEAF_ERR_INVALID, "n=%d too large", n);
  score_argmax_kernel<<<B, 256, static_cast<size_t>(n) * 4, static_cast<cudaStream_t>(stream)>>>(
      feat, anchor, n, e->cfg.embed_dim, objective, loss_out, best_out, best_feat_out);
  e->launches++;
  CK(cudaGetLastError());
  return LEAF_OK;
}

extern "C" int leaf_topk(leaf_handle_t e, const float* score_a, const float* score_b, int32_t m, int32_t k, int32_t* idx_out,
                         float* val_out, void* stream) {
  if (!e || !score_a || !idx_out) return fail(LEAF_ERR_INVALID, "null argument");
  if (m <= 0 || k <= 0 || k > m) return fail(LEAF_ERR_INVALID, "top-k of m=%d, k=%d", m, k);
  const size_t smem = static_cast<size_t>(m) * 4;
  if (smem > 200 * 1024) return fail(LEAF_ERR_INVALID, "m=%d too large (max %d)", m, 200 * 1024 / 4);
  topk_kernel<<<1, 1024, smem, static_cast<cudaStream_t>(stream)>>>(score_a, score_b, m, k, idx_out, val_out);
  e->launches++;
  CK(cudaGetLastError());
  return LEAF_OK;
}

extern "C" int leaf_gemm_bf16(leaf_handle_t e, const void* A, const void* Bt, const float* bias, void* C, int32_t M, int32_t N,
                              int32_t K, int32_t epilogue, int32_t act, const int32_t* m_dev, void* stream) {
  if (!e || !A || !Bt || !C) return fail(LEAF_ERR_INVALID, "null argument");
  return launch_gemm(e, static_cast<const __nv_bfloat16*>(A), M, static_cast<const __nv_bfloat16*>(Bt), bias, C, N, M, N, K,
                     epilogue, act, m_dev, static_cast<cudaStream_t>(stream));
}

extern "C" int leaf_gemm_bf16_mn(leaf_handle_t e, const void* A, const void* B, const float* bias, void* C, int32_t M, int32_t N,
                                 int32_t K, int32_t epilogue, int32_t a_mn, void* stream) {
  if (!e || !A || !B || !C) return fail(LEAF_ERR_INVALID, "null argument");
  return launch_gemm(e, static_cast<const __nv_bfloat16*>(A), a_mn ? K : M, static_cast<const __nv_bfloat16*>(B), bias, C, N, M, N, K,
                     epilogue, 0, nullptr, static_cast<cudaStream_t>(stream), nullptr, GEMM_B_MN | (a_mn ? GEMM_A_MN : 0));
}

extern "C" int leaf_test_layernorm(leaf_handle_t e, const float* x, int32_t rows, const float* gamma, const float* beta, void* y,
                                   void* stream) {
  if (!e || !x || !gamma || !beta || !y || rows <= 0) return fail(LEAF_ERR_INVALID, "bad argument");
  return launch_layernorm(e, x, nullptr, rows, nullptr, gamma, beta, static_cast<__nv_bfloat16*>(y), static_cast<cudaStream_t>(stream));
}

extern "C" int leaf_test_attention(leaf_handle_t e, const void* qkv, const int32_t* meta, int32_t N, void* out, void* stream) {
  if (!e || !qkv || !meta || !out || N <= 0) return fail(LEAF_ERR_INVALID, "bad argument");
  return launch_attention(e, static_cast<const __nv_bfloat16*>(qkv), reinterpret_cast<const int4*>(meta), N,
                          static_cast<__nv_bfloat16*>(out), 0, static_cast<cudaStream_t>(stream));
}

extern "C" int leaf_test_attention_bwd(leaf_handle_t e, const void* qkv, const void* o, const float* dout, const int32_t* meta,
                                       int32_t N, int32_t T, void* dqkv, void* stream) {
  if (!e || !qkv || !o || !dout || !meta || !dqkv || N <= 0 || T <= 0 || T > LEAF_CTX) return fail(LEAF_ERR_INVALID, "bad argument");
  attention_bwd_kernel<false><<<dim3(N, e->cfg.heads), ATTB_WARPS * 32, attb_smem_bytes(T), static_cast<cudaStream_t>(stream)>>>(
      static_cast<const __nv_bfloat16*>(qkv), static_cast<const __nv_bfloat16*>(o), dout, reinterpret_cast<const int4*>(meta),
      e->cfg.width, T, static_cast<__nv_bfloat16*>(dqkv));
  e->launches++;
  CK(cudaGetLastError());
  return LEAF_OK;
}

extern "C" int leaf_set_prune_last(leaf_handle_t e, int32_t on) {
  if (!e) return fail(LEAF_ERR_INVALID, "null handle");
  e->prune_last = on != 0;
  return LEAF_OK;
}

extern "C" int64_t leaf_launch_count(leaf_handle_t e, int32_t reset) {
  if (!e) return 0;
  const int64_t v = e->launches;
  if (reset) e->launches = 0;
  return v;
}

extern "C" int64_t leaf_last_rows(leaf_handle_t e) {
  if (!e || !e->total_rows) return 0;
  int v = 0;
  if (cudaMemcpy(&v, e->total_rows, 4, cudaMemcpyDeviceToHost) != cudaSuccess) return -1;
  return v;
}

extern "C" double leaf_timing_ms(leaf_handle_t e, int32_t which, int32_t* launches);
extern "C" int leaf_set_timing(leaf_handle_t e, int32_t on) {
  if (!e) return fail(LEAF_ERR_INVALID, "null handle");
  e->timing = on != 0;
  if (e->timing) {                               // a new measurement starts from zero
    int32_t dummy;
    leaf_timing_ms(e, 0, &dummy);
    for (int i = 0; i < 10; ++i) { e->span_ms[i] = 0; e->span_n[i] = 0; }
  }
  return LEAF_OK;
}

extern "C" double leaf_timing_ms(leaf_handle_t e, int32_t which, int32_t* launches) {
  if (!e || which < 0 || which > 9) return 0.0;
  if (!e->spans.empty()) {                       // fold the recorded spans into the per-category totals
    for (auto& sp : e->spans) {
      cudaEventSynchronize(sp.b);
      float ms = 0.f;
      if (cudaEventElapsedTime(&ms, sp.a, sp.b) == cudaSuccess) {
        e->span_ms[sp.cat] += ms; e->span_n[sp.cat]++;
        if (sp.cat >= 4) { e->span_ms[0] += ms; e->span_n[0]++; }
        if (sp.cat == 8) { e->span_ms[4 + EPI_F32_RESIDUAL] += ms; e->span_n[4 + EPI_F32_RESIDUAL]++; }
      }
      e->event_pool.push_back(sp.a);
      e->event_pool.push_back(sp.b);
    }
    e->spans.clear();
  }
  if (launches) *launches = e->span_n[which];
  return e->span_ms[which];
}

// =====================================================================================================================
// K4: forward in train mode (activations kept) and backward of the selected adversarial batch
// (/root/reference/utils_AT.py:312-337). Every product is a TN GEMM on the tcgen05 kernel:
//   dgrad  dX[M,in]   = dY[M,out] . W[out,in]            -> A = dY (bf16),        Bt = W^T copy [in,out]
//   wgrad  dW[out,in] += dY^T[out,M] . X[M,in]           -> A = dY^T [out,Mp],    Bt = X^T [in,Mp]   (fp32 accumulate into .grad)
// =====================================================================================================================
template <typename Tp>
static int tw_alloc(TrainWs& t, Tp** p, size_t count) {
  void* d = nullptr;
  CK(cudaMalloc(&d, count * sizeof(Tp)));
  t.allocs.push_back(d);
  *p = static_cast<Tp*>(d);
  return LEAF_OK;
}

static void free_train(leaf_engine* e) {
  for (void* p : e->tw.allocs) cudaFree(p);
  e->tw = TrainWs();
  e->tmaps.clear();
}

// Workspace of the deterministic backward for the reserved training shape (a no-op when it exists or nothing is reserved).
// Largest user of each buffer: the split-K partial tiles (two waves of work units at the device's pair count), fc1's bias
// (one row of column sums per 32 packed rows), the LayerNorm bands (at most 2 x SMs / column blocks + 1), the attention
// bias partials (one per sequence and warp).
static int reserve_deterministic(leaf_engine* e) {
  TrainWs& t = e->tw;
  if (t.det_ws || t.max_seqs == 0) return LEAF_OK;
  const size_t W = e->cfg.width, rows = static_cast<size_t>(t.rows_cap), pairs = static_cast<size_t>(e->sm_count / 2);
  const size_t cbx = (W + 255) / 256;
  size_t f = 2 * pairs * GEMM2_BM * GEMM_BN;
  f = std::max(f, (rows + 31) / 32 * 4 * W);
  f = std::max(f, (2 * static_cast<size_t>(e->sm_count) + cbx) * 3 * 256);
  f = std::max(f, static_cast<size_t>(t.max_seqs) * ATTB_WARPS * 3 * W);
  size_t c = std::max(pairs * 2 * EPI_WARPS, (4 * W + GEMM_BN - 1) / GEMM_BN * 4);
  c = std::max(c, std::max(cbx, static_cast<size_t>(e->cfg.heads)));
  int rc;
  if ((rc = tw_alloc(t, &t.det_ws, f))) return rc;
  if ((rc = tw_alloc(t, &t.det_cnt, c))) return rc;
  if ((rc = tw_alloc(t, &t.det_idx, 3 * rows))) return rc;
  CK(cudaMemset(t.det_cnt, 0, c * 4));
  CK(cudaDeviceSynchronize());
  t.det_ws_floats = f;
  t.det_cnt_ints = c;
  return LEAF_OK;
}

extern "C" int leaf_train_reserve(leaf_handle_t e, int32_t max_seqs) {
  if (!e || max_seqs <= 0) return fail(LEAF_ERR_INVALID, "max_seqs");
  if (!e->bound) return fail(LEAF_ERR_STATE, "weights not bound");
  const size_t W = e->cfg.width, E = e->cfg.embed_dim;
  int rc;
  if (max_seqs <= e->tw.max_seqs) return LEAF_OK;
  cudaDeviceSynchronize();
  free_train(e);
  TrainWs& t = e->tw;
  const size_t rows = ((static_cast<size_t>(max_seqs) * LEAF_CTX + 127) / 128) * 128;
  const size_t wide = 4 * W > E ? 4 * W : E;
  t.L.resize(e->cfg.layers);
  for (auto& l : t.L) {
    if ((rc = tw_alloc(t, &l.x_in, rows * W))) return rc;
    if ((rc = tw_alloc(t, &l.x_mid, rows * W))) return rc;
    if ((rc = tw_alloc(t, &l.h1, rows * W))) return rc;
    if ((rc = tw_alloc(t, &l.qkv, rows * 3 * W))) return rc;
    if ((rc = tw_alloc(t, &l.o, rows * W))) return rc;
    if ((rc = tw_alloc(t, &l.h2, rows * W))) return rc;
    if ((rc = tw_alloc(t, &l.u, rows * 4 * W))) return rc;
    if ((rc = tw_alloc(t, &l.g, rows * 4 * W))) return rc;
  }
  if ((rc = tw_alloc(t, &t.x_out, rows * W))) return rc;
  if ((rc = tw_alloc(t, &t.dx, rows * W))) return rc;
  if ((rc = tw_alloc(t, &t.dtmp, rows * wide))) return rc;
  if ((rc = tw_alloc(t, &t.scratch, 2 * W))) return rc;
  if ((rc = tw_alloc(t, &t.pooled, (static_cast<size_t>(max_seqs) + 128) * W))) return rc;
  if ((rc = tw_alloc(t, &t.d16, rows * wide))) return rc;
  if ((rc = tw_alloc(t, &t.dx16, rows * W))) return rc;
  if ((rc = tw_alloc(t, &t.ln_stats, rows * 2))) return rc;
  if ((rc = tw_alloc(t, &t.tok, static_cast<size_t>(max_seqs) * LEAF_CTX))) return rc;
  if ((rc = tw_alloc(t, &t.cu, static_cast<size_t>(max_seqs) + 1))) return rc;
  if ((rc = tw_alloc(t, &t.eos_row, static_cast<size_t>(max_seqs)))) return rc;
  if ((rc = tw_alloc(t, &t.total_rows, 2))) return rc;
  if ((rc = tw_alloc(t, &t.pfx, static_cast<size_t>(max_seqs)))) return rc;
  if ((rc = tw_alloc(t, &t.own_len, static_cast<size_t>(max_seqs)))) return rc;
  if ((rc = tw_alloc(t, &t.meta, static_cast<size_t>(max_seqs)))) return rc;
  t.max_seqs = max_seqs;
  t.rows_cap = static_cast<long>(rows);
  return e->deterministic ? reserve_deterministic(e) : LEAF_OK;
}

static int launch_ew(leaf_engine* e, size_t n) {      // grid for the grid-stride element-wise kernels
  size_t b = (n + 255) / 256;
  const size_t cap = static_cast<size_t>(e->sm_count) * 16;
  return static_cast<int>(b < cap ? (b ? b : 1) : cap);
}

// traps (a CUDA error at the next synchronisation) when the caller's row-count hints are not what the device computed
__global__ void check_train_hints_kernel(const int* __restrict__ total_rows, int rows, int max_len) {
  if (total_rows[0] != rows || total_rows[1] > max_len) __trap();
}

extern "C" int leaf_forward_train(leaf_handle_t e, const int32_t* tok, const int32_t* len, int32_t N, float* feat_out,
                                  int32_t rows_hint, int32_t max_len_hint, int64_t* generation_out, void* stream) {
  if (!e || !tok || !len || !feat_out || N <= 0) return fail(LEAF_ERR_INVALID, "bad argument");
  if (!e->bound) return fail(LEAF_ERR_STATE, "weights not bound");
  if (N > e->tw.max_seqs) return fail(LEAF_ERR_STATE, "training workspace reserved for %d sequences, need %d (leaf_train_reserve)", e->tw.max_seqs, N);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  TrainWs& t = e->tw;
  const int W = e->cfg.width, E = e->cfg.embed_dim;
  int rc;
  t.have_forward = false;
  t.generation = ++e->train_generation;
  CK(cudaMemcpyAsync(t.tok, tok, static_cast<size_t>(N) * LEAF_CTX * 4, cudaMemcpyDeviceToDevice, st));
  prefix_kernel<<<(N + 7) / 8, 256, 0, st>>>(tok, len, nullptr, nullptr, N, t.pfx, t.own_len);
  scan_lengths_kernel<<<1, 1024, 0, st>>>(t.own_len, N, t.cu, t.total_rows, t.total_rows + 1);
  meta_kernel<<<(N + 255) / 256, 256, 0, st>>>(t.cu, t.pfx, nullptr, nullptr, N, t.meta, t.eos_row);
  e->launches += 3;
  int mt[2] = {rows_hint, max_len_hint};
  if (rows_hint > 0 && max_len_hint > 0) {             // the caller knows the lengths (e.g. from the tokenizer's status read): no sync
    check_train_hints_kernel<<<1, 1, 0, st>>>(t.total_rows, rows_hint, max_len_hint);
    e->launches++;
  } else {
    CK(cudaMemcpyAsync(mt, t.total_rows, 8, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));                     // packed row count (sizes the wgrad contractions) + longest sequence
  }
  const int M = mt[0];
  if (M <= 0 || M > t.rows_cap || mt[1] <= 0 || mt[1] > LEAF_CTX) return fail(LEAF_ERR_STATE, "bad packed row count %d / length %d", M, mt[1]);
  t.N = N; t.M = M; t.T = mt[1];
  embed_kernel<<<N, 256, 0, st>>>(tok, t.meta, N, W, e->wp.token_embedding, e->wp.positional_embedding, t.L[0].x_in);
  e->launches++;
  for (int l = 0; l < e->cfg.layers; ++l) {
    const leaf_layer_ptrs_t& p = e->layer_ptrs[l];
    const LayerW& w = e->lw[l];
    TrainLayer& a = t.L[l];
    float* x_next = (l + 1 < e->cfg.layers) ? t.L[l + 1].x_in : t.x_out;
    if ((rc = launch_layernorm(e, a.x_in, nullptr, M, nullptr, p.ln1_w, p.ln1_b, a.h1, st))) return rc;
    if ((rc = launch_gemm(e, a.h1, t.rows_cap, w.qkv_w, w.qkv_b, a.qkv, 3 * W, M, 3 * W, W, EPI_BF16, 0, nullptr, st))) return rc;
    if ((rc = launch_attention(e, a.qkv, t.meta, N, a.o, 0, st))) return rc;
    if ((rc = launch_gemm(e, a.o, t.rows_cap, w.out_w, p.out_b, a.x_mid, W, M, W, W, EPI_F32_RESIDUAL, 0, nullptr, st, nullptr, 0, 0, a.x_in))) return rc;
    if ((rc = launch_layernorm(e, a.x_mid, nullptr, M, nullptr, p.ln2_w, p.ln2_b, a.h2, st))) return rc;
    // one epilogue stores fc1's output twice: the pre-activation u (kept for act'(u) in the backward) and act(u)
    if ((rc = launch_gemm(e, a.h2, t.rows_cap, w.fc1_w, p.fc1_b, a.g, 4 * W, M, 4 * W, W, EPI_BF16_ACT, e->cfg.activation, nullptr, st,
                          nullptr, 0, 0, nullptr, a.u))) return rc;
    if ((rc = launch_gemm(e, a.g, t.rows_cap, w.fc2_w, p.fc2_b, x_next, W, M, W, 4 * W, EPI_F32_RESIDUAL, 0, nullptr, st, nullptr, 0, 0, a.x_mid))) return rc;
  }
  if ((rc = launch_layernorm(e, t.x_out, nullptr, N, t.eos_row, e->wp.lnf_w, e->wp.lnf_b, t.pooled, st))) return rc;
  if ((rc = launch_gemm(e, t.pooled, t.max_seqs + 128, e->proj_w, nullptr, feat_out, E, N, E, W, EPI_F32, 0, nullptr, st))) return rc;
  CK(cudaGetLastError());
  t.have_forward = true;
  if (generation_out) *generation_out = t.generation;
  return LEAF_OK;
}

static int launch_layernorm_bwd(leaf_engine* e, const float* dy, const float* x, const int* gather, int rows, const float* gamma,
                                float* dx, int accumulate, float* dgamma, float* dbeta, float* scratch, cudaStream_t st,
                                __nv_bfloat16* dx16 = nullptr, float* dxsum = nullptr) {
  const int W = e->cfg.width;
  // frozen LayerNorm parameters (NULL grads) still need somewhere to add to: the scratch row pair
  if (!dgamma) dgamma = scratch;
  if (!dbeta) dbeta = scratch + W;
  // rows kernel (dx, dx16, per-row mean / rstd) + column kernel (dgamma, dbeta, dxsum from the saved statistics): train_kernels.cuh
  float2* stats = reinterpret_cast<float2*>(e->tw.ln_stats);
  int blocks = (rows + 7) / 8;
  if (blocks > 2 * e->sm_count) blocks = 2 * e->sm_count;
  if (blocks < 1) blocks = 1;
#define LNB_CASE(V) case V: layernorm_bwd_rows_kernel<V><<<blocks, 256, 0, st>>>(dy, x, gather, rows, W, gamma, e->cfg.ln_eps, dx, accumulate, dx16, stats); break;
  switch (W / 128) {
    LNB_CASE(1) LNB_CASE(2) LNB_CASE(3) LNB_CASE(4) LNB_CASE(5) LNB_CASE(6) LNB_CASE(7) LNB_CASE(8)
    LNB_CASE(9) LNB_CASE(10) LNB_CASE(11) LNB_CASE(12) LNB_CASE(13) LNB_CASE(14) LNB_CASE(15) LNB_CASE(16)
    default: return fail(LEAF_ERR_INVALID, "unsupported width %d", W);
  }
#undef LNB_CASE
  const int cbx = (W + 255) / 256;
  int bands = (2 * e->sm_count + cbx - 1) / cbx;
  if (bands > (rows + 7) / 8) bands = (rows + 7) / 8;
  if (bands < 1) bands = 1;
  if (e->deterministic) {                              // band sums added in band order (train_kernels.cuh)
    if (static_cast<size_t>(bands) * 3 * W > e->tw.det_ws_floats || static_cast<size_t>(cbx) > e->tw.det_cnt_ints)
      return fail(LEAF_ERR_STATE, "deterministic workspace too small for the LayerNorm backward (%d bands)", bands);
    CK(launch_pdl(e, layernorm_bwd_cols_kernel<true>, dim3(cbx, bands), dim3(256), st, dy, x, gather, stats, dx, rows, W, dgamma, dbeta,
                  dxsum, e->tw.det_ws, e->tw.det_cnt));
  } else {
    CK(launch_pdl(e, layernorm_bwd_cols_kernel<false>, dim3(cbx, bands), dim3(256), st, dy, x, gather, stats, dx, rows, W, dgamma, dbeta,
                  dxsum, nullptr, nullptr));
  }
  e->launches += 2;
  CK(cudaGetLastError());
  return LEAF_OK;
}

// grads mirrors leaf_weight_ptrs_t: fp32 device buffers that are ACCUMULATED into (+=); NULL = parameter is frozen.
extern "C" int leaf_backward(leaf_handle_t e, int64_t generation, const float* dfeat, int32_t dfeat_rows,
                             const leaf_weight_ptrs_t* grads, void* stream) {
  if (!e || !dfeat || !grads || !grads->layers) return fail(LEAF_ERR_INVALID, "null argument");
  TrainWs& t = e->tw;
  if (!t.have_forward) return fail(LEAF_ERR_STATE, "leaf_backward needs a preceding leaf_forward_train (the activation store is empty or already consumed)");
  if (generation != 0 && generation != t.generation)
    return fail(LEAF_ERR_STATE, "the activation store holds forward #%lld, this backward belongs to forward #%lld: the engine keeps ONE "
                "saved forward (run each encode_text's backward before the next encode_text with gradients enabled)",
                (long long)t.generation, (long long)generation);
  if (dfeat_rows != t.N) return fail(LEAF_ERR_INVALID, "dfeat has %d rows, the saved forward has %d sequences", dfeat_rows, t.N);
  if (e->deterministic && !t.det_ws) return fail(LEAF_ERR_STATE, "deterministic mode without its workspace (leaf_train_reserve)");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int W = e->cfg.width, E = e->cfg.embed_dim, N = t.N, M = t.M;
  const long cap = t.rows_cap;
  int rc;
  auto F = [](const float* p) { return const_cast<float*>(p); };
  float* scratch = t.scratch;                        // sink for the LayerNorm gradients of frozen parameters
  // Every product reads its operands as they lie (MN-major UMMA operands, gemm_sm100.cuh): the data gradients take the
  // forward's bf16 weight copy W[out,in] as B[k = out][n = in], the weight gradients take dY[rows,out] and X[rows,in] as
  // A[k = rows][m = out] and B[k = rows][n = in]. No transposed copies of weights or activations exist.
  auto dgrad = [&](const __nv_bfloat16* dy, long dy_rows, const __nv_bfloat16* w_oi, float* dx_out, int rows, int in, int out) {
    return launch_gemm(e, dy, dy_rows, w_oi, nullptr, dx_out, in, rows, in, out, EPI_F32, 0, nullptr, st, nullptr, GEMM_B_MN);
  };
  auto wgrad = [&](const __nv_bfloat16* dy, long dy_pitch, const __nv_bfloat16* x, float* dw, int rows, int in, int out) {
    return launch_gemm(e, dy, rows, x, nullptr, dw, in, out, in, rows, EPI_F32_RESIDUAL, 0, nullptr, st, nullptr,
                       GEMM_A_MN | GEMM_B_MN, dy_pitch, nullptr, nullptr, /*allow_split_k=*/true);
  };
  // ---- projection + ln_final on the pooled rows ----
  const size_t nfe = static_cast<size_t>(N) * E;
  cast_f32_bf16_kernel<<<launch_ew(e, nfe), 256, 0, st>>>(dfeat, t.d16, nfe);
  e->launches++;
  if ((rc = dgrad(t.d16, N, e->proj_w, t.dtmp, N, W, E))) return rc;                                        // dpooled [N,W] = dfeat . P[E,W]
  if (grads->text_projection) {
    if (grads->projection_is_ew) {
      if ((rc = wgrad(t.d16, 0, t.pooled, F(grads->text_projection), N, W, E))) return rc;                 // dP[E,W] += dfeat^T . pooled
    } else if ((rc = launch_gemm(e, t.pooled, N, t.d16, nullptr, F(grads->text_projection), E, W, E, N, EPI_F32_RESIDUAL, 0, nullptr, st,
                                 nullptr, GEMM_A_MN | GEMM_B_MN))) return rc;                              // dP[W,E] += pooled^T . dfeat
  }
  // dx and its bf16 copy dx16 (the A operand of the next dgrad GEMM) are written together by the LayerNorm backward
  CK(cudaMemsetAsync(t.dx, 0, static_cast<size_t>(M) * W * 4, st));
  CK(cudaMemsetAsync(t.dx16, 0, static_cast<size_t>(M) * W * 2, st));
  CK(cudaMemsetAsync(scratch, 0, 2 * W * 4, st));
  // the bias gradients that are column sums of dx (fc2's, out-proj's) are accumulated by the LayerNorm backward that writes
  // that dx: ln_final / the layer above's ln_1 for fc2, this layer's ln_2 for out-proj
  if ((rc = launch_layernorm_bwd(e, t.dtmp, t.x_out, t.eos_row, N, e->wp.lnf_w, t.dx, 0, F(grads->lnf_w), F(grads->lnf_b), scratch, st, t.dx16,
                                 F(grads->layers[e->cfg.layers - 1].fc2_b)))) return rc;
  if (e->bwd_hook) e->bwd_hook(e->cfg.layers, e->bwd_hook_user);          // projection + ln_final gradients are enqueued
  for (int l = e->cfg.layers - 1; l >= 0; --l) {
    const leaf_layer_ptrs_t& p = e->layer_ptrs[l];
    const leaf_layer_ptrs_t& g = grads->layers[l];
    const LayerW& w = e->lw[l];
    TrainLayer& a = t.L[l];
    // ================= MLP branch: x_next = x_mid + fc2(act(fc1(ln_2(x_mid)))) =================
    // du [M,4W] = (dx . W2[W,4W]) * act'(u), bf16, with fc1's bias gradient (its column sums): one GEMM, the activation
    // backward is its epilogue (EPI_BF16_ACTBWD; a separate pass over an fp32 dg [M,4W] before)
    if ((rc = launch_gemm(e, t.dx16, cap, w.fc2_w, nullptr, t.d16, 4 * W, M, 4 * W, W, EPI_BF16_ACTBWD, e->cfg.activation, nullptr, st,
                          a.u, GEMM_B_MN, 0, nullptr, F(g.fc1_b)))) return rc;
    if (g.fc2_w && (rc = wgrad(t.dx16, 0, a.g, F(g.fc2_w), M, 4 * W, W))) return rc;
    if ((rc = dgrad(t.d16, cap, w.fc1_w, t.dtmp, M, W, 4 * W))) return rc;                                  // dh2 [M,W]
    if (g.fc1_w && (rc = wgrad(t.d16, 0, a.h2, F(g.fc1_w), M, W, 4 * W))) return rc;
    if ((rc = launch_layernorm_bwd(e, t.dtmp, a.x_mid, nullptr, M, p.ln2_w, t.dx, 1, F(g.ln2_w), F(g.ln2_b), scratch, st, t.dx16, F(g.out_b)))) return rc;
    // ================= attention branch: x_mid = x_in + out_proj(attn(in_proj(ln_1(x_in)))) =================
    if ((rc = dgrad(t.dx16, cap, w.out_w, t.dtmp, M, W, W))) return rc;                                     // do [M,W]
    if (g.out_w && (rc = wgrad(t.dx16, 0, a.o, F(g.out_w), M, W, W))) return rc;
    {                                                                                                        // dqkv [M,3W] bf16 (+ in-projection bias grads)
      float* bq = p.in_proj_w ? F(g.in_proj_b) : F(g.q_b);
      float* bk = p.in_proj_w ? (g.in_proj_b ? F(g.in_proj_b) + W : nullptr) : F(g.k_b);
      float* bv = p.in_proj_w ? (g.in_proj_b ? F(g.in_proj_b) + 2 * W : nullptr) : F(g.v_b);
      if (e->deterministic && (bq || bk || bv))         // bias column sums added in (sequence, warp) order
        attention_bwd_kernel<true><<<dim3(N, e->cfg.heads), ATTB_WARPS * 32, attb_smem_bytes(t.T), st>>>(a.qkv, a.o, t.dtmp, t.meta, W, t.T, t.d16,
                                                                                                      bq, bk, bv, t.det_ws, t.det_cnt);
      else
        attention_bwd_kernel<false><<<dim3(N, e->cfg.heads), ATTB_WARPS * 32, attb_smem_bytes(t.T), st>>>(a.qkv, a.o, t.dtmp, t.meta, W, t.T, t.d16,
                                                                                                       bq, bk, bv);
    }
    e->launches++;
    CK(cudaGetLastError());
    if ((rc = dgrad(t.d16, cap, w.qkv_w, t.dtmp, M, W, 3 * W))) return rc;                                  // dh1 [M,W]
    if (p.in_proj_w) {                                                                                       // layout of the bound parameters
      if (g.in_proj_w && (rc = wgrad(t.d16, 0, a.h1, F(g.in_proj_w), M, W, 3 * W))) return rc;
    } else {                                                                                                 // HF: q, k, v are column blocks of dqkv
      const float* dw[3] = {g.q_w, g.k_w, g.v_w};
      for (int j = 0; j < 3; ++j)
        if (dw[j] && (rc = wgrad(t.d16 + j * W, 3 * W, a.h1, F(dw[j]), M, W, W))) return rc;
    }
    if ((rc = launch_layernorm_bwd(e, t.dtmp, a.x_in, nullptr, M, p.ln1_w, t.dx, 1, F(g.ln1_w), F(g.ln1_b), scratch, st, t.dx16,
                                   l > 0 ? F(grads->layers[l - 1].fc2_b) : nullptr))) return rc;
    // layer l's weight gradients (and every bias / LayerNorm gradient of layers > l) are complete on the stream from here on
    if (e->bwd_hook) e->bwd_hook(l, e->bwd_hook_user);
  }
  if (grads->token_embedding || grads->positional_embedding) {
    // a frozen table still needs a target for the atomics: reuse dtmp as a sink is not possible (49408 rows) -> require both
    if (!grads->token_embedding || !grads->positional_embedding)
      return fail(LEAF_ERR_INVALID, "token and positional embedding gradients must be given together");
    if (e->deterministic) {                            // rows grouped by token id, one writer per table row (train_kernels.cuh)
      int* row_tok = t.det_idx;
      int* order = row_tok + t.rows_cap;
      int* key = order + t.rows_cap;
      embed_sort_kernel<<<1, 1024, LEAF_VOCAB * 4, st>>>(t.tok, t.meta, N, M, row_tok, order, key);
      embed_bwd_det_kernel<<<dim3(M + LEAF_CTX, (W + 255) / 256), 256, 0, st>>>(order, key, t.meta, N, M, W, t.dx, F(grads->token_embedding),
                                                                                F(grads->positional_embedding));
      e->launches += 2;
    } else {
      embed_bwd_kernel<<<N, 256, 0, st>>>(t.tok, t.meta, N, W, t.dx, F(grads->token_embedding), F(grads->positional_embedding));
      e->launches++;
    }
  }
  CK(cudaGetLastError());
  t.have_forward = false;                              // consumed: dx / dtmp were overwritten, a second backward would be wrong
  if (e->bwd_hook) e->bwd_hook(-1, e->bwd_hook_user);  // everything, embeddings included
  return LEAF_OK;
}

// The persistent GEMM grids normally take every SM (one CTA pair per TPC). While a collective runs next to the backward
// (leaf_set_backward_hook + an all-reduce on a side stream) its CTAs need SMs of their own: n_sms > 0 caps the GEMM grids at
// n_sms SMs, 0 restores the full device.
extern "C" int leaf_set_sm_budget(leaf_handle_t e, int32_t n_sms) {
  if (!e || n_sms < 0) return fail(LEAF_ERR_INVALID, "bad argument");
  e->gemm_sm_budget = n_sms >= 2 ? n_sms : 0;
  return LEAF_OK;
}

extern "C" int leaf_set_deterministic(leaf_handle_t e, int32_t on) {
  if (!e) return fail(LEAF_ERR_INVALID, "null handle");
  if (on) {
    if (!e->det_sum_ws) {
      CK(cudaMalloc(&e->det_sum_ws, static_cast<size_t>(e->sm_count) * 16 * 4));
      CK(cudaMalloc(&e->det_sum_cnt, 4));
      CK(cudaMemset(e->det_sum_cnt, 0, 4));
      CK(cudaDeviceSynchronize());
    }
    e->deterministic = true;
    int rc = reserve_deterministic(e);
    if (rc) { e->deterministic = false; return rc; }
  } else {
    e->deterministic = false;
  }
  return LEAF_OK;
}

extern "C" int leaf_set_backward_hook(leaf_handle_t e, leaf_backward_hook_t fn, void* user) {
  if (!e) return fail(LEAF_ERR_INVALID, "null handle");
  e->bwd_hook = fn;
  e->bwd_hook_user = user;
  return LEAF_OK;
}

// AdamW step over a flat fp32 parameter buffer (n a multiple of 4, 16-byte aligned): train_AT_text_only.py:326-341,
// utils_AT.py:358-362. Elements [0, n_nodecay) take no weight decay.
extern "C" int leaf_adamw(leaf_handle_t e, float* params, const float* grads, float* exp_avg, float* exp_avg_sq, int64_t n,
                          int64_t n_nodecay, float lr, float beta1, float beta2, float eps, float weight_decay, int32_t step,
                          float grad_scale, void* stream) {
  if (!e || !params || !grads || !exp_avg || !exp_avg_sq) return fail(LEAF_ERR_INVALID, "null argument");
  if (n <= 0 || n % 4 != 0 || n_nodecay < 0 || n_nodecay > n || step < 1) return fail(LEAF_ERR_INVALID, "n=%lld n_nodecay=%lld step=%d", (long long)n, (long long)n_nodecay, step);
  if ((reinterpret_cast<uintptr_t>(params) | reinterpret_cast<uintptr_t>(grads) | reinterpret_cast<uintptr_t>(exp_avg) |
       reinterpret_cast<uintptr_t>(exp_avg_sq)) & 15)
    return fail(LEAF_ERR_INVALID, "AdamW buffers must be 16-byte aligned");
  const float bc1 = 1.f - powf(beta1, static_cast<float>(step));
  const float bc2s = sqrtf(1.f - powf(beta2, static_cast<float>(step)));
  adamw_kernel<<<launch_ew(e, static_cast<size_t>(n) / 4), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      params, grads, exp_avg, exp_avg_sq, static_cast<size_t>(n), static_cast<size_t>(n_nodecay), lr, beta1, beta2, eps,
      weight_decay, bc1, bc2s, grad_scale);
  e->launches++;
  CK(cudaGetLastError());
  return LEAF_OK;
}

// out[0] (device fp32, zeroed by the caller) += sum of squares of g[0, n)
extern "C" int leaf_sumsq(leaf_handle_t e, const float* g, int64_t n, float* out, void* stream) {
  if (!e || !g || !out || n <= 0 || n % 4 != 0) return fail(LEAF_ERR_INVALID, "bad argument");
  const int grid = launch_ew(e, static_cast<size_t>(n) / 4);       // <= 16 x SMs: leaf_set_deterministic sizes det_sum_ws for it
  if (e->deterministic)
    sumsq_kernel<true><<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(g, static_cast<size_t>(n), out, e->det_sum_ws, e->det_sum_cnt);
  else
    sumsq_kernel<false><<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(g, static_cast<size_t>(n), out);
  e->launches++;
  CK(cudaGetLastError());
  return LEAF_OK;
}

// g[0, n) *= s (in place): torch.nn.utils.clip_grad_norm_'s rescale of the accumulated gradients after a micro-batch that
// is not followed by an optimizer step (utils_AT.py:356-357 runs it after EVERY micro-batch)
extern "C" int leaf_scale(leaf_handle_t e, float* g, int64_t n, float s, void* stream) {
  if (!e || !g || n <= 0 || n % 4 != 0) return fail(LEAF_ERR_INVALID, "bad argument");
  scale_f32_kernel<<<launch_ew(e, static_cast<size_t>(n) / 4), 256, 0, static_cast<cudaStream_t>(stream)>>>(g, static_cast<size_t>(n), s);
  e->launches++;
  CK(cudaGetLastError());
  return LEAF_OK;
}

// ---- on-device --constrain filter (constrain_core.cuh) ---------------------------------------------------------------------
extern "C" int leaf_load_words(leaf_handle_t e, const uint8_t* words_blob, const int32_t* words_off, int32_t n_words,
                               const uint8_t* abbrev_blob, const int32_t* abbrev_off, int32_t n_abbrev) {
  if (!e || !words_blob || !words_off || n_words <= 0) return fail(LEAF_ERR_INVALID, "word list required");
  if (n_abbrev > 0 && (!abbrev_blob || !abbrev_off)) return fail(LEAF_ERR_INVALID, "abbreviation list");
  CnTables T{};
  std::vector<uint64_t> w = cn_build_table(words_blob, words_off, n_words, &T.words_bits);
  int rc;
  if ((rc = upload(e, w.data(), w.size(), &T.words))) return rc;
  if (n_abbrev > 0) {
    std::vector<uint64_t> ab = cn_build_table(abbrev_blob, abbrev_off, n_abbrev, &T.abbrev_bits);
    if ((rc = upload(e, ab.data(), ab.size(), &T.abbrev))) return rc;
  }
  e->cn = T;
  e->words_loaded = true;
  return LEAF_OK;
}

extern "C" int leaf_constrain_mask(leaf_handle_t e, const uint8_t* caps, const int32_t* cap_off, int32_t B, int32_t n,
                                   const int32_t* pos, const int32_t* chr, const int32_t* sel, uint8_t* valid_out,
                                   int32_t* count_out, int32_t* status_out, void* stream) {
  if (!e || !caps || !cap_off || !pos || !chr || !valid_out) return fail(LEAF_ERR_INVALID, "null argument");
  if (!e->words_loaded) return fail(LEAF_ERR_STATE, "leaf_load_words has not been called");
  if (B <= 0 || n <= 0) return fail(LEAF_ERR_INVALID, "B=%d n=%d", B, n);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int R = B * n + B;
  int32_t* cnt = count_out;
  if (!cnt) {
    if (R > e->cn_count_cap) {
      CK(cudaStreamSynchronize(st));
      cudaFree(e->cn_count);
      e->cn_count = nullptr;
      CK(cudaMalloc(&e->cn_count, static_cast<size_t>(R) * 4));
      e->cn_count_cap = R;
    }
    cnt = e->cn_count;
  }
  CnArgs a{caps, cap_off, B, n, pos, chr, sel, cnt, status_out};
  constrain_count_kernel<<<(R + 63) / 64, 64, 0, st>>>(e->cn, a);
  constrain_valid_kernel<<<(B * n + 255) / 256, 256, 0, st>>>(cnt, B, n, valid_out);
  e->launches += 2;
  CK(cudaGetLastError());
  return LEAF_OK;
}

// Captions longer than LEAF_MAX_CAPTION_BYTES (up to LEAF_MAX_CAPTION_BYTES_LONG) switch leaf_expand_tokenize to its
// long-text variant (one warp per CTA, 4 KB text buffers: ~4 x slower on a kernel that takes 0.15 ms per 6 528 rows).
extern "C" int leaf_set_max_caption_bytes(leaf_handle_t e, int32_t bytes) {
  if (!e || bytes <= 0 || bytes > LEAF_MAX_CAPTION_BYTES_LONG) return fail(LEAF_ERR_INVALID, "caption limit %d (max %d)", bytes, LEAF_MAX_CAPTION_BYTES_LONG);
  e->max_caption_bytes = bytes;
  return LEAF_OK;
}

// 0 = open_clip SimpleTokenizer (default), 1 = transformers CLIPTokenizer (no html.unescape, <|startoftext|> spellings)
extern "C" int leaf_set_tokenizer_mode(leaf_handle_t e, int32_t mode) {
  if (!e || (mode != 0 && mode != 1)) return fail(LEAF_ERR_INVALID, "tokenizer mode %d", mode);
  e->hf_tokenizer = mode == 1;
  return LEAF_OK;
}
