// tcgen05 / TMEM / TMA GEMM for the CLIP text tower (sm_100a only).
//
//   C[M,N] = A[M,K] . Bt[N,K]^T  (+ bias, activation, residual)      A, Bt bf16 K-major, fp32 accumulate
//
// This is the kernel behind every nn.Linear of the reference's text tower
// (/root/reference/src/open_clip/transformer.py:225 in_proj/out_proj, :233-235 c_fc/c_proj,
// /root/reference/src/open_clip/model.py:282 text_projection). nn.Linear weights are [out,in] row-major,
// i.e. already the K-major "B" operand, so no transpose is ever made.
//
// This header holds the PTX wrappers, descriptors and the fused epilogue; the kernel itself (CTA-pair,
// cta_group::2) is gemm2_sm100.cuh. Roles per CTA (640 threads):
//   warp 16     TMA producer   : cp.async.bulk.tensor, 128B-swizzled 128x64 boxes of A and B into a shared-memory
//                                ring, completion on mbarriers
//   warp 17     MMA issuer     : one thread (leader CTA) issues tcgen05.mma.kind::f16, accumulators in TMEM,
//                                double buffered (2 x 256 columns)
//   warp 18     TMEM allocator
//   warps 0-15  epilogue       : tcgen05.ld 32 lanes x 32 columns -> registers -> fused bias / GELU / residual
//                                -> coalesced global store; overlaps the next tile's MMAs (TMEM double buffer)
// M may be a device-side value (packed token rows are only known on the device).
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace leaf {

// Programmatic dependent launch. Every GEMM, LayerNorm and attention launch carries
// cudaLaunchAttributeProgrammaticStreamSerialization (engine.cu: launch_gemm, launch_pdl), and the non-GEMM kernels call
// pdl_trigger() on entry: the GEMM that follows becomes resident while they drain, runs its prologue (barrier init, TMEM
// allocation, descriptor prefetch) and blocks in pdl_wait() until its predecessor has completed and its writes are visible.
// Rule: nothing that a predecessor of the same per-layer chain writes may be read, and nothing may be written, before
// pdl_wait() (the packed row count m_dev is written before the chain starts). Both are no-ops under an ordinary launch.
// Worth 0.9 ms of the 13.0 ms K4 step (27 us kernels); neutral on the attack step (profiles/r2_25_pdl_ab.txt).
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

constexpr int GEMM_BN = 256;
constexpr int GEMM_BK = 64;

enum { EPI_BF16 = 0, EPI_BF16_ACT = 1, EPI_F32_RESIDUAL = 2, EPI_F32 = 3, EPI_F32_SPLITK = 4,   // 4: C += partial sums (red.global.add)
       EPI_BF16_ACTBWD = 5,     // 5: C = bf16(acc * act'(U)), U = GemmParams::delta (bf16 [M, ldc]); C2 (fp32 [N], may be null) += column sums
       // Deterministic variants of 4 and 5 (leaf_set_deterministic): the partial sums go to GemmParams::ws, and the epilogue warp
       // that arrives last at a region (per-region counter in GemmParams::cnt) adds them to C / C2 in index order, so the result
       // does not depend on which work unit finished first. Own template instances: 4 and 5 keep their code and registers.
       EPI_F32_SPLITK_DET = 6, EPI_BF16_ACTBWD_DET = 7 };
enum { ACT_GELU_ERF = 0, ACT_QUICK_GELU = 1 };

struct GemmParams {
  int M;                  // rows (upper bound when m_dev != nullptr)
  const int* m_dev;       // optional device-side row count
  int N, K;
  const float* bias;      // [N] or nullptr
  void* C;                // bf16 or fp32 [M, ldc]
  const __nv_bfloat16* delta;   // EPI_F32_RESIDUAL only, may be null: bf16 [M, ldc] added to the residual as well
  const float* res;             // EPI_F32_RESIDUAL only, may be null: the residual is read from res [M, ldc] instead of C
                                // (C = res + acc + bias: the training forward keeps the block input, so no copy first)
  int ldc;
  int act;
  uint32_t tx_bytes;      // bytes one pipeline stage receives (TMA boxes are clamped to small tensors)
  // mn_major: bit 0 = A is given MN-major ([K, M] row-major), bit 1 = B is given MN-major ([K, N] row-major) instead of the
  // K-major [M, K] / [N, K]. The wgrad product dW[out,in] = dY[rows,out]^T . X[rows,in] reads dY and X as they lie (3), the
  // dgrad product dX[rows,in] = dY[rows,out] . W[out,in] reads the forward's weight copy as it lies (2): no transposes.
  int mn_major;
  // EPI_BF16_ACT only, may be null: the PRE-activation (acc + bias) is stored here as bf16 as well, same shape as C. The
  // training forward keeps fc1's output for the backward (act'(u)), so one epilogue writes u and act(u): no separate
  // activation pass over [rows, 4W] (utils_AT.py:317-319 forward of the winners).
  void* C2;
  // split-K (EPI_F32_SPLITK only, no bias): the k-blocks of one output tile are divided over `split_k` work units whose
  // epilogues ADD their partial sums into C with red.global.add.v4.f32 (C += A.B is what the weight-gradient products want
  // anyway). Its own template instance, so the hot fc2 epilogue (EPI_F32_RESIDUAL) keeps its register budget. 1 = off.
  int split_k;
  // EPI_F32_SPLITK_DET: ws holds one 256 x 256 fp32 partial tile per work unit, cnt one arrival counter per (output tile, epilogue
  // warp of the pair). EPI_BF16_ACTBWD_DET: ws holds the column sums of every 32-row chunk [ceil(M / 32), N], cnt one counter per
  // 64 columns. Counters are zero before the launch and are left at zero.
  float* ws;
  int* cnt;
};
constexpr int GEMM_A_MN = 1, GEMM_B_MN = 2;
// MN-major 128B-swizzled tile as TMA lays it down from a [K, MN] row-major tensor with a 64 (MN) x 64 (k) box: one 128-byte
// line per k, 8-line groups 1 KB apart (SBO), the next 64 MN elements in the next box 8 KB on (LBO); 16 k = 2 KB.
constexpr uint32_t GEMM_MN_LBO = 8192, GEMM_MN_SBO = 1024, GEMM_MN_KSTEP = 2048;

// ---------------------------------------------------------------------------------------------
// PTX wrappers
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
// Bounded wait: a protocol bug must end in a trap (reported as a CUDA error), never in a hung GPU.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t done = 0;
  long long t0 = 0;
  for (uint32_t it = 0;; ++it) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(bar), "r"(parity)
        : "memory");
    if (done) return;
    if (it == 1024) t0 = clock64();
    if (it > 1024 && (it & 1023) == 0 && clock64() - t0 > 4000000000LL) __trap();
  }
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* tmap) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(tmap)) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t* v) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
        "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
        "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// K-major, 128-byte swizzled operand tile whose rows are 128 bytes (64 bf16): 8-row groups are 1024 B apart
// (SBO), LBO is unused by swizzled K-major layouts (encoded 1), descriptor version 1 (Blackwell), layout 2.
__device__ __forceinline__ uint64_t make_smem_desc_sw128(uint32_t saddr) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((saddr & 0x3FFFF) >> 4);
  d |= static_cast<uint64_t>(1) << 16;
  d |= static_cast<uint64_t>(1024 >> 4) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(2) << 61;
  return d;
}
// kind::f16 instruction descriptor: D fp32, A/B bf16, both K-major, N>>3 at [17,23), M>>4 at [24,29).
__host__ __device__ constexpr uint32_t make_idesc_bf16(int m, int n) {
  return (1u << 4) | (1u << 7) | (1u << 10) | (static_cast<uint32_t>(n >> 3) << 17) | (static_cast<uint32_t>(m >> 4) << 24);
}
constexpr uint32_t IDESC_A_MN_MAJOR = 1u << 15, IDESC_B_MN_MAJOR = 1u << 16;
// MN-major, 128-byte swizzled operand tile: 64 MN elements (128 B) contiguous, one 128-byte line per k, 8-line groups
// `sbo` bytes apart, the next 64 MN elements `lbo` bytes away.
__device__ __forceinline__ uint64_t make_smem_desc_mn_sw128(uint32_t saddr, uint32_t lbo, uint32_t sbo) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((saddr & 0x3FFFF) >> 4);
  d |= static_cast<uint64_t>(lbo >> 4) << 16;
  d |= static_cast<uint64_t>(sbo >> 4) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(2) << 61;
  return d;
}

// sum of p[0], p[stride], ..., p[(n - 1) stride], added one after another in index order (the fixed order of the deterministic
// reductions' last step), with U loads in flight: these sums read L2-resident partials written by other SMs (hence .cg).
template <int U>
__device__ __forceinline__ float ordered_sum(const float* p, size_t stride, int n) {
  float t = 0.f;
  int i = 0;
  for (; i + U <= n; i += U) {
    float v[U];
#pragma unroll
    for (int u = 0; u < U; ++u) v[u] = __ldcg(p + static_cast<size_t>(i + u) * stride);
#pragma unroll
    for (int u = 0; u < U; ++u) t += v[u];
  }
  for (; i < n; ++i) t += __ldcg(p + static_cast<size_t>(i) * stride);
  return t;
}

__device__ __forceinline__ float fast_ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float fast_rcp(float x) {
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// nn.GELU (erf form) x Phi(x), written as x sigmoid(q(x)) with q(x) = x (c0 + c1 x^2 + c2 x^4) an odd polynomial fitted to
// 2 atanh(erf(x / sqrt 2)) (x^2 clamped at 36, beyond which sigmoid is 1 or 0 to 1e-9): 7 FP32 ops + 2 MUFU per element, the
// cost of QuickGELU plus three. No cancellation anywhere (the negative tail is a product, not a difference), so the error
// is the fit's: |error| <= 7e-5 absolute, relative 4e-4 where |y| > 0.01, 3e-3 where |y| > 0.001 - at or below the bf16
// rounding the result gets anyway (2^-9 relative); tools/fit_gelu.py reproduces the coefficients and these bounds.
// Before: max(x, 0) - 0.5 |x| erfc(|x| / sqrt 2) with Abramowitz-Stegun 7.1.26 (13 FP32 + 2 MUFU, |error| 1.5e-7) - exact
// beyond need for a bf16 result, and the fc1 GEMM ran 13 % below the QKV GEMM's rate per FLOP in situ because its
// epilogue's FP32 / MUFU work costs power under the board's cap; libdevice's erff (~39 instructions) before that.
__device__ __forceinline__ float gelu_erf(float x) {
  const float x2 = fminf(x * x, 36.0f);
  const float r = fmaf(x2, fmaf(x2, 0.0011236976601259265f, -0.10762115607988151f), -2.299969046114191f);   // -log2(e) q(x) / x
  return x * fast_rcp(1.0f + fast_ex2(x * r));
}
__device__ __forceinline__ float quick_gelu(float x) {                   // x sigmoid(1.702 x), transformer.py:33-36
  return x * fast_rcp(1.0f + fast_ex2(-1.702f * 1.4426950408889634f * x));
}
// Derivatives for the backward's fused epilogue (EPI_BF16_ACTBWD): Phi(x) + x phi(x) with Phi as in gelu_erf above (|error|
// <= 7e-5, the result is rounded to bf16), s + 1.702 x s (1 - s) for QuickGELU. 3 resp. 2 MUFU per element: exact erff / expf
// forms would make the epilogue four times the tile's MMA time. tests/test_gpu_backward.py compares with autograd's.
__device__ __forceinline__ float gelu_erf_grad(float x) {
  const float x2 = fminf(x * x, 36.0f);
  const float r = fmaf(x2, fmaf(x2, 0.0011236976601259265f, -0.10762115607988151f), -2.299969046114191f);
  const float cdf = fast_rcp(1.0f + fast_ex2(x * r));
  const float pdf = 0.3989422804014327f * fast_ex2(-0.5f * 1.4426950408889634f * x2);
  return fmaf(x, pdf, cdf);
}
__device__ __forceinline__ float quick_gelu_grad(float x) {
  const float s = fast_rcp(1.0f + fast_ex2(-1.702f * 1.4426950408889634f * x));
  return fmaf(1.702f * x * s, 1.0f - s, s);
}
// Fused epilogue of one 32-row x 32-column chunk of the accumulator. Each lane arrives with one ROW of the chunk
// (v = raw fp32 bits from TMEM, tcgen05.ld 32x32b); storing that directly would touch 32 different 128-byte lines per
// instruction (ncu r3: LSU wavefronts, not the tensor pipe, paced the K=1024 GEMMs). The chunk is bounced through a
// padded per-warp staging buffer (rows of 64 B at a stride of 80 B: the 16-byte accesses of 8 consecutive lanes hit 8
// distinct bank groups) and written with 8 rows x 64 B per instruction. bf16 outputs take one pass (32 columns),
// fp32 outputs two passes of 16 columns. The fp32 residual is loaded with the same mapping BEFORE the accumulator is
// read from TMEM, so its latency hides behind the TMEM load and the bias/activation math.
constexpr int EPI_WARPS = 16;                    // 4 per TMEM lane quadrant, 64 accumulator columns each
constexpr int EPI_STAGE_BYTES = 32 * 80;         // per warp
constexpr int GEMM_THREADS = 128 + 32 * EPI_WARPS;

struct ResidualRegs { float4 x[8]; };

template <int EPI>
__device__ __forceinline__ void epilogue_load_residual(const GemmParams& p, ResidualRegs& r, int lane, int row0, int col0, int M) {
  if (EPI != EPI_F32_RESIDUAL) return;
  const int c = lane & 3;
#pragma unroll
  for (int h = 0; h < 2; ++h) {
#pragma unroll
    for (int it = 0; it < 4; ++it) {
      const int row = row0 + it * 8 + (lane >> 2);
      const int col = col0 + h * 16 + c * 4;
      if (row < M && col < p.N)
        r.x[h * 4 + it] = *reinterpret_cast<const float4*>((p.res ? p.res : reinterpret_cast<const float*>(p.C)) + static_cast<size_t>(row) * p.ldc + col);
    }
  }
}

template <int EPI>
__device__ __forceinline__ void epilogue_chunk(const GemmParams& p, const uint32_t* v, const ResidualRegs& res, uint8_t* stage,
                                               int lane, int row0, int col0, int M) {
  float f[32];
#pragma unroll
  for (int j = 0; j < 32; ++j) f[j] = __uint_as_float(v[j]);
  if (p.bias) {
#pragma unroll
    for (int j = 0; j < 32; j += 4) {
      if (col0 + j < p.N) {
        const float4 b = __ldg(reinterpret_cast<const float4*>(p.bias + col0 + j));
        f[j] += b.x; f[j + 1] += b.y; f[j + 2] += b.z; f[j + 3] += b.w;
      }
    }
  }
  const int c = lane & 3;
  // bf16 tile store: 32 rows x 32 columns through the padded staging buffer, 8 rows x 64 B per store instruction
  auto store_bf16 = [&](void* dst) {
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      uint4 pk;
      __nv_bfloat162 t0 = __floats2bfloat162_rn(f[8 * q], f[8 * q + 1]);
      __nv_bfloat162 t1 = __floats2bfloat162_rn(f[8 * q + 2], f[8 * q + 3]);
      __nv_bfloat162 t2 = __floats2bfloat162_rn(f[8 * q + 4], f[8 * q + 5]);
      __nv_bfloat162 t3 = __floats2bfloat162_rn(f[8 * q + 6], f[8 * q + 7]);
      pk.x = *reinterpret_cast<uint32_t*>(&t0);
      pk.y = *reinterpret_cast<uint32_t*>(&t1);
      pk.z = *reinterpret_cast<uint32_t*>(&t2);
      pk.w = *reinterpret_cast<uint32_t*>(&t3);
      *reinterpret_cast<uint4*>(stage + lane * 80 + q * 16) = pk;
    }
    __syncwarp();
    const bool col_ok = col0 + c * 8 < p.N;
#pragma unroll
    for (int it = 0; it < 4; ++it) {
      const int r = it * 8 + (lane >> 2);
      const uint4 pk = *reinterpret_cast<const uint4*>(stage + r * 80 + c * 16);
      if (col_ok && row0 + r < M)
        *reinterpret_cast<uint4*>(reinterpret_cast<__nv_bfloat16*>(dst) + static_cast<size_t>(row0 + r) * p.ldc + col0 + c * 8) = pk;
    }
    __syncwarp();                                 // the staging buffer is reused by the next store / chunk
  };
  if (EPI == EPI_BF16_ACT) {
    if (p.C2) store_bf16(p.C2);                   // the pre-activation, kept for the backward
    if (p.act == ACT_QUICK_GELU) {
#pragma unroll
      for (int j = 0; j < 32; ++j) f[j] = quick_gelu(f[j]);
    } else {
#pragma unroll
      for (int j = 0; j < 32; ++j) f[j] = gelu_erf(f[j]);
    }
  }
  if (EPI == EPI_BF16_ACTBWD || EPI == EPI_BF16_ACTBWD_DET) {
    // du = dg * act'(u) (the backward's dgrad through fc2, fused with what was a separate activation-backward pass). The u tile comes in through the
    // staging buffer (8 rows x 64 B per load instruction), each lane then reads its own row; rows past M are zeroed (their
    // accumulators are whatever lay behind the operand) so that the column sums below - the gradient of fc1's bias - see
    // exactly the values stored, rounded to bf16.
#pragma unroll
    for (int it = 0; it < 4; ++it) {
      const int r = it * 8 + (lane >> 2);
      uint4 pk = make_uint4(0u, 0u, 0u, 0u);
      if (col0 + c * 8 < p.N && row0 + r < M)
        pk = *reinterpret_cast<const uint4*>(p.delta + static_cast<size_t>(row0 + r) * p.ldc + col0 + c * 8);
      *reinterpret_cast<uint4*>(stage + r * 80 + c * 16) = pk;
    }
    __syncwarp();
    const bool live = row0 + lane < M;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const uint4 pk = *reinterpret_cast<const uint4*>(stage + lane * 80 + q * 16);
      const uint32_t w[4] = {pk.x, pk.y, pk.z, pk.w};
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const float2 u = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&w[k]));
        const float g0 = p.act == ACT_QUICK_GELU ? quick_gelu_grad(u.x) : gelu_erf_grad(u.x);
        const float g1 = p.act == ACT_QUICK_GELU ? quick_gelu_grad(u.y) : gelu_erf_grad(u.y);
        const int j = 8 * q + 2 * k;
        f[j] = live ? __bfloat162float(__float2bfloat16_rn(f[j] * g0)) : 0.f;
        f[j + 1] = live ? __bfloat162float(__float2bfloat16_rn(f[j + 1] * g1)) : 0.f;
      }
    }
    __syncwarp();                                 // every lane has read its row before the store reuses the buffer
    store_bf16(p.C);
    if (p.C2) {
      // column sums over the 32 rows of the chunk: transpose-reduce by recursive halving (31 shuffles), lane j ends with column j
#pragma unroll
      for (int off = 16; off >= 1; off >>= 1) {
        const bool up = lane & off;
#pragma unroll
        for (int j = 0; j < off; ++j) {
          const float keep = up ? f[j + off] : f[j];
          const float send = up ? f[j] : f[j + off];
          f[j] = keep + __shfl_xor_sync(0xffffffffu, send, off);
        }
      }
      if (EPI == EPI_BF16_ACTBWD_DET) {
        if (col0 + lane < p.N) p.ws[static_cast<size_t>(row0 >> 5) * p.N + col0 + lane] = f[0];
      } else if (col0 + lane < p.N) {
        atomicAdd(reinterpret_cast<float*>(p.C2) + col0 + lane, f[0]);
      }
    }
  } else if (EPI == EPI_BF16 || EPI == EPI_BF16_ACT) {
    store_bf16(p.C);
  } else {
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      // the bf16 delta is fetched per pass (8 registers) rather than with the residual: the kernel sits at its register
      // cap, and the only user (fc2, K = 4W) has four times the mainloop time of the other GEMMs to hide the latency in
      uint2 dl[4];
      if (EPI == EPI_F32_RESIDUAL && p.delta) {
#pragma unroll
        for (int it = 0; it < 4; ++it) {
          const int row = row0 + it * 8 + (lane >> 2), col = col0 + h * 16 + c * 4;
          dl[it] = (row < M && col < p.N) ? *reinterpret_cast<const uint2*>(p.delta + static_cast<size_t>(row) * p.ldc + col)
                                          : make_uint2(0u, 0u);
        }
      }
#pragma unroll
      for (int q = 0; q < 4; ++q)
        *reinterpret_cast<float4*>(stage + lane * 80 + q * 16) =
            make_float4(f[16 * h + 4 * q], f[16 * h + 4 * q + 1], f[16 * h + 4 * q + 2], f[16 * h + 4 * q + 3]);
      __syncwarp();
      const int col = col0 + h * 16 + c * 4;
#pragma unroll
      for (int it = 0; it < 4; ++it) {
        const int r = it * 8 + (lane >> 2);
        float4 o = *reinterpret_cast<const float4*>(stage + r * 80 + c * 16);
        if (EPI == EPI_F32_SPLITK) {                        // partial sum of a split-K part: C += o, no read-modify-write
          if (col < p.N && row0 + r < M)
            atomicAdd(reinterpret_cast<float4*>(reinterpret_cast<float*>(p.C) + static_cast<size_t>(row0 + r) * p.ldc + col), o);
        } else if (col < p.N && row0 + r < M) {
          if (EPI == EPI_F32_RESIDUAL) {
            float4 x = res.x[h * 4 + it];
            if (p.delta) {                              // x + delta first: the sum LayerNorm saw (leaf_encode)
              const uint2 d = dl[it];
              const float2 d0 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&d.x));
              const float2 d1 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&d.y));
              x.x += d0.x; x.y += d0.y; x.z += d1.x; x.w += d1.y;
            }
            o.x += x.x; o.y += x.y; o.z += x.z; o.w += x.w;
          }
          *reinterpret_cast<float4*>(reinterpret_cast<float*>(p.C) + static_cast<size_t>(row0 + r) * p.ldc + col) = o;
        }
      }
      __syncwarp();
    }
  }
}

}  // namespace leaf
