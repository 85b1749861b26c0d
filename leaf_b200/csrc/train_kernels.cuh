// K4: kernels of the backward pass of the selected adversarial batch (the FARE-style update,
// /root/reference/utils_AT.py:312-337: encode_text(adv) in train mode, mse(...).sum(-1).mean(), backward).
// All matrix products (dgrad and wgrad) run on the tcgen05 GEMM (gemm2_sm100.cuh), which reads weights and activations as
// they lie (MN-major operands where the contraction runs over rows); the kernels here are the element-wise / per-row
// pieces around them.
// The batch is the B winners only (~3 % of the step's FLOPs), so these kernels are written for clarity and exact
// fp32 math, not for the roofline.
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "tower_kernels.cuh"

namespace leaf {

// The activation backward du = dg * act'(u) and fc1's bias gradient are the epilogue of the dgrad GEMM through fc2
// (gemm_sm100.cuh, EPI_BF16_ACTBWD); the training forward's fc1 epilogue stores u and act(u) together.
__global__ void scale_f32_kernel(float* __restrict__ g, size_t n, float s) {
  for (size_t i = (static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x) * 4; i + 3 < n; i += static_cast<size_t>(gridDim.x) * blockDim.x * 4) {
    float4 v = *reinterpret_cast<float4*>(g + i);
    v.x *= s; v.y *= s; v.z *= s; v.w *= s;
    *reinterpret_cast<float4*>(g + i) = v;
  }
}
__global__ void cast_f32_bf16_kernel(const float* __restrict__ src, __nv_bfloat16* __restrict__ dst, size_t n) {
  for (size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += static_cast<size_t>(gridDim.x) * blockDim.x)
    dst[i] = __float2bfloat16_rn(src[i]);
}

template <typename T>
__device__ __forceinline__ float to_f32(T v);
template <>
__device__ __forceinline__ float to_f32<float>(float v) { return v; }
template <>
__device__ __forceinline__ float to_f32<__nv_bfloat16>(__nv_bfloat16 v) { return __bfloat162float(v); }

// ---- LayerNorm backward: dx[row] (+)= rstd * (g*dy - mean(g*dy) - xhat * mean(g*dy*xhat)); dgamma += dy*xhat; dbeta += dy
// gather != nullptr: row r reads x[gather[r]] and WRITES dx[gather[r]] (final LN on the pooled rows).
// accumulate: dx += (residual branch) instead of dx = .
// Two kernels. (1) A row kernel, one warp per row: dx, its bf16 copy (the A operand of the next dgrad GEMM) and the row's
// (mean, rstd) saved to `stats`; no per-column accumulators, so two 8-warp CTAs fit an SM. (2) A column kernel in which a thread
// owns four adjacent columns over a band of rows and rebuilds dy * xhat from the saved statistics (dy, x, dx are L2-resident at
// K4's sizes): dgamma, dbeta and dxsum - the bias gradient of the Linear whose output gradient this dx is (fc2 of the layer below
// for ln_1 / ln_final, out-proj for ln_2) - with 2 x SMs x 3 x 256 global atomics per launch. The single kernel this replaces
// carried 3 x W/32 accumulators per lane through its row loop (255 registers, one CTA per SM) and ended in 3 W atomics per CTA:
// 33 us per launch at 4 k rows against 24 for the pair (profiles/r2_33_lnb_split_ab.txt).
template <int VPL>
__global__ void __launch_bounds__(256, VPL <= 10 ? 2 : 1) layernorm_bwd_rows_kernel(const float* __restrict__ dy, const float* __restrict__ x,
                                                                    const int* __restrict__ gather, int rows, int W,
                                                                    const float* __restrict__ gamma, float eps, float* __restrict__ dx,
                                                                    int accumulate, __nv_bfloat16* __restrict__ dx16,
                                                                    float2* __restrict__ stats) {
  pdl_trigger();
  const int lane = threadIdx.x & 31;
  const int warps_total = (gridDim.x * blockDim.x) >> 5;
  const float invW = 1.f / static_cast<float>(W);
  for (int r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; r < rows; r += warps_total) {
    const int xr = gather ? gather[r] : r;
    const float4* xin = reinterpret_cast<const float4*>(x + static_cast<size_t>(xr) * W);
    const float4* din = reinterpret_cast<const float4*>(dy + static_cast<size_t>(r) * W);
    float4* out = reinterpret_cast<float4*>(dx + static_cast<size_t>(xr) * W);
    float4 xv[VPL], dv[VPL];
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < VPL; ++i) {
      xv[i] = xin[lane + 32 * i];
      dv[i] = din[lane + 32 * i];
      s += (xv[i].x + xv[i].y) + (xv[i].z + xv[i].w);
    }
    const float mean = warp_sum(s) * invW;
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < VPL; ++i) {
      xv[i].x -= mean; xv[i].y -= mean; xv[i].z -= mean; xv[i].w -= mean;
      q += (xv[i].x * xv[i].x + xv[i].y * xv[i].y) + (xv[i].z * xv[i].z + xv[i].w * xv[i].w);
    }
    const float rstd = rsqrtf(warp_sum(q) * invW + eps);
    if (lane == 0) stats[r] = make_float2(mean, rstd);
    float s1 = 0.f, s2 = 0.f;                 // sum(g*dy), sum(g*dy*xhat)
#pragma unroll
    for (int i = 0; i < VPL; ++i) {
      const float4 g = __ldg(reinterpret_cast<const float4*>(gamma) + lane + 32 * i);
      xv[i].x *= rstd; xv[i].y *= rstd; xv[i].z *= rstd; xv[i].w *= rstd;      // xhat
      dv[i].x *= g.x; dv[i].y *= g.y; dv[i].z *= g.z; dv[i].w *= g.w;           // g*dy
      s1 += (dv[i].x + dv[i].y) + (dv[i].z + dv[i].w);
      s2 += (dv[i].x * xv[i].x + dv[i].y * xv[i].y) + (dv[i].z * xv[i].z + dv[i].w * xv[i].w);
    }
    s1 = warp_sum(s1) * invW;
    s2 = warp_sum(s2) * invW;
#pragma unroll
    for (int i = 0; i < VPL; ++i) {
      float4 o;
      o.x = rstd * (dv[i].x - s1 - xv[i].x * s2);
      o.y = rstd * (dv[i].y - s1 - xv[i].y * s2);
      o.z = rstd * (dv[i].z - s1 - xv[i].z * s2);
      o.w = rstd * (dv[i].w - s1 - xv[i].w * s2);
      if (accumulate) {
        const float4 p = out[lane + 32 * i];
        o.x += p.x; o.y += p.y; o.z += p.z; o.w += p.w;
      }
      out[lane + 32 * i] = o;
      if (dx16) {                              // bf16 copy: the A operand of the next dgrad GEMM
        uint2 pk;
        pk.x = pack_bf16x2(o.x, o.y);
        pk.y = pack_bf16x2(o.z, o.w);
        reinterpret_cast<uint2*>(dx16 + static_cast<size_t>(xr) * W)[lane + 32 * i] = pk;
      }
    }
  }
}

// dgamma[c] += sum_r dy[r,c] xhat[r,c], dbeta[c] += sum_r dy[r,c], dxsum[c] += sum_r dx[row(r),c] (dxsum may be null) over the
// rows of this CTA's band. CTA = 64 column quads (256 columns) x 4 row phases; grid = (ceil(W / 256), bands).
// Launched behind layernorm_bwd_rows_kernel with programmatic stream serialization: it reads that kernel's stats and dx.
// DET (leaf_set_deterministic): each band writes its sums to ws [bands][3][W] instead of adding them, and the last band of a
// column block to finish (counter cnt[blockIdx.x], zero before and after) adds them to the gradients in band order.
template <bool DET>
__global__ void __launch_bounds__(256) layernorm_bwd_cols_kernel(const float* __restrict__ dy, const float* __restrict__ x,
                                                                 const int* __restrict__ gather, const float2* __restrict__ stats,
                                                                 const float* __restrict__ dx, int rows, int W,
                                                                 float* __restrict__ dgamma, float* __restrict__ dbeta,
                                                                 float* __restrict__ dxsum, float* __restrict__ ws = nullptr,
                                                                 int* __restrict__ cnt = nullptr) {
  pdl_wait();
  pdl_trigger();
  __shared__ float4 red[3][4][64];
  const int quad = threadIdx.x & 63, ph = threadIdx.x >> 6;
  const int c = blockIdx.x * 256 + quad * 4;
  const int band = (rows + gridDim.y - 1) / gridDim.y, r0 = blockIdx.y * band, r1 = min(r0 + band, rows);
  float4 ag = make_float4(0.f, 0.f, 0.f, 0.f), ab = ag, as = ag;
  if (c < W) {
    auto one = [&](int r) {
      const int xr = gather ? gather[r] : r;
      const float2 st = __ldg(stats + r);
      const float4 d = *reinterpret_cast<const float4*>(dy + static_cast<size_t>(r) * W + c);
      const float4 v = *reinterpret_cast<const float4*>(x + static_cast<size_t>(xr) * W + c);
      ag.x += d.x * ((v.x - st.x) * st.y); ag.y += d.y * ((v.y - st.x) * st.y);
      ag.z += d.z * ((v.z - st.x) * st.y); ag.w += d.w * ((v.w - st.x) * st.y);
      ab.x += d.x; ab.y += d.y; ab.z += d.z; ab.w += d.w;
      if (dxsum) {
        const float4 o = *reinterpret_cast<const float4*>(dx + static_cast<size_t>(xr) * W + c);
        as.x += o.x; as.y += o.y; as.z += o.z; as.w += o.w;
      }
    };
    int r = r0 + ph;
    for (; r + 4 < r1; r += 8) { one(r); one(r + 4); }       // two independent rows in flight
    if (r < r1) one(r);
  }
  red[0][ph][quad] = ag;
  red[1][ph][quad] = ab;
  red[2][ph][quad] = as;
  __syncthreads();
  // 768 sums per CTA (3 arrays x 256 columns): thread t takes column t of each array
  const int col = blockIdx.x * 256 + threadIdx.x;
  const float* f = reinterpret_cast<const float*>(&red[0][0][0]);        // [array][phase][256 floats]
  float* dst[3] = {dgamma, dbeta, dxsum};
  if constexpr (DET) {
    __shared__ bool last;
    if (col < W) {
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        const float* a = f + (k * 4) * 256 + threadIdx.x;
        ws[(static_cast<size_t>(blockIdx.y) * 3 + k) * W + col] = (a[0] + a[256]) + (a[512] + a[768]);
      }
    }
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) last = atomicAdd(cnt + blockIdx.x, 1) == static_cast<int>(gridDim.y) - 1;
    __syncthreads();
    if (!last) return;
    __threadfence();
    if (col < W) {
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        if (!dst[k]) continue;
        dst[k][col] += ordered_sum<8>(ws + static_cast<size_t>(k) * W + col, static_cast<size_t>(3) * W, gridDim.y);
      }
    }
    if (threadIdx.x == 0) cnt[blockIdx.x] = 0;
  } else if (col < W && r1 > r0) {
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      if (!dst[k]) continue;
      const float* a = f + (k * 4) * 256 + threadIdx.x;
      atomicAdd(dst[k] + col, (a[0] + a[256]) + (a[512] + a[768]));
    }
  }
}

// ---- causal attention backward on the tensor cores: two warps per (sequence, head) ------------------------------------------
// qkv bf16 [rows,3W], o bf16 [rows,W] (forward output), dout fp32 [rows,W] -> dqkv bf16 [rows,3W].
//   P = softmax(scale Q K^T + causal), D_i = sum_d dO_id O_id, dP = dO V^T, dS = P o (dP - D),
//   dV = P^T dO, dQ = scale dS K, dK = scale dS^T Q.
// Q, K, V and dO (rounded to bf16, like every other GEMM operand of the backward) are staged in shared memory with rows
// padded to 72 elements (ldmatrix conflict-free), zero beyond the sequence. Pass 1 walks the 16-query tiles: S and dP of
// the whole (<= 5 key tiles) row block sit in registers (mma.sync.m16n8k16, fp32 accumulate), softmax and dS in fp32, dQ
// straight from the dS accumulator registers (a C fragment pair IS the next product's A fragment); P and dS go to
// shared memory as bf16. Pass 2 walks the key tiles and reads them back TRANSPOSED (ldmatrix.trans) for dV and dK.
// The scalar fp32 version this replaces (one CTA per pair, 221 us per layer at B = 128) was the largest K4 kernel.
// T16 = longest sequence of the batch rounded up to 16 (sizes the shared-memory arrays).
constexpr int ATTB_PITCH = 72;
__host__ __device__ constexpr int attb_smem_bytes(int T) {
  const int T16 = (T + 15) / 16 * 16;
  return 4 * T16 * ATTB_PITCH * 2 + 2 * T16 * (T16 + 8) * 2 + T16 * 4;
}
__device__ __forceinline__ void ldsm_x4(uint32_t (&r)[4], uint32_t addr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
__device__ __forceinline__ void ldsm_x4_t(uint32_t (&r)[4], uint32_t addr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}

// Pass 1 for the query tile qi (NKT = qi + 1 key tiles under the causal mask, no shared prefix in training batches)
template <int NKT>
__device__ __forceinline__ void attb_query_tile(uint32_t sQ, uint32_t sK, uint32_t sV, uint32_t sdO, __nv_bfloat16* Ps, __nv_bfloat16* dSs,
                                                const float* Dv, int PP, int lane, float (&dq)[8][4]) {
  constexpr int qi = NKT - 1;
  const int g = lane >> 2, c = lane & 3;
  const float sl2 = 0.125f * 1.4426950408889634f;
  // A fragments of Q and dO rows 16qi.., four k-steps of 16 over d
  const uint32_t a_off = static_cast<uint32_t>(((16 * qi + (lane & 7) + 8 * ((lane >> 3) & 1)) * ATTB_PITCH + 8 * (lane >> 4)) * 2);
  uint32_t aq[4][4], ado[4][4];
#pragma unroll
  for (int ks = 0; ks < 4; ++ks) {
    ldsm_x4(aq[ks], sQ + a_off + ks * 32);
    ldsm_x4(ado[ks], sdO + a_off + ks * 32);
  }
  float s[NKT][2][4], dp[NKT][2][4];
  // B fragments of K / V stored [key][d]: matrices (keys 0-7, d 0-7), (keys 0-7, d 8-15), (keys 8-15, d 0-7), (keys 8-15, d 8-15)
  const uint32_t b_off = static_cast<uint32_t>((((lane & 7) + 8 * (lane >> 4)) * ATTB_PITCH + 8 * ((lane >> 3) & 1)) * 2);
#pragma unroll
  for (int kj = 0; kj < NKT; ++kj) {
#pragma unroll
    for (int nt = 0; nt < 2; ++nt)
#pragma unroll
      for (int e = 0; e < 4; ++e) s[kj][nt][e] = dp[kj][nt][e] = 0.f;
#pragma unroll
    for (int ks = 0; ks < 4; ++ks) {
      uint32_t bk[4], bv[4];
      ldsm_x4(bk, sK + b_off + (16 * kj * ATTB_PITCH + 16 * ks) * 2);
      ldsm_x4(bv, sV + b_off + (16 * kj * ATTB_PITCH + 16 * ks) * 2);
      mma_bf16_16816(s[kj][0], aq[ks], bk[0], bk[1]);
      mma_bf16_16816(s[kj][1], aq[ks], bk[2], bk[3]);
      mma_bf16_16816(dp[kj][0], ado[ks], bv[0], bv[1]);
      mma_bf16_16816(dp[kj][1], ado[ks], bv[2], bv[3]);
    }
  }
  // causal mask, softmax rows g and g+8 of the tile
  const int i0 = 16 * qi + g, i1 = i0 + 8;
  float mx0 = -INFINITY, mx1 = -INFINITY;
#pragma unroll
  for (int kj = 0; kj < NKT; ++kj)
#pragma unroll
    for (int nt = 0; nt < 2; ++nt)
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const int j = 16 * kj + 8 * nt + 2 * c + e;
        if (j > i0) s[kj][nt][e] = -INFINITY;
        if (j > i1) s[kj][nt][2 + e] = -INFINITY;
        mx0 = fmaxf(mx0, s[kj][nt][e]);
        mx1 = fmaxf(mx1, s[kj][nt][2 + e]);
      }
  mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 1));
  mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 2));
  mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 1));
  mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 2));
  float l0 = 0.f, l1 = 0.f;
#pragma unroll
  for (int kj = 0; kj < NKT; ++kj)
#pragma unroll
    for (int nt = 0; nt < 2; ++nt)
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        s[kj][nt][e] = att_ex2((s[kj][nt][e] - mx0) * sl2);
        s[kj][nt][2 + e] = att_ex2((s[kj][nt][2 + e] - mx1) * sl2);
        l0 += s[kj][nt][e];
        l1 += s[kj][nt][2 + e];
      }
  l0 += __shfl_xor_sync(0xffffffffu, l0, 1);
  l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
  l1 += __shfl_xor_sync(0xffffffffu, l1, 1);
  l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
  const float inv0 = 1.f / l0, inv1 = 1.f / l1, d0 = Dv[i0], d1 = Dv[i1];
#pragma unroll
  for (int i = 0; i < 8; ++i) dq[i][0] = dq[i][1] = dq[i][2] = dq[i][3] = 0.f;
  // K stored [key][d] read as the B operand [k = key][n = d]: transposed 8x8 loads
  const uint32_t bt_off = static_cast<uint32_t>((((lane & 7) + 8 * ((lane >> 3) & 1)) * ATTB_PITCH + 8 * (lane >> 4)) * 2);
#pragma unroll
  for (int kj = 0; kj < NKT; ++kj) {
    uint32_t ads[4];                                       // dS tile as the A fragment of dQ += dS K
#pragma unroll
    for (int nt = 0; nt < 2; ++nt) {
      const float p00 = s[kj][nt][0] * inv0, p01 = s[kj][nt][1] * inv0, p10 = s[kj][nt][2] * inv1, p11 = s[kj][nt][3] * inv1;
      const float t00 = 0.125f * p00 * (dp[kj][nt][0] - d0), t01 = 0.125f * p01 * (dp[kj][nt][1] - d0);
      const float t10 = 0.125f * p10 * (dp[kj][nt][2] - d1), t11 = 0.125f * p11 * (dp[kj][nt][3] - d1);
      const uint32_t pp0 = pack_bf16x2(p00, p01), pp1 = pack_bf16x2(p10, p11);
      ads[2 * nt] = pack_bf16x2(t00, t01);
      ads[2 * nt + 1] = pack_bf16x2(t10, t11);
      const int col = 16 * kj + 8 * nt + 2 * c;
      *reinterpret_cast<uint32_t*>(Ps + i0 * PP + col) = pp0;
      *reinterpret_cast<uint32_t*>(Ps + i1 * PP + col) = pp1;
      *reinterpret_cast<uint32_t*>(dSs + i0 * PP + col) = ads[2 * nt];
      *reinterpret_cast<uint32_t*>(dSs + i1 * PP + col) = ads[2 * nt + 1];
    }
#pragma unroll
    for (int nd = 0; nd < 4; ++nd) {                       // d blocks of 16: two n8 tiles each
      uint32_t bk[4];
      ldsm_x4_t(bk, sK + bt_off + (16 * kj * ATTB_PITCH + 16 * nd) * 2);
      mma_bf16_16816(dq[2 * nd], ads, bk[0], bk[1]);
      mma_bf16_16816(dq[2 * nd + 1], ads, bk[2], bk[3]);
    }
  }
}

// Column sums of a 16 x 64 accumulator tile (8 n8 blocks) over its 16 rows, left on the lanes with g == 0 (lane c holds
// columns 8 n8 + 2c, +1): the bias gradient of the in-projection is the column sum of dQ | dK | dV.
__device__ __forceinline__ void attb_colsum(const float (&acc)[8][4], float (&sum)[8][2]) {
#pragma unroll
  for (int n8 = 0; n8 < 8; ++n8) {
    float a = acc[n8][0] + acc[n8][2], b = acc[n8][1] + acc[n8][3];
#pragma unroll
    for (int o = 4; o < 32; o <<= 1) {
      a += __shfl_xor_sync(0xffffffffu, a, o);
      b += __shfl_xor_sync(0xffffffffu, b, o);
    }
    sum[n8][0] += a;
    sum[n8][1] += b;
  }
}

// db_q / db_k / db_v (each may be null): [W] fp32, += the column sums of dQ / dK / dV (the in-projection's bias gradient;
// the rows beyond a sequence's length are exactly zero in all three, so they do not disturb the sums)
// Two warps per (sequence, head): they split the staging rows, the query tiles of pass 1 and the key tiles of pass 2 (round
// robin; the shared-memory footprint - what limits the CTAs per SM - is per item, so the second warp doubles the warps in flight).
// DET (leaf_set_deterministic): each warp writes its column sums to ws [sequence][warp][q|k|v][W] instead of adding them, and
// the last CTA of a head to finish (counter cnt[head], zero before and after) adds them in (sequence, warp) order.
constexpr int ATTB_WARPS = 2;
template <bool DET>
__global__ void __launch_bounds__(ATTB_WARPS * 32) attention_bwd_kernel(const __nv_bfloat16* __restrict__ qkv, const __nv_bfloat16* __restrict__ o,
                                                           const float* __restrict__ dout, const int4* __restrict__ meta,
                                                           int W, int T, __nv_bfloat16* __restrict__ dqkv,
                                                           float* __restrict__ db_q = nullptr, float* __restrict__ db_k = nullptr,
                                                           float* __restrict__ db_v = nullptr, float* __restrict__ ws = nullptr,
                                                           int* __restrict__ cnt = nullptr) {
  pdl_trigger();
  extern __shared__ __align__(16) uint8_t attb_sm[];
  const int T16 = (T + 15) / 16 * 16, PP = T16 + 8;
  __nv_bfloat16* Qs = reinterpret_cast<__nv_bfloat16*>(attb_sm);
  __nv_bfloat16* Ks = Qs + T16 * ATTB_PITCH;
  __nv_bfloat16* Vs = Ks + T16 * ATTB_PITCH;
  __nv_bfloat16* dOs = Vs + T16 * ATTB_PITCH;
  __nv_bfloat16* Ps = dOs + T16 * ATTB_PITCH;
  __nv_bfloat16* dSs = Ps + T16 * PP;
  float* Dv = reinterpret_cast<float*>(dSs + T16 * PP);
  const int seq = blockIdx.x, head = blockIdx.y, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int4 mt = meta[seq];
  const int row0 = mt.x, t = min(mt.y, T);              // training batches are packed without prefix sharing (p = 0)
  const int nt16 = (t + 15) / 16;                        // 16-row tiles of this sequence
  const size_t ld = static_cast<size_t>(3) * W;
  // ---- stage Q, K, V, dO (bf16) and D_i; 8 lanes per row, 16 bytes (8 elements) per lane ----
  const int sub = lane & 7;
  for (int r = threadIdx.x >> 3; r < nt16 * 16; r += 4 * ATTB_WARPS) {
    uint4 q = make_uint4(0, 0, 0, 0), k = q, v = q, d = q;
    float dsum = 0.f;
    if (r < t) {
      const __nv_bfloat16* b = qkv + static_cast<size_t>(row0 + r) * ld + head * 64 + sub * 8;
      q = *reinterpret_cast<const uint4*>(b);
      k = *reinterpret_cast<const uint4*>(b + W);
      v = *reinterpret_cast<const uint4*>(b + 2 * W);
      const float* dr = dout + static_cast<size_t>(row0 + r) * W + head * 64 + sub * 8;
      const float4 f0 = *reinterpret_cast<const float4*>(dr), f1 = *reinterpret_cast<const float4*>(dr + 4);
      const uint4 ob = *reinterpret_cast<const uint4*>(o + static_cast<size_t>(row0 + r) * W + head * 64 + sub * 8);
      const __nv_bfloat162* o2 = reinterpret_cast<const __nv_bfloat162*>(&ob);
      const float2 o0 = __bfloat1622float2(o2[0]), o1 = __bfloat1622float2(o2[1]), o2f = __bfloat1622float2(o2[2]), o3 = __bfloat1622float2(o2[3]);
      dsum = (f0.x * o0.x + f0.y * o0.y) + (f0.z * o1.x + f0.w * o1.y) + (f1.x * o2f.x + f1.y * o2f.y) + (f1.z * o3.x + f1.w * o3.y);
      d.x = pack_bf16x2(f0.x, f0.y); d.y = pack_bf16x2(f0.z, f0.w); d.z = pack_bf16x2(f1.x, f1.y); d.w = pack_bf16x2(f1.z, f1.w);
    }
    dsum += __shfl_xor_sync(0xffffffffu, dsum, 1);
    dsum += __shfl_xor_sync(0xffffffffu, dsum, 2);
    dsum += __shfl_xor_sync(0xffffffffu, dsum, 4);
    *reinterpret_cast<uint4*>(Qs + r * ATTB_PITCH + sub * 8) = q;
    *reinterpret_cast<uint4*>(Ks + r * ATTB_PITCH + sub * 8) = k;
    *reinterpret_cast<uint4*>(Vs + r * ATTB_PITCH + sub * 8) = v;
    *reinterpret_cast<uint4*>(dOs + r * ATTB_PITCH + sub * 8) = d;
    if (sub == 0) Dv[r] = dsum;
  }
  __syncthreads();
  const uint32_t sQ = smem_u32(Qs), sK = smem_u32(Ks), sV = smem_u32(Vs), sdO = smem_u32(dOs);
  const int g = lane >> 2, c = lane & 3;
  // ---- pass 1: per query tile S, dP, softmax, dS, dQ; P and dS to shared memory ----
  float sq[8][2], sk[8][2], sv[8][2];
#pragma unroll
  for (int i = 0; i < 8; ++i) sq[i][0] = sq[i][1] = sk[i][0] = sk[i][1] = sv[i][0] = sv[i][1] = 0.f;
  for (int qi = warp; qi < nt16; qi += ATTB_WARPS) {
    float dq[8][4];
    switch (qi) {                                          // warp-uniform
      case 0: attb_query_tile<1>(sQ, sK, sV, sdO, Ps, dSs, Dv, PP, lane, dq); break;
      case 1: attb_query_tile<2>(sQ, sK, sV, sdO, Ps, dSs, Dv, PP, lane, dq); break;
      case 2: attb_query_tile<3>(sQ, sK, sV, sdO, Ps, dSs, Dv, PP, lane, dq); break;
      case 3: attb_query_tile<4>(sQ, sK, sV, sdO, Ps, dSs, Dv, PP, lane, dq); break;
      default: attb_query_tile<5>(sQ, sK, sV, sdO, Ps, dSs, Dv, PP, lane, dq); break;
    }
    const int i0 = 16 * qi + g, i1 = i0 + 8;
    if (db_q) attb_colsum(dq, sq);
#pragma unroll
    for (int n8 = 0; n8 < 8; ++n8) {
      __nv_bfloat16* dst = dqkv + head * 64 + 8 * n8 + 2 * c;
      if (i0 < t) *reinterpret_cast<uint32_t*>(dst + static_cast<size_t>(row0 + i0) * ld) = pack_bf16x2(dq[n8][0], dq[n8][1]);
      if (i1 < t) *reinterpret_cast<uint32_t*>(dst + static_cast<size_t>(row0 + i1) * ld) = pack_bf16x2(dq[n8][2], dq[n8][3]);
    }
  }
  __syncthreads();
  // ---- pass 2: per key tile dV = sum_qi P^T dO, dK = sum_qi dS^T Q over the query tiles qi >= kj ----
  const uint32_t sP = smem_u32(Ps), sdS = smem_u32(dSs);
  // A operand from transposed storage: matrices (i 0-7, j 0-7), (i 0-7, j 8-15), (i 8-15, j 0-7), (i 8-15, j 8-15) of the [i][j] tile
  const int mi = lane >> 3;
  const uint32_t at_row = static_cast<uint32_t>((lane & 7) + 8 * (mi >> 1)), at_col = static_cast<uint32_t>(8 * (mi & 1));
  const uint32_t bt_off = static_cast<uint32_t>((((lane & 7) + 8 * ((lane >> 3) & 1)) * ATTB_PITCH + 8 * (lane >> 4)) * 2);
  for (int kj = warp; kj < nt16; kj += ATTB_WARPS) {
    float dv[8][4], dk[8][4];
#pragma unroll
    for (int i = 0; i < 8; ++i) dv[i][0] = dv[i][1] = dv[i][2] = dv[i][3] = dk[i][0] = dk[i][1] = dk[i][2] = dk[i][3] = 0.f;
    for (int qi = kj; qi < nt16; ++qi) {
      uint32_t ap[4], ads[4];
      const uint32_t off = ((16 * qi + at_row) * PP + 16 * kj + at_col) * 2;
      ldsm_x4_t(ap, sP + off);
      ldsm_x4_t(ads, sdS + off);
#pragma unroll
      for (int nd = 0; nd < 4; ++nd) {
        uint32_t bo[4], bq[4];
        ldsm_x4_t(bo, sdO + bt_off + (16 * qi * ATTB_PITCH + 16 * nd) * 2);
        ldsm_x4_t(bq, sQ + bt_off + (16 * qi * ATTB_PITCH + 16 * nd) * 2);
        mma_bf16_16816(dv[2 * nd], ap, bo[0], bo[1]);
        mma_bf16_16816(dv[2 * nd + 1], ap, bo[2], bo[3]);
        mma_bf16_16816(dk[2 * nd], ads, bq[0], bq[1]);
        mma_bf16_16816(dk[2 * nd + 1], ads, bq[2], bq[3]);
      }
    }
    const int j0 = 16 * kj + g, j1 = j0 + 8;
    if (db_k) attb_colsum(dk, sk);
    if (db_v) attb_colsum(dv, sv);
#pragma unroll
    for (int n8 = 0; n8 < 8; ++n8) {
      __nv_bfloat16* dst = dqkv + head * 64 + 8 * n8 + 2 * c;
      if (j0 < t) {
        *reinterpret_cast<uint32_t*>(dst + static_cast<size_t>(row0 + j0) * ld + W) = pack_bf16x2(dk[n8][0], dk[n8][1]);
        *reinterpret_cast<uint32_t*>(dst + static_cast<size_t>(row0 + j0) * ld + 2 * W) = pack_bf16x2(dv[n8][0], dv[n8][1]);
      }
      if (j1 < t) {
        *reinterpret_cast<uint32_t*>(dst + static_cast<size_t>(row0 + j1) * ld + W) = pack_bf16x2(dk[n8][2], dk[n8][3]);
        *reinterpret_cast<uint32_t*>(dst + static_cast<size_t>(row0 + j1) * ld + 2 * W) = pack_bf16x2(dv[n8][2], dv[n8][3]);
      }
    }
  }
  if constexpr (DET) {
    if (!db_q && !db_k && !db_v) return;                 // uniform over the grid
    __shared__ bool last;
    if (g == 0) {
      float* w = ws + static_cast<size_t>(seq * ATTB_WARPS + warp) * 3 * W;
#pragma unroll
      for (int n8 = 0; n8 < 8; ++n8) {
        const int col = head * 64 + 8 * n8 + 2 * c;
        *reinterpret_cast<float2*>(w + col) = make_float2(sq[n8][0], sq[n8][1]);
        *reinterpret_cast<float2*>(w + W + col) = make_float2(sk[n8][0], sk[n8][1]);
        *reinterpret_cast<float2*>(w + 2 * W + col) = make_float2(sv[n8][0], sv[n8][1]);
      }
    }
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) last = atomicAdd(cnt + head, 1) == static_cast<int>(gridDim.x) - 1;
    __syncthreads();
    if (!last) return;
    __threadfence();
    float* dst[3] = {db_q, db_k, db_v};
    for (int j = threadIdx.x; j < 3 * 64; j += ATTB_WARPS * 32) {
      const int k = j >> 6, col = head * 64 + (j & 63);
      if (!dst[k]) continue;
      dst[k][col] += ordered_sum<16>(ws + static_cast<size_t>(k) * W + col, static_cast<size_t>(3) * W, gridDim.x * ATTB_WARPS);
    }
    if (threadIdx.x == 0) cnt[head] = 0;
  } else if (g == 0) {
#pragma unroll
    for (int n8 = 0; n8 < 8; ++n8) {
      const int col = head * 64 + 8 * n8 + 2 * c;
      if (db_q) { atomicAdd(db_q + col, sq[n8][0]); atomicAdd(db_q + col + 1, sq[n8][1]); }
      if (db_k) { atomicAdd(db_k + col, sk[n8][0]); atomicAdd(db_k + col + 1, sk[n8][1]); }
      if (db_v) { atomicAdd(db_v + col, sv[n8][0]); atomicAdd(db_v + col + 1, sv[n8][1]); }
    }
  }
}

// ---- embedding backward: dtok[id] += dx[row], dpos[pos] += dx[row] -------------------------------------------------------
__global__ void __launch_bounds__(256) embed_bwd_kernel(const int* __restrict__ tok, const int4* __restrict__ meta, int N, int W,
                                                        const float* __restrict__ dx, float* __restrict__ dtok,
                                                        float* __restrict__ dpos) {
  const int seq = blockIdx.x;
  if (seq >= N) return;
  const int4 mt = meta[seq];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarp = blockDim.x >> 5;
  for (int pos = mt.z + warp; pos < mt.y; pos += nwarp) {
    const int id = tok[seq * 77 + pos];
    const float* g = dx + static_cast<size_t>(mt.x + pos - mt.z) * W;
    for (int c = lane; c < W; c += 32) {
      const float v = g[c];
      atomicAdd(dtok + static_cast<size_t>(id) * W + c, v);
      atomicAdd(dpos + static_cast<size_t>(pos) * W + c, v);
    }
  }
}

// ---- deterministic embedding backward (leaf_set_deterministic): one writer per table row, summing in packed-row order ---------
// embed_sort_kernel (one CTA, LEAF_VOCAB ints of shared memory) groups the packed rows by token id with a stable counting sort:
// row_tok[r] = token id of packed row r, order[] = the rows sorted by (id, row), key[i] = row_tok[order[i]].
__global__ void __launch_bounds__(1024) embed_sort_kernel(const int* __restrict__ tok, const int4* __restrict__ meta, int N, int M,
                                                          int* __restrict__ row_tok, int* __restrict__ order, int* __restrict__ key) {
  extern __shared__ int cursor[];                          // [LEAF_VOCAB]: counts, then the next free slot of each id
  __shared__ int wsum[32];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (int i = tid; i < LEAF_VOCAB; i += 1024) cursor[i] = 0;
  __syncthreads();
  for (int i = tid; i < N * LEAF_CTX; i += 1024) {
    const int seq = i / LEAF_CTX, pos = i - seq * LEAF_CTX;
    const int4 mt = meta[seq];
    if (pos >= mt.z && pos < mt.y) {
      const int id = tok[i];
      row_tok[mt.x + pos - mt.z] = id;
      atomicAdd(cursor + id, 1);
    }
  }
  __syncthreads();
  // exclusive scan of the counts: thread t owns ids [t * per, (t + 1) * per)
  constexpr int per = (LEAF_VOCAB + 1023) / 1024;
  const int lo = tid * per, hi = min(lo + per, static_cast<int>(LEAF_VOCAB));
  int s = 0;
  for (int i = lo; i < hi; ++i) s += cursor[i];
  int incl = s;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int v = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += v;
  }
  if (lane == 31) wsum[warp] = incl;
  __syncthreads();
  if (warp == 0) {
    int w = wsum[lane];
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int v = __shfl_up_sync(0xffffffffu, w, o);
      if (lane >= o) w += v;
    }
    wsum[lane] = w;                                        // inclusive over warps
  }
  __syncthreads();
  int run = incl - s + (warp ? wsum[warp - 1] : 0);
  for (int i = lo; i < hi; ++i) { const int c = cursor[i]; cursor[i] = run; run += c; }
  __syncthreads();
  // stable scatter in row order by one warp, 32 rows per step (ids of 8 steps loaded ahead)
  if (warp == 0) {
    for (int b0 = 0; b0 < M; b0 += 256) {
      int ids[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) ids[u] = (b0 + 32 * u + lane < M) ? row_tok[b0 + 32 * u + lane] : -1;
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const int r = b0 + 32 * u + lane, id = ids[u];
        const unsigned peers = __match_any_sync(0xffffffffu, id);
        const int start = id >= 0 ? cursor[id] : 0;
        __syncwarp();
        if (id >= 0) {
          const int at = start + __popc(peers & ((1u << lane) - 1u));
          order[at] = r;
          key[at] = id;
          if (lane == 31 - __clz(peers)) cursor[id] = start + __popc(peers);
        }
        __syncwarp();
      }
    }
  }
}

// grid (M + LEAF_CTX, ceil(W / 256)): block x < M that starts a run of equal keys adds dtok[id] += the run's dx rows in row
// order; block x = M + pos adds dpos[pos] += the dx rows of position pos in sequence order.
__global__ void __launch_bounds__(256) embed_bwd_det_kernel(const int* __restrict__ order, const int* __restrict__ key,
                                                            const int4* __restrict__ meta, int N, int M, int W,
                                                            const float* __restrict__ dx, float* __restrict__ dtok,
                                                            float* __restrict__ dpos) {
  const int c = blockIdx.y * 256 + threadIdx.x;
  const int i = blockIdx.x;
  if (i < M) {
    const int id = key[i];
    if ((i > 0 && key[i - 1] == id) || c >= W) return;
    float t = 0.f;
    for (int j = i; j < M; j += 8) {
      int rows[8];
      bool in[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        in[u] = j + u < M && key[j + u] == id;
        rows[u] = in[u] ? order[j + u] : 0;
      }
      float v[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) v[u] = in[u] ? dx[static_cast<size_t>(rows[u]) * W + c] : 0.f;
#pragma unroll
      for (int u = 0; u < 8; ++u)
        if (in[u]) t += v[u];
      if (!in[7]) break;
    }
    dtok[static_cast<size_t>(id) * W + c] += t;
    return;
  }
  const int pos = i - M;
  if (c >= W) return;
  float t = 0.f;
  for (int s0 = 0; s0 < N; s0 += 8) {                      // 8 sequences' loads in flight, added in sequence order
    float v[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const int4 mt = s0 + u < N ? meta[s0 + u] : make_int4(0, 0, 0, 0);
      v[u] = (pos >= mt.z && pos < mt.y) ? dx[static_cast<size_t>(mt.x + pos - mt.z) * W + c] : 0.f;
    }
#pragma unroll
    for (int u = 0; u < 8; ++u) t += v[u];
  }
  dpos[static_cast<size_t>(pos) * W + c] += t;
}

// ---- AdamW over the tower's flat parameter buffer (torch.optim.AdamW semantics, decoupled weight decay;
// train_AT_text_only.py:326-341: gains / biases / LayerNorm parameters form a group with weight_decay = 0 and are laid
// out first, elements [0, n_nodecay)). g is multiplied by grad_scale first (1/accum_freq, or the clipping
// coefficient). bc1 = 1 - beta1^t, bc2s = sqrt(1 - beta2^t). HBM bound: 28 B per element.
__global__ void __launch_bounds__(256) adamw_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                                                    float* __restrict__ v, size_t n, size_t n_nodecay, float lr, float beta1,
                                                    float beta2, float eps, float wd, float bc1, float bc2s, float grad_scale) {
  const size_t stride = static_cast<size_t>(gridDim.x) * blockDim.x * 4;
  for (size_t i = (static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x) * 4; i < n; i += stride) {
    float4 pv = *reinterpret_cast<const float4*>(p + i), gv = *reinterpret_cast<const float4*>(g + i);
    float4 mv = *reinterpret_cast<const float4*>(m + i), vv = *reinterpret_cast<const float4*>(v + i);
    float* pp = &pv.x; float* gg = &gv.x; float* mm = &mv.x; float* vs = &vv.x;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float gj = gg[j] * grad_scale;
      if (i + j >= n_nodecay) pp[j] *= 1.f - lr * wd;
      mm[j] = beta1 * mm[j] + (1.f - beta1) * gj;              // lerp(m, g, 1 - beta1)
      vs[j] = beta2 * vs[j] + (1.f - beta2) * gj * gj;
      const float denom = sqrtf(vs[j]) / bc2s + eps;
      pp[j] -= (lr / bc1) * (mm[j] / denom);
    }
    *reinterpret_cast<float4*>(p + i) = pv;
    *reinterpret_cast<float4*>(m + i) = mv;
    *reinterpret_cast<float4*>(v + i) = vv;
  }
}

// sum of squares of a flat fp32 buffer (gradient-norm clipping, utils_AT.py:349-357): out[0] += sum(g^2)
// DET (leaf_set_deterministic): every block writes its sum to ws[blockIdx.x]; the last block to finish (counter *cnt, zero before
// and after) adds them up in a fixed order: thread t takes blocks t, t + 256, ..., then the block reduction below.
template <bool DET>
__global__ void __launch_bounds__(256) sumsq_kernel(const float* __restrict__ g, size_t n, float* __restrict__ out,
                                                    float* __restrict__ ws = nullptr, int* __restrict__ cnt = nullptr) {
  __shared__ float part[8];
  float s = 0.f;
  const size_t stride = static_cast<size_t>(gridDim.x) * blockDim.x * 4;
  for (size_t i = (static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x) * 4; i < n; i += stride) {
    const float4 v = *reinterpret_cast<const float4*>(g + i);
    s += (v.x * v.x + v.y * v.y) + (v.z * v.z + v.w * v.w);
  }
  s = warp_sum(s);
  if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) t += part[i];
    if constexpr (DET) ws[blockIdx.x] = t;
    else atomicAdd(out, t);
  }
  if constexpr (DET) {
    __shared__ bool last;
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) last = atomicAdd(cnt, 1) == static_cast<int>(gridDim.x) - 1;
    __syncthreads();
    if (!last) return;
    __threadfence();
    float u = 0.f;
    for (int b = threadIdx.x; b < static_cast<int>(gridDim.x); b += 256) u += __ldcg(ws + b);
    u = warp_sum(u);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = u;
    __syncthreads();
    if (threadIdx.x == 0) {
      float t = 0.f;
#pragma unroll
      for (int i = 0; i < 8; ++i) t += part[i];
      out[0] += t;
      *cnt = 0;
    }
  }
}

// dst[r, :] += src[r, :] (fp32), used to add the attention/MLP branch gradient into the running dx
__global__ void add_f32_kernel(const float* __restrict__ src, float* __restrict__ dst, size_t n) {
  for (size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += static_cast<size_t>(gridDim.x) * blockDim.x)
    dst[i] += src[i];
}

// dst[W,E] += src[E,W]^T (HF projection layout -> open_clip layout or back), fp32
__global__ void add_transposed_f32_kernel(const float* __restrict__ src, float* __restrict__ dst, int R, int C) {
  __shared__ float tile[32][33];
  const int c0 = blockIdx.x * 32, r0 = blockIdx.y * 32;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int r = r0 + i, c = c0 + threadIdx.x;
    tile[i][threadIdx.x] = (r < R && c < C) ? src[static_cast<size_t>(r) * C + c] : 0.f;
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int c = c0 + i, r = r0 + threadIdx.x;
    if (c < C && r < R) dst[static_cast<size_t>(c) * R + r] += tile[threadIdx.x][i];
  }
}

}  // namespace leaf
