// Non-GEMM kernels of the text tower and the TextFARE score (sm_100a).
// Token rows are PACKED: sequence i owns rows [cu[i], cu[i] + len[i]) where len[i] = argmax(ids)+1; positions
// after the pooled EOS row cannot influence it under the causal mask (transformer.py:758-764) and are skipped.
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "gemm_sm100.cuh"   // pdl_wait / pdl_trigger

namespace leaf {

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// ---------------------------------------------------------------------------------------------
// exclusive scan of the (own) row lengths -> cu[N+1]; clamps to [0, 77]. Single CTA (N <= ~10^5).
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(1024) scan_lengths_kernel(const int* __restrict__ len, int N, int* __restrict__ cu,
                                                            int* __restrict__ total_rows, int* __restrict__ max_len = nullptr) {
  __shared__ int warp_tot[32];
  __shared__ int carry;
  __shared__ int vmax_s;
  if (threadIdx.x == 0) { carry = 0; vmax_s = 0; }
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int base = 0; base < N; base += 1024) {
    const int i = base + threadIdx.x;
    int v = (i < N) ? min(max(len[i], 0), 77) : 0;      // 0 = duplicate row, encoded with its first occurrence
    if (max_len) atomicMax(&vmax_s, v);
    int inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      int t = __shfl_up_sync(0xffffffffu, inc, o);
      if (lane >= o) inc += t;
    }
    if (lane == 31) warp_tot[warp] = inc;
    __syncthreads();
    if (warp == 0) {
      int w = warp_tot[lane];
      int winc = w;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        int t = __shfl_up_sync(0xffffffffu, winc, o);
        if (lane >= o) winc += t;
      }
      warp_tot[lane] = winc - w;   // exclusive
    }
    __syncthreads();
    const int excl = carry + warp_tot[warp] + inc - v;
    if (i < N) cu[i] = excl;
    __syncthreads();
    if (threadIdx.x == 1023) carry = excl + v;
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    cu[N] = carry;
    *total_rows = carry;
    if (max_len) *max_len = vmax_s;
  }
}

// ---------------------------------------------------------------------------------------------
// shared-prefix analysis. Row i may name a base row base[i] of the same batch (the unedited caption of its
// sample): hidden states of the positions where both token rows agree are identical under the causal mask, so only
// positions [p, t) of row i are computed and its attention reads the base's keys/values for [0, p).
// own_len[i] = t - p with p = min(common prefix, t - 1) (the pooled EOS row is always computed). One warp per row.
// ---------------------------------------------------------------------------------------------
// dup_of[i] >= 0 (from dedup_kernel): row i has the same tokens as an earlier row and owns NO rows at all.
// need != nullptr: need[b] = max over the rows that name b as their base of the prefix length they read from it (zeroed by
// the caller); trim_providers_kernel then cuts the base rows down to that many positions.
__global__ void __launch_bounds__(256) prefix_kernel(const int* __restrict__ tok, const int* __restrict__ len,
                                                     const int* __restrict__ base, const int* __restrict__ dup_of, int N,
                                                     int* __restrict__ pfx, int* __restrict__ own_len, int* __restrict__ need = nullptr) {
  const int i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (i >= N) return;
  const int t = min(max(len[i], 1), 77);
  if (dup_of && dup_of[i] >= 0) {
    if (lane == 0) { pfx[i] = t; own_len[i] = 0; }
    return;
  }
  int p = 0;
  const int b = base ? base[i] : -1;
  if (b >= 0 && b < N && b != i) {
    const int tb = min(max(len[b], 1), 77);
    const int lim = min(t, tb);
    p = lim;
    for (int c = 0; c < 96; c += 32) {
      const int k = c + lane;
      const bool diff = (k < lim) && (tok[i * 77 + k] != tok[b * 77 + k]);
      const unsigned m = __ballot_sync(0xffffffffu, diff);
      if (m) { p = c + __ffs(m) - 1; break; }
    }
    p = min(p, t - 1);
    if (need && lane == 0 && p > 0) atomicMax(need + b, p);
  }
  if (lane == 0) { pfx[i] = p; own_len[i] = t - p; }
}

// Rows [first, N) with base == -1 are PROVIDERS when the caller does not read their features (the unedited captions of an
// attack phase, which exist only so that the candidates can share their prefix): only the positions some candidate
// actually reads are kept (at least one, so that the row still has a pooled position). With the TextFARE objective the
// winning edit position of phase 1 sits in the first words, so in phase 2 a caption shrinks from ~32 rows to ~3.
__global__ void trim_providers_kernel(const int* __restrict__ base, const int* __restrict__ need, int first, int N,
                                      int* __restrict__ own_len) {
  const int i = first + blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N || (base && base[i] >= 0)) return;
  own_len[i] = max(1, min(own_len[i], need[i]));
}

// Duplicate candidates inside a sample (e.g. 'a' and 'A' written at the same position: the tokenizer lower-cases, so
// ~14 % of the phase-2 rows repeat an earlier row) are encoded once: dup_of[i] = first earlier row of the same group of
// `group` consecutive rows with identical length and tokens, else -1. One warp per row; rows >= n_rows are never grouped.
__global__ void __launch_bounds__(256) dedup_kernel(const int* __restrict__ tok, const int* __restrict__ len, int n_rows,
                                                    int group, int N, int* __restrict__ dup_of) {
  const int i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (i >= N) return;
  int found = -1;
  if (i < n_rows) {
    const int t = len[i];
    const int a0 = tok[i * 77 + lane], a1 = tok[i * 77 + 32 + lane], a2 = lane < 13 ? tok[i * 77 + 64 + lane] : 0;
    for (int j = (i / group) * group; j < i; ++j) {
      if (len[j] != t) continue;                                          // warp-uniform
      const bool same = a0 == tok[j * 77 + lane] && a1 == tok[j * 77 + 32 + lane] && (lane >= 13 || a2 == tok[j * 77 + 64 + lane]);
      if (__all_sync(0xffffffffu, same)) { found = j; break; }
    }
  }
  if (lane == 0) dup_of[i] = found;
}

// meta[i] = {own_row, t, p, base_row}; eos_row[i] = last own row (of the first occurrence for a duplicate);
// first_of[i] = the sequence whose rows stand for sequence i (itself unless it is a duplicate)
__global__ void meta_kernel(const int* __restrict__ cu, const int* __restrict__ pfx, const int* __restrict__ base,
                            const int* __restrict__ dup_of, int N, int4* __restrict__ meta, int* __restrict__ eos_row,
                            int* __restrict__ first_of = nullptr) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  const int own = cu[i], n_own = cu[i + 1] - own, p = pfx[i];
  const int b = (base && p > 0 && base[i] >= 0) ? base[i] : i;
  meta[i] = make_int4(own, p + n_own, p, cu[b]);
  const int d = (dup_of && dup_of[i] >= 0) ? dup_of[i] : i;
  eos_row[i] = cu[d + 1] - 1;
  if (first_of) first_of[i] = d;
}

// ---------------------------------------------------------------------------------------------
// x[row,:] = token_embedding[id] + positional_embedding[pos]      (model.py:272-274), fp32
// one warp per packed row; grid = sequences
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) embed_kernel(const int* __restrict__ tok, const int4* __restrict__ meta, int N, int W,
                                                    const float* __restrict__ tok_emb, const float* __restrict__ pos_emb,
                                                    float* __restrict__ x) {
  const int seq = blockIdx.x;
  if (seq >= N) return;
  const int4 mt = meta[seq];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarp = blockDim.x >> 5;
  for (int pos = mt.z + warp; pos < mt.y; pos += nwarp) {
    const int id = tok[seq * 77 + pos];
    const float4* e = reinterpret_cast<const float4*>(tok_emb + static_cast<size_t>(id) * W);
    const float4* pe = reinterpret_cast<const float4*>(pos_emb + static_cast<size_t>(pos) * W);
    float4* o = reinterpret_cast<float4*>(x + static_cast<size_t>(mt.x + pos - mt.z) * W);
    for (int c = lane; c < W / 4; c += 32) {
      float4 a = __ldg(e + c), b = __ldg(pe + c);
      o[c] = make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w);
    }
  }
}

// ---------------------------------------------------------------------------------------------
// LayerNorm over fp32 rows -> bf16 (F.layer_norm, transformer.py:24-30), two-pass in registers.
// W = 128 * V4 floats... one warp per row, lane owns W/32 contiguous-by-4 elements. Rows from a device count.
// gather != nullptr: output row r reads input row gather[r] (EOS pooling, transformer.py:661).
// delta != nullptr: the row normalised is x[row] + delta[row] (bf16): the attention branch's out-proj result, which
// leaf_encode keeps apart from the fp32 residual stream until fc2's epilogue folds both in (see leaf_encode).
// ---------------------------------------------------------------------------------------------
template <int VPL /* float4 per lane */>
__global__ void __launch_bounds__(256) layernorm_bf16_kernel(const float* __restrict__ x, const int* __restrict__ rows_dev,
                                                            int rows_max, const int* __restrict__ gather, int W,
                                                            const float* __restrict__ gamma, const float* __restrict__ beta,
                                                            float eps, __nv_bfloat16* __restrict__ y,
                                                            const __nv_bfloat16* __restrict__ delta = nullptr,
                                                            __nv_bfloat16* __restrict__ y_lo = nullptr) {
  pdl_wait();
  pdl_trigger();     // the GEMM that follows sets itself up (barriers, TMEM, descriptors) while this grid runs
  const int rows = rows_dev ? min(*rows_dev, rows_max) : rows_max;
  const int lane = threadIdx.x & 31;
  const int warps_total = (gridDim.x * blockDim.x) >> 5;
  for (int r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; r < rows; r += warps_total) {
    const int src = gather ? gather[r] : r;
    const float4* in = reinterpret_cast<const float4*>(x + static_cast<size_t>(src) * W);
    float4 v[VPL];
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < VPL; ++i) v[i] = in[lane + 32 * i];
    if (delta) {
      const uint2* dp = reinterpret_cast<const uint2*>(delta + static_cast<size_t>(src) * W);
#pragma unroll
      for (int i = 0; i < VPL; ++i) {
        const uint2 d = dp[lane + 32 * i];
        const float2 d0 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&d.x));
        const float2 d1 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&d.y));
        v[i].x += d0.x; v[i].y += d0.y; v[i].z += d1.x; v[i].w += d1.y;
      }
    }
#pragma unroll
    for (int i = 0; i < VPL; ++i) s += (v[i].x + v[i].y) + (v[i].z + v[i].w);
    const float mean = warp_sum(s) / static_cast<float>(W);
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < VPL; ++i) {
      const float a = v[i].x - mean, b = v[i].y - mean, c = v[i].z - mean, d = v[i].w - mean;
      q += (a * a + b * b) + (c * c + d * d);
    }
    const float rstd = rsqrtf(warp_sum(q) / static_cast<float>(W) + eps);
    uint2* out = reinterpret_cast<uint2*>(y + static_cast<size_t>(r) * W);
#pragma unroll
    for (int i = 0; i < VPL; ++i) {
      const float4 g = __ldg(reinterpret_cast<const float4*>(gamma) + lane + 32 * i);
      const float4 b = __ldg(reinterpret_cast<const float4*>(beta) + lane + 32 * i);
      __nv_bfloat162 lo = __floats2bfloat162_rn((v[i].x - mean) * rstd * g.x + b.x, (v[i].y - mean) * rstd * g.y + b.y);
      __nv_bfloat162 hi = __floats2bfloat162_rn((v[i].z - mean) * rstd * g.z + b.z, (v[i].w - mean) * rstd * g.w + b.w);
      uint2 pk;
      pk.x = *reinterpret_cast<uint32_t*>(&lo);
      pk.y = *reinterpret_cast<uint32_t*>(&hi);
      out[lane + 32 * i] = pk;
      if (y_lo) {                                // what the bf16 rounding dropped, as a second bf16 operand (final projection)
        const float2 l = __bfloat1622float2(lo), h = __bfloat1622float2(hi);
        __nv_bfloat162 lo2 = __floats2bfloat162_rn((v[i].x - mean) * rstd * g.x + b.x - l.x, (v[i].y - mean) * rstd * g.y + b.y - l.y);
        __nv_bfloat162 hi2 = __floats2bfloat162_rn((v[i].z - mean) * rstd * g.z + b.z - h.x, (v[i].w - mean) * rstd * g.w + b.w - h.y);
        uint2 pk2;
        pk2.x = *reinterpret_cast<uint32_t*>(&lo2);
        pk2.y = *reinterpret_cast<uint32_t*>(&hi2);
        reinterpret_cast<uint2*>(y_lo + static_cast<size_t>(r) * W)[lane + 32 * i] = pk2;
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------
// causal attention over packed rows, head_dim 64 (nn.MultiheadAttention with the additive -inf mask,
// transformer.py:225,250-252,758-764; scale 1/sqrt(64)).
//
// One warp per (sequence, head); everything stays in registers: mma.sync.m16n8k16 (bf16, fp32 accumulate) for
// Q.K^T and P.V, fp32 softmax (exp2 with the scale folded in). A sequence has at most 77 positions, so the whole score
// row of a 16-query tile fits in registers (<= 5 key tiles): plain two-pass softmax, no running maximum, no rescaling.
// Operand fragments are read straight from global memory with sm_100's 256-BIT loads (LDG.E.256): a lane reads 32
// contiguous bytes, a quad one whole 128-byte head row, so a warp-wide load touches 8 full lines. With 128-bit loads
// (8 half lines per instruction) the L1 tag stage was the busiest unit (ncu r19: L1/TEX 65 %, 56 % of the stall cycles
// on its scoreboard); halving the requests per byte bought 15 % (tools/ab_attention.py, profiles/r34_attention_ab.log).
// Lane (g, c) owns d = 16c .. 16c+15 of a head row; register i holds d = 16c + 2i, +1. The contraction index of Q.K^T is
// permuted identically for Q and K (k-step j uses registers 2j, 2j+1), and the movmatrix-transposed V registers leave a
// lane with 16 contiguous output columns (one 32-byte store per row).
// The key tiles and then the value tiles form ONE stream of 2*NKT fragment sets that runs DEPTH sets ahead of the MMAs
// through a register ring, so the first value tiles are in flight during the softmax (+6 % over loading at the point of
// use; more registers per thread for occupancy, or fewer with spills, both measured slower).
// tcgen05's 128-row tiles do not fit 2..77-row problems (1.2 % of the tower's FLOPs).
//
// meta[seq] = {own_row, t, p, base_row}: the sequence has t positions; positions [p, t) are its own packed rows
// starting at own_row (they are the queries); keys/values of positions [0, p) are read from the rows of another
// sequence starting at base_row (shared prefix under the causal mask), p = 0 when nothing is shared.
// qkv: bf16 [rows, 3W] (q | k | v), out: bf16 [rows, W].
// ---------------------------------------------------------------------------------------------
constexpr int ATT_WARPS = 4;

__device__ __forceinline__ void mma_bf16_16816(float* c, const uint32_t* a, uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ uint32_t movmatrix_trans(uint32_t x) {
  uint32_t y;
  asm volatile("movmatrix.sync.aligned.m8n8.trans.b16 %0, %1;" : "=r"(y) : "r"(x));
  return y;
}
__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 t = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&t);
}
__device__ __forceinline__ float att_ex2(float x) {            // ex2.approx(-inf) = +0: masked keys drop out exactly
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

struct U8 { uint32_t r[8]; };
__device__ __forceinline__ U8 ldg256(const void* p) {
  U8 v;
  asm volatile("ld.global.nc.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(v.r[0]), "=r"(v.r[1]), "=r"(v.r[2]), "=r"(v.r[3]), "=r"(v.r[4]), "=r"(v.r[5]), "=r"(v.r[6]), "=r"(v.r[7])
               : "l"(p));
  return v;
}
__device__ __forceinline__ void stg256(void* p, const U8& v) {
  asm volatile("st.global.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p), "r"(v.r[0]), "r"(v.r[1]), "r"(v.r[2]), "r"(v.r[3]),
               "r"(v.r[4]), "r"(v.r[5]), "r"(v.r[6]), "r"(v.r[7])
               : "memory");
}

template <int NKT, int DEPTH>
__device__ __forceinline__ void attention_tile(const __nv_bfloat16* __restrict__ kbase, const __nv_bfloat16* __restrict__ vbase,
                                                  size_t ld, const U8& qa, const U8& qb, int pos0, int pos1, int t, int p,
                                                  int own_row, int base_row, int g, int c, float (&o)[8][4], float& inv0, float& inv1) {
  const float sl2 = 0.125f * 1.4426950408889634f;          // 1/sqrt(64) * log2(e)
  constexpr int NS = 2 * NKT;                              // stream: K tiles 0..NKT-1, then V tiles 0..NKT-1
  U8 ring[DEPTH][2];                                       // [slot][key half: keys 16kt+g, 16kt+8+g]
  auto issue = [&](int si) {
    const int kt = si < NKT ? si : si - NKT;
    const __nv_bfloat16* src = si < NKT ? kbase : vbase;
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int j = min(kt * 16 + h * 8 + g, t - 1);
      ring[si % DEPTH][h] = ldg256(src + static_cast<size_t>(j < p ? base_row + j : own_row + (j - p)) * ld);
    }
  };
#pragma unroll
  for (int si = 0; si < DEPTH && si < NS; ++si) issue(si);
  // ---- S = Q.K^T ----
  float s[NKT][2][4];
#pragma unroll
  for (int kt = 0; kt < NKT; ++kt) {
#pragma unroll
    for (int nt = 0; nt < 2; ++nt) {
      s[kt][nt][0] = s[kt][nt][1] = s[kt][nt][2] = s[kt][nt][3] = 0.f;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const uint32_t a[4] = {qa.r[2 * j], qb.r[2 * j], qa.r[2 * j + 1], qb.r[2 * j + 1]};
        mma_bf16_16816(s[kt][nt], a, ring[kt % DEPTH][nt].r[2 * j], ring[kt % DEPTH][nt].r[2 * j + 1]);
      }
    }
    if (kt + DEPTH < NS) issue(kt + DEPTH);
  }
  // ---- causal mask and row maxima (rows g and g+8 live on the 4 lanes of a quad) ----
  float mx0 = -INFINITY, mx1 = -INFINITY;
#pragma unroll
  for (int kt = 0; kt < NKT; ++kt)
#pragma unroll
    for (int nt = 0; nt < 2; ++nt)
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const int j = kt * 16 + nt * 8 + 2 * c + e;
        if (j > pos0) s[kt][nt][e] = -INFINITY;
        if (j > pos1) s[kt][nt][2 + e] = -INFINITY;
        mx0 = fmaxf(mx0, s[kt][nt][e]);
        mx1 = fmaxf(mx1, s[kt][nt][2 + e]);
      }
  mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 1));
  mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 2));
  mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 1));
  mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 2));
  const float nm0 = -mx0 * sl2, nm1 = -mx1 * sl2;          // finite: key 0 is visible to every query
  // ---- P = exp2((S - max) * scale), row sums, bf16 A fragments ----
  float l0 = 0.f, l1 = 0.f;
  uint32_t pf[NKT][4];
#pragma unroll
  for (int kt = 0; kt < NKT; ++kt)
#pragma unroll
    for (int nt = 0; nt < 2; ++nt) {
      const float p00 = att_ex2(fmaf(s[kt][nt][0], sl2, nm0)), p01 = att_ex2(fmaf(s[kt][nt][1], sl2, nm0));
      const float p10 = att_ex2(fmaf(s[kt][nt][2], sl2, nm1)), p11 = att_ex2(fmaf(s[kt][nt][3], sl2, nm1));
      l0 += p00 + p01;
      l1 += p10 + p11;
      pf[kt][2 * nt] = pack_bf16x2(p00, p01);
      pf[kt][2 * nt + 1] = pack_bf16x2(p10, p11);
    }
  l0 += __shfl_xor_sync(0xffffffffu, l0, 1);
  l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
  l1 += __shfl_xor_sync(0xffffffffu, l1, 1);
  l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
  inv0 = 1.f / l0;
  inv1 = 1.f / l1;
  // ---- O = P.V : V fragments transposed in registers; MMA i yields d = 16c + 2i, +1 ----
#pragma unroll
  for (int i = 0; i < 8; ++i) o[i][0] = o[i][1] = o[i][2] = o[i][3] = 0.f;
#pragma unroll
  for (int kt = 0; kt < NKT; ++kt) {
#pragma unroll
    for (int i = 0; i < 8; ++i)
      mma_bf16_16816(o[i], pf[kt], movmatrix_trans(ring[(NKT + kt) % DEPTH][0].r[i]), movmatrix_trans(ring[(NKT + kt) % DEPTH][1].r[i]));
    if (NKT + kt + DEPTH < NS) issue(NKT + kt + DEPTH);
  }
}

// last_only (final layer): only the pooled EOS position feeds the output (transformer.py:661), so only the query tile
// that holds it is computed and its row is written to out[seq] (one compact row per sequence).
constexpr int ATT_DEPTH = 3;
__global__ void __launch_bounds__(ATT_WARPS * 32, 4) attention_kernel(const __nv_bfloat16* __restrict__ qkv,
                                                                       const int4* __restrict__ meta, int n_seq, int heads,
                                                                       int W, __nv_bfloat16* __restrict__ out,
                                                                       int last_only = 0) {
  pdl_wait();
  pdl_trigger();     // the GEMM that follows sets itself up (barriers, TMEM, descriptors) while this grid runs
  const int pair = blockIdx.x * ATT_WARPS + (threadIdx.x >> 5);
  if (pair >= n_seq * heads) return;
  const int seq = pair / heads, head = pair - seq * heads;
  const int lane = threadIdx.x & 31, g = lane >> 2, c = lane & 3;
  const int4 mt = __ldg(meta + seq);
  const int own_row = mt.x, t = mt.y, p = mt.z, base_row = mt.w;
  const int nq = t - p;
  if (nq <= 0) return;                                       // duplicate of an earlier sequence: owns no rows
  const size_t ld = static_cast<size_t>(3) * W;
  const __nv_bfloat16* qbase = qkv + head * 64 + c * 16;
  const __nv_bfloat16* kbase = qbase + W;
  const __nv_bfloat16* vbase = qbase + 2 * W;
  for (int q0 = last_only ? ((nq - 1) & ~15) : 0; q0 < nq; q0 += 16) {
    const int qi0 = min(q0 + g, nq - 1), qi1 = min(q0 + g + 8, nq - 1);
    const U8 qa = ldg256(qbase + static_cast<size_t>(own_row + qi0) * ld);
    const U8 qb = ldg256(qbase + static_cast<size_t>(own_row + qi1) * ld);
    const int pos0 = p + qi0, pos1 = p + qi1;               // absolute positions of the two query rows
    const int kmax = min(t - 1, p + q0 + 15);               // last key any query of the tile may see
    float o[8][4];
    float inv0, inv1;
#define ATT_ARGS kbase, vbase, ld, qa, qb, pos0, pos1, t, p, own_row, base_row, g, c, o, inv0, inv1
    switch (kmax >> 4) {                                     // warp-uniform
      case 0: attention_tile<1, ATT_DEPTH>(ATT_ARGS); break;
      case 1: attention_tile<2, ATT_DEPTH>(ATT_ARGS); break;
      case 2: attention_tile<3, ATT_DEPTH>(ATT_ARGS); break;
      case 3: attention_tile<4, ATT_DEPTH>(ATT_ARGS); break;
      default: attention_tile<5, ATT_DEPTH>(ATT_ARGS); break;
    }
#undef ATT_ARGS
    U8 w0, w1;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      w0.r[i] = pack_bf16x2(o[i][0] * inv0, o[i][1] * inv0);
      w1.r[i] = pack_bf16x2(o[i][2] * inv1, o[i][3] * inv1);
    }
    __nv_bfloat16* ob = out + head * 64 + c * 16;
    if (last_only) {
      if (q0 + g == nq - 1) stg256(ob + static_cast<size_t>(seq) * W, w0);
      if (q0 + g + 8 == nq - 1) stg256(ob + static_cast<size_t>(seq) * W, w1);
    } else {
      if (q0 + g < nq) stg256(ob + static_cast<size_t>(own_row + q0 + g) * W, w0);
      if (q0 + g + 8 < nq) stg256(ob + static_cast<size_t>(own_row + q0 + g + 8) * W, w1);
    }
  }
}

// dst[r,:] = src[rows[r],:] (fp32): the residual rows of the pooled EOS positions, compacted for the final layer's MLP.
__global__ void __launch_bounds__(256) gather_rows_f32_kernel(const float* __restrict__ src, const int* __restrict__ rows, int N,
                                                             int W, float* __restrict__ dst) {
  const int r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (r >= N) return;
  const float4* in = reinterpret_cast<const float4*>(src + static_cast<size_t>(rows[r]) * W);
  float4* o = reinterpret_cast<float4*>(dst + static_cast<size_t>(r) * W);
  for (int c = lane; c < W / 4; c += 32) o[c] = in[c];
}

// F.normalize(x, dim=-1) in place (model.py:284): x / max(||x||, 1e-12). One warp per row.
__global__ void __launch_bounds__(256) l2_normalize_kernel(float* __restrict__ f, int N, int E) {
  const int r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (r >= N) return;
  float* row = f + static_cast<size_t>(r) * E;
  float s = 0.f;
  for (int c = lane; c < E; c += 32) s += row[c] * row[c];
  const float inv = 1.f / fmaxf(sqrtf(warp_sum(s)), 1e-12f);
  for (int c = lane; c < E; c += 32) row[c] *= inv;
}

// ---------------------------------------------------------------------------------------------
// K3: score[b,j] and per-sample argmax (utils_attacks.py:332-348, :370-386, :393).
// One CTA per sample; each warp reduces whole candidates (float4 loads), then a CTA-level argmax with the
// FIRST maximal index winning, as torch.argmax does. objective: 0 l2, 1 negl2, 2 sim, 3 dissim.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) score_argmax_kernel(const float* __restrict__ feat, const float* __restrict__ anchor,
                                                          int n, int E, int objective, float* __restrict__ loss_out,
                                                          int* __restrict__ best_out, float* __restrict__ best_feat_out) {
  extern __shared__ float sc[];     // [n] scores
  __shared__ float red_v[8];
  __shared__ int red_i[8];
  __shared__ int best_s;
  const int b = blockIdx.x;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarp = blockDim.x >> 5;
  const float4* a4 = reinterpret_cast<const float4*>(anchor + static_cast<size_t>(b) * E);
  for (int j = warp; j < n; j += nwarp) {
    const float4* f4 = reinterpret_cast<const float4*>(feat + (static_cast<size_t>(b) * n + j) * E);
    float s = 0.f;
    for (int c = lane; c < E / 4; c += 32) {
      const float4 f = f4[c], a = __ldg(a4 + c);
      if (objective <= 1) {
        const float dx = f.x - a.x, dy = f.y - a.y, dz = f.z - a.z, dw = f.w - a.w;
        s += (dx * dx + dy * dy) + (dz * dz + dw * dw);
      } else {
        s += (f.x * a.x + f.y * a.y) + (f.z * a.z + f.w * a.w);
      }
    }
    s = warp_sum(s);
    if (objective == 1 || objective == 3) s = -s;
    if (lane == 0) {
      sc[j] = s;
      if (loss_out) loss_out[static_cast<size_t>(b) * n + j] = s;
    }
  }
  __syncthreads();
  // argmax, first index on ties; NaN never wins over a number (torch treats NaN as max - not reachable here)
  float bv = -INFINITY;
  int bi = 0x7fffffff;
  for (int j = threadIdx.x; j < n; j += blockDim.x) {
    const float v = sc[j];
    if (v > bv || (v == bv && j < bi)) { bv = v; bi = j; }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
    const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
    if (ov > bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
  }
  if (lane == 0) { red_v[warp] = bv; red_i[warp] = bi; }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < nwarp; ++w)
      if (red_v[w] > bv || (red_v[w] == bv && red_i[w] < bi)) { bv = red_v[w]; bi = red_i[w]; }
    if (bi == 0x7fffffff) bi = 0;
    best_s = bi;
    best_out[b] = bi;
  }
  __syncthreads();
  if (best_feat_out) {
    const float* src = feat + (static_cast<size_t>(b) * n + best_s) * E;
    float* dst = best_feat_out + static_cast<size_t>(b) * E;
    for (int c = threadIdx.x; c < E; c += blockDim.x) dst[c] = src[c];
  }
}

// ---------------------------------------------------------------------------------------------
// Top-k of a score vector (Charmer's position selection, utils_attacks.py:519, and the argmax over the whole candidate
// list, :447/:575, with k = 1). v[i] = a[i], or (a[i] + b[i]) / 2 when a second tower scores the same candidates
// (:498-513). Order: value descending, ties by ascending index (torch.argmax's first-index rule for k = 1; torch.topk
// leaves the order of ties unspecified). One CTA; the working copy of the scores lives in shared memory.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(1024) topk_kernel(const float* __restrict__ a, const float* __restrict__ b, int m, int k,
                                                    int* __restrict__ idx_out, float* __restrict__ val_out) {
  extern __shared__ float tk[];     // [m]
  __shared__ float red_v[32];
  __shared__ int red_i[32];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarp = blockDim.x >> 5;
  for (int i = threadIdx.x; i < m; i += blockDim.x) tk[i] = b ? (a[i] + b[i]) / 2.f : a[i];
  __syncthreads();
  for (int r = 0; r < k; ++r) {
    float bv = -INFINITY;
    int bi = 0x7fffffff;
    for (int i = threadIdx.x; i < m; i += blockDim.x) {
      const float v = tk[i];
      if (v > bv || (v == bv && i < bi)) { bv = v; bi = i; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
      const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
      if (ov > bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
    }
    if (lane == 0) { red_v[warp] = bv; red_i[warp] = bi; }
    __syncthreads();
    if (warp == 0) {
      bv = lane < nwarp ? red_v[lane] : -INFINITY;
      bi = lane < nwarp ? red_i[lane] : 0x7fffffff;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
        const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
        if (ov > bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
      }
      if (lane == 0) {
        if (bi == 0x7fffffff) bi = 0;             // every remaining score is -inf
        idx_out[r] = bi;
        if (val_out) val_out[r] = bv;
        tk[bi] = -INFINITY;                       // taken (a genuine -inf score can be returned twice; not reachable here)
      }
    }
    __syncthreads();
  }
}

// fp32 -> bf16 cast (weight refresh), optional transpose for text_projection [W,E] -> [E,W]
// residual = 1: dst = bf16(src - float(bf16(src))), the part of src its bf16 copy dropped (second operand of the final projection)
__device__ __forceinline__ float bf16_residual(float v) { return v - __bfloat162float(__float2bfloat16_rn(v)); }
__global__ void cast_bf16_kernel(const float* __restrict__ src, __nv_bfloat16* __restrict__ dst, size_t n, int residual = 0) {
  size_t i = (static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x) * 4;
  const size_t stride = static_cast<size_t>(gridDim.x) * blockDim.x * 4;
  for (; i + 3 < n; i += stride) {
    float4 v = *reinterpret_cast<const float4*>(src + i);
    if (residual) { v.x = bf16_residual(v.x); v.y = bf16_residual(v.y); v.z = bf16_residual(v.z); v.w = bf16_residual(v.w); }
    __nv_bfloat162 lo = __floats2bfloat162_rn(v.x, v.y), hi = __floats2bfloat162_rn(v.z, v.w);
    uint2 pk;
    pk.x = *reinterpret_cast<uint32_t*>(&lo);
    pk.y = *reinterpret_cast<uint32_t*>(&hi);
    *reinterpret_cast<uint2*>(dst + i) = pk;
  }
}
__global__ void cast_bf16_transpose_kernel(const float* __restrict__ src /*[R,C]*/, __nv_bfloat16* __restrict__ dst /*[C,R]*/,
                                           int R, int C, int residual = 0) {
  __shared__ float tile[32][33];
  const int c0 = blockIdx.x * 32, r0 = blockIdx.y * 32;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int r = r0 + i, c = c0 + threadIdx.x;
    const float v = (r < R && c < C) ? src[static_cast<size_t>(r) * C + c] : 0.f;
    tile[i][threadIdx.x] = residual ? bf16_residual(v) : v;
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int c = c0 + i, r = r0 + threadIdx.x;
    if (c < C && r < R) dst[static_cast<size_t>(c) * R + r] = __float2bfloat16_rn(tile[threadIdx.x][i]);
  }
}
}  // namespace leaf
