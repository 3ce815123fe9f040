// vit_attn_tc.cuh -- tensor-core attention core of the CLIP ViT (head dim 64, T <= 256), forward and backward.
//
// softmax(Q K^T / 8) V per (sample, head); one CTA per (sample, head). The sequence is tiny (T = 50 for
// ViT-B/32, 197 for ViT-B/16), so K and V of a head stay resident in shared memory and the whole problem is a
// handful of 16x8x16 bf16 MMAs per warp (mma.sync, fp32 accumulate); softmax statistics live in registers.
//   forward : S = Q K^T -> softmax (exp2, fp32) -> O = P V                       (P never leaves registers)
//   backward: 3 register-light passes per query block recompute S / P / dP = dO V^T tile by tile
//             (row max+sum, then delta = rowsum(P o dP), then dS = P o (dP - delta)): dQ = dS K from registers;
//             P and dS are parked in shared memory (bf16) and re-read TRANSPOSED (ldmatrix.trans) so that each warp
//             owns key tiles and reduces dV = P^T dO, dK = dS^T Q over all query rows without atomics.
// Shared-memory tiles are 128-byte rows with the 16-byte chunk index XOR-swizzled by (row & 7): ldmatrix is
// bank-conflict free. qkv is bf16 [S*T, 3*D] (q | k | v), out / dout bf16 [S*T, D], dqkv bf16 [S*T, 3*D].
#pragma once
#include "tc_gemm.cuh"
#include <stdlib.h>

namespace aph {

__device__ __forceinline__ void ldsm4(uint32_t (&r)[4], uint32_t saddr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0, %1, %2, %3}, [%4];" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(saddr));
}
__device__ __forceinline__ void ldsm4t(uint32_t (&r)[4], uint32_t saddr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0, %1, %2, %3}, [%4];" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(saddr));
}
__device__ __forceinline__ void mma16816(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3]) : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ uint32_t pack2(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}
// byte offset of 16-byte chunk `chunk` of row `row` in a tile with `pitch` bytes per row (pitch % 128 == 0)
__device__ __forceinline__ uint32_t swz(int row, int chunk, int pitch) {
  return (uint32_t)(row * pitch + ((((chunk & ~7) | ((chunk ^ row) & 7))) << 4));
}
__device__ __forceinline__ float quad_max(float v) { v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, 1)); return fmaxf(v, __shfl_xor_sync(0xffffffffu, v, 2)); }
__device__ __forceinline__ float quad_sum(float v) { v += __shfl_xor_sync(0xffffffffu, v, 1); return v + __shfl_xor_sync(0xffffffffu, v, 2); }

constexpr float kAttnScaleLog2 = 0.125f * 1.4426950408889634f;   // (1/sqrt(64)) * log2(e)

// copies `rows` rows of 64 bf16 (128 B) from global (row stride ld elements) into a swizzled tile; rows >= valid are zeroed
__device__ __forceinline__ void load_tile64(uint8_t* tile, const bf16* __restrict__ src, size_t ld, int rows, int valid, int nthreads) {
  for (int idx = threadIdx.x; idx < rows * 8; idx += nthreads) {
    const int r = idx >> 3, c = idx & 7;
    uint4 v = make_uint4(0u, 0u, 0u, 0u);
    if (r < valid) v = __ldg(reinterpret_cast<const uint4*>(src + (size_t)r * ld) + c);
    *reinterpret_cast<uint4*>(tile + swz(r, c, 128)) = v;
  }
}

// A fragments (16 rows x 64 k) of the rows r0.. of a 64-col tile
__device__ __forceinline__ void load_a_frags(uint32_t (&a)[4][4], uint32_t tile, int r0, int lane) {
#pragma unroll
  for (int ks = 0; ks < 4; ++ks) ldsm4(a[ks], tile + swz(r0 + (lane & 15), ks * 2 + (lane >> 4), 128));
}

// S tile for 16 keys (two n-tiles) = A(16 x 64) . Keys(16 x 64)^T
__device__ __forceinline__ void qk_tile(float (&c0)[4], float (&c1)[4], const uint32_t (&a)[4][4], uint32_t ktile, int key0, int lane) {
#pragma unroll
  for (int i = 0; i < 4; ++i) { c0[i] = 0.f; c1[i] = 0.f; }
#pragma unroll
  for (int ks = 0; ks < 4; ++ks) {
    uint32_t b[4];
    ldsm4(b, ktile + swz(key0 + (lane & 7) + ((lane >> 4) << 3), ks * 2 + ((lane >> 3) & 1), 128));
    mma16816(c0, a[ks], b[0], b[1]);
    mma16816(c1, a[ks], b[2], b[3]);
  }
}

// acc(16 x 64) += A(16 x 16, registers) . Rows(16 x 64) where the B operand rows are the k index (V, K, dO or Q tile rows)
__device__ __forceinline__ void av_step(float (&acc)[8][4], const uint32_t (&a)[4], uint32_t tile, int row0, int lane) {
#pragma unroll
  for (int dt2 = 0; dt2 < 4; ++dt2) {
    uint32_t b[4];
    ldsm4t(b, tile + swz(row0 + (lane & 7) + (((lane >> 3) & 1) << 3), dt2 * 2 + (lane >> 4), 128));
    mma16816(acc[2 * dt2], a, b[0], b[1]);
    mma16816(acc[2 * dt2 + 1], a, b[2], b[3]);
  }
}

// ---------------------------------------------------------------------------------------------
// CAUSAL (the CLIP text tower): query row i sees keys j <= i only; key tiles wholly above the warp's rows are skipped.
template <int NW, int NT2, bool CAUSAL = false>
__global__ void __launch_bounds__(NW * 32) k_attn_fwd_tc(const bf16* __restrict__ qkv, bf16* __restrict__ out, int T, int D, int heads) {
  pdl_trigger(); pdl_wait();
  extern __shared__ __align__(128) uint8_t sm[];
  constexpr int TK = NT2 * 16, QB = NW * 16;
  uint8_t* Ks = sm; uint8_t* Vs = Ks + TK * 128; uint8_t* Qs = Vs + TK * 128;
  const int s = blockIdx.x / heads, h = blockIdx.x - s * heads;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  const size_t ld = (size_t)3 * D;
  const bf16* base = qkv + (size_t)s * T * ld + h * 64;
  load_tile64(Ks, base + D, ld, TK, T, NW * 32);
  load_tile64(Vs, base + 2 * D, ld, TK, T, NW * 32);
  load_tile64(Qs, base, ld, QB, T, NW * 32);                 // first query block rides along with K / V
  const uint32_t ks_a = smem_u32(Ks), vs_a = smem_u32(Vs), qs_a = smem_u32(Qs);
  for (int q0 = 0; q0 < T; q0 += QB) {
    if (q0 > 0) {
      __syncthreads();
      load_tile64(Qs, base + (size_t)q0 * ld, ld, QB, T - q0, NW * 32);
    }
    __syncthreads();
    const int r0 = warp * 16;
    if (q0 + r0 >= T) continue;
    uint32_t qa[4][4];
    load_a_frags(qa, qs_a, r0, lane);
    float c[2 * NT2][4];
    float m0 = -INFINITY, m1 = -INFINITY;
#pragma unroll
    for (int n2 = 0; n2 < NT2; ++n2) {
      if (CAUSAL && n2 * 16 > q0 + r0 + 15) {          // every key of the tile lies above the diagonal of this warp's rows
#pragma unroll
        for (int u = 0; u < 2; ++u) c[2 * n2 + u][0] = c[2 * n2 + u][1] = c[2 * n2 + u][2] = c[2 * n2 + u][3] = -INFINITY;
        continue;
      }
      qk_tile(c[2 * n2], c[2 * n2 + 1], qa, ks_a, n2 * 16, lane);
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        const int col = n2 * 16 + u * 8 + 2 * t;
        float* cc = c[2 * n2 + u];
        if (CAUSAL) {      // rows q0 + r0 + g and + 8 see keys j <= i; key 0 always, so m0, m1 stay finite
          const int qi = q0 + r0 + g;
          if (col > qi) cc[0] = -INFINITY;
          if (col + 1 > qi) cc[1] = -INFINITY;
          if (col > qi + 8) cc[2] = -INFINITY;
          if (col + 1 > qi + 8) cc[3] = -INFINITY;
        }
        cc[0] = (col < T) ? cc[0] * kAttnScaleLog2 : -INFINITY; cc[1] = (col + 1 < T) ? cc[1] * kAttnScaleLog2 : -INFINITY;
        cc[2] = (col < T) ? cc[2] * kAttnScaleLog2 : -INFINITY; cc[3] = (col + 1 < T) ? cc[3] * kAttnScaleLog2 : -INFINITY;
        m0 = fmaxf(m0, fmaxf(cc[0], cc[1])); m1 = fmaxf(m1, fmaxf(cc[2], cc[3]));
      }
    }
    m0 = quad_max(m0); m1 = quad_max(m1);
    float l0 = 0.f, l1 = 0.f;
#pragma unroll
    for (int n = 0; n < 2 * NT2; ++n) {
      c[n][0] = exp2f(c[n][0] - m0); c[n][1] = exp2f(c[n][1] - m0); c[n][2] = exp2f(c[n][2] - m1); c[n][3] = exp2f(c[n][3] - m1);
      l0 += c[n][0] + c[n][1]; l1 += c[n][2] + c[n][3];
    }
    l0 = quad_sum(l0); l1 = quad_sum(l1);
    float o[8][4];
#pragma unroll
    for (int i = 0; i < 8; ++i) { o[i][0] = o[i][1] = o[i][2] = o[i][3] = 0.f; }
#pragma unroll
    for (int kk = 0; kk < NT2; ++kk) {
      if (CAUSAL && kk * 16 > q0 + r0 + 15) continue;   // P is exactly zero there
      uint32_t pa[4] = {pack2(c[2 * kk][0], c[2 * kk][1]), pack2(c[2 * kk][2], c[2 * kk][3]),
                        pack2(c[2 * kk + 1][0], c[2 * kk + 1][1]), pack2(c[2 * kk + 1][2], c[2 * kk + 1][3])};
      av_step(o, pa, vs_a, kk * 16, lane);
    }
    const float i0 = 1.f / l0, i1 = 1.f / l1;
    const int row0 = q0 + r0 + g, row1 = row0 + 8;
#pragma unroll
    for (int dt = 0; dt < 8; ++dt) {
      const int col = h * 64 + dt * 8 + 2 * t;
      if (row0 < T) *reinterpret_cast<__nv_bfloat162*>(out + ((size_t)s * T + row0) * D + col) = __floats2bfloat162_rn(o[dt][0] * i0, o[dt][1] * i0);
      if (row1 < T) *reinterpret_cast<__nv_bfloat162*>(out + ((size_t)s * T + row1) * D + col) = __floats2bfloat162_rn(o[dt][2] * i1, o[dt][3] * i1);
    }
  }
}

// ---------------------------------------------------------------------------------------------
template <int NW, int NT2>
__global__ void __launch_bounds__(NW * 32, NW == 4 ? 3 : 1) k_attn_bwd_tc(const bf16* __restrict__ qkv, const bf16* __restrict__ dout, bf16* __restrict__ dqkv,
                                                         int T, int D, int heads) {
  pdl_trigger(); pdl_wait();
  extern __shared__ __align__(128) uint8_t sm[];
  constexpr int TK = NT2 * 16, QB = NW * 16, KT = (NT2 + NW - 1) / NW, PB = ((TK + 63) / 64) * 128;
  uint8_t* Ks = sm; uint8_t* Vs = Ks + TK * 128; uint8_t* Qs = Vs + TK * 128; uint8_t* Gs = Qs + QB * 128;
  uint8_t* Ps = Gs + QB * 128; uint8_t* Ds = Ps + QB * PB;
  const int s = blockIdx.x / heads, h = blockIdx.x - s * heads;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  const size_t ld = (size_t)3 * D;
  const bf16* base = qkv + (size_t)s * T * ld + h * 64;
  const bf16* gbase = dout + (size_t)s * T * D + h * 64;
  bf16* obase = dqkv + (size_t)s * T * ld + h * 64;
  load_tile64(Ks, base + D, ld, TK, T, NW * 32);
  load_tile64(Vs, base + 2 * D, ld, TK, T, NW * 32);
  const uint32_t ks_a = smem_u32(Ks), vs_a = smem_u32(Vs), qs_a = smem_u32(Qs), gs_a = smem_u32(Gs), ps_a = smem_u32(Ps), ds_a = smem_u32(Ds);
  constexpr bool ONE_BLOCK = (TK <= QB);       // all queries in one block (ViT-B/32): key-side accumulators only live in phase B
  float dv[KT][8][4], dk[KT][8][4];
  if (!ONE_BLOCK) {
#pragma unroll
    for (int i = 0; i < KT; ++i)
#pragma unroll
      for (int j = 0; j < 8; ++j) { dv[i][j][0] = dv[i][j][1] = dv[i][j][2] = dv[i][j][3] = 0.f; dk[i][j][0] = dk[i][j][1] = dk[i][j][2] = dk[i][j][3] = 0.f; }
  }

  load_tile64(Qs, base, ld, QB, T, NW * 32);                 // first query block rides along with K / V
  load_tile64(Gs, gbase, (size_t)D, QB, T, NW * 32);
  for (int q0 = 0; q0 < T; q0 += QB) {
    if (q0 > 0) {
      __syncthreads();
      load_tile64(Qs, base + (size_t)q0 * ld, ld, QB, T - q0, NW * 32);
      load_tile64(Gs, gbase + (size_t)q0 * D, (size_t)D, QB, T - q0, NW * 32);
    }
    __syncthreads();
    // ---------------- phase A: query rows r0 .. r0+15 of this block
    const int r0 = warp * 16;
    {
      uint32_t qa[4][4], ga[4][4];
      load_a_frags(qa, qs_a, r0, lane);
      load_a_frags(ga, gs_a, r0, lane);
      float dq[8][4];
#pragma unroll
      for (int i = 0; i < 8; ++i) { dq[i][0] = dq[i][1] = dq[i][2] = dq[i][3] = 0.f; }
      if (NT2 <= 4) {
        // ---- register-resident variant: S and dP are computed once
        float c[2 * NT2][4], e[2 * NT2][4];
        float m0 = -INFINITY, m1 = -INFINITY;
#pragma unroll
        for (int n2 = 0; n2 < NT2; ++n2) {
          qk_tile(c[2 * n2], c[2 * n2 + 1], qa, ks_a, n2 * 16, lane);
          qk_tile(e[2 * n2], e[2 * n2 + 1], ga, vs_a, n2 * 16, lane);
#pragma unroll
          for (int u = 0; u < 2; ++u) {
            const int cl = n2 * 16 + u * 8 + 2 * t;
            float* cc = c[2 * n2 + u];
            cc[0] = (cl < T) ? cc[0] * kAttnScaleLog2 : -INFINITY; cc[1] = (cl + 1 < T) ? cc[1] * kAttnScaleLog2 : -INFINITY;
            cc[2] = (cl < T) ? cc[2] * kAttnScaleLog2 : -INFINITY; cc[3] = (cl + 1 < T) ? cc[3] * kAttnScaleLog2 : -INFINITY;
            m0 = fmaxf(m0, fmaxf(cc[0], cc[1])); m1 = fmaxf(m1, fmaxf(cc[2], cc[3]));
          }
        }
        m0 = quad_max(m0); m1 = quad_max(m1);
        float l0 = 0.f, l1 = 0.f, d0 = 0.f, d1 = 0.f;
#pragma unroll
        for (int n = 0; n < 2 * NT2; ++n) {
          c[n][0] = exp2f(c[n][0] - m0); c[n][1] = exp2f(c[n][1] - m0); c[n][2] = exp2f(c[n][2] - m1); c[n][3] = exp2f(c[n][3] - m1);
          l0 += c[n][0] + c[n][1]; l1 += c[n][2] + c[n][3];
          d0 += c[n][0] * e[n][0] + c[n][1] * e[n][1]; d1 += c[n][2] * e[n][2] + c[n][3] * e[n][3];
        }
        l0 = quad_sum(l0); l1 = quad_sum(l1); d0 = quad_sum(d0); d1 = quad_sum(d1);
        const float i0 = 1.f / l0, i1 = 1.f / l1;
        d0 *= i0; d1 *= i1;
#pragma unroll
        for (int n2 = 0; n2 < NT2; ++n2) {
          uint32_t pa[4], da[4];
#pragma unroll
          for (int u = 0; u < 2; ++u) {
            const float* cc = c[2 * n2 + u]; const float* ee = e[2 * n2 + u];
            const float p0 = cc[0] * i0, p1 = cc[1] * i0, p2 = cc[2] * i1, p3 = cc[3] * i1;
            pa[2 * u] = pack2(p0, p1); pa[2 * u + 1] = pack2(p2, p3);
            da[2 * u] = pack2(p0 * (ee[0] - d0) * 0.125f, p1 * (ee[1] - d0) * 0.125f);
            da[2 * u + 1] = pack2(p2 * (ee[2] - d1) * 0.125f, p3 * (ee[3] - d1) * 0.125f);
            const int chunk = n2 * 2 + u;
            *reinterpret_cast<uint32_t*>(Ps + swz(r0 + g, chunk, PB) + 4 * t) = pa[2 * u];
            *reinterpret_cast<uint32_t*>(Ps + swz(r0 + g + 8, chunk, PB) + 4 * t) = pa[2 * u + 1];
            *reinterpret_cast<uint32_t*>(Ds + swz(r0 + g, chunk, PB) + 4 * t) = da[2 * u];
            *reinterpret_cast<uint32_t*>(Ds + swz(r0 + g + 8, chunk, PB) + 4 * t) = da[2 * u + 1];
          }
          av_step(dq, da, ks_a, n2 * 16, lane);
        }
      } else {
      // pass 1: row max and sum
      float m0 = -INFINITY, m1 = -INFINITY;
#pragma unroll 1
      for (int n2 = 0; n2 < NT2; ++n2) {
        float c0[4], c1[4];
        qk_tile(c0, c1, qa, ks_a, n2 * 16, lane);
        const int col = n2 * 16 + 2 * t;
        if (col < T) { m0 = fmaxf(m0, c0[0]); m1 = fmaxf(m1, c0[2]); }
        if (col + 1 < T) { m0 = fmaxf(m0, c0[1]); m1 = fmaxf(m1, c0[3]); }
        if (col + 8 < T) { m0 = fmaxf(m0, c1[0]); m1 = fmaxf(m1, c1[2]); }
        if (col + 9 < T) { m0 = fmaxf(m0, c1[1]); m1 = fmaxf(m1, c1[3]); }
      }
      m0 = quad_max(m0) * kAttnScaleLog2; m1 = quad_max(m1) * kAttnScaleLog2;
      float l0 = 0.f, l1 = 0.f, d0 = 0.f, d1 = 0.f;
      // pass 2: l = sum exp, delta_unnorm = sum exp * dP     (dP = dO V^T)
#pragma unroll 1
      for (int n2 = 0; n2 < NT2; ++n2) {
        float c0[4], c1[4], e0[4], e1[4];
        qk_tile(c0, c1, qa, ks_a, n2 * 16, lane);
        qk_tile(e0, e1, ga, vs_a, n2 * 16, lane);
        const int col = n2 * 16 + 2 * t;
#pragma unroll
        for (int u = 0; u < 2; ++u) {
          float* cc = u ? c1 : c0; float* ee = u ? e1 : e0;
          const int cl = col + u * 8;
          const float p0 = (cl < T) ? exp2f(cc[0] * kAttnScaleLog2 - m0) : 0.f, p1 = (cl + 1 < T) ? exp2f(cc[1] * kAttnScaleLog2 - m0) : 0.f;
          const float p2 = (cl < T) ? exp2f(cc[2] * kAttnScaleLog2 - m1) : 0.f, p3 = (cl + 1 < T) ? exp2f(cc[3] * kAttnScaleLog2 - m1) : 0.f;
          l0 += p0 + p1; l1 += p2 + p3;
          d0 += p0 * ee[0] + p1 * ee[1]; d1 += p2 * ee[2] + p3 * ee[3];
        }
      }
      l0 = quad_sum(l0); l1 = quad_sum(l1); d0 = quad_sum(d0); d1 = quad_sum(d1);
      const float i0 = 1.f / l0, i1 = 1.f / l1;
      d0 *= i0; d1 *= i1;                        // delta_i = sum_j P_ij dP_ij
      // pass 3: P, dS (scaled by 1/8) -> smem (bf16) and dQ = dS K
#pragma unroll 1
      for (int n2 = 0; n2 < NT2; ++n2) {
        float c0[4], c1[4], e0[4], e1[4];
        qk_tile(c0, c1, qa, ks_a, n2 * 16, lane);
        qk_tile(e0, e1, ga, vs_a, n2 * 16, lane);
        const int col = n2 * 16 + 2 * t;
        uint32_t pa[4], da[4];
#pragma unroll
        for (int u = 0; u < 2; ++u) {
          float* cc = u ? c1 : c0; float* ee = u ? e1 : e0;
          const int cl = col + u * 8;
          const float p0 = (cl < T) ? exp2f(cc[0] * kAttnScaleLog2 - m0) * i0 : 0.f, p1 = (cl + 1 < T) ? exp2f(cc[1] * kAttnScaleLog2 - m0) * i0 : 0.f;
          const float p2 = (cl < T) ? exp2f(cc[2] * kAttnScaleLog2 - m1) * i1 : 0.f, p3 = (cl + 1 < T) ? exp2f(cc[3] * kAttnScaleLog2 - m1) * i1 : 0.f;
          pa[2 * u] = pack2(p0, p1); pa[2 * u + 1] = pack2(p2, p3);
          da[2 * u] = pack2(p0 * (ee[0] - d0) * 0.125f, p1 * (ee[1] - d0) * 0.125f);
          da[2 * u + 1] = pack2(p2 * (ee[2] - d1) * 0.125f, p3 * (ee[3] - d1) * 0.125f);
          const int chunk = n2 * 2 + u;
          *reinterpret_cast<uint32_t*>(Ps + swz(r0 + g, chunk, PB) + 4 * t) = pa[2 * u];
          *reinterpret_cast<uint32_t*>(Ps + swz(r0 + g + 8, chunk, PB) + 4 * t) = pa[2 * u + 1];
          *reinterpret_cast<uint32_t*>(Ds + swz(r0 + g, chunk, PB) + 4 * t) = da[2 * u];
          *reinterpret_cast<uint32_t*>(Ds + swz(r0 + g + 8, chunk, PB) + 4 * t) = da[2 * u + 1];
        }
        av_step(dq, da, ks_a, n2 * 16, lane);
      }
      }
      const int row0 = q0 + r0 + g, row1 = row0 + 8;
#pragma unroll
      for (int dt = 0; dt < 8; ++dt) {
        const int col = dt * 8 + 2 * t;
        if (row0 < T) *reinterpret_cast<__nv_bfloat162*>(obase + (size_t)row0 * ld + col) = __floats2bfloat162_rn(dq[dt][0], dq[dt][1]);
        if (row1 < T) *reinterpret_cast<__nv_bfloat162*>(obase + (size_t)row1 * ld + col) = __floats2bfloat162_rn(dq[dt][2], dq[dt][3]);
      }
    }
    __syncthreads();
    // ---------------- phase B: key tiles owned by this warp, reduced over the block's query rows
    if (ONE_BLOCK) {
#pragma unroll
      for (int i = 0; i < KT; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) { dv[i][j][0] = dv[i][j][1] = dv[i][j][2] = dv[i][j][3] = 0.f; dk[i][j][0] = dk[i][j][1] = dk[i][j][2] = dk[i][j][3] = 0.f; }
    }
#pragma unroll
    for (int i = 0; i < KT; ++i) {
      const int kt = warp + i * NW;
      if (kt < NT2) {
#pragma unroll
        for (int ks = 0; ks < QB / 16; ++ks) {
          uint32_t pa[4], da[4];
          const int srow = ks * 16 + (lane & 7) + ((lane >> 4) << 3), chunk = kt * 2 + ((lane >> 3) & 1);
          ldsm4t(pa, ps_a + swz(srow, chunk, PB));
          ldsm4t(da, ds_a + swz(srow, chunk, PB));
          av_step(dv[i], pa, gs_a, ks * 16, lane);
          av_step(dk[i], da, qs_a, ks * 16, lane);
        }
      }
    }
  }
#pragma unroll
  for (int i = 0; i < KT; ++i) {
    const int kt = warp + i * NW;
    if (kt < NT2) {
      const int key0 = kt * 16 + g, key1 = key0 + 8;
#pragma unroll
      for (int dt = 0; dt < 8; ++dt) {
        const int col = dt * 8 + 2 * t;
        if (key0 < T) {
          *reinterpret_cast<__nv_bfloat162*>(obase + (size_t)key0 * ld + D + col) = __floats2bfloat162_rn(dk[i][dt][0], dk[i][dt][1]);
          *reinterpret_cast<__nv_bfloat162*>(obase + (size_t)key0 * ld + 2 * D + col) = __floats2bfloat162_rn(dv[i][dt][0], dv[i][dt][1]);
        }
        if (key1 < T) {
          *reinterpret_cast<__nv_bfloat162*>(obase + (size_t)key1 * ld + D + col) = __floats2bfloat162_rn(dk[i][dt][2], dk[i][dt][3]);
          *reinterpret_cast<__nv_bfloat162*>(obase + (size_t)key1 * ld + 2 * D + col) = __floats2bfloat162_rn(dv[i][dt][2], dv[i][dt][3]);
        }
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------
// Pipelined variants for T <= 64 (ViT-B/32: T = 50): the per-(sample, head) problem is so small that a CTA is dominated by
// the global-load latency of its 24-32 KB of operands (ncu: long-scoreboard stalls, 17 % warps active). Here a CTA walks a
// strided list of (sample, head) items and prefetches the NEXT item's tiles into the other half of a double buffer while it
// computes the current one. The tiles are fetched by TMA (one thread, 3-4 cp.async.bulk.tensor.3d per item, completion on an
// mbarrier) from a [S][T][cols] view of the token matrix whose out-of-range token rows arrive zero-filled; the per-thread
// cp.async loop this replaced was 20 % of the backward kernel's instructions (profiles/r1l_ncu_full_summary.md).
template <int NT2>
__global__ void __launch_bounds__(128) k_attn_fwd_tc1(const __grid_constant__ CUtensorMap tm_kv, const __grid_constant__ CUtensorMap tm_q,
                                                      bf16* __restrict__ out, int T, int D, int heads, int items) {
  pdl_trigger(); pdl_wait();
  extern __shared__ __align__(1024) uint8_t sm_raw[];
  __shared__ __align__(8) uint64_t full[2];
  constexpr int TK = NT2 * 16, QB = 64, BUF = (2 * TK + QB) * 128;
  const uint32_t sm_a = (smem_u32(sm_raw) + 1023u) & ~1023u;     // 128B-swizzled TMA tiles want 1024-byte aligned bases
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  if (threadIdx.x == 0) { mbar_init(&full[0], 1); mbar_init(&full[1], 1); fence_barrier_init(); tma_prefetch_desc(&tm_kv); tma_prefetch_desc(&tm_q); }
  __syncthreads();
  // one thread asks TMA for the K, V, Q tiles of an item: rows >= T of the 3-D view come back as zeros
  auto issue = [&](int item, int b) {
    const int s = item / heads, h = item - s * heads;
    const uint32_t a = sm_a + b * BUF;
    mbar_expect_tx(&full[b], BUF);
    tma_load_3d(a, &tm_kv, &full[b], D + h * 64, 0, s);
    tma_load_3d(a + TK * 128, &tm_kv, &full[b], 2 * D + h * 64, 0, s);
    tma_load_3d(a + 2 * TK * 128, &tm_q, &full[b], h * 64, 0, s);
  };
  int item = blockIdx.x, b = 0;
  uint32_t phases = 0u;                                          // bit b = parity of the next fill of buffer b
  if (item < items && threadIdx.x == 0) issue(item, 0);
  for (; item < items; item += gridDim.x, b ^= 1) {
    const int nxt = item + gridDim.x;
    if (nxt < items && threadIdx.x == 0) issue(nxt, b ^ 1);      // buffer b^1 was released by the barrier that ended the previous item
    mbar_wait(&full[b], (phases >> b) & 1u); phases ^= 1u << b;
    const int s = item / heads, h = item - s * heads;
    const uint32_t ks_a = sm_a + b * BUF, vs_a = ks_a + TK * 128, qs_a = vs_a + TK * 128;
    const int r0 = warp * 16;
    if (r0 < T) {
      uint32_t qa[4][4];
      load_a_frags(qa, qs_a, r0, lane);
      float c[2 * NT2][4];
      float m0 = -INFINITY, m1 = -INFINITY;
#pragma unroll
      for (int n2 = 0; n2 < NT2; ++n2) {
        qk_tile(c[2 * n2], c[2 * n2 + 1], qa, ks_a, n2 * 16, lane);
#pragma unroll
        for (int u = 0; u < 2; ++u) {
          const int col = n2 * 16 + u * 8 + 2 * t;
          float* cc = c[2 * n2 + u];
          cc[0] = (col < T) ? cc[0] * kAttnScaleLog2 : -INFINITY; cc[1] = (col + 1 < T) ? cc[1] * kAttnScaleLog2 : -INFINITY;
          cc[2] = (col < T) ? cc[2] * kAttnScaleLog2 : -INFINITY; cc[3] = (col + 1 < T) ? cc[3] * kAttnScaleLog2 : -INFINITY;
          m0 = fmaxf(m0, fmaxf(cc[0], cc[1])); m1 = fmaxf(m1, fmaxf(cc[2], cc[3]));
        }
      }
      m0 = quad_max(m0); m1 = quad_max(m1);
      float l0 = 0.f, l1 = 0.f;
#pragma unroll
      for (int n = 0; n < 2 * NT2; ++n) {
        c[n][0] = exp2f(c[n][0] - m0); c[n][1] = exp2f(c[n][1] - m0); c[n][2] = exp2f(c[n][2] - m1); c[n][3] = exp2f(c[n][3] - m1);
        l0 += c[n][0] + c[n][1]; l1 += c[n][2] + c[n][3];
      }
      l0 = quad_sum(l0); l1 = quad_sum(l1);
      float o[8][4];
#pragma unroll
      for (int i = 0; i < 8; ++i) { o[i][0] = o[i][1] = o[i][2] = o[i][3] = 0.f; }
#pragma unroll
      for (int kk = 0; kk < NT2; ++kk) {
        uint32_t pa[4] = {pack2(c[2 * kk][0], c[2 * kk][1]), pack2(c[2 * kk][2], c[2 * kk][3]),
                          pack2(c[2 * kk + 1][0], c[2 * kk + 1][1]), pack2(c[2 * kk + 1][2], c[2 * kk + 1][3])};
        av_step(o, pa, vs_a, kk * 16, lane);
      }
      const float i0 = 1.f / l0, i1 = 1.f / l1;
      const int row0 = r0 + g, row1 = row0 + 8;
#pragma unroll
      for (int dt = 0; dt < 8; ++dt) {
        const int col = h * 64 + dt * 8 + 2 * t;
        if (row0 < T) *reinterpret_cast<__nv_bfloat162*>(out + ((size_t)s * T + row0) * D + col) = __floats2bfloat162_rn(o[dt][0] * i0, o[dt][1] * i0);
        if (row1 < T) *reinterpret_cast<__nv_bfloat162*>(out + ((size_t)s * T + row1) * D + col) = __floats2bfloat162_rn(o[dt][2] * i1, o[dt][3] * i1);
      }
    }
    __syncthreads();          // everyone is done with buffer b before the next-next prefetch overwrites it
  }
}

template <int NT2>
__global__ void __launch_bounds__(128, 2) k_attn_bwd_tc1(const __grid_constant__ CUtensorMap tm_kv, const __grid_constant__ CUtensorMap tm_q,
                                                         const __grid_constant__ CUtensorMap tm_do, bf16* __restrict__ dqkv,
                                                         int T, int D, int heads, int items) {
  pdl_trigger(); pdl_wait();
  extern __shared__ __align__(1024) uint8_t sm_raw[];
  __shared__ __align__(8) uint64_t full[2];
  constexpr int TK = NT2 * 16, QB = 64, PB = 128, BUF = (2 * TK + 2 * QB) * 128;
  uint8_t* sm = sm_raw + (((smem_u32(sm_raw) + 1023u) & ~1023u) - smem_u32(sm_raw));
  const uint32_t sm_a = smem_u32(sm);
  uint8_t* Ps = sm + 2 * BUF; uint8_t* Ds = Ps + QB * PB;
  const uint32_t ps_a = smem_u32(Ps), ds_a = smem_u32(Ds);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  const size_t ld = (size_t)3 * D;
  if (threadIdx.x == 0) {
    mbar_init(&full[0], 1); mbar_init(&full[1], 1); fence_barrier_init();
    tma_prefetch_desc(&tm_kv); tma_prefetch_desc(&tm_q); tma_prefetch_desc(&tm_do);
  }
  __syncthreads();
  auto issue = [&](int item, int b) {
    const int s = item / heads, h = item - s * heads;
    const uint32_t a = sm_a + b * BUF;
    mbar_expect_tx(&full[b], BUF);
    tma_load_3d(a, &tm_kv, &full[b], D + h * 64, 0, s);
    tma_load_3d(a + TK * 128, &tm_kv, &full[b], 2 * D + h * 64, 0, s);
    tma_load_3d(a + 2 * TK * 128, &tm_q, &full[b], h * 64, 0, s);
    tma_load_3d(a + (2 * TK + QB) * 128, &tm_do, &full[b], h * 64, 0, s);
  };
  int item = blockIdx.x, b = 0;
  uint32_t phases = 0u;                                          // bit b = parity of the next fill of buffer b
  if (item < items && threadIdx.x == 0) issue(item, 0);
  for (; item < items; item += gridDim.x, b ^= 1) {
    const int nxt = item + gridDim.x;
    if (nxt < items && threadIdx.x == 0) issue(nxt, b ^ 1);
    mbar_wait(&full[b], (phases >> b) & 1u); phases ^= 1u << b;
    const int s = item / heads, h = item - s * heads;
    bf16* obase = dqkv + (size_t)s * T * ld + h * 64;
    const uint32_t ks_a = sm_a + b * BUF, vs_a = ks_a + TK * 128, qs_a = vs_a + TK * 128, gs_a = qs_a + QB * 128;
    const int r0 = warp * 16;
    {
      uint32_t qa[4][4], ga[4][4];
      load_a_frags(qa, qs_a, r0, lane);
      load_a_frags(ga, gs_a, r0, lane);
      float dq[8][4];
#pragma unroll
      for (int i = 0; i < 8; ++i) { dq[i][0] = dq[i][1] = dq[i][2] = dq[i][3] = 0.f; }
      float c[2 * NT2][4], e[2 * NT2][4];
      float m0 = -INFINITY, m1 = -INFINITY;
#pragma unroll
      for (int n2 = 0; n2 < NT2; ++n2) {
        qk_tile(c[2 * n2], c[2 * n2 + 1], qa, ks_a, n2 * 16, lane);
        qk_tile(e[2 * n2], e[2 * n2 + 1], ga, vs_a, n2 * 16, lane);
#pragma unroll
        for (int u = 0; u < 2; ++u) {
          const int cl = n2 * 16 + u * 8 + 2 * t;
          float* cc = c[2 * n2 + u];
          cc[0] = (cl < T) ? cc[0] * kAttnScaleLog2 : -INFINITY; cc[1] = (cl + 1 < T) ? cc[1] * kAttnScaleLog2 : -INFINITY;
          cc[2] = (cl < T) ? cc[2] * kAttnScaleLog2 : -INFINITY; cc[3] = (cl + 1 < T) ? cc[3] * kAttnScaleLog2 : -INFINITY;
          m0 = fmaxf(m0, fmaxf(cc[0], cc[1])); m1 = fmaxf(m1, fmaxf(cc[2], cc[3]));
        }
      }
      m0 = quad_max(m0); m1 = quad_max(m1);
      float l0 = 0.f, l1 = 0.f, d0 = 0.f, d1 = 0.f;
#pragma unroll
      for (int n = 0; n < 2 * NT2; ++n) {
        c[n][0] = exp2f(c[n][0] - m0); c[n][1] = exp2f(c[n][1] - m0); c[n][2] = exp2f(c[n][2] - m1); c[n][3] = exp2f(c[n][3] - m1);
        l0 += c[n][0] + c[n][1]; l1 += c[n][2] + c[n][3];
        d0 += c[n][0] * e[n][0] + c[n][1] * e[n][1]; d1 += c[n][2] * e[n][2] + c[n][3] * e[n][3];
      }
      l0 = quad_sum(l0); l1 = quad_sum(l1); d0 = quad_sum(d0); d1 = quad_sum(d1);
      const float i0 = 1.f / l0, i1 = 1.f / l1;
      d0 *= i0; d1 *= i1;
#pragma unroll
      for (int n2 = 0; n2 < NT2; ++n2) {
        uint32_t pa[4], da[4];
#pragma unroll
        for (int u = 0; u < 2; ++u) {
          const float* cc = c[2 * n2 + u]; const float* ee = e[2 * n2 + u];
          const float p0 = cc[0] * i0, p1 = cc[1] * i0, p2 = cc[2] * i1, p3 = cc[3] * i1;
          pa[2 * u] = pack2(p0, p1); pa[2 * u + 1] = pack2(p2, p3);
          da[2 * u] = pack2(p0 * (ee[0] - d0) * 0.125f, p1 * (ee[1] - d0) * 0.125f);
          da[2 * u + 1] = pack2(p2 * (ee[2] - d1) * 0.125f, p3 * (ee[3] - d1) * 0.125f);
          const int chunk = n2 * 2 + u;
          *reinterpret_cast<uint32_t*>(Ps + swz(r0 + g, chunk, PB) + 4 * t) = pa[2 * u];
          *reinterpret_cast<uint32_t*>(Ps + swz(r0 + g + 8, chunk, PB) + 4 * t) = pa[2 * u + 1];
          *reinterpret_cast<uint32_t*>(Ds + swz(r0 + g, chunk, PB) + 4 * t) = da[2 * u];
          *reinterpret_cast<uint32_t*>(Ds + swz(r0 + g + 8, chunk, PB) + 4 * t) = da[2 * u + 1];
        }
        av_step(dq, da, ks_a, n2 * 16, lane);
      }
      const int row0 = r0 + g, row1 = row0 + 8;
#pragma unroll
      for (int dt = 0; dt < 8; ++dt) {
        const int col = dt * 8 + 2 * t;
        if (row0 < T) *reinterpret_cast<__nv_bfloat162*>(obase + (size_t)row0 * ld + col) = __floats2bfloat162_rn(dq[dt][0], dq[dt][1]);
        if (row1 < T) *reinterpret_cast<__nv_bfloat162*>(obase + (size_t)row1 * ld + col) = __floats2bfloat162_rn(dq[dt][2], dq[dt][3]);
      }
    }
    __syncthreads();
    if (warp < NT2) {          // key tile kt = warp
      float dv[8][4], dk[8][4];
#pragma unroll
      for (int j = 0; j < 8; ++j) { dv[j][0] = dv[j][1] = dv[j][2] = dv[j][3] = 0.f; dk[j][0] = dk[j][1] = dk[j][2] = dk[j][3] = 0.f; }
#pragma unroll
      for (int ks = 0; ks < QB / 16; ++ks) {
        uint32_t pa[4], da[4];
        const int srow = ks * 16 + (lane & 7) + ((lane >> 4) << 3), chunk = warp * 2 + ((lane >> 3) & 1);
        ldsm4t(pa, ps_a + swz(srow, chunk, PB));
        ldsm4t(da, ds_a + swz(srow, chunk, PB));
        av_step(dv, pa, gs_a, ks * 16, lane);
        av_step(dk, da, qs_a, ks * 16, lane);
      }
      const int key0 = warp * 16 + g, key1 = key0 + 8;
#pragma unroll
      for (int dt = 0; dt < 8; ++dt) {
        const int col = dt * 8 + 2 * t;
        if (key0 < T) {
          *reinterpret_cast<__nv_bfloat162*>(obase + (size_t)key0 * ld + D + col) = __floats2bfloat162_rn(dk[dt][0], dk[dt][1]);
          *reinterpret_cast<__nv_bfloat162*>(obase + (size_t)key0 * ld + 2 * D + col) = __floats2bfloat162_rn(dv[dt][0], dv[dt][1]);
        }
        if (key1 < T) {
          *reinterpret_cast<__nv_bfloat162*>(obase + (size_t)key1 * ld + D + col) = __floats2bfloat162_rn(dk[dt][2], dk[dt][3]);
          *reinterpret_cast<__nv_bfloat162*>(obase + (size_t)key1 * ld + 2 * D + col) = __floats2bfloat162_rn(dv[dt][2], dv[dt][3]);
        }
      }
    }
    __syncthreads();          // buffer b and Ps / Ds are free again
  }
}

template <int NT2>
static int attn_launch1(bool fwd, const bf16* qkv, const bf16* dout, bf16* out_or_dqkv, int S, int T, int D, int heads, cudaStream_t st) {
  constexpr size_t smem_f = (size_t)2 * (2 * NT2 * 16 + 64) * 128 + 1024;                                // + alignment slack
  constexpr size_t smem_b = (size_t)2 * (2 * NT2 * 16 + 128) * 128 + (size_t)2 * 64 * 128 + 1024;
  static bool cfg = false;
  if (!cfg) {
    APH_CUDA_OK(cudaFuncSetAttribute(k_attn_fwd_tc1<NT2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_f));
    APH_CUDA_OK(cudaFuncSetAttribute(k_attn_bwd_tc1<NT2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_b));
    APH_CUDA_OK(cudaFuncSetAttribute(k_attn_fwd_tc1<NT2>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    APH_CUDA_OK(cudaFuncSetAttribute(k_attn_bwd_tc1<NT2>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    cfg = true;
  }
  const int items = S * heads;
  CUtensorMap tm_kv, tm_q, tm_do;
  if (int e = make_tmap_bf16_tokens(&tm_kv, qkv, 3 * D, T, S, NT2 * 16)) return e;
  if (int e = make_tmap_bf16_tokens(&tm_q, qkv, 3 * D, T, S, 64)) return e;
  if (fwd) {
    const int per_sm = (int)(220 * 1024 / smem_f) < 6 ? (int)(220 * 1024 / smem_f) : 6;
    const int grid = items < kNumSMs * per_sm ? items : kNumSMs * per_sm;
    APH_CUDA_OK(launch_k(k_attn_fwd_tc1<NT2>, dim3(grid), dim3(128), smem_f, st, 1, tm_kv, tm_q, out_or_dqkv, T, D, heads, items));
  } else {
    if (int e = make_tmap_bf16_tokens(&tm_do, dout, D, T, S, 64)) return e;
    const int per_sm = (int)(220 * 1024 / smem_b) < 3 ? (int)(220 * 1024 / smem_b) : 3;
    const int grid = items < kNumSMs * per_sm ? items : kNumSMs * per_sm;
    APH_CUDA_OK(launch_k(k_attn_bwd_tc1<NT2>, dim3(grid), dim3(128), smem_b, st, 1, tm_kv, tm_q, tm_do, out_or_dqkv, T, D, heads, items));
  }
  APH_LAUNCH_OK();
  return 0;
}

template <int NW, int NT2> constexpr size_t attn_tc_fwd_smem() { return (size_t)(2 * NT2 * 16 + NW * 16) * 128; }
template <int NW, int NT2> constexpr size_t attn_tc_bwd_smem() {
  return (size_t)(2 * NT2 * 16 + 2 * NW * 16) * 128 + (size_t)2 * NW * 16 * (((NT2 * 16 + 63) / 64) * 128);
}

// Host dispatch over the supported (warps, key-tile) shapes: T <= 32, 64, 112, 208, 256.
template <int NW, int NT2>
static int attn_launch(bool fwd, const bf16* qkv, const bf16* dout, bf16* out_or_dqkv, int S, int T, int D, int heads, cudaStream_t st) {
  static bool cfg = false;
  if (!cfg) {
    APH_CUDA_OK(cudaFuncSetAttribute(k_attn_fwd_tc<NW, NT2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)attn_tc_fwd_smem<NW, NT2>()));
    APH_CUDA_OK(cudaFuncSetAttribute(k_attn_bwd_tc<NW, NT2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)attn_tc_bwd_smem<NW, NT2>()));
    APH_CUDA_OK(cudaFuncSetAttribute(k_attn_fwd_tc<NW, NT2>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    APH_CUDA_OK(cudaFuncSetAttribute(k_attn_bwd_tc<NW, NT2>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    cfg = true;
  }
  if (fwd) APH_CUDA_OK(launch_k(k_attn_fwd_tc<NW, NT2>, dim3(S * heads), dim3(NW * 32), attn_tc_fwd_smem<NW, NT2>(), st, 1, qkv, out_or_dqkv, T, D, heads));
  else APH_CUDA_OK(launch_k(k_attn_bwd_tc<NW, NT2>, dim3(S * heads), dim3(NW * 32), attn_tc_bwd_smem<NW, NT2>(), st, 1, qkv, dout, out_or_dqkv, T, D, heads));
  APH_LAUNCH_OK();
  return 0;
}

static int attn_dispatch(bool fwd, const bf16* qkv, const bf16* dout, bf16* out_or_dqkv, int S, int T, int D, int heads, cudaStream_t st) {
  static int nopipe = -1;
  if (nopipe < 0) { const char* e = getenv("APH_ATTN_NOPIPE"); nopipe = (e && e[0] == '1') ? 1 : 0; }
  if (!nopipe && T <= 32) return attn_launch1<2>(fwd, qkv, dout, out_or_dqkv, S, T, D, heads, st);
  if (!nopipe && T <= 64) return attn_launch1<4>(fwd, qkv, dout, out_or_dqkv, S, T, D, heads, st);
  if (T <= 32) return attn_launch<4, 2>(fwd, qkv, dout, out_or_dqkv, S, T, D, heads, st);
  if (T <= 64) return attn_launch<4, 4>(fwd, qkv, dout, out_or_dqkv, S, T, D, heads, st);
  if (T <= 112) return attn_launch<8, 7>(fwd, qkv, dout, out_or_dqkv, S, T, D, heads, st);
  if (T <= 208) return attn_launch<8, 13>(fwd, qkv, dout, out_or_dqkv, S, T, D, heads, st);
  if (T <= 256) return attn_launch<8, 16>(fwd, qkv, dout, out_or_dqkv, S, T, D, heads, st);
  set_error("attention: T=%d > 256 unsupported", T);
  return 2;
}

}  // namespace aph
