// ln_rows.cuh -- LayerNorm building blocks shared by the CLIP image encoder (vit.cu) and text encoder (text.cu):
// one warp per row of width D = 128*NCH held in registers, the row load/store helpers and the bf16-output LayerNorm.
#pragma once
#include "tc_gemm.cuh"

namespace aph {

// ---------------------------------------------------------------------------------------------
// LayerNorm row helpers: one warp per row, width D (multiple of 128), each lane holds D/32 values.

struct RowStats { float mean, rstd; };

template <int N>
__device__ __forceinline__ RowStats row_stats(const float (&v)[N], int D) {
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < N; ++i) s += v[i];
  const float mean = warp_sum(s) / (float)D;
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < N; ++i) { const float d = v[i] - mean; q += d * d; }
  const float var = warp_sum(q) / (float)D;
  return {mean, rsqrtf(var + 1e-5f)};
}

// lane owns float4 chunks: element index of chunk k = (k*32 + lane)*4
template <int N>
__device__ __forceinline__ void load_row(const float* __restrict__ row, float (&v)[N], int lane) {
#pragma unroll
  for (int k = 0; k < N / 4; ++k) {
    const float4 a = *reinterpret_cast<const float4*>(row + (k * 32 + lane) * 4);
    v[4 * k] = a.x; v[4 * k + 1] = a.y; v[4 * k + 2] = a.z; v[4 * k + 3] = a.w;
  }
}
// bf16 row -> fp32 registers (same lane ownership as load_row: chunk k holds elements (k*32 + lane)*4 .. +3)
template <int N>
__device__ __forceinline__ void load_row(const bf16* __restrict__ row, float (&v)[N], int lane) {
#pragma unroll
  for (int k = 0; k < N / 4; ++k) {
    const uint2 u = *reinterpret_cast<const uint2*>(row + (k * 32 + lane) * 4);
    const float2 a = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u.x)), b = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u.y));
    v[4 * k] = a.x; v[4 * k + 1] = a.y; v[4 * k + 2] = b.x; v[4 * k + 3] = b.y;
  }
}
template <int N>
__device__ __forceinline__ void store_row_f32(float* __restrict__ row, const float (&v)[N], int lane) {
#pragma unroll
  for (int k = 0; k < N / 4; ++k)
    *reinterpret_cast<float4*>(row + (k * 32 + lane) * 4) = make_float4(v[4 * k], v[4 * k + 1], v[4 * k + 2], v[4 * k + 3]);
}
template <int N>
__device__ __forceinline__ void store_row_bf16(bf16* __restrict__ row, const float (&v)[N], int lane) {
#pragma unroll
  for (int k = 0; k < N / 4; ++k) {
    __nv_bfloat162 p0 = __floats2bfloat162_rn(v[4 * k], v[4 * k + 1]), p1 = __floats2bfloat162_rn(v[4 * k + 2], v[4 * k + 3]);
    uint2 u; u.x = *reinterpret_cast<uint32_t*>(&p0); u.y = *reinterpret_cast<uint32_t*>(&p1);
    *reinterpret_cast<uint2*>(row + (k * 32 + lane) * 4) = u;
  }
}

// y = LN(x) as bf16. Input row r lives at x + r*in_stride (in_stride = D for all tokens, T*D for the cls rows).
template <int NCH>
__global__ void __launch_bounds__(256) k_ln_fwd(const float* __restrict__ x, size_t in_stride, const float* __restrict__ gamma,
                                                const float* __restrict__ beta, bf16* __restrict__ y, float* __restrict__ mean_out,
                                                float* __restrict__ rstd_out, int rows, int D) {
  pdl_trigger(); pdl_wait();
  const int row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (row >= rows) return;
  constexpr int N = 4 * NCH;
  float v[N], gm[N], bt[N];
  load_row(x + (size_t)row * in_stride, v, lane);
  const RowStats st = row_stats(v, D);
  load_row(gamma, gm, lane); load_row(beta, bt, lane);
  #pragma unroll
  for (int i = 0; i < N; ++i) v[i] = (v[i] - st.mean) * st.rstd * gm[i] + bt[i];
  store_row_bf16(y + (size_t)row * D, v, lane);
  if (lane == 0) { mean_out[row] = st.mean; rstd_out[row] = st.rstd; }
}

#define NCH_DISPATCH(D, ...)                                                           \
  switch ((D) / 128) {                                                                 \
    case 1: { constexpr int NCH = 1; __VA_ARGS__; } break;                             \
    case 2: { constexpr int NCH = 2; __VA_ARGS__; } break;                             \
    case 4: { constexpr int NCH = 4; __VA_ARGS__; } break;                             \
    case 6: { constexpr int NCH = 6; __VA_ARGS__; } break;                             \
    case 8: { constexpr int NCH = 8; __VA_ARGS__; } break;                             \
    default: set_error("unsupported width %d", (D)); return 2;                         \
  }

// blocks of 256 threads (8 warps) covering `rows` one-warp rows
static inline int rows_grid(int rows) { return (rows * 32 + 255) / 256; }

}  // namespace aph
