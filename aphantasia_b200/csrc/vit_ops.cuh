// vit_ops.cu -- the non-GEMM kernels of the CLIP ViT-B image encoder, forward and data-gradient.
//
// Restates OpenAI clip/model.py VisionTransformer (third-party; SURVEY.md A5): patchify (conv1 with
// stride = kernel is an im2col permutation), cls/pos embedding + ln_pre, LayerNorm (fp32 statistics),
// multi-head attention core softmax(QK^T/sqrt(64))V, and their backward passes (no weight gradients).
// Token rows are sample-major: row = s*T + t.  Width D = 128*NCH (template), so rows live in registers.
#pragma once
#include "ln_rows.cuh"

namespace aph {

// ---------------------------------------------------------------------------------------------
// images fp32 [S,3,R,R] -> patches bf16 [S*g*g, 3*p*p], col = c*p*p + py*p + px  (conv1 weight layout)
__global__ void __launch_bounds__(256) k_patchify(const float* __restrict__ img, bf16* __restrict__ out, int S, int p, int g) {
  pdl_trigger(); pdl_wait();
  const int R = p * g, Kp = 3 * p * p;
  const size_t total = (size_t)S * g * g * Kp / 8;
  for (size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
    const size_t e = idx * 8;
    const int row = (int)(e / Kp), col = (int)(e - (size_t)row * Kp);
    const int s = row / (g * g), pr = row - s * g * g, gy = pr / g, gx = pr - gy * g;
    const int c = col / (p * p), rem = col - c * p * p, py = rem / p, px = rem - py * p;
    const float* src = img + (((size_t)s * 3 + c) * R + gy * p + py) * R + gx * p + px;
    const float4 a = __ldg(reinterpret_cast<const float4*>(src)), b = __ldg(reinterpret_cast<const float4*>(src) + 1);
    __nv_bfloat162 p0 = __floats2bfloat162_rn(a.x, a.y), p1 = __floats2bfloat162_rn(a.z, a.w);
    __nv_bfloat162 p2 = __floats2bfloat162_rn(b.x, b.y), p3 = __floats2bfloat162_rn(b.z, b.w);
    uint4 u; u.x = *reinterpret_cast<uint32_t*>(&p0); u.y = *reinterpret_cast<uint32_t*>(&p1);
    u.z = *reinterpret_cast<uint32_t*>(&p2); u.w = *reinterpret_cast<uint32_t*>(&p3);
    *reinterpret_cast<uint4*>(out + e) = u;
  }
}

__global__ void __launch_bounds__(256) k_f32_to_bf16(const float* __restrict__ in, bf16* __restrict__ out, size_t n) {
  pdl_trigger(); pdl_wait();
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    out[i] = __float2bfloat16_rn(in[i]);
}

// e = [cls; tok] + pos (saved), x0 = ln_pre(e). tok fp32 [S*(T-1), D].
template <int NCH>
__global__ void __launch_bounds__(256) k_embed_lnpre(const float* __restrict__ tok, const float* __restrict__ cls,
                                                     const float* __restrict__ pos, const float* __restrict__ gamma,
                                                     const float* __restrict__ beta, float* __restrict__ e_out,
                                                     float* __restrict__ x0, float* __restrict__ mean_out, float* __restrict__ rstd_out,
                                                     int S, int T, int D) {
  pdl_trigger(); pdl_wait();
  const int row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (row >= S * T) return;
  const int s = row / T, t = row - s * T;
  constexpr int N = 4 * NCH;
  const float* src = (t == 0) ? cls : tok + ((size_t)s * (T - 1) + (t - 1)) * D;
  float v[N], pz[N];
  load_row(src, v, lane);
  load_row(pos + (size_t)t * D, pz, lane);
  #pragma unroll
  for (int i = 0; i < N; ++i) v[i] += pz[i];
  store_row_f32(e_out + (size_t)row * D, v, lane);
  const RowStats st = row_stats(v, D);
  float gm[N], bt[N];
  load_row(gamma, gm, lane); load_row(beta, bt, lane);
  #pragma unroll
  for (int i = 0; i < N; ++i) v[i] = (v[i] - st.mean) * st.rstd * gm[i] + bt[i];
  store_row_f32(x0 + (size_t)row * D, v, lane);
  if (lane == 0) { mean_out[row] = st.mean; rstd_out[row] = st.rstd; }
}

// LayerNorm data-gradient for one row: returns dx in v (input: dy in v, x in xv).
template <int N>
__device__ __forceinline__ void ln_bwd_row(float (&v)[N], const float (&xv)[N], const float (&gm)[N], float mean, float rstd, int D) {
  float s1 = 0.f, s2 = 0.f;
#pragma unroll
  for (int i = 0; i < N; ++i) {
    const float xh = (xv[i] - mean) * rstd, dxh = v[i] * gm[i];
    s1 += dxh; s2 += dxh * xh;
  }
  s1 = warp_sum(s1) / (float)D; s2 = warp_sum(s2) / (float)D;
#pragma unroll
  for (int i = 0; i < N; ++i) {
    const float xh = (xv[i] - mean) * rstd, dxh = v[i] * gm[i];
    v[i] = rstd * (dxh - s1 - xh * s2);
  }
}

// mode 0: all rows: dx[row] (+)= LNbwd(dy[row]); writes dx (fp32) and dx_bf16.        (ln_1 / ln_2)
// mode 1: ln_post: dy has S rows (cls only); dx[s*T] = LNbwd, other rows were zeroed by the caller.
// mode 2: ln_pre : dy = dx itself (all rows); writes only non-cls rows as bf16 into dtok [S*(T-1), D].
template <int NCH, typename DY = float>
__global__ void __launch_bounds__(256) k_ln_bwd(const DY* __restrict__ dy, const float* __restrict__ x, const float* __restrict__ mean,
                                                const float* __restrict__ rstd, const float* __restrict__ gamma,
                                                float* __restrict__ dx, bf16* __restrict__ dx_bf16, int rows, int T, int D,
                                                int mode, int accumulate) {
  pdl_trigger(); pdl_wait();
  const int r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (r >= rows) return;
  constexpr int N = 4 * NCH;
  const size_t row = (mode == 1) ? (size_t)r * T : (size_t)r;      // token row in x / dx
  if (mode == 2 && (r % T) == 0) return;                           // the cls row has no patch behind it
  float v[N], xv[N], gm[N];
  load_row(dy + (size_t)r * D, v, lane);
  load_row(x + row * D, xv, lane);
  load_row(gamma, gm, lane);
  const int sidx = (mode == 1) ? r : (int)row;
  ln_bwd_row(v, xv, gm, mean[sidx], rstd[sidx], D);
  if (mode == 2) {
    const int s = r / T, t = r - s * T;
    store_row_bf16(dx_bf16 + ((size_t)s * (T - 1) + (t - 1)) * D, v, lane);
    return;
  }
  if (accumulate) {
    float a[N];
    load_row(dx + row * D, a, lane);
    #pragma unroll
  for (int i = 0; i < N; ++i) v[i] += a[i];
  }
  store_row_f32(dx + row * D, v, lane);
  store_row_bf16(dx_bf16 + row * D, v, lane);
}

// ---------------------------------------------------------------------------------------------
// Attention core, one CTA per (sample, head), head dim 64, T <= 256. qkv bf16 [S*T, 3*D]: q | k | v.
// Forward: warp per query row; lanes own keys for the scores, dims for the output.
constexpr int HD = 64;

__global__ void __launch_bounds__(256) k_attn_fwd(const bf16* __restrict__ qkv, bf16* __restrict__ out, int T, int D, int heads) {
  extern __shared__ uint8_t sm_raw[];
  const int Tp = (T + 31) & ~31;
  const int Tq = Tp + 2;                                 // padded leading dim of transposed arrays (bank spread)
  bf16* Kt = reinterpret_cast<bf16*>(sm_raw);            // [HD][Tq]
  bf16* V = Kt + HD * Tq;                                // [T][HD]
  float* qs = reinterpret_cast<float*>(V + (size_t)Tp * HD);   // [8][HD]
  float* ps = qs + 8 * HD;                               // [8][Tp]
  const int s = blockIdx.x / heads, h = blockIdx.x - s * heads;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const size_t ld = (size_t)3 * D;
  const bf16* base = qkv + (size_t)s * T * ld + h * HD;
  for (int idx = threadIdx.x; idx < Tp * HD; idx += blockDim.x) {
    const int j = idx / HD, d = idx - j * HD;
    const bool ok = j < T;
    Kt[d * Tq + j] = ok ? base[(size_t)j * ld + D + d] : __float2bfloat16(0.f);
    if (ok) V[j * HD + d] = base[(size_t)j * ld + 2 * D + d];
  }
  __syncthreads();
  const int nj = Tp / 32;
  for (int i = warp; i < T; i += 8) {
    const __nv_bfloat162 q2 = *reinterpret_cast<const __nv_bfloat162*>(base + (size_t)i * ld + 2 * lane);
    const float2 qf = __bfloat1622float2(q2);
    qs[warp * HD + 2 * lane] = qf.x * 0.125f; qs[warp * HD + 2 * lane + 1] = qf.y * 0.125f;
    __syncwarp();
    float sc[8];
    float mx = -INFINITY;
    #pragma unroll
    for (int jj = 0; jj < 8; ++jj) if (jj < nj) {
      const int j = jj * 32 + lane;
      float a = 0.f;
#pragma unroll 16
      for (int d = 0; d < HD; ++d) a += qs[warp * HD + d] * __bfloat162float(Kt[d * Tq + j]);
      sc[jj] = (j < T) ? a : -INFINITY;
      mx = fmaxf(mx, sc[jj]);
    }
    mx = warp_max(mx);
    float sum = 0.f;
    #pragma unroll
    for (int jj = 0; jj < 8; ++jj) if (jj < nj) { const float p = __expf(sc[jj] - mx); sc[jj] = p; sum += p; }
    sum = warp_sum(sum);
    const float inv = 1.f / sum;
    #pragma unroll
    for (int jj = 0; jj < 8; ++jj) if (jj < nj) ps[warp * Tp + jj * 32 + lane] = sc[jj] * inv;
    __syncwarp();
    float o0 = 0.f, o1 = 0.f;
    for (int j = 0; j < T; ++j) {
      const float p = ps[warp * Tp + j];
      const float2 v = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(V + j * HD + 2 * lane));
      o0 += p * v.x; o1 += p * v.y;
    }
    *reinterpret_cast<__nv_bfloat162*>(out + ((size_t)s * T + i) * D + h * HD + 2 * lane) = __floats2bfloat162_rn(o0, o1);
    __syncwarp();
  }
}

// Backward: pass 1 (warp per query row) -> dQ and the row statistics (max, 1/sum, delta);
//           pass 2 (warp per key) recomputes its column of P / dS and reduces dK, dV without atomics.
__global__ void __launch_bounds__(256) k_attn_bwd(const bf16* __restrict__ qkv, const bf16* __restrict__ dout, bf16* __restrict__ dqkv,
                                                  int T, int D, int heads) {
  extern __shared__ uint8_t sm_raw[];
  const int Tp = (T + 31) & ~31;
  const int Tq = Tp + 2;                       // padded leading dim of transposed arrays (bank spread)
  bf16* Q = reinterpret_cast<bf16*>(sm_raw);   // [Tp][HD]
  bf16* K = Q + (size_t)Tp * HD;               // [Tp][HD]
  bf16* dO = K + (size_t)Tp * HD;              // [Tp][HD]
  bf16* Qt = dO + (size_t)Tp * HD;             // [HD][Tq]
  bf16* Kt = Qt + (size_t)Tq * HD;
  bf16* Vt = Kt + (size_t)Tq * HD;
  bf16* dOt = Vt + (size_t)Tq * HD;
  float* rmax = reinterpret_cast<float*>(dOt + (size_t)Tq * HD);   // [Tp]
  float* rinv = rmax + Tp;
  float* rdel = rinv + Tp;
  float* va = rdel + Tp;                       // [8][HD] per-warp vector a (q or k, pre-scaled)
  float* vb = va + 8 * HD;                     // [8][HD] per-warp vector b (dO row or v)
  float* s1 = vb + 8 * HD;                     // [8][Tp] strip 1 (p)
  float* s2 = s1 + 8 * Tp;                     // [8][Tp] strip 2 (ds)
  const int s = blockIdx.x / heads, h = blockIdx.x - s * heads;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const size_t ld = (size_t)3 * D;
  const bf16* base = qkv + (size_t)s * T * ld + h * HD;
  const bf16* dbase = dout + (size_t)s * T * D + h * HD;
  const bf16 zero = __float2bfloat16(0.f);
  for (int idx = threadIdx.x; idx < Tp * HD; idx += blockDim.x) {
    const int j = idx / HD, d = idx - j * HD;
    const bool ok = j < T;
    const bf16 q = ok ? base[(size_t)j * ld + d] : zero, k = ok ? base[(size_t)j * ld + D + d] : zero;
    const bf16 v = ok ? base[(size_t)j * ld + 2 * D + d] : zero, g = ok ? dbase[(size_t)j * D + d] : zero;
    Q[j * HD + d] = q; Qt[d * Tq + j] = q; K[j * HD + d] = k; Kt[d * Tq + j] = k; Vt[d * Tq + j] = v;
    dO[j * HD + d] = g; dOt[d * Tq + j] = g;
  }
  __syncthreads();
  const int nj = Tp / 32;
  float* a = va + warp * HD; float* b = vb + warp * HD;
  float* p1 = s1 + warp * Tp; float* p2 = s2 + warp * Tp;
  // ---- pass 1: query rows
  for (int i = warp; i < T; i += 8) {
    {
      const float2 qf = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(Q + i * HD + 2 * lane));
      const float2 gf = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(dO + i * HD + 2 * lane));
      a[2 * lane] = qf.x * 0.125f; a[2 * lane + 1] = qf.y * 0.125f; b[2 * lane] = gf.x; b[2 * lane + 1] = gf.y;
    }
    __syncwarp();
    float sc[8], dp[8];
    float mx = -INFINITY;
    #pragma unroll
    for (int jj = 0; jj < 8; ++jj) if (jj < nj) {
      const int j = jj * 32 + lane;
      float x = 0.f, y = 0.f;
#pragma unroll 16
      for (int d = 0; d < HD; ++d) { x += a[d] * __bfloat162float(Kt[d * Tq + j]); y += b[d] * __bfloat162float(Vt[d * Tq + j]); }
      sc[jj] = (j < T) ? x : -INFINITY; dp[jj] = y;
      mx = fmaxf(mx, sc[jj]);
    }
    mx = warp_max(mx);
    float sum = 0.f;
    #pragma unroll
    for (int jj = 0; jj < 8; ++jj) if (jj < nj) { sc[jj] = __expf(sc[jj] - mx); sum += sc[jj]; }
    sum = warp_sum(sum);
    const float inv = 1.f / sum;
    float del = 0.f;
    #pragma unroll
    for (int jj = 0; jj < 8; ++jj) if (jj < nj) { sc[jj] *= inv; del += sc[jj] * dp[jj]; }
    del = warp_sum(del);
    #pragma unroll
    for (int jj = 0; jj < 8; ++jj) if (jj < nj) p2[jj * 32 + lane] = sc[jj] * (dp[jj] - del);     // dS (w.r.t. scaled logits)
    if (lane == 0) { rmax[i] = mx; rinv[i] = inv; rdel[i] = del; }
    __syncwarp();
    float g0 = 0.f, g1 = 0.f;
    for (int j = 0; j < T; ++j) {
      const float ds = p2[j];
      const float2 kf = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(K + j * HD + 2 * lane));
      g0 += ds * kf.x; g1 += ds * kf.y;
    }
    *reinterpret_cast<__nv_bfloat162*>(dqkv + ((size_t)s * T + i) * ld + h * HD + 2 * lane) = __floats2bfloat162_rn(g0 * 0.125f, g1 * 0.125f);
    __syncwarp();
  }
  __syncthreads();
  // ---- pass 2: key rows
  for (int j = warp; j < T; j += 8) {
    {
      const float2 kf = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(K + j * HD + 2 * lane));
      a[2 * lane] = kf.x * 0.125f; a[2 * lane + 1] = kf.y * 0.125f;
      b[2 * lane] = __bfloat162float(Vt[(2 * lane) * Tq + j]); b[2 * lane + 1] = __bfloat162float(Vt[(2 * lane + 1) * Tq + j]);
    }
    __syncwarp();
    for (int ii = 0; ii < nj; ++ii) {
      const int i = ii * 32 + lane;
      float x = 0.f, y = 0.f;
#pragma unroll 16
      for (int d = 0; d < HD; ++d) { x += a[d] * __bfloat162float(Qt[d * Tq + i]); y += b[d] * __bfloat162float(dOt[d * Tq + i]); }
      float p = 0.f, ds = 0.f;
      if (i < T) { p = __expf(x - rmax[i]) * rinv[i]; ds = p * (y - rdel[i]); }
      p1[i] = p; p2[i] = ds;
    }
    __syncwarp();
    float k0 = 0.f, k1 = 0.f, v0 = 0.f, v1 = 0.f;
    for (int i = 0; i < T; ++i) {
      const float p = p1[i], ds = p2[i];
      const float2 qf = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(Q + i * HD + 2 * lane));
      const float2 gf = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(dO + i * HD + 2 * lane));
      k0 += ds * qf.x; k1 += ds * qf.y; v0 += p * gf.x; v1 += p * gf.y;
    }
    bf16* orow = dqkv + ((size_t)s * T + j) * ld + h * HD + 2 * lane;
    *reinterpret_cast<__nv_bfloat162*>(orow + D) = __floats2bfloat162_rn(k0 * 0.125f, k1 * 0.125f);
    *reinterpret_cast<__nv_bfloat162*>(orow + 2 * D) = __floats2bfloat162_rn(v0, v1);
    __syncwarp();
  }
}

inline size_t attn_fwd_smem(int T) { const int Tp = (T + 31) & ~31; return (size_t)(Tp + 2 + Tp) * HD * 2 + (8 * HD + 8 * Tp) * 4; }
inline size_t attn_bwd_smem(int T) { const int Tp = (T + 31) & ~31; return (size_t)(3 * Tp + 4 * (Tp + 2)) * HD * 2 + (3 * Tp + 16 * HD + 16 * Tp) * 4; }

}  // namespace aph
