// Region-level kernels of the ESAT backbone (DualTrans_HS, reference model/backbone.py:171-196): LayerNorm + ReLU +
// 16-row region mean for embeddings wider than one GEMM tile, sincos positional embedding, residual add + LayerNorm,
// and multi-head self-attention over the regions of each bag (forward and backward).  Everything here works on
// rows/16 "region" rows; the N-row contraction of the embedding runs on the GEMM engines (gemm_stages.cu).
#include <limits.h>
#include "stages.cuh"
#include "esat_attn.cuh"

namespace advmil {

__device__ __forceinline__ float to_f32(float v) { return v; }
__device__ __forceinline__ float to_f32(bf16 v) { return __bfloat162float(v); }
template <typename T> __device__ __forceinline__ T from_f32(float v);
template <> __device__ __forceinline__ float from_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ bf16 from_f32<bf16>(float v) { return __float2bfloat16_rn(v); }

// ---- a row of width d = 32 * NPL held by one warp: lane l owns columns l, l + 32, ... -----------------------------
template <typename T, int NPL>
__device__ __forceinline__ void row_load(const T* __restrict__ p, int lane, float (&v)[NPL]) {
#pragma unroll
  for (int k = 0; k < NPL; ++k) v[k] = to_f32(p[lane + 32 * k]);
}
// mean and 1/sqrt(var + eps) (biased variance, two passes over the registers: nn.LayerNorm)
template <int NPL>
__device__ __forceinline__ void row_stats(const float (&v)[NPL], float eps, float& mean, float& rstd) {
  float s = 0.f;
#pragma unroll
  for (int k = 0; k < NPL; ++k) s += v[k];
  mean = warp_sum(s) * (1.0f / (32 * NPL));
  float q = 0.f;
#pragma unroll
  for (int k = 0; k < NPL; ++k) { const float c = v[k] - mean; q = fmaf(c, c, q); }
  rstd = rsqrtf(warp_sum(q) * (1.0f / (32 * NPL)) + eps);
}

// ---- vector-friendly column ownership for the N-row streams (y_pre, d_y): lane l owns CONTIGUOUS chunks so that a row moves
// in 16-byte (bf16: 8 columns) / 8-byte pieces instead of 2-byte scalars.  LayerNorm does not care which lane owns which
// column; only gamma / beta / the outputs are indexed through col().  NPL = 12 in bf16: columns [0, 256) in chunks of 8,
// [256, 384) in chunks of 4.  Widths without a vector layout keep the strided ownership (lane, lane + 32, ...).
template <typename T, int NPL> struct RowMap {
  static constexpr int C0 = (sizeof(T) == 2) ? (NPL >= 8 ? 8 : (NPL == 4 ? 4 : 0)) : (NPL % 4 == 0 ? 4 : 0);     // first chunk size
  static constexpr bool VEC = C0 != 0 && (sizeof(T) == 2 ? (NPL == 4 || NPL == 8 || NPL == 12) : true);
  // column of this lane's k-th element
  __device__ __forceinline__ static int col(int lane, int k) {
    if (!VEC) return lane + 32 * k;
    if (sizeof(T) == 2) return k < 8 ? (NPL >= 8 ? 8 * lane + k : 4 * lane + k) : 256 + 4 * lane + (k - 8);
    return 128 * (k >> 2) + 4 * lane + (k & 3);
  }
  __device__ __forceinline__ static void load(const T* __restrict__ p, int lane, float (&v)[NPL]) {
    if constexpr (!VEC) {
#pragma unroll
      for (int k = 0; k < NPL; ++k) v[k] = to_f32(p[lane + 32 * k]);
    } else if constexpr (sizeof(T) == 2) {
      if constexpr (NPL >= 8) {
        const uint4 u = *reinterpret_cast<const uint4*>(p + 8 * lane);
        v[0] = bf_lo(u.x); v[1] = bf_hi(u.x); v[2] = bf_lo(u.y); v[3] = bf_hi(u.y); v[4] = bf_lo(u.z); v[5] = bf_hi(u.z); v[6] = bf_lo(u.w); v[7] = bf_hi(u.w);
        if constexpr (NPL == 12) {
          const uint2 w = *reinterpret_cast<const uint2*>(p + 256 + 4 * lane);
          v[8] = bf_lo(w.x); v[9] = bf_hi(w.x); v[10] = bf_lo(w.y); v[11] = bf_hi(w.y);
        }
      } else {
        const uint2 w = *reinterpret_cast<const uint2*>(p + 4 * lane);
        v[0] = bf_lo(w.x); v[1] = bf_hi(w.x); v[2] = bf_lo(w.y); v[3] = bf_hi(w.y);
      }
    } else {
#pragma unroll
      for (int c = 0; c < NPL / 4; ++c) {
        const float4 f = *reinterpret_cast<const float4*>(reinterpret_cast<const float*>(p) + 128 * c + 4 * lane);
        v[4 * c] = f.x; v[4 * c + 1] = f.y; v[4 * c + 2] = f.z; v[4 * c + 3] = f.w;
      }
    }
  }
  __device__ __forceinline__ static void store(T* __restrict__ p, int lane, const float (&v)[NPL]) {
    if constexpr (!VEC) {
#pragma unroll
      for (int k = 0; k < NPL; ++k) p[lane + 32 * k] = from_f32<T>(v[k]);
    } else if constexpr (sizeof(T) == 2) {
      if constexpr (NPL >= 8) {
        *reinterpret_cast<uint4*>(p + 8 * lane) = make_uint4(pack_bf2(v[0], v[1]), pack_bf2(v[2], v[3]), pack_bf2(v[4], v[5]), pack_bf2(v[6], v[7]));
        if constexpr (NPL == 12) *reinterpret_cast<uint2*>(p + 256 + 4 * lane) = make_uint2(pack_bf2(v[8], v[9]), pack_bf2(v[10], v[11]));
      } else {
        *reinterpret_cast<uint2*>(p + 4 * lane) = make_uint2(pack_bf2(v[0], v[1]), pack_bf2(v[2], v[3]));
      }
    } else {
#pragma unroll
      for (int c = 0; c < NPL / 4; ++c)
        *reinterpret_cast<float4*>(reinterpret_cast<float*>(p) + 128 * c + 4 * lane) = make_float4(v[4 * c], v[4 * c + 1], v[4 * c + 2], v[4 * c + 3]);
    }
  }
};

// =============================================================================================
// emb[r] = mean_{k<16} relu(LayerNorm(y_pre[16 r + k]))  (AVGPoolPatchEmbedding, model/backbone_utils.py:160-167)
// one warp per region; optional positional embedding added to the result (model/backbone.py:192-194)
// =============================================================================================
template <typename T, int NPL>
__global__ void __launch_bounds__(256) ln_relu_mean16_fwd_kernel(const T* __restrict__ y_pre, const float* __restrict__ gamma,
                                                                 const float* __restrict__ beta, int R, float eps,
                                                                 const float* __restrict__ pe, float* __restrict__ emb) {
  pdl_prologue();
  constexpr int d = 32 * NPL;
  const int lane = threadIdx.x & 31, r = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (r >= R) return;
  using Map = RowMap<T, NPL>;
  float g[NPL], b[NPL], acc[NPL];
#pragma unroll
  for (int k = 0; k < NPL; ++k) { g[k] = gamma[Map::col(lane, k)]; b[k] = beta[Map::col(lane, k)]; acc[k] = 0.f; }
#pragma unroll 2
  for (int i = 0; i < 16; ++i) {
    float v[NPL], mean, rstd;
    Map::load(y_pre + ((size_t)r * 16 + i) * d, lane, v);
    row_stats<NPL>(v, eps, mean, rstd);
#pragma unroll
    for (int k = 0; k < NPL; ++k) acc[k] += fmaxf(fmaf((v[k] - mean) * rstd, g[k], b[k]), 0.f);
  }
#pragma unroll
  for (int k = 0; k < NPL; ++k) {
    const size_t o = (size_t)r * d + Map::col(lane, k);
    emb[o] = acc[k] * (1.0f / 16.0f) + (pe ? pe[o] : 0.f);
  }
}

// backward: de = d_emb[r] / 16 where relu was active; LayerNorm backward per row; column sums of d(gamma), d(beta) and
// d_y (the conv bias gradient) per CTA into part[blockIdx.x][3 d]
template <typename T, int NPL>
__global__ void __launch_bounds__(256) ln_relu_mean16_bwd_kernel(const T* __restrict__ y_pre, const float* __restrict__ d_emb,
                                                                 const float* __restrict__ gamma, const float* __restrict__ beta,
                                                                 int R, float eps, T* __restrict__ d_y, float* __restrict__ part) {
  pdl_prologue();
  constexpr int d = 32 * NPL;
  __shared__ float red[8][3 * d];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
  using Map = RowMap<T, NPL>;
  float g[NPL], b[NPL], dg[NPL], db[NPL], dc[NPL];
#pragma unroll
  for (int k = 0; k < NPL; ++k) { g[k] = gamma[Map::col(lane, k)]; b[k] = beta[Map::col(lane, k)]; dg[k] = db[k] = dc[k] = 0.f; }
  for (int r = blockIdx.x * nw + wid; r < R; r += gridDim.x * nw) {
    float de[NPL];
#pragma unroll
    for (int k = 0; k < NPL; ++k) de[k] = d_emb[(size_t)r * d + Map::col(lane, k)] * (1.0f / 16.0f);
#pragma unroll 1
    for (int i = 0; i < 16; ++i) {
      const size_t row = (size_t)r * 16 + i;
      float v[NPL], mean, rstd;
      Map::load(y_pre + row * d, lane, v);
      row_stats<NPL>(v, eps, mean, rstd);
      float gy[NPL], s1 = 0.f, s2 = 0.f;
#pragma unroll
      for (int k = 0; k < NPL; ++k) {
        const float xh = (v[k] - mean) * rstd;
        const float dek = fmaf(xh, g[k], b[k]) > 0.f ? de[k] : 0.f;
        dg[k] = fmaf(dek, xh, dg[k]);
        db[k] += dek;
        gy[k] = dek * g[k];
        s1 += gy[k];
        s2 = fmaf(gy[k], xh, s2);
        v[k] = xh;
      }
      s1 = warp_sum(s1) * (1.0f / d);
      s2 = warp_sum(s2) * (1.0f / d);
      float dy[NPL];
#pragma unroll
      for (int k = 0; k < NPL; ++k) {
        dy[k] = rstd * (gy[k] - s1 - v[k] * s2);
        dc[k] += dy[k];
      }
      Map::store(d_y + row * d, lane, dy);
    }
  }
#pragma unroll
  for (int k = 0; k < NPL; ++k) {
    const int c = Map::col(lane, k);
    red[wid][c] = dg[k]; red[wid][d + c] = db[k]; red[wid][2 * d + c] = dc[k];
  }
  __syncthreads();
  for (int c = threadIdx.x; c < 3 * d; c += blockDim.x) {
    float t = 0.f;
    for (int w = 0; w < nw; ++w) t += red[w][c];
    part[(size_t)blockIdx.x * 3 * d + c] = t;
  }
}

// =============================================================================================
// out = LayerNorm(a + b) per region row; s = a + b is written over b (the backward pass needs s, not b)
// (nn.TransformerEncoderLayer, post-norm: x = norm(x + dropout(sublayer(x))))
// =============================================================================================
template <int NPL>
__global__ void __launch_bounds__(256) add_ln_fwd_kernel(const float* __restrict__ a, float* __restrict__ b_s,
                                                         const float* __restrict__ gamma, const float* __restrict__ beta, int R,
                                                         float eps, float* __restrict__ out) {
  pdl_prologue();
  constexpr int d = 32 * NPL;
  const int lane = threadIdx.x & 31, r = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (r >= R) return;
  float v[NPL], mean, rstd;
#pragma unroll
  for (int k = 0; k < NPL; ++k) {
    const size_t o = (size_t)r * d + lane + 32 * k;
    v[k] = a[o] + b_s[o];
    b_s[o] = v[k];
  }
  row_stats<NPL>(v, eps, mean, rstd);
#pragma unroll
  for (int k = 0; k < NPL; ++k)
    out[(size_t)r * d + lane + 32 * k] = fmaf((v[k] - mean) * rstd, gamma[lane + 32 * k], beta[lane + 32 * k]);
}

// d_s = LayerNorm backward of d_out at s; column sums of d(gamma), d(beta) per CTA into part[blockIdx.x][2 d]
template <int NPL>
__global__ void __launch_bounds__(256) add_ln_bwd_kernel(const float* __restrict__ s, const float* __restrict__ gamma,
                                                         const float* __restrict__ d_out, int R, float eps,
                                                         float* __restrict__ d_s, float* __restrict__ part) {
  pdl_prologue();
  constexpr int d = 32 * NPL;
  __shared__ float red[8][2 * d];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
  float g[NPL], dg[NPL], db[NPL];
#pragma unroll
  for (int k = 0; k < NPL; ++k) { g[k] = gamma[lane + 32 * k]; dg[k] = db[k] = 0.f; }
  for (int r = blockIdx.x * nw + wid; r < R; r += gridDim.x * nw) {
    float v[NPL], gy[NPL], mean, rstd, s1 = 0.f, s2 = 0.f;
    row_load<float, NPL>(s + (size_t)r * d, lane, v);
    row_stats<NPL>(v, eps, mean, rstd);
#pragma unroll
    for (int k = 0; k < NPL; ++k) {
      const float xh = (v[k] - mean) * rstd, dn = d_out[(size_t)r * d + lane + 32 * k];
      dg[k] = fmaf(dn, xh, dg[k]);
      db[k] += dn;
      gy[k] = dn * g[k];
      s1 += gy[k];
      s2 = fmaf(gy[k], xh, s2);
      v[k] = xh;
    }
    s1 = warp_sum(s1) * (1.0f / d);
    s2 = warp_sum(s2) * (1.0f / d);
#pragma unroll
    for (int k = 0; k < NPL; ++k) d_s[(size_t)r * d + lane + 32 * k] = rstd * (gy[k] - s1 - v[k] * s2);
  }
#pragma unroll
  for (int k = 0; k < NPL; ++k) { red[wid][lane + 32 * k] = dg[k]; red[wid][d + lane + 32 * k] = db[k]; }
  __syncthreads();
  for (int c = threadIdx.x; c < 2 * d; c += blockDim.x) {
    float t = 0.f;
    for (int w = 0; w < nw; ++w) t += red[w][c];
    part[(size_t)blockIdx.x * 2 * d + c] = t;
  }
}

__global__ void add_rows_kernel(float* __restrict__ a, const float* __restrict__ b, size_t n4) {
  pdl_prologue();
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n4) return;
  float4 x = reinterpret_cast<float4*>(a)[i];
  const float4 y = reinterpret_cast<const float4*>(b)[i];
  x.x += y.x; x.y += y.y; x.z += y.z; x.w += y.w;
  reinterpret_cast<float4*>(a)[i] = x;
}

// =============================================================================================
// sincos positional embedding of the region coordinates (model/backbone_utils.py:79-99): coordinates relative to the
// bag's minimum; pe[r] = [sin(x w) | cos(x w) | sin(y w) | cos(y w)], w = omega[d/4] (computed by the caller exactly as
// the reference does).  One CTA per bag.
// =============================================================================================
__global__ void __launch_bounds__(256) sincos_pe_kernel(const int64_t* __restrict__ coord, const int32_t* __restrict__ ro,
                                                        int d, const float* __restrict__ omega, float* __restrict__ pe) {
  pdl_prologue();
  __shared__ long long mn[2][8];
  const int b = blockIdx.x, r0 = ro[b], r1 = ro[b + 1];
  long long mx = LLONG_MAX, my = LLONG_MAX;
  for (int r = r0 + threadIdx.x; r < r1; r += blockDim.x) { mx = min(mx, (long long)coord[2 * (size_t)r]); my = min(my, (long long)coord[2 * (size_t)r + 1]); }
  for (int o = 16; o > 0; o >>= 1) { mx = min(mx, __shfl_xor_sync(0xffffffffu, mx, o)); my = min(my, __shfl_xor_sync(0xffffffffu, my, o)); }
  if ((threadIdx.x & 31) == 0) { mn[0][threadIdx.x >> 5] = mx; mn[1][threadIdx.x >> 5] = my; }
  __syncthreads();
  mx = mn[0][0]; my = mn[1][0];
  for (int w = 1; w < (int)(blockDim.x >> 5); ++w) { mx = min(mx, mn[0][w]); my = min(my, mn[1][w]); }
  const int q = d / 4;
  for (size_t i = threadIdx.x; i < (size_t)(r1 - r0) * q; i += blockDim.x) {
    const int r = r0 + (int)(i / q), k = (int)(i % q);
    const float xv = (float)((long long)coord[2 * (size_t)r] - mx) * omega[k];
    const float yv = (float)((long long)coord[2 * (size_t)r + 1] - my) * omega[k];
    float* o = pe + (size_t)r * d;
    o[k] = sinf(xv); o[q + k] = cosf(xv); o[2 * q + k] = sinf(yv); o[3 * q + k] = cosf(yv);
  }
}

// =============================================================================================
// multi-head self-attention over the regions of each bag (nn.MultiheadAttention inside the encoder layer):
//   P = softmax(q k^T / sqrt(hd)) over the bag's regions, dropout on P, ctx = P v.
// qkv [R, 3 d] (q | k | v, head h = columns h*hd .. of each third).  Flash-style: one thread per query, keys/values
// stream through shared memory in tiles, online softmax; lse = log sum exp is kept for the backward pass.
// grid (ceil(max regions per bag / ATT_BQ), bags, heads)
// =============================================================================================
constexpr int ATT_BQ = 128;
constexpr int ATT_BK = 32;

template <int HD>
__global__ void __launch_bounds__(ATT_BQ) mha_fwd_kernel(const float* __restrict__ qkv, const int32_t* __restrict__ ro, int d,
                                                         float scale, AttDrop ad, float* __restrict__ ctx,
                                                         float* __restrict__ lse, int Rtot) {
  pdl_prologue();
  __shared__ __align__(16) float Ks[ATT_BK][HD];
  __shared__ __align__(16) float Vs[ATT_BK][HD];
  const int b = blockIdx.y, head = blockIdx.z, r0 = ro[b], Rb = ro[b + 1] - r0;
  const int q0 = blockIdx.x * ATT_BQ;
  if (q0 >= Rb) return;
  const int qi = q0 + threadIdx.x;
  const bool valid = qi < Rb;
  const size_t ld = 3 * (size_t)d;
  float q[HD], acc[HD];
#pragma unroll
  for (int c = 0; c < HD; ++c) { q[c] = valid ? qkv[(size_t)(r0 + qi) * ld + head * HD + c] * scale : 0.f; acc[c] = 0.f; }
  float m = -INFINITY, l = 0.f;
  for (int k0 = 0; k0 < Rb; k0 += ATT_BK) {
    const int nk = min(ATT_BK, Rb - k0);
    __syncthreads();
    for (int i = threadIdx.x; i < nk * (HD / 4); i += ATT_BQ) {
      const int j = i / (HD / 4), c4 = i % (HD / 4);
      const float* src = qkv + (size_t)(r0 + k0 + j) * ld + head * HD + 4 * c4;
      *reinterpret_cast<float4*>(&Ks[j][4 * c4]) = *reinterpret_cast<const float4*>(src + d);
      *reinterpret_cast<float4*>(&Vs[j][4 * c4]) = *reinterpret_cast<const float4*>(src + 2 * d);
    }
    __syncthreads();
    if (!valid) continue;
    float s[ATT_BK], tm = -INFINITY;
#pragma unroll
    for (int j = 0; j < ATT_BK; ++j) {
      float t = 0.f;
      if (j < nk) {
#pragma unroll
        for (int c4 = 0; c4 < HD / 4; ++c4) {
          const float4 kk = *reinterpret_cast<const float4*>(&Ks[j][4 * c4]);
          t = fmaf(q[4 * c4], kk.x, t); t = fmaf(q[4 * c4 + 1], kk.y, t); t = fmaf(q[4 * c4 + 2], kk.z, t); t = fmaf(q[4 * c4 + 3], kk.w, t);
        }
        tm = fmaxf(tm, t);
      }
      s[j] = t;
    }
    const float mn = fmaxf(m, tm), corr = expf(m - mn);
    l *= corr;
#pragma unroll
    for (int c = 0; c < HD; ++c) acc[c] *= corr;
#pragma unroll
    for (int j = 0; j < ATT_BK; ++j) {
      if (j < nk) {
        const float p = expf(s[j] - mn);
        l += p;
        if (ad.keep(b, head, qi, k0 + j, Rb, r0 + qi)) {
#pragma unroll
          for (int c4 = 0; c4 < HD / 4; ++c4) {
            const float4 vv = *reinterpret_cast<const float4*>(&Vs[j][4 * c4]);
            acc[4 * c4] = fmaf(p, vv.x, acc[4 * c4]); acc[4 * c4 + 1] = fmaf(p, vv.y, acc[4 * c4 + 1]);
            acc[4 * c4 + 2] = fmaf(p, vv.z, acc[4 * c4 + 2]); acc[4 * c4 + 3] = fmaf(p, vv.w, acc[4 * c4 + 3]);
          }
        }
      }
    }
    m = mn;
  }
  if (!valid) return;
  const float inv = ad.drop.inv_keep / l;
#pragma unroll
  for (int c = 0; c < HD; ++c) ctx[(size_t)(r0 + qi) * d + head * HD + c] = acc[c] * inv;
  lse[(size_t)head * Rtot + r0 + qi] = m + logf(l);
}

// backward, pass 1 (one thread per query): D_i = dO_i . O_i, dq_i = scale * sum_j dS_ij k_j with
// dS_ij = P_ij (keep_ij dO_i . v_j / (1-p) - D_i), P_ij = exp(s_ij - lse_i)
template <int HD>
__global__ void __launch_bounds__(ATT_BQ) mha_bwd_q_kernel(const float* __restrict__ qkv, const float* __restrict__ ctx,
                                                           const float* __restrict__ d_ctx, const float* __restrict__ lse,
                                                           const int32_t* __restrict__ ro, int d, float scale, AttDrop ad,
                                                           float* __restrict__ d_qkv, float* __restrict__ Dq, int Rtot) {
  pdl_prologue();
  __shared__ __align__(16) float Ks[ATT_BK][HD];
  __shared__ __align__(16) float Vs[ATT_BK][HD];
  const int b = blockIdx.y, head = blockIdx.z, r0 = ro[b], Rb = ro[b + 1] - r0;
  const int q0 = blockIdx.x * ATT_BQ;
  if (q0 >= Rb) return;
  const int qi = q0 + threadIdx.x;
  const bool valid = qi < Rb;
  const size_t ld = 3 * (size_t)d;
  float q[HD], go[HD], dq[HD];
  float Di = 0.f, li = 0.f;
#pragma unroll
  for (int c = 0; c < HD; ++c) {
    q[c] = valid ? qkv[(size_t)(r0 + qi) * ld + head * HD + c] * scale : 0.f;
    go[c] = valid ? d_ctx[(size_t)(r0 + qi) * d + head * HD + c] : 0.f;
    dq[c] = 0.f;
    if (valid) Di = fmaf(go[c], ctx[(size_t)(r0 + qi) * d + head * HD + c], Di);
  }
  if (valid) { li = lse[(size_t)head * Rtot + r0 + qi]; Dq[(size_t)head * Rtot + r0 + qi] = Di; }
  for (int k0 = 0; k0 < Rb; k0 += ATT_BK) {
    const int nk = min(ATT_BK, Rb - k0);
    __syncthreads();
    for (int i = threadIdx.x; i < nk * (HD / 4); i += ATT_BQ) {
      const int j = i / (HD / 4), c4 = i % (HD / 4);
      const float* src = qkv + (size_t)(r0 + k0 + j) * ld + head * HD + 4 * c4;
      *reinterpret_cast<float4*>(&Ks[j][4 * c4]) = *reinterpret_cast<const float4*>(src + d);
      *reinterpret_cast<float4*>(&Vs[j][4 * c4]) = *reinterpret_cast<const float4*>(src + 2 * d);
    }
    __syncthreads();
    if (!valid) continue;
    for (int j = 0; j < nk; ++j) {
      float t = 0.f, gv = 0.f;
#pragma unroll
      for (int c4 = 0; c4 < HD / 4; ++c4) {
        const float4 kk = *reinterpret_cast<const float4*>(&Ks[j][4 * c4]);
        const float4 vv = *reinterpret_cast<const float4*>(&Vs[j][4 * c4]);
        t = fmaf(q[4 * c4], kk.x, t); t = fmaf(q[4 * c4 + 1], kk.y, t); t = fmaf(q[4 * c4 + 2], kk.z, t); t = fmaf(q[4 * c4 + 3], kk.w, t);
        gv = fmaf(go[4 * c4], vv.x, gv); gv = fmaf(go[4 * c4 + 1], vv.y, gv); gv = fmaf(go[4 * c4 + 2], vv.z, gv); gv = fmaf(go[4 * c4 + 3], vv.w, gv);
      }
      const float p = expf(t - li);
      const float dp = ad.keep(b, head, qi, k0 + j, Rb, r0 + qi) ? gv * ad.drop.inv_keep : 0.f;
      const float ds = p * (dp - Di);
#pragma unroll
      for (int c4 = 0; c4 < HD / 4; ++c4) {
        const float4 kk = *reinterpret_cast<const float4*>(&Ks[j][4 * c4]);
        dq[4 * c4] = fmaf(ds, kk.x, dq[4 * c4]); dq[4 * c4 + 1] = fmaf(ds, kk.y, dq[4 * c4 + 1]);
        dq[4 * c4 + 2] = fmaf(ds, kk.z, dq[4 * c4 + 2]); dq[4 * c4 + 3] = fmaf(ds, kk.w, dq[4 * c4 + 3]);
      }
    }
  }
  if (!valid) return;
#pragma unroll
  for (int c = 0; c < HD; ++c) d_qkv[(size_t)(r0 + qi) * ld + head * HD + c] = dq[c] * scale;
}

// backward, pass 2 (one thread per key): dv_j = sum_i keep_ij P_ij / (1-p) dO_i;  dk_j = scale * sum_i dS_ij q_i
template <int HD>
__global__ void __launch_bounds__(ATT_BQ) mha_bwd_kv_kernel(const float* __restrict__ qkv, const float* __restrict__ d_ctx,
                                                            const float* __restrict__ lse, const float* __restrict__ Dq,
                                                            const int32_t* __restrict__ ro, int d, float scale, AttDrop ad,
                                                            float* __restrict__ d_qkv, int Rtot) {
  pdl_prologue();
  __shared__ __align__(16) float Qs[ATT_BK][HD];
  __shared__ __align__(16) float Gs[ATT_BK][HD];
  __shared__ float Ls[ATT_BK], Ds[ATT_BK];
  const int b = blockIdx.y, head = blockIdx.z, r0 = ro[b], Rb = ro[b + 1] - r0;
  const int k0 = blockIdx.x * ATT_BQ;
  if (k0 >= Rb) return;
  const int kj = k0 + threadIdx.x;
  const bool valid = kj < Rb;
  const size_t ld = 3 * (size_t)d;
  float kk[HD], vv[HD], dk[HD], dv[HD];
#pragma unroll
  for (int c = 0; c < HD; ++c) {
    kk[c] = valid ? qkv[(size_t)(r0 + kj) * ld + d + head * HD + c] : 0.f;
    vv[c] = valid ? qkv[(size_t)(r0 + kj) * ld + 2 * d + head * HD + c] : 0.f;
    dk[c] = 0.f; dv[c] = 0.f;
  }
  for (int q0 = 0; q0 < Rb; q0 += ATT_BK) {
    const int nq = min(ATT_BK, Rb - q0);
    __syncthreads();
    for (int i = threadIdx.x; i < nq * (HD / 4); i += ATT_BQ) {
      const int j = i / (HD / 4), c4 = i % (HD / 4);
      float4 qv = *reinterpret_cast<const float4*>(qkv + (size_t)(r0 + q0 + j) * ld + head * HD + 4 * c4);
      qv.x *= scale; qv.y *= scale; qv.z *= scale; qv.w *= scale;
      *reinterpret_cast<float4*>(&Qs[j][4 * c4]) = qv;
      *reinterpret_cast<float4*>(&Gs[j][4 * c4]) = *reinterpret_cast<const float4*>(d_ctx + (size_t)(r0 + q0 + j) * d + head * HD + 4 * c4);
    }
    if (threadIdx.x < nq) {
      Ls[threadIdx.x] = lse[(size_t)head * Rtot + r0 + q0 + threadIdx.x];
      Ds[threadIdx.x] = Dq[(size_t)head * Rtot + r0 + q0 + threadIdx.x];
    }
    __syncthreads();
    if (!valid) continue;
    for (int i = 0; i < nq; ++i) {
      float t = 0.f, gv = 0.f;
#pragma unroll
      for (int c4 = 0; c4 < HD / 4; ++c4) {
        const float4 qq = *reinterpret_cast<const float4*>(&Qs[i][4 * c4]);
        const float4 gg = *reinterpret_cast<const float4*>(&Gs[i][4 * c4]);
        t = fmaf(kk[4 * c4], qq.x, t); t = fmaf(kk[4 * c4 + 1], qq.y, t); t = fmaf(kk[4 * c4 + 2], qq.z, t); t = fmaf(kk[4 * c4 + 3], qq.w, t);
        gv = fmaf(vv[4 * c4], gg.x, gv); gv = fmaf(vv[4 * c4 + 1], gg.y, gv); gv = fmaf(vv[4 * c4 + 2], gg.z, gv); gv = fmaf(vv[4 * c4 + 3], gg.w, gv);
      }
      const float p = expf(t - Ls[i]);
      const bool keep = ad.keep(b, head, q0 + i, kj, Rb, r0 + q0 + i);
      const float pd = keep ? p * ad.drop.inv_keep : 0.f;
      const float ds = p * ((keep ? gv * ad.drop.inv_keep : 0.f) - Ds[i]);
#pragma unroll
      for (int c4 = 0; c4 < HD / 4; ++c4) {
        const float4 qq = *reinterpret_cast<const float4*>(&Qs[i][4 * c4]);
        const float4 gg = *reinterpret_cast<const float4*>(&Gs[i][4 * c4]);
        dv[4 * c4] = fmaf(pd, gg.x, dv[4 * c4]); dv[4 * c4 + 1] = fmaf(pd, gg.y, dv[4 * c4 + 1]);
        dv[4 * c4 + 2] = fmaf(pd, gg.z, dv[4 * c4 + 2]); dv[4 * c4 + 3] = fmaf(pd, gg.w, dv[4 * c4 + 3]);
        dk[4 * c4] = fmaf(ds, qq.x, dk[4 * c4]); dk[4 * c4 + 1] = fmaf(ds, qq.y, dk[4 * c4 + 1]);
        dk[4 * c4 + 2] = fmaf(ds, qq.z, dk[4 * c4 + 2]); dk[4 * c4 + 3] = fmaf(ds, qq.w, dk[4 * c4 + 3]);
      }
    }
  }
  if (!valid) return;
#pragma unroll
  for (int c = 0; c < HD; ++c) {
    d_qkv[(size_t)(r0 + kj) * ld + d + head * HD + c] = dk[c];        // Qs already carries the 1/sqrt(hd) factor
    d_qkv[(size_t)(r0 + kj) * ld + 2 * d + head * HD + c] = dv[c];
  }
}

// ---- host launchers ---------------------------------------------------------------------------
#define ESAT_NPL_SWITCH(d, CALL)                                                                        \
  switch ((d) / 32) {                                                                                   \
    case 1: { constexpr int NPL = 1; CALL; break; }                                                     \
    case 2: { constexpr int NPL = 2; CALL; break; }                                                     \
    case 4: { constexpr int NPL = 4; CALL; break; }                                                     \
    case 8: { constexpr int NPL = 8; CALL; break; }                                                     \
    case 12: { constexpr int NPL = 12; CALL; break; }                                                   \
    default: ADVMIL_REQUIRE(false, "esat: width %d unsupported (32, 64, 128, 256 or 384)", (int)(d)); \
  }
#define ESAT_HD_SWITCH(hd, CALL)                                                                        \
  switch (hd) {                                                                                         \
    case 4: { constexpr int HD = 4; CALL; break; }                                                      \
    case 8: { constexpr int HD = 8; CALL; break; }                                                      \
    case 16: { constexpr int HD = 16; CALL; break; }                                                    \
    case 32: { constexpr int HD = 32; CALL; break; }                                                    \
    case 48: { constexpr int HD = 48; CALL; break; }                                                    \
    case 64: { constexpr int HD = 64; CALL; break; }                                                    \
    default: ADVMIL_REQUIRE(false, "esat: head width %d unsupported (4, 8, 16, 32, 48 or 64)", (int)(hd)); \
  }

static bool npl_ok(int d) { return d % 32 == 0; }
constexpr int LN_BWD_MAX_CTAS = 592;   // 4 per SM; partial sums [ctas][k d] are folded by reduce_rows

int esat_ln_bwd_ctas(int R) { return min(LN_BWD_MAX_CTAS, cdiv(R, 8)); }

int ln_relu_mean16_fwd(const void* y_pre, const float* gamma, const float* beta, int rows, int d, float eps, const float* pe,
                       float* emb, int dt, cudaStream_t st) {
  ADVMIL_REQUIRE(rows % 16 == 0 && npl_ok(d), "ln_relu_mean16: rows %d (%%16), d %d (%%32)", rows, d);
  const int R = rows / 16;
  if (R == 0) return ADVMIL_OK;
  if (dt == ELEM_BF16) {
    ESAT_NPL_SWITCH(d, (launch_k(ln_relu_mean16_fwd_kernel<bf16, NPL>, dim3(cdiv(R, 8)), dim3(256), 0, st, (const bf16*)y_pre, gamma, beta, R, eps, pe, emb)));
  } else {
    ESAT_NPL_SWITCH(d, (launch_k(ln_relu_mean16_fwd_kernel<float, NPL>, dim3(cdiv(R, 8)), dim3(256), 0, st, (const float*)y_pre, gamma, beta, R, eps, pe, emb)));
  }
  ADVMIL_CHECK_LAUNCH();
  return ADVMIL_OK;
}

// ws >= esat_ln_bwd_ctas(R) * 3 * d floats
int ln_relu_mean16_bwd(const void* y_pre, const float* d_emb, const float* gamma, const float* beta, int rows, int d, float eps,
                       void* d_y, float* dgamma, float* dbeta, float* dbias, float* ws, int dt, cudaStream_t st) {
  ADVMIL_REQUIRE(rows % 16 == 0 && npl_ok(d), "ln_relu_mean16: rows %d (%%16), d %d (%%32)", rows, d);
  const int R = rows / 16;
  if (R == 0) return ADVMIL_OK;
  const int ctas = esat_ln_bwd_ctas(R);
  if (dt == ELEM_BF16) {
    ESAT_NPL_SWITCH(d, (launch_k(ln_relu_mean16_bwd_kernel<bf16, NPL>, dim3(ctas), dim3(256), 0, st, (const bf16*)y_pre, d_emb, gamma, beta, R, eps, (bf16*)d_y, ws)));
  } else {
    ESAT_NPL_SWITCH(d, (launch_k(ln_relu_mean16_bwd_kernel<float, NPL>, dim3(ctas), dim3(256), 0, st, (const float*)y_pre, d_emb, gamma, beta, R, eps, (float*)d_y, ws)));
  }
  ADVMIL_CHECK_LAUNCH();
  ADVMIL_TRY(reduce_rows_strided(ws, ctas, 3 * d, d, dgamma, 0, st));
  ADVMIL_TRY(reduce_rows_strided(ws + d, ctas, 3 * d, d, dbeta, 0, st));
  return reduce_rows_strided(ws + 2 * d, ctas, 3 * d, d, dbias, 0, st);
}

int add_ln_fwd(const float* a, float* b_s, const float* gamma, const float* beta, int R, int d, float eps, float* out,
               cudaStream_t st) {
  ADVMIL_REQUIRE(npl_ok(d), "add_ln: d %d (%%32)", d);
  if (R == 0) return ADVMIL_OK;
  ESAT_NPL_SWITCH(d, (launch_k(add_ln_fwd_kernel<NPL>, dim3(cdiv(R, 8)), dim3(256), 0, st, a, b_s, gamma, beta, R, eps, out)));
  ADVMIL_CHECK_LAUNCH();
  return ADVMIL_OK;
}

// ws >= esat_ln_bwd_ctas(R) * 2 * d floats
int add_ln_bwd(const float* s, const float* gamma, const float* d_out, int R, int d, float eps, float* d_s, float* dgamma,
               float* dbeta, float* ws, cudaStream_t st) {
  ADVMIL_REQUIRE(npl_ok(d), "add_ln: d %d (%%32)", d);
  if (R == 0) return ADVMIL_OK;
  const int ctas = esat_ln_bwd_ctas(R);
  ESAT_NPL_SWITCH(d, (launch_k(add_ln_bwd_kernel<NPL>, dim3(ctas), dim3(256), 0, st, s, gamma, d_out, R, eps, d_s, ws)));
  ADVMIL_CHECK_LAUNCH();
  ADVMIL_TRY(reduce_rows_strided(ws, ctas, 2 * d, d, dgamma, 0, st));
  return reduce_rows_strided(ws + d, ctas, 2 * d, d, dbeta, 0, st);
}

int add_rows(float* a, const float* b, size_t n, cudaStream_t st) {
  ADVMIL_REQUIRE(n % 4 == 0, "add_rows: n %zu (%%4)", n);
  if (n == 0) return ADVMIL_OK;
  launch_k(add_rows_kernel, dim3(cdiv(n / 4, 256)), dim3(256), 0, st, a, b, n / 4);
  ADVMIL_CHECK_LAUNCH();
  return ADVMIL_OK;
}

int sincos_pe(const int64_t* coord, const int32_t* ro, int bags, int d, const float* omega, float* pe, cudaStream_t st) {
  ADVMIL_REQUIRE(d % 4 == 0, "sincos_pe: d %d must be a multiple of 4 (model/backbone_utils.py:82)", d);
  launch_k(sincos_pe_kernel, dim3(bags), dim3(256), 0, st, coord, ro, d, omega, pe);
  ADVMIL_CHECK_LAUNCH();
  return ADVMIL_OK;
}

static AttDrop make_att_drop(const Drop& drop, const uint8_t* mask, const int64_t* mask_off, int heads) {
  AttDrop ad;
  ad.drop = drop; ad.drop.mask = nullptr; ad.mask = mask; ad.mask_off = mask_off; ad.heads = heads;
  return ad;
}

// the tf32 / bf16 modes run attention on the tcgen05 kernels when the head width allows it; the exact-fp32 mode and the
// other head widths run the FFMA kernels
static bool mha_use_tc(int precision, int hd, int d) { return precision != ADVMIL_FP32 && mha_tcgen05_supported(hd, d); }

int mha_fwd(const float* qkv, const int32_t* ro, const int32_t* ro_host, int bags, int Rtot, int d, int heads, const Drop& drop,
            const uint8_t* mask, const int64_t* mask_off, float* ctx, float* lse, int precision, cudaStream_t st) {
  ADVMIL_REQUIRE(d % heads == 0 && (!mask || mask_off), "mha: d %d / heads %d; injected masks need their offsets", d, heads);
  if (Rtot == 0) return ADVMIL_OK;
  const int hd = d / heads;
  int mx = 0;
  for (int b = 0; b < bags; ++b) mx = max(mx, ro_host[b + 1] - ro_host[b]);
  const AttDrop ad = make_att_drop(drop, mask, mask_off, heads);
  const float scale = 1.0f / sqrtf((float)hd);
  if (mha_use_tc(precision, hd, d))     // tcgen05 / TMEM / TMA kernel (esat_attn_tc.cu)
    return mha_fwd_tcgen05(qkv, ro, bags, Rtot, d, heads, mx, scale, ad, ctx, lse, st);
  ESAT_HD_SWITCH(hd, (launch_k(mha_fwd_kernel<HD>, dim3(cdiv(mx, ATT_BQ), bags, heads), dim3(ATT_BQ), 0, st, qkv, ro, d, scale, ad, ctx, lse, Rtot)));
  ADVMIL_CHECK_LAUNCH();
  return ADVMIL_OK;
}

// Dq: [heads, Rtot] scratch
int mha_bwd(const float* qkv, const float* ctx, const float* d_ctx, const float* lse, const int32_t* ro, const int32_t* ro_host,
            int bags, int Rtot, int d, int heads, const Drop& drop, const uint8_t* mask, const int64_t* mask_off, float* d_qkv,
            float* Dq, int precision, cudaStream_t st) {
  ADVMIL_REQUIRE(d % heads == 0 && (!mask || mask_off), "mha: d %d / heads %d; injected masks need their offsets", d, heads);
  if (Rtot == 0) return ADVMIL_OK;
  const int hd = d / heads;
  int mx = 0;
  for (int b = 0; b < bags; ++b) mx = max(mx, ro_host[b + 1] - ro_host[b]);
  const AttDrop ad = make_att_drop(drop, mask, mask_off, heads);
  const float scale = 1.0f / sqrtf((float)hd);
  if (mha_use_tc(precision, hd, d))     // esat_attn_bwd_tc.cu
    return mha_bwd_tcgen05(qkv, ctx, d_ctx, lse, ro, bags, Rtot, d, heads, mx, scale, ad, d_qkv, Dq, st);
  const dim3 grid(cdiv(mx, ATT_BQ), bags, heads);
  ESAT_HD_SWITCH(hd, (launch_k(mha_bwd_q_kernel<HD>, grid, dim3(ATT_BQ), 0, st, qkv, ctx, d_ctx, lse, ro, d, scale, ad, d_qkv, Dq, Rtot)));
  ADVMIL_CHECK_LAUNCH();
  ESAT_HD_SWITCH(hd, (launch_k(mha_bwd_kv_kernel<HD>, grid, dim3(ATT_BQ), 0, st, qkv, d_ctx, lse, Dq, ro, d, scale, ad, d_qkv, Rtot)));
  ADVMIL_CHECK_LAUNCH();
  return ADVMIL_OK;
}

}  // namespace advmil
