// Segmented (per-bag) kernels and row-streaming backward kernels.  HBM-bound: coalesced float4 streams,
// warp-shuffle reductions, deterministic two-level reductions (no atomics).
#include <stdarg.h>
#include <stdlib.h>
#include "stages.cuh"

namespace advmil {

// =============================================================================================
// small utilities
// =============================================================================================
__global__ void fill_zero_kernel(float* p, size_t n) {
  pdl_prologue();
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  size_t stride = (size_t)gridDim.x * blockDim.x;
  for (; i < n; i += stride) p[i] = 0.f;
}
int fill_zero(float* p, size_t n, cudaStream_t st) {
  if (n == 0) return ADVMIL_OK;
  int grid = (int)min((size_t)148 * 8, (n + 255) / 256);
  launch_k(fill_zero_kernel, dim3(grid), dim3(256), 0, st, p, n);
  ADVMIL_CHECK_LAUNCH();
  return ADVMIL_OK;
}

__global__ void cast_bf16_kernel(const float* __restrict__ in, size_t n, bf16* __restrict__ out) {
  pdl_prologue();
  size_t i = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) * 8;
  const size_t stride = (size_t)gridDim.x * blockDim.x * 8;
  for (; i < n; i += stride) {
    if (i + 7 < n) {
      const float4 a = *reinterpret_cast<const float4*>(in + i), b = *reinterpret_cast<const float4*>(in + i + 4);
      const float o[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
      stv(out + i, o);
    } else {
      for (size_t j = i; j < n; ++j) out[j] = __float2bfloat16_rn(in[j]);
    }
  }
}
int cast_f32_to_bf16(const float* in, size_t n, void* out, cudaStream_t st) {
  if (n == 0) return ADVMIL_OK;
  ADVMIL_REQUIRE((((uintptr_t)in | (uintptr_t)out) & 15) == 0, "cast_f32_to_bf16: pointers must be 16-byte aligned");
  const int grid = (int)min((size_t)148 * 16, (n / 8 + 255) / 256 + 1);
  launch_k(cast_bf16_kernel, dim3(grid), dim3(256), 0, st, in, n, (bf16*)out);
  ADVMIL_CHECK_LAUNCH();
  return ADVMIL_OK;
}

// out[c] (+)= sum_p part[p][c]; block (8 columns, 128 part lanes): one 32-byte sector per part row, every thread's
// <= 16 loads independent, grid = ceil(ncols / 8) CTAs
__global__ void __launch_bounds__(1024) reduce_rows_kernel(const float* __restrict__ part, int nparts, int width /*row stride*/,
                                                           int ncols, float* __restrict__ out, int accumulate) {
  pdl_prologue();
  __shared__ float sm[128][9];
  const int c = blockIdx.x * 8 + threadIdx.x;
  float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
  if (c < ncols) {
    int p = threadIdx.y;
    for (; p + 7 * 128 < nparts; p += 8 * 128) {     // 8 independent loads in flight
      const float v0 = part[(size_t)p * width + c], v1 = part[(size_t)(p + 128) * width + c];
      const float v2 = part[(size_t)(p + 256) * width + c], v3 = part[(size_t)(p + 384) * width + c];
      const float v4 = part[(size_t)(p + 512) * width + c], v5 = part[(size_t)(p + 640) * width + c];
      const float v6 = part[(size_t)(p + 768) * width + c], v7 = part[(size_t)(p + 896) * width + c];
      a0 += v0 + v4; a1 += v1 + v5; a2 += v2 + v6; a3 += v3 + v7;
    }
    for (; p < nparts; p += 128) a0 += part[(size_t)p * width + c];
  }
  sm[threadIdx.y][threadIdx.x] = (a0 + a1) + (a2 + a3);
  __syncthreads();
  for (int s = 64; s > 0; s >>= 1) {
    if (threadIdx.y < s) sm[threadIdx.y][threadIdx.x] += sm[threadIdx.y + s][threadIdx.x];
    __syncthreads();
  }
  if (threadIdx.y == 0 && c < ncols) out[c] = accumulate ? out[c] + sm[0][threadIdx.x] : sm[0][threadIdx.x];
}
// several column-sum reductions over the same number of partial rows in one launch
struct ReduceSeg { const float* part; int width; int ncols; float* out; int accumulate; };
struct ReduceBatch { ReduceSeg s[4]; int first_block[5]; int n; };
__global__ void __launch_bounds__(1024) reduce_rows_multi_kernel(ReduceBatch rb, int nparts) {
  pdl_prologue();
  __shared__ float sm[128][9];
  int k = 0;
  while (k + 1 < rb.n && (int)blockIdx.x >= rb.first_block[k + 1]) ++k;
  const ReduceSeg q = rb.s[k];
  const int c = (blockIdx.x - rb.first_block[k]) * 8 + threadIdx.x;
  float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
  if (c < q.ncols) {
    int p = threadIdx.y;
    for (; p + 7 * 128 < nparts; p += 8 * 128) {
      const float v0 = q.part[(size_t)p * q.width + c], v1 = q.part[(size_t)(p + 128) * q.width + c];
      const float v2 = q.part[(size_t)(p + 256) * q.width + c], v3 = q.part[(size_t)(p + 384) * q.width + c];
      const float v4 = q.part[(size_t)(p + 512) * q.width + c], v5 = q.part[(size_t)(p + 640) * q.width + c];
      const float v6 = q.part[(size_t)(p + 768) * q.width + c], v7 = q.part[(size_t)(p + 896) * q.width + c];
      a0 += v0 + v4; a1 += v1 + v5; a2 += v2 + v6; a3 += v3 + v7;
    }
    for (; p < nparts; p += 128) a0 += q.part[(size_t)p * q.width + c];
  }
  sm[threadIdx.y][threadIdx.x] = (a0 + a1) + (a2 + a3);
  __syncthreads();
  for (int s_ = 64; s_ > 0; s_ >>= 1) {
    if (threadIdx.y < s_) sm[threadIdx.y][threadIdx.x] += sm[threadIdx.y + s_][threadIdx.x];
    __syncthreads();
  }
  if (threadIdx.y == 0 && c < q.ncols) q.out[c] = q.accumulate ? q.out[c] + sm[0][threadIdx.x] : sm[0][threadIdx.x];
}
static int reduce_rows_multi(const ReduceSeg* segs, int n, int nparts, cudaStream_t st) {
  ReduceBatch rb;
  rb.n = n;
  int blocks = 0;
  for (int k = 0; k < n; ++k) { rb.s[k] = segs[k]; rb.first_block[k] = blocks; blocks += cdiv(segs[k].ncols, 8); }
  rb.first_block[n] = blocks;
  launch_k(reduce_rows_multi_kernel, dim3(blocks), dim3(dim3(8, 128)), 0, st, rb, nparts);
  ADVMIL_CHECK_LAUNCH();
  return ADVMIL_OK;
}

int reduce_rows_strided(const float* part, int nparts, int stride, int ncols, float* out, int accumulate, cudaStream_t st) {
  launch_k(reduce_rows_kernel, dim3(cdiv(ncols, 8)), dim3(dim3(8, 128)), 0, st, part, nparts, stride, ncols, out, accumulate);
  ADVMIL_CHECK_LAUNCH();
  return ADVMIL_OK;
}
int reduce_rows(const float* part, int nparts, int width, float* out, int accumulate, cudaStream_t st) {
  launch_k(reduce_rows_kernel, dim3(cdiv(width, 8)), dim3(dim3(8, 128)), 0, st, part, nparts, width, width, out, accumulate);
  ADVMIL_CHECK_LAUNCH();
  return ADVMIL_OK;
}

__global__ void splitk_reduce_kernel(const float* __restrict__ ws, int splits, size_t n, float* __restrict__ out,
                                     int accumulate) {
  pdl_prologue();
  size_t i = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) * 4;
  if (i >= n) return;
  if (i + 3 < n) {
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int z = 0; z < splits; ++z) {
      float4 v = *reinterpret_cast<const float4*>(ws + (size_t)z * n + i);
      acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
    }
    float4* o = reinterpret_cast<float4*>(out + i);
    if (accumulate) { float4 p = *o; acc.x += p.x; acc.y += p.y; acc.z += p.z; acc.w += p.w; }
    *o = acc;
  } else {
    for (; i < n; ++i) {
      float acc = 0.f;
      for (int z = 0; z < splits; ++z) acc += ws[(size_t)z * n + i];
      out[i] = accumulate ? out[i] + acc : acc;
    }
  }
}
// out[c][r] (+)= sum_z ws[z][r][c]  (ws slices are [R][Cc]; out is [Cc][R]): split-K reduce of a product computed transposed
__global__ void splitk_reduce_t_kernel(const float* __restrict__ ws, int splits, int R, int Cc, float* __restrict__ out,
                                       int accumulate) {
  pdl_prologue();
  __shared__ float t[32][33];
  const int c = blockIdx.x * 32 + threadIdx.x, r0 = blockIdx.y * 32;
  float acc[4] = {0.f, 0.f, 0.f, 0.f};
  for (int z = 0; z < splits; ++z) {
    const float* src = ws + (size_t)z * R * Cc;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int r = r0 + threadIdx.y + 8 * j;
      if (r < R && c < Cc) acc[j] += src[(size_t)r * Cc + c];
    }
  }
#pragma unroll
  for (int j = 0; j < 4; ++j) t[threadIdx.y + 8 * j][threadIdx.x] = acc[j];
  __syncthreads();
  const int orr = r0 + threadIdx.x;           // output column (= input row)
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int oc = blockIdx.x * 32 + threadIdx.y + 8 * j;   // output row (= input column)
    if (oc < Cc && orr < R) {
      float* dst = out + (size_t)oc * R + orr;
      const float v = t[threadIdx.x][threadIdx.y + 8 * j];
      *dst = accumulate ? *dst + v : v;
    }
  }
}
int splitk_reduce_t(const float* ws, int splits, int R, int Cc, float* out, int accumulate, cudaStream_t st) {
  launch_k(splitk_reduce_t_kernel, dim3(dim3(cdiv(Cc, 32), cdiv(R, 32))), dim3(dim3(32, 8)), 0, st, ws, splits, R, Cc, out, accumulate);
  ADVMIL_CHECK_LAUNCH();
  return ADVMIL_OK;
}

int splitk_reduce(const float* ws, int splits, size_t n, float* out, int accumulate, cudaStream_t st) {
  launch_k(splitk_reduce_kernel, dim3(cdiv((n + 3) / 4, 256)), dim3(256), 0, st, ws, splits, n, out, accumulate);
  ADVMIL_CHECK_LAUNCH();
  return ADVMIL_OK;
}

// out[o][c][tap] (+)= sum_z ws[z][o][tap * C + c]: the tap-major partials of a 3x3 weight gradient into the Conv2d layout
// [N1, C, 3, 3].  One block per (o, 128 channels): coalesced reads per tap, a [128][9] shared tile, coalesced writes.
__global__ void splitk_reduce_conv3_kernel(const float* __restrict__ ws, int splits, int N1, int C, float* __restrict__ out,
                                           int accumulate) {
  pdl_prologue();
  __shared__ float t[128 * 9];
  const int o = blockIdx.y, c0 = blockIdx.x * 128, c = c0 + threadIdx.x;
  const size_t n = (size_t)N1 * 9 * C;
  for (int tap = 0; tap < 9; ++tap) {
    float acc = 0.f;
    if (c < C)
      for (int z = 0; z < splits; ++z) acc += ws[(size_t)z * n + ((size_t)o * 9 + tap) * C + c];
    t[threadIdx.x * 9 + tap] = acc;
  }
  __syncthreads();
  const int nc = min(128, C - c0);
  float* dst = out + ((size_t)o * C + c0) * 9;
  for (int j = threadIdx.x; j < nc * 9; j += 128) dst[j] = accumulate ? dst[j] + t[j] : t[j];
}
int splitk_reduce_conv3(const float* ws, int splits, int N1, int C, float* out, int accumulate, cudaStream_t st) {
  launch_k(splitk_reduce_conv3_kernel, dim3(dim3(cdiv(C, 128), N1)), dim3(128), 0, st, ws, splits, N1, C, out, accumulate);
  ADVMIL_CHECK_LAUNCH();
  return ADVMIL_OK;
}

template <typename T>
__global__ void apply_dropout_kernel(const T* __restrict__ src, size_t nvec, int vec_per_row, Drop drop, T* __restrict__ dst) {
  pdl_prologue();
  constexpr int VEC = VecN<T>::N;
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (; i < nvec; i += stride) {
    float v[VEC];
    ldv(src + i * VEC, v);
    const uint32_t row = (uint32_t)(i / vec_per_row), col = (uint32_t)(i % vec_per_row) * VEC;
    if (drop.active) {
      if (drop.mask == nullptr) {
#pragma unroll
        for (int e = 0; e < VEC; e += 2) {
          const uint32_t hb = drop.bits(row, col + e);
          v[e] = (hb & 0xFFFFu) >= drop.thresh16 ? v[e] * drop.inv_keep : 0.f;
          v[e + 1] = (hb >> 16) >= drop.thresh16 ? v[e + 1] * drop.inv_keep : 0.f;
        }
      } else {
#pragma unroll
        for (int e = 0; e < VEC; ++e) v[e] = drop.keep(row, col + e) ? v[e] * drop.inv_keep : 0.f;
      }
    }
    stv(dst + i * VEC, v);
  }
}
template <typename T>
static int apply_dropout_t(const T* src, int rows, int width, const Drop& drop, T* dst, cudaStream_t st) {
  constexpr int VEC = VecN<T>::N;
  ADVMIL_REQUIRE(width % VEC == 0, "apply_dropout: width %d must be a multiple of %d", width, VEC);
  const size_t nvec = (size_t)rows * width / VEC;
  if (nvec == 0) return ADVMIL_OK;
  const int grid = (int)min((size_t)148 * 16, (nvec + 255) / 256);
  launch_k(apply_dropout_kernel<T>, dim3(grid), dim3(256), 0, st, src, nvec, width / VEC, drop, dst);
  ADVMIL_CHECK_LAUNCH();
  return ADVMIL_OK;
}
int apply_dropout(const void* src, int rows, int width, const Drop& drop, void* dst, int dt, cudaStream_t st) {
  if (dt == ELEM_BF16) return apply_dropout_t<bf16>((const bf16*)src, rows, width, drop, (bf16*)dst, st);
  return apply_dropout_t<float>((const float*)src, rows, width, drop, (float*)dst, st);
}

// =============================================================================================
// gate weight packing: Wp[abw, L] rows = (64 tanh rows | 64 sigmoid rows) per 128-block, zero padded
// =============================================================================================
__global__ void gate_pack_kernel(const float* __restrict__ Wa, const float* __restrict__ ba,
                                 const float* __restrict__ Wb, const float* __restrict__ bb, int L, int D, int abw,
                                 float* __restrict__ Wp, float* __restrict__ bp) {
  pdl_prologue();
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  size_t n = (size_t)abw * L;
  if (i < n) {
    int pr = (int)(i / L), l = (int)(i % L);
    int tile = pr >> 7, within = pr & 127;
    int j = tile * 64 + (within & 63);
    float v = 0.f;
    if (j < D) v = (within < 64) ? Wa[(size_t)j * L + l] : Wb[(size_t)j * L + l];
    Wp[i] = v;
  }
  if (i < (size_t)abw) {
    int pr = (int)i;
    int tile = pr >> 7, within = pr & 127;
    int j = tile * 64 + (within & 63);
    bp[pr] = (j < D) ? ((within < 64) ? ba[j] : bb[j]) : 0.f;
  }
}
int gate_pack_weights(const float* Wa, const float* ba, const float* Wb, const float* bb, int L, int D, float* Wp,
                      float* bp, cudaStream_t st) {
  int abw = gate_width(D);
  size_t n = (size_t)abw * L;
  launch_k(gate_pack_kernel, dim3(cdiv(n, 256)), dim3(256), 0, st, Wa, ba, Wb, bb, L, D, abw, Wp, bp);
  ADVMIL_CHECK_LAUNCH();
  return ADVMIL_OK;
}

__global__ void gate_unpack_kernel(const float* __restrict__ dWp, const float* __restrict__ dbp, int L, int D,
                                   float* __restrict__ dWa, float* __restrict__ dba, float* __restrict__ dWb,
                                   float* __restrict__ dbb, int accumulate) {
  pdl_prologue();
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  size_t n = (size_t)D * L;
  if (i < n) {
    int j = (int)(i / L), l = (int)(i % L);
    int pa = gate_col_a(j);
    float va = dWp[(size_t)pa * L + l], vb = dWp[(size_t)(pa + 64) * L + l];
    dWa[i] = accumulate ? dWa[i] + va : va;
    dWb[i] = accumulate ? dWb[i] + vb : vb;
  }
  if (i < (size_t)D) {
    int pa = gate_col_a((int)i);
    dba[i] = accumulate ? dba[i] + dbp[pa] : dbp[pa];
    dbb[i] = accumulate ? dbb[i] + dbp[pa + 64] : dbp[pa + 64];
  }
}
int gate_unpack_grads(const float* dWp, const float* dbp, int L, int D, float* dWa, float* dba, float* dWb, float* dbb,
                      int accumulate, cudaStream_t st) {
  size_t n = (size_t)D * L;
  launch_k(gate_unpack_kernel, dim3(cdiv(n, 256)), dim3(256), 0, st, dWp, dbp, L, D, dWa, dba, dWb, dbb, accumulate);
  ADVMIL_CHECK_LAUNCH();
  return ADVMIL_OK;
}

__global__ void gate_score_finish_kernel(const float* __restrict__ part, int ntiles, int rows,
                                         const float* __restrict__ bc, float* __restrict__ s) {
  pdl_prologue();
  int m = blockIdx.x * blockDim.x + threadIdx.x;
  if (m >= rows) return;
  float acc = 0.f;
  for (int t = 0; t < ntiles; ++t) acc += part[(size_t)t * rows + m];
  s[m] = acc + bc[0];
}
int gate_score_finish(const float* part, int ntiles, int rows, const float* bc, float* s, cudaStream_t st) {
  launch_k(gate_score_finish_kernel, dim3(cdiv(rows, 256)), dim3(256), 0, st, part, ntiles, rows, bc, s);
  ADVMIL_CHECK_LAUNCH();
  return ADVMIL_OK;
}

// =============================================================================================
// K3: segmented softmax + attention pooling (model/backbone.py:82-84; backbone_utils.py:53-55)
// =============================================================================================
constexpr int POOL_CH = 256;  // rows per pooling chunk (1024 CTAs at the benchmark size: ~7 per SM)

// One pass over v (online softmax): chunk c of a bag computes its own max m_c, l_c = sum exp(s - m_c) and the partial
// z_c = sum exp(s - m_c) v; the final kernel rescales by exp(m_c - M).  When `sparts` is given the logits are first
// assembled from the gate kernel's per-tile partial scores (s = sum_t sparts[t][row] + bc) and written to s.
// grid (maxchunks, bags); threads = RG row groups x WV 16-byte vectors per row
// 16-byte vector of T kept packed in four registers until it is consumed (the bf16 stream holds 4 rows = 16 registers in
// flight instead of 32 unpacked floats: the register count decides how many CTAs stream per SM)
__device__ __forceinline__ uint4 ld_raw16(const void* p) { return __ldg(reinterpret_cast<const uint4*>(p)); }
template <typename T, bool MEAN>
__device__ __forceinline__ void acc_raw(const uint4& q, float w, float (&acc)[VecN<T>::N], float (&accm)[VecN<T>::N]) {
  if constexpr (sizeof(T) == 4) {
    const float x[4] = {__uint_as_float(q.x), __uint_as_float(q.y), __uint_as_float(q.z), __uint_as_float(q.w)};
#pragma unroll
    for (int e = 0; e < 4; ++e) { acc[e] = fmaf(w, x[e], acc[e]); if (MEAN) accm[e] += x[e]; }
  } else {
    const uint32_t u[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const float lo = __uint_as_float(u[k] << 16), hi = __uint_as_float(u[k] & 0xFFFF0000u);
      acc[2 * k] = fmaf(w, lo, acc[2 * k]); acc[2 * k + 1] = fmaf(w, hi, acc[2 * k + 1]);
      if (MEAN) { accm[2 * k] += lo; accm[2 * k + 1] += hi; }
    }
  }
}

template <typename T, bool MEAN>
__global__ void __launch_bounds__(512) seg_pool_partial_kernel(
    float* __restrict__ s, const float* __restrict__ sparts, int ntiles, int rows, const float* __restrict__ bc,
    const T* __restrict__ v, const int32_t* __restrict__ offsets, int width,
    float* __restrict__ cstats /*[chunk][2] = m_c, l_c*/, float* __restrict__ part /*[offsets[b]/POOL_CH + b + chunk][width]*/,
    float* __restrict__ part_mean) {
  pdl_prologue();
  constexpr int VEC = VecN<T>::N;
  extern __shared__ float sm[];  // w_s[POOL_CH] + red[RG][width] (+ red_mean)
  __shared__ float redb[33];
  int b = blockIdx.y, chunk = blockIdx.x;
  int beg = offsets[b] + chunk * POOL_CH, end = min(offsets[b + 1], beg + POOL_CH);
  if (beg >= offsets[b + 1]) return;
  int nrows = end - beg;
  const size_t ci = (size_t)(offsets[b] / POOL_CH + b + chunk);
  float* w_s = sm;
  float mx = -INFINITY;
  for (int r = threadIdx.x; r < nrows; r += blockDim.x) {
    float sv;
    if (sparts) {
      float acc = 0.f;
      for (int t = 0; t < ntiles; ++t) acc += sparts[(size_t)t * rows + beg + r];
      sv = acc + bc[0];
      s[beg + r] = sv;
    } else {
      sv = s[beg + r];
    }
    w_s[r] = sv;
    mx = fmaxf(mx, sv);
  }
  mx = block_max(mx, redb);
  float lsum = 0.f;
  for (int r = threadIdx.x; r < nrows; r += blockDim.x) {
    const float pv = expf(w_s[r] - mx);
    w_s[r] = pv;
    lsum += pv;
  }
  lsum = block_sum(lsum, redb);   // (ends with a barrier: w_s is visible to every thread below)
  if (threadIdx.x == 0) { cstats[2 * ci] = mx; cstats[2 * ci + 1] = lsum; }
  const int WV = width / VEC;
  int RG = blockDim.x / WV; if (RG > POOL_CH) RG = POOL_CH;
  const int cv = threadIdx.x % WV, rg = threadIdx.x / WV;
  float acc[VEC], accm[VEC];
#pragma unroll
  for (int e = 0; e < VEC; ++e) { acc[e] = 0.f; accm[e] = 0.f; }
  if (rg < RG) {
    const T* vp = v + (size_t)beg * width + cv * VEC;
    int r = rg;
    for (; r + 3 * RG < nrows; r += 4 * RG) {
      const uint4 q0 = ld_raw16(vp + (size_t)r * width), q1 = ld_raw16(vp + (size_t)(r + RG) * width);
      const uint4 q2 = ld_raw16(vp + (size_t)(r + 2 * RG) * width), q3 = ld_raw16(vp + (size_t)(r + 3 * RG) * width);
      const float w0 = w_s[r], w1 = w_s[r + RG], w2 = w_s[r + 2 * RG], w3 = w_s[r + 3 * RG];
      if constexpr (sizeof(T) == 4) {      // fp32: the vectors are the floats themselves; four independent products per element
        const float x0[4] = {__uint_as_float(q0.x), __uint_as_float(q0.y), __uint_as_float(q0.z), __uint_as_float(q0.w)};
        const float x1[4] = {__uint_as_float(q1.x), __uint_as_float(q1.y), __uint_as_float(q1.z), __uint_as_float(q1.w)};
        const float x2[4] = {__uint_as_float(q2.x), __uint_as_float(q2.y), __uint_as_float(q2.z), __uint_as_float(q2.w)};
        const float x3[4] = {__uint_as_float(q3.x), __uint_as_float(q3.y), __uint_as_float(q3.z), __uint_as_float(q3.w)};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          acc[e] += w0 * x0[e] + w1 * x1[e] + w2 * x2[e] + w3 * x3[e];
          if (MEAN) accm[e] += (x0[e] + x1[e]) + (x2[e] + x3[e]);
        }
      } else {
        acc_raw<T, MEAN>(q0, w0, acc, accm); acc_raw<T, MEAN>(q1, w1, acc, accm);
        acc_raw<T, MEAN>(q2, w2, acc, accm); acc_raw<T, MEAN>(q3, w3, acc, accm);
      }
    }
    for (; r < nrows; r += RG) acc_raw<T, MEAN>(ld_raw16(vp + (size_t)r * width), w_s[r], acc, accm);
  }
  float* red = sm + POOL_CH;
  float* redm = red + (size_t)RG * width;
  if (rg < RG) {
#pragma unroll
    for (int e = 0; e < VEC; ++e) {
      red[(size_t)rg * width + cv * VEC + e] = acc[e];
      if (MEAN) redm[(size_t)rg * width + cv * VEC + e] = accm[e];
    }
  }
  __syncthreads();
  for (int c = threadIdx.x; c < width; c += blockDim.x) {
    float t = 0.f, tm = 0.f;
    for (int g = 0; g < RG; ++g) { t += red[(size_t)g * width + c]; if (MEAN) tm += redm[(size_t)g * width + c]; }
    part[ci * width + c] = t;
    if (MEAN) part_mean[ci * width + c] = tm;
  }
}

// grid (max(maxchunks, ceil(width/32)), bags), 256 threads.  Every CTA derives the bag statistics M = max m_c,
// L = sum l_c exp(m_c - M) from the chunk statistics; CTA x < #chunks writes the softmax weights of chunk x; CTA
// x < ceil(width/32) combines 32 columns of z (8 chunk groups, then a shared-memory fold).
__global__ void __launch_bounds__(256) seg_pool_final_kernel(const float* __restrict__ s, const float* __restrict__ cstats,
                                                             const float* __restrict__ part, const float* __restrict__ part_mean,
                                                             const int32_t* __restrict__ offsets, int width,
                                                             float* __restrict__ w, float* __restrict__ z, float* __restrict__ mean) {
  pdl_prologue();
  __shared__ float redb[33];
  __shared__ float sm[2][8][33];
  const int b = blockIdx.y, x = blockIdx.x;
  const int beg_bag = offsets[b], len = offsets[b + 1] - beg_bag;
  const int nch = (len + POOL_CH - 1) / POOL_CH;
  const size_t base = (size_t)(beg_bag / POOL_CH + b);
  const bool wrole = x < nch, zrole = x * 32 < width;
  if (!wrole && !zrole) return;
  float mx = -INFINITY;
  for (int c = threadIdx.x; c < nch; c += blockDim.x) mx = fmaxf(mx, cstats[2 * (base + c)]);
  mx = block_max(mx, redb);
  float L = 0.f;
  for (int c = threadIdx.x; c < nch; c += blockDim.x) L += cstats[2 * (base + c) + 1] * expf(cstats[2 * (base + c)] - mx);
  L = block_sum(L, redb);
  const float invL = 1.0f / L;
  if (wrole) {
    const int beg = beg_bag + x * POOL_CH, nrows = min(POOL_CH, len - x * POOL_CH);
    for (int r = threadIdx.x; r < nrows; r += blockDim.x) w[beg + r] = expf(s[beg + r] - mx) * invL;
  }
  if (zrole) {
    const int lane = threadIdx.x & 31, g = threadIdx.x >> 5, col = x * 32 + lane;
    float t = 0.f, tm = 0.f;
    if (col < width) {
      for (int c = g; c < nch; c += 8) {
        const float f = expf(cstats[2 * (base + c)] - mx);
        t = fmaf(part[(base + c) * width + col], f, t);
        if (mean) tm += part_mean[(base + c) * width + col];
      }
    }
    sm[0][g][lane] = t; sm[1][g][lane] = tm;
    __syncthreads();
    if (g == 0 && col < width) {
      float a = 0.f, am = 0.f;
#pragma unroll
      for (int k = 0; k < 8; ++k) { a += sm[0][k][lane]; am += sm[1][k][lane]; }
      z[(size_t)b * width + col] = a * invL;
      if (mean) mean[(size_t)b * width + col] = am / (float)len;
    }
  }
}

static int pool_maxchunks(const int32_t* offsets_host, int bags) {
  int mx = 0;
  for (int b = 0; b < bags; ++b) mx = max(mx, offsets_host[b + 1] - offsets_host[b]);
  return cdiv(mx, POOL_CH);
}
size_t seg_pool_ws_floats(int rows, int bags, int width) {
  size_t nparts = (size_t)rows / POOL_CH + bags + 1;  // sum_b ceil(len_b / POOL_CH) <= rows/POOL_CH + bags
  return align_up(2 * nparts, 64) + 2 * nparts * width;
}
template <typename T>
static int seg_softmax_pool_fwd_t(float* s, const float* sparts, int ntiles, const float* bc, const T* v, const int32_t* offsets,
                                  const int32_t* offsets_host, int rows, int bags, int width, float* w, float* z, float* mean,
                                  float* ws, cudaStream_t st) {
  constexpr int VEC = VecN<T>::N;
  ADVMIL_REQUIRE(width % VEC == 0 && width <= 1024, "seg_softmax_pool: width %d must be a multiple of %d and <= 1024", width, VEC);
  for (int b = 0; b < bags; ++b)
    ADVMIL_REQUIRE(offsets_host[b + 1] > offsets_host[b], "seg_softmax_pool: bag %d is empty", b);
  int maxchunks = pool_maxchunks(offsets_host, bags);
  const size_t nparts = (size_t)rows / POOL_CH + bags + 1;
  float* cstats = ws;
  float* part = ws + align_up(2 * nparts, 64);
  float* part_mean = part + nparts * width;
  const int WV = width / VEC;
  int threads = 256;                                   // whole row groups when the row divides a 512/384-thread block
  if ((8 * WV) % 32 == 0 && 8 * WV <= 512) threads = 8 * WV;
  else if ((4 * WV) % 32 == 0 && 4 * WV <= 512) threads = 4 * WV;
  int RG = min(threads / WV, POOL_CH);
  size_t smem = (POOL_CH + (size_t)RG * width * (mean ? 2 : 1)) * sizeof(float);
  if (mean) launch_k(seg_pool_partial_kernel<T, true>, dim3(maxchunks, bags), dim3(threads), smem, st, s, sparts, ntiles, rows, bc, v, offsets, width, cstats, part, part_mean);
  else launch_k(seg_pool_partial_kernel<T, false>, dim3(maxchunks, bags), dim3(threads), smem, st, s, sparts, ntiles, rows, bc, v, offsets, width, cstats, part, part_mean);
  ADVMIL_CHECK_LAUNCH();
  launch_k(seg_pool_final_kernel, dim3(dim3(max(maxchunks, cdiv(width, 32)), bags)), dim3(256), 0, st, s, cstats, part, mean ? part_mean : nullptr,
                                                                                     offsets, width, w, z, mean);
  ADVMIL_CHECK_LAUNCH();
  return ADVMIL_OK;
}
int seg_softmax_pool_fwd(float* s, const float* sparts, int ntiles, const float* bc, const void* v, int dt, const int32_t* offsets,
                         const int32_t* offsets_host, int rows, int bags, int width, float* w, float* z, float* mean, float* ws,
                         cudaStream_t st) {
  if (dt == ELEM_BF16)
    return seg_softmax_pool_fwd_t<bf16>(s, sparts, ntiles, bc, (const bf16*)v, offsets, offsets_host, rows, bags, width, w, z, mean, ws, st);
  return seg_softmax_pool_fwd_t<float>(s, sparts, ntiles, bc, (const float*)v, offsets, offsets_host, rows, bags, width, w, z, mean, ws, st);
}

// =============================================================================================
// backward of pooling + gated attention (SURVEY.md A.2):
//   ds_n = w_n (dz.v_n - dz.z);  du_j = ds wc_j;  da_pre = du b_d sa (1-a^2);  db_pre = du a_d sb b(1-b)
// =============================================================================================
__global__ void bag_dot_kernel(const float* __restrict__ a, const float* __restrict__ b, int width, float* __restrict__ out) {
  pdl_prologue();
  __shared__ float red[33];
  int bag = blockIdx.x;
  float acc = 0.f;
  for (int c = threadIdx.x; c < width; c += blockDim.x) acc += a[(size_t)bag * width + c] * b[(size_t)bag * width + c];
  acc = block_sum(acc, red);
  if (threadIdx.x == 0) out[bag] = acc;
}

// pass 1: ds[row] = w[row] (dz[bag] . v[row] - dz[bag] . z[bag]).  8 lanes per row (16-byte vectors interleaved across
// the 8 lanes: 128 contiguous bytes per row per load instruction), 8 rows in flight per warp, 16 rows per warp in total
template <typename T>
__global__ void __launch_bounds__(256) pool_ds_kernel(const T* __restrict__ v, const float* __restrict__ w,
                                                      const float* __restrict__ dz, const float* __restrict__ gz,
                                                      const int32_t* __restrict__ offsets, int rows, int bags, int L,
                                                      float* __restrict__ ds) {
  pdl_prologue();
  constexpr int VEC = VecN<T>::N;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int sub = lane & 7, slot = lane >> 3;
  const int row0 = blockIdx.x * ROWS_PER_CTA + wid * (ROWS_PER_CTA / 8);
  const int rend = min(rows, row0 + ROWS_PER_CTA / 8);
  if (row0 >= rend) return;
  const int bag0 = bag_of_row(offsets, bags, row0);          // one search per warp; rows are visited in order
#pragma unroll 1
  for (int rb = row0; rb < rend; rb += 8) {
    int r[2], bag[2];
    bool ok[2];
    float acc[2] = {0.f, 0.f};
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      r[u] = rb + u * 4 + slot;
      ok[u] = r[u] < rend;
      int bg = bag0;
      if (ok[u]) { while (r[u] >= offsets[bg + 1]) ++bg; }
      bag[u] = bg;
    }
    for (int c = sub * VEC; c < L; c += 8 * VEC) {
      float x[2][VEC];
#pragma unroll
      for (int u = 0; u < 2; ++u) {
#pragma unroll
        for (int e = 0; e < VEC; ++e) x[u][e] = 0.f;
        if (ok[u]) ldv(v + (size_t)r[u] * L + c, x[u]);
      }
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        const float* dzr = dz + (size_t)bag[u] * L + c;
#pragma unroll
        for (int q4 = 0; q4 < VEC / 4; ++q4) {
          const float4 g = *reinterpret_cast<const float4*>(dzr + 4 * q4);
          acc[u] += x[u][4 * q4] * g.x + x[u][4 * q4 + 1] * g.y + x[u][4 * q4 + 2] * g.z + x[u][4 * q4 + 3] * g.w;
        }
      }
    }
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      const float t = oct_sum(acc[u]);
      if (sub == 0 && ok[u]) ds[r[u]] = w[r[u]] * (t - gz[bag[u]]);
    }
  }
}

// pass 2 (pure stream): thread (rg, pv) owns VEC consecutive gate-column pairs of every RGN-th row of a 128-row chunk:
// 16-byte loads of the tanh / sigmoid vectors, 16-byte stores of dA / dB.  Also accumulates dwc and the column sums of
// dAB (the packed gate-bias gradient), so no separate pass over dAB is needed.
template <typename T>
__global__ void __launch_bounds__(256, 4) pool_gate_bwd_kernel(
    const float* __restrict__ ds_g, const T* __restrict__ ab, const float* __restrict__ wc, int rows, int D, int abw, int RGN,
    Drop da, Drop db, T* __restrict__ dAB, float* __restrict__ part /*[chunks][D+1]*/, float* __restrict__ part_b /*[chunks][abw] or null*/) {
  pdl_prologue();
  constexpr int VEC = VecN<T>::N;
  extern __shared__ float red3[];              // [RGN][3][npairs]
  __shared__ float ds_s[ROWS_PER_CTA];
  __shared__ float red[33];
  const int row0 = blockIdx.x * ROWS_PER_CTA;
  const int nrows = min(ROWS_PER_CTA, rows - row0);
  for (int r = threadIdx.x; r < nrows; r += blockDim.x) ds_s[r] = ds_g[row0 + r];
  __syncthreads();
  const int npairs = abw >> 1, TPR = npairs / VEC;
  const int rg = threadIdx.x / TPR, pv = threadIdx.x % TPR;
  if (rg < RGN) {
    const int q0 = pv * VEC, ca = gate_col_a(q0);
    float wcj[VEC], dwc[VEC], sa_sum[VEC], sb_sum[VEC];
#pragma unroll
    for (int e = 0; e < VEC; ++e) { wcj[e] = (q0 + e < D) ? wc[q0 + e] : 0.f; dwc[e] = 0.f; sa_sum[e] = 0.f; sb_sum[e] = 0.f; }
#pragma unroll 2
    for (int r = rg; r < nrows; r += RGN) {
      const size_t row = (size_t)(row0 + r);
      float a[VEC], b[VEC], oa[VEC], ob[VEC];
      ldv(ab + row * abw + ca, a);
      ldv(ab + row * abw + ca + 64, b);
      const float ds = ds_s[r];
#pragma unroll
      for (int e = 0; e < VEC; ++e) {
        const bool valid = q0 + e < D;
        // train mode: the forward stored the joint keep bit of the pair in the sign of the sigmoid
        const bool keep = (__float_as_uint(b[e]) >> 31) == 0u;
        const float sa = keep ? da.inv_keep : 0.f, sb = keep ? db.inv_keep : 0.f;
        const float av = valid ? a[e] : 0.f, bv = valid ? fabsf(b[e]) : 0.f;
        const float ad = av * sa, bd = bv * sb, du = ds * wcj[e];
        oa[e] = du * bd * sa * (1.f - av * av);
        ob[e] = du * ad * sb * bv * (1.f - bv);
        dwc[e] = fmaf(ds, ad * bd, dwc[e]);
        sa_sum[e] += oa[e]; sb_sum[e] += ob[e];
      }
      stv(dAB + row * abw + ca, oa);
      stv(dAB + row * abw + ca + 64, ob);
    }
    // element e of thread pv at [e][pv]-style offsets: consecutive lanes hit consecutive banks
#pragma unroll
    for (int e = 0; e < VEC; ++e) {
      red3[((size_t)rg * 3 + 0) * npairs + e * TPR + pv] = dwc[e];
      red3[((size_t)rg * 3 + 1) * npairs + e * TPR + pv] = sa_sum[e];
      red3[((size_t)rg * 3 + 2) * npairs + e * TPR + pv] = sb_sum[e];
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < npairs; i += blockDim.x) {   // i = e * TPR + pv  ->  pair q = pv * VEC + e
    float t0 = 0.f, t1 = 0.f, t2 = 0.f;
    for (int g = 0; g < RGN; ++g) {
      t0 += red3[((size_t)g * 3 + 0) * npairs + i]; t1 += red3[((size_t)g * 3 + 1) * npairs + i]; t2 += red3[((size_t)g * 3 + 2) * npairs + i];
    }
    const int q = (i % TPR) * VEC + i / TPR;
    const int ca = gate_col_a(q);
    if (q < D) part[(size_t)blockIdx.x * (D + 1) + q] = t0;
    if (part_b) { part_b[(size_t)blockIdx.x * abw + ca] = t1; part_b[(size_t)blockIdx.x * abw + ca + 64] = t2; }
  }
  float t = 0.f;
  for (int r = threadIdx.x; r < nrows; r += blockDim.x) t += ds_s[r];
  t = block_sum(t, red);
  if (threadIdx.x == 0) part[(size_t)blockIdx.x * (D + 1) + D] = t;
}

template <typename T>
static int pool_gate_bwd_t(const T* v, const float* w, const float* z, const float* dz, const T* ab, const float* wc,
                           const int32_t* offsets, int rows, int bags, int L, int D, const Drop& da, const Drop& db, T* dAB,
                           float* dwc, float* dbc, float* dbp, int accumulate, float* ws, cudaStream_t st) {
  constexpr int VEC = VecN<T>::N;
  ADVMIL_REQUIRE(L % VEC == 0, "pool_gate_bwd: L %d must be a multiple of %d", L, VEC);
  const int chunks = row_chunks(rows);
  const int abw = gate_width(D);
  float* gz = ws;
  float* part = ws + align_up((size_t)bags, 64);
  float* part_b = dbp ? part + align_up((size_t)chunks * (D + 1), 64) : nullptr;
  float* ds = part + align_up((size_t)chunks * (D + 1), 64) + (size_t)chunks * abw;
  launch_k(bag_dot_kernel, dim3(bags), dim3(128), 0, st, dz, z, L, gz);
  ADVMIL_CHECK_LAUNCH();
  launch_k(pool_ds_kernel<T>, dim3(chunks), dim3(256), 0, st, v, w, dz, gz, offsets, rows, bags, L, ds);
  ADVMIL_CHECK_LAUNCH();
  const int npairs = abw / 2, TPR = npairs / VEC;
  ADVMIL_REQUIRE(TPR >= 1 && TPR <= 256, "pool_gate_bwd: gate width %d unsupported", abw);
  const int RGN = max(1, min(192 / TPR, 16));
  const int threads = max(64, ((TPR * RGN + 31) / 32) * 32);
  const size_t smem = (size_t)RGN * 3 * npairs * sizeof(float);
  ADVMIL_REQUIRE(smem <= 48 * 1024, "pool_gate_bwd: gate width %d needs too much shared memory", abw);
  launch_k(pool_gate_bwd_kernel<T>, dim3(chunks), dim3(threads), smem, st, ds, ab, wc, rows, D, abw, RGN, da, db, dAB, part, part_b);
  ADVMIL_CHECK_LAUNCH();
  // dwc | dbc | packed gate-bias gradient (never accumulated: the caller unpacks it with its own accumulate flag)
  ReduceSeg segs[3] = {{part, D + 1, D, dwc, accumulate}, {part + D, D + 1, 1, dbc, accumulate}, {part_b, abw, abw, dbp, 0}};
  return reduce_rows_multi(segs, dbp ? 3 : 2, chunks, st);
}
int pool_gate_bwd(const void* v, const float* w, const float* z, const float* dz, const void* ab, const float* wc,
                  const int32_t* offsets, int rows, int bags, int L, int D, const Drop& da, const Drop& db, void* dAB,
                  float* dwc, float* dbc, float* dbp, int accumulate, float* ws, int dt, cudaStream_t st) {
  if (dt == ELEM_BF16)
    return pool_gate_bwd_t<bf16>((const bf16*)v, w, z, dz, (const bf16*)ab, wc, offsets, rows, bags, L, D, da, db, (bf16*)dAB,
                                 dwc, dbc, dbp, accumulate, ws, st);
  return pool_gate_bwd_t<float>((const float*)v, w, z, dz, (const float*)ab, wc, offsets, rows, bags, L, D, da, db,
                                (float*)dAB, dwc, dbc, dbp, accumulate, ws, st);
}

// =============================================================================================
// K5/K6 backward per row: region mean (1/16), ReLU, LayerNorm (biased variance, eps) -> d_y
// =============================================================================================
// T = element type of y_pre / d_y (fp32, or bf16 at d = 64 and 256; d = 128 has its own kernel below)
template <typename T, int VPL>  // values per lane: d <= 32*VPL
__global__ void __launch_bounds__(256) ln_pool_bwd_kernel(
    const T* __restrict__ y_pre, const float* __restrict__ d_emb, const float* __restrict__ d_emb2,
    const float* __restrict__ gamma, const float* __restrict__ beta, int rows, int d, float eps, T* __restrict__ d_y,
    float* __restrict__ part /*[chunks][3][d]*/) {
  pdl_prologue();
  extern __shared__ float sm[];  // [8 warps][3][d]
  int row0 = blockIdx.x * ROWS_PER_CTA;
  int nrows = min(ROWS_PER_CTA, rows - row0);
  int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  float g[VPL], be[VPL], pg[VPL], pb[VPL], pbias[VPL];
#pragma unroll
  for (int k = 0; k < VPL; ++k) {
    int c = lane + 32 * k;
    g[k] = c < d ? gamma[c] : 0.f;
    be[k] = c < d ? beta[c] : 0.f;
    pg[k] = pb[k] = pbias[k] = 0.f;
  }
  const float inv_d = 1.0f / (float)d;
  for (int r = wid; r < nrows; r += 8) {
    size_t row = (size_t)(row0 + r);
    float y[VPL];
    float s = 0.f;
#pragma unroll
    for (int k = 0; k < VPL; ++k) { int c = lane + 32 * k; y[k] = c < d ? ld1(y_pre + row * d + c) : 0.f; s += y[k]; }
    float mean = warp_sum(s) * inv_d;
    float q = 0.f;
#pragma unroll
    for (int k = 0; k < VPL; ++k) { int c = lane + 32 * k; float cc = c < d ? y[k] - mean : 0.f; q = fmaf(cc, cc, q); }
    float rstd = rsqrtf(warp_sum(q) * inv_d + eps);
    float xh[VPL], dxh[VPL];
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int k = 0; k < VPL; ++k) {
      int c = lane + 32 * k;
      xh[k] = 0.f; dxh[k] = 0.f;
      if (c < d) {
        xh[k] = (y[k] - mean) * rstd;
        float e = fmaf(xh[k], g[k], be[k]);
        float de = e > 0.f ? (d_emb[(row >> 4) * d + c] + (d_emb2 ? d_emb2[(row >> 4) * d + c] : 0.f)) * (1.0f / 16.0f) : 0.f;
        pg[k] = fmaf(de, xh[k], pg[k]);
        pb[k] += de;
        dxh[k] = de * g[k];
        s1 += dxh[k];
        s2 = fmaf(dxh[k], xh[k], s2);
      }
    }
    float m1 = warp_sum(s1) * inv_d, m2 = warp_sum(s2) * inv_d;
#pragma unroll
    for (int k = 0; k < VPL; ++k) {
      int c = lane + 32 * k;
      if (c < d) {
        float dy = rstd * (dxh[k] - m1 - xh[k] * m2);
        st1(d_y + row * d + c, dy);
        pbias[k] += dy;
      }
    }
  }
#pragma unroll
  for (int k = 0; k < VPL; ++k) {
    int c = lane + 32 * k;
    if (c < d) {
      sm[(wid * 3 + 0) * d + c] = pg[k];
      sm[(wid * 3 + 1) * d + c] = pb[k];
      sm[(wid * 3 + 2) * d + c] = pbias[k];
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 3 * d; i += blockDim.x) {
    float t = 0.f;
#pragma unroll
    for (int wv = 0; wv < 8; ++wv) t += sm[wv * 3 * d + i];
    part[(size_t)blockIdx.x * 3 * d + i] = t;
  }
}

// d == 128: 16 lanes per row (8 columns per lane as 16-byte vectors interleaved across the 16 lanes, so every load
// instruction covers 256 contiguous bytes per row), 2 rows per warp and 4 such pairs in flight: 8 rows = half a region
// per warp iteration; 24 partial-sum registers per lane keep the occupancy at 4+ CTAs per SM
template <typename T, int OCC>
__global__ void __launch_bounds__(128, OCC) ln_pool_bwd128_kernel(
    const T* __restrict__ y_pre, const float* __restrict__ d_emb, const float* __restrict__ d_emb2,
    const float* __restrict__ gamma, const float* __restrict__ beta, int rows, float eps, T* __restrict__ d_y,
    float* __restrict__ part) {
  pdl_prologue();
  constexpr int VEC = VecN<T>::N, NV = 8 / VEC;           // vectors per lane (2 for fp32, 1 for bf16)
  __shared__ float sm[4 * 3 * 128];
  const int row0 = blockIdx.x * ROWS_PER_CTA;
  const int nrows = min(ROWS_PER_CTA, rows - row0);
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int sub = lane & 15, slot = lane >> 4;            // column group, row slot within the warp
  // column of element (k, e): k * 16 * VEC + sub * VEC + e
  float g[8], be[8], pg[8], pb[8], pbias[8];
#pragma unroll
  for (int k = 0; k < NV; ++k)
#pragma unroll
    for (int e = 0; e < VEC; ++e) {
      const int c = k * 16 * VEC + sub * VEC + e, i = k * VEC + e;
      g[i] = gamma[c]; be[i] = beta[c]; pg[i] = 0.f; pb[i] = 0.f; pbias[i] = 0.f;
    }
  for (int rb = wid * 8; rb < nrows; rb += 32) {
    // rb is a multiple of 8: the 8 rows of this warp iteration lie in ONE 16-row region
    float ge[8];
#pragma unroll
    for (int k = 0; k < NV; ++k)
#pragma unroll
      for (int q4 = 0; q4 < VEC / 4; ++q4) {
        const size_t go = ((size_t)(row0 + rb) >> 4) * 128 + k * 16 * VEC + sub * VEC + 4 * q4;
        float4 d4 = *reinterpret_cast<const float4*>(d_emb + go);
        if (d_emb2) { const float4 e4 = *reinterpret_cast<const float4*>(d_emb2 + go); d4.x += e4.x; d4.y += e4.y; d4.z += e4.z; d4.w += e4.w; }
        const int i = k * VEC + 4 * q4;
        ge[i] = d4.x * 0.0625f; ge[i + 1] = d4.y * 0.0625f; ge[i + 2] = d4.z * 0.0625f; ge[i + 3] = d4.w * 0.0625f;
      }
    float y[4][8];
    bool ok[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int r = rb + u * 2 + slot;
      ok[u] = r < nrows;
      const size_t row = (size_t)(row0 + r);
#pragma unroll
      for (int k = 0; k < NV; ++k) {
        float t[VEC];
#pragma unroll
        for (int e = 0; e < VEC; ++e) t[e] = 0.f;
        if (ok[u]) ldv(y_pre + row * 128 + k * 16 * VEC + sub * VEC, t);
#pragma unroll
        for (int e = 0; e < VEC; ++e) y[u][k * VEC + e] = t[e];
      }
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const size_t row = (size_t)(row0 + rb + u * 2 + slot);
      float sacc = 0.f;
#pragma unroll
      for (int i = 0; i < 8; ++i) sacc += y[u][i];
      const float mean = half_warp_sum(sacc) * (1.0f / 128.0f);
      float q = 0.f;
#pragma unroll
      for (int i = 0; i < 8; ++i) { const float c = y[u][i] - mean; q = fmaf(c, c, q); }
      const float rstd = rsqrtf(half_warp_sum(q) * (1.0f / 128.0f) + eps);
      float xh[8], dxh[8], s1 = 0.f, s2 = 0.f;
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        xh[i] = (y[u][i] - mean) * rstd;
        const float e = fmaf(xh[i], g[i], be[i]);
        const float de = (e > 0.f && ok[u]) ? ge[i] : 0.f;
        pg[i] = fmaf(de, xh[i], pg[i]);
        pb[i] += de;
        dxh[i] = de * g[i];
        s1 += dxh[i];
        s2 = fmaf(dxh[i], xh[i], s2);
      }
      const float m1 = half_warp_sum(s1) * (1.0f / 128.0f), m2 = half_warp_sum(s2) * (1.0f / 128.0f);
      float dy[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) { dy[i] = rstd * (dxh[i] - m1 - xh[i] * m2); if (ok[u]) pbias[i] += dy[i]; }
      if (ok[u]) {
#pragma unroll
        for (int k = 0; k < NV; ++k) {
          float t[VEC];
#pragma unroll
          for (int e = 0; e < VEC; ++e) t[e] = dy[k * VEC + e];
          stv(d_y + row * 128 + k * 16 * VEC + sub * VEC, t);
        }
      }
    }
  }
  // fold the 2 row slots of the warp, then the 4 warps
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    pg[i] += __shfl_xor_sync(0xffffffffu, pg[i], 16);
    pb[i] += __shfl_xor_sync(0xffffffffu, pb[i], 16);
    pbias[i] += __shfl_xor_sync(0xffffffffu, pbias[i], 16);
  }
  if (slot == 0) {
#pragma unroll
    for (int k = 0; k < NV; ++k)
#pragma unroll
      for (int e = 0; e < VEC; ++e) {
        const int c = k * 16 * VEC + sub * VEC + e, i = k * VEC + e;
        sm[(wid * 3 + 0) * 128 + c] = pg[i];
        sm[(wid * 3 + 1) * 128 + c] = pb[i];
        sm[(wid * 3 + 2) * 128 + c] = pbias[i];
      }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 3 * 128; i += blockDim.x) {
    float t = 0.f;
#pragma unroll
    for (int wv = 0; wv < 4; ++wv) t += sm[wv * 3 * 128 + i];
    part[(size_t)blockIdx.x * 3 * 128 + i] = t;
  }
}

int ln_pool_bwd(const void* y_pre, const float* d_emb, const float* d_emb2, const float* gamma, const float* beta, int rows,
                int d, float eps, void* d_y, float* dgamma, float* dbeta, float* dbias, int accumulate, float* ws, int dt,
                cudaStream_t st) {
  ADVMIL_REQUIRE(d <= 256, "ln_pool_bwd: d %d > 256 unsupported", d);
  ADVMIL_REQUIRE(dt == ELEM_F32 || d == 64 || d == 128 || d == 256, "ln_pool_bwd: the bf16 mode supports d = 64, 128 and 256 only (d=%d)", d);
  int chunks = row_chunks(rows);
  size_t smem = (size_t)8 * 3 * d * sizeof(float);
  if (d == 128 && dt == ELEM_BF16)      // 96 registers (32 bytes of spills), 5 CTAs per SM: 58 -> 56 us
    launch_k(ln_pool_bwd128_kernel<bf16, 5>, dim3(chunks), dim3(128), 0, st, (const bf16*)y_pre, d_emb, d_emb2, gamma, beta, rows, eps, (bf16*)d_y, ws);
  else if (d == 128)
    launch_k(ln_pool_bwd128_kernel<float, 4>, dim3(chunks), dim3(128), 0, st, (const float*)y_pre, d_emb, d_emb2, gamma, beta, rows, eps, (float*)d_y, ws);
  else if (dt == ELEM_BF16 && d == 64)
    launch_k(ln_pool_bwd_kernel<bf16, 2>, dim3(chunks), dim3(256), smem, st, (const bf16*)y_pre, d_emb, d_emb2, gamma, beta, rows, d, eps, (bf16*)d_y, ws);
  else if (dt == ELEM_BF16)
    launch_k(ln_pool_bwd_kernel<bf16, 8>, dim3(chunks), dim3(256), smem, st, (const bf16*)y_pre, d_emb, d_emb2, gamma, beta, rows, d, eps, (bf16*)d_y, ws);
  else if (d <= 128) launch_k(ln_pool_bwd_kernel<float, 4>, dim3(chunks), dim3(256), smem, st, (const float*)y_pre, d_emb, d_emb2, gamma, beta, rows, d, eps, (float*)d_y, ws);
  else launch_k(ln_pool_bwd_kernel<float, 8>, dim3(chunks), dim3(256), smem, st, (const float*)y_pre, d_emb, d_emb2, gamma, beta, rows, d, eps, (float*)d_y, ws);
  ADVMIL_CHECK_LAUNCH();
  ReduceSeg segs[3] = {{ws, 3 * d, d, dgamma, accumulate}, {ws + d, 3 * d, d, dbeta, accumulate}, {ws + 2 * d, 3 * d, d, dbias, accumulate}};
  return reduce_rows_multi(segs, 3, chunks, st);
}

// =============================================================================================
// column sums (bias gradients): each thread owns 4 / sizeof(T) ... one 4-byte word of every row = 1 fp32 or 2 bf16 columns
// =============================================================================================
// 1024 threads = 4 row groups x 256 column threads: a 128-row chunk is summed by four groups of 32 rows and folded through
// shared memory (one partial row per chunk, as before).  With one group per chunk the region-level calls (rows / 16 = 16384
// rows -> 128 CTAs of 8 warps) left most of the chip idle: 36 us for 25 MB.
constexpr int COLSUM_GROUPS = 4;
template <typename T>
__global__ void __launch_bounds__(256 * COLSUM_GROUPS) colsum_partial_kernel(const T* __restrict__ dY, int rows, int N, int ld,
                                                                             float* __restrict__ part) {
  pdl_prologue();
  constexpr int CPT = 4 / (int)sizeof(T);
  extern __shared__ float cs_sm[];                       // [COLSUM_GROUPS][N]
  const int tc = threadIdx.x & 255, tg = threadIdx.x >> 8;
  const int row0 = blockIdx.x * ROWS_PER_CTA;
  const int nrows = min(ROWS_PER_CTA, rows - row0);
  constexpr int RPG = ROWS_PER_CTA / COLSUM_GROUPS;
  const int rbeg = tg * RPG, rend = min(nrows, rbeg + RPG);
  for (int c = tc * CPT; c < N; c += 256 * CPT) {
    const T* p = dY + (size_t)row0 * ld + c;
    float a[4][CPT];
#pragma unroll
    for (int u = 0; u < 4; ++u)
#pragma unroll
      for (int e = 0; e < CPT; ++e) a[u][e] = 0.f;
    int r = rbeg;
    for (; r + 3 < rend; r += 4) {
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        float t[CPT];
        ldw(p + (size_t)(r + u) * ld, t);
#pragma unroll
        for (int e = 0; e < CPT; ++e) a[u][e] += t[e];
      }
    }
    for (; r < rend; ++r) {
      float t[CPT];
      ldw(p + (size_t)r * ld, t);
#pragma unroll
      for (int e = 0; e < CPT; ++e) a[0][e] += t[e];
    }
#pragma unroll
    for (int e = 0; e < CPT; ++e) cs_sm[tg * N + c + e] = (a[0][e] + a[1][e]) + (a[2][e] + a[3][e]);
  }
  __syncthreads();
  for (int c = threadIdx.x; c < N; c += blockDim.x) {
    float t = 0.f;
#pragma unroll
    for (int g = 0; g < COLSUM_GROUPS; ++g) t += cs_sm[g * N + c];
    part[(size_t)blockIdx.x * N + c] = t;
  }
}
int colsum(const void* dY, int dt, int rows, int N, int ld, float* out, int accumulate, float* ws, cudaStream_t st) {
  int chunks = row_chunks(rows);
  const size_t smem = (size_t)COLSUM_GROUPS * N * sizeof(float);
  ADVMIL_REQUIRE(smem <= 48 * 1024, "colsum: N=%d too wide", N);
  if (dt == ELEM_BF16) {
    ADVMIL_REQUIRE(N % 2 == 0 && ld % 2 == 0, "colsum: bf16 needs even N (%d) and ld (%d)", N, ld);
    launch_k(colsum_partial_kernel<bf16>, dim3(chunks), dim3(256 * COLSUM_GROUPS), smem, st, (const bf16*)dY, rows, N, ld, ws);
  } else {
    launch_k(colsum_partial_kernel<float>, dim3(chunks), dim3(256 * COLSUM_GROUPS), smem, st, (const float*)dY, rows, N, ld, ws);
  }
  ADVMIL_CHECK_LAUNCH();
  return reduce_rows(ws, chunks, N, out, accumulate, st);
}

}  // namespace advmil
