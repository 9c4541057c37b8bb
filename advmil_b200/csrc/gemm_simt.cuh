// fp32 FFMA tile GEMM with pluggable epilogues (exact-fp32 engine; also serves the small region-level and
// head contractions in every precision mode).  C[M,N] = sum_k A(m,k) * B(k,n).
//   A_KC: A(m,k) = A[m*lda + k]   (activations [rows,K])        else A(m,k) = A[k*lda + m]  (dY^T for weight grads)
//   B_KC: B(k,n) = B[n*ldb + k]   (weights W[N,K], y = x W^T)   else B(k,n) = B[k*ldb + n]  (dX = dY W, dW = dY^T X)
// CTA tile 128x128x16, 256 threads, 8x8 outputs per thread: rows ty*8+i, columns tx*4+j and 64+tx*4+j.
// Requirements: pointers 16-byte aligned, lda/ldb multiples of 4, the contiguous extent (K or M/N) multiple of 4.
#pragma once
#include "common.cuh"

namespace advmil {

constexpr int BM = 128, BN = 128, BK = 16, GEMM_THREADS = 256;

struct GemmArgs {
  const float* A;
  const float* B;
  int M, N, K;
  int lda, ldb;
  int kchunk;  // K range per blockIdx.z (split-K); == K when grid.z == 1
};

template <bool KC>
struct TileLoader {
  // loads this thread's two float4 of a [128 (mn) x 16 (k)] tile into v[2], zero-filling out of range
  __device__ __forceinline__ static void load(const float* __restrict__ P, int ld, int mn0, int MN, int k0, int kend,
                                              int t, float4 (&v)[2]) {
    if (KC) {
#pragma unroll
      for (int i = 0; i < 2; ++i) {
        int mn = mn0 + (t >> 2) + 64 * i;
        int k = k0 + (t & 3) * 4;
        float4 r = make_float4(0.f, 0.f, 0.f, 0.f);
        if (mn < MN && k < kend) {
          const float* src = P + (size_t)mn * ld + k;
          if (k + 3 < kend) r = *reinterpret_cast<const float4*>(src);
          else { r.x = src[0]; if (k + 1 < kend) r.y = src[1]; if (k + 2 < kend) r.z = src[2]; }
        }
        v[i] = r;
      }
    } else {
#pragma unroll
      for (int i = 0; i < 2; ++i) {
        int k = k0 + (t >> 5) + 8 * i;
        int mn = mn0 + (t & 31) * 4;
        float4 r = make_float4(0.f, 0.f, 0.f, 0.f);
        if (k < kend && mn < MN) {
          const float* src = P + (size_t)k * ld + mn;
          if (mn + 3 < MN) r = *reinterpret_cast<const float4*>(src);
          else { r.x = src[0]; if (mn + 1 < MN) r.y = src[1]; if (mn + 2 < MN) r.z = src[2]; }
        }
        v[i] = r;
      }
    }
  }
  __device__ __forceinline__ static void store(float (*S)[BM + 4], int t, const float4 (&v)[2]) {
    if (KC) {
#pragma unroll
      for (int i = 0; i < 2; ++i) {
        int mn = (t >> 2) + 64 * i;
        int k = (t & 3) * 4;
        S[k + 0][mn] = v[i].x; S[k + 1][mn] = v[i].y; S[k + 2][mn] = v[i].z; S[k + 3][mn] = v[i].w;
      }
    } else {
#pragma unroll
      for (int i = 0; i < 2; ++i) {
        int k = (t >> 5) + 8 * i;
        int mn = (t & 31) * 4;
        *reinterpret_cast<float4*>(&S[k][mn]) = v[i];
      }
    }
  }
};

// Implicit-GEMM loaders of the 3x3 convolution inside every 4x4 region of 16 rows (row 16r + 4i + j = grid cell (i, j) of
// region r), for x [rows, C] with ld == C and a tap-major K or N index tap * C + c (tap = 3 kh + kw).  The row read for
// row m and tap is m's neighbour at (i + kh - 1, j + kw - 1), or zero outside the grid: no im2col copy of x.  C % 16 == 0,
// so a BK = 16 block or a float4 never spans two taps.
__device__ __forceinline__ int conv3_src_row(int m, int tap) {
  const int di = tap / 3 - 1, dj = tap % 3 - 1, i = ((m >> 2) & 3) + di, j = (m & 3) + dj;
  return ((unsigned)i < 4u && (unsigned)j < 4u) ? m + 4 * di + dj : -1;
}
// A(m, k) = x[nbr(m, tap)][c], k = tap * C + c   (the forward's activation operand, K-contiguous like TileLoader<true>)
struct Conv3LoaderA : TileLoader<true> {
  __device__ __forceinline__ static void load(const float* __restrict__ P, int ld, int mn0, int MN, int k0, int kend,
                                              int t, float4 (&v)[2]) {
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      const int mn = mn0 + (t >> 2) + 64 * i, k = k0 + (t & 3) * 4;
      const int tap = k / ld, src = (mn < MN && k < kend) ? conv3_src_row(mn, tap) : -1;
      v[i] = src >= 0 ? *reinterpret_cast<const float4*>(P + (size_t)src * ld + (k - tap * ld)) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
  }
};
// B(k, n) = x[nbr(k, tap)][c], n = tap * C + c   (the weight gradient's X operand, N-contiguous like TileLoader<false>)
struct Conv3LoaderB : TileLoader<false> {
  __device__ __forceinline__ static void load(const float* __restrict__ P, int ld, int mn0, int MN, int k0, int kend,
                                              int t, float4 (&v)[2]) {
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      const int k = k0 + (t >> 5) + 8 * i, mn = mn0 + (t & 31) * 4;
      const int tap = mn / ld, src = (k < kend && mn < MN) ? conv3_src_row(k, tap) : -1;
      v[i] = src >= 0 ? *reinterpret_cast<const float4*>(P + (size_t)src * ld + (mn - tap * ld)) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
  }
};

template <bool A_KC, bool B_KC, class Epi, class LA = TileLoader<A_KC>, class LB = TileLoader<B_KC>>
__global__ void __launch_bounds__(GEMM_THREADS) gemm_simt_kernel(GemmArgs g, Epi epi) {
  pdl_prologue();
  __shared__ __align__(16) float As[2][BK][BM + 4];
  __shared__ __align__(16) float Bs[2][BK][BN + 4];
  const int t = threadIdx.x;
  const int tx = t & 15, ty = t >> 4;
  const int m0 = blockIdx.x * BM, n0 = blockIdx.y * BN;
  const int kbeg = blockIdx.z * g.kchunk;
  const int kend = min(g.K, kbeg + g.kchunk);

  float acc[8][8];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;

  float4 ra[2], rb[2];
  LA::load(g.A, g.lda, m0, g.M, kbeg, kend, t, ra);
  LB::load(g.B, g.ldb, n0, g.N, kbeg, kend, t, rb);
  LA::store(As[0], t, ra);
  LB::store(Bs[0], t, rb);
  __syncthreads();

  int buf = 0;
  for (int k0 = kbeg; k0 < kend; k0 += BK) {
    const bool more = (k0 + BK) < kend;
    if (more) {
      LA::load(g.A, g.lda, m0, g.M, k0 + BK, kend, t, ra);
      LB::load(g.B, g.ldb, n0, g.N, k0 + BK, kend, t, rb);
    }
#pragma unroll
    for (int kk = 0; kk < BK; ++kk) {
      float4 a0 = *reinterpret_cast<const float4*>(&As[buf][kk][ty * 8]);
      float4 a1 = *reinterpret_cast<const float4*>(&As[buf][kk][ty * 8 + 4]);
      float4 b0 = *reinterpret_cast<const float4*>(&Bs[buf][kk][tx * 4]);
      float4 b1 = *reinterpret_cast<const float4*>(&Bs[buf][kk][64 + tx * 4]);
      float a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
      float b[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    if (more) {
      LA::store(As[buf ^ 1], t, ra);
      LB::store(Bs[buf ^ 1], t, rb);
    }
    __syncthreads();
    buf ^= 1;
  }
  epi(acc, m0 + ty * 8, n0, tx, g.M, g.N);
}

// column owned by (tx, j): j<4 -> n0 + tx*4 + j ; j>=4 -> n0 + 64 + tx*4 + (j-4)
__device__ __forceinline__ int epi_col(int n0, int tx, int j) { return n0 + ((j >> 2) << 6) + tx * 4 + (j & 3); }

// ---- epilogues --------------------------------------------------------------------------------
// y = act(acc + bias) * dropout
struct EpiLinear {
  float* out; int ldo;
  const float* bias;
  int relu;
  Drop drop;
  int drop_width;  // logical row width of the dropout mask index (== N)
  __device__ __forceinline__ void operator()(float (&acc)[8][8], int mrow0, int n0, int tx, int M, int N) const {
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      int m = mrow0 + i;
      if (m >= M) continue;
#pragma unroll
      for (int jh = 0; jh < 2; ++jh) {
        int n = epi_col(n0, tx, jh * 4);
        if (n >= N) continue;
        float v[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          float val = acc[i][jh * 4 + j];
          if (n + j < N) {
            if (bias) val += bias[n + j];
            if (relu) val = fmaxf(val, 0.f);
            val *= drop.scale(m, n + j);
          }
          v[j] = val;
        }
        float* dst = out + (size_t)m * ldo + n;
        if (n + 3 < N) *reinterpret_cast<float4*>(dst) = make_float4(v[0], v[1], v[2], v[3]);
        else for (int j = 0; j < 4 && n + j < N; ++j) dst[j] = v[j];
      }
    }
  }
};

// gated attention: packed weights (tanh block | sigmoid block per 128 columns); writes undropped activations
// (optional) and the partial score of this column tile: part[tile][m] = sum_j a_j b_j wc_j
struct EpiGate {
  float* ab; int ld_ab;       // [M, Npacked] or nullptr
  const float* bias_packed;   // [Npacked]
  const float* wc;            // [D]
  float* part;                // [ntiles, M]
  int D;
  Drop drop_a, drop_b;
  __device__ __forceinline__ void operator()(float (&acc)[8][8], int mrow0, int n0, int tx, int M, int N) const {
    const int tile = n0 >> 7;
    const int j0 = tile * 64 + tx * 4;  // logical gate column of acc[.][0]
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      int m = mrow0 + i;
      float partial = 0.f;
      float av[4], bv[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        float a = tanhf(acc[i][j] + bias_packed[n0 + tx * 4 + j]);
        float b = sigmoidf_(acc[i][4 + j] + bias_packed[n0 + 64 + tx * 4 + j]);
        av[j] = a; bv[j] = b;
        int jj = j0 + j;
        if (jj < D && m < M) {
          float ad = a, bd = b;
          if (drop_a.active) {
            bool ka, kb;
            gate_keep(drop_a, drop_b, m, jj, ka, kb);
            ad = ka ? a * drop_a.inv_keep : 0.f;
            bd = kb ? b * drop_b.inv_keep : 0.f;
            if (!(ka && kb)) bv[j] = -b;      // joint keep bit in the sign of the stored sigmoid (see gemm_tc.cu)
          }
          partial = fmaf(ad * bd, wc[jj], partial);
        }
      }
      partial = half_warp_sum(partial);
      if (m < M) {
        if (ab) {
          *reinterpret_cast<float4*>(ab + (size_t)m * ld_ab + n0 + tx * 4) = make_float4(av[0], av[1], av[2], av[3]);
          *reinterpret_cast<float4*>(ab + (size_t)m * ld_ab + n0 + 64 + tx * 4) = make_float4(bv[0], bv[1], bv[2], bv[3]);
        }
        if (tx == 0) part[(size_t)tile * M + m] = partial;
      }
    }
  }
};

// K5+K6: LayerNorm over the d (<=128) columns of the tile, ReLU, mean over the 16 rows of each region.
// Thread rows ty*8..+7: region q of the tile = rows 16q..16q+15 = the two half-warps of warp q.
struct EpiLNPool {
  float* y_pre; // [M,d] or nullptr
  float* emb;   // [M/16,d]
  const float* bias; const float* gamma; const float* beta;
  int d; float eps;
  __device__ __forceinline__ void operator()(float (&acc)[8][8], int mrow0, int n0, int tx, int M, int N) const {
    float colsum[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) colsum[j] = 0.f;
    float bj[8], gj[8], bej[8];
    int cols[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      cols[j] = epi_col(n0, tx, j);
      bool ok = cols[j] < d;
      bj[j] = ok ? bias[cols[j]] : 0.f;
      gj[j] = ok ? gamma[cols[j]] : 0.f;
      bej[j] = ok ? beta[cols[j]] : 0.f;
    }
    const float inv_d = 1.0f / (float)d;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      int m = mrow0 + i;
      float y[8];
      float s = 0.f;
#pragma unroll
      for (int j = 0; j < 8; ++j) { y[j] = (cols[j] < d) ? acc[i][j] + bj[j] : 0.f; s += y[j]; }
      float mean = half_warp_sum(s) * inv_d;
      float q = 0.f;
#pragma unroll
      for (int j = 0; j < 8; ++j) { float c = (cols[j] < d) ? y[j] - mean : 0.f; q = fmaf(c, c, q); }
      float rstd = rsqrtf(half_warp_sum(q) * inv_d + eps);
      if (m < M) {
        if (y_pre) {
#pragma unroll
          for (int jh = 0; jh < 2; ++jh) {
            int n = cols[jh * 4];
            float* dst = y_pre + (size_t)m * d + n;
            if (n + 3 < d) *reinterpret_cast<float4*>(dst) = make_float4(y[jh * 4], y[jh * 4 + 1], y[jh * 4 + 2], y[jh * 4 + 3]);
            else for (int j = 0; j < 4 && n + j < d; ++j) dst[j] = y[jh * 4 + j];
          }
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) colsum[j] += fmaxf(fmaf((y[j] - mean) * rstd, gj[j], bej[j]), 0.f);
      }
    }
    // combine the two half-warps (rows 16q..16q+7 and 16q+8..16q+15)
#pragma unroll
    for (int j = 0; j < 8; ++j) colsum[j] += __shfl_xor_sync(0xffffffffu, colsum[j], 16);
    int region_row0 = mrow0 & ~15;
    if ((threadIdx.x & 16) == 0 && region_row0 < M) {
      float* dst = emb + (size_t)(region_row0 >> 4) * d;
#pragma unroll
      for (int j = 0; j < 8; ++j) if (cols[j] < d) dst[cols[j]] = colsum[j] * (1.0f / 16.0f);
    }
  }
};

// backward-data epilogue: dX = (acc + w[m]*dz[bag,n] + invn[bag]*dmean[bag,n]) * relu'(src) [+ dX]
struct EpiBwdData {
  float* out; int ldo;
  const float* w;       // [M] or nullptr     (softmax weights)
  const float* dz;      // [bags,N] or nullptr
  const float* dmean;   // [bags,N] or nullptr (gradient of the plain per-bag mean)
  const int32_t* offsets; int bags;
  const float* relu_src; int ld_src;  // forward output (post relu/dropout) or nullptr
  float inv_keep;
  int accumulate;
  __device__ __forceinline__ void operator()(float (&acc)[8][8], int mrow0, int n0, int tx, int M, int N) const {
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      int m = mrow0 + i;
      if (m >= M) continue;
      int bag = 0; float wm = 0.f, invn = 0.f;
      if (dz || dmean) {
        bag = bag_of_row(offsets, bags, m);
        if (w) wm = w[m];
        if (dmean) invn = 1.0f / (float)(offsets[bag + 1] - offsets[bag]);
      }
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        int n = epi_col(n0, tx, j);
        if (n >= N) continue;
        float v = acc[i][j];
        if (dz) v = fmaf(wm, dz[(size_t)bag * N + n], v);
        if (dmean) v = fmaf(invn, dmean[(size_t)bag * N + n], v);
        if (relu_src) v = (relu_src[(size_t)m * ld_src + n] > 0.f) ? v * inv_keep : 0.f;
        float* dst = out + (size_t)m * ldo + n;
        *dst = accumulate ? (*dst + v) : v;
      }
    }
  }
};

// split-K partial tile store: ws[z][M][N]
struct EpiPartial {
  float* ws;
  __device__ __forceinline__ void operator()(float (&acc)[8][8], int mrow0, int n0, int tx, int M, int N) const {
    float* base = ws + (size_t)blockIdx.z * M * N;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      int m = mrow0 + i;
      if (m >= M) continue;
#pragma unroll
      for (int jh = 0; jh < 2; ++jh) {
        int n = epi_col(n0, tx, jh * 4);
        if (n >= N) continue;
        float* dst = base + (size_t)m * N + n;
        if (n + 3 < N) *reinterpret_cast<float4*>(dst) = make_float4(acc[i][jh * 4], acc[i][jh * 4 + 1], acc[i][jh * 4 + 2], acc[i][jh * 4 + 3]);
        else for (int j = 0; j < 4 && n + j < N; ++j) dst[j] = acc[i][jh * 4 + j];
      }
    }
  }
};

template <bool A_KC, bool B_KC, class Epi, class LA = TileLoader<A_KC>, class LB = TileLoader<B_KC>>
inline int launch_gemm(const GemmArgs& g, const Epi& epi, int splits, cudaStream_t st) {
  dim3 grid(cdiv(g.M, BM), cdiv(g.N, BN), splits);
  launch_k(gemm_simt_kernel<A_KC, B_KC, Epi, LA, LB>, dim3(grid), dim3(GEMM_THREADS), 0, st, g, epi);
  ADVMIL_CHECK_LAUNCH();
  return ADVMIL_OK;
}

}  // namespace advmil
