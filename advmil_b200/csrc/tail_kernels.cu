// Per-bag "tail" kernels (latency-bound: one CTA per bag), losses, fused Adam, DeepAttMISL cluster pooling and the
// region index map.  All vectors live in shared memory; mat-vecs are warp-per-output-row with coalesced weight reads.
#include <cooperative_groups.h>
#include "stages.cuh"

namespace cg = cooperative_groups;

namespace advmil {

// sum_r W[r*ld + col] * v[r], r < n: transposed mat-vec column owned by one thread (coalesced across threads);
// four independent accumulators so the loads of consecutive rows are in flight together
__device__ __forceinline__ float col_dot(const float* __restrict__ W, int ld, int col, const float* __restrict__ v, int n) {
  float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
  int r = 0;
  for (; r + 7 < n; r += 8) {
    const float w0 = __ldg(W + (size_t)r * ld + col), w1 = __ldg(W + (size_t)(r + 1) * ld + col);
    const float w2 = __ldg(W + (size_t)(r + 2) * ld + col), w3 = __ldg(W + (size_t)(r + 3) * ld + col);
    const float w4 = __ldg(W + (size_t)(r + 4) * ld + col), w5 = __ldg(W + (size_t)(r + 5) * ld + col);
    const float w6 = __ldg(W + (size_t)(r + 6) * ld + col), w7 = __ldg(W + (size_t)(r + 7) * ld + col);
    a0 = fmaf(w0, v[r], a0); a1 = fmaf(w1, v[r + 1], a1); a2 = fmaf(w2, v[r + 2], a2); a3 = fmaf(w3, v[r + 3], a3);
    a0 = fmaf(w4, v[r + 4], a0); a1 = fmaf(w5, v[r + 5], a1); a2 = fmaf(w6, v[r + 6], a2); a3 = fmaf(w7, v[r + 7], a3);
  }
  for (; r < n; ++r) a0 = fmaf(__ldg(W + (size_t)r * ld + col), v[r], a0);
  return (a0 + a1) + (a2 + a3);
}

// out[r] = dot(W[r, 0:n], v) for r handled by this warp; caller adds bias/activation
__device__ __forceinline__ float warp_dot(const float* __restrict__ Wrow, const float* __restrict__ v, int n, int lane) {
  float acc = 0.f;
  for (int c = lane; c < n; c += 32) acc = fmaf(Wrow[c], v[c], acc);
  return warp_sum(acc);
}

// Four output rows r0..r0+3 of y = W v at once (W row-major [*, ld], n % 4 == 0, rows and v 16-byte aligned): 4 x n/128
// independent 16-byte loads in flight per lane instead of one dependent 4-byte chain per row.  Rows >= rmax are skipped.
__device__ __forceinline__ void warp_dot4(const float* __restrict__ W, int ld, int r0, int rmax, const float* __restrict__ v,
                                          int n, int lane, float (&out)[4]) {
  float acc[4] = {0.f, 0.f, 0.f, 0.f};
  for (int c = lane * 4; c < n; c += 128) {
    const float4 x = *reinterpret_cast<const float4*>(v + c);
    float4 w[4];
#pragma unroll
    for (int u = 0; u < 4; ++u)
      w[u] = (r0 + u < rmax) ? __ldg(reinterpret_cast<const float4*>(W + (size_t)(r0 + u) * ld + c)) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int u = 0; u < 4; ++u) acc[u] += w[u].x * x.x + w[u].y * x.y + w[u].z * x.z + w[u].w * x.w;
  }
#pragma unroll
  for (int u = 0; u < 4; ++u) out[u] = warp_sum(acc[u]);
}

// y[c] = sum_{r<n} W[r*ld + c] v[r] for c < ncols (ncols % 4 == 0, W 16-byte aligned): the whole block cooperates, thread
// (g, cv) accumulates column vector cv over rows g, g+G, ...; partials meet in `scratch` ([G][ncols] floats).  v, scratch
// and out live in shared memory; ends with a __syncthreads().
__device__ __forceinline__ void block_colmat(const float* __restrict__ W, int ld, int ncols, const float* __restrict__ v,
                                             int n, float* __restrict__ scratch, float* __restrict__ out) {
  const int CV = ncols >> 2;
  const int G = max(1, min((int)blockDim.x / CV, n));
  const int cv = threadIdx.x % CV, g = threadIdx.x / CV;
  if (g < G) {
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    int r = g;
    for (; r + 3 * G < n; r += 4 * G) {
      const float4 w0 = __ldg(reinterpret_cast<const float4*>(W + (size_t)r * ld) + cv);
      const float4 w1 = __ldg(reinterpret_cast<const float4*>(W + (size_t)(r + G) * ld) + cv);
      const float4 w2 = __ldg(reinterpret_cast<const float4*>(W + (size_t)(r + 2 * G) * ld) + cv);
      const float4 w3 = __ldg(reinterpret_cast<const float4*>(W + (size_t)(r + 3 * G) * ld) + cv);
      const float v0 = v[r], v1 = v[r + G], v2 = v[r + 2 * G], v3 = v[r + 3 * G];
      acc.x += w0.x * v0 + w1.x * v1 + w2.x * v2 + w3.x * v3;
      acc.y += w0.y * v0 + w1.y * v1 + w2.y * v2 + w3.y * v3;
      acc.z += w0.z * v0 + w1.z * v1 + w2.z * v2 + w3.z * v3;
      acc.w += w0.w * v0 + w1.w * v1 + w2.w * v2 + w3.w * v3;
    }
    for (; r < n; r += G) {
      const float4 w0 = __ldg(reinterpret_cast<const float4*>(W + (size_t)r * ld) + cv);
      const float v0 = v[r];
      acc.x += w0.x * v0; acc.y += w0.y * v0; acc.z += w0.z * v0; acc.w += w0.w * v0;
    }
    *reinterpret_cast<float4*>(scratch + (size_t)g * ncols + cv * 4) = acc;
  }
  __syncthreads();
  for (int c = threadIdx.x; c < ncols; c += blockDim.x) {
    float t = 0.f;
    for (int k = 0; k < G; ++k) t += scratch[(size_t)k * ncols + c];
    out[c] = t;
  }
  __syncthreads();
}

// =============================================================================================
// K4: generator head  (model/backbone.py:73-77,85; model/GANSurv.py:32-49; model/model_utils.py:116-133)
// One thread-block CLUSTER of HEAD_CS CTAs per (bag, sample): the per-bag chain rho -> MLP0 -> out streams ~0.9 MB of
// weights through a dependent mat-vec chain, which one CTA can only pull at one SM's L2 bandwidth.  Each CTA of the cluster
// owns a slice of every layer's output rows and pushes its results into its peers' shared memory (DSMEM).
// grid (bags * HEAD_CS, samples)
// =============================================================================================
constexpr int HEAD_CS = 8;
// slice [beg, end) of n outputs owned by cluster rank r (multiples of 4 so that the float4 paths stay 16-byte aligned)
__device__ __forceinline__ void head_slice(int n, int rank, int& beg, int& end) {
  const int per = ((n + HEAD_CS - 1) / HEAD_CS + 3) & ~3;
  beg = min(n, rank * per);
  end = min(n, beg + per);
}

__global__ void __launch_bounds__(384) gen_head_fwd_kernel(AdvmilGenParams p, const float* __restrict__ z,
                                                          const float* __restrict__ noise0,
                                                          const float* __restrict__ noise1, int bags, Drop drho,
                                                          Drop dmlp0, float* __restrict__ H, float* __restrict__ H1,
                                                          float* __restrict__ pre, float* __restrict__ pred) {
  pdl_prologue();
  cg::cluster_group cluster = cg::this_cluster();
  const int rank = (int)cluster.block_rank();
  extern __shared__ __align__(16) float sm[];
  const int b = blockIdx.x / HEAD_CS, smp = blockIdx.y;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
  const int h = p.h, o = p.o, hid = p.hid;
  float* zs = sm;            // [h]
  float* Hs = zs + h;        // [2*o]   (H | noise0)
  float* H1s = Hs + 2 * o;   // [2*hid] (H1 | noise1)
  float* red = H1s + 2 * hid;  // [33]
  for (int c = threadIdx.x; c < h; c += blockDim.x) zs[c] = z[(size_t)b * h + c];
  cluster.sync();            // zs visible; every CTA of the cluster is running before anyone writes into a peer
  const bool vec_ok = (h % 4 == 0) && (o % 4 == 0) && (hid % 4 == 0);   // 16-byte aligned rows for warp_dot4
  if (p.Wrho) {
    int ib, ie;
    head_slice(o, rank, ib, ie);
    if (vec_ok) {
      for (int i0 = ib + wid * 4; i0 < ie; i0 += nw * 4) {
        float v4[4];
        warp_dot4(p.Wrho, h, i0, ie, zs, h, lane, v4);
        const int u = lane & 3, dst = lane >> 2;             // lane (dst, u) hands output i0 + u to CTA dst
        const float vv = u == 0 ? v4[0] : u == 1 ? v4[1] : u == 2 ? v4[2] : v4[3];
        if (i0 + u < ie) cluster.map_shared_rank(Hs, dst)[i0 + u] = fmaxf(vv + p.brho[i0 + u], 0.f) * drho.scale(b, i0 + u);
      }
    } else {
      for (int i = ib + wid; i < ie; i += nw) {
        float v = warp_dot(p.Wrho + (size_t)i * h, zs, h, lane);
        if (lane < HEAD_CS) cluster.map_shared_rank(Hs, lane)[i] = fmaxf(v + p.brho[i], 0.f) * drho.scale(b, i);
      }
    }
  } else {
    for (int c = threadIdx.x; c < o; c += blockDim.x) Hs[c] = zs[c];
  }
  const int in0 = o * (1 + p.noise0);
  if (p.noise0)
    for (int c = threadIdx.x; c < o; c += blockDim.x)
      Hs[o + c] = noise0 ? noise0[((size_t)smp * bags + b) * o + c] : 0.f;
  cluster.sync();            // Hs complete in every CTA
  if (H && smp == 0 && rank == 0) for (int c = threadIdx.x; c < o; c += blockDim.x) H[(size_t)b * o + c] = Hs[c];
  if (p.W0 == nullptr) return;  // backbone-only mode (ABMIL.forward without the Generator head)
  {
    int jb, je;
    head_slice(hid, rank, jb, je);
    float* H1s0 = cluster.map_shared_rank(H1s, 0);           // only rank 0 consumes H1
    if (vec_ok) {
      for (int j0 = jb + wid * 4; j0 < je; j0 += nw * 4) {
        float v4[4];
        warp_dot4(p.W0, in0, j0, je, Hs, in0, lane, v4);
        const float vv = lane == 0 ? v4[0] : lane == 1 ? v4[1] : lane == 2 ? v4[2] : v4[3];
        if (lane < 4 && j0 + lane < je) H1s0[j0 + lane] = fmaxf(vv + p.b0[j0 + lane], 0.f) * dmlp0.scale(b, j0 + lane);
      }
    } else {
      for (int j = jb + wid; j < je; j += nw) {
        float v = warp_dot(p.W0 + (size_t)j * in0, Hs, in0, lane);
        if (lane == 0) H1s0[j] = fmaxf(v + p.b0[j], 0.f) * dmlp0.scale(b, j);
      }
    }
  }
  cluster.sync();            // H1s complete in rank 0; nobody touches a peer's shared memory after this point
  if (rank != 0) return;
  const int in1 = hid * (1 + p.noise1);
  if (p.noise1)
    for (int c = threadIdx.x; c < hid; c += blockDim.x)
      H1s[hid + c] = noise1 ? noise1[((size_t)smp * bags + b) * hid + c] : 0.f;
  __syncthreads();
  if (H1 && smp == 0) for (int c = threadIdx.x; c < hid; c += blockDim.x) H1[(size_t)b * hid + c] = H1s[c];
  float acc = 0.f;
  for (int c = threadIdx.x; c < in1; c += blockDim.x) acc = fmaf(p.Wl[c], H1s[c], acc);
  acc = block_sum(acc, red);
  if (threadIdx.x == 0) {
    float v = acc + p.bl[0];
    if (pre && smp == 0) pre[b] = v;
    float out = v;
    if (p.out_scale == 1) out = sigmoidf_(v);
    else if (p.out_scale == 2) out = expf(v);
    pred[(size_t)smp * bags + b] = out;
  }
}

int gen_head_fwd(const AdvmilGenParams& p, const float* z, const float* noise0, const float* noise1, int bags,
                 int samples, const Drop& drho, const Drop& dmlp0, float* H, float* H1, float* pre, float* pred,
                 cudaStream_t st) {
  ADVMIL_REQUIRE(p.Wrho != nullptr || p.o == p.h, "gen_head: no rho layer requires o == h");
  size_t smem = (size_t)(p.h + 2 * p.o + 2 * p.hid + 40) * sizeof(float);
  ADVMIL_REQUIRE(smem <= 48 * 1024, "gen_head: dims too large for the head kernel (h=%d o=%d)", p.h, p.o);
  launch_kc(gen_head_fwd_kernel, dim3(bags * HEAD_CS, samples), dim3(384), smem, st, HEAD_CS, p, z, noise0, noise1, bags, drho, dmlp0,
           H, H1, pre, pred);
  ADVMIL_CHECK_LAUNCH();
  return ADVMIL_OK;
}

// backward of the head: dz = Wrho^T (relu' (W0[:, :o]^T d1)), one cluster per bag; rank r owns a column slice of each
// transposed mat-vec (W rows are read as contiguous slices) and pushes its part of dH to every peer.
__global__ void __launch_bounds__(256) gen_head_bwd_kernel(AdvmilGenParams p, const float* __restrict__ d_pred,
                                                           const float* __restrict__ H, const float* __restrict__ H1,
                                                           const float* __restrict__ pred, float inv_keep_rho,
                                                           float inv_keep_mlp0, float* __restrict__ dz,
                                                           float* __restrict__ dHpre, float* __restrict__ dH1pre,
                                                           float* __restrict__ dpre) {
  pdl_prologue();
  cg::cluster_group cluster = cg::this_cluster();
  const int rank = (int)cluster.block_rank();
  extern __shared__ __align__(16) float sm[];
  const int b = blockIdx.x / HEAD_CS;
  const int h = p.h, o = p.o, hid = p.hid;
  float* d1 = sm;                        // [hid]
  float* dH = d1 + ((hid + 3) & ~3);     // [o]      (complete after the exchange)
  float* loc = dH + ((o + 3) & ~3);      // [slice]  this CTA's part of a transposed mat-vec
  float* scratch = loc + (((max(o, h) + HEAD_CS - 1) / HEAD_CS + 7) & ~3);   // [4 * blockDim.x] block_colmat partials
  const bool head = p.W0 != nullptr;  // else d_pred is dL/dH [bags,o] (backbone-only mode)
  if (head) {
    float dp = d_pred[b];
    float pr = pred[b];
    if (p.out_scale == 1) dp *= pr * (1.f - pr);
    else if (p.out_scale == 2) dp *= pr;
    if (threadIdx.x == 0 && rank == 0) dpre[b] = dp;
    for (int j = threadIdx.x; j < hid; j += blockDim.x) {
      float hv = H1[(size_t)b * hid + j];
      float g = hv > 0.f ? dp * p.Wl[j] * inv_keep_mlp0 : 0.f;
      d1[j] = g;
      if (rank == 0) dH1pre[(size_t)b * hid + j] = g;
    }
  }
  cluster.sync();            // d1 visible; every CTA of the cluster is running
  const int in0 = o * (1 + p.noise0);
  const bool vec_ok = (o % 4 == 0) && (h % 4 == 0) && (in0 % 4 == 0);
  int cb, ce;
  head_slice(o, rank, cb, ce);
  if (head && ce > cb) {
    if (vec_ok) block_colmat(p.W0 + cb, in0, ce - cb, d1, hid, scratch, loc);          // dH[slice] = W0[:, slice]^T d1
    else { for (int i = cb + threadIdx.x; i < ce; i += blockDim.x) loc[i - cb] = col_dot(p.W0, in0, i, d1, hid); __syncthreads(); }
  }
  for (int i = cb + threadIdx.x; i < ce; i += blockDim.x) {
    float acc = head ? loc[i - cb] : d_pred[(size_t)b * o + i];
    if (p.Wrho) acc = H[(size_t)b * o + i] > 0.f ? acc * inv_keep_rho : 0.f;
    dHpre[(size_t)b * o + i] = acc;
#pragma unroll
    for (int dst = 0; dst < HEAD_CS; ++dst) cluster.map_shared_rank(dH, dst)[i] = acc;
  }
  cluster.sync();            // dH complete in every CTA; no peer access after this point
  int kb, ke;
  head_slice(h, rank, kb, ke);
  if (ke <= kb) return;
  if (p.Wrho && vec_ok) {
    block_colmat(p.Wrho + kb, h, ke - kb, dH, o, scratch, loc);                         // dz[slice] = Wrho[:, slice]^T dH
    for (int k = kb + threadIdx.x; k < ke; k += blockDim.x) dz[(size_t)b * h + k] = loc[k - kb];
  } else {
    for (int k = kb + threadIdx.x; k < ke; k += blockDim.x)
      dz[(size_t)b * h + k] = p.Wrho ? col_dot(p.Wrho, h, k, dH, o) : dH[k];
  }
}

int gen_head_bwd(const AdvmilGenParams& p, const float* d_pred, const float* H, const float* H1, const float* pred,
                 int bags, float inv_keep_rho, float inv_keep_mlp0, float* dz, float* dHpre, float* dH1pre, float* dpre,
                 cudaStream_t st) {
  const int threads = 256;
  const size_t slice = ((size_t)(max(p.o, p.h) + HEAD_CS - 1) / HEAD_CS + 7) & ~(size_t)3;
  size_t smem = ((size_t)(p.hid + p.o) + 8 + slice + 4 * (size_t)threads + 16) * sizeof(float);
  ADVMIL_REQUIRE(smem <= 48 * 1024, "gen_head_bwd: dims too large for the head kernel (h=%d o=%d)", p.h, p.o);
  launch_kc(gen_head_bwd_kernel, dim3(bags * HEAD_CS), dim3(threads), smem, st, HEAD_CS, p, d_pred, H, H1, pred, inv_keep_rho,
           inv_keep_mlp0, dz, dHpre, dH1pre, dpre);
  ADVMIL_CHECK_LAUNCH();
  return ADVMIL_OK;
}

// acc += sum_b g[b * ldg] * x[b * ldx], accb += sum_b g[b * ldg], in bag order (bit-identical to the plain loop): the
// 2 x 8 loads of a block of bags are issued together -- the loop is a chain of dependent global-memory latencies otherwise
// (16-32 bags: 14 us for a few KFLOP)
__device__ __forceinline__ void outer_accumulate(const float* __restrict__ g, int ldg, const float* __restrict__ x, int ldx, int bags,
                                                 float& acc, float& accb) {
  int b = 0;
  for (; b + 8 <= bags; b += 8) {
    float gv[8], xv[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) { gv[u] = g[(size_t)(b + u) * ldg]; xv[u] = x ? x[(size_t)(b + u) * ldx] : 0.f; }
#pragma unroll
    for (int u = 0; u < 8; ++u) { acc = fmaf(gv[u], xv[u], acc); accb += gv[u]; }
  }
  for (; b < bags; ++b) {
    const float gv = g[(size_t)b * ldg], xv = x ? x[(size_t)b * ldx] : 0.f;
    acc = fmaf(gv, xv, acc);
    accb += gv;
  }
}

// dW[o, i] (+)= sum_b dy[b,o] * xcat[b,i];  db[o] (+)= sum_b dy[b,o]
__global__ void outer_sum_kernel(const float* __restrict__ dy, const float* __restrict__ x1, int in1,
                                 const float* __restrict__ x2, int in2, int bags, int out, float* __restrict__ dW,
                                 float* __restrict__ db, int accumulate) {
  pdl_prologue();
  const int in = in1 + in2;
  size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (size_t)out * in) return;
  int o = (int)(idx / in), i = (int)(idx % in);
  float acc = 0.f, accb = 0.f;
  const float* xs = i < in1 ? x1 + i : (x2 ? x2 + (i - in1) : nullptr);
  outer_accumulate(dy + o, out, xs, i < in1 ? in1 : in2, bags, acc, accb);
  if (dW) dW[idx] = accumulate ? dW[idx] + acc : acc;
  if (db && i == 0) db[o] = accumulate ? db[o] + accb : accb;
}
int outer_sum(const float* dy, const float* x1, int in1, const float* x2, int in2, int bags, int out, float* dW,
              float* db, int accumulate, cudaStream_t st) {
  size_t n = (size_t)out * (in1 + in2);
  launch_k(outer_sum_kernel, dim3(cdiv(n, 256)), dim3(256), 0, st, dy, x1, in1, x2, in2, bags, out, dW, db, accumulate);
  ADVMIL_CHECK_LAUNCH();
  return ADVMIL_OK;
}

// several outer-sum problems in one launch (the per-bag head layers of one backward pass)
struct OuterBatch { OuterProb p[OUTER_MAX]; int first_block[OUTER_MAX + 1]; int n; };
__global__ void outer_sum_multi_kernel(OuterBatch ob, int bags, int accumulate) {
  pdl_prologue();
  int k = 0;
  while (k + 1 < ob.n && (int)blockIdx.x >= ob.first_block[k + 1]) ++k;
  const OuterProb q = ob.p[k];
  const int in = q.in1 + q.in2;
  const size_t idx = (size_t)(blockIdx.x - ob.first_block[k]) * blockDim.x + threadIdx.x;
  if (idx >= (size_t)q.out * in) return;
  const int o = (int)(idx / in), i = (int)(idx % in);
  float acc = 0.f, accb = 0.f;
  const float* xs = i < q.in1 ? q.x1 + i : (q.x2 ? q.x2 + (i - q.in1) : nullptr);
  outer_accumulate(q.dy + o, q.out, xs, i < q.in1 ? q.in1 : q.in2, bags, acc, accb);
  if (q.dW) q.dW[idx] = accumulate ? q.dW[idx] + acc : acc;
  if (q.db && i == 0) q.db[o] = accumulate ? q.db[o] + accb : accb;
}
int outer_sum_multi(const OuterProb* probs, int n, int bags, int accumulate, cudaStream_t st) {
  ADVMIL_REQUIRE(n >= 0 && n <= OUTER_MAX, "outer_sum_multi: at most %d problems", OUTER_MAX);
  if (n == 0) return ADVMIL_OK;
  OuterBatch ob;
  ob.n = n;
  int blocks = 0;
  for (int k = 0; k < n; ++k) {
    ob.p[k] = probs[k];
    ob.first_block[k] = blocks;
    blocks += cdiv((size_t)probs[k].out * (probs[k].in1 + probs[k].in2), 256);
  }
  ob.first_block[n] = blocks;
  launch_k(outer_sum_multi_kernel, dim3(blocks), dim3(256), 0, st, ob, bags, accumulate);
  ADVMIL_CHECK_LAUNCH();
  return ADVMIL_OK;
}

// =============================================================================================
// K7/K8 tail: bag MLP fc2, time embedding, inner product, projection
// (model/model_utils.py:200-206; model/GANSurv.py:89-105)
// =============================================================================================
__global__ void __launch_bounds__(512) rlip_tail_fwd_kernel(AdvmilDiscParams p, const float* __restrict__ bagv,
                                                            const float* __restrict__ fbar, const float* __restrict__ t,
                                                            Drop dfc2, float* __restrict__ g1, float* __restrict__ hx,
                                                            float* __restrict__ u1, float* __restrict__ ht,
                                                            float* __restrict__ out) {
  pdl_prologue();
  extern __shared__ __align__(16) float sm[];
  const int b = blockIdx.x;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
  const int d = p.d, dh = p.d / 2, t1 = p.t1, t2 = p.t2;
  float* bv = sm;           // [d]
  float* g1s = bv + d;      // [dh]
  float* hxs = g1s + dh;    // [d]
  float* u1s = hxs + d;     // [t1]
  float* hts = u1s + t1;    // [t2]
  float* red = hts + t2;    // [33]
  for (int c = threadIdx.x; c < d; c += blockDim.x) bv[c] = bagv[(size_t)b * d + c];
  const float tv = t[b];
  for (int c = threadIdx.x; c < t1; c += blockDim.x) {
    float v = fmaxf(fmaf(p.T1_w[c], tv, p.T1_b[c]), 0.f);
    u1s[c] = v;
    u1[(size_t)b * t1 + c] = v;
  }
  __syncthreads();
  const bool vec_ok = (d % 8 == 0) && (t1 % 4 == 0) && (t2 % 4 == 0);
  for (int j0 = wid * 4; j0 < dh; j0 += nw * 4) {
    float v4[4];
    if (vec_ok) warp_dot4(p.F2a_w, d, j0, dh, bv, d, lane, v4);
    else for (int u = 0; u < 4; ++u) v4[u] = j0 + u < dh ? warp_dot(p.F2a_w + (size_t)(j0 + u) * d, bv, d, lane) : 0.f;
    const float vv = lane == 0 ? v4[0] : lane == 1 ? v4[1] : lane == 2 ? v4[2] : v4[3];
    const int j = j0 + lane;
    if (lane < 4 && j < dh) {
      const float v = fmaxf(vv + p.F2a_b[j], 0.f) * dfc2.scale(b, j);
      g1s[j] = v;
      g1[(size_t)b * dh + j] = v;
    }
  }
  for (int j0 = wid * 4; j0 < t2; j0 += nw * 4) {
    float v4[4];
    if (vec_ok) warp_dot4(p.T2_w, t1, j0, t2, u1s, t1, lane, v4);
    else for (int u = 0; u < 4; ++u) v4[u] = j0 + u < t2 ? warp_dot(p.T2_w + (size_t)(j0 + u) * t1, u1s, t1, lane) : 0.f;
    const float vv = lane == 0 ? v4[0] : lane == 1 ? v4[1] : lane == 2 ? v4[2] : v4[3];
    const int j = j0 + lane;
    if (lane < 4 && j < t2) {
      const float v = fmaxf(vv + p.T2_b[j], 0.f);
      hts[j] = v;
      ht[(size_t)b * t2 + j] = v;
    }
  }
  __syncthreads();
  for (int j0 = wid * 4; j0 < d; j0 += nw * 4) {
    float v4[4];
    if (vec_ok) warp_dot4(p.F2b_w, dh, j0, d, g1s, dh, lane, v4);
    else for (int u = 0; u < 4; ++u) v4[u] = j0 + u < d ? warp_dot(p.F2b_w + (size_t)(j0 + u) * dh, g1s, dh, lane) : 0.f;
    const float vv = lane == 0 ? v4[0] : lane == 1 ? v4[1] : lane == 2 ? v4[2] : v4[3];
    const int j = j0 + lane;
    if (lane < 4 && j < d) {
      const float v = vv + p.F2b_b[j];
      hxs[j] = v;
      hx[(size_t)b * d + j] = v;
    }
  }
  __syncthreads();
  float acc = 0.f;
  for (int c = threadIdx.x; c < d; c += blockDim.x) {
    if (p.prj_path == 3) {      // concat discriminator (model/GANSurv.py:52-68): out = fc([hx | ht]), no inner product
      acc = fmaf(p.Pr_w[c], hxs[c], acc);
      acc = fmaf(p.Pr_w[d + c], hts[c], acc);
      continue;
    }
    float left = p.inner_instance ? fbar[(size_t)b * d + c] : hxs[c];
    acc = fmaf(left, hts[c], acc);
    if (p.prj_path == 1) acc = fmaf(p.Pr_w[c], hxs[c], acc);
    else if (p.prj_path == 2) acc = fmaf(p.Pr_w[c], hts[c], acc);
  }
  acc = block_sum(acc, red);
  if (threadIdx.x == 0) out[b] = acc + (p.prj_path ? p.Pr_b[0] : 0.f);
}

int rlip_tail_fwd(const AdvmilDiscParams& p, const float* bagv, const float* fbar, const float* t, int bags,
                  const Drop& dfc2, float* g1, float* hx, float* u1, float* ht, float* out, cudaStream_t st) {
  ADVMIL_REQUIRE(p.t2 == p.d, "rlip_tail: time embedding width %d must equal d %d", p.t2, p.d);
  size_t smem = (size_t)(p.d * 2 + p.d / 2 + p.t1 + p.t2 + 40) * sizeof(float);
  launch_k(rlip_tail_fwd_kernel, dim3(bags), dim3(512), smem, st, p, bagv, fbar, t, dfc2, g1, hx, u1, ht, out);
  ADVMIL_CHECK_LAUNCH();
  return ADVMIL_OK;
}

__global__ void __launch_bounds__(512) rlip_tail_bwd_kernel(
    AdvmilDiscParams p, const float* __restrict__ d_out, const float* __restrict__ bagv, const float* __restrict__ fbar,
    const float* __restrict__ g1, const float* __restrict__ hx, const float* __restrict__ u1,
    const float* __restrict__ ht, float inv_keep_fc2, float* __restrict__ d_fbar, float* __restrict__ d_bagv,
    float* __restrict__ d_hx, float* __restrict__ d_g1pre, float* __restrict__ d_htpre, float* __restrict__ d_u1pre,
    float* __restrict__ d_t) {
  pdl_prologue();
  extern __shared__ __align__(16) float sm[];
  const int b = blockIdx.x;
  const int d = p.d, dh = p.d / 2, t1 = p.t1, t2 = p.t2;
  float* dhx = sm;          // [d]
  float* dg1 = dhx + d;     // [dh]
  float* dht = dg1 + dh;    // [t2]
  float* du1 = dht + t2;    // [t1]
  float* red = du1 + t1;    // [33]
  const float go = d_out[b];
  for (int c = threadIdx.x; c < d; c += blockDim.x) {
    float hxv = hx[(size_t)b * d + c], htv = ht[(size_t)b * t2 + c], fb = fbar[(size_t)b * d + c];
    float g_hx = 0.f, g_ht = 0.f, g_fb = 0.f;
    if (p.prj_path == 3) { g_hx = go * p.Pr_w[c]; g_ht = go * p.Pr_w[d + c]; }
    else if (p.inner_instance) { g_fb = go * htv; g_ht = go * fb; }
    else { g_hx = go * htv; g_ht = go * hxv; }
    if (p.prj_path == 1) g_hx += go * p.Pr_w[c];
    else if (p.prj_path == 2) g_ht += go * p.Pr_w[c];
    g_ht = htv > 0.f ? g_ht : 0.f;  // ReLU of the last time-MLP layer
    dhx[c] = g_hx; dht[c] = g_ht;
    d_hx[(size_t)b * d + c] = g_hx;
    d_htpre[(size_t)b * t2 + c] = g_ht;
    d_fbar[(size_t)b * d + c] = g_fb;
  }
  __syncthreads();
  float* scratch = red + 40;      // [G][ncols] partials of the transposed mat-vecs (<= 2048 floats when vec_ok)
  const bool vec_ok = (d % 8 == 0) && (t1 % 4 == 0) && (t2 % 4 == 0);
  if (vec_ok) {
    block_colmat(p.F2b_w, dh, dh, dhx, d, scratch, dg1);       // dg1 = F2b_w^T dhx
    block_colmat(p.T2_w, t1, t1, dht, t2, scratch, du1);       // du1 = T2_w^T dht
  } else {
    for (int j = threadIdx.x; j < dh; j += blockDim.x) dg1[j] = col_dot(p.F2b_w, dh, j, dhx, d);
    for (int k = threadIdx.x; k < t1; k += blockDim.x) du1[k] = col_dot(p.T2_w, t1, k, dht, t2);
    __syncthreads();
  }
  for (int j = threadIdx.x; j < dh; j += blockDim.x) {
    const float acc = g1[(size_t)b * dh + j] > 0.f ? dg1[j] * inv_keep_fc2 : 0.f;
    dg1[j] = acc;
    d_g1pre[(size_t)b * dh + j] = acc;
  }
  for (int k = threadIdx.x; k < t1; k += blockDim.x) {
    const float acc = u1[(size_t)b * t1 + k] > 0.f ? du1[k] : 0.f;
    du1[k] = acc;
    d_u1pre[(size_t)b * t1 + k] = acc;
  }
  __syncthreads();
  if (vec_ok) {
    float* dbv = scratch + 2048;
    block_colmat(p.F2a_w, d, d, dg1, dh, scratch, dbv);        // d_bagv = F2a_w^T dg1
    for (int c = threadIdx.x; c < d; c += blockDim.x) d_bagv[(size_t)b * d + c] = dbv[c];
  } else {
    for (int c = threadIdx.x; c < d; c += blockDim.x) d_bagv[(size_t)b * d + c] = col_dot(p.F2a_w, d, c, dg1, dh);
  }
  float acc = 0.f;
  for (int k = threadIdx.x; k < t1; k += blockDim.x) acc = fmaf(p.T1_w[k], du1[k], acc);
  acc = block_sum(acc, red);
  if (threadIdx.x == 0 && d_t) d_t[b] = acc;
}

int rlip_tail_bwd(const AdvmilDiscParams& p, const float* d_out, const float* bagv, const float* fbar, const float* g1,
                  const float* hx, const float* u1, const float* ht, int bags, float inv_keep_fc2, float* d_fbar,
                  float* d_bagv, float* d_hx, float* d_g1pre, float* d_htpre, float* d_u1pre, float* d_t,
                  cudaStream_t st) {
  // scratch of block_colmat: G * ncols <= threads * 4 floats per call, + one [d] result vector
  size_t smem = (size_t)(p.d + p.d / 2 + p.t2 + p.t1 + 40 + 40 + 2048 + p.d + 16) * sizeof(float);
  ADVMIL_REQUIRE(smem <= 48 * 1024 && p.d <= 2048, "rlip_tail_bwd: d=%d too large", p.d);
  launch_k(rlip_tail_bwd_kernel, dim3(bags), dim3(512), smem, st, p, d_out, bagv, fbar, g1, hx, u1, ht, inv_keep_fc2, d_fbar, d_bagv,
                                                 d_hx, d_g1pre, d_htpre, d_u1pre, d_t);
  ADVMIL_CHECK_LAUNCH();
  return ADVMIL_OK;
}

// =============================================================================================
// losses (loss/utils.py:21-41,182-208) — one CTA, bags <= a few thousand
// =============================================================================================
__global__ void disc_loss_kernel(const float* __restrict__ f_real, const float* __restrict__ f_fake,
                                 const uint8_t* __restrict__ real_mask, int bags, int which, float n_real, float n_fake,
                                 float* __restrict__ loss_out, float* __restrict__ d_real, float* __restrict__ d_fake) {
  pdl_prologue();
  __shared__ float red[33];
  float acc = 0.f;
  for (int b = threadIdx.x; b < bags; b += blockDim.x) {
    float f = f_fake[b];
    float lf, gf;
    if (which == 0) {
      float sg = sigmoidf_(f);
      lf = -(1.0f - logf(sg + 1e-8f));
      gf = sg * (1.f - sg) / (sg + 1e-8f);
    } else if (which == 1) {
      lf = fmaxf(1.f + f, 0.f);
      gf = (1.f + f) > 0.f ? 1.f : 0.f;
    } else {
      lf = f; gf = 1.f;
    }
    acc += lf / n_fake;
    if (d_fake) d_fake[b] = gf / n_fake;
    float gr = 0.f;
    if (real_mask && real_mask[b] && n_real > 0.f) {
      float r = f_real[b];
      float lr;
      if (which == 0) {
        float sg = sigmoidf_(r);
        lr = -logf(sg + 1e-8f);
        gr = -sg * (1.f - sg) / (sg + 1e-8f);
      } else if (which == 1) {
        lr = fmaxf(1.f - r, 0.f);
        gr = (1.f - r) > 0.f ? -1.f : 0.f;
      } else {
        lr = -r; gr = -1.f;
      }
      acc += lr / n_real;
      gr /= n_real;
    }
    if (d_real) d_real[b] = gr;
  }
  acc = block_sum(acc, red);
  if (threadIdx.x == 0) loss_out[0] += acc;
}

__global__ void gen_loss_kernel(const float* __restrict__ pred, const float* __restrict__ t, const float* __restrict__ e,
                                const uint8_t* __restrict__ visible, const float* __restrict__ f_fake, int bags,
                                float n_visible, float n_fake, float coef_gan, float alpha, float gamma, int norm,
                                float* __restrict__ losses, float* __restrict__ d_pred, float* __restrict__ d_fake) {
  pdl_prologue();
  __shared__ float red[33];
  float rec = 0.f, gen = 0.f;
  for (int b = threadIdx.x; b < bags; b += blockDim.x) {
    float g = 0.f;
    if (visible[b] && n_visible > 0.f) {
      float diff = pred[b] - t[b], ev = e[b];
      float sgn = diff > 0.f ? 1.f : (diff < 0.f ? -1.f : 0.f);
      float lo = ev * fabsf(diff);
      float glo = ev * sgn;
      float marg = gamma - diff;
      float lc = (1.f - ev) * fmaxf(marg, 0.f);
      float glc = marg > 0.f ? -(1.f - ev) : 0.f;
      if (norm == 1) { glo = 2.f * lo * glo; glc = 2.f * lc * glc; lo = lo * lo; lc = lc * lc; }
      rec += ((1.f - alpha) * (lo + lc) + alpha * lo) / n_visible;
      g = ((1.f - alpha) * (glo + glc) + alpha * glo) / n_visible;
    }
    d_pred[b] = g;
    gen += -f_fake[b] / n_fake;
    d_fake[b] = coef_gan == 0.f ? 0.f : -coef_gan / n_fake;
  }
  rec = block_sum(rec, red);
  gen = block_sum(gen, red);
  if (threadIdx.x == 0) {
    losses[0] += rec;
    losses[1] += gen;
    losses[2] += coef_gan == 0.f ? rec : rec + coef_gan * gen;
  }
}

// =============================================================================================
// fused Adam (+L2 weight decay mask, +L1 sub-gradient) over a flat buffer
// =============================================================================================
__global__ void adam_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                            float* __restrict__ v, const uint8_t* __restrict__ wd_mask, int64_t n, float step_size,
                            float beta1, float beta2, float eps, float weight_decay, float l1_coef, float inv_sqrt_bc2,
                            float grad_scale) {
  pdl_prologue();
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float pv = p[i];
  float gv = g[i] * grad_scale;
  if (l1_coef != 0.f) gv += l1_coef * (pv > 0.f ? 1.f : (pv < 0.f ? -1.f : 0.f));
  if (wd_mask && wd_mask[i]) gv = fmaf(weight_decay, pv, gv);
  float mv = beta1 * m[i] + (1.f - beta1) * gv;
  float vv = beta2 * v[i] + (1.f - beta2) * gv * gv;
  m[i] = mv; v[i] = vv;
  float denom = sqrtf(vv) * inv_sqrt_bc2 + eps;
  p[i] = pv - step_size * (mv / denom);
}

// one cluster of ABS_CS CTAs; partial sums meet in rank 0's shared memory and are added in rank order (deterministic,
// no atomics)
constexpr int ABS_CS = 8;
__global__ void __launch_bounds__(1024) abs_sum_kernel(const float* __restrict__ p, int64_t n, float* __restrict__ out) {
  pdl_prologue();
  cg::cluster_group cluster = cg::this_cluster();
  __shared__ float red[33];
  __shared__ float parts[ABS_CS];
  float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if ((reinterpret_cast<uintptr_t>(p) & 15) == 0) {   // 16-byte loads, four in flight per thread
    const float4* p4 = reinterpret_cast<const float4*>(p);
    const int64_t n4 = n >> 2;
    for (; i + 3 * stride < n4; i += 4 * stride) {
      const float4 v0 = p4[i], v1 = p4[i + stride], v2 = p4[i + 2 * stride], v3 = p4[i + 3 * stride];
      a0 += (fabsf(v0.x) + fabsf(v0.y)) + (fabsf(v0.z) + fabsf(v0.w));
      a1 += (fabsf(v1.x) + fabsf(v1.y)) + (fabsf(v1.z) + fabsf(v1.w));
      a2 += (fabsf(v2.x) + fabsf(v2.y)) + (fabsf(v2.z) + fabsf(v2.w));
      a3 += (fabsf(v3.x) + fabsf(v3.y)) + (fabsf(v3.z) + fabsf(v3.w));
    }
    for (; i < n4; i += stride) { const float4 v = p4[i]; a0 += (fabsf(v.x) + fabsf(v.y)) + (fabsf(v.z) + fabsf(v.w)); }
    i = (n4 << 2) + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;   // scalar tail
  }
  for (; i < n; i += stride) a0 += fabsf(p[i]);
  float acc = block_sum((a0 + a1) + (a2 + a3), red);
  cluster.sync();                                     // every CTA of the cluster is running
  if (threadIdx.x == 0) cluster.map_shared_rank(parts, 0)[cluster.block_rank()] = acc;
  cluster.sync();
  if (cluster.block_rank() == 0 && threadIdx.x == 0) {
    float t = 0.f;
    for (int r = 0; r < ABS_CS; ++r) t += parts[r];
    out[0] += t;
  }
}

// =============================================================================================
// K9: DeepAttMISL cluster pooling (model/backbone.py:105-117): per (bag, cluster) mean of rows
// =============================================================================================
constexpr int CL_CH = 128;
constexpr int CL_MAX = 64;                            // most clusters per bag
// the partial kernel's static shared memory (cnt_s, cid_s): it counts against the 48 KB a block may use without opting in
constexpr size_t SEG_MEAN_STATIC_SMEM = (CL_MAX + CL_CH) * sizeof(int);
template <typename T>
__global__ void __launch_bounds__(256) seg_mean_id_partial_kernel(const T* __restrict__ v,
                                                                  const int32_t* __restrict__ cid,
                                                                  const int32_t* __restrict__ offsets, int width,
                                                                  int ncl, float* __restrict__ part,
                                                                  int32_t* __restrict__ part_cnt) {
  pdl_prologue();
  extern __shared__ float sm[];  // [ncl][width] sums
  __shared__ int cnt_s[CL_MAX];
  __shared__ int cid_s[CL_CH];
  int b = blockIdx.y, chunk = blockIdx.x;
  int beg = offsets[b] + chunk * CL_CH, end = min(offsets[b + 1], beg + CL_CH);
  if (beg >= offsets[b + 1]) return;
  int nrows = end - beg;
  for (int i = threadIdx.x; i < ncl * width; i += blockDim.x) sm[i] = 0.f;
  if (threadIdx.x < ncl) cnt_s[threadIdx.x] = 0;
  for (int r = threadIdx.x; r < nrows; r += blockDim.x) cid_s[r] = cid[beg + r];
  __syncthreads();
  // each thread owns a fixed set of columns -> no conflicts while rows are visited in order
  for (int c = threadIdx.x; c < width; c += blockDim.x) {
    for (int r = 0; r < nrows; ++r) {
      int k = cid_s[r];
      if (k >= 0 && k < ncl) sm[k * width + c] += ld1(v + (size_t)(beg + r) * width + c);
    }
  }
  if (threadIdx.x == 0)
    for (int r = 0; r < nrows; ++r) { int k = cid_s[r]; if (k >= 0 && k < ncl) cnt_s[k]++; }
  __syncthreads();
  size_t o = ((size_t)(offsets[b] / CL_CH + b + chunk)) * ncl;
  for (int i = threadIdx.x; i < ncl * width; i += blockDim.x) part[o * width + i] = sm[i];
  if (threadIdx.x < ncl) part_cnt[o + threadIdx.x] = cnt_s[threadIdx.x];
}
__global__ void seg_mean_id_final_kernel(const float* __restrict__ part, const int32_t* __restrict__ part_cnt,
                                         const int32_t* __restrict__ offsets, int width, int ncl,
                                         float* __restrict__ out, int32_t* __restrict__ counts) {
  pdl_prologue();
  int b = blockIdx.x / ncl, k = blockIdx.x % ncl;
  int len = offsets[b + 1] - offsets[b];
  int nch = (len + CL_CH - 1) / CL_CH;
  int cnt = 0;
  const size_t pbase = (size_t)(offsets[b] / CL_CH + b);
  for (int ch = 0; ch < nch; ++ch) cnt += part_cnt[(pbase + ch) * ncl + k];
  for (int c = threadIdx.x; c < width; c += blockDim.x) {
    float t = 0.f;
    for (int ch = 0; ch < nch; ++ch) t += part[((pbase + ch) * ncl + k) * width + c];
    out[((size_t)b * ncl + k) * width + c] = cnt > 0 ? t / (float)cnt : 0.f;  // zeros for an empty cluster (backbone.py:114-115)
  }
  if (threadIdx.x == 0) counts[b * ncl + k] = cnt;
}
template <typename T>
__global__ void seg_mean_id_bwd_kernel(const float* __restrict__ d_out, const T* __restrict__ v,
                                       const int32_t* __restrict__ cid, const int32_t* __restrict__ offsets,
                                       const int32_t* __restrict__ counts, int rows, int bags, int width, int ncl,
                                       int relu_mask, T* __restrict__ d_v) {
  pdl_prologue();
  int row = blockIdx.x;
  int b = bag_of_row(offsets, bags, row);
  int k = cid[row];
  bool ok = k >= 0 && k < ncl;
  float inv = ok ? 1.0f / (float)max(counts[b * ncl + k], 1) : 0.f;
  for (int c = threadIdx.x; c < width; c += blockDim.x) {
    float g = ok ? d_out[((size_t)b * ncl + k) * width + c] * inv : 0.f;
    if (relu_mask && !(ld1(v + (size_t)row * width + c) > 0.f)) g = 0.f;
    st1(d_v + (size_t)row * width + c, g);
  }
}

// =============================================================================================
// region <-> patch index map (tools/big_to_small_patching.py:40-46,59-76)
// =============================================================================================
__global__ void region_index_map_kernel(const int64_t* __restrict__ c2, int m, int psize, int scale, double* __restrict__ c1) {
  pdl_prologue();
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  int s2 = scale * scale;
  if (i >= m * s2) return;
  int k = i / s2, within = i % s2;
  int jj = within / scale, ii = within % scale;  // j outer (y), i inner (x)
  c1[2 * (size_t)i + 0] = (double)c2[2 * (size_t)k + 0] + (double)(ii * psize);
  c1[2 * (size_t)i + 1] = (double)c2[2 * (size_t)k + 1] + (double)(jj * psize);
}
__global__ void region_of_rows_kernel(int rows, int scale, int32_t* __restrict__ out) {
  pdl_prologue();
  int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= rows) return;
  int s2 = scale * scale;
  out[3 * (size_t)n + 0] = n / s2;
  out[3 * (size_t)n + 1] = (n % s2) / scale;
  out[3 * (size_t)n + 2] = n % scale;
}

}  // namespace advmil

// =============================================================================================
// C ABI for the kernels of this file
// =============================================================================================
using namespace advmil;

extern "C" int advmil_disc_loss(const float* f_real, const float* f_fake, const uint8_t* real_mask, int32_t bags,
                                int32_t which, float n_real, float n_fake, float* loss_out, float* d_real, float* d_fake,
                                void* stream) {
  ProfScope ps_(PROF_LOSS_OPT, (cudaStream_t)stream);
  ADVMIL_REQUIRE(bags > 0 && which >= 0 && which <= 2 && n_fake > 0.f, "disc_loss: bad arguments");
  launch_k(disc_loss_kernel, dim3(1), dim3(256), 0, (cudaStream_t)stream, f_real, f_fake, real_mask, bags, which, n_real, n_fake, loss_out, d_real, d_fake);
  ADVMIL_CHECK_LAUNCH();
  return ADVMIL_OK;
}

extern "C" int advmil_gen_loss(const float* pred, const float* t, const float* e, const uint8_t* visible,
                               const float* f_fake, int32_t bags, float n_visible, float n_fake, float coef_gan,
                               float alpha, float gamma, int32_t norm, float* losses, float* d_pred, float* d_fake,
                               void* stream) {
  ProfScope ps_(PROF_LOSS_OPT, (cudaStream_t)stream);
  ADVMIL_REQUIRE(bags > 0 && n_fake > 0.f && (norm == 0 || norm == 1), "gen_loss: bad arguments");
  launch_k(gen_loss_kernel, dim3(1), dim3(256), 0, (cudaStream_t)stream, pred, t, e, visible, f_fake, bags, n_visible, n_fake, coef_gan, alpha, gamma, norm, losses, d_pred, d_fake);
  ADVMIL_CHECK_LAUNCH();
  return ADVMIL_OK;
}

extern "C" int advmil_adam_step(float* param, const float* grad, float* m, float* v, const uint8_t* wd_mask, int64_t n,
                                float lr, float beta1, float beta2, float eps, float weight_decay, float l1_coef,
                                int32_t step, float grad_scale, void* stream) {
  ProfScope ps_(PROF_LOSS_OPT, (cudaStream_t)stream);
  ADVMIL_REQUIRE(n >= 0 && step >= 1, "adam_step: bad arguments");
  if (n == 0) return ADVMIL_OK;
  double bc1 = 1.0 - pow((double)beta1, (double)step);
  double bc2 = 1.0 - pow((double)beta2, (double)step);
  launch_k(adam_kernel, dim3(cdiv(n, 256)), dim3(256), 0, (cudaStream_t)stream, param, grad, m, v, wd_mask, n, (float)(lr / bc1), beta1,
                                                                beta2, eps, weight_decay, l1_coef,
                                                                (float)(1.0 / sqrt(bc2)), grad_scale);
  ADVMIL_CHECK_LAUNCH();
  return ADVMIL_OK;
}

extern "C" int advmil_abs_sum(const float* p, int64_t n, float* out, void* stream) {
  ProfScope ps_(PROF_LOSS_OPT, (cudaStream_t)stream);
  if (n <= 0) return ADVMIL_OK;
  launch_kc(abs_sum_kernel, dim3(ABS_CS), dim3(1024), 0, (cudaStream_t)stream, ABS_CS, p, n, out);
  ADVMIL_CHECK_LAUNCH();
  return ADVMIL_OK;
}

extern "C" size_t advmil_segment_mean_workspace_bytes(int32_t rows, int32_t bags, int32_t width, int32_t num_clusters) {
  size_t nparts = (size_t)rows / CL_CH + bags + 1;
  return align_up(nparts * num_clusters * width * sizeof(float), 256) + align_up(nparts * num_clusters * sizeof(int32_t), 256);
}

extern "C" int advmil_segment_mean_by_id_fwd(const void* v, int32_t elem, const int32_t* cid, const int32_t* offsets,
                                             const int32_t* offsets_host, int32_t rows, int32_t bags, int32_t width,
                                             int32_t num_clusters, float* out, int32_t* counts, void* workspace,
                                             size_t workspace_bytes, void* stream) {
  ADVMIL_REQUIRE(num_clusters > 0 && num_clusters <= CL_MAX && width > 0, "segment_mean_by_id: bad arguments");
  ADVMIL_REQUIRE((size_t)num_clusters * width * sizeof(float) <= 96 * 1024, "segment_mean_by_id: clusters*width too large");
  cudaStream_t st = (cudaStream_t)stream;
  size_t nparts = (size_t)rows / CL_CH + bags + 1;
  Workspace ws(workspace, workspace_bytes);
  float* part = ws.take<float>(nparts * num_clusters * width);
  int32_t* part_cnt = ws.take<int32_t>(nparts * num_clusters);
  if (!part || !part_cnt) { set_error("segment_mean_by_id: workspace too small"); return ADVMIL_ERR_WORKSPACE; }
  int maxlen = 0;
  for (int b = 0; b < bags; ++b) maxlen = max(maxlen, offsets_host[b + 1] - offsets_host[b]);
  int maxchunks = max(1, cdiv(maxlen, CL_CH));
  size_t smem = (size_t)num_clusters * width * sizeof(float);
  if (smem + SEG_MEAN_STATIC_SMEM > 48 * 1024) {
    ADVMIL_CHECK_CUDA(cudaFuncSetAttribute(seg_mean_id_partial_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    ADVMIL_CHECK_CUDA(cudaFuncSetAttribute(seg_mean_id_partial_kernel<bf16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  }
  if (elem == ELEM_BF16)
    launch_k(seg_mean_id_partial_kernel<bf16>, dim3(dim3(maxchunks, bags)), dim3(256), smem, st, (const bf16*)v, cid, offsets, width, num_clusters, part, part_cnt);
  else
    launch_k(seg_mean_id_partial_kernel<float>, dim3(dim3(maxchunks, bags)), dim3(256), smem, st, (const float*)v, cid, offsets, width, num_clusters, part, part_cnt);
  ADVMIL_CHECK_LAUNCH();
  launch_k(seg_mean_id_final_kernel, dim3(bags * num_clusters), dim3(128), 0, st, part, part_cnt, offsets, width, num_clusters, out, counts);
  ADVMIL_CHECK_LAUNCH();
  return ADVMIL_OK;
}

extern "C" int advmil_segment_mean_by_id_bwd(const float* d_out, const void* v, int32_t elem, const int32_t* cid,
                                             const int32_t* offsets, const int32_t* counts, int32_t rows, int32_t bags,
                                             int32_t width, int32_t num_clusters, int32_t relu_mask, void* d_v,
                                             void* stream) {
  if (rows == 0) return ADVMIL_OK;
  if (elem == ELEM_BF16)
    launch_k(seg_mean_id_bwd_kernel<bf16>, dim3(rows), dim3(128), 0, (cudaStream_t)stream, d_out, (const bf16*)v, cid, offsets, counts, rows, bags, width, num_clusters, relu_mask, (bf16*)d_v);
  else
    launch_k(seg_mean_id_bwd_kernel<float>, dim3(rows), dim3(128), 0, (cudaStream_t)stream, d_out, (const float*)v, cid, offsets, counts, rows, bags, width, num_clusters, relu_mask, (float*)d_v);
  ADVMIL_CHECK_LAUNCH();
  return ADVMIL_OK;
}

__global__ void dropout_mask_kernel(Drop d, Drop d2, int role, int rows, int width, uint8_t* __restrict__ out) {
  pdl_prologue();
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (size_t)rows * width) return;
  const uint32_t row = (uint32_t)(i / width), col = (uint32_t)(i % width);
  bool k;
  if (role == 0) k = d.keep(row, col);
  else { bool ka, kb; gate_keep(d, d2, row, col, ka, kb); k = role == 1 ? ka : kb; }
  out[i] = k ? 1 : 0;
}
extern "C" int advmil_dropout_mask(uint64_t seed, int32_t site, float p, int32_t rows, int32_t width, uint8_t* out, void* stream) {
  ADVMIL_REQUIRE(out && rows >= 0 && width > 0 && p >= 0.f && p < 1.f, "dropout_mask: bad arguments");
  const bool gate_a = site == SITE_A || site == SITE_GA, gate_b = site == SITE_B || site == SITE_GS;
  const int role = gate_a ? 1 : gate_b ? 2 : 0;
  Drop d = Drop::make(nullptr, seed, gate_b ? site - 1 : site, p, 1, width);   // the pair is keyed by the tanh site
  Drop d2 = Drop::make(nullptr, seed, gate_b ? site : site + 1, p, 1, width);
  if (role != 0) Drop::pair_gate(d, d2);      // joint keep bit on the tanh site, all-ones on the sigmoid site
  const size_t n = (size_t)rows * width;
  if (n == 0) return ADVMIL_OK;
  launch_k(dropout_mask_kernel, dim3(cdiv(n, 256)), dim3(256), 0, (cudaStream_t)stream, d, d2, role, rows, width, out);
  ADVMIL_CHECK_LAUNCH();
  return ADVMIL_OK;
}

// =============================================================================================
// Harrell's C (eval/cindex.py:82-143): one thread per event sample i, all j; integer counts via block reduce + atomics
// =============================================================================================
template <typename T>
__global__ void __launch_bounds__(256) cindex_kernel(const T* __restrict__ t, const T* __restrict__ e,
                                                     const T* __restrict__ pred, int n, T tol,
                                                     unsigned long long* __restrict__ counts) {
  pdl_prologue();
  __shared__ unsigned long long sm[3][8];
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  unsigned long long con = 0, tie = 0, cmp = 0;
  if (i < n && e[i] != (T)0) {
    const T ti = t[i], ri = -pred[i];
    for (int j = 0; j < n; ++j) {
      const T tj = t[j];
      const bool comparable = (tj > ti) || (tj == ti && e[j] == (T)0);   // j == i: equal time and an event -> false
      if (!comparable) continue;
      const T rj = -pred[j];
      const T diff = rj - ri;
      const bool is_tie = (diff < (T)0 ? -diff : diff) <= tol;
      cmp += 1;
      tie += is_tie ? 1 : 0;
      con += (!is_tie && rj < ri) ? 1 : 0;
    }
  }
  for (int o = 16; o > 0; o >>= 1) {
    con += __shfl_xor_sync(0xffffffffu, con, o); tie += __shfl_xor_sync(0xffffffffu, tie, o); cmp += __shfl_xor_sync(0xffffffffu, cmp, o);
  }
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  if (lane == 0) { sm[0][wid] = con; sm[1][wid] = tie; sm[2][wid] = cmp; }
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned long long c0 = 0, c1 = 0, c2 = 0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) { c0 += sm[0][w]; c1 += sm[1][w]; c2 += sm[2][w]; }
    atomicAdd(counts + 0, c0); atomicAdd(counts + 1, c1); atomicAdd(counts + 2, c2); atomicAdd(counts + 3, c2 - c0 - c1);
  }
}
extern "C" int advmil_cindex_counts(const float* t, const float* e, const float* pred, int32_t n, float tied_tol,
                                    int64_t* counts, void* stream) {
  ADVMIL_REQUIRE(t && e && pred && counts && n >= 2, "cindex_counts: need at least two samples (eval/cindex.py:72-73)");
  cudaStream_t st = (cudaStream_t)stream;
  ADVMIL_CHECK_CUDA(cudaMemsetAsync(counts, 0, 4 * sizeof(int64_t), st));
  launch_k(cindex_kernel<float>, dim3(cdiv(n, 256)), dim3(256), 0, st, t, e, pred, n, tied_tol, (unsigned long long*)counts);
  ADVMIL_CHECK_LAUNCH();
  return ADVMIL_OK;
}
extern "C" int advmil_cindex_counts_f64(const double* t, const double* e, const double* pred, int32_t n, double tied_tol,
                                        int64_t* counts, void* stream) {
  ADVMIL_REQUIRE(t && e && pred && counts && n >= 2, "cindex_counts_f64: need at least two samples (eval/cindex.py:72-73)");
  cudaStream_t st = (cudaStream_t)stream;
  ADVMIL_CHECK_CUDA(cudaMemsetAsync(counts, 0, 4 * sizeof(int64_t), st));
  launch_k(cindex_kernel<double>, dim3(cdiv(n, 256)), dim3(256), 0, st, t, e, pred, n, tied_tol, (unsigned long long*)counts);
  ADVMIL_CHECK_LAUNCH();
  return ADVMIL_OK;
}

extern "C" int advmil_region_index_map(const int64_t* coords_l2, int32_t m, int32_t patch_size, int32_t scale,
                                       double* coords_l1, void* stream) {
  ADVMIL_REQUIRE(m >= 0 && scale > 0, "region_index_map: bad arguments");
  if (m == 0) return ADVMIL_OK;
  launch_k(region_index_map_kernel, dim3(cdiv((long long)m * scale * scale, 256)), dim3(256), 0, (cudaStream_t)stream, coords_l2, m, patch_size, scale, coords_l1);
  ADVMIL_CHECK_LAUNCH();
  return ADVMIL_OK;
}

extern "C" int advmil_region_of_rows(int32_t rows, int32_t scale, int32_t* out, void* stream) {
  if (rows == 0) return ADVMIL_OK;
  launch_k(region_of_rows_kernel, dim3(cdiv(rows, 256)), dim3(256), 0, (cudaStream_t)stream, rows, scale, out);
  ADVMIL_CHECK_LAUNCH();
  return ADVMIL_OK;
}
