// K9 of the DeepAttMISL generator (model/backbone.py:105-117): hc[b, c] = mean over the rows n of bag b with cid[n] == c of
// relu(x[n] W^T + bias), zeros for an empty cluster.  The tcgen05 pass (gemm_tc.cu, EPI_POOL) reduces the activation in its
// epilogue into one partial per (128-row tile, bag, cluster); the finalize kernel below adds a bag's partials in tile order
// and divides by the count.  The [rows, h] activation never reaches HBM: only its ReLU keep bits (1 bit per element) are
// kept for the backward, which expands d_hc into d_hx[n] = keep(n) * d_hc[bag(n), cid(n)] / count.
#include "gemm_tc.cuh"

namespace advmil {

// one CTA per (bag, cluster): the count over the bag's ids, then the column sums of the bag's tiles t in [beg / 128,
// (end - 1) / 128] (partial index t + bag, as the epilogue writes them).  Per 32-column chunk warp w adds tiles t0 + w,
// t0 + w + 8, ... and warp 0 adds the 8 warp sums in order: a fixed order, 8 independent load chains per column.
__global__ void __launch_bounds__(256) cluster_pool_finalize_kernel(const float* __restrict__ part, const int32_t* __restrict__ cid,
                                                                    const int32_t* __restrict__ offsets, int N, int ncl,
                                                                    float* __restrict__ out, int32_t* __restrict__ counts) {
  pdl_prologue();
  __shared__ int red[8];
  __shared__ float psum[8][32];
  const int b = blockIdx.x / ncl, k = blockIdx.x % ncl;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int beg = offsets[b], end = offsets[b + 1];
  int c = 0;
  for (int r = beg + threadIdx.x; r < end; r += blockDim.x) c += cid[r] == k ? 1 : 0;
  for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
  if (lane == 0) red[warp] = c;
  __syncthreads();
  int cnt = 0;
  for (int w = 0; w < 8; ++w) cnt += red[w];
  const int t0 = beg / 128, t1 = end > beg ? (end - 1) / 128 : t0 - 1;
  for (int c0 = 0; c0 < N; c0 += 32) {             // N % 32 == 0
    float t = 0.f;
#pragma unroll 4
    for (int tl = t0 + warp; tl <= t1; tl += 8) t += part[((size_t)(tl + b) * ncl + k) * N + c0 + lane];
    psum[warp][lane] = t;
    __syncthreads();
    if (warp == 0) {
      float s = 0.f;
#pragma unroll
      for (int w = 0; w < 8; ++w) s += psum[w][lane];
      out[((size_t)b * ncl + k) * N + c0 + lane] = cnt > 0 ? s / (float)cnt : 0.f;   // zeros for an empty cluster (backbone.py:114-115)
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) counts[b * ncl + k] = cnt;
}

// d_hx[n, 8 g .. 8 g + 7] from the keep bits; rows whose id is outside [0, ncl) get zeros
template <typename T>
__global__ void cluster_pool_bwd_kernel(const float* __restrict__ d_hc, const uint32_t* __restrict__ keep, const int32_t* __restrict__ cid,
                                        const int32_t* __restrict__ offsets, const int32_t* __restrict__ counts, int rows, int bags,
                                        int N, int ncl, T* __restrict__ d_hx) {
  pdl_prologue();
  const int G = N / 8;
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (size_t)rows * G) return;
  const int row = (int)(i / G), g = (int)(i - (size_t)row * G);
  const int k = cid[row];
  float v[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) v[e] = 0.f;
  if (k >= 0 && k < ncl) {
    const int b = bag_of_row(offsets, bags, row);
    const float inv = 1.0f / (float)max(counts[b * ncl + k], 1);
    const uint32_t bits = (keep[(size_t)row * (N / 32) + (g >> 2)] >> ((g & 3) * 8)) & 0xFFu;
    const float4* src = reinterpret_cast<const float4*>(d_hc + ((size_t)b * ncl + k) * N + 8 * g);
    const float4 a = src[0], c = src[1];
    const float d[8] = {a.x, a.y, a.z, a.w, c.x, c.y, c.z, c.w};
#pragma unroll
    for (int e = 0; e < 8; ++e) v[e] = ((bits >> e) & 1u) ? d[e] * inv : 0.f;
  }
  T* dst = d_hx + (size_t)row * N + 8 * g;
  if constexpr (sizeof(T) == 2) {
    stv(dst, v);
  } else {
    stv(dst, *reinterpret_cast<const float(*)[4]>(v));
    stv(dst + 4, *reinterpret_cast<const float(*)[4]>(v + 4));
  }
}

static int check_cluster_bags(const int32_t* offsets_host, int rows, int bags, int ncl) {
  ADVMIL_REQUIRE(ncl >= 1 && ncl <= CLUSTER_POOL_MAX, "cluster_pool: num_clusters %d outside 1..%d", ncl, CLUSTER_POOL_MAX);
  ADVMIL_REQUIRE(bags >= 1 && offsets_host && offsets_host[0] == 0 && offsets_host[bags] == rows, "cluster_pool: bad bag offsets");
  for (int i = 0; i < bags; ++i)
    ADVMIL_REQUIRE((offsets_host[i + 1] - offsets_host[i]) % 16 == 0 && offsets_host[i + 1] >= offsets_host[i],
                   "bags: bag %d has a length that is not a multiple of 16 (model/backbone_utils.py:65)", i);
  return ADVMIL_OK;
}

bool cluster_pool_fused(int rows, int C, int h, int precision) {
  return precision != ADVMIL_FP32 && h % 32 == 0 && tc_proj_pool_supported(rows, C, h, elem_of_precision(precision));
}
size_t cluster_pool_ws_floats(int rows, int bags, int h, int ncl) { return ((size_t)rows / 128 + bags + 1) * ncl * h; }

int cluster_pool_fwd(const void* x, const float* W, const float* b, const int32_t* cid, const int32_t* offsets,
                     const int32_t* offsets_host, int rows, int bags, int C, int h, int ncl, int precision, float* hc,
                     int32_t* counts, uint32_t* keep, float* ws, cudaStream_t st) {
  ADVMIL_TRY(check_cluster_bags(offsets_host, rows, bags, ncl));
  ADVMIL_REQUIRE(cluster_pool_fused(rows, C, h, precision),
                 "cluster_pool_fwd: no tcgen05 pass for rows=%d C=%d h=%d precision=%d (the fp32 mode composes linear_fwd and "
                 "segment_mean_by_id)", rows, C, h, precision);
  ADVMIL_TRY(tc_proj_pool_fwd(x, W, b, cid, offsets, bags, rows, C, h, ncl, keep, ws, precision, st));
  launch_k(cluster_pool_finalize_kernel, dim3(bags * ncl), dim3(256), 0, st, (const float*)ws, cid, offsets, h, ncl, hc, counts);
  ADVMIL_CHECK_LAUNCH();
  return ADVMIL_OK;
}

int cluster_pool_bwd(const float* d_hc, const uint32_t* keep, const int32_t* cid, const int32_t* offsets, const int32_t* counts,
                     int rows, int bags, int h, int ncl, int precision, void* d_hx, cudaStream_t st) {
  ADVMIL_REQUIRE(h % 32 == 0 && ncl >= 1 && ncl <= CLUSTER_POOL_MAX, "cluster_pool_bwd: h=%d (%%32) num_clusters=%d unsupported", h, ncl);
  if (rows == 0) return ADVMIL_OK;
  const size_t n = (size_t)rows * (h / 8);
  if (precision == ADVMIL_BF16)
    launch_k(cluster_pool_bwd_kernel<bf16>, dim3(cdiv(n, 256)), dim3(256), 0, st, d_hc, keep, cid, offsets, counts, rows, bags, h, ncl, (bf16*)d_hx);
  else
    launch_k(cluster_pool_bwd_kernel<float>, dim3(cdiv(n, 256)), dim3(256), 0, st, d_hc, keep, cid, offsets, counts, rows, bags, h, ncl, (float*)d_hx);
  ADVMIL_CHECK_LAUNCH();
  return ADVMIL_OK;
}

}  // namespace advmil

using namespace advmil;

extern "C" size_t advmil_cluster_pool_workspace_bytes(int32_t rows, int32_t bags, int32_t h, int32_t num_clusters) {
  return align_up(cluster_pool_ws_floats(rows, bags, h, num_clusters) * sizeof(float), 256) + 256;
}

extern "C" int advmil_cluster_pool_fwd(const void* x, const float* W, const float* b, const int32_t* cid, const int32_t* offsets,
                                       const int32_t* offsets_host, int32_t rows, int32_t bags, int32_t C, int32_t h,
                                       int32_t num_clusters, int32_t precision, float* hc, int32_t* counts, uint32_t* keep,
                                       void* workspace, size_t workspace_bytes, void* stream) {
  ADVMIL_REQUIRE(x && W && b && cid && offsets && hc && counts && workspace, "cluster_pool_fwd: null argument");
  cudaStream_t st = (cudaStream_t)stream;
  ProfScope ps(PROF_PROJ_SEGMEAN, st);
  Workspace ws(workspace, workspace_bytes);
  float* part = ws.take<float>(cluster_pool_ws_floats(rows, bags, h, num_clusters));
  if (!part) { set_error("cluster_pool_fwd: workspace too small (have %zu bytes)", workspace_bytes); return ADVMIL_ERR_WORKSPACE; }
  return cluster_pool_fwd(x, W, b, cid, offsets, offsets_host, rows, bags, C, h, num_clusters, precision, hc, counts, keep, part, st);
}

extern "C" int advmil_cluster_pool_bwd(const float* d_hc, const uint32_t* keep, const int32_t* cid, const int32_t* offsets,
                                       const int32_t* counts, int32_t rows, int32_t bags, int32_t h, int32_t num_clusters,
                                       int32_t precision, void* d_hx, void* stream) {
  ADVMIL_REQUIRE(d_hc && keep && cid && offsets && counts && d_hx, "cluster_pool_bwd: null argument");
  return cluster_pool_bwd(d_hc, keep, cid, offsets, counts, rows, bags, h, num_clusters, precision, d_hx, (cudaStream_t)stream);
}
