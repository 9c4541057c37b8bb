// Shared device/host helpers for the advmil_b200 kernels (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>
#include <math.h>
#include "../../include/advmil_b200.h"

namespace advmil {

// ---- error plumbing -------------------------------------------------------------------------
void set_error(const char* fmt, ...);
void count_launch(int n = 1);

#define ADVMIL_CHECK_CUDA(expr)                                                        \
  do {                                                                                 \
    cudaError_t _e = (expr);                                                           \
    if (_e != cudaSuccess) {                                                           \
      ::advmil::set_error("%s:%d %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e)); \
      return ADVMIL_ERR_CUDA;                                                          \
    }                                                                                  \
  } while (0)

#define ADVMIL_CHECK_LAUNCH()                                                          \
  do {                                                                                 \
    ::advmil::count_launch();                                                          \
    cudaError_t _e = cudaGetLastError();                                               \
    if (_e != cudaSuccess) {                                                           \
      ::advmil::set_error("%s:%d launch -> %s", __FILE__, __LINE__, cudaGetErrorString(_e)); \
      return ADVMIL_ERR_CUDA;                                                          \
    }                                                                                  \
  } while (0)

#define ADVMIL_REQUIRE(cond, ...)                                                      \
  do {                                                                                 \
    if (!(cond)) {                                                                     \
      ::advmil::set_error(__VA_ARGS__);                                                \
      return ADVMIL_ERR_INVALID;                                                       \
    }                                                                                  \
  } while (0)

#define ADVMIL_TRY(expr)                                                               \
  do {                                                                                 \
    int _s = (expr);                                                                   \
    if (_s != ADVMIL_OK) return _s;                                                    \
  } while (0)

// ---- programmatic dependent launch (PDL) -----------------------------------------------------------------------------
// A step is ~85 dependent launches, half of them region-level kernels of a few microseconds.  Every kernel is launched
// with cudaLaunchAttributeProgrammaticStreamSerialization and starts with pdl_prologue(): it lets ITS dependents be
// scheduled right away (their CTAs become resident while this grid still runs) and then waits until the grid(s) it
// depends on have completed and flushed, so no kernel touches memory before its predecessor in the stream is done.  The
// gain is the launch/scheduling latency between dependent kernels.
__device__ __forceinline__ void pdl_prologue() {
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  asm volatile("griddepcontrol.wait;" ::: "memory");
}
template <typename... Exp, typename... Act>
static inline void launch_kc(void (*kern)(Exp...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, unsigned cluster_x,
                             Act&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute at[2];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  unsigned n = 1;
  if (cluster_x > 1) {
    at[n].id = cudaLaunchAttributeClusterDimension;
    at[n].val.clusterDim.x = cluster_x; at[n].val.clusterDim.y = 1; at[n].val.clusterDim.z = 1;
    ++n;
  }
  cfg.attrs = at; cfg.numAttrs = n;
  (void)cudaLaunchKernelEx(&cfg, kern, static_cast<Act&&>(args)...);   // the status is read by ADVMIL_CHECK_LAUNCH()
}
template <typename... Exp, typename... Act>
static inline void launch_k(void (*kern)(Exp...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Act&&... args) {
  launch_kc(kern, grid, block, smem, st, 1u, static_cast<Act&&>(args)...);
}

// ---- optional per-stage CUDA-event profiling (bench.py roofline) ---------------------------------
enum ProfTag : int {
  PROF_PROJ = 0,        // K1  x.W1^T + bias + ReLU (+dropout)
  PROF_GATE = 1,        // K2  gated attention scores
  PROF_POOL = 2,        // K3  segmented softmax + pooling
  PROF_EMBED = 3,       // K5+K6 projection + LN + ReLU + region mean
  PROF_POOL_BWD = 4,    // pooling + gate backward (row stream)
  PROF_BWD_DATA = 5,    // dh = dAB.[Wa;Wb] (+pool term, ReLU mask)
  PROF_BWD_W_GATE = 6,  // d[Wa;Wb] = dAB^T h
  PROF_BWD_W_PROJ = 7,  // dW1 = dh^T x
  PROF_LN_BWD = 8,      // LN/ReLU/region-mean backward (row stream)
  PROF_BWD_W_EMBED = 9, // dWc = dy^T x
  PROF_COLSUM = 10,     // bias gradients
  PROF_DROPOUT = 11,    // dropout re-application on cached eval activations
  PROF_HEAD_FWD = 12,   // RLIP head forward (region MLP, GAPool, bag MLP, time embedding, inner product)
  PROF_HEAD_BWD = 13,   // RLIP head backward
  PROF_GEN_TAIL = 14,   // generator per-bag head fwd/bwd, small outer products, gate weight packing
  PROF_LOSS_OPT = 15,   // losses, Adam, L1 value
  PROF_PROJ_EMBED = 16, // K1 + K5/K6 fused over stacked weights (bf16 fused step)
  PROF_ATTN_FWD = 17,   // ESAT self-attention forward
  PROF_ATTN_BWD = 18,   // ESAT self-attention backward (dQ pass + dK/dV pass)
  PROF_PROJ_SEGMEAN = 19, // K9: DeepAttMISL projection + ReLU + per-(bag, cluster) mean in one pass (+ finalize)
  PROF_NTAGS = 20
};
struct ProfScope {
  int tag; cudaStream_t st; void* rec;
  ProfScope(int tag, cudaStream_t st);
  ~ProfScope();
};

static inline int cdiv(long long a, long long b) { return (int)((a + b - 1) / b); }
static inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// Bump allocator over the caller-provided workspace.
struct Workspace {
  char* base;
  size_t cap, used;
  Workspace(void* p, size_t n) : base((char*)p), cap(n), used(0) {}
  template <class T>
  T* take(size_t count) {
    size_t bytes = align_up(count * sizeof(T), 256);
    if (used + bytes > cap || base == nullptr) return nullptr;
    T* r = (T*)(base + used);
    used += bytes;
    return r;
  }
};

// ---- dropout keep bits: counter-based, identical in forward and backward ----------------------
// Sites (one id per dropout layer of the reference):
enum DropSite : int {
  SITE_H = 1, SITE_A = 2, SITE_B = 3, SITE_RHO = 4, SITE_MLP0 = 5,           // generator
  SITE_FC1 = 11, SITE_GA = 12, SITE_GS = 13, SITE_FC2 = 14,                   // discriminator
  SITE_ATT = 21, SITE_SA = 22, SITE_FF1 = 23, SITE_FF2 = 24,                  // ESAT encoder layer
  SITE_USER = 100
};

__host__ __device__ __forceinline__ uint64_t mix64(uint64_t z) {
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL;
  return z ^ (z >> 31);
}

// uniform in [0,1) with 24 bits from (seed, site, element index)
__host__ __device__ __forceinline__ float rng_uniform(uint64_t seed, int site, uint64_t idx) {
  uint64_t r = mix64(seed + 0x9E3779B97F4A7C15ULL * (uint64_t)(site + 1) + mix64(idx + 0xD1B54A32D192ED03ULL));
  return (float)(r >> 40) * (1.0f / 16777216.0f);
}

struct Drop {          // one dropout site
  const uint8_t* mask; // injected keep mask [rows, width] or nullptr
  uint64_t seed;
  float p;             // drop probability
  float inv_keep;      // 1/(1-p)
  int site;
  int active;          // train && p > 0
  int width;           // logical row width of the dropped tensor (index of an injected mask = row * width + col)
  uint32_t key;        // per-(seed, site) 32-bit key of the counter-based generator
  uint32_t thresh16;   // an element is dropped when its 16 random bits < thresh16 (= round(p * 2^16))
  uint32_t thresh8j;   // gate sites (Drop::pair_gate): a (tanh_j, sigmoid_j) pair is dropped when its 8 random bits < thresh8j
  __host__ static Drop make(const uint8_t* mask, uint64_t seed, int site, float p, int train, int width) {
    Drop d;
    d.mask = mask; d.seed = seed; d.site = site; d.p = p; d.width = width;
    d.active = (train && p > 0.f) ? 1 : 0;
    d.inv_keep = d.active ? 1.0f / (1.0f - p) : 1.0f;
    d.key = (uint32_t)(mix64(seed + 0x9E3779B97F4A7C15ULL * (uint64_t)(site + 1)) >> 32);
    double t = (double)p * 65536.0 + 0.5;
    d.thresh16 = t >= 65536.0 ? 65536u : (uint32_t)t;
    d.thresh8j = 0;
    return d;
  }
  // The two dropouts of a gated-attention pair (tanh_j and sigmoid_j, reference model/backbone_utils.py:15-22) only ever act
  // through their product: a_j b_j contributes, forward and backward, iff BOTH units are kept.  The in-kernel generator
  // therefore draws the JOINT keep bit, Bernoulli((1-p_a)(1-p_b)) -- the same distribution as two independent draws --
  // from 8 random bits per pair (one 32-bit draw serves 4 pairs; the joint drop probability is quantised to 2^-8:
  // p = 0.25 -> 112/256 exactly).  Materialised masks (advmil_dropout_mask) carry the joint bit on the tanh site and
  // all-ones on the sigmoid site.  Injected masks are used as given.
  __host__ static void pair_gate(Drop& a, Drop& b) {
    const double pj = 1.0 - (1.0 - (a.active ? (double)a.p : 0.0)) * (1.0 - (b.active ? (double)b.p : 0.0));
    const double t = pj * 256.0 + 0.5;
    a.thresh8j = b.thresh8j = t >= 256.0 ? 256u : (uint32_t)t;
  }
  // 32 random bits of the counter (row, col): 2-D multiply-xor counter + murmur3 finaliser, ~9 integer instructions.
  // One draw serves TWO elements (16 bits each; the keep probability is quantised to 2^-16, a relative bias < 2e-5):
  // columns (2k, 2k+1) of a plain site, or the (tanh_j, sigmoid_j) pair of a gate.  Forward and backward regenerate the
  // same bits from (seed, site, row, col).
  __device__ __forceinline__ uint32_t bits(uint32_t row, uint32_t col) const {
    uint32_t x = (row * 0x9E3779B1u) ^ (col * 0x85EBCA77u + key);
    x ^= x >> 16; x *= 0x85EBCA6Bu; x ^= x >> 13; x *= 0xC2B2AE35u; x ^= x >> 16;
    return x;
  }
  __device__ __forceinline__ bool keep(uint32_t row, uint32_t col) const {
    if (mask) return mask[(size_t)row * width + col] != 0;
    const uint32_t h = bits(row, col & ~1u);
    return ((col & 1u) ? (h >> 16) : (h & 0xFFFFu)) >= thresh16;
  }
  // columns col (even) and col + 1 from one draw
  __device__ __forceinline__ void keep2(uint32_t row, uint32_t col_even, bool& k0, bool& k1) const {
    if (mask) { k0 = mask[(size_t)row * width + col_even] != 0; k1 = mask[(size_t)row * width + col_even + 1] != 0; return; }
    const uint32_t h = bits(row, col_even);
    k0 = (h & 0xFFFFu) >= thresh16; k1 = (h >> 16) >= thresh16;
  }
  // multiplicative factor: 0 or 1/(1-p); 1 when inactive
  __device__ __forceinline__ float scale(uint32_t row, uint32_t col) const {
    if (!active) return 1.0f;
    return keep(row, col) ? inv_keep : 0.0f;
  }
};

// keep bits of the (tanh_j, sigmoid_j) pair of a gated-attention row: the joint bit of Drop::pair_gate (byte j % 4 of the
// draw of pair group j / 4, keyed by the tanh site) when neither site has an injected mask
__device__ __forceinline__ void gate_keep(const Drop& da, const Drop& db, uint32_t row, uint32_t j, bool& ka, bool& kb) {
  if (!da.mask && !db.mask) {
    const uint32_t h = da.bits(row, j & ~3u);
    ka = ((h >> (8u * (j & 3u))) & 0xFFu) >= da.thresh8j;
    kb = true;
    return;
  }
  uint32_t h = 0;
  if (!da.mask || !db.mask) h = da.bits(row, j);
  ka = da.mask ? da.mask[(size_t)row * da.width + j] != 0 : (h & 0xFFFFu) >= da.thresh16;
  kb = db.mask ? db.mask[(size_t)row * db.width + j] != 0 : (h >> 16) >= db.thresh16;
}

// ---- element types of the [rows, width] activation tensors ------------------------------------------
// fp32 / tf32 modes keep them in fp32; the bf16 mode (ADVMIL_BF16) keeps x, h, ab, dAB, dh, y_pre, d_y in bfloat16
// (half the HBM bytes, kind::f16 tensor-core rate) while every accumulation, statistic and parameter stays fp32.
typedef __nv_bfloat16 bf16;
enum ElemType : int { ELEM_F32 = 0, ELEM_BF16 = 1 };
template <typename T> struct ElemOf;
template <> struct ElemOf<float> { static constexpr int value = ELEM_F32; };
template <> struct ElemOf<bf16> { static constexpr int value = ELEM_BF16; };
static inline size_t elem_bytes(int dt) { return dt == ELEM_BF16 ? 2 : 4; }
static inline int elem_of_precision(int precision) { return precision == ADVMIL_BF16 ? ELEM_BF16 : ELEM_F32; }

__device__ __forceinline__ float bf_lo(uint32_t u) { return __uint_as_float(u << 16); }
__device__ __forceinline__ float bf_hi(uint32_t u) { return __uint_as_float(u & 0xFFFF0000u); }
__device__ __forceinline__ uint32_t pack_bf2(float lo, float hi) {
  __nv_bfloat162 t = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&t);
}
__device__ __forceinline__ float ld1(const float* p) { return *p; }
__device__ __forceinline__ float ld1(const bf16* p) { return __bfloat162float(*p); }
__device__ __forceinline__ void st1(float* p, float v) { *p = v; }
__device__ __forceinline__ void st1(bf16* p, float v) { *p = __float2bfloat16_rn(v); }
// 4 consecutive elements (16-byte / 8-byte aligned)
__device__ __forceinline__ float4 ld4(const float* p) { return *reinterpret_cast<const float4*>(p); }
__device__ __forceinline__ float4 ld4(const bf16* p) {
  const uint2 u = *reinterpret_cast<const uint2*>(p);
  return make_float4(bf_lo(u.x), bf_hi(u.x), bf_lo(u.y), bf_hi(u.y));
}
__device__ __forceinline__ void st4(float* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }
__device__ __forceinline__ void st4(bf16* p, float4 v) {
  *reinterpret_cast<uint2*>(p) = make_uint2(pack_bf2(v.x, v.y), pack_bf2(v.z, v.w));
}
// one 16-byte vector = VecN<T>::N consecutive elements
template <typename T> struct VecN { static constexpr int N = 16 / (int)sizeof(T); };
__device__ __forceinline__ void ldv(const float* p, float (&o)[4]) {
  const float4 v = *reinterpret_cast<const float4*>(p);
  o[0] = v.x; o[1] = v.y; o[2] = v.z; o[3] = v.w;
}
__device__ __forceinline__ void ldv(const bf16* p, float (&o)[8]) {
  const uint4 u = *reinterpret_cast<const uint4*>(p);
  o[0] = bf_lo(u.x); o[1] = bf_hi(u.x); o[2] = bf_lo(u.y); o[3] = bf_hi(u.y);
  o[4] = bf_lo(u.z); o[5] = bf_hi(u.z); o[6] = bf_lo(u.w); o[7] = bf_hi(u.w);
}
__device__ __forceinline__ void stv(float* p, const float (&o)[4]) {
  *reinterpret_cast<float4*>(p) = make_float4(o[0], o[1], o[2], o[3]);
}
__device__ __forceinline__ void stv(bf16* p, const float (&o)[8]) {
  *reinterpret_cast<uint4*>(p) = make_uint4(pack_bf2(o[0], o[1]), pack_bf2(o[2], o[3]), pack_bf2(o[4], o[5]), pack_bf2(o[6], o[7]));
}

// one 4-byte word = 1 fp32 or 2 bf16 consecutive elements
__device__ __forceinline__ void ldw(const float* p, float (&o)[1]) { o[0] = *p; }
__device__ __forceinline__ void ldw(const bf16* p, float (&o)[2]) {
  const uint32_t u = *reinterpret_cast<const uint32_t*>(p);
  o[0] = bf_lo(u); o[1] = bf_hi(u);
}

// ---- warp helpers -----------------------------------------------------------------------------
__device__ __forceinline__ float oct_sum(float v) {  // over 8 consecutive lanes (aligned groups)
#pragma unroll
  for (int o = 4; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ float half_warp_sum(float v) {  // over 16 consecutive lanes
#pragma unroll
  for (int o = 8; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// block-wide sum / max through shared memory (blockDim.x multiple of 32, <= 1024); all threads get the result
__device__ __forceinline__ float block_sum(float v, float* red /*[33]*/) {
  int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
  v = warp_sum(v);
  __syncthreads();
  if (lane == 0) red[wid] = v;
  __syncthreads();
  if (wid == 0) {
    float t = lane < nw ? red[lane] : 0.f;
    t = warp_sum(t);
    if (lane == 0) red[32] = t;
  }
  __syncthreads();
  return red[32];
}
__device__ __forceinline__ float block_max(float v, float* red) {
  int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
  v = warp_max(v);
  __syncthreads();
  if (lane == 0) red[wid] = v;
  __syncthreads();
  if (wid == 0) {
    float t = lane < nw ? red[lane] : -INFINITY;
    t = warp_max(t);
    if (lane == 0) red[32] = t;
  }
  __syncthreads();
  return red[32];
}

__device__ __forceinline__ float sigmoidf_(float v) { return 1.0f / (1.0f + expf(-v)); }

// bag of a packed row by binary search over offsets[0..bags]
__device__ __forceinline__ int bag_of_row(const int32_t* __restrict__ offsets, int bags, int row) {
  int lo = 0, hi = bags;  // invariant: offsets[lo] <= row < offsets[hi]
  while (hi - lo > 1) {
    int mid = (lo + hi) >> 1;
    if (offsets[mid] <= row) lo = mid; else hi = mid;
  }
  return lo;
}

// packed gate layout: tanh_j at 128*(j/64) + j%64, sigmoid_j at +64
__host__ __device__ __forceinline__ int gate_width(int D) { return 128 * ((D + 63) / 64); }
__host__ __device__ __forceinline__ int gate_col_a(int j) { return 128 * (j >> 6) + (j & 63); }

}  // namespace advmil
