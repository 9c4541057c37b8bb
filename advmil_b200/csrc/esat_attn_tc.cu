// ESAT self-attention on the Blackwell tensor path (tcgen05 / TMEM / TMA), forward.
// Reference: nn.MultiheadAttention inside nn.TransformerEncoderLayer (reference model/backbone.py:171-196,
// model/backbone_utils.py:112-127): softmax(q k^T / sqrt(hd)) -> dropout -> . v per (bag, head) over the regions of a bag.
//
// One CTA owns 128 queries of one (bag, head) and walks the bag's keys in tiles of 128 (flash style, nothing of size
// R x R touches HBM).  q, k and v are read straight out of the packed projection qkv [R, 3d] (fp32) by TMA -- head h is
// columns [h hd, (h+1) hd) of each third -- as 128-byte-swizzled blocks of 32 columns (hd = 48: two blocks, the second half
// used), and consumed by tcgen05.mma.kind::tf32 as they are:
//   S  = Q K^T      A = Q (K-major), B = K tile (K-major)                      -> TMEM, 128 columns, double-buffered
//   P  = 2^(S c - m)  one query row per thread, written back over S IN TENSOR MEMORY (tcgen05.st), after dropout
//   Ot = P V        A = P (tensor memory), B = V tile (MN-major: v rows are the contraction index)
//                                                                            -> TMEM, 64 columns, double-buffered
//   o  = o * 2^(m_old - m_new) + Ot   in registers (the tile result is read back, the running output never leaves registers)
// Warp roles (608 threads): warps 0-7 and 8-15 are two softmax groups that own the even and the odd key tiles (each with its
// own S / P and P V columns in tensor memory, its own running maximum, sum and output; two threads -- column halves -- per
// query row exchange the row maximum inside the group; one group computes while the other waits for its MMAs; the two
// partial results are merged at the end), warp 16 MMA issuer, warp 17 TMA producer of q and the k tiles, warp 18 TMA producer of the v tiles (a k slot is free as soon as its S has
// retired, a v slot only after P V: separate rings keep the next S from waiting behind a P V plus a TMA round trip).
// Dropout keep bits: the same counter generator and indices as the FFMA kernels (esat_kernels.cu), so the backward
// pass regenerates them.
#include "stages.cuh"
#include "tc_ptx.cuh"
#include "esat_attn.cuh"

namespace advmil {
using namespace tc;

namespace {

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn get_encode() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess && qres == cudaDriverEntryPointSuccess)
      fn = (EncodeTiledFn)p;
  }
  return fn;
}
// row-major fp32 matrix [rows, cols]; box = 128 rows x 32 columns (128 bytes)
int make_map(CUtensorMap* m, const float* base, long long rows, long long cols, CUtensorMapSwizzle swz) {
  EncodeTiledFn enc = get_encode();
  if (!enc) { set_error("cuTensorMapEncodeTiled unavailable"); return ADVMIL_ERR_CUDA; }
  cuuint64_t gdim[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t gstr[1] = {(cuuint64_t)cols * sizeof(float)};
  cuuint32_t box[2] = {32u, 128u};
  cuuint32_t estr[2] = {1u, 1u};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, (void*)base, gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, swz,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { set_error("attention: cuTensorMapEncodeTiled failed (%d) rows=%lld cols=%lld", (int)r, rows, cols); return ADVMIL_ERR_CUDA; }
  return ADVMIL_OK;
}

constexpr int AT_TILE = 128;                 // queries per CTA = keys per tile
constexpr int AT_NH = 2;                     // threads per query row inside a softmax group (column halves of a key tile)
constexpr int AT_GW = 4 * AT_NH;             // warps per softmax group (TMEM lane quarter = warp % 4)
constexpr int AT_SOFT = 2 * AT_GW;           // softmax warps: two groups
constexpr int AT_THREADS = 32 * (AT_SOFT + 3);
constexpr int AT_BLK = 128 * 128;            // bytes of one [128 rows x 128 B] operand block
constexpr float kLog2eA = 1.4426950408889634f, kLn2A = 0.6931471805599453f;

template <int HD> struct AttCfg {
  static_assert(HD % 16 == 0 && HD >= 16 && HD <= 64, "head width");
  static constexpr int NB = (HD + 31) / 32;                  // 32-column blocks per operand
  static constexpr int Q_BYTES = NB * AT_BLK, KV_BYTES = NB * AT_BLK;
  static constexpr int OH = HD / AT_NH;                      // output columns per softmax thread
  static constexpr size_t USED = (size_t)Q_BYTES + 4 * (size_t)KV_BYTES + 2 * 2 * AT_NH * AT_TILE * 4 /*xm*/ + 16 * 8 /*barriers, TMEM address*/;
  static constexpr size_t SMEM = USED + 1024;                // + alignment slack
  static_assert((size_t)(HD + 1 + 2 * AT_NH) * AT_TILE * 4 <= (size_t)Q_BYTES + KV_BYTES, "merge buffer");
};

__device__ __forceinline__ float ex2a(float x) { float y; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
// tf32 rounding of a probability (0 <= p <= 1: finite, no overflow): the tensor core drops the low 13 mantissa bits, so
// half an ulp is added first -- one integer add instead of cvt.rna's four instructions
__device__ __forceinline__ uint32_t round_tf32_pos(float x) { return __float_as_uint(x) + 0x1000u; }
__device__ __forceinline__ void soft_bar() { asm volatile("bar.sync 1, %0;" ::"n"(32 * AT_SOFT) : "memory"); }
__device__ __forceinline__ void group_bar(int g) { asm volatile("bar.sync %0, %1;" ::"r"(2 + g), "n"(32 * AT_GW) : "memory"); }

// TMEM <-> registers, this warp's 32 lanes x N consecutive 32-bit columns
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float* v) {
  uint32_t r[16];
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
                 "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
               : "r"(taddr) : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, float* v) {
  uint32_t r[8];
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr) : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 8; ++i) v[i] = __uint_as_float(r[i]);
}
template <int N> __device__ __forceinline__ void tmem_ldn(uint32_t taddr, float (&v)[N]) {
  static_assert(N % 8 == 0 && N <= 64, "column count");
#pragma unroll
  for (int c = 0; c + 16 <= N; c += 16) tmem_ld16(taddr + c, v + c);
  if constexpr (N % 16 == 8) tmem_ld8(taddr + N - 8, v + N - 8);
}
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]), "r"(r[10]),
      "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]), "r"(r[18]), "r"(r[19]), "r"(r[20]),
      "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]),
      "r"(r[31])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
// D[tmem] (+)= A[tmem] * B[smem desc]: the A operand (128 lanes x K 32-bit columns) is read from tensor memory
__device__ __forceinline__ void mma_tf32_ta(uint32_t d_tmem, uint32_t a_tmem, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}" ::"r"(d_tmem),
      "r"(a_tmem), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}

template <int HD>
__global__ void __launch_bounds__(AT_THREADS, 1)
mha_fwd_tcgen05_kernel(const __grid_constant__ CUtensorMap tmK /*q, k: K-major*/, const __grid_constant__ CUtensorMap tmV /*v: MN-major*/,
                       const int32_t* __restrict__ ro, int d, float scale, AttDrop ad, float* __restrict__ ctx,
                       float* __restrict__ lse, int Rtot) {
  pdl_prologue();
  using Cfg = AttCfg<HD>;
  constexpr int NB = Cfg::NB;
  const int b = blockIdx.y, head = blockIdx.z, r0 = ro[b], Rb = ro[b + 1] - r0;
  const int q0 = blockIdx.x * AT_TILE;
  if (q0 >= Rb) return;
  const int T = (Rb + AT_TILE - 1) / AT_TILE;        // key tiles

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* Q_s = smem;
  uint8_t* K_s = Q_s + Cfg::Q_BYTES;                 // [2][NB blocks]
  uint8_t* V_s = K_s + 2 * Cfg::KV_BYTES;            // [2][NB blocks]
  float* xm = (float*)(V_s + 2 * Cfg::KV_BYTES);     // [2 groups][2 (iteration parity)][AT_NH][128] row maxima of the column halves
  uint64_t* bars = (uint64_t*)(xm + 2 * 2 * AT_NH * AT_TILE);
  uint64_t* qfull = bars;            // [1]
  uint64_t* kfull = bars + 1;        // [2]
  uint64_t* kfree = bars + 3;        // [2]
  uint64_t* vfull = bars + 5;        // [2]
  uint64_t* vfree = bars + 7;        // [2]
  uint64_t* sfull = bars + 9;        // [2]  S of the group's tile is in TMEM
  uint64_t* pfull = bars + 11;       // [2]  the group has replaced S by P (4 warp arrivals)
  uint64_t* ofull = bars + 13;       // [2]  P V of the group's tile is in TMEM
  uint32_t* tmem_ptr = (uint32_t*)(bars + 15);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    prefetch_tmap(&tmK);
    prefetch_tmap(&tmV);
    mbar_init(qfull, 1);
    for (int i = 0; i < 2; ++i) {
      mbar_init(&kfull[i], 1); mbar_init(&kfree[i], 1); mbar_init(&vfull[i], 1); mbar_init(&vfree[i], 1);
      mbar_init(&sfull[i], 1); mbar_init(&pfull[i], AT_GW); mbar_init(&ofull[i], 1);
    }
    fence_barrier_init();
  }
  if (warp == AT_SOFT) tmem_alloc(tmem_ptr, 512);     // S / P: 2 x 128 columns, P V: 2 x 64 columns
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;
  constexpr uint32_t S_COL = 0, O_COL = 256;

  if (warp == AT_SOFT + 1) {
    // ---------------- TMA producer: q once, then the k tiles ----------------
    if (lane == 0) {
      const int cq = head * HD, ck = d + head * HD;
      mbar_arrive_expect_tx(qfull, Cfg::Q_BYTES);
#pragma unroll
      for (int g = 0; g < NB; ++g) tma_load_2d(Q_s + g * AT_BLK, &tmK, qfull, cq + 32 * g, r0 + q0);
      for (int j = 0; j < T; ++j) {
        const int s = j & 1;
        if (j >= 2) mbar_wait(&kfree[s], (uint32_t)(((j >> 1) & 1) ^ 1));
        mbar_arrive_expect_tx(&kfull[s], Cfg::KV_BYTES);
#pragma unroll
        for (int g = 0; g < NB; ++g) tma_load_2d(K_s + s * Cfg::KV_BYTES + g * AT_BLK, &tmK, &kfull[s], ck + 32 * g, r0 + j * AT_TILE);
      }
    }
  } else if (warp == AT_SOFT + 2) {
    // ---------------- TMA producer: the v tiles ----------------
    if (lane == 0) {
      const int cv = 2 * d + head * HD;
      for (int j = 0; j < T; ++j) {
        const int s = j & 1;
        if (j >= 2) mbar_wait(&vfree[s], (uint32_t)(((j >> 1) & 1) ^ 1));
        mbar_arrive_expect_tx(&vfull[s], Cfg::KV_BYTES);
#pragma unroll
        for (int g = 0; g < NB; ++g) tma_load_2d(V_s + s * Cfg::KV_BYTES + g * AT_BLK, &tmV, &vfull[s], cv + 32 * g, r0 + j * AT_TILE);
      }
    }
  } else if (warp == AT_SOFT) {
    // ---------------- MMA issuer ----------------
    if (lane == 0) {
      constexpr uint32_t IDESC_S = idesc_tf32(AT_TILE, AT_TILE, 0, 0);
      constexpr uint32_t IDESC_O = idesc_tf32(AT_TILE, HD, 0, 1);
      const uint32_t q_addr = smem_u32(Q_s);
      auto issue_s = [&](int j) {
        const int s = j & 1;
        mbar_wait(&kfull[s], (uint32_t)((j >> 1) & 1));
        tc_fence_after();
        const uint32_t k_addr = smem_u32(K_s + s * Cfg::KV_BYTES);
        uint32_t acc = 0;
#pragma unroll
        for (int kk = 0; kk < HD / 8; ++kk) {
          const int g = kk >> 2, k8 = kk & 3;
          mma_tf32(tmem_base + S_COL + 128 * s, smem_desc_sw128(q_addr + g * AT_BLK + k8 * 32, 16, 1024),
                   smem_desc_sw128(k_addr + g * AT_BLK + k8 * 32, 16, 1024), IDESC_S, acc);
          acc = 1;
        }
        mma_commit(&sfull[s]);
        mma_commit(&kfree[s]);
      };
      mbar_wait(qfull, 0);
      issue_s(0);
      if (T > 1) issue_s(1);
      for (int j = 0; j < T; ++j) {
        const int s = j & 1;
        mbar_wait(&vfull[s], (uint32_t)((j >> 1) & 1));
        mbar_wait(&pfull[s], (uint32_t)((j >> 1) & 1));
        tc_fence_after();
        const uint32_t v_addr = smem_u32(V_s + s * Cfg::KV_BYTES);
#pragma unroll
        for (int k8 = 0; k8 < AT_TILE / 8; ++k8) {
          // A: 8 columns of P in tensor memory; B: 8 key rows (two 512-byte swizzle groups) of every 32-column group of V
          mma_tf32_ta(tmem_base + O_COL + 64 * s, tmem_base + S_COL + 128 * s + 8 * k8, smem_desc_sw128(v_addr + k8 * 1024, AT_BLK, 512, 1),
                      IDESC_O, k8 != 0 ? 1u : 0u);
        }
        mma_commit(&ofull[s]);
        mma_commit(&vfree[s]);
        if (j + 2 < T) issue_s(j + 2);       // in order behind P V of tile j: overwrites the group's S / P columns only after they were read
      }
    }
  } else {
    // ---------------- softmax: group g owns the tiles j = g, g + 2, ...; AT_NH threads (column halves) per query row ----------------
    constexpr int OH = Cfg::OH, CPT = 4 / AT_NH;        // 32-column chunks per thread and tile
    const int qt = warp & 3, half = (warp >> 2) % AT_NH, g = warp / AT_GW, row = qt * 32 + lane;
    const int qi = q0 + row;
    const uint32_t lane_base = tmem_base + ((uint32_t)(qt * 32) << 16);
    const uint32_t s_addr = lane_base + S_COL + 128 * g + 32 * CPT * half, o_addr = lane_base + O_COL + 64 * g + OH * half;
    const float sc = scale * kLog2eA;                 // logits in log2 units
    const uint32_t drow = (uint32_t)(r0 + min(qi, Rb - 1)) * (uint32_t)ad.heads + (uint32_t)head;
    float* xmg = xm + g * 2 * AT_NH * AT_TILE;
    float o[OH];
#pragma unroll
    for (int c = 0; c < OH; ++c) o[c] = 0.f;
    float m = -INFINITY, l = 0.f;
    for (int j = g; j < T; j += 2) {
      const uint32_t par = (uint32_t)((j >> 1) & 1);
      const int nk = min(AT_TILE, Rb - j * AT_TILE);
      const int kb0 = 32 * CPT * half;                 // first key column of this thread inside the tile
      mbar_wait(&sfull[g], par);
      tc_fence_after();
      // pass 1: row maximum (exchanged between the column halves)
      float mx4[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
#pragma unroll 1
      for (int ch = 0; ch < CPT; ++ch) {
        float sv[32];
        tmem_ld32(s_addr + 32 * ch, sv);
        if (nk < AT_TILE) {
#pragma unroll
          for (int i = 0; i < 32; ++i) if (kb0 + 32 * ch + i >= nk) sv[i] = -INFINITY;
        }
#pragma unroll
        for (int i = 0; i < 32; ++i) mx4[i & 3] = fmaxf(mx4[i & 3], sv[i]);
      }
      float mx = fmaxf(fmaxf(mx4[0], mx4[1]), fmaxf(mx4[2], mx4[3]));
      if (AT_NH > 1) {
        float* xmp = xmg + par * AT_NH * AT_TILE;      // double-buffered by iteration parity: one barrier per tile
        xmp[half * AT_TILE + row] = mx;
        group_bar(g);
#pragma unroll
        for (int h = 0; h < AT_NH; ++h) mx = fmaxf(mx, xmp[h * AT_TILE + row]);
      }
      const float mn = fmaxf(m, mx * sc);              // sc > 0
      const float cj = ex2a(m - mn);
      l *= cj;
      // pass 2: probabilities, in place
#pragma unroll 1
      for (int ch = 0; ch < CPT; ++ch) {
        float sv[32];
        tmem_ld32(s_addr + 32 * ch, sv);
        if (nk < AT_TILE) {
#pragma unroll
          for (int i = 0; i < 32; ++i) if (kb0 + 32 * ch + i >= nk) sv[i] = -INFINITY;
        }
        float ls4[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int i = 0; i < 32; ++i) { sv[i] = ex2a(fmaf(sv[i], sc, -mn)); ls4[i & 3] += sv[i]; }
        l += (ls4[0] + ls4[1]) + (ls4[2] + ls4[3]);
        if (ad.drop.active) {
          const int kg = j * AT_TILE + kb0 + 32 * ch;  // key index inside the bag
          if (ad.mask) {
#pragma unroll
            for (int i = 0; i < 32; ++i)
              if (!ad.keep(b, head, min(qi, Rb - 1), min(kg + i, Rb - 1), Rb, 0)) sv[i] = 0.f;
          } else {
#pragma unroll
            for (int i = 0; i < 32; i += 2) {
              bool ka, kb;
              ad.drop.keep2(drow, (uint32_t)(kg + i), ka, kb);
              if (!ka) sv[i] = 0.f;
              if (!kb) sv[i + 1] = 0.f;
            }
          }
        }
        uint32_t pw[32];
#pragma unroll
        for (int i = 0; i < 32; ++i) pw[i] = round_tf32_pos(sv[i]);
        tmem_st32(s_addr + 32 * ch, pw);
      }
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&pfull[g]);
      // this tile's P V joins the running output
      mbar_wait(&ofull[g], par);
      tc_fence_after();
      float ot[OH];
      tmem_ldn<OH>(o_addr, ot);
#pragma unroll
      for (int c = 0; c < OH; ++c) o[c] = fmaf(o[c], cj, ot[c]);
      m = mn;
    }
    // ---- merge the two groups (every MMA has retired and every TMA load has landed: the operand buffers are free) ----
    tc_fence_before();
    soft_bar();
    float* xch = (float*)Q_s;      // column-major [.][128]: 0 = m of group 1, 1 + (2 g + half) = l parts, 1 + 2 AT_NH + c = o of group 1
    xch[(1 + AT_NH * g + half) * AT_TILE + row] = l;
    if (g == 1) {
      if (half == 0) xch[row] = m;
#pragma unroll
      for (int c = 0; c < OH; ++c) xch[(1 + 2 * AT_NH + OH * half + c) * AT_TILE + row] = o[c];
    }
    soft_bar();
    if (g == 0 && qi < Rb) {
      const float m1 = xch[row];
      float l0 = 0.f, l1 = 0.f;
#pragma unroll
      for (int h = 0; h < AT_NH; ++h) { l0 += xch[(1 + h) * AT_TILE + row]; l1 += xch[(1 + AT_NH + h) * AT_TILE + row]; }
      const float M = fmaxf(m, m1), w0 = ex2a(m - M), w1 = ex2a(m1 - M);     // group 0 always has a tile: M is finite
      const float lt = l0 * w0 + l1 * w1;
      const float inv = ad.drop.inv_keep / lt;
      float* dst = ctx + (size_t)(r0 + qi) * d + head * HD + OH * half;
      const float* x1 = xch + (size_t)(1 + 2 * AT_NH + OH * half) * AT_TILE + row;
#pragma unroll
      for (int c = 0; c < OH; c += 4) {
        float4 v;
        v.x = (o[c] * w0 + x1[(c) * AT_TILE] * w1) * inv;
        v.y = (o[c + 1] * w0 + x1[(c + 1) * AT_TILE] * w1) * inv;
        v.z = (o[c + 2] * w0 + x1[(c + 2) * AT_TILE] * w1) * inv;
        v.w = (o[c + 3] * w0 + x1[(c + 3) * AT_TILE] * w1) * inv;
        *reinterpret_cast<float4*>(dst + c) = v;
      }
      if (half == 0) lse[(size_t)head * Rtot + r0 + qi] = M * kLn2A + __logf(lt);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == AT_SOFT) { tc_fence_after(); tmem_dealloc(tmem_base, 512); }
}

}  // namespace

bool mha_tcgen05_supported(int hd, int d) {
  return (hd == 16 || hd == 32 || hd == 48 || hd == 64) && (3 * (long long)d * 4) % 16 == 0;
}

template <int HD>
static int launch_fwd(const float* qkv, const int32_t* ro, int bags, int Rtot, int d, int heads, int mx, float scale, const AttDrop& ad,
                      float* ctx, float* lse, cudaStream_t st) {
  CUtensorMap tmK, tmV;
  ADVMIL_TRY(make_map(&tmK, qkv, Rtot, 3LL * d, CU_TENSOR_MAP_SWIZZLE_128B));
  ADVMIL_TRY(make_map(&tmV, qkv, Rtot, 3LL * d, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B));
  static bool attr_set[64] = {};
  int dev = 0;
  ADVMIL_CHECK_CUDA(cudaGetDevice(&dev));
  if (dev < 0 || dev >= 64 || !attr_set[dev]) {
    ADVMIL_CHECK_CUDA(cudaFuncSetAttribute(mha_fwd_tcgen05_kernel<HD>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)AttCfg<HD>::SMEM));
    if (dev >= 0 && dev < 64) attr_set[dev] = true;
  }
  launch_k(mha_fwd_tcgen05_kernel<HD>, dim3(cdiv(mx, AT_TILE), bags, heads), dim3(AT_THREADS), AttCfg<HD>::SMEM, st, tmK, tmV, ro, d, scale,
           ad, ctx, lse, Rtot);
  ADVMIL_CHECK_LAUNCH();
  return ADVMIL_OK;
}

int mha_fwd_tcgen05(const float* qkv, const int32_t* ro, int bags, int Rtot, int d, int heads, int mx, float scale, const AttDrop& ad,
                    float* ctx, float* lse, cudaStream_t st) {
  ADVMIL_REQUIRE(((uintptr_t)qkv) % 16 == 0, "attention: qkv must be 16-byte aligned");
  switch (d / heads) {
    case 16: return launch_fwd<16>(qkv, ro, bags, Rtot, d, heads, mx, scale, ad, ctx, lse, st);
    case 32: return launch_fwd<32>(qkv, ro, bags, Rtot, d, heads, mx, scale, ad, ctx, lse, st);
    case 48: return launch_fwd<48>(qkv, ro, bags, Rtot, d, heads, mx, scale, ad, ctx, lse, st);
    case 64: return launch_fwd<64>(qkv, ro, bags, Rtot, d, heads, mx, scale, ad, ctx, lse, st);
  }
  set_error("attention: head width %d unsupported on tcgen05", d / heads);
  return ADVMIL_ERR_INVALID;
}

}  // namespace advmil
