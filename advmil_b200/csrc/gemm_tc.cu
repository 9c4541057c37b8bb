// tcgen05 / TMEM / TMA engine for the N-row contractions (sm_100a).
//
//  tc_rows_kernel   C[rows, N] = A[rows, K] . W[N, K]^T with a fused epilogue.  A (activations, fp32 in HBM) and W are
//                   K-major; 128 x BLOCK_N output tiles; TMA (SWIZZLE_128B boxes of 32 fp32 = 128 B per row) feeds a 4-stage
//                   shared-memory ring; one elected thread issues tcgen05.mma.kind::tf32 (fp32 bits are consumed directly:
//                   no conversion pass over x); accumulators are double-buffered in TMEM so the epilogue of tile i overlaps
//                   the MMAs of tile i+1; persistent over tiles with the N-tiles of one row block adjacent in time so x is
//                   fetched from HBM once and re-read from L2.
//                   Epilogues: bias+ReLU+dropout (K1), tanh*sigmoid gate + w_c score (K2), LayerNorm+ReLU+16-row region mean
//                   (K5+K6), backward-data with pooling term and ReLU mask.
//  tc_wgrad_kernel  dW[N1, N2] = dY[rows, N1]^T . X[rows, N2]: both operands MN-major straight from their row-major
//                   activations (no transposes of the big tensors), split-K over rows, fp32 partial tiles reduced afterwards.
//
// Warp roles (256 threads): warp 0 TMA producer, warp 1 MMA issuer, warp 2 TMEM allocator, warps 4-7 epilogue
// (TMEM lane quarter = warp % 4).
#include <mutex>
#include "gemm_tc.cuh"
#include "tc_ptx.cuh"

namespace advmil {
using namespace tc;

// ------------------------------------------------------------------------------------------------
// tensor maps (driver entry point resolved at run time: no link-time dependency on libcuda)
// ------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn get_encode() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = (EncodeTiledFn)p;
  }
  return fn;
}
// per-element-type constants of the engine: one 128-byte swizzle row holds KBLK elements; one MMA consumes 32 bytes of K
template <typename T> struct TcElem;
template <> struct TcElem<float> {
  static constexpr int KBLK = 32;
  static constexpr CUtensorMapDataType DT = CU_TENSOR_MAP_DATA_TYPE_FLOAT32;
  static constexpr CUtensorMapSwizzle MN_SWZ = CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B;   // MN-major 32-bit operands
  static constexpr uint32_t MN_LAYOUT = 1;      // SWIZZLE_128B_BASE32B
  static constexpr int MN_SBO = 512;            // 4 k-rows x 128 B per swizzle group
  __host__ __device__ static constexpr uint32_t idesc(int M, int N, int am, int bm) { return idesc_tf32(M, N, am, bm); }
  __device__ __forceinline__ static void mma(uint32_t d, uint64_t a, uint64_t b, uint32_t i, uint32_t acc) { mma_tf32(d, a, b, i, acc); }
};
template <> struct TcElem<bf16> {
  static constexpr int KBLK = 64;
  static constexpr CUtensorMapDataType DT = CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
  static constexpr CUtensorMapSwizzle MN_SWZ = CU_TENSOR_MAP_SWIZZLE_128B;
  static constexpr uint32_t MN_LAYOUT = 2;      // SWIZZLE_128B
  static constexpr int MN_SBO = 1024;           // 8 k-rows x 128 B per swizzle atom
  __host__ __device__ static constexpr uint32_t idesc(int M, int N, int am, int bm) { return idesc_bf16(M, N, am, bm); }
  __device__ __forceinline__ static void mma(uint32_t d, uint64_t a, uint64_t b, uint32_t i, uint32_t acc) { mma_f16(d, a, b, i, acc); }
};

// row-major matrix [rows, cols] of T; box = box_rows x (128 B of elements), 128-byte swizzle, OOB reads return zeros
template <typename T>
static int make_tmap(CUtensorMap* m, const T* base, long long rows, long long cols, int box_rows,
                     CUtensorMapSwizzle swz = CU_TENSOR_MAP_SWIZZLE_128B) {
  EncodeTiledFn enc = get_encode();
  if (!enc) { set_error("cuTensorMapEncodeTiled unavailable"); return ADVMIL_ERR_CUDA; }
  cuuint64_t gdim[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t gstr[1] = {(cuuint64_t)cols * sizeof(T)};
  cuuint32_t box[2] = {(cuuint32_t)TcElem<T>::KBLK, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1u, 1u};
  CUresult r = enc(m, TcElem<T>::DT, 2, (void*)base, gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   swz, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled failed (%d) rows=%lld cols=%lld", (int)r, rows, cols); return ADVMIL_ERR_CUDA; }
  return ADVMIL_OK;
}
// x [16 R, C] viewed as R regions of 4 x 4 patches (row 16r + 4i + j = region r, grid row i, grid column j), innermost first:
// {C, j, i, r}.  A box {KBLK, 4, 4, box_regions} is box_regions * 16 rows x 128 B: in shared memory the same image as a
// 2-D box of that many rows.  A box shifted by (di, dj) in the grid lands partly outside it and TMA fills those elements
// with zeros: that is the 3x3 convolution's zero padding at every region border (and the tail past the last region).
template <typename T>
static int make_tmap_regions(CUtensorMap* m, const T* base, long long regions, long long C, int box_regions,
                             CUtensorMapSwizzle swz = CU_TENSOR_MAP_SWIZZLE_128B) {
  EncodeTiledFn enc = get_encode();
  if (!enc) { set_error("cuTensorMapEncodeTiled unavailable"); return ADVMIL_ERR_CUDA; }
  const cuuint64_t rb = (cuuint64_t)C * sizeof(T);
  cuuint64_t gdim[4] = {(cuuint64_t)C, 4, 4, (cuuint64_t)regions};
  cuuint64_t gstr[3] = {rb, 4 * rb, 16 * rb};
  cuuint32_t box[4] = {(cuuint32_t)TcElem<T>::KBLK, 4, 4, (cuuint32_t)box_regions};
  cuuint32_t estr[4] = {1u, 1u, 1u, 1u};
  CUresult r = enc(m, TcElem<T>::DT, 4, (void*)base, gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   swz, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled failed (%d) regions=%lld C=%lld", (int)r, regions, C); return ADVMIL_ERR_CUDA; }
  return ADVMIL_OK;
}

static int sm_count() {
  static int n = 0;
  if (!n) { int dev = 0; cudaGetDevice(&dev); cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev); if (n <= 0) n = 148; }
  return n;
}

// ------------------------------------------------------------------------------------------------
// epilogue parameter block
// ------------------------------------------------------------------------------------------------
enum RowEpiKind : int { EPI_LINEAR = 0, EPI_GATE = 1, EPI_LN = 2, EPI_BWD = 3, EPI_PE = 4 /* K1 + K5/K6 on stacked weights */,
                        EPI_POOL = 5 /* K9: relu(x W^T + b) -> per-(tile, bag, cluster) column sums */ };

// out / ab / y_pre / relu_src are [rows, *] activation tensors of the kernel's element type T (fp32 or bf16)
struct RowEpi {
  void* out; int ldo; const float* bias;
  int relu; Drop drop;                                                           // EPI_LINEAR
  void* out2; Drop drop2;                                                        // EPI_LINEAR: optional second output = dropout(out) under drop2
  void* ab; const float* wc; float* part; int D; Drop drop_a, drop_b;            // EPI_GATE (bias = packed gate bias)
  void* y_pre; float* emb; const float* gamma; const float* beta; float eps;     // EPI_LN
  int h_cols; const float* bias2;                                                // EPI_PE: columns [0, h_cols) = K1, last 128 = K5 (bias2 = conv bias)
  const float* w; const float* dz; const int32_t* offsets; int bags;             // EPI_BWD
  const float* dmean; int accumulate;
  float* colpart;                                                                // EPI_BWD: [4 * num_m][N] column sums of dX per 32 rows
  const void* relu_src; int ld_src; float inv_keep;
  // EPI_POOL reuses fields of the block above (its layout, and so every other instantiation, stays as it is):
  //   out = optional ReLU keep bits uint32 [rows][N / 32] (bit i of word c = column 32 c + i), ldo = N / 32, bias,
  //   part = column sums [(m-tile + bag) * D + cluster][N] (fp32), D = number of clusters, relu_src = cluster ids int32
  //   [rows], offsets / bags = the packed bags (every bag length a multiple of 16)
};

constexpr int TILE_M = 128;
constexpr int A_STAGE_BYTES = TILE_M * 128;            // 128 rows x one 128-byte swizzle row = 16 KB
constexpr int STG_LD = 36;                             // staging row stride (floats) for 32-column chunks
constexpr int STG_LD_LN = 132;                         // staging row stride for full 128-column rows

// ES = element size of the activation type.  The smem ring takes whatever the epilogue's staging leaves: the TMA -> MMA
// pipeline is latency-bound (ncu: tensor pipe ~50 % busy with no memory level saturated), so depth matters more than
// anything else here; the bf16 epilogues stage 80-byte rows (2.5 KB per warp) and leave room for 5 / 4 stages at
// BLOCK_N = 192 / 256.
// X3 = split-tf32 ("3xTF32") variant of the fp32-element kernels: every operand is split into a tf32-exact high part and a
// tf32-rounded low part (x = hi + lo + O(2^-22 x)) and each K step issues three MMAs, hi.hi + lo.hi + hi.lo, accumulated in
// fp32 in TMEM: fp32-grade products (the dropped lo.lo term is 2^-22 relative) on the tensor pipe.  The activation tile's
// split happens in shared memory (two converter warps rewrite the TMA-written tile in place as `hi` and fill a second
// buffer with `lo`; fence.proxy.async hands both to the tensor core); the weight's two parts are prepared in global
// memory by a small kernel and arrive by TMA.  A stage therefore holds 2 x (A + B): 2 stages at 256 / 192 columns, with
// 4 epilogue warps, which is enough because every stage now carries 12 MMAs.
template <int ES, int BLOCK_N, int EPI, bool X3 = false> struct RowCfg {
  static_assert(!X3 || ES == 4, "split-tf32 runs on fp32 elements");
  // Epilogue warps per TMEM lane quarter (NSUB).  The bf16 epilogues are chains of dependent ALU / shared / global
  // instructions: with 2 warps per scheduler the epilogue issued ~1 instruction per 8 cycles per warp and the tensor pipe
  // idled behind it (ncu r02: dh 35 % tensor-active at 0.26 IPC per scheduler).  4 warps per quarter (3 at 192 columns, where
  // 6 chunks divide evenly) give the schedulers the warps to hide those latencies; registers: 65536 / 640 threads = 102.
  static constexpr bool WIDE_EPI = ES == 2 && (EPI == EPI_GATE || EPI == EPI_BWD || EPI == EPI_LINEAR);
  static constexpr int NSUB = (EPI == EPI_LN || EPI == EPI_POOL || X3) ? 1 : (!WIDE_EPI ? 2 : (EPI != EPI_GATE && BLOCK_N == 192 ? 3 : (BLOCK_N >= 128 ? 4 : 2)));
  static constexpr int EPI_WARPS = 4 * NSUB;
  static constexpr int THREADS = 128 + 32 * EPI_WARPS;
  static constexpr int B_STAGE_BYTES = BLOCK_N * 128;
  static constexpr int STAGE_BYTES = (X3 ? 2 : 1) * (A_STAGE_BYTES + B_STAGE_BYTES);
  static constexpr int TMA_BYTES = A_STAGE_BYTES + (X3 ? 2 : 1) * B_STAGE_BYTES;     // what TMA delivers per stage
  // bf16 staging: 32 rows x 64 bytes, XOR-swizzled (2 KB per warp); fp32 staging: 32 x 36 floats; LN: full 128-column rows
  // (the 64- and 256-column LN epilogues work chunk by chunk and stage 32 columns)
  static constexpr int STG_FLOATS_PER_WARP = (EPI == EPI_LN) ? (BLOCK_N == 128 ? 32 * STG_LD_LN : 32 * STG_LD)
                                                             : ((ES == 2 && EPI != EPI_PE && EPI != EPI_POOL) ? 32 * 64 / 4 : 32 * STG_LD);
  // gate: per 32-pair chunk 32 tanh biases | 32 sigmoid biases | 32 w_c (4 / NSUB chunks per warp);
  // proj+embed: conv bias | gamma | beta (128 each); cluster pool: per-cluster column sums of the warp's two 16-row halves
  static constexpr int COEF_FLOATS_PER_WARP = (EPI == EPI_GATE) ? 384 / NSUB : (EPI == EPI_PE) ? 384 : (EPI == EPI_POOL) ? 2 * 16 * 32 : 0;
  static constexpr int GPART_FLOATS = (EPI == EPI_GATE && NSUB == 4) ? 2 * 8 * 32 : 0;   // partial-score exchange between warp pairs
  static constexpr int TMEM_COLS = (2 * BLOCK_N <= 64) ? 64 : (2 * BLOCK_N <= 128) ? 128 : (2 * BLOCK_N <= 256) ? 256 : 512;
  static constexpr size_t FIXED = 1024 /*align slack*/ + (size_t)EPI_WARPS * (STG_FLOATS_PER_WARP + COEF_FLOATS_PER_WARP + 96) * 4 +
                                  GPART_FLOATS * 4 + 256 /*barriers*/;
  static constexpr int FIT = (int)((227 * 1024 - FIXED - 64) / STAGE_BYTES);
  static constexpr int STAGES = FIT > 8 ? 8 : FIT;
  static_assert(STAGES >= (X3 ? 2 : 3), "shared-memory ring too shallow");
  static constexpr size_t SMEM = FIXED + (size_t)STAGES * STAGE_BYTES;
};

__device__ __forceinline__ float fast_tanh(float x) { float y; asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }

// stage one 32-column chunk: thread `lane` owns row `lane`
__device__ __forceinline__ void stage_chunk(float* stg, int ld, int col0, const float (&v)[32], int lane) {
#pragma unroll
  for (int j = 0; j < 8; ++j)
    *reinterpret_cast<float4*>(stg + lane * ld + col0 + 4 * j) = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
}

// raw 16-byte vector -> floats
__device__ __forceinline__ void raw_floats(const uint4& u, float (&o)[4]) {
  o[0] = __uint_as_float(u.x); o[1] = __uint_as_float(u.y); o[2] = __uint_as_float(u.z); o[3] = __uint_as_float(u.w);
}
__device__ __forceinline__ void raw_floats(const uint4& u, float (&o)[8]) {
  o[0] = bf_lo(u.x); o[1] = bf_hi(u.x); o[2] = bf_lo(u.y); o[3] = bf_hi(u.y);
  o[4] = bf_lo(u.z); o[5] = bf_hi(u.z); o[6] = bf_lo(u.w); o[7] = bf_hi(u.w);
}
// staged [32 rows][ncols] fp32 block (row stride ld floats) -> global rows of T, 16-byte stores, consecutive lanes along a row
template <typename T, int NCOLS>
__device__ __forceinline__ void store_staged(const float* stg, int ld, T* __restrict__ out, size_t ldo, int m_base, int M,
                                             int col0, int lane) {
  constexpr int VEC = VecN<T>::N, LPR = NCOLS / VEC, RPI = 32 / LPR, NIT = 32 / RPI;
  static_assert(LPR <= 32 && 32 % LPR == 0, "row must be covered by at most one warp");
#pragma unroll
  for (int it = 0; it < NIT; ++it) {
    const int r = lane / LPR + RPI * it, cv = lane % LPR, m = m_base + r;
    if (m < M) {
      float o[VEC];
#pragma unroll
      for (int q = 0; q < VEC / 4; ++q) {
        const float4 t = *reinterpret_cast<const float4*>(stg + r * ld + cv * VEC + 4 * q);
        o[4 * q] = t.x; o[4 * q + 1] = t.y; o[4 * q + 2] = t.z; o[4 * q + 3] = t.w;
      }
      stv(out + (size_t)m * ldo + col0 + cv * VEC, o);
    }
  }
}

// bf16 outputs: a warp's [32 rows][32 columns] chunk, one row per lane in registers, is rounded to bf16 FIRST and staged
// as 64-byte rows, i.e. half the shared-memory traffic of fp32 staging -- the tensor pipe's operand fetch already uses
// most of the shared-memory bandwidth.  The 16-byte piece q of row r lives at r * 64 + ((q ^ ((r >> 1) & 3)) * 16): the
// row-per-lane writes (8 consecutive rows per quarter-warp) and the transposed reads (2 rows x 4 pieces per quarter-warp)
// both touch 8 distinct 16-byte bank groups -- conflict-free (the 80-byte stride of round 1 cost 2.5 wavefronts per read).
// Lane l then stores 16 bytes of row l/4 + 8*it: 4 lanes cover one 64-byte row segment.
__device__ __forceinline__ uint32_t stgb_off(int r, int q) { return (uint32_t)(r * 64 + ((q ^ ((r >> 1) & 3)) << 4)); }
__device__ __forceinline__ void stage_words_bf16(uint8_t* stgb, const uint32_t (&w)[16], int lane) {
#pragma unroll
  for (int q = 0; q < 4; ++q)
    *reinterpret_cast<uint4*>(stgb + stgb_off(lane, q)) = make_uint4(w[4 * q], w[4 * q + 1], w[4 * q + 2], w[4 * q + 3]);
}
__device__ __forceinline__ void stage_rows_bf16(uint8_t* stgb, const float (&v)[32], int lane) {
#pragma unroll
  for (int q = 0; q < 4; ++q)
    *reinterpret_cast<uint4*>(stgb + stgb_off(lane, q)) =
        make_uint4(pack_bf2(v[8 * q], v[8 * q + 1]), pack_bf2(v[8 * q + 2], v[8 * q + 3]), pack_bf2(v[8 * q + 4], v[8 * q + 5]),
                   pack_bf2(v[8 * q + 6], v[8 * q + 7]));
}
__device__ __forceinline__ void store_rows_bf16(uint8_t* stgb, const float (&v)[32], bf16* __restrict__ out, size_t ldo, int m_base,
                                                int M, int col0, int lane) {
  stage_rows_bf16(stgb, v, lane);
  __syncwarp();
#pragma unroll
  for (int it = 0; it < 4; ++it) {
    const int r = (lane >> 2) + 8 * it, cv = lane & 3, m = m_base + r;
    const uint4 qv = *reinterpret_cast<const uint4*>(stgb + stgb_off(r, cv));
    if (m < M) *reinterpret_cast<uint4*>(out + (size_t)m * ldo + col0 + cv * 8) = qv;
  }
  __syncwarp();
}

// gate math on one 32-pair chunk: va/vb hold pre-activations on entry and tanh / sigmoid values on exit.
// MODE 0 = eval; 1 = train, in-kernel generator; 2 = train, injected masks (kept out of the hot instantiation: the
// compiler otherwise issues both paths predicated for every element)
template <bool FAST, int MODE>
__device__ __forceinline__ float gate_chunk(float (&va)[32], float (&vb)[32], const float* __restrict__ cba,
                                            const float* __restrict__ cbb, const float* __restrict__ cwc, const Drop& da,
                                            const Drop& db, uint32_t row, uint32_t j0, float partial, bool row_valid = true) {
  const uint32_t rowterm = row * 0x9E3779B1u, tj = da.thresh8j, key = da.key;
#pragma unroll
  for (int i0 = 0; i0 < 32; i0 += 4) {
    uint32_t x = 0;
    if (MODE == 1) {     // one draw per 4 pairs, 8 bits each: the JOINT keep bit of the pair (Drop::pair_gate; == gate_keep)
      x = rowterm ^ ((j0 + i0) * 0x85EBCA77u + key);               // == Drop::bits(row, j0 + i0)
      x ^= x >> 16; x *= 0x85EBCA6Bu; x ^= x >> 13; x *= 0xC2B2AE35u; x ^= x >> 16;
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int i = i0 + k;
      const float xa = va[i] + cba[i], xb = vb[i] + cbb[i];
      float a, b;
      if (FAST) { a = fast_tanh(xa); b = fmaf(0.5f, fast_tanh(0.5f * xb), 0.5f); }
      else { a = tanhf(xa); b = sigmoidf_(xb); }
      va[i] = a; vb[i] = b;
      if (MODE != 0) {
        // either unit dropped => the pair contributes nothing forward or backward: the stored sigmoid carries the joint
        // keep bit in its (otherwise unused) sign, so the backward pass needs no generator
        bool keep;
        if (MODE == 1) {
          keep = ((x >> (8 * k)) & 0xFFu) >= tj;
        } else {
          bool ka = false, kb = false;
          if (row_valid) gate_keep(da, db, row, j0 + i, ka, kb);      // rows past M of the last tile have no mask entries
          keep = ka && kb;
        }
        vb[i] = keep ? b : -b;
        partial = fmaf(keep ? a * b : 0.f, cwc[i], partial);
      } else {
        partial = fmaf(a * b, cwc[i], partial);
      }
    }
  }
  return partial;
}

// tf32-exact high part and tf32-rounded low part of an fp32 value (cvt.rna.tf32.f32: low 13 mantissa bits zero)
__device__ __forceinline__ uint32_t tf32_rna(float x) { uint32_t r; asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x)); return r; }
__device__ __forceinline__ void split_tf32(uint32_t raw, uint32_t& hi, uint32_t& lo) {
  const float x = __uint_as_float(raw);
  hi = tf32_rna(x);
  lo = tf32_rna(x - __uint_as_float(hi));
}
__device__ __forceinline__ void split_tf32(const uint4& v, uint4& hi, uint4& lo) {
  split_tf32(v.x, hi.x, lo.x); split_tf32(v.y, hi.y, lo.y); split_tf32(v.z, hi.z, lo.z); split_tf32(v.w, hi.w, lo.w);
}

// One CTA per SM, persistent over its 128 x BLOCK_N tiles.  Barriers: full (the stage's TMA bytes landed), empty (the
// MMAs that read the stage retired), conv (X3: the converter warps split the stage's A tile), tfull (an accumulator
// buffer is complete), tempty (every epilogue thread drained it).
// CONV: implicit-GEMM 3x3 convolution inside each 4x4 region, K = 9 C.  tmA is the region view of x (make_tmap_regions),
// W the tap-major repacked weight [N, 9 C]; k block kb = 9 kc + tap reads channel block kc of x shifted by the tap, so
// the nine boxes of one channel block cover the same 128 rows back to back and x is read from HBM about once.
template <typename T, int BLOCK_N, int EPI, bool FAST, bool X3 = false, bool CONV = false>
__global__ void __launch_bounds__(RowCfg<(int)sizeof(T), BLOCK_N, EPI, X3>::THREADS, 1)
tc_rows_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
               const __grid_constant__ CUtensorMap tmBlo, int M, int N, int K, RowEpi ea) {
  pdl_prologue();
  using Cfg = RowCfg<(int)sizeof(T), BLOCK_N, EPI, X3>;
  constexpr int STAGES = Cfg::STAGES;
  constexpr int KBLK = TcElem<T>::KBLK;
  constexpr int VEC = VecN<T>::N;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);   // pointer arithmetic keeps the shared address space
  uint8_t* A_s = smem;
  uint8_t* AL_s = A_s + STAGES * A_STAGE_BYTES;                        // X3: low parts of the A tiles
  uint8_t* B_s = AL_s + (X3 ? STAGES * A_STAGE_BYTES : 0);
  uint8_t* BL_s = B_s + STAGES * Cfg::B_STAGE_BYTES;                   // X3: low parts of the weight tiles
  float* stg_all = (float*)(BL_s + (X3 ? STAGES * Cfg::B_STAGE_BYTES : 0));
  float* coef_all = stg_all + Cfg::EPI_WARPS * Cfg::STG_FLOATS_PER_WARP;
  int* rowbag = (int*)(coef_all + Cfg::EPI_WARPS * Cfg::COEF_FLOATS_PER_WARP);
  float* roww = (float*)(rowbag + Cfg::EPI_WARPS * 32);
  float* rowinv = roww + Cfg::EPI_WARPS * 32;
  float* gpart = rowinv + Cfg::EPI_WARPS * 32;            // [2][8][32] partial-score exchange (gate, 4 warps per quarter)
  uint64_t* bars = (uint64_t*)(gpart + Cfg::GPART_FLOATS);
  uint64_t* full = bars;                 // [STAGES]
  uint64_t* empty = bars + STAGES;       // [STAGES]
  uint64_t* conv = bars + 2 * STAGES;    // [STAGES] X3: the activation tile has been split
  uint64_t* tfull = bars + 3 * STAGES;   // [2]
  uint64_t* tempty = tfull + 2;          // [2]
  uint32_t* tmem_ptr = (uint32_t*)(tempty + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int num_m = (M + TILE_M - 1) / TILE_M, num_n = N / BLOCK_N;
  const int total = num_m * num_n, kblocks = K / KBLK;
  const int work0 = blockIdx.x, work_stride = gridDim.x;

  if (threadIdx.x == 0) {
    prefetch_tmap(&tmA);
    prefetch_tmap(&tmB);
    for (int i = 0; i < STAGES; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); mbar_init(&conv[i], X3 ? 64 : 1); }
    if (X3) prefetch_tmap(&tmBlo);
    // accumulator release: every epilogue thread arrives
    for (int i = 0; i < 2; ++i) { mbar_init(&tfull[i], 1); mbar_init(&tempty[i], 32 * Cfg::EPI_WARPS); }
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc(tmem_ptr, Cfg::TMEM_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      int stage = 0; uint32_t phase = 0;
      for (int tile = work0; tile < total; tile += work_stride) {
        const int m0 = (tile / num_n) * TILE_M, n0 = (tile % num_n) * BLOCK_N;
        for (int kb = 0; kb < kblocks; ++kb) {
          mbar_wait(&empty[stage], phase ^ 1);          // the MMAs that read this slot retired
          mbar_arrive_expect_tx(&full[stage], Cfg::TMA_BYTES);
          int kw = kb * KBLK;                             // k coordinate of the weight tile
          if constexpr (CONV) {
            const int kc = kb / 9, tap = kb - 9 * kc;
            tma_load_4d(A_s + stage * A_STAGE_BYTES, &tmA, &full[stage], kc * KBLK, tap % 3 - 1, tap / 3 - 1, m0 >> 4);
            kw = tap * (K / 9) + kc * KBLK;
          } else {
            tma_load_2d(A_s + stage * A_STAGE_BYTES, &tmA, &full[stage], kb * KBLK, m0);
          }
          tma_load_2d(B_s + stage * Cfg::B_STAGE_BYTES, &tmB, &full[stage], kw, n0);
          if (X3) tma_load_2d(BL_s + stage * Cfg::B_STAGE_BYTES, &tmBlo, &full[stage], kw, n0);
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    constexpr uint32_t IDESC = TcElem<T>::idesc(TILE_M, BLOCK_N, 0, 0);
    int stage = 0; uint32_t phase = 0; int it = 0;
    for (int tile = work0; tile < total; tile += work_stride, ++it) {
      // split tf32: ONE accumulator pair per CTA -- columns [0, BLOCK_N) take the hi.hi chain, [BLOCK_N, 2 BLOCK_N) the two
      // small terms -- instead of two alternating tiles.  The tensor core accumulates with truncation: every MMA into a large
      // accumulator costs up to one ulp of it, one-sided, so the small terms must not be chained into the main sum (the
      // epilogue adds the two accumulators once, in round-to-nearest fp32).
      const int acc = X3 ? 0 : (it & 1); const uint32_t aphase = X3 ? (it & 1) : ((it >> 1) & 1);
      mbar_wait(&tempty[acc], aphase ^ 1);
      tc_fence_after();
      const uint32_t d_tmem = tmem_base + acc * BLOCK_N;
      for (int kb = 0; kb < kblocks; ++kb) {
        if (X3) mbar_wait(&conv[stage], phase);         // split-tf32: TMA landed AND the converter warps split the A tile
        else mbar_wait(&full[stage], phase);
        tc_fence_after();
        if (lane == 0) {
          const uint32_t a_addr = smem_u32(A_s + stage * A_STAGE_BYTES), b_addr = smem_u32(B_s + stage * Cfg::B_STAGE_BYTES);
#pragma unroll
          for (int kk = 0; kk < 4; ++kk) {   // one MMA = 32 bytes of K (8 tf32 / 16 bf16) inside the 128-byte swizzle row
            uint64_t ad = smem_desc_sw128(a_addr + kk * 32, 16, 1024);
            uint64_t bd = smem_desc_sw128(b_addr + kk * 32, 16, 1024);
            TcElem<T>::mma(d_tmem, ad, bd, IDESC, (kb | kk) != 0 ? 1u : 0u);
            if constexpr (X3) {              // + lo.hi + hi.lo
              const uint64_t ald = smem_desc_sw128(smem_u32(AL_s + stage * A_STAGE_BYTES) + kk * 32, 16, 1024);
              const uint64_t bld = smem_desc_sw128(smem_u32(BL_s + stage * Cfg::B_STAGE_BYTES) + kk * 32, 16, 1024);
              TcElem<T>::mma(d_tmem + BLOCK_N, ald, bd, IDESC, (kb | kk) != 0 ? 1u : 0u);
              TcElem<T>::mma(d_tmem + BLOCK_N, ad, bld, IDESC, 1u);
            }
          }
          mma_commit(&empty[stage]);                 // smem slot is free once these MMAs retire
          if (kb == kblocks - 1) mma_commit(&tfull[acc]);
        }
        __syncwarp();
        if (++stage == STAGES) { stage = 0; phase ^= 1; }
      }
    }
  } else if (X3 && (warp == 2 || warp == 3)) {
    // ===================== split-tf32 converter (64 threads): A tile -> hi in place, lo beside it =====================
    if constexpr (X3) {
      const int ct = threadIdx.x - 64;
      int stage = 0; uint32_t phase = 0;
      for (int tile = work0; tile < total; tile += work_stride) {
        for (int kb = 0; kb < kblocks; ++kb) {
          mbar_wait(&full[stage], phase);
          uint4* hi = reinterpret_cast<uint4*>(A_s + stage * A_STAGE_BYTES);
          uint4* lo = reinterpret_cast<uint4*>(AL_s + stage * A_STAGE_BYTES);
#pragma unroll 4
          for (int i = ct; i < A_STAGE_BYTES / 16; i += 64) {
            uint4 h4, l4;
            split_tf32(hi[i], h4, l4);
            hi[i] = h4; lo[i] = l4;
          }
          fence_proxy_async();                   // generic-proxy writes -> visible to the tensor core's async-proxy reads
          mbar_arrive(&conv[stage]);
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp >= 4) {
    // ===================== epilogue =====================
    constexpr int NSUB = Cfg::NSUB;        // epilogue warps per TMEM lane quarter
    const int ew = warp - 4;               // 0..EPI_WARPS-1
    const int wq = warp & 3;               // TMEM lane quarter this warp may read
    const int sub = ew >> 2;               // which share of the tile's column chunks this warp drains (0..NSUB-1)
    const int half = sub;                  // the 2-warps-per-quarter epilogues: which half of the tile's columns
    // this warp no longer needs the TMEM accumulator buffer: tell the MMA issuer
    auto release_acc = [&](uint64_t* bar) {
      tc_fence_before();
      mbar_arrive(bar);
    };
    float* stg = stg_all + ew * Cfg::STG_FLOATS_PER_WARP;
    float* coef = coef_all + ew * Cfg::COEF_FLOATS_PER_WARP;
    int* mybag = rowbag + ew * 32;
    float* myw = roww + ew * 32;
    float* myinv = rowinv + ew * 32;
    if constexpr (EPI == EPI_PE) {           // LayerNorm coefficients of the embed block: constant for the whole launch
      if (half == 1) {
        for (int t = lane; t < 128; t += 32) {
          coef[t] = __ldg(ea.bias2 + t); coef[128 + t] = __ldg(ea.gamma + t); coef[256 + t] = __ldg(ea.beta + t);
        }
      }
      __syncwarp();
    }
    int it = 0;
    for (int tile = work0; tile < total; tile += work_stride, ++it) {
      const int acc = X3 ? 0 : (it & 1); const uint32_t aphase = X3 ? (it & 1) : ((it >> 1) & 1);
      const int mt = tile / num_n, nt = tile % num_n;
      const int m_base = mt * TILE_M + wq * 32, n0 = nt * BLOCK_N;
      const int m_row = m_base + lane;                     // the row this thread owns in TMEM
      if constexpr (EPI == EPI_BWD) {                      // per-row pooling operands (independent of the accumulator)
        int bg = 0; float wv = 0.f, inv = 0.f;
        if ((ea.dz || ea.dmean) && m_row < M) {
          bg = bag_of_row(ea.offsets, ea.bags, m_row);
          const float ik = ea.relu_src ? ea.inv_keep : 1.0f;     // folded here and into W^T (see tc_bwd_data_t)
          if (ea.dz) wv = ea.w[m_row] * ik;
          if (ea.dmean) inv = ik / (float)(ea.offsets[bg + 1] - ea.offsets[bg]);
        }
        mybag[lane] = bg; myw[lane] = wv; myinv[lane] = inv;
      }
      int pool_cid = -1;
      if constexpr (EPI == EPI_POOL) {                     // cluster id and bag of this thread's row (-1: past the last row)
        int bg = -1;
        if (m_row < M) { pool_cid = reinterpret_cast<const int32_t*>(ea.relu_src)[m_row]; bg = bag_of_row(ea.offsets, ea.bags, m_row); }
        mybag[lane] = bg;
      }
      if constexpr (EPI == EPI_GATE) {                     // this warp's 32-pair chunks: biases and w_c into shared memory
        constexpr int PCW = 4 / NSUB;                      // pair chunks per warp (a 256-column tile holds 4)
#pragma unroll
        for (int q = 0; q < PCW; ++q) {
          const int pc = sub * PCW + q;                    // pair chunk: gate block pc / 2, pairs (pc % 2) * 32 .. + 31 of it
          const int cb0 = n0 + (pc >> 1) * 128 + (pc & 1) * 32, j0 = (n0 >> 1) + pc * 32;
          coef[q * 96 + lane] = __ldg(ea.bias + cb0 + lane);
          coef[q * 96 + 32 + lane] = __ldg(ea.bias + cb0 + 64 + lane);
          coef[q * 96 + 64 + lane] = (j0 + lane < ea.D) ? __ldg(ea.wc + j0 + lane) : 0.f;
        }
      }
      __syncwarp();
      // bf16 backward-data: the ReLU-mask operand (this lane's own row of the forward activation, 64 bytes per chunk) does
      // not depend on the accumulator: fetch it for every chunk of the tile BEFORE waiting for the MMAs
      constexpr int NCHW = (BLOCK_N / 32 + NSUB - 1) / NSUB;      // chunks this warp drains per tile
      uint4 hpre[(EPI == EPI_BWD && sizeof(T) == 2) ? NCHW : 1][4];
      if constexpr (EPI == EPI_BWD && sizeof(T) == 2) {
        const bf16* srcp0 = reinterpret_cast<const bf16*>(ea.relu_src);
        if (srcp0) {
#pragma unroll
          for (int k = 0; k < NCHW; ++k) {
            const int chk = sub + NSUB * k;
#pragma unroll
            for (int q = 0; q < 4; ++q)
              hpre[k][q] = (m_row < M && chk < BLOCK_N / 32)
                               ? *reinterpret_cast<const uint4*>(srcp0 + (size_t)m_row * ea.ld_src + n0 + chk * 32 + q * 8)
                               : make_uint4(0u, 0u, 0u, 0u);
          }
        }
      }
      mbar_wait(&tfull[acc], aphase);
      tc_fence_after();
      const uint32_t taddr = tmem_base + ((uint32_t)(wq * 32) << 16) + acc * BLOCK_N;
      // one 32-column chunk of this warp's accumulator rows (split tf32: main chain + small-term accumulator)
      auto ld_acc = [&](uint32_t col, float (&v)[32]) {
        tmem_ld32(taddr + col, v);
        if constexpr (X3) {
          float w[32];
          tmem_ld32(taddr + BLOCK_N + col, w);
#pragma unroll
          for (int i = 0; i < 32; ++i) v[i] += w[i];
        }
      };

      if constexpr ((EPI == EPI_LINEAR || EPI == EPI_BWD) && sizeof(T) == 2) {
        // bf16: all epilogue math in the TMEM (row-per-lane) layout, then bf16 staging (see stage_rows_bf16)
        constexpr int NCH = BLOCK_N / 32;
        bf16* outp = reinterpret_cast<bf16*>(ea.out);
        const bf16* srcp = reinterpret_cast<const bf16*>(ea.relu_src);
        uint8_t* stgb = reinterpret_cast<uint8_t*>(stg);
        const bool rowok = m_row < M;
        int bg = 0; float wv = 0.f, inv = 0.f;
        if constexpr (EPI == EPI_BWD) { bg = mybag[lane]; wv = myw[lane]; inv = myinv[lane]; }
#pragma unroll
        for (int kk = 0; kk < NCHW; ++kk) {
          const int ch = sub + NSUB * kk;
          if (ch >= NCH) break;
          const int col0 = n0 + ch * 32;
          uint4 hsrc[4];
          if constexpr (EPI == EPI_BWD) {
#pragma unroll
            for (int q = 0; q < 4; ++q) hsrc[q] = hpre[kk][q];
          }
          float v[32];
          tmem_ld32(taddr + ch * 32, v);
          if (ch + NSUB >= NCH) { release_acc(&tempty[acc]); }
          if constexpr (EPI == EPI_LINEAR) {
            if (ea.bias) {
#pragma unroll
              for (int q = 0; q < 8; ++q) {
                const float4 b4 = __ldg(reinterpret_cast<const float4*>(ea.bias + col0) + q);
                v[4 * q] += b4.x; v[4 * q + 1] += b4.y; v[4 * q + 2] += b4.z; v[4 * q + 3] += b4.w;
              }
            }
            if (ea.relu) {
#pragma unroll
              for (int i = 0; i < 32; ++i) v[i] = fmaxf(v[i], 0.f);
            }
            if (ea.drop.active) {
              if (ea.drop.mask == nullptr) {
#pragma unroll
                for (int i = 0; i < 32; i += 2) {
                  const uint32_t hb = ea.drop.bits(m_row, col0 + i);
                  v[i] = (hb & 0xFFFFu) >= ea.drop.thresh16 ? v[i] * ea.drop.inv_keep : 0.f;
                  v[i + 1] = (hb >> 16) >= ea.drop.thresh16 ? v[i + 1] * ea.drop.inv_keep : 0.f;
                }
              } else if (rowok) {
#pragma unroll
                for (int i = 0; i < 32; ++i) v[i] = ea.drop.keep(m_row, col0 + i) ? v[i] * ea.drop.inv_keep : 0.f;
              }
            }
          } else {
            if (ea.dz) {
#pragma unroll
              for (int q = 0; q < 8; ++q) {
                const float4 d4 = *(reinterpret_cast<const float4*>(ea.dz + (size_t)bg * N + col0) + q);
                v[4 * q] = fmaf(wv, d4.x, v[4 * q]); v[4 * q + 1] = fmaf(wv, d4.y, v[4 * q + 1]);
                v[4 * q + 2] = fmaf(wv, d4.z, v[4 * q + 2]); v[4 * q + 3] = fmaf(wv, d4.w, v[4 * q + 3]);
              }
            }
            if (ea.dmean) {
#pragma unroll
              for (int q = 0; q < 8; ++q) {
                const float4 d4 = *(reinterpret_cast<const float4*>(ea.dmean + (size_t)bg * N + col0) + q);
                v[4 * q] = fmaf(inv, d4.x, v[4 * q]); v[4 * q + 1] = fmaf(inv, d4.y, v[4 * q + 1]);
                v[4 * q + 2] = fmaf(inv, d4.z, v[4 * q + 2]); v[4 * q + 3] = fmaf(inv, d4.w, v[4 * q + 3]);
              }
            }
            // ReLU / dropout mask of the forward activation (1 / keep is folded into W^T and the per-row pooling weights).
            // Without accumulation the mask is applied AFTER rounding, on packed pairs: one HSET2 + one LOP per two elements
            if (srcp && ea.accumulate) {
#pragma unroll
              for (int q = 0; q < 4; ++q) {
                float sv[8];
                raw_floats(hsrc[q], sv);
#pragma unroll
                for (int e = 0; e < 8; ++e) v[8 * q + e] = sv[e] > 0.f ? v[8 * q + e] : 0.f;
              }
            }
            if (ea.accumulate && rowok) {
#pragma unroll
              for (int q = 0; q < 4; ++q) {
                float pv[8];
                ldv(outp + (size_t)m_row * ea.ldo + col0 + q * 8, pv);
#pragma unroll
                for (int e = 0; e < 8; ++e) v[8 * q + e] += pv[e];
              }
            }
          }
          if constexpr (EPI == EPI_LINEAR) {
            if (ea.out2) {     // second output: the same activations under another dropout draw (the G step's train pass)
              store_rows_bf16(stgb, v, outp, ea.ldo, m_base, M, col0, lane);
              if (ea.drop2.mask == nullptr) {
#pragma unroll
                for (int i = 0; i < 32; i += 2) {
                  const uint32_t hb = ea.drop2.bits(m_row, col0 + i);
                  v[i] = (hb & 0xFFFFu) >= ea.drop2.thresh16 ? v[i] * ea.drop2.inv_keep : 0.f;
                  v[i + 1] = (hb >> 16) >= ea.drop2.thresh16 ? v[i + 1] * ea.drop2.inv_keep : 0.f;
                }
              } else if (rowok) {
#pragma unroll
                for (int i = 0; i < 32; ++i) v[i] = ea.drop2.keep(m_row, col0 + i) ? v[i] * ea.drop2.inv_keep : 0.f;
              }
              store_rows_bf16(stgb, v, reinterpret_cast<bf16*>(ea.out2), ea.ldo, m_base, M, col0, lane);
              continue;
            }
          }
          bool staged = false;
          if constexpr (EPI == EPI_BWD) {
           if (srcp && !ea.accumulate) {
            uint32_t pw[16];
            const __nv_bfloat162 zero2 = __floats2bfloat162_rn(0.f, 0.f);
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              const uint32_t hw[4] = {hsrc[q].x, hsrc[q].y, hsrc[q].z, hsrc[q].w};
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                const uint32_t keep2 = __hgt2_mask(*reinterpret_cast<const __nv_bfloat162*>(&hw[e]), zero2);
                pw[4 * q + e] = pack_bf2(v[8 * q + 2 * e], v[8 * q + 2 * e + 1]) & keep2;
              }
            }
            stage_words_bf16(stgb, pw, lane);
            staged = true;
           }
          }
          if (!staged) stage_rows_bf16(stgb, v, lane);
          __syncwarp();
          float cs[8];
#pragma unroll
          for (int e = 0; e < 8; ++e) cs[e] = 0.f;
#pragma unroll
          for (int it2 = 0; it2 < 4; ++it2) {
            const int r = (lane >> 2) + 8 * it2, cv = lane & 3, m = m_base + r;
            const uint4 qv = *reinterpret_cast<const uint4*>(stgb + stgb_off(r, cv));
            if (m < M) {
              *reinterpret_cast<uint4*>(outp + (size_t)m * ea.ldo + col0 + cv * 8) = qv;
              if constexpr (EPI == EPI_BWD) {
                float o[8];
                raw_floats(qv, o);
#pragma unroll
                for (int e = 0; e < 8; ++e) cs[e] += o[e];
              }
            }
          }
          if constexpr (EPI == EPI_BWD) {
            if (ea.colpart) {      // column sums of this warp's 32 rows: halving butterfly over the 8 lanes that share cv
              const bool up0 = (lane >> 2) & 1, up1 = (lane >> 3) & 1, up2 = (lane >> 4) & 1;
              float k4[4], k2[2];
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                const float recv = __shfl_xor_sync(0xffffffffu, up0 ? cs[e] : cs[e + 4], 4);
                k4[e] = (up0 ? cs[e + 4] : cs[e]) + recv;
              }
#pragma unroll
              for (int e = 0; e < 2; ++e) {
                const float recv = __shfl_xor_sync(0xffffffffu, up1 ? k4[e] : k4[e + 2], 8);
                k2[e] = (up1 ? k4[e + 2] : k4[e]) + recv;
              }
              const float recv = __shfl_xor_sync(0xffffffffu, up2 ? k2[0] : k2[1], 16);
              const float tot = (up2 ? k2[1] : k2[0]) + recv;
              ea.colpart[(size_t)(mt * 4 + wq) * N + col0 + (lane & 3) * 8 + (up0 ? 4 : 0) + (up1 ? 2 : 0) + (up2 ? 1 : 0)] = tot;
            }
          }
          __syncwarp();
        }
      } else if constexpr (EPI == EPI_LINEAR || EPI == EPI_BWD) {
        constexpr int NCH = BLOCK_N / 32;
        constexpr int LPR = 32 / VEC, RPI = 32 / LPR, NIT = 32 / RPI;   // lanes per row, rows per pass, passes per chunk
        T* outp = reinterpret_cast<T*>(ea.out);
        const T* srcp = reinterpret_cast<const T*>(ea.relu_src);
#pragma unroll 1
        for (int ch = sub; ch < NCH; ch += NSUB) {
          uint4 src[NIT];
          if constexpr (EPI == EPI_BWD) {                  // issue the ReLU-mask loads before touching TMEM
            if (srcp) {
#pragma unroll
              for (int it2 = 0; it2 < NIT; ++it2) {
                const int r = lane / LPR + RPI * it2, m = m_base + r, col = n0 + ch * 32 + (lane % LPR) * VEC;
                src[it2] = (m < M) ? *reinterpret_cast<const uint4*>(srcp + (size_t)m * ea.ld_src + col) : make_uint4(0u, 0u, 0u, 0u);
              }
            }
          }
          float v[32];
          ld_acc(ch * 32, v);
          if (ch + NSUB >= NCH) { release_acc(&tempty[acc]); }
          stage_chunk(stg, STG_LD, 0, v, lane);
          __syncwarp();
          float cs[VEC];
#pragma unroll
          for (int e = 0; e < VEC; ++e) cs[e] = 0.f;
#pragma unroll
          for (int it2 = 0; it2 < NIT; ++it2) {
            const int r = lane / LPR + RPI * it2, cv = lane % LPR;
            const int m = m_base + r, col = n0 + ch * 32 + cv * VEC;
            if (m < M) {
              float o[VEC];
#pragma unroll
              for (int q = 0; q < VEC / 4; ++q) {
                const float4 t4 = *reinterpret_cast<const float4*>(stg + r * STG_LD + cv * VEC + 4 * q);
                o[4 * q] = t4.x; o[4 * q + 1] = t4.y; o[4 * q + 2] = t4.z; o[4 * q + 3] = t4.w;
              }
              if constexpr (EPI == EPI_LINEAR) {
                if (ea.bias) {
#pragma unroll
                  for (int q = 0; q < VEC / 4; ++q) {
                    const float4 b4 = *reinterpret_cast<const float4*>(ea.bias + col + 4 * q);
                    o[4 * q] += b4.x; o[4 * q + 1] += b4.y; o[4 * q + 2] += b4.z; o[4 * q + 3] += b4.w;
                  }
                }
                if (ea.relu) {
#pragma unroll
                  for (int e = 0; e < VEC; ++e) o[e] = fmaxf(o[e], 0.f);
                }
                if (ea.drop.active) {
                  if (ea.drop.mask == nullptr) {
#pragma unroll
                    for (int e = 0; e < VEC; e += 2) {
                      const uint32_t hb = ea.drop.bits(m, col + e);
                      o[e] = (hb & 0xFFFFu) >= ea.drop.thresh16 ? o[e] * ea.drop.inv_keep : 0.f;
                      o[e + 1] = (hb >> 16) >= ea.drop.thresh16 ? o[e + 1] * ea.drop.inv_keep : 0.f;
                    }
                  } else {
#pragma unroll
                    for (int e = 0; e < VEC; ++e) o[e] = ea.drop.keep(m, col + e) ? o[e] * ea.drop.inv_keep : 0.f;
                  }
                }
              } else {
                if (ea.dz) {
                  const float wv = myw[r];
#pragma unroll
                  for (int q = 0; q < VEC / 4; ++q) {
                    const float4 d4 = *reinterpret_cast<const float4*>(ea.dz + (size_t)mybag[r] * N + col + 4 * q);
                    o[4 * q] = fmaf(wv, d4.x, o[4 * q]); o[4 * q + 1] = fmaf(wv, d4.y, o[4 * q + 1]);
                    o[4 * q + 2] = fmaf(wv, d4.z, o[4 * q + 2]); o[4 * q + 3] = fmaf(wv, d4.w, o[4 * q + 3]);
                  }
                }
                if (ea.dmean) {
                  const float iv = myinv[r];
#pragma unroll
                  for (int q = 0; q < VEC / 4; ++q) {
                    const float4 d4 = *reinterpret_cast<const float4*>(ea.dmean + (size_t)mybag[r] * N + col + 4 * q);
                    o[4 * q] = fmaf(iv, d4.x, o[4 * q]); o[4 * q + 1] = fmaf(iv, d4.y, o[4 * q + 1]);
                    o[4 * q + 2] = fmaf(iv, d4.z, o[4 * q + 2]); o[4 * q + 3] = fmaf(iv, d4.w, o[4 * q + 3]);
                  }
                }
                if (srcp) {
                  float sv[VEC];
                  raw_floats(src[it2], sv);
#pragma unroll
                  for (int e = 0; e < VEC; ++e) o[e] = sv[e] > 0.f ? o[e] : 0.f;
                }
                if (ea.accumulate) {
                  float pv[VEC];
                  ldv(outp + (size_t)m * ea.ldo + col, pv);
#pragma unroll
                  for (int e = 0; e < VEC; ++e) o[e] += pv[e];
                }
#pragma unroll
                for (int e = 0; e < VEC; ++e) cs[e] += o[e];
              }
              stv(outp + (size_t)m * ea.ldo + col, o);
              if constexpr (EPI == EPI_LINEAR) {
                if (ea.out2) {
#pragma unroll
                  for (int e = 0; e < VEC; ++e) o[e] = ea.drop2.keep(m, col + e) ? o[e] * ea.drop2.inv_keep : 0.f;
                  stv(reinterpret_cast<T*>(ea.out2) + (size_t)m * ea.ldo + col, o);
                }
              }
            }
          }
          if constexpr (EPI == EPI_BWD) {
            if (ea.colpart) {
              // bias gradient for free: column sums of this warp's 32 rows.  The RPI lanes that share a column vector
              // (lane = cv + LPR * k) fold with a halving butterfly: each step exchanges half of the remaining values, so
              // VEC - 1 shuffles leave ONE column sum per lane and the 32 lanes store 32 distinct columns (128 bytes).
              int colsel = 0;
              if constexpr (VEC == 8) {
                const bool up0 = (lane / LPR) & 1;
                float k4[4];
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                  const float recv = __shfl_xor_sync(0xffffffffu, up0 ? cs[e] : cs[e + 4], LPR);
                  k4[e] = (up0 ? cs[e + 4] : cs[e]) + recv;
                }
                const bool up1 = (lane / (2 * LPR)) & 1;
                float k2[2];
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                  const float recv = __shfl_xor_sync(0xffffffffu, up1 ? k4[e] : k4[e + 2], 2 * LPR);
                  k2[e] = (up1 ? k4[e + 2] : k4[e]) + recv;
                }
                const bool up2 = (lane / (4 * LPR)) & 1;
                const float recv = __shfl_xor_sync(0xffffffffu, up2 ? k2[0] : k2[1], 4 * LPR);
                cs[0] = (up2 ? k2[1] : k2[0]) + recv;
                colsel = (up0 ? 4 : 0) + (up1 ? 2 : 0) + (up2 ? 1 : 0);
              } else {
                const bool up0 = (lane / LPR) & 1;
                float k2[2];
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                  const float recv = __shfl_xor_sync(0xffffffffu, up0 ? cs[e] : cs[e + 2], LPR);
                  k2[e] = (up0 ? cs[e + 2] : cs[e]) + recv;
                }
                const bool up1 = (lane / (2 * LPR)) & 1;
                const float recv = __shfl_xor_sync(0xffffffffu, up1 ? k2[0] : k2[1], 2 * LPR);
                cs[0] = (up1 ? k2[1] : k2[0]) + recv;
                colsel = (up0 ? 2 : 0) + (up1 ? 1 : 0);
              }
              ea.colpart[(size_t)(mt * 4 + wq) * N + n0 + ch * 32 + (lane % LPR) * VEC + colsel] = cs[0];
            }
          }
          __syncwarp();
        }
      } else if constexpr (EPI == EPI_PE) {
        // Stacked weights [W1; Wc]: this warp owns 128 columns of the 256-wide tile.  Columns below h_cols are the
        // generator projection h = relu(x W1^T + b1) (plus the G step's dropped copy); the last 128 columns are the
        // discriminator's y = x Wc^T + bc -> LayerNorm -> ReLU -> 16-row region mean.  x is read from HBM once for both.
        static_assert(EPI != EPI_PE || (BLOCK_N == 256 && sizeof(T) == 2), "proj+embed epilogue: bf16, 256-column tiles");
        const int cb = n0 + half * 128;
        uint8_t* stgb = reinterpret_cast<uint8_t*>(stg);
        const bool rowok = m_row < M;
        const uint32_t tcol = taddr + half * 128;
        if (cb < ea.h_cols) {
          bf16* outp = reinterpret_cast<bf16*>(ea.out);
#pragma unroll 1
          for (int k = 0; k < 4; ++k) {
            const int col0 = cb + k * 32;
            float v[32];
            tmem_ld32(tcol + k * 32, v);
            if (k == 3) { release_acc(&tempty[acc]); }
#pragma unroll
            for (int q = 0; q < 8; ++q) {
              const float4 b4 = __ldg(reinterpret_cast<const float4*>(ea.bias + col0) + q);
              v[4 * q] = fmaxf(v[4 * q] + b4.x, 0.f); v[4 * q + 1] = fmaxf(v[4 * q + 1] + b4.y, 0.f);
              v[4 * q + 2] = fmaxf(v[4 * q + 2] + b4.z, 0.f); v[4 * q + 3] = fmaxf(v[4 * q + 3] + b4.w, 0.f);
            }
            store_rows_bf16(stgb, v, outp, ea.ldo, m_base, M, col0, lane);
            if (ea.out2) {
              if (ea.drop2.mask == nullptr) {
#pragma unroll
                for (int i = 0; i < 32; i += 2) {
                  const uint32_t hb = ea.drop2.bits(m_row, col0 + i);
                  v[i] = (hb & 0xFFFFu) >= ea.drop2.thresh16 ? v[i] * ea.drop2.inv_keep : 0.f;
                  v[i + 1] = (hb >> 16) >= ea.drop2.thresh16 ? v[i + 1] * ea.drop2.inv_keep : 0.f;
                }
              } else if (rowok) {
#pragma unroll
                for (int i = 0; i < 32; ++i) v[i] = ea.drop2.keep(m_row, col0 + i) ? v[i] * ea.drop2.inv_keep : 0.f;
              }
              store_rows_bf16(stgb, v, reinterpret_cast<bf16*>(ea.out2), ea.ldo, m_base, M, col0, lane);
            }
          }
        } else {
          // three sweeps over the 128 TMEM columns of this row (sum -> mean, squares -> rstd, normalise) keep the register
          // footprint at one 32-column chunk; y is rounded to bf16 first: y_pre IS a bf16 tensor (see EPI_LN)
          float ssum = 0.f;
#pragma unroll 1
          for (int k = 0; k < 4; ++k) {
            float v[32];
            tmem_ld32(tcol + k * 32, v);
#pragma unroll
            for (int i = 0; i < 32; ++i) ssum += __bfloat162float(__float2bfloat16_rn(v[i] + coef[k * 32 + i]));
          }
          const float mean = ssum * (1.0f / 128.0f);
          float qsum = 0.f;
#pragma unroll 1
          for (int k = 0; k < 4; ++k) {
            float v[32];
            tmem_ld32(tcol + k * 32, v);
#pragma unroll
            for (int i = 0; i < 32; ++i) {
              const float c = __bfloat162float(__float2bfloat16_rn(v[i] + coef[k * 32 + i])) - mean;
              qsum = fmaf(c, c, qsum);
            }
          }
          const float rstd = rsqrtf(qsum * (1.0f / 128.0f) + ea.eps);
#pragma unroll 1
          for (int k = 0; k < 4; ++k) {
            float v[32];
            tmem_ld32(tcol + k * 32, v);
            if (k == 3) { release_acc(&tempty[acc]); }
#pragma unroll
            for (int i = 0; i < 32; ++i) v[i] = __bfloat162float(__float2bfloat16_rn(v[i] + coef[k * 32 + i]));
            if (ea.y_pre) store_rows_bf16(stgb, v, reinterpret_cast<bf16*>(ea.y_pre), 128, m_base, M, k * 32, lane);
#pragma unroll
            for (int i = 0; i < 32; ++i)
              v[i] = rowok ? fmaxf(fmaf((v[i] - mean) * rstd, coef[128 + k * 32 + i], coef[256 + k * 32 + i]), 0.f) : 0.f;
            stage_chunk(stg, STG_LD, 0, v, lane);
            __syncwarp();
            const int rg = lane >> 4, c2 = (lane & 15) * 2;      // two 16-row regions per warp, two columns per lane
            float a0 = 0.f, a1 = 0.f;
#pragma unroll
            for (int r = 0; r < 16; ++r) {
              const float2 t2 = *reinterpret_cast<const float2*>(stg + (rg * 16 + r) * STG_LD + c2);
              a0 += t2.x; a1 += t2.y;
            }
            const int m = m_base + rg * 16;
            if (m < M) *reinterpret_cast<float2*>(ea.emb + (size_t)(m >> 4) * 128 + k * 32 + c2) = make_float2(a0 * 0.0625f, a1 * 0.0625f);
            __syncwarp();
          }
        }
      } else if constexpr (EPI == EPI_POOL) {
        // K9 (DeepAttMISL, model/backbone.py:105-117): v = relu(x W^T + b) is summed per (bag, cluster id) here and never
        // written.  Bag lengths are multiples of 16 and a warp owns 32 aligned rows, so each 16-row half of a warp lies in
        // one bag; a tile is 8 such segments.  Per 32-column chunk: lane c adds column c of its two halves, row by row, into
        // per-cluster sums in shared memory; then (named barrier over the 4 epilogue warps) the 4 warps, a quarter of the
        // clusters each, add each bag's segments in row order and write one partial per (tile, bag, cluster).
        // No atomics: the result does not depend on scheduling.  cluster_pool_finalize adds the partials in a fixed order.
        constexpr int NCH = BLOCK_N / 32;
        const int ncl = ea.D;
        float* sacc = coef;                                 // [2 halves][16 clusters][32 columns] of this warp
        uint32_t* keep = reinterpret_cast<uint32_t*>(ea.out);
        auto seg_bag = [&](int sg) { return rowbag[(sg >> 1) * 32 + (sg & 1) * 16]; };
#pragma unroll 1
        for (int ch = 0; ch < NCH; ++ch) {
          const int col0 = n0 + ch * 32;
          float v[32];
          ld_acc(ch * 32, v);
          if (ch == NCH - 1) { release_acc(&tempty[acc]); }
#pragma unroll
          for (int q = 0; q < 8; ++q) {
            const float4 b4 = __ldg(reinterpret_cast<const float4*>(ea.bias + col0) + q);
            v[4 * q] += b4.x; v[4 * q + 1] += b4.y; v[4 * q + 2] += b4.z; v[4 * q + 3] += b4.w;
          }
          if (keep && m_row < M) {
            uint32_t kw = 0;
#pragma unroll
            for (int i = 0; i < 32; ++i) kw |= (v[i] > 0.f ? 1u : 0u) << i;
            keep[(size_t)m_row * ea.ldo + (col0 >> 5)] = kw;
          }
#pragma unroll
          for (int i = 0; i < 32; ++i) v[i] = fmaxf(v[i], 0.f);
          stage_chunk(stg, STG_LD, 0, v, lane);
          for (int k = 0; k < ncl; ++k) { sacc[k * 32 + lane] = 0.f; sacc[(16 + k) * 32 + lane] = 0.f; }
          __syncwarp();
#pragma unroll 4
          for (int r = 0; r < 32; ++r) {
            const int k = __shfl_sync(0xffffffffu, pool_cid, r);
            const float xv = stg[r * STG_LD + lane];
            if ((unsigned)k < (unsigned)ncl) sacc[((r >> 4) * 16 + k) * 32 + lane] += xv;
          }
          asm volatile("bar.sync 1, 128;" ::: "memory");      // the tile's 8 segments of this chunk are summed
          // every warp writes the clusters k = wq, wq + 4, ... of each bag in the tile: the bag's segments (adjacent) are
          // added in row order; the 8 loads are issued before the adds
#pragma unroll 1
          for (int sg = 0; sg < 8; ++sg) {
            const int b = seg_bag(sg);
            if (b < 0 || (sg > 0 && seg_bag(sg - 1) == b)) continue;     // not the first segment of its bag in this tile
            int se = sg;
            while (se < 7 && seg_bag(se + 1) == b) ++se;
            float* dst = ea.part + (size_t)(mt + b) * ncl * N + col0 + lane;
#pragma unroll 1
            for (int k = wq; k < ncl; k += 4) {
              float xs[8];
#pragma unroll
              for (int s2 = 0; s2 < 8; ++s2) xs[s2] = coef_all[(s2 >> 1) * Cfg::COEF_FLOATS_PER_WARP + ((s2 & 1) * 16 + k) * 32 + lane];
              float t = 0.f;
#pragma unroll
              for (int s2 = 0; s2 < 8; ++s2) if (s2 >= sg && s2 <= se) t += xs[s2];
              dst[(size_t)k * N] = t;
            }
          }
          asm volatile("bar.sync 1, 128;" ::: "memory");      // before the next chunk overwrites the sums and the staging
        }
      } else if constexpr (EPI == EPI_GATE) {
        // BLOCK_N = 256 = two packed gate blocks (64 tanh | 64 sigmoid columns) = four 32-pair chunks; this warp owns
        // 4 / NSUB of them.  One partial score per 128-column gate block: with 4 warps per lane quarter the warps of
        // chunks 2k and 2k+1 meet on a named barrier and the even one stores the sum (same order as the 2-warp variant's
        // sequential accumulation up to one rounding).
        static_assert(EPI != EPI_GATE || BLOCK_N == 256, "gate epilogue expects 256-column tiles");
        constexpr int PCW = 4 / NSUB;
        float partial = 0.f;
        const bool train = ea.drop_a.active != 0;
        const bool masked = ea.drop_a.mask != nullptr || ea.drop_b.mask != nullptr;
#pragma unroll 1
        for (int q = 0; q < PCW; ++q) {
          const int pc = sub * PCW + q;
          const int ca = (pc >> 1) * 128 + (pc & 1) * 32, cb = ca + 64;
          const int j0 = (n0 >> 1) + pc * 32;               // logical gate column of element 0
          const float* cf = coef + q * 96;
          float va[32], vb[32];
          ld_acc(ca, va);
          ld_acc(cb, vb);
          if (q == PCW - 1) { release_acc(&tempty[acc]); }
          if (!train) partial = gate_chunk<FAST, 0>(va, vb, cf, cf + 32, cf + 64, ea.drop_a, ea.drop_b, m_row, j0, partial);
          else if (!masked) partial = gate_chunk<FAST, 1>(va, vb, cf, cf + 32, cf + 64, ea.drop_a, ea.drop_b, m_row, j0, partial);
          else partial = gate_chunk<FAST, 2>(va, vb, cf, cf + 32, cf + 64, ea.drop_a, ea.drop_b, m_row, j0, partial, m_row < M);
          if constexpr (sizeof(T) == 2) {
            if (ea.ab) {
              store_rows_bf16(reinterpret_cast<uint8_t*>(stg), va, reinterpret_cast<bf16*>(ea.ab), ea.ldo, m_base, M, n0 + ca, lane);
              store_rows_bf16(reinterpret_cast<uint8_t*>(stg), vb, reinterpret_cast<bf16*>(ea.ab), ea.ldo, m_base, M, n0 + cb, lane);
            }
          } else if (ea.ab) {
#pragma unroll 1
            for (int hb = 0; hb < 2; ++hb) {
              if (hb == 0) stage_chunk(stg, STG_LD, 0, va, lane); else stage_chunk(stg, STG_LD, 0, vb, lane);
              __syncwarp();
              store_staged<T, 32>(stg, STG_LD, reinterpret_cast<T*>(ea.ab), ea.ldo, m_base, M, n0 + (hb == 0 ? ca : cb), lane);
              __syncwarp();
            }
          }
          if constexpr (NSUB != 4) {        // this warp just finished a whole 128-column gate block: one partial per block
            if (pc & 1) {
              if (train) partial *= ea.drop_a.inv_keep * ea.drop_b.inv_keep;
              if (m_row < M) ea.part[(size_t)(nt * 2 + (pc >> 1)) * M + m_row] = partial;
              partial = 0.f;
            }
          }
        }
        if constexpr (NSUB == 4) {
          if (train) partial *= ea.drop_a.inv_keep * ea.drop_b.inv_keep;
          const int blk = sub >> 1;                          // gate block (128 columns) of this warp's chunk
          float* slot = gpart + ((it & 1) * 8 + wq * 2 + blk) * 32;
          if (sub & 1) slot[lane] = partial;
          asm volatile("bar.sync %0, 64;" ::"r"(1 + wq * 2 + blk) : "memory");     // the two warps of (quarter, block)
          if (!(sub & 1) && m_row < M) ea.part[(size_t)(nt * 2 + blk) * M + m_row] = partial + slot[lane];
        }
      } else if constexpr (EPI == EPI_LN && BLOCK_N != 128) {
        // BLOCK_N == d == 64 or 256: three sweeps over this row's TMEM columns (sum -> mean, squared deviations -> rstd,
        // normalise + store), one 32-column chunk in registers at a time.  A 256-float row would not fit the register file
        // the 128-column variant below already fills.  The accumulator stays allocated for the three sweeps.
        constexpr int NCH = BLOCK_N / 32;
        const bool rowok = m_row < M;
        auto ld_y = [&](int ch, float (&v)[32]) {
          ld_acc(ch * 32, v);
#pragma unroll
          for (int i = 0; i < 32; ++i) {
            float y = v[i] + __ldg(ea.bias + ch * 32 + i);
            if constexpr (sizeof(T) == 2) y = __bfloat162float(__float2bfloat16_rn(y));      // y_pre is bf16: see below
            v[i] = y;
          }
        };
        float ssum = 0.f;
#pragma unroll 1
        for (int ch = 0; ch < NCH; ++ch) {
          float v[32];
          ld_y(ch, v);
#pragma unroll
          for (int i = 0; i < 32; ++i) ssum += v[i];
        }
        const float mean = ssum * (1.0f / BLOCK_N);
        float qsum = 0.f;
#pragma unroll 1
        for (int ch = 0; ch < NCH; ++ch) {
          float v[32];
          ld_y(ch, v);
#pragma unroll
          for (int i = 0; i < 32; ++i) { const float c = v[i] - mean; qsum = fmaf(c, c, qsum); }
        }
        const float rstd = rsqrtf(qsum * (1.0f / BLOCK_N) + ea.eps);
#pragma unroll 1
        for (int ch = 0; ch < NCH; ++ch) {
          float v[32];
          ld_y(ch, v);
          if (ch == NCH - 1) { release_acc(&tempty[acc]); }
          if (ea.y_pre) {
            if constexpr (sizeof(T) == 2) {
              store_rows_bf16(reinterpret_cast<uint8_t*>(stg), v, reinterpret_cast<bf16*>(ea.y_pre), BLOCK_N, m_base, M, ch * 32, lane);
            } else {
              stage_chunk(stg, STG_LD, 0, v, lane);
              __syncwarp();
              store_staged<T, 32>(stg, STG_LD, reinterpret_cast<T*>(ea.y_pre), BLOCK_N, m_base, M, ch * 32, lane);
              __syncwarp();
            }
          }
#pragma unroll
          for (int i = 0; i < 32; ++i)
            v[i] = rowok ? fmaxf(fmaf((v[i] - mean) * rstd, __ldg(ea.gamma + ch * 32 + i), __ldg(ea.beta + ch * 32 + i)), 0.f) : 0.f;
          stage_chunk(stg, STG_LD, 0, v, lane);
          __syncwarp();
          const int rg = lane >> 4, c2 = (lane & 15) * 2;      // two 16-row regions per warp, two columns per lane
          float a0 = 0.f, a1 = 0.f;
#pragma unroll
          for (int r = 0; r < 16; ++r) {
            const float2 t2 = *reinterpret_cast<const float2*>(stg + (rg * 16 + r) * STG_LD + c2);
            a0 += t2.x; a1 += t2.y;
          }
          const int m = m_base + rg * 16;
          if (m < M) *reinterpret_cast<float2*>(ea.emb + (size_t)(m >> 4) * BLOCK_N + ch * 32 + c2) = make_float2(a0 * 0.0625f, a1 * 0.0625f);
          __syncwarp();
        }
      } else if constexpr (EPI == EPI_LN) {
        // BLOCK_N == 128 == d: the whole row lives in this thread's registers
        float v[128];
#pragma unroll
        for (int ch = 0; ch < 4; ++ch) {
          float t[32];
          ld_acc(ch * 32, t);
#pragma unroll
          for (int i = 0; i < 32; ++i) {
            float y = t[i] + __ldg(ea.bias + ch * 32 + i);
            // bf16 mode: y_pre IS a bf16 tensor -- LayerNorm sees the rounded values, so that the backward pass (which
            // re-derives the statistics and the ReLU mask from the stored y_pre) sees exactly what the forward saw
            if constexpr (sizeof(T) == 2) y = __bfloat162float(__float2bfloat16_rn(y));
            v[ch * 32 + i] = y;
          }
        }
        release_acc(&tempty[acc]);
        float s = 0.f;
#pragma unroll
        for (int i = 0; i < 128; ++i) s += v[i];
        const float mean = s * (1.0f / 128.0f);
        float q = 0.f;
#pragma unroll
        for (int i = 0; i < 128; ++i) { const float c = v[i] - mean; q = fmaf(c, c, q); }
        const float rstd = rsqrtf(q * (1.0f / 128.0f) + ea.eps);
        if (ea.y_pre) {
#pragma unroll
          for (int j = 0; j < 32; ++j)
            *reinterpret_cast<float4*>(stg + lane * STG_LD_LN + 4 * j) = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
          __syncwarp();
          store_staged<T, 128>(stg, STG_LD_LN, reinterpret_cast<T*>(ea.y_pre), 128, m_base, M, 0, lane);
          __syncwarp();
        }
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          float e[4];
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const int c = 4 * j + k;
            e[k] = (m_row < M) ? fmaxf(fmaf((v[c] - mean) * rstd, __ldg(ea.gamma + c), __ldg(ea.beta + c)), 0.f) : 0.f;
          }
          *reinterpret_cast<float4*>(stg + lane * STG_LD_LN + 4 * j) = make_float4(e[0], e[1], e[2], e[3]);
        }
        __syncwarp();
#pragma unroll
        for (int rg = 0; rg < 2; ++rg) {          // two 16-row regions per warp
          float4 a4 = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
          for (int r = 0; r < 16; ++r) {
            const float4 t4 = *reinterpret_cast<const float4*>(stg + (rg * 16 + r) * STG_LD_LN + lane * 4);
            a4.x += t4.x; a4.y += t4.y; a4.z += t4.z; a4.w += t4.w;
          }
          const int m = m_base + rg * 16;
          if (m < M)
            *reinterpret_cast<float4*>(ea.emb + (size_t)(m >> 4) * 128 + lane * 4) =
                make_float4(a4.x * 0.0625f, a4.y * 0.0625f, a4.z * 0.0625f, a4.w * 0.0625f);
        }
        __syncwarp();
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) { tc_fence_after(); tmem_dealloc(tmem_base, Cfg::TMEM_COLS); }
}

// CTA pairs (tcgen05.mma.cta_group::2, M = 256, each CTA loading half of the weight tile) were measured, no gain: within
// 3 % of this kernel and mostly slower on B200 (the epilogue's HBM writes and latency bound it, not operand ingress).
// CONV: A is x [rows, K / 9] (rows % 16 == 0), read through its region view
template <typename T, int BLOCK_N, int EPI, bool FAST, bool X3 = false, bool CONV = false>
static int launch_rows(const T* A, const T* W, int rows, int K, int N, const RowEpi& ea, cudaStream_t st, const T* Wlo = nullptr) {
  using Cfg = RowCfg<(int)sizeof(T), BLOCK_N, EPI, X3>;
  const int num_m = cdiv(rows, TILE_M), num_n = N / BLOCK_N;
  CUtensorMap tmA, tmB, tmBlo;
  if constexpr (CONV) ADVMIL_TRY(make_tmap_regions<T>(&tmA, A, rows / 16, K / 9, TILE_M / 16));
  else ADVMIL_TRY(make_tmap<T>(&tmA, A, rows, K, TILE_M));
  ADVMIL_TRY(make_tmap<T>(&tmB, W, N, K, BLOCK_N));
  ADVMIL_TRY(make_tmap<T>(&tmBlo, X3 ? Wlo : W, N, K, BLOCK_N));
  auto kern = tc_rows_kernel<T, BLOCK_N, EPI, FAST, X3, CONV>;
  static bool attr_set = false;
  if (!attr_set) {
    ADVMIL_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Cfg::SMEM));
    attr_set = true;
  }
  const int grid = min(num_m * num_n, sm_count());
  launch_k(kern, dim3(grid), dim3(Cfg::THREADS), Cfg::SMEM, st, tmA, tmB, tmBlo, rows, N, K, ea);
  ADVMIL_CHECK_LAUNCH();
  return ADVMIL_OK;
}

// ------------------------------------------------------------------------------------------------
// weight-gradient kernel: dW[N1,N2] partial over a row range; both operands MN-major
//   fp32 (tf32): MN groups of 32 elements, 32 k-rows per stage, SWIZZLE_128B with 32-byte atoms (the only swizzle the
//                hardware accepts for MN-major 32-bit operands), 8 k-rows (two 512-byte groups) per MMA;
//   bf16:        MN groups of 64 elements, 64 k-rows per stage, plain SWIZZLE_128B, 16 k-rows (two 1024-byte atoms) per MMA.
// Either way one MN group of one stage is a TMA box of KR rows x 128 bytes and a stage holds 4 MMAs.
// ------------------------------------------------------------------------------------------------
template <typename T, int BLOCK_N, bool X3 = false> struct WgCfg {
  static constexpr int STAGES = X3 ? 2 : 4;                      // split-tf32: a stage holds hi and lo of both operands
  static constexpr int MNG = TcElem<T>::KBLK;                    // elements per 128-byte MN group
  static constexpr int KR = TcElem<T>::KBLK;                     // k-rows (= instance rows) per stage
  static constexpr int A_GROUPS = TILE_M / MNG, B_GROUPS = BLOCK_N / MNG;
  static constexpr int GROUP_BYTES = KR * 128;
  static constexpr int A_BYTES = A_GROUPS * GROUP_BYTES;         // 16 KB
  static constexpr int B_BYTES = B_GROUPS * GROUP_BYTES;
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;          // what TMA delivers per stage
  static constexpr int MMA_BYTES = (KR / 4) * 128;               // k-rows per MMA x 128 B
  static constexpr int ACC_COLS = BLOCK_N <= 128 ? 128 : 256;
  static constexpr int TMEM_COLS = X3 ? 2 * ACC_COLS : ACC_COLS;   // split tf32: second accumulator for the small terms
  static constexpr size_t SMEM = 1024 + (size_t)STAGES * STAGE_BYTES * (X3 ? 2 : 1) + 4 * 32 * STG_LD * 4 + 256;
};

// CONV: dWc of the 3x3 region convolution, N2 = 9 C tap-major (column tap * C + c); tmB is the region view of x with
// KR / 16 regions per box, and a BLOCK_N-column tile (C % BLOCK_N == 0) reads x shifted by its tap
template <typename T, int BLOCK_N, bool X3 = false, bool CONV = false>
__global__ void __launch_bounds__(256, 1)
tc_wgrad_kernel(const __grid_constant__ CUtensorMap tmA /*dY*/, const __grid_constant__ CUtensorMap tmB /*X*/,
                int rows, int N1, int N2, int rows_per_split, float* __restrict__ ws) {
  pdl_prologue();
  using Cfg = WgCfg<T, BLOCK_N, X3>;
  constexpr int STAGES = Cfg::STAGES, KR = Cfg::KR, MNG = Cfg::MNG;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);   // pointer arithmetic keeps the shared address space
  // A and B of a stage are contiguous ([A | B] per stage) so that the split-tf32 converter sweeps one range; the low parts
  // mirror that layout in a second region
  constexpr int SB = Cfg::STAGE_BYTES;
  uint8_t* S_s = smem;                                  // [STAGES][A | B]            (hi / raw)
  uint8_t* L_s = smem + STAGES * SB;                    // [STAGES][A_lo | B_lo]      (X3 only)
  float* stg_all = (float*)(L_s + (X3 ? STAGES * SB : 0));
  uint64_t* bars = (uint64_t*)(stg_all + 4 * 32 * STG_LD);
  uint64_t* full = bars;
  uint64_t* empty = bars + STAGES;
  uint64_t* conv = bars + 2 * STAGES;                   // X3: both operands of the stage have been split
  uint64_t* tfull = bars + 3 * STAGES;
  uint32_t* tmem_ptr = (uint32_t*)(tfull + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int num_n = N2 / BLOCK_N;
  const int mt = blockIdx.x / num_n, nt = blockIdx.x % num_n;
  const int m0 = mt * TILE_M, n0 = nt * BLOCK_N;
  const int r_beg = blockIdx.y * rows_per_split, r_end = min(rows, r_beg + rows_per_split);
  const int kblocks = (r_end - r_beg + KR - 1) / KR;     // rows past `rows` are zero-filled by TMA

  if (threadIdx.x == 0) {
    prefetch_tmap(&tmA);
    prefetch_tmap(&tmB);
    for (int i = 0; i < STAGES; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); mbar_init(&conv[i], 128); }
    mbar_init(tfull, 1);
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc(tmem_ptr, Cfg::TMEM_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  if (warp == 0) {
    if (lane == 0) {
      int stage = 0; uint32_t phase = 0;
      for (int kb = 0; kb < kblocks; ++kb) {
        const int r0 = r_beg + kb * KR;
        mbar_wait(&empty[stage], phase ^ 1);
        mbar_arrive_expect_tx(&full[stage], Cfg::STAGE_BYTES);
#pragma unroll
        for (int g = 0; g < Cfg::A_GROUPS; ++g)
          tma_load_2d(S_s + stage * SB + g * Cfg::GROUP_BYTES, &tmA, &full[stage], m0 + g * MNG, r0);
        if constexpr (CONV) {
          const int C = N2 / 9, tap = n0 / C, c0 = n0 - tap * C;
#pragma unroll
          for (int g = 0; g < Cfg::B_GROUPS; ++g)
            tma_load_4d(S_s + stage * SB + Cfg::A_BYTES + g * Cfg::GROUP_BYTES, &tmB, &full[stage], c0 + g * MNG, tap % 3 - 1,
                        tap / 3 - 1, r0 >> 4);
        } else {
#pragma unroll
          for (int g = 0; g < Cfg::B_GROUPS; ++g)
            tma_load_2d(S_s + stage * SB + Cfg::A_BYTES + g * Cfg::GROUP_BYTES, &tmB, &full[stage], n0 + g * MNG, r0);
        }
        if (++stage == STAGES) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp == 1) {
    constexpr uint32_t IDESC = TcElem<T>::idesc(TILE_M, BLOCK_N, 1, 1);
    int stage = 0; uint32_t phase = 0;
    for (int kb = 0; kb < kblocks; ++kb) {
      if (X3) mbar_wait(&conv[stage], phase); else mbar_wait(&full[stage], phase);
      tc_fence_after();
      if (lane == 0) {
        const uint32_t a_addr = smem_u32(S_s + stage * SB), b_addr = a_addr + Cfg::A_BYTES;
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) {   // LBO = stride between MN groups, SBO = stride between k-row swizzle groups
          uint64_t ad = smem_desc_sw128(a_addr + kk * Cfg::MMA_BYTES, Cfg::GROUP_BYTES, TcElem<T>::MN_SBO, TcElem<T>::MN_LAYOUT);
          uint64_t bd = smem_desc_sw128(b_addr + kk * Cfg::MMA_BYTES, Cfg::GROUP_BYTES, TcElem<T>::MN_SBO, TcElem<T>::MN_LAYOUT);
          TcElem<T>::mma(tmem_base, ad, bd, IDESC, (kb | kk) != 0 ? 1u : 0u);
          if constexpr (X3) {              // + lo.hi + hi.lo
            const uint32_t al_addr = smem_u32(L_s + stage * SB), bl_addr = al_addr + Cfg::A_BYTES;
            uint64_t ald = smem_desc_sw128(al_addr + kk * Cfg::MMA_BYTES, Cfg::GROUP_BYTES, TcElem<T>::MN_SBO, TcElem<T>::MN_LAYOUT);
            uint64_t bld = smem_desc_sw128(bl_addr + kk * Cfg::MMA_BYTES, Cfg::GROUP_BYTES, TcElem<T>::MN_SBO, TcElem<T>::MN_LAYOUT);
            TcElem<T>::mma(tmem_base + Cfg::ACC_COLS, ald, bd, IDESC, (kb | kk) != 0 ? 1u : 0u);   // own accumulator: see tc_rows_kernel
            TcElem<T>::mma(tmem_base + Cfg::ACC_COLS, ad, bld, IDESC, 1u);
          }
        }
        mma_commit(&empty[stage]);
        if (kb == kblocks - 1) mma_commit(tfull);
      }
      __syncwarp();
      if (++stage == STAGES) { stage = 0; phase ^= 1; }
    }
  } else if (warp >= 4) {
    if constexpr (X3) {     // during the main loop the (otherwise idle) epilogue warps are the split-tf32 converter: 128 threads
      const int ct = threadIdx.x - 128;
      int stage = 0; uint32_t phase = 0;
      for (int kb = 0; kb < kblocks; ++kb) {
        mbar_wait(&full[stage], phase);
        uint4* hi = reinterpret_cast<uint4*>(S_s + stage * SB);
        uint4* lo = reinterpret_cast<uint4*>(L_s + stage * SB);
#pragma unroll 4
        for (int i = ct; i < SB / 16; i += 128) {
          uint4 h4, l4;
          split_tf32(hi[i], h4, l4);
          hi[i] = h4; lo[i] = l4;
        }
        fence_proxy_async();
        mbar_arrive(&conv[stage]);
        if (++stage == STAGES) { stage = 0; phase ^= 1; }
      }
    }
    const int wq = warp & 3;
    float* stg = stg_all + wq * 32 * STG_LD;
    float* out = ws + (size_t)blockIdx.y * N1 * N2;
    const int m_base = m0 + wq * 32;
    if (kblocks > 0) {
      mbar_wait(tfull, 0);
      tc_fence_after();
    }
    const uint32_t taddr = tmem_base + ((uint32_t)(wq * 32) << 16);
#pragma unroll 1
    for (int ch = 0; ch < BLOCK_N / 32; ++ch) {
      float v[32];
      if (kblocks > 0) {
        tmem_ld32(taddr + ch * 32, v);
        if constexpr (X3) {
          float w[32];
          tmem_ld32(taddr + Cfg::ACC_COLS + ch * 32, w);
#pragma unroll
          for (int i = 0; i < 32; ++i) v[i] += w[i];
        }
      } else {
#pragma unroll
        for (int i = 0; i < 32; ++i) v[i] = 0.f;
      }
      stage_chunk(stg, STG_LD, 0, v, lane);
      __syncwarp();
      store_staged<float, 32>(stg, STG_LD, out, N2, m_base, N1, n0 + ch * 32, lane);
      __syncwarp();
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) { tc_fence_after(); tmem_dealloc(tmem_base, Cfg::TMEM_COLS); }
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
static int pick_block_n(int N) {
  if (N % 192 == 0 && N % 256 != 0) return 192;
  if (N % 256 == 0) return 256;
  if (N % 128 == 0) return 128;
  if (N == 64) return 64;
  return 0;
}
static int kblk_of(int dt) { return dt == ELEM_BF16 ? TcElem<bf16>::KBLK : TcElem<float>::KBLK; }

// library-owned, grow-only scratch for operand copies of the (small) weights: bf16 conversions, W^T and the split-tf32
// parts.  At most a few MB per device; the "no allocation" rule of the ABI is about activations.  One buffer per
// (device, STREAM, use): two operands of one call never alias, reuse along one stream is ordered by that stream, and the
// fused step's side stream (the G step's train forward, which overlaps the D phase's head chain on the caller's stream)
// never shares a buffer with the main stream -- a shared slot would let one stream overwrite, or a growing reallocation
// free, weights that a kernel of the other stream is still reading.  Growing a buffer synchronises its own stream first.
enum WSlot : int { WS_LINEAR = 0, WS_GATE = 1, WS_EMBED = 2, WS_BWD_T = 3, WS_NSLOTS = 4 };
static int weight_scratch(int slot, size_t bytes, cudaStream_t st, void** out) {
  struct Entry { int dev; cudaStream_t st; int slot; void* buf; size_t cap; };
  constexpr int MAX_ENTRIES = 256;
  static Entry tab[MAX_ENTRIES];
  static int n = 0;
  static std::mutex mu;
  int dev = 0;
  ADVMIL_CHECK_CUDA(cudaGetDevice(&dev));
  std::lock_guard<std::mutex> lock(mu);
  Entry* e = nullptr;
  for (int i = 0; i < n; ++i)
    if (tab[i].dev == dev && tab[i].st == st && tab[i].slot == slot) { e = &tab[i]; break; }
  if (!e) {
    ADVMIL_REQUIRE(n < MAX_ENTRIES, "weight_scratch: more than %d (device, stream, use) combinations", MAX_ENTRIES);
    e = &tab[n++];
    *e = Entry{dev, st, slot, nullptr, 0};
  }
  if (bytes > e->cap) {
    ADVMIL_CHECK_CUDA(cudaStreamSynchronize(st));
    if (e->buf) cudaFree(e->buf);
    e->buf = nullptr; e->cap = 0;
    const size_t want = bytes + bytes / 2;                 // headroom: fewer reallocations when shapes vary
    ADVMIL_CHECK_CUDA(cudaMalloc(&e->buf, want));
    e->cap = want;
  }
  *out = e->buf;
  return ADVMIL_OK;
}

// split-tf32 parts of a weight matrix: hi = rna_tf32(W), lo = rna_tf32(W - hi), both [n] fp32 in library scratch
__global__ void split_tf32_kernel(const float* __restrict__ in, size_t n, float* __restrict__ hi, float* __restrict__ lo) {
  pdl_prologue();
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) {
    uint32_t h, l;
    split_tf32(__float_as_uint(in[i]), h, l);
    hi[i] = __uint_as_float(h); lo[i] = __uint_as_float(l);
  }
}
static int weight_split(const float* W, size_t n, int slot, cudaStream_t st, const float** hi, const float** lo) {
  void* p = nullptr;
  ADVMIL_TRY(weight_scratch(slot, 2 * n * sizeof(float), st, &p));
  float* h = (float*)p;
  launch_k(split_tf32_kernel, dim3(cdiv(n, 256)), dim3(256), 0, st, W, n, h, h + n);
  ADVMIL_CHECK_LAUNCH();
  *hi = h; *lo = h + n;
  return ADVMIL_OK;
}

__global__ void to_bf16_kernel(const float* __restrict__ in, size_t n, bf16* __restrict__ out) {
  pdl_prologue();
  size_t i = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) * 4;
  if (i + 3 < n) st4(out + i, *reinterpret_cast<const float4*>(in + i));
  else for (; i < n; ++i) out[i] = __float2bfloat16_rn(in[i]);
}
// operand copy of a weight matrix for element type T: fp32 weights are used in place, bf16 gets a converted copy
template <typename T>
static int weight_operand(const float* W, size_t n, int slot, cudaStream_t st, const T** out);
template <>
int weight_operand<float>(const float* W, size_t, int, cudaStream_t, const float** out) { *out = W; return ADVMIL_OK; }
template <>
int weight_operand<bf16>(const float* W, size_t n, int slot, cudaStream_t st, const bf16** out) {
  void* p = nullptr;
  ADVMIL_TRY(weight_scratch(slot, n * sizeof(bf16), st, &p));
  launch_k(to_bf16_kernel, dim3(cdiv((n + 3) / 4, 256)), dim3(256), 0, st, W, n, (bf16*)p);
  ADVMIL_CHECK_LAUNCH();
  *out = (const bf16*)p;
  return ADVMIL_OK;
}

// TMA zero-fills rows past the end of the tensor, so the engine is correct for any rows >= 1; below one tile the fp32 modes
// prefer the FFMA engine (exact fp32), the bf16 mode has no other engine
static bool rows_ok(int rows, int dt) { return dt == ELEM_BF16 ? rows >= 1 : rows >= TILE_M; }
bool tc_linear_supported(int rows, int K, int N, int dt) { return rows_ok(rows, dt) && K % kblk_of(dt) == 0 && pick_block_n(N) != 0; }

template <typename T, int EPI, bool FAST, bool X3 = false>
static int launch_rows_any(const T* A, const T* W, int rows, int K, int N, const RowEpi& ea, cudaStream_t st, const T* Wlo = nullptr) {
  switch (pick_block_n(N)) {
    case 64: return launch_rows<T, 64, EPI, FAST, X3>(A, W, rows, K, N, ea, st, Wlo);
    case 128: return launch_rows<T, 128, EPI, FAST, X3>(A, W, rows, K, N, ea, st, Wlo);
    case 192: return launch_rows<T, 192, EPI, FAST, X3>(A, W, rows, K, N, ea, st, Wlo);
    case 256: return launch_rows<T, 256, EPI, FAST, X3>(A, W, rows, K, N, ea, st, Wlo);
  }
  set_error("tc: unsupported N=%d", N);
  return ADVMIL_ERR_INVALID;
}

template <typename T>
static int tc_linear_fwd_t(const void* x, const float* W, const float* b, int rows, int K, int N, int relu, const Drop& drop,
                           void* y, void* y2, const Drop* drop2, cudaStream_t st) {
  const T* Wt;
  ADVMIL_TRY(weight_operand<T>(W, (size_t)N * K, WS_LINEAR, st, &Wt));
  RowEpi ea{};
  ea.out = y; ea.ldo = N; ea.bias = b; ea.relu = relu; ea.drop = drop;
  if (y2 && drop2) { ea.out2 = y2; ea.drop2 = *drop2; }
  return launch_rows_any<T, EPI_LINEAR, true>((const T*)x, Wt, rows, K, N, ea, st);
}
int tc_linear_fwd(const void* x, const float* W, const float* b, int rows, int K, int N, int relu, const Drop& drop,
                  void* y, int precision, cudaStream_t st, void* y2, const Drop* drop2) {
  if (precision == ADVMIL_BF16) return tc_linear_fwd_t<bf16>(x, W, b, rows, K, N, relu, drop, y, y2, drop2, st);
  if (precision == ADVMIL_TF32X3) {
    const float *Wh, *Wl;
    ADVMIL_TRY(weight_split(W, (size_t)N * K, WS_LINEAR, st, &Wh, &Wl));
    RowEpi ea{};
    ea.out = y; ea.ldo = N; ea.bias = b; ea.relu = relu; ea.drop = drop;
    if (y2 && drop2) { ea.out2 = y2; ea.drop2 = *drop2; }
    return launch_rows_any<float, EPI_LINEAR, true, true>((const float*)x, Wh, rows, K, N, ea, st, Wl);
  }
  return tc_linear_fwd_t<float>(x, W, b, rows, K, N, relu, drop, y, y2, drop2, st);
}

// K1 + K5/K6 in one pass over x (bf16 mode): stacked weights [W1; Wc] -> 256-wide tiles, the widest the single-CTA pipeline
// can feed (profiles/exp_tile_width.py: 1.2 PFLOP/s vs 1.05 at 192), and x leaves HBM once instead of twice
bool tc_proj_embed_supported(int rows, int C, int h, int d, int dt) {
  return dt == ELEM_BF16 && rows >= 1 && C % TcElem<bf16>::KBLK == 0 && d == 128 && h % 128 == 0 && (h + d) % 256 == 0;
}
int tc_proj_embed_fwd(const void* x, const float* W1, const float* b1, const float* Wc, const float* bc, const float* gamma,
                      const float* beta, int rows, int C, int h, int d, float eps, void* hout, void* hdrop, const Drop* drop2,
                      void* y_pre, float* emb, cudaStream_t st) {
  void* wp = nullptr;
  ADVMIL_TRY(weight_scratch(WS_LINEAR, (size_t)(h + d) * C * sizeof(bf16), st, &wp));
  bf16* Wt = (bf16*)wp;
  launch_k(to_bf16_kernel, dim3(cdiv(((size_t)h * C + 3) / 4, 256)), dim3(256), 0, st, W1, (size_t)h * C, Wt);
  ADVMIL_CHECK_LAUNCH();
  launch_k(to_bf16_kernel, dim3(cdiv(((size_t)d * C + 3) / 4, 256)), dim3(256), 0, st, Wc, (size_t)d * C, Wt + (size_t)h * C);
  ADVMIL_CHECK_LAUNCH();
  RowEpi ea{};
  ea.out = hout; ea.ldo = h; ea.bias = b1; ea.relu = 1;
  if (hdrop && drop2) { ea.out2 = hdrop; ea.drop2 = *drop2; }
  ea.h_cols = h; ea.bias2 = bc; ea.gamma = gamma; ea.beta = beta; ea.eps = eps; ea.y_pre = y_pre; ea.emb = emb;
  return launch_rows<bf16, 256, EPI_PE, true>((const bf16*)x, Wt, rows, C, h + d, ea, st);
}

// K9: relu(x W^T + b) reduced per (bag, cluster id) in the epilogue; part = [(rows / 128 + bags + 1) * ncl][N] column sums
bool tc_proj_pool_supported(int rows, int C, int N, int dt) { return rows_ok(rows, dt) && C % kblk_of(dt) == 0 && pick_block_n(N) != 0; }
template <typename T, bool X3>
static int tc_proj_pool_t(const void* x, const T* W, const T* Wlo, const float* b, const int32_t* cid, const int32_t* offsets,
                          int bags, int rows, int C, int N, int ncl, uint32_t* keep, float* part, cudaStream_t st) {
  RowEpi ea{};
  ea.out = keep; ea.ldo = N / 32; ea.bias = b; ea.part = part; ea.D = ncl; ea.relu_src = cid; ea.offsets = offsets; ea.bags = bags;
  int bn = pick_block_n(N);
  if (X3 && bn == 256) bn = 128;      // split tf32 doubles a stage: 256 columns leave room for one stage only
  switch (bn) {
    case 64: return launch_rows<T, 64, EPI_POOL, true, X3>((const T*)x, W, rows, C, N, ea, st, Wlo);
    case 128: return launch_rows<T, 128, EPI_POOL, true, X3>((const T*)x, W, rows, C, N, ea, st, Wlo);
    case 192: return launch_rows<T, 192, EPI_POOL, true, X3>((const T*)x, W, rows, C, N, ea, st, Wlo);
    case 256: if constexpr (!X3) return launch_rows<T, 256, EPI_POOL, true, X3>((const T*)x, W, rows, C, N, ea, st, Wlo);
  }
  set_error("tc: unsupported N=%d", N);
  return ADVMIL_ERR_INVALID;
}
int tc_proj_pool_fwd(const void* x, const float* W, const float* b, const int32_t* cid, const int32_t* offsets, int bags, int rows,
                     int C, int N, int ncl, uint32_t* keep, float* part, int precision, cudaStream_t st) {
  if (precision == ADVMIL_BF16) {
    const bf16* Wt;
    ADVMIL_TRY(weight_operand<bf16>(W, (size_t)N * C, WS_LINEAR, st, &Wt));
    return tc_proj_pool_t<bf16, false>(x, Wt, nullptr, b, cid, offsets, bags, rows, C, N, ncl, keep, part, st);
  }
  if (precision == ADVMIL_TF32X3) {
    const float *Wh, *Wl;
    ADVMIL_TRY(weight_split(W, (size_t)N * C, WS_LINEAR, st, &Wh, &Wl));
    return tc_proj_pool_t<float, true>(x, Wh, Wl, b, cid, offsets, bags, rows, C, N, ncl, keep, part, st);
  }
  return tc_proj_pool_t<float, false>(x, W, nullptr, b, cid, offsets, bags, rows, C, N, ncl, keep, part, st);
}

bool tc_gate_supported(int rows, int L, int D, int dt) { return rows_ok(rows, dt) && L % kblk_of(dt) == 0 && D % 128 == 0; }

template <typename T, bool FAST>
static int tc_gate_t(const void* v, const float* Wp, const float* bp, const float* wc, int rows, int L, int D,
                     const Drop& da, const Drop& db, void* ab, float* part, cudaStream_t st) {
  const int abw = gate_width(D);
  const T* Wt;
  ADVMIL_TRY(weight_operand<T>(Wp, (size_t)abw * L, WS_GATE, st, &Wt));
  RowEpi ea{};
  ea.bias = bp; ea.ab = ab; ea.ldo = abw; ea.wc = wc; ea.part = part; ea.D = D; ea.drop_a = da; ea.drop_b = db;
  return launch_rows<T, 256, EPI_GATE, FAST>((const T*)v, Wt, rows, L, abw, ea, st);
}
int tc_gated_score_fwd(const void* v, const float* Wp, const float* bp, const float* wc, const float* bc, int rows,
                       int L, int D, const Drop& da, const Drop& db, void* ab, float* s, float* part, int precision,
                       cudaStream_t st) {
  if (precision == ADVMIL_BF16) ADVMIL_TRY((tc_gate_t<bf16, true>(v, Wp, bp, wc, rows, L, D, da, db, ab, part, st)));
  else if (precision == ADVMIL_TF32) ADVMIL_TRY((tc_gate_t<float, true>(v, Wp, bp, wc, rows, L, D, da, db, ab, part, st)));
  else {      // split tf32: exact tanh / sigmoid in the epilogue as well
    const int abw = gate_width(D);
    const float *Wh, *Wl;
    ADVMIL_TRY(weight_split(Wp, (size_t)abw * L, WS_GATE, st, &Wh, &Wl));
    RowEpi ea{};
    ea.bias = bp; ea.ab = ab; ea.ldo = abw; ea.wc = wc; ea.part = part; ea.D = D; ea.drop_a = da; ea.drop_b = db;
    ADVMIL_TRY((launch_rows<float, 256, EPI_GATE, false, true>((const float*)v, Wh, rows, L, abw, ea, st, Wl)));
  }
  if (s == nullptr) return ADVMIL_OK;      // the pooling kernel assembles the logits from the partials
  return gate_score_finish(part, gate_width(D) / 128, rows, bc, s, st);
}

// d = 64 / 128 / 256: one tile holds the whole row that LayerNorm needs (a 256-column split-tf32 tile has room for two
// stages: see RowCfg)
bool tc_embed_supported(int rows, int C, int d, int dt) {
  return rows_ok(rows, dt) && C % kblk_of(dt) == 0 && (d == 64 || d == 128 || d == 256);
}
template <typename T, bool X3 = false, bool CONV = false>
static int launch_embed(const T* x, const T* W, int rows, int K, int d, const RowEpi& ea, cudaStream_t st, const T* Wlo = nullptr) {
  switch (d) {
    case 64: return launch_rows<T, 64, EPI_LN, true, X3, CONV>(x, W, rows, K, d, ea, st, Wlo);
    case 128: return launch_rows<T, 128, EPI_LN, true, X3, CONV>(x, W, rows, K, d, ea, st, Wlo);
    case 256: return launch_rows<T, 256, EPI_LN, true, X3, CONV>(x, W, rows, K, d, ea, st, Wlo);
  }
  set_error("tc: region embedding width d=%d unsupported (64, 128 or 256)", d);
  return ADVMIL_ERR_INVALID;
}

template <typename T>
static int tc_embed_t(const void* x, const float* Wc, const float* bc, const float* gamma, const float* beta, int rows, int C,
                      int d, float eps, void* y_pre, float* emb, cudaStream_t st) {
  const T* Wt;
  ADVMIL_TRY(weight_operand<T>(Wc, (size_t)d * C, WS_EMBED, st, &Wt));
  RowEpi ea{};
  ea.bias = bc; ea.y_pre = y_pre; ea.emb = emb; ea.gamma = gamma; ea.beta = beta; ea.eps = eps;
  return launch_embed<T>((const T*)x, Wt, rows, C, d, ea, st);
}
int tc_region_embed_fwd(const void* x, const float* Wc, const float* bc, const float* gamma, const float* beta,
                        int rows, int C, int d, float eps, void* y_pre, float* emb, int precision, cudaStream_t st) {
  if (precision == ADVMIL_BF16) return tc_embed_t<bf16>(x, Wc, bc, gamma, beta, rows, C, d, eps, y_pre, emb, st);
  if (precision == ADVMIL_TF32X3) {
    const float *Wh, *Wl;
    ADVMIL_TRY(weight_split(Wc, (size_t)d * C, WS_EMBED, st, &Wh, &Wl));
    RowEpi ea{};
    ea.bias = bc; ea.y_pre = y_pre; ea.emb = emb; ea.gamma = gamma; ea.beta = beta; ea.eps = eps;
    return launch_embed<float, true>((const float*)x, Wh, rows, C, d, ea, st, Wl);
  }
  return tc_embed_t<float>(x, Wc, bc, gamma, beta, rows, C, d, eps, y_pre, emb, st);
}

// tap-major K-major operand of a 3x3 weight W [N, C, 3, 3]: out[o, tap * C + c] = W[o, c, kh, kw], tap = 3 kh + kw;
// out_lo != nullptr (fp32 only): split-tf32 parts, hi to `out`, lo to `out_lo`
template <typename T>
__global__ void conv3_pack_kernel(const float* __restrict__ W, int N, int C, T* __restrict__ out, T* __restrict__ out_lo) {
  pdl_prologue();
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (size_t)N * 9 * C) return;
  const int o = (int)(i / (9 * (size_t)C)), r = (int)(i - (size_t)o * 9 * C), tap = r / C, c = r - tap * C;
  const float v = W[((size_t)o * C + c) * 9 + tap];
  if constexpr (sizeof(T) == 4) {
    if (out_lo) {
      uint32_t h, l;
      split_tf32(__float_as_uint(v), h, l);
      out[i] = __uint_as_float(h); out_lo[i] = __uint_as_float(l);
      return;
    }
  }
  st1(out + i, v);
}
template <typename T>
static int conv3_operand(const float* W, int N, int C, bool split, cudaStream_t st, const T** hi, const T** lo) {
  const size_t n = (size_t)N * 9 * C;
  void* p = nullptr;
  ADVMIL_TRY(weight_scratch(WS_EMBED, n * sizeof(T) * (split ? 2 : 1), st, &p));
  T* h = (T*)p;
  T* l = split ? h + n : nullptr;
  launch_k(conv3_pack_kernel<T>, dim3(cdiv(n, 256)), dim3(256), 0, st, W, N, C, h, l);
  ADVMIL_CHECK_LAUNCH();
  *hi = h;
  if (lo) *lo = l;
  return ADVMIL_OK;
}
int conv3_weight_f32(const float* W, int N, int C, cudaStream_t st, const float** out) {
  return conv3_operand<float>(W, N, C, false, st, out, nullptr);
}

template <typename T, bool X3 = false>
static int tc_conv3_embed_t(const void* x, const float* Wc, const float* bc, const float* gamma, const float* beta, int rows,
                            int C, int d, float eps, void* y_pre, float* emb, cudaStream_t st) {
  const T *Wt, *Wl;
  ADVMIL_TRY(conv3_operand<T>(Wc, d, C, X3, st, &Wt, &Wl));
  RowEpi ea{};
  ea.bias = bc; ea.y_pre = y_pre; ea.emb = emb; ea.gamma = gamma; ea.beta = beta; ea.eps = eps;
  return launch_embed<T, X3, true>((const T*)x, Wt, rows, 9 * C, d, ea, st, Wl);
}
int tc_conv3_embed_fwd(const void* x, const float* Wc, const float* bc, const float* gamma, const float* beta,
                       int rows, int C, int d, float eps, void* y_pre, float* emb, int precision, cudaStream_t st) {
  if (precision == ADVMIL_BF16) return tc_conv3_embed_t<bf16>(x, Wc, bc, gamma, beta, rows, C, d, eps, y_pre, emb, st);
  if (precision == ADVMIL_TF32X3) return tc_conv3_embed_t<float, true>(x, Wc, bc, gamma, beta, rows, C, d, eps, y_pre, emb, st);
  return tc_conv3_embed_t<float>(x, Wc, bc, gamma, beta, rows, C, d, eps, y_pre, emb, st);
}

// dX = dY . W with W [Ny, Nx] row-major fp32: the engine needs W^T [Nx, Ny] K-major in the operand type; the transpose
// of the (small) weight goes to library scratch
// out_lo != nullptr (fp32 only): split-tf32 parts of the scaled transpose -- hi to `out`, lo to `out_lo`
template <typename T>
__global__ void transpose_kernel(const float* __restrict__ in, int R, int Cc, T* __restrict__ out, float scale, T* __restrict__ out_lo = nullptr) {
  pdl_prologue();
  __shared__ float t[32][33];
  int x = blockIdx.x * 32 + threadIdx.x, y0 = blockIdx.y * 32;
  for (int j = threadIdx.y; j < 32; j += 8)
    if (x < Cc && y0 + j < R) t[j][threadIdx.x] = in[(size_t)(y0 + j) * Cc + x];
  __syncthreads();
  int ox = blockIdx.y * 32 + threadIdx.x, oy0 = blockIdx.x * 32;
  for (int j = threadIdx.y; j < 32; j += 8)
    if (ox < R && oy0 + j < Cc) {
      const float v = t[threadIdx.x][j] * scale;
      if constexpr (sizeof(T) == 4) {
        if (out_lo) {
          uint32_t h, l;
          split_tf32(__float_as_uint(v), h, l);
          out[(size_t)(oy0 + j) * R + ox] = __uint_as_float(h); out_lo[(size_t)(oy0 + j) * R + ox] = __uint_as_float(l);
          continue;
        }
      }
      st1(out + (size_t)(oy0 + j) * R + ox, v);
    }
}

bool tc_bwd_data_supported(int rows, int Ny, int Nx, int dt) {
  return rows_ok(rows, dt) && Ny % kblk_of(dt) == 0 && pick_block_n(Nx) != 0 && (size_t)Ny * Nx <= (size_t)1 << 20;
}

template <typename T, bool X3 = false>
static int tc_bwd_data_t(const void* dY, const float* W, int rows, int Ny, int Nx, void* dX, const BwdDataExtras& ex,
                         cudaStream_t st) {
  void* wt = nullptr;
  const size_t nW = (size_t)Ny * Nx;
  ADVMIL_TRY(weight_scratch(WS_BWD_T, nW * sizeof(T) * (X3 ? 2 : 1), st, &wt));
  T* wlo = X3 ? (T*)wt + nW : nullptr;
  // the ReLU/dropout mask's 1 / keep is folded into the transposed operand (and into the per-row pooling weights)
  launch_k(transpose_kernel<T>, dim3(dim3(cdiv(Nx, 32), cdiv(Ny, 32))), dim3(dim3(32, 8)), 0, st, W, Ny, Nx, (T*)wt,
           ex.relu_src ? ex.inv_keep : 1.0f, wlo);
  ADVMIL_CHECK_LAUNCH();
  RowEpi ea{};
  ea.out = dX; ea.ldo = Nx; ea.w = ex.w; ea.dz = ex.dz; ea.offsets = ex.offsets; ea.bags = ex.bags;
  ea.dmean = ex.dmean; ea.accumulate = ex.accumulate; ea.colpart = ex.colsum_part;
  ea.relu_src = ex.relu_src; ea.ld_src = ex.ld_src; ea.inv_keep = ex.inv_keep;
  return launch_rows_any<T, EPI_BWD, true, X3>((const T*)dY, (const T*)wt, rows, Ny, Nx, ea, st, (const T*)wlo);
}
int tc_bwd_data(const void* dY, const float* W, int rows, int Ny, int Nx, void* dX, const BwdDataExtras& ex,
                int precision, cudaStream_t st) {
  if (precision == ADVMIL_BF16) return tc_bwd_data_t<bf16>(dY, W, rows, Ny, Nx, dX, ex, st);
  if (precision == ADVMIL_TF32X3) return tc_bwd_data_t<float, true>(dY, W, rows, Ny, Nx, dX, ex, st);
  return tc_bwd_data_t<float>(dY, W, rows, Ny, Nx, dX, ex, st);
}

static int wgrad_block_n(int N2) {
  if (N2 % 256 == 0) return 256;
  if (N2 % 128 == 0) return 128;
  if (N2 == 64) return 64;
  return 0;
}
// split tf32 (x3): the tensor core's accumulation truncates, so the error of a partial sum grows with the number of MMAs
// chained into it; a split covers at most X3_WGRAD_ROWS rows (256 chained MMAs), the fp32 split-K reduce does the rest
constexpr int X3_WGRAD_ROWS = 2048;
static int wgrad_splits(int rows, int N1, int N2, bool x3 = false) {
  int bn = wgrad_block_n(N2);
  int tiles = cdiv(N1, TILE_M) * (N2 / bn);
  int s = max(1, sm_count() / tiles);
  int max_by_rows = max(1, rows / 1024);
  s = min(s, max_by_rows);
  if (x3) s = max(s, cdiv(rows, X3_WGRAD_ROWS));
  return s;
}
bool tc_bwd_weight_supported(int rows, int N1, int N2, int dt) {
  return (dt == ELEM_BF16 ? rows >= 1 : rows >= 4096) && N1 % kblk_of(dt) == 0 && N1 >= 64 && wgrad_block_n(N2) != 0;
}
// dW^T = X^T dY is computed instead (and transposed in the split-K reduce) when that turns 128-wide N tiles, which are
// bound by shared-memory operand bandwidth, into 256-wide ones: d[Wa;Wb] (N1 = 768, N2 = 384) -> 128 x 256 tiles
static bool wgrad_swap(int N1, int N2) { return wgrad_block_n(N2) == 128 && N1 % 256 == 0 && N2 % 128 == 0; }
size_t tc_bwd_weight_ws_floats(int rows, int N1, int N2) {
  if (wgrad_block_n(N2) == 0 || N1 < 64) return 0;
  size_t a = (size_t)(wgrad_splits(rows, N1, N2, true) + 1) * N1 * N2;      // sized for the split-tf32 mode's shorter splits
  size_t b = wgrad_swap(N1, N2) ? (size_t)(wgrad_splits(rows, N2, N1, true) + 1) * N1 * N2 : 0;
  return a > b ? a : b;
}

// CONV: X is x [rows, N2 / 9], read through its region view
template <typename T, int BLOCK_N, bool X3 = false, bool CONV = false>
static int launch_wgrad(const T* dY, const T* X, int rows, int N1, int N2, int rows_per_split, int nsplit, float* ws,
                        cudaStream_t st) {
  using Cfg = WgCfg<T, BLOCK_N, X3>;
  CUtensorMap tmA, tmB;
  ADVMIL_TRY(make_tmap<T>(&tmA, dY, rows, N1, Cfg::KR, TcElem<T>::MN_SWZ));
  if constexpr (CONV) ADVMIL_TRY(make_tmap_regions<T>(&tmB, X, rows / 16, N2 / 9, Cfg::KR / 16, TcElem<T>::MN_SWZ));
  else ADVMIL_TRY(make_tmap<T>(&tmB, X, rows, N2, Cfg::KR, TcElem<T>::MN_SWZ));
  auto kern = tc_wgrad_kernel<T, BLOCK_N, X3, CONV>;
  static bool attr_set = false;
  if (!attr_set) {
    ADVMIL_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Cfg::SMEM));
    attr_set = true;
  }
  dim3 grid(cdiv(N1, TILE_M) * (N2 / BLOCK_N), nsplit);
  launch_k(kern, dim3(grid), dim3(256), Cfg::SMEM, st, tmA, tmB, rows, N1, N2, rows_per_split, ws);
  ADVMIL_CHECK_LAUNCH();
  return ADVMIL_OK;
}

template <typename T, bool X3 = false>
static int tc_bwd_weight_t(const void* dY, const void* X, int rows, int N1, int N2, float* dW, int accumulate, float* ws,
                           cudaStream_t st) {
  constexpr int KR = TcElem<T>::KBLK;
  if (wgrad_swap(N1, N2) && N2 % TcElem<T>::KBLK == 0) {
    const int splits = wgrad_splits(rows, N2, N1, X3);
    const int rows_per_split = cdiv(cdiv(rows, splits), KR) * KR;
    const int nsplit = cdiv(rows, rows_per_split);
    ADVMIL_TRY((launch_wgrad<T, 256, X3>((const T*)X, (const T*)dY, rows, N2, N1, rows_per_split, nsplit, ws, st)));
    return splitk_reduce_t(ws, nsplit, N2, N1, dW, accumulate, st);
  }
  const int splits = wgrad_splits(rows, N1, N2, X3);
  const int rows_per_split = cdiv(cdiv(rows, splits), KR) * KR;
  const int nsplit = cdiv(rows, rows_per_split);
  if (wgrad_block_n(N2) == 256) ADVMIL_TRY((launch_wgrad<T, 256, X3>((const T*)dY, (const T*)X, rows, N1, N2, rows_per_split, nsplit, ws, st)));
  else if (wgrad_block_n(N2) == 64) ADVMIL_TRY((launch_wgrad<T, 64, X3>((const T*)dY, (const T*)X, rows, N1, N2, rows_per_split, nsplit, ws, st)));
  else ADVMIL_TRY((launch_wgrad<T, 128, X3>((const T*)dY, (const T*)X, rows, N1, N2, rows_per_split, nsplit, ws, st)));
  return splitk_reduce(ws, nsplit, (size_t)N1 * N2, dW, accumulate, st);
}
int tc_bwd_weight(const void* dY, const void* X, int rows, int N1, int N2, float* dW, int accumulate, float* ws,
                  int precision, cudaStream_t st) {
  if (precision == ADVMIL_BF16) return tc_bwd_weight_t<bf16>(dY, X, rows, N1, N2, dW, accumulate, ws, st);
  if (precision == ADVMIL_TF32X3) return tc_bwd_weight_t<float, true>(dY, X, rows, N1, N2, dW, accumulate, ws, st);
  return tc_bwd_weight_t<float>(dY, X, rows, N1, N2, dW, accumulate, ws, st);
}

// 9 C columns tap-major: a 256- or 128-column tile never straddles two taps because C is a multiple of the tile width
bool tc_conv3_bwd_weight_supported(int rows, int N1, int C, int dt) {
  const int bn = wgrad_block_n(9 * C);
  return tc_bwd_weight_supported(rows, N1, 9 * C, dt) && bn != 0 && C % bn == 0;
}
template <typename T, bool X3 = false>
static int tc_conv3_bwd_weight_t(const void* dY, const void* X, int rows, int N1, int C, float* dW, int accumulate, float* ws,
                                 cudaStream_t st) {
  constexpr int KR = TcElem<T>::KBLK;
  const int N2 = 9 * C;
  const int splits = wgrad_splits(rows, N1, N2, X3);
  const int rows_per_split = cdiv(cdiv(rows, splits), KR) * KR;
  const int nsplit = cdiv(rows, rows_per_split);
  if (wgrad_block_n(N2) == 256) ADVMIL_TRY((launch_wgrad<T, 256, X3, true>((const T*)dY, (const T*)X, rows, N1, N2, rows_per_split, nsplit, ws, st)));
  else ADVMIL_TRY((launch_wgrad<T, 128, X3, true>((const T*)dY, (const T*)X, rows, N1, N2, rows_per_split, nsplit, ws, st)));
  return splitk_reduce_conv3(ws, nsplit, N1, C, dW, accumulate, st);
}
int tc_conv3_bwd_weight(const void* dY, const void* X, int rows, int N1, int C, float* dW, int accumulate, float* ws,
                        int precision, cudaStream_t st) {
  if (precision == ADVMIL_BF16) return tc_conv3_bwd_weight_t<bf16>(dY, X, rows, N1, C, dW, accumulate, ws, st);
  if (precision == ADVMIL_TF32X3) return tc_conv3_bwd_weight_t<float, true>(dY, X, rows, N1, C, dW, accumulate, ws, st);
  return tc_conv3_bwd_weight_t<float>(dY, X, rows, N1, C, dW, accumulate, ws, st);
}

}  // namespace advmil
