// Region-level chain of the RLIP discriminator head in ONE kernel (forward):
//   f1  = dropout(relu(emb F1a^T + b))            EmbedXLayer.fc1.0-2   (reference model/model_utils.py:202-210)
//   fi  = f1 F1b^T + b                            EmbedXLayer.fc1.3     (the "instance embeddings", quirk A.4#2)
//   a,b = tanh(fi Pg^T + b), sigmoid(fi Ps^T + b) GAPool gate           (reference model/backbone_utils.py:47-56)
//   rep = sum_j drop(a_j) drop(b_j) Pc_j                                (bias and softmax: seg_softmax_pool_fwd)
// over R = rows / 16 regions of width d = 64, 128 or 256 (128: 49 152 multiply-adds per region): far too little to fill the
// tensor pipe kernel by kernel (round 1: four launches of 10-25 us, tensor pipe 2-10 %, a quarter of the step for 0.2 % of
// its FLOPs).  One CTA owns 32 or 64 regions and walks the three contractions with the intermediates in shared memory; the
// weights (192 KB, L2-resident) stream through a double-buffered stage.  The chain is fp32-grade in EVERY precision mode (no
// tf32 truncation in the discriminator outputs, whose real/fake cancellation amplifies forward errors in the gradients).
//
// The contractions run on the tensor cores as warp-level mma.sync m16n8k8 tf32 with SPLIT operands ("3xTF32").  Every fp32
// operand is split in registers into hi = rna_tf32(x) and lo = x - hi (exact in fp32; the tensor core reads its top 19
// bits), each K step issues lo.hi + hi.lo into a small-term accumulator and hi.hi into the main one (the tensor core's
// fp32 accumulation truncates, so the small terms are never chained into the large sum), and the epilogue adds the two
// once in round-to-nearest fp32: products are exact to ~2^-21 relative, i.e. fp32-grade, in every precision mode.
// An exact-FFMA kernel tops out at the FFMA rate (128 MAC / clk / SM at ~50 % pipe utilisation); the warp-level tf32 MMA
// does 512 MAC / clk / SM, i.e. 1.33x the FFMA peak after the three-fold split, with a tenth of the issue slots.
// FFMA chain (118 + 58 us against 84 + 46 us on B200): measured, slower, removed.
//
// One CTA = 32 x WM regions with WM x 4 warps as WM (rows) x 4 (columns): a warp owns 32 rows (two 16-row MMA tiles) and a
// quarter of the output columns of the phase.  Activations stay row-major in shared memory (stride K + 4 floats: the
// A-fragment loads of a quarter-warp hit 32 distinct banks), weights stream through a double-buffered [rows n][KC k] stage
// filled with cp.async straight from their [N, K] row-major global layout (stride KC + 4 floats: conflict-free B-fragment
// loads) -- no transposes anywhere.  In the gate phase a warp's four n-tiles are two tanh tiles and the two sigmoid tiles
// of the SAME columns, so that a thread holds both halves of each (tanh_j, sigmoid_j) pair in matching fragment slots.
// Measured (ncu, B200): 84 us for 32768 regions with <WM, KC> = <1, 16> (4 CTAs per SM), 46 us for 16384 regions with <2, 32>
// (2 CTAs per SM); legacy tensor pipe 43-47 % busy, HMMA.1688.F32.TF32 at ~10.6 cycles per instruction and sub-core.
// Other widths: phase 1 has d / 2 columns (d / 64 n-tiles per warp); phase 2 runs its d columns in groups of at most 128
// (4 n-tiles per warp, as at d = 128: the accumulators of a 256-column phase would not fit beside the fragments); the gate
// has d / 64 blocks.  Weight stages hold at most 128 rows at every width.
#include "stages.cuh"

namespace advmil {

namespace {

namespace mm {
constexpr int WROWS = 128;
// D = region width (64, 128 or 256), DH = D / 2.
// WM = warp rows per CTA (a warp owns 32 regions): 64 regions / 256 threads or 32 regions / 128 threads; KC = K extent of a
// weight stage.  Smaller CTAs balance better over the 148 SMs (16384 regions = 110.7 per SM) and decouple the phases of the
// CTAs that share an SM (one CTA's epilogue runs under another's MMAs).
template <int D, int WM, int KC>
struct Cfg {
  static constexpr int DH = D / 2, LDA = D + 4, LDF = DH + 4;
  static constexpr int TM = 32 * WM, THREADS = 128 * WM, LDW = KC + 4;
  static constexpr int W2 = D < 128 ? D : 128, G2 = D / W2;      // phase 2: G2 column groups of W2 columns
  static constexpr int NB = D / 64;                               // gate blocks of 64 (tanh, sigmoid) pairs
  static constexpr int NC1 = D / KC, NC2 = DH / KC, NCHUNK = NC1 + G2 * NC2 + NB * NC1;
  static constexpr size_t SMEM_FLOATS = (size_t)TM * LDA + (size_t)TM * LDF + 2 * (size_t)WROWS * LDW + (size_t)NB * 4 * TM;
  static constexpr int MIN_CTAS = WM == 2 ? 2 : 4;
  static_assert(NC2 >= 1 && DH <= WROWS, "unsupported chain width");
};

__device__ __forceinline__ void split3(float x, uint32_t& hi, uint32_t& lo) {
  hi = (__float_as_uint(x) + 0x1000u) & 0xFFFFE000u;       // cvt.rna.tf32.f32 for finite x
  lo = __float_as_uint(x - __uint_as_float(hi));           // exact; truncated to tf32 by the tensor core
}
__device__ __forceinline__ void mma_tf32(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void cp_async16(float* dst_smem, const float* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(dst_smem)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }

// [NROWS (n)][KC (k)] weight chunk -> stage; rows < 64 from W0, rows >= 64 from W1 (both [.., K] row-major).  Every loop
// bound is a compile-time constant: a thread's pieces are NROWS * KC / 4 / THREADS fixed (row, column) slots.
template <int KC, int THREADS, int NROWS>
__device__ __forceinline__ void load_w_chunk(float* stage, const float* __restrict__ W0, const float* __restrict__ W1, int K, int k0,
                                             int tid) {
  constexpr int PPR = KC / 4, LDW = KC + 4, PIECES = NROWS * PPR;      // 16-byte pieces per row / per chunk
  static_assert(PIECES % THREADS == 0 && THREADS % PPR == 0, "weight chunk must divide evenly over the CTA");
  const int r0 = tid / PPR, c4 = tid % PPR;
#pragma unroll
  for (int k = 0; k < PIECES / THREADS; ++k) {
    const int r = r0 + k * (THREADS / PPR);
    const float* src = (r < 64 ? W0 + (size_t)r * K : W1 + (size_t)(r - 64) * K) + k0 + 4 * c4;
    cp_async16(stage + r * LDW + 4 * c4, src);
  }
}

// one KC-wide chunk of the contraction: accm += hi.hi, accs += lo.hi + hi.lo.  A: activations [row][lda] (this warp's 32
// rows start at Aw), columns k0 .. k0 + KC; Ws: weight stage; nrow[nt]: stage row of n-tile nt's first column.  The two
// MMAs into the same small-term accumulator are issued three MMAs apart.
template <int NT, int KC>
__device__ __forceinline__ void mma_chunk(float (&accm)[2][NT][4], float (&accs)[2][NT][4], const float* __restrict__ Aw, int lda,
                                          int k0, const float* __restrict__ Ws, const int (&nrow)[NT], int g, int t) {
  constexpr int LDW = KC + 4;
#pragma unroll
  for (int ks = 0; ks < KC / 8; ++ks) {
    uint32_t ah[2][4], al[2][4];
#pragma unroll
    for (int mt = 0; mt < 2; ++mt) {
      const float* p = Aw + (size_t)(mt * 16 + g) * lda + k0 + ks * 8 + t;
      split3(p[0], ah[mt][0], al[mt][0]);
      split3(p[8 * lda], ah[mt][1], al[mt][1]);
      split3(p[4], ah[mt][2], al[mt][2]);
      split3(p[8 * lda + 4], ah[mt][3], al[mt][3]);
    }
#pragma unroll
    for (int nt = 0; nt < NT; ++nt) {
      const float* q = Ws + (size_t)(nrow[nt] + g) * LDW + ks * 8 + t;
      uint32_t bh0, bl0, bh1, bl1;
      split3(q[0], bh0, bl0);
      split3(q[4], bh1, bl1);
      mma_tf32(accs[0][nt], al[0], bh0, bh1);
      mma_tf32(accs[1][nt], al[1], bh0, bh1);
      mma_tf32(accm[0][nt], ah[0], bh0, bh1);
      mma_tf32(accm[1][nt], ah[1], bh0, bh1);
      mma_tf32(accs[0][nt], ah[0], bl0, bl1);
      mma_tf32(accs[1][nt], ah[1], bl0, bl1);
    }
  }
}
template <int NT>
__device__ __forceinline__ void zero_acc(float (&a)[2][NT][4], float (&b)[2][NT][4]) {
#pragma unroll
  for (int i = 0; i < 2; ++i)
#pragma unroll
    for (int j = 0; j < NT; ++j)
#pragma unroll
      for (int e = 0; e < 4; ++e) { a[i][j][e] = 0.f; b[i][j][e] = 0.f; }
}

template <int D, int WM, int KC>
__global__ void __launch_bounds__(Cfg<D, WM, KC>::THREADS, Cfg<D, WM, KC>::MIN_CTAS)
rlip_chain_mma_kernel(const float* __restrict__ emb, const float* __restrict__ F1a_w, const float* __restrict__ F1a_b,
                      const float* __restrict__ F1b_w, const float* __restrict__ F1b_b, const float* __restrict__ Pg_w,
                      const float* __restrict__ Pg_b, const float* __restrict__ Ps_w, const float* __restrict__ Ps_b,
                      const float* __restrict__ Pc_w, int R, Drop dfc1, Drop dga, Drop dgs, float* __restrict__ f1,
                      float* __restrict__ fi, float* __restrict__ ab, float* __restrict__ part) {
  pdl_prologue();
  using C = Cfg<D, WM, KC>;
  constexpr int DH = C::DH, ABW = 2 * D, TM = C::TM, THREADS = C::THREADS, LDW = C::LDW, NC1 = C::NC1, NC2 = C::NC2;
  constexpr int LDA = C::LDA, LDF = C::LDF, W2 = C::W2, NT1 = DH / 32, NT2 = W2 / 32;
  extern __shared__ __align__(16) float smem[];
  float* actA = smem;                                   // [TM][LDA]: emb, later fi
  float* f1A = actA + (size_t)TM * LDA;                 // [TM][LDF]
  float* wst = f1A + (size_t)TM * LDF;                  // [2][WROWS][LDW]
  float* red = wst + 2 * (size_t)WROWS * LDW;           // [2 (c)][4 (warp column)][TM]
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, g = lane >> 2, t = lane & 3;
  const int wm = warp % WM, wn = warp / WM;
  const int m0 = blockIdx.x * TM;
  const int rbase = wm * 32;                            // this warp's first row of the tile

  // weight chunk q of the schedule: F1a (NC1 chunks of K = D), F1b (G2 column groups of NC2 chunks, K = DH), then the
  // NB gate blocks (NC1 chunks each)
  auto issue_chunk = [&](int q) {
    float* stage = wst + (size_t)(q & 1) * WROWS * LDW;
    if (q < NC1) load_w_chunk<KC, THREADS, DH>(stage, F1a_w, DH > 64 ? F1a_w + (size_t)64 * D : nullptr, D, q * KC, tid);
    else if (q < NC1 + C::G2 * NC2) {
      const int grp = C::G2 == 1 ? 0 : (q - NC1) / NC2, kq = C::G2 == 1 ? q - NC1 : (q - NC1) % NC2;
      const float* W0 = F1b_w + (size_t)grp * W2 * DH;
      load_w_chunk<KC, THREADS, W2>(stage, W0, W0 + (size_t)64 * DH, DH, kq * KC, tid);
    } else {
      const int c = (q - NC1 - C::G2 * NC2) / NC1, kq = (q - NC1 - C::G2 * NC2) % NC1;
      load_w_chunk<KC, THREADS, 128>(stage, Pg_w + (size_t)c * 64 * D, Ps_w + (size_t)c * 64 * D, D, kq * KC, tid);
    }
    cp_async_commit();
  };
  // chunk q has landed and is visible to every thread; the other stage buffer is free: prefetch chunk q + 1 into it
  auto advance = [&](int q) -> const float* {
    cp_async_wait_all();
    __syncthreads();
    if (q + 1 < C::NCHUNK) issue_chunk(q + 1);
    return wst + (size_t)(q & 1) * WROWS * LDW;
  };

  // ---- emb tile (row-major, zero beyond R) + first weight chunk ----
  for (int i = tid; i < TM * (D / 4); i += THREADS) {
    const int r = i / (D / 4), c4 = i % (D / 4);
    if (m0 + r < R) cp_async16(actA + (size_t)r * LDA + 4 * c4, emb + (size_t)(m0 + r) * D + 4 * c4);
    else *reinterpret_cast<float4*>(actA + (size_t)r * LDA + 4 * c4) = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  issue_chunk(0);

  // ---- phase 1: f1 = dropout(relu(emb F1a^T + b)), DH columns: NT1 n-tiles per warp ----
  {
    float accm[2][NT1][4], accs[2][NT1][4];
    zero_acc<NT1>(accm, accs);
    int nrow[NT1];
#pragma unroll
    for (int nt = 0; nt < NT1; ++nt) nrow[nt] = wn * (DH / 4) + nt * 8;
#pragma unroll 1
    for (int q = 0; q < NC1; ++q) {
      const float* Ws = advance(q);
      mma_chunk<NT1, KC>(accm, accs, actA + (size_t)rbase * LDA, LDA, q * KC, Ws, nrow, g, t);
    }
#pragma unroll
    for (int nt = 0; nt < NT1; ++nt) {
      const int n = nrow[nt] + 2 * t;
      const float2 bv = *reinterpret_cast<const float2*>(F1a_b + n);
#pragma unroll
      for (int mt = 0; mt < 2; ++mt)
#pragma unroll
        for (int hh = 0; hh < 2; ++hh) {
          const int row = rbase + mt * 16 + g + 8 * hh, m = m0 + row;
          float v0 = fmaxf(accm[mt][nt][2 * hh] + accs[mt][nt][2 * hh] + bv.x, 0.f);
          float v1 = fmaxf(accm[mt][nt][2 * hh + 1] + accs[mt][nt][2 * hh + 1] + bv.y, 0.f);
          if (dfc1.active) {
            bool k0 = true, k1 = true;
            if (m < R) dfc1.keep2(m, n, k0, k1);
            v0 = k0 ? v0 * dfc1.inv_keep : 0.f;
            v1 = k1 ? v1 * dfc1.inv_keep : 0.f;
          }
          if (m < R) *reinterpret_cast<float2*>(f1 + (size_t)m * DH + n) = make_float2(v0, v1);
          *reinterpret_cast<float2*>(f1A + (size_t)row * LDF + n) = make_float2(v0, v1);
        }
    }
  }

  // ---- phase 2: fi = f1 F1b^T + b, D columns in G2 groups of W2: NT2 n-tiles per warp; fi replaces emb in shared memory.
  //      With 4 n-tiles per warp the accumulators are those of phase 3 ----
  float accm[2][4][4], accs[2][4][4];
  float am1[2][NT2 == 4 ? 1 : NT2][4], as1[2][NT2 == 4 ? 1 : NT2][4];
  auto& am = *reinterpret_cast<float (*)[2][NT2][4]>(NT2 == 4 ? (void*)accm : (void*)am1);
  auto& as = *reinterpret_cast<float (*)[2][NT2][4]>(NT2 == 4 ? (void*)accs : (void*)as1);
#pragma unroll 1
  for (int grp = 0; grp < C::G2; ++grp) {
    zero_acc<NT2>(am, as);
    int nrow[NT2];
#pragma unroll
    for (int nt = 0; nt < NT2; ++nt) nrow[nt] = wn * (W2 / 4) + nt * 8;
    const int q0 = NC1 + grp * NC2;
#pragma unroll 1
    for (int q = q0; q < q0 + NC2; ++q) {
      const float* Ws = advance(q);
      mma_chunk<NT2, KC>(am, as, f1A + (size_t)rbase * LDF, LDF, (q - q0) * KC, Ws, nrow, g, t);
    }
    // every warp has finished reading emb (phase 1) before any thread got past the barriers of this phase
#pragma unroll
    for (int nt = 0; nt < NT2; ++nt) {
      const int n = grp * W2 + nrow[nt] + 2 * t;
      const float2 bv = *reinterpret_cast<const float2*>(F1b_b + n);
#pragma unroll
      for (int mt = 0; mt < 2; ++mt)
#pragma unroll
        for (int hh = 0; hh < 2; ++hh) {
          const int row = rbase + mt * 16 + g + 8 * hh, m = m0 + row;
          const float v0 = am[mt][nt][2 * hh] + as[mt][nt][2 * hh] + bv.x;
          const float v1 = am[mt][nt][2 * hh + 1] + as[mt][nt][2 * hh + 1] + bv.y;
          if (m < R) *reinterpret_cast<float2*>(fi + (size_t)m * D + n) = make_float2(v0, v1);
          *reinterpret_cast<float2*>(actA + (size_t)row * LDA + n) = make_float2(v0, v1);
        }
    }
  }

  // ---- phase 3: the gate, 64 (tanh_j, sigmoid_j) pairs per block; n-tiles 0,1 = tanh columns, 2,3 = the sigmoid columns of
  //      the same pairs.  Conventions as in EpiGate (gemm_simt.cuh) ----
  const bool hashed = dga.active && !dga.mask && !dgs.mask;
#pragma unroll 1
  for (int c = 0; c < D / 64; ++c) {
    zero_acc<4>(accm, accs);
    const int nrow[4] = {wn * 16, wn * 16 + 8, 64 + wn * 16, 64 + wn * 16 + 8};
    const int q0 = NC1 + C::G2 * NC2 + c * NC1;
#pragma unroll 1
    for (int q = q0; q < q0 + NC1; ++q) {
      const float* Ws = advance(q);
      mma_chunk<4, KC>(accm, accs, actA + (size_t)rbase * LDA, LDA, (q - q0) * KC, Ws, nrow, g, t);
    }
    float partial[2][2] = {{0.f, 0.f}, {0.f, 0.f}};
#pragma unroll
    for (int nt = 0; nt < 2; ++nt) {
      const int jl = wn * 16 + nt * 8 + 2 * t, j0 = c * 64 + jl;      // pair index inside the block / logical gate column (even)
      const float2 ba = *reinterpret_cast<const float2*>(Pg_b + j0), bb = *reinterpret_cast<const float2*>(Ps_b + j0);
      const float2 wc = *reinterpret_cast<const float2*>(Pc_w + j0);
#pragma unroll
      for (int mt = 0; mt < 2; ++mt)
#pragma unroll
        for (int hh = 0; hh < 2; ++hh) {
          const int row = rbase + mt * 16 + g + 8 * hh, m = m0 + row;
          uint32_t h = 0;
          if (hashed) h = dga.bits(m, (uint32_t)j0 & ~3u);
          float av[2], bv[2];
#pragma unroll
          for (int e = 0; e < 2; ++e) {
            const float a = tanhf(accm[mt][nt][2 * hh + e] + accs[mt][nt][2 * hh + e] + (e ? ba.y : ba.x));
            const float b = sigmoidf_(accm[mt][nt + 2][2 * hh + e] + accs[mt][nt + 2][2 * hh + e] + (e ? bb.y : bb.x));
            av[e] = a; bv[e] = b;
            float ad = a, bd = b;
            if (dga.active && m < R) {
              bool ka, kb;
              if (hashed) { ka = ((h >> (8 * ((j0 + e) & 3))) & 0xFFu) >= dga.thresh8j; kb = true; }
              else gate_keep(dga, dgs, m, j0 + e, ka, kb);
              ad = ka ? a * dga.inv_keep : 0.f;
              bd = kb ? b * dgs.inv_keep : 0.f;
              if (!(ka && kb)) bv[e] = -b;          // joint keep bit in the sign of the stored sigmoid
            }
            partial[mt][hh] = fmaf(ad * bd, e ? wc.y : wc.x, partial[mt][hh]);
          }
          if (ab && m < R) {
            *reinterpret_cast<float2*>(ab + (size_t)m * ABW + c * 128 + jl) = make_float2(av[0], av[1]);
            *reinterpret_cast<float2*>(ab + (size_t)m * ABW + c * 128 + 64 + jl) = make_float2(bv[0], bv[1]);
          }
        }
    }
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
      for (int hh = 0; hh < 2; ++hh) {
        float p = partial[mt][hh];
        p += __shfl_xor_sync(0xffffffffu, p, 1);
        p += __shfl_xor_sync(0xffffffffu, p, 2);
        if (t == 0) red[(size_t)(c * 4 + wn) * TM + rbase + mt * 16 + g + 8 * hh] = p;
      }
  }
  __syncthreads();
  static_assert(C::NB * TM <= THREADS, "one thread per (gate block, region)");
  if (tid < C::NB * TM) {
    const int c = tid / TM, row = tid % TM, m = m0 + row;
    const float* rp = red + (size_t)c * 4 * TM + row;
    if (m < R) part[(size_t)c * R + m] = (rp[0] + rp[TM]) + (rp[2 * TM] + rp[3 * TM]);
  }
}

template <int D, int WM, int KC>
static int launch_chain_mma(const float* emb, const AdvmilDiscParams& p, int R, const Drop& dfc1, const Drop& dga, const Drop& dgs,
                            float* f1, float* fi, float* ab, float* part, cudaStream_t st) {
  using C = Cfg<D, WM, KC>;
  const size_t smem = C::SMEM_FLOATS * sizeof(float);
  static bool attr_set[64] = {};
  int dev = 0;
  ADVMIL_CHECK_CUDA(cudaGetDevice(&dev));
  if (dev < 0 || dev >= 64 || !attr_set[dev]) {
    ADVMIL_CHECK_CUDA(cudaFuncSetAttribute(rlip_chain_mma_kernel<D, WM, KC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    if (dev >= 0 && dev < 64) attr_set[dev] = true;
  }
  launch_k(rlip_chain_mma_kernel<D, WM, KC>, dim3(cdiv(R, C::TM)), dim3(C::THREADS), smem, st, emb, p.F1a_w, p.F1a_b, p.F1b_w, p.F1b_b,
           p.Pg_w, p.Pg_b, p.Ps_w, p.Ps_b, p.Pc_w, R, dfc1, dga, dgs, f1, fi, ab, part);
  ADVMIL_CHECK_LAUNCH();
  return ADVMIL_OK;
}
}  // namespace mm

}  // namespace

bool rlip_chain_supported(int d) { return d == 64 || d == 128 || d == 256; }

int rlip_chain_fwd(const float* emb, const AdvmilDiscParams& p, int R, const Drop& dfc1, const Drop& dga, const Drop& dgs,
                   float* f1, float* fi, float* ab, float* part, cudaStream_t st) {
  ADVMIL_REQUIRE(rlip_chain_supported(p.d), "rlip_chain_fwd: d=%d unsupported (64, 128 or 256)", p.d);
  if (R == 0) return ADVMIL_OK;
  // 64-region CTAs while they fit one wave of 2 CTAs per SM (R = 16384: 46 us against 49 us), 32-region CTAs with 16-deep
  // weight stages (4 CTAs per SM) beyond that (the batched real + fake launch, 2R = 32768: 86 us against 91 us)
  static int sms = 0;
  if (!sms) { int dev = 0; cudaGetDevice(&dev); cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev); if (sms <= 0) sms = 148; }
  // d = 64: the same choice with 32-deep stages (a 16-deep stage of the 32-row F1a chunk does not divide over 256 threads);
  // d = 256: 32-region CTAs only (a 64-region CTA needs 138 KB of shared memory: one per SM)
  if (p.d == 64) {
    if (cdiv(R, 64) <= 2 * sms) return mm::launch_chain_mma<64, 2, 32>(emb, p, R, dfc1, dga, dgs, f1, fi, ab, part, st);
    return mm::launch_chain_mma<64, 1, 32>(emb, p, R, dfc1, dga, dgs, f1, fi, ab, part, st);
  }
  if (p.d == 256) return mm::launch_chain_mma<256, 1, 16>(emb, p, R, dfc1, dga, dgs, f1, fi, ab, part, st);
  if (cdiv(R, 64) <= 2 * sms) return mm::launch_chain_mma<128, 2, 32>(emb, p, R, dfc1, dga, dgs, f1, fi, ab, part, st);
  return mm::launch_chain_mma<128, 1, 16>(emb, p, R, dfc1, dga, dgs, f1, fi, ab, part, st);
}

}  // namespace advmil
