// Launchers for the N-row contractions.  precision == ADVMIL_FP32 runs the FFMA tile engine (gemm_simt.cuh);
// ADVMIL_TF32 / ADVMIL_TF32X3 run the tcgen05 engine (gemm_tc.cu) for the shapes it supports and fall through to
// the FFMA engine for the small region-level shapes, where the tensor pipe cannot be filled anyway.
#include "gemm_simt.cuh"
#include "stages.cuh"
#include "gemm_tc.cuh"

namespace advmil {

static bool gemm_ok(int K, int N, const void* a, const void* b) {
  return (K % 4 == 0) && (N % 4 == 0) && (((uintptr_t)a | (uintptr_t)b) % 16 == 0);
}

static const char* kBf16Shape = "%s: the bf16 mode runs only on the tcgen05 engine and this shape is unsupported by it (rows=%d K=%d N=%d)";

int linear_fwd(const void* x, const float* W, const float* b, int rows, int K, int N, int relu, const Drop& drop,
               void* y, int precision, cudaStream_t st, void* y2, const Drop* drop2) {
  ADVMIL_REQUIRE(gemm_ok(K, N, x, W), "linear_fwd: K=%d N=%d must be multiples of 4 and pointers 16B aligned", K, N);
  if (rows == 0) return ADVMIL_OK;
  if (precision != ADVMIL_FP32 && tc_linear_supported(rows, K, N, elem_of_precision(precision)))
    return tc_linear_fwd(x, W, b, rows, K, N, relu, drop, y, precision, st, y2, drop2);
  ADVMIL_REQUIRE(precision != ADVMIL_BF16, kBf16Shape, "linear_fwd", rows, K, N);
  GemmArgs g{(const float*)x, W, rows, N, K, K, K, K};
  EpiLinear epi{(float*)y, N, b, relu, drop, N};
  ADVMIL_TRY((launch_gemm<true, true>(g, epi, 1, st)));
  if (y2 && drop2) return apply_dropout(y, rows, N, *drop2, y2, ELEM_F32, st);
  return ADVMIL_OK;
}

bool proj_embed_supported(int rows, int C, int h, int d, int precision) {
  return precision == ADVMIL_BF16 && rows % 16 == 0 && tc_proj_embed_supported(rows, C, h, d, ELEM_BF16);
}
int proj_embed_fwd(const void* x, const float* W1, const float* b1, const float* Wc, const float* bc, const float* gamma,
                   const float* beta, int rows, int C, int h, int d, float eps, void* hout, void* hdrop, const Drop* drop2,
                   void* y_pre, float* emb, cudaStream_t st) {
  ADVMIL_REQUIRE(tc_proj_embed_supported(rows, C, h, d, ELEM_BF16) && rows % 16 == 0, "proj_embed_fwd: unsupported shape rows=%d C=%d h=%d d=%d", rows, C, h, d);
  return tc_proj_embed_fwd(x, W1, b1, Wc, bc, gamma, beta, rows, C, h, d, eps, hout, hdrop, drop2, y_pre, emb, st);
}

int gated_score_fwd(const void* v, const float* Wp, const float* bp, const float* wc, const float* bc, int rows, int L,
                    int D, const Drop& da, const Drop& db, void* ab, float* s, float* part_ws, int precision,
                    cudaStream_t st) {
  ADVMIL_REQUIRE(L % 4 == 0, "gated_score_fwd: L=%d must be a multiple of 4", L);
  if (rows == 0) return ADVMIL_OK;
  int abw = gate_width(D);
  if (precision != ADVMIL_FP32 && tc_gate_supported(rows, L, D, elem_of_precision(precision)))
    return tc_gated_score_fwd(v, Wp, bp, wc, bc, rows, L, D, da, db, ab, s, part_ws, precision, st);
  ADVMIL_REQUIRE(precision != ADVMIL_BF16, kBf16Shape, "gated_score_fwd", rows, L, D);
  GemmArgs g{(const float*)v, Wp, rows, abw, L, L, L, L};
  EpiGate epi{(float*)ab, abw, bp, wc, part_ws, D, da, db};
  ADVMIL_TRY((launch_gemm<true, true>(g, epi, 1, st)));
  if (s == nullptr) return ADVMIL_OK;
  return gate_score_finish(part_ws, abw / 128, rows, bc, s, st);
}

int region_embed_fwd(const void* x, const float* Wc, const float* bc, const float* gamma, const float* beta, int rows,
                     int C, int d, float eps, void* y_pre, float* emb, int precision, cudaStream_t st, int ksize, float* y_ws) {
  ADVMIL_REQUIRE(rows % 16 == 0, "region_embed: rows %d not a multiple of 16 (backbone_utils.py:65)", rows);
  ADVMIL_REQUIRE(((d <= 128 && d % 4 == 0) || d == 256) && C % 4 == 0, "region_embed: d=%d (<=128 and %%4, or 256) C=%d (%%4) unsupported", d, C);
  ADVMIL_REQUIRE(ksize == 1 || C % 16 == 0, "region_embed: the 3x3 embedding needs C %% 16 == 0 (C=%d)", C);
  // rejected here rather than in the backward: bf16 runs only on tcgen05, and the 3x3 weight gradient tiles its 9 C columns
  // by 128 or 256 without straddling a tap
  ADVMIL_REQUIRE(ksize == 1 || precision != ADVMIL_BF16 || C % 128 == 0,
                 "region_embed: the bf16 3x3 embedding needs C %% 128 == 0 (C=%d)", C);
  if (rows == 0) return ADVMIL_OK;
  if (precision != ADVMIL_FP32 && tc_embed_supported(rows, C, d, elem_of_precision(precision)))
    return ksize == 3 ? tc_conv3_embed_fwd(x, Wc, bc, gamma, beta, rows, C, d, eps, y_pre, emb, precision, st)
                      : tc_region_embed_fwd(x, Wc, bc, gamma, beta, rows, C, d, eps, y_pre, emb, precision, st);
  ADVMIL_REQUIRE(precision != ADVMIL_BF16, kBf16Shape, "region_embed_fwd", rows, C, d);
  if (d > 128) {
    // EpiLNPool needs the whole row in one 128-column tile: y = x Wc^T + bc first, then LayerNorm + ReLU + region mean
    // per row (the same two passes as the ESAT patch embedding)
    float* y = y_pre ? (float*)y_pre : y_ws;
    ADVMIL_REQUIRE(y, "region_embed: the fp32 embedding at d=%d needs y_pre or %d x %d floats of workspace", d, rows, d);
    EpiLinear lin{y, d, bc, 0, Drop::make(nullptr, 0, 0, 0.f, 0, 0), d};
    if (ksize == 3) {
      const float* Wk;
      ADVMIL_TRY(conv3_weight_f32(Wc, d, C, st, &Wk));
      GemmArgs g{(const float*)x, Wk, rows, d, 9 * C, C, 9 * C, 9 * C};
      ADVMIL_TRY((launch_gemm<true, true, EpiLinear, Conv3LoaderA>(g, lin, 1, st)));
    } else {
      GemmArgs g{(const float*)x, Wc, rows, d, C, C, C, C};
      ADVMIL_TRY((launch_gemm<true, true>(g, lin, 1, st)));
    }
    return ln_relu_mean16_fwd(y, gamma, beta, rows, d, eps, nullptr, emb, ELEM_F32, st);
  }
  EpiLNPool epi{(float*)y_pre, emb, bc, gamma, beta, d, eps};
  if (ksize == 3) {
    const float* Wk;
    ADVMIL_TRY(conv3_weight_f32(Wc, d, C, st, &Wk));
    GemmArgs g{(const float*)x, Wk, rows, d, 9 * C, C, 9 * C, 9 * C};
    return launch_gemm<true, true, EpiLNPool, Conv3LoaderA>(g, epi, 1, st);
  }
  GemmArgs g{(const float*)x, Wc, rows, d, C, C, C, C};
  return launch_gemm<true, true>(g, epi, 1, st);
}

bool bwd_data_fuses_colsum(int rows, int Ny, int Nx, int precision) {
  return rows > 0 && precision != ADVMIL_FP32 && tc_bwd_data_supported(rows, Ny, Nx, elem_of_precision(precision));
}

int bwd_data(const void* dY, const float* W, int rows, int Ny, int Nx, void* dX, const BwdDataExtras& ex,
             int precision, cudaStream_t st) {
  ADVMIL_REQUIRE(gemm_ok(Ny, Nx, dY, W), "bwd_data: Ny=%d Nx=%d must be multiples of 4", Ny, Nx);
  if (rows == 0) return ADVMIL_OK;
  if (precision != ADVMIL_FP32 && tc_bwd_data_supported(rows, Ny, Nx, elem_of_precision(precision)))
    return tc_bwd_data(dY, W, rows, Ny, Nx, dX, ex, precision, st);
  ADVMIL_REQUIRE(precision != ADVMIL_BF16, kBf16Shape, "bwd_data", rows, Ny, Nx);
  GemmArgs g{(const float*)dY, W, rows, Nx, Ny, Ny, Nx, Ny};
  EpiBwdData epi{(float*)dX, Nx, ex.w, ex.dz, ex.dmean, ex.offsets, ex.bags, (const float*)ex.relu_src, ex.ld_src, ex.inv_keep, ex.accumulate};
  return launch_gemm<true, false>(g, epi, 1, st);
}

static int pick_splits(int rows, int N1, int N2) {
  int tiles = cdiv(N1, BM) * cdiv(N2, BN);
  int want = cdiv(148 * 4, tiles);                  // ~4 CTAs per SM
  int max_by_k = max(1, rows / 256);                // at least 256 rows per split
  int s = min(want, max_by_k);
  return max(1, min(s, 256));
}
size_t bwd_weight_ws_floats(int rows, int N1, int N2) {
  size_t simt = (size_t)pick_splits(rows, N1, N2) * N1 * N2;
  size_t tcw = tc_bwd_weight_ws_floats(rows, N1, N2);
  return simt > tcw ? simt : tcw;
}
int bwd_weight(const void* dY, const void* X, int rows, int N1, int N2, float* dW, int accumulate, float* ws,
               int precision, cudaStream_t st) {
  ADVMIL_REQUIRE(gemm_ok(N1, N2, dY, X), "bwd_weight: N1=%d N2=%d must be multiples of 4", N1, N2);
  if (rows == 0) { if (!accumulate) return fill_zero(dW, (size_t)N1 * N2, st); return ADVMIL_OK; }
  if (precision != ADVMIL_FP32 && tc_bwd_weight_supported(rows, N1, N2, elem_of_precision(precision)))
    return tc_bwd_weight(dY, X, rows, N1, N2, dW, accumulate, ws, precision, st);
  ADVMIL_REQUIRE(precision != ADVMIL_BF16, kBf16Shape, "bwd_weight", rows, N1, N2);
  int splits = pick_splits(rows, N1, N2);
  int kchunk = cdiv(cdiv(rows, splits), BK) * BK;
  splits = cdiv(rows, kchunk);
  GemmArgs g{(const float*)dY, (const float*)X, N1, N2, rows, N1, N2, kchunk};
  EpiPartial epi{ws};
  ADVMIL_TRY((launch_gemm<false, false>(g, epi, splits, st)));
  return splitk_reduce(ws, splits, (size_t)N1 * N2, dW, accumulate, st);
}

int bwd_weight_conv3(const void* dY, const void* X, int rows, int N1, int C, float* dW, int accumulate, float* ws,
                     int precision, cudaStream_t st) {
  ADVMIL_REQUIRE(N1 % 4 == 0 && C % 16 == 0 && rows % 16 == 0 && (((uintptr_t)dY | (uintptr_t)X) % 16 == 0),
                 "bwd_weight_conv3: N1=%d (%%4) C=%d (%%16) rows=%d (%%16) unsupported", N1, C, rows);
  if (rows == 0) { if (!accumulate) return fill_zero(dW, (size_t)N1 * C * 9, st); return ADVMIL_OK; }
  if (precision != ADVMIL_FP32 && tc_conv3_bwd_weight_supported(rows, N1, C, elem_of_precision(precision)))
    return tc_conv3_bwd_weight(dY, X, rows, N1, C, dW, accumulate, ws, precision, st);
  ADVMIL_REQUIRE(precision != ADVMIL_BF16, kBf16Shape, "bwd_weight_conv3", rows, N1, 9 * C);
  const int N2 = 9 * C;
  int splits = pick_splits(rows, N1, N2);
  int kchunk = cdiv(cdiv(rows, splits), BK) * BK;
  splits = cdiv(rows, kchunk);
  GemmArgs g{(const float*)dY, (const float*)X, N1, N2, rows, N1, C, kchunk};
  EpiPartial epi{ws};
  ADVMIL_TRY((launch_gemm<false, false, EpiPartial, TileLoader<false>, Conv3LoaderB>(g, epi, splits, st)));
  return splitk_reduce_conv3(ws, splits, N1, C, dW, accumulate, st);
}

}  // namespace advmil
