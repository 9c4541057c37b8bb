// tcgen05 / TMEM / TMA engine for the N-row contractions (declarations; implementation in gemm_tc.cu).
// dt = ELEM_F32 / ELEM_BF16 element type of the activation tensors (`void*` arguments); precision picks the MMA kind.
#pragma once
#include "stages.cuh"

namespace advmil {

bool tc_linear_supported(int rows, int K, int N, int dt);
int tc_linear_fwd(const void* x, const float* W, const float* b, int rows, int K, int N, int relu, const Drop& drop,
                  void* y, int precision, cudaStream_t st, void* y2 = nullptr, const Drop* drop2 = nullptr);
bool tc_proj_embed_supported(int rows, int C, int h, int d, int dt);
int tc_proj_embed_fwd(const void* x, const float* W1, const float* b1, const float* Wc, const float* bc, const float* gamma,
                      const float* beta, int rows, int C, int h, int d, float eps, void* hout, void* hdrop, const Drop* drop2,
                      void* y_pre, float* emb, cudaStream_t st);
// K9: part[(m-tile + bag) * ncl + cluster][N] = column sums of relu(x W^T + b) over the tile's rows of that bag and cluster;
// keep (optional) = the ReLU keep bits [rows][N / 32].  Every bag length a multiple of 16; ncl <= 16.
bool tc_proj_pool_supported(int rows, int C, int N, int dt);
int tc_proj_pool_fwd(const void* x, const float* W, const float* b, const int32_t* cid, const int32_t* offsets, int bags, int rows,
                     int C, int N, int ncl, uint32_t* keep, float* part, int precision, cudaStream_t st);
bool tc_gate_supported(int rows, int L, int D, int dt);
int tc_gated_score_fwd(const void* v, const float* Wp, const float* bp, const float* wc, const float* bc, int rows,
                       int L, int D, const Drop& da, const Drop& db, void* ab, float* s, float* part, int precision,
                       cudaStream_t st);
bool tc_embed_supported(int rows, int C, int d, int dt);
int tc_region_embed_fwd(const void* x, const float* Wc, const float* bc, const float* gamma, const float* beta,
                        int rows, int C, int d, float eps, void* y_pre, float* emb, int precision, cudaStream_t st);
// 3x3 region convolution (Wc [d, C, 3, 3]; same support rule as tc_embed_supported, rows % 16 == 0)
int tc_conv3_embed_fwd(const void* x, const float* Wc, const float* bc, const float* gamma, const float* beta,
                       int rows, int C, int d, float eps, void* y_pre, float* emb, int precision, cudaStream_t st);
// fp32 tap-major repack [N, 9 C] of a 3x3 weight in library scratch (the FFMA engine's operand)
int conv3_weight_f32(const float* W, int N, int C, cudaStream_t st, const float** out);
bool tc_bwd_data_supported(int rows, int Ny, int Nx, int dt);
int tc_bwd_data(const void* dY, const float* W, int rows, int Ny, int Nx, void* dX, const BwdDataExtras& ex,
                int precision, cudaStream_t st);
bool tc_bwd_weight_supported(int rows, int N1, int N2, int dt);
size_t tc_bwd_weight_ws_floats(int rows, int N1, int N2);
int tc_bwd_weight(const void* dY, const void* X, int rows, int N1, int N2, float* dW, int accumulate, float* ws,
                  int precision, cudaStream_t st);
bool tc_conv3_bwd_weight_supported(int rows, int N1, int C, int dt);
int tc_conv3_bwd_weight(const void* dY, const void* X, int rows, int N1, int C, float* dW, int accumulate, float* ws,
                        int precision, cudaStream_t st);

}  // namespace advmil
