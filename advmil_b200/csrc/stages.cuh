// Internal stage launchers shared by the C-ABI composites (api.cu).  All asynchronous on `st`.
#pragma once
#include "common.cuh"

namespace advmil {

// Precision of the RLIP head's region-level (rows / 16) and bag-level contractions.  fp32 stays fp32 (FFMA) and the tf32
// mode runs them on plain tf32 (the mode's definition).  The split-tf32 mode runs them on split tf32; so does the bf16
// mode in the FORWARD pass of a training discriminator (`exact`): the discriminator's parameter gradients are sums in which
// real and fake pair terms cancel, which amplifies the error of the forward outputs f (through dL/df) -- with plain tf32
// (operands truncated to 10 mantissa bits) some tensors were 3-12 % off the bf16-storage oracle, with split tf32 every
// tensor agrees with it to 1.4e-3 (profiles/r02_bf16_parity.md).  These contractions are a fraction of a percent of the
// step's FLOPs and latency-bound; the backward contractions and the eval-mode passes (G step, inference) keep plain tf32.
static inline int region_precision(int precision, bool exact) {
  if (precision == ADVMIL_FP32 || precision == ADVMIL_TF32) return precision;
  if (precision == ADVMIL_TF32X3) return ADVMIL_TF32X3;
  return exact ? ADVMIL_TF32X3 : ADVMIL_TF32;      // bf16 mode
}
// ESAT self-attention: FFMA kernels in the exact modes (fp32, split tf32), tcgen05 tf32 kernels otherwise (esat_kernels.cu:
// head widths other than 16 / 32 / 48 / 64 also run the FFMA kernels)
static inline int attention_precision(int precision) {
  return (precision == ADVMIL_FP32 || precision == ADVMIL_TF32X3) ? ADVMIL_FP32 : ADVMIL_TF32;
}


// ---- gemm_stages.cu ---------------------------------------------------------------------------
// Activation tensors ([rows, *]: x, y, v, ab, y_pre, dY, dX, X, relu_src) are `const void*` / `void*`: bf16 when
// precision == ADVMIL_BF16 (or dt == ELEM_BF16), fp32 otherwise.  Weights, biases, statistics and outputs at bag / region
// granularity are always fp32.
// y2 / drop2 (optional): a second output y2 = dropout(y) under drop2, written by the same pass (the tcgen05 epilogue
// stores both; the FFMA engine adds an apply_dropout pass)
int linear_fwd(const void* x, const float* W, const float* b, int rows, int K, int N, int relu, const Drop& drop,
               void* y, int precision, cudaStream_t st, void* y2 = nullptr, const Drop* drop2 = nullptr);
// K1 (generator projection) and K5+K6 (discriminator region embedding) of the same x in ONE pass (bf16 mode, tcgen05 only):
// hout = relu(x W1^T + b1), hdrop = dropout(hout) under drop2 (optional), y_pre / emb as region_embed_fwd
bool proj_embed_supported(int rows, int C, int h, int d, int precision);
int proj_embed_fwd(const void* x, const float* W1, const float* b1, const float* Wc, const float* bc, const float* gamma,
                   const float* beta, int rows, int C, int h, int d, float eps, void* hout, void* hdrop, const Drop* drop2,
                   void* y_pre, float* emb, cudaStream_t st);
// packed gate weights Wp [abw, L], bp [abw] (zero padded) must have been built by gate_pack_weights.
// s == nullptr: only the per-tile partial scores part_ws [abw/128][rows] are produced (seg_softmax_pool_fwd finishes them)
int gated_score_fwd(const void* v, const float* Wp, const float* bp, const float* wc, const float* bc, int rows, int L,
                    int D, const Drop& da, const Drop& db, void* ab, float* s, float* part_ws, int precision,
                    cudaStream_t st);
// ksize 1: y = x Wc^T + bc (Wc [d, C]); ksize 3: y = 3x3 convolution, zero padded, inside every 4x4 region of 16 rows
// (Wc [d, C, 3, 3], the Conv2d layout).  d <= 128 (%4) or d == 256; the bf16 mode runs d = 64, 128 and 256 only.
// y_ws: rows x d floats of scratch for the FFMA path at d = 256 when y_pre is NULL (the LayerNorm there runs as a
// second pass over y; at every other width the statistics are taken in the GEMM's epilogue)
int region_embed_fwd(const void* x, const float* Wc, const float* bc, const float* gamma, const float* beta, int rows,
                     int C, int d, float eps, void* y_pre, float* emb, int precision, cudaStream_t st, int ksize = 1,
                     float* y_ws = nullptr);
// dX[rows,Nx] = (dY[rows,Ny] . W[Ny,Nx] + pool terms) * relu'  (W row-major [Ny, Nx])
struct BwdDataExtras {
  const float* w = nullptr; const float* dz = nullptr; const float* dmean = nullptr;
  const int32_t* offsets = nullptr; int bags = 0;
  const void* relu_src = nullptr; int ld_src = 0; float inv_keep = 1.f;
  int accumulate = 0;
  float* colsum_part = nullptr;   // tcgen05 engine only: [4 * ceil(rows/128)][Nx] column sums of dX per 32 rows (bias gradient)
};
// true when bwd_data(..., precision) will run on the tcgen05 engine and therefore fills ex.colsum_part
bool bwd_data_fuses_colsum(int rows, int Ny, int Nx, int precision);
int bwd_data(const void* dY, const float* W, int rows, int Ny, int Nx, void* dX, const BwdDataExtras& ex,
             int precision, cudaStream_t st);
// dW[N1,N2] (+)= dY[rows,N1]^T . X[rows,N2]   (split-K over rows; ws >= bwd_weight_ws_floats floats)
size_t bwd_weight_ws_floats(int rows, int N1, int N2);
int bwd_weight(const void* dY, const void* X, int rows, int N1, int N2, float* dW, int accumulate, float* ws,
               int precision, cudaStream_t st);
// dW[N1, C, 3, 3] (+)= the weight gradient of the 3x3 region convolution of X[rows, C] (rows % 16 == 0) under dY[rows, N1]
// (ws >= bwd_weight_ws_floats(rows, N1, 9 C) floats)
int bwd_weight_conv3(const void* dY, const void* X, int rows, int N1, int C, float* dW, int accumulate, float* ws,
                     int precision, cudaStream_t st);

// ---- cluster_pool.cu: K9 of the DeepAttMISL generator ------------------------------------------------------------------
constexpr int CLUSTER_POOL_MAX = 16;     // clusters per bag the tcgen05 epilogue keeps sums for
// true when cluster_pool_fwd runs for this shape and mode (tcgen05 engine; the fp32 mode composes linear_fwd and the
// segment mean instead)
bool cluster_pool_fused(int rows, int C, int h, int precision);
size_t cluster_pool_ws_floats(int rows, int bags, int h, int ncl);
// hc [bags * ncl, h] = per-(bag, cluster) mean of relu(x W^T + b), counts [bags * ncl]; keep (optional) [rows, h / 32] ReLU
// keep bits; ws >= cluster_pool_ws_floats.  Every bag length a multiple of 16, 1 <= ncl <= CLUSTER_POOL_MAX.
int cluster_pool_fwd(const void* x, const float* W, const float* b, const int32_t* cid, const int32_t* offsets,
                     const int32_t* offsets_host, int rows, int bags, int C, int h, int ncl, int precision, float* hc,
                     int32_t* counts, uint32_t* keep, float* ws, cudaStream_t st);
// d_hx [rows, h] (T of precision) = keep * d_hc[bag, cid] / count
int cluster_pool_bwd(const float* d_hc, const uint32_t* keep, const int32_t* cid, const int32_t* offsets, const int32_t* counts,
                     int rows, int bags, int h, int ncl, int precision, void* d_hx, cudaStream_t st);

// ---- rlip_chain.cu ----------------------------------------------------------------------------
// fc1 MLP + GAPool gate of the RLIP head over R regions in one split-tf32 mma.sync kernel (d = 64, 128 or 256): writes
// f1 [R, d/2], fi [R, d],
// ab [R, 2d] packed (optional) and the per-64-pair partial logits part [d/64][R] (finished by seg_softmax_pool_fwd)
bool rlip_chain_supported(int d);
int rlip_chain_fwd(const float* emb, const AdvmilDiscParams& p, int R, const Drop& dfc1, const Drop& dga, const Drop& dgs,
                   float* f1, float* fi, float* ab, float* part, cudaStream_t st);

// ---- seg_kernels.cu ---------------------------------------------------------------------------
int gate_pack_weights(const float* Wa, const float* ba, const float* Wb, const float* bb, int L, int D, float* Wp,
                      float* bp, cudaStream_t st);
int gate_unpack_grads(const float* dWp, const float* dbp, int L, int D, float* dWa, float* dba, float* dWb, float* dbb,
                      int accumulate, cudaStream_t st);
int gate_score_finish(const float* part, int ntiles, int rows, const float* bc, float* s, cudaStream_t st);
size_t seg_pool_ws_floats(int rows, int bags, int width);
// sparts != nullptr: the logits are assembled here from the gate kernel's per-tile partial scores (sparts [ntiles][rows],
// + bc[0]) and written to s (gated_score_fwd was called with s == nullptr); else s is read.
int seg_softmax_pool_fwd(float* s, const float* sparts, int ntiles, const float* bc, const void* v, int dt, const int32_t* offsets,
                         const int32_t* offsets_host, int rows, int bags, int width, float* w, float* z, float* mean, float* ws,
                         cudaStream_t st);
// rows_per_cta used by the row-chunked backward kernels (partials are [nchunks, ...])
constexpr int ROWS_PER_CTA = 128;
inline int row_chunks(int rows) { return cdiv(rows, ROWS_PER_CTA); }
// pooling + gate backward: ds = w (dz.v - dz.z); dAB packed; partial dwc/dbc per chunk -> reduced into dwc, dbc
int pool_gate_bwd(const void* v, const float* w, const float* z, const float* dz, const void* ab, const float* wc,
                  const int32_t* offsets, int rows, int bags, int L, int D, const Drop& da, const Drop& db, void* dAB,
                  float* dwc, float* dbc, float* dbp /* packed gate-bias grad [abw] or null */, int accumulate,
                  float* ws /* >= pool_gate_ws_floats */, int dt, cudaStream_t st);
inline size_t pool_gate_ws_floats(int rows, int bags, int D) {
  return align_up((size_t)bags, 64) + align_up((size_t)row_chunks(rows) * (D + 1), 64) + (size_t)row_chunks(rows) * gate_width(D) +
         align_up((size_t)rows, 64) + 64;
}
// LayerNorm + ReLU + region-mean backward per row; partials of dgamma/dbeta/dbias reduced into the outputs
// d_emb2 (optional): a second upstream gradient that is added to d_emb (real + fake halves of a batched D step)
int ln_pool_bwd(const void* y_pre, const float* d_emb, const float* d_emb2, const float* gamma, const float* beta, int rows,
                int d, float eps, void* d_y, float* dgamma, float* dbeta, float* dbias, int accumulate,
                float* ws /* >= row_chunks*3*d floats */, int dt, cudaStream_t st);

// ---- api.cu ---------------------------------------------------------------------------------
int disc_embed_bwd_impl(const AdvmilDiscParams* p, const AdvmilBags* bags, const AdvmilEmbedActs* a, const float* d_emb,
                        const float* d_emb2, AdvmilDiscGrads* g, int accumulate, cudaStream_t st);
int colsum(const void* dY, int dt, int rows, int N, int ld, float* out, int accumulate, float* ws /* >= row_chunks*N */,
           cudaStream_t st);
int reduce_rows(const float* part, int nparts, int width, float* out, int accumulate, cudaStream_t st);
// out[c] (+)= sum_p part[p * stride + c], c < ncols
int reduce_rows_strided(const float* part, int nparts, int stride, int ncols, float* out, int accumulate, cudaStream_t st);
int splitk_reduce(const float* ws, int splits, size_t n, float* out, int accumulate, cudaStream_t st);
int splitk_reduce_t(const float* ws, int splits, int R, int Cc, float* out, int accumulate, cudaStream_t st);
// ws slices [N1][9 C] tap-major -> out [N1][C][3][3]
int splitk_reduce_conv3(const float* ws, int splits, int N1, int C, float* out, int accumulate, cudaStream_t st);
int apply_dropout(const void* src, int rows, int width, const Drop& drop, void* dst, int dt, cudaStream_t st);
int fill_zero(float* p, size_t n, cudaStream_t st);
int cast_f32_to_bf16(const float* in, size_t n, void* out, cudaStream_t st);

// ---- esat_kernels.cu (region-level stages of the ESAT backbone, model/backbone.py:171-196) ---------------------------
// emb[r] = mean_{k<16} relu(LN(y_pre[16r+k])) (+ pe[r]);  y_pre: T [rows, d], d % 32 == 0
int ln_relu_mean16_fwd(const void* y_pre, const float* gamma, const float* beta, int rows, int d, float eps, const float* pe,
                       float* emb, int dt, cudaStream_t st);
int esat_ln_bwd_ctas(int R);   // partial-sum rows the two LayerNorm backward kernels write (workspace sizing)
int ln_relu_mean16_bwd(const void* y_pre, const float* d_emb, const float* gamma, const float* beta, int rows, int d, float eps,
                       void* d_y, float* dgamma, float* dbeta, float* dbias, float* ws /* >= ctas*3*d */, int dt, cudaStream_t st);
// out = LN(a + b); b is overwritten with s = a + b
int add_ln_fwd(const float* a, float* b_s, const float* gamma, const float* beta, int R, int d, float eps, float* out, cudaStream_t st);
int add_ln_bwd(const float* s, const float* gamma, const float* d_out, int R, int d, float eps, float* d_s, float* dgamma,
               float* dbeta, float* ws /* >= ctas*2*d */, cudaStream_t st);
int add_rows(float* a, const float* b, size_t n, cudaStream_t st);   // a += b
int sincos_pe(const int64_t* coord, const int32_t* ro, int bags, int d, const float* omega, float* pe, cudaStream_t st);
// self-attention over the regions of each bag: qkv [R, 3d] -> ctx [R, d], lse [heads, R]; ro = region offsets [bags+1]
int mha_fwd(const float* qkv, const int32_t* ro, const int32_t* ro_host, int bags, int Rtot, int d, int heads, const Drop& drop,
            const uint8_t* mask, const int64_t* mask_off, float* ctx, float* lse, int precision, cudaStream_t st);
int mha_bwd(const float* qkv, const float* ctx, const float* d_ctx, const float* lse, const int32_t* ro, const int32_t* ro_host,
            int bags, int Rtot, int d, int heads, const Drop& drop, const uint8_t* mask, const int64_t* mask_off, float* d_qkv,
            float* Dq /* [heads, R] */, int precision, cudaStream_t st);

// ---- esat.cu ------------------------------------------------------------------------------------
void esat_request_overlap(int on);   // this thread's next advmil_esat_bwd calls may use the backward side stream (C-fused step)

// ---- tail_kernels.cu --------------------------------------------------------------------------
int gen_head_fwd(const AdvmilGenParams& p, const float* z, const float* noise0, const float* noise1, int bags,
                 int samples, const Drop& drho, const Drop& dmlp0, float* H, float* H1, float* pre, float* pred,
                 cudaStream_t st);
// per-bag vector backward; writes dz [bags,h], dHpre [bags,o], dH1pre [bags,hid], dpre [bags]
int gen_head_bwd(const AdvmilGenParams& p, const float* d_pred, const float* H, const float* H1, const float* pred,
                 int bags, float inv_keep_rho, float inv_keep_mlp0, float* dz, float* dHpre, float* dH1pre, float* dpre,
                 cudaStream_t st);
// dW[out, in1+in2] (+)= sum_b dy[b,out] * concat(x1[b,:in1], x2[b,:in2]);  db[out] (+)= sum_b dy[b,out]
int outer_sum(const float* dy, const float* x1, int in1, const float* x2, int in2, int bags, int out, float* dW,
              float* db, int accumulate, cudaStream_t st);
// up to OUTER_MAX outer-sum problems (same bags, same accumulate flag) in one launch
constexpr int OUTER_MAX = 6;
struct OuterProb { const float* dy; const float* x1; int in1; const float* x2; int in2; int out; float* dW; float* db; };
int outer_sum_multi(const OuterProb* probs, int n, int bags, int accumulate, cudaStream_t st);
int rlip_tail_fwd(const AdvmilDiscParams& p, const float* bagv, const float* fbar, const float* t, int bags,
                  const Drop& dfc2, float* g1, float* hx, float* u1, float* ht, float* out, cudaStream_t st);
int rlip_tail_bwd(const AdvmilDiscParams& p, const float* d_out, const float* bagv, const float* fbar, const float* g1,
                  const float* hx, const float* u1, const float* ht, int bags, float inv_keep_fc2, float* d_fbar,
                  float* d_bagv, float* d_hx, float* d_g1pre, float* d_htpre, float* d_u1pre, float* d_t,
                  cudaStream_t st);

}  // namespace advmil
