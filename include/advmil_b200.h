/*
 * advmil_b200 — C ABI of the B200-native AdvMIL hot path (libadvmil_b200.so).
 *
 * This is the drop-in boundary: plain pointers and sizes, no torch types.  The reference
 * (liupei101/AdvMIL) is pure Python/PyTorch and has no FFI of its own; each entry point below
 * replaces the named reference interface (file:line relative to the reference root) and is bound
 * from Python with ctypes (advmil_b200/_lib.py; INTEGRATION.md shows the stub).
 *
 * Conventions (SURVEY.md §8b):
 *   - every entry point returns int: 0 = ok, non-zero = AdvmilStatus; never throws;
 *   - no entry point allocates device memory: all outputs, saved activations and scratch are
 *     caller-owned (sizes via advmil_*_workspace_bytes);
 *   - every entry point takes an explicit cudaStream_t (passed as void*) and is asynchronous;
 *   - all device tensors are dense row-major fp32 unless stated; "bags" are packed:
 *     x[rows, C] with int32 offsets[bags+1] (offsets[0] = 0, offsets[bags] = rows), which is
 *     dataset/PatchWSI.py:65-94's per-patient [N,1024] tensors concatenated.
 *   - dropout sites take either an injected keep-mask (uint8, 1 = keep; parity tests) or, when the
 *     mask pointer is NULL and train != 0, a counter-based in-kernel generator keyed by `seed`
 *     (forward and backward regenerate identical bits).
 */
#ifndef ADVMIL_B200_H_
#define ADVMIL_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum AdvmilStatus {
  ADVMIL_OK = 0,
  ADVMIL_ERR_INVALID = 1,   /* bad argument / unsupported shape (reference: AssertionError / ValueError) */
  ADVMIL_ERR_CUDA = 2,      /* a CUDA runtime call or launch failed; advmil_last_error() has the text */
  ADVMIL_ERR_WORKSPACE = 3, /* workspace too small */
  ADVMIL_ERR_NO_DEVICE = 4  /* no sm_100 device */
} AdvmilStatus;

#define ADVMIL_ABI_VERSION 3
#if defined(__GNUC__)
#define ADVMIL_API __attribute__((visibility("default")))
#else
#define ADVMIL_API
#endif

/* GEMM engine selection for the N-row contractions (K1/K2/K5 and their backward):
 *   0 = fp32 FFMA tiles (exact-fp32 mode, rtol 1e-5 parity)
 *   1 = tcgen05 kind::tf32 single pass, TMA-fed, TMEM accumulators (fast mode, <= 2e-2 parity)
 *   2 = reserved (3xTF32); currently served by mode 1
 *   3 = bf16 storage mode: x and every [rows, *] activation tensor that crosses the ABI (h, ab, h_eval, y_pre; and the
 *       library's own dAB / dh / dy scratch) are bfloat16, tcgen05 kind::f16 with fp32 accumulation in TMEM; all
 *       statistics, region/bag-level tensors, parameters, gradients and optimiser state stay fp32 (<= 2e-2 parity).
 * Pointers documented as "T" below are float in modes 0-2 and bfloat16 (2-byte) in mode 3.                    */
typedef enum AdvmilPrecision { ADVMIL_FP32 = 0, ADVMIL_TF32 = 1, ADVMIL_TF32X3 = 2, ADVMIL_BF16 = 3 } AdvmilPrecision;
typedef enum AdvmilElem { ADVMIL_ELEM_F32 = 0, ADVMIL_ELEM_BF16 = 1 } AdvmilElem;

/* ---- packed bags ------------------------------------------------------------------------- */
typedef struct AdvmilBags {
  const void* x;               /* [rows, C] device, element type `elem` */
  const int32_t* offsets;      /* [bags+1] device */
  const int32_t* offsets_host; /* [bags+1] host copy (grid sizing, validation) */
  int32_t rows, bags, C, max_bag_rows;
  int32_t elem;                /* AdvmilElem of x: must be BF16 with precision ADVMIL_BF16 and F32 otherwise */
} AdvmilBags;

/* ---- generator: ABMIL encoder + noise head (model/GANSurv.py:13-49, model/backbone.py:54-86,
 *      model/backbone_utils.py:11-29, model/model_utils.py:116-133) ------------------------- */
typedef struct AdvmilGenParams {
  const float *W1, *b1;       /* backbone.attention_net.0        [h,C],[h]  */
  const float *Wa, *ba;       /* ...attention_net.3.attention_a.0 [h,h],[h] */
  const float *Wb, *bb;       /* ...attention_net.3.attention_b.0 [h,h],[h] */
  const float *wc, *bc;       /* ...attention_net.3.attention_c   [1,h],[1] */
  const float *Wrho, *brho;   /* backbone.rho.0                   [o,h],[o] (NULL for DeepAttMISL) */
  const float *W0, *b0;       /* MLPs.0.0  [hid, o*(1+noise0)],[hid] */
  const float *Wl, *bl;       /* MLPs.1.0  [1, hid*(1+noise1)],[1]   */
  int32_t C, h, o, hid;
  int32_t noise0, noise1;     /* gen_noi_noise "n0-n1" (config/cfg_nlst.yaml:30) */
  int32_t out_scale;          /* 0 none, 1 sigmoid, 2 exp (GANSurv.py:43-48) */
  float p_backbone, p_head;   /* dropout probabilities 0.25 / gen_dropout */
} AdvmilGenParams;

typedef struct AdvmilGenGrads { /* same tensors as AdvmilGenParams, written (not accumulated) */
  float *W1, *b1, *Wa, *ba, *Wb, *bb, *wc, *bc, *Wrho, *brho, *W0, *b0, *Wl, *bl;
  float *dx; /* optional [rows,C]: gradient w.r.t. the bag features (NULL = skipped; the WSI features never need it,
                the DeepAttMISL cluster path does for its pooled cluster rows) */
} AdvmilGenGrads;

typedef struct AdvmilGenActs {
  void* h;      /* T [rows,h]   relu(+dropout) of the projection; pooled tensor (backbone.py:81-84) */
  void* ab;     /* T [rows,abw] tanh|sigmoid gate activations, packed column order (see advmil_gate_packed_width); NULL = not
                   saved.  Train mode: the sign of a stored sigmoid is the joint dropout keep bit of its (tanh, sigmoid)
                   pair (negative = the pair was dropped); its magnitude is the undropped activation. */
  float* s;     /* [rows] attention logits */
  float* w;     /* [rows] softmax weights within each bag */
  float* z;     /* [bags,h] pooled */
  float* H;     /* [bags,o] rho output (post dropout) */
  float* H1;    /* [bags,hid] MLPs.0 output (post dropout) */
  float* pre;   /* [bags] last-layer pre-activation */
  float* pred;  /* [bags] output */
  const float* noise0; /* [bags,o]   or NULL (zero / unused) */
  const float* noise1; /* [bags,hid] or NULL */
  const void* h_eval;  /* optional T [rows,h]: eval-mode h of the same x and W1 (dropout is applied to it instead of recomputing K1) */
  const uint8_t *mask_h, *mask_a, *mask_b, *mask_rho, *mask_mlp0; /* optional injected keep masks */
  uint64_t seed;
  int32_t train;       /* 0 eval (no dropout), 1 train */
  int32_t precision;   /* AdvmilPrecision */
  void* workspace; size_t workspace_bytes;
  /* projection sharing between an eval pass and a later train pass over the same x and W1 (the fused step):
   *   eval pass : h_drop_out != NULL -> the projection kernel also writes dropout(h) under (seed_drop | mask_h_drop) there;
   *   train pass: h_ready != 0       -> `h` already holds that dropped projection: neither K1 nor a dropout pass runs.   */
  void* h_drop_out; uint64_t seed_drop; const uint8_t* mask_h_drop;
  int32_t h_ready;
} AdvmilGenActs;

/* ---- discriminator: RLIP (model/GANSurv.py:71-105, model/model_utils.py:157-210,
 *      model/backbone_utils.py:31-77,129-168) ----------------------------------------------- */
typedef struct AdvmilDiscParams {
  const float *Wc, *bc;        /* net_pair_one.embedding.conv [d,C(,1,1)] (ksize 0 / 1) or [d,C,3,3] (ksize 3),[d] */
  const float *ln_g, *ln_b;    /* net_pair_one.embedding.norm [d],[d] */
  const float *F1a_w, *F1a_b;  /* net_pair_one.fc1.0 [d/2,d] */
  const float *F1b_w, *F1b_b;  /* net_pair_one.fc1.3 [d,d/2] */
  const float *Pg_w, *Pg_b;    /* net_pair_one.pool.fc1.0   [d,d] (tanh branch)    */
  const float *Ps_w, *Ps_b;    /* net_pair_one.pool.score.0 [d,d] (sigmoid branch) */
  const float *Pc_w, *Pc_b;    /* net_pair_one.pool.fc2     [1,d],[1] */
  const float *F2a_w, *F2a_b;  /* net_pair_one.fc2.0 [d/2,d] */
  const float *F2b_w, *F2b_b;  /* net_pair_one.fc2.3 [d,d/2] */
  const float *T1_w, *T1_b;    /* net_pair_two.0.0 [t1,1] */
  const float *T2_w, *T2_b;    /* net_pair_two.1.0 [t2,t1] */
  const float *Pr_w, *Pr_b;    /* prj_layer [1,d] (or NULL); prj_path 3: the concat discriminator's fc [1, d + t2] */
  int32_t C, d, t1, t2;
  int32_t inner_instance;      /* 1 = 'instance' (RLIP), 0 = 'bag' (GANSurv.py:92-98) */
  int32_t prj_path;            /* 0 none, 1 'x', 2 'y' (PrjDiscriminator); 3 = Discriminator (GANSurv.py:52-68):
                                  out = fc(cat[hx, ht]) with no inner product (inner_instance ignored) */
  float p;                     /* disc_netx_dropout */
  float ln_eps;
  int32_t ksize;               /* disc_netx_ksize: kernel size of the patch-embedding conv.  0 or 1 = per-patch linear;
                                  3 = 3x3 convolution (stride 1, padding 1) over each region's 4x4 grid of patches, zero
                                  padded at the region border (needs C % 16 == 0, and C % 128 == 0 in ADVMIL_BF16);
                                  anything else = ADVMIL_ERR_INVALID */
} AdvmilDiscParams;

typedef struct AdvmilDiscGrads {
  float *Wc, *bc, *ln_g, *ln_b, *F1a_w, *F1a_b, *F1b_w, *F1b_b, *Pg_w, *Pg_b, *Ps_w, *Ps_b, *Pc_w, *Pc_b,
        *F2a_w, *F2a_b, *F2b_w, *F2b_b, *T1_w, *T1_b, *T2_w, *T2_b, *Pr_w, *Pr_b;
} AdvmilDiscGrads;

typedef struct AdvmilEmbedActs {      /* K5+K6: region embedding */
  float* emb;    /* [rows/16, d] */
  void* y_pre;   /* T [rows, d] pre-LayerNorm projection, NULL = not saved (no D-param backward) */
  int32_t precision;
  /* workspace: required by advmil_disc_embed_bwd (advmil_disc_workspace_bytes(p, rows, bags, 1) bytes).  The forward reads
   * it only on the exact-fp32 FFMA path at d = 256 with y_pre == NULL (fp32 mode, or tf32 / tf32x3 below 128 rows), where
   * it needs rows * d * 4 bytes for y before the LayerNorm pass; the backward size above covers that. */
  void* workspace; size_t workspace_bytes;
} AdvmilEmbedActs;

typedef struct AdvmilHeadActs {       /* K7+K8: region MLP, GAPool, bag MLP, time embedding, inner product */
  const float* emb; /* [R,d] */
  const float* t;   /* [bags] time fed to D (real label or generator output) */
  float* f1;    /* [R,d/2] fc1 hidden (post relu+dropout) */
  float* fi;    /* [R,d] instance embeddings (post fc1; quirk A.4#2) */
  float* ab;    /* [R,abw] GAPool gate activations packed */
  float* rep;   /* [R] GAPool logits */
  float* attn;  /* [R] GAPool softmax */
  float* bagv;  /* [bags,d] attention-pooled */
  float* fbar;  /* [bags,d] mean_r fi */
  float* g1;    /* [bags,d/2] fc2 hidden (post relu+dropout) */
  float* hx;    /* [bags,d] */
  float* u1;    /* [bags,t1] */
  float* ht;    /* [bags,t2] */
  float* out;   /* [bags] */
  const uint8_t *mask_fc1, *mask_ga, *mask_gs, *mask_fc2;
  uint64_t seed;
  int32_t train;
  int32_t precision;  /* AdvmilPrecision of the step: FP32 = exact FFMA; any other mode runs the region-level contractions
                         (all tensors here are fp32) on tcgen05 kind::tf32 */
  void* workspace; size_t workspace_bytes;
} AdvmilHeadActs;

/* ---- version / diagnostics ---------------------------------------------------------------- */
ADVMIL_API int advmil_abi_version(void);
ADVMIL_API const char* advmil_last_error(void);
/* sizeof() of the ABI structs, for binding self-checks: which = 0 Bags, 1 GenParams, 2 GenGrads, 3 GenActs,
 * 4 DiscParams, 5 DiscGrads, 6 EmbedActs, 7 HeadActs, 8 StepArgs, 9 EsatParams, 10 EsatGrads, 11 EsatActs, 12 EsatStepArgs,
 * 13 ClusterStepArgs */
ADVMIL_API size_t advmil_abi_sizeof(int which);
/* counts kernel launches issued by this library since the last reset (bench "gpu_launches") */
ADVMIL_API int64_t advmil_launch_count(int reset);
/* per-stage CUDA-event profiling of the N-row kernels (bench.py roofline): enable, run steps, read.  read() synchronises
 * the device and returns accumulated milliseconds / launch counts per AdvmilProfTag, then clears the records. */
typedef enum AdvmilProfTag {
  ADVMIL_PROF_PROJ = 0, ADVMIL_PROF_GATE = 1, ADVMIL_PROF_POOL = 2, ADVMIL_PROF_EMBED = 3, ADVMIL_PROF_POOL_BWD = 4,
  ADVMIL_PROF_BWD_DATA = 5, ADVMIL_PROF_BWD_W_GATE = 6, ADVMIL_PROF_BWD_W_PROJ = 7, ADVMIL_PROF_LN_BWD = 8,
  ADVMIL_PROF_BWD_W_EMBED = 9, ADVMIL_PROF_COLSUM = 10, ADVMIL_PROF_DROPOUT = 11,
  /* composites of the region-level / bag-level (latency-bound) work, reported in microseconds, not as roofline fractions */
  ADVMIL_PROF_HEAD_FWD = 12, ADVMIL_PROF_HEAD_BWD = 13, ADVMIL_PROF_GEN_TAIL = 14, ADVMIL_PROF_LOSS_OPT = 15,
  ADVMIL_PROF_PROJ_EMBED = 16, /* K1 + K5/K6 in one pass over x (fused step, bf16 mode) */
  ADVMIL_PROF_NTAGS = 17
} AdvmilProfTag;
ADVMIL_API int advmil_profile_enable(int on);
ADVMIL_API int advmil_profile_read(double* ms, int64_t* counts, int32_t ntags);
/* packed gate width: 128 * ceil(D/64) columns; column of tanh_j = 128*(j/64)+j%64, sigmoid_j = +64 */
ADVMIL_API int32_t advmil_gate_packed_width(int32_t D);

/* ---- generator (replaces Generator.forward, model/GANSurv.py:30-49, with backbone ABMIL.forward,
 *      model/backbone.py:79-86) over packed bags; backward = autograd of the same (K10) ---------- */
ADVMIL_API size_t advmil_generator_workspace_bytes(const AdvmilGenParams* p, int32_t rows, int32_t bags, int32_t backward);
ADVMIL_API int advmil_generator_fwd(const AdvmilGenParams* p, const AdvmilBags* bags, AdvmilGenActs* acts, void* stream);
/* d_pred: [bags] dL/dpred. Writes all parameter gradients (summed over the bags).
 * Backbone-only mode: when p->W0 == NULL the forward stops at H (ABMIL.forward, model/backbone.py:79-86) and d_pred is
 * dL/dH [bags,o]. */
ADVMIL_API int advmil_generator_bwd(const AdvmilGenParams* p, const AdvmilBags* bags, const AdvmilGenActs* acts,
                         const float* d_pred, AdvmilGenGrads* grads, void* stream);
/* Head only: S noise draws per bag from one backbone pass (replaces the 30 redundant Generator forwards of
 * MyHandler.test_model, model/model_handler.py:624-636).  H: [bags,o]; noise1: [S,bags,hid]; out: [S,bags] */
ADVMIL_API int advmil_generator_sample(const AdvmilGenParams* p, const float* H, const float* noise0, const float* noise1,
                            int32_t bags, int32_t samples, float* out, void* stream);

/* ---- discriminator ------------------------------------------------------------------------ */
/* K5+K6 (AVGPoolPatchEmbedding.forward, model/backbone_utils.py:158-168): emb[r] = mean_{k<16} relu(LN(x[16r+k]Wc^T+bc)),
 * or with ksize 3 the same over y = conv3x3(region r's 4x4 grid of rows) + bc.
 * Every bag length must be a multiple of 16 (backbone_utils.py:65) else ADVMIL_ERR_INVALID. */
ADVMIL_API size_t advmil_disc_workspace_bytes(const AdvmilDiscParams* p, int32_t rows, int32_t bags, int32_t backward);
ADVMIL_API int advmil_disc_embed_fwd(const AdvmilDiscParams* p, const AdvmilBags* bags, AdvmilEmbedActs* acts, void* stream);
/* d_emb [R,d] -> dWc, dbc, dln_g, dln_b (accumulate != 0 adds into grads) */
ADVMIL_API int advmil_disc_embed_bwd(const AdvmilDiscParams* p, const AdvmilBags* bags, const AdvmilEmbedActs* acts,
                          const float* d_emb, AdvmilDiscGrads* grads, int32_t accumulate, void* stream);
/* K7+K8 (EmbedXLayer.forward model/model_utils.py:202-210 after the embedding; PrjDiscriminator.forward
 * model/GANSurv.py:89-105) */
ADVMIL_API int advmil_disc_head_fwd(const AdvmilDiscParams* p, const AdvmilBags* bags, AdvmilHeadActs* acts, void* stream);
/* d_out [bags] -> d_emb [R,d] (NULL = skip), d_t [bags] (NULL = skip), parameter grads (NULL = skip).
 * accumulate != 0 adds into d_emb and grads instead of overwriting. */
ADVMIL_API int advmil_disc_head_bwd(const AdvmilDiscParams* p, const AdvmilBags* bags, const AdvmilHeadActs* acts,
                         const float* d_out, float* d_emb, float* d_t, AdvmilDiscGrads* grads,
                         int32_t accumulate, void* stream);

/* ---- DeepAttMISL cluster pooling (model/backbone.py:105-117): hc[b,c] = mean_{n in bag b, cid[n]==c} v[n,:], zeros if empty.
 * v: [rows,width]; cid: [rows] int32 in [0,num_clusters); out: [bags*num_clusters,width]; counts: [bags*num_clusters] int32 */
ADVMIL_API size_t advmil_segment_mean_workspace_bytes(int32_t rows, int32_t bags, int32_t width, int32_t num_clusters);
ADVMIL_API int advmil_segment_mean_by_id_fwd(const void* v /*elem*/, int32_t elem, const int32_t* cid, const int32_t* offsets,
                                  const int32_t* offsets_host, int32_t rows, int32_t bags, int32_t width,
                                  int32_t num_clusters, float* out, int32_t* counts, void* workspace,
                                  size_t workspace_bytes, void* stream);
/* d_v[n,:] = d_out[bag(n), cid[n], :] / count, optionally masked by (v > 0) (ReLU before the mean) */
ADVMIL_API int advmil_segment_mean_by_id_bwd(const float* d_out, const void* v /*elem*/, int32_t elem, const int32_t* cid,
                                  const int32_t* offsets, const int32_t* counts, int32_t rows, int32_t bags, int32_t width,
                                  int32_t num_clusters, int32_t relu_mask, void* d_v /*elem*/, void* stream);

/* The same K9 as ONE tcgen05 pass (ADVMIL_TF32 / ADVMIL_TF32X3 / ADVMIL_BF16; the fp32 mode has no such pass): hc[b,c] =
 * per-(bag, cluster) mean of relu(x W^T + b) (x [rows,C] of the precision's element type, W [h,C], b [h]), counts
 * [bags*num_clusters] int32; keep (optional, device uint32 [rows, h/32]): the ReLU keep bits (pre-activation > 0), bit i of
 * word j = column 32 j + i.  The [rows,h] activation is never written.  Rows whose id is outside [0, num_clusters) count
 * nowhere.  Every bag length must be a multiple of 16 and 1 <= num_clusters <= 16, else ADVMIL_ERR_INVALID.  Deterministic
 * (no floating-point atomics).  workspace >= advmil_cluster_pool_workspace_bytes. */
ADVMIL_API size_t advmil_cluster_pool_workspace_bytes(int32_t rows, int32_t bags, int32_t h, int32_t num_clusters);
ADVMIL_API int advmil_cluster_pool_fwd(const void* x, const float* W, const float* b, const int32_t* cid, const int32_t* offsets,
                                       const int32_t* offsets_host, int32_t rows, int32_t bags, int32_t C, int32_t h,
                                       int32_t num_clusters, int32_t precision, float* hc, int32_t* counts, uint32_t* keep,
                                       void* workspace, size_t workspace_bytes, void* stream);
/* its backward: d_hx[n,:] = keep(n,:) * d_hc[bag(n), cid[n], :] / count (element type of precision; zeros for ids outside
 * [0, num_clusters)) */
ADVMIL_API int advmil_cluster_pool_bwd(const float* d_hc, const uint32_t* keep, const int32_t* cid, const int32_t* offsets,
                                       const int32_t* counts, int32_t rows, int32_t bags, int32_t h, int32_t num_clusters,
                                       int32_t precision, void* d_hx, void* stream);

/* ---- stage-level entry points (also used by the DeepAttMISL path and by the kernel unit tests) ---- */
/* y = act(x W^T + b): act 0 none, 1 relu; optional dropout (p, mask or seed/site) -> y [rows,N].  W: [N,K] fp32.
 * x, y (and dY, X, dX, v, ab below): element type T of `precision` (bf16 in ADVMIL_BF16, else fp32). */
ADVMIL_API int advmil_linear_fwd(const void* x, const float* W, const float* b, int32_t rows, int32_t K, int32_t N, int32_t act,
                      float p_drop, const uint8_t* mask, uint64_t seed, int32_t site, int32_t train,
                      int32_t precision, void* y, void* stream);
/* dX = dY W, dW = dY^T X, db = colsum(dY); any output may be NULL (dX needs W, dW needs X).  accumulate != 0 adds
 * into dX, dW and db instead of overwriting them. */
ADVMIL_API int advmil_linear_bwd(const void* dY, const void* X, const float* W, int32_t rows, int32_t K, int32_t N,
                      void* dX, float* dW, float* db, int32_t accumulate, int32_t precision,
                      void* workspace, size_t workspace_bytes, void* stream);
ADVMIL_API size_t advmil_linear_bwd_workspace_bytes(int32_t rows, int32_t K, int32_t N);
/* gated attention scores (Attn_Net_Gated.forward, model/backbone_utils.py:24-29) */
ADVMIL_API int advmil_gated_score_fwd(const void* v, const float* Wa, const float* ba, const float* Wb, const float* bb,
                           const float* wc, const float* bc, int32_t rows, int32_t L, int32_t D, float p_drop,
                           const uint8_t* mask_a, const uint8_t* mask_b, uint64_t seed, int32_t site, int32_t train,
                           int32_t precision, void* ab, float* s, void* workspace, size_t workspace_bytes, void* stream);
/* segmented softmax + attention pooling (model/backbone.py:82-84): w = softmax over each bag of s; z[b] = sum w v */
ADVMIL_API int advmil_seg_softmax_pool_fwd(const float* s, const void* v /*elem*/, int32_t elem, const int32_t* offsets,
                                const int32_t* offsets_host, int32_t rows, int32_t bags, int32_t width, float* w, float* z,
                                float* mean, void* workspace, size_t workspace_bytes, void* stream);
ADVMIL_API size_t advmil_seg_pool_workspace_bytes(int32_t rows, int32_t bags, int32_t width);

/* Materialises the keep mask (uint8, 1 = keep) that the kernels generate on the fly for one dropout site when no mask is
 * injected: out[rows, width].  site: 1 h, 2 gate tanh, 3 gate sigmoid, 4 rho, 5 MLPs.0 (generator); 11 fc1, 12 GAPool
 * tanh, 13 GAPool sigmoid, 14 fc2 (discriminator).  The two gate sites of a row share one draw keyed by the tanh site.
 * Test / debugging aid: feeding these masks back through the mask_* pointers must reproduce the seeded run exactly. */
ADVMIL_API int advmil_dropout_mask(uint64_t seed, int32_t site, float p, int32_t rows, int32_t width, uint8_t* out, void* stream);

/* fp32 -> bf16 (round to nearest even) of n contiguous elements: how fp32 features enter the ADVMIL_BF16 mode when the
 * loader did not already store them as bf16 */
ADVMIL_API int advmil_cast_f32_to_bf16(const float* in, int64_t n, void* out_bf16, void* stream);

/* ---- region <-> patch index map (tools/big_to_small_patching.py:40-46,59-76) ---------------- */
/* coords_l2 [m,2] int64 (device) -> coords_l1 [16m,2] float64 (device): row 16k+4j+i = c_k + (i*psize, j*psize) */
ADVMIL_API int advmil_region_index_map(const int64_t* coords_l2, int32_t m, int32_t patch_size, int32_t scale, double* coords_l1, void* stream);
/* region id (n / scale^2) and in-region (j,i) of every level-1 row: out [rows,3] int32 */
ADVMIL_API int advmil_region_of_rows(int32_t rows, int32_t scale, int32_t* out, void* stream);

/* ---- losses (loss/utils.py:21-41,182-208) with gradients, over the per-bag scores of one step ---- */
/* which: 0 bce (the reference's non-standard form), 1 hinge, 2 wasserstein.  real_mask[b] != 0 marks bags that
 * contribute a real pair (e==1 && label visible, model_handler.py:373-377).  n_real / n_fake are GLOBAL counts (data
 * parallel: sums over ranks) used as the mean denominators.  Outputs: loss_out[0] += local contribution (caller zeroes). */
ADVMIL_API int advmil_disc_loss(const float* f_real, const float* f_fake, const uint8_t* real_mask, int32_t bags, int32_t which,
                     float n_real, float n_fake, float* loss_out, float* d_real, float* d_fake, void* stream);
/* G loss: recon (norm 0=l1,1=l2; alpha; gamma) over visible bags + coef_gan * (-mean f_fake).  Outputs: losses[3] =
 * {recon, gen, total-without-L1} local contributions, d_pred (recon part) and d_fake. */
ADVMIL_API int advmil_gen_loss(const float* pred, const float* t, const float* e, const uint8_t* visible, const float* f_fake,
                    int32_t bags, float n_visible, float n_fake, float coef_gan, float alpha, float gamma, int32_t norm,
                    float* losses, float* d_pred, float* d_fake, void* stream);

/* ---- fused multi-tensor Adam on a flat parameter buffer (torch.optim.Adam semantics as configured at
 *      model/model_handler.py:104-107, optim/optim_factory.py:25-37): g += wd[i]*p (L2) + l1*sign(p) (loss_reg_l1,
 *      loss/utils.py:6-14), then Adam with bias correction.  wd_mask: per-element uint8 (1 = decayed). -------------- */
ADVMIL_API int advmil_adam_step(float* param, const float* grad, float* m, float* v, const uint8_t* wd_mask, int64_t n,
                     float lr, float beta1, float beta2, float eps, float weight_decay, float l1_coef, int32_t step,
                     float grad_scale, void* stream);
/* sum |p| over a flat buffer (the L1 term's value), out[0] += result */
ADVMIL_API int advmil_abs_sum(const float* p, int64_t n, float* out, void* stream);

/* ---- Harrell's C on the device (replaces eval/cindex.py:106-143 `_estimate_concordance_index` with unit weights, as
 *      reached from concordance_index(y_true, y_pred) :10-40 with estimate = -y_pred).  t, e, pred: [n] fp32 device.
 *      counts (device int64[4], overwritten): concordant, tied_risk, comparable, discordant -- integer exact;
 *      C = (concordant + 0.5 * tied_risk) / comparable.  Pair (i, j) is comparable when e_i and (t_j > t_i or
 *      (t_j == t_i and !e_j)); concordant when pred_j > pred_i (risk = -pred), tied when |pred_i - pred_j| <= tied_tol. */
ADVMIL_API int advmil_cindex_counts(const float* t, const float* e, const float* pred, int32_t n, float tied_tol,
                         int64_t* counts, void* stream);
/* same in float64 (the reference counts in the caller's dtype: float64 inputs are compared as float64) */
ADVMIL_API int advmil_cindex_counts_f64(const double* t, const double* e, const double* pred, int32_t n, double tied_tol,
                                        int64_t* counts, void* stream);

/* ---- fused adversarial step (replaces the bodies of MyHandler._update_disc / _update_gen, model/model_handler.py:349-498,
 *      for one optimiser step of `bags`; the Adam updates and the data-parallel gradient all-reduce stay with the caller,
 *      between the two phases).  One host call per phase instead of ~70: the launch sequence is issued from C.
 *
 *  advmil_adv_step_disc: D.train / G.eval (:355-356).  pred_d = G(x, noise_d) (detached); the real pair (x, t) of every
 *      bag with real_mask and the fake pair (x, pred_d) of every bag run through ONE batched RLIP head pass over a shared
 *      region embedding; D loss (loss/utils.py:182-203) with GLOBAL pair counts; writes all 24 D gradients.
 *  advmil_adv_step_gen:  D.eval / G.train (:432-433), D already updated by the caller.  Re-uses the eval projection of the
 *      disc phase (kept in the workspace: call both phases with the SAME workspace), new dropout draw; G loss = recon +
 *      coef_gan * (-mean f_fake) (:478-484; the L1 term lives in advmil_adam_step); writes all 14 G gradients.
 *  advmil_adv_step_gen_next: one more G update of the same step (gen_updates > 1, model_handler.py:328-335), called after
 *      advmil_adv_step_gen and the caller's G Adam step, on the same workspace.  The caller sets that update's noise_g,
 *      seed_g, g_mask_*, pred_g, f_fake_g and losses.  K1 is recomputed from G's current parameters; D's region embedding
 *      of x is read back from the workspace (advmil_adv_step_gen left it there: D does not change between G updates).   */
typedef struct AdvmilStepArgs {
  const AdvmilGenParams* gen; const AdvmilDiscParams* disc;
  AdvmilGenGrads* gen_grads; AdvmilDiscGrads* disc_grads;
  const AdvmilBags* bags;
  const float* t; const float* e;      /* [bags] time label in [0,1], event indicator */
  const uint8_t* visible;              /* [bags] label_visible_mask (model_handler.py:591-596) */
  const float* noise_d; const float* noise_g;   /* [bags, hid] noise of the last head layer for the two generator passes */
  /* optional injected dropout keep masks (parity tests); NULL = in-kernel generator keyed by the seeds below.
   * d_masks_*: fc1 [2R, d/2] | ga [2R, d] | gs [2R, d] | fc2 [2*bags, d/2] with the FAKE pairs first, then the REAL pairs */
  const uint8_t *g_mask_h, *g_mask_a, *g_mask_b, *g_mask_rho, *g_mask_mlp0;
  const uint8_t *d_mask_fc1, *d_mask_ga, *d_mask_gs, *d_mask_fc2;
  uint64_t seed_d, seed_g;
  float n_real, n_fake, n_visible;     /* GLOBAL counts (sums over data-parallel ranks) */
  int32_t loss_d;                      /* 0 bce (reference form), 1 hinge, 2 wasserstein */
  float coef_gan, recon_alpha, recon_gamma; int32_t recon_norm;
  int32_t precision;
  /* outputs (device) */
  float* losses;      /* [8]: [0] dis_loss, [1] recon, [2] gen, [3] recon + coef_gan*gen; the caller zeroes it per step */
  float* pred_d;      /* [bags] G output of the disc phase */
  float* f_fake_d;    /* [2*bags]: D(x, pred_d) then D(x, t) (the real half is meaningful where real_mask != 0) */
  uint8_t* real_mask; /* [bags] e == 1 && visible */
  float* pred_g;      /* [bags] G output of the gen phase */
  float* f_fake_g;    /* [bags] D(x, pred_g) */
  void* workspace; size_t workspace_bytes;
} AdvmilStepArgs;
ADVMIL_API size_t advmil_adv_step_workspace_bytes(const AdvmilGenParams* gen, const AdvmilDiscParams* disc, int32_t rows,
                                       int32_t bags, int32_t precision);
ADVMIL_API int advmil_adv_step_disc(const AdvmilStepArgs* a, void* stream);
ADVMIL_API int advmil_adv_step_gen(const AdvmilStepArgs* a, void* stream);
ADVMIL_API int advmil_adv_step_gen_next(const AdvmilStepArgs* a, void* stream);

/* ---- the same two-phase step for the DeepAttMISL generator (bcb_mode `cluster`, model/backbone.py:89-123) with the RLIP
 *      discriminator.  The disc phase runs K9 (advmil_cluster_pool_fwd) once and keeps hc, counts and the ReLU keep bits in
 *      the workspace (the fp32 mode keeps relu(x Wphi^T + b) itself); the eval and the train pass of the attention stage
 *      (num_clusters rows per bag, always ADVMIL_FP32) both start from that hc: phis has no dropout and G's parameters do
 *      not change between the phases.  Same semantics, outputs and loss layout as advmil_adv_step_disc / _gen.
 *      base.gen: the attention stage (C = h) and the noise head, Wrho == NULL; base.gen_grads its gradients (dx is set by
 *      the step).  g_mask_h / _a / _b: [bags * num_clusters, h], g_mask_mlp0 as in AdvmilStepArgs.  K9 runs as the
 *      single tcgen05 pass in ADVMIL_TF32 / _TF32X3 / _BF16 wherever that pass covers the shape; elsewhere (ADVMIL_FP32,
 *      and fp32 features with fewer than 128 rows) the step composes advmil_linear_fwd and advmil_segment_mean_by_id_fwd,
 *      reported under the ADVMIL_PROF_PROJ tag instead of the K9 tag.  Every bag length a
 *      multiple of 16, 1 <= num_clusters <= 16, noise0 == 0, ksize-1 discriminator: else ADVMIL_ERR_INVALID.
 *      advmil_adv_step_cluster_gen_next: one more G update, as advmil_adv_step_gen_next; it runs K9 again from the updated
 *      Wphi / bphi (rewriting hc, the counts and the keep bits in the workspace). */
typedef struct AdvmilClusterStepArgs {
  AdvmilStepArgs base;
  const float *Wphi, *bphi;            /* backbone.phis.0 [h, C(,1,1)], [h] */
  float *dWphi, *dbphi;                /* their gradients (written) */
  const int32_t* cid;                  /* [rows] cluster id of every row */
  int32_t num_clusters;
} AdvmilClusterStepArgs;
ADVMIL_API size_t advmil_adv_step_cluster_workspace_bytes(const AdvmilGenParams* gen, const AdvmilDiscParams* disc, int32_t rows,
                                                          int32_t bags, int32_t num_clusters, int32_t precision);
ADVMIL_API int advmil_adv_step_cluster_disc(const AdvmilClusterStepArgs* a, void* stream);
ADVMIL_API int advmil_adv_step_cluster_gen(const AdvmilClusterStepArgs* a, void* stream);
ADVMIL_API int advmil_adv_step_cluster_gen_next(const AdvmilClusterStepArgs* a, void* stream);

/* ---- ESAT backbone: DualTrans_HS (model/backbone.py:171-196) as load_backbone('patch', dims) builds it (:31-35):
 *      AVGPoolPatchEmbedding(C -> d, scale 4, ksize 1; model/backbone_utils.py:129-168) -> optional sincos positional
 *      embedding (:79-99) -> one post-norm nn.TransformerEncoderLayer(d, nhead, dim_feedforward = ff, dropout p, relu)
 *      (make_transformer_layer, model/backbone_utils.py:112-127) -> GAPool(d, d) (:31-56), followed by the Generator's
 *      noise head (model/GANSurv.py:32-49) when `head` is given.  Parameter names are the reference state_dict's. ---- */
typedef struct AdvmilEsatParams {
  const float *Wc, *bc, *ln_g, *ln_b;     /* patch_embedding_layer.conv [d,C(,1,1)],[d]; .norm [d],[d] */
  const float *Win, *bin;                 /* patch_encoder_layer.layers.0.self_attn.in_proj_weight [3d,d], in_proj_bias [3d] */
  const float *Wout, *bout;               /* ...self_attn.out_proj [d,d],[d] */
  const float *W1, *b1, *W2, *b2;         /* ...linear1 [ff,d],[ff]; linear2 [d,ff],[d] */
  const float *n1_g, *n1_b, *n2_g, *n2_b; /* ...norm1, norm2 [d] */
  const float *Pa_w, *Pa_b;               /* pool.fc1.0   [d,d],[d] (tanh branch)    */
  const float *Ps_w, *Ps_b;               /* pool.score.0 [d,d],[d] (sigmoid branch) */
  const float *Pc_w, *Pc_b;               /* pool.fc2     [1,d],[1] */
  int32_t C, d, ff, nhead;
  float p;                                /* dropout of the encoder layer (attention probabilities, both residual branches,
                                             feed-forward) and of GAPool */
  float ln_eps;
} AdvmilEsatParams;

typedef struct AdvmilEsatGrads {          /* same tensors, written (not accumulated) */
  float *Wc, *bc, *ln_g, *ln_b, *Win, *bin, *Wout, *bout, *W1, *b1, *W2, *b2, *n1_g, *n1_b, *n2_g, *n2_b,
        *Pa_w, *Pa_b, *Ps_w, *Ps_b, *Pc_w, *Pc_b;
} AdvmilEsatGrads;

typedef struct AdvmilEsatActs {           /* caller-allocated; R = rows / 16 region rows, packed like the bags */
  void* y_pre;    /* T [rows,d] pre-LayerNorm projection */
  float* emb;     /* [R,d] region embedding (+ pe) */
  float* qkv;     /* [R,3d] */
  float* lse;     /* [nhead,R] log-sum-exp of the attention logits */
  float* ctx;     /* [R,d] attention output before out_proj */
  float* s1;      /* [R,d] emb + dropout1(out_proj(ctx)) */
  float* x1;      /* [R,d] norm1(s1) */
  float* f;       /* [R,ff] dropout(relu(linear1(x1))) */
  float* s2;      /* [R,d] x1 + dropout2(linear2(f)) */
  float* x2;      /* [R,d] norm2(s2): the encoder output that GAPool pools */
  float* ab;      /* [R,abw] GAPool gate activations (advmil_gate_packed_width(d)) */
  float* rep;     /* [R] GAPool logits */
  float* attn;    /* [R] GAPool softmax weights */
  float* H;       /* [bags,d] backbone output */
  float* H1;      /* [bags,hid] head (NULL without head) */
  float* pre;     /* [bags] */
  float* pred;    /* [bags] */
  const float* pe;       /* optional [R,d] positional embedding (advmil_sincos_pe), added to emb */
  const float* noise0;   /* [bags,d] or NULL */
  const float* noise1;   /* [bags,hid] or NULL */
  /* optional injected keep masks: attention probabilities per bag [nhead, R_b, R_b] at mask_attn_off[bag] (int64 element
   * offsets, device); sa / ff2 / ga / gs [R,d]; ff1 [R,ff]; mlp0 [bags,hid] */
  const uint8_t* mask_attn; const int64_t* mask_attn_off;
  const uint8_t *mask_sa, *mask_ff1, *mask_ff2, *mask_ga, *mask_gs, *mask_mlp0;
  uint64_t seed;
  int32_t train, precision;
  void* workspace; size_t workspace_bytes;
  int32_t emb_ready;  /* != 0: y_pre and emb already hold the patch embedding of these bags under the current conv / norm
                         parameters (written by an earlier call, e.g. the eval pass of the D step): the projection and its
                         LayerNorm stream are skipped (the embedding has no dropout, so eval and train passes share it) */
} AdvmilEsatActs;

ADVMIL_API size_t advmil_esat_workspace_bytes(const AdvmilEsatParams* p, const AdvmilGenParams* head, int32_t rows, int32_t bags,
                                   int32_t backward);
/* head == NULL: backbone only (DualTrans_HS.forward), result in acts->H.  head: AdvmilGenParams with Wrho == NULL,
 * h == o == d and the MLPs tensors (W0, b0, Wl, bl, hid, noise0/1, out_scale, p_head); result in acts->pred. */
ADVMIL_API int advmil_esat_fwd(const AdvmilEsatParams* p, const AdvmilGenParams* head, const AdvmilBags* bags, AdvmilEsatActs* acts,
                    void* stream);
/* d_out: dL/dpred [bags] with a head, dL/dH [bags,d] without.  head_grads: W0, b0, Wl, bl are written. */
ADVMIL_API int advmil_esat_bwd(const AdvmilEsatParams* p, const AdvmilGenParams* head, const AdvmilBags* bags, const AdvmilEsatActs* acts,
                    const float* d_out, AdvmilEsatGrads* grads, AdvmilGenGrads* head_grads, void* stream);
/* compute_pe (model/backbone_utils.py:90-99): coord [R,2] int64 region coordinates (packed like the regions), made
 * relative to each bag's minimum; omega [d/4] = 1 / 10000^(k / (d/4 - 1)) as the reference computes it; pe [R,d]. */
ADVMIL_API int advmil_sincos_pe(const int64_t* coord, const int32_t* offsets /* bag row offsets [bags+1], device */, int32_t bags,
                     int32_t d, const float* omega, float* pe, void* workspace, size_t workspace_bytes, void* stream);

/* ---- the fused adversarial step for the ESAT generator (the launch sequence of step.ModuleAdvStep issued from C; same
 *      semantics, outputs and loss layout as advmil_adv_step_disc / _gen; in-kernel dropout only).  pe: optional [R, d]
 *      positional embedding (advmil_sincos_pe).  The two calls share one workspace: the D phase's eval pass leaves the patch
 *      embedding of the bags in it for the G phase's train pass.  advmil_adv_step_esat_gen_next: one more G update, as
 *      advmil_adv_step_gen_next; it recomputes the patch embedding from the updated parameters. */
typedef struct AdvmilEsatStepArgs {
  const AdvmilEsatParams* esat; const AdvmilGenParams* head; const AdvmilDiscParams* disc;
  AdvmilEsatGrads* esat_grads; AdvmilGenGrads* head_grads; AdvmilDiscGrads* disc_grads;
  const AdvmilBags* bags;
  const float* t; const float* e; const uint8_t* visible;
  const float* noise_d; const float* noise_g;
  const float* pe;
  uint64_t seed_d, seed_g;
  float n_real, n_fake, n_visible;
  int32_t loss_d;
  float coef_gan, recon_alpha, recon_gamma; int32_t recon_norm;
  int32_t precision;
  float* losses; float* pred_d; float* f_fake_d; uint8_t* real_mask; float* pred_g; float* f_fake_g;
  void* workspace; size_t workspace_bytes;
} AdvmilEsatStepArgs;
ADVMIL_API size_t advmil_adv_step_esat_workspace_bytes(const AdvmilEsatParams* esat, const AdvmilGenParams* head, const AdvmilDiscParams* disc,
                                            int32_t rows, int32_t bags, int32_t precision);
ADVMIL_API int advmil_adv_step_esat_disc(const AdvmilEsatStepArgs* a, void* stream);
ADVMIL_API int advmil_adv_step_esat_gen(const AdvmilEsatStepArgs* a, void* stream);
ADVMIL_API int advmil_adv_step_esat_gen_next(const AdvmilEsatStepArgs* a, void* stream);

/* ---- ESAT self-attention, stage level (nn.MultiheadAttention inside the encoder layer, model/backbone_utils.py:112-127):
 *      qkv [R, 3d] fp32 (the packed in-projection), region offsets [bags+1] on the device and on the host, -> ctx [R, d],
 *      lse [heads, R].  Dropout on the probabilities by the counter generator (seed, train, p_drop) or injected per-bag masks
 *      [heads, Rb, Rb] at mask_off[bag].  precision FP32 / TF32X3 = FFMA kernels, TF32 / BF16 = tensor-core kernels (forward on
 *      tcgen05 for head widths 16/32/48/64).  Used by the kernel unit tests; the model goes through advmil_esat_fwd/bwd. */
ADVMIL_API int advmil_mha_fwd(const float* qkv, const int32_t* region_offsets, const int32_t* region_offsets_host, int32_t bags,
                   int32_t d, int32_t heads, float p_drop, uint64_t seed, int32_t train, const uint8_t* mask,
                   const int64_t* mask_off, int32_t precision, float* ctx, float* lse, void* stream);
ADVMIL_API int advmil_mha_bwd(const float* qkv, const float* ctx, const float* d_ctx, const float* lse, const int32_t* region_offsets,
                   const int32_t* region_offsets_host, int32_t bags, int32_t d, int32_t heads, float p_drop, uint64_t seed,
                   int32_t train, const uint8_t* mask, const int64_t* mask_off, int32_t precision, float* d_qkv,
                   float* scratch /* [heads * R] */, void* stream);

/* ---- lossless 12-bit transport format of bf16 features (the packed loader that replaces dataset/PatchWSI.py:65-94 +
 *      model_handler.py:315-316's `.cuda()`): lo[n] = sign<<7 | mantissa, hi[n/2] = two 4-bit exponent codes, table16 (HOST
 *      pointer, code -> exponent byte, code 15 = escape), escapes (element index, exponent byte).  Decodes n elements
 *      (n % 8 == 0) into out_bf16 exactly; see advmil_b200/dataset/codec.py for the encoder. */
ADVMIL_API int advmil_bf16p12_decode(const uint8_t* lo, const uint8_t* hi, const uint8_t* table16_host, const int32_t* esc_idx,
                          const uint8_t* esc_exp, int64_t n, int32_t n_esc, void* out_bf16, void* stream);

/* ---- "vl": the same transport format with the exponent plane entropy-coded (canonical Huffman, <= 8 bits, LSB-first; ~10.9
 *      instead of 12 bits per element on Gaussian-like features).  Elements are dealt to 32 sub-streams per super-block of 4096
 *      (lane t owns elements r*128 + 4t + {0..3}) so that the decoder's loads and stores stay coalesced: lo[n] as in p12,
 *      stream[] uint32 words (+2 guard words), sbase[n/4096] word offset of a super-block, loff[n/128] word offset of a
 *      sub-stream inside its super-block, tables (HOST pointers: symbol -> exponent byte / code length / LSB-first code), escapes
 *      as in p12.  n % 4096 == 0, n < 2^31.
 *      advmil_bf16vl_encode and advmil_bf16vl_decode_host are HOST functions (packing time / tests; no GPU needed):
 *      x = n bf16 words; stream_cap_words >= n/4 + n/128 + 2 always suffices; returns the words and escapes written. */
ADVMIL_API int advmil_bf16vl_encode(const uint16_t* x, int64_t n, uint8_t* lo, uint32_t* stream, int64_t stream_cap_words, uint32_t* sbase,
                         uint16_t* loff, uint8_t* tab_exp16, uint8_t* tab_len16, uint16_t* tab_code16, int32_t* esc_idx,
                         uint8_t* esc_exp, int64_t esc_cap, int64_t* stream_words, int64_t* n_esc);
/* tables from an exponent histogram (hist256[e] = number of elements with exponent byte e), e.g. of a whole packed file, and
 * the encoder with GIVEN tables: every bag of a file then shares one table and the streams of any selection of bags
 * concatenate into a step without re-encoding (advmil_b200/dataset/packed_file.py, transport "vl") */
ADVMIL_API int advmil_bf16vl_tables(const uint64_t* hist256, uint8_t* tab_exp16, uint8_t* tab_len16, uint16_t* tab_code16);
ADVMIL_API int advmil_bf16vl_encode_with_tables(const uint16_t* x, int64_t n, uint8_t* lo, uint32_t* stream, int64_t stream_cap_words,
                                     uint32_t* sbase, uint16_t* loff, const uint8_t* tab_exp16, const uint8_t* tab_len16,
                                     const uint16_t* tab_code16, int32_t* esc_idx, uint8_t* esc_exp, int64_t esc_cap,
                                     int64_t* stream_words, int64_t* n_esc);
ADVMIL_API int advmil_bf16vl_decode_host(const uint8_t* lo, const uint32_t* stream, const uint32_t* sbase, const uint16_t* loff,
                              const uint8_t* tab_exp16, const uint8_t* tab_len16, const uint16_t* tab_code16,
                              const int32_t* esc_idx, const uint8_t* esc_exp, int64_t n, int64_t n_esc, uint16_t* out);
ADVMIL_API int advmil_bf16vl_decode(const uint8_t* lo, const uint32_t* stream, const uint32_t* sbase, const uint16_t* loff,
                         const uint8_t* tab_exp16_host, const uint8_t* tab_len16_host, const uint16_t* tab_code16_host,
                         const int32_t* esc_idx, const uint8_t* esc_exp, int64_t n, int32_t n_esc, void* out_bf16, void* cuda_stream);

#ifdef __cplusplus
}
#endif
#endif /* ADVMIL_B200_H_ */
