// C-ABI composites of the ESAT backbone (DualTrans_HS, reference model/backbone.py:171-196; encoder layer built by
// make_transformer_layer, model/backbone_utils.py:112-127; GAPool :31-56; noise head model/GANSurv.py:32-49).
// The N-row projection runs on the GEMM engines in the caller's precision mode; everything after the region mean works
// on rows/16 region rows in fp32 (contractions on tcgen05 kind::tf32 outside the exact-fp32 mode, like the RLIP head).
#include <mutex>
#include <vector>
#include "stages.cuh"

namespace advmil {

__global__ void region_offsets_kernel(const int32_t* __restrict__ offs, int n, int32_t* __restrict__ out) {
  pdl_prologue();
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = offs[i] / 16;
}

#define ESAT_TAKE(var, type, count)                                                                           \
  type* var = ws.take<type>(count);                                                                           \
  if (!var) { set_error("%s: workspace too small (have %zu bytes)", __func__, ws.cap); return ADVMIL_ERR_WORKSPACE; }

// ---- side stream of the backward pass ------------------------------------------------------------------------------------
// Each region-level layer's backward is three independent pieces of work once dY exists: dX = dY W (the chain the next layer
// waits for), dW = dY^T X and db = colsum(dY).  They are all 10-30 us kernels on 16 k region rows that leave most of the chip
// idle, so the weight / bias gradients can run on a second stream beside the data-gradient chain.  The C-fused step
// (advmil_adv_step_esat_gen) requests it: 3.40 -> 3.32 ms per step.  The module path does not: the generator's forward +
// backward alone gains 4 % (2.22 -> 2.13 ms), but the Python-composed ModuleAdvStep is within a few percent of being
// host-bound and the six extra event record / wait pairs per backward cost it more host time than the overlap saves
// (4.42 -> 4.60 ms per step).
struct EsatSide {
  cudaStream_t st = nullptr;
  cudaEvent_t fork = nullptr, join = nullptr;
};
static EsatSide g_esat_side[64];
static std::mutex g_esat_mu;
static thread_local int g_esat_overlap_request = 0;      // set by the C-fused step around its backward call
void esat_request_overlap(int on) { g_esat_overlap_request = on; }
static int esat_side_get(EsatSide** out) {
  *out = nullptr;
  if (!g_esat_overlap_request) return ADVMIL_OK;
  int dev = 0;
  ADVMIL_CHECK_CUDA(cudaGetDevice(&dev));
  if (dev < 0 || dev >= 64) return ADVMIL_OK;
  EsatSide& s = g_esat_side[dev];
  if (!s.st) {
    ADVMIL_CHECK_CUDA(cudaStreamCreateWithFlags(&s.st, cudaStreamNonBlocking));
    ADVMIL_CHECK_CUDA(cudaEventCreateWithFlags(&s.fork, cudaEventDisableTiming));
    ADVMIL_CHECK_CUDA(cudaEventCreateWithFlags(&s.join, cudaEventDisableTiming));
  }
  *out = &s;
  return ADVMIL_OK;
}

static int esat_check(const AdvmilEsatParams* p, const AdvmilGenParams* head, const AdvmilBags* b, int precision) {
  ADVMIL_REQUIRE(p && b && b->x && b->offsets && b->offsets_host, "esat: null argument");
  ADVMIL_REQUIRE(p->Wc && p->Win && p->Wout && p->W1 && p->W2 && p->n1_g && p->n2_g && p->Pa_w && p->Ps_w && p->Pc_w, "esat: missing parameter tensor");
  ADVMIL_REQUIRE(precision >= ADVMIL_FP32 && precision <= ADVMIL_BF16, "unknown precision mode %d", precision);
  ADVMIL_REQUIRE(b->elem == elem_of_precision(precision), "bags: x element type %d does not match precision mode %d", b->elem, precision);
  ADVMIL_REQUIRE(b->C == p->C, "bags: feature width %d != model input width %d", b->C, p->C);
  ADVMIL_REQUIRE(b->bags > 0 && b->rows > 0 && b->offsets_host[0] == 0 && b->offsets_host[b->bags] == b->rows, "bags: offsets must span [0, rows]");
  ADVMIL_REQUIRE(p->nhead > 0 && p->d % p->nhead == 0 && (p->d / p->nhead) % 4 == 0, "esat: d %d / nhead %d must give a head width that is a multiple of 4", p->d, p->nhead);
  for (int i = 0; i < b->bags; ++i) {
    const int len = b->offsets_host[i + 1] - b->offsets_host[i];
    ADVMIL_REQUIRE(len > 0 && len % 16 == 0, "bags: bag %d has %d rows, not a positive multiple of 16 (model/backbone_utils.py:65)", i, len);
  }
  if (head) ADVMIL_REQUIRE(head->Wrho == nullptr && head->h == p->d && head->o == p->d && head->W0 && head->Wl,
                           "esat: the head must be AdvmilGenParams with Wrho == NULL, h == o == d and the MLPs tensors");
  return ADVMIL_OK;
}

struct EsatDrops { Drop att, sa, ff1, ff2, ga, gs, mlp0, none; };
static EsatDrops esat_drops(const AdvmilEsatParams* p, const AdvmilGenParams* head, const AdvmilEsatActs* a) {
  EsatDrops d;
  d.att = Drop::make(nullptr, a->seed, SITE_ATT, p->p, a->train, 0);
  d.sa = Drop::make(a->mask_sa, a->seed, SITE_SA, p->p, a->train, p->d);
  d.ff1 = Drop::make(a->mask_ff1, a->seed, SITE_FF1, p->p, a->train, p->ff);
  d.ff2 = Drop::make(a->mask_ff2, a->seed, SITE_FF2, p->p, a->train, p->d);
  d.ga = Drop::make(a->mask_ga, a->seed, SITE_GA, p->p, a->train, p->d);
  d.gs = Drop::make(a->mask_gs, a->seed, SITE_GS, p->p, a->train, p->d);
  Drop::pair_gate(d.ga, d.gs);
  d.mlp0 = Drop::make(a->mask_mlp0, a->seed, SITE_MLP0, head ? head->p_head : 0.f, a->train, head ? head->hid : 0);
  d.none = Drop::make(nullptr, 0, 0, 0.f, 0, 0);
  return d;
}

static int region_offsets(const AdvmilBags* bags, std::vector<int32_t>& host, int32_t* dev, cudaStream_t st) {
  host.resize(bags->bags + 1);
  for (int i = 0; i <= bags->bags; ++i) host[i] = bags->offsets_host[i] / 16;
  launch_k(region_offsets_kernel, dim3(cdiv(bags->bags + 1, 128)), dim3(128), 0, st, bags->offsets, bags->bags + 1, dev);
  ADVMIL_CHECK_LAUNCH();
  return ADVMIL_OK;
}

}  // namespace advmil

using namespace advmil;

extern "C" size_t advmil_esat_workspace_bytes(const AdvmilEsatParams* p, const AdvmilGenParams* head, int32_t rows, int32_t bags,
                                              int32_t backward) {
  const size_t d = p->d, ff = p->ff, R = rows / 16, abw = gate_width(p->d), nb = bags;
  size_t f = 64 + abw * d + abw + (abw / 128) * R + seg_pool_ws_floats((int)R, bags, p->d);   // ro, Wp, bp, score parts, pool scratch
  if (backward) {
    const size_t hid = head ? head->hid : 0;
    f += nb * (2 * d + hid + 1) + R * abw + abw * d + abw + pool_gate_ws_floats((int)R, bags, p->d);
    size_t bw = bwd_weight_ws_floats((int)R, (int)abw, p->d);
    bw = bw > bwd_weight_ws_floats((int)R, p->d, p->ff) ? bw : bwd_weight_ws_floats((int)R, p->d, p->ff);
    bw = bw > bwd_weight_ws_floats((int)R, p->ff, p->d) ? bw : bwd_weight_ws_floats((int)R, p->ff, p->d);
    bw = bw > bwd_weight_ws_floats((int)R, 3 * p->d, p->d) ? bw : bwd_weight_ws_floats((int)R, 3 * p->d, p->d);
    bw = bw > bwd_weight_ws_floats(rows, p->d, p->C) ? bw : bwd_weight_ws_floats(rows, p->d, p->C);
    f += bw + (size_t)row_chunks((int)R) * 3 * (d > ff ? d : ff) + (size_t)esat_ln_bwd_ctas((int)R) * 3 * d;
    f += R * (8 * d + ff + 3 * d) + (size_t)p->nhead * R + (size_t)rows * d;   // region-level gradients, Dq, d_y (as fp32 upper bound)
  }
  return f * sizeof(float) + 64 * 256;
}

extern "C" int advmil_esat_fwd(const AdvmilEsatParams* p, const AdvmilGenParams* head, const AdvmilBags* bags, AdvmilEsatActs* a,
                               void* stream) {
  ADVMIL_REQUIRE(a, "esat_fwd: null argument");
  ADVMIL_TRY(esat_check(p, head, bags, a->precision));
  ADVMIL_REQUIRE(a->y_pre && a->emb && a->qkv && a->lse && a->ctx && a->s1 && a->x1 && a->f && a->s2 && a->x2 && a->ab && a->rep &&
                 a->attn && a->H, "esat_fwd: missing activation buffers");
  ADVMIL_REQUIRE(!head || (a->H1 && a->pre && a->pred), "esat_fwd: missing head buffers");
  cudaStream_t st = (cudaStream_t)stream;
  const int rows = bags->rows, nb = bags->bags, R = rows / 16, d = p->d, ff = p->ff, C = p->C;
  const int abw = gate_width(d);
  const int dt = elem_of_precision(a->precision);
  const int rp = region_precision(a->precision, false);      // region-level contractions
  const EsatDrops dr = esat_drops(p, head, a);
  Workspace ws(a->workspace, a->workspace_bytes);
  ESAT_TAKE(ro, int32_t, nb + 1);
  ESAT_TAKE(Wp, float, (size_t)abw * d);
  ESAT_TAKE(bp, float, abw);
  ESAT_TAKE(part, float, (size_t)(abw / 128) * R);
  ESAT_TAKE(poolws, float, seg_pool_ws_floats(R, nb, d));
  std::vector<int32_t> ro_host;
  ADVMIL_TRY(region_offsets(bags, ro_host, ro, st));
  // patch embedding (model/backbone_utils.py:158-168) + positional embedding (model/backbone.py:192-194)
  if (!a->emb_ready) {
    ProfScope ps(PROF_EMBED, st);
    ADVMIL_TRY(linear_fwd(bags->x, p->Wc, p->bc, rows, C, d, 0, dr.none, a->y_pre, a->precision, st));
    ADVMIL_TRY(ln_relu_mean16_fwd(a->y_pre, p->ln_g, p->ln_b, rows, d, p->ln_eps, a->pe, a->emb, dt, st));
  }
  ProfScope ps(PROF_HEAD_FWD, st);
  // encoder layer, post-norm
  ADVMIL_TRY(linear_fwd(a->emb, p->Win, p->bin, R, d, 3 * d, 0, dr.none, a->qkv, rp, st));
  { ProfScope pa(PROF_ATTN_FWD, st);
    ADVMIL_TRY(mha_fwd(a->qkv, ro, ro_host.data(), nb, R, d, p->nhead, dr.att, a->mask_attn, a->mask_attn_off, a->ctx, a->lse, attention_precision(a->precision), st)); }
  ADVMIL_TRY(linear_fwd(a->ctx, p->Wout, p->bout, R, d, d, 0, dr.sa, a->s1, rp, st));
  ADVMIL_TRY(add_ln_fwd(a->emb, a->s1, p->n1_g, p->n1_b, R, d, p->ln_eps, a->x1, st));
  ADVMIL_TRY(linear_fwd(a->x1, p->W1, p->b1, R, d, ff, 1, dr.ff1, a->f, rp, st));
  ADVMIL_TRY(linear_fwd(a->f, p->W2, p->b2, R, ff, d, 0, dr.ff2, a->s2, rp, st));
  ADVMIL_TRY(add_ln_fwd(a->x1, a->s2, p->n2_g, p->n2_b, R, d, p->ln_eps, a->x2, st));
  // GAPool over the regions of each bag (model/backbone_utils.py:47-56)
  ADVMIL_TRY(gate_pack_weights(p->Pa_w, p->Pa_b, p->Ps_w, p->Ps_b, d, d, Wp, bp, st));
  ADVMIL_TRY(gated_score_fwd(a->x2, Wp, bp, p->Pc_w, p->Pc_b, R, d, d, dr.ga, dr.gs, a->ab, nullptr, part, rp, st));
  ADVMIL_TRY(seg_softmax_pool_fwd(a->rep, part, abw / 128, p->Pc_b, a->x2, ELEM_F32, ro, ro_host.data(), R, nb, d, a->attn, a->H,
                                  nullptr, poolws, st));
  if (head)
    ADVMIL_TRY(gen_head_fwd(*head, a->H, a->noise0, a->noise1, nb, 1, dr.none, dr.mlp0, nullptr, a->H1, a->pre, a->pred, st));
  return ADVMIL_OK;
}

extern "C" int advmil_esat_bwd(const AdvmilEsatParams* p, const AdvmilGenParams* head, const AdvmilBags* bags, const AdvmilEsatActs* a,
                               const float* d_out, AdvmilEsatGrads* g, AdvmilGenGrads* hg, void* stream) {
  ADVMIL_REQUIRE(a && d_out && g, "esat_bwd: null argument");
  ADVMIL_TRY(esat_check(p, head, bags, a->precision));
  ADVMIL_REQUIRE(!head || hg, "esat_bwd: head gradients missing");
  cudaStream_t st = (cudaStream_t)stream;
  std::lock_guard<std::mutex> side_lock(g_esat_mu);
  EsatSide* side = nullptr;
  ADVMIL_TRY(esat_side_get(&side));
  cudaStream_t sw = side ? side->st : st;                 // stream of the weight / bias gradients
  // everything issued on `st` so far is visible to the side stream from here on
  auto fork = [&]() -> int {
    if (!side) return ADVMIL_OK;
    ADVMIL_CHECK_CUDA(cudaEventRecord(side->fork, st));
    ADVMIL_CHECK_CUDA(cudaStreamWaitEvent(side->st, side->fork, 0));
    return ADVMIL_OK;
  };
  const int rows = bags->rows, nb = bags->bags, R = rows / 16, d = p->d, ff = p->ff, C = p->C;
  const int abw = gate_width(d);
  const int dt = elem_of_precision(a->precision);
  const int rp = region_precision(a->precision, false);
  const EsatDrops dr = esat_drops(p, head, a);
  const float ik = dr.sa.inv_keep;
  Workspace ws(a->workspace, a->workspace_bytes);
  ESAT_TAKE(ro, int32_t, nb + 1);
  ESAT_TAKE(Wp, float, (size_t)abw * d);
  ESAT_TAKE(bp, float, abw);
  std::vector<int32_t> ro_host;
  ADVMIL_TRY(region_offsets(bags, ro_host, ro, st));
  ProfScope ps(PROF_HEAD_BWD, st);
  // ---- noise head ----
  const float* dH = d_out;
  if (head) {
    const int hid = head->hid;
    ESAT_TAKE(dz, float, (size_t)nb * d);
    ESAT_TAKE(dHpre, float, (size_t)nb * d);
    ESAT_TAKE(dH1pre, float, (size_t)nb * hid);
    ESAT_TAKE(dpre, float, nb);
    ADVMIL_TRY(gen_head_bwd(*head, d_out, a->H, a->H1, a->pred, nb, 1.f, dr.mlp0.inv_keep, dz, dHpre, dH1pre, dpre, st));
    OuterProb op[2];
    op[0] = OuterProb{dpre, a->H1, hid, a->noise1, head->noise1 ? hid : 0, 1, hg->Wl, hg->bl};
    op[1] = OuterProb{dH1pre, a->H, d, a->noise0, head->noise0 ? d : 0, hid, hg->W0, hg->b0};
    ADVMIL_TRY(outer_sum_multi(op, 2, nb, 0, st));
    dH = dz;
  }
  // ---- GAPool ----
  ESAT_TAKE(dAB, float, (size_t)R * abw);
  ESAT_TAKE(dWp, float, (size_t)abw * d);
  ESAT_TAKE(dbp, float, abw);
  ESAT_TAKE(pgws, float, pool_gate_ws_floats(R, nb, d));
  size_t bw = bwd_weight_ws_floats(R, abw, d);
  bw = max(bw, bwd_weight_ws_floats(R, d, ff)); bw = max(bw, bwd_weight_ws_floats(R, ff, d));
  bw = max(bw, bwd_weight_ws_floats(R, 3 * d, d)); bw = max(bw, bwd_weight_ws_floats(rows, d, C));
  ESAT_TAKE(bwws, float, bw);
  ESAT_TAKE(csws, float, (size_t)row_chunks(R) * 3 * max(d, ff));
  ESAT_TAKE(lnws, float, (size_t)esat_ln_bwd_ctas(R) * 3 * d);
  ESAT_TAKE(d_x2, float, (size_t)R * d);
  ESAT_TAKE(d_s2, float, (size_t)R * d);
  ESAT_TAKE(g2, float, (size_t)R * d);
  ESAT_TAKE(d_fpre, float, (size_t)R * ff);
  ESAT_TAKE(d_x1, float, (size_t)R * d);
  ESAT_TAKE(d_s1, float, (size_t)R * d);
  ESAT_TAKE(gsa, float, (size_t)R * d);
  ESAT_TAKE(d_ctx, float, (size_t)R * d);
  ESAT_TAKE(d_qkv, float, (size_t)R * 3 * d);
  ESAT_TAKE(Dq, float, (size_t)p->nhead * R);
  ESAT_TAKE(d_emb, float, (size_t)R * d);
  ESAT_TAKE(d_y, char, (size_t)rows * d * elem_bytes(dt));
  ADVMIL_TRY(gate_pack_weights(p->Pa_w, p->Pa_b, p->Ps_w, p->Ps_b, d, d, Wp, bp, st));
  ADVMIL_TRY(pool_gate_bwd(a->x2, a->attn, a->H, dH, a->ab, p->Pc_w, ro, R, nb, d, d, dr.ga, dr.gs, dAB, g->Pc_w, g->Pc_b, dbp, 0, pgws,
                           ELEM_F32, st));
  { BwdDataExtras ex;
    ex.w = a->attn; ex.dz = dH; ex.offsets = ro; ex.bags = nb;
    ADVMIL_TRY(bwd_data(dAB, Wp, R, abw, d, d_x2, ex, rp, st)); }
  ADVMIL_TRY(fork());
  ADVMIL_TRY(bwd_weight(dAB, a->x2, R, abw, d, dWp, 0, bwws, rp, sw));
  ADVMIL_TRY(gate_unpack_grads(dWp, dbp, d, d, g->Pa_w, g->Pa_b, g->Ps_w, g->Ps_b, 0, sw));
  // ---- norm2 and the feed-forward block ----
  ADVMIL_TRY(add_ln_bwd(a->s2, p->n2_g, d_x2, R, d, p->ln_eps, d_s2, g->n2_g, g->n2_b, lnws, st));
  ADVMIL_TRY(apply_dropout(d_s2, R, d, dr.ff2, g2, ELEM_F32, st));
  ADVMIL_TRY(fork());
  ADVMIL_TRY(bwd_weight(g2, a->f, R, d, ff, g->W2, 0, bwws, rp, sw));
  ADVMIL_TRY(colsum(g2, ELEM_F32, R, d, d, g->b2, 0, csws, sw));
  { BwdDataExtras ex;
    ex.relu_src = a->f; ex.ld_src = ff; ex.inv_keep = ik;
    ADVMIL_TRY(bwd_data(g2, p->W2, R, d, ff, d_fpre, ex, rp, st)); }
  ADVMIL_TRY(fork());
  ADVMIL_TRY(bwd_weight(d_fpre, a->x1, R, ff, d, g->W1, 0, bwws, rp, sw));
  ADVMIL_TRY(colsum(d_fpre, ELEM_F32, R, ff, ff, g->b1, 0, csws, sw));
  { BwdDataExtras ex;
    ADVMIL_TRY(bwd_data(d_fpre, p->W1, R, ff, d, d_x1, ex, rp, st)); }
  ADVMIL_TRY(add_rows(d_x1, d_s2, (size_t)R * d, st));                          // residual branch of norm2
  // ---- norm1 and self-attention ----
  ADVMIL_TRY(add_ln_bwd(a->s1, p->n1_g, d_x1, R, d, p->ln_eps, d_s1, g->n1_g, g->n1_b, lnws, st));
  ADVMIL_TRY(apply_dropout(d_s1, R, d, dr.sa, gsa, ELEM_F32, st));
  ADVMIL_TRY(fork());
  ADVMIL_TRY(bwd_weight(gsa, a->ctx, R, d, d, g->Wout, 0, bwws, rp, sw));
  ADVMIL_TRY(colsum(gsa, ELEM_F32, R, d, d, g->bout, 0, csws, sw));
  { BwdDataExtras ex;
    ADVMIL_TRY(bwd_data(gsa, p->Wout, R, d, d, d_ctx, ex, rp, st)); }
  { ProfScope pa(PROF_ATTN_BWD, st);
    ADVMIL_TRY(mha_bwd(a->qkv, a->ctx, d_ctx, a->lse, ro, ro_host.data(), nb, R, d, p->nhead, dr.att, a->mask_attn, a->mask_attn_off,
                       d_qkv, Dq, attention_precision(a->precision), st)); }
  ADVMIL_TRY(fork());
  ADVMIL_TRY(bwd_weight(d_qkv, a->emb, R, 3 * d, d, g->Win, 0, bwws, rp, sw));
  ADVMIL_TRY(colsum(d_qkv, ELEM_F32, R, 3 * d, 3 * d, g->bin, 0, csws, sw));
  { BwdDataExtras ex;
    ADVMIL_TRY(bwd_data(d_qkv, p->Win, R, 3 * d, d, d_emb, ex, rp, st)); }
  ADVMIL_TRY(add_rows(d_emb, d_s1, (size_t)R * d, st));                         // residual branch of norm1
  // ---- patch embedding ----
  { ProfScope ps2(PROF_LN_BWD, st);
    ADVMIL_TRY(ln_relu_mean16_bwd(a->y_pre, d_emb, p->ln_g, p->ln_b, rows, d, p->ln_eps, d_y, g->ln_g, g->ln_b, g->bc, lnws, dt, st)); }
  if (side) {      // join: the weight-gradient scratch is reused below, and the caller's stream owns every result after the call
    ADVMIL_CHECK_CUDA(cudaEventRecord(side->join, side->st));
    ADVMIL_CHECK_CUDA(cudaStreamWaitEvent(st, side->join, 0));
  }
  { ProfScope ps2(PROF_BWD_W_EMBED, st);
    ADVMIL_TRY(bwd_weight(d_y, bags->x, rows, d, C, g->Wc, 0, bwws, a->precision, st)); }
  return ADVMIL_OK;
}

extern "C" int advmil_sincos_pe(const int64_t* coord, const int32_t* offsets, int32_t bags, int32_t d, const float* omega, float* pe,
                                void* workspace, size_t workspace_bytes, void* stream) {
  ADVMIL_REQUIRE(coord && offsets && omega && pe && bags > 0, "sincos_pe: bad arguments");
  cudaStream_t st = (cudaStream_t)stream;
  Workspace ws(workspace, workspace_bytes);
  ESAT_TAKE(ro, int32_t, bags + 1);
  launch_k(region_offsets_kernel, dim3(cdiv(bags + 1, 128)), dim3(128), 0, st, offsets, bags + 1, ro);
  ADVMIL_CHECK_LAUNCH();
  return sincos_pe(coord, ro, bags, d, omega, pe, st);
}

// ---- stage-level entry points of the self-attention (kernel unit tests: every head width / ragged region counts) ----------
extern "C" int advmil_mha_fwd(const float* qkv, const int32_t* region_offsets, const int32_t* region_offsets_host, int32_t bags,
                              int32_t d, int32_t heads, float p_drop, uint64_t seed, int32_t train, const uint8_t* mask,
                              const int64_t* mask_off, int32_t precision, float* ctx, float* lse, void* stream) {
  ADVMIL_REQUIRE(qkv && region_offsets && region_offsets_host && ctx && lse && bags > 0 && heads > 0 && d % heads == 0,
                 "mha_fwd: bad arguments");
  const int R = region_offsets_host[bags];
  const Drop dr = Drop::make(nullptr, seed, SITE_ATT, p_drop, train, 0);
  return mha_fwd(qkv, region_offsets, region_offsets_host, bags, R, d, heads, dr, mask, mask_off, ctx, lse, attention_precision(precision),
                 (cudaStream_t)stream);
}

extern "C" int advmil_mha_bwd(const float* qkv, const float* ctx, const float* d_ctx, const float* lse, const int32_t* region_offsets,
                              const int32_t* region_offsets_host, int32_t bags, int32_t d, int32_t heads, float p_drop, uint64_t seed,
                              int32_t train, const uint8_t* mask, const int64_t* mask_off, int32_t precision, float* d_qkv,
                              float* scratch /* [heads * R] */, void* stream) {
  ADVMIL_REQUIRE(qkv && ctx && d_ctx && lse && region_offsets && region_offsets_host && d_qkv && scratch && bags > 0 && heads > 0 &&
                 d % heads == 0, "mha_bwd: bad arguments");
  const int R = region_offsets_host[bags];
  const Drop dr = Drop::make(nullptr, seed, SITE_ATT, p_drop, train, 0);
  return mha_bwd(qkv, ctx, d_ctx, lse, region_offsets, region_offsets_host, bags, R, d, heads, dr, mask, mask_off, d_qkv, scratch,
                 attention_precision(precision), (cudaStream_t)stream);
}
