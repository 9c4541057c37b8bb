// Fused adversarial step: the launch sequence of one D update + one G update (model/model_handler.py:349-498) issued from
// C in two host calls (advmil_adv_step_disc / advmil_adv_step_gen) over one caller-owned workspace.  gen_updates > 1 (more
// G updates per D update, model/model_handler.py:328-335): advmil_adv_step_gen_next runs each further G update on the same
// workspace; the G phase is one function (gen_phase) with a `first` flag.
//
//  * real and fake pairs of the D step share one region-embedding pass and run through ONE batched RLIP head pass: the
//    head sees 2 x bags "virtual bags" (fake pairs first, then real pairs) over a duplicated [2R, d] embedding;
//  * the D-step generator forward (eval) and the G-step generator forward (train) share relu(x W1^T + b1): the projection
//    kernel of the D phase writes both the eval activations and the G step's dropped copy (its seed is known up front);
//  * the G step asks D only for dL/dt and never touches D-parameter gradients.
#include <mutex>
#include <vector>
#include "stages.cuh"

namespace advmil {

__global__ void real_mask_kernel(const float* __restrict__ e, const uint8_t* __restrict__ visible, int n, uint8_t* __restrict__ out) {
  pdl_prologue();
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = (e[i] == 1.0f && visible[i] != 0) ? 1 : 0;   // model_handler.py:373-375
}
__global__ void dup_offsets_kernel(const int32_t* __restrict__ offs, int nb, int rows, int32_t* __restrict__ out) {
  pdl_prologue();
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i <= nb) { out[i] = offs[i]; out[nb + i] = offs[i] + rows; }
}
__global__ void add_inplace_kernel(float* __restrict__ a, const float* __restrict__ b, int n) {
  pdl_prologue();
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) a[i] += b[i];
}

// head activation buffers for nr region rows / nbv (virtual) bags
static bool take_head(Workspace& ws, const AdvmilDiscParams& p, size_t nr, size_t nbv, AdvmilHeadActs& h) {
  const size_t d = p.d, dh = p.d / 2, abw = gate_width(p.d);
  h.f1 = ws.take<float>(nr * dh); h.fi = ws.take<float>(nr * d); h.ab = ws.take<float>(nr * abw);
  h.rep = ws.take<float>(nr); h.attn = ws.take<float>(nr);
  h.bagv = ws.take<float>(nbv * d); h.fbar = ws.take<float>(nbv * d); h.g1 = ws.take<float>(nbv * dh);
  h.hx = ws.take<float>(nbv * d); h.u1 = ws.take<float>(nbv * p.t1); h.ht = ws.take<float>(nbv * p.t2);
  return h.f1 && h.fi && h.ab && h.rep && h.attn && h.bagv && h.fbar && h.g1 && h.hx && h.u1 && h.ht;
}
static size_t head_bytes(const AdvmilDiscParams& p, size_t nr, size_t nbv) {
  const size_t d = p.d, dh = p.d / 2, abw = gate_width(p.d);
  const size_t f = nr * (dh + d + abw + 2) + nbv * (3 * d + dh + p.t1 + p.t2);
  return f * sizeof(float) + 16 * 256;
}

struct GenBufs { float *s, *w, *z, *H, *H1, *pre; };
static bool take_gen(Workspace& ws, const AdvmilGenParams& g, size_t rows, size_t nb, GenBufs& b) {
  b.s = ws.take<float>(rows); b.w = ws.take<float>(rows); b.z = ws.take<float>(nb * g.h); b.H = ws.take<float>(nb * g.o);
  b.H1 = ws.take<float>(nb * (g.hid > 0 ? g.hid : 1)); b.pre = ws.take<float>(nb);
  return b.s && b.w && b.z && b.H && b.H1 && b.pre;
}
static size_t gen_bufs_bytes(const AdvmilGenParams& g, size_t rows, size_t nb) {
  return (2 * rows + nb * (g.h + g.o + g.hid + 2)) * sizeof(float) + 8 * 256;
}

// ---- overlap of the D phase's region-level chain with the G phase's first half --------------------------------------
// After the eval projection exists, the train-mode generator forward of the G step (dropout on the cached projection, gate
// GEMM, pooling, head) depends on nothing the D phase still has to do, while the D phase's head forward/backward is a
// chain of small region-level kernels that leaves most SMs idle.  The disc call therefore issues that forward on a side
// stream; the gen call joins it.
struct SideState {
  static constexpr int SLOTS = 4;       // engines (workspaces) with a forked forward in flight at the same time
  cudaStream_t stream = nullptr;
  cudaEvent_t fork = nullptr, done[SLOTS] = {nullptr, nullptr, nullptr, nullptr};
  const void* pending_ws[SLOTS] = {nullptr, nullptr, nullptr, nullptr};   // workspace whose train forward was forked
  int find(const void* ws) const { for (int i = 0; i < SLOTS; ++i) if (pending_ws[i] == ws) return i; return -1; }
};
// One side stream and event set PER DEVICE (created on the device that is current at the call, which is the device of the
// caller's stream and workspace), guarded by a mutex: several engines, devices or host threads in one process never
// share a stream of the wrong device or race on the slot table.
static constexpr int MAX_DEVICES = 64;
static SideState g_side[MAX_DEVICES];
static std::mutex g_side_mu;
static int side_get(SideState** out) {
  *out = nullptr;
  int dev = 0;
  ADVMIL_CHECK_CUDA(cudaGetDevice(&dev));
  if (dev < 0 || dev >= MAX_DEVICES) return ADVMIL_OK;     // no overlap on an out-of-range ordinal: the gen call runs the forward
  SideState& s = g_side[dev];
  if (!s.stream) {
    ADVMIL_CHECK_CUDA(cudaStreamCreateWithFlags(&s.stream, cudaStreamNonBlocking));
    ADVMIL_CHECK_CUDA(cudaEventCreateWithFlags(&s.fork, cudaEventDisableTiming));
    for (int i = 0; i < SideState::SLOTS; ++i) ADVMIL_CHECK_CUDA(cudaEventCreateWithFlags(&s.done[i], cudaEventDisableTiming));
  }
  *out = &s;
  return ADVMIL_OK;
}

#define STEP_TAKE(var, type, count)                                                                         \
  type* var = ws.take<type>(count);                                                                         \
  if (!var) { set_error("%s: workspace too small (have %zu bytes)", __func__, ws.cap); return ADVMIL_ERR_WORKSPACE; }

// ---- the RLIP discriminator's part of the two phases, shared by the ABMIL, ESAT and DeepAttMISL steps ----------------
// Scratch bytes of the D phase from the region embedding on, and of the G phase's D(x, pred_g) with the caller's d_pred.
// `who` names the public entry point in error messages.
static size_t disc_part_bytes(const AdvmilDiscParams* d, size_t rows, size_t nb, int precision) {
  const size_t es = elem_bytes(elem_of_precision(precision)), R = rows / 16;
  return align_up(2 * R * d->d * sizeof(float), 256) + align_up(rows * d->d * es, 256) + head_bytes(*d, 2 * R, 2 * nb) +
         align_up(2 * R * d->d * sizeof(float), 256) + 8 * 256 + 6 * nb * sizeof(float) + align_up((2 * nb + 2) * sizeof(int32_t), 256) +
         advmil_disc_workspace_bytes(d, 2 * rows, 2 * nb, 1) + 256;
}
static size_t gen_part_bytes(const AdvmilDiscParams* d, size_t rows, size_t nb) {
  const size_t R = rows / 16;
  return head_bytes(*d, R, nb) + 8 * 256 + 4 * nb * sizeof(float) + advmil_disc_workspace_bytes(d, rows, nb, 1) + 256;
}
// D's region embedding of x for the G phase, [R, d] fp32: a persistent slot of every step's workspace.  D does not change
// between the G updates of one step, so the first G update writes it and the later ones read it back.
static size_t gen_emb_bytes(const AdvmilDiscParams* d, size_t rows) { return align_up(rows / 16 * d->d * sizeof(float), 256); }
// D phase, region embedding: ea.emb has room for the [2R, d] copy that disc_rlip duplicates for the batched head.  With
// run == false the caller writes ea.emb / ea.y_pre itself (the ABMIL step: fused with its projection, or after its forward).
static int disc_embed(const AdvmilStepArgs* a, Workspace& ws, bool run, AdvmilEmbedActs& ea, const char* who, cudaStream_t st) {
  const size_t rows = a->bags->rows, d = a->disc->d;
  ea = AdvmilEmbedActs{};
  ea.emb = ws.take<float>(2 * (rows / 16) * d);
  ea.y_pre = ws.take<char>(rows * d * elem_bytes(elem_of_precision(a->precision)));
  ea.precision = a->precision;
  if (!ea.emb || !ea.y_pre) { set_error("%s: workspace too small (have %zu bytes)", who, ws.cap); return ADVMIL_ERR_WORKSPACE; }
  return run ? advmil_disc_embed_fwd(a->disc, a->bags, &ea, (void*)st) : ADVMIL_OK;
}
// D phase after pred_d and the region embedding exist: batched head over [fake | real] pairs, D loss, D backward
static int disc_rlip(const AdvmilStepArgs* a, Workspace& ws, AdvmilEmbedActs& ea, const char* who, cudaStream_t st) {
  const AdvmilDiscParams& dp = *a->disc;
  const AdvmilBags* bags = a->bags;
  const int rows = bags->rows, nb = bags->bags, R = rows / 16, d = dp.d;
  const bool batched = a->n_real > 0.f;                 // no real pair anywhere: only the fake half runs
  AdvmilHeadActs ha{};
  const bool head_ok = take_head(ws, dp, 2 * (size_t)R, 2 * (size_t)nb, ha);
  float* d_emb2 = ws.take<float>((size_t)2 * R * d);
  float* t2 = ws.take<float>(2 * nb);
  float* d_out2 = ws.take<float>(2 * nb);
  int32_t* offs2 = ws.take<int32_t>(2 * nb + 2);
  const size_t dws_bytes = advmil_disc_workspace_bytes(&dp, 2 * rows, 2 * nb, 1);
  char* dws = ws.take<char>(dws_bytes);
  if (!head_ok || !d_emb2 || !t2 || !d_out2 || !offs2 || !dws) {
    set_error("%s: workspace too small (have %zu bytes)", who, ws.cap);
    return ADVMIL_ERR_WORKSPACE;
  }
  float* emb2 = ea.emb;
  std::vector<int32_t> offs2_host(2 * nb + 1);
  for (int i = 0; i <= nb; ++i) { offs2_host[i] = bags->offsets_host[i]; offs2_host[nb + i] = bags->offsets_host[i] + rows; }
  launch_k(dup_offsets_kernel, dim3(cdiv(nb + 1, 128)), dim3(128), 0, st, bags->offsets, nb, rows, offs2);
  ADVMIL_CHECK_LAUNCH();
  launch_k(real_mask_kernel, dim3(cdiv(nb, 128)), dim3(128), 0, st, a->e, a->visible, nb, a->real_mask);
  ADVMIL_CHECK_LAUNCH();
  ADVMIL_CHECK_CUDA(cudaMemcpyAsync(t2, a->pred_d, nb * sizeof(float), cudaMemcpyDeviceToDevice, st));
  if (batched) {
    ADVMIL_CHECK_CUDA(cudaMemcpyAsync(t2 + nb, a->t, nb * sizeof(float), cudaMemcpyDeviceToDevice, st));
    ADVMIL_CHECK_CUDA(cudaMemcpyAsync(emb2 + (size_t)R * d, emb2, (size_t)R * d * sizeof(float), cudaMemcpyDeviceToDevice, st));
  }
  AdvmilBags vb = *bags;
  vb.offsets = offs2; vb.offsets_host = offs2_host.data(); vb.rows = batched ? 2 * rows : rows; vb.bags = batched ? 2 * nb : nb;
  ha.emb = emb2; ha.t = t2; ha.out = a->f_fake_d;
  ha.mask_fc1 = a->d_mask_fc1; ha.mask_ga = a->d_mask_ga; ha.mask_gs = a->d_mask_gs; ha.mask_fc2 = a->d_mask_fc2;
  ha.seed = a->seed_d; ha.train = 1; ha.precision = a->precision; ha.workspace = dws; ha.workspace_bytes = dws_bytes;
  ADVMIL_TRY(advmil_disc_head_fwd(&dp, &vb, &ha, (void*)st));
  // ---- loss (loss/utils.py:182-203) and backward ----
  ADVMIL_TRY(advmil_disc_loss(a->f_fake_d + nb, a->f_fake_d, a->real_mask, nb, a->loss_d, a->n_real, a->n_fake, a->losses,
                              d_out2 + nb, d_out2, (void*)st));
  ADVMIL_TRY(advmil_disc_head_bwd(&dp, &vb, &ha, d_out2, d_emb2, nullptr, a->disc_grads, 0, (void*)st));
  ea.workspace = dws; ea.workspace_bytes = dws_bytes;
  return disc_embed_bwd_impl(&dp, bags, &ea, d_emb2, batched ? d_emb2 + (size_t)R * d : nullptr, a->disc_grads, 0, st);
}
// G phase after pred_g exists: D(x, pred_g) with the updated discriminator in eval mode, G loss, and dL/dpred_g (recon +
// the adversarial term through D) into d_pred [bags].  emb: the persistent [R, d] slot of D's region embedding, computed
// here unless emb_ready (a later G update of the same step).
static int gen_rlip(const AdvmilStepArgs* a, Workspace& ws, float* emb, bool emb_ready, float* d_pred, const char* who,
                    cudaStream_t st) {
  const AdvmilDiscParams& dp = *a->disc;
  const AdvmilBags* bags = a->bags;
  const int rows = bags->rows, nb = bags->bags, R = rows / 16;
  AdvmilHeadActs ha{};
  const bool head_ok = take_head(ws, dp, R, nb, ha);
  float* d_fake = ws.take<float>(nb);
  float* d_t = ws.take<float>(nb);
  const size_t dws_bytes = advmil_disc_workspace_bytes(&dp, rows, nb, 1);
  char* dws = ws.take<char>(dws_bytes);
  if (!head_ok || !d_fake || !d_t || !dws) { set_error("%s: workspace too small (have %zu bytes)", who, ws.cap); return ADVMIL_ERR_WORKSPACE; }
  if (!emb_ready) {
    AdvmilEmbedActs ea{};
    ea.emb = emb; ea.y_pre = nullptr; ea.precision = a->precision;
    ea.workspace = dws; ea.workspace_bytes = dws_bytes;      // the head forward below reuses it
    ADVMIL_TRY(advmil_disc_embed_fwd(&dp, bags, &ea, (void*)st));
  }
  ha.ab = nullptr;      // the G step asks D only for dL/dt: the gate activations are never read back
  ha.emb = emb; ha.t = a->pred_g; ha.out = a->f_fake_g; ha.seed = 0; ha.train = 0; ha.precision = a->precision;
  ha.workspace = dws; ha.workspace_bytes = dws_bytes;
  ADVMIL_TRY(advmil_disc_head_fwd(&dp, bags, &ha, (void*)st));
  // ---- loss (loss/utils.py:21-41,205-208) and backward: D hands back only dL/dt ----
  ADVMIL_TRY(advmil_gen_loss(a->pred_g, a->t, a->e, a->visible, a->f_fake_g, nb, a->n_visible, a->n_fake, a->coef_gan,
                             a->recon_alpha, a->recon_gamma, a->recon_norm, a->losses + 1, d_pred, d_fake, (void*)st));
  ADVMIL_TRY(advmil_disc_head_bwd(&dp, bags, &ha, d_fake, nullptr, d_t, nullptr, 0, (void*)st));
  launch_k(add_inplace_kernel, dim3(cdiv(nb, 128)), dim3(128), 0, st, d_pred, d_t, nb);
  ADVMIL_CHECK_LAUNCH();
  return ADVMIL_OK;
}

}  // namespace advmil

using namespace advmil;

// persistent region (same layout in every call): eval projection and everything the G step's train forward writes (it may
// run on the side stream while the D phase uses the scratch region), and D's region embedding for the G phase
struct Persist {
  char* h_eval; char* h; char* ab; GenBufs gb; char* gws; size_t gws_bytes; float* demb;
};
static int take_persist(Workspace& ws, const AdvmilGenParams& gp, const AdvmilDiscParams& dp, int rows, int nb, size_t es, Persist& P) {
  const size_t abw = gate_width(gp.h);
  P.h_eval = ws.take<char>((size_t)rows * gp.h * es);
  P.h = ws.take<char>((size_t)rows * gp.h * es);
  P.ab = ws.take<char>((size_t)rows * abw * es);
  const bool ok = take_gen(ws, gp, rows, nb, P.gb);
  P.gws_bytes = advmil_generator_workspace_bytes(&gp, rows, nb, 1);
  P.gws = ws.take<char>(P.gws_bytes);
  P.demb = ws.take<float>((size_t)(rows / 16) * dp.d);
  if (!P.h_eval || !P.h || !P.ab || !ok || !P.gws || !P.demb) { set_error("adv_step: workspace too small (have %zu bytes)", ws.cap); return ADVMIL_ERR_WORKSPACE; }
  return ADVMIL_OK;
}
static void fill_train_acts(const AdvmilStepArgs* a, const Persist& P, AdvmilGenActs& ga) {
  ga = AdvmilGenActs{};
  ga.h = P.h; ga.ab = P.ab; ga.s = P.gb.s; ga.w = P.gb.w; ga.z = P.gb.z; ga.H = P.gb.H; ga.H1 = P.gb.H1; ga.pre = P.gb.pre;
  ga.pred = a->pred_g; ga.noise0 = nullptr; ga.noise1 = a->noise_g;
  ga.h_eval = nullptr; ga.h_ready = 1;   // the disc phase's projection kernel already wrote dropout(h_eval) into P.h
  ga.mask_h = a->g_mask_h; ga.mask_a = a->g_mask_a; ga.mask_b = a->g_mask_b; ga.mask_rho = a->g_mask_rho; ga.mask_mlp0 = a->g_mask_mlp0;
  ga.seed = a->seed_g; ga.train = 1; ga.precision = a->precision; ga.workspace = P.gws; ga.workspace_bytes = P.gws_bytes;
}

extern "C" size_t advmil_adv_step_workspace_bytes(const AdvmilGenParams* g, const AdvmilDiscParams* d, int32_t rows,
                                                  int32_t bags, int32_t precision) {
  const size_t es = elem_bytes(elem_of_precision(precision));
  const size_t nb = bags, abw = gate_width(g->h);
  size_t persistent = 2 * align_up((size_t)rows * g->h * es, 256) + align_up((size_t)rows * abw * es, 256) + gen_bufs_bytes(*g, rows, nb) +
                      advmil_generator_workspace_bytes(g, rows, bags, 1) + gen_emb_bytes(d, rows) + 2048;
  size_t disc = gen_bufs_bytes(*g, rows, nb) + advmil_generator_workspace_bytes(g, rows, bags, 0) + 256 + disc_part_bytes(d, rows, nb, precision);
  size_t gen = gen_part_bytes(d, rows, nb);
  return persistent + (disc > gen ? disc : gen) + 4096;
}

static int step_check(const AdvmilStepArgs* a) {
  ADVMIL_REQUIRE(a && a->gen && a->disc && a->bags && a->t && a->e && a->visible && a->losses, "adv_step: null argument");
  ADVMIL_REQUIRE(a->gen->W0 && a->gen->Wrho, "adv_step: the fused step covers the ABMIL generator with its noise head");
  ADVMIL_REQUIRE(a->gen->noise0 == 0, "adv_step: noise on the first head layer (gen_noi_noise '1-*') is not covered by the fused step");
  ADVMIL_REQUIRE(a->workspace, "adv_step: workspace missing");
  return ADVMIL_OK;
}

extern "C" int advmil_adv_step_disc(const AdvmilStepArgs* a, void* stream) {
  ADVMIL_TRY(step_check(a));
  ADVMIL_REQUIRE(a->disc_grads && a->pred_d && a->f_fake_d && a->real_mask, "adv_step_disc: missing output buffers");
  cudaStream_t st = (cudaStream_t)stream;
  const AdvmilGenParams& gp = *a->gen;
  const AdvmilDiscParams& dp = *a->disc;
  const AdvmilBags* bags = a->bags;
  const int rows = bags->rows, nb = bags->bags, d = dp.d;
  const size_t es = elem_bytes(elem_of_precision(a->precision));
  Workspace ws(a->workspace, a->workspace_bytes);
  Persist P;
  ADVMIL_TRY(take_persist(ws, gp, dp, rows, nb, es, P));
  char* h_eval = P.h_eval;
  std::lock_guard<std::mutex> side_lock(g_side_mu);
  SideState* side = nullptr;
  ADVMIL_TRY(side_get(&side));
  if (side) {
    // a gen call never came for this workspace (exception between the phases): the forked forward may still be reading
    // and writing the persistent region -- the new step must not overwrite it before that forward has drained
    const int old = side->find(a->workspace);
    if (old >= 0) { ADVMIL_CHECK_CUDA(cudaStreamWaitEvent(st, side->done[old], 0)); side->pending_ws[old] = nullptr; }
  }
  // ---- generator, eval mode, detached (model_handler.py:383-387) ----
  GenBufs gb;
  if (!take_gen(ws, gp, rows, nb, gb)) { set_error("adv_step_disc: workspace too small"); return ADVMIL_ERR_WORKSPACE; }
  const size_t gws_bytes = advmil_generator_workspace_bytes(&gp, rows, nb, 0);
  STEP_TAKE(gws, char, gws_bytes);
  AdvmilGenActs ga{};
  ga.h = h_eval; ga.ab = nullptr; ga.s = gb.s; ga.w = gb.w; ga.z = gb.z; ga.H = gb.H; ga.H1 = gb.H1; ga.pre = gb.pre;
  ga.pred = a->pred_d; ga.noise0 = nullptr; ga.noise1 = a->noise_d; ga.h_eval = nullptr;
  ga.seed = 0; ga.train = 0; ga.precision = a->precision; ga.workspace = gws; ga.workspace_bytes = gws_bytes;
  ga.h_drop_out = P.h; ga.seed_drop = a->seed_g; ga.mask_h_drop = a->g_mask_h;   // the G step's dropped projection, same pass
  // ---- shared region embedding (K5+K6), duplicated for the batched head ----
  AdvmilEmbedActs ea;
  ADVMIL_TRY(disc_embed(a, ws, false, ea, __func__, st));
  const bool fused = gp.C == dp.C && (dp.ksize == 0 || dp.ksize == 1) && proj_embed_supported(rows, gp.C, gp.h, d, a->precision);
  if (fused) {     // K1 and K5+K6 read the same x: one pass over stacked weights, then the generator forward skips K1
    for (int i = 0; i < nb; ++i)
      ADVMIL_REQUIRE((bags->offsets_host[i + 1] - bags->offsets_host[i]) % 16 == 0,
                     "bags: bag %d has a length that is not a multiple of 16 (model/backbone_utils.py:65)", i);
    Drop d2 = Drop::make(a->g_mask_h, a->seed_g, SITE_H, gp.p_backbone, 1, gp.h);
    { ProfScope ps(PROF_PROJ_EMBED, st);
      ADVMIL_TRY(proj_embed_fwd(bags->x, gp.W1, gp.b1, dp.Wc, dp.bc, dp.ln_g, dp.ln_b, rows, gp.C, gp.h, d, dp.ln_eps, h_eval, P.h, &d2,
                                ea.y_pre, ea.emb, st)); }
    ga.h_ready = 1; ga.h_drop_out = nullptr;
  }
  ADVMIL_TRY(advmil_generator_fwd(&gp, bags, &ga, stream));
  if (!fused) ADVMIL_TRY(advmil_disc_embed_fwd(&dp, bags, &ea, stream));
  // ---- fork: the G step's train-mode generator forward runs on the side stream from here on ----
  const int slot = side ? side->find(nullptr) : -1;      // no free slot: the gen call runs the forward itself
  if (slot >= 0 && a->gen_grads && a->pred_g && a->noise_g) {
    ADVMIL_CHECK_CUDA(cudaEventRecord(side->fork, st));
    ADVMIL_CHECK_CUDA(cudaStreamWaitEvent(side->stream, side->fork, 0));
    AdvmilGenActs gt;
    fill_train_acts(a, P, gt);
    ADVMIL_TRY(advmil_generator_fwd(&gp, bags, &gt, (void*)side->stream));
    ADVMIL_CHECK_CUDA(cudaEventRecord(side->done[slot], side->stream));
    side->pending_ws[slot] = a->workspace;
  }
  // ---- batched head over the virtual bags [fake pairs | real pairs], loss and backward ----
  return disc_rlip(a, ws, ea, __func__, st);
}

// One G update (model_handler.py:432-498 up to the caller's Adam step).  first: the update after the D phase, which reuses
// the dropped projection of the disc call (side stream or not); a later update recomputes K1 from G's current parameters.
static int gen_phase(const AdvmilStepArgs* a, bool first, const char* who, cudaStream_t st) {
  ADVMIL_TRY(step_check(a));
  ADVMIL_REQUIRE(a->gen_grads && a->pred_g && a->f_fake_g, "%s: missing output buffers", who);
  const AdvmilGenParams& gp = *a->gen;
  const AdvmilBags* bags = a->bags;
  const int rows = bags->rows, nb = bags->bags;
  const size_t es = elem_bytes(elem_of_precision(a->precision));
  Workspace ws(a->workspace, a->workspace_bytes);
  Persist P;                                                  // h_eval was written by advmil_adv_step_disc on this workspace
  ADVMIL_TRY(take_persist(ws, gp, *a->disc, rows, nb, es, P));
  // ---- generator, train mode: join the side stream's forward on the cached eval projection, or run it here ----
  AdvmilGenActs ga;
  fill_train_acts(a, P, ga);
  if (!first) ga.h_ready = 0;        // K1 with this update's dropout: G's parameters moved at the previous update
  std::unique_lock<std::mutex> side_lock(g_side_mu);
  SideState* side = nullptr;
  ADVMIL_TRY(side_get(&side));
  const int slot = side ? side->find(a->workspace) : -1;
  if (slot >= 0) {
    ADVMIL_CHECK_CUDA(cudaStreamWaitEvent(st, side->done[slot], 0));
    side->pending_ws[slot] = nullptr;
  }
  side_lock.unlock();
  if (slot < 0 || !first) ADVMIL_TRY(advmil_generator_fwd(&gp, bags, &ga, (void*)st));
  // ---- D(x, pred_g) with the updated discriminator, G loss, dL/dpred_g ----
  float* d_pred = ws.take<float>(nb);
  if (!d_pred) { set_error("%s: workspace too small (have %zu bytes)", who, ws.cap); return ADVMIL_ERR_WORKSPACE; }
  ADVMIL_TRY(gen_rlip(a, ws, P.demb, !first, d_pred, who, st));
  return advmil_generator_bwd(&gp, bags, &ga, d_pred, a->gen_grads, (void*)st);
}

extern "C" int advmil_adv_step_gen(const AdvmilStepArgs* a, void* stream) {
  return gen_phase(a, true, __func__, (cudaStream_t)stream);
}
extern "C" int advmil_adv_step_gen_next(const AdvmilStepArgs* a, void* stream) {
  return gen_phase(a, false, __func__, (cudaStream_t)stream);
}


// =====================================================================================================================
// The same two-phase step for the ESAT generator (bcb_mode `patch`: DualTrans_HS + noise head, advmil_esat_fwd / _bwd) with
// the RLIP discriminator: the launch sequence of ModuleAdvStep (step.py) issued from C.  The eval pass of the D phase and the
// train pass of the G phase share ONE activation set in the persistent region: the patch embedding (y_pre, emb) has no
// dropout and G's parameters do not change between the phases, so the train pass runs with emb_ready = 1; real and fake D
// pairs share the region embedding and run through one batched head pass, exactly like the ABMIL step above.
// In-kernel dropout only (seed_d / seed_g); injected masks go through the module path.
// =====================================================================================================================
namespace advmil {
struct EsatBufs {
  char* y_pre; float *emb, *qkv, *lse, *ctx, *s1, *x1, *f, *s2, *x2, *ab, *rep, *attn, *H, *H1, *pre;
  char* ews; size_t ews_bytes;
  float* demb;      // D's region embedding for the G phase
};
static size_t esat_acts_bytes(const AdvmilEsatParams& p, const AdvmilGenParams& h, size_t rows, size_t nb, size_t es) {
  const size_t R = rows / 16, d = p.d, abw = gate_width(p.d);
  return align_up(rows * d * es, 256) + (R * (d * 9 + p.ff + abw + 2) + (size_t)p.nhead * R + nb * (d + h.hid + 1)) * sizeof(float) + 20 * 256;
}
static int take_esat(Workspace& ws, const AdvmilEsatParams& p, const AdvmilGenParams& h, const AdvmilDiscParams& dp, int rows, int nb,
                     size_t es, EsatBufs& b) {
  const size_t R = rows / 16, d = p.d, abw = gate_width(p.d);
  b.y_pre = ws.take<char>((size_t)rows * d * es);
  b.emb = ws.take<float>(R * d); b.qkv = ws.take<float>(R * 3 * d); b.lse = ws.take<float>((size_t)p.nhead * R); b.ctx = ws.take<float>(R * d);
  b.s1 = ws.take<float>(R * d); b.x1 = ws.take<float>(R * d); b.f = ws.take<float>(R * p.ff); b.s2 = ws.take<float>(R * d);
  b.x2 = ws.take<float>(R * d); b.ab = ws.take<float>(R * abw); b.rep = ws.take<float>(R); b.attn = ws.take<float>(R);
  b.H = ws.take<float>((size_t)nb * d); b.H1 = ws.take<float>((size_t)nb * (h.hid > 0 ? h.hid : 1)); b.pre = ws.take<float>(nb);
  const size_t e0 = advmil_esat_workspace_bytes(&p, &h, rows, nb, 0), e1 = advmil_esat_workspace_bytes(&p, &h, rows, nb, 1);
  b.ews_bytes = e0 > e1 ? e0 : e1;
  b.ews = ws.take<char>(b.ews_bytes);
  b.demb = ws.take<float>(R * dp.d);
  if (!b.y_pre || !b.emb || !b.qkv || !b.lse || !b.ctx || !b.s1 || !b.x1 || !b.f || !b.s2 || !b.x2 || !b.ab || !b.rep || !b.attn || !b.H ||
      !b.H1 || !b.pre || !b.ews || !b.demb) {
    set_error("adv_step_esat: workspace too small (have %zu bytes)", ws.cap);
    return ADVMIL_ERR_WORKSPACE;
  }
  return ADVMIL_OK;
}
static void fill_esat_acts(const AdvmilEsatStepArgs* a, const EsatBufs& b, int train, AdvmilEsatActs& ea) {
  ea = AdvmilEsatActs{};
  ea.y_pre = b.y_pre; ea.emb = b.emb; ea.qkv = b.qkv; ea.lse = b.lse; ea.ctx = b.ctx; ea.s1 = b.s1; ea.x1 = b.x1; ea.f = b.f; ea.s2 = b.s2;
  ea.x2 = b.x2; ea.ab = b.ab; ea.rep = b.rep; ea.attn = b.attn; ea.H = b.H; ea.H1 = b.H1; ea.pre = b.pre;
  ea.pred = train ? a->pred_g : a->pred_d;
  ea.pe = a->pe; ea.noise0 = nullptr; ea.noise1 = train ? a->noise_g : a->noise_d;
  ea.seed = train ? a->seed_g : 0; ea.train = train; ea.precision = a->precision;
  ea.workspace = b.ews; ea.workspace_bytes = b.ews_bytes;
  ea.emb_ready = train;        // the eval pass of the D phase wrote y_pre / emb of these bags under the same parameters
}
static int esat_step_check(const AdvmilEsatStepArgs* a) {
  ADVMIL_REQUIRE(a && a->esat && a->head && a->disc && a->bags && a->t && a->e && a->visible && a->losses && a->workspace,
                 "adv_step_esat: null argument");
  ADVMIL_REQUIRE(a->head->W0 && a->head->noise0 == 0, "adv_step_esat: needs the noise head with gen_noi_noise '0-1'");
  return ADVMIL_OK;
}
// the fields disc_rlip / gen_rlip read, as an AdvmilStepArgs view of the ESAT step's arguments (no injected D masks)
static AdvmilStepArgs rlip_args(const AdvmilEsatStepArgs* a) {
  AdvmilStepArgs v{};
  v.disc = a->disc; v.disc_grads = a->disc_grads; v.bags = a->bags; v.t = a->t; v.e = a->e; v.visible = a->visible;
  v.seed_d = a->seed_d; v.n_real = a->n_real; v.n_fake = a->n_fake; v.n_visible = a->n_visible;
  v.loss_d = a->loss_d; v.coef_gan = a->coef_gan; v.recon_alpha = a->recon_alpha; v.recon_gamma = a->recon_gamma;
  v.recon_norm = a->recon_norm; v.precision = a->precision;
  v.losses = a->losses; v.pred_d = a->pred_d; v.f_fake_d = a->f_fake_d; v.real_mask = a->real_mask;
  v.pred_g = a->pred_g; v.f_fake_g = a->f_fake_g;
  return v;
}
}  // namespace advmil

extern "C" size_t advmil_adv_step_esat_workspace_bytes(const AdvmilEsatParams* g, const AdvmilGenParams* head, const AdvmilDiscParams* d,
                                                       int32_t rows, int32_t bags, int32_t precision) {
  const size_t es = elem_bytes(elem_of_precision(precision));
  const size_t nb = bags;
  const size_t e0 = advmil_esat_workspace_bytes(g, head, rows, bags, 0), e1 = advmil_esat_workspace_bytes(g, head, rows, bags, 1);
  size_t persistent = esat_acts_bytes(*g, *head, rows, nb, es) + (e0 > e1 ? e0 : e1) + gen_emb_bytes(d, rows) + 512;
  size_t disc = disc_part_bytes(d, rows, nb, precision), gen = gen_part_bytes(d, rows, nb);
  return persistent + (disc > gen ? disc : gen) + 4096;
}

extern "C" int advmil_adv_step_esat_disc(const AdvmilEsatStepArgs* a, void* stream) {
  ADVMIL_TRY(esat_step_check(a));
  ADVMIL_REQUIRE(a->disc_grads && a->pred_d && a->f_fake_d && a->real_mask, "adv_step_esat_disc: missing output buffers");
  cudaStream_t st = (cudaStream_t)stream;
  const AdvmilBags* bags = a->bags;
  const int rows = bags->rows, nb = bags->bags;
  const size_t es = elem_bytes(elem_of_precision(a->precision));
  Workspace ws(a->workspace, a->workspace_bytes);
  EsatBufs B;
  ADVMIL_TRY(take_esat(ws, *a->esat, *a->head, *a->disc, rows, nb, es, B));
  // ---- generator, eval mode, detached (model_handler.py:383-387) ----
  AdvmilEsatActs ea;
  fill_esat_acts(a, B, 0, ea);
  ADVMIL_TRY(advmil_esat_fwd(a->esat, a->head, bags, &ea, stream));
  // ---- shared region embedding, batched head over [fake | real] pairs, D loss and backward ----
  const AdvmilStepArgs v = rlip_args(a);
  AdvmilEmbedActs da;
  ADVMIL_TRY(disc_embed(&v, ws, true, da, __func__, st));
  return disc_rlip(&v, ws, da, __func__, st);
}

// One G update; first: the update after the D phase, on the patch embedding of the disc call's eval pass.  A later update
// recomputes the embedding from G's current parameters (emb_ready = 0).
static int esat_gen_phase(const AdvmilEsatStepArgs* a, bool first, const char* who, cudaStream_t st) {
  ADVMIL_TRY(esat_step_check(a));
  ADVMIL_REQUIRE(a->esat_grads && a->head_grads && a->pred_g && a->f_fake_g, "%s: missing output buffers", who);
  const AdvmilBags* bags = a->bags;
  const int rows = bags->rows, nb = bags->bags;
  const size_t es = elem_bytes(elem_of_precision(a->precision));
  Workspace ws(a->workspace, a->workspace_bytes);
  EsatBufs B;                                      // y_pre / emb were written by advmil_adv_step_esat_disc on this workspace
  ADVMIL_TRY(take_esat(ws, *a->esat, *a->head, *a->disc, rows, nb, es, B));
  // ---- generator, train mode ----
  AdvmilEsatActs ea;
  fill_esat_acts(a, B, 1, ea);
  ea.emb_ready = first;
  ADVMIL_TRY(advmil_esat_fwd(a->esat, a->head, bags, &ea, (void*)st));
  // ---- D(x, pred_g) with the updated discriminator, G loss, dL/dpred_g ----
  float* d_pred = ws.take<float>(nb);
  if (!d_pred) { set_error("%s: workspace too small (have %zu bytes)", who, ws.cap); return ADVMIL_ERR_WORKSPACE; }
  const AdvmilStepArgs v = rlip_args(a);
  ADVMIL_TRY(gen_rlip(&v, ws, B.demb, !first, d_pred, who, st));
  esat_request_overlap(1);     // weight / bias gradients of the region-level layers on the backward side stream
  const int rc = advmil_esat_bwd(a->esat, a->head, bags, &ea, d_pred, a->esat_grads, a->head_grads, (void*)st);
  esat_request_overlap(0);
  return rc;
}

extern "C" int advmil_adv_step_esat_gen(const AdvmilEsatStepArgs* a, void* stream) {
  return esat_gen_phase(a, true, __func__, (cudaStream_t)stream);
}
extern "C" int advmil_adv_step_esat_gen_next(const AdvmilEsatStepArgs* a, void* stream) {
  return esat_gen_phase(a, false, __func__, (cudaStream_t)stream);
}


// =====================================================================================================================
// The same two-phase step for the DeepAttMISL generator (bcb_mode `cluster`, model/backbone.py:89-123) with the RLIP
// discriminator.  The disc phase runs K9 once -- projection, ReLU and the per-(bag, cluster) mean in one tcgen05 pass that
// never writes the [rows, h] activation (cluster_pool.cu) -- and keeps hc, the counts and the ReLU keep bits in the
// persistent region; the eval pass (disc phase) and the train pass (gen phase) of the attention stage both start from that
// hc: phis has no dropout and G's parameters do not change between the phases.  The attention stage sees num_clusters rows
// per bag and always runs in fp32 (like Generator.forward).  The fp32 mode (and any shape without the tcgen05 pass) composes
// linear_fwd and the segment mean instead and keeps relu(x Wphi^T + b) itself for the backward.  The D part of both
// phases is that of the ABMIL step: one shared region embedding, one batched head pass over [fake | real] pairs.
// =====================================================================================================================
namespace advmil {

__global__ void iota_scaled_kernel(int n, int step, int32_t* __restrict__ out) {
  pdl_prologue();
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i <= n) out[i] = i * step;
}

struct ClusterBufs { float* hc; int32_t* counts; uint32_t* keep; char* hx; int32_t* hoffs; float* demb; };
static size_t cluster_persist_bytes(int rows, int nb, int C, int h, int ncl, int precision) {
  const size_t nbc = (size_t)nb * ncl;
  const size_t act = cluster_pool_fused(rows, C, h, precision) ? (size_t)rows * (h / 32) * sizeof(uint32_t)
                                                                : (size_t)rows * h * elem_bytes(elem_of_precision(precision));
  return align_up(nbc * h * sizeof(float), 256) + align_up(nbc * sizeof(int32_t), 256) + align_up(act, 256) +
         align_up((nb + 1) * sizeof(int32_t), 256) + 4 * 256;
}
static int take_cluster(Workspace& ws, const AdvmilDiscParams& dp, int rows, int nb, int C, int h, int ncl, int precision, ClusterBufs& B) {
  const size_t nbc = (size_t)nb * ncl;
  B = ClusterBufs{};
  B.hc = ws.take<float>(nbc * h);
  B.counts = ws.take<int32_t>(nbc);
  if (cluster_pool_fused(rows, C, h, precision)) B.keep = ws.take<uint32_t>((size_t)rows * (h / 32));
  else B.hx = ws.take<char>((size_t)rows * h * elem_bytes(elem_of_precision(precision)));
  B.hoffs = ws.take<int32_t>(nb + 1);
  B.demb = ws.take<float>((size_t)(rows / 16) * dp.d);
  if (!B.hc || !B.counts || !(B.keep || B.hx) || !B.hoffs || !B.demb) { set_error("adv_step_cluster: workspace too small (have %zu bytes)", ws.cap); return ADVMIL_ERR_WORKSPACE; }
  return ADVMIL_OK;
}
// packed view of hc: num_clusters fp32 rows of width h per bag
static AdvmilBags cluster_bags(const ClusterBufs& B, int nb, int ncl, int h, std::vector<int32_t>& offs_host) {
  offs_host.resize(nb + 1);
  for (int i = 0; i <= nb; ++i) offs_host[i] = i * ncl;
  AdvmilBags cb{};
  cb.x = B.hc; cb.offsets = B.hoffs; cb.offsets_host = offs_host.data();
  cb.rows = nb * ncl; cb.bags = nb; cb.C = h; cb.max_bag_rows = ncl; cb.elem = ELEM_F32;
  return cb;
}
// K9: hc, counts and the backward's ReLU keep bits (or relu(x Wphi^T + b) itself) into the persistent region, from the
// current Wphi / bphi.  Its partials come from the scratch region.
static size_t cluster_k9_bytes(int rows, int nb, int C, int h, int ncl, int precision) {
  return cluster_pool_fused(rows, C, h, precision) ? align_up(cluster_pool_ws_floats(rows, nb, h, ncl) * sizeof(float), 256)
                                                   : advmil_segment_mean_workspace_bytes(rows, nb, h, ncl) + 256;
}
static int cluster_k9(const AdvmilClusterStepArgs* ca, Workspace& ws, const ClusterBufs& B, const char* who, cudaStream_t st) {
  const AdvmilBags* bags = ca->base.bags;
  const int rows = bags->rows, nb = bags->bags, C = bags->C, h = ca->base.gen->h, ncl = ca->num_clusters, prec = ca->base.precision;
  if (cluster_pool_fused(rows, C, h, prec)) {
    float* part = ws.take<float>(cluster_pool_ws_floats(rows, nb, h, ncl));
    if (!part) { set_error("%s: workspace too small (have %zu bytes)", who, ws.cap); return ADVMIL_ERR_WORKSPACE; }
    ProfScope ps(PROF_PROJ_SEGMEAN, st);
    return cluster_pool_fwd(bags->x, ca->Wphi, ca->bphi, ca->cid, bags->offsets, bags->offsets_host, rows, nb, C, h, ncl, prec,
                            B.hc, B.counts, B.keep, part, st);
  }
  const size_t sm_bytes = advmil_segment_mean_workspace_bytes(rows, nb, h, ncl);
  char* smws = ws.take<char>(sm_bytes);
  if (!smws) { set_error("%s: workspace too small (have %zu bytes)", who, ws.cap); return ADVMIL_ERR_WORKSPACE; }
  Drop none = Drop::make(nullptr, 0, 0, 0.f, 0, 0);
  { ProfScope ps(PROF_PROJ, st); ADVMIL_TRY(linear_fwd(bags->x, ca->Wphi, ca->bphi, rows, C, h, 1, none, B.hx, prec, st)); }
  return advmil_segment_mean_by_id_fwd(B.hx, elem_of_precision(prec), ca->cid, bags->offsets, bags->offsets_host, rows, nb, h, ncl,
                                       B.hc, B.counts, smws, sm_bytes, (void*)st);
}
static int cluster_step_check(const AdvmilClusterStepArgs* ca) {
  ADVMIL_REQUIRE(ca, "adv_step_cluster: null argument");
  const AdvmilStepArgs* a = &ca->base;
  ADVMIL_REQUIRE(a->gen && a->disc && a->bags && a->t && a->e && a->visible && a->losses && a->workspace && ca->Wphi && ca->bphi && ca->cid,
                 "adv_step_cluster: null argument");
  ADVMIL_REQUIRE(a->gen->W0 && !a->gen->Wrho, "adv_step_cluster: the attention stage has no rho layer and needs the noise head");
  ADVMIL_REQUIRE(a->gen->noise0 == 0, "adv_step_cluster: noise on the first head layer (gen_noi_noise '1-*') is not covered by the fused step");
  ADVMIL_REQUIRE(a->gen->C == a->gen->h, "adv_step_cluster: the attention stage reads the h-wide cluster means (C %d != h %d)", a->gen->C, a->gen->h);
  ADVMIL_REQUIRE(a->disc->ksize == 0 || a->disc->ksize == 1, "adv_step_cluster: the fused step covers the ksize-1 discriminator");
  ADVMIL_REQUIRE(ca->num_clusters >= 1 && ca->num_clusters <= CLUSTER_POOL_MAX, "adv_step_cluster: num_clusters %d outside 1..%d",
                 ca->num_clusters, CLUSTER_POOL_MAX);
  const AdvmilBags* b = a->bags;
  ADVMIL_REQUIRE(b->offsets_host && b->bags > 0 && b->offsets_host[0] == 0 && b->offsets_host[b->bags] == b->rows, "bags: bad offsets");
  for (int i = 0; i < b->bags; ++i)
    ADVMIL_REQUIRE((b->offsets_host[i + 1] - b->offsets_host[i]) % 16 == 0,
                   "bags: bag %d has a length that is not a multiple of 16 (model/backbone_utils.py:65)", i);
  return ADVMIL_OK;
}
}  // namespace advmil

extern "C" size_t advmil_adv_step_cluster_workspace_bytes(const AdvmilGenParams* g, const AdvmilDiscParams* d, int32_t rows,
                                                          int32_t bags, int32_t num_clusters, int32_t precision) {
  const int C = d->C, h = g->h, ncl = num_clusters;
  const size_t nb = bags, nbc = nb * ncl, abw = gate_width(h);
  const size_t es = elem_bytes(elem_of_precision(precision));
  const size_t persistent = cluster_persist_bytes(rows, bags, C, h, ncl, precision) + gen_emb_bytes(d, rows);
  const size_t k9 = cluster_k9_bytes(rows, bags, C, h, ncl, precision);      // the disc phase, and every G update after the first
  const size_t disc = k9 + gen_bufs_bytes(*g, nbc, nb) + align_up(nbc * h * sizeof(float), 256) +
                      advmil_generator_workspace_bytes(g, (int)nbc, bags, 0) + 256 + disc_part_bytes(d, rows, nb, precision);
  const size_t gen = k9 + gen_bufs_bytes(*g, nbc, nb) + align_up(nbc * h * sizeof(float), 256) + align_up(nbc * abw * sizeof(float), 256) +
                     advmil_generator_workspace_bytes(g, (int)nbc, bags, 1) + 256 + align_up(nb * sizeof(float), 256) +
                     align_up(nbc * h * sizeof(float), 256) + align_up((size_t)rows * h * es, 256) +
                     align_up(bwd_weight_ws_floats(rows, h, C) * sizeof(float), 256) + align_up((size_t)row_chunks(rows) * h * sizeof(float), 256) +
                     gen_part_bytes(d, rows, nb);
  return persistent + (disc > gen ? disc : gen) + 4096;
}

extern "C" int advmil_adv_step_cluster_disc(const AdvmilClusterStepArgs* ca, void* stream) {
  ADVMIL_TRY(cluster_step_check(ca));
  const AdvmilStepArgs* a = &ca->base;
  ADVMIL_REQUIRE(a->disc_grads && a->pred_d && a->f_fake_d && a->real_mask && a->noise_d, "adv_step_cluster_disc: missing buffers");
  cudaStream_t st = (cudaStream_t)stream;
  const AdvmilGenParams& gp = *a->gen;
  const AdvmilBags* bags = a->bags;
  const int rows = bags->rows, nb = bags->bags, C = bags->C, h = gp.h, ncl = ca->num_clusters, nbc = nb * ncl;
  const int prec = a->precision;
  ADVMIL_REQUIRE(C == a->disc->C && bags->elem == elem_of_precision(prec), "adv_step_cluster_disc: x width %d / element type do not match", C);
  Workspace ws(a->workspace, a->workspace_bytes);
  ClusterBufs B;
  ADVMIL_TRY(take_cluster(ws, *a->disc, rows, nb, C, h, ncl, prec, B));
  // ---- K9: hc, counts and the backward's ReLU mask stay in the persistent region for the first G update ----
  ADVMIL_TRY(cluster_k9(ca, ws, B, __func__, st));
  launch_k(iota_scaled_kernel, dim3(cdiv(nb + 1, 128)), dim3(128), 0, st, nb, ncl, B.hoffs);
  ADVMIL_CHECK_LAUNCH();
  // ---- attention stage, eval mode, detached (model_handler.py:383-387) ----
  std::vector<int32_t> hoffs_host;
  const AdvmilBags cb = cluster_bags(B, nb, ncl, h, hoffs_host);
  GenBufs gb;
  if (!take_gen(ws, gp, nbc, nb, gb)) { set_error("adv_step_cluster_disc: workspace too small"); return ADVMIL_ERR_WORKSPACE; }
  STEP_TAKE(hh, float, (size_t)nbc * h);
  const size_t gws_bytes = advmil_generator_workspace_bytes(&gp, nbc, nb, 0);
  STEP_TAKE(gws, char, gws_bytes);
  AdvmilGenActs ga{};
  ga.h = hh; ga.ab = nullptr; ga.s = gb.s; ga.w = gb.w; ga.z = gb.z; ga.H = gb.H; ga.H1 = gb.H1; ga.pre = gb.pre;
  ga.pred = a->pred_d; ga.noise0 = nullptr; ga.noise1 = a->noise_d;
  ga.seed = 0; ga.train = 0; ga.precision = ADVMIL_FP32; ga.workspace = gws; ga.workspace_bytes = gws_bytes;
  ADVMIL_TRY(advmil_generator_fwd(&gp, &cb, &ga, stream));
  AdvmilEmbedActs ea;
  ADVMIL_TRY(disc_embed(a, ws, true, ea, __func__, st));
  return disc_rlip(a, ws, ea, __func__, st);
}

// One G update; first: the update after the D phase, on the hc of the disc call's K9.  A later update runs K9 again from
// G's current Wphi / bphi.
static int cluster_gen_phase(const AdvmilClusterStepArgs* ca, bool first, const char* who, cudaStream_t st) {
  ADVMIL_TRY(cluster_step_check(ca));
  const AdvmilStepArgs* a = &ca->base;
  ADVMIL_REQUIRE(a->gen_grads && a->pred_g && a->f_fake_g && a->noise_g && ca->dWphi && ca->dbphi, "%s: missing buffers", who);
  void* stream = (void*)st;
  const AdvmilGenParams& gp = *a->gen;
  const AdvmilBags* bags = a->bags;
  const int rows = bags->rows, nb = bags->bags, C = bags->C, h = gp.h, ncl = ca->num_clusters, nbc = nb * ncl;
  const int prec = a->precision, dt = elem_of_precision(prec);
  Workspace ws(a->workspace, a->workspace_bytes);
  ClusterBufs B;                                    // hc / counts / keep bits were written by advmil_adv_step_cluster_disc
  ADVMIL_TRY(take_cluster(ws, *a->disc, rows, nb, C, h, ncl, prec, B));
  if (!first) ADVMIL_TRY(cluster_k9(ca, ws, B, who, st));
  // ---- attention stage, train mode, on the same hc ----
  std::vector<int32_t> hoffs_host;
  const AdvmilBags cb = cluster_bags(B, nb, ncl, h, hoffs_host);
  GenBufs gb;
  if (!take_gen(ws, gp, nbc, nb, gb)) { set_error("adv_step_cluster_gen: workspace too small"); return ADVMIL_ERR_WORKSPACE; }
  STEP_TAKE(hh, float, (size_t)nbc * h);
  STEP_TAKE(ab, float, (size_t)nbc * gate_width(h));
  const size_t gws_bytes = advmil_generator_workspace_bytes(&gp, nbc, nb, 1);
  STEP_TAKE(gws, char, gws_bytes);
  AdvmilGenActs ga{};
  ga.h = hh; ga.ab = ab; ga.s = gb.s; ga.w = gb.w; ga.z = gb.z; ga.H = gb.H; ga.H1 = gb.H1; ga.pre = gb.pre;
  ga.pred = a->pred_g; ga.noise0 = nullptr; ga.noise1 = a->noise_g;
  ga.mask_h = a->g_mask_h; ga.mask_a = a->g_mask_a; ga.mask_b = a->g_mask_b; ga.mask_rho = nullptr; ga.mask_mlp0 = a->g_mask_mlp0;
  ga.seed = a->seed_g; ga.train = 1; ga.precision = ADVMIL_FP32; ga.workspace = gws; ga.workspace_bytes = gws_bytes;
  ADVMIL_TRY(advmil_generator_fwd(&gp, &cb, &ga, stream));
  // ---- D(x, pred_g), G loss, dL/dpred_g ----
  STEP_TAKE(d_pred, float, nb);
  ADVMIL_TRY(gen_rlip(a, ws, B.demb, !first, d_pred, who, st));
  // ---- attention stage backward down to d_hc, then K9's backward and dWphi / dbphi ----
  STEP_TAKE(d_hc, float, (size_t)nbc * h);
  AdvmilGenGrads gg = *a->gen_grads;
  gg.dx = d_hc;
  ADVMIL_TRY(advmil_generator_bwd(&gp, &cb, &ga, d_pred, &gg, stream));
  STEP_TAKE(d_hx, char, (size_t)rows * h * elem_bytes(dt));
  if (B.keep) {
    ProfScope ps(PROF_BWD_DATA, st);
    ADVMIL_TRY(cluster_pool_bwd(d_hc, B.keep, ca->cid, bags->offsets, B.counts, rows, nb, h, ncl, prec, d_hx, st));
  } else {
    ADVMIL_TRY(advmil_segment_mean_by_id_bwd(d_hc, B.hx, dt, ca->cid, bags->offsets, B.counts, rows, nb, h, ncl, 1, d_hx, stream));
  }
  STEP_TAKE(bwws, float, bwd_weight_ws_floats(rows, h, C));
  { ProfScope ps(PROF_BWD_W_PROJ, st); ADVMIL_TRY(bwd_weight(d_hx, bags->x, rows, h, C, ca->dWphi, 0, bwws, prec, st)); }
  STEP_TAKE(csws, float, (size_t)row_chunks(rows) * h);
  { ProfScope ps(PROF_COLSUM, st); ADVMIL_TRY(colsum(d_hx, dt, rows, h, h, ca->dbphi, 0, csws, st)); }
  return ADVMIL_OK;
}

extern "C" int advmil_adv_step_cluster_gen(const AdvmilClusterStepArgs* ca, void* stream) {
  return cluster_gen_phase(ca, true, __func__, (cudaStream_t)stream);
}
extern "C" int advmil_adv_step_cluster_gen_next(const AdvmilClusterStepArgs* ca, void* stream) {
  return cluster_gen_phase(ca, false, __func__, (cudaStream_t)stream);
}
