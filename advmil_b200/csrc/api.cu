// C-ABI composites: generator fwd/bwd, discriminator embed/head fwd/bwd, stage-level entry points.
// Host orchestration only — every kernel lives in gemm_*.cu / seg_kernels.cu / tail_kernels.cu.
#include <stdarg.h>
#include <string.h>
#include <atomic>
#include <mutex>
#include <vector>
#include "stages.cuh"

namespace advmil {

static thread_local char g_err[512] = "";
static std::atomic<long long> g_launches{0};

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
void count_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }

// ---- per-stage event profiling ------------------------------------------------------------------
struct ProfRec { int tag; cudaEvent_t a, b; };
static std::atomic<int> g_prof_on{0};
static std::mutex g_prof_mu;
static std::vector<ProfRec*> g_prof;
ProfScope::ProfScope(int tag_, cudaStream_t st_) : tag(tag_), st(st_), rec(nullptr) {
  if (!g_prof_on.load(std::memory_order_relaxed)) return;
  ProfRec* r = new ProfRec{tag, nullptr, nullptr};
  if (cudaEventCreate(&r->a) != cudaSuccess || cudaEventCreate(&r->b) != cudaSuccess) { delete r; return; }
  cudaEventRecord(r->a, st);
  rec = r;
}
ProfScope::~ProfScope() {
  if (!rec) return;
  ProfRec* r = (ProfRec*)rec;
  cudaEventRecord(r->b, st);
  std::lock_guard<std::mutex> lk(g_prof_mu);
  g_prof.push_back(r);
}

__global__ void scale_offsets_kernel(const int32_t* __restrict__ in, int n, int div, int32_t* __restrict__ out) {
  pdl_prologue();
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = in[i] / div;
}

static int check_bags(const AdvmilBags* b, int C, bool need16, int precision) {
  ADVMIL_REQUIRE(b && b->x && b->offsets && b->offsets_host, "bags: null pointer");
  ADVMIL_REQUIRE(precision >= ADVMIL_FP32 && precision <= ADVMIL_BF16, "unknown precision mode %d", precision);
  ADVMIL_REQUIRE(b->elem == elem_of_precision(precision), "bags: x element type %d does not match precision mode %d (bf16 x <=> ADVMIL_BF16)",
                 b->elem, precision);
  ADVMIL_REQUIRE(b->bags > 0 && b->rows > 0, "bags: empty batch (rows=%d bags=%d)", b->rows, b->bags);
  ADVMIL_REQUIRE(b->C == C, "bags: feature width %d != model input width %d", b->C, C);
  ADVMIL_REQUIRE(b->offsets_host[0] == 0 && b->offsets_host[b->bags] == b->rows, "bags: offsets must span [0, rows]");
  for (int i = 0; i < b->bags; ++i) {
    int len = b->offsets_host[i + 1] - b->offsets_host[i];
    ADVMIL_REQUIRE(len > 0, "bags: bag %d is empty", i);
    if (need16) ADVMIL_REQUIRE(len % 16 == 0, "bags: bag %d has %d rows, not a multiple of 16 (model/backbone_utils.py:65)", i, len);
  }
  return ADVMIL_OK;
}

#define WS_TAKE(var, type, count)                                                        \
  type* var = ws.take<type>(count);                                                      \
  if (!var) { set_error("%s: workspace too small (need > %zu bytes)", __func__, ws.cap); return ADVMIL_ERR_WORKSPACE; }

}  // namespace advmil

using namespace advmil;

extern "C" int advmil_abi_version(void) { return ADVMIL_ABI_VERSION; }
extern "C" const char* advmil_last_error(void) { return g_err; }
extern "C" size_t advmil_abi_sizeof(int which) {
  switch (which) {
    case 0: return sizeof(AdvmilBags);
    case 1: return sizeof(AdvmilGenParams);
    case 2: return sizeof(AdvmilGenGrads);
    case 3: return sizeof(AdvmilGenActs);
    case 4: return sizeof(AdvmilDiscParams);
    case 5: return sizeof(AdvmilDiscGrads);
    case 6: return sizeof(AdvmilEmbedActs);
    case 7: return sizeof(AdvmilHeadActs);
    case 8: return sizeof(AdvmilStepArgs);
    case 9: return sizeof(AdvmilEsatParams);
    case 10: return sizeof(AdvmilEsatGrads);
    case 11: return sizeof(AdvmilEsatActs);
    case 12: return sizeof(AdvmilEsatStepArgs);
    case 13: return sizeof(AdvmilClusterStepArgs);
    default: return 0;
  }
}
extern "C" int64_t advmil_launch_count(int reset) {
  long long v = g_launches.load();
  if (reset) g_launches.store(0);
  return v;
}
extern "C" int32_t advmil_gate_packed_width(int32_t D) { return gate_width(D); }
extern "C" int advmil_profile_enable(int on) { g_prof_on.store(on ? 1 : 0); return ADVMIL_OK; }
extern "C" int advmil_profile_read(double* ms, int64_t* counts, int32_t ntags) {
  ADVMIL_CHECK_CUDA(cudaDeviceSynchronize());
  std::lock_guard<std::mutex> lk(g_prof_mu);
  for (int i = 0; i < ntags; ++i) { ms[i] = 0.0; counts[i] = 0; }
  for (ProfRec* r : g_prof) {
    float t = 0.f;
    if (cudaEventElapsedTime(&t, r->a, r->b) == cudaSuccess && r->tag < ntags) { ms[r->tag] += t; counts[r->tag] += 1; }
    cudaEventDestroy(r->a); cudaEventDestroy(r->b);
    delete r;
  }
  g_prof.clear();
  return ADVMIL_OK;
}

// =============================================================================================
// generator
// =============================================================================================
extern "C" size_t advmil_generator_workspace_bytes(const AdvmilGenParams* p, int32_t rows, int32_t bags, int32_t backward) {
  const size_t h = p->h, C = p->C, o = p->o, hid = p->hid;
  const size_t abw = gate_width(p->h);
  size_t f = 0;  // floats
  f += abw * h + abw + 512;                                   // packed gate weights
  f += (abw / 128) * (size_t)rows + 256;                      // gate score partials
  f += seg_pool_ws_floats(rows, bags, (int)h) + 256;
  if (backward) {
    f += (size_t)bags * (h + o + hid + 1) + 1024;             // per-bag gradient vectors
    f += (size_t)rows * abw + (size_t)rows * h + 512;         // dAB, dh_pre
    f += abw * h + abw + 512;                                 // packed gate weight grads
    f += pool_gate_ws_floats(rows, bags, (int)h) + 256;       // pool_gate partials
    f += max(bwd_weight_ws_floats(rows, (int)abw, (int)h), bwd_weight_ws_floats(rows, (int)h, (int)C)) + 256;
    f += (size_t)4 * row_chunks(rows) * max(abw, h) + 256;    // colsum partials
  }
  return f * sizeof(float) + 64 * 256;
}

extern "C" int advmil_generator_fwd(const AdvmilGenParams* p, const AdvmilBags* bags, AdvmilGenActs* a, void* stream) {
  ADVMIL_REQUIRE(p && a, "generator_fwd: null argument");
  ADVMIL_TRY(check_bags(bags, p->C, false, a->precision));
  ADVMIL_REQUIRE(p->h % 4 == 0 && p->C % 4 == 0, "generator_fwd: C=%d and h=%d must be multiples of 4", p->C, p->h);
  ADVMIL_REQUIRE(a->h && a->s && a->w && a->z && (a->pred || !p->W0), "generator_fwd: missing output buffers");
  cudaStream_t st = (cudaStream_t)stream;
  const int rows = bags->rows, nb = bags->bags, h = p->h;
  const int abw = gate_width(h);
  Workspace ws(a->workspace, a->workspace_bytes);
  WS_TAKE(Wp, float, (size_t)abw * h);
  WS_TAKE(bp, float, abw);
  WS_TAKE(part, float, (size_t)(abw / 128) * rows);
  WS_TAKE(poolws, float, seg_pool_ws_floats(rows, nb, h));
  Drop dh = Drop::make(a->mask_h, a->seed, SITE_H, p->p_backbone, a->train, p->h);
  Drop da = Drop::make(a->mask_a, a->seed, SITE_A, p->p_backbone, a->train, p->h);
  Drop db = Drop::make(a->mask_b, a->seed, SITE_B, p->p_backbone, a->train, p->h);
  Drop::pair_gate(da, db);
  Drop drho = Drop::make(a->mask_rho, a->seed, SITE_RHO, p->p_backbone, a->train, p->o);
  Drop dmlp0 = Drop::make(a->mask_mlp0, a->seed, SITE_MLP0, p->p_head, a->train, p->hid);
  const int dt = elem_of_precision(a->precision);
  if (a->h_ready) { /* `h` was written by an earlier eval pass (h_drop_out) */ }
  else if (a->h_eval) { ProfScope ps(PROF_DROPOUT, st); ADVMIL_TRY(apply_dropout(a->h_eval, rows, h, dh, a->h, dt, st)); }
  else {
    ProfScope ps(PROF_PROJ, st);
    Drop d2 = Drop::make(a->mask_h_drop, a->seed_drop, SITE_H, p->p_backbone, 1, p->h);
    ADVMIL_TRY(linear_fwd(bags->x, p->W1, p->b1, rows, p->C, h, 1, dh, a->h, a->precision, st, a->h_drop_out,
                          a->h_drop_out ? &d2 : nullptr));
  }
  { ProfScope ps(PROF_GEN_TAIL, st); ADVMIL_TRY(gate_pack_weights(p->Wa, p->ba, p->Wb, p->bb, h, h, Wp, bp, st)); }
  { ProfScope ps(PROF_GATE, st);
    ADVMIL_TRY(gated_score_fwd(a->h, Wp, bp, p->wc, p->bc, rows, h, h, da, db, a->ab, nullptr, part, a->precision, st)); }
  { ProfScope ps(PROF_POOL, st);
    ADVMIL_TRY(seg_softmax_pool_fwd(a->s, part, abw / 128, p->bc, a->h, dt, bags->offsets, bags->offsets_host, rows, nb, h, a->w,
                                    a->z, nullptr, poolws, st)); }
  { ProfScope ps(PROF_GEN_TAIL, st);
    ADVMIL_TRY(gen_head_fwd(*p, a->z, a->noise0, a->noise1, nb, 1, drho, dmlp0, a->H, a->H1, a->pre, a->pred, st)); }
  return ADVMIL_OK;
}

extern "C" int advmil_generator_bwd(const AdvmilGenParams* p, const AdvmilBags* bags, const AdvmilGenActs* a,
                                    const float* d_pred, AdvmilGenGrads* g, void* stream) {
  ADVMIL_REQUIRE(p && a && g && d_pred, "generator_bwd: null argument");
  ADVMIL_TRY(check_bags(bags, p->C, false, a->precision));
  ADVMIL_REQUIRE(!(g->dx && a->precision == ADVMIL_BF16), "generator_bwd: dx is not available in the bf16 mode");
  ADVMIL_REQUIRE(a->ab && a->H && (a->H1 || !p->W0), "generator_bwd: forward was run without saving activations (ab/H/H1)");
  cudaStream_t st = (cudaStream_t)stream;
  const int rows = bags->rows, nb = bags->bags, h = p->h, o = p->o, hid = p->hid, C = p->C;
  const int abw = gate_width(h);
  const int prec = a->precision, dt = elem_of_precision(a->precision);
  Workspace ws(a->workspace, a->workspace_bytes);
  WS_TAKE(Wp, float, (size_t)abw * h);
  WS_TAKE(bp, float, abw);
  WS_TAKE(dz, float, (size_t)nb * h);
  WS_TAKE(dHpre, float, (size_t)nb * o);
  WS_TAKE(dH1pre, float, (size_t)nb * hid);
  WS_TAKE(dpre, float, nb);
  WS_TAKE(dAB, float, (size_t)rows * abw);
  WS_TAKE(dhpre, float, (size_t)rows * h);
  WS_TAKE(dWp, float, (size_t)abw * h);
  WS_TAKE(dbp, float, abw);
  WS_TAKE(pgws, float, pool_gate_ws_floats(rows, nb, h));
  WS_TAKE(bwws, float, max(bwd_weight_ws_floats(rows, abw, h), bwd_weight_ws_floats(rows, h, C)));
  WS_TAKE(csws, float, (size_t)4 * row_chunks(rows) * max(abw, h));
  const float ik_bb = (a->train && p->p_backbone > 0.f) ? 1.f / (1.f - p->p_backbone) : 1.f;
  const float ik_hd = (a->train && p->p_head > 0.f) ? 1.f / (1.f - p->p_head) : 1.f;
  Drop da = Drop::make(a->mask_a, a->seed, SITE_A, p->p_backbone, a->train, p->h);
  Drop db = Drop::make(a->mask_b, a->seed, SITE_B, p->p_backbone, a->train, p->h);
  Drop::pair_gate(da, db);
  // head
  { ProfScope ps(PROF_GEN_TAIL, st);
    ADVMIL_TRY(gen_head_bwd(*p, d_pred, a->H, a->H1, a->pred, nb, ik_bb, ik_hd, dz, dHpre, dH1pre, dpre, st));
    OuterProb op[OUTER_MAX];
    int nop = 0;
    if (p->W0) {
      op[nop++] = OuterProb{dpre, a->H1, hid, a->noise1, p->noise1 ? hid : 0, 1, g->Wl, g->bl};
      op[nop++] = OuterProb{dH1pre, a->H, o, a->noise0, p->noise0 ? o : 0, hid, g->W0, g->b0};
    }
    if (p->Wrho) op[nop++] = OuterProb{dHpre, a->z, h, nullptr, 0, o, g->Wrho, g->brho};
    ADVMIL_TRY(outer_sum_multi(op, nop, nb, 0, st));
    // pooling + gate
    ADVMIL_TRY(gate_pack_weights(p->Wa, p->ba, p->Wb, p->bb, h, h, Wp, bp, st));
  }
  { ProfScope ps(PROF_POOL_BWD, st);
    ADVMIL_TRY(pool_gate_bwd(a->h, a->w, a->z, dz, a->ab, p->wc, bags->offsets, rows, nb, h, h, da, db, dAB, g->wc, g->bc, dbp, 0, pgws, dt, st)); }
  BwdDataExtras ex;
  ex.w = a->w; ex.dz = dz; ex.offsets = bags->offsets; ex.bags = nb; ex.relu_src = a->h; ex.ld_src = h; ex.inv_keep = ik_bb;
  const bool fused_b1 = bwd_data_fuses_colsum(rows, abw, h, prec);   // db1 = column sums of dh: from the GEMM epilogue
  if (fused_b1) ex.colsum_part = csws;
  { ProfScope ps(PROF_BWD_DATA, st); ADVMIL_TRY(bwd_data(dAB, Wp, rows, abw, h, dhpre, ex, prec, st)); }
  { ProfScope ps(PROF_BWD_W_GATE, st); ADVMIL_TRY(bwd_weight(dAB, a->h, rows, abw, h, dWp, 0, bwws, prec, st)); }
  { ProfScope ps(PROF_GEN_TAIL, st); ADVMIL_TRY(gate_unpack_grads(dWp, dbp, h, h, g->Wa, g->ba, g->Wb, g->bb, 0, st)); }
  // first layer
  { ProfScope ps(PROF_BWD_W_PROJ, st); ADVMIL_TRY(bwd_weight(dhpre, bags->x, rows, h, C, g->W1, 0, bwws, prec, st)); }
  { ProfScope ps(PROF_COLSUM, st);
    if (fused_b1) ADVMIL_TRY(reduce_rows(csws, 4 * cdiv(rows, 128), h, g->b1, 0, st));
    else ADVMIL_TRY(colsum(dhpre, dt, rows, h, h, g->b1, 0, csws, st)); }
  if (g->dx) {
    BwdDataExtras exx;
    ADVMIL_TRY(bwd_data(dhpre, p->W1, rows, h, C, g->dx, exx, prec, st));
  }
  return ADVMIL_OK;
}

extern "C" int advmil_generator_sample(const AdvmilGenParams* p, const float* H, const float* noise0,
                                       const float* noise1, int32_t bags, int32_t samples, float* out, void* stream) {
  ADVMIL_REQUIRE(p && H && out && bags > 0 && samples > 0, "generator_sample: bad arguments");
  // H is the backbone output (post rho); run only MLPs + out scale: present H as "z" with the rho layer disabled
  AdvmilGenParams q = *p;
  q.Wrho = nullptr; q.brho = nullptr; q.h = p->o;
  Drop none = Drop::make(nullptr, 0, 0, 0.f, 0, 0);
  return gen_head_fwd(q, H, noise0, noise1, bags, samples, none, none, nullptr, nullptr, nullptr, out, (cudaStream_t)stream);
}

// =============================================================================================
// discriminator
// =============================================================================================
// the patch embedding's kernel size: 1 (ksize 0 = the ABI's zero default) or 3
static int disc_ksize(const AdvmilDiscParams* p) { return p->ksize == 0 ? 1 : p->ksize; }
static int check_ksize(const AdvmilDiscParams* p) {
  ADVMIL_REQUIRE(p->ksize == 0 || p->ksize == 1 || p->ksize == 3, "disc: patch-embedding ksize %d unsupported (0, 1 or 3)", p->ksize);
  return ADVMIL_OK;
}

extern "C" size_t advmil_disc_workspace_bytes(const AdvmilDiscParams* p, int32_t rows, int32_t bags, int32_t backward) {
  const size_t d = p->d, dh = p->d / 2, R = rows / 16;
  const size_t Kc = (size_t)p->C * disc_ksize(p) * disc_ksize(p);     // columns of the embedding's weight operand
  const size_t abw = gate_width(p->d);
  size_t f = 0;
  // head forward
  f += abw * d + abw + 512 + (abw / 128) * R + 256 + seg_pool_ws_floats((int)R, bags, (int)d) + 256 + (bags + 1) + 64;
  if (backward) {
    // embed backward
    size_t e = (size_t)rows * d + (size_t)row_chunks(rows) * 3 * d + bwd_weight_ws_floats(rows, (int)d, (int)Kc) + 1024;
    // head backward
    size_t hb = (size_t)bags * (3 * d + dh + p->t2 + p->t1 + 2) + 2048;
    hb += R * abw + R * d + R * dh + abw * d + abw + 1024;
    hb += pool_gate_ws_floats((int)R, bags, (int)d) + 256;
    hb += max(bwd_weight_ws_floats((int)R, (int)abw, (int)d), bwd_weight_ws_floats((int)R, (int)d, (int)dh)) + 256;
    hb += (size_t)row_chunks((int)R) * abw + 256 + (size_t)8 * row_chunks((int)R) * d + 512;
    f += max(e, hb);
  }
  return f * sizeof(float) + 64 * 256;
}

extern "C" int advmil_disc_embed_fwd(const AdvmilDiscParams* p, const AdvmilBags* bags, AdvmilEmbedActs* a, void* stream) {
  ADVMIL_REQUIRE(p && a && a->emb, "disc_embed_fwd: null argument");
  ADVMIL_TRY(check_bags(bags, p->C, true, a->precision));
  ADVMIL_TRY(check_ksize(p));
  ProfScope ps(PROF_EMBED, (cudaStream_t)stream);
  // the fp32 embedding at d = 256 writes y before its LayerNorm pass: into y_pre, or into the workspace when y_pre is not saved
  const size_t y_bytes = (size_t)bags->rows * p->d * sizeof(float);
  float* y_ws = (a->workspace && a->workspace_bytes >= y_bytes) ? (float*)a->workspace : nullptr;
  return region_embed_fwd(bags->x, p->Wc, p->bc, p->ln_g, p->ln_b, bags->rows, p->C, p->d, p->ln_eps, a->y_pre, a->emb,
                          a->precision, (cudaStream_t)stream, disc_ksize(p), y_ws);
}

namespace advmil {
int disc_embed_bwd_impl(const AdvmilDiscParams* p, const AdvmilBags* bags, const AdvmilEmbedActs* a, const float* d_emb,
                        const float* d_emb2, AdvmilDiscGrads* g, int accumulate, cudaStream_t st) {
  ADVMIL_REQUIRE(p && a && d_emb && g, "disc_embed_bwd: null argument");
  ADVMIL_REQUIRE(a->y_pre, "disc_embed_bwd: forward was run without saving y_pre");
  ADVMIL_TRY(check_bags(bags, p->C, true, a->precision));
  ADVMIL_TRY(check_ksize(p));
  const int rows = bags->rows, d = p->d, C = p->C, ks = disc_ksize(p);
  Workspace ws(a->workspace, a->workspace_bytes);
  WS_TAKE(d_y, float, (size_t)rows * d);
  WS_TAKE(lnws, float, (size_t)row_chunks(rows) * 3 * d);
  WS_TAKE(bwws, float, bwd_weight_ws_floats(rows, d, ks * ks * C));
  { ProfScope ps(PROF_LN_BWD, st);
    ADVMIL_TRY(ln_pool_bwd(a->y_pre, d_emb, d_emb2, p->ln_g, p->ln_b, rows, d, p->ln_eps, d_y, g->ln_g, g->ln_b, g->bc, accumulate, lnws,
                           elem_of_precision(a->precision), st)); }
  { ProfScope ps(PROF_BWD_W_EMBED, st);
    if (ks == 3) ADVMIL_TRY(bwd_weight_conv3(d_y, bags->x, rows, d, C, g->Wc, accumulate, bwws, a->precision, st));
    else ADVMIL_TRY(bwd_weight(d_y, bags->x, rows, d, C, g->Wc, accumulate, bwws, a->precision, st)); }
  return ADVMIL_OK;
}
}  // namespace advmil

extern "C" int advmil_disc_embed_bwd(const AdvmilDiscParams* p, const AdvmilBags* bags, const AdvmilEmbedActs* a,
                                     const float* d_emb, AdvmilDiscGrads* g, int32_t accumulate, void* stream) {
  return disc_embed_bwd_impl(p, bags, a, d_emb, nullptr, g, accumulate, (cudaStream_t)stream);
}

namespace {
struct RegionOffsets {
  std::vector<int32_t> host;
  int32_t* dev;
};
}  // namespace

static int make_region_offsets(const AdvmilBags* bags, Workspace& ws, cudaStream_t st, RegionOffsets& ro) {
  ro.host.resize(bags->bags + 1);
  for (int i = 0; i <= bags->bags; ++i) ro.host[i] = bags->offsets_host[i] / 16;
  ro.dev = ws.take<int32_t>(bags->bags + 1);
  if (!ro.dev) { set_error("disc_head: workspace too small"); return ADVMIL_ERR_WORKSPACE; }
  launch_k(scale_offsets_kernel, dim3(cdiv(bags->bags + 1, 128)), dim3(128), 0, st, bags->offsets, bags->bags + 1, 16, ro.dev);
  ADVMIL_CHECK_LAUNCH();
  return ADVMIL_OK;
}

extern "C" int advmil_disc_head_fwd(const AdvmilDiscParams* p, const AdvmilBags* bags, AdvmilHeadActs* a, void* stream) {
  ADVMIL_REQUIRE(p && a && a->emb && a->t && a->out, "disc_head_fwd: null argument");
  ADVMIL_TRY(check_bags(bags, p->C, true, bags ? (bags->elem == ELEM_BF16 ? ADVMIL_BF16 : ADVMIL_FP32) : 0));
  ADVMIL_REQUIRE(a->f1 && a->fi && a->rep && a->attn && a->bagv && a->fbar && a->g1 && a->hx && a->u1 && a->ht,
                 "disc_head_fwd: missing activation buffers");
  cudaStream_t st = (cudaStream_t)stream;
  ProfScope ps(PROF_HEAD_FWD, st);
  const int nb = bags->bags, d = p->d, dh = p->d / 2, R = bags->rows / 16;
  const int abw = gate_width(d);
  Workspace ws(a->workspace, a->workspace_bytes);
  RegionOffsets ro;
  ADVMIL_TRY(make_region_offsets(bags, ws, st, ro));
  WS_TAKE(Wp, float, (size_t)abw * d);
  WS_TAKE(bp, float, abw);
  WS_TAKE(part, float, (size_t)(abw / 128) * R);
  WS_TAKE(poolws, float, seg_pool_ws_floats(R, nb, d));
  Drop dfc1 = Drop::make(a->mask_fc1, a->seed, SITE_FC1, p->p, a->train, p->d / 2);
  Drop dga = Drop::make(a->mask_ga, a->seed, SITE_GA, p->p, a->train, p->d);
  Drop dgs = Drop::make(a->mask_gs, a->seed, SITE_GS, p->p, a->train, p->d);
  Drop::pair_gate(dga, dgs);
  Drop dfc2 = Drop::make(a->mask_fc2, a->seed, SITE_FC2, p->p, a->train, p->d / 2);
  Drop none = Drop::make(nullptr, 0, 0, 0.f, 0, 0);
  // region-level tensors are fp32; outside the exact-fp32 mode their contractions run on the tcgen05 tf32 pipe
  const int rp = region_precision(a->precision, a->train != 0);
  if (rlip_chain_supported(d)) {      // one fp32-grade kernel for the region-level chain (rlip_chain.cu: split-tf32 mma.sync), every precision mode
    ADVMIL_TRY(rlip_chain_fwd(a->emb, *p, R, dfc1, dga, dgs, a->f1, a->fi, a->ab, part, st));
  } else {
    ADVMIL_TRY(linear_fwd(a->emb, p->F1a_w, p->F1a_b, R, d, dh, 1, dfc1, a->f1, rp, st));
    ADVMIL_TRY(linear_fwd(a->f1, p->F1b_w, p->F1b_b, R, dh, d, 0, none, a->fi, rp, st));
    ADVMIL_TRY(gate_pack_weights(p->Pg_w, p->Pg_b, p->Ps_w, p->Ps_b, d, d, Wp, bp, st));
    ADVMIL_TRY(gated_score_fwd(a->fi, Wp, bp, p->Pc_w, p->Pc_b, R, d, d, dga, dgs, a->ab, nullptr, part, rp, st));
  }
  ADVMIL_TRY(seg_softmax_pool_fwd(a->rep, part, abw / 128, p->Pc_b, a->fi, ELEM_F32, ro.dev, ro.host.data(), R, nb, d, a->attn,
                                  a->bagv, a->fbar, poolws, st));
  ADVMIL_TRY(rlip_tail_fwd(*p, a->bagv, a->fbar, a->t, nb, dfc2, a->g1, a->hx, a->u1, a->ht, a->out, st));
  return ADVMIL_OK;
}

extern "C" int advmil_disc_head_bwd(const AdvmilDiscParams* p, const AdvmilBags* bags, const AdvmilHeadActs* a,
                                    const float* d_out, float* d_emb, float* d_t, AdvmilDiscGrads* g,
                                    int32_t accumulate, void* stream) {
  ADVMIL_REQUIRE(p && a && d_out, "disc_head_bwd: null argument");
  ADVMIL_TRY(check_bags(bags, p->C, true, bags ? (bags->elem == ELEM_BF16 ? ADVMIL_BF16 : ADVMIL_FP32) : 0));
  cudaStream_t st = (cudaStream_t)stream;
  ProfScope ps(PROF_HEAD_BWD, st);
  const int nb = bags->bags, d = p->d, dh = p->d / 2, R = bags->rows / 16, t1 = p->t1, t2 = p->t2;
  const int abw = gate_width(d);
  const float ik = (a->train && p->p > 0.f) ? 1.f / (1.f - p->p) : 1.f;
  // backward: plain tf32 in the bf16 mode -- its 1e-3 relative errors land in the gradients unamplified; what the real/fake
  // cancellation amplifies is the error of the FORWARD outputs f (through dL/df), and the training forward runs split tf32
  const int rp = region_precision(a->precision, false);
  Workspace ws(a->workspace, a->workspace_bytes);
  RegionOffsets ro;
  ADVMIL_TRY(make_region_offsets(bags, ws, st, ro));
  WS_TAKE(d_fbar, float, (size_t)nb * d);
  WS_TAKE(d_bagv, float, (size_t)nb * d);
  WS_TAKE(d_hx, float, (size_t)nb * d);
  WS_TAKE(d_g1pre, float, (size_t)nb * dh);
  WS_TAKE(d_htpre, float, (size_t)nb * t2);
  WS_TAKE(d_u1pre, float, (size_t)nb * t1);
  WS_TAKE(d_t_scratch, float, nb);
  ADVMIL_TRY(rlip_tail_bwd(*p, d_out, a->bagv, a->fbar, a->g1, a->hx, a->u1, a->ht, nb, ik, d_fbar, d_bagv, d_hx, d_g1pre,
                           d_htpre, d_u1pre, d_t ? d_t : d_t_scratch, st));
  if (!d_emb && !g) return ADVMIL_OK;  // G step: only dL/dt is needed from D (SURVEY.md A.2)
  if (g) {
    OuterProb op[OUTER_MAX];
    int nop = 0;
    op[nop++] = OuterProb{d_hx, a->g1, dh, nullptr, 0, d, g->F2b_w, g->F2b_b};
    op[nop++] = OuterProb{d_g1pre, a->bagv, d, nullptr, 0, dh, g->F2a_w, g->F2a_b};
    op[nop++] = OuterProb{d_htpre, a->u1, t1, nullptr, 0, t2, g->T2_w, g->T2_b};
    op[nop++] = OuterProb{d_u1pre, a->t, 1, nullptr, 0, t1, g->T1_w, g->T1_b};
    if (p->prj_path == 1) op[nop++] = OuterProb{d_out, a->hx, d, nullptr, 0, 1, g->Pr_w, g->Pr_b};
    else if (p->prj_path == 2) op[nop++] = OuterProb{d_out, a->ht, t2, nullptr, 0, 1, g->Pr_w, g->Pr_b};
    else if (p->prj_path == 3) op[nop++] = OuterProb{d_out, a->hx, d, a->ht, t2, 1, g->Pr_w, g->Pr_b};
    ADVMIL_TRY(outer_sum_multi(op, nop, nb, accumulate, st));
  }
  WS_TAKE(Wp, float, (size_t)abw * d);
  WS_TAKE(bp, float, abw);
  WS_TAKE(dAB, float, (size_t)R * abw);
  WS_TAKE(d_fi, float, (size_t)R * d);
  WS_TAKE(d_f1pre, float, (size_t)R * dh);
  WS_TAKE(dWp, float, (size_t)abw * d);
  WS_TAKE(dbp, float, abw);
  WS_TAKE(dwc_scratch, float, d + 1);
  WS_TAKE(pgws, float, pool_gate_ws_floats(R, nb, d));
  WS_TAKE(bwws, float, max(bwd_weight_ws_floats(R, abw, d), bwd_weight_ws_floats(R, d, dh)));
  WS_TAKE(csws, float, (size_t)row_chunks(R) * abw);
  WS_TAKE(cp_fi, float, (size_t)4 * row_chunks(R) * d);      // column-sum partials from the backward-data epilogues
  WS_TAKE(cp_f1, float, (size_t)4 * row_chunks(R) * d);
  Drop dga = Drop::make(a->mask_ga, a->seed, SITE_GA, p->p, a->train, p->d);
  Drop dgs = Drop::make(a->mask_gs, a->seed, SITE_GS, p->p, a->train, p->d);
  Drop::pair_gate(dga, dgs);
  ADVMIL_TRY(gate_pack_weights(p->Pg_w, p->Pg_b, p->Ps_w, p->Ps_b, d, d, Wp, bp, st));
  ADVMIL_TRY(pool_gate_bwd(a->fi, a->attn, a->bagv, d_bagv, a->ab, p->Pc_w, ro.dev, R, nb, d, d, dga, dgs, dAB,
                           g ? g->Pc_w : dwc_scratch, g ? g->Pc_b : dwc_scratch + d, g ? dbp : nullptr, g ? accumulate : 0, pgws,
                           ELEM_F32, st));
  BwdDataExtras ex;
  ex.w = a->attn; ex.dz = d_bagv; ex.dmean = (p->inner_instance && p->prj_path != 3) ? d_fbar : nullptr; ex.offsets = ro.dev; ex.bags = nb;
  const bool fuse_fi = g && bwd_data_fuses_colsum(R, abw, d, rp), fuse_f1 = g && bwd_data_fuses_colsum(R, d, dh, rp);
  if (fuse_fi) ex.colsum_part = cp_fi;
  ADVMIL_TRY(bwd_data(dAB, Wp, R, abw, d, d_fi, ex, rp, st));
  if (g) {
    ADVMIL_TRY(bwd_weight(dAB, a->fi, R, abw, d, dWp, 0, bwws, rp, st));
    ADVMIL_TRY(gate_unpack_grads(dWp, dbp, d, d, g->Pg_w, g->Pg_b, g->Ps_w, g->Ps_b, accumulate, st));
  }
  BwdDataExtras ex1;
  ex1.relu_src = a->f1; ex1.ld_src = dh; ex1.inv_keep = ik;
  if (fuse_f1) ex1.colsum_part = cp_f1;
  ADVMIL_TRY(bwd_data(d_fi, p->F1b_w, R, d, dh, d_f1pre, ex1, rp, st));
  if (g) {
    ADVMIL_TRY(bwd_weight(d_fi, a->f1, R, d, dh, g->F1b_w, accumulate, bwws, rp, st));
    if (fuse_fi) ADVMIL_TRY(reduce_rows(cp_fi, 4 * cdiv(R, 128), d, g->F1b_b, accumulate, st));
    else ADVMIL_TRY(colsum(d_fi, ELEM_F32, R, d, d, g->F1b_b, accumulate, csws, st));
    ADVMIL_TRY(bwd_weight(d_f1pre, a->emb, R, dh, d, g->F1a_w, accumulate, bwws, rp, st));
    if (fuse_f1) ADVMIL_TRY(reduce_rows(cp_f1, 4 * cdiv(R, 128), dh, g->F1a_b, accumulate, st));
    else ADVMIL_TRY(colsum(d_f1pre, ELEM_F32, R, dh, dh, g->F1a_b, accumulate, csws, st));
  }
  if (d_emb) {
    BwdDataExtras ex2;
    ex2.accumulate = accumulate;
    ADVMIL_TRY(bwd_data(d_f1pre, p->F1a_w, R, dh, d, d_emb, ex2, rp, st));
  }
  return ADVMIL_OK;
}

// =============================================================================================
// stage-level entry points
// =============================================================================================
extern "C" int advmil_linear_fwd(const void* x, const float* W, const float* b, int32_t rows, int32_t K, int32_t N,
                                 int32_t act, float p_drop, const uint8_t* mask, uint64_t seed, int32_t site,
                                 int32_t train, int32_t precision, void* y, void* stream) {
  ADVMIL_REQUIRE(x && W && y && rows >= 0, "linear_fwd: null argument");
  Drop dr = Drop::make(mask, seed, SITE_USER + site, p_drop, train, N);
  return linear_fwd(x, W, b, rows, K, N, act, dr, y, precision, (cudaStream_t)stream);
}

extern "C" size_t advmil_linear_bwd_workspace_bytes(int32_t rows, int32_t K, int32_t N) {
  return (bwd_weight_ws_floats(rows, N, K) + (size_t)row_chunks(rows) * N + 1024) * sizeof(float);
}

extern "C" int advmil_linear_bwd(const void* dY, const void* X, const float* W, int32_t rows, int32_t K, int32_t N,
                                 void* dX, float* dW, float* db, int32_t accumulate, int32_t precision, void* workspace,
                                 size_t workspace_bytes, void* stream) {
  ADVMIL_REQUIRE(dY, "linear_bwd: null dY");
  cudaStream_t st = (cudaStream_t)stream;
  Workspace ws(workspace, workspace_bytes);
  if (dX) {
    ADVMIL_REQUIRE(W, "linear_bwd: dX needs W");
    BwdDataExtras ex; ex.accumulate = accumulate;
    ADVMIL_TRY(bwd_data(dY, W, rows, N, K, dX, ex, precision, st));
  }
  if (dW) {
    ADVMIL_REQUIRE(X, "linear_bwd: dW needs X");
    WS_TAKE(bwws, float, bwd_weight_ws_floats(rows, N, K));
    ADVMIL_TRY(bwd_weight(dY, X, rows, N, K, dW, accumulate, bwws, precision, st));
  }
  if (db) {
    WS_TAKE(csws, float, (size_t)row_chunks(rows) * N);
    ADVMIL_TRY(colsum(dY, elem_of_precision(precision), rows, N, N, db, accumulate, csws, st));
  }
  return ADVMIL_OK;
}

extern "C" int advmil_gated_score_fwd(const void* v, const float* Wa, const float* ba, const float* Wb, const float* bb,
                                      const float* wc, const float* bc, int32_t rows, int32_t L, int32_t D, float p_drop,
                                      const uint8_t* mask_a, const uint8_t* mask_b, uint64_t seed, int32_t site,
                                      int32_t train, int32_t precision, void* ab, float* s, void* workspace,
                                      size_t workspace_bytes, void* stream) {
  ADVMIL_REQUIRE(v && Wa && Wb && wc && bc && s, "gated_score_fwd: null argument");
  cudaStream_t st = (cudaStream_t)stream;
  const int abw = gate_width(D);
  Workspace ws(workspace, workspace_bytes);
  WS_TAKE(Wp, float, (size_t)abw * L);
  WS_TAKE(bp, float, abw);
  WS_TAKE(part, float, (size_t)(abw / 128) * rows);
  Drop da = Drop::make(mask_a, seed, SITE_USER + site, p_drop, train, D);
  Drop db = Drop::make(mask_b, seed, SITE_USER + site + 1, p_drop, train, D);
  Drop::pair_gate(da, db);
  ADVMIL_TRY(gate_pack_weights(Wa, ba, Wb, bb, L, D, Wp, bp, st));
  return gated_score_fwd(v, Wp, bp, wc, bc, rows, L, D, da, db, ab, s, part, precision, st);
}

extern "C" int advmil_cast_f32_to_bf16(const float* in, int64_t n, void* out_bf16, void* stream) {
  ADVMIL_REQUIRE(in && out_bf16 && n >= 0, "cast_f32_to_bf16: bad arguments");
  return cast_f32_to_bf16(in, (size_t)n, out_bf16, (cudaStream_t)stream);
}

extern "C" size_t advmil_seg_pool_workspace_bytes(int32_t rows, int32_t bags, int32_t width) {
  return seg_pool_ws_floats(rows, bags, width) * sizeof(float) + 1024;
}

extern "C" int advmil_seg_softmax_pool_fwd(const float* s, const void* v, int32_t elem, const int32_t* offsets,
                                           const int32_t* offsets_host, int32_t rows, int32_t bags, int32_t width,
                                           float* w, float* z, float* mean, void* workspace, size_t workspace_bytes,
                                           void* stream) {
  ADVMIL_REQUIRE(s && v && offsets && offsets_host && w && z, "seg_softmax_pool_fwd: null argument");
  Workspace ws(workspace, workspace_bytes);
  WS_TAKE(poolws, float, seg_pool_ws_floats(rows, bags, width));
  ADVMIL_REQUIRE(elem == ELEM_F32 || elem == ELEM_BF16, "seg_softmax_pool_fwd: unknown element type %d", elem);
  return seg_softmax_pool_fwd(const_cast<float*>(s), nullptr, 0, nullptr, v, elem, offsets, offsets_host, rows, bags, width, w, z,
                              mean, poolws, (cudaStream_t)stream);
}
