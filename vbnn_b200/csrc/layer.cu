// layer.cu -- context + the nn.VBLinear entry points of include/vbnn.h.
// Every exported function cites the reference call it replaces in the header.
#include <math.h>
#include <stdarg.h>
#include <string.h>

#include <vector>

#include "knobs.h"
#include "state.h"

namespace vbnn {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

template <typename T>
static int dev_zalloc(T** p, size_t count, cudaStream_t st) {
  VB_TRY(dev_alloc(p, count));
  if (count) VB_CUDA(cudaMemsetAsync(*p, 0, count * sizeof(T), st));
  return VBNN_OK;
}
#define DEV_FREE(p) do { if (p) { cudaFree(p); (p) = nullptr; } } while (0)

PhiloxStream layer_stream(const vbnn_layer* L, uint32_t kind, int sample) {
  PhiloxStream ps;
  ps.key0 = (uint32_t)(L->ctx->seed & 0xFFFFFFFFu);
  ps.key1 = (uint32_t)(L->ctx->seed >> 32);
  ps.stream = kind | (uint32_t)L->id;
  ps.sample = (uint32_t)sample;
  ps.step = 0;
  return ps;
}

static inline bool is_bf16(const vbnn_layer* L) { return L->opts.precision == VBNN_PREC_BF16; }
static inline size_t esz(const vbnn_layer* L) { return is_bf16(L) ? 2 : 4; }
// peer mode: mu / log sigma^2 of rows owned by other ranks are only kept current when the forward pass
// needs them in fp32 (weight sampling); otherwise whole-layer reads need vbnn_mlp_sync_replicas first
static int check_params_fresh(const vbnn_layer* L, const char* what) {
  VB_CHECK(!(L->shard_stale && *L->shard_stale && layer_is_lrt(L)), VBNN_E_STATE,
           "%s in peer mode: rows owned by other ranks are out of date; call vbnn_mlp_sync_replicas on every rank first", what);
  return VBNN_OK;
}

int layer_refresh_copies(vbnn_layer* L) {
  cudaStream_t st = L->ctx->stream;
  if (L->kind == VBNN_KIND_LINEAR) {
    if (L->w_bf16) VB_TRY(launch_cast(L->weight, L->I, L->O, L->I, L->w_bf16, nullptr, L->ldI, st));
    return VBNN_OK;
  }
  if (L->mu_bf16 || L->s2_bf16 || L->s2_f32)
    VB_TRY(launch_param_copies(L->means, L->lvars, L->O, L->I, L->mu_bf16, L->s2_bf16, L->ldI, L->s2_f32,
                               st));
  return VBNN_OK;
}

PriorArgs layer_prior(const vbnn_layer* L, size_t row_off) {
  PriorArgs pr;
  memset(&pr, 0, sizeof(pr));
  pr.kind = L->prior_kind;
  if (L->prior_kind == VBNN_PRIOR_FIXED) { pr.mu0 = L->prior_mu0; pr.var0 = L->prior_var0; pr.lvar0 = logf(L->prior_var0); }
  if (L->prior_kind == VBNN_PRIOR_PER_WEIGHT) { pr.mu = L->prior_means + row_off; pr.lvar = L->prior_lvars + row_off; }
  return pr;
}

int layer_compute_prior_internal(vbnn_layer* L) {
  vbnn_ctx* c = L->ctx;
  int np = 0;
  const long long W = (long long)L->O * L->I;
  const bool empirical = L->prior_kind == VBNN_PRIOR_EMPIRICAL;
  if (empirical) VB_TRY(launch_prior_partials(L->means, L->lvars, W, c->d_partials, &np, c->stream));
  VB_TRY(launch_prior_finalize(c->d_partials, np, W, L->var_hat_dev, L->means, L->lvars, L->stdv,
                               L->mu_sqe, layer_prior(L, 0), c->stream));
  c->launches += empirical ? 2 : 1;
  L->prior_valid = true;
  return VBNN_OK;
}

// (re)compute the ping-pong partial sums the next update will read; called whenever mu / lvar / t
// change outside update() so that update() itself never needs a separate reduction pass
int layer_refresh_prior_partials(vbnn_layer* L) {
  if (L->kind != VBNN_KIND_VB) return VBNN_OK;
  VB_TRY(launch_prior_partials_pp(L->means, L->lvars, (long long)L->O * L->I, L->prior_partials, L->t_dev,
                                  L->n_part, L->ctx->stream));
  L->ctx->launches++;
  return VBNN_OK;
}

int layer_create_internal(vbnn_ctx* ctx, int I, int O, int kind, const vbnn_opts* opts, int S_alloc,
                          float* gW, float* gS, float* gb, int id, vbnn_layer** out) {
  VB_CHECK(ctx && out && opts, VBNN_E_INVALID, "layer_create: null argument");
  VB_CHECK(I > 0 && O > 0, VBNN_E_INVALID, "layer_create: bad sizes %d x %d", O, I);
  VB_CHECK(kind == VBNN_KIND_VB || kind == VBNN_KIND_LINEAR, VBNN_E_INVALID, "layer_create: bad kind");
  // the epsilon counter is uint32(o * ceil(I/4) + i/4) (philox.cuh): refuse layers where it would wrap
  VB_CHECK((unsigned long long)O * (unsigned long long)((I + 3) / 4) <= 0xFFFFFFFFull, VBNN_E_UNSUPPORTED,
           "layer_create: %d x %d weights exceed the 2^32-quad Philox counter", O, I);
  VB_CUDA(cudaSetDevice(ctx->device));
  vbnn_layer* L = new vbnn_layer();
  L->ctx = ctx; L->I = I; L->O = O; L->kind = kind; L->opts = *opts;
  // Philox stream id: position inside an mlp (identical on every rank / rebuild) or a ctx counter
  L->id = id >= 0 ? id : 0x1000 + ctx->next_layer_id++;
  L->ldI = round_up(I, 8); L->ldO = round_up(O, 8);
  L->S_alloc = S_alloc < 1 ? 1 : S_alloc;
  L->n_part = update_grid(O, I);
  cudaStream_t st = ctx->stream;
  const size_t W = (size_t)O * I;
  const bool vb = kind == VBNN_KIND_VB, b16 = is_bf16(L), lrt = layer_is_lrt(L);
  int r = VBNN_OK;
#define A_(expr) do { if (r == VBNN_OK) r = (expr); } while (0)
  A_(dev_zalloc(&L->bias, O, st));
  A_(dev_zalloc(&L->t_dev, 1, st));
  A_(dev_alloc(&L->hp, 1));
  if (gW) { L->gW = gW; L->gS = gS; L->gb = gb; L->grads_external = true; }
  else {
    A_(dev_zalloc(&L->gW, W, st));
    if (vb) A_(dev_zalloc(&L->gS, W, st));
    A_(dev_zalloc(&L->gb, O, st));
  }
  if (vb) {
    A_(dev_alloc(&L->means, W)); A_(dev_alloc(&L->lvars, W));
    A_(dev_zalloc(&L->m_mu, W, st)); A_(dev_zalloc(&L->v_mu, W, st));
    A_(dev_zalloc(&L->m_var, W, st)); A_(dev_zalloc(&L->v_var, W, st));
    A_(dev_zalloc(&L->var_hat_dev, 1, st));
    A_(dev_alloc(&L->prior_partials, (size_t)2 * kMaxPartials));
    if (opts->strict_reference) { A_(dev_alloc(&L->stdv, W)); A_(dev_alloc(&L->mu_sqe, W)); }
    if (!lrt && !b16) A_(dev_zalloc(&L->weight, W * L->S_alloc, st));
    if (!lrt && b16) A_(dev_zalloc(&L->w_bf16, (size_t)O * L->ldI * L->S_alloc, st));
    if (!lrt && b16 && gW) {                       // mlp-owned: the fused minibatch keeps epsilon for the dW epilogue
      uint16_t* e16 = nullptr;
      A_(dev_zalloc(&e16, (size_t)O * L->ldI * L->S_alloc, st));
      L->eps16 = e16;
    }
    if (lrt && b16) A_(dev_zalloc(&L->mu_bf16, (size_t)O * L->ldI, st));
    if (lrt && b16) A_(dev_zalloc(&L->s2_bf16, (size_t)O * L->ldI, st));
    if (lrt && !b16) A_(dev_alloc(&L->s2_f32, W));
  } else {
    A_(dev_alloc(&L->weight, W));
    if (b16) A_(dev_zalloc(&L->w_bf16, (size_t)O * L->ldI, st));
  }
#undef A_
  if (r != VBNN_OK) { vbnn_layer_destroy(L); return r; }
  // before any graph can capture a kernel that reads it
  VB_TRY(launch_set_live_opts(L->hp, live_opts(*opts), st));
  // ---- initial values: VBLinear.lua:12-29 ----
  if (vb) {
    float var_init = opts->msr_init ? 2.0f / (float)I : opts->var_init;                 // :12-16
    VB_TRY(launch_fill(L->lvars, W, logf(var_init), st));                               // :18
    if (opts->mu_init == 0.f) VB_CUDA(cudaMemsetAsync(L->means, 0, W * 4, st));         // :23
    else VB_TRY(launch_init_normal(L->means, W, 0.f, sqrtf(var_init), layer_stream(L, kStreamInit, 0), st));  // :25-28
    VB_TRY(layer_compute_prior_internal(L));                                            // :46
    VB_TRY(layer_refresh_prior_partials(L));
  } else {
    // nn.Linear weights as re-initialised by mlp.lua:47-55: N(0, sqrt(2/fan_in)), bias 0
    VB_TRY(launch_init_normal(L->weight, W, 0.f, sqrtf(2.0f / (float)I), layer_stream(L, kStreamInit, 0), st));
  }
  VB_TRY(layer_refresh_copies(L));
  ctx->launches += 4;
  *out = L;
  return VBNN_OK;
}

static int ensure_scratch(vbnn_layer* L, int N) {
  if (N <= L->cap_N) return VBNN_OK;
  VB_CUDA(cudaStreamSynchronize(L->ctx->stream));
  DEV_FREE(L->xs); DEV_FREE(L->xs2); DEV_FREE(L->gs_); DEV_FREE(L->hs); DEV_FREE(L->R);
  const size_t e = esz(L);
  char* p;
  VB_TRY(dev_alloc(&p, (size_t)N * L->ldI * e)); L->xs = p;
  VB_TRY(dev_alloc(&p, (size_t)N * L->ldO * e)); L->gs_ = p;
  if (layer_is_lrt(L)) {
    VB_TRY(dev_alloc(&p, (size_t)N * L->ldI * e)); L->xs2 = p;
    VB_TRY(dev_alloc(&p, (size_t)N * L->ldO * e)); L->hs = p;
    VB_TRY(dev_alloc(&p, (size_t)N * L->ldO * e)); L->R = p;
  }
  L->cap_N = N;
  return VBNN_OK;
}

// stage the caller's fp32 X (and X^2) into operand form
static int stage_x(vbnn_layer* L, const float* X, int N) {
  cudaStream_t st = L->ctx->stream;
  if (is_bf16(L)) {
    VB_TRY(launch_cast(X, L->I, N, L->I, (bf16*)L->xs, layer_is_lrt(L) ? (bf16*)L->xs2 : nullptr, L->ldI, st));
    L->ctx->launches++;
  } else if (layer_is_lrt(L)) {
    VB_TRY(launch_square(X, (float*)L->xs2, (long long)N * L->I, st));   // dense [N x I]
    L->ctx->launches++;
  }
  return VBNN_OK;
}

// The caller's X [N x I] and G [N x O] as GEMM operands: the bf16 copies stage_x / stage_g made, or the dense fp32
// buffers themselves
static GemmOperand x_operand(const vbnn_layer* L, const float* X, int kmajor) {
  return is_bf16(L) ? GemmOperand{L->xs, L->ldI, kmajor, 0} : GemmOperand{X, L->I, kmajor, 0};
}
static GemmOperand g_operand(const vbnn_layer* L, const float* G, int kmajor) {
  return is_bf16(L) ? GemmOperand{L->gs_, L->ldO, kmajor, 0} : GemmOperand{G, L->O, kmajor, 0};
}

static void fill_noise(vbnn_layer* L, EpiParams& p, uint32_t kind, const float* injected) {
  p.noise = injected;
  p.zs_noise = 0;
  p.ps = layer_stream(L, kind, L->cur_sample);
  p.step_ptr = L->ctx->d_step;
  p.row0 = 0;
}

static int bump_layer_t(vbnn_layer* L) {
  vbnn_ctx* c = L->ctx;
  VB_CUDA(cudaMemcpyAsync(c->h_scalars, L->t_dev, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
  VB_CUDA(cudaStreamSynchronize(c->stream));
  int t = *reinterpret_cast<int*>(c->h_scalars) + 1;
  VB_CUDA(cudaMemcpyAsync(L->t_dev, &t, sizeof(int), cudaMemcpyHostToDevice, c->stream));
  VB_CUDA(cudaStreamSynchronize(c->stream));
  return VBNN_OK;
}

int layer_update_internal(vbnn_layer* L, vbnn_stats* stats, bool bump_t) {
  vbnn_ctx* c = L->ctx;
  cudaStream_t st = c->stream;
  const long long W = (long long)L->O * L->I;
  if (L->kind == VBNN_KIND_LINEAR) {
    // optim.sgd over the whole output layer (mlp.lua:120-123; quirk Q4: intent, not the 110 slice)
    VB_TRY(launch_sgd(L->weight, L->gW, W, &L->hp->lr_bias, L->w_bf16, L->I, L->ldI, st));
    VB_TRY(launch_sgd(L->bias, L->gb, L->O, &L->hp->lr_bias, nullptr, 1, 1, st));
    c->launches += 2;
    if (bump_t) VB_TRY(bump_layer_t(L));
    return VBNN_OK;
  }
  VB_TRY(launch_sgd(L->bias, L->gb, L->O, &L->hp->lr_bias, nullptr, 1, 1, st));         // VBLinear.lua:125-128
  // compute_prior (:130): the per-block sums of exp(lvar)+mu^2 were left behind by the previous
  // update of this layer (or by layer_refresh_prior_partials after set / init)
  UpdateParams u;
  memset(&u, 0, sizeof(u));
  u.mu = L->means; u.lvar = L->lvars; u.gW = L->gW; u.gS = L->gS;
  u.m_mu = L->m_mu; u.v_mu = L->v_mu; u.m_var = L->m_var; u.v_var = L->v_var;
  u.stdv = L->stdv; u.mu_sqe = L->mu_sqe;
  u.mu_bf16 = L->mu_bf16; u.s2_bf16 = L->s2_bf16; u.ld_bf16 = L->ldI; u.s2_f32 = L->s2_f32;
  u.O = L->O; u.I = L->I;
  u.partials = L->prior_partials; u.n_partials = L->n_part;
  u.next_partials = L->prior_partials; u.partials_pingpong = 1;
  u.var_hat_dev = L->var_hat_dev; u.t_dev = L->t_dev;
  u.S = (float)L->opts.S;
  u.hp = L->hp;
  u.lrt = layer_is_lrt(L);
  u.prior = layer_prior(L, 0);
  // the grid that writes the next partials must be the one whose count (n_part, fixed at creation) the next update
  // reads: update_grid() under a later upd_bps would write more or fewer of them
  u.grid_override = L->n_part;
  u.coresident = knobs().upd_coresident != 0;
  double* stat_dev = stats ? c->d_partials + kMaxPartials : nullptr;
  u.stat_partials = stat_dev;
  int grid = 0;
  // bench.py's HBM roofline: class 7 = fused update, "flops" slot = algorithmic bytes (56 B / weight, + the 8 B of
  // the prior's mean and log-variance under PER_WEIGHT)
  const double bytes = (L->prior_kind == VBNN_PRIOR_PER_WEIGHT ? 64.0 : 56.0) * (double)W;
  VB_TRY(prof_launch(c, 7, bytes, [&] { return launch_update(u, &grid, st); }));         // :131-143
  c->launches += 2;
  L->prior_valid = true;
  // single counter bump: the layer owns t_dev.  The kernel left the new sums in half
  // ((t_old + 1) & 1) == (t & 1): consistent with the bump
  if (bump_t) VB_TRY(bump_layer_t(L));
  if (stats) {
    VB_CUDA(cudaMemcpyAsync(c->h_partials, stat_dev, (size_t)grid * kStatSlots * sizeof(double),
                            cudaMemcpyDeviceToHost, st));
    VB_CUDA(cudaMemcpyAsync(c->h_scalars, L->var_hat_dev, sizeof(float), cudaMemcpyDeviceToHost, st));
    VB_CUDA(cudaStreamSynchronize(st));
    double s[kStatSlots] = {0};
    s[11] = 3e38; s[12] = -3e38; s[13] = 3e38; s[14] = -3e38;
    for (int b = 0; b < grid; ++b) {
      const double* q = c->h_partials + (size_t)b * kStatSlots;
      for (int i = 0; i < 10; ++i) s[i] += q[i];
      s[11] = fmin(s[11], q[11]); s[12] = fmax(s[12], q[12]);
      s[13] = fmin(s[13], q[13]); s[14] = fmax(s[14], q[14]);
    }
    const double n = (double)W, nl = sqrt(s[4]), nm = sqrt(s[5]);
    stats->vlc_grad = (float)(sqrt(s[0]) / nl);                     // VBLinear.lua:150
    stats->vle_grad = (float)(sqrt(s[1]) / nl);                     // :151
    stats->mlc_grad = (float)(sqrt(s[2]) / nm);                     // :152
    stats->mle_grad = (float)(sqrt(s[3]) / nm);                     // :153
    stats->min_variance = (float)s[11];                             // :154
    stats->max_variance = (float)s[12];                             // :155
    stats->mean_variance = (float)(s[6] / n);                       // :156
    stats->var_hat = c->h_scalars[0];                               // :157
    const double mean = s[7] / n;
    stats->mean_means = (float)mean;                                // :158
    stats->std_means = (float)sqrt(fmax(0.0, (s[5] - n * mean * mean) / (n - 1.0)));   // :159
    stats->min_means = (float)s[13];                                // :160
    stats->max_means = (float)s[14];                                // :161
    stats->mu_normratio = (float)(sqrt(s[8]) / nm);                 // :162
    stats->var_normratio = (float)(sqrt(s[9]) / nl);                // :163
  }
  return VBNN_OK;
}

void weight_operands(GemmArgs& g, const vbnn_layer* L, int kmajor, bool batched, bool lrt) {
  const bool b16 = is_bf16(L), mu = layer_is_lrt(L);
  const int ld = b16 ? L->ldI : L->I;
  const void* w = b16 ? (mu ? (const void*)L->mu_bf16 : L->w_bf16) : (mu ? L->means : L->weight);
  g.B1 = {w, ld, kmajor, batched ? (long long)L->O * ld : 0};
  if (lrt) g.B2 = {b16 ? (const void*)L->s2_bf16 : L->s2_f32, ld, kmajor, 0};
}

int gemm(vbnn_ctx* c, bool bf16, int mode, const GemmArgs& g, const EpiParams& p, int prof_cls) {
  if (!bf16) return gemm_simt_launch(mode, g, p, c->stream, &c->launches);
  const int cls = (prof_cls >= 0 ? prof_cls : mode) & 7;        // GEMM classes 0-7; class 8 is predict (mlp.cu)
  const double flops = 2.0 * g.M * (double)g.N * g.K * g.batch * (epi_is_dual(mode) ? 2.0 : 1.0);
  return prof_launch(c, cls, flops, [&] { return gemm_tc_launch(mode, g, p, c->stream, &c->launches); });
}

int prof_mark(vbnn_ctx* c, int id) {
  if (!c->profiling) return VBNN_OK;
  cudaEvent_t e;
  if (!c->prof_pool.empty()) { e = c->prof_pool.back(); c->prof_pool.pop_back(); }
  else VB_CUDA(cudaEventCreate(&e));
  VB_CUDA(cudaEventRecord(e, c->stream));
  c->marks.push_back({e, id});
  return VBNN_OK;
}

int prof_collect(vbnn_ctx* c) {
  if (c->prof_recs.empty() && c->marks.empty()) return VBNN_OK;
  VB_CUDA(cudaStreamSynchronize(c->stream));
  for (size_t i = 0; i < c->marks.size(); ++i) {
    const int id = c->marks[i].id & 15;
    if (i > 0 && id != 0) {
      float ms = 0.f;
      VB_CUDA(cudaEventElapsedTime(&ms, c->marks[i - 1].e, c->marks[i].e));
      c->phase_ms[id] += ms; c->phase_n[id] += 1;
    }
  }
  for (auto& mk : c->marks) c->prof_pool.push_back(mk.e);
  c->marks.clear();
  for (auto& r : c->prof_recs) {
    float ms = 0.f;
    VB_CUDA(cudaEventElapsedTime(&ms, r.a, r.b));
    c->prof_ms[r.cls] += ms; c->prof_flops[r.cls] += r.flops; c->prof_n[r.cls] += 1;
    c->prof_pool.push_back(r.a); c->prof_pool.push_back(r.b);
  }
  c->prof_recs.clear();
  return VBNN_OK;
}

}  // namespace vbnn

using namespace vbnn;

// ============================================================ library ======================
extern "C" int vbnn_abi_version(void) { return VBNN_ABI_VERSION; }
extern "C" const char* vbnn_last_error(void) { return g_err; }

extern "C" void vbnn_opts_default(vbnn_opts* o) {
  if (!o) return;
  memset(o, 0, sizeof(*o));
  o->var_init = 0.001f;     // config.lua:44
  o->msr_init = 0;          // config.lua:45 (commented out)
  o->mu_init = 0.f;         // config.lua:43
  o->B = 1000000.f;         // config.lua:30
  o->S = 30;                // config.lua:32
  o->lr_bias = 0.001f;      // config.lua:53
  o->lr_mu = 0.0001f;       // config.lua:62
  o->lr_var = 0.05f;        // config.lua:57
  o->adam_beta1 = 0.9f; o->adam_beta2 = 0.999f; o->adam_eps = 1e-8f;
  o->reparam = VBNN_REPARAM_WEIGHT;
  o->precision = VBNN_PREC_FP32;
  o->strict_reference = 1;
}

// ============================================================ context ======================
extern "C" int vbnn_ctx_create(int device, void* stream, uint64_t seed, vbnn_ctx** out) {
  return vbnn_ctx_create_ex(device, stream, VBNN_CTX_STREAM_GIVEN, seed, out);
}

extern "C" int vbnn_ctx_create_ex(int device, void* stream, int stream_mode, uint64_t seed, vbnn_ctx** out) {
  VB_CHECK(out != nullptr, VBNN_E_INVALID, "vbnn_ctx_create: out is null");
  VB_CHECK(stream_mode >= VBNN_CTX_STREAM_GIVEN && stream_mode <= VBNN_CTX_STREAM_PRIVATE_BLOCKING, VBNN_E_INVALID,
           "vbnn_ctx_create_ex: bad stream_mode %d", stream_mode);
  VB_CHECK(stream_mode == VBNN_CTX_STREAM_GIVEN || stream == nullptr, VBNN_E_INVALID,
           "vbnn_ctx_create_ex: stream must be NULL with stream_mode %d", stream_mode);
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0) {
    set_error("no CUDA device available (%s); libvbnn has no CPU fallback",
              e != cudaSuccess ? cudaGetErrorString(e) : "device count 0");
    return VBNN_E_CUDA;
  }
  VB_CHECK(device >= 0 && device < ndev, VBNN_E_INVALID, "vbnn_ctx_create: device %d of %d", device, ndev);
  VB_CUDA(cudaSetDevice(device));
  cudaDeviceProp prop;
  VB_CUDA(cudaGetDeviceProperties(&prop, device));
  VB_CHECK(prop.major == 10, VBNN_E_UNSUPPORTED,
           "libvbnn.so is built for sm_100a only; device %d is sm_%d%d", device, prop.major, prop.minor);
  vbnn_ctx* c = new vbnn_ctx();
  c->device = device; c->seed = seed;
  if (stream_mode == VBNN_CTX_STREAM_LEGACY_DEFAULT) {
    c->stream = cudaStreamLegacy;          // stream 0: ordered with the caller's cutorch-style default-stream work
    c->capturable = false;
  } else if (stream_mode == VBNN_CTX_STREAM_PRIVATE_BLOCKING) {
    VB_CUDA(cudaStreamCreateWithFlags(&c->stream, cudaStreamDefault));   // implicit sync with stream 0
    c->own_stream = true;
  } else if (stream) {
    c->stream = (cudaStream_t)stream;
    c->capturable = c->stream != cudaStreamLegacy && c->stream != cudaStreamPerThread;
  } else {
    VB_CUDA(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
    c->own_stream = true;
  }
  VB_CUDA(cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking));
  VB_TRY(dev_zalloc(&c->d_step, 1, c->stream));
  VB_TRY(dev_alloc(&c->d_partials, (size_t)kMaxPartials * (1 + kStatSlots)));
  VB_CUDA(cudaMallocHost((void**)&c->h_partials, (size_t)kMaxPartials * kStatSlots * sizeof(double)));
  VB_CUDA(cudaMallocHost((void**)&c->h_scalars, 4096 * sizeof(float)));
  *out = c;
  return VBNN_OK;
}

extern "C" int vbnn_ctx_destroy(vbnn_ctx* c) {
  if (!c) return VBNN_OK;
  cudaSetDevice(c->device);
  cudaStreamSynchronize(c->stream);
  prof_collect(c);
  for (cudaEvent_t e : c->prof_pool) cudaEventDestroy(e);
  vbnn_comm_destroy(c);
  DEV_FREE(c->d_step); DEV_FREE(c->d_partials);
  if (c->h_partials) cudaFreeHost(c->h_partials);
  if (c->h_scalars) cudaFreeHost(c->h_scalars);
  if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
  if (c->own_stream) cudaStreamDestroy(c->stream);
  delete c;
  return VBNN_OK;
}

extern "C" int vbnn_ctx_synchronize(vbnn_ctx* c) {
  VB_CHECK(c, VBNN_E_INVALID, "null ctx");
  VB_CUDA(cudaStreamSynchronize(c->stream));
  return VBNN_OK;
}
extern "C" int vbnn_ctx_profile(vbnn_ctx* c, int enable) {
  VB_CHECK(c, VBNN_E_INVALID, "null ctx");
  VB_TRY(prof_collect(c));
  c->profiling = enable != 0;
  if (enable) for (int i = 0; i < vbnn_ctx::kProfClasses; ++i) { c->prof_ms[i] = 0; c->prof_flops[i] = 0; c->prof_n[i] = 0; }
  if (enable) for (int i = 0; i < 16; ++i) { c->phase_ms[i] = 0; c->phase_n[i] = 0; }
  return VBNN_OK;
}
extern "C" int vbnn_ctx_profile_read(vbnn_ctx* c, int cls, double* total_ms, long long* launches, double* flops) {
  VB_CHECK(c && cls >= 0 && cls < vbnn_ctx::kProfClasses, VBNN_E_INVALID, "vbnn_ctx_profile_read: bad argument");
  VB_TRY(prof_collect(c));
  if (total_ms) *total_ms = c->prof_ms[cls];
  if (launches) *launches = c->prof_n[cls];
  if (flops) *flops = c->prof_flops[cls];
  return VBNN_OK;
}
extern "C" int vbnn_ctx_phase_read(vbnn_ctx* c, int id, double* total_ms, long long* count) {
  VB_CHECK(c && id >= 0 && id < 16, VBNN_E_INVALID, "vbnn_ctx_phase_read: bad argument");
  VB_TRY(prof_collect(c));
  if (total_ms) *total_ms = c->phase_ms[id];
  if (count) *count = c->phase_n[id];
  return VBNN_OK;
}
extern "C" int vbnn_ctx_set_step(vbnn_ctx* c, uint32_t step) {
  VB_CHECK(c, VBNN_E_INVALID, "null ctx");
  VB_CUDA(cudaMemcpyAsync(c->d_step, &step, sizeof(step), cudaMemcpyHostToDevice, c->stream));
  VB_CUDA(cudaStreamSynchronize(c->stream));
  return VBNN_OK;
}
extern "C" int vbnn_ctx_get_step(vbnn_ctx* c, uint32_t* step) {
  VB_CHECK(c && step, VBNN_E_INVALID, "null argument");
  VB_CUDA(cudaMemcpyAsync(step, c->d_step, sizeof(*step), cudaMemcpyDeviceToHost, c->stream));
  VB_CUDA(cudaStreamSynchronize(c->stream));
  return VBNN_OK;
}

// ============================================================ layer ========================
extern "C" int vbnn_layer_create(vbnn_ctx* ctx, int inputSize, int outputSize, int kind,
                                 const vbnn_opts* opts, vbnn_layer** out) {
  return layer_create_internal(ctx, inputSize, outputSize, kind, opts, 1, nullptr, nullptr, nullptr, -1, out);
}

extern "C" int vbnn_layer_destroy(vbnn_layer* L) {
  if (!L) return VBNN_OK;
  cudaSetDevice(L->ctx->device);
  cudaStreamSynchronize(L->ctx->stream);
  DEV_FREE(L->means); DEV_FREE(L->lvars);
  if (!L->ext_bias) DEV_FREE(L->bias);
  if (!L->ext_weight) DEV_FREE(L->weight);
  if (!L->grads_external) {
    if (!L->ext_gW) DEV_FREE(L->gW);
    DEV_FREE(L->gS);
    if (!L->ext_gb) DEV_FREE(L->gb);
  }
  DEV_FREE(L->m_mu); DEV_FREE(L->v_mu); DEV_FREE(L->m_var); DEV_FREE(L->v_var);
  DEV_FREE(L->eps); DEV_FREE(L->stdv); DEV_FREE(L->mu_sqe); DEV_FREE(L->s2_f32);
  DEV_FREE(L->var_hat_dev); DEV_FREE(L->t_dev); DEV_FREE(L->hp); DEV_FREE(L->prior_partials);
  DEV_FREE(L->w_bf16); DEV_FREE(L->mu_bf16); DEV_FREE(L->s2_bf16); DEV_FREE(L->eps16);
  DEV_FREE(L->xs); DEV_FREE(L->xs2); DEV_FREE(L->gs_); DEV_FREE(L->hs); DEV_FREE(L->R);
  DEV_FREE(L->zeta_keep);
  DEV_FREE(L->prior_means); DEV_FREE(L->prior_lvars);
  delete L;
  return VBNN_OK;
}

extern "C" int vbnn_layer_dims(const vbnn_layer* L, int* I, int* O) {
  VB_CHECK(L, VBNN_E_INVALID, "null layer");
  if (I) *I = L->I;
  if (O) *O = L->O;
  return VBNN_OK;
}

extern "C" int vbnn_layer_sample(vbnn_layer* L, int sample_idx, const float* eps_dev) {
  VB_CHECK(L && L->kind == VBNN_KIND_VB, VBNN_E_INVALID, "vbnn_layer_sample: not a VB layer");
  L->cur_sample = sample_idx;
  L->map_mode = false;
  L->eps_injected = eps_dev != nullptr;
  L->eps16_valid = false;
  if (layer_is_lrt(L)) return VBNN_OK;     // local reparameterisation draws its noise in forward()
  cudaStream_t st = L->ctx->stream;
  const size_t W = (size_t)L->O * L->I;
  if (eps_dev && !L->eps) VB_TRY(dev_alloc(&L->eps, W));
  SampleParams p;
  memset(&p, 0, sizeof(p));
  p.mu = L->means;
  if (L->opts.strict_reference) { p.sig = L->stdv; p.sig_is_lvar = 0; }     // quirk Q1
  else { p.sig = L->lvars; p.sig_is_lvar = 1; }
  p.O = L->O; p.I = L->I; p.S = 1;
  p.ps = layer_stream(L, kStreamEps, sample_idx);
  p.step_ptr = L->ctx->d_step;
  p.eps_in = eps_dev;
  p.eps_out = eps_dev ? L->eps : nullptr;                                   // self.e
  p.w_f32 = L->weight;
  p.w_bf16 = L->w_bf16; p.ld_bf16 = L->ldI; p.zs_bf16 = 0;
  VB_TRY(launch_sample_w(p, st));
  L->ctx->launches++;
  return VBNN_OK;
}

extern "C" int vbnn_layer_clamp_to_map(vbnn_layer* L) {
  VB_CHECK(L && L->kind == VBNN_KIND_VB, VBNN_E_INVALID, "vbnn_layer_clamp_to_map: not a VB layer");
  VB_TRY(check_params_fresh(L, "vbnn_layer_clamp_to_map"));
  cudaStream_t st = L->ctx->stream;
  L->map_mode = true;
  if (layer_is_lrt(L)) {
    if (L->mu_bf16) VB_TRY(layer_refresh_copies(L));
    return VBNN_OK;
  }
  if (L->weight)
    VB_CUDA(cudaMemcpyAsync(L->weight, L->means, (size_t)L->O * L->I * 4, cudaMemcpyDeviceToDevice, st));
  if (L->w_bf16) VB_TRY(launch_cast(L->means, L->I, L->O, L->I, L->w_bf16, nullptr, L->ldI, st));
  L->ctx->launches++;
  return VBNN_OK;
}

extern "C" int vbnn_layer_forward(vbnn_layer* L, const float* X, int N, float* Y, const float* zeta) {
  VB_CHECK(L && X && Y && N > 0, VBNN_E_INVALID, "vbnn_layer_forward: bad argument");
  VB_TRY(ensure_scratch(L, N));
  VB_TRY(stage_x(L, X, N));
  const bool lrt = layer_is_lrt(L) && !L->map_mode;
  EpiParams p;
  memset(&p, 0, sizeof(p));
  p.M = N; p.N = L->O;
  p.out_f32 = Y; p.ld_f32 = L->O;
  p.bias = L->bias; p.relu = 0;
  p.ld_act = L->ldO;
  int mode = EPI_FWD;
  if (lrt) {
    mode = EPI_FWD_LRT;
    p.r_out = L->R;
    fill_noise(L, p, kStreamZeta, zeta);
    VB_CHECK((unsigned long long)N * (unsigned long long)((L->O + 3) / 4) <= 0xFFFFFFFFull, VBNN_E_UNSUPPORTED,
             "Philox zeta counter would wrap: %d rows x %d outputs", N, L->O);
  }
  GemmArgs g;
  memset(&g, 0, sizeof(g));
  g.M = N; g.N = L->O; g.K = L->I; g.batch = 1;
  g.A1 = x_operand(L, X, 1);
  if (lrt) g.A2 = {L->xs2, g.A1.ld, 1, 0};
  weight_operands(g, L, 1, false, lrt);
  return gemm(L->ctx, is_bf16(L), mode, g, p);
}

// H = G .* R for the local-reparameterisation backward; also stages G in operand form
static int stage_g(vbnn_layer* L, const float* G, int N) {
  cudaStream_t st = L->ctx->stream;
  const bool lrt = layer_is_lrt(L) && !L->map_mode;
  if (is_bf16(L)) {
    VB_TRY(launch_cast(G, L->O, N, L->O, (bf16*)L->gs_, nullptr, L->ldO, st));
    L->ctx->launches++;
  }
  if (lrt) {
    VB_TRY(launch_mul_act(G, L->O, 0, L->R, L->ldO, L->hs, L->ldO, N, L->O, is_bf16(L), st));
    L->ctx->launches++;
  }
  return VBNN_OK;
}

extern "C" int vbnn_layer_backward_data(vbnn_layer* L, const float* X, const float* G, int N, float* dX) {
  VB_CHECK(L && X && G && dX && N > 0, VBNN_E_INVALID, "vbnn_layer_backward_data: bad argument");
  VB_CHECK(N <= L->cap_N, VBNN_E_STATE, "vbnn_layer_backward_data before forward (N=%d)", N);
  const bool lrt = layer_is_lrt(L) && !L->map_mode;
  VB_TRY(stage_g(L, G, N));
  EpiParams p;
  memset(&p, 0, sizeof(p));
  p.M = N; p.N = L->I;
  p.out_f32 = dX; p.ld_f32 = L->I;
  p.ld_act = L->ldI;
  p.mask = 0;
  const int mode = lrt ? EPI_DX_LRT : EPI_DX;
  GemmArgs g;
  memset(&g, 0, sizeof(g));
  g.M = N; g.N = L->I; g.K = L->O; g.batch = 1;
  g.A1 = g_operand(L, G, 1);
  if (lrt) {
    const GemmOperand x = x_operand(L, X, 1);
    p.xprev = x.ptr; p.ld_x = x.ld;
    g.A2 = {L->hs, L->ldO, 1, 0};
  }
  weight_operands(g, L, 0, false, lrt);
  return gemm(L->ctx, is_bf16(L), mode, g, p);
}

extern "C" int vbnn_layer_acc_grad(vbnn_layer* L, const float* X, const float* G, int N, float scale) {
  VB_CHECK(L && X && G && N > 0, VBNN_E_INVALID, "vbnn_layer_acc_grad: bad argument");
  VB_TRY(ensure_scratch(L, N));
  cudaStream_t st = L->ctx->stream;
  const bool lrt = layer_is_lrt(L) && !L->map_mode;
  // operands may not have been staged by forward/backward_data of this call sequence
  VB_TRY(stage_x(L, X, N));
  VB_TRY(stage_g(L, G, N));
  EpiParams p;
  memset(&p, 0, sizeof(p));
  p.M = L->O; p.N = L->I;
  p.gW = L->gW; p.gS = L->kind == VBNN_KIND_VB ? L->gS : nullptr; p.ld_g = L->I;
  p.scale = scale; p.accumulate = 1;
  fill_noise(L, p, kStreamEps, L->eps_injected ? L->eps : nullptr);
  if (L->map_mode) { p.gS = nullptr; }
  const int mode = lrt ? EPI_DW_LRT : EPI_DW;
  GemmArgs g;
  memset(&g, 0, sizeof(g));
  g.M = L->O; g.N = L->I; g.K = N; g.batch = 1;
  g.A1 = g_operand(L, G, 0);
  g.B1 = x_operand(L, X, 0);
  if (lrt) { g.A2 = {L->hs, L->ldO, 0, 0}; g.B2 = {L->xs2, g.B1.ld, 0, 0}; }
  VB_TRY(gemm(L->ctx, is_bf16(L), mode, g, p));
  VB_TRY(launch_colsum(G, 0, N, L->O, L->O, scale, L->gb, st));       // gradBias += scale * G^T 1
  L->ctx->launches++;
  return VBNN_OK;
}

extern "C" int vbnn_layer_reset_acc(vbnn_layer* L) {
  VB_CHECK(L, VBNN_E_INVALID, "null layer");
  cudaStream_t st = L->ctx->stream;
  const size_t W = (size_t)L->O * L->I;
  VB_CUDA(cudaMemsetAsync(L->gW, 0, W * 4, st));                       // mlp.lua:63
  if (L->gS) VB_CUDA(cudaMemsetAsync(L->gS, 0, W * 4, st));            // VBLinear.lua:121
  VB_CUDA(cudaMemsetAsync(L->gb, 0, (size_t)L->O * 4, st));
  return VBNN_OK;
}

extern "C" int vbnn_layer_compute_prior(vbnn_layer* L, float* mu_hat, float* var_hat) {
  VB_CHECK(L && L->kind == VBNN_KIND_VB, VBNN_E_INVALID, "vbnn_layer_compute_prior: not a VB layer");
  VB_TRY(check_params_fresh(L, "vbnn_layer_compute_prior"));
  VB_TRY(layer_compute_prior_internal(L));
  cudaStream_t st = L->ctx->stream;
  VB_CUDA(cudaMemcpyAsync(L->ctx->h_scalars, L->var_hat_dev, 4, cudaMemcpyDeviceToHost, st));
  VB_CUDA(cudaStreamSynchronize(st));
  if (mu_hat) *mu_hat = L->prior_kind == VBNN_PRIOR_EMPIRICAL ? 0.f             // VBLinear.lua:81
                      : L->prior_kind == VBNN_PRIOR_FIXED ? L->prior_mu0 : nanf("");
  if (var_hat) *var_hat = L->ctx->h_scalars[0];                        // FIXED: var0, PER_WEIGHT: NaN
  return VBNN_OK;
}

extern "C" int vbnn_layer_grads(vbnn_layer* L, float* mleg, float* mlcg, float* vleg, float* vlcg) {
  VB_CHECK(L && L->kind == VBNN_KIND_VB, VBNN_E_INVALID, "vbnn_layer_grads: not a VB layer");
  VB_CHECK(L->prior_valid, VBNN_E_STATE, "vbnn_layer_grads before compute_prior");
  VB_TRY(launch_grads(L->means, L->lvars, L->gW, L->gS, (long long)L->O * L->I, L->var_hat_dev, layer_prior(L, 0),
                      L->hp, (float)L->opts.S, layer_is_lrt(L), mleg, mlcg, vleg, vlcg, L->ctx->stream));
  L->ctx->launches++;
  return VBNN_OK;
}

extern "C" int vbnn_layer_update(vbnn_layer* L, vbnn_stats* stats) {
  VB_CHECK(L, VBNN_E_INVALID, "null layer");
  return layer_update_internal(L, stats, true);
}

extern "C" int vbnn_layer_calc_lc(vbnn_layer* L, float* lc_dev, float* sum_host) {
  VB_CHECK(L && L->kind == VBNN_KIND_VB, VBNN_E_INVALID, "vbnn_layer_calc_lc: not a VB layer");
  VB_TRY(check_params_fresh(L, "vbnn_layer_calc_lc"));
  vbnn_ctx* c = L->ctx;
  cudaStream_t st = c->stream;
  const long long W = (long long)L->O * L->I;
  int np = 0;
  if (L->opts.strict_reference && L->stdv && L->mu_sqe) {
    // quirk Q6: tensors cached by the last compute_prior (VBLinear.lua:100-101 read self.vars etc.)
    VB_TRY(launch_calc_lc(L->stdv, 1, L->mu_sqe, 1, W, L->var_hat_dev, layer_prior(L, 0), L->hp, lc_dev,
                          c->d_partials, &np, st));
  } else {
    VB_TRY(layer_compute_prior_internal(L));
    VB_TRY(launch_calc_lc(L->lvars, 0, L->means, 0, W, L->var_hat_dev, layer_prior(L, 0), L->hp, lc_dev,
                          c->d_partials, &np, st));
  }
  c->launches++;
  if (sum_host) {
    VB_CUDA(cudaMemcpyAsync(c->h_partials, c->d_partials, np * sizeof(double), cudaMemcpyDeviceToHost, st));
    VB_CUDA(cudaStreamSynchronize(st));
    double s = 0;
    for (int i = 0; i < np; ++i) s += c->h_partials[i];
    *sum_host = (float)s;
  }
  return VBNN_OK;
}

extern "C" int vbnn_layer_set_prior(vbnn_layer* L, int kind, float mu0, float var0) {
  VB_CHECK(L && L->kind == VBNN_KIND_VB, VBNN_E_INVALID, "vbnn_layer_set_prior: not a VB layer");
  VB_CHECK(kind == VBNN_PRIOR_EMPIRICAL || kind == VBNN_PRIOR_FIXED || kind == VBNN_PRIOR_PER_WEIGHT, VBNN_E_INVALID,
           "vbnn_layer_set_prior: unknown kind %d", kind);
  VB_CHECK(kind != VBNN_PRIOR_FIXED || (isfinite(mu0) && isfinite(var0) && var0 > 0.f), VBNN_E_INVALID,
           "vbnn_layer_set_prior: FIXED needs a finite mu0 and a finite var0 > 0 (got %g, %g)", mu0, var0);
  VB_CHECK(!(L->owner && L->owner->step_open), VBNN_E_STATE,
           "vbnn_layer_set_prior: the net has an open vbnn_mlp_forward_train step");
  VB_CHECK(!(kind == VBNN_PRIOR_PER_WEIGHT && L->shard_stale && *L->shard_stale), VBNN_E_STATE,
           "vbnn_layer_set_prior(PER_WEIGHT) in peer mode: rows owned by other ranks are out of date; call "
           "vbnn_mlp_sync_replicas on every rank first");
  vbnn_ctx* c = L->ctx;
  cudaStream_t st = c->stream;
  const size_t W = (size_t)L->O * L->I;
  const int old = L->prior_kind;
  if (kind == VBNN_PRIOR_PER_WEIGHT) {
    if (!L->prior_means) {
      VB_TRY(dev_alloc(&L->prior_means, W));
      int r = dev_alloc(&L->prior_lvars, W);
      if (r != VBNN_OK) { DEV_FREE(L->prior_means); return r; }
    }
    // the snapshot: this posterior becomes the prior (variational continual learning)
    VB_CUDA(cudaMemcpyAsync(L->prior_means, L->means, W * 4, cudaMemcpyDeviceToDevice, st));
    VB_CUDA(cudaMemcpyAsync(L->prior_lvars, L->lvars, W * 4, cudaMemcpyDeviceToDevice, st));
  }
  // the arrays, once allocated, stay until vbnn_layer_destroy: pointers handed out by vbnn_layer_device_ptr stay valid
  // across kind changes (VBNN_BUF_PRIOR_* are refused while the kind is not PER_WEIGHT)
  L->prior_kind = kind;
  L->prior_mu0 = kind == VBNN_PRIOR_FIXED ? mu0 : 0.f;
  L->prior_var0 = kind == VBNN_PRIOR_FIXED ? var0 : 0.f;
  if (kind == VBNN_PRIOR_FIXED || kind == VBNN_PRIOR_PER_WEIGHT) {
    // the scalar vbnn_layer_grads / calc_lc / compute_prior / vbnn_stats read: var0, or NaN (no scalar prior)
    VB_TRY(launch_fill(L->var_hat_dev, 1, kind == VBNN_PRIOR_FIXED ? var0 : nanf(""), st));
    c->launches++;
  } else if (old != VBNN_PRIOR_EMPIRICAL) {
    // back to the reference's prior: var_hat of the current parameters, the strict_reference caches untouched
    int np = 0;
    VB_TRY(launch_prior_partials(L->means, L->lvars, (long long)W, c->d_partials, &np, st));
    VB_TRY(launch_prior_finalize(c->d_partials, np, (long long)W, L->var_hat_dev, L->means, L->lvars, nullptr,
                                 nullptr, layer_prior(L, 0), st));
    c->launches += 2;
  }
  if (L->owner) mlp_drop_graphs(L->owner);   // the update kernels of the step graphs bake the prior in
  return VBNN_OK;
}

extern "C" int vbnn_layer_get_prior(const vbnn_layer* L, int* kind, float* mu0, float* var0) {
  VB_CHECK(L && L->kind == VBNN_KIND_VB, VBNN_E_INVALID, "vbnn_layer_get_prior: not a VB layer");
  const bool fixed = L->prior_kind == VBNN_PRIOR_FIXED;
  if (kind) *kind = L->prior_kind;
  if (mu0) *mu0 = fixed ? L->prior_mu0 : nanf("");
  if (var0) *var0 = fixed ? L->prior_var0 : nanf("");
  return VBNN_OK;
}

LiveOpts vbnn::live_opts(const vbnn_opts& o) {
  return LiveOpts{o.B, o.lr_bias, o.lr_mu, o.lr_var, o.adam_beta1, o.adam_beta2, o.adam_eps};
}

// vbnn_layer_set_opts / vbnn_mlp_set_opts: the fields that size buffers or choose kernels must be the layer's own, and
// every live value must be one the update can use
static int check_opts(const vbnn_layer* L, const vbnn_opts* o, const char* who) {
  const vbnn_opts& c = L->opts;
#define FIXED_(f) VB_CHECK(memcmp(&o->f, &c.f, sizeof(c.f)) == 0, VBNN_E_INVALID, "%s: %s cannot change on a live layer", \
                           who, #f)
  FIXED_(var_init); FIXED_(msr_init); FIXED_(mu_init); FIXED_(S); FIXED_(reparam); FIXED_(precision);
  FIXED_(strict_reference);
#undef FIXED_
  VB_CHECK(isfinite(o->B) && o->B > 0.f, VBNN_E_INVALID, "%s: B must be finite and > 0 (got %g)", who, o->B);
#define RATE_(f) VB_CHECK(isfinite(o->f) && o->f >= 0.f, VBNN_E_INVALID, "%s: %s must be finite and >= 0 (got %g)", \
                          who, #f, o->f)
  RATE_(lr_bias); RATE_(lr_mu); RATE_(lr_var);
#undef RATE_
#define BETA_(f) VB_CHECK(o->f >= 0.f && o->f < 1.f, VBNN_E_INVALID, "%s: %s must be in [0, 1) (got %g)", who, #f, o->f)
  BETA_(adam_beta1); BETA_(adam_beta2);
#undef BETA_
  VB_CHECK(isfinite(o->adam_eps) && o->adam_eps > 0.f, VBNN_E_INVALID, "%s: adam_eps must be finite and > 0 (got %g)",
           who, o->adam_eps);
  return VBNN_OK;
}

// the host copy would disagree with a graph that captured the write
static int refuse_set_in_capture(const vbnn_ctx* c, const char* who) {
  cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
  VB_CUDA(cudaStreamIsCapturing(c->stream, &cs));
  VB_CHECK(cs == cudaStreamCaptureStatusNone, VBNN_E_STATE, "%s: the context's stream is being captured", who);
  return VBNN_OK;
}

static int write_opts(vbnn_layer* L, const vbnn_opts* o) {
  VB_TRY(launch_set_live_opts(L->hp, live_opts(*o), L->ctx->stream));
  L->ctx->launches++;
  L->opts = *o;
  return VBNN_OK;
}

extern "C" int vbnn_layer_get_opts(const vbnn_layer* L, vbnn_opts* out) {
  VB_CHECK(L && out, VBNN_E_INVALID, "vbnn_layer_get_opts: null argument");
  *out = L->opts;
  return VBNN_OK;
}

extern "C" int vbnn_layer_set_opts(vbnn_layer* L, const vbnn_opts* opts) {
  VB_CHECK(L && opts, VBNN_E_INVALID, "vbnn_layer_set_opts: null argument");
  VB_TRY(refuse_set_in_capture(L->ctx, "vbnn_layer_set_opts"));
  VB_TRY(check_opts(L, opts, "vbnn_layer_set_opts"));
  VB_CUDA(cudaSetDevice(L->ctx->device));
  if (L->owner) VB_TRY(mlp_wait_side(L->owner));
  return write_opts(L, opts);
}

extern "C" int vbnn_mlp_set_opts(vbnn_mlp* m, const vbnn_opts* opts) {
  VB_CHECK(m && opts, VBNN_E_INVALID, "vbnn_mlp_set_opts: null argument");
  VB_TRY(refuse_set_in_capture(m->ctx, "vbnn_mlp_set_opts"));
  for (const vbnn_layer* L : m->layers) VB_TRY(check_opts(L, opts, "vbnn_mlp_set_opts"));
  VB_CUDA(cudaSetDevice(m->ctx->device));
  VB_TRY(mlp_wait_side(m));
  for (vbnn_layer* L : m->layers) VB_TRY(write_opts(L, opts));
  m->opts = *opts;
  return VBNN_OK;
}

static int buf_lookup(vbnn_layer* L, int which, float** p, size_t* n) {
  const size_t W = (size_t)L->O * L->I;
  *p = nullptr; *n = W;
  switch (which) {
    case VBNN_BUF_MEANS: *p = L->means; break;
    case VBNN_BUF_LVARS: *p = L->lvars; break;
    case VBNN_BUF_BIAS: *p = L->bias; *n = L->O; break;
    case VBNN_BUF_WEIGHT: *p = L->weight; break;
    case VBNN_BUF_GRAD_WEIGHT: *p = L->gW; break;
    case VBNN_BUF_GRAD_SUM: *p = L->gS; break;
    case VBNN_BUF_GRAD_BIAS: *p = L->gb; *n = L->O; break;
    case VBNN_BUF_ADAM_M_MU: *p = L->m_mu; break;
    case VBNN_BUF_ADAM_V_MU: *p = L->v_mu; break;
    case VBNN_BUF_ADAM_M_VAR: *p = L->m_var; break;
    case VBNN_BUF_ADAM_V_VAR: *p = L->v_var; break;
    case VBNN_BUF_EPS: *p = L->eps; break;
    case VBNN_BUF_STDV: *p = L->stdv; break;
    case VBNN_BUF_MU_SQE: *p = L->mu_sqe; break;
    case VBNN_BUF_PRIOR_MEANS:
    case VBNN_BUF_PRIOR_LVARS:
      VB_CHECK(L->prior_kind == VBNN_PRIOR_PER_WEIGHT, VBNN_E_STATE,
               "buffer %d: the layer's prior is not VBNN_PRIOR_PER_WEIGHT (vbnn_layer_set_prior)", which);
      *p = which == VBNN_BUF_PRIOR_MEANS ? L->prior_means : L->prior_lvars;
      break;
    default:
      set_error("unknown buffer id %d", which);
      return VBNN_E_INVALID;
  }
  return VBNN_OK;
}

extern "C" int vbnn_layer_device_ptr(vbnn_layer* L, int which, float** ptr, size_t* count) {
  VB_CHECK(L && ptr, VBNN_E_INVALID, "null argument");
  size_t n;
  VB_TRY(buf_lookup(L, which, ptr, &n));
  if (count) *count = n;
  return VBNN_OK;
}

extern "C" int vbnn_layer_bind(vbnn_layer* L, int which, float* ptr) {
  VB_CHECK(L, VBNN_E_INVALID, "null layer");
  VB_CHECK(!L->owned_by_mlp, VBNN_E_STATE, "vbnn_layer_bind: the layer belongs to a vbnn_mlp (its gradients live in the mlp's arena)");
  float** slot = nullptr; bool* ext = nullptr;
  size_t n = (size_t)L->O * L->I;
  switch (which) {
    case VBNN_BUF_WEIGHT: slot = &L->weight; ext = &L->ext_weight; n *= (size_t)L->S_alloc; break;
    case VBNN_BUF_BIAS: slot = &L->bias; ext = &L->ext_bias; n = L->O; break;
    case VBNN_BUF_GRAD_WEIGHT: slot = &L->gW; ext = &L->ext_gW; break;
    case VBNN_BUF_GRAD_BIAS: slot = &L->gb; ext = &L->ext_gb; n = L->O; break;
    default:
      set_error("vbnn_layer_bind: buffer %d cannot be caller-owned (weight, bias, gradWeight, gradBias only)", which);
      return VBNN_E_INVALID;
  }
  VB_CHECK(*slot != nullptr, VBNN_E_STATE, "vbnn_layer_bind: buffer %d is not materialised in this mode", which);
  VB_CHECK(ptr == nullptr || (reinterpret_cast<uintptr_t>(ptr) & 3) == 0, VBNN_E_INVALID, "vbnn_layer_bind: unaligned pointer");
  if (ptr == *slot) return VBNN_OK;
  cudaStream_t st = L->ctx->stream;
  if (ptr) {
    // adopt the caller's tensor AS IS: Torch moved the values itself when it re-flattened the storage, and
    // whatever the caller wrote since (mlp.lua:48-54 re-initialises weight / bias after getParameters) wins
    if (!*ext) {
      VB_CUDA(cudaStreamSynchronize(st));          // nothing of ours may still read the old buffer
      cudaFree(*slot);
    }
    *slot = ptr;
    *ext = true;
    return VBNN_OK;
  }
  if (!*ext) return VBNN_OK;
  float* fresh = nullptr;                          // hand the buffer back to the library, contents kept
  VB_TRY(dev_alloc(&fresh, n));
  VB_CUDA(cudaMemcpyAsync(fresh, *slot, n * 4, cudaMemcpyDeviceToDevice, st));
  VB_CUDA(cudaStreamSynchronize(st));
  *slot = fresh;
  *ext = false;
  return VBNN_OK;
}

extern "C" int vbnn_debug_knob(const char* name, int value, int* old_value) {
  int old = 0;
  VB_CHECK(knob_get(name, &old) == 0, VBNN_E_INVALID, "vbnn_debug_knob: unknown knob '%s'", name ? name : "(null)");
  if (old_value) *old_value = old;
  knob_set(name, value);
  return VBNN_OK;
}

extern "C" int vbnn_layer_get(vbnn_layer* L, int which, float* dst) {
  VB_CHECK(L && dst, VBNN_E_INVALID, "null argument");
  cudaStream_t st = L->ctx->stream;
  float* p; size_t n;
  VB_TRY(buf_lookup(L, which, &p, &n));
  if (L->shard_stale && *L->shard_stale) {
    const bool sharded = which == VBNN_BUF_MEANS || which == VBNN_BUF_LVARS || which == VBNN_BUF_ADAM_M_MU ||
                         which == VBNN_BUF_ADAM_V_MU || which == VBNN_BUF_ADAM_M_VAR || which == VBNN_BUF_ADAM_V_VAR ||
                         (which == VBNN_BUF_WEIGHT && L->kind == VBNN_KIND_LINEAR);
    VB_CHECK(!sharded, VBNN_E_STATE,
             "peer mode: rows owned by other ranks are out of date; call vbnn_mlp_sync_replicas on every rank first");
  }
  if (which == VBNN_BUF_WEIGHT && !p && L->w_bf16) {
    // bf16 precision keeps the sampled weights only as tensor-core operands: widen on the host
    std::vector<uint16_t> tmp((size_t)L->O * L->ldI);
    VB_CUDA(cudaMemcpyAsync(tmp.data(), L->w_bf16, tmp.size() * 2, cudaMemcpyDeviceToHost, st));
    VB_CUDA(cudaStreamSynchronize(st));
    for (int o = 0; o < L->O; ++o)
      for (int i = 0; i < L->I; ++i) {
        uint32_t u = (uint32_t)tmp[(size_t)o * L->ldI + i] << 16;
        memcpy(&dst[(size_t)o * L->I + i], &u, 4);
      }
    return VBNN_OK;
  }
  VB_CHECK(p != nullptr, VBNN_E_STATE, "buffer %d is not materialised in this mode", which);
  VB_CUDA(cudaMemcpyAsync(dst, p, n * 4, cudaMemcpyDeviceToHost, st));
  VB_CUDA(cudaStreamSynchronize(st));
  return VBNN_OK;
}

extern "C" int vbnn_layer_set(vbnn_layer* L, int which, const float* src) {
  VB_CHECK(L && src, VBNN_E_INVALID, "null argument");
  cudaStream_t st = L->ctx->stream;
  float* p; size_t n;
  if (which == VBNN_BUF_EPS && !L->eps) VB_TRY(dev_alloc(&L->eps, (size_t)L->O * L->I));
  VB_TRY(buf_lookup(L, which, &p, &n));
  VB_CHECK(p != nullptr, VBNN_E_STATE, "buffer %d is not materialised in this mode", which);
  VB_CUDA(cudaMemcpyAsync(p, src, n * 4, cudaMemcpyHostToDevice, st));
  VB_CUDA(cudaStreamSynchronize(st));
  if (which == VBNN_BUF_MEANS || which == VBNN_BUF_LVARS || (which == VBNN_BUF_WEIGHT && L->kind == VBNN_KIND_LINEAR)) {
    VB_TRY(layer_refresh_copies(L));
    L->prior_valid = false;
    VB_TRY(layer_refresh_prior_partials(L));
  }
  if (which == VBNN_BUF_WEIGHT && L->kind == VBNN_KIND_VB && L->w_bf16)
    VB_TRY(launch_cast(L->weight, L->I, L->O, L->I, L->w_bf16, nullptr, L->ldI, st));
  return VBNN_OK;
}

extern "C" int vbnn_layer_get_t(vbnn_layer* L, int* t) {
  VB_CHECK(L && t, VBNN_E_INVALID, "null argument");
  VB_CUDA(cudaMemcpyAsync(t, L->t_dev, sizeof(int), cudaMemcpyDeviceToHost, L->ctx->stream));
  VB_CUDA(cudaStreamSynchronize(L->ctx->stream));
  return VBNN_OK;
}
extern "C" int vbnn_layer_set_t(vbnn_layer* L, int t) {
  VB_CHECK(L, VBNN_E_INVALID, "null argument");
  VB_CUDA(cudaMemcpyAsync(L->t_dev, &t, sizeof(int), cudaMemcpyHostToDevice, L->ctx->stream));
  VB_CUDA(cudaStreamSynchronize(L->ctx->stream));
  return layer_refresh_prior_partials(L);
}

extern "C" int vbnn_layer_snr_count(vbnn_layer* L, float thresh, uint8_t* mask_dev, long long* count) {
  VB_CHECK(L && L->kind == VBNN_KIND_VB, VBNN_E_INVALID, "vbnn_layer_snr_count: not a VB layer");
  VB_TRY(check_params_fresh(L, "vbnn_layer_snr_count"));
  vbnn_ctx* c = L->ctx;
  unsigned long long* cnt = reinterpret_cast<unsigned long long*>(c->d_partials);
  VB_CUDA(cudaMemsetAsync(cnt, 0, 8, c->stream));
  VB_TRY(launch_snr(L->means, L->lvars, (long long)L->O * L->I, thresh, mask_dev, cnt, c->stream));
  c->launches++;
  if (count) {
    unsigned long long h = 0;
    VB_CUDA(cudaMemcpyAsync(&h, cnt, 8, cudaMemcpyDeviceToHost, c->stream));
    VB_CUDA(cudaStreamSynchronize(c->stream));
    *count = (long long)h;
  }
  return VBNN_OK;
}

extern "C" int vbnn_layer_draw_noise(vbnn_layer* L, uint32_t step, int sample_idx, int rows, int row0,
                                     float* out_dev) {
  VB_CHECK(L && out_dev, VBNN_E_INVALID, "null argument");
  PhiloxStream ps;
  if (layer_is_lrt(L)) {
    ps = layer_stream(L, kStreamZeta, sample_idx);
    ps.step = step;
    VB_TRY(launch_philox_matrix(out_dev, rows, L->O, row0, ps, L->ctx->stream));
  } else {
    ps = layer_stream(L, kStreamEps, sample_idx);
    ps.step = step;
    VB_TRY(launch_philox_matrix(out_dev, L->O, L->I, 0, ps, L->ctx->stream));
  }
  L->ctx->launches++;
  return VBNN_OK;
}

extern "C" int vbnn_philox_normal(vbnn_ctx* ctx, uint64_t seed, uint32_t step, uint32_t stream,
                                  uint32_t sample, int rows, int cols, int row0, float* out_dev) {
  VB_CHECK(ctx && out_dev && rows > 0 && cols > 0, VBNN_E_INVALID, "vbnn_philox_normal: bad argument");
  PhiloxStream ps;
  ps.key0 = (uint32_t)(seed & 0xFFFFFFFFu); ps.key1 = (uint32_t)(seed >> 32);
  ps.stream = stream; ps.sample = sample; ps.step = step;
  VB_TRY(launch_philox_matrix(out_dev, rows, cols, row0, ps, ctx->stream));
  ctx->launches++;
  return VBNN_OK;
}

extern "C" int vbnn_gemm_bf16(vbnn_ctx* ctx, const uint16_t* A, int lda, int a_kmajor, const uint16_t* B,
                              int ldb, int b_kmajor, float* D, int ldd, int M, int N, int K, int batch,
                              long long strideA, long long strideB, long long strideD) {
  VB_CHECK(ctx && A && B && D, VBNN_E_INVALID, "vbnn_gemm_bf16: null argument");
  GemmArgs g;
  memset(&g, 0, sizeof(g));
  g.M = M; g.N = N; g.K = K; g.batch = batch < 1 ? 1 : batch;
  g.A1 = {A, lda, a_kmajor, strideA};
  g.B1 = {B, ldb, b_kmajor, strideB};
  EpiParams p;
  memset(&p, 0, sizeof(p));
  p.M = M; p.N = N; p.out_f32 = D; p.ld_f32 = ldd; p.zs_f32 = strideD;
  return gemm(ctx, true, EPI_STORE, g, p);
}
