// mlp.cu -- the mlp.lua net object (mlp.lua:5-143) and the per-minibatch loop of
// main.lua:28-40 as device-resident sequences: all S Monte-Carlo samples are batched through
// each GEMM launch, the whole minibatch is replayed as one CUDA graph, and nothing returns to
// the host except the two scalars main.lua:38-39 accumulates.
#include <string.h>

#include "knobs.h"
#include "state.h"

using namespace vbnn;

namespace {

inline size_t esz(const vbnn_mlp* m) { return m->bf16 ? 2 : 4; }
inline int nlayers(const vbnn_mlp* m) { return (int)m->layers.size(); }
// LRT forward / backward-data as two single-accumulator GEMMs (default) or one dual-accumulator GEMM
// (VBNN_LRT_SPLIT bit 0: forward, bit 1: backward-data).  Measured on C3 under the 1000 W cap: the split
// forward is 7 % faster (its Philox-heavy epilogue hides under the MMAs), the split backward-data 3 %
// slower (its light epilogue gains nothing and the extra fp32 round trip costs energy) -> default 1.
inline bool lrt_split(const vbnn_mlp* m, int which) {
  return (knobs().lrt_split & which) != 0 && m->aux != nullptr;
}

// ---- stage the caller's minibatch into operand form (outside the graph: pointers vary) ----
int stage_input(vbnn_mlp* m, const float* X, const float* T, int N) {
  cudaStream_t st = m->ctx->stream;
  const int I0 = m->sizes[0], ld0 = m->ld[0];
  if (m->bf16) {
    VB_TRY(launch_cast(X, I0, N, I0, (bf16*)m->act[0], m->lrt ? (bf16*)m->act2[0] : nullptr, ld0, st));
    m->ctx->launches++;
  } else {
    VB_CUDA(cudaMemcpy2DAsync(m->act[0], (size_t)ld0 * 4, X, (size_t)I0 * 4, (size_t)I0 * 4, N,
                              cudaMemcpyDeviceToDevice, st));
    if (m->lrt) {
      if (ld0 != I0) VB_CUDA(cudaMemsetAsync(m->act2[0], 0, (size_t)N * ld0 * 4, st));
      VB_TRY(launch_square((const float*)m->act[0], (float*)m->act2[0], (long long)N * ld0, st));
      m->ctx->launches++;
    }
  }
  if (T) VB_CUDA(cudaMemcpyAsync(m->targets, T, (size_t)N * 4, cudaMemcpyDeviceToDevice, st));
  m->last_N = N;
  m->outputs_external = false;
  return VBNN_OK;
}

// the same from uint8 pixels, data.lua's normalisation fused (vbnn_mlp_submit_host_u8)
int stage_input_u8(vbnn_mlp* m, const uint8_t* X, const float* T, int N, float mean, float inv_std) {
  cudaStream_t st = m->ctx->stream;
  const int I0 = m->sizes[0], ld0 = m->ld[0];
  if (m->bf16)
    VB_TRY(launch_cast_u8(X, N, I0, mean, inv_std, (bf16*)m->act[0], m->lrt ? (bf16*)m->act2[0] : nullptr, ld0,
                          nullptr, nullptr, 0, st));
  else
    VB_TRY(launch_cast_u8(X, N, I0, mean, inv_std, nullptr, nullptr, 0, (float*)m->act[0],
                          m->lrt ? (float*)m->act2[0] : nullptr, ld0, st));
  m->ctx->launches++;
  if (T) VB_CUDA(cudaMemcpyAsync(m->targets, T, (size_t)N * 4, cudaMemcpyDeviceToDevice, st));
  m->last_N = N;
  m->outputs_external = false;
  return VBNN_OK;
}

// mlp:sample() for Zrun samples at once (mlp.lua:69-74 x main.lua:32-33)
int sample_all(vbnn_mlp* m, int sample0, int Zrun) {
  for (vbnn_layer* L : m->layers) {
    if (L->kind != VBNN_KIND_VB || layer_is_lrt(L)) continue;
    SampleParams p;
    memset(&p, 0, sizeof(p));
    p.mu = L->means;
    if (L->opts.strict_reference) { p.sig = L->stdv; p.sig_is_lvar = 0; }    // quirk Q1
    else { p.sig = L->lvars; p.sig_is_lvar = 1; }
    p.O = L->O; p.I = L->I; p.S = Zrun;
    p.ps = layer_stream(L, kStreamEps, sample0);
    p.step_ptr = m->ctx->d_step;
    p.w_f32 = L->weight;
    p.w_bf16 = L->w_bf16; p.ld_bf16 = L->ldI; p.zs_bf16 = (long long)L->O * L->ldI;
    p.eps16 = knobs().dw_eps16 ? L->eps16 : nullptr;
    VB_TRY(launch_sample_w(p, m->ctx->stream));
    m->ctx->launches++;
    L->map_mode = false;
    L->eps_injected = false;
    L->eps16_valid = p.eps16 != nullptr;
  }
  return VBNN_OK;
}

int clamp_all(vbnn_mlp* m) {
  for (vbnn_layer* L : m->layers)
    if (L->kind == VBNN_KIND_VB) VB_TRY(vbnn_layer_clamp_to_map(L));
  return VBNN_OK;
}

// The split form of the dual LRT GEMM g (mode EPI_FWD_LRT or EPI_DX_LRT, bf16 only): one product alone into aux as a
// plain fp32 store, then the other with the LRT2 epilogue joining it -- forward: X mu^T first, then the variance
// X^2 s2^T; backward-data: H s2 first, then G mu with the 2 X .* T join.  Each GEMM has a single TMEM accumulator,
// double-buffered, so the epilogue of tile i runs under the MMAs of tile i+1 (the dual kernel fills all 512 TMEM
// columns and cannot).  Both launches are profiled under `mode`.
int gemm_lrt_split(vbnn_mlp* m, int mode, const GemmArgs& g, EpiParams p) {
  const bool fwd = mode == EPI_FWD_LRT;
  GemmArgs first = g, second = g;
  first.A2 = first.B2 = second.A2 = second.B2 = GemmOperand{};
  if (fwd) { second.A1 = g.A2; second.B1 = g.B2; }
  else { first.A1 = g.A2; first.B1 = g.B2; }
  const long long zs_aux = g.zsum ? 0 : (long long)p.M * m->ld_aux;       // summing form: the z = 0 slice only
  EpiParams p0;
  memset(&p0, 0, sizeof(p0));
  p0.M = p.M; p0.N = p.N;
  p0.out_f32 = m->aux; p0.ld_f32 = m->ld_aux; p0.zs_f32 = zs_aux;
  VB_TRY(gemm(m->ctx, m->bf16, EPI_STORE, first, p0, mode));
  p.aux = m->aux; p.ld_aux = m->ld_aux; p.zs_aux = zs_aux;
  return gemm(m->ctx, m->bf16, fwd ? EPI_FWD_LRT2 : EPI_DX_LRT2, second, p, mode);
}

// One layer forward for Zrun batched samples.
int forward_layer(vbnn_mlp* m, int j, int N, int Zrun, int sample0, bool map_mode) {
  vbnn_layer* L = m->layers[j];
  const bool last = j == nlayers(m) - 1;
  const bool lrt = layer_is_lrt(L) && !map_mode;
  const int ldi = m->ld[j], ldo = m->ld[j + 1];
  const long long zs_in = j == 0 ? 0 : (long long)N * ldi;
  const bool w_batched = L->kind == VBNN_KIND_VB && !layer_is_lrt(L) && !map_mode;
  EpiParams p;
  memset(&p, 0, sizeof(p));
  p.M = N; p.N = L->O;
  p.bias = L->bias;
  p.relu = last ? 0 : 1;
  p.ld_act = ldo; p.zs_act = (long long)N * ldo;
  if (last && m->ext_logits) {            // vbnn_mlp_forward_train: straight into the caller's dense [Z x N x C]
    p.out_f32 = m->ext_logits; p.ld_f32 = L->O; p.zs_f32 = (long long)N * L->O;
  } else if (last) {
    p.out_f32 = m->logits; p.ld_f32 = m->ld_logits; p.zs_f32 = (long long)N * m->ld_logits;
  } else {
    p.out_act = m->act[j + 1];
  }
  int mode = EPI_FWD;
  if (lrt) {
    mode = EPI_FWD_LRT;
    if (!last) p.out_act2 = m->act2[j + 1];
    p.r_out = m->R[j];
    p.ps = layer_stream(L, kStreamZeta, sample0);
    p.step_ptr = m->ctx->d_step;
    p.row0 = m->ctx->rank * N;
    // the zeta counter is uint32(global row * ceil(O/4) + col/4): refuse shapes where it would wrap
    VB_CHECK((unsigned long long)m->ctx->nranks * (unsigned long long)N * (unsigned long long)((L->O + 3) / 4) <= 0xFFFFFFFFull,
             VBNN_E_UNSUPPORTED, "Philox zeta counter would wrap: %d ranks x %d rows x %d outputs", m->ctx->nranks, N, L->O);
  }
  GemmArgs g;
  memset(&g, 0, sizeof(g));
  g.M = N; g.N = L->O; g.K = L->I; g.batch = Zrun;
  g.A1 = {m->act[j], ldi, 1, zs_in};
  if (lrt) g.A2 = {m->act2[j], ldi, 1, zs_in};
  weight_operands(g, L, 1, w_batched, lrt);
  if (lrt && lrt_split(m, 1)) return gemm_lrt_split(m, mode, g, p);
  return gemm(m->ctx, m->bf16, mode, g, p);
}

int loss_all(vbnn_mlp* m, int N, int Zrun, bool backward, float* logp_out, float* result) {
  const int Lc = nlayers(m);
  vbnn_layer* Lo = m->layers[Lc - 1];
  LossParams lp;
  memset(&lp, 0, sizeof(lp));
  lp.logits = m->logits; lp.ld_logits = m->ld_logits;
  lp.targets = m->targets;
  lp.N = N; lp.C = Lo->O; lp.Z = Zrun;
  lp.grad_scale = 1.0f / ((float)N * (float)m->ctx->nranks);     // ClassNLL size-average, global batch
  if (backward) {
    if (m->bf16) lp.g_bf16 = (bf16*)m->G[Lc - 1]; else lp.g_f32 = (float*)m->G[Lc - 1];
    lp.ld_g = m->ld[Lc];
  }
  lp.logp_out = logp_out;
  lp.result = result;
  lp.z_slot0 = 0;
  VB_TRY(launch_loss(lp, m->ctx->stream));
  m->ctx->launches++;
  if (backward && layer_is_lrt(Lo)) {
    VB_TRY(launch_mul_act(m->G[Lc - 1], m->ld[Lc], m->bf16, m->R[Lc - 1], m->ld[Lc], m->H[Lc - 1], m->ld[Lc],
                          (long long)Zrun * N, Lo->O, m->bf16, m->ctx->stream));
    m->ctx->launches++;
  }
  return VBNN_OK;
}

// updateGradInput of layer j (its gradInput is layer j-1's gradOutput, ReLU backward fused)
int backward_data_layer(vbnn_mlp* m, int j, int N, int Zrun) {
  if (j == 0 && !m->dX) return VBNN_OK;
  vbnn_layer* L = m->layers[j];
  const bool lrt = layer_is_lrt(L);
  const int ldi = m->ld[j], ldo = m->ld[j + 1];
  const long long zs_out = (long long)N * ldo;
  GemmArgs g;
  memset(&g, 0, sizeof(g));
  g.M = N; g.N = L->I; g.K = L->O; g.batch = Zrun;
  g.A1 = {m->G[j], ldo, 1, zs_out};
  if (lrt) g.A2 = {m->H[j], ldo, 1, zs_out};
  weight_operands(g, L, 0, L->kind == VBNN_KIND_VB && !lrt, lrt);
  EpiParams p;
  memset(&p, 0, sizeof(p));
  p.M = N; p.N = L->I;
  if (j > 0) {
    p.out_act = m->G[j - 1]; p.ld_act = ldi; p.zs_act = (long long)N * ldi;
    p.xprev = m->act[j]; p.ld_x = ldi; p.zs_x = (long long)N * ldi;
    p.mask = 1;                                                    // nn.ReLU backward
    if (layer_is_lrt(m->layers[j - 1])) { p.rprev = m->R[j - 1]; p.out_act2 = m->H[j - 1]; }
  } else {
    // vbnn_mlp_step_grad_input: the first layer's gradInput summed over the Z samples, dX = sum_z dl_z/dX, written
    // straight into the caller's [N x I0] buffer by ONE GEMM whose contraction runs over the samples too (no atomics,
    // no partials).  Nothing below the input: no ReLU mask.  The staged input act[0] is shared by every sample
    // (zs_x = 0), so the LRT join is exact on the sums: sum_z (G_z mu + 2 X .* H_z s2) = (sum_z G_z) mu +
    // 2 X .* ((sum_z H_z) s2).
    g.zsum = 1;
    p.out_f32 = m->dX; p.ld_f32 = L->I;
    if (lrt) { p.xprev = m->act[0]; p.ld_x = ldi; p.zs_x = 0; }
  }
  const int mode = lrt ? EPI_DX_LRT : EPI_DX;
  if (lrt && lrt_split(m, 2)) return gemm_lrt_split(m, mode, g, p);
  return gemm(m->ctx, m->bf16, mode, g, p);
}

// accGradParameters of layer j (+ gradBias column sums)
int backward_weight_layer(vbnn_mlp* m, int j, int N, int Zrun, int sample0, int accumulate, bool scatter = false) {
  vbnn_layer* L = m->layers[j];
  const bool lrt = layer_is_lrt(L);
  const int ldi = m->ld[j], ldo = m->ld[j + 1];
  const long long zs_in = j == 0 ? 0 : (long long)N * ldi;
  const long long zs_out = (long long)N * ldo;
  cudaStream_t st = m->ctx->stream;
  {
    EpiParams p;
    memset(&p, 0, sizeof(p));
    p.M = L->O; p.N = L->I;
    p.gW = L->gW; p.gS = L->kind == VBNN_KIND_VB ? L->gS : nullptr; p.ld_g = L->I;
    p.scale = 1.f; p.accumulate = accumulate;
    p.ps = layer_stream(L, kStreamEps, sample0);
    p.step_ptr = m->ctx->d_step;
    if (L->eps_injected && Zrun == 1 && L->eps) p.noise = L->eps;      // parity mode: injected epsilon
    else if (L->eps16_valid && L->kind == VBNN_KIND_VB && !lrt) {      // this minibatch's epsilon, kept by sample_all
      p.eps16 = L->eps16; p.ld_e16 = L->ldI; p.zs_e16 = (long long)L->O * L->ldI;
    }
    if (scatter) peer_scatter(m, j, N, p);                             // reduce-scatter fused into the epilogue (or staged for the copy engines)
    const int mode = lrt ? EPI_DW_LRT : EPI_DW;
    // Dual dW (one launch, two accumulators, single-buffered TMEM) or two single-accumulator GEMMs
    // (double-buffered: the epilogue of tile i overlaps the MMAs of tile i+1).  On one GPU they tie; in
    // peer mode the epilogue's stores cross NVLink and the split form hides them (8 GPUs: 6.14 -> 5.97 ms).
    const int split_knob = knobs().dw_split;
    const bool split = split_knob >= 0 ? split_knob != 0 : (scatter && !peer_transport_ce(m, N));
    GemmArgs g;
    memset(&g, 0, sizeof(g));
    g.M = L->O; g.N = L->I; g.K = N; g.batch = Zrun;
    g.A1 = {m->G[j], ldo, 0, zs_out};
    g.B1 = {m->act[j], ldi, 0, zs_in};
    if (lrt) { g.A2 = {m->H[j], ldo, 0, zs_out}; g.B2 = {m->act2[j], ldi, 0, zs_in}; }
    const int lin_tiles = ceil_div(L->O, 128) * ceil_div(L->I, 128);
    if (m->bf16 && lrt && split) {
      // The two LRT parameter gradients are independent (g_mu = G^T X, g_s = H^T X^2): as two
      // single-accumulator GEMMs each tile needs half the TMEM, so the accumulator is double-buffered
      // and the epilogue of tile i hides behind the MMAs of tile i+1 (the dual kernel cannot).
      GemmArgs g1 = g;
      g1.A2 = g1.B2 = GemmOperand{};
      EpiParams p1 = p;
      p1.gS = nullptr;
      p1.noise = nullptr;
      VB_TRY(gemm(m->ctx, m->bf16, EPI_DW, g1, p1));
      g1.A1 = g.A2; g1.B1 = g.B2;
      p1.gW = L->gS;                      // plain accumulate of H^T X^2 into gradSum
      if (p1.scatter_rows)                // ... or into the owners' gradSum receive slots
        for (int q = 0; q < 8; ++q) p1.gW_peer[q] = p.gS_peer[q];
      p1.scale = 1.f;
      VB_TRY(gemm(m->ctx, m->bf16, EPI_DW, g1, p1));
    } else if (m->bf16 && L->kind == VBNN_KIND_LINEAR && Zrun > 1 && !scatter && m->dw_partials &&
               lin_tiles * 2 <= kNumSMs && (L->I & 3) == 0) {
      // plain nn.Linear with few output tiles (the 10 x 1200 output layer of C2: 10 tiles): one tile would walk
      // all Z * N rows serially (50 us for 0.25 GFLOP).  Instead every (tile, sample) pair is its own work unit
      // -- a batched plain-store GEMM into per-sample partial products -- and a fixed-order reduction adds them.
      EpiParams p0;
      memset(&p0, 0, sizeof(p0));
      p0.M = L->O; p0.N = L->I;
      p0.out_f32 = m->dw_partials; p0.ld_f32 = L->I; p0.zs_f32 = (long long)L->O * L->I;
      VB_TRY(gemm(m->ctx, m->bf16, EPI_STORE, g, p0, EPI_DW));
      VB_TRY(launch_sum_partials(m->dw_partials, Zrun, (long long)L->O * L->I, (long long)L->O * L->I, p.scale, accumulate,
                                 L->gW, st));
      m->ctx->launches++;
    } else {
      if (m->bf16 && L->kind == VBNN_KIND_LINEAR && Zrun > 1 && zs_in == (long long)N * ldi) {
        // plain nn.Linear (no per-sample epsilon): sum_z G_z^T X_z is ONE GEMM over K = Z * N rows, the
        // samples being contiguous in both operands -- no per-sample accumulator round trips
        g.K = N * Zrun; g.batch = 1;
        g.A1.zs = 0; g.B1.zs = 0;
      }
      VB_TRY(gemm(m->ctx, m->bf16, mode, g, p));
    }
  }
  // gradBias += G^T 1 summed over all samples (quirk Q3: never divided by S)
  VB_TRY(launch_colsum(m->G[j], m->bf16, (long long)Zrun * N, L->O, ldo, 1.f, L->gb, st));
  m->ctx->launches++;
  return VBNN_OK;
}

// model:backward for layer j (mlp.lua:79): updateGradInput (for the first layer only when the caller asked for
// the input gradient, vbnn_mlp_step_grad_input) + accGradParameters.
int backward_layer(vbnn_mlp* m, int j, int N, int Zrun, int sample0, int accumulate) {
  VB_TRY(backward_data_layer(m, j, N, Zrun));
  return backward_weight_layer(m, j, N, Zrun, sample0, accumulate, false);
}

// model:forward of Zrun samples (mlp.lua:77) up to the output layer's pre-LogSoftMax outputs
int forward_samples(vbnn_mlp* m, int N, int Zrun, int sample0, bool peer = false) {
  const int Lc = nlayers(m);
  vbnn_ctx* c = m->ctx;
  for (int j = 0; j < Lc; ++j) {
    // peer mode: layer j's operands of the previous minibatch must have landed from every owner -- waited for
    // per layer, right before they are first read, so that the exchange of the layers updated last (see the
    // backward order below) hides behind the forward GEMMs of the layers before them
    if (peer && !m->peer_waited_all) { VB_TRY(peer_wait_params(m, j, true)); VB_TRY(prof_mark(c, 1)); }
    VB_TRY(forward_layer(m, j, N, Zrun, sample0, false));
    VB_TRY(prof_mark(c, 3));
  }
  return VBNN_OK;
}

// model:backward of Zrun samples (mlp.lua:79) from the output layer's gradient G[L-1] (and H[L-1])
int backward_samples(vbnn_mlp* m, int N, int Zrun, int sample0, int accumulate, bool reduce_overlap = false,
                     bool peer = false) {
  const int Lc = nlayers(m);
  vbnn_ctx* c = m->ctx;
  if (peer) {
    // Peer mode runs the backward-data chain first and the parameter-gradient GEMMs afterwards in FORWARD order
    // (same GEMMs, same operands: G_j / H_j stay in their per-layer buffers).  Layer 0 -- the first one the next
    // minibatch's forward needs -- then finishes its exchange (reduce-scatter in the dW epilogue, owner update,
    // operand all-gather on the side stream) while the dW GEMMs of the layers above still run, and the tail
    // after the last dW belongs to the output layer, which the next forward reads last.
    // The input gradient (m->dX, layer 0's backward-data) belongs to this chain and must stay before
    // backward_weight_layer(0): once layer 0 raises grad_ready, its owners may update it and all-gather the new
    // operands into this rank's mu_bf16 / s2_bf16 / w_bf16, which that GEMM reads.
    for (int j = Lc - 1; j >= (m->dX ? 0 : 1); --j) { VB_TRY(backward_data_layer(m, j, N, Zrun)); VB_TRY(prof_mark(c, 5)); }
    for (int j = 0; j < Lc; ++j) {
      VB_TRY(backward_weight_layer(m, j, N, Zrun, sample0, accumulate, true));
      VB_TRY(prof_mark(c, 5));
      VB_TRY(peer_after_dw(m, j));       // signal; owner update + all-gather of layer j on the side stream
    }
    return VBNN_OK;
  }
  for (int j = Lc - 1; j >= 0; --j) {
    VB_TRY(backward_layer(m, j, N, Zrun, sample0, accumulate));
    VB_TRY(prof_mark(c, 5));
    // reduce_overlap: the allreduce of layer j's {gW, gS, gb} slice starts on the communication stream as soon as
    // its dW is done and overlaps the backward of the layers below
    if (reduce_overlap) {
      VB_CUDA(cudaEventRecord(m->ev_bwd[j], c->stream));
      VB_CUDA(cudaStreamWaitEvent(c->comm_stream, m->ev_bwd[j], 0));
      VB_TRY(comm_allreduce_internal(c, m->grad_arena + m->grad_off[j], m->grad_len[j], c->comm_stream));
      VB_CUDA(cudaEventRecord(m->ev_red[j], c->comm_stream));
    }
  }
  return VBNN_OK;
}

int update_all(vbnn_mlp* m, bool wait_reduce = false) {
  const int Lc = nlayers(m);
  cudaStream_t st = m->ctx->stream;
  // mlp.lua:117-142: SGD on the output layer first, then the VB layers.  The layers are independent,
  // so with the overlapped allreduce they are updated top-down, each as soon as its reduction lands.
  if (m->layers[Lc - 1]->kind == VBNN_KIND_LINEAR) {
    if (wait_reduce) VB_CUDA(cudaStreamWaitEvent(st, m->ev_red[Lc - 1], 0));
    VB_TRY(layer_update_internal(m->layers[Lc - 1], nullptr, false));
  }
  if (wait_reduce) {
    for (int j = Lc - 1; j >= 0; --j) {
      if (m->layers[j]->kind != VBNN_KIND_VB) continue;
      VB_CUDA(cudaStreamWaitEvent(st, m->ev_red[j], 0));
      VB_TRY(layer_update_internal(m->layers[j], nullptr, false));
    }
  } else {
    for (vbnn_layer* L : m->layers)
      if (L->kind == VBNN_KIND_VB) VB_TRY(layer_update_internal(L, nullptr, false));
  }
  return VBNN_OK;
}

// The first half of one minibatch after input staging (main.lua:28-34 up to the criterion): the gradBias reset, the
// peer waits, mlp:sample() and the forward of the S samples.
int step_forward(vbnn_mlp* m, int N) {
  cudaStream_t st = m->ctx->stream;
  for (vbnn_layer* L : m->layers) VB_CUDA(cudaMemsetAsync(L->gb, 0, (size_t)L->O * 4, st));   // main.lua:28
  const bool peer = m->peer && m->peer->active;
  if (peer) {
    // data parallel over NVLink peer memory (peer.cu): no collective call anywhere in the step
    VB_TRY(peer_check(m));
    m->peer_waited_all = !m->lrt;
    if (!m->lrt) {                                   // weight sampling reads mu / log sigma^2 of every layer up front
      VB_TRY(peer_wait_params(m, -1, true));
      VB_TRY(prof_mark(m->ctx, 1));
    }
  } else {
    VB_TRY(prof_mark(m->ctx, 1));
  }
  VB_TRY(sample_all(m, 0, m->Z));                                                              // :33
  VB_TRY(prof_mark(m->ctx, 2));
  return forward_samples(m, N, m->Z, 0, peer);                                                 // :34
}

// The second half, from the output layer's gradient on: backward, [exchange], update, [the fused loss's result] and
// the step-counter bump.
int step_backward(vbnn_mlp* m, int N, bool finalize) {
  cudaStream_t st = m->ctx->stream;
  if (m->peer && m->peer->active) {
    VB_TRY(backward_samples(m, N, m->Z, 0, 0, false, true));
    if (finalize) { VB_TRY(launch_finalize_result(m->result_acc, m->Z, N, m->result, st)); m->ctx->launches++; }
    VB_TRY(launch_bump(m->ctx->d_step, m->t_list_dev, 0, st));    // the layers' t counters advance on the side stream
    m->ctx->launches++;
    VB_TRY(prof_mark(m->ctx, 7));
    return VBNN_OK;
  }
  const bool dp = m->ctx->nranks > 1;
  const bool overlap = dp && knobs().dp_overlap && m->ctx->comm_stream != nullptr;
  VB_TRY(backward_samples(m, N, m->Z, 0, /*accumulate=*/0, overlap));                          // :34
  if (dp && !overlap) VB_TRY(comm_allreduce_internal(m->ctx, m->grad_arena, m->grad_count, st));
  VB_TRY(update_all(m, overlap));                                                              // :40
  VB_TRY(prof_mark(m->ctx, 6));
  if (finalize) {                                                                              // :38-39
    VB_TRY(launch_finalize_result(m->result_acc, m->Z, N, m->result, st));
    m->ctx->launches++;
  }
  VB_TRY(launch_bump(m->ctx->d_step, m->t_list_dev, m->n_t, st));
  m->ctx->launches++;
  VB_TRY(prof_mark(m->ctx, 7));
  return VBNN_OK;
}

// everything of one minibatch after input staging: main.lua:28-40
int step_body(vbnn_mlp* m, int N) {
  VB_TRY(prof_mark(m->ctx, 0));
  VB_CUDA(cudaMemsetAsync(m->result_acc, 0, (size_t)2 * m->Z * 4, m->ctx->stream));
  VB_TRY(step_forward(m, N));
  VB_TRY(loss_all(m, N, m->Z, true, nullptr, m->result_acc));
  VB_TRY(prof_mark(m->ctx, 4));
  return step_backward(m, N, true);
}

// vbnn_mlp_backward_update's half: the caller's dL/dY becomes the output layer's gradient operand, then the rest of
// the step.  Phase mark 0 first, so that the caller's loss since the forward half is not timed as this step's.
int split_backward_body(vbnn_mlp* m, int N, const float* grad) {
  const int Lc = nlayers(m);
  vbnn_layer* Lo = m->layers[Lc - 1];
  VB_TRY(prof_mark(m->ctx, 0));
  VB_TRY(launch_grad_logits(grad, (long long)m->Z * N, Lo->O, m->G[Lc - 1], m->ld[Lc],
                            layer_is_lrt(Lo) ? m->R[Lc - 1] : nullptr, m->H[Lc - 1], m->bf16, m->ctx->stream));
  m->ctx->launches++;
  VB_TRY(prof_mark(m->ctx, 4));
  return step_backward(m, N, false);
}

// body() enqueued eagerly, or captured once into sg and replayed while (N, key) stays the same: one GPU, a
// capturable stream, profiling off, and never on the first call (which warms up and allocates lazily)
template <typename Body>
int graph_enqueue(vbnn_mlp* m, vbnn_mlp::StepGraph& sg, int N, const void* key0, const void* key1, Body&& body) {
  vbnn_ctx* c = m->ctx;
  cudaStream_t st = c->stream;
  const bool graphable = m->use_graph && c->capturable && c->nranks == 1 && !c->profiling;
  if (!graphable || sg.eager_steps < 1) {
    sg.eager_steps++;
    return body();
  }
  if (sg.exec && (sg.N != N || sg.key[0] != key0 || sg.key[1] != key1)) {
    cudaGraphExecDestroy(sg.exec);
    sg.exec = nullptr;
  }
  if (!sg.exec) {
    const long long before = c->launches;
    VB_CUDA(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
    int r = body();
    cudaGraph_t gr = nullptr;
    cudaError_t e = cudaStreamEndCapture(st, &gr);
    if (r != VBNN_OK) { if (gr) cudaGraphDestroy(gr); return r; }
    if (e != cudaSuccess) { set_error("cudaStreamEndCapture: %s", cudaGetErrorString(e)); return VBNN_E_CUDA; }
    e = cudaGraphInstantiate(&sg.exec, gr, 0);
    cudaGraphDestroy(gr);
    if (e != cudaSuccess) { set_error("cudaGraphInstantiate: %s", cudaGetErrorString(e)); sg.exec = nullptr; return VBNN_E_CUDA; }
    sg.N = N;
    sg.key[0] = key0; sg.key[1] = key1;
    sg.launches = c->launches - before;
    c->launches = before;
    m->graph_captures++;
  }
  VB_CUDA(cudaGraphLaunch(sg.exec, st));
  c->launches += sg.launches;
  return VBNN_OK;
}

int step_enqueue(vbnn_mlp* m, int N) {
  // m->dX set: vbnn_mlp_step_grad_input, whose graph bakes the caller's buffer into its first-layer dX GEMM
  return graph_enqueue(m, m->graphs[m->dX ? vbnn_mlp::kGraphStepDx : vbnn_mlp::kGraphStep], N, m->dX, nullptr,
                       [&] { return step_body(m, N); });
}

// While a split step is open, only vbnn_mlp_backward_update and vbnn_mlp_reset_gradients may enqueue work.
int refuse_open_step(const vbnn_mlp* m, const char* who) {
  VB_CHECK(!m->step_open, VBNN_E_STATE,
           "%s: a vbnn_mlp_forward_train step is open: close it with vbnn_mlp_backward_update (or abandon it with "
           "vbnn_mlp_reset_gradients)", who);
  return VBNN_OK;
}

// The evaluation forward of vbnn_mlp_test and vbnn_mlp_predict (mlp.lua:86-107): stage the input, wait for the
// peers' parameters, then one MAP pass (n_samples == 0, quicktest) or n_samples sampled passes in chunks of Z whose
// noise indices (1 << 20) + t never reuse a training sample.  consume(zc, first, last) runs after each chunk.
// samples (vbnn_mlp_predict_outputs): the output layer's epilogue stores sample t into the caller's dense
// [T x N x C] buffer at t * N * C instead of `logits`; the caller resets m->ext_logits afterwards, error or not.
template <typename Consume>
int eval_forward(vbnn_mlp* m, const float* X, const float* T, int N, int n_samples, const char* who,
                 Consume&& consume, float* samples = nullptr) {
  VB_TRY(stage_input(m, X, T, N));
  if (m->peer && m->peer->active) {
    VB_CHECK(n_samples > 0 || !m->peer->stale, VBNN_E_STATE,
             "%s(quicktest) in peer mode: call vbnn_mlp_sync_replicas on every rank first", who);
    VB_TRY(peer_wait_params(m, -1, false));
  }
  const int Lc = nlayers(m);
  const long long C = m->sizes.back();
  if (n_samples == 0) {
    if (samples) m->ext_logits = samples;
    VB_TRY(clamp_all(m));                                                    // mlp.lua:88-90 (quicktest)
    for (int j = 0; j < Lc; ++j) VB_TRY(forward_layer(m, j, N, 1, 0, true));
    VB_TRY(consume(1, true, true));
    for (vbnn_layer* L : m->layers) L->map_mode = false;
    return VBNN_OK;
  }
  const int base = 1 << 20;                                                  // test noise never reuses train samples
  for (int s0 = 0; s0 < n_samples; s0 += m->Z) {                             // mlp.lua:94-100
    const int zc = n_samples - s0 < m->Z ? n_samples - s0 : m->Z;
    if (samples) m->ext_logits = samples + (long long)s0 * N * C;
    VB_TRY(sample_all(m, base + s0, zc));
    for (int j = 0; j < Lc; ++j) VB_TRY(forward_layer(m, j, N, zc, base + s0, false));
    VB_TRY(consume(zc, s0 == 0, s0 + zc == n_samples));
  }
  return VBNN_OK;
}

// the first call of an evaluation entry point allocates its state: not while the stream is being captured
int refuse_capture(cudaStream_t st, const char* who) {
  cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
  VB_CUDA(cudaStreamIsCapturing(st, &cs));
  VB_CHECK(cs == cudaStreamCaptureStatusNone, VBNN_E_STATE, "%s: the first call allocates its state and cannot be captured",
           who);
  return VBNN_OK;
}

// per-block {sum, sum} partials of vbnn_mlp_predict and vbnn_mlp_predict_outputs [kMaxPartials x 2]
int ensure_pred_partials(vbnn_mlp* m) {
  if (m->pred_partials) return VBNN_OK;
  return dev_alloc(&m->pred_partials, (size_t)kMaxPartials * 2);
}

}  // namespace

// a prior change (vbnn_layer_set_prior): the update kernels the graphs captured bake the old prior in
void vbnn::mlp_drop_graphs(vbnn_mlp* m) {
  for (vbnn_mlp::StepGraph& sg : m->graphs)
    if (sg.exec) { cudaGraphExecDestroy(sg.exec); sg.exec = nullptr; }
}

// ============================================================ create / destroy =============
extern "C" int vbnn_mlp_create(vbnn_ctx* ctx, const int* sizes, int n_sizes, int vb_output, int max_batch,
                               const vbnn_opts* opts, vbnn_mlp** out) {
  VB_CHECK(ctx && sizes && opts && out, VBNN_E_INVALID, "vbnn_mlp_create: null argument");
  VB_CHECK(n_sizes >= 2 && max_batch > 0 && opts->S >= 1 && opts->S <= 2048, VBNN_E_INVALID,
           "vbnn_mlp_create: need >= 2 sizes, max_batch > 0, 1 <= S <= 2048");
  VB_CUDA(cudaSetDevice(ctx->device));
  vbnn_mlp* m = new vbnn_mlp();
  m->ctx = ctx; m->opts = *opts; m->vb_output = vb_output; m->max_batch = max_batch;
  m->bf16 = opts->precision == VBNN_PREC_BF16;
  m->lrt = opts->reparam == VBNN_REPARAM_LOCAL;
  m->Z = opts->S;
  m->sizes.assign(sizes, sizes + n_sizes);
  for (int k = 0; k < n_sizes; ++k) {
    VB_CHECK(sizes[k] > 0, VBNN_E_INVALID, "vbnn_mlp_create: size[%d] = %d", k, sizes[k]);
    m->ld.push_back(round_up(sizes[k], 8));
  }
  const int Lc = n_sizes - 1;
  cudaStream_t st = ctx->stream;
  int r = VBNN_OK;
  // ---- gradient arena {gW, gS, gb} per layer, contiguous: one allreduce (SURVEY 8e) ----
  std::vector<size_t> off_gW(Lc), off_gS(Lc), off_gb(Lc);
  size_t off = 0;
  auto take = [&](size_t n) { size_t o = off; off += (n + 63) / 64 * 64; return o; };
  for (int j = 0; j < Lc; ++j) {
    const bool vb = j < Lc - 1 || vb_output;
    const size_t W = (size_t)sizes[j] * sizes[j + 1];
    off_gW[j] = take(W);
    off_gS[j] = vb ? take(W) : 0;
    off_gb[j] = take(sizes[j + 1]);
    m->grad_off.push_back(off_gW[j]);
    m->grad_len.push_back(off - off_gW[j]);
  }
  m->grad_count = off;
  r = dev_alloc(&m->grad_arena, off);
  if (r == VBNN_OK && cudaMemsetAsync(m->grad_arena, 0, off * 4, st) != cudaSuccess) r = VBNN_E_CUDA;
  for (int j = 0; j < Lc && r == VBNN_OK; ++j) {
    const bool vb = j < Lc - 1 || vb_output;
    vbnn_layer* L = nullptr;
    r = layer_create_internal(ctx, sizes[j], sizes[j + 1], vb ? VBNN_KIND_VB : VBNN_KIND_LINEAR, opts,
                              (vb && !m->lrt) ? m->Z : 1, m->grad_arena + off_gW[j],
                              vb ? m->grad_arena + off_gS[j] : nullptr, m->grad_arena + off_gb[j], j, &L);
    if (r == VBNN_OK) { L->owned_by_mlp = true; L->owner = m; m->layers.push_back(L); }
  }
  // ---- activations ----
  const size_t e = esz(m);
  const size_t ZN = (size_t)m->Z * max_batch;
  m->act.assign(n_sizes, nullptr); m->act2.assign(n_sizes, nullptr);
  m->R.assign(Lc, nullptr); m->G.assign(Lc, nullptr); m->H.assign(Lc, nullptr);
  auto A_ = [&](void** p, size_t bytes) { if (r == VBNN_OK) { char* q; r = dev_alloc(&q, bytes); *p = q; } };
  A_(&m->act[0], (size_t)max_batch * m->ld[0] * e);
  if (m->lrt) A_(&m->act2[0], (size_t)max_batch * m->ld[0] * e);
  for (int j = 0; j < Lc; ++j) {
    const bool vb = j < Lc - 1 || vb_output;
    const size_t bytes = ZN * m->ld[j + 1] * e;
    if (j < Lc - 1) {
      A_(&m->act[j + 1], bytes);
      if (m->lrt) A_(&m->act2[j + 1], bytes);
    }
    A_(&m->G[j], bytes);
    if (m->lrt && vb) { A_(&m->R[j], bytes); A_(&m->H[j], bytes); }
  }
  if (m->lrt && m->bf16) {
    int mx = 0;
    for (int k = 0; k < n_sizes; ++k) mx = m->ld[k] > mx ? m->ld[k] : mx;
    m->ld_aux = mx;
    A_((void**)&m->aux, ZN * (size_t)mx * 4);
  }
  if (m->bf16 && m->Z > 1 && !vb_output)
    A_((void**)&m->dw_partials, (size_t)m->Z * sizes[Lc - 1] * sizes[Lc] * 4);
  m->ld_logits = m->ld[Lc];
  A_((void**)&m->logits, ZN * m->ld_logits * 4);
  A_((void**)&m->targets, (size_t)max_batch * 4);
  A_((void**)&m->result_acc, (size_t)2 * m->Z * 4);
  A_((void**)&m->result, 2 * 4);
  // Adam/SGD step counters of all layers, bumped by one tiny kernel per minibatch
  if (r == VBNN_OK) {
    std::vector<int*> ts;
    for (vbnn_layer* L : m->layers) ts.push_back(L->t_dev);
    m->n_t = (int)ts.size();
    r = dev_alloc(&m->t_list_dev, ts.size());
    if (r == VBNN_OK &&
        cudaMemcpyAsync(m->t_list_dev, ts.data(), ts.size() * sizeof(int*), cudaMemcpyHostToDevice, st) != cudaSuccess)
      r = VBNN_E_CUDA;
    if (r == VBNN_OK) cudaStreamSynchronize(st);
  }
  for (int s = 0; s < 2; ++s) { m->slots[s].busy = false; m->slots[s].h_result = nullptr; m->slots[s].copied = nullptr; }
  for (int j = 0; j < Lc && r == VBNN_OK; ++j) {
    cudaEvent_t a, b;
    if (cudaEventCreateWithFlags(&a, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&b, cudaEventDisableTiming) != cudaSuccess) { r = VBNN_E_CUDA; break; }
    m->ev_bwd.push_back(a); m->ev_red.push_back(b);
  }
  if (knobs().no_graph) m->use_graph = false;
  if (r != VBNN_OK) { vbnn_mlp_destroy(m); return r; }
  *out = m;
  return VBNN_OK;
}

extern "C" int vbnn_mlp_destroy(vbnn_mlp* m) {
  if (!m) return VBNN_OK;
  cudaSetDevice(m->ctx->device);
  cudaStreamSynchronize(m->ctx->stream);
  cudaStreamSynchronize(m->ctx->copy_stream);
  for (vbnn_mlp::StepGraph& sg : m->graphs)
    if (sg.exec) cudaGraphExecDestroy(sg.exec);
  peer_destroy(m);
  for (cudaEvent_t e : m->ev_bwd) cudaEventDestroy(e);
  for (cudaEvent_t e : m->ev_red) cudaEventDestroy(e);
  for (vbnn_layer* L : m->layers) vbnn_layer_destroy(L);
  for (void* p : m->act) if (p) cudaFree(p);
  for (void* p : m->act2) if (p) cudaFree(p);
  for (void* p : m->R) if (p) cudaFree(p);
  for (void* p : m->G) if (p) cudaFree(p);
  for (void* p : m->H) if (p) cudaFree(p);
  if (m->aux) cudaFree(m->aux);
  if (m->dw_partials) cudaFree(m->dw_partials);
  if (m->logits) cudaFree(m->logits);
  if (m->logp) cudaFree(m->logp);
  if (m->pred_max) cudaFree(m->pred_max);
  if (m->pred_sum) cudaFree(m->pred_sum);
  if (m->pred_ent) cudaFree(m->pred_ent);
  if (m->pred_partials) cudaFree(m->pred_partials);
  if (m->mom_state) cudaFree(m->mom_state);
  if (m->targets) cudaFree(m->targets);
  if (m->result_acc) cudaFree(m->result_acc);
  if (m->result) cudaFree(m->result);
  if (m->grad_arena) cudaFree(m->grad_arena);
  if (m->t_list_dev) cudaFree(m->t_list_dev);
  for (int s = 0; s < 2; ++s) {
    if (m->xstage[s]) cudaFree(m->xstage[s]);
    if (m->xstage_u8[s]) cudaFree(m->xstage_u8[s]);
    if (m->tstage[s]) cudaFree(m->tstage[s]);
    if (m->pipeline_ready) {
      cudaEventDestroy(m->slots[s].copied); cudaEventDestroy(m->slots[s].consumed); cudaEventDestroy(m->slots[s].done);
      if (m->slots[s].h_result) cudaFreeHost(m->slots[s].h_result);
    }
  }
  delete m;
  return VBNN_OK;
}

extern "C" int vbnn_mlp_num_layers(const vbnn_mlp* m) { return m ? (int)m->layers.size() : VBNN_E_INVALID; }

extern "C" int vbnn_mlp_layer(vbnn_mlp* m, int k, vbnn_layer** out) {
  VB_CHECK(m && out && k >= 0 && k < nlayers(m), VBNN_E_INVALID, "vbnn_mlp_layer: bad index %d", k);
  *out = m->layers[k];
  return VBNN_OK;
}

extern "C" int vbnn_mlp_init_params(vbnn_mlp* m, uint64_t seed, int he_means) {
  VB_CHECK(m, VBNN_E_INVALID, "null mlp");
  VB_TRY(refuse_open_step(m, "vbnn_mlp_init_params"));
  cudaStream_t st = m->ctx->stream;
  for (vbnn_layer* L : m->layers) {
    const long long W = (long long)L->O * L->I;
    PhiloxStream ps = layer_stream(L, kStreamInit, 1);
    ps.key0 = (uint32_t)(seed & 0xFFFFFFFFu); ps.key1 = (uint32_t)(seed >> 32);
    VB_CUDA(cudaMemsetAsync(L->bias, 0, (size_t)L->O * 4, st));                    // mlp.lua:49-50
    if (L->kind == VBNN_KIND_LINEAR) {
      VB_TRY(launch_init_normal(L->weight, W, 0.f, sqrtf(2.0f / (float)L->I), ps, st));   // mlp.lua:52-54
    } else {
      const float var_init = (L->opts.msr_init || he_means) ? 2.0f / (float)L->I : L->opts.var_init;
      if (he_means || L->opts.mu_init != 0.f)
        VB_TRY(launch_init_normal(L->means, W, 0.f, sqrtf(var_init), ps, st));     // VBLinear.lua:25-28
      else
        VB_CUDA(cudaMemsetAsync(L->means, 0, (size_t)W * 4, st));                  // VBLinear.lua:23
      VB_TRY(layer_compute_prior_internal(L));
      VB_TRY(layer_refresh_prior_partials(L));
    }
    VB_TRY(layer_refresh_copies(L));
    m->ctx->launches += 2;
  }
  return VBNN_OK;
}

// ============================================================ step pieces ==================
extern "C" int vbnn_mlp_reset_gradients(vbnn_mlp* m) {
  VB_CHECK(m, VBNN_E_INVALID, "null mlp");
  if (m->step_open) {
    // abandon the split step: no update, the step counter stays.  In peer mode the forward half has already
    // advanced the peers' flag protocol, so the step must be closed by vbnn_mlp_backward_update.
    VB_CHECK(!(m->peer && m->peer->active), VBNN_E_STATE,
             "vbnn_mlp_reset_gradients: an open step cannot be abandoned in peer mode; pass a zero gradient to "
             "vbnn_mlp_backward_update instead");
    m->step_open = false;
  }
  cudaStream_t st = m->ctx->stream;
  VB_CUDA(cudaMemsetAsync(m->grad_arena, 0, m->grad_count * 4, st));     // mlp.lua:63-66
  VB_CUDA(cudaMemsetAsync(m->result_acc, 0, (size_t)2 * m->Z * 4, st));
  return VBNN_OK;
}

extern "C" int vbnn_mlp_sample(vbnn_mlp* m, int sample_idx) {
  VB_CHECK(m, VBNN_E_INVALID, "null mlp");
  VB_TRY(refuse_open_step(m, "vbnn_mlp_sample"));
  for (vbnn_layer* L : m->layers) L->cur_sample = sample_idx;
  return sample_all(m, sample_idx, 1);
}

extern "C" int vbnn_mlp_run(vbnn_mlp* m, const float* X, const float* T, int N, int sample_idx,
                            float* err_host, float* acc_host) {
  VB_CHECK(m && X && T, VBNN_E_INVALID, "vbnn_mlp_run: null argument");
  VB_CHECK(N > 0 && N <= m->max_batch, VBNN_E_INVALID, "vbnn_mlp_run: N=%d exceeds max_batch=%d", N, m->max_batch);
  VB_TRY(refuse_open_step(m, "vbnn_mlp_run"));
  vbnn_ctx* c = m->ctx;
  cudaStream_t st = c->stream;
  VB_TRY(stage_input(m, X, T, N));
  float* racc = reinterpret_cast<float*>(c->d_partials);       // private slot: run() returns its own scalars
  VB_CUDA(cudaMemsetAsync(racc, 0, 8, st));
  const int Lc = nlayers(m);
  for (int j = 0; j < Lc; ++j) VB_TRY(forward_layer(m, j, N, 1, sample_idx, m->layers[j]->map_mode));
  VB_TRY(loss_all(m, N, 1, true, nullptr, racc));
  for (int j = Lc - 1; j >= 0; --j) VB_TRY(backward_layer(m, j, N, 1, sample_idx, 1));
  if (err_host || acc_host) {
    VB_CUDA(cudaMemcpyAsync(c->h_scalars, racc, 8, cudaMemcpyDeviceToHost, st));
    VB_CUDA(cudaStreamSynchronize(st));
    if (err_host) *err_host = c->h_scalars[0] / (float)N;                    // mlp.lua:80
    if (acc_host) *acc_host = c->h_scalars[1] / (float)N * 100.f;            // mlp.lua:82
  }
  return VBNN_OK;
}

extern "C" int vbnn_mlp_update(vbnn_mlp* m) {
  VB_CHECK(m, VBNN_E_INVALID, "null mlp");
  VB_TRY(refuse_open_step(m, "vbnn_mlp_update"));
  VB_CHECK(!(m->peer && m->peer->active), VBNN_E_UNSUPPORTED,
           "peer mode drives the whole minibatch through vbnn_mlp_step / vbnn_mlp_submit_host");
  if (m->ctx->nranks > 1)
    VB_TRY(comm_allreduce_internal(m->ctx, m->grad_arena, m->grad_count, m->ctx->stream));
  VB_TRY(update_all(m));
  VB_TRY(launch_bump(m->ctx->d_step, m->t_list_dev, m->n_t, m->ctx->stream));
  m->ctx->launches++;
  return VBNN_OK;
}

extern "C" int vbnn_mlp_calc_lc(vbnn_mlp* m, float* lc_host) {
  VB_CHECK(m && lc_host, VBNN_E_INVALID, "null argument");
  VB_TRY(refuse_open_step(m, "vbnn_mlp_calc_lc"));
  double lc = 0;
  for (vbnn_layer* L : m->layers) {
    if (L->kind != VBNN_KIND_VB) continue;
    float s = 0;
    VB_TRY(vbnn_layer_calc_lc(L, nullptr, &s));                              // mlp.lua:112
    lc += s;
  }
  *lc_host = (float)lc;
  return VBNN_OK;
}

extern "C" int vbnn_mlp_step(vbnn_mlp* m, const float* X, const float* T, int N, float* result_dev) {
  VB_CHECK(m && X && T, VBNN_E_INVALID, "vbnn_mlp_step: null argument");
  VB_CHECK(N > 0 && N <= m->max_batch, VBNN_E_INVALID, "vbnn_mlp_step: N=%d exceeds max_batch=%d", N, m->max_batch);
  VB_TRY(refuse_open_step(m, "vbnn_mlp_step"));
  VB_CUDA(cudaSetDevice(m->ctx->device));
  VB_TRY(stage_input(m, X, T, N));
  VB_TRY(step_enqueue(m, N));
  if (result_dev)
    VB_CUDA(cudaMemcpyAsync(result_dev, m->result, 8, cudaMemcpyDeviceToDevice, m->ctx->stream));
  return VBNN_OK;
}

extern "C" int vbnn_mlp_step_grad_input(vbnn_mlp* m, const float* X, const float* T, int N, float* result_dev,
                                        float* dX) {
  VB_CHECK(m && X && T && dX, VBNN_E_INVALID, "vbnn_mlp_step_grad_input: null argument");
  VB_CHECK(N > 0 && N <= m->max_batch, VBNN_E_INVALID, "vbnn_mlp_step_grad_input: N=%d exceeds max_batch=%d", N,
           m->max_batch);
  VB_TRY(refuse_open_step(m, "vbnn_mlp_step_grad_input"));
  VB_CUDA(cudaSetDevice(m->ctx->device));
  VB_TRY(stage_input(m, X, T, N));
  m->dX = dX;                             // read by backward_data_layer(0) and step_enqueue while the step is enqueued
  const int r = step_enqueue(m, N);
  m->dX = nullptr;
  VB_TRY(r);
  if (result_dev)
    VB_CUDA(cudaMemcpyAsync(result_dev, m->result, 8, cudaMemcpyDeviceToDevice, m->ctx->stream));
  return VBNN_OK;
}

extern "C" int vbnn_mlp_forward_train(vbnn_mlp* m, const float* X, int N, float* logits_dev) {
  VB_CHECK(m && X && logits_dev, VBNN_E_INVALID, "vbnn_mlp_forward_train: null argument");
  VB_CHECK(N > 0 && N <= m->max_batch, VBNN_E_INVALID, "vbnn_mlp_forward_train: N=%d outside 1..max_batch=%d", N,
           m->max_batch);
  VB_CHECK((reinterpret_cast<uintptr_t>(logits_dev) & 15) == 0, VBNN_E_INVALID,
           "vbnn_mlp_forward_train: logits_dev must be 16-byte aligned");
  VB_CHECK(!m->step_open, VBNN_E_STATE, "vbnn_mlp_forward_train: a step is already open: call "
           "vbnn_mlp_backward_update (or vbnn_mlp_reset_gradients) first");
  VB_CHECK(m->inflight == 0, VBNN_E_STATE, "vbnn_mlp_forward_train: %d host-pipeline minibatch(es) not collected",
           m->inflight);
  VB_CUDA(cudaSetDevice(m->ctx->device));
  VB_TRY(stage_input(m, X, nullptr, N));
  m->ext_logits = logits_dev;             // read by forward_layer(L-1) and the graph key while the half is enqueued
  const int r = graph_enqueue(m, m->graphs[vbnn_mlp::kGraphFwd], N, logits_dev, nullptr, [&] {
    VB_TRY(prof_mark(m->ctx, 0));
    return step_forward(m, N);
  });
  m->ext_logits = nullptr;
  VB_TRY(r);
  m->step_open = true;
  m->open_N = N;
  m->outputs_external = true;
  return VBNN_OK;
}

extern "C" int vbnn_mlp_backward_update(vbnn_mlp* m, const float* grad_dev, float* dX_dev) {
  VB_CHECK(m && grad_dev, VBNN_E_INVALID, "vbnn_mlp_backward_update: null argument");
  VB_CHECK(m->step_open, VBNN_E_STATE, "vbnn_mlp_backward_update: no open step: call vbnn_mlp_forward_train first");
  VB_CUDA(cudaSetDevice(m->ctx->device));
  const int N = m->open_N;
  m->step_open = false;                   // closed whatever the outcome: an error leaves the net to be re-initialised
  m->dX = dX_dev;                         // read by backward_data_layer(0) and the graph key while the half is enqueued
  // with and without dX in graphs of their own, so that each form runs eagerly once before it is captured (as
  // vbnn_mlp_step / vbnn_mlp_step_grad_input do) and alternating the two never re-captures
  vbnn_mlp::StepGraph& sg = m->graphs[dX_dev ? vbnn_mlp::kGraphBwdDx : vbnn_mlp::kGraphBwd];
  const int r = graph_enqueue(m, sg, N, grad_dev, dX_dev, [&] { return split_backward_body(m, N, grad_dev); });
  m->dX = nullptr;
  return r;
}

static int ensure_pipeline(vbnn_mlp* m) {
  if (m->pipeline_ready) return VBNN_OK;
  for (int s = 0; s < 2; ++s) {
    VB_TRY(dev_alloc(&m->xstage[s], (size_t)m->max_batch * m->sizes[0]));
    VB_TRY(dev_alloc(&m->tstage[s], (size_t)m->max_batch));
    VB_CUDA(cudaEventCreateWithFlags(&m->slots[s].copied, cudaEventDisableTiming));
    VB_CUDA(cudaEventCreateWithFlags(&m->slots[s].consumed, cudaEventDisableTiming));
    VB_CUDA(cudaEventCreateWithFlags(&m->slots[s].done, cudaEventDisableTiming));
    VB_CUDA(cudaMallocHost((void**)&m->slots[s].h_result, 16));
    m->slots[s].busy = false;
  }
  m->pipeline_ready = true;
  return VBNN_OK;
}

static int submit_host_any(vbnn_mlp* m, const float* X_host, const uint8_t* X8_host, const float* T_host, int N,
                           float mean, float inv_std) {
  VB_CHECK(m && (X_host || X8_host) && T_host, VBNN_E_INVALID, "vbnn_mlp_submit_host: null argument");
  VB_CHECK(N > 0 && N <= m->max_batch, VBNN_E_INVALID, "vbnn_mlp_submit_host: N=%d exceeds max_batch=%d", N, m->max_batch);
  VB_TRY(refuse_open_step(m, "vbnn_mlp_submit_host"));
  VB_CUDA(cudaSetDevice(m->ctx->device));
  VB_TRY(ensure_pipeline(m));
  VB_CHECK(m->inflight < 2, VBNN_E_STATE, "vbnn_mlp_submit_host: two minibatches in flight, collect first");
  vbnn_ctx* c = m->ctx;
  const int s = m->submit_idx & 1;
  vbnn_mlp::Slot& sl = m->slots[s];
  if (X8_host && !m->xstage_u8[s]) VB_TRY(dev_alloc(&m->xstage_u8[s], (size_t)m->max_batch * m->sizes[0]));
  // copy engine: wait until the previous user of this staging buffer has been consumed
  if (m->submit_idx >= 2) VB_CUDA(cudaStreamWaitEvent(c->copy_stream, sl.consumed, 0));
  if (X8_host)
    VB_CUDA(cudaMemcpyAsync(m->xstage_u8[s], X8_host, (size_t)N * m->sizes[0], cudaMemcpyHostToDevice, c->copy_stream));
  else
    VB_CUDA(cudaMemcpyAsync(m->xstage[s], X_host, (size_t)N * m->sizes[0] * 4, cudaMemcpyHostToDevice, c->copy_stream));
  VB_CUDA(cudaMemcpyAsync(m->tstage[s], T_host, (size_t)N * 4, cudaMemcpyHostToDevice, c->copy_stream));
  VB_CUDA(cudaEventRecord(sl.copied, c->copy_stream));
  // compute stream
  VB_CUDA(cudaStreamWaitEvent(c->stream, sl.copied, 0));
  if (X8_host) VB_TRY(stage_input_u8(m, m->xstage_u8[s], m->tstage[s], N, mean, inv_std));
  else VB_TRY(stage_input(m, m->xstage[s], m->tstage[s], N));
  VB_CUDA(cudaEventRecord(sl.consumed, c->stream));
  VB_TRY(step_enqueue(m, N));
  VB_CUDA(cudaMemcpyAsync(sl.h_result, m->result, 8, cudaMemcpyDeviceToHost, c->stream));
  VB_CUDA(cudaEventRecord(sl.done, c->stream));
  sl.busy = true; sl.N = N;
  m->submit_idx++; m->inflight++;
  return VBNN_OK;
}

extern "C" int vbnn_mlp_submit_host(vbnn_mlp* m, const float* X_host, const float* T_host, int N) {
  VB_CHECK(X_host, VBNN_E_INVALID, "vbnn_mlp_submit_host: null argument");
  return submit_host_any(m, X_host, nullptr, T_host, N, 0.f, 1.f);
}

extern "C" int vbnn_mlp_submit_host_u8(vbnn_mlp* m, const uint8_t* X_host, const float* T_host, int N, float mean,
                                       float inv_std) {
  VB_CHECK(X_host, VBNN_E_INVALID, "vbnn_mlp_submit_host_u8: null argument");
  return submit_host_any(m, nullptr, X_host, T_host, N, mean, inv_std);
}

int vbnn::mlp_wait_side(vbnn_mlp* m) {
  if (m->peer && m->peer->active) {
    VB_CUDA(cudaEventRecord(m->peer->ev_side, m->peer->side));     // the side stream already waits for the transfer stream
    VB_CUDA(cudaStreamWaitEvent(m->ctx->stream, m->peer->ev_side, 0));
  }
  return VBNN_OK;
}

extern "C" int vbnn_mlp_join_streams(vbnn_mlp* m) {
  VB_CHECK(m, VBNN_E_INVALID, "null mlp");
  vbnn_ctx* c = m->ctx;
  VB_TRY(mlp_wait_side(m));
  if (c->comm_stream && !m->ev_red.empty()) {
    VB_CUDA(cudaEventRecord(m->ev_red[0], c->comm_stream));
    VB_CUDA(cudaStreamWaitEvent(c->stream, m->ev_red[0], 0));
  }
  return VBNN_OK;
}

extern "C" int vbnn_mlp_collect(vbnn_mlp* m, float* err_host, float* acc_host) {
  VB_CHECK(m, VBNN_E_INVALID, "null mlp");
  VB_CHECK(m->inflight > 0, VBNN_E_STATE, "vbnn_mlp_collect: nothing in flight");
  vbnn_mlp::Slot& sl = m->slots[m->collect_idx & 1];
  VB_CUDA(cudaEventSynchronize(sl.done));
  VB_TRY(peer_check(m));
  if (err_host) *err_host = sl.h_result[0];
  if (acc_host) *acc_host = sl.h_result[1];
  sl.busy = false;
  m->collect_idx++; m->inflight--;
  return VBNN_OK;
}

extern "C" int vbnn_mlp_step_host(vbnn_mlp* m, const float* X_host, const float* T_host, int N,
                                  float* err_host, float* acc_host) {
  VB_TRY(vbnn_mlp_submit_host(m, X_host, T_host, N));
  return vbnn_mlp_collect(m, err_host, acc_host);
}

extern "C" int vbnn_mlp_test(vbnn_mlp* m, const float* X, const float* T, int N, int n_samples,
                             float* err_host, float* acc_host) {
  VB_CHECK(m && X && T, VBNN_E_INVALID, "vbnn_mlp_test: null argument");
  VB_CHECK(N > 0 && N <= m->max_batch && n_samples >= 0, VBNN_E_INVALID, "vbnn_mlp_test: bad N/n_samples");
  VB_TRY(refuse_open_step(m, "vbnn_mlp_test"));
  vbnn_ctx* c = m->ctx;
  cudaStream_t st = c->stream;
  VB_CUDA(cudaMemsetAsync(m->result_acc, 0, (size_t)2 * m->Z * 4, st));
  VB_TRY(eval_forward(m, X, T, N, n_samples, "vbnn_mlp_test",
                      [&](int zc, bool, bool) { return loss_all(m, N, zc, false, nullptr, m->result_acc); }));
  const int total = n_samples == 0 ? 1 : n_samples;
  VB_CUDA(cudaMemcpyAsync(c->h_scalars, m->result_acc, (size_t)2 * m->Z * 4, cudaMemcpyDeviceToHost, st));
  VB_CUDA(cudaStreamSynchronize(st));
  double e = 0, a = 0;
  for (int z = 0; z < m->Z; ++z) { e += c->h_scalars[2 * z]; a += c->h_scalars[2 * z + 1]; }
  if (err_host) *err_host = (float)(e / ((double)total * N));               // mlp.lua:101
  if (acc_host) *acc_host = (float)(a / ((double)total * N) * 100.0);
  return VBNN_OK;
}

extern "C" int vbnn_mlp_predict(vbnn_mlp* m, const float* X, int N, int n_samples, const float* targets,
                                float* logp_dev, float* unc_dev, float* nll_host, float* acc_host) {
  VB_CHECK(m && X, VBNN_E_INVALID, "vbnn_mlp_predict: null argument");
  VB_CHECK(N > 0 && N <= m->max_batch && n_samples >= 0, VBNN_E_INVALID,
           "vbnn_mlp_predict: N=%d (max_batch %d), n_samples=%d", N, m->max_batch, n_samples);
  VB_CHECK(targets || !(nll_host || acc_host), VBNN_E_INVALID, "vbnn_mlp_predict: nll / accuracy need targets");
  VB_TRY(refuse_open_step(m, "vbnn_mlp_predict"));
  vbnn_ctx* c = m->ctx;
  cudaStream_t st = c->stream;
  VB_CUDA(cudaSetDevice(c->device));
  const int C = m->sizes.back();
  if (!m->pred_ent) {                     // allocated last: set only once all of predict's state is
    VB_TRY(refuse_capture(st, "vbnn_mlp_predict"));
    VB_TRY(ensure_pred_partials(m));
    for (float** q : {&m->pred_max, &m->pred_sum})
      if (*q) { cudaFree(*q); *q = nullptr; }
    VB_TRY(dev_alloc(&m->pred_max, (size_t)m->max_batch * C));
    VB_TRY(dev_alloc(&m->pred_sum, (size_t)m->max_batch * C));
    VB_TRY(dev_alloc(&m->pred_ent, (size_t)m->max_batch));
  }
  const bool reduce = nll_host || acc_host;
  int grid = 0;
  auto consume = [&](int zc, bool first, bool last) -> int {
    PredictParams p;
    memset(&p, 0, sizeof(p));
    p.logits = m->logits; p.ld_logits = m->ld_logits;
    p.N = N; p.C = C; p.zc = zc; p.first = first; p.last = last;
    p.T = n_samples == 0 ? 1 : n_samples;
    p.st_max = m->pred_max; p.st_sum = m->pred_sum; p.st_ent = m->pred_ent;
    if (last) {
      p.logp_out = logp_dev; p.unc_out = unc_dev;
      p.targets = reduce ? targets : nullptr; p.partials = m->pred_partials;
    }
    // profile class 8; its "flops" slot holds the algorithmic bytes: 4 B of logits + 16 B of state read and
    // write per (row, class, sample)
    return prof_launch(c, 8, 20.0 * zc * (double)N * C, [&] { return launch_predict(p, &grid, st); });
  };
  VB_TRY(eval_forward(m, X, nullptr, N, n_samples, "vbnn_mlp_predict", consume));
  if (reduce) {
    VB_CUDA(cudaMemcpyAsync(c->h_partials, m->pred_partials, (size_t)grid * 2 * sizeof(double), cudaMemcpyDeviceToHost,
                            st));
    VB_CUDA(cudaStreamSynchronize(st));
    double nll = 0, corr = 0;
    for (int b = 0; b < grid; ++b) { nll += c->h_partials[2 * b]; corr += c->h_partials[2 * b + 1]; }   // fixed order
    if (nll_host) *nll_host = (float)(nll / N);
    if (acc_host) *acc_host = (float)(corr / N * 100.0);
  }
  return VBNN_OK;
}

extern "C" int vbnn_mlp_predict_outputs(vbnn_mlp* m, const float* X, int N, int n_samples, int output_model,
                                        const float* targets, float* samples_dev, float* mean_dev, float* epi_dev,
                                        float* ale_dev, float* nll_host, float* rmse_host) {
  VB_CHECK(m && X, VBNN_E_INVALID, "vbnn_mlp_predict_outputs: null argument");
  VB_CHECK(N > 0 && N <= m->max_batch && n_samples >= 0, VBNN_E_INVALID,
           "vbnn_mlp_predict_outputs: N=%d (max_batch %d), n_samples=%d", N, m->max_batch, n_samples);
  VB_CHECK(output_model == VBNN_OUTPUT_RAW || output_model == VBNN_OUTPUT_GAUSSIAN, VBNN_E_INVALID,
           "vbnn_mlp_predict_outputs: unknown output model %d", output_model);
  const int C = m->sizes.back();
  const bool gaussian = output_model == VBNN_OUTPUT_GAUSSIAN;
  VB_CHECK(!gaussian || C % 2 == 0, VBNN_E_INVALID,
           "vbnn_mlp_predict_outputs: VBNN_OUTPUT_GAUSSIAN needs an even number of outputs, the net has %d", C);
  VB_CHECK(gaussian || !(ale_dev || nll_host), VBNN_E_INVALID,
           "vbnn_mlp_predict_outputs: aleatoric variance and nll need VBNN_OUTPUT_GAUSSIAN");
  VB_CHECK(targets || !(nll_host || rmse_host), VBNN_E_INVALID, "vbnn_mlp_predict_outputs: nll / rmse need targets");
  VB_CHECK((reinterpret_cast<uintptr_t>(samples_dev) & 15) == 0, VBNN_E_INVALID,
           "vbnn_mlp_predict_outputs: samples_dev must be 16-byte aligned");
  VB_TRY(refuse_open_step(m, "vbnn_mlp_predict_outputs"));
  vbnn_ctx* c = m->ctx;
  cudaStream_t st = c->stream;
  VB_CUDA(cudaSetDevice(c->device));
  if (!m->mom_state) {
    VB_TRY(refuse_capture(st, "vbnn_mlp_predict_outputs"));
    VB_TRY(ensure_pred_partials(m));
    VB_TRY(dev_alloc(&m->mom_state, (size_t)m->max_batch * (3 * (size_t)C + 2)));
  }
  const int K = gaussian ? C / 2 : C;
  const size_t NC = (size_t)N * C;
  const bool reduce = nll_host || rmse_host;
  const bool lse = gaussian && nll_host;
  int grid = 0, done = 0;
  auto consume = [&](int zc, bool first, bool last) -> int {
    MomentsParams p;
    memset(&p, 0, sizeof(p));
    if (samples_dev) { p.out = samples_dev + (size_t)done * NC; p.ld_out = C; }
    else { p.out = m->logits; p.ld_out = m->ld_logits; }
    done += zc;
    p.N = N; p.K = K; p.gaussian = gaussian; p.zc = zc; p.first = first; p.last = last;
    p.T = n_samples == 0 ? 1 : n_samples;
    p.st_f0 = m->mom_state; p.st_sum = p.st_f0 + NC; p.st_sq = p.st_sum + NC;
    p.st_lmax = p.st_sq + NC; p.st_lsum = p.st_lmax + N;
    p.lse = lse;
    p.targets = lse || (last && rmse_host) ? targets : nullptr;
    if (last) {
      p.mean_out = mean_dev; p.epi_out = epi_dev; p.ale_out = ale_dev;
      p.partials = reduce ? m->pred_partials : nullptr;
    }
    // profile class 8; its "flops" slot holds the algorithmic bytes, counted as if every sample read and wrote the
    // state: per (row, sample) 28 B per mean column (4 B output, 12 B state read, 12 B written) and, under GAUSSIAN,
    // 12 B per log-variance column (4 B output, 4 B state read, 4 B written)
    const double bytes = (double)zc * N * (gaussian ? 40.0 * K : 28.0 * C);
    return prof_launch(c, 8, bytes, [&] { return launch_predict_moments(p, &grid, st); });
  };
  const int r = eval_forward(m, X, nullptr, N, n_samples, "vbnn_mlp_predict_outputs", consume, samples_dev);
  m->ext_logits = nullptr;
  if (samples_dev) m->outputs_external = true;      // get_outputs: the outputs are in the caller's buffer
  VB_TRY(r);
  if (reduce) {
    VB_CUDA(cudaMemcpyAsync(c->h_partials, m->pred_partials, (size_t)grid * 2 * sizeof(double), cudaMemcpyDeviceToHost,
                            st));
    VB_CUDA(cudaStreamSynchronize(st));
    double nll = 0, se = 0;
    for (int b = 0; b < grid; ++b) { nll += c->h_partials[2 * b]; se += c->h_partials[2 * b + 1]; }   // fixed order
    if (nll_host) *nll_host = (float)(nll / N);
    if (rmse_host) *rmse_host = (float)sqrt(se / ((double)N * K));
  }
  return VBNN_OK;
}

extern "C" int vbnn_mlp_get_outputs(vbnn_mlp* m, int sample_idx, float* logp_host) {
  VB_CHECK(m && logp_host, VBNN_E_INVALID, "null argument");
  VB_CHECK(m->last_N > 0 && sample_idx >= 0 && sample_idx < m->Z, VBNN_E_STATE, "vbnn_mlp_get_outputs: no forward yet");
  VB_TRY(refuse_open_step(m, "vbnn_mlp_get_outputs"));
  VB_CHECK(!m->outputs_external, VBNN_E_STATE,
           "vbnn_mlp_get_outputs: the last forward was vbnn_mlp_forward_train, whose outputs are in the caller's buffer");
  vbnn_ctx* c = m->ctx;
  const int N = m->last_N, C = m->sizes.back();
  if (!m->logp) VB_TRY(dev_alloc(&m->logp, (size_t)m->max_batch * C));
  LossParams lp;
  memset(&lp, 0, sizeof(lp));
  lp.logits = m->logits + (size_t)sample_idx * N * m->ld_logits; lp.ld_logits = m->ld_logits;
  lp.targets = m->targets; lp.N = N; lp.C = C; lp.Z = 1; lp.grad_scale = 0.f;
  lp.logp_out = m->logp;
  lp.result = reinterpret_cast<float*>(c->d_partials) + 16;
  VB_TRY(launch_loss(lp, c->stream));
  c->launches++;
  VB_CUDA(cudaMemcpyAsync(logp_host, m->logp, (size_t)N * C * 4, cudaMemcpyDeviceToHost, c->stream));
  VB_CUDA(cudaStreamSynchronize(c->stream));
  return VBNN_OK;
}

extern "C" int vbnn_mlp_launch_count(vbnn_mlp* m, long long* count) {
  VB_CHECK(m && count, VBNN_E_INVALID, "null argument");
  *count = m->ctx->launches;
  return VBNN_OK;
}

extern "C" int vbnn_mlp_graph_captures(vbnn_mlp* m, long long* count) {
  VB_CHECK(m && count, VBNN_E_INVALID, "null argument");
  *count = m->graph_captures;
  return VBNN_OK;
}

extern "C" int vbnn_mlp_grad_arena(vbnn_mlp* m, float** ptr, size_t* count) {
  VB_CHECK(m && ptr, VBNN_E_INVALID, "null argument");
  *ptr = m->grad_arena;
  if (count) *count = m->grad_count;
  return VBNN_OK;
}
