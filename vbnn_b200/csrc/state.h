// state.h -- the opaque handle types behind include/vbnn.h.
#pragma once
#include <vector>

#include "common.cuh"
#include "gemm.h"
#include "kernels.h"

struct vbnn_ctx {
  int device = 0;
  cudaStream_t stream = nullptr;
  bool own_stream = false;
  bool capturable = true;            // false on the legacy default stream (CUDA graphs cannot capture stream 0)
  cudaStream_t copy_stream = nullptr;
  uint64_t seed = 0;
  uint32_t* d_step = nullptr;        // Philox "minibatch" counter, lives on the device (graph-safe)
  double* d_partials = nullptr;      // kMaxPartials * kStatSlots doubles of reduction scratch
  double* h_partials = nullptr;      // pinned mirror
  float* h_scalars = nullptr;        // pinned scratch for scalar read-backs
  int next_layer_id = 0;
  long long launches = 0;
  // per-launch device timing of the tensor-core GEMM (bench.py roofline), the fused update (7) and predict (8)
  static constexpr int kProfClasses = 9;
  bool profiling = false;
  struct ProfRec { cudaEvent_t a, b; int cls; double flops; };
  std::vector<ProfRec> prof_recs;
  std::vector<cudaEvent_t> prof_pool;
  double prof_ms[kProfClasses] = {0}; double prof_flops[kProfClasses] = {0}; long long prof_n[kProfClasses] = {0};
  // phase marks of one minibatch (same switch): time from the previous mark to mark `id`
  struct Mark { cudaEvent_t e; int id; };
  std::vector<Mark> marks;
  double phase_ms[16] = {0}; long long phase_n[16] = {0};
  // data parallel
  void* nccl_comm = nullptr;
  int rank = 0, nranks = 1;
  cudaStream_t comm_stream = nullptr;   // per-layer gradient allreduce overlaps the rest of backward
};

struct vbnn_layer {
  vbnn_ctx* ctx = nullptr;
  int I = 0, O = 0, kind = VBNN_KIND_VB, id = 0;
  vbnn_opts opts;
  int ldI = 0, ldO = 0;              // padded leading dims (multiples of 8) of operand buffers
  int S_alloc = 1;                   // weight samples held at once
  bool owned_by_mlp = false;
  bool grads_external = false;       // gW/gS/gb live in the mlp's allreduce arena
  bool ext_weight = false, ext_bias = false, ext_gW = false, ext_gb = false;   // caller-owned (vbnn_layer_bind)
  // fp32 master state, dense [O x I] / [O]
  float *means = nullptr, *lvars = nullptr, *bias = nullptr, *weight = nullptr;
  float *gW = nullptr, *gS = nullptr, *gb = nullptr;
  float *m_mu = nullptr, *v_mu = nullptr, *m_var = nullptr, *v_var = nullptr;
  float *eps = nullptr, *stdv = nullptr, *mu_sqe = nullptr, *s2_f32 = nullptr;
  float* var_hat_dev = nullptr;
  int n_part = 0;                    // partial sums per half (update_grid(O, I); peer mode: G x blocks per shard)
  double* prior_partials = nullptr;  // 2 x kMaxPartials: per-block sums written by the last update (ping-pong:
                                     // an update reads one half while its blocks write the other)
  // half (t & 1) holds the sums of the CURRENT parameters, t = the layer's device step counter
  int* t_dev = nullptr;              // meanState.t == varState.t == biasState.evalCounter
  vbnn::LiveOpts* hp = nullptr;      // B, rates, Adam constants the update kernels read (vbnn_layer_set_opts)
  // bf16 tensor-core operand copies [.. x ldI]
  bf16 *w_bf16 = nullptr, *mu_bf16 = nullptr, *s2_bf16 = nullptr;
  void* eps16 = nullptr;             // fp16 [S_alloc x O x ldI]: this minibatch's epsilon for the dW epilogue (mlp-owned layers)
  bool eps16_valid = false;
  // layer-API scratch (grown on demand)
  int cap_N = 0;
  void *xs = nullptr, *xs2 = nullptr, *gs_ = nullptr, *hs = nullptr, *R = nullptr;
  float* zeta_keep = nullptr;
  int cur_sample = 0;
  bool eps_injected = false;
  bool map_mode = false;
  bool prior_valid = false;
  const bool* shard_stale = nullptr;  // peer mode: fp32 state of the rows other ranks own is out of date
  vbnn_mlp* owner = nullptr;         // the net whose step graphs bake this layer's prior in (mlp-owned layers)
  // prior of the KL terms (vbnn_layer_set_prior): kind, FIXED scalars, PER_WEIGHT arrays [O x I]
  int prior_kind = VBNN_PRIOR_EMPIRICAL;
  float prior_mu0 = 0.f, prior_var0 = 0.f;
  float *prior_means = nullptr, *prior_lvars = nullptr;
};

// ---- peer mode (peer.cu): the data-parallel gradient exchange over NVLink peer memory -------
// Rows [q*rpo, (q+1)*rpo) of every layer's parameters belong to rank q.  The dW GEMM epilogue
// stores each gradient tile straight into its owner's receive slot (reduce-scatter fused into the
// GEMM), the owner sums the G slots inside the fused KL + Adam update of its shard, and the copy
// engines push the refreshed operands back to every rank (all-gather) while backward continues.
constexpr int kMaxPeers = 8;
struct PeerBuf { void* ptr[kMaxPeers] = {nullptr}; };   // ptr[q]: the buffer as mapped from rank q (ptr[me]: local)
struct PeerLayer {
  int rpo = 0, row0 = 0, rows = 0;       // rows per owner (multiple of 32), this rank's shard
  size_t slot_floats = 0;                // floats per source slot {gW [, gS]}: rpo * I (* 2)
  size_t off_recv = 0;                   // byte offset of slot 0 inside the comm block
  size_t off_gb = 0;                     // byte offset of the [G][O] gradBias slots
  PeerBuf means, lvars, s2_f32, mu_bf16, s2_bf16, weight, w_bf16, partials, m_mu, v_mu, m_var, v_var;
  uint32_t *mseq = nullptr, *sseq = nullptr;   // step counters owned by the main / side stream
  cudaEvent_t ev_dw = nullptr;
  float* stage = nullptr;                // copy-engine transport: local gradient tiles laid out like the G receive slots
};
struct vbnn_peer {
  int G = 1, me = 0;
  char* block = nullptr; size_t block_bytes = 0;     // local comm block: flags | gb slots | receive slots
  char* peer_block[kMaxPeers] = {nullptr};
  size_t off_grad_ready = 0, off_param_ready = 0;    // uint32 [L][G] each
  std::vector<PeerLayer> layers;
  uint32_t* seq = nullptr;                           // local counters: {mseq, sseq} x L, then wseq[L]
  int* h_err = nullptr; int* d_err = nullptr;        // pinned + mapped: set when a peer wait times out
  cudaStream_t side = nullptr;
  cudaStream_t xfer = nullptr;                       // copy-engine transport of gradient slabs
  cudaEvent_t ev_xfer = nullptr;
  unsigned int* xfer_done = nullptr;                 // copy-kernel transport: CTAs finished per peer
  cudaEvent_t ev_side = nullptr;
  std::vector<void*> opened;                         // IPC mappings to close
  bool exported = false, active = false, stale = false;
};

struct vbnn_mlp {
  vbnn_ctx* ctx = nullptr;
  vbnn_peer* peer = nullptr;
  std::vector<int> sizes;
  std::vector<vbnn_layer*> layers;   // hidden VB layers..., then the output layer
  int vb_output = 0, max_batch = 0, Z = 1;
  vbnn_opts opts;
  bool bf16 = false, lrt = false;
  std::vector<int> ld;               // padded width of sizes[k]
  // activations, element type float (FP32) or bf16 (BF16); index k = features sizes[k]
  std::vector<void*> act, act2;      // act[0] = staged input [N x ld0]; act[k>0] = [Z x N x ld_k]
  std::vector<void*> R, G, H;        // per layer output k+1: [Z x N x ld_{k+1}]
  float* aux = nullptr; int ld_aux = 0;     // fp32 [Z x N x ld_aux]: first product of the split LRT GEMMs
  float* dw_partials = nullptr;             // fp32 [Z x O x I] of the plain output layer: per-sample dW products (Z > 1)
  float* logits = nullptr; int ld_logits = 0;
  float* logp = nullptr;
  // vbnn_mlp_predict state, allocated by the first call: log-sum-exp max / sum [max_batch x C], entropy sum
  // [max_batch], per-block {nll, correct} partials [kMaxPartials x 2]
  float *pred_max = nullptr, *pred_sum = nullptr, *pred_ent = nullptr;
  double* pred_partials = nullptr;   // shared with vbnn_mlp_predict_outputs
  // vbnn_mlp_predict_outputs state, allocated by its first call: {f0, sum d, sum d^2} [3 x max_batch x C], then the
  // per-row log-sum-exp max / sum [2 x max_batch]
  float* mom_state = nullptr;
  float* targets = nullptr;          // staged targets [N]
  float* xstage[2] = {nullptr, nullptr};   // fp32 H2D staging for the host-buffer API
  float* tstage[2] = {nullptr, nullptr};
  uint8_t* xstage_u8[2] = {nullptr, nullptr};   // uint8 H2D staging (vbnn_mlp_submit_host_u8)
  float* result_acc = nullptr;       // [2*Z] loss sums / correct counts
  float* result = nullptr;           // [2] {error, accuracy}
  float* grad_arena = nullptr; size_t grad_count = 0;
  std::vector<size_t> grad_off, grad_len;       // per-layer slice {gW, gS, gb} of the arena
  std::vector<cudaEvent_t> ev_bwd, ev_red;      // dW of layer j done / its allreduce done
  int** t_list_dev = nullptr; int n_t = 0;
  // CUDA graphs of one step: vbnn_mlp_step's keyed by N, vbnn_mlp_step_grad_input's by (N, dX), the forward half of
  // the split step by (N, logits), its backward half by (N, grad) without and (N, grad, dX) with an input gradient;
  // no call destroys or re-captures another's.  Each graph runs its body eagerly once before it captures.
  struct StepGraph {
    cudaGraphExec_t exec = nullptr; int N = -1; const void* key[2] = {nullptr, nullptr}; int eager_steps = 0;
    long long launches = 0;
  };
  enum { kGraphStep, kGraphStepDx, kGraphFwd, kGraphBwd, kGraphBwdDx, kNumGraphs };
  StepGraph graphs[kNumGraphs];
  long long graph_captures = 0;      // captures made by all of them (vbnn_mlp_graph_captures)
  bool use_graph = true;
  // vbnn_mlp_step_grad_input's / vbnn_mlp_backward_update's output [N x I0] fp32, set only while that call enqueues
  float* dX = nullptr;
  // vbnn_mlp_forward_train's output [Z x N x C] fp32, set only while that call enqueues its forward half
  float* ext_logits = nullptr;
  // split step (vbnn_mlp_forward_train .. vbnn_mlp_backward_update): open, its N, and whether the last forward's
  // outputs went to the caller's buffer instead of `logits` (vbnn_mlp_get_outputs has nothing to return)
  bool step_open = false;
  int open_N = 0;
  bool outputs_external = false;
  // host-buffer pipeline
  struct Slot { cudaEvent_t copied, consumed, done; float* h_result; bool busy; int N; };
  Slot slots[2];
  int submit_idx = 0, collect_idx = 0, inflight = 0;
  bool pipeline_ready = false;
  int last_N = 0;
  bool peer_waited_all = false;      // this step already waited for (and counted) every layer's operands up front
};

namespace vbnn {
// cudaMalloc of count elements (none: nullptr) with the library's error reporting
template <typename T>
int dev_alloc(T** p, size_t count) {
  *p = nullptr;
  if (count == 0) return VBNN_OK;
  cudaError_t e = cudaMalloc((void**)p, count * sizeof(T));
  if (e != cudaSuccess) {
    set_error("cudaMalloc(%zu bytes) failed: %s", count * sizeof(T), cudaGetErrorString(e));
    return e == cudaErrorMemoryAllocation ? VBNN_E_NOMEM : VBNN_E_CUDA;
  }
  return VBNN_OK;
}
// the layer runs the local reparameterisation: its forward reads mu and sigma^2 and draws the noise per output
inline bool layer_is_lrt(const vbnn_layer* L) {
  return L->kind == VBNN_KIND_VB && L->opts.reparam == VBNN_REPARAM_LOCAL;
}
int layer_create_internal(vbnn_ctx* ctx, int I, int O, int kind, const vbnn_opts* opts, int S_alloc,
                          float* gW, float* gS, float* gb, int id, vbnn_layer** out);
int layer_update_internal(vbnn_layer* L, vbnn_stats* stats, bool bump_t);
int layer_refresh_copies(vbnn_layer* L);
int layer_compute_prior_internal(vbnn_layer* L);
int layer_refresh_prior_partials(vbnn_layer* L);
PriorArgs layer_prior(const vbnn_layer* L, size_t row_off);   // row_off: first element of a peer-mode row shard
void mlp_drop_graphs(vbnn_mlp* m);                            // each step graph re-captures at its next use
int mlp_wait_side(vbnn_mlp* m);                               // peer mode: the context's stream waits for the side stream
LiveOpts live_opts(const vbnn_opts& o);                       // the fields of o the update reads at every call
PhiloxStream layer_stream(const vbnn_layer* L, uint32_t kind, int sample);
int comm_allreduce_internal(vbnn_ctx* ctx, float* buf, size_t count, cudaStream_t st);
// peer mode (peer.cu)
void peer_destroy(vbnn_mlp* m);
void peer_scatter(const vbnn_mlp* m, int j, int N, EpiParams& p);         // dW epilogue -> owners' slots (or the local staging copy of them)
bool peer_transport_ce(const vbnn_mlp* m, int N);
bool peer_wire_bf16(const vbnn_mlp* m, int j, int N);                     // layer j's gradient tiles travel as bf16 for this batch size                         // gradient slabs travel by copy engine for this batch size
int peer_wait_params(vbnn_mlp* m, int j, bool bump);                      // main stream, before layer j's forward (-1: all layers)
int peer_after_dw(vbnn_mlp* m, int j);                                    // signal + owner update + push
int peer_check(vbnn_mlp* m);                                              // host: a peer wait timed out?
// The weight operands of the forward (kmajor = 1: B = W^T) and backward-data (kmajor = 0: B = W) GEMMs in the
// layer's precision: B1 = mu for an LRT layer (MAP mode included), else W -- per sample when `batched`; with
// `lrt` (the layer runs the LRT form) also B2 = sigma^2.
void weight_operands(GemmArgs& g, const vbnn_layer* L, int kmajor, bool batched, bool lrt);
// GEMM launch on the bf16 tcgen05 engine or the fp32 CUDA-core engine.  While ctx->profiling, a bf16 launch is
// timed and accounted under prof_cls (default: its mode).
int gemm(vbnn_ctx* ctx, bool bf16, int mode, const GemmArgs& g, const EpiParams& p, int prof_cls = -1);
int prof_collect(vbnn_ctx* ctx);
int prof_mark(vbnn_ctx* ctx, int id);     // id 0 starts a minibatch; no-op unless profiling
// launch() under a pair of CUDA events while ctx->profiling, accounted to class cls with `work` in its flops slot
template <typename Launch>
int prof_launch(vbnn_ctx* c, int cls, double work, Launch&& launch) {
  if (!c->profiling) return launch();
  vbnn_ctx::ProfRec r;
  for (cudaEvent_t* e : {&r.a, &r.b}) {
    if (!c->prof_pool.empty()) { *e = c->prof_pool.back(); c->prof_pool.pop_back(); }
    else VB_CUDA(cudaEventCreate(e));
  }
  r.cls = cls; r.flops = work;
  VB_CUDA(cudaEventRecord(r.a, c->stream));
  const int rc = launch();
  VB_CUDA(cudaEventRecord(r.b, c->stream));
  c->prof_recs.push_back(r);
  if (c->prof_recs.size() + c->marks.size() >= 4096) VB_TRY(prof_collect(c));
  return rc;
}
}  // namespace vbnn
