// peer.cu -- data-parallel gradient exchange fused into the hot path over NVLink peer memory
// (new functionality: the reference is single-GPU, SURVEY.md section 2.2 / 8e).
//
// One process per GPU; every rank maps the others' buffers with CUDA IPC.  Per layer j and step:
//
//   reduce-scatter  fused into the dW GEMM: rows [q*rpo, (q+1)*rpo) of gradWeight / gradSum belong
//                   to rank q, and the tcgen05 epilogue stores each finished tile straight into
//                   rank q's receive slot for this rank (posted stores over NVLink, no staging
//                   buffer, no separate collective kernel)                    -> peer_scatter()
//   owner update    rank q's fused KL + Adam kernel sums the G slots of its shard while it reads
//                   them; the update costs 1/G of the replicated one         -> peer_after_dw()
//   all-gather      the refreshed operands of the shard (bf16 mu / sigma^2, or fp32 mu / log
//                   sigma^2 for weight sampling) are pushed to every rank by the copy engines on a
//                   side stream while the SMs continue with the backward pass of the layers below
//
// Ordering uses per-layer flags in peer memory (release/acquire at system scope): grad_ready[j][r]
// is set on every rank by rank r once its dW tile stores and gradBias of layer j are out;
// param_ready[j][q] is set on every rank by owner q once its pushes of layer j have completed.
// Counters are per stream (wseq: main stream's waits, mseq: the stream that signals gradients -- main or transfer --,
// sseq: side), so nothing races with the host, a graph or another stream.
// Every wait is bounded: a rank that does not show up sets an error word instead of hanging.
#include <cuda.h>
#include <string.h>

#include "knobs.h"
#include "state.h"

namespace vbnn {

namespace {

constexpr uint32_t kBlobMagic = 0x56424E50u;   // "VBNP"
constexpr int kBufsPerLayer = 12;
constexpr unsigned long long kWaitTimeoutNs = 30ull * 1000ull * 1000ull * 1000ull;

struct BlobHeader { uint32_t magic, rank, nranks, n_entries; };
struct BlobEntry { cudaIpcMemHandle_t handle; uint64_t offset, bytes; };

inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// ------------------------------------------------------------------ device side -----------
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_sys(uint32_t* p, uint32_t v) {
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned long long globaltimer_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
__device__ __forceinline__ void spin_until(const uint32_t* flag, uint32_t need, int* err) {
  if (ld_acquire_sys(flag) >= need) return;
  const unsigned long long t0 = globaltimer_ns();
  while (ld_acquire_sys(flag) < need) {
    __nanosleep(200);
    if (globaltimer_ns() - t0 > kWaitTimeoutNs) { *err = 1; return; }
  }
}

// main stream, before layer j's operands are first read in a step: every owner's operands of the previous step have
// landed in this rank's buffers.  ready: [L][G]; wseq: [L] steps this stream has started per layer -- a counter of its
// OWN (the gradient signal that advances mseq may run on the transfer stream, whose progress the main stream must not
// race with); bump: training steps advance it, evaluation only looks.
__global__ void k_wait_params(const uint32_t* ready, uint32_t* wseq, int L, int G, int* err, int bump) {
  for (int t = threadIdx.x; t < L * G; t += blockDim.x) spin_until(ready + t, wseq[t / G], err);
  __syncthreads();
  if (bump)
    for (int j = threadIdx.x; j < L; j += blockDim.x) wseq[j] += 1u;
}

struct SignalGrad {
  const float* gb; int O;          // this rank's gradBias of the layer
  float* gb_dst[kMaxPeers];        // rank q's gradBias slot for this rank
  uint32_t* ready_dst[kMaxPeers];  // rank q's grad_ready[j][me]
  uint32_t* mseq;
  int G;
};
// main stream, after the dW GEMM + gradBias column sums of layer j
__global__ void k_signal_grad(SignalGrad s) {
  const uint32_t v = *s.mseq + 1u;
  for (int q = 0; q < s.G; ++q)
    for (int i = threadIdx.x; i < s.O; i += blockDim.x) s.gb_dst[q][i] = s.gb[i];
  __threadfence_system();
  __syncthreads();
  if (threadIdx.x < s.G) st_release_sys(s.ready_dst[threadIdx.x], v);
  if (threadIdx.x == 0) *s.mseq = v;
}

// Copy-kernel transport (strong-scaling regime): the dW GEMM left this rank's gradient tiles in a local staging copy
// of the slot layout; this kernel -- a few small CTAs that fit beside the persistent GEMM CTAs of the next layers --
// streams slab q to owner q over NVLink with 16-byte loads / stores (every peer link busy at once: blockIdx.x picks
// the peer), and the last CTA of each peer also delivers gradBias and raises grad_ready there: transfer and signal in
// ONE launch (the copy-engine form needs 2 G API calls per layer and runs the slabs one after another).
struct PushSlabs {
  const float* stage;              // [G][slot_floats]
  float* dst[kMaxPeers];           // rank q's receive slot for this rank
  size_t slot_floats;              // distance between slots (floats)
  size_t slot_bytes;               // bytes of a slot that carry data (half of it with bf16 tiles)
  const float* gb; int O;
  float* gb_dst[kMaxPeers];
  uint32_t* ready_dst[kMaxPeers];
  uint32_t* mseq;
  unsigned int* done;              // [G] CTAs finished per peer (reset by the last one)
  int G, me;
};
__global__ void __launch_bounds__(128, 8) k_push_slabs(PushSlabs s) {
  const int q = (s.me + 1 + (int)blockIdx.x) % s.G;                 // staggered start: no two ranks hit the same peer first
  const uint4* src = reinterpret_cast<const uint4*>(s.stage + (size_t)q * s.slot_floats);
  uint4* dst = reinterpret_cast<uint4*>(s.dst[q]);
  const size_t n16 = s.slot_bytes / 16;                             // a multiple of 16 bytes (rpo % 32 == 0)
  const size_t stride = (size_t)gridDim.y * blockDim.x;
  size_t i = (size_t)blockIdx.y * blockDim.x + threadIdx.x;
  for (; i + 3 * stride < n16; i += 4 * stride) {                   // 4 x 16 B in flight per thread
    const uint4 a = __ldcs(src + i), b = __ldcs(src + i + stride), c = __ldcs(src + i + 2 * stride), d = __ldcs(src + i + 3 * stride);
    dst[i] = a; dst[i + stride] = b; dst[i + 2 * stride] = c; dst[i + 3 * stride] = d;
  }
  for (; i < n16; i += stride) dst[i] = __ldcs(src + i);
  __threadfence_system();
  __syncthreads();
  __shared__ bool last;
  if (threadIdx.x == 0) last = atomicAdd(s.done + q, 1u) + 1u == gridDim.y;
  __syncthreads();
  if (!last) return;
  for (int k = threadIdx.x; k < s.O; k += blockDim.x) s.gb_dst[q][k] = s.gb[k];
  __threadfence_system();
  __syncthreads();
  if (threadIdx.x == 0) {
    s.done[q] = 0;
    const uint32_t v = *s.mseq + 1u;
    st_release_sys(s.ready_dst[q], v);
    // the counter advances once every peer has been signalled
    if (atomicAdd(s.done + s.G, 1u) + 1u == (unsigned)s.G) { s.done[s.G] = 0; *s.mseq = v; }
  }
}

// side stream: every rank's gradient tiles of layer j have landed in this rank's receive slots
__global__ void k_wait_grad(const uint32_t* ready /*[G]*/, const uint32_t* sseq, int G, int* err) {
  if (threadIdx.x < G) spin_until(ready + threadIdx.x, *sseq + 1u, err);
}

struct SignalParam {
  uint32_t* ready_dst[kMaxPeers];  // rank q's param_ready[j][me]
  uint32_t* sseq;
  int* t_dev;                      // the layer's optimiser step counter
  int G;
};
// side stream, after the shard update and its copy-engine pushes
__global__ void k_signal_param(SignalParam s) {
  const uint32_t v = *s.sseq + 1u;
  __threadfence_system();
  __syncthreads();
  if (threadIdx.x < s.G) st_release_sys(s.ready_dst[threadIdx.x], v);
  if (threadIdx.x == 0) { *s.sseq = v; if (s.t_dev) *s.t_dev += 1; }
}

// ------------------------------------------------------------------ host helpers ----------
typedef CUresult (*PFN_getRange)(CUdeviceptr*, size_t*, CUdeviceptr);
PFN_getRange get_range_fn() {
  static PFN_getRange fn = nullptr;
  static bool tried = false;
  if (tried) return fn;
  tried = true;
  void* p = nullptr;
  cudaDriverEntryPointQueryResult qr;
  if (cudaGetDriverEntryPoint("cuMemGetAddressRange", &p, cudaEnableDefault, &qr) == cudaSuccess &&
      qr == cudaDriverEntryPointSuccess)
    fn = reinterpret_cast<PFN_getRange>(p);
  return fn;
}

int make_entry(const void* ptr, size_t bytes, BlobEntry* e) {
  memset(e, 0, sizeof(*e));
  if (!ptr || !bytes) return VBNN_OK;
  char* base = (char*)ptr;
  if (PFN_getRange fn = get_range_fn()) {
    CUdeviceptr b = 0; size_t sz = 0;
    if (fn(&b, &sz, (CUdeviceptr)ptr) == CUDA_SUCCESS && b) base = (char*)b;
  }
  VB_CUDA(cudaIpcGetMemHandle(&e->handle, base));
  e->offset = (uint64_t)((const char*)ptr - base);
  e->bytes = bytes;
  return VBNN_OK;
}

PeerBuf* layer_bufs(PeerLayer& pl, int k) {
  PeerBuf* t[kBufsPerLayer] = {&pl.means, &pl.lvars, &pl.s2_f32, &pl.mu_bf16, &pl.s2_bf16, &pl.weight,
                               &pl.w_bf16, &pl.partials, &pl.m_mu, &pl.v_mu, &pl.m_var, &pl.v_var};
  return t[k];
}
void local_bufs(const vbnn_layer* L, const void* (&ptr)[kBufsPerLayer], size_t (&bytes)[kBufsPerLayer]) {
  const size_t W = (size_t)L->O * L->I, Wb = (size_t)L->O * L->ldI;
  const bool vb = L->kind == VBNN_KIND_VB;
  const void* p[kBufsPerLayer] = {L->means, L->lvars, L->s2_f32, L->mu_bf16, L->s2_bf16,
                                  vb ? nullptr : L->weight, vb ? nullptr : L->w_bf16, L->prior_partials,
                                  L->m_mu, L->v_mu, L->m_var, L->v_var};
  const size_t b[kBufsPerLayer] = {W * 4, W * 4, W * 4, Wb * 2, Wb * 2, W * 4, Wb * 2,
                                   (size_t)2 * kMaxPartials * sizeof(double), W * 4, W * 4, W * 4, W * 4};
  for (int k = 0; k < kBufsPerLayer; ++k) { ptr[k] = p[k]; bytes[k] = p[k] ? b[k] : 0; }
}

inline uint32_t* flag_ptr(const vbnn_peer* P, int q, size_t off, int j, int r) {
  return reinterpret_cast<uint32_t*>(P->peer_block[q] + off) + (size_t)j * P->G + r;
}

// device-to-device copy of this rank's shard of one buffer to every other rank (copy engines)
int push_shard(vbnn_peer* P, const PeerBuf& b, size_t off_bytes, size_t bytes) {
  if (!b.ptr[P->me] || !bytes) return VBNN_OK;
  for (int q = 0; q < P->G; ++q) {
    if (q == P->me) continue;
    VB_CUDA(cudaMemcpyAsync((char*)b.ptr[q] + off_bytes, (const char*)b.ptr[P->me] + off_bytes, bytes,
                            cudaMemcpyDefault, P->side));
  }
  return VBNN_OK;
}
// the reverse: fetch every other owner's shard of a buffer that is not pushed during training
int pull_shards(vbnn_peer* P, const PeerBuf& b, int O, size_t row_bytes, int rpo, cudaStream_t st) {
  if (!b.ptr[P->me]) return VBNN_OK;
  for (int q = 0; q < P->G; ++q) {
    if (q == P->me) continue;
    int r0, rows;
    vbnn_peer_shard(O, P->G, q, &r0, &rows);
    (void)rpo;
    if (rows <= 0) continue;
    VB_CUDA(cudaMemcpyAsync((char*)b.ptr[P->me] + (size_t)r0 * row_bytes, (const char*)b.ptr[q] + (size_t)r0 * row_bytes,
                            (size_t)rows * row_bytes, cudaMemcpyDefault, st));
  }
  return VBNN_OK;
}

}  // namespace

// ------------------------------------------------------------------ used by mlp.cu --------
// Which way the gradient tiles travel.  Fused: the dW epilogue stores every tile straight into its owner's receive
// slot -- no staging, no extra kernel, the transfer rides on the GEMM; right while the GEMM is compute-bound (per-rank
// batch large: the stores need a fraction of NVLink).  With a small per-rank batch (strong scaling) the same bytes
// must leave within a few microseconds per tile, the epilogue warps stall on posted remote stores and the tensor pipe
// waits for its TMEM buffers (measured, C3 at 8 x 1024 rows: dW 196 TFLOP/s, 345 GB/s out of 900): there the tiles
// are written to a LOCAL staging copy of the slot layout at full GEMM speed and a small co-resident copy kernel (or,
// knob 2, the copy engines) moves one contiguous slab per owner over NVLink while the GEMMs go on.
bool peer_transport_ce(const vbnn_mlp* m, int N) {
  const int t = knobs().peer_transport;
  if (t == 1) return false;
  if (!m->peer || m->peer->layers.empty() || !m->peer->layers[0].stage) return false;   // set up without a staging copy
  if (t == 2 || t == 3) return true;
  // Per layer and rank the dW GEMMs take t_dw ~ 4 * rows * O * I / 1.3e15 s while 8 * O * I * (G - 1) / G bytes must leave over
  // NVLink (t_link at ~700 GB/s): the fused stores hide while t_link < t_dw / 2, i.e. rows > 7428 * (G - 1) / G
  // (measured: G = 2, 4096 rows: fused 3.62 ms vs staged 3.84; G = 8, 1024 rows: fused 2.74 ms vs staged 2.17)
  const int G = m->peer ? m->peer->G : 1;
  return (long long)N * m->Z < 7428LL * (G - 1) / G;
}

bool peer_wire_bf16(const vbnn_mlp* m, int j, int N) {
  const vbnn_layer* L = m->layers[j];
  return knobs().peer_wire_bf16 != 0 && peer_transport_ce(m, N) && m->bf16 && m->Z == 1 && layer_is_lrt(L) && (L->I & 7) == 0;
}

void peer_scatter(const vbnn_mlp* m, int j, int N, EpiParams& p) {
  const vbnn_peer* P = m->peer;
  const PeerLayer& pl = P->layers[j];
  const vbnn_layer* L = m->layers[j];
  const bool ce = peer_transport_ce(m, N);
  const bool wire16 = peer_wire_bf16(m, j, N);
  p.scatter_rows = pl.rpo;
  for (int q = 0; q < 8; ++q) { p.gW_peer[q] = nullptr; p.gS_peer[q] = nullptr; }
  for (int q = 0; q < P->G; ++q) {
    float* slot = ce ? pl.stage + (size_t)q * pl.slot_floats
                     : reinterpret_cast<float*>(P->peer_block[q] + pl.off_recv) + (size_t)P->me * pl.slot_floats;
    // pre-biased: the epilogue indexes with the GLOBAL row
    if (wire16) {                                        // bf16 tiles in the first half of the slot's bytes
      bf16* s16 = reinterpret_cast<bf16*>(slot) - (long long)q * pl.rpo * L->I;
      p.gW_peer[q] = reinterpret_cast<float*>(s16);
      p.gS_peer[q] = reinterpret_cast<float*>(s16 + (size_t)pl.rpo * L->I);
    } else {
      p.gW_peer[q] = slot - (long long)q * pl.rpo * L->I;
      p.gS_peer[q] = L->kind == VBNN_KIND_VB ? p.gW_peer[q] + (size_t)pl.rpo * L->I : nullptr;
    }
  }
  p.grads_bf16 = wire16 ? 1 : 0;
}

int peer_wait_params(vbnn_mlp* m, int j, bool bump) {
  vbnn_peer* P = m->peer;
  const int Lc = (int)m->layers.size();
  const uint32_t* ready = reinterpret_cast<const uint32_t*>(P->block + P->off_param_ready);
  uint32_t* wseq = P->seq + 2 * Lc;
  if (j < 0) k_wait_params<<<1, 256, 0, m->ctx->stream>>>(ready, wseq, Lc, P->G, P->d_err, bump ? 1 : 0);
  else k_wait_params<<<1, 32, 0, m->ctx->stream>>>(ready + (size_t)j * P->G, wseq + j, 1, P->G, P->d_err, bump ? 1 : 0);
  VB_CUDA(cudaGetLastError());
  m->ctx->launches++;
  return VBNN_OK;
}

int peer_after_dw(vbnn_mlp* m, int j) {
  vbnn_peer* P = m->peer;
  vbnn_ctx* c = m->ctx;
  vbnn_layer* L = m->layers[j];
  PeerLayer& pl = P->layers[j];
  const int G = P->G, me = P->me;
  // ---- main stream: gradBias to every rank, then "my gradients of layer j are out" ----
  SignalGrad sg;
  memset(&sg, 0, sizeof(sg));
  sg.gb = L->gb; sg.O = L->O; sg.mseq = pl.mseq; sg.G = G;
  for (int q = 0; q < G; ++q) {
    sg.gb_dst[q] = reinterpret_cast<float*>(P->peer_block[q] + pl.off_gb) + (size_t)me * L->O;
    sg.ready_dst[q] = flag_ptr(P, q, P->off_grad_ready, j, me);
  }
  cudaStream_t sd = P->side;
  const bool wire16 = peer_wire_bf16(m, j, m->last_N);
  const size_t slot_bytes = pl.slot_floats * (wire16 ? 2 : 4);       // bytes of a slot that carry data
  if (peer_transport_ce(m, m->last_N)) {
    // copy-engine transport: one contiguous slab {gW rows, gS rows} per owner from the local staging copy, on
    // its own stream so that the slabs of successive layers queue back to back on NVLink; the flag follows them
    cudaStream_t xf = knobs().peer_one_stream ? sd : P->xfer;
    VB_CUDA(cudaEventRecord(pl.ev_dw, c->stream));
    VB_CUDA(cudaStreamWaitEvent(xf, pl.ev_dw, 0));
    if (knobs().peer_transport == 2) {
      // copy engines: 2 G API calls, slabs one after another
      for (int k = 1; k <= G; ++k) {
        const int q = (me + k) % G;                                // staggered: own shard last
        float* dst = reinterpret_cast<float*>(P->peer_block[q] + pl.off_recv) + (size_t)me * pl.slot_floats;
        VB_CUDA(cudaMemcpyAsync(dst, pl.stage + (size_t)q * pl.slot_floats, slot_bytes, cudaMemcpyDefault, xf));
      }
      k_signal_grad<<<1, 256, 0, xf>>>(sg);
    } else {
      PushSlabs ps;
      memset(&ps, 0, sizeof(ps));
      ps.stage = pl.stage; ps.slot_floats = pl.slot_floats; ps.slot_bytes = slot_bytes; ps.gb = L->gb; ps.O = L->O; ps.mseq = pl.mseq;
      ps.done = P->xfer_done; ps.G = G; ps.me = me;
      for (int q = 0; q < G; ++q) {
        ps.dst[q] = reinterpret_cast<float*>(P->peer_block[q] + pl.off_recv) + (size_t)me * pl.slot_floats;
        ps.gb_dst[q] = sg.gb_dst[q]; ps.ready_dst[q] = sg.ready_dst[q];
      }
      // ~144 small CTAs: one per SM beside the GEMM CTAs; the slab of a small layer needs fewer
      int per_peer = (int)((slot_bytes / 16 + 4 * 128 - 1) / (4 * 128));
      int cap = kNumSMs / G > 0 ? kNumSMs / G : 1;
      if (knobs().peer_push_ctas > 0) cap = knobs().peer_push_ctas;
      if (per_peer > cap) per_peer = cap;
      if (per_peer < 1) per_peer = 1;
      k_push_slabs<<<dim3(G, per_peer), 128, 0, xf>>>(ps);
    }
    VB_CUDA(cudaGetLastError());
    if (xf != sd) {
      VB_CUDA(cudaEventRecord(P->ev_xfer, xf));
      VB_CUDA(cudaStreamWaitEvent(sd, P->ev_xfer, 0));
    }
  } else {
    k_signal_grad<<<1, 256, 0, c->stream>>>(sg);
    VB_CUDA(cudaGetLastError());
    VB_CUDA(cudaEventRecord(pl.ev_dw, c->stream));
    VB_CUDA(cudaStreamWaitEvent(sd, pl.ev_dw, 0));
  }
  // ---- side stream: wait for every rank, update this rank's rows, push, signal ----
  k_wait_grad<<<1, 32, 0, sd>>>(flag_ptr(P, me, P->off_grad_ready, j, 0), pl.sseq, G, P->d_err);
  VB_CUDA(cudaGetLastError());
  const float* gb_slots = reinterpret_cast<const float*>(P->block + pl.off_gb);
  float* slot0 = reinterpret_cast<float*>(P->block + pl.off_recv);
  const size_t roff = (size_t)pl.row0 * L->I, roffb = (size_t)pl.row0 * L->ldI;
  // bias (and the plain nn.Linear output layer): optim.sgd, VBLinear.lua:125-128 / mlp.lua:120-123;
  // the bias is O floats: every rank applies the summed gradient itself
  VB_TRY(launch_sgd_slots(L->bias, gb_slots, G, L->O, L->O, &L->hp->lr_bias, nullptr, 1, 1, sd));
  c->launches += 3;
  if (L->kind == VBNN_KIND_LINEAR) {
    if (pl.rows > 0) {
      VB_TRY(launch_sgd_slots(L->weight + roff, slot0, G, (long long)pl.slot_floats, (long long)pl.rows * L->I,
                              &L->hp->lr_bias, L->w_bf16 ? L->w_bf16 + roffb : nullptr, L->I, L->ldI, sd));
      c->launches++;
      if (L->w_bf16) VB_TRY(push_shard(P, pl.w_bf16, roffb * 2, (size_t)pl.rows * L->ldI * 2));
      else VB_TRY(push_shard(P, pl.weight, roff * 4, (size_t)pl.rows * L->I * 4));
    }
  } else {
    UpdateParams u;
    memset(&u, 0, sizeof(u));
    u.mu = L->means + roff; u.lvar = L->lvars + roff;
    u.gW = slot0; u.gS = slot0 + (size_t)pl.rpo * L->I;
    u.n_src = G; u.src_stride = (long long)pl.slot_floats;
    if (wire16) {                                        // bf16 tiles: gS follows gW inside the first half of each slot
      u.grads_bf16 = 1;
      u.gS = reinterpret_cast<const float*>(reinterpret_cast<const bf16*>(slot0) + (size_t)pl.rpo * L->I);
      u.src_stride = (long long)pl.slot_floats * 2;
    }
    u.m_mu = L->m_mu + roff; u.v_mu = L->v_mu + roff; u.m_var = L->m_var + roff; u.v_var = L->v_var + roff;
    u.mu_bf16 = L->mu_bf16 ? L->mu_bf16 + roffb : nullptr;
    u.s2_bf16 = L->s2_bf16 ? L->s2_bf16 + roffb : nullptr;
    u.ld_bf16 = L->ldI;
    u.s2_f32 = L->s2_f32 ? L->s2_f32 + roff : nullptr;
    u.O = pl.rows; u.I = L->I; u.W_total = (long long)L->O * L->I;
    const int gq = L->n_part / G;
    u.partials = L->prior_partials; u.n_partials = L->n_part;
    u.next_partials = L->prior_partials; u.partials_pingpong = 1;
    u.grid_override = gq; u.part_off = me * gq;
    // The shard updates run while the persistent GEMM CTAs of the main stream (the dW GEMMs of the layers above,
    // then the next minibatch's forward) own every SM: use the 128-thread / 80-register variant that fits beside
    // them (a full-width kernel would only start at the next kernel boundary and stall the whole chain).
    u.coresident = 1;
    for (int q = 0; q < G; ++q)
      if (q != me) u.peer_partials[u.n_peer++] = (double*)pl.partials.ptr[q];
    u.var_hat_dev = L->var_hat_dev; u.t_dev = L->t_dev;
    u.S = (float)L->opts.S;
    u.hp = L->hp;
    u.lrt = layer_is_lrt(L);
    u.prior = layer_prior(L, roff);
    // knob peer_fused_push: the update kernel stores the refreshed operands to every rank itself instead of
    // 2 x (G-1) copy-engine copies.  It paid when layer 0's update was the tail of the minibatch (idle SMs); with
    // the dW GEMMs issued in forward order every update runs under GEMMs, where SM-free copy engines win.
    const int fp_knob = knobs().peer_fused_push;         // 1: always, -1: never, 0: with the copy-kernel transport
    const bool fused_push = (fp_knob > 0 || (fp_knob == 0 && peer_transport_ce(m, m->last_N) && knobs().peer_transport != 2)) &&
                            pl.rows > 0;
    if (fused_push) {
      for (int q = 0; q < G; ++q) {
        if (q == me) continue;
        const int i = u.n_push++;
        if (!layer_is_lrt(L)) {
          u.push_mu[i] = (float*)pl.means.ptr[q] + roff; u.push_lv[i] = (float*)pl.lvars.ptr[q] + roff;
        } else if (L->mu_bf16) {
          u.push_mu16[i] = (bf16*)pl.mu_bf16.ptr[q] + roffb; u.push_s216[i] = (bf16*)pl.s2_bf16.ptr[q] + roffb;
        } else {
          u.push_mu[i] = (float*)pl.means.ptr[q] + roff; u.push_s2[i] = (float*)pl.s2_f32.ptr[q] + roff;
        }
      }
    }
    VB_TRY(launch_update(u, nullptr, sd));                                   // VBLinear.lua:130-143 on rows [row0, row0+rows)
    c->launches++;
    L->prior_valid = true;
    if (pl.rows > 0 && !fused_push) {
      if (!layer_is_lrt(L)) {                    // weight sampling reads mu / log sigma^2 (VBLinear.lua:59)
        VB_TRY(push_shard(P, pl.means, roff * 4, (size_t)pl.rows * L->I * 4));
        VB_TRY(push_shard(P, pl.lvars, roff * 4, (size_t)pl.rows * L->I * 4));
      } else if (L->mu_bf16) {                   // tensor-core operands of the LRT GEMMs
        VB_TRY(push_shard(P, pl.mu_bf16, roffb * 2, (size_t)pl.rows * L->ldI * 2));
        VB_TRY(push_shard(P, pl.s2_bf16, roffb * 2, (size_t)pl.rows * L->ldI * 2));
      } else {                                   // fp32 LRT GEMM operands
        VB_TRY(push_shard(P, pl.means, roff * 4, (size_t)pl.rows * L->I * 4));
        VB_TRY(push_shard(P, pl.s2_f32, roff * 4, (size_t)pl.rows * L->I * 4));
      }
    }
  }
  SignalParam sp;
  memset(&sp, 0, sizeof(sp));
  for (int q = 0; q < G; ++q) sp.ready_dst[q] = flag_ptr(P, q, P->off_param_ready, j, me);
  sp.sseq = pl.sseq; sp.t_dev = L->t_dev; sp.G = G;
  k_signal_param<<<1, 32, 0, sd>>>(sp);
  VB_CUDA(cudaGetLastError());
  c->launches++;
  P->stale = true;
  return VBNN_OK;
}

int peer_check(vbnn_mlp* m) {
  if (m->peer && m->peer->h_err && *m->peer->h_err) {
    set_error("peer mode: a rank did not signal within %llu s (wait timed out); results are invalid",
              kWaitTimeoutNs / 1000000000ull);
    return VBNN_E_STATE;
  }
  return VBNN_OK;
}

void peer_destroy(vbnn_mlp* m) {
  vbnn_peer* P = m->peer;
  if (!P) return;
  if (P->xfer) { cudaStreamSynchronize(P->xfer); cudaStreamDestroy(P->xfer); }
  if (P->side) { cudaStreamSynchronize(P->side); cudaStreamDestroy(P->side); }
  if (P->ev_xfer) cudaEventDestroy(P->ev_xfer);
  if (P->xfer_done) cudaFree(P->xfer_done);
  for (PeerLayer& pl : P->layers) if (pl.stage) cudaFree(pl.stage);
  for (void* p : P->opened) cudaIpcCloseMemHandle(p);
  for (PeerLayer& pl : P->layers) if (pl.ev_dw) cudaEventDestroy(pl.ev_dw);
  if (P->ev_side) cudaEventDestroy(P->ev_side);
  if (P->block) cudaFree(P->block);
  if (P->h_err) cudaFreeHost(P->h_err);
  for (vbnn_layer* L : m->layers) L->shard_stale = nullptr;
  delete P;
  m->peer = nullptr;
}

}  // namespace vbnn

using namespace vbnn;

// rows [row0, row0 + rows) of an O-row parameter matrix belong to `rank` of `nranks`; the shard
// height is a multiple of 32 so that a 32-row epilogue chunk never straddles two owners
extern "C" int vbnn_peer_shard(int O, int nranks, int rank, int* row0, int* rows) {
  VB_CHECK(O > 0 && nranks >= 1 && rank >= 0 && rank < nranks, VBNN_E_INVALID, "vbnn_peer_shard: bad argument");
  const int rpo = round_up(ceil_div(O, nranks), 32);
  int r0 = rank * rpo;
  if (r0 > O) r0 = O;
  int r1 = r0 + rpo;
  if (r1 > O) r1 = O;
  if (row0) *row0 = r0;
  if (rows) *rows = r1 - r0;
  return rpo;
}

extern "C" int vbnn_mlp_peer_export(vbnn_mlp* m, void* blob, size_t capacity, size_t* blob_len) {
  VB_CHECK(m && blob_len, VBNN_E_INVALID, "vbnn_mlp_peer_export: null argument");
  vbnn_ctx* c = m->ctx;
  const int G = c->nranks, Lc = (int)m->layers.size();
  const size_t need = sizeof(BlobHeader) + (size_t)(1 + Lc * kBufsPerLayer) * sizeof(BlobEntry);
  *blob_len = need;
  if (!blob) return VBNN_OK;                                    // size query
  VB_CHECK(capacity >= need, VBNN_E_INVALID, "vbnn_mlp_peer_export: blob needs %zu bytes", need);
  VB_CHECK(G > 1 && G <= kMaxPeers, VBNN_E_UNSUPPORTED, "peer mode needs 2..%d ranks (vbnn_comm_init first)", kMaxPeers);
  VB_CHECK(!m->opts.strict_reference, VBNN_E_UNSUPPORTED,
           "peer mode does not shard the stdv / mu_sqe caches of strict_reference");
  VB_CHECK(m->peer == nullptr, VBNN_E_STATE, "peer mode already set up");
  VB_CUDA(cudaSetDevice(c->device));
  vbnn_peer* P = new vbnn_peer();
  m->peer = P;
  P->G = G; P->me = c->rank;
  P->layers.resize(Lc);
  // ---- comm block layout (identical on every rank) ----
  size_t off = 0;
  P->off_grad_ready = off; off = align_up(off + (size_t)Lc * G * 4, 256);
  P->off_param_ready = off; off = align_up(off + (size_t)Lc * G * 4, 256);
  const size_t off_seq = off; off = align_up(off + (size_t)3 * Lc * 4, 256);   // mseq, sseq per layer, then wseq[L]
  for (int j = 0; j < Lc; ++j) {
    vbnn_layer* L = m->layers[j];
    PeerLayer& pl = P->layers[j];
    pl.rpo = vbnn_peer_shard(L->O, G, P->me, &pl.row0, &pl.rows);
    pl.slot_floats = (size_t)pl.rpo * L->I * (L->kind == VBNN_KIND_VB ? 2 : 1);
    pl.off_gb = off; off = align_up(off + (size_t)G * L->O * 4, 256);
    pl.off_recv = off; off = align_up(off + (size_t)G * pl.slot_floats * 4, 256);
  }
  P->block_bytes = off;
  cudaError_t e = cudaMalloc((void**)&P->block, off);
  if (e != cudaSuccess) {
    set_error("peer mode: cudaMalloc(%zu bytes) failed: %s", off, cudaGetErrorString(e));
    peer_destroy(m);
    return VBNN_E_NOMEM;
  }
  VB_CUDA(cudaMemsetAsync(P->block, 0, off, c->stream));
  VB_CUDA(cudaStreamSynchronize(c->stream));
  P->seq = reinterpret_cast<uint32_t*>(P->block + off_seq);
  for (int j = 0; j < Lc; ++j) { P->layers[j].mseq = P->seq + 2 * j; P->layers[j].sseq = P->seq + 2 * j + 1; }
  VB_CUDA(cudaHostAlloc((void**)&P->h_err, sizeof(int), cudaHostAllocMapped));
  *P->h_err = 0;
  VB_CUDA(cudaHostGetDevicePointer((void**)&P->d_err, P->h_err, 0));
  // ---- the blob: IPC handle + offset of every buffer another rank touches ----
  BlobHeader* h = reinterpret_cast<BlobHeader*>(blob);
  h->magic = kBlobMagic; h->rank = (uint32_t)P->me; h->nranks = (uint32_t)G; h->n_entries = (uint32_t)(1 + Lc * kBufsPerLayer);
  BlobEntry* en = reinterpret_cast<BlobEntry*>(h + 1);
  VB_TRY(make_entry(P->block, P->block_bytes, &en[0]));
  for (int j = 0; j < Lc; ++j) {
    const void* ptr[kBufsPerLayer]; size_t bytes[kBufsPerLayer];
    local_bufs(m->layers[j], ptr, bytes);
    for (int k = 0; k < kBufsPerLayer; ++k) VB_TRY(make_entry(ptr[k], bytes[k], &en[1 + j * kBufsPerLayer + k]));
  }
  P->exported = true;
  return VBNN_OK;
}

extern "C" int vbnn_mlp_peer_import(vbnn_mlp* m, const void* blobs, size_t blob_len) {
  VB_CHECK(m && blobs, VBNN_E_INVALID, "vbnn_mlp_peer_import: null argument");
  VB_CHECK(!m->step_open, VBNN_E_STATE, "vbnn_mlp_peer_import: a vbnn_mlp_forward_train step is open");
  vbnn_peer* P = m->peer;
  VB_CHECK(P && P->exported && !P->active, VBNN_E_STATE, "vbnn_mlp_peer_import: call vbnn_mlp_peer_export first");
  vbnn_ctx* c = m->ctx;
  const int G = P->G, Lc = (int)m->layers.size();
  VB_CUDA(cudaSetDevice(c->device));
  struct Opened { cudaIpcMemHandle_t h; char* base; };
  for (int q = 0; q < G; ++q) {
    const BlobHeader* h = reinterpret_cast<const BlobHeader*>((const char*)blobs + (size_t)q * blob_len);
    VB_CHECK(h->magic == kBlobMagic && (int)h->rank == q && (int)h->nranks == G &&
                 (int)h->n_entries == 1 + Lc * kBufsPerLayer,
             VBNN_E_INVALID, "vbnn_mlp_peer_import: blob %d is not rank %d's export of the same network", q, q);
    const BlobEntry* en = reinterpret_cast<const BlobEntry*>(h + 1);
    std::vector<Opened> cache;
    auto map = [&](const BlobEntry& e, void** out) -> int {
      *out = nullptr;
      if (!e.bytes) return VBNN_OK;
      for (const Opened& o : cache)
        if (memcmp(&o.h, &e.handle, sizeof(e.handle)) == 0) { *out = o.base + e.offset; return VBNN_OK; }
      void* base = nullptr;
      cudaError_t err = cudaIpcOpenMemHandle(&base, e.handle, cudaIpcMemLazyEnablePeerAccess);
      if (err != cudaSuccess) {
        set_error("cudaIpcOpenMemHandle (rank %d's buffer) failed: %s", q, cudaGetErrorString(err));
        return VBNN_E_CUDA;
      }
      cache.push_back({e.handle, (char*)base});
      P->opened.push_back(base);
      *out = (char*)base + e.offset;
      return VBNN_OK;
    };
    if (q == P->me) {
      P->peer_block[q] = P->block;
      for (int j = 0; j < Lc; ++j) {
        const void* ptr[kBufsPerLayer]; size_t bytes[kBufsPerLayer];
        local_bufs(m->layers[j], ptr, bytes);
        for (int k = 0; k < kBufsPerLayer; ++k) layer_bufs(P->layers[j], k)->ptr[q] = const_cast<void*>(ptr[k]);
      }
      continue;
    }
    void* p = nullptr;
    VB_TRY(map(en[0], &p));
    P->peer_block[q] = (char*)p;
    for (int j = 0; j < Lc; ++j)
      for (int k = 0; k < kBufsPerLayer; ++k) {
        VB_TRY(map(en[1 + j * kBufsPerLayer + k], &p));
        layer_bufs(P->layers[j], k)->ptr[q] = p;
      }
  }
  // the sigma_hat^2 partial sums: G x (blocks per shard) entries per half from now on
  for (int j = 0; j < Lc; ++j) {
    vbnn_layer* L = m->layers[j];
    L->shard_stale = &P->stale;
    if (L->kind != VBNN_KIND_VB) continue;
    int gq = update_grid(P->layers[j].rpo, L->I);
    if (gq > kMaxPartials / G) gq = kMaxPartials / G;
    if (gq > kNumSMs) gq = kNumSMs;      // one co-resident CTA per SM (see peer_after_dw)
    if (gq < 1) gq = 1;
    L->n_part = gq * G;
    VB_TRY(layer_refresh_prior_partials(L));
  }
  int lo = 0, hi = 0;
  VB_CUDA(cudaDeviceGetStreamPriorityRange(&lo, &hi));
  VB_CUDA(cudaStreamCreateWithPriority(&P->side, cudaStreamNonBlocking, hi));
  VB_CUDA(cudaStreamCreateWithPriority(&P->xfer, cudaStreamNonBlocking, hi));
  VB_CUDA(cudaEventCreateWithFlags(&P->ev_xfer, cudaEventDisableTiming));
  VB_CUDA(cudaMalloc((void**)&P->xfer_done, (kMaxPeers + 1) * sizeof(unsigned int)));
  VB_CUDA(cudaMemsetAsync(P->xfer_done, 0, (kMaxPeers + 1) * sizeof(unsigned int), c->stream));
  for (int j = 0; j < Lc; ++j) {
    PeerLayer& pl = P->layers[j];
    if (knobs().peer_transport == 1) continue;                     // fused stores only: no staging copy
    cudaError_t e = cudaMalloc((void**)&pl.stage, (size_t)G * pl.slot_floats * 4);
    if (e != cudaSuccess) { set_error("peer mode: cudaMalloc of the gradient staging copy failed: %s", cudaGetErrorString(e)); return VBNN_E_NOMEM; }
    VB_CUDA(cudaMemsetAsync(pl.stage, 0, (size_t)G * pl.slot_floats * 4, c->stream));
  }
  VB_CUDA(cudaEventCreateWithFlags(&P->ev_side, cudaEventDisableTiming));
  for (PeerLayer& pl : P->layers) VB_CUDA(cudaEventCreateWithFlags(&pl.ev_dw, cudaEventDisableTiming));
  VB_CUDA(cudaStreamSynchronize(c->stream));
  P->active = true;
  return VBNN_OK;
}

// Collective (host barrier before and after, on every rank): bring the fp32 state of the rows the
// other ranks own up to date -- whatever training does not push: Adam moments always, plus mu /
// log sigma^2 (LRT) or the nn.Linear weights (bf16) -- so that get / checkpoint / clamp_to_map see
// the whole layer (utils.lua:73-80, main.lua:181).
extern "C" int vbnn_mlp_sync_replicas(vbnn_mlp* m) {
  VB_CHECK(m, VBNN_E_INVALID, "null mlp");
  VB_CHECK(!m->step_open, VBNN_E_STATE, "vbnn_mlp_sync_replicas: a vbnn_mlp_forward_train step is open");
  vbnn_peer* P = m->peer;
  if (!P || !P->active) return VBNN_OK;
  vbnn_ctx* c = m->ctx;
  VB_CUDA(cudaSetDevice(c->device));
  VB_CUDA(cudaStreamSynchronize(c->stream));
  VB_CUDA(cudaStreamSynchronize(P->xfer));
  VB_CUDA(cudaStreamSynchronize(P->side));
  VB_TRY(peer_check(m));
  for (size_t j = 0; j < m->layers.size(); ++j) {
    vbnn_layer* L = m->layers[j];
    PeerLayer& pl = P->layers[j];
    const size_t rb = (size_t)L->I * 4;
    if (L->kind == VBNN_KIND_LINEAR) {
      if (L->w_bf16) VB_TRY(pull_shards(P, pl.weight, L->O, rb, pl.rpo, c->stream));
      continue;
    }
    if (layer_is_lrt(L)) {
      if (L->mu_bf16) VB_TRY(pull_shards(P, pl.means, L->O, rb, pl.rpo, c->stream));
      VB_TRY(pull_shards(P, pl.lvars, L->O, rb, pl.rpo, c->stream));
    }
    VB_TRY(pull_shards(P, pl.m_mu, L->O, rb, pl.rpo, c->stream));
    VB_TRY(pull_shards(P, pl.v_mu, L->O, rb, pl.rpo, c->stream));
    VB_TRY(pull_shards(P, pl.m_var, L->O, rb, pl.rpo, c->stream));
    VB_TRY(pull_shards(P, pl.v_var, L->O, rb, pl.rpo, c->stream));
  }
  VB_CUDA(cudaStreamSynchronize(c->stream));
  P->stale = false;
  return VBNN_OK;
}

extern "C" int vbnn_mlp_peer_active(const vbnn_mlp* m) { return m && m->peer && m->peer->active ? 1 : 0; }
