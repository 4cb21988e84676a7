// gemm_simt.cu -- fp32-operand / fp32-accumulate CUDA-core GEMM with the fused VB epilogues.
//
// This is the VBNN_PREC_FP32 "exact parity" mode: the reference computes everything in fp32
// (main.lua:10), so this path is directly comparable with the oracle to ~1e-6.  It is also what
// serves the tiny launch-bound C1 config.  The throughput path is gemm_tc.cu (tcgen05).
//
// D[m,n] = sum_k A(m,k) * B(k,n) with arbitrary element strides, so one kernel covers
//   forward   Y  = X W^T      (A = X [N x I], B(k,n) = W[n*ldw + k])          nn.Linear:updateOutput
//   backward  dX = G W        (A = G [N x O], B(k,n) = W[k*ldw + n])          nn.Linear:updateGradInput
//   wgrad     dW = G^T X      (A(m,k) = G[k*ldg + m], B(k,n) = X[k*ldx + n])  VBLinear.lua:113-115
#include <map>
#include <utility>

#include "gemm.h"

namespace vbnn {

// The kernel's view of GemmArgs: element (m,k) of A at A[m*sAm + k*sAk], (k,n) of B at B[k*sBk + n*sBn].
struct SimtGemmArgs {
  const float* A1; long long sA1m, sA1k, zsA1;
  const float* B1; long long sB1n, sB1k, zsB1;
  const float* A2; long long sA2m, sA2k, zsA2;
  const float* B2; long long sB2n, sB2k, zsB2;
  int M, N, K;
  // > 1: sum the products of samples z = 0 .. zsum-1 into ONE output (z = 0 of the epilogue), register
  // accumulation in a fixed order; launch with batch = 1
  int zsum;
};

constexpr int TM = 64, TN = 64, TK = 16;
__device__ __forceinline__ int ceil_div_dev(int a, int b) { return (a + b - 1) / b; }
__device__ __forceinline__ int round_up_dev(int a, int b) { return (a + b - 1) / b * b; }

template <bool DUAL>
struct SimtSmem {
  float a[DUAL ? 2 : 1][TK][TM + 4];
  float b[DUAL ? 2 : 1][TK][TN + 4];
};

__device__ __forceinline__ void load_tile(float (*dst)[TM + 4], const float* __restrict__ src,
                                          long long s_mn, long long s_k, int mn0, int k0, int MN,
                                          int K) {
  // 64 (mn) x 16 (k) elements, 256 threads -> 4 each; make the unit-stride dim the fastest.
  const int tid = threadIdx.x;
  if (s_k == 1) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      int e = tid + i * 256;
      int k = e & 15, mn = e >> 4;
      int gm = mn0 + mn, gk = k0 + k;
      dst[k][mn] = (gm < MN && gk < K) ? src[gm * s_mn + gk] : 0.f;
    }
  } else {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      int e = tid + i * 256;
      int mn = e & 63, k = e >> 6;
      int gm = mn0 + mn, gk = k0 + k;
      dst[k][mn] = (gm < MN && gk < K) ? src[gm * s_mn + gk * s_k] : 0.f;
    }
  }
}

// ksplit > 1: blockIdx.z = z * ksplit + ks and CTA ks contracts only its slice of K, leaving raw partial accumulators in
// `scratch` [(z * ksplit + ks) * NACC + a][M x N]; k_simt_finish then adds the slices in a fixed order and runs the fused
// epilogue.  For the tiny launch-bound configs (C1: 100 x 100 outputs, K = 784 -- 4 CTAs walking 49 k-steps serially)
// this turns one long dependent chain into ksplit short ones.
template <int MODE, bool DUAL>
__global__ void __launch_bounds__(256) gemm_simt_kernel(SimtGemmArgs g, EpiParams p, int ksplit, float* scratch) {
  __shared__ SimtSmem<DUAL> sm;
  const int z = blockIdx.z / ksplit, ks = blockIdx.z - z * ksplit;
  const int m0 = blockIdx.y * TM, n0 = blockIdx.x * TN;
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const int kchunk = ksplit > 1 ? round_up_dev(ceil_div_dev(g.K, ksplit), TK) : g.K;
  const int k_begin = ks * kchunk, k_end = min(g.K, k_begin + kchunk);

  float acc1[4][4] = {}, acc2[4][4] = {};
  // sample-summing form (g.zsum > 1, z = 0): the samples' products accumulate in registers, sample by sample
  const int nz = g.zsum > 1 ? g.zsum : 1;
  for (int zz = z; zz < z + nz; ++zz) {
    const float* A1 = g.A1 + zz * g.zsA1;
    const float* B1 = g.B1 + zz * g.zsB1;
    const float* A2 = DUAL ? g.A2 + zz * g.zsA2 : nullptr;
    const float* B2 = DUAL ? g.B2 + zz * g.zsB2 : nullptr;
    for (int k0 = k_begin; k0 < k_end; k0 += TK) {
      load_tile(sm.a[0], A1, g.sA1m, g.sA1k, m0, k0, g.M, k_end);
      load_tile(sm.b[0], B1, g.sB1n, g.sB1k, n0, k0, g.N, k_end);
      if (DUAL) {
        load_tile(sm.a[DUAL ? 1 : 0], A2, g.sA2m, g.sA2k, m0, k0, g.M, k_end);
        load_tile(sm.b[DUAL ? 1 : 0], B2, g.sB2n, g.sB2k, n0, k0, g.N, k_end);
      }
      __syncthreads();
#pragma unroll
      for (int k = 0; k < TK; ++k) {
        float4 av = *reinterpret_cast<const float4*>(&sm.a[0][k][ty * 4]);
        float4 bv = *reinterpret_cast<const float4*>(&sm.b[0][k][tx * 4]);
        float a[4] = {av.x, av.y, av.z, av.w}, b[4] = {bv.x, bv.y, bv.z, bv.w};
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j) acc1[i][j] = fmaf(a[i], b[j], acc1[i][j]);
        if (DUAL) {
          float4 av2 = *reinterpret_cast<const float4*>(&sm.a[DUAL ? 1 : 0][k][ty * 4]);
          float4 bv2 = *reinterpret_cast<const float4*>(&sm.b[DUAL ? 1 : 0][k][tx * 4]);
          float a2[4] = {av2.x, av2.y, av2.z, av2.w}, b2[4] = {bv2.x, bv2.y, bv2.z, bv2.w};
#pragma unroll
          for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) acc2[i][j] = fmaf(a2[i], b2[j], acc2[i][j]);
        }
      }
      __syncthreads();
    }
  }
  if (ksplit > 1) {
    constexpr int NACC = DUAL ? 2 : 1;
    const long long MN = (long long)g.M * g.N;
    float* s1 = scratch + ((long long)blockIdx.z * NACC) * MN;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int row = m0 + ty * 4 + i;
      if (row >= g.M) continue;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int col = n0 + tx * 4 + j;
        if (col >= g.N) continue;
        s1[(long long)row * g.N + col] = acc1[i][j];
        if (DUAL) s1[MN + (long long)row * g.N + col] = acc2[i][j];
      }
    }
    return;
  }
  const PhiloxStream ps = epi_stream(p);
#pragma unroll
  for (int i = 0; i < 4; ++i) epi_quad<MODE, float>(p, ps, z, m0 + ty * 4 + i, n0 + tx * 4, acc1[i], acc2[i]);
}

// one thread per quad: add the K slices in slice order, then the same fused epilogue
template <int MODE, bool DUAL>
__global__ void __launch_bounds__(256) k_simt_finish(int M, int N, int batch, int ksplit, const float* scratch, EpiParams p) {
  constexpr int NACC = DUAL ? 2 : 1;
  const int Q = (N + 3) >> 2;
  const long long quads = (long long)batch * M * Q, MN = (long long)M * N;
  const PhiloxStream ps = epi_stream(p);
  for (long long qd = blockIdx.x * (long long)blockDim.x + threadIdx.x; qd < quads; qd += (long long)gridDim.x * blockDim.x) {
    const int z = (int)(qd / ((long long)M * Q));
    const long long r = qd - (long long)z * M * Q;
    const int row = (int)(r / Q), col = (int)(r - (long long)row * Q) * 4;
    float a1[4] = {0.f, 0.f, 0.f, 0.f}, a2[4] = {0.f, 0.f, 0.f, 0.f};
    for (int ks = 0; ks < ksplit; ++ks) {
      const float* s1 = scratch + ((long long)(z * ksplit + ks) * NACC) * MN + (long long)row * N + col;
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (col + j < N) { a1[j] += s1[j]; if (DUAL) a2[j] += s1[MN + j]; }
    }
    epi_quad<MODE, float>(p, ps, z, row, col, a1, a2);
  }
}

// Scratch for the K-split partials: one fixed-size buffer per (device, stream), allocated on first use and never moved
// (a captured CUDA graph bakes the pointer into its kernel nodes).  The heuristic below bounds the need:
// <= 32 CTAs x 64 x 64 outputs x 8 slices x 2 accumulators.
constexpr size_t kScratchFloats = (size_t)32 * TM * TN * 8 * 2;
static std::map<std::pair<int, cudaStream_t>, float*> g_scratch;
static int get_scratch(cudaStream_t st, bool may_allocate, float** out) {
  int dev = 0;
  cudaGetDevice(&dev);
  auto it = g_scratch.find({dev, st});
  if (it != g_scratch.end()) { *out = it->second; return VBNN_OK; }
  *out = nullptr;
  if (!may_allocate) return VBNN_OK;
  float* p = nullptr;
  VB_CUDA(cudaMalloc((void**)&p, kScratchFloats * sizeof(float)));
  g_scratch[{dev, st}] = p;
  *out = p;
  return VBNN_OK;
}

static int choose_ksplit(const SimtGemmArgs& g, int batch) {
  const long long ctas = (long long)ceil_div(g.N, TN) * ceil_div(g.M, TM) * batch;
  if (ctas > 32 || g.K < 256) return 1;
  int ks = g.K / 128;
  return ks < 1 ? 1 : (ks > 8 ? 8 : ks);
}

template <int MODE>
static int launch_one(const SimtGemmArgs& g, const EpiParams& p, int batch, cudaStream_t st) {
  constexpr bool DUAL = epi_is_dual(MODE);
  int ksplit = choose_ksplit(g, batch);
  float* scratch = nullptr;
  if (ksplit > 1) {
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    cudaStreamIsCapturing(st, &cs);
    VB_TRY(get_scratch(st, cs == cudaStreamCaptureStatusNone, &scratch));      // never allocate inside a capture
    const size_t need = (size_t)batch * ksplit * (DUAL ? 2 : 1) * g.M * g.N;
    if (!scratch || need > kScratchFloats) ksplit = 1;
  }
  dim3 grid(ceil_div(g.N, TN), ceil_div(g.M, TM), batch * ksplit);
  gemm_simt_kernel<MODE, DUAL><<<grid, 256, 0, st>>>(g, p, ksplit, scratch);
  if (ksplit > 1) {
    const long long quads = (long long)batch * g.M * ((g.N + 3) / 4);
    int blocks = (int)((quads + 255) / 256);
    if (blocks > kNumSMs * 4) blocks = kNumSMs * 4;
    k_simt_finish<MODE, DUAL><<<blocks, 256, 0, st>>>(g.M, g.N, batch, ksplit, scratch, p);
  }
  VB_CUDA(cudaGetLastError());
  return VBNN_OK;
}

template <int MODE>
static int launch_mode(const SimtGemmArgs& g, const EpiParams& p, int batch, cudaStream_t st) {
  constexpr bool DUAL = epi_is_dual(MODE);
  if (g.M <= 0 || g.N <= 0) return VBNN_OK;
  if (epi_z_accumulates(MODE)) {
    // z = MC sample accumulates into one output: serialise over z (deterministic order)
    for (int z = 0; z < batch; ++z) {
      SimtGemmArgs gz = g;
      gz.A1 += z * g.zsA1; gz.B1 += z * g.zsB1;
      if (DUAL) { gz.A2 += z * g.zsA2; gz.B2 += z * g.zsB2; }
      EpiParams pz = p;
      pz.ps.sample += z;
      if (pz.noise) pz.noise += z * p.zs_noise;
      if (pz.eps16) pz.eps16 = reinterpret_cast<const char*>(pz.eps16) + (long long)z * p.zs_e16 * 2;
      pz.accumulate = p.accumulate || z > 0;
      VB_TRY(launch_one<MODE>(gz, pz, 1, st));
    }
    return VBNN_OK;
  }
  return launch_one<MODE>(g, p, batch, st);
}

// A (m,k) / B (k,n) of a GemmOperand as a stride pair
static void simt_operand(const GemmOperand& o, const float** ptr, long long* s_mn, long long* s_k, long long* zs) {
  *ptr = static_cast<const float*>(o.ptr);
  *s_mn = o.kmajor ? o.ld : 1;
  *s_k = o.kmajor ? 1 : o.ld;
  *zs = o.zs;
}

int gemm_simt_launch(int mode, const GemmArgs& a, const EpiParams& p, cudaStream_t st, long long* launches) {
  SimtGemmArgs g = {};
  simt_operand(a.A1, &g.A1, &g.sA1m, &g.sA1k, &g.zsA1);
  simt_operand(a.B1, &g.B1, &g.sB1n, &g.sB1k, &g.zsB1);
  if (epi_is_dual(mode)) {
    simt_operand(a.A2, &g.A2, &g.sA2m, &g.sA2k, &g.zsA2);
    simt_operand(a.B2, &g.B2, &g.sB2n, &g.sB2k, &g.zsB2);
  }
  g.M = a.M; g.N = a.N; g.K = a.K;
  // the sample-summing form runs the samples inside one CTA: zsum = batch, launched with batch 1
  g.zsum = a.zsum ? a.batch : 0;
  const int batch = a.zsum ? 1 : a.batch;
  VB_CHECK(g.zsum <= 1 || (batch == 1 && !epi_z_accumulates(mode)), VBNN_E_INVALID,
           "gemm_simt: the sample-summing form runs with batch 1 and no dW mode");
  if (launches) {
    const bool zacc = epi_z_accumulates(mode);
    *launches += (long long)(zacc ? batch : 1) * (choose_ksplit(g, zacc ? 1 : batch) > 1 ? 2 : 1);   // + the K-split finish kernel
  }
  switch (mode) {
    case EPI_STORE: return launch_mode<EPI_STORE>(g, p, batch, st);
    case EPI_FWD: return launch_mode<EPI_FWD>(g, p, batch, st);
    case EPI_FWD_LRT: return launch_mode<EPI_FWD_LRT>(g, p, batch, st);
    case EPI_DX: return launch_mode<EPI_DX>(g, p, batch, st);
    case EPI_DX_LRT: return launch_mode<EPI_DX_LRT>(g, p, batch, st);
    case EPI_DW: return launch_mode<EPI_DW>(g, p, batch, st);
    case EPI_DW_LRT: return launch_mode<EPI_DW_LRT>(g, p, batch, st);
  }
  set_error("gemm_simt_launch: bad mode %d", mode);
  return VBNN_E_INVALID;
}

}  // namespace vbnn
