// gemm.h -- host-side interface of the two GEMM engines (gemm_simt.cu, gemm_tc.cu).
#pragma once
#include "common.cuh"
#include "epilogue.cuh"

namespace vbnn {

// ---- fp32 CUDA-core engine (VBNN_PREC_FP32) ---------------------------------------------
// D[m,n] = sum_k A(m,k) B(k,n); element (m,k) of A at A[m*sAm + k*sAk], (k,n) of B at
// B[k*sBk + n*sBn].  A2/B2 are the second operand pair of the dual (LRT) modes.
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
int gemm_simt_launch(int mode, const SimtGemmArgs& g, const EpiParams& p, int batch,
                     cudaStream_t st, long long* launches);

// ---- bf16 tcgen05 engine (VBNN_PREC_BF16) --------------------------------------------------
// An operand is a row-major bf16 matrix.  kmajor = 1: stored [MN x K] (K contiguous);
// kmajor = 0: stored [K x MN] (MN contiguous; fed to the tensor core through an MN-major
// shared-memory descriptor, no transpose pass).  ld in elements, multiple of 8 (16-byte rows
// for TMA); zs = batch stride in elements (multiple of 8).
struct TcOperand {
  const bf16* ptr;
  int ld;
  int kmajor;
  long long zs;
};
struct TcGemmArgs {
  TcOperand A1, B1, A2, B2;
  int M, N, K, batch;
  // 1: sample-summing form (not for the z-accumulating dW modes): D = sum_z A_z B_z as ONE contraction over
  // K = batch x K (the accumulate bit stays set across z in TMEM), one work unit and one epilogue (z = 0) per tile
  int zsum;
};
int gemm_tc_launch(int mode, const TcGemmArgs& g, const EpiParams& p, cudaStream_t st,
                   long long* launches);
// debugging knobs for the descriptor probe (tests/tools only)
void gemm_tc_set_debug(int block_n_override);

}  // namespace vbnn
