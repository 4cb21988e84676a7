// gemm.h -- host-side interface of the two GEMM engines (gemm_simt.cu, gemm_tc.cu).
#pragma once
#include "common.cuh"
#include "epilogue.cuh"

namespace vbnn {

// D[m,n] = sum_k A(m,k) B(k,n) (+ the A2 B2 product of the dual LRT modes) over `batch` samples.
// An operand is a row-major matrix of the engine's element type: bf16 for the tcgen05 engine
// (VBNN_PREC_BF16), fp32 for the CUDA-core engine (VBNN_PREC_FP32).  A with kmajor = 1 is stored
// [M x K], otherwise [K x M]; B with kmajor = 1 is stored [N x K], otherwise [K x N].  ld and zs (the
// batch stride) in elements; the tcgen05 engine feeds kmajor = 0 operands to the tensor core through an
// MN-major shared-memory descriptor (no transpose pass) and needs ld and zs to be multiples of 8
// (16-byte rows for TMA).
struct GemmOperand {
  const void* ptr;
  int ld;
  int kmajor;
  long long zs;
};
struct GemmArgs {
  GemmOperand A1, B1, A2, B2;
  int M, N, K, batch;
  // 1: sample-summing form (not for the z-accumulating dW modes): D = sum_z A_z B_z into ONE output (z = 0 of the
  // epilogue), summed in a fixed order
  int zsum;
};
int gemm_simt_launch(int mode, const GemmArgs& g, const EpiParams& p, cudaStream_t st, long long* launches);
int gemm_tc_launch(int mode, const GemmArgs& g, const EpiParams& p, cudaStream_t st, long long* launches);

}  // namespace vbnn
