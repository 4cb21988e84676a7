// epilogue.cuh -- the fused GEMM epilogues of the VBLinear hot path, shared by the tcgen05
// tensor-core kernel (gemm_tc.cu) and the fp32 CUDA-core kernel (gemm_simt.cu).
//
// One "quad" = 4 consecutive output columns of one output row; col % 4 == 0 so that a quad is
// exactly one Philox counter (philox.cuh).  What each mode replaces in the reference:
//   EPI_FWD      nn.Linear:updateOutput bias add (addr) + nn.ReLU           (mlp.lua:19,27,77)
//   EPI_FWD_LRT  local reparameterisation forward (SURVEY.md 8a A12; not in the reference)
//   EPI_DX       nn.Linear:updateGradInput + nn.ReLU backward               (mlp.lua:79)
//   EPI_DX_LRT   A12 backward-data
//   EPI_DW       VBLinear:accGradParameters: gradWeight += s*G^T X and
//                gradSum += (G^T X) .* eps from ONE GEMM                    (VBLinear.lua:113-115)
//   EPI_DW_LRT   A12 parameter gradients (two accumulators)
//   EPI_FWD_LRT2 / EPI_DX_LRT2  the same A12 forward / backward-data maths with one of the two products
//                read back from global memory instead of a second TMEM accumulator
#pragma once
#include <cuda_fp16.h>

#include "common.cuh"
#include "philox.cuh"

namespace vbnn {

enum EpiMode : int {
  EPI_STORE = 0,
  EPI_FWD = 1,
  EPI_FWD_LRT = 2,
  EPI_DX = 3,
  EPI_DX_LRT = 4,
  EPI_DW = 5,
  EPI_DW_LRT = 6,
  // Second halves of the SPLIT local-reparameterisation GEMMs (tensor-core engine): the first half is a
  // plain EPI_STORE GEMM that leaves its fp32 accumulator in `aux`; the second half's single accumulator
  // (TMEM double-buffered, so this heavy epilogue overlaps the next tile's MMAs) is joined with `aux`.
  EPI_FWD_LRT2 = 7,          // acc = X^2 s2^T (variance), aux = X mu^T (mean)
  EPI_DX_LRT2 = 8,           // acc = G mu, aux = H s2
};

__host__ __device__ constexpr bool epi_is_dual(int mode) {
  return mode == EPI_FWD_LRT || mode == EPI_DX_LRT || mode == EPI_DW_LRT;
}
// DW modes accumulate over the batch index z (MC samples) into one output.
__host__ __device__ constexpr bool epi_z_accumulates(int mode) {
  return mode == EPI_DW || mode == EPI_DW_LRT;
}

struct EpiParams {
  int M, N;                  // logical output extent (rows, cols)
  // generic outputs; "act" pointers are AT (float or bf16), selected by the kernel template
  float* out_f32; int ld_f32; long long zs_f32;
  void* out_act; void* out_act2; void* r_out; int ld_act; long long zs_act;
  // inputs read by the epilogue
  const float* bias;         // [N]               (FWD, FWD_LRT)
  int relu;                  // apply ReLU        (FWD, FWD_LRT)
  const void* xprev;         // AT [M x ld_x]     (DX: mask source; DX_LRT: X and mask source)
  const void* rprev;         // AT [M x ld_x]     (DX_LRT: R of the previous layer, nullable)
  int ld_x; long long zs_x;
  int mask;                  // DX/DX_LRT: multiply by (xprev > 0)
  const float* noise;        // injected eps [M x N] (DW) / zeta [M x N] (FWD_LRT); NULL -> Philox
  long long zs_noise;
  // DW, weight sampling on the tensor-core path: the epsilon k_sample_w drew for this minibatch, kept as fp16
  // [Z x M x ld_e16] (2 B per weight and sample instead of regenerating Philox + Box-Muller in the epilogue, which made
  // the multi-sample dW epilogue-bound 2:1).  One more operand rounding of the bf16 mode: |d eps| <= 2^-11 |eps|.
  const void* eps16; int ld_e16; long long zs_e16;
  PhiloxStream ps;           // Philox stream (sample = ps.sample + z)
  const uint32_t* step_ptr;  // device step counter (overrides ps.step when non-null)
  int row0;                  // global row offset of this rank's shard (FWD_LRT zeta)
  // DW outputs
  float* gW; float* gS; int ld_g;
  float scale;               // accGradParameters' scale
  int accumulate;            // 0: first z overwrites (saves the memset), 1: always +=
  // peer mode: rows [q*scatter_rows, (q+1)*scatter_rows) go to rank q's receive slot (pointers are
  // pre-biased so that row * ld_g + col indexes them like gW / gS); 0 = plain local gW / gS
  int scatter_rows;
  float* gW_peer[8]; float* gS_peer[8];
  // bf16 gradient tiles (peer mode, staged transports, knob peer_wire_bf16): gW / gS (and the per-owner pointers) are bf16
  // buffers written ONCE (accumulate == 0, one sample); halves the NVLink bytes of the reduce-scatter at the price of one
  // more rounding point (each rank's partial sum, 2^-9 relative), stated separately in dp_parity
  int grads_bf16;
  // split LRT modes: the other product, fp32 [M x ld_aux] (+ z * zs_aux)
  const float* aux; int ld_aux; long long zs_aux;
};

// destination of a dW tile whose rows all share one owner (32-row warp chunks: scatter_rows % 32 == 0)
__device__ __forceinline__ void dw_dest(const EpiParams& p, int row, float*& gW, float*& gS) {
  if (p.scatter_rows == 0) { gW = p.gW; gS = p.gS; return; }
  const int q = row / p.scatter_rows;
  gW = p.gW_peer[q];
  gS = p.gS_peer[q];
}

template <typename AT> struct Vec4;
template <> struct Vec4<float> {
  static __device__ __forceinline__ void load(const float* p, float (&v)[4]) {
    float4 t = *reinterpret_cast<const float4*>(p);
    v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
  }
  static __device__ __forceinline__ void store(float* p, const float (&v)[4]) {
    *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
  }
};
template <> struct Vec4<bf16> {
  static __device__ __forceinline__ void load(const bf16* p, float (&v)[4]) {
    uint2 t = *reinterpret_cast<const uint2*>(p);
    __nv_bfloat162 a = *reinterpret_cast<__nv_bfloat162*>(&t.x);
    __nv_bfloat162 b = *reinterpret_cast<__nv_bfloat162*>(&t.y);
    v[0] = __low2float(a); v[1] = __high2float(a); v[2] = __low2float(b); v[3] = __high2float(b);
  }
  static __device__ __forceinline__ void store(bf16* p, const float (&v)[4]) {
    __nv_bfloat162 a = __floats2bfloat162_rn(v[0], v[1]);
    __nv_bfloat162 b = __floats2bfloat162_rn(v[2], v[3]);
    uint2 t;
    t.x = *reinterpret_cast<uint32_t*>(&a);
    t.y = *reinterpret_cast<uint32_t*>(&b);
    *reinterpret_cast<uint2*>(p) = t;
  }
};

template <typename T>
__device__ __forceinline__ void load4(const T* p, float (&v)[4], int nvalid, bool vec) {
  if (vec && nvalid == 4) {
    Vec4<T>::load(p, v);
  } else {
#pragma unroll
    for (int j = 0; j < 4; ++j) v[j] = j < nvalid ? to_f32(p[j]) : 0.f;
  }
}
template <typename T>
__device__ __forceinline__ void store4(T* p, const float (&v)[4], int nvalid, bool vec) {
  if (vec && nvalid == 4) {
    Vec4<T>::store(p, v);
  } else {
#pragma unroll
    for (int j = 0; j < 4; ++j)
      if (j < nvalid) p[j] = from_f32<T>(v[j]);
  }
}

// Philox stream of this launch with the device-side step counter resolved ONCE per thread (the
// kernels call this at entry; doing it per quad put a dependent global load in front of every
// Philox chain).
__device__ __forceinline__ PhiloxStream epi_stream(const EpiParams& p) {
  PhiloxStream ps = p.ps;
  if (p.step_ptr) ps.step = *p.step_ptr;
  return ps;
}

__device__ __forceinline__ void load_bias4(const float* bias, int col, int nvalid, float (&b)[4]) {
  if (bias == nullptr) { b[0] = b[1] = b[2] = b[3] = 0.f; return; }
  if (nvalid == 4) {
    float4 t = __ldg(reinterpret_cast<const float4*>(bias + col));   // col % 4 == 0, cudaMalloc-aligned
    b[0] = t.x; b[1] = t.y; b[2] = t.z; b[3] = t.w;
  } else {
#pragma unroll
    for (int j = 0; j < 4; ++j) b[j] = j < nvalid ? __ldg(bias + col + j) : 0.f;
  }
}

// 1/sqrt(V) of the local-reparameterisation forward, from which sqrt(V) = V * rs and R = zeta * rs / 2 follow.
// V >= FLT_MIN: one MUFU.RSQ.  0 < V < FLT_MIN (a row whose inputs are all below ~1e-19): the .ftz of that
// instruction would flush V to 0 and return +inf, turning Y and R into +-inf; V * 2^64 is exact and normal, and
// rsqrt(V * 2^64) * 2^32 = rsqrt(V).  V = 0 (an all-zero input row): 0, so that R = 0 (include/vbnn.h).
__device__ __forceinline__ float lrt_rsqrt(float v) {
  if (v >= 1.17549435e-38f) return rsqrt_fast(v);
  return v > 0.f ? rsqrt_fast(v * 18446744073709551616.f) * 4294967296.f : 0.f;
}

// Process one quad.  a1/a2: accumulator values (a2 only for dual modes).
template <int MODE, typename AT>
__device__ __forceinline__ void epi_quad(const EpiParams& p, const PhiloxStream& ps0, int z, int row, int col,
                                         const float (&a1)[4], const float (&a2)[4]);

// split modes: fetch the other product, then run the dual-mode code
template <int MODE, typename AT>
__device__ __forceinline__ void epi_quad_split(const EpiParams& p, const PhiloxStream& ps0, int z, int row, int col,
                                               const float (&acc)[4]) {
  if (row >= p.M || col >= p.N) return;
  float o[4];
  load4<float>(p.aux + z * p.zs_aux + (long long)row * p.ld_aux + col, o, min(4, p.N - col), (p.ld_aux & 3) == 0);
  if constexpr (MODE == EPI_FWD_LRT2) epi_quad<EPI_FWD_LRT, AT>(p, ps0, z, row, col, o, acc);     // (mean, variance)
  else epi_quad<EPI_DX_LRT, AT>(p, ps0, z, row, col, acc, o);                                    // (G mu, H s2)
}

template <int MODE, typename AT>
__device__ __forceinline__ void epi_quad(const EpiParams& p, const PhiloxStream& ps0, int z, int row, int col,
                                         const float (&a1)[4], const float (&a2)[4]) {
  if constexpr (MODE == EPI_FWD_LRT2 || MODE == EPI_DX_LRT2) { epi_quad_split<MODE, AT>(p, ps0, z, row, col, a1); return; }
  if (row >= p.M || col >= p.N) return;
  const int nvalid = min(4, p.N - col);
  const bool vec_act = (p.ld_act & 3) == 0;
  const bool vec_f32 = (p.ld_f32 & 3) == 0;

  if constexpr (MODE == EPI_STORE) {
    store4<float>(p.out_f32 + z * p.zs_f32 + (long long)row * p.ld_f32 + col, a1, nvalid, vec_f32);
  } else if constexpr (MODE == EPI_FWD) {
    float y[4], b[4];
    load_bias4(p.bias, col, nvalid, b);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      y[j] = a1[j] + b[j];
      if (p.relu) y[j] = fmaxf(y[j], 0.f);
    }
    if (p.out_f32)
      store4<float>(p.out_f32 + z * p.zs_f32 + (long long)row * p.ld_f32 + col, y, nvalid, vec_f32);
    if (p.out_act)
      store4<AT>((AT*)p.out_act + z * p.zs_act + (long long)row * p.ld_act + col, y, nvalid, vec_act);
  } else if constexpr (MODE == EPI_FWD_LRT) {
    float zt[4];
    if (p.noise) {
      load4<float>(p.noise + z * p.zs_noise + (long long)row * p.N + col, zt, nvalid, (p.N & 3) == 0);
    } else {
      PhiloxStream ps = ps0;
      ps.sample += (uint32_t)z;
      uint32_t q = (uint32_t)((p.N + 3) >> 2);
      philox_normal4(ps, (uint32_t)(row + p.row0) * q + (uint32_t)(col >> 2), zt);
    }
    float y[4], y2[4], r[4], b[4];
    load_bias4(p.bias, col, nvalid, b);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      // sqrt(V) and zeta / (2 sqrt(V)) from one MUFU.RSQ (V = 0 only for an all-zero input row)
      const float v = a2[j];
      const float rs = lrt_rsqrt(v);
      const float sq = v * rs;
      y[j] = a1[j] + b[j] + sq * zt[j];
      r[j] = 0.5f * zt[j] * rs;
    }
    if (p.out_f32)
      store4<float>(p.out_f32 + z * p.zs_f32 + (long long)row * p.ld_f32 + col, y, nvalid, vec_f32);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      if (p.relu) y[j] = fmaxf(y[j], 0.f);
      // square the value the next layer will actually read (after rounding to AT)
      float yr = to_f32(from_f32<AT>(y[j]));
      y2[j] = yr * yr;
    }
    long long off = z * p.zs_act + (long long)row * p.ld_act + col;
    if (p.out_act) store4<AT>((AT*)p.out_act + off, y, nvalid, vec_act);
    if (p.out_act2) store4<AT>((AT*)p.out_act2 + off, y2, nvalid, vec_act);
    if (p.r_out) store4<AT>((AT*)p.r_out + off, r, nvalid, vec_act);
  } else if constexpr (MODE == EPI_DX || MODE == EPI_DX_LRT) {
    const bool vec_x = (p.ld_x & 3) == 0;
    long long xoff = z * p.zs_x + (long long)row * p.ld_x + col;
    float x[4] = {0.f, 0.f, 0.f, 0.f};
    if (p.xprev) load4<AT>((const AT*)p.xprev + xoff, x, nvalid, vec_x);
    float g[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      g[j] = a1[j];
      if constexpr (MODE == EPI_DX_LRT) g[j] += 2.f * x[j] * a2[j];
      if (p.mask) g[j] = x[j] > 0.f ? g[j] : 0.f;
    }
    if (p.out_f32)
      store4<float>(p.out_f32 + z * p.zs_f32 + (long long)row * p.ld_f32 + col, g, nvalid, vec_f32);
    long long off = z * p.zs_act + (long long)row * p.ld_act + col;
    if (p.out_act) store4<AT>((AT*)p.out_act + off, g, nvalid, vec_act);
    if (p.out_act2 && p.rprev) {
      float r[4], h[4];
      load4<AT>((const AT*)p.rprev + xoff, r, nvalid, vec_x);
#pragma unroll
      for (int j = 0; j < 4; ++j) h[j] = to_f32(from_f32<AT>(g[j])) * r[j];
      store4<AT>((AT*)p.out_act2 + off, h, nvalid, vec_act);
    }
  } else if constexpr (MODE == EPI_DW || MODE == EPI_DW_LRT) {
    const bool vec_g = (p.ld_g & 3) == 0;
    long long goff = (long long)row * p.ld_g + col;
    const bool acc = p.accumulate || z > 0;
    float *gWd, *gSd;
    dw_dest(p, row, gWd, gSd);
    if (p.grads_bf16) {
      float w[4], sv[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) { w[j] = p.scale * a1[j]; sv[j] = MODE == EPI_DW_LRT ? a2[j] : 0.f; }
      store4<bf16>(reinterpret_cast<bf16*>(gWd) + goff, w, nvalid, (p.ld_g & 3) == 0);
      if (p.gS) {
        if constexpr (MODE == EPI_DW_LRT) store4<bf16>(reinterpret_cast<bf16*>(gSd) + goff, sv, nvalid, (p.ld_g & 3) == 0);
      }
      return;
    }
    float w[4] = {0.f, 0.f, 0.f, 0.f};
    if (acc) load4<float>(gWd + goff, w, nvalid, vec_g);
#pragma unroll
    for (int j = 0; j < 4; ++j) w[j] += p.scale * a1[j];
    store4<float>(gWd + goff, w, nvalid, vec_g);
    if (p.gS) {
      float s[4] = {0.f, 0.f, 0.f, 0.f};
      if (acc) load4<float>(gSd + goff, s, nvalid, vec_g);
      if constexpr (MODE == EPI_DW) {
        float e[4];
        if (p.noise) {
          load4<float>(p.noise + z * p.zs_noise + (long long)row * p.N + col, e, nvalid, (p.N & 3) == 0);
        } else if (p.eps16) {
          const __half* ep = reinterpret_cast<const __half*>(p.eps16) + z * p.zs_e16 + (long long)row * p.ld_e16 + col;
#pragma unroll
          for (int j = 0; j < 4; ++j) e[j] = j < nvalid ? __half2float(ep[j]) : 0.f;
        } else {
          PhiloxStream ps = ps0;
          ps.sample += (uint32_t)z;
          uint32_t q = (uint32_t)((p.N + 3) >> 2);
          philox_normal4(ps, (uint32_t)row * q + (uint32_t)(col >> 2), e);
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) s[j] += a1[j] * e[j];     // VBLinear.lua:115 (ignores scale)
      } else {
#pragma unroll
        for (int j = 0; j < 4; ++j) s[j] += a2[j];
      }
      store4<float>(gSd + goff, s, nvalid, vec_g);
    }
  }
}

}  // namespace vbnn
