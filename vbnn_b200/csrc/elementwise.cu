// elementwise.cu -- the HBM-bound kernels of the VBLinear path: one pass each, 128-bit
// accesses where rows allow it, warp-shuffle + block reductions, results stay on the device.
// Each kernel replaces a chain of THC pointwise/reduction launches in the reference; the
// citations name the chain.
#include <cuda_fp16.h>

#include "kernels.h"
#include "knobs.h"

namespace vbnn {

namespace {

constexpr int kThreads = 256;

inline int grid_for(long long work_items, int per_sm = 8) {
  long long blocks = (work_items + kThreads - 1) / kThreads;
  long long cap = (long long)kNumSMs * per_sm;
  if (blocks < 1) blocks = 1;
  return (int)(blocks < cap ? blocks : cap);
}

__device__ __forceinline__ float4 ld4(const float* p) { return *reinterpret_cast<const float4*>(p); }
__device__ __forceinline__ void st4(float* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }
__device__ __forceinline__ void st4_bf16(bf16* p, float a, float b, float c, float d) {
  __nv_bfloat162 lo = __floats2bfloat162_rn(a, b), hi = __floats2bfloat162_rn(c, d);
  uint2 t;
  t.x = *reinterpret_cast<uint32_t*>(&lo);
  t.y = *reinterpret_cast<uint32_t*>(&hi);
  *reinterpret_cast<uint2*>(p) = t;
}

// ------------------------------------------------------------------ sample --------------
// VBLinear.lua:55-63: CPU randomkit fill + H2D + cmul + add + copy  ->  one pass.
// One thread = one quad (4 consecutive i of one row o) = one Philox counter.
template <bool VEC>
__global__ void __launch_bounds__(kThreads) k_sample_w(SampleParams p) {
  const int Q = (p.I + 3) >> 2;
  const long long quads = (long long)p.O * Q;
  PhiloxStream ps0 = p.ps;
  if (p.step_ptr) ps0.step = *p.step_ptr;
  const long long OI = (long long)p.O * p.I;
  for (long long qd = blockIdx.x * (long long)blockDim.x + threadIdx.x; qd < quads;
       qd += (long long)gridDim.x * blockDim.x) {
    const int o = (int)(qd / Q), c = (int)(qd - (long long)o * Q);
    const int i0 = c * 4;
    const long long e0 = (long long)o * p.I + i0;
    const int nv = min(4, p.I - i0);
    // mu and sigma are read (and sigma exponentiated) once for ALL samples of the minibatch
    float mu[4], sd[4];
    if (VEC) {
      float4 a = ld4(p.mu + e0), b = ld4(p.sig + e0);
      mu[0] = a.x; mu[1] = a.y; mu[2] = a.z; mu[3] = a.w;
      sd[0] = b.x; sd[1] = b.y; sd[2] = b.z; sd[3] = b.w;
    } else {
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        mu[j] = j < nv ? p.mu[e0 + j] : 0.f;
        sd[j] = j < nv ? p.sig[e0 + j] : 0.f;
      }
    }
    if (p.sig_is_lvar) {
#pragma unroll
      for (int j = 0; j < 4; ++j) sd[j] = __expf(0.5f * sd[j]);
    }
#pragma unroll 2
    for (int s = blockIdx.y; s < p.S; s += gridDim.y) {
      float ep[4], w[4];
      if (p.eps_in) {
        if (VEC) {
          float4 e = ld4(p.eps_in + s * OI + e0);
          ep[0] = e.x; ep[1] = e.y; ep[2] = e.z; ep[3] = e.w;
        } else {
#pragma unroll
          for (int j = 0; j < 4; ++j) ep[j] = j < nv ? p.eps_in[s * OI + e0 + j] : 0.f;
        }
      } else {
        PhiloxStream ps = ps0;
        ps.sample += (uint32_t)s;
        philox_normal4(ps, (uint32_t)qd, ep);
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) w[j] = fmaf(sd[j], ep[j], mu[j]);          // VBLinear.lua:59
      if (p.eps_out) {
        if (VEC) st4(p.eps_out + s * OI + e0, make_float4(ep[0], ep[1], ep[2], ep[3]));
        else
          for (int j = 0; j < nv; ++j) p.eps_out[s * OI + e0 + j] = ep[j];
      }
      if (p.w_f32) {
        if (VEC) st4(p.w_f32 + s * OI + e0, make_float4(w[0], w[1], w[2], w[3]));
        else
          for (int j = 0; j < nv; ++j) p.w_f32[s * OI + e0 + j] = w[j];
      }
      if (p.w_bf16) {
        bf16* dst = p.w_bf16 + s * p.zs_bf16 + (long long)o * p.ld_bf16 + i0;
        if (nv == 4) st4_bf16(dst, w[0], w[1], w[2], w[3]);
        else
          for (int j = 0; j < nv; ++j) dst[j] = __float2bfloat16_rn(w[j]);
      }
      if (p.eps16) {
        __half* dst = reinterpret_cast<__half*>(p.eps16) + s * p.zs_bf16 + (long long)o * p.ld_bf16 + i0;
        if (nv == 4) {
          const __half2 lo = __floats2half2_rn(ep[0], ep[1]), hi = __floats2half2_rn(ep[2], ep[3]);
          uint2 t;
          t.x = *reinterpret_cast<const uint32_t*>(&lo);
          t.y = *reinterpret_cast<const uint32_t*>(&hi);
          *reinterpret_cast<uint2*>(dst) = t;
        } else {
          for (int j = 0; j < nv; ++j) dst[j] = __float2half_rn(ep[j]);
        }
      }
    }
  }
}

// ------------------------------------------------------------------ prior ---------------
// VBLinear.lua:78-86: exp, sqrt, add, pow, add, sum + D2H sync  ->  one read pass, no sync.
__global__ void __launch_bounds__(kThreads) k_prior_partials(const float* __restrict__ mu,
                                                             const float* __restrict__ lvar,
                                                             long long n, double* partials,
                                                             const int* t_dev) {
  __shared__ double sh[32];
  if (t_dev) partials += (size_t)(*t_dev & 1) * kMaxPartials;
  float acc = 0.f;
  double dacc = 0.0;
  const long long n4 = n >> 2;
  const long long stride = (long long)gridDim.x * blockDim.x;
  int cnt = 0;
  for (long long q = blockIdx.x * (long long)blockDim.x + threadIdx.x; q < n4; q += stride) {
    float4 m = ld4(mu + 4 * q), l = ld4(lvar + 4 * q);
    acc += __expf(l.x) + m.x * m.x;
    acc += __expf(l.y) + m.y * m.y;
    acc += __expf(l.z) + m.z * m.z;
    acc += __expf(l.w) + m.w * m.w;
    if (++cnt == 64) { dacc += acc; acc = 0.f; cnt = 0; }
  }
  dacc += acc;
  if (blockIdx.x == 0 && threadIdx.x < (n & 3)) {
    long long e = (n4 << 2) + threadIdx.x;
    dacc += (double)(__expf(lvar[e]) + mu[e] * mu[e]);
  }
  double r = block_sum(dacc, sh);
  if (threadIdx.x == 0) partials[blockIdx.x] = r;
}

__global__ void __launch_bounds__(kThreads) k_prior_finalize(const double* partials, int np,
                                                             long long W, float* var_hat,
                                                             const float* mu, const float* lvar,
                                                             float* stdv, float* mu_sqe, PriorArgs pr) {
  __shared__ double sh[32];
  if (blockIdx.x == 0) {
    if (pr.kind == VBNN_PRIOR_EMPIRICAL) {
      double a = 0.0;
      for (int i = threadIdx.x; i < np; i += blockDim.x) a += partials[i];
      double r = block_sum(a, sh);
      if (threadIdx.x == 0) *var_hat = (float)(r / (double)W);        // VBLinear.lua:86
    } else if (threadIdx.x == 0) {
      *var_hat = pr.kind == VBNN_PRIOR_FIXED ? pr.var0 : __int_as_float(0x7fc00000);
    }
  }
  if (stdv || mu_sqe) {
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < W;
         e += (long long)gridDim.x * blockDim.x) {
      if (stdv) stdv[e] = __expf(0.5f * lvar[e]);                       // VBLinear.lua:78-79
      if (mu_sqe) {                                                     // VBLinear.lua:82
        const float d = mu[e] - (pr.mu ? pr.mu[e] : pr.mu0);
        mu_sqe[e] = d * d;
      }
    }
  }
}

// ------------------------------------------------------------------ fused update --------
// VBLinear.lua:130-143 (+150-163 when STATS): compute_prior caches, compute_mugrads,
// compute_vargrads, two optim.adam calls (~45 pointwise launches, >= 13 host syncs)
//   -> one pass: 32 B read + 24 B written per weight (+ caches / operand copies).
struct AdamCoef { float step_mu, step_var; };

// The KL terms of a prior given by mu_hat and l0 = log var_hat (FIXED and PER_WEIGHT; k_update, k_grads), without a
// division.  The mean term (mu - mu_hat) / (B var_hat) applies exp(-l0) as two factors exp(-l0 / 2) after the 1/B scale,
// so it stays finite for l0 >= -177 wherever the exact value is representable; it is exactly 0 where mu == mu_hat for
// any l0 (no 0 * inf).  The log-variance term (var / var_hat - 1) / (2B) is exp(lvar - l0): exactly 0 where
// lvar == l0, finite whatever the two are when their difference is.
__device__ __forceinline__ float kl_mu(float d, float l0, float inv_B) {
  const float e = __expf(-0.5f * l0);
  return d == 0.f ? 0.f : d * inv_B * e * e;
}
__device__ __forceinline__ float kl_lvar(float lv, float l0, float inv_2B) { return (__expf(lv - l0) - 1.f) * inv_2B; }

// PK (enum vbnn_prior) selects where the prior N(mu_hat, var_hat) of the KL terms comes from:
//   EMPIRICAL   the reduction of the partials below (VBLinear.lua:81-86), the reference's arithmetic;
//   FIXED       p.prior.mu0 and l0 = p.prior.lvar0 = log var0, no reduction;
//   PER_WEIGHT  mu_hat, l0 read next to mu / lvar (+8 B per weight).
// FIXED and PER_WEIGHT share kl_mu / kl_lvar.
template <bool VEC, bool STATS, int TPB, int PK>
__global__ void __launch_bounds__(TPB, TPB == 128 ? 6 : 1) k_update(UpdateParams p) {
  __shared__ double sh[32];
  __shared__ float s_var_hat;
  __shared__ AdamCoef s_coef;
  __shared__ LiveOpts s_hp;             // the layer's hyper-parameters, read once per block
  // t for the epilogue's partials half: kept in shared memory, not in a register live across the main loop (the
  // 128-thread variant is at its 80-register cap)
  __shared__ int s_t;
  const int t_now = *p.t_dev;
  {
    LiveOpts hp;
    if (threadIdx.x == 0) hp = *p.hp;
    double r = 0.0;
    if (PK == VBNN_PRIOR_EMPIRICAL) {
      const double* part = p.partials + (p.partials_pingpong ? (size_t)(t_now & 1) * kMaxPartials : 0);
      double a = 0.0;
      for (int i = threadIdx.x; i < p.n_partials; i += blockDim.x) a += part[i];
      r = block_sum(a, sh);
    }
    if (threadIdx.x == 0) {
      if (PK == VBNN_PRIOR_EMPIRICAL) {
        const long long W = p.W_total > 0 ? p.W_total : (long long)p.O * p.I;
        float vh = (float)(r / (double)W);
        s_var_hat = vh;
        if (blockIdx.x == 0) *p.var_hat_dev = vh;
      } else {
        s_var_hat = 1.f;                                                // unused: kl_mu / kl_lvar
      }
      const int t = t_now + 1;                                          // state.t = state.t + 1
      s_t = t;
      double bc1 = 1.0 - pow((double)hp.beta1, (double)t);
      double bc2 = 1.0 - pow((double)hp.beta2, (double)t);
      s_coef.step_mu = (float)((double)hp.lr_mu * sqrt(bc2) / bc1);
      s_coef.step_var = (float)((double)hp.lr_var * sqrt(bc2) / bc1);
      s_hp = hp;
    }
    __syncthreads();
  }
  const float var_hat = s_var_hat;
  const float B = s_hp.B, eps = s_hp.eps;
  const float inv_S = 1.f / p.S, inv_BV = 1.f / (B * var_hat), inv_2B = 1.f / (2.f * B);
  const float inv_vh = 1.f / var_hat;
  const float b1 = s_hp.beta1, b2 = s_hp.beta2, omb1 = 1.f - s_hp.beta1, omb2 = 1.f - s_hp.beta2;

  float nxt = 0.f;                       // sigma_hat^2 numerator of the next minibatch
  double st[kStatSlots];
  if (STATS) {
#pragma unroll
    for (int i = 0; i < kStatSlots; ++i) st[i] = 0.0;
    st[11] = 3.0e38; st[12] = -3.0e38; st[13] = 3.0e38; st[14] = -3.0e38;
  }

  const int Q = (p.I + 3) >> 2;
  const long long quads = (long long)p.O * Q;
  for (long long qd = blockIdx.x * (long long)blockDim.x + threadIdx.x; qd < quads;
       qd += (long long)gridDim.x * blockDim.x) {
    const int o = (int)(qd / Q), c = (int)(qd - (long long)o * Q);
    const int i0 = c * 4;
    const long long e0 = (long long)o * p.I + i0;
    const int nv = VEC ? 4 : min(4, p.I - i0);
    float mu[4], lv[4], gw[4], gs[4], mm[4], vm[4], mv[4], vv[4];
    auto load = [&](const float* src, float (&d)[4]) {
      if (VEC) { float4 t = ld4(src + e0); d[0] = t.x; d[1] = t.y; d[2] = t.z; d[3] = t.w; }
      else {
#pragma unroll
        for (int j = 0; j < 4; ++j) d[j] = j < nv ? src[e0 + j] : 0.f;
      }
    };
    auto store = [&](float* dst, const float (&d)[4]) {
      if (VEC) st4(dst + e0, make_float4(d[0], d[1], d[2], d[3]));
      else
        for (int j = 0; j < nv; ++j) dst[e0 + j] = d[j];
    };
    load(p.mu, mu); load(p.lvar, lv);
    if (p.grads_bf16) {                                  // peer mode, bf16 gradient tiles on the wire (I % 4 == 0)
      const bf16* gWb = reinterpret_cast<const bf16*>(p.gW);
      const bf16* gSb = reinterpret_cast<const bf16*>(p.gS);
#pragma unroll
      for (int j = 0; j < 4; ++j) { gw[j] = 0.f; gs[j] = 0.f; }
      for (int src = 0; src < p.n_src; ++src) {
        const uint2 a = *reinterpret_cast<const uint2*>(gWb + src * p.src_stride + e0);
        const uint2 b = *reinterpret_cast<const uint2*>(gSb + src * p.src_stride + e0);
        gw[0] += __uint_as_float(a.x << 16); gw[1] += __uint_as_float(a.x & 0xFFFF0000u);
        gw[2] += __uint_as_float(a.y << 16); gw[3] += __uint_as_float(a.y & 0xFFFF0000u);
        gs[0] += __uint_as_float(b.x << 16); gs[1] += __uint_as_float(b.x & 0xFFFF0000u);
        gs[2] += __uint_as_float(b.y << 16); gs[3] += __uint_as_float(b.y & 0xFFFF0000u);
      }
    } else {
      load(p.gW, gw); load(p.gS, gs);
      for (int src = 1; src < p.n_src; ++src) {          // peer mode: sum the ranks' receive slots
        float a[4], b[4];
        load(p.gW + src * p.src_stride, a); load(p.gS + src * p.src_stride, b);
#pragma unroll
        for (int j = 0; j < 4; ++j) { gw[j] += a[j]; gs[j] += b[j]; }
      }
    }
    float sd_old[4], musq[4], s2_new[4];
    // FIXED / PER_WEIGHT: the KL terms are formed first (without STATS: added to the data terms in gw / gs).  The
    // co-resident variant (80 registers) also stores the caches and only then loads the Adam state, so that the prior
    // quads are dead by then; the others load the Adam state up front, as EMPIRICAL does, and keep every load in
    // flight at once.  EMPIRICAL keeps the parent's statements: they compile to the same instructions.
    constexpr bool kl_first = TPB == 128 && PK != VBNN_PRIOR_EMPIRICAL;
    if constexpr (!kl_first) { load(p.m_mu, mm); load(p.v_mu, vm); load(p.m_var, mv); load(p.v_var, vv); }
    float klm[4], klv[4], kvar[4];
    if constexpr (PK != VBNN_PRIOR_EMPIRICAL) {
      float pm[4], pl[4];
      if constexpr (PK == VBNN_PRIOR_PER_WEIGHT) { load(p.prior.mu, pm); load(p.prior.lvar, pl); }
      else {
#pragma unroll
        for (int j = 0; j < 4; ++j) { pm[j] = p.prior.mu0; pl[j] = p.prior.lvar0; }
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float var = __expf(lv[j]);                                // :78
        kvar[j] = var;
        sd_old[j] = sqrtf(var);                                         // :79
        const float dmu0 = mu[j] - pm[j];                               // mu - mu_hat, :81-82
        musq[j] = dmu0 * dmu0;
        klm[j] = kl_mu(dmu0, pl[j], 2.f * inv_2B);                      // :91; 2 * inv_2B == 1/B in fp32
        klv[j] = kl_lvar(lv[j], pl[j], inv_2B);                         // :96-97
        if (!STATS) {
          gw[j] = gw[j] * inv_S + klm[j];
          gs[j] = (p.lrt ? gs[j] * inv_S * var : gs[j] * (0.5f * inv_S) * sd_old[j]) + klv[j];
        }
      }
      if constexpr (kl_first) {
        if (p.stdv) store(p.stdv, sd_old);
        if (p.mu_sqe) store(p.mu_sqe, musq);
      }
    }
    if constexpr (kl_first) { load(p.m_mu, mm); load(p.v_mu, vm); load(p.m_var, mv); load(p.v_var, vv); }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float var = PK == VBNN_PRIOR_EMPIRICAL ? __expf(lv[j]) : kvar[j];   // :78
      const float sd = PK == VBNN_PRIOR_EMPIRICAL ? sqrtf(var) : sd_old[j];      // :79
      sd_old[j] = sd;
      if (PK == VBNN_PRIOR_EMPIRICAL) musq[j] = mu[j] * mu[j];          // :82
      const float mleg = gw[j] * inv_S;                                 // :92
      const float mlcg = PK == VBNN_PRIOR_EMPIRICAL ? mu[j] * inv_BV : klm[j];   // :91
      const float vleg = p.lrt ? gs[j] * inv_S * var : gs[j] * (0.5f * inv_S) * sd;   // :97 / A12
      // :96-97, (1/var_hat - 1/var) * var / (2B) without the division: var = __expf(lv) is 0 for lv < ln(FLT_MIN),
      // where the reference's form is inf * 0 = NaN and this one is the finite limit -1/(2B)
      const float vlcg = PK == VBNN_PRIOR_EMPIRICAL ? (var * inv_vh - 1.f) * inv_2B : klv[j];
      const bool folded = PK != VBNN_PRIOR_EMPIRICAL && !STATS;
      const float gmu = folded ? gw[j] : mleg + mlcg;                   // :132
      const float gvar = folded ? gs[j] : vleg + vlcg;                  // :134
      // optim.adam on means (:135-138)
      mm[j] = b1 * mm[j] + omb1 * gmu;
      vm[j] = b2 * vm[j] + omb2 * gmu * gmu;
      const float dmu = -s_coef.step_mu * mm[j] / (sqrtf(vm[j]) + eps);
      // optim.adam on lvars (:140-143)
      mv[j] = b1 * mv[j] + omb1 * gvar;
      vv[j] = b2 * vv[j] + omb2 * gvar * gvar;
      const float dlv = -s_coef.step_var * mv[j] / (sqrtf(vv[j]) + eps);
      mu[j] += dmu;
      lv[j] += dlv;
      s2_new[j] = __expf(lv[j]);
      if (j < nv) nxt += s2_new[j] + mu[j] * mu[j];
      if (STATS && j < nv) {
        st[0] += (double)vlcg * vlcg; st[1] += (double)vleg * vleg;
        st[2] += (double)mlcg * mlcg; st[3] += (double)mleg * mleg;
        st[4] += (double)lv[j] * lv[j]; st[5] += (double)mu[j] * mu[j];
        st[6] += (double)s2_new[j]; st[7] += (double)mu[j];
        st[8] += (double)dmu * dmu; st[9] += (double)dlv * dlv;
        st[11] = fmin(st[11], (double)s2_new[j]); st[12] = fmax(st[12], (double)s2_new[j]);
        st[13] = fmin(st[13], (double)mu[j]); st[14] = fmax(st[14], (double)mu[j]);
      }
    }
    store(p.mu, mu); store(p.lvar, lv);
    store(p.m_mu, mm); store(p.v_mu, vm); store(p.m_var, mv); store(p.v_var, vv);
    if (!kl_first && p.stdv) store(p.stdv, sd_old);
    if (!kl_first && p.mu_sqe) store(p.mu_sqe, musq);
    if (p.s2_f32) store(p.s2_f32, s2_new);
    if (p.mu_bf16) {
      bf16* d1 = p.mu_bf16 + (long long)o * p.ld_bf16 + i0;
      bf16* d2 = p.s2_bf16 + (long long)o * p.ld_bf16 + i0;
      if (nv == 4) {
        st4_bf16(d1, mu[0], mu[1], mu[2], mu[3]);
        st4_bf16(d2, s2_new[0], s2_new[1], s2_new[2], s2_new[3]);
      } else {
        for (int j = 0; j < nv; ++j) { d1[j] = __float2bfloat16_rn(mu[j]); d2[j] = __float2bfloat16_rn(s2_new[j]); }
      }
    }
    for (int q = 0; q < p.n_push; ++q) {                 // peer mode, layer 0: all-gather by NVLink stores
      if (p.push_mu[q]) store(p.push_mu[q], mu);
      if (p.push_lv[q]) store(p.push_lv[q], lv);
      if (p.push_s2[q]) store(p.push_s2[q], s2_new);
      if (p.push_mu16[q]) {
        bf16* d1 = p.push_mu16[q] + (long long)o * p.ld_bf16 + i0;
        bf16* d2 = p.push_s216[q] + (long long)o * p.ld_bf16 + i0;
        if (nv == 4) {
          st4_bf16(d1, mu[0], mu[1], mu[2], mu[3]);
          st4_bf16(d2, s2_new[0], s2_new[1], s2_new[2], s2_new[3]);
        } else {
          for (int j = 0; j < nv; ++j) { d1[j] = __float2bfloat16_rn(mu[j]); d2[j] = __float2bfloat16_rn(s2_new[j]); }
        }
      }
    }
  }
  if (p.n_push > 0 || p.n_peer > 0) __threadfence_system();   // peer stores of this thread are out before the flag kernel
  if (p.next_partials) {
    double r = block_sum((double)nxt, sh);
    if (threadIdx.x == 0) {
      const size_t idx = (p.partials_pingpong ? (size_t)(s_t & 1) * kMaxPartials : 0) + p.part_off + blockIdx.x;
      p.next_partials[idx] = r;
      for (int q = 0; q < p.n_peer; ++q) p.peer_partials[q][idx] = r;
      if (p.n_peer > 0) __threadfence_system();
    }
  }
  if (STATS) {
    // sums in slots 0..9, min/max in 11..14
#pragma unroll
    for (int i = 0; i < 10; ++i) {
      double r = block_sum(st[i], sh);
      if (threadIdx.x == 0) p.stat_partials[blockIdx.x * kStatSlots + i] = r;
    }
#pragma unroll
    for (int i = 11; i < 15; ++i) {
      const bool is_min = (i == 11 || i == 13);
      float v = (float)st[i];
      v = is_min ? warp_min(v) : warp_max(v);
      __shared__ float shf[32];
      __syncthreads();
      if ((threadIdx.x & 31) == 0) shf[threadIdx.x >> 5] = v;
      __syncthreads();
      if (threadIdx.x == 0) {
        float r = shf[0];
        for (int w = 1; w < (blockDim.x >> 5); ++w) r = is_min ? fminf(r, shf[w]) : fmaxf(r, shf[w]);
        p.stat_partials[blockIdx.x * kStatSlots + i] = (double)r;
      }
    }
  }
}

// ------------------------------------------------------------------ grads (API parity) ---
__global__ void __launch_bounds__(kThreads) k_grads(const float* mu, const float* lvar, float* gW,
                                                    float* gS, long long n, const float* var_hat_dev,
                                                    PriorArgs pr, const LiveOpts* hp, float S, int lrt,
                                                    float* mleg, float* mlcg, float* vleg, float* vlcg) {
  const float var_hat = *var_hat_dev;                                   // EMPIRICAL
  const float B = hp->B;
  const bool args = pr.kind != VBNN_PRIOR_EMPIRICAL;                    // mu_hat, l0 from pr: as k_update
  const bool do_mu = mleg || mlcg, do_var = vleg || vlcg;
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n;
       e += (long long)gridDim.x * blockDim.x) {
    const float var = __expf(lvar[e]), sd = sqrtf(var);
    const float l0 = pr.lvar ? pr.lvar[e] : pr.lvar0;
    if (do_mu) {
      const float a = gW[e] / S;                                        // :92 (in place)
      gW[e] = a;
      if (mleg) mleg[e] = a;
      if (mlcg) {                                                       // :91
        const float d = mu[e] - (pr.mu ? pr.mu[e] : pr.mu0);
        mlcg[e] = args ? kl_mu(d, l0, 1.f / B) : d / (B * var_hat);
      }
    }
    if (do_var) {
      const float b = lrt ? gS[e] / S * var : gS[e] / (2.f * S) * sd;   // :97 (in place)
      gS[e] = b;
      if (vleg) vleg[e] = b;
      if (vlcg)                                                         // :96-97, finite at var = 0 (k_update)
        vlcg[e] = args ? kl_lvar(lvar[e], l0, 1.f / (2.f * B)) : (var * (1.f / var_hat) - 1.f) / (2.f * B);
    }
  }
}

// ------------------------------------------------------------------ calc_lc -------------
__global__ void __launch_bounds__(kThreads) k_calc_lc(const float* var_src, int var_kind,
                                                      const float* mu_src, int mu_is_sq, long long n,
                                                      const float* var_hat_dev, PriorArgs pr, const LiveOpts* hp,
                                                      float* lc_out, double* partials) {
  __shared__ double sh[32];
  const float var_hat = *var_hat_dev;                                   // EMPIRICAL
  const float B = hp->B;
  const float log_sd_hat = 0.5f * logf(var_hat);
  const bool args = pr.kind != VBNN_PRIOR_EMPIRICAL;                    // mu_hat, l0 from pr
  double acc = 0.0;
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n;
       e += (long long)gridDim.x * blockDim.x) {
    float var, log_sd, sd = 0.f;
    if (var_kind == 0) { log_sd = 0.5f * var_src[e]; var = expf(var_src[e]); }
    else { sd = var_src[e]; var = sd * sd; log_sd = logf(sd); }
    float m = mu_src[e];
    float musq = m;
    if (!mu_is_sq) { const float d = m - (pr.mu ? pr.mu[e] : pr.mu0); musq = d * d; }
    float first, second;
    if (args) {
      // (l0 - log var) / 2 + ((mu - mu_hat)^2 e^-l0 + var e^-l0 - 1) / 2 with e^-l0 as two factors e^(-l0/2), as kl_mu:
      // finite at any representable l0 down to -177, and exactly 0 at a snapshot from the log-variances
      // (exp(lvar - l0) = 1, mu == mu_hat)
      const float l0 = pr.lvar ? pr.lvar[e] : pr.lvar0;
      const float eh = expf(-0.5f * l0);
      const float ratio = var_kind == 0 ? expf(var_src[e] - l0) : (sd * eh) * (sd * eh);
      first = 0.5f * l0 - log_sd;                                       // :100
      second = 0.5f * ((musq == 0.f ? 0.f : musq * eh * eh) + (ratio - 1.f));   // :101
    } else {
      first = -log_sd + log_sd_hat;                                     // :100
      second = (musq + (var - var_hat)) / (2.f * var_hat);              // :101
    }
    float lc = (first + second) * (1.f / B);                            // :102
    if (lc_out) lc_out[e] = lc;
    acc += (double)lc;
  }
  double r = block_sum(acc, sh);
  if (threadIdx.x == 0) partials[blockIdx.x] = r;
}

// ------------------------------------------------------------------ sgd -----------------
__global__ void __launch_bounds__(kThreads) k_sgd(float* x, const float* g, long long n, const float* lr_dev,
                                                  bf16* xb, int I, int ld) {
  const float lr = *lr_dev;
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n;
       e += (long long)gridDim.x * blockDim.x) {
    float v = x[e] - lr * g[e];
    x[e] = v;
    if (xb) {
      long long o = e / I;
      int i = (int)(e - o * I);
      xb[o * ld + i] = __float2bfloat16_rn(v);
    }
  }
}

// peer mode: the gradient is the sum of the ranks' receive slots
__global__ void __launch_bounds__(kThreads) k_sgd_slots(float* x, const float* g, int n_src, long long src_stride,
                                                        long long n, const float* lr_dev, bf16* xb, int I, int ld) {
  const float lr = *lr_dev;
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n;
       e += (long long)gridDim.x * blockDim.x) {
    float gs = 0.f;
    for (int s = 0; s < n_src; ++s) gs += g[e + s * src_stride];
    float v = x[e] - lr * gs;
    x[e] = v;
    if (xb) {
      long long o = e / I;
      int i = (int)(e - o * I);
      xb[o * ld + i] = __float2bfloat16_rn(v);
    }
  }
}

// ------------------------------------------------------------------ loss ----------------
// One warp per row: LogSoftMax + ClassNLL (size-averaged) forward and backward + argmax match.
// Replaces cunn LogSoftMax/ClassNLLCriterion kernels plus the host accuracy loop of
// utils.lua:11-27 (N device syncs per run()).
__global__ void __launch_bounds__(kThreads) k_loss(LossParams p) {
  const int warps_per_block = blockDim.x >> 5;
  const int lane = threadIdx.x & 31;
  const long long rows = (long long)p.Z * p.N;
  for (long long r0 = (long long)blockIdx.x * warps_per_block; r0 < rows;
       r0 += (long long)gridDim.x * warps_per_block) {
    const long long r = r0 + (threadIdx.x >> 5);
    float my_loss = 0.f, my_corr = 0.f;
    int z = 0;
    if (r < rows) {
      z = (int)(r / p.N);
      const int n = (int)(r - (long long)z * p.N);
      const float* x = p.logits + r * p.ld_logits;
      const int tgt = (int)p.targets[n] - 1;                            // 1-based (data.lua:16)
      float mx = -3.0e38f; int arg = 0x7fffffff;
      for (int c = lane; c < p.C; c += 32) {
        float v = x[c];
        if (v > mx) { mx = v; arg = c; }
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        float om = __shfl_xor_sync(0xffffffffu, mx, o);
        int oa = __shfl_xor_sync(0xffffffffu, arg, o);
        if (om > mx || (om == mx && oa < arg)) { mx = om; arg = oa; }
      }
      float se = 0.f;
      for (int c = lane; c < p.C; c += 32) se += __expf(x[c] - mx);
      se = warp_sum(se);
      const float lse = mx + __logf(se);
      for (int c = lane; c < p.C; c += 32) {
        const float lp = x[c] - lse;
        const float g = (__expf(lp) - (c == tgt ? 1.f : 0.f)) * p.grad_scale;
        if (p.g_f32) p.g_f32[r * p.ld_g + c] = g;
        if (p.g_bf16) p.g_bf16[r * p.ld_g + c] = __float2bfloat16_rn(g);
        if (p.logp_out) p.logp_out[r * p.C + c] = lp;
      }
      // zero the padding columns of G so the bf16 GEMMs read clean operands
      for (int c = p.C + lane; c < p.ld_g; c += 32) {
        if (p.g_f32) p.g_f32[r * p.ld_g + c] = 0.f;
        if (p.g_bf16) p.g_bf16[r * p.ld_g + c] = __float2bfloat16_rn(0.f);
      }
      if (lane == 0) {
        my_loss = (tgt >= 0 && tgt < p.C) ? -(x[tgt] - lse) : 0.f;
        my_corr = (arg == tgt) ? 1.f : 0.f;
      }
    }
    // One atomic pair per block instead of per row (8192 rows hammering two addresses serialised the
    // whole kernel): the rows of one block almost always share z; per-warp atomics otherwise.
    __shared__ float sh_loss[kThreads / 32], sh_corr[kThreads / 32];
    __shared__ int sh_z[kThreads / 32];
    const int w = threadIdx.x >> 5;
    if (lane == 0) { sh_loss[w] = my_loss; sh_corr[w] = my_corr; sh_z[w] = r < rows ? z : -1; }
    __syncthreads();
    if (threadIdx.x == 0) {
      int z0 = -1; bool same = true;
      for (int k = 0; k < warps_per_block; ++k) {
        if (sh_z[k] < 0) continue;
        if (z0 < 0) z0 = sh_z[k];
        same &= sh_z[k] == z0;
      }
      if (same && z0 >= 0) {
        float a = 0.f, c = 0.f;
        for (int k = 0; k < warps_per_block; ++k) if (sh_z[k] >= 0) { a += sh_loss[k]; c += sh_corr[k]; }
        atomicAdd(p.result + 2 * (p.z_slot0 + z0), a);
        atomicAdd(p.result + 2 * (p.z_slot0 + z0) + 1, c);
      } else {
        for (int k = 0; k < warps_per_block; ++k)
          if (sh_z[k] >= 0) {
            atomicAdd(p.result + 2 * (p.z_slot0 + sh_z[k]), sh_loss[k]);
            atomicAdd(p.result + 2 * (p.z_slot0 + sh_z[k]) + 1, sh_corr[k]);
          }
      }
    }
    __syncthreads();
  }
}

// ------------------------------------------------------------------ predict -------------
// acc - exp(lp) * lp: one entropy term.  The per-sample and the averaged entropy both use it, so that a
// one-sample average, whose log p-bar is bitwise logp, has a mutual information of exactly 0.
__device__ __forceinline__ float sub_plogp(float acc, float lp) { return acc - expf(lp) * lp; }

// One warp per row, like k_loss.  The warp folds the chunk's samples in order z = 0..zc-1 and every sum has a
// fixed order (no atomics), so two launches on the same logits give the same bits.
__global__ void __launch_bounds__(kThreads) k_predict(PredictParams p) {
  const int warps_per_block = blockDim.x >> 5;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const float log_t = logf((float)p.T);
  const bool reduce = p.last && p.targets;                              // block-uniform
  double blk_nll = 0.0, blk_corr = 0.0;                                 // thread 0: the block's rows in order
  __shared__ float sh_nll[kThreads / 32], sh_corr[kThreads / 32];
  for (long long r0 = (long long)blockIdx.x * warps_per_block; r0 < p.N;
       r0 += (long long)gridDim.x * warps_per_block) {
    const long long n = r0 + w;
    float my_nll = 0.f, my_corr = 0.f;
    if (n < p.N) {
      float* smax = p.st_max + n * p.C;
      float* ssum = p.st_sum + n * p.C;
      const int tgt = p.targets ? (int)p.targets[n] - 1 : -1;          // 1-based (data.lua:16)
      float ent = p.first ? 0.f : p.st_ent[n];
      float hbar = 0.f, best = -3.0e38f, nll = 0.f;
      int arg = 0x7fffffff;
      for (int z = 0; z < p.zc; ++z) {
        const float* x = p.logits + ((long long)z * p.N + n) * p.ld_logits;
        // lse formed exactly as k_loss forms it: logp_t is bitwise the LogSoftMax that get_outputs returns
        float mx = -3.0e38f;
        for (int c = lane; c < p.C; c += 32) mx = fmaxf(mx, x[c]);
        mx = warp_max(mx);
        float se = 0.f;
        for (int c = lane; c < p.C; c += 32) se += __expf(x[c] - mx);
        se = warp_sum(se);
        const float lse = mx + __logf(se);
        const bool init = p.first && z == 0, fin = p.last && z == p.zc - 1;
        float h = 0.f;
        for (int c = lane; c < p.C; c += 32) {
          const float lp = x[c] - lse;
          h = sub_plogp(h, lp);
          float m = lp, s = 1.f;
          if (!init) {
            m = smax[c]; s = ssum[c];
            if (lp > m) { s = s * expf(m - lp) + 1.f; m = lp; }
            else s += expf(lp - m);
          }
          if (!fin) { smax[c] = m; ssum[c] = s; continue; }
          const float lpb = (m + logf(s)) - log_t;                      // log p-bar(c | x)
          hbar = sub_plogp(hbar, lpb);
          if (lpb > best) { best = lpb; arg = c; }
          if (c == tgt) nll = -lpb;
          if (p.logp_out) p.logp_out[n * p.C + c] = lpb;
        }
        ent += warp_sum(h);
      }
      if (p.last) {
        hbar = warp_sum(hbar);
        nll = warp_sum(nll);                                            // one lane holds the target's term
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {                              // lowest index on ties, as k_loss
          float ob = __shfl_xor_sync(0xffffffffu, best, o);
          int oa = __shfl_xor_sync(0xffffffffu, arg, o);
          if (ob > best || (ob == best && oa < arg)) { best = ob; arg = oa; }
        }
        const float e = ent / (float)p.T;
        if (lane == 0 && p.unc_out) {
          float* u = p.unc_out + n * 4;
          u[0] = hbar; u[1] = e; u[2] = fmaxf(hbar - e, 0.f); u[3] = (float)(arg + 1);
        }
        if (lane == 0 && reduce) {
          my_nll = (tgt >= 0 && tgt < p.C) ? nll : 0.f;
          my_corr = arg == tgt ? 1.f : 0.f;
        }
      } else if (lane == 0) {
        p.st_ent[n] = ent;
      }
    }
    if (reduce) {
      if (lane == 0) { sh_nll[w] = my_nll; sh_corr[w] = my_corr; }
      __syncthreads();
      if (threadIdx.x == 0)
        for (int k = 0; k < warps_per_block; ++k) { blk_nll += sh_nll[k]; blk_corr += sh_corr[k]; }
      __syncthreads();
    }
  }
  if (reduce && threadIdx.x == 0) { p.partials[2 * blockIdx.x] = blk_nll; p.partials[2 * blockIdx.x + 1] = blk_corr; }
}

// Moments of the raw outputs over sampled forward passes (vbnn_mlp_predict_outputs).  One warp per row as in
// k_predict; lane l owns the output columns l, l + 32, ...  Per (row, mean column) the state is the first sample's
// value f0 and the sums of d = m_t - f0 and d^2: f0 is within the spread of the samples, so the variance formed from
// those sums does not cancel when |mean| >> spread (m_t - f0 is exact by Sterbenz wherever m_t and f0 are within a
// factor 2).  GAUSSIAN keeps sum_t exp(s_t) in the log-variance column's first state slot and, with targets, a
// per-row online log-sum-exp (running max, scaled sum) of l_t = sum_k log N(y_k; m_tk, e^{s_tk}).  Samples are
// folded in order and every sum has a fixed order, so the result depends neither on the chunking nor on the launch.
__global__ void __launch_bounds__(kThreads) k_predict_moments(MomentsParams p) {
  const int warps_per_block = blockDim.x >> 5;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int C = p.gaussian ? 2 * p.K : p.K;
  const float inv_t = 1.f / (float)p.T;
  const float half_log_2pi = 0.91893853320467274f;
  const bool reduce = p.last && p.partials;                             // block-uniform
  double blk_nll = 0.0, blk_se = 0.0;                                   // thread 0: the block's rows in order
  __shared__ float sh_nll[kThreads / 32], sh_se[kThreads / 32];
  for (long long r0 = (long long)blockIdx.x * warps_per_block; r0 < p.N;
       r0 += (long long)gridDim.x * warps_per_block) {
    const long long n = r0 + w;
    float my_nll = 0.f, my_se = 0.f;
    if (n < p.N) {
      float* s0 = p.st_f0 + n * C;
      float* s1 = p.st_sum + n * C;
      float* s2 = p.st_sq + n * C;
      const float* y = p.targets ? p.targets + n * p.K : nullptr;
      float lmax = 0.f, lsum = 0.f;
      if (p.lse && !p.first) { lmax = p.st_lmax[n]; lsum = p.st_lsum[n]; }
      float se = 0.f;
      for (int z = 0; z < p.zc; ++z) {
        const float* x = p.out + ((long long)z * p.N + n) * p.ld_out;
        const bool init = p.first && z == 0, fin = p.last && z == p.zc - 1;
        float ll = 0.f;                                                 // this lane's part of l_t
        for (int k = lane; k < p.K; k += 32) {
          const float m = x[k];
          float f0 = m, a = 0.f, b = 0.f;
          if (!init) {
            f0 = s0[k];
            const float d = m - f0;
            a = s1[k] + d;
            b = fmaf(d, d, s2[k]);
          }
          float sv = 0.f, ev = 0.f;
          if (p.gaussian) {
            sv = x[p.K + k];
            ev = expf(sv);
            if (!init) ev += s1[p.K + k];
            if (p.lse) {
              // log N formed in the log domain: (y - m)^2 e^{-s} as (d e^{-s/2})^2, 0 where y == m
              const float dy = y[k] - m;
              const float q = dy == 0.f ? 0.f : dy * expf(-0.5f * sv);
              ll -= half_log_2pi + 0.5f * (sv + q * q);
            }
          }
          if (!fin) {
            s0[k] = f0; s1[k] = a; s2[k] = b;
            if (p.gaussian) s1[p.K + k] = ev;
            continue;
          }
          const float mean = f0 + a * inv_t;
          if (p.mean_out) p.mean_out[n * p.K + k] = mean;
          if (p.epi_out) p.epi_out[n * p.K + k] = fmaxf((b - a * (a * inv_t)) * inv_t, 0.f);
          if (p.ale_out) p.ale_out[n * p.K + k] = ev * inv_t;
          if (reduce) { const float e = y[k] - mean; se = fmaf(e, e, se); }
        }
        if (p.lse) {
          ll = warp_sum(ll);
          // l_t = -inf (a density that underflows, (y - m)^2 e^{-s} beyond fp32) adds 0, not exp(-inf + inf) = NaN
          if (init) { lmax = ll; lsum = 1.f; }
          else if (ll > lmax) { lsum = lsum * expf(lmax - ll) + 1.f; lmax = ll; }
          else if (ll > -INFINITY) lsum += expf(ll - lmax);
        }
      }
      if (p.last) {
        if (reduce) {
          se = warp_sum(se);
          if (lane == 0) {
            my_se = se;
            my_nll = p.lse ? -((lmax + logf(lsum)) - logf((float)p.T)) : 0.f;
          }
        }
      } else if (p.lse && lane == 0) {
        p.st_lmax[n] = lmax; p.st_lsum[n] = lsum;
      }
    }
    if (reduce) {
      if (lane == 0) { sh_nll[w] = my_nll; sh_se[w] = my_se; }
      __syncthreads();
      if (threadIdx.x == 0)
        for (int k = 0; k < warps_per_block; ++k) { blk_nll += sh_nll[k]; blk_se += sh_se[k]; }
      __syncthreads();
    }
  }
  if (reduce && threadIdx.x == 0) { p.partials[2 * blockIdx.x] = blk_nll; p.partials[2 * blockIdx.x + 1] = blk_se; }
}

__global__ void k_finalize_result(const float* acc, int Z, int N, float* out2) {
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    float e = 0.f, a = 0.f;
    for (int z = 0; z < Z; ++z) {
      e += acc[2 * z] / (float)N;                                       // ClassNLL size-average
      a += acc[2 * z + 1] / (float)N * 100.f;                           // utils.lua:26
    }
    out2[0] = e / (float)Z;                                             // main.lua:39
    out2[1] = a / (float)Z;                                             // main.lua:38
  }
}

// ------------------------------------------------------------------ colsum --------------
template <typename T>
__global__ void __launch_bounds__(256) k_colsum(const T* G, long long rows, int cols, int ld,
                                                float scale, float* gb) {
  __shared__ float sh[8][33];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int col = blockIdx.x * 32 + tx;
  float acc = 0.f;
  if (col < cols)
    for (long long r = (long long)blockIdx.y * 8 + ty; r < rows; r += (long long)gridDim.y * 8)
      acc += to_f32(G[r * ld + col]);
  sh[ty][tx] = acc;
  __syncthreads();
  if (ty == 0 && col < cols) {
    float s = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) s += sh[k][tx];
    atomicAdd(gb + col, scale * s);
  }
}

// ------------------------------------------------------------------ staging -------------
__global__ void __launch_bounds__(kThreads) k_cast(const float* src, int src_ld, long long rows,
                                                   int cols, bf16* dst, bf16* dst_sq, int ld) {
  const int Q = ld >> 2;   // ld % 8 == 0; padding columns are written as zeros
  const long long quads = rows * Q;
  for (long long qd = blockIdx.x * (long long)blockDim.x + threadIdx.x; qd < quads;
       qd += (long long)gridDim.x * blockDim.x) {
    const long long r = qd / Q;
    const int c0 = (int)(qd - r * Q) * 4;
    float v[4];
    if (c0 + 3 < cols && (src_ld & 3) == 0) {
      float4 t = ld4(src + r * src_ld + c0);
      v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
    } else {
#pragma unroll
      for (int j = 0; j < 4; ++j) v[j] = (c0 + j < cols) ? src[r * src_ld + c0 + j] : 0.f;
    }
    st4_bf16(dst + r * ld + c0, v[0], v[1], v[2], v[3]);
    if (dst_sq) {
      // square what the GEMM will actually read (the bf16-rounded value)
      float w[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) { float b = __bfloat162float(__float2bfloat16_rn(v[j])); w[j] = b * b; }
      st4_bf16(dst_sq + r * ld + c0, w[0], w[1], w[2], w[3]);
    }
  }
}

// uint8 pixels -> normalised operands.  One thread = 8 consecutive columns (ld % 8 == 0): one 8-byte load when
// the row pitch allows it, one 16-byte bf16 store.
__global__ void __launch_bounds__(kThreads) k_cast_u8(const uint8_t* src, long long rows, int cols, float mean,
                                                      float inv_std, bf16* dst, bf16* dst_sq, int ld,
                                                      float* dst_f32, float* dst_sq_f32, int ld_f32) {
  const int ldw = dst ? ld : ld_f32;
  const int O = (ldw + 7) >> 3;
  const long long octs = rows * O;
  const bool vec = (cols & 7) == 0;
  for (long long od = blockIdx.x * (long long)blockDim.x + threadIdx.x; od < octs;
       od += (long long)gridDim.x * blockDim.x) {
    const long long r = od / O;
    const int c0 = (int)(od - r * O) * 8;
    uint8_t b[8];
    if (vec && c0 + 7 < cols) {
      const uint2 t = *reinterpret_cast<const uint2*>(src + r * cols + c0);
      *reinterpret_cast<uint2*>(b) = t;
    } else {
#pragma unroll
      for (int j = 0; j < 8; ++j) b[j] = c0 + j < cols ? src[r * cols + c0 + j] : 0;
    }
    float v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = c0 + j < cols ? ((float)b[j] - mean) * inv_std : 0.f;
    if (dst) {
      st4_bf16(dst + r * ld + c0, v[0], v[1], v[2], v[3]);
      st4_bf16(dst + r * ld + c0 + 4, v[4], v[5], v[6], v[7]);
      if (dst_sq) {
        float w[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) { const float q = __bfloat162float(__float2bfloat16_rn(v[j])); w[j] = q * q; }
        st4_bf16(dst_sq + r * ld + c0, w[0], w[1], w[2], w[3]);
        st4_bf16(dst_sq + r * ld + c0 + 4, w[4], w[5], w[6], w[7]);
      }
    } else {
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        if (c0 + j >= ld_f32) break;
        dst_f32[r * ld_f32 + c0 + j] = v[j];
        if (dst_sq_f32) dst_sq_f32[r * ld_f32 + c0 + j] = v[j] * v[j];
      }
    }
  }
}

__global__ void __launch_bounds__(kThreads) k_sum_partials(const float* __restrict__ src, int Z, long long stride, long long n,
                                                           float scale, int accumulate, float* dst) {
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x) {
    float a = 0.f;
    for (int z = 0; z < Z; ++z) a += src[z * stride + e];
    dst[e] = accumulate ? dst[e] + scale * a : scale * a;
  }
}

__global__ void __launch_bounds__(kThreads) k_square(const float* src, float* dst, long long n) {
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n;
       e += (long long)gridDim.x * blockDim.x) {
    float v = src[e];
    dst[e] = v * v;
  }
}

__global__ void __launch_bounds__(kThreads) k_param_copies(const float* mu, const float* lvar, int O,
                                                           int I, bf16* mu_b, bf16* s2_b, int ld,
                                                           float* s2_f32) {
  const long long n = (long long)O * I;
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n;
       e += (long long)gridDim.x * blockDim.x) {
    const long long o = e / I;
    const int i = (int)(e - o * I);
    const float s2 = __expf(lvar[e]);
    if (mu_b) mu_b[o * ld + i] = __float2bfloat16_rn(mu[e]);
    if (s2_b) s2_b[o * ld + i] = __float2bfloat16_rn(s2);
    if (s2_f32) s2_f32[e] = s2;
  }
}

template <typename TA, typename T>
__global__ void __launch_bounds__(kThreads) k_mul_act(const TA* a, int lda, const T* b, int ldb, T* out,
                                                      int ldo, long long rows, int cols) {
  const long long n = rows * cols;
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n;
       e += (long long)gridDim.x * blockDim.x) {
    const long long r = e / cols;
    const int c = (int)(e - r * cols);
    const float av = to_f32(from_f32<T>(to_f32(a[r * lda + c])));
    out[r * ldo + c] = from_f32<T>(av * to_f32(b[r * ldb + c]));
  }
}

// The caller's dL/dY (vbnn_mlp_backward_update) into the output layer's gradient operand: G = T(grad) over the
// padded width (the padding columns zeroed exactly as k_loss leaves them) and, for an LRT output layer, H = T(G .* R)
// as k_mul_act forms it from the stored G.  One thread per 4 columns: ld_g is a multiple of 8, so G / R / H quads are
// aligned for one vector access each; the caller's rows of C floats carry no alignment and are read per element.
template <typename T>
struct alignas(4 * sizeof(T)) Quad { T v[4]; };

template <typename T>
__global__ void __launch_bounds__(kThreads) k_grad_logits(const float* __restrict__ grad, long long rows, int C,
                                                          T* __restrict__ g, int ld_g, const T* __restrict__ r,
                                                          T* __restrict__ h) {
  const int qpr = ld_g >> 2;
  const long long n = rows * qpr;
  const bool narrow = n <= 0xFFFFFFFFll;                            // 32-bit index division where it fits
  for (long long q = blockIdx.x * (long long)blockDim.x + threadIdx.x; q < n; q += (long long)gridDim.x * blockDim.x) {
    const long long row = narrow ? (long long)((uint32_t)q / (uint32_t)qpr) : q / qpr;
    const int c0 = (int)(q - row * qpr) * 4;
    const float* src = grad + row * C;
    Quad<T> gq;
#pragma unroll
    for (int e = 0; e < 4; ++e) gq.v[e] = from_f32<T>(c0 + e < C ? src[c0 + e] : 0.f);
    const long long off = row * ld_g + c0;
    *reinterpret_cast<Quad<T>*>(g + off) = gq;
    if (r && c0 < C) {
      const Quad<T> rq = *reinterpret_cast<const Quad<T>*>(r + off);
      Quad<T> hq;
#pragma unroll
      for (int e = 0; e < 4; ++e) hq.v[e] = from_f32<T>(to_f32(gq.v[e]) * to_f32(rq.v[e]));
      if (c0 + 4 <= C) {
        *reinterpret_cast<Quad<T>*>(h + off) = hq;
      } else {
        for (int e = 0; c0 + e < C; ++e) h[off + e] = hq.v[e];      // H's padding is left as k_mul_act leaves it
      }
    }
  }
}

__global__ void __launch_bounds__(kThreads) k_fill(float* dst, long long n, float v) {
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n;
       e += (long long)gridDim.x * blockDim.x)
    dst[e] = v;
}

__global__ void k_set_live_opts(LiveOpts* dst, LiveOpts v) { *dst = v; }

__global__ void __launch_bounds__(kThreads) k_init_normal(float* dst, long long n, float mean,
                                                          float std, PhiloxStream ps) {
  const long long quads = (n + 3) >> 2;
  for (long long q = blockIdx.x * (long long)blockDim.x + threadIdx.x; q < quads;
       q += (long long)gridDim.x * blockDim.x) {
    float v[4];
    philox_normal4(ps, (uint32_t)q, v);
#pragma unroll
    for (int j = 0; j < 4; ++j)
      if (4 * q + j < n) dst[4 * q + j] = mean + std * v[j];
  }
}

__global__ void __launch_bounds__(kThreads) k_philox_matrix(float* dst, int rows, int cols, int row0,
                                                            PhiloxStream ps) {
  const int Q = (cols + 3) >> 2;
  const long long quads = (long long)rows * Q;
  for (long long qd = blockIdx.x * (long long)blockDim.x + threadIdx.x; qd < quads;
       qd += (long long)gridDim.x * blockDim.x) {
    const int r = (int)(qd / Q), c = (int)(qd - (long long)r * Q);
    float v[4];
    philox_normal4(ps, (uint32_t)(r + row0) * (uint32_t)Q + (uint32_t)c, v);
#pragma unroll
    for (int j = 0; j < 4; ++j)
      if (4 * c + j < cols) dst[(long long)r * cols + 4 * c + j] = v[j];
  }
}

__global__ void k_bump(uint32_t* step, int** t_ptrs, int n_t) {
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    if (step) *step += 1u;
    for (int i = 0; i < n_t; ++i) *t_ptrs[i] += 1;
  }
}

__global__ void __launch_bounds__(kThreads) k_snr(const float* mu, const float* lvar, long long n,
                                                  float thresh, uint8_t* mask,
                                                  unsigned long long* count) {
  unsigned long long c = 0;
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n;
       e += (long long)gridDim.x * blockDim.x) {
    const float snr = fabsf(mu[e]) / __expf(0.5f * lvar[e]);            // mainviz.lua:20-23
    const bool prune = snr < thresh;
    if (mask) mask[e] = prune ? 1 : 0;
    c += prune ? 1ull : 0ull;
  }
  for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
  if ((threadIdx.x & 31) == 0 && c) atomicAdd(count, c);
}

}  // namespace

// ------------------------------------------------------------------ launchers -----------
int launch_sample_w(const SampleParams& p, cudaStream_t st) {
  const long long quads = (long long)p.O * ((p.I + 3) / 4);
  // enough quads to fill the GPU: one thread draws all S samples of its quad; small layers spread the
  // samples over grid.y instead
  const int gx = grid_for(quads);
  dim3 grid(gx, gx >= kNumSMs * 4 ? 1 : p.S);
  if ((p.I & 3) == 0) k_sample_w<true><<<grid, kThreads, 0, st>>>(p);
  else k_sample_w<false><<<grid, kThreads, 0, st>>>(p);
  VB_CUDA(cudaGetLastError());
  return VBNN_OK;
}

int launch_prior_partials(const float* mu, const float* lvar, long long n, double* partials,
                          int* n_partials_out, cudaStream_t st) {
  int grid = grid_for((n + 3) / 4, 4);
  if (grid > kMaxPartials) grid = kMaxPartials;
  k_prior_partials<<<grid, kThreads, 0, st>>>(mu, lvar, n, partials, nullptr);
  VB_CUDA(cudaGetLastError());
  *n_partials_out = grid;
  return VBNN_OK;
}

int update_grid(int O, int I) {
  const long long quads = (long long)O * ((I + 3) / 4);
  int grid = grid_for(quads, knobs().upd_bps > 0 ? knobs().upd_bps : 4);
  return grid > kMaxPartials ? kMaxPartials : grid;
}

int launch_prior_partials_pp(const float* mu, const float* lvar, long long n, double* partials2,
                             const int* t_dev, int grid, cudaStream_t st) {
  k_prior_partials<<<grid, kThreads, 0, st>>>(mu, lvar, n, partials2, t_dev);
  VB_CUDA(cudaGetLastError());
  return VBNN_OK;
}

int launch_prior_finalize(const double* partials, int n_partials, long long W, float* var_hat_dev,
                          const float* mu, const float* lvar, float* stdv, float* mu_sqe, const PriorArgs& pr,
                          cudaStream_t st) {
  int grid = (stdv || mu_sqe) ? grid_for(W) : 1;
  k_prior_finalize<<<grid, kThreads, 0, st>>>(partials, n_partials, W, var_hat_dev, mu, lvar, stdv,
                                              mu_sqe, pr);
  VB_CUDA(cudaGetLastError());
  return VBNN_OK;
}

template <int PK>
static void launch_update_kind(const UpdateParams& p, int grid, cudaStream_t st) {
  const bool vec = (p.I & 3) == 0;
  const bool stats = p.stat_partials != nullptr;
  if (p.coresident && vec && !stats) k_update<true, false, 128, PK><<<grid, 128, 0, st>>>(p);
  else if (vec && stats) k_update<true, true, kThreads, PK><<<grid, kThreads, 0, st>>>(p);
  else if (vec) k_update<true, false, kThreads, PK><<<grid, kThreads, 0, st>>>(p);
  else if (stats) k_update<false, true, kThreads, PK><<<grid, kThreads, 0, st>>>(p);
  else k_update<false, false, kThreads, PK><<<grid, kThreads, 0, st>>>(p);
}

int launch_update(const UpdateParams& p, int* grid_out, cudaStream_t st) {
  const int grid = p.grid_override > 0 ? p.grid_override : update_grid(p.O, p.I);
  switch (p.prior.kind) {
    case VBNN_PRIOR_EMPIRICAL: launch_update_kind<VBNN_PRIOR_EMPIRICAL>(p, grid, st); break;
    case VBNN_PRIOR_FIXED: launch_update_kind<VBNN_PRIOR_FIXED>(p, grid, st); break;
    case VBNN_PRIOR_PER_WEIGHT: launch_update_kind<VBNN_PRIOR_PER_WEIGHT>(p, grid, st); break;
    default: set_error("launch_update: unknown prior kind %d", p.prior.kind); return VBNN_E_INVALID;
  }
  VB_CUDA(cudaGetLastError());
  if (grid_out) *grid_out = grid;
  return VBNN_OK;
}

int launch_grads(const float* mu, const float* lvar, float* gW, float* gS, long long n,
                 const float* var_hat_dev, const PriorArgs& pr, const LiveOpts* hp, float S, int lrt, float* mleg,
                 float* mlcg, float* vleg, float* vlcg, cudaStream_t st) {
  k_grads<<<grid_for(n), kThreads, 0, st>>>(mu, lvar, gW, gS, n, var_hat_dev, pr, hp, S, lrt, mleg, mlcg,
                                            vleg, vlcg);
  VB_CUDA(cudaGetLastError());
  return VBNN_OK;
}

int launch_calc_lc(const float* var_src, int var_kind, const float* mu_src, int mu_is_sq, long long n,
                   const float* var_hat_dev, const PriorArgs& pr, const LiveOpts* hp, float* lc_out, double* partials,
                   int* n_partials_out, cudaStream_t st) {
  int grid = grid_for(n, 4);
  if (grid > kMaxPartials) grid = kMaxPartials;
  k_calc_lc<<<grid, kThreads, 0, st>>>(var_src, var_kind, mu_src, mu_is_sq, n, var_hat_dev, pr, hp, lc_out,
                                       partials);
  VB_CUDA(cudaGetLastError());
  *n_partials_out = grid;
  return VBNN_OK;
}

int launch_sgd(float* x, const float* g, long long n, const float* lr, bf16* x_bf16, int I, int ld_bf16,
               cudaStream_t st) {
  if (n <= 0) return VBNN_OK;
  k_sgd<<<grid_for(n), kThreads, 0, st>>>(x, g, n, lr, x_bf16, I, ld_bf16);
  VB_CUDA(cudaGetLastError());
  return VBNN_OK;
}

int launch_sgd_slots(float* x, const float* g, int n_src, long long src_stride, long long n, const float* lr,
                     bf16* x_bf16, int I, int ld_bf16, cudaStream_t st) {
  if (n <= 0) return VBNN_OK;
  k_sgd_slots<<<grid_for(n), kThreads, 0, st>>>(x, g, n_src, src_stride, n, lr, x_bf16, I, ld_bf16);
  VB_CUDA(cudaGetLastError());
  return VBNN_OK;
}

int launch_loss(const LossParams& p, cudaStream_t st) {
  const long long rows = (long long)p.Z * p.N;
  const int wpb = kThreads / 32;
  long long blocks = (rows + wpb - 1) / wpb;
  if (blocks > kNumSMs * 8) blocks = kNumSMs * 8;
  k_loss<<<(int)blocks, kThreads, 0, st>>>(p);
  VB_CUDA(cudaGetLastError());
  return VBNN_OK;
}

int launch_predict(const PredictParams& p, int* grid_out, cudaStream_t st) {
  const int wpb = kThreads / 32;
  long long blocks = ((long long)p.N + wpb - 1) / wpb;
  if (blocks > kMaxPartials) blocks = kMaxPartials;
  k_predict<<<(int)blocks, kThreads, 0, st>>>(p);
  VB_CUDA(cudaGetLastError());
  if (grid_out) *grid_out = (int)blocks;
  return VBNN_OK;
}

int launch_predict_moments(const MomentsParams& p, int* grid_out, cudaStream_t st) {
  const int wpb = kThreads / 32;
  long long blocks = ((long long)p.N + wpb - 1) / wpb;
  if (blocks > kMaxPartials) blocks = kMaxPartials;
  k_predict_moments<<<(int)blocks, kThreads, 0, st>>>(p);
  VB_CUDA(cudaGetLastError());
  if (grid_out) *grid_out = (int)blocks;
  return VBNN_OK;
}

int launch_grad_logits(const float* grad, long long rows, int C, void* g, int ld_g, const void* r, void* h, int is_bf16,
                       cudaStream_t st) {
  const int grid = grid_for(rows * (ld_g / 4));
  if (is_bf16)
    k_grad_logits<bf16><<<grid, kThreads, 0, st>>>(grad, rows, C, (bf16*)g, ld_g, (const bf16*)r, (bf16*)h);
  else
    k_grad_logits<float><<<grid, kThreads, 0, st>>>(grad, rows, C, (float*)g, ld_g, (const float*)r, (float*)h);
  VB_CUDA(cudaGetLastError());
  return VBNN_OK;
}

int launch_finalize_result(const float* acc, int Z, int N, float* out2, cudaStream_t st) {
  k_finalize_result<<<1, 32, 0, st>>>(acc, Z, N, out2);
  VB_CUDA(cudaGetLastError());
  return VBNN_OK;
}

// bf16 rows with 16-byte pitch: one thread owns 8 consecutive columns (one 16-byte load per row), a
// warp covers 512 contiguous bytes of a row, a block 8 rows per iteration
__global__ void __launch_bounds__(256) k_colsum_bf16x8(const bf16* G, long long rows, int cols, int ld, float scale,
                                                        float* gb) {
  __shared__ float sh[8][32][9];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int col0 = (blockIdx.x * 32 + tx) * 8;
  float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  if (col0 < ld) {
    for (long long r = (long long)blockIdx.y * 8 + ty; r < rows; r += (long long)gridDim.y * 8) {
      const uint4 v = *reinterpret_cast<const uint4*>(G + r * ld + col0);
      const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        acc[2 * k] += __uint_as_float(w[k] << 16);
        acc[2 * k + 1] += __uint_as_float(w[k] & 0xFFFF0000u);
      }
    }
  }
#pragma unroll
  for (int k = 0; k < 8; ++k) sh[ty][tx][k] = acc[k];
  __syncthreads();
  // 256 threads reduce the 8 row-groups of the block's 256 columns
  const int c = threadIdx.x;
  float s = 0.f;
#pragma unroll
  for (int g = 0; g < 8; ++g) s += sh[g][c >> 3][c & 7];
  const int col = blockIdx.x * 256 + c;
  if (col < cols) atomicAdd(gb + col, scale * s);
}

int launch_colsum(const void* G, int is_bf16, long long rows, int cols, int ld, float scale, float* gb,
                  cudaStream_t st) {
  if (is_bf16 && (ld & 7) == 0 && (reinterpret_cast<uintptr_t>(G) & 15) == 0 && cols >= 256) {
    long long ry = (rows + 63) / 64;
    if (ry < 1) ry = 1;
    const int gx = ceil_div(cols, 256);
    const long long cap = (long long)kNumSMs * 4 / gx > 1 ? (long long)kNumSMs * 4 / gx : 1;
    if (ry > cap) ry = cap;
    k_colsum_bf16x8<<<dim3(gx, (int)ry), 256, 0, st>>>((const bf16*)G, rows, cols, ld, scale, gb);
    VB_CUDA(cudaGetLastError());
    return VBNN_OK;
  }
  long long ry = (rows + 255) / 256;
  if (ry < 1) ry = 1;
  if (ry > 64) ry = 64;
  dim3 grid(ceil_div(cols, 32), (int)ry);
  if (is_bf16) k_colsum<bf16><<<grid, 256, 0, st>>>((const bf16*)G, rows, cols, ld, scale, gb);
  else k_colsum<float><<<grid, 256, 0, st>>>((const float*)G, rows, cols, ld, scale, gb);
  VB_CUDA(cudaGetLastError());
  return VBNN_OK;
}

int launch_cast(const float* src, int src_ld, long long rows, int cols, bf16* dst, bf16* dst_sq, int ld,
                cudaStream_t st) {
  k_cast<<<grid_for(rows * (ld / 4)), kThreads, 0, st>>>(src, src_ld, rows, cols, dst, dst_sq, ld);
  VB_CUDA(cudaGetLastError());
  return VBNN_OK;
}

int launch_cast_u8(const uint8_t* src, long long rows, int cols, float mean, float inv_std, bf16* dst, bf16* dst_sq,
                   int ld, float* dst_f32, float* dst_sq_f32, int ld_f32, cudaStream_t st) {
  const int ldw = dst ? ld : ld_f32;
  k_cast_u8<<<grid_for(rows * ((ldw + 7) / 8)), kThreads, 0, st>>>(src, rows, cols, mean, inv_std, dst, dst_sq, ld,
                                                                  dst_f32, dst_sq_f32, ld_f32);
  VB_CUDA(cudaGetLastError());
  return VBNN_OK;
}

int launch_sum_partials(const float* src, int Z, long long stride, long long n, float scale, int accumulate, float* dst,
                        cudaStream_t st) {
  k_sum_partials<<<grid_for(n), kThreads, 0, st>>>(src, Z, stride, n, scale, accumulate, dst);
  VB_CUDA(cudaGetLastError());
  return VBNN_OK;
}

int launch_square(const float* src, float* dst, long long n, cudaStream_t st) {
  k_square<<<grid_for(n), kThreads, 0, st>>>(src, dst, n);
  VB_CUDA(cudaGetLastError());
  return VBNN_OK;
}

int launch_param_copies(const float* mu, const float* lvar, int O, int I, bf16* mu_bf16, bf16* s2_bf16,
                        int ld, float* s2_f32, cudaStream_t st) {
  k_param_copies<<<grid_for((long long)O * I), kThreads, 0, st>>>(mu, lvar, O, I, mu_bf16, s2_bf16, ld,
                                                                 s2_f32);
  VB_CUDA(cudaGetLastError());
  return VBNN_OK;
}

int launch_mul_act(const void* a, int lda, int a_is_bf16, const void* b, int ldb, void* out, int ldo,
                   long long rows, int cols, int is_bf16, cudaStream_t st) {
  const int grid = grid_for(rows * cols);
  if (is_bf16 && a_is_bf16)
    k_mul_act<bf16, bf16><<<grid, kThreads, 0, st>>>((const bf16*)a, lda, (const bf16*)b, ldb, (bf16*)out, ldo, rows, cols);
  else if (is_bf16)
    k_mul_act<float, bf16><<<grid, kThreads, 0, st>>>((const float*)a, lda, (const bf16*)b, ldb, (bf16*)out, ldo, rows, cols);
  else
    k_mul_act<float, float><<<grid, kThreads, 0, st>>>((const float*)a, lda, (const float*)b, ldb, (float*)out, ldo, rows, cols);
  VB_CUDA(cudaGetLastError());
  return VBNN_OK;
}

int launch_fill(float* dst, long long n, float v, cudaStream_t st) {
  if (n <= 0) return VBNN_OK;
  k_fill<<<grid_for(n), kThreads, 0, st>>>(dst, n, v);
  VB_CUDA(cudaGetLastError());
  return VBNN_OK;
}

int launch_set_live_opts(LiveOpts* dst, const LiveOpts& v, cudaStream_t st) {
  k_set_live_opts<<<1, 1, 0, st>>>(dst, v);
  VB_CUDA(cudaGetLastError());
  return VBNN_OK;
}

int launch_init_normal(float* dst, long long n, float mean, float std, PhiloxStream ps,
                       cudaStream_t st) {
  k_init_normal<<<grid_for((n + 3) / 4), kThreads, 0, st>>>(dst, n, mean, std, ps);
  VB_CUDA(cudaGetLastError());
  return VBNN_OK;
}

int launch_philox_matrix(float* dst, int rows, int cols, int row0, PhiloxStream ps, cudaStream_t st) {
  k_philox_matrix<<<grid_for((long long)rows * ((cols + 3) / 4)), kThreads, 0, st>>>(dst, rows, cols,
                                                                                   row0, ps);
  VB_CUDA(cudaGetLastError());
  return VBNN_OK;
}

int launch_bump(uint32_t* step, int** t_ptrs_dev, int n_t, cudaStream_t st) {
  k_bump<<<1, 32, 0, st>>>(step, t_ptrs_dev, n_t);
  VB_CUDA(cudaGetLastError());
  return VBNN_OK;
}

int launch_snr(const float* mu, const float* lvar, long long n, float thresh, uint8_t* mask,
               unsigned long long* count_dev, cudaStream_t st) {
  k_snr<<<grid_for(n), kThreads, 0, st>>>(mu, lvar, n, thresh, mask, count_dev);
  VB_CUDA(cudaGetLastError());
  return VBNN_OK;
}

}  // namespace vbnn
