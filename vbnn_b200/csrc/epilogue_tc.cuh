// epilogue_tc.cuh -- coalesced I/O for the tcgen05 kernel's fused epilogues.
//
// tcgen05.ld hands every epilogue thread ONE accumulator row (32 consecutive columns).  Writing
// that straight to global memory makes each warp store touch 32 different rows with 8-16 bytes
// each: partial-sector writes that L2 must read-modify-write (ncu r01b: dw_lrt read 0.70 GB from
// DRAM for a 256 MB problem).  Here every tensor the epilogue reads or writes goes through a
// per-warp 32x32 staging tile in shared memory (16-byte pieces, XOR-swizzled, conflict-free), so
// that global accesses are full 64-128 B row segments: thread = row for the math, thread = piece
// for the memory traffic.  The math is the same as epilogue.cuh (shared with the fp32 kernel).
#pragma once
#include "epilogue.cuh"

namespace vbnn {

constexpr int kStageBytes = 4096;   // per epilogue warp: 32 rows x 32 fp32

// physical byte offset of 16-byte piece `piece` of row `row`; P = pieces per row (4: bf16, 8: fp32)
template <int P>
__device__ __forceinline__ uint32_t stage_off(int row, int piece) {
  if constexpr (P == 8) return (uint32_t)(row * 128 + ((piece ^ (row & 7)) << 4));
  else return (uint32_t)(row * 64 + ((piece ^ ((row >> 1) & 3)) << 4));
}
__device__ __forceinline__ void sts128(uint32_t addr, uint4 v) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ uint4 lds128(uint32_t addr) {
  uint4 v;
  asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr) : "memory");
  return v;
}
__device__ __forceinline__ uint32_t pack_bf16(float a, float b) {
  __nv_bfloat162 t = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&t);
}
__device__ __forceinline__ uint32_t bf16x2_square(uint32_t w) {
  const __nv_bfloat162 t = *reinterpret_cast<const __nv_bfloat162*>(&w);
  const __nv_bfloat162 r = __hmul2(t, t);
  return *reinterpret_cast<const uint32_t*>(&r);
}
__device__ __forceinline__ float bf16_lo(uint32_t w) { return __uint_as_float(w << 16); }
__device__ __forceinline__ float bf16_hi(uint32_t w) { return __uint_as_float(w & 0xFFFF0000u); }

// ---- row-owner side: this thread's 32 values <-> its row of the staging tile ----
__device__ __forceinline__ void stage_put_bf16(uint32_t stage, int lane, const uint32_t (&w)[16]) {
#pragma unroll
  for (int pc = 0; pc < 4; ++pc)
    sts128(stage + stage_off<4>(lane, pc), make_uint4(w[4 * pc], w[4 * pc + 1], w[4 * pc + 2], w[4 * pc + 3]));
}
__device__ __forceinline__ void stage_put_f32(uint32_t stage, int lane, const float (&v)[32]) {
#pragma unroll
  for (int pc = 0; pc < 8; ++pc)
    sts128(stage + stage_off<8>(lane, pc),
           make_uint4(__float_as_uint(v[4 * pc]), __float_as_uint(v[4 * pc + 1]), __float_as_uint(v[4 * pc + 2]),
                      __float_as_uint(v[4 * pc + 3])));
}
__device__ __forceinline__ void stage_get_bf16(uint32_t stage, int lane, uint32_t (&w)[16]) {
#pragma unroll
  for (int pc = 0; pc < 4; ++pc) {
    uint4 t = lds128(stage + stage_off<4>(lane, pc));
    w[4 * pc] = t.x; w[4 * pc + 1] = t.y; w[4 * pc + 2] = t.z; w[4 * pc + 3] = t.w;
  }
}
__device__ __forceinline__ void stage_get_f32(uint32_t stage, int lane, float (&v)[32]) {
#pragma unroll
  for (int pc = 0; pc < 8; ++pc) {
    uint4 t = lds128(stage + stage_off<8>(lane, pc));
    v[4 * pc] = __uint_as_float(t.x); v[4 * pc + 1] = __uint_as_float(t.y);
    v[4 * pc + 2] = __uint_as_float(t.z); v[4 * pc + 3] = __uint_as_float(t.w);
  }
}

// ---- memory side: the 32 x (P*16 B) tile <-> global, 16-byte piece per lane, row segments contiguous
// g points at element (row 0 of the tile, first column of the chunk); ld_bytes = row pitch.
template <int P>
__device__ __forceinline__ void stage_to_global(uint32_t stage, int lane, char* g, long long ld_bytes, int rows_valid) {
#pragma unroll
  for (int it = 0; it < P; ++it) {
    const int idx = it * 32 + lane, row = idx / P, pc = idx % P;
    const uint4 v = lds128(stage + stage_off<P>(row, pc));
    // streaming store (evict-first): epilogue outputs are not re-read by this kernel; keeping them out of the way
    // leaves L2 to the operand tiles the CTAs in flight share (ncu r01e: dx-lrt / dw-lrt moved 1.9x their
    // algorithmic DRAM bytes, the excess being operand tiles evicted by output write-allocates)
    if (row < rows_valid) __stcs(reinterpret_cast<uint4*>(g + row * ld_bytes + pc * 16), v);
  }
}
template <int P>
__device__ __forceinline__ void global_to_stage(uint32_t stage, int lane, const char* g, long long ld_bytes, int rows_valid) {
  uint4 v[P];
#pragma unroll
  for (int it = 0; it < P; ++it) {
    const int idx = it * 32 + lane, row = idx / P, pc = idx % P;
    v[it] = row < rows_valid ? __ldcs(reinterpret_cast<const uint4*>(g + row * ld_bytes + pc * 16)) : make_uint4(0, 0, 0, 0);
  }
#pragma unroll
  for (int it = 0; it < P; ++it) {
    const int idx = it * 32 + lane, row = idx / P, pc = idx % P;
    sts128(stage + stage_off<P>(row, pc), v[it]);
  }
}

// write this thread's row of 32 bf16 (packed) / fp32 values to a [rows x ld] global tensor, coalesced
__device__ __forceinline__ void put_tile_bf16(uint32_t stage, int lane, bf16* g, long long ld, int rows_valid,
                                              const uint32_t (&w)[16]) {
  __syncwarp();
  stage_put_bf16(stage, lane, w);
  __syncwarp();
  stage_to_global<4>(stage, lane, reinterpret_cast<char*>(g), ld * 2, rows_valid);
}
__device__ __forceinline__ void put_tile_f32(uint32_t stage, int lane, float* g, long long ld, int rows_valid,
                                             const float (&v)[32]) {
  __syncwarp();
  stage_put_f32(stage, lane, v);
  __syncwarp();
  stage_to_global<8>(stage, lane, reinterpret_cast<char*>(g), ld * 4, rows_valid);
}
__device__ __forceinline__ void get_tile_bf16(uint32_t stage, int lane, const bf16* g, long long ld, int rows_valid,
                                              uint32_t (&w)[16]) {
  __syncwarp();
  global_to_stage<4>(stage, lane, reinterpret_cast<const char*>(g), ld * 2, rows_valid);
  __syncwarp();
  stage_get_bf16(stage, lane, w);
}
__device__ __forceinline__ void get_tile_f32(uint32_t stage, int lane, const float* g, long long ld, int rows_valid,
                                             float (&v)[32]) {
  __syncwarp();
  global_to_stage<8>(stage, lane, reinterpret_cast<const char*>(g), ld * 4, rows_valid);
  __syncwarp();
  stage_get_f32(stage, lane, v);
}

// Host-side predicate: every tensor this mode touches has 16-byte aligned rows, so the staged path
// applies (otherwise the kernel uses epi_quad's direct path; ragged right-edge chunks always do).
inline bool epi_can_stage(int mode, const EpiParams& p) {
  auto ok_act = [&](const void* ptr, int ld) { return ptr == nullptr || ((ld % 8) == 0 && (reinterpret_cast<uintptr_t>(ptr) % 16) == 0); };
  auto ok_f32 = [&](const void* ptr, int ld) { return ptr == nullptr || ((ld % 4) == 0 && (reinterpret_cast<uintptr_t>(ptr) % 16) == 0); };
  if (p.noise != nullptr) return false;                       // injected-noise parity mode: direct path
  if (!ok_f32(p.out_f32, p.ld_f32) || (p.zs_f32 % 4) != 0) return false;
  if (!ok_act(p.out_act, p.ld_act) || !ok_act(p.out_act2, p.ld_act) || !ok_act(p.r_out, p.ld_act) || (p.zs_act % 8) != 0) return false;
  if (!ok_act(p.xprev, p.ld_x) || !ok_act(p.rprev, p.ld_x) || (p.zs_x % 8) != 0) return false;
  if (p.grads_bf16 && (p.ld_g % 8) != 0) return false;
  if (!ok_f32(p.gW, p.ld_g) || !ok_f32(p.gS, p.ld_g)) return false;
  if (!ok_f32(p.aux, p.ld_aux) || (p.zs_aux % 4) != 0) return false;
  if (!ok_act(p.eps16, p.ld_e16) || (p.zs_e16 % 8) != 0) return false;
  if (p.scatter_rows)
    for (int q = 0; q < 8; ++q)
      if (!ok_f32(p.gW_peer[q], p.ld_g) || !ok_f32(p.gS_peer[q], p.ld_g)) return false;
  if (p.bias != nullptr && (reinterpret_cast<uintptr_t>(p.bias) % 16) != 0) return false;
  (void)mode;
  return true;
}

// One full 32-column chunk of one warp (rows row0 .. row0+31, columns col0 .. col0+31 all < N).
// v1 / v2: this thread's accumulator row (lane = row).  AT = bf16.
template <int MODE>
__device__ __forceinline__ void epi_chunk_staged(const EpiParams& p, const PhiloxStream& ps0, int z, int row0, int lane,
                                                 int col0, const float (&v1)[32], const float (&v2)[32], uint32_t stage) {
  const int rows_valid = min(32, p.M - row0);        // <= 0 never happens: the caller skips such warps
  const int row = row0 + lane;
  if constexpr (MODE == EPI_FWD_LRT2 || MODE == EPI_DX_LRT2) {
    // split LRT: the other product comes from global memory (coalesced through the staging tile)
    float o[32];
    get_tile_f32(stage, lane, p.aux + z * p.zs_aux + (long long)row0 * p.ld_aux + col0, p.ld_aux, rows_valid, o);
    if constexpr (MODE == EPI_FWD_LRT2) epi_chunk_staged<EPI_FWD_LRT>(p, ps0, z, row0, lane, col0, o, v1, stage);
    else epi_chunk_staged<EPI_DX_LRT>(p, ps0, z, row0, lane, col0, v1, o, stage);
    return;
  }
  if constexpr (MODE == EPI_STORE) {
    put_tile_f32(stage, lane, p.out_f32 + z * p.zs_f32 + (long long)row0 * p.ld_f32 + col0, p.ld_f32, rows_valid, v1);
  } else if constexpr (MODE == EPI_FWD) {
    float y[32];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      float b[4];
      load_bias4(p.bias, col0 + 4 * j, 4, b);
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        float t = v1[4 * j + e] + b[e];
        y[4 * j + e] = p.relu ? fmaxf(t, 0.f) : t;
      }
    }
    if (p.out_f32)
      put_tile_f32(stage, lane, p.out_f32 + z * p.zs_f32 + (long long)row0 * p.ld_f32 + col0, p.ld_f32, rows_valid, y);
    if (p.out_act) {
      uint32_t w[16];
#pragma unroll
      for (int j = 0; j < 16; ++j) w[j] = pack_bf16(y[2 * j], y[2 * j + 1]);
      put_tile_bf16(stage, lane, (bf16*)p.out_act + z * p.zs_act + (long long)row0 * p.ld_act + col0, p.ld_act, rows_valid, w);
    }
  } else if constexpr (MODE == EPI_FWD_LRT) {
    PhiloxStream ps = ps0;
    ps.sample += (uint32_t)z;
    const uint32_t q = (uint32_t)((p.N + 3) >> 2);
    uint32_t wa[16], w2[16], wr[16];
    float yf[32];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      float zt[4], b[4];
      philox_normal4(ps, (uint32_t)(row + p.row0) * q + (uint32_t)((col0 >> 2) + j), zt);
      load_bias4(p.bias, col0 + 4 * j, 4, b);
      float ya[4], rr[4];
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const float v = v2[4 * j + e];
        const float rs = lrt_rsqrt(v);
        const float y = v1[4 * j + e] + b[e] + (v * rs) * zt[e];
        yf[4 * j + e] = y;
        ya[e] = p.relu ? fmaxf(y, 0.f) : y;
        rr[e] = 0.5f * zt[e] * rs;
      }
      wa[2 * j] = pack_bf16(ya[0], ya[1]); wa[2 * j + 1] = pack_bf16(ya[2], ya[3]);
      wr[2 * j] = pack_bf16(rr[0], rr[1]); wr[2 * j + 1] = pack_bf16(rr[2], rr[3]);
      // square the value the next layer will actually read (the bf16-rounded activation): one packed bf16 multiply
      // per pair -- the exact product of two bf16 fits fp32, so rounding it once to bf16 (HMUL2.BF16) equals the
      // unpack / FMUL / pack sequence bit for bit
      w2[2 * j] = bf16x2_square(wa[2 * j]); w2[2 * j + 1] = bf16x2_square(wa[2 * j + 1]);
    }
    const long long off = z * p.zs_act + (long long)row0 * p.ld_act + col0;
    if (p.out_f32)
      put_tile_f32(stage, lane, p.out_f32 + z * p.zs_f32 + (long long)row0 * p.ld_f32 + col0, p.ld_f32, rows_valid, yf);
    if (p.out_act) put_tile_bf16(stage, lane, (bf16*)p.out_act + off, p.ld_act, rows_valid, wa);
    if (p.out_act2) put_tile_bf16(stage, lane, (bf16*)p.out_act2 + off, p.ld_act, rows_valid, w2);
    if (p.r_out) put_tile_bf16(stage, lane, (bf16*)p.r_out + off, p.ld_act, rows_valid, wr);
  } else if constexpr (MODE == EPI_DX || MODE == EPI_DX_LRT) {
    const long long xoff = z * p.zs_x + (long long)row0 * p.ld_x + col0;
    uint32_t wx[16];
    const bool need_x = p.xprev != nullptr && (p.mask || MODE == EPI_DX_LRT);
    if (need_x) get_tile_bf16(stage, lane, (const bf16*)p.xprev + xoff, p.ld_x, rows_valid, wx);
    float g[32];
#pragma unroll
    for (int j = 0; j < 16; ++j) {
      const float x0 = need_x ? bf16_lo(wx[j]) : 0.f, x1 = need_x ? bf16_hi(wx[j]) : 0.f;
      float g0 = v1[2 * j], g1 = v1[2 * j + 1];
      if constexpr (MODE == EPI_DX_LRT) { g0 += 2.f * x0 * v2[2 * j]; g1 += 2.f * x1 * v2[2 * j + 1]; }
      if (p.mask) { g0 = x0 > 0.f ? g0 : 0.f; g1 = x1 > 0.f ? g1 : 0.f; }
      g[2 * j] = g0; g[2 * j + 1] = g1;
    }
    if (p.out_f32)
      put_tile_f32(stage, lane, p.out_f32 + z * p.zs_f32 + (long long)row0 * p.ld_f32 + col0, p.ld_f32, rows_valid, g);
    const long long off = z * p.zs_act + (long long)row0 * p.ld_act + col0;
    uint32_t wg[16];
#pragma unroll
    for (int j = 0; j < 16; ++j) wg[j] = pack_bf16(g[2 * j], g[2 * j + 1]);
    if (p.out_act) put_tile_bf16(stage, lane, (bf16*)p.out_act + off, p.ld_act, rows_valid, wg);
    if (p.out_act2 && p.rprev) {
      uint32_t wr[16];
      get_tile_bf16(stage, lane, (const bf16*)p.rprev + xoff, p.ld_x, rows_valid, wr);
#pragma unroll
      for (int j = 0; j < 16; ++j)
        wr[j] = pack_bf16(bf16_lo(wg[j]) * bf16_lo(wr[j]), bf16_hi(wg[j]) * bf16_hi(wr[j]));
      put_tile_bf16(stage, lane, (bf16*)p.out_act2 + off, p.ld_act, rows_valid, wr);
    }
  } else if constexpr (MODE == EPI_DW || MODE == EPI_DW_LRT) {
    const long long goff = (long long)row0 * p.ld_g + col0;
    const bool acc = p.accumulate || z > 0;
    float *gWd, *gSd;
    dw_dest(p, row0, gWd, gSd);
    if (p.grads_bf16) {                                   // write-once bf16 tiles (LRT, one sample)
      uint32_t w[16];
#pragma unroll
      for (int j = 0; j < 16; ++j) w[j] = pack_bf16(p.scale * v1[2 * j], p.scale * v1[2 * j + 1]);
      put_tile_bf16(stage, lane, reinterpret_cast<bf16*>(gWd) + goff, p.ld_g, rows_valid, w);
      if constexpr (MODE == EPI_DW_LRT) {
        if (p.gS) {
#pragma unroll
          for (int j = 0; j < 16; ++j) w[j] = pack_bf16(v2[2 * j], v2[2 * j + 1]);
          put_tile_bf16(stage, lane, reinterpret_cast<bf16*>(gSd) + goff, p.ld_g, rows_valid, w);
        }
      }
      return;
    }
    float t[32];
    if (acc) {
      get_tile_f32(stage, lane, gWd + goff, p.ld_g, rows_valid, t);
#pragma unroll
      for (int j = 0; j < 32; ++j) t[j] += p.scale * v1[j];
    } else {
#pragma unroll
      for (int j = 0; j < 32; ++j) t[j] = p.scale * v1[j];
    }
    put_tile_f32(stage, lane, gWd + goff, p.ld_g, rows_valid, t);
    if (p.gS) {
      if (acc) get_tile_f32(stage, lane, gSd + goff, p.ld_g, rows_valid, t);
      else {
#pragma unroll
        for (int j = 0; j < 32; ++j) t[j] = 0.f;
      }
      if constexpr (MODE == EPI_DW) {
        if (p.eps16) {
          uint32_t we[16];
          get_tile_bf16(stage, lane, reinterpret_cast<const bf16*>(p.eps16) + z * p.zs_e16 + (long long)row0 * p.ld_e16 + col0,
                        p.ld_e16, rows_valid, we);
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const float2 e = __half22float2(*reinterpret_cast<const __half2*>(&we[j]));
            t[2 * j] += v1[2 * j] * e.x; t[2 * j + 1] += v1[2 * j + 1] * e.y;     // VBLinear.lua:115
          }
        } else {
          PhiloxStream ps = ps0;
          ps.sample += (uint32_t)z;
          const uint32_t q = (uint32_t)((p.N + 3) >> 2);
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            float e[4];
            philox_normal4(ps, (uint32_t)row * q + (uint32_t)((col0 >> 2) + j), e);
#pragma unroll
            for (int k = 0; k < 4; ++k) t[4 * j + k] += v1[4 * j + k] * e[k];      // VBLinear.lua:115
          }
        }
      } else {
#pragma unroll
        for (int j = 0; j < 32; ++j) t[j] += v2[j];
      }
      put_tile_f32(stage, lane, gSd + goff, p.ld_g, rows_valid, t);
    }
  }
}

}  // namespace vbnn
