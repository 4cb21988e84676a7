// gemm_tc.cu -- bf16 x bf16 -> fp32 GEMM on the 5th-gen tensor cores (tcgen05), sm_100a only.
//
// The dense work of the VBLinear hot path (reference call sites: nn.Linear:updateOutput /
// updateGradInput via mlp.lua:77,79 and VBLinear:accGradParameters VBLinear.lua:113-115, all of
// which reach cublasSgemm in the reference) as ONE warp-specialised persistent kernel:
//
//   warp 0        TMA producer   cp.async.bulk.tensor (128B-swizzled boxes) -> smem ring
//   warp 1        MMA issuer     one thread: tcgen05.mma.cta_group::{1,2}.kind::f16, fp32 accumulators in TMEM
//   warps 2..9    epilogue       tcgen05.ld TMEM -> registers -> fused VB epilogue (epilogue.cuh /
//                                epilogue_tc.cuh: coalesced I/O through per-warp swizzled smem tiles)
//
// Tiles: a CTA pair (cta_group::2) owns a 256 x 256 tile -- each CTA stages its 128 rows of A and half
// of B, the leader issues the MMAs for both -- or one CTA a 128 x {64,128,256} tile for small problems.
// Pipelines (mbarriers): smem full/empty (TMA <-> MMA), TMEM full/empty (MMA <-> epilogue; two
// accumulator stages whenever 2 x accumulators x BLOCK_N <= 512 columns, so tile i's epilogue overlaps
// tile i+1's MMAs), and the tile scheduler: cluster launch control (one cluster per tile is launched, the
// resident clusters cancel and absorb the pending ones) or a static round-robin.  The "dual" modes
// (local reparameterisation) run two GEMMs with different operands into two TMEM accumulators and join
// them in the epilogue; the multi-sample dW keeps its running sums in spare TMEM columns.
//
// Operands may be K-major or MN-major in global memory; MN-major tiles are fetched as
// {64 x BK} boxes and handed to the MMA through an MN-major shared-memory descriptor, so the
// batch-contracting dW GEMM (D = G^T X) and dX = G W need no transposed copies.
#include "gemm.h"
#include "epilogue_tc.cuh"
#include "knobs.h"

#include <cuda.h>
#include <stdlib.h>
#include <string.h>

namespace vbnn {

namespace {

constexpr int BM = 128;   // UMMA M (cta_group::1)
constexpr int BK = 64;    // one 128-byte swizzle row of bf16
constexpr int UK = 16;    // UMMA K for 16-bit inputs
constexpr int EPIW = 8;   // epilogue warps
constexpr int NTHREADS = (2 + EPIW) * 32;
constexpr int EPI_STAGE_BYTES = EPIW * kStageBytes;            // per-warp epilogue staging tiles
constexpr int SMEM_BUDGET = 227 * 1024 - 2048 - EPI_STAGE_BYTES;   // minus barriers + alignment slack + staging

// ------------------------------------------------------------------ PTX wrappers ---------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
// arrive on the barrier at the same smem offset in CTA `cta` of this cluster
__device__ __forceinline__ void mbar_arrive_remote(uint32_t bar, uint32_t cta) {
  asm volatile(
      "{\n\t.reg .b32 ra;\n\t"
      "mapa.shared::cluster.u32 ra, %0, %1;\n\t"
      "mbarrier.arrive.release.cluster.shared::cluster.b64 _, [ra];\n\t}"
      ::"r"(bar), "r"(cta)
      : "memory");
}
// arm the barrier at the same offset in CTA `cta` of the cluster for `bytes` of async transactions
__device__ __forceinline__ void mbar_expect_tx_remote(uint32_t bar, uint32_t cta, uint32_t bytes) {
  asm volatile(
      "{\n\t.reg .b32 ra;\n\t"
      "mapa.shared::cluster.u32 ra, %0, %1;\n\t"
      "mbarrier.arrive.expect_tx.shared::cluster.b64 _, [ra], %2;\n\t}"
      ::"r"(bar), "r"(cta), "r"(bytes)
      : "memory");
}
// Cluster launch control (Blackwell): ask the hardware to cancel one not-yet-launched cluster of
// this grid and hand its block index to us; the 16-byte response lands in every CTA of the cluster.
__device__ __forceinline__ void clc_try_cancel(uint32_t resp, uint32_t bar) {
  asm volatile(
      "clusterlaunchcontrol.try_cancel.async.shared::cta.mbarrier::complete_tx::bytes.multicast::cluster::all.b128 [%0], [%1];"
      ::"r"(resp), "r"(bar)
      : "memory");
}
// returns the first blockIdx.x of the cancelled cluster, or -1 when nothing was left to cancel
__device__ __forceinline__ int clc_read(uint32_t resp) {
  uint32_t x, y, z, valid;
  asm volatile(
      "{\n\t.reg .pred p1;\n\t.reg .b128 r;\n\t"
      "ld.shared.b128 r, [%4];\n\t"
      "clusterlaunchcontrol.query_cancel.is_canceled.pred.b128 p1, r;\n\t"
      "selp.u32 %3, 1, 0, p1;\n\t"
      "mov.u32 %0, 0; mov.u32 %1, 0; mov.u32 %2, 0;\n\t"
      "@p1 clusterlaunchcontrol.query_cancel.get_first_ctaid.v4.b32.b128 {%0, %1, %2, _}, r;\n\t}"
      : "=r"(x), "=r"(y), "=r"(z), "=r"(valid)
      : "r"(resp)
      : "memory");
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  return valid ? (int)x : -1;
}
__device__ __forceinline__ uint32_t mbar_try(uint32_t bar, uint32_t parity) {
  uint32_t done;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.b32 %0, 1, 0, p;\n\t}"
      : "=r"(done)
      : "r"(bar), "r"(parity)
      : "memory");
  return done;
}
// Bounded wait: a protocol bug traps (the launch fails) instead of hanging the GPU.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  if (mbar_try(bar, parity)) return;
  long long t0 = 0;
  for (uint32_t spins = 1; !mbar_try(bar, parity); ++spins) {
    if ((spins & 1023u) != 0) continue;       // look at the clock once per 1024 polls: the poll loop shares
    if (t0 == 0) { t0 = clock64(); continue; }   // issue slots with the epilogue warps
    if (clock64() - t0 > 4000000000LL) {
      printf("vbnn gemm_tc: mbarrier timeout (block %d thread %d bar %u parity %u)\n", blockIdx.x,
             threadIdx.x, bar, parity);
      __trap();
    }
  }
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
// CG == 2: both CTAs of the pair load into their own smem but complete the transaction on the
// LEADER's barrier (the CTA-rank bit of the shared::cluster address is cleared).
// L2 eviction-priority hints for TMA loads (createpolicy encodings, as in CUTLASS' CacheHintSm90)
constexpr uint64_t kL2EvictNormal = 0x1000000000000000ull;
constexpr uint64_t kL2EvictFirst = 0x12F0000000000000ull;
constexpr uint64_t kL2EvictLast = 0x14F0000000000000ull;
template <int CG>
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* tm, uint32_t bar,
                                            int c0, int c1, int c2, uint64_t hint) {
  if constexpr (CG == 1) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint"
        " [%0], [%1, {%3, %4, %5}], [%2], %6;"
        ::"r"(dst), "l"(reinterpret_cast<uint64_t>(tm)), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "l"(hint)
        : "memory");
  } else {
    asm volatile(
        "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint"
        " [%0], [%1, {%3, %4, %5}], [%2], %6;"
        ::"r"(dst), "l"(reinterpret_cast<uint64_t>(tm)), "r"(bar & 0xFEFFFFFFu), "r"(c0), "r"(c1), "r"(c2), "l"(hint)
        : "memory");
  }
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* tm) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(tm)) : "memory");
}
template <int CG>
__device__ __forceinline__ void tmem_alloc(uint32_t dst_smem, uint32_t cols) {
  if constexpr (CG == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  } else {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
}
template <int CG>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t cols) {
  if constexpr (CG == 1)
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
  else
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
// arrive on `bar` once every MMA issued so far has retired; CG == 2: on the same barrier of both CTAs
template <int CG>
__device__ __forceinline__ void tc_commit(uint32_t bar) {
  if constexpr (CG == 1) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
  } else {
    asm volatile(
        "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
        ::"r"(bar), "h"((uint16_t)3)
        : "memory");
  }
}
template <int CG>
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc,
                                          uint32_t idesc, uint32_t accumulate) {
  if constexpr (CG == 1) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
  } else {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
  }
}
// 32 lanes x 32 consecutive fp32 columns: thread t gets lane (base_lane + t), columns col..col+31
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float (&v)[32]) {
  uint32_t* r = reinterpret_cast<uint32_t*>(v);
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
        "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]),
        "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]),
        "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
        "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() {
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
// the reverse: thread t writes its 32 registers to lane (base_lane + t), columns col..col+31
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const float (&v)[32]) {
  const uint32_t* r = reinterpret_cast<const uint32_t*>(v);
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]),
        "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]),
        "r"(r[16]), "r"(r[17]), "r"(r[18]), "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]),
        "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() {
  asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
}

// ---- UMMA shared-memory descriptor (SWIZZLE_128B) ---------------------------------------------
// bits [0,14) start>>4 | [16,30) LBO>>4 | [32,46) SBO>>4 | [46,48) version=1 | [61,64) layout=2
// K-major  tile [rows x 64]: 8-row groups of 128-byte rows, SBO = 1024, LBO unused (=16 B);
//          the k-th UMMA_K slice starts 32 bytes further along the swizzled row.
// MN-major tile [64 k-rows x 64*c]: each k-row is 128 bytes of 64 MN elements, 8 k-rows = one
//          1024-byte swizzle atom (SBO), the next 64-wide MN chunk is a separate TMA box LBO =
//          BK*128 bytes away; the k-th UMMA_K slice starts 16 rows = 2048 bytes further.
template <bool KMAJOR>
__device__ __forceinline__ uint64_t make_sdesc(uint32_t saddr) {
  constexpr uint64_t lbo = KMAJOR ? 16 : (uint64_t)BK * 128;
  constexpr uint64_t sbo = 1024;
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFFu) >> 4);
  d |= (lbo >> 4) << 16;
  d |= (sbo >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
template <bool KMAJOR>
__device__ __forceinline__ constexpr uint32_t kslice_bytes() {
  return KMAJOR ? UK * 2 : UK * 128;
}
// instruction descriptor: c=F32 [4,6), a=b=BF16 [7,10),[10,13), a_major 15, b_major 16,
// N>>3 [17,23), M>>4 [24,29).  M = 128 per CTA of the group (256 for cta_group::2).
template <int BN, int CG, bool AK, bool BKM>
__device__ __forceinline__ constexpr uint32_t make_idesc() {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((AK ? 0u : 1u) << 15) | ((BKM ? 0u : 1u) << 16) |
         ((uint32_t)(BN >> 3) << 17) | ((uint32_t)((BM * CG) >> 4) << 24);
}

struct TcShape {
  int M, N, K, batch;
  int mt, nt, num_kb;       // mt counts (128*CG)-row tiles
  int gm;                   // rasterisation band height in m-tiles
  int staged;               // every epilogue tensor is 16-byte aligned: coalesced staged I/O
  int clc;                  // dynamic scheduling: one cluster per work unit, resident clusters steal pending ones
  int zA1, zB1, zA2, zB2;   // 0: the operand is shared by every batch index z (stride 0), 1: batched
  int hintA, hintB;         // L2 eviction priority of the A / B operand tiles: 0 normal, 1 evict-last, 2 evict-first
  int zsum;                 // sample-summing form: one work unit per tile walks every z into one TMEM accumulator
};

// Tile rasterisation: bands of `gm` m-tiles, inside a band n-major.  The ~#SM/CG tiles in flight
// then form a gm x (slots/gm) block of the tile grid, so their A rows and B rows are shared
// through L2 (M-fastest order streamed the whole A operand from DRAM once per wave: 1.05 GB read
// for a 192 MB problem, ncu r01b).
__device__ __forceinline__ void decode_tile(const TcShape& sh, int tile, int& mi, int& ni) {
  const int band_tiles = sh.gm * sh.nt;
  const int band = tile / band_tiles;
  const int r = tile - band * band_tiles;
  const int rows = min(sh.gm, sh.mt - band * sh.gm);
  ni = r / rows;
  mi = band * sh.gm + (r - ni * rows);
}

// CG = CTAs per MMA (cta_group).  With CG == 2 a CTA pair owns a (256 x BN) tile: CTA r holds rows
// [128r, 128r+128) of A and of the accumulator and rows [r*BN/2, (r+1)*BN/2) of B; the leader
// (rank 0) issues tcgen05.mma.cta_group::2, which reads both CTAs' shared memory.
template <int MODE, int BN, int CG>
struct TcCfg {
  static constexpr bool DUAL = epi_is_dual(MODE);
  static constexpr int NACC = DUAL ? 2 : 1;
  static constexpr int A_BYTES = BM * BK * 2;
  static constexpr int B_ROWS = BN / CG;
  static constexpr int B_BYTES = B_ROWS * BK * 2;
  static constexpr int STAGE_BYTES = NACC * (A_BYTES + B_BYTES);
  static constexpr int STAGES_RAW = SMEM_BUDGET / STAGE_BYTES;
  static constexpr int STAGES = STAGES_RAW > 6 ? 6 : STAGES_RAW;
  static constexpr int ACC_COLS = NACC * BN;                        // TMEM columns per accumulator stage
  static constexpr int ACC_STAGES = 2 * ACC_COLS <= 512 ? 2 : 1;    // double-buffered when it fits
  // ZACC with BN == 128: columns [256, 384) / [384, 512) hold the running gradWeight / gradSum of the tile
  // across the Monte-Carlo samples (written by the epilogue warps with tcgen05.st, never by the MMA)
  static constexpr bool TACC = epi_z_accumulates(MODE) && !DUAL && BN == 128;
  static constexpr int TMEM_COLS = TACC ? 512 : ACC_STAGES * ACC_COLS;
  // barriers + CLC ring live in the last 512 bytes; the dynamic window is declared 1024-byte aligned, so
  // no alignment slack: together with the 1 KB the system reserves per CTA this leaves room on the SM
  // for one small co-resident CTA of an HBM-bound kernel (the fused update overlaps the backward GEMMs)
  static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + EPI_STAGE_BYTES + 512;
  static_assert(TMEM_COLS == 128 || TMEM_COLS == 256 || TMEM_COLS == 512, "TMEM allocation must be a power of two");
  static_assert(STAGES >= 2, "need at least a double-buffered smem ring");
  static_assert(B_ROWS % 64 == 0, "B tile rows per CTA must be a multiple of 64");
};

// One operand tile: K-major -> one {64 x ROWS} box; MN-major -> ROWS/64 boxes of {64 x BK}.
template <int CG, bool KMAJOR, int ROWS>
__device__ __forceinline__ void load_operand(const CUtensorMap* tm, uint32_t dst, uint32_t bar,
                                             int mn0, int k0, int z, uint64_t hint) {
  if constexpr (KMAJOR) {
    tma_load_3d<CG>(dst, tm, bar, k0, mn0, z, hint);
  } else {
#pragma unroll
    for (int c = 0; c < ROWS / 64; ++c) tma_load_3d<CG>(dst + c * (BK * 128), tm, bar, mn0 + c * 64, k0, z, hint);
  }
}

template <int MODE, int BN, int CG, bool AK, bool BKM>
__global__ void __launch_bounds__(NTHREADS, 1)
gemm_tc_kernel(const __grid_constant__ CUtensorMap tmA1, const __grid_constant__ CUtensorMap tmB1,
               const __grid_constant__ CUtensorMap tmA2, const __grid_constant__ CUtensorMap tmB2,
               TcShape sh, EpiParams p) {
  using C = TcCfg<MODE, BN, CG>;
  constexpr bool DUAL = C::DUAL;
  constexpr bool ZACC = epi_z_accumulates(MODE);
  constexpr int AS = C::ACC_STAGES;

  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const uint32_t smem_base = smem_u32(smem_raw);
  if ((smem_base & 1023u) != 0) {        // SWIZZLE_128B tiles need 1024-byte alignment
    if (threadIdx.x == 0) printf("vbnn gemm_tc: dynamic shared memory base %u is not 1024-byte aligned\n", smem_base);
    __trap();
  }
  const uint32_t epi_stage_base = smem_base + C::STAGES * C::STAGE_BYTES;
  const uint32_t bar_base = epi_stage_base + EPI_STAGE_BYTES;
  // barriers: full[STAGES], empty[STAGES], tmem_full[2], tmem_empty[2]; then the TMEM address
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (C::STAGES + s); };
  auto tfull_bar = [&](int s) { return bar_base + 8u * (2 * C::STAGES + s); };
  auto tempty_bar = [&](int s) { return bar_base + 8u * (2 * C::STAGES + 2 + s); };
  const uint32_t tmem_slot = bar_base + 8u * (2 * C::STAGES + 4);
  // cluster-launch-control ring (2 slots): 16-byte responses, full barriers (one per CTA), empty
  // barriers (the leader's collect every consumer of the cluster)
  auto clc_resp = [&](int s) { return bar_base + 256u + 16u * s; };
  auto clc_full = [&](int s) { return bar_base + 320u + 8u * s; };
  auto clc_empty = [&](int s) { return bar_base + 336u + 8u * s; };
  constexpr uint32_t kClcConsumers = CG * (1 + EPIW) + 1;   // producers + epilogue warps of every CTA + the MMA thread

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int rank = CG == 2 ? (int)cluster_ctarank() : 0;     // position inside the CTA pair
  const bool leader = rank == 0;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA1);
    tma_prefetch_desc(&tmB1);
    if (DUAL) { tma_prefetch_desc(&tmA2); tma_prefetch_desc(&tmB2); }
    for (int s = 0; s < C::STAGES; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
    // the leader's MMA thread waits for the epilogue warps of every CTA of the group
    for (int s = 0; s < 2; ++s) { mbar_init(tfull_bar(s), 1); mbar_init(tempty_bar(s), EPIW * CG); }
    for (int s = 0; s < 2; ++s) { mbar_init(clc_full(s), 1); mbar_init(clc_empty(s), kClcConsumers); }
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc<CG>(tmem_slot, C::TMEM_COLS);
  tc_fence_before();
  if constexpr (CG == 2) cluster_sync_all(); else __syncthreads();
  tc_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.b32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));

  const int tiles = sh.mt * sh.nt;
  // one work unit per tile when the unit walks every z (ZACC, zsum): w < tiles, so z = w / tiles = 0 below
  const int num_work = (ZACC || sh.zsum) ? tiles : tiles * sh.batch;
  const int group = blockIdx.x / CG, num_groups = gridDim.x / CG;
  const bool dyn = sh.clc != 0;
  // next work unit of a role: static round-robin, or the response of the CLC query issued by the
  // leader's producer thread (every role consumes every response, including the final "nothing left")
  auto next_work = [&](int w, int& cs, uint32_t& cp, bool whole_warp) -> int {
    if (!dyn) { w += num_groups; return w < num_work ? w : -1; }
    mbar_wait(clc_full(cs), cp);
    const int first = clc_read(clc_resp(cs));
    if (whole_warp) __syncwarp();
    if (!whole_warp || lane == 0) {
      if (CG == 1 || leader) mbar_arrive(clc_empty(cs)); else mbar_arrive_remote(clc_empty(cs), 0);
    }
    if (++cs == 2) { cs = 0; cp ^= 1; }
    return first >= 0 ? first / CG : -1;
  };

  if (warp == 0) {
    // ======================= TMA producer (one per CTA) =======================
    if (lane == 0) {
      int stage = 0; uint32_t phase = 0;
      int cs = 0; uint32_t cp = 0;          // CLC ring position as consumer
      int is = 0; uint32_t ip = 0;          // ... and as issuer (leader only)
      const uint64_t hA = sh.hintA == 1 ? kL2EvictLast : sh.hintA == 2 ? kL2EvictFirst : kL2EvictNormal;
      const uint64_t hB = sh.hintB == 1 ? kL2EvictLast : sh.hintB == 2 ? kL2EvictFirst : kL2EvictNormal;
      for (int w = group; w >= 0 && w < num_work; w = next_work(w, cs, cp, false)) {
        if (dyn && leader) {
          // ask for the unit after this one now, so the answer is there when the loads are out
          mbar_wait(clc_empty(is), ip ^ 1);
          mbar_expect_tx(clc_full(is), 16);
          if (CG == 2) mbar_expect_tx_remote(clc_full(is), 1, 16);
          clc_try_cancel(clc_resp(is), clc_full(is));
          if (++is == 2) { is = 0; ip ^= 1; }
        }
        const int tile = ZACC ? w : w % tiles;
        const int zb = ZACC ? 0 : w / tiles, zn = (ZACC || sh.zsum) ? sh.batch : 1;
        int mi, ni;
        decode_tile(sh, tile, mi, ni);
        const int m0 = mi * (BM * CG) + rank * BM;
        const int n0 = ni * BN + rank * C::B_ROWS;
        for (int z = zb; z < zb + zn; ++z) {
          for (int kb = 0; kb < sh.num_kb; ++kb) {
            mbar_wait(empty_bar(stage), phase ^ 1);
            // the leader arms its barrier for the bytes of the whole group
            if (leader) mbar_expect_tx(full_bar(stage), C::STAGE_BYTES * CG);
            const uint32_t sa = smem_base + stage * C::STAGE_BYTES;
            const uint32_t sb = sa + C::NACC * C::A_BYTES;
            load_operand<CG, AK, BM>(&tmA1, sa, full_bar(stage), m0, kb * BK, z * sh.zA1, hA);
            load_operand<CG, BKM, C::B_ROWS>(&tmB1, sb, full_bar(stage), n0, kb * BK, z * sh.zB1, hB);
            if (DUAL) {
              load_operand<CG, AK, BM>(&tmA2, sa + C::A_BYTES, full_bar(stage), m0, kb * BK, z * sh.zA2, hA);
              load_operand<CG, BKM, C::B_ROWS>(&tmB2, sb + C::B_BYTES, full_bar(stage), n0, kb * BK, z * sh.zB2, hB);
            }
            if (++stage == C::STAGES) { stage = 0; phase ^= 1; }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ======================= MMA issuer (one thread of the leader CTA) =======================
    if (lane == 0 && leader) {
      constexpr uint32_t idesc = make_idesc<BN, CG, AK, BKM>();
      int stage = 0; uint32_t phase = 0;
      int as = 0; uint32_t aphase = 0;
      int cs = 0; uint32_t cp = 0;
      for (int w = group; w >= 0 && w < num_work; w = next_work(w, cs, cp, false)) {
        const int zn = (ZACC || sh.zsum) ? sh.batch : 1;
        for (int zi = 0; zi < zn; ++zi) {
          // ZACC: one accumulator (and epilogue pass) per z; zsum: the samples are K-concatenated into one
          // accumulator, claimed before z = 0 and handed to the epilogue after the last z
          const bool first_z = zi == 0 || !sh.zsum, last_z = zi + 1 == zn || !sh.zsum;
          const int kz = sh.zsum ? zi : 0;
          if (first_z) {
            mbar_wait(tempty_bar(as), aphase ^ 1);
            tc_fence_after();
          }
          const uint32_t d1 = tmem_base + as * C::ACC_COLS;
          for (int kb = 0; kb < sh.num_kb; ++kb) {
            mbar_wait(full_bar(stage), phase);
            tc_fence_after();
            const uint32_t sa = smem_base + stage * C::STAGE_BYTES;
            const uint32_t sb = sa + C::NACC * C::A_BYTES;
#pragma unroll
            for (int k = 0; k < BK / UK; ++k) {
              const uint32_t acc = (kz | kb | k) != 0 ? 1u : 0u;
              umma_bf16<CG>(d1, make_sdesc<AK>(sa + k * kslice_bytes<AK>()),
                            make_sdesc<BKM>(sb + k * kslice_bytes<BKM>()), idesc, acc);
              if (DUAL)
                umma_bf16<CG>(d1 + BN, make_sdesc<AK>(sa + C::A_BYTES + k * kslice_bytes<AK>()),
                              make_sdesc<BKM>(sb + C::B_BYTES + k * kslice_bytes<BKM>()), idesc, acc);
            }
            tc_commit<CG>(empty_bar(stage));     // smem slot free (in every CTA) once these MMAs retire
            if (++stage == C::STAGES) { stage = 0; phase ^= 1; }
          }
          if (last_z) {
            tc_commit<CG>(tfull_bar(as));        // accumulator ready for the epilogue warps
            if (++as == AS) { as = 0; aphase ^= 1; }
          }
        }
      }
    }
  } else {
    // ======================= epilogue warps (every CTA drains its own 128 TMEM lanes) ==========
    const int q = warp & 3;                  // TMEM lane quarter this warp may access
    const int half = (warp - 2) >> 2;        // two warps share a quarter, split the columns
    const PhiloxStream ps = epi_stream(p);
    const uint32_t my_stage = epi_stage_base + (uint32_t)(warp - 2) * kStageBytes;
    int as = 0; uint32_t aphase = 0;
    int cs = 0; uint32_t cp = 0;
    for (int w = group; w >= 0 && w < num_work; w = next_work(w, cs, cp, true)) {
      const int tile = ZACC ? w : w % tiles;
      const int zb = ZACC ? 0 : w / tiles, zn = ZACC ? sh.batch : 1;
      int mi, ni;
      decode_tile(sh, tile, mi, ni);
      const int m0 = mi * (BM * CG) + rank * BM, n0 = ni * BN;
      const int row = m0 + q * 32 + lane;
      if (C::TACC && zn > 1) {
        // Multi-sample dW with TMEM-RESIDENT accumulators: a 128 x 128 tile (half the operand traffic per MAC
        // of the 128 x 64 register-accumulating form, which is L2-bandwidth-bound), each warp owning two
        // 32 x 32 chunks whose running gradWeight / gradSum live in spare TMEM columns between samples --
        // tcgen05.ld the sample's product, fold it in, tcgen05.st it back; global memory once per tile.
        const uint32_t lane_base = (uint32_t)(q * 32) << 16;
        const uint32_t tW = tmem_base + lane_base + 256u, tS = tmem_base + lane_base + 384u;
        const uint32_t qn = (uint32_t)((p.N + 3) >> 2);
        for (int z = zb; z < zb + zn; ++z) {
          const bool first = z == zb, last = z + 1 == zb + zn;
          mbar_wait(tfull_bar(as), aphase);
          tc_fence_after();
          const uint32_t tz = tmem_base + lane_base + as * C::ACC_COLS;
          PhiloxStream psz = ps;
          psz.sample += (uint32_t)z;
#pragma unroll 1
          for (int c = half; c < BN / 32; c += EPIW / 4) {
            const int col0 = n0 + c * 32;
            if (col0 >= sh.N) break;                       // warp-uniform
            const int row0 = m0 + q * 32;
            const bool full = sh.staged && col0 + 32 <= sh.N;
            const int rows_valid = min(32, p.M - row0);
            float *gWd, *gSd;
            dw_dest(p, row0, gWd, gSd);
            auto emit = [&](float* dst, float (&a)[32]) {   // the tile's final value of one accumulator -> global
              const long long goff = (long long)row0 * p.ld_g + col0;
              if (full) {
                if (p.accumulate) {
                  float t[32];
                  get_tile_f32(my_stage, lane, dst + goff, p.ld_g, rows_valid, t);
#pragma unroll
                  for (int j = 0; j < 32; ++j) a[j] += t[j];
                }
                put_tile_f32(my_stage, lane, dst + goff, p.ld_g, rows_valid, a);
              } else if (row < p.M) {
                const bool vec_g = (p.ld_g & 3) == 0;
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                  const int cq = col0 + 4 * j;
                  if (cq >= p.N) break;
                  const int nvalid = min(4, p.N - cq);
                  float* gp = dst + (long long)row * p.ld_g + cq;
                  float w4[4] = {a[4 * j], a[4 * j + 1], a[4 * j + 2], a[4 * j + 3]};
                  if (p.accumulate) { float o[4]; load4<float>(gp, o, nvalid, vec_g); for (int k = 0; k < 4; ++k) w4[k] += o[k]; }
                  store4<float>(gp, w4, nvalid, vec_g);
                }
              }
            };
            float v1[32], acc[32];
            tmem_ld32(tz + c * 32, v1);
            if (!first && p.gS) tmem_ld32(tS + c * 32, acc);
            tmem_ld_wait();
            if (p.gS) {
              if (first) {
#pragma unroll
                for (int j = 0; j < 32; ++j) acc[j] = 0.f;
              }
              if (p.eps16 && full) {
                // epsilon as k_sample_w drew it (fp16), one coalesced 2 KB tile instead of 8 Philox + 16 Box-Muller
                // (fetching the tile before the accumulator wait changed nothing: the kernel is bound by the L2 -> SM
                // operand traffic of 128 x 128 tiles, not by this load)
                uint32_t we[16];
                get_tile_bf16(my_stage, lane,
                              reinterpret_cast<const bf16*>(p.eps16) + z * p.zs_e16 + (long long)row0 * p.ld_e16 + col0,
                              p.ld_e16, rows_valid, we);
#pragma unroll
                for (int j = 0; j < 16; ++j) {
                  const float2 e = __half22float2(*reinterpret_cast<const __half2*>(&we[j]));
                  acc[2 * j] += v1[2 * j] * e.x; acc[2 * j + 1] += v1[2 * j + 1] * e.y;   // VBLinear.lua:115
                }
              } else if (p.eps16) {
                const __half* ep = reinterpret_cast<const __half*>(p.eps16) + z * p.zs_e16 + (long long)row * p.ld_e16 + col0;
#pragma unroll
                for (int j = 0; j < 32; ++j)
                  if (row < p.M && col0 + j < p.N) acc[j] += v1[j] * __half2float(ep[j]);
              } else {
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                  float e[4];
                  philox_normal4(psz, (uint32_t)row * qn + (uint32_t)((col0 >> 2) + j), e);
#pragma unroll
                  for (int k = 0; k < 4; ++k) acc[4 * j + k] += v1[4 * j + k] * e[k];       // VBLinear.lua:115
                }
              }
              if (last) emit(gSd, acc); else tmem_st32(tS + c * 32, acc);
            }
            if (first) {
#pragma unroll
              for (int j = 0; j < 32; ++j) acc[j] = p.scale * v1[j];                     // VBLinear.lua:113
            } else {
              tmem_ld32(tW + c * 32, acc);
              tmem_ld_wait();
#pragma unroll
              for (int j = 0; j < 32; ++j) acc[j] += p.scale * v1[j];
            }
            if (last) emit(gWd, acc); else tmem_st32(tW + c * 32, acc);
          }
          if (!last) tmem_st_wait();
          tc_fence_before();
          __syncwarp();
          if (lane == 0) {
            if constexpr (CG == 1) mbar_arrive(tempty_bar(as));
            else mbar_arrive_remote(tempty_bar(as), 0);
          }
          if (++as == AS) { as = 0; aphase ^= 1; }
        }
      } else if constexpr (ZACC && BN == 64) {
        // Multi-sample dW (weight-space sampling, S > 1): this warp owns ONE 32 x 32 chunk of the
        // tile and keeps its gradWeight / gradSum values in registers across all samples, so the
        // per-sample work is TMEM load + Philox + FMA; global memory is touched once per tile
        // (the per-sample read-modify-write was a ~1 us dependent chain per sample).
        const int col0 = n0 + half * 32;
        float accW[32], accS[32];
#pragma unroll
        for (int j = 0; j < 32; ++j) { accW[j] = 0.f; accS[j] = 0.f; }
        const uint32_t qn = (uint32_t)((p.N + 3) >> 2);
        for (int z = zb; z < zb + zn; ++z) {
          mbar_wait(tfull_bar(as), aphase);
          tc_fence_after();
          const uint32_t t0 = tmem_base + ((uint32_t)(q * 32) << 16) + as * C::ACC_COLS;
          if (col0 < sh.N) {
            float v1[32], v2[32];
            tmem_ld32(t0 + half * 32, v1);
            if (DUAL) tmem_ld32(t0 + BN + half * 32, v2);
            tmem_ld_wait();
            PhiloxStream psz = ps;
            psz.sample += (uint32_t)z;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              if constexpr (MODE == EPI_DW) {
                float e[4];
                if (p.noise) {
                  const int cq = col0 + 4 * j;
                  if (row < p.M && cq < p.N)
                    load4<float>(p.noise + z * p.zs_noise + (long long)row * p.N + cq, e, min(4, p.N - cq), (p.N & 3) == 0);
                  else e[0] = e[1] = e[2] = e[3] = 0.f;
                } else {
                  philox_normal4(psz, (uint32_t)row * qn + (uint32_t)((col0 >> 2) + j), e);
                }
#pragma unroll
                for (int k = 0; k < 4; ++k) accS[4 * j + k] += v1[4 * j + k] * e[k];     // VBLinear.lua:115
              } else {
#pragma unroll
                for (int k = 0; k < 4; ++k) accS[4 * j + k] += v2[DUAL ? 4 * j + k : 0];
              }
#pragma unroll
              for (int k = 0; k < 4; ++k) accW[4 * j + k] += p.scale * v1[4 * j + k];   // VBLinear.lua:113
            }
          }
          tc_fence_before();
          __syncwarp();
          if (lane == 0) {
            if constexpr (CG == 1) mbar_arrive(tempty_bar(as));
            else mbar_arrive_remote(tempty_bar(as), 0);
          }
          if (++as == AS) { as = 0; aphase ^= 1; }
        }
        if (col0 < sh.N) {
          const int row0 = m0 + q * 32;
          const long long goff = (long long)row0 * p.ld_g + col0;
          float *gWd, *gSd;
          dw_dest(p, row0, gWd, gSd);
          if (sh.staged && col0 + 32 <= sh.N) {
            const int rows_valid = min(32, p.M - row0);
            float t[32];
            if (p.accumulate) {
              get_tile_f32(my_stage, lane, gWd + goff, p.ld_g, rows_valid, t);
#pragma unroll
              for (int j = 0; j < 32; ++j) accW[j] += t[j];
            }
            put_tile_f32(my_stage, lane, gWd + goff, p.ld_g, rows_valid, accW);
            if (p.gS) {
              if (p.accumulate) {
                get_tile_f32(my_stage, lane, gSd + goff, p.ld_g, rows_valid, t);
#pragma unroll
                for (int j = 0; j < 32; ++j) accS[j] += t[j];
              }
              put_tile_f32(my_stage, lane, gSd + goff, p.ld_g, rows_valid, accS);
            }
          } else if (row < p.M) {
            const bool vec_g = (p.ld_g & 3) == 0;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const int cq = col0 + 4 * j;
              if (cq >= p.N) break;
              const int nvalid = min(4, p.N - cq);
              float* gw = gWd + (long long)row * p.ld_g + cq;
              float w4[4] = {accW[4 * j], accW[4 * j + 1], accW[4 * j + 2], accW[4 * j + 3]};
              if (p.accumulate) { float o[4]; load4<float>(gw, o, nvalid, vec_g); for (int k = 0; k < 4; ++k) w4[k] += o[k]; }
              store4<float>(gw, w4, nvalid, vec_g);
              if (p.gS) {
                float* gs = gSd + (long long)row * p.ld_g + cq;
                float s4[4] = {accS[4 * j], accS[4 * j + 1], accS[4 * j + 2], accS[4 * j + 3]};
                if (p.accumulate) { float o[4]; load4<float>(gs, o, nvalid, vec_g); for (int k = 0; k < 4; ++k) s4[k] += o[k]; }
                store4<float>(gs, s4, nvalid, vec_g);
              }
            }
          }
        }
      } else {
      for (int z = zb; z < zb + zn; ++z) {
        mbar_wait(tfull_bar(as), aphase);
        tc_fence_after();
        const uint32_t t0 = tmem_base + ((uint32_t)(q * 32) << 16) + as * C::ACC_COLS;
#pragma unroll 1
        for (int c = half; c < BN / 32; c += EPIW / 4) {
          if (n0 + c * 32 >= sh.N) break;    // warp-uniform
          float v1[32], v2[32];
          tmem_ld32(t0 + c * 32, v1);
          if (DUAL) tmem_ld32(t0 + BN + c * 32, v2);
          tmem_ld_wait();
          if (sh.staged && n0 + c * 32 + 32 <= sh.N) {
            epi_chunk_staged<MODE>(p, ps, z, m0 + q * 32, lane, n0 + c * 32, v1, v2, my_stage);
          } else {
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              epi_quad<MODE, bf16>(p, ps, z, row, n0 + c * 32 + j * 4,
                                   *reinterpret_cast<const float(*)[4]>(&v1[j * 4]),
                                   *reinterpret_cast<const float(*)[4]>(&v2[DUAL ? j * 4 : 0]));
            }
          }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) {
          if constexpr (CG == 1) mbar_arrive(tempty_bar(as));
          else mbar_arrive_remote(tempty_bar(as), 0);      // the leader's barrier
        }
        if (++as == AS) { as = 0; aphase ^= 1; }
      }
      }
    }
  }

  // peer mode: this CTA's gradient tiles went to other GPUs; make them visible system-wide before the
  // kernel retires (the flag that announces them is raised by a later kernel of the same stream)
  if constexpr (ZACC) { if (p.scatter_rows) __threadfence_system(); }
  tc_fence_before();
  if constexpr (CG == 2) cluster_sync_all(); else __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc<CG>(tmem_base, C::TMEM_COLS);
  }
}

// ------------------------------------------------------------------ host side -------------
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*,
                                    const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                    const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                    CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

PFN_encodeTiled get_encode() {
  static PFN_encodeTiled fn = nullptr;
  if (fn) return fn;
  void* p = nullptr;
  cudaDriverEntryPointQueryResult qr;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qr) != cudaSuccess ||
      qr != cudaDriverEntryPointSuccess)
    return nullptr;
  fn = reinterpret_cast<PFN_encodeTiled>(p);
  return fn;
}

// rows_mn: MN extent, K: contraction extent, box_mn: tile rows for a K-major operand
int make_tmap(CUtensorMap* tm, const GemmOperand& op, int rows_mn, int K, int batch, int box_mn) {
  PFN_encodeTiled enc = get_encode();
  VB_CHECK(enc != nullptr, VBNN_E_CUDA, "cuTensorMapEncodeTiled unavailable (no CUDA driver?)");
  VB_CHECK(op.ptr != nullptr, VBNN_E_INVALID, "gemm_tc: null operand");
  VB_CHECK((op.ld % 8) == 0 && (reinterpret_cast<uintptr_t>(op.ptr) % 16) == 0, VBNN_E_INVALID,
           "gemm_tc: operand rows must be 16-byte aligned (ld=%d)", op.ld);
  VB_CHECK(batch == 1 || (op.zs % 8) == 0, VBNN_E_INVALID, "gemm_tc: batch stride %% 8 != 0");
  cuuint64_t dims[3], strides[2];
  cuuint32_t box[3], estr[3] = {1, 1, 1};
  if (op.kmajor) {
    dims[0] = (cuuint64_t)K; dims[1] = (cuuint64_t)rows_mn;
    box[0] = BK; box[1] = (cuuint32_t)box_mn;
  } else {
    dims[0] = (cuuint64_t)rows_mn; dims[1] = (cuuint64_t)K;
    box[0] = 64; box[1] = BK;
  }
  const bool batched = batch > 1 && op.zs != 0;
  dims[2] = batched ? (cuuint64_t)batch : 1;
  box[2] = 1;
  strides[0] = (cuuint64_t)op.ld * 2;
  strides[1] = batched ? (cuuint64_t)op.zs * 2 : strides[0] * dims[1];
  CUresult r = enc(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(op.ptr), dims, strides,
                   box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  VB_CHECK(r == CUDA_SUCCESS, VBNN_E_CUDA,
           "cuTensorMapEncodeTiled failed (%d): dims %llu x %llu x %llu ld %d kmajor %d", (int)r,
           (unsigned long long)dims[0], (unsigned long long)dims[1], (unsigned long long)dims[2],
           op.ld, op.kmajor);
  return VBNN_OK;
}

struct TcChoice { int bn, cg; };   // bn == 64: multi-sample dW with register accumulation

template <int MODE, int BN, int CG, bool AK, bool BKM>
int launch_cfg(const GemmArgs& g, const EpiParams& p, cudaStream_t st) {
  using C = TcCfg<MODE, BN, CG>;
  TcShape sh;
  sh.M = g.M; sh.N = g.N; sh.K = g.K; sh.batch = g.batch;
  sh.mt = ceil_div(g.M, BM * CG); sh.nt = ceil_div(g.N, BN); sh.num_kb = ceil_div(g.K, BK);
  sh.zA1 = g.A1.zs != 0; sh.zB1 = g.B1.zs != 0; sh.zA2 = g.A2.zs != 0; sh.zB2 = g.B2.zs != 0;
  sh.zsum = g.zsum && g.batch > 1;
  {
    const Knobs& k = knobs();
    sh.gm = k.tc_gm > 0 ? k.tc_gm : 8;
    if (sh.gm > sh.mt) sh.gm = sh.mt;
    sh.staged = k.tc_staged && epi_can_stage(MODE, p);
    sh.clc = k.tc_clc;
    // L2 priorities (knob tc_l2hint, default on).  Band rasterisation keeps a band of gm m-tiles of A in flight
    // while the n-tiles of B sweep past: the A band is what every tile of the band re-reads, so it is evict-last;
    // B tiles are shared only by the tiles running at the same time: normal priority.  A weight operand that is
    // small enough to stay resident for the whole kernel (B of the forward / backward-data GEMMs) is evict-last too.
    sh.hintA = 0; sh.hintB = 0;
    if (k.tc_l2hint == 1) {
      const double a_band = (double)sh.gm * BM * CG * g.K * 2.0 * C::NACC;       // bytes of one A band
      const double b_all = (double)g.N * g.K * 2.0 * C::NACC;                    // bytes of the whole B operand
      if (b_all <= 72e6 && g.B1.zs == 0) sh.hintB = 1;
      if (a_band <= 40e6) sh.hintA = sh.hintB == 1 && a_band + b_all > 100e6 ? 0 : 1;
    } else if (k.tc_l2hint > 1) {              // experiments: 2 = A evict-last, 3 = B evict-last, 4 = both, 5 = A last + B first
      sh.hintA = (k.tc_l2hint == 2 || k.tc_l2hint >= 4) ? 1 : 0;
      sh.hintB = (k.tc_l2hint == 3 || k.tc_l2hint == 4) ? 1 : (k.tc_l2hint == 5 ? 2 : 0);
    }
  }
  CUtensorMap tA1, tB1, tA2, tB2;
  VB_TRY(make_tmap(&tA1, g.A1, g.M, g.K, g.batch, BM));
  VB_TRY(make_tmap(&tB1, g.B1, g.N, g.K, g.batch, C::B_ROWS));
  if (C::DUAL) {
    VB_TRY(make_tmap(&tA2, g.A2, g.M, g.K, g.batch, BM));
    VB_TRY(make_tmap(&tB2, g.B2, g.N, g.K, g.batch, C::B_ROWS));
  } else {
    tA2 = tA1; tB2 = tB1;
  }
  auto kern = gemm_tc_kernel<MODE, BN, CG, AK, BKM>;
  static bool attr_set = false;
  if (!attr_set) {
    VB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM_BYTES));
    attr_set = true;
  }
  const int tiles = sh.mt * sh.nt;
  const int num_work = (epi_z_accumulates(MODE) || sh.zsum) ? tiles : tiles * g.batch;
  static int sms = 0;
  if (!sms) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (sms <= 0) sms = kNumSMs;
  }
  // static: one persistent cluster per SM group; CLC: one cluster per work unit (the hardware keeps
  // #SM/CG resident, the rest are cancelled and absorbed by the resident ones)
  const int groups = sh.clc ? num_work : (num_work < sms / CG ? num_work : sms / CG);
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(groups * CG);
  cfg.blockDim = dim3(NTHREADS);
  cfg.dynamicSmemBytes = C::SMEM_BYTES;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CG; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  VB_CUDA(cudaLaunchKernelEx(&cfg, kern, tA1, tB1, tA2, tB2, sh, p));
  return VBNN_OK;
}

// Tile choice.  A CTA pair (cta_group::2) on a 256 x 256 tile halves the operand traffic per MAC
// (the 128 x 128 tile needs more L2->SM bandwidth than the chip has), so it wins whenever the
// problem has enough 256 x 256 tiles to fill the 74 pairs; small problems quantise better on
// 128 x 128 single-CTA tiles.  cost = waves x (tile MACs / relative per-MAC speed).
template <int MODE>
TcChoice choose_cfg(const GemmArgs& g) {
  const Knobs& k = knobs();
  TcChoice c{k.tc_bn, k.tc_cg};
  if ((c.bn == 128 || c.bn == 256) && (c.cg == 1 || c.cg == 2) && !(c.bn == 128 && c.cg == 2 && !epi_is_dual(MODE))) return c;
  if (epi_z_accumulates(MODE) && g.batch > 1) {
    // TMEM-resident accumulators: 128 x 128 tiles (1), or 256 x 128 CTA-pair tiles (2) when M allows
    if (k.tc_tacc && !epi_is_dual(MODE)) return TcChoice{128, k.tc_tacc == 2 && g.M >= 256 ? 2 : 1};
    if (k.tc_dw64) return TcChoice{64, 1};
  }
  const long long zmul = (epi_z_accumulates(MODE) || g.zsum) ? 1 : g.batch;
  auto cost = [&](int bn, int cg, double speed) {
    const long long work = (long long)ceil_div(g.M, BM * cg) * ceil_div(g.N, bn) * zmul;
    const long long slots = kNumSMs / cg;
    const long long waves = (work + slots - 1) / slots;
    return (double)waves * (double)bn / speed;      // each CTA computes 128 x bn per tile
  };
  const double c1 = cost(128, 1, 1.0), c2 = cost(256, 2, 1.45);
  return c2 <= c1 ? TcChoice{256, 2} : TcChoice{128, 1};
}

template <int MODE, bool AK, bool BKM>
int launch_any(const GemmArgs& g, const EpiParams& p, cudaStream_t st) {
  const TcChoice c = choose_cfg<MODE>(g);
  if constexpr (epi_z_accumulates(MODE)) {
    if (c.bn == 64) return launch_cfg<MODE, 64, 1, AK, BKM>(g, p, st);
    if constexpr (!epi_is_dual(MODE)) {
      if (c.bn == 128 && c.cg == 2) return launch_cfg<MODE, 128, 2, AK, BKM>(g, p, st);
    }
  }
  if constexpr (epi_is_dual(MODE)) {
    // 256 x 128 pair tile: two accumulators use 256 TMEM columns, so the accumulator is double-buffered
    if (c.cg == 2 && c.bn == 128) return launch_cfg<MODE, 128, 2, AK, BKM>(g, p, st);
  }
  if (c.cg == 2) return launch_cfg<MODE, 256, 2, AK, BKM>(g, p, st);
  if (c.bn == 256 && !epi_is_dual(MODE)) return launch_cfg<MODE, epi_is_dual(MODE) ? 128 : 256, 1, AK, BKM>(g, p, st);
  return launch_cfg<MODE, 128, 1, AK, BKM>(g, p, st);
}

}  // namespace

int gemm_tc_launch(int mode, const GemmArgs& g, const EpiParams& p, cudaStream_t st, long long* launches) {
  VB_CHECK(g.M > 0 && g.N > 0 && g.K > 0 && g.batch > 0, VBNN_E_INVALID,
           "gemm_tc: empty problem %d x %d x %d (batch %d)", g.M, g.N, g.K, g.batch);
  VB_CHECK(!g.zsum || !epi_z_accumulates(mode), VBNN_E_INVALID, "gemm_tc: the dW modes already sum over z");
  if (launches) *launches += 1;
  const bool ak = g.A1.kmajor != 0, bk = g.B1.kmajor != 0;
  switch (mode) {
    case EPI_STORE:
      if (ak && bk) return launch_any<EPI_STORE, true, true>(g, p, st);
      if (ak && !bk) return launch_any<EPI_STORE, true, false>(g, p, st);
      if (!ak && bk) return launch_any<EPI_STORE, false, true>(g, p, st);
      return launch_any<EPI_STORE, false, false>(g, p, st);
    case EPI_FWD:
      VB_CHECK(ak && bk, VBNN_E_INVALID, "EPI_FWD expects K-major operands");
      return launch_any<EPI_FWD, true, true>(g, p, st);
    case EPI_FWD_LRT:
      VB_CHECK(ak && bk, VBNN_E_INVALID, "EPI_FWD_LRT expects K-major operands");
      return launch_any<EPI_FWD_LRT, true, true>(g, p, st);
    case EPI_DX:
      VB_CHECK(ak && !bk, VBNN_E_INVALID, "EPI_DX expects K-major A, MN-major B");
      return launch_any<EPI_DX, true, false>(g, p, st);
    case EPI_DX_LRT:
      VB_CHECK(ak && !bk, VBNN_E_INVALID, "EPI_DX_LRT expects K-major A, MN-major B");
      return launch_any<EPI_DX_LRT, true, false>(g, p, st);
    case EPI_FWD_LRT2:
      VB_CHECK(ak && bk && p.aux, VBNN_E_INVALID, "EPI_FWD_LRT2 expects K-major operands and the mean product");
      return launch_any<EPI_FWD_LRT2, true, true>(g, p, st);
    case EPI_DX_LRT2:
      VB_CHECK(ak && !bk && p.aux, VBNN_E_INVALID, "EPI_DX_LRT2 expects K-major A, MN-major B and the H s2 product");
      return launch_any<EPI_DX_LRT2, true, false>(g, p, st);
    case EPI_DW:
      VB_CHECK(!ak && !bk, VBNN_E_INVALID, "EPI_DW expects MN-major operands");
      return launch_any<EPI_DW, false, false>(g, p, st);
    case EPI_DW_LRT:
      VB_CHECK(!ak && !bk, VBNN_E_INVALID, "EPI_DW_LRT expects MN-major operands");
      return launch_any<EPI_DW_LRT, false, false>(g, p, st);
  }
  set_error("gemm_tc_launch: bad mode %d", mode);
  return VBNN_E_INVALID;
}

}  // namespace vbnn
