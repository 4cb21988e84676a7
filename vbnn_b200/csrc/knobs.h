// knobs.h -- experiment / debugging switches of libvbnn.so.
//
// Every knob has a measured-best default; the environment variable VBNN_<NAME> (read once per
// process) or vbnn_debug_knob("<name>", value) (include/vbnn.h, self-test hooks; what the parity
// tests use to force a tile shape or a GEMM form in-process) overrides it.  None of them changes
// results beyond fp32 summation order, except dw_eps16, which also rounds epsilon to fp16 in the
// weight-mode gradSum (<= 2^-11 relative per product).  On operands where every fp32 partial sum is
// exact, every GEMM knob gives bit-identical logits, dX, gradWeight and gradBias
// (tests/test_gpu_multiwave.py).
#pragma once

namespace vbnn {

struct Knobs {
  int tc_bn = 0;        // force BLOCK_N of the tcgen05 kernel (128 / 256); 0 = cost model
  int tc_cg = 0;        // force the CTA-group size (1 / 2); 0 = cost model
  int tc_gm = 0;        // raster band height in m-tiles; 0 = per-class default
  int tc_clc = 1;       // cluster launch control (dynamic tile scheduling)
  int tc_l2hint = 0;    // L2 eviction priorities on the TMA operand loads (1: A band / resident weights evict-last; measured neutral, profiles/r02_traffic_sweep.md)
  int tc_staged = 1;    // coalesced epilogue I/O through the per-warp staging tiles
  int tc_tacc = 1;      // multi-sample dW: TMEM-resident accumulators (1: 128x128, 2: 256x128 pair)
  int tc_dw64 = 1;      // ... else the 128x64 register-accumulating form
  int dw_eps16 = 1;     // weight sampling, bf16: keep epsilon as fp16 for the dW epilogue instead of regenerating it
  int lrt_split = 1;    // bit 0: split LRT forward, bit 1: split LRT backward-data
  int dw_split = -1;    // LRT dW as two single-accumulator GEMMs: -1 = only in peer mode
  int dp_overlap = 1;   // NCCL mode: per-layer allreduce overlapped with backward
  int upd_bps = 4;      // fused update: 256-thread blocks per SM in its grid; read when a layer is created, so it applies
                        // to layers created after it is set (a layer's update grid and partial count stay fixed)
  int upd_coresident = 0;  // one GPU: run the 128-thread co-resident update variant (peer mode's) where it applies
                           // (I % 4 == 0, no diagnostics); for testing it without a second GPU
  int no_graph = 0;     // eager launches instead of CUDA graph replay
  int peer_transport = 0;  // gradient reduce-scatter: 0 = auto, 1 = NVLink stores from the dW epilogue, 2 = local staging + copy engines,
                           // 3 = local staging + one co-resident copy kernel per layer (transfer + signal fused)
  int peer_wire_bf16 = 0;  // staged transports, LRT layers: gradient tiles travel as bf16 (half the NVLink bytes; opt-in)
  int peer_one_stream = 0; // staged transports: run the gradient transfer on the update stream (one co-resident kernel at a time)
  int peer_push_ctas = 0;  // copy-kernel transport: CTAs per peer (0 = #SM / G)
  int peer_fused_push = 0; // operand all-gather: 0 = copy engines (SM-free), 1 = NVLink stores from the update kernel
};

Knobs& knobs();
// returns 0 on success, -1 for an unknown name; value == INT_MIN restores the env / default value
int knob_set(const char* name, int value);
int knob_get(const char* name, int* value);

}  // namespace vbnn
