// Engine knobs.  Every XPGNN_* environment variable is read ONCE, at the first use of the library; after that a knob
// changes only through xpgnn_set_option (include/xpgnn_b200.h) -- which is how the tests and the sweep tools compare
// kernel variants in one process.  All knobs select between implementations that compute the same function; nothing here
// skips work (the experiment switches of round 1 -- XPGNN_DENSE_EXP and friends -- are compiled out, see dense_tc.cu).
#pragma once
#include <stdint.h>

namespace xpgnn {

struct Knobs {
  int compact = 1;         // XPGNN_COMPACT: compact path for homogeneous stacks in full mode
  int compact_hetero = 1;  // XPGNN_COMPACT_HETERO
  int cw = 32;             // XPGNN_CW: 32 | 16 floats per activation chunk
  int l0_lists = 0;        // XPGNN_L0=lists: list-driven layer 0 instead of the row-outer kernels
  int occ = 8;             // XPGNN_OCC: CTAs / SM of the row-lockstep SpMM
  int seg = 7;             // XPGNN_SEG: 0 row-lockstep SpMM | 4 / 6 / 7 / 8 / 12 / 16 segmented SpMM with that many gathers in flight per lane
                           // (C3, ms per tile: 7 at 7 CTAs / SM 9.08, 8 at 7: 9.11, 8 at 6: 9.42, 6 at 7: 9.20, 12 at 5: 10.0, row-lockstep 11.7)
  int seg_skew = 0;        // XPGNN_SEG_SKEW: the `seg` value used instead when the graph has hub rows (skewed degrees: many short rows
                           // next to the long ones; R-MAT C3: 13.2 ms per tile with 4 in flight at 8 CTAs against 13.8 with 8 at 6); 0: same as seg
  int seg_pf = 0;          // XPGNN_SEG_PF: list entries per row the segmented kernel prefetches into registers during the previous block's epilogue (0 | 8 | 12 | 16); measured slower (register spills: 9.58 / 10.22 / 10.82 vs 9.50 ms per C3 tile)
  int seg_carve = 0;       // XPGNN_SEG_CARVE: > 0 = preferred shared-memory carve-out of the segmented kernel in percent (experiment: L1 size)
  int seg_occ = 0;         // XPGNN_SEG_OCC: 0 default CTAs / SM of the chosen segmented variant
  int seg_tma = 0;         // XPGNN_SEG_TMA: 1 = a small TMA gather4 kernel (compact_bulk.cu) runs next to the segmented SpMM on a second stream;
                           // both take blocks from the same in-order counter (bit-identical results)
  int l2_stream = 1;       // XPGNN_L2_STREAM / XPGNN_L2_GATHER: L2 eviction priority of streamed / gathered accesses
  int l2_gather = 0;
  int sched_static = 0;    // XPGNN_SCHED=static: static round-robin instead of the in-order work counter
  int act_column = 1;      // XPGNN_ACT_COLUMN: the compact path copies the tile's word of the coalition matrix into a dense [N] array first
  int l0_slices = 1;       // XPGNN_L0_SLICES: hub rows of layer 0 cut into 4096-in-edge slices, one CTA each (0: one CTA per hub row)
  int long_rows = 1;       // XPGNN_LONG=0: hub rows through the row-per-warp kernels
  int occ16 = 8;           // XPGNN_OCC16
  int l0_multi = 1;        // XPGNN_L0_MULTI
  int l1_multi = 0;        // XPGNN_L1_MULTI
  int l0_ws = 3;           // XPGNN_L0_WS: 0 one warp per row | 1 warp specialised, cp.async staging | 2 slot x column tiling |
                           // 3 (default) = 1 with the Z pieces staged by TMA bulk copies (UBLKCP): same arithmetic, bit-identical;
                           // measured at C3 4.91 vs 4.93 ms per tile, R-MAT 10.27 vs 10.32 (profiles/r02_summary.md)
  int l0_wait_ns = 2000;    // XPGNN_L0_WAIT_NS: the same for the warp-specialised layer-0 kernel
  int dense_wait_ns = 2000;  // XPGNN_DENSE_WAIT_NS: > 0 = waiting warps of dense_tc suspend inside mbarrier.try_wait (hint in ns) instead of polling
                           // (0 = poll + nanosleep; measured 3.94 -> 3.89 ms per C3 tile launch, layer 0 4.96 -> 4.95)
  int dense_tma = 1;       // XPGNN_DENSE_TMA: TF32x3 transforms of chunk-major 32-float inputs with tile-table rows load A by TMA gather4
                           // and feed the landed rows to the tensor core as the hi operand (bit-identical; 0: the register loaders)
  int dense_simt = 0;      // XPGNN_DENSE=simt: exact fp32 FMA transforms instead of 3xTF32 tensor-core products
  int prune_l0 = 1;        // XPGNN_PRUNE_L0
  int fused = 0;           // XPGNN_FUSED
  int fused_sb = 0;        // XPGNN_FUSED_SB
};

Knobs& knobs();                               // first call reads the environment
int set_knob(const char* name, int value);    // 0 ok, 1 unknown name
int get_knob(const char* name, int* value);

}  // namespace xpgnn
