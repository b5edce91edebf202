// Arguments of the dense row transform, shared by the SIMT (engine.cu) and tensor-core (dense_tc.cu) paths.
#pragma once
#include <cuda.h>

#include "common.cuh"

namespace xpgnn {

// out[m][n] (+)= act(sum_k in[m][k] w[n][k] + b[n]) (* row scale); m enumerates (coalition slot s, row) pairs.
//
// Two ways of naming the rows:
//   flat     : m = s * rows_per_s + rr, row = rows ? rows[rr] : row_lo + rr            (legacy tile path)
//   tile map : 128-row tile t -> (slot, first list position) = tile_map[t]; the slot's row list
//              slot_rows[slot][..] has slot_nrows[slot] live entries, known only on the device
//              (active nodes of a coalition: compact path, compact.cu)
// Two operand layouts: row-major (cw == 0, element k of a row at +k) and chunk-major (cw = 16 | 32:
// element k at (k / cw) * chunk_stride + k % cw, rows cw floats apart -- the layout the masked SpMM
// gathers from so that one (coalition, chunk) pass has an L2-resident working set).
struct DenseArgs {
  const float* in;
  int64_t in_s_stride;
  int ld_in, k;
  const float* w;  // [n_out][k]
  const float* b;
  int n_out;
  float* out;
  int64_t out_s_stride;
  int ld_out;
  const int32_t* rows;
  int rows_per_s, row_lo;  // rows == NULL: row = row_lo + (m % rows_per_s)
  int64_t M;               // n_slots * rows_per_s (flat) | worst-case tiles * 128 (tile map)
  int accumulate, act_fn;
  int dst_lo, dst_hi;      // rows outside [dst_lo, dst_hi) are skipped (row lists of hetero layers)
  // ---- chunk-major operands ----
  int cw_in, cw_in_lg, cw_out, cw_out_lg;  // 0: row-major
  int64_t in_chunk_stride, out_chunk_stride;
  // ---- tile table (device-side row counts): entry [tile * 128 + r] = slot << 26 | node id, or -1 ----
  const int32_t* rows_packed;
  const int32_t* n_tiles_dev;
  const float* rs_packed;      // optional row scale per entry: (1 + masked in-degree)^-1/2 (GCN operand of the next layer)
  // ---- bf16 activation storage (tensor-core bf16 mode only): `in` / `out` point at __nv_bfloat16, all strides in elements ----
  int in16, out16;
  int exp_flags;               // experiments only (XPGNN_DENSE_EXP): 1 skip stores, 2 skip loads, 4 skip MMAs
};
constexpr int kPackShift = 26;  // node ids < 2^26 in the packed tile table

__device__ __forceinline__ float apply_act(float x, int a) {
  if (a == XPGNN_ACT_RELU) return fmaxf(x, 0.0f);
  if (a == XPGNN_ACT_SIGMOID) return 1.0f / (1.0f + expf(-x));
  return x;
}

__device__ __forceinline__ float gcn_dinv(uint32_t masked_in_degree) { return 1.0f / sqrtf(1.0f + (float)masked_in_degree); }

struct DenseRow {
  int64_t io, oo;  // element offsets of the row's first element in `in` / `out`
  float rs;        // row scale of the epilogue
};

// row r (0..127) of 128-row tile `tile`; false: the row does not exist / is outside the destination range
__device__ __forceinline__ bool dense_resolve_row(const DenseArgs& a, int64_t tile, int r, DenseRow& o) {
  o.rs = 1.0f;
  if (a.rows_packed) {
    const int64_t pos = tile * 128 + r;
    const int32_t e = a.rows_packed[pos];
    if (e < 0) return false;
    const int64_t slot = (uint32_t)e >> kPackShift, v = e & ((1 << kPackShift) - 1);
    o.io = slot * a.in_s_stride + v * a.ld_in;
    o.oo = slot * a.out_s_stride + v * a.ld_out;
    if (a.rs_packed) o.rs = a.rs_packed[pos];
    return true;
  }
  const uint32_t m = (uint32_t)tile * 128u + (uint32_t)r;  // M < 2^31 (checked on the host): 32-bit div, not 64-bit
  if (m >= (uint32_t)a.M) return false;
  const uint32_t sl = m / (uint32_t)a.rows_per_s;
  const int rr = (int)(m - sl * (uint32_t)a.rows_per_s);
  const int v = a.rows ? a.rows[rr] : a.row_lo + rr;
  if (v < a.dst_lo || v >= a.dst_hi) return false;
  o.io = (int64_t)sl * a.in_s_stride + (int64_t)v * a.ld_in;
  o.oo = (int64_t)sl * a.out_s_stride + (int64_t)v * a.ld_out;
  return true;
}

__device__ __forceinline__ int64_t dense_in_off(const DenseArgs& a, int kk) {
  return a.cw_in ? (int64_t)(kk >> a.cw_in_lg) * a.in_chunk_stride + (kk & (a.cw_in - 1)) : (int64_t)kk;
}
__device__ __forceinline__ int64_t dense_out_off(const DenseArgs& a, int n) {
  return a.cw_out ? (int64_t)(n >> a.cw_out_lg) * a.out_chunk_stride + (n & (a.cw_out - 1)) : (int64_t)n;
}

enum { DENSE_SIMT = 0, DENSE_TC_BF16 = 1, DENSE_TC_TF32X3 = 2 };
bool dense_tc_eligible(const DenseArgs& d, int mode /*0 tf32x3, 1 bf16*/);
// 2-D tensor map over a float buffer seen as [rows][32 floats] with a 128-byte pitch, box = one row (the gather4 form loads
// four of them per instruction); swizzle128: land the rows in the K-major SWIZZLE_128B layout.  Cached per (base, rows, swizzle).
int rows128_tensor_map(const float* base, uint64_t rows, bool swizzle128, CUtensorMap* out);
int launch_dense_tc(const DenseArgs& d, int mode, cudaStream_t st);

}  // namespace xpgnn
