// Coalition-batched masked message passing (the hot path).
//
// Replaces, without materialising anything, the reference's block-diagonal perturbation
//   Data.perturbator / build_edge_mask / perturb_node / concat_features   (data.py:390-648)
// and the black-box forward it feeds
//   Model.infer / predict_hetero_output / extract_node_edge_output        (model.py:62-328)
// for stacks of PyG GCNConv / SAGEConv(mean) / HeteroConv(sum) + MLP head.
//
// Formulation (SURVEY.md section 7, verified against the materialised path by the oracle):
//   edge e=(u->v) is active in coalition s iff bit_s(act[u]) & bit_s(act[v]);
//   GCN : deg_s[v] = 1 + #active in-edges (input self loops dropped, one unit loop added),
//         out_s[v] = dinv_s[v] * ( sum_e a_e dinv_s[u] Z[u] + dinv_s[v] Z[v] ) + b
//   SAGE: out_s[v] = W_l * ( sum_e a_e x[u] / max(1, #active) ) + b_l + W_r x[v]
//   HeteroConv(sum): relations into the same destination type are summed.
// Layer 0 is transform-first (Z = X W^T is coalition invariant, computed once); deeper layers are
// aggregate-first (masked SpMM on the coalition-specific activations, then the dense transform).
// 32 coalitions share one bit word per node, so one AND per edge decides 32 coalitions.
#include <algorithm>
#include <vector>

#include <cstdlib>

#include "common.cuh"
#include "dense_args.cuh"
#include "fused.cuh"
#include "compact_internal.cuh"

namespace xpgnn {

// ------------------------------------------------------------------------------------------
// masked degrees -> per (node, coalition-in-word) normalisation
// ------------------------------------------------------------------------------------------
// CTA_ROW: rows above long_threshold in-edges (hub rows of power-law graphs) -- the CTA's warps take interleaved 32-edge
// batches and add their per-slot counts through shared memory; the warp-per-row launch skips those rows.
template <bool CTA_ROW>
__global__ void __launch_bounds__(256) masked_scale_kernel(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col,
                                                           const uint32_t* __restrict__ act, int W, int w, int row_lo, int row_hi,
                                                           int kind, float* __restrict__ scale, uint32_t* __restrict__ ebits,
                                                           unsigned long long* __restrict__ tile_active, int long_threshold) {
  __shared__ unsigned long long s_active[32];
  __shared__ int s_cnt[8][32];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5, wpb = blockDim.x >> 5;
  if (threadIdx.x < 32) s_active[threadIdx.x] = 0;
  __syncthreads();
  unsigned long long my_active = 0;
  for (int v = row_lo + (CTA_ROW ? blockIdx.x : blockIdx.x * wpb + wib); v < row_hi; v += CTA_ROW ? gridDim.x : gridDim.x * wpb) {
    const int e0 = rowptr[v], e1 = rowptr[v + 1];
    if (long_threshold > 0 && (CTA_ROW ? e1 - e0 <= long_threshold : e1 - e0 > long_threshold)) continue;  // CTA uniform when CTA_ROW
    const uint32_t av = act[(int64_t)v * W + w];
    int cnt = 0;
    for (int base = e0 + (CTA_ROW ? 32 * wib : 0); base < e1; base += CTA_ROW ? 32 * wpb : 32) {
      const int e = base + lane;
      uint32_t bits = 0;
      if (e < e1) {
        bits = act[(int64_t)col[e] * W + w] & av;
        ebits[e] = bits;  // bit b: edge e is active in coalition 32 w + b (read by every SpMM of the tile)
      }
      const int n = min(32, e1 - base);
      for (int j = 0; j < n; ++j) cnt += (__shfl_sync(0xffffffffu, bits, j) >> lane) & 1u;
    }
    if (CTA_ROW) {
      s_cnt[wib][lane] = cnt;
      __syncthreads();
      cnt = 0;
      for (int k = 0; k < wpb; ++k) cnt += s_cnt[k][lane];
      __syncthreads();
      if (wib != 0) continue;
    }
    scale[(int64_t)v * 32 + lane] = (kind == XPGNN_CONV_GCN) ? 1.0f / sqrtf(1.0f + (float)cnt) : 1.0f / (float)max(cnt, 1);
    my_active += cnt;
  }
  if (tile_active) {
    atomicAdd(&s_active[lane], my_active);
    __syncthreads();
    if (threadIdx.x < 32 && s_active[threadIdx.x]) atomicAdd(&tile_active[threadIdx.x], s_active[threadIdx.x]);
  }
}

// ------------------------------------------------------------------------------------------
// masked SpMM: one warp per destination row, lanes across the feature dimension, coalitions of
// the tile looped inside so that the row's column indices / activity words are read once.
// ------------------------------------------------------------------------------------------
constexpr int kLongRowTile = 1024;  // in-edges above which the tile path hands a row to a whole CTA
constexpr int kHubRows = 16;        // launches with at most this many rows split their hub rows over kHubSlices CTAs each
constexpr int kHubSlices = 64;

struct SpmmArgs {
  const int32_t* rowptr;
  const int32_t* col;
  const uint32_t* ebits;     // [E] per-edge activity word of the current 32-coalition word
  int b0, n_bits;            // first bit, coalitions in this tile
  const float* in;           // gathered operand; in[s * in_s_stride + u * ld_in + c]
  int64_t in_s_stride;       // 0: coalition-invariant operand (layer 0)
  int ld_in;
  const float* scale;        // [N][32] for this relation's CSR
  int kind;
  const int32_t* rows;       // optional row list
  int n_rows, row_lo;        // rows == NULL: rows [row_lo, row_lo + n_rows)
  int dst_lo, dst_hi;
  const float* addend;       // optional coalition-invariant addend [N][ld_add]
  int ld_add;
  float* out;                // out[s * out_s_stride + v * ld_out + c]
  int64_t out_s_stride;
  int ld_out;
  int accumulate, act_fn, H;
  int has_long_rows;         // the CSR has rows above kLongRowTile in-edges (host knows: max degree per unique CSR)
  float* hub_partial;        // [kHubRows][kHubSlices][32][H] scratch of the sliced hub-row path (tiny launches), or NULL
};

template <int VEC>
struct Vec;
template <>
struct Vec<4> {
  float v[4];
  __device__ __forceinline__ void load(const float* p) {
    const float4 t = __ldg(reinterpret_cast<const float4*>(p));
    v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
  }
  __device__ __forceinline__ void store(float* p) const { *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]); }
};
template <>
struct Vec<1> {
  float v[1];
  __device__ __forceinline__ void load(const float* p) { v[0] = __ldg(p); }
  __device__ __forceinline__ void store(float* p) const { *p = v[0]; }
};

template <int VEC>
__device__ __forceinline__ void gather_edges(const SpmmArgs& a, uint32_t m, int my_u, int b, const float* in_s, int c0, bool colok,
                                             float (&acc)[VEC]) {
  // m is warp uniform: every lane walks the same active edges
  while (m) {
    const int l0 = __ffs(m) - 1;
    m &= m - 1;
    const int l1 = m ? __ffs(m) - 1 : l0;
    const bool two = m != 0;
    m &= m - 1;
    const int u0 = __shfl_sync(0xffffffffu, my_u, l0);
    const int u1 = __shfl_sync(0xffffffffu, my_u, l1);
    float k0 = 1.0f, k1 = 1.0f;
    if (a.kind == XPGNN_CONV_GCN) {
      k0 = __ldg(a.scale + (int64_t)u0 * 32 + b);
      k1 = __ldg(a.scale + (int64_t)u1 * 32 + b);
    }
    if (colok) {
      Vec<VEC> x0, x1;
      x0.load(in_s + (int64_t)u0 * a.ld_in + c0);
      if (two) x1.load(in_s + (int64_t)u1 * a.ld_in + c0);
#pragma unroll
      for (int i = 0; i < VEC; ++i) acc[i] = fmaf(k0, x0.v[i], acc[i]);
      if (two) {
#pragma unroll
        for (int i = 0; i < VEC; ++i) acc[i] = fmaf(k1, x1.v[i], acc[i]);
      }
    }
  }
}

// CTA_ROW: hub rows (more than long_threshold in-edges) -- a whole CTA takes the row and its warps split the coalition
// slots, instead of one warp walking e.g. 82 K in-edges x 32 slots alone (the pruned last layer of a hub query is
// exactly one such row).
template <int VEC, bool CTA_ROW>
__global__ void __launch_bounds__(256, 4) spmm_masked_kernel(const SpmmArgs a) {
  // Row-outer, coalition-inner: a row's column indices and edge-activity words are read once and stay
  // in registers for all coalitions of the tile (<= 64 in-edges; longer rows re-read them from L1).
  // (The coalition-outer order was measured in round 1: 32x more row visits made it latency bound,
  //  l1 23.7 -> 29.5 ms, l0 12.2 -> 29.9 ms -- see DESIGN.md.)
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5, wpb = blockDim.x >> 5;
  const int chunks = (a.H + 32 * VEC - 1) / (32 * VEC);
  for (int r = CTA_ROW ? blockIdx.x : blockIdx.x * wpb + wib; r < a.n_rows; r += CTA_ROW ? gridDim.x : gridDim.x * wpb) {
    const int v = a.rows ? a.rows[r] : a.row_lo + r;
    if (v < a.dst_lo || v >= a.dst_hi) continue;
    const int e0 = a.rowptr[v], e1 = a.rowptr[v + 1], deg = e1 - e0;
    if (CTA_ROW ? deg <= kLongRowTile : deg > kLongRowTile) continue;  // hub rows belong to the CTA_ROW launch
    const float sc_lane = a.scale[(int64_t)v * 32 + lane];
    int u_reg[2] = {-1, -1};
    uint32_t bits_reg[2] = {0u, 0u};
    if (deg <= 64) {
#pragma unroll
      for (int k = 0; k < 2; ++k) {
        const int e = e0 + 32 * k + lane;
        if (e < e1) {
          u_reg[k] = __ldg(a.col + e);
          bits_reg[k] = __ldg(a.ebits + e);
        }
      }
    }
    for (int cc = 0; cc < chunks; ++cc) {
      const int c0 = cc * 32 * VEC + lane * VEC;
      const bool colok = c0 < a.H;
      for (int s = CTA_ROW ? wib : 0; s < a.n_bits; s += CTA_ROW ? wpb : 1) {
        const int b = a.b0 + s;
        const float* in_s = a.in + (int64_t)s * a.in_s_stride;
        float acc[VEC];
#pragma unroll
        for (int i = 0; i < VEC; ++i) acc[i] = 0.0f;
        if (deg <= 64) {
          gather_edges<VEC>(a, __ballot_sync(0xffffffffu, (bits_reg[0] >> b) & 1u), u_reg[0], b, in_s, c0, colok, acc);
          if (deg > 32)
            gather_edges<VEC>(a, __ballot_sync(0xffffffffu, (bits_reg[1] >> b) & 1u), u_reg[1], b, in_s, c0, colok, acc);
        } else {
          for (int base = e0; base < e1; base += 32) {
            const int e = base + lane;
            int u = -1;
            uint32_t bits = 0;
            if (e < e1) {
              u = __ldg(a.col + e);
              bits = __ldg(a.ebits + e);
            }
            gather_edges<VEC>(a, __ballot_sync(0xffffffffu, (bits >> b) & 1u), u, b, in_s, c0, colok, acc);
          }
        }
        const float dv = __shfl_sync(0xffffffffu, sc_lane, b);
        if (colok) {
          Vec<VEC> o;
          if (a.kind == XPGNN_CONV_GCN) {
            Vec<VEC> self;
            self.load(in_s + (int64_t)v * a.ld_in + c0);
#pragma unroll
            for (int i = 0; i < VEC; ++i) o.v[i] = dv * fmaf(dv, self.v[i], acc[i]);
          } else {
#pragma unroll
            for (int i = 0; i < VEC; ++i) o.v[i] = dv * acc[i];
          }
          if (a.addend) {
            Vec<VEC> ad;
            ad.load(a.addend + (int64_t)v * a.ld_add + c0);
#pragma unroll
            for (int i = 0; i < VEC; ++i) o.v[i] += ad.v[i];
          }
          float* op = a.out + (int64_t)s * a.out_s_stride + (int64_t)v * a.ld_out + c0;
          if (a.accumulate) {
            Vec<VEC> prev;
            prev.load(op);
#pragma unroll
            for (int i = 0; i < VEC; ++i) o.v[i] += prev.v[i];
          }
#pragma unroll
          for (int i = 0; i < VEC; ++i) o.v[i] = apply_act(o.v[i], a.act_fn);
          o.store(op);
        }
      }
    }
  }
}

// Hub rows of a TINY launch (the pruned last layer of a query is one row; a hub query's row has e.g. 82 K in-edges): one
// CTA per row leaves 147 SMs idle, so the row's in-edges are cut into kHubSlices slices, one CTA each (its warps split the
// slots as above), partial sums go to scratch and a second kernel adds the slices in a fixed order (deterministic) and
// runs the row epilogue.
template <int VEC>
__global__ void __launch_bounds__(256, 4) spmm_hub_slices_kernel(const SpmmArgs a) {
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5, wpb = blockDim.x >> 5;
  const int r = blockIdx.x / kHubSlices, j = blockIdx.x % kHubSlices;
  const int v = a.rows ? a.rows[r] : a.row_lo + r;
  if (v < a.dst_lo || v >= a.dst_hi) return;
  const int e0 = a.rowptr[v], e1 = a.rowptr[v + 1], deg = e1 - e0;
  if (deg <= kLongRowTile) return;
  const int per = ((deg + kHubSlices - 1) / kHubSlices + 31) & ~31;  // slice length, whole 32-edge batches
  const int bs = e0 + j * per, be = min(e1, bs + per);
  const int chunks = (a.H + 32 * VEC - 1) / (32 * VEC);
  for (int cc = 0; cc < chunks; ++cc) {
    const int c0 = cc * 32 * VEC + lane * VEC;
    const bool colok = c0 < a.H;
    for (int s = wib; s < a.n_bits; s += wpb) {
      const int b = a.b0 + s;
      const float* in_s = a.in + (int64_t)s * a.in_s_stride;
      float acc[VEC];
#pragma unroll
      for (int i = 0; i < VEC; ++i) acc[i] = 0.0f;
      for (int base = bs; base < be; base += 32) {
        const int e = base + lane;
        int u = -1;
        uint32_t bits = 0;
        if (e < be) {
          u = __ldg(a.col + e);
          bits = __ldg(a.ebits + e);
        }
        gather_edges<VEC>(a, __ballot_sync(0xffffffffu, (bits >> b) & 1u), u, b, in_s, c0, colok, acc);
      }
      if (colok) {
        Vec<VEC> o;
#pragma unroll
        for (int i = 0; i < VEC; ++i) o.v[i] = acc[i];
        o.store(a.hub_partial + (((int64_t)r * kHubSlices + j) * 32 + s) * a.H + c0);
      }
    }
  }
}

template <int VEC>
__global__ void __launch_bounds__(256) spmm_hub_reduce_kernel(const SpmmArgs a) {
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5, wpb = blockDim.x >> 5;
  const int r = blockIdx.x;
  const int v = a.rows ? a.rows[r] : a.row_lo + r;
  if (v < a.dst_lo || v >= a.dst_hi) return;
  if (a.rowptr[v + 1] - a.rowptr[v] <= kLongRowTile) return;
  const int chunks = (a.H + 32 * VEC - 1) / (32 * VEC);
  for (int cc = 0; cc < chunks; ++cc) {
    const int c0 = cc * 32 * VEC + lane * VEC;
    if (c0 >= a.H) continue;
    for (int s = wib; s < a.n_bits; s += wpb) {
      const float* in_s = a.in + (int64_t)s * a.in_s_stride;
      float acc[VEC];
#pragma unroll
      for (int i = 0; i < VEC; ++i) acc[i] = 0.0f;
      for (int j = 0; j < kHubSlices; ++j) {
        Vec<VEC> pj;
        pj.load(a.hub_partial + (((int64_t)r * kHubSlices + j) * 32 + s) * a.H + c0);
#pragma unroll
        for (int i = 0; i < VEC; ++i) acc[i] += pj.v[i];
      }
      const float dv = a.scale[(int64_t)v * 32 + a.b0 + s];
      Vec<VEC> o;
      if (a.kind == XPGNN_CONV_GCN) {
        Vec<VEC> self;
        self.load(in_s + (int64_t)v * a.ld_in + c0);
#pragma unroll
        for (int i = 0; i < VEC; ++i) o.v[i] = dv * fmaf(dv, self.v[i], acc[i]);
      } else {
#pragma unroll
        for (int i = 0; i < VEC; ++i) o.v[i] = dv * acc[i];
      }
      if (a.addend) {
        Vec<VEC> ad;
        ad.load(a.addend + (int64_t)v * a.ld_add + c0);
#pragma unroll
        for (int i = 0; i < VEC; ++i) o.v[i] += ad.v[i];
      }
      float* op = a.out + (int64_t)s * a.out_s_stride + (int64_t)v * a.ld_out + c0;
      if (a.accumulate) {
        Vec<VEC> prev;
        prev.load(op);
#pragma unroll
        for (int i = 0; i < VEC; ++i) o.v[i] += prev.v[i];
      }
#pragma unroll
      for (int i = 0; i < VEC; ++i) o.v[i] = apply_act(o.v[i], a.act_fn);
      o.store(op);
    }
  }
}

// ------------------------------------------------------------------------------------------
// dense row transform, exact fp32 SIMT path (tensor-core path: dense_tc.cu)
// ------------------------------------------------------------------------------------------
constexpr int DBM = 64, DBN = 64, DBK = 16;

__global__ void __launch_bounds__(256) dense_rows_kernel(const DenseArgs a) {
  __shared__ float As[DBK][DBM + 4];
  __shared__ float Bs[DBK][DBN + 4];
  __shared__ int64_t in_off[DBM], out_off[DBM];
  __shared__ float row_scale[DBM];
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int64_t tile = blockIdx.x >> 1;  // 128-row tile of the shared row naming (dense_args.cuh); this CTA takes one half
  if (a.rows_packed && tile >= *a.n_tiles_dev) return;
  const int n0 = blockIdx.y * DBN;
  if (tid < DBM) {
    DenseRow row;
    const bool ok = dense_resolve_row(a, tile, (blockIdx.x & 1) * DBM + tid, row);
    in_off[tid] = ok ? row.io : -1;
    out_off[tid] = ok ? row.oo : -1;
    row_scale[tid] = row.rs;
  }
  __syncthreads();
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.0f;
  const int lr = tid >> 2, lk = (tid & 3) * 4;  // each thread stages 4 consecutive k of one row
  for (int k0 = 0; k0 < a.k; k0 += DBK) {
    const int64_t io = in_off[lr];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int kk = k0 + lk + i;
      As[lk + i][lr] = (io >= 0 && kk < a.k) ? __ldg(a.in + io + dense_in_off(a, kk)) : 0.0f;
      const int n = n0 + lr;
      Bs[lk + i][lr] = (n < a.n_out && kk < a.k) ? __ldg(a.w + (int64_t)n * a.k + kk) : 0.0f;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < DBK; ++kk) {
      float av[4], bv[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) av[i] = As[kk][ty * 4 + i];
#pragma unroll
      for (int j = 0; j < 4; ++j) bv[j] = Bs[kk][tx * 4 + j];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int64_t oo = out_off[ty * 4 + i];
    if (oo < 0) continue;
    const float rs = row_scale[ty * 4 + i];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int n = n0 + tx * 4 + j;
      if (n >= a.n_out) continue;
      float x = acc[i][j] + (a.b ? __ldg(a.b + n) : 0.0f);
      float* op = a.out + oo + dense_out_off(a, n);
      if (a.accumulate) x += *op;
      *op = apply_act(x, a.act_fn) * rs;
    }
  }
}

// ------------------------------------------------------------------------------------------
// MLP head on the query rows (one CTA per (coalition slot, query)).
// ------------------------------------------------------------------------------------------
constexpr int kMaxHead = 8;
struct HeadArgs {
  int n_layers;
  xpgnn_dense_t l[kMaxHead];
  const float* in;
  int64_t in_s_stride;
  int ld_in, dim0;
  const int32_t* query;
  int n_query, out_col;
  float* y;        // y[slot * n_query + q]
  const unsigned long long* tile_active;  // zero-edge rule (NULL: off)
  int b0;
};

__global__ void __launch_bounds__(128) head_kernel(const HeadArgs a, int max_dim) {
  extern __shared__ float sm[];
  float* x0 = sm;
  float* x1 = sm + max_dim;
  const int slot = blockIdx.x / a.n_query, q = blockIdx.x % a.n_query;
  const float* src = a.in + (int64_t)slot * a.in_s_stride + (int64_t)a.query[q] * a.ld_in;
  for (int i = threadIdx.x; i < a.dim0; i += blockDim.x) x0[i] = src[i];
  __syncthreads();
  for (int li = 0; li < a.n_layers; ++li) {
    const xpgnn_dense_t& L = a.l[li];
    for (int n = threadIdx.x; n < L.out; n += blockDim.x) {
      float s = 0.0f;
      const float* wr = L.w + (int64_t)n * L.in;
      for (int k = 0; k < L.in; ++k) s = fmaf(x0[k], __ldg(wr + k), s);
      if (L.b) s += __ldg(L.b + n);
      x1[n] = apply_act(s, L.act);
    }
    __syncthreads();
    float* t = x0; x0 = x1; x1 = t;
  }
  if (threadIdx.x == 0) {
    float r = x0[a.out_col];
    if (a.tile_active && a.tile_active[a.b0 + slot] == 0ull) r = 0.0f;  // model.py:213-215
    a.y[(int64_t)slot * a.n_query + q] = r;
  }
}

__global__ void add_into_kernel(float* __restrict__ acc, const float* __restrict__ x, int n, int first) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) acc[i] = first ? x[i] : acc[i] + x[i];
}

__global__ void max_degree_kernel(const int32_t* __restrict__ rowptr, int lo, int hi, int32_t* __restrict__ out) {
  const int v = lo + blockIdx.x * blockDim.x + threadIdx.x;
  int d = v < hi ? rowptr[v + 1] - rowptr[v] : 0;
  d = __reduce_max_sync(0xffffffffu, d);
  if ((threadIdx.x & 31) == 0 && d > kLongRowTile) atomicMax(out, d);
}

__global__ void rows_by_hop_kernel(const int8_t* __restrict__ hop, int N, int max_hop, int32_t* __restrict__ rows, int32_t* __restrict__ count) {
  const int v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v < N && hop[v] >= 0 && hop[v] <= max_hop) rows[atomicAdd(count, 1)] = v;
}

// hub rows (more than `threshold` in-edges) among the rows of a list
__global__ void long_rows_of_list_kernel(const int32_t* __restrict__ rows, int n, const int32_t* __restrict__ rowptr, int threshold,
                                         int32_t* __restrict__ out, int32_t* __restrict__ count) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int v = rows[i];
  if (rowptr[v + 1] - rowptr[v] > threshold) out[atomicAdd(count, 1)] = v;
}

__global__ void stats_accum_kernel(const unsigned long long* tile_active, int n_bits, int b0, long long mult, int64_t* stats) {
  unsigned long long t = 0;
  for (int b = 0; b < n_bits; ++b) t += tile_active[b0 + b];
  stats[1] += (int64_t)t * mult;
  stats[3] += 1;
}

// ------------------------------------------------------------------------------------------ host side
Profile g_prof;

// precision: DENSE_SIMT exact fp32 FMA | DENSE_TC_TF32X3 fp32 via 3 TF32 MMAs | DENSE_TC_BF16
int launch_dense(const DenseArgs& d, cudaStream_t st, int precision) {
  if (d.M <= 0 || d.n_out <= 0) return 0;
  ProfScope ps(PROF_DENSE, st);
  if (precision != DENSE_SIMT && (d.M >= 1024 || d.in16 || d.out16)) {
    const int mode = precision == DENSE_TC_BF16 ? 1 : 0;
    if (dense_tc_eligible(d, mode)) return launch_dense_tc(d, mode, st);
  }
  XP_REQUIRE(!d.in16 && !d.out16, "bf16 activation storage needs the tensor-core transform (shape not eligible)");
  dim3 grid((unsigned)(2 * ceil_div(d.M, 2 * DBM)), (unsigned)ceil_div(d.n_out, DBN));
  XP_LAUNCH(dense_rows_kernel, grid, 256, 0, st, d);
  return 0;
}

static int launch_spmm(const SpmmArgs& s, cudaStream_t st) {
  if (s.n_rows <= 0 || s.n_bits <= 0) return 0;
  ProfScope ps(s.in_s_stride == 0 ? PROF_SPMM_INVARIANT : PROF_SPMM_TILE, st);
  const int grid = (int)std::min<int64_t>(ceil_div(s.n_rows, 8), (int64_t)kNumSMs * 16);
  const bool vec4 = (s.H % 4 == 0) && (s.ld_in % 4 == 0) && (s.ld_out % 4 == 0) && (s.in_s_stride % 4 == 0) &&
                    (s.out_s_stride % 4 == 0) && (((uintptr_t)s.in | (uintptr_t)s.out) % 16 == 0) &&
                    (!s.addend || (s.ld_add % 4 == 0 && (uintptr_t)s.addend % 16 == 0));
  void (*k)(const SpmmArgs) = vec4 ? spmm_masked_kernel<4, false> : spmm_masked_kernel<1, false>;
  XP_LAUNCH(k, grid, 256, 0, st, s);
  if (s.has_long_rows && s.hub_partial && s.n_rows <= kHubRows) {  // few rows: every hub row over kHubSlices CTAs
    void (*ks)(const SpmmArgs) = vec4 ? spmm_hub_slices_kernel<4> : spmm_hub_slices_kernel<1>;
    void (*kr)(const SpmmArgs) = vec4 ? spmm_hub_reduce_kernel<4> : spmm_hub_reduce_kernel<1>;
    XP_LAUNCH(ks, s.n_rows * kHubSlices, 256, 0, st, s);
    XP_LAUNCH(kr, s.n_rows, 256, 0, st, s);
  } else if (s.has_long_rows) {  // hub rows: one CTA per row, warps split the slots
    const int grid_long = (int)std::min<int64_t>(s.n_rows, (int64_t)kNumSMs * 8);
    void (*kl)(const SpmmArgs) = vec4 ? spmm_masked_kernel<4, true> : spmm_masked_kernel<1, true>;
    XP_LAUNCH(kl, grid_long, 256, 0, st, s);
  }
  return 0;
}

struct Layout {
  std::vector<float*> zn;      // layer-0 per-relation transformed sources (biased pointer: index by global id)
  float* r0 = nullptr;         // layer-0 coalition-invariant addend
  std::vector<float*> scale;   // per unique CSR
  std::vector<uint32_t*> ebits; // per unique CSR: activity word of every edge for the current coalition word
  unsigned long long* tile_active = nullptr;
  float* hbuf[2] = {nullptr, nullptr};
  float* agg = nullptr;
  std::vector<std::vector<float*>> wimg;  // per layer >= 1, per relation: TF32 hi/lo image of W for the fused kernel
  std::vector<std::vector<float*>> wroot; // per layer >= 1, per relation: sum of the SAGE root weights of its destination group
  std::vector<int32_t*> rows;  // per layer (prune)
  int32_t* row_counts = nullptr;
  float* hub_partial = nullptr;  // sliced hub rows of tiny launches (prune)
  int32_t* l0_counter = nullptr; // row counter of the layer-0 row kernel (prune)
  int32_t* l0_long = nullptr;    // hub rows among the layer-0 row list (prune)
  int32_t *l0_item_row = nullptr, *l0_item_slice = nullptr, *l0_row_item0 = nullptr;  // their slices (compact_l0.cu)
  float2* l0_slice_scratch = nullptr;
  int64_t bytes = 0;
};

struct UniqueCsr {
  const int32_t* rowptr;
  const int32_t* col;
  int kind, lo, hi, n_edges;
};

static void collect_unique(const xpgnn_plan_t* p, std::vector<UniqueCsr>& uniq, std::vector<std::vector<int>>& map) {
  map.resize(p->n_layers);
  for (int l = 0; l < p->n_layers; ++l) {
    const xpgnn_layer_t& L = p->layers_host[l];
    map[l].resize(L.n_rel);
    for (int r = 0; r < L.n_rel; ++r) {
      const xpgnn_relation_t& R = L.rel_host[r];
      int id = -1;
      for (size_t i = 0; i < uniq.size(); ++i)
        if (uniq[i].rowptr == R.rowptr && uniq[i].col == R.col && uniq[i].kind == R.conv_kind) id = (int)i;
      if (id < 0) {
        uniq.push_back({R.rowptr, R.col, R.conv_kind, R.dst_lo, R.dst_hi, R.n_edges});
        id = (int)uniq.size() - 1;
      }
      map[l][r] = id;
    }
  }
}

static Layout carve(const xpgnn_plan_t* p, void* ws, int64_t cap, int tile, const std::vector<UniqueCsr>& uniq) {
  Layout lay;
  Bump b(ws, cap);
  const int64_t N = p->n_nodes;
  const xpgnn_layer_t& L0 = p->layers_host[0];
  for (int r = 0; r < L0.n_rel; ++r) {
    const xpgnn_relation_t& R = L0.rel_host[r];
    float* z = b.take<float>((int64_t)(R.src_hi - R.src_lo) * L0.h_out);
    lay.zn.push_back(z ? z - (int64_t)R.src_lo * L0.h_out : nullptr);
  }
  lay.r0 = b.take<float>(N * L0.h_out);
  for (size_t i = 0; i < uniq.size(); ++i) {
    lay.scale.push_back(b.take<float>(N * 32));
    lay.ebits.push_back(b.take<uint32_t>(std::max(uniq[i].n_edges, 1)));
  }
  lay.tile_active = b.take<unsigned long long>(32);
  int hmax = 0, kmax = 0;
  for (int l = 0; l < p->n_layers; ++l) {
    hmax = std::max(hmax, p->layers_host[l].h_out);
    if (l > 0) kmax = std::max(kmax, p->layers_host[l].h_in);
  }
  lay.hbuf[0] = b.take<float>((int64_t)tile * N * hmax);
  if (p->n_layers > 1) {
    lay.hbuf[1] = b.take<float>((int64_t)tile * N * hmax);
    lay.agg = b.take<float>((int64_t)tile * N * kmax);
  }
  lay.wroot.resize(p->n_layers);
  for (int l = 1; l < p->n_layers; ++l)
    for (int r = 0; r < p->layers_host[l].n_rel; ++r)
      lay.wroot[l].push_back(b.take<float>((int64_t)p->layers_host[l].h_out * p->layers_host[l].h_in));
  lay.wimg.resize(p->n_layers);
  for (int l = 1; l < p->n_layers; ++l)
    for (int r = 0; r < p->layers_host[l].n_rel; ++r)
      lay.wimg[l].push_back(b.take<float>(fused_w_image_bytes((p->layers_host[l].h_in + 31) / 32 * 32, p->layers_host[l].h_out) / 4));
  if (p->prune) {
    for (int l = 0; l < p->n_layers; ++l) lay.rows.push_back(b.take<int32_t>(N));
    lay.row_counts = b.take<int32_t>(p->n_layers);
    lay.hub_partial = b.take<float>((int64_t)kHubRows * kHubSlices * 32 * std::max(hmax, kmax));
    lay.l0_counter = b.take<int32_t>(64);
    lay.l0_long = b.take<int32_t>(N);
    if (p->n_layers > 0 && p->layers_host[0].n_rel == 1) {  // sliced hub rows of the pruned layer 0 (homogeneous stacks)
      const int64_t e0 = std::max(p->layers_host[0].rel_host[0].n_edges, 1), items = l0_long_items_max(e0);
      lay.l0_item_row = b.take<int32_t>(items);
      lay.l0_item_slice = b.take<int32_t>(items);
      lay.l0_row_item0 = b.take<int32_t>(e0 / kLongRowTile + 2);
      lay.l0_slice_scratch = b.take<float2>(l0_slice_scratch_items(e0) * (p->layers_host[0].h_out / 64 + 1) * 1024);
    }
  }
  lay.bytes = (b.off + 255) & ~255ll;
  return lay;
}

}  // namespace xpgnn

using namespace xpgnn;

extern "C" {

int xpgnn_profile(int32_t enable) {
  g_prof.reset();
  g_prof.on = enable != 0;
  return 0;
}

int xpgnn_profile_read(double* ms_host, int64_t* launches_host) {
  XP_REQUIRE(ms_host && launches_host, "null argument");
  for (int c = 0; c < PROF_N; ++c) {
    double tot = 0.0;
    for (auto& e : g_prof.ev[c]) {
      XP_CHECK(cudaEventSynchronize(e.second));
      float ms = 0.f;
      XP_CHECK(cudaEventElapsedTime(&ms, e.first, e.second));
      tot += ms;
    }
    ms_host[c] = tot;
    launches_host[c] = (int64_t)g_prof.ev[c].size();
  }
  return 0;
}

int64_t xpgnn_forward_workspace_bytes(const xpgnn_plan_t* plan, int32_t tile_coalitions) {
  if (!plan || plan->n_layers < 1 || tile_coalitions < 1 || tile_coalitions > 32) return -1;
  if (compact_eligible(plan)) return compact_workspace_bytes(plan, tile_coalitions);
  if (compact_hetero_eligible(plan)) return compact_hetero_workspace_bytes(plan, tile_coalitions);
  std::vector<UniqueCsr> uniq;
  std::vector<std::vector<int>> map;
  collect_unique(plan, uniq, map);
  return carve(plan, nullptr, 0, tile_coalitions, uniq).bytes;
}

int xpgnn_dense_rows(const float* in, int64_t rows, int32_t k, int32_t ld_in, const float* w, const float* b, int32_t n_out,
                     int32_t act, float* out, int32_t ld_out, int32_t accumulate, int32_t precision, void* stream) {
  XP_REQUIRE(in && w && out && rows >= 0 && rows < (1ll << 31) && k > 0 && n_out > 0, "bad argument");
  XP_REQUIRE(precision >= 0 && precision <= 2, "precision must be 0 (fp32 SIMT), 1 (bf16 tcgen05) or 2 (tf32x3 tcgen05)");
  if (rows == 0) return 0;  // nothing to transform, in every precision (the tensor-core shape check wants rows > 0)
  DenseArgs d{};
  d.in = in; d.ld_in = ld_in; d.k = k; d.w = w; d.b = b; d.n_out = n_out; d.out = out; d.ld_out = ld_out;
  d.rows_per_s = (int)rows; d.M = rows; d.accumulate = accumulate; d.act_fn = act; d.dst_lo = 0; d.dst_hi = (int)rows;
  if (precision != DENSE_SIMT) {
    XP_REQUIRE(dense_tc_eligible(d, precision == DENSE_TC_BF16 ? 1 : 0), "shape not eligible for the tensor-core path");
    ProfScope ps(PROF_DENSE, (cudaStream_t)stream);
    return launch_dense_tc(d, precision == DENSE_TC_BF16 ? 1 : 0, (cudaStream_t)stream);
  }
  return launch_dense(d, (cudaStream_t)stream, DENSE_SIMT);
}

int xpgnn_forward(const xpgnn_plan_t* p, const uint32_t* act, int32_t W, int32_t s0, int32_t n_s, float* y, void* workspace,
                  int64_t workspace_bytes, int64_t* stats, void* stream) {
  XP_REQUIRE(p && act && workspace && (y || n_s == 0), "null argument");  // an empty range may come with an empty output
  XP_REQUIRE(p->n_layers >= 1 && p->n_nodes > 0 && p->n_query > 0 && p->query, "empty plan");
  XP_REQUIRE(s0 % 32 == 0 && n_s >= 0 && (int64_t)W * 32 >= (int64_t)s0 + n_s, "coalition range outside the bit matrix");
  XP_REQUIRE(p->n_head <= kMaxHead, "head deeper than 8 layers");
  XP_REQUIRE(p->precision >= 0 && p->precision <= 2, "plan precision must be 0 (fp32), 1 (bf16 transforms) or 2 (bf16 transforms + bf16 activation storage)");
  // fp32 plans use the 3xTF32 tensor-core transform (error ~2^-20) unless XPGNN_DENSE=simt forces exact FMA
  const int dense_prec = p->precision >= 1 ? DENSE_TC_BF16 : (knobs().dense_simt ? DENSE_SIMT : DENSE_TC_TF32X3);
  XP_REQUIRE(!p->prune || p->hop, "prune = 1 needs the hop levels");
  if (n_s == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  if (compact_eligible(p)) return forward_compact(p, act, W, s0, n_s, y, workspace, workspace_bytes, stats, st, dense_prec);
  if (compact_hetero_eligible(p)) return forward_compact_hetero(p, act, W, s0, n_s, y, workspace, workspace_bytes, stats, st, dense_prec);
  const int N = p->n_nodes, NL = p->n_layers;

  std::vector<UniqueCsr> uniq;
  std::vector<std::vector<int>> umap;
  collect_unique(p, uniq, umap);
  int tile = 32;
  while (tile > 1 && carve(p, nullptr, 0, tile, uniq).bytes > workspace_bytes) tile >>= 1;
  XP_REQUIRE(carve(p, nullptr, 0, tile, uniq).bytes <= workspace_bytes, "workspace too small even for one coalition per tile");
  Layout lay = carve(p, workspace, workspace_bytes, tile, uniq);
  int hmax = 0;
  for (int l = 0; l < NL; ++l) hmax = std::max(hmax, p->layers_host[l].h_out);
  const int64_t hstride = (int64_t)N * hmax;  // per-slot stride of the activation buffers

  // ---- hub rows (a property of the graph): which CSRs have rows above kLongRowTile in-edges ----
  std::vector<int32_t> max_deg(uniq.size(), 0);
  {
    Scratch sc(st);
    XP_CHECK(sc.alloc(sizeof(int32_t) * uniq.size()));
    XP_CHECK(cudaMemsetAsync(sc.p, 0, sizeof(int32_t) * uniq.size(), st));
    for (size_t i = 0; i < uniq.size(); ++i) {
      const int rows = uniq[i].hi - uniq[i].lo;
      if (rows > 0) XP_LAUNCH(max_degree_kernel, (int)ceil_div(rows, 256), 256, 0, st, uniq[i].rowptr, uniq[i].lo, uniq[i].hi, sc.as<int32_t>() + i);
    }
    XP_CHECK(cudaMemcpyAsync(max_deg.data(), sc.p, sizeof(int32_t) * uniq.size(), cudaMemcpyDeviceToHost, st));
    XP_CHECK(cudaStreamSynchronize(st));
  }

  // ---- needed rows per layer (prune) ----
  std::vector<int> n_rows(NL, N);
  if (p->prune) {
    XP_CHECK(cudaMemsetAsync(lay.row_counts, 0, sizeof(int32_t) * NL, st));
    for (int l = 0; l < NL; ++l)
      XP_LAUNCH(rows_by_hop_kernel, (int)ceil_div(N, 256), 256, 0, st, p->hop, N, NL - 1 - l, lay.rows[l], lay.row_counts + l);
    std::vector<int32_t> h(NL);
    XP_CHECK(cudaMemcpyAsync(h.data(), lay.row_counts, sizeof(int32_t) * NL, cudaMemcpyDeviceToHost, st));
    XP_CHECK(cudaStreamSynchronize(st));
    for (int l = 0; l < NL; ++l) n_rows[l] = h[l];
  }

  // ---- coalition-invariant part of layer 0: Z_r = X W_r^T, R0 = sum_r (b_r + X W_root,r^T) ----
  const xpgnn_layer_t& L0 = p->layers_host[0];
  // pruned homogeneous stacks run layer 0 through the row-outer kernels of compact_l0.cu (see the layer loop)
  const bool prune_l0_env = knobs().prune_l0 != 0;
  const bool prune_l0 = prune_l0_env && p->prune && NL > 1 && L0.n_rel == 1 && L0.rel_host[0].src_lo == 0 && L0.rel_host[0].src_hi == N &&
                        L0.rel_host[0].dst_lo == 0 && L0.rel_host[0].dst_hi == N && L0.h_out % 64 == 0 &&
                        (int64_t)N * L0.h_out < (int64_t(1) << 31) && n_rows[0] > n_rows[1];
  int32_t n_long0 = 0, n_items0 = 0;
  const bool l0_slices = knobs().l0_slices != 0 && lay.l0_item_row != nullptr && L0.h_out / 64 <= 4 && kLongRowTile == kLongRow;
  if (prune_l0 && max_deg[umap[0][0]] > kLongRowTile) {
    XP_CHECK(cudaMemsetAsync(lay.l0_counter + 1, 0, sizeof(int32_t), st));
    XP_LAUNCH(long_rows_of_list_kernel, (int)ceil_div(n_rows[0], 256), 256, 0, st, lay.rows[0], n_rows[0], L0.rel_host[0].rowptr, kLongRowTile,
              lay.l0_long, lay.l0_counter + 1);
    XP_CHECK(cudaMemcpyAsync(&n_long0, lay.l0_counter + 1, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    if (l0_slices) {
      if (build_l0_long_items(L0.rel_host[0].rowptr, lay.l0_long, lay.l0_counter + 1, lay.l0_item_row, lay.l0_item_slice, lay.l0_row_item0,
                              lay.l0_counter + 2, st))
        return 1;
      XP_CHECK(cudaMemcpyAsync(&n_items0, lay.l0_counter + 2, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    }
    XP_CHECK(cudaStreamSynchronize(st));
  }
  XP_REQUIRE(L0.h_in == p->f_in, "layer 0 input width != feature width");
  XP_CHECK(cudaMemsetAsync(lay.r0, 0, sizeof(float) * (int64_t)N * L0.h_out, st));
  for (int r = 0; r < L0.n_rel; ++r) {
    const xpgnn_relation_t& R = L0.rel_host[r];
    DenseArgs z{};
    z.in = p->x; z.ld_in = p->f_in; z.k = p->f_in; z.w = R.w_nbr; z.n_out = L0.h_out; z.out = lay.zn[r]; z.ld_out = L0.h_out;
    z.rows_per_s = R.src_hi - R.src_lo; z.row_lo = R.src_lo; z.M = z.rows_per_s; z.dst_lo = 0; z.dst_hi = N;
    if (launch_dense(z, st, dense_prec)) return 1;
    // R0 += b_r (+ X W_root,r^T for SAGE) on the destination range; k = 0 degenerates to "add the bias"
    const bool sage_root = R.conv_kind == XPGNN_CONV_SAGE_MEAN && R.w_root;
    if (sage_root || R.b_nbr) {
      DenseArgs rt = z;
      rt.k = sage_root ? p->f_in : 0; rt.w = sage_root ? R.w_root : R.w_nbr; rt.b = R.b_nbr; rt.out = lay.r0;
      rt.rows_per_s = R.dst_hi - R.dst_lo; rt.row_lo = R.dst_lo; rt.M = rt.rows_per_s; rt.accumulate = 1;
      if (launch_dense(rt, st, dense_prec)) return 1;
    }
  }

  // first / last relation touching each destination range, per layer
  auto first_last = [&](const xpgnn_layer_t& L, std::vector<char>& first, std::vector<char>& last) {
    first.assign(L.n_rel, 1);
    last.assign(L.n_rel, 1);
    for (int r = 0; r < L.n_rel; ++r)
      for (int q = 0; q < L.n_rel; ++q)
        if (q != r && L.rel_host[q].dst_lo == L.rel_host[r].dst_lo && L.rel_host[q].dst_hi == L.rel_host[r].dst_hi) {
          if (q < r) first[r] = 0;
          if (q > r) last[r] = 0;
        }
  };

  // ---- fused SpMM + tcgen05 transform for layers >= 1 (single relation per destination range, no row list) ----

  // opt-in (XPGNN_FUSED=1): at one 512-thread CTA per SM its gather / MMA / epilogue phases do not overlap and it
  // measured 49.7 ms per C3 tile against 23.1 + 18.8 ms for the unfused pair (profiles/r01_summary.md)
  const bool fused_on = dense_prec == DENSE_TC_TF32X3 && !p->prune && knobs().fused == 1;
  const int fused_sb = knobs().fused_sb;
  std::vector<std::vector<char>> use_fused(NL);
  for (int l = 1; l < NL; ++l) {
    const xpgnn_layer_t& L = p->layers_host[l];
    std::vector<char> first, last;
    first_last(L, first, last);
    use_fused[l].assign(L.n_rel, 0);
    for (int r = 0; r < L.n_rel; ++r) {
      const xpgnn_relation_t& R = L.rel_host[r];
      const bool sage_root = R.conv_kind == XPGNN_CONV_SAGE_MEAN && R.w_root;
      if (fused_on && first[r] && last[r] && !sage_root &&
          fused_eligible(L.h_in, L.h_out, hmax, hmax, hstride, hstride, lay.hbuf[0], lay.hbuf[1])) {
        use_fused[l][r] = 1;
        if (fused_build_w_image(R.w_nbr, L.h_out, L.h_in, lay.wimg[l][r], st)) return 1;
      }
    }
  }

  // HeteroConv(sum) adds W_root,r x[v] once per relation into the same destination type: one transform with the summed
  // root weights per destination group instead (at C4: 15 of the 40 dense launches of a layer)
  std::vector<std::vector<char>> group_root(NL);
  for (int l = 1; l < NL; ++l) {
    const xpgnn_layer_t& L = p->layers_host[l];
    std::vector<char> first, last;
    first_last(L, first, last);
    group_root[l].assign(L.n_rel, 0);
    for (int r = 0; r < L.n_rel; ++r) {
      if (!last[r]) continue;
      int n_root = 0;
      const int nw = L.h_out * L.h_in;
      for (int q = 0; q <= r; ++q) {
        const xpgnn_relation_t& Q = L.rel_host[q];
        if (Q.dst_lo != L.rel_host[r].dst_lo || Q.dst_hi != L.rel_host[r].dst_hi) continue;
        if (Q.conv_kind != XPGNN_CONV_SAGE_MEAN || !Q.w_root) continue;
        XP_LAUNCH(add_into_kernel, (int)ceil_div(nw, 256), 256, 0, st, lay.wroot[l][r], Q.w_root, nw, n_root == 0);
        ++n_root;
      }
      group_root[l][r] = n_root > 0;
    }
  }

  const int w_first = s0 / 32, w_last = (s0 + n_s - 1) / 32;
  for (int w = w_first; w <= w_last; ++w) {
    const int bits_in_word = std::min(32, s0 + n_s - w * 32);
    XP_CHECK(cudaMemsetAsync(lay.tile_active, 0, sizeof(unsigned long long) * 32, st));
    for (size_t i = 0; i < uniq.size(); ++i) {
      const int rows = uniq[i].hi - uniq[i].lo;
      const int grid = (int)std::min<int64_t>(std::max<int64_t>(ceil_div(rows, 8), 1), (int64_t)kNumSMs * 8);
      ProfScope ps(PROF_SCALE, st);
      const int thr = max_deg[i] > kLongRowTile ? kLongRowTile : 0;
      XP_LAUNCH(masked_scale_kernel<false>, grid, 256, 0, st, uniq[i].rowptr, uniq[i].col, act, W, w, uniq[i].lo, uniq[i].hi,
                uniq[i].kind, lay.scale[i], lay.ebits[i], lay.tile_active, thr);
      if (thr > 0)
        XP_LAUNCH(masked_scale_kernel<true>, (int)std::min<int64_t>(rows, (int64_t)kNumSMs * 8), 256, 0, st, uniq[i].rowptr, uniq[i].col, act, W,
                  w, uniq[i].lo, uniq[i].hi, uniq[i].kind, lay.scale[i], lay.ebits[i], lay.tile_active, thr);
    }
    for (int b0 = 0; b0 < bits_in_word; b0 += tile) {
      const int nb = std::min(tile, bits_in_word - b0);
      float* cur = lay.hbuf[0];
      float* nxt = lay.hbuf[1];
      for (int l = 0; l < NL; ++l) {
        const xpgnn_layer_t& L = p->layers_host[l];
        std::vector<char> first, last;
        first_last(L, first, last);
        for (int r = 0; r < L.n_rel; ++r) {
          const xpgnn_relation_t& R = L.rel_host[r];
          SpmmArgs s{};
          s.rowptr = R.rowptr; s.col = R.col; s.ebits = lay.ebits[umap[l][r]]; s.b0 = b0; s.n_bits = nb;
          s.scale = lay.scale[umap[l][r]]; s.kind = R.conv_kind; s.has_long_rows = max_deg[umap[l][r]] > kLongRowTile;
          s.rows = p->prune ? lay.rows[l] : nullptr;
          s.n_rows = p->prune ? n_rows[l] : (R.dst_hi - R.dst_lo);
          s.row_lo = R.dst_lo; s.dst_lo = R.dst_lo; s.dst_hi = R.dst_hi; s.hub_partial = lay.hub_partial;
          if (l == 0) {  // transform-first: gather the coalition-invariant Z_r, accumulate relations in place
            s.in = lay.zn[r]; s.in_s_stride = 0; s.ld_in = L.h_out; s.H = L.h_out;
            s.addend = first[r] ? lay.r0 : nullptr; s.ld_add = L.h_out;
            s.out = cur; s.out_s_stride = hstride; s.ld_out = hmax;
            s.accumulate = !first[r]; s.act_fn = last[r] ? L.act : XPGNN_ACT_NONE;
            // Pruned homogeneous stacks (what Explainer.run builds for GCN / SAGE models): the needed rows of layer 0 through
            // the row-outer kernel of the compact path (a source row crosses the fabric once per destination row, not once per
            // (row, slot)), writing the row-major tile buffer.  It produces the (row, slot) pairs in which the row is ACTIVE --
            // all that active edges of the next layer gather; the rows the next layer reads in EVERY slot (self / root term
            // of its own row list) and the hub rows follow through the tile kernel.
            if (prune_l0) {
              L0RowsArgs a{};
              a.rowptr = R.rowptr; a.col = R.col; a.ebits = s.ebits; a.act = act; a.W = W; a.w = w; a.b0 = b0; a.nb = nb; a.N = N;
              a.scale = s.scale; a.z = lay.zn[r]; a.h0 = L.h_out; a.bias = nullptr;
              a.r0c = lay.r0; a.r0_chunk_stride = 32; a.r0_row_stride = L.h_out;
              a.out = cur; a.out_s_stride = hstride; a.out_chunk_stride = 32; a.out_row_stride = hmax;
              a.kind = R.conv_kind; a.act_fn = L.act; a.prescale = 0;
              a.long_threshold = n_long0 > 0 ? kLongRowTile : 0; a.counter = lay.l0_counter;
              a.row_lo = 0; a.row_hi = N; a.rows = lay.rows[0]; a.n_list = n_rows[0]; a.accumulate = 0; a.finish = 1;
              XP_CHECK(cudaMemsetAsync(lay.l0_counter, 0, sizeof(int32_t), st));
              {
                ProfScope ps(PROF_SPMM_INVARIANT, st);
                if (launch_l0_rows(a, L.act == XPGNN_ACT_SIGMOID, false, n_rows[0], st)) return 1;
              }
              if (n_long0 > 0) {  // hub rows of the list: one CTA per row
                a.long_rows = lay.l0_long;
                if (l0_slices && n_items0 <= l0_slice_scratch_items(std::max(R.n_edges, 1))) {
                  a.item_row = lay.l0_item_row; a.item_slice = lay.l0_item_slice; a.row_item0 = lay.l0_row_item0;
                  a.slice_scratch = lay.l0_slice_scratch;
                }
                ProfScope ps(PROF_SPMM_INVARIANT, st);
                if (launch_l0_long_rows(a, L.act == XPGNN_ACT_SIGMOID, false, n_long0, st, n_items0)) return 1;
              }
              s.rows = lay.rows[1]; s.n_rows = n_rows[1];  // every slot of the rows the next layer reads as its own
            }
            if (launch_spmm(s, st)) return 1;
          } else if (use_fused[l][r]) {  // aggregate + transform in one kernel, the aggregate never leaves the SM
            FusedArgs f{};
            f.rowptr = R.rowptr; f.col = R.col; f.ebits = lay.ebits[umap[l][r]]; f.scale = lay.scale[umap[l][r]];
            f.kind = R.conv_kind; f.in = cur; f.in_s_stride = hstride; f.ld_in = hmax; f.K = L.h_in;
            f.w_image = lay.wimg[l][r]; f.b = R.b_nbr; f.n_out = L.h_out; f.out = nxt; f.out_s_stride = hstride;
            f.ld_out = hmax; f.act_fn = L.act; f.row_lo = R.dst_lo; f.n_rows = R.dst_hi - R.dst_lo;
            f.b0 = b0; f.n_bits = nb; f.SB = fused_sb; f.slot_major = fused_sb > 0 && fused_sb < 32;
            ProfScope ps(PROF_SPMM_TILE, st);
            if (launch_fused(f, st)) return 1;
          } else {       // aggregate-first: masked SpMM on the activations, then the dense transform
            s.in = cur; s.in_s_stride = hstride; s.ld_in = hmax; s.H = L.h_in;
            s.addend = nullptr; s.ld_add = 0;
            s.out = lay.agg; s.out_s_stride = (int64_t)N * L.h_in; s.ld_out = L.h_in;
            s.accumulate = 0; s.act_fn = XPGNN_ACT_NONE;
            if (launch_spmm(s, st)) return 1;
            const bool sage_root = last[r] && group_root[l][r];  // merged root transform of the destination group
            DenseArgs d{};
            d.in = lay.agg; d.in_s_stride = (int64_t)N * L.h_in; d.ld_in = L.h_in; d.k = L.h_in; d.w = R.w_nbr; d.b = R.b_nbr;
            d.n_out = L.h_out; d.out = nxt; d.out_s_stride = hstride; d.ld_out = hmax;
            d.rows = p->prune ? lay.rows[l] : nullptr;
            d.rows_per_s = p->prune ? n_rows[l] : (R.dst_hi - R.dst_lo); d.row_lo = R.dst_lo;
            d.M = (int64_t)nb * d.rows_per_s; d.accumulate = !first[r];
            d.act_fn = (last[r] && !sage_root) ? L.act : XPGNN_ACT_NONE;
            d.dst_lo = R.dst_lo; d.dst_hi = R.dst_hi;  // a pruned row list may hold rows of other node types
            if (launch_dense(d, st, dense_prec)) return 1;
            if (sage_root) {
              DenseArgs rt = d;
              rt.in = cur; rt.in_s_stride = hstride; rt.ld_in = hmax; rt.w = lay.wroot[l][r]; rt.b = nullptr;
              rt.accumulate = 1; rt.act_fn = L.act;
              if (launch_dense(rt, st, dense_prec)) return 1;
            }
          }
        }
        if (l > 0) std::swap(cur, nxt);
        if (l == 0 && NL > 1) { /* layer-0 output lives in hbuf[0] == cur */ }
      }
      // ---- head on the query rows ----
      HeadArgs h{};
      h.n_layers = p->n_head;
      int max_dim = p->layers_host[NL - 1].h_out;
      for (int i = 0; i < p->n_head; ++i) {
        h.l[i] = p->head_host[i];
        max_dim = std::max(max_dim, std::max(p->head_host[i].in, p->head_host[i].out));
      }
      h.in = cur; h.in_s_stride = hstride; h.ld_in = hmax; h.dim0 = p->layers_host[NL - 1].h_out;
      h.query = p->query; h.n_query = p->n_query; h.out_col = p->out_col;
      h.y = y + ((int64_t)(w * 32 + b0) - s0) * p->n_query;
      h.tile_active = p->zero_edge_rule ? lay.tile_active : nullptr;
      h.b0 = b0;
      {
        ProfScope ps(PROF_HEAD, st);
        XP_LAUNCH(head_kernel, nb * p->n_query, 128, sizeof(float) * 2 * max_dim, st, h, max_dim);
      }
      if (stats) {
        long long mult = 0;
        for (int l = 0; l < NL; ++l) mult += p->layers_host[l].n_rel;  // every layer walks every relation once
        XP_LAUNCH(stats_accum_kernel, 1, 1, 0, st, lay.tile_active, nb, b0, mult / std::max<size_t>(uniq.size(), 1), stats);
      }
    }
  }
  return 0;
}

}  // extern "C"
