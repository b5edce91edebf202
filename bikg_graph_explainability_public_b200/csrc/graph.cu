// k-hop computational graph (frontier BFS over the COO edge list) and CSR construction.
//
// Replaces Data.comp_graph (data.py:281-361) and the PyG k_hop_subgraph it calls: per hop one
// coalesced pass over the E edges marks the sources of edges whose target is in the frontier
// (flow = source_to_target); the final pass keeps every edge with both ends in the node set, in
// original order, relabelled by the rank of the node id (subset is ascending, like torch.unique).
// Stream compaction / sorting use CUB device primitives (plumbing, not the hot path).
#include <cub/cub.cuh>

#include "common.cuh"

namespace xpgnn {

__global__ void khop_init_kernel(int8_t* hop, uint8_t* frontier, int64_t N, int64_t query) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i < N) {
    hop[i] = (i == query) ? 0 : -1;
    frontier[i] = (i == query) ? 1 : 0;
  }
}

// one pass: next[src] = 1 for every edge whose dst is in cur.  PyG re-expands the whole previous
// layer (visited nodes included), so `next` is not filtered by `hop`.
__global__ void __launch_bounds__(256) khop_expand_kernel(const int64_t* __restrict__ src, const int64_t* __restrict__ dst, int64_t E,
                                                          int64_t N, const uint8_t* __restrict__ cur, uint8_t* __restrict__ next) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < E; e += stride) {
    const int64_t s = src[e], d = dst[e];
    if ((uint64_t)s >= (uint64_t)N || (uint64_t)d >= (uint64_t)N) continue;  // counted by khop_validate_kernel
    if (cur[d]) next[s] = 1;
  }
}

// endpoints outside [0, N): PyG raises an index error; here they are counted (counts[2]) and the edge is ignored
__global__ void __launch_bounds__(256) khop_validate_kernel(const int64_t* __restrict__ src, const int64_t* __restrict__ dst, int64_t E,
                                                            int64_t N, int64_t* __restrict__ n_bad) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  int bad = 0;
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < E; e += stride)
    bad += ((uint64_t)src[e] >= (uint64_t)N) || ((uint64_t)dst[e] >= (uint64_t)N);
  bad = __reduce_add_sync(0xffffffffu, bad);
  if ((threadIdx.x & 31) == 0 && bad) atomicAdd(reinterpret_cast<unsigned long long*>(n_bad), (unsigned long long)bad);
}

__global__ void khop_mark_kernel(int8_t* hop, const uint8_t* next, int64_t N, int level) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i < N && next[i] && hop[i] < 0) hop[i] = (int8_t)level;
}

__global__ void khop_nodeflag_kernel(const int8_t* hop, int32_t* flag, int64_t N) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i < N) flag[i] = hop[i] >= 0;
}

__global__ void khop_relabel_kernel(const int8_t* hop, const int32_t* rank, int64_t N, int32_t* relabel, int64_t* subset) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i < N) {
    if (hop[i] >= 0) {
      relabel[i] = rank[i];
      subset[rank[i]] = i;
    } else {
      relabel[i] = -1;
    }
  }
}

__global__ void __launch_bounds__(256) khop_edgeflag_kernel(const int64_t* __restrict__ src, const int64_t* __restrict__ dst, int64_t E,
                                                            int64_t N, const int8_t* __restrict__ hop, uint8_t* __restrict__ edge_mask,
                                                            int32_t* __restrict__ flag) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < E; e += stride) {
    const int64_t s = src[e], d = dst[e];
    const bool ok = (uint64_t)s < (uint64_t)N && (uint64_t)d < (uint64_t)N;
    const int k = ok && (hop[s] >= 0) && (hop[d] >= 0);
    edge_mask[e] = (uint8_t)k;
    flag[e] = k;
  }
}

__global__ void __launch_bounds__(256) khop_edgewrite_kernel(const int64_t* __restrict__ src, const int64_t* __restrict__ dst, int64_t E,
                                                             const int32_t* __restrict__ flag, const int32_t* __restrict__ rank,
                                                             const int32_t* __restrict__ relabel, int64_t* __restrict__ out) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < E; e += stride)
    if (flag[e]) {
      out[rank[e]] = relabel[src[e]];
      out[E + rank[e]] = relabel[dst[e]];
    }
}

__global__ void khop_counts_kernel(const int32_t* nflag, const int32_t* nrank, int64_t N, const int32_t* eflag, const int32_t* erank,
                                   int64_t E, const int32_t* relabel, int64_t query, int64_t* sub_edge_index, int64_t* counts) {
  const int64_t ns = N > 0 ? nrank[N - 1] + nflag[N - 1] : 0;
  int64_t es = E > 0 ? erank[E - 1] + eflag[E - 1] : 0;
  if (es == 0) {  // data.py:337-339: leave at least the node self connected
    sub_edge_index[0] = relabel[query];
    sub_edge_index[E > 0 ? E : 1] = relabel[query];
    es = 1;
  }
  counts[0] = ns;
  counts[1] = es;
}

// ---------------------------------------------------------------- CSR
__global__ void __launch_bounds__(256) csr_key_kernel(const int64_t* __restrict__ src, const int64_t* __restrict__ dst, int64_t E, int drop,
                                                      int32_t sentinel, int32_t* __restrict__ key, int32_t* __restrict__ val) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < E; e += stride) {
    const int64_t s = src[e], d = dst[e];
    key[e] = (drop && s == d) ? sentinel : (int32_t)d;  // dropped edges sort behind every row
    val[e] = (int32_t)s;
  }
}

__global__ void __launch_bounds__(256) csr_rowptr_kernel(const int32_t* __restrict__ sorted_key, int64_t E, int32_t N, int32_t* __restrict__ rowptr,
                                                         int64_t* __restrict__ n_kept) {
  // rowptr[r] = first position whose key >= r  (keys sorted ascending; sentinel N sorts last)
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; r <= N; r += stride) {
    int64_t lo = 0, hi = E;
    while (lo < hi) {
      int64_t mid = (lo + hi) >> 1;
      if (sorted_key[mid] < r) lo = mid + 1; else hi = mid;
    }
    rowptr[r] = (int32_t)lo;
    if (r == N) n_kept[0] = lo;
  }
}

// ---------------------------------------------------------------- multi-query k-hop
// F[h][v] bit q: v is in the level-h frontier of query q.  The union of the levels is the reach word.
constexpr int kMqBlocks = kNumSMs * 4;  // count / emit grids: each block owns one contiguous chunk

__device__ __forceinline__ uint64_t mq_reach(const uint64_t* __restrict__ F, int levels, int64_t N, int64_t v) {
  uint64_t r = 0;
  for (int h = 0; h < levels; ++h) r |= F[(int64_t)h * N + v];
  return r;
}

// bit q of item i: node i is in query q's graph (nodes) / edge i has both ends in it (edges)
template <bool EDGES>
__device__ __forceinline__ uint64_t mq_item(const uint64_t* __restrict__ F, int levels, int64_t N, const int64_t* __restrict__ src,
                                            const int64_t* __restrict__ dst, int64_t i) {
  if (!EDGES) return mq_reach(F, levels, N, i);
  const int64_t s = src[i], d = dst[i];
  if ((uint64_t)s >= (uint64_t)N || (uint64_t)d >= (uint64_t)N) return 0;
  return mq_reach(F, levels, N, s) & mq_reach(F, levels, N, d);
}

__device__ __forceinline__ uint64_t warp_or64(uint64_t m) {
  const uint32_t lo = __reduce_or_sync(0xffffffffu, (uint32_t)m), hi = __reduce_or_sync(0xffffffffu, (uint32_t)(m >> 32));
  return ((uint64_t)hi << 32) | lo;
}

__global__ void mq_init_kernel(uint64_t* F0, const int64_t* __restrict__ queries, int Q, int64_t N) {
  const int q = threadIdx.x;
  if (q < Q && (uint64_t)queries[q] < (uint64_t)N) atomicOr(reinterpret_cast<unsigned long long*>(F0 + queries[q]), 1ull << q);
}

// one pass over the edges for every query: next[src] |= cur[dst].  The read filters the atomics: a hub source already
// holding the bits is not written again.
__global__ void __launch_bounds__(256) mq_expand_kernel(const int64_t* __restrict__ src, const int64_t* __restrict__ dst, int64_t E,
                                                        int64_t N, const uint64_t* __restrict__ cur, uint64_t* next) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < E; e += stride) {
    const int64_t s = src[e], d = dst[e];
    if ((uint64_t)s >= (uint64_t)N || (uint64_t)d >= (uint64_t)N) continue;
    const uint64_t b = cur[d];
    if (b && (b & ~*((volatile uint64_t*)(next + s)))) atomicOr(reinterpret_cast<unsigned long long*>(next + s), b);
  }
}

// per block and query: number of items (nodes / edges) of the block's chunk that belong to the query (warp ballots per
// query bit present in the warp)
template <bool EDGES>
__global__ void __launch_bounds__(256) mq_count_kernel(const uint64_t* __restrict__ F, int levels, int64_t N, const int64_t* __restrict__ src,
                                                       const int64_t* __restrict__ dst, int64_t total, int64_t chunk,
                                                       int32_t* __restrict__ blk) {
  __shared__ int32_t cnt[64];
  if (threadIdx.x < 64) cnt[threadIdx.x] = 0;
  __syncthreads();
  const int64_t lo = blockIdx.x * chunk, hi = min(total, lo + chunk);
  for (int64_t base = lo; base < hi; base += 256) {
    const int64_t i = base + threadIdx.x;
    const uint64_t m = i < hi ? mq_item<EDGES>(F, levels, N, src, dst, i) : 0;
    uint64_t wor = warp_or64(m);
    while (wor) {
      const int q = __ffsll((long long)wor) - 1;
      wor &= wor - 1;
      const uint32_t b = __ballot_sync(0xffffffffu, (m >> q) & 1);
      if ((threadIdx.x & 31) == 0) atomicAdd(&cnt[q], __popc(b));
    }
  }
  __syncthreads();
  if (threadIdx.x < 64) blk[blockIdx.x * 64 + threadIdx.x] = cnt[threadIdx.x];
}

// grid (Q, 2): one warp scans query q's block counts (y = 0 nodes, 1 edges) into exclusive bases; totals -> counts
__global__ void mq_scan_kernel(int32_t* __restrict__ node_blk, int32_t* __restrict__ edge_blk, int G, int Q, int64_t* __restrict__ counts) {
  const int q = blockIdx.x, lane = threadIdx.x;
  int32_t* c = blockIdx.y ? edge_blk : node_blk;
  int32_t run = 0;
  for (int g0 = 0; g0 < G; g0 += 32) {
    const int g = g0 + lane;
    const int32_t v = g < G ? c[g * 64 + q] : 0;
    int32_t incl = v;
    for (int o = 1; o < 32; o <<= 1) {
      const int32_t t = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += t;
    }
    if (g < G) c[g * 64 + q] = run + incl - v;
    run += __shfl_sync(0xffffffffu, incl, 31);
  }
  if (lane == 0) counts[blockIdx.y * Q + q] = run;
}

__device__ __forceinline__ int64_t lower_bound_i64(const int64_t* __restrict__ a, int64_t n, int64_t x) {
  int64_t lo = 0, hi = n;
  while (lo < hi) {
    const int64_t mid = (lo + hi) >> 1;
    if (a[mid] < x) lo = mid + 1; else hi = mid;
  }
  return lo;
}

struct MqEmitArgs {
  const int64_t* node_off;
  const int64_t* edge_off;
  int64_t n_union_edges;
  int64_t* subset;
  int8_t* level;
  int64_t* sub_ind;
  int64_t* sub_ei;
  int64_t* edge_id;
};

// same chunks and tile order as mq_count_kernel; the position of an item inside its query's block is the scanned block
// base + the running count of earlier tiles + the counts of earlier warps + the ballot prefix inside the warp
template <bool EDGES>
__global__ void __launch_bounds__(256) mq_emit_kernel(const uint64_t* __restrict__ F, int levels, int64_t N, const int64_t* __restrict__ src,
                                                      const int64_t* __restrict__ dst, int64_t total, int64_t chunk,
                                                      const int32_t* __restrict__ blk, MqEmitArgs a) {
  __shared__ uint32_t bal[8][64];
  __shared__ int32_t wcnt[8][64];
  __shared__ int32_t run[64];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  if (threadIdx.x < 64) run[threadIdx.x] = blk[blockIdx.x * 64 + threadIdx.x];
  const int64_t lo = blockIdx.x * chunk, hi = min(total, lo + chunk);
  const int64_t* off = EDGES ? a.edge_off : a.node_off;
  for (int64_t base = lo; base < hi; base += 256) {
    const int64_t i = base + threadIdx.x;
    const uint64_t m = i < hi ? mq_item<EDGES>(F, levels, N, src, dst, i) : 0;
    wcnt[wib][lane] = 0;
    wcnt[wib][lane + 32] = 0;
    __syncwarp();
    uint64_t wor = warp_or64(m);
    while (wor) {
      const int q = __ffsll((long long)wor) - 1;
      wor &= wor - 1;
      const uint32_t b = __ballot_sync(0xffffffffu, (m >> q) & 1);
      if (lane == 0) {
        bal[wib][q] = b;
        wcnt[wib][q] = __popc(b);
      }
    }
    __syncthreads();
    uint64_t own = m;
    while (own) {
      const int q = __ffsll((long long)own) - 1;
      own &= own - 1;
      int32_t r = run[q] + __popc(bal[wib][q] & ((1u << lane) - 1u));
      for (int w = 0; w < wib; ++w) r += wcnt[w][q];
      const int64_t pos = off[q] + r;
      if (!EDGES) {
        int h = 0;
        while (!((F[(int64_t)h * N + i] >> q) & 1)) ++h;
        a.subset[pos] = i;
        a.level[pos] = (int8_t)h;
        if (h == 0) a.sub_ind[q] = r;
      } else {
        const int64_t n0 = a.node_off[q], nq = a.node_off[q + 1] - n0;
        a.sub_ei[pos] = n0 + lower_bound_i64(a.subset + n0, nq, src[i]);
        a.sub_ei[a.n_union_edges + pos] = n0 + lower_bound_i64(a.subset + n0, nq, dst[i]);
        if (a.edge_id) a.edge_id[pos] = i;
      }
    }
    __syncthreads();
    if (threadIdx.x < 64) {
      int32_t t = 0;
      for (int w = 0; w < 8; ++w) t += wcnt[w][threadIdx.x];
      run[threadIdx.x] += t;
    }
    __syncthreads();
  }
}

// data.py:337-339 per query: a query without an induced edge keeps one self loop
__global__ void mq_self_loop_kernel(const int64_t* __restrict__ counts, int Q, MqEmitArgs a) {
  const int q = threadIdx.x;
  if (q >= Q || counts[Q + q] != 0) return;
  const int64_t pos = a.edge_off[q], v = a.node_off[q] + a.sub_ind[q];
  a.sub_ei[pos] = v;
  a.sub_ei[a.n_union_edges + pos] = v;
  if (a.edge_id) a.edge_id[pos] = -1;
}

inline int64_t mq_chunk(int64_t total) { return std::max<int64_t>(ceil_div(ceil_div(total, kMqBlocks), 256) * 256, 256); }

}  // namespace xpgnn

using namespace xpgnn;

extern "C" {

int xpgnn_khop_subgraph(const int64_t* edge_index, int64_t E, int64_t N, int64_t query, int32_t hops, int64_t* subset,
                        int32_t* relabel, int8_t* hop, uint8_t* edge_mask, int64_t* sub_edge_index, int64_t* counts,
                        void* stream) {
  XP_REQUIRE(N > 0 && query >= 0 && query < N, "query outside [0, N)");
  XP_REQUIRE(E >= 0 && hops >= 0 && hops < 127, "bad E / hops");
  XP_REQUIRE(N < (1ll << 31) - 1 && E < (1ll << 31) - 1, "N/E out of int32 range (the scans and ranks are 32-bit)");
  XP_REQUIRE(subset && relabel && hop && counts && sub_edge_index && (edge_mask || E == 0), "null output");
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t* src = edge_index;
  const int64_t* dst = edge_index + E;
  Scratch fr(st), nflag(st), nrank(st), eflag(st), erank(st), tmp(st);
  XP_CHECK(fr.alloc(2 * N));
  XP_CHECK(nflag.alloc(sizeof(int32_t) * N));
  XP_CHECK(nrank.alloc(sizeof(int32_t) * N));
  XP_CHECK(eflag.alloc(sizeof(int32_t) * (E + 1)));
  XP_CHECK(erank.alloc(sizeof(int32_t) * (E + 1)));
  uint8_t* cur = fr.as<uint8_t>();
  uint8_t* nxt = cur + N;
  const int nb = (int)ceil_div(N, 256);
  const int eb = (int)std::min<int64_t>(std::max<int64_t>(ceil_div(E, 256), 1), kNumSMs * 16);
  XP_CHECK(cudaMemsetAsync(counts + 2, 0, sizeof(int64_t), st));
  if (E > 0) XP_LAUNCH(khop_validate_kernel, eb, 256, 0, st, src, dst, E, N, counts + 2);
  XP_LAUNCH(khop_init_kernel, nb, 256, 0, st, hop, cur, N, query);
  for (int h = 1; h <= hops; ++h) {
    XP_CHECK(cudaMemsetAsync(nxt, 0, N, st));
    if (E > 0) XP_LAUNCH(khop_expand_kernel, eb, 256, 0, st, src, dst, E, N, cur, nxt);
    XP_LAUNCH(khop_mark_kernel, nb, 256, 0, st, hop, nxt, N, h);
    std::swap(cur, nxt);
  }
  size_t tb = 0, tb2 = 0;
  XP_CHECK(cub::DeviceScan::ExclusiveSum(nullptr, tb, nflag.as<int32_t>(), nrank.as<int32_t>(), (int)N, st));
  if (E > 0) XP_CHECK(cub::DeviceScan::ExclusiveSum(nullptr, tb2, eflag.as<int32_t>(), erank.as<int32_t>(), (int)E, st));
  XP_CHECK(tmp.alloc(std::max(tb, tb2)));
  tb = tb2 = std::max(tb, tb2);
  XP_LAUNCH(khop_nodeflag_kernel, nb, 256, 0, st, hop, nflag.as<int32_t>(), N);
  XP_CHECK(cub::DeviceScan::ExclusiveSum(tmp.p, tb, nflag.as<int32_t>(), nrank.as<int32_t>(), (int)N, st));
  XP_LAUNCH(khop_relabel_kernel, nb, 256, 0, st, hop, nrank.as<int32_t>(), N, relabel, subset);
  if (E > 0) {
    XP_LAUNCH(khop_edgeflag_kernel, eb, 256, 0, st, src, dst, E, N, hop, edge_mask, eflag.as<int32_t>());
    XP_CHECK(cub::DeviceScan::ExclusiveSum(tmp.p, tb2, eflag.as<int32_t>(), erank.as<int32_t>(), (int)E, st));
    XP_LAUNCH(khop_edgewrite_kernel, eb, 256, 0, st, src, dst, E, eflag.as<int32_t>(), erank.as<int32_t>(), relabel,
              sub_edge_index);
  }
  XP_LAUNCH(khop_counts_kernel, 1, 1, 0, st, nflag.as<int32_t>(), nrank.as<int32_t>(), N, eflag.as<int32_t>(),
            erank.as<int32_t>(), E, relabel, query, sub_edge_index, counts);
  return 0;
}

int64_t xpgnn_khop_multi_workspace_bytes(int64_t N, int32_t hops) {
  if (N <= 0 || hops < 0 || hops >= 127) return -1;
  return (int64_t)sizeof(uint64_t) * N * (hops + 1) + 2 * (int64_t)sizeof(int32_t) * kMqBlocks * 64;
}

static int khop_multi_check(const int64_t* edge_index, int64_t E, int64_t N, const int64_t* queries, int32_t Q, int32_t hops,
                            const void* workspace, int64_t workspace_bytes) {
  XP_REQUIRE(N > 0 && E >= 0 && hops >= 0 && hops < 127, "bad N / E / hops");
  XP_REQUIRE(N < (1ll << 31) - 1 && E < (1ll << 31) - 1, "N/E out of int32 range (the per-query ranks are 32-bit)");
  XP_REQUIRE(Q >= 1 && Q <= 64, "1 <= Q <= 64 queries per call");
  XP_REQUIRE(queries && workspace && (edge_index || E == 0), "null argument");
  XP_REQUIRE(workspace_bytes >= xpgnn_khop_multi_workspace_bytes(N, hops), "workspace too small");
  return 0;
}

int xpgnn_khop_multi_count(const int64_t* edge_index, int64_t E, int64_t N, const int64_t* queries, int32_t Q, int32_t hops,
                           void* workspace, int64_t workspace_bytes, int64_t* counts, void* stream) {
  if (int rc = khop_multi_check(edge_index, E, N, queries, Q, hops, workspace, workspace_bytes)) return rc;
  XP_REQUIRE(counts, "null counts");
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t* src = edge_index;
  const int64_t* dst = edge_index + E;
  uint64_t* F = static_cast<uint64_t*>(workspace);
  int32_t* node_blk = reinterpret_cast<int32_t*>(F + N * (hops + 1));
  int32_t* edge_blk = node_blk + kMqBlocks * 64;
  const int levels = hops + 1;
  const int eb = (int)std::min<int64_t>(std::max<int64_t>(ceil_div(E, 256), 1), kNumSMs * 16);
  // queries are device data: one outside [0, N) is skipped here (it reaches nothing, N_q = 0); callers check them first
  XP_CHECK(cudaMemsetAsync(F, 0, sizeof(uint64_t) * N * levels, st));
  XP_CHECK(cudaMemsetAsync(counts + 2 * Q, 0, sizeof(int64_t), st));
  if (E > 0) XP_LAUNCH(khop_validate_kernel, eb, 256, 0, st, src, dst, E, N, counts + 2 * Q);
  XP_LAUNCH(mq_init_kernel, 1, 64, 0, st, F, queries, Q, N);
  for (int h = 1; h <= hops; ++h)
    if (E > 0) XP_LAUNCH(mq_expand_kernel, eb, 256, 0, st, src, dst, E, N, F + (h - 1) * N, F + h * N);
  XP_LAUNCH(mq_count_kernel<false>, kMqBlocks, 256, 0, st, F, levels, N, src, dst, N, mq_chunk(N), node_blk);
  if (E > 0) XP_LAUNCH(mq_count_kernel<true>, kMqBlocks, 256, 0, st, F, levels, N, src, dst, E, mq_chunk(E), edge_blk);
  else XP_CHECK(cudaMemsetAsync(edge_blk, 0, sizeof(int32_t) * kMqBlocks * 64, st));
  XP_LAUNCH(mq_scan_kernel, dim3((unsigned)Q, 2), 32, 0, st, node_blk, edge_blk, kMqBlocks, Q, counts);
  return 0;
}

int xpgnn_khop_multi_emit(const int64_t* edge_index, int64_t E, int64_t N, const int64_t* queries, int32_t Q, int32_t hops,
                          const void* workspace, int64_t workspace_bytes, const int64_t* counts, const int64_t* node_off,
                          const int64_t* edge_off, int64_t n_union_edges, int64_t* subset, int8_t* level, int64_t* sub_ind,
                          int64_t* sub_edge_index, int64_t* edge_id, void* stream) {
  if (int rc = khop_multi_check(edge_index, E, N, queries, Q, hops, workspace, workspace_bytes)) return rc;
  XP_REQUIRE(counts && node_off && edge_off && subset && level && sub_ind && sub_edge_index && n_union_edges >= Q,
             "null output / bad union size");
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t* src = edge_index;
  const int64_t* dst = edge_index + E;
  const uint64_t* F = static_cast<const uint64_t*>(workspace);
  const int32_t* node_blk = reinterpret_cast<const int32_t*>(F + N * (hops + 1));
  const int32_t* edge_blk = node_blk + kMqBlocks * 64;
  const int levels = hops + 1;
  MqEmitArgs a{node_off, edge_off, n_union_edges, subset, level, sub_ind, sub_edge_index, edge_id};
  XP_LAUNCH(mq_emit_kernel<false>, kMqBlocks, 256, 0, st, F, levels, N, src, dst, N, mq_chunk(N), node_blk, a);
  if (E > 0) XP_LAUNCH(mq_emit_kernel<true>, kMqBlocks, 256, 0, st, F, levels, N, src, dst, E, mq_chunk(E), edge_blk, a);
  XP_LAUNCH(mq_self_loop_kernel, 1, 64, 0, st, counts, Q, a);
  return 0;
}

int xpgnn_build_csr(const int64_t* src, const int64_t* dst, int64_t E, int64_t N, int32_t drop_self_loops, int32_t* rowptr,
                    int32_t* col, int64_t* n_kept, void* stream) {
  XP_REQUIRE(N > 0 && N < (1ll << 31) - 1 && E >= 0 && E < (1ll << 31) - 1, "N/E out of int32 range");
  XP_REQUIRE(rowptr && n_kept && (col || E == 0), "null output");
  cudaStream_t st = (cudaStream_t)stream;
  if (E == 0) {
    XP_CHECK(cudaMemsetAsync(rowptr, 0, sizeof(int32_t) * (N + 1), st));
    XP_CHECK(cudaMemsetAsync(n_kept, 0, sizeof(int64_t), st));
    return 0;
  }
  Scratch key(st), key2(st), val(st), tmp(st);
  XP_CHECK(key.alloc(sizeof(int32_t) * E));
  XP_CHECK(key2.alloc(sizeof(int32_t) * E));
  XP_CHECK(val.alloc(sizeof(int32_t) * E));
  const int eb = (int)std::min<int64_t>(ceil_div(E, 256), kNumSMs * 16);
  XP_LAUNCH(csr_key_kernel, eb, 256, 0, st, src, dst, E, drop_self_loops, (int32_t)N, key.as<int32_t>(), val.as<int32_t>());
  int bits = 1;
  while ((1ll << bits) <= N) ++bits;  // keys in [0, N]
  size_t tb = 0;
  XP_CHECK(cub::DeviceRadixSort::SortPairs(nullptr, tb, key.as<int32_t>(), key2.as<int32_t>(), val.as<int32_t>(), col, (int)E, 0,
                                           bits, st));
  XP_CHECK(tmp.alloc(tb));
  XP_CHECK(cub::DeviceRadixSort::SortPairs(tmp.p, tb, key.as<int32_t>(), key2.as<int32_t>(), val.as<int32_t>(), col, (int)E, 0,
                                           bits, st));  // LSD radix sort is stable: edge order kept inside a row
  const int rb = (int)std::min<int64_t>(ceil_div(N + 1, 256), kNumSMs * 16);
  XP_LAUNCH(csr_rowptr_kernel, rb, 256, 0, st, key2.as<int32_t>(), E, (int32_t)N, rowptr, n_kept);
  return 0;
}

}  // extern "C"
