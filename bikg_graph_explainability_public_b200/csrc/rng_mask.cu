// MT19937 stream replay + community-coalition mask generation on device.
//
// Replaces the torch CPU-generator draws and the Python loops of
//   masks.py:80-136 (get_internal_mask), :138-194 (get_external_indices), :231-260 (shapley_mask),
//   :262-397 (mask_generator) and pathways.py:234-385 of the reference.
// The (rows x N) bool matrix of the reference is never needed by the engine: bits are emitted
// directly in the packed node-major layout the masked SpMM reads (act[v][w]).
#include <cstdlib>

#include "common.cuh"
#include "knobs.cuh"

namespace xpgnn {
thread_local std::string g_last_error;

namespace {
struct KnobEntry { const char* name; int Knobs::*field; };
const KnobEntry kKnobTable[] = {
    {"compact", &Knobs::compact}, {"compact_hetero", &Knobs::compact_hetero}, {"cw", &Knobs::cw}, {"l0_lists", &Knobs::l0_lists},
    {"occ", &Knobs::occ}, {"seg", &Knobs::seg}, {"seg_occ", &Knobs::seg_occ}, {"seg_tma", &Knobs::seg_tma}, {"seg_skew", &Knobs::seg_skew}, {"seg_pf", &Knobs::seg_pf}, {"seg_carve", &Knobs::seg_carve}, {"l0_slices", &Knobs::l0_slices}, {"act_column", &Knobs::act_column}, {"l2_stream", &Knobs::l2_stream},
    {"l2_gather", &Knobs::l2_gather}, {"sched_static", &Knobs::sched_static}, {"long_rows", &Knobs::long_rows}, {"occ16", &Knobs::occ16},
    {"l0_multi", &Knobs::l0_multi}, {"l1_multi", &Knobs::l1_multi}, {"l0_ws", &Knobs::l0_ws}, {"dense_simt", &Knobs::dense_simt}, {"dense_wait_ns", &Knobs::dense_wait_ns}, {"dense_tma", &Knobs::dense_tma}, {"l0_wait_ns", &Knobs::l0_wait_ns},
    {"prune_l0", &Knobs::prune_l0}, {"fused", &Knobs::fused}, {"fused_sb", &Knobs::fused_sb}};
int env_int(const char* name, int dflt) {
  const char* e = getenv(name);
  return e && *e ? atoi(e) : dflt;
}
bool env_is(const char* name, const char* value) {
  const char* e = getenv(name);
  return e && std::string(e) == value;
}
}  // namespace

Knobs& knobs() {
  static Knobs k = [] {
    Knobs d;
    d.compact = env_int("XPGNN_COMPACT", d.compact);
    d.compact_hetero = env_int("XPGNN_COMPACT_HETERO", d.compact_hetero);
    d.cw = env_int("XPGNN_CW", d.cw) == 16 ? 16 : 32;
    d.l0_lists = env_is("XPGNN_L0", "lists");
    d.occ = env_int("XPGNN_OCC", d.occ);
    d.seg = env_int("XPGNN_SEG", d.seg);
    d.seg_occ = env_int("XPGNN_SEG_OCC", d.seg_occ);
    d.seg_tma = env_int("XPGNN_SEG_TMA", d.seg_tma);
    d.seg_skew = env_int("XPGNN_SEG_SKEW", d.seg_skew);
    d.seg_pf = env_int("XPGNN_SEG_PF", d.seg_pf);
    d.dense_wait_ns = env_int("XPGNN_DENSE_WAIT_NS", d.dense_wait_ns);
    d.dense_tma = env_int("XPGNN_DENSE_TMA", d.dense_tma);
    d.l0_wait_ns = env_int("XPGNN_L0_WAIT_NS", d.l0_wait_ns);
    d.l0_slices = env_int("XPGNN_L0_SLICES", d.l0_slices);
    d.act_column = env_int("XPGNN_ACT_COLUMN", d.act_column);
    d.l2_stream = env_int("XPGNN_L2_STREAM", d.l2_stream);
    d.l2_gather = env_int("XPGNN_L2_GATHER", d.l2_gather);
    d.sched_static = env_is("XPGNN_SCHED", "static");
    d.long_rows = env_int("XPGNN_LONG", d.long_rows);
    d.occ16 = env_int("XPGNN_OCC16", d.occ16);
    d.l0_multi = env_int("XPGNN_L0_MULTI", d.l0_multi);
    d.l1_multi = env_int("XPGNN_L1_MULTI", d.l1_multi);
    d.l0_ws = env_int("XPGNN_L0_WS", d.l0_ws);
    d.dense_simt = env_is("XPGNN_DENSE", "simt");
    d.prune_l0 = env_int("XPGNN_PRUNE_L0", d.prune_l0);
    d.fused = env_int("XPGNN_FUSED", d.fused);
    d.fused_sb = env_int("XPGNN_FUSED_SB", d.fused_sb);
    return d;
  }();
  return k;
}
int set_knob(const char* name, int value) {
  for (const KnobEntry& e : kKnobTable)
    if (std::string(e.name) == name) { knobs().*(e.field) = value; return 0; }
  return 1;
}
int get_knob(const char* name, int* value) {
  for (const KnobEntry& e : kKnobTable)
    if (std::string(e.name) == name) { *value = knobs().*(e.field); return 0; }
  return 1;
}
std::atomic<int64_t> g_launches{0};

// ------------------------------------------------------------------------------------------
// at::mt19937: 624-word state, block-parallel twist (three dependent phases of <=227 lanes).
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t mt_mix(uint32_t cur, uint32_t nxt, uint32_t far) {
  uint32_t y = (cur & 0x80000000u) | (nxt & 0x7fffffffu);
  return far ^ (y >> 1) ^ ((y & 1u) ? 0x9908b0dfu : 0u);
}
__device__ __forceinline__ uint32_t mt_temper(uint32_t y) {
  y ^= y >> 11;
  y ^= (y << 7) & 0x9d2c5680u;
  y ^= (y << 15) & 0xefc60000u;
  return y ^ (y >> 18);
}

constexpr int MT_N = 624, MT_M = 397, MT_D = MT_N - MT_M;  // 227

__global__ void __launch_bounds__(256) mt19937_draw_kernel(uint32_t* __restrict__ state, int32_t* __restrict__ pos_io,
                                                           uint32_t* __restrict__ out, int64_t n) {
  __shared__ uint32_t mt[MT_N];
  const int tid = threadIdx.x;
  for (int i = tid; i < MT_N; i += blockDim.x) mt[i] = state[i];
  int pos = *pos_io;
  __syncthreads();
  int64_t done = 0;
  while (done < n) {
    if (pos == MT_N) {
      // phase A: i in [0,227) uses old mt[i+397]; phase B: [227,454) uses new mt[i-227];
      // phase C: [454,623) uses new mt[i-227]; element 623 uses new mt[0] and new mt[396].
      uint32_t v = 0;
      if (tid < MT_D) v = mt_mix(mt[tid], mt[tid + 1], mt[tid + MT_M]);
      __syncthreads();
      if (tid < MT_D) mt[tid] = v;
      __syncthreads();
      if (tid < MT_D) v = mt_mix(mt[tid + MT_D], mt[tid + MT_D + 1], mt[tid]);
      __syncthreads();
      if (tid < MT_D) mt[tid + MT_D] = v;
      __syncthreads();
      const int i = tid + 2 * MT_D;  // 454 ..
      if (i < MT_N - 1) v = mt_mix(mt[i], mt[i + 1], mt[i - MT_D]);
      else if (i == MT_N - 1) v = mt_mix(mt[MT_N - 1], mt[0], mt[MT_M - 1]);
      __syncthreads();
      if (i < MT_N) mt[i] = v;
      __syncthreads();
      pos = 0;
    }
    const int take = (int)min((int64_t)(MT_N - pos), n - done);
    for (int i = tid; i < take; i += blockDim.x) out[done + i] = mt_temper(mt[pos + i]);
    pos += take;
    done += take;
  }
  __syncthreads();
  for (int i = tid; i < MT_N; i += blockDim.x) state[i] = mt[i];
  if (tid == 0) *pos_io = pos;
}

// ------------------------------------------------------------------------------------------
// torch.randperm: Fisher-Yates, z = u32 % (n - i) for i < n-1  (masks.py:385, pathways.py:318)
// ------------------------------------------------------------------------------------------
__device__ void fisher_yates(const uint32_t* __restrict__ draws, int n, int32_t* perm /*global*/, int32_t* smem_perm,
                             int smem_cap) {
  // called by the whole block; thread 0 walks the dependent chain
  int32_t* p = (n <= smem_cap) ? smem_perm : perm;
  for (int i = threadIdx.x; i < n; i += blockDim.x) p[i] = i;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int i = 0; i < n - 1; ++i) {
      uint32_t z = draws[i] % (uint32_t)(n - i);
      int32_t a = p[i], b = p[i + z];
      p[i] = b;
      p[i + z] = a;
    }
  }
  __syncthreads();
  if (p != perm)
    for (int i = threadIdx.x; i < n; i += blockDim.x) perm[i] = p[i];
  __syncthreads();
}

__global__ void __launch_bounds__(256) randperm_kernel(const uint32_t* __restrict__ draws, int n, int32_t* perm, int smem_cap) {
  extern __shared__ int32_t sperm[];
  fisher_yates(draws, n, perm, sperm, smem_cap);
}

// ------------------------------------------------------------------------------------------
// Stream-offset resolution (sequential over community blocks; data dependent only through the
// dead-mask repair of pathways.py:285-334, which can fire only when a block has no antithetic
// pair, i.e. (size - size_int) < 2).
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) mask_resolve_kernel(const int32_t* __restrict__ com_ptr, const int32_t* __restrict__ order,
                                                           const int32_t* __restrict__ size, const int32_t* __restrict__ size_int,
                                                           int n_pos, int C, int n_rows, const uint32_t* __restrict__ draws,
                                                           int64_t* __restrict__ offsets, int64_t* __restrict__ consumed, int shuffle,
                                                           int32_t* ind, int smem_cap) {
  extern __shared__ int32_t sperm[];
  int64_t cur = 0;
  for (int p = 0; p < n_pos; ++p) {
    const int cid = order[p];
    const int L = com_ptr[cid + 1] - com_ptr[cid];
    const int sz = size[p], si = size_int[p];
    const int n_ext = sz - si, half = n_ext >> 1, odd = n_ext & 1;
    const int64_t off_int = cur;
    cur += (int64_t)sz * L;
    const int64_t off_ext = cur;
    cur += (int64_t)half * C;
    const int64_t off_odd = odd ? cur : -1;
    cur += odd ? C : 0;
    int dead = -1;
    if (C > 1 && half == 0) {
      int any = 0;
      if (odd)
        for (int c = threadIdx.x; c < C; c += blockDim.x)
          if (c != p && (draws[off_odd + c] & 1u)) any = 1;
      any = __syncthreads_or(any);
      if (!any) {  // activate_dead_mask: randperm(C), drop `p`, first survivor goes to the only row
        if (odd) {
          uint32_t z0 = draws[cur] % (uint32_t)C;
          int first = (int)z0;
          if (first == p) {
            if (C == 2) first = (z0 == 1u) ? 0 : 1;
            else {
              int idx = 1 + (int)(draws[cur + 1] % (uint32_t)(C - 1));
              first = (z0 != 0u && idx == (int)z0) ? 0 : idx;
            }
          }
          dead = first;
        }
        cur += C - 1;
      }
    }
    if (threadIdx.x == 0) {
      offsets[4 * p + 0] = off_int;
      offsets[4 * p + 1] = off_ext;
      offsets[4 * p + 2] = off_odd;
      offsets[4 * p + 3] = dead;
    }
  }
  if (shuffle) {
    fisher_yates(draws + cur, n_rows, ind, sperm, smem_cap);
    cur += n_rows > 0 ? n_rows - 1 : 0;
  }
  if (threadIdx.x == 0) consumed[0] = cur;
}

// ------------------------------------------------------------------------------------------
// Expansion: one thread = one node x one 32-coalition word.
// ------------------------------------------------------------------------------------------
struct RowDesc {
  int64_t off_int, off_ext, off_odd;
  int32_t pos, cid, L, local, size_int, half, dead, valid;
};

__global__ void __launch_bounds__(256) mask_expand_kernel(xpgnn_mask_plan_t plan, const uint32_t* __restrict__ draws,
                                                          const int64_t* __restrict__ offsets, const int32_t* __restrict__ ind, int n_out,
                                                          uint8_t* __restrict__ mask_rm, uint32_t* __restrict__ act, int W,
                                                          int32_t* __restrict__ pathway_rows, int32_t* __restrict__ popcount) {
  __shared__ RowDesc rd[32];
  __shared__ int32_t cnt[32];
  const int w = blockIdx.y;
  const int N = plan.n_elements, C = plan.n_communities;
  if (threadIdx.x < 32) {
    const int s = w * 32 + threadIdx.x;
    RowDesc d;
    d.valid = s < n_out;
    cnt[threadIdx.x] = 0;
    if (d.valid) {
      const int r = ind ? ind[s] : s;
      int lo = 0, hi = plan.n_positions;  // last position with row_start <= r
      while (hi - lo > 1) {
        int mid = (lo + hi) >> 1;
        if (plan.row_start[mid] <= r) lo = mid; else hi = mid;
      }
      d.pos = lo;
      d.cid = plan.order[lo];
      d.L = plan.com_ptr[d.cid + 1] - plan.com_ptr[d.cid];
      d.local = r - plan.row_start[lo];
      d.size_int = plan.size_int[lo];
      d.half = (plan.size[lo] - d.size_int) >> 1;
      d.off_int = offsets[4 * lo + 0];
      d.off_ext = offsets[4 * lo + 1];
      d.off_odd = offsets[4 * lo + 2];
      d.dead = (int)offsets[4 * lo + 3];
      if (pathway_rows && blockIdx.x == 0) pathway_rows[s] = d.cid;
    }
    rd[threadIdx.x] = d;
  }
  __syncthreads();
  const int v = blockIdx.x * blockDim.x + threadIdx.x;
  uint32_t word = 0;
  if (v < N) {
    const int m0 = plan.node_ptr[v], m1 = plan.node_ptr[v + 1];
    for (int b = 0; b < 32; ++b) {
      const RowDesc& d = rd[b];
      if (!d.valid) break;
      int bit = 0, internal = 0;
      for (int m = m0; m < m1; ++m) {
        const int c = plan.node_com[m];
        if (c == d.cid) {  // masks.py:338 -- internal bits overwrite every row of the block
          bit = (int)(draws[d.off_int + (int64_t)d.local * d.L + plan.node_slot[m]] & 1u);
          internal = 1;
          break;
        }
      }
      if (!internal && d.local >= d.size_int) {
        const int j = d.local - d.size_int;
        for (int m = m0; m < m1 && !bit; ++m) {
          const int c = plan.node_com[m];
          if (c == d.pos) continue;  // masks.py:178: column = sorted position (quirk kept)
          if (j < d.half) bit = (int)(draws[d.off_ext + (int64_t)j * C + c] & 1u);
          else if (j < 2 * d.half) bit = (int)((draws[d.off_ext + (int64_t)(j - d.half) * C + c] & 1u) ^ 1u);
          else bit = (int)(draws[d.off_odd + c] & 1u) | (int)(c == d.dead);
        }
      }
      word |= (uint32_t)bit << b;
    }
    if (act) act[(int64_t)v * W + w] = word;
    if (mask_rm)
      for (int b = 0; b < 32 && rd[b].valid; ++b) mask_rm[(int64_t)(w * 32 + b) * N + v] = (word >> b) & 1u;
  }
  if (popcount) {
    for (int b = 0; b < 32; ++b) {
      const uint32_t ball = __ballot_sync(0xffffffffu, (word >> b) & 1u);
      if ((threadIdx.x & 31) == 0 && ball) atomicAdd(&cnt[b], __popc(ball));
    }
    __syncthreads();
    if (threadIdx.x < 32 && rd[threadIdx.x].valid && cnt[threadIdx.x])
      atomicAdd(&popcount[w * 32 + threadIdx.x], cnt[threadIdx.x]);
  }
}

__global__ void __launch_bounds__(256) shapley_expand_kernel(const uint32_t* __restrict__ draws, const int32_t* __restrict__ ind, int n_out, int N,
                                                             uint8_t* __restrict__ mask_rm, uint32_t* __restrict__ act, int W,
                                                             int32_t* __restrict__ popcount) {
  __shared__ int32_t cnt[32];
  const int w = blockIdx.y;
  if (threadIdx.x < 32) cnt[threadIdx.x] = 0;
  __syncthreads();
  const int v = blockIdx.x * blockDim.x + threadIdx.x;
  uint32_t word = 0;
  if (v < N) {
    for (int b = 0; b < 32; ++b) {
      const int s = w * 32 + b;
      if (s >= n_out) break;
      const int r = ind ? ind[s] : s;
      word |= (draws[(int64_t)r * N + v] & 1u) << b;
    }
    if (act) act[(int64_t)v * W + w] = word;
    if (mask_rm)
      for (int b = 0; b < 32 && w * 32 + b < n_out; ++b) mask_rm[(int64_t)(w * 32 + b) * N + v] = (word >> b) & 1u;
  }
  if (popcount) {
    for (int b = 0; b < 32; ++b) {
      const uint32_t ball = __ballot_sync(0xffffffffu, (word >> b) & 1u);
      if ((threadIdx.x & 31) == 0 && ball) atomicAdd(&cnt[b], __popc(ball));
    }
    __syncthreads();
    if (threadIdx.x < 32 && w * 32 + (int)threadIdx.x < n_out && cnt[threadIdx.x])
      atomicAdd(&popcount[w * 32 + threadIdx.x], cnt[threadIdx.x]);
  }
}

__global__ void __launch_bounds__(256) pack_mask_kernel(const uint8_t* __restrict__ mask_rm, int S, int N, uint32_t* __restrict__ act, int W,
                                                        int32_t* __restrict__ popcount) {
  __shared__ int32_t cnt[32];
  const int w = blockIdx.y;
  if (threadIdx.x < 32) cnt[threadIdx.x] = 0;
  __syncthreads();
  const int v = blockIdx.x * blockDim.x + threadIdx.x;
  uint32_t word = 0;
  if (v < N) {
    for (int b = 0; b < 32 && w * 32 + b < S; ++b) word |= (uint32_t)(mask_rm[(int64_t)(w * 32 + b) * N + v] != 0) << b;
    act[(int64_t)v * W + w] = word;
  }
  if (popcount) {
    for (int b = 0; b < 32; ++b) {
      const uint32_t ball = __ballot_sync(0xffffffffu, (word >> b) & 1u);
      if ((threadIdx.x & 31) == 0 && ball) atomicAdd(&cnt[b], __popc(ball));
    }
    __syncthreads();
    if (threadIdx.x < 32 && w * 32 + (int)threadIdx.x < S && cnt[threadIdx.x])
      atomicAdd(&popcount[w * 32 + threadIdx.x], cnt[threadIdx.x]);
  }
}

}  // namespace xpgnn

using namespace xpgnn;

extern "C" {

const char* xpgnn_last_error(void) { return g_last_error.c_str(); }
int xpgnn_abi_version(void) { return XPGNN_ABI_VERSION; }
int xpgnn_set_option(const char* name, int32_t value) {
  XP_REQUIRE(name && set_knob(name, value) == 0, "unknown engine option");
  return 0;
}
int xpgnn_get_option(const char* name, int32_t* value) {
  int v = 0;
  XP_REQUIRE(name && value && get_knob(name, &v) == 0, "unknown engine option");
  *value = v;
  return 0;
}
int64_t xpgnn_launch_count(void) { return g_launches.load(); }

int xpgnn_mt19937_draw(uint32_t* state624, int32_t* pos, uint32_t* draws, int64_t n, void* stream) {
  XP_REQUIRE(state624 && pos && (draws || n == 0), "null argument");
  if (n <= 0) return 0;
  XP_LAUNCH(mt19937_draw_kernel, 1, 256, 0, (cudaStream_t)stream, state624, pos, draws, n);
  return 0;
}

static const int kPermSmemInts = 48 * 1024;  // 192 KiB of dynamic shared memory for the shuffle

int xpgnn_randperm(const uint32_t* draws, int32_t n, int32_t* perm, void* stream) {
  XP_REQUIRE(perm && n >= 0, "bad argument");
  if (n == 0) return 0;
  const int cap = n <= kPermSmemInts ? n : 0;
  XP_CHECK(cudaFuncSetAttribute(randperm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kPermSmemInts * 4));
  XP_LAUNCH(randperm_kernel, 1, 256, (size_t)cap * 4, (cudaStream_t)stream, draws, n, perm, cap);
  return 0;
}

int64_t xpgnn_mask_max_draws(const int32_t* size_host, const int32_t* size_int_host, const int32_t* len_host,
                             int32_t n_positions, int32_t n_communities, int32_t shuffle) {
  int64_t tot = 0, rows = 0;
  for (int p = 0; p < n_positions; ++p) {
    const int64_t n_ext = size_host[p] - size_int_host[p];
    tot += (int64_t)size_host[p] * len_host[p] + (n_ext / 2) * n_communities + (n_ext & 1) * n_communities;
    if (n_communities > 1 && n_ext < 2) tot += n_communities - 1;  // possible dead-mask repair
    rows += size_host[p];
  }
  if (shuffle && rows > 0) tot += rows - 1;
  return tot;
}

int xpgnn_mask_resolve(const xpgnn_mask_plan_t* plan, const uint32_t* draws, int64_t* offsets, int64_t* consumed,
                       int32_t shuffle, int32_t* ind, void* stream) {
  XP_REQUIRE(plan && draws && offsets && consumed, "null argument");
  XP_REQUIRE(!shuffle || ind, "shuffle requested without an output permutation");
  const int cap = (shuffle && plan->n_rows <= kPermSmemInts) ? plan->n_rows : 0;
  XP_CHECK(cudaFuncSetAttribute(mask_resolve_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kPermSmemInts * 4));
  XP_LAUNCH(mask_resolve_kernel, 1, 256, (size_t)cap * 4, (cudaStream_t)stream, plan->com_ptr, plan->order, plan->size,
            plan->size_int, plan->n_positions, plan->n_communities, plan->n_rows, draws, offsets, consumed, shuffle, ind, cap);
  return 0;
}

int xpgnn_mask_expand(const xpgnn_mask_plan_t* plan, const uint32_t* draws, const int64_t* offsets, const int32_t* ind,
                      int32_t n_out, uint8_t* mask_rowmajor, uint32_t* act, int32_t W, int32_t* pathway_rows,
                      int32_t* popcount, void* stream) {
  XP_REQUIRE(plan && draws && offsets, "null argument");
  XP_REQUIRE(!act || W * 32 >= n_out, "W too small");
  if (n_out <= 0 || plan->n_elements <= 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  if (popcount) XP_CHECK(cudaMemsetAsync(popcount, 0, sizeof(int32_t) * n_out, st));
  dim3 grid((unsigned)ceil_div(plan->n_elements, 256), (unsigned)ceil_div(n_out, 32));
  XP_LAUNCH(mask_expand_kernel, grid, 256, 0, st, *plan, draws, offsets, ind, n_out, mask_rowmajor, act, W, pathway_rows,
            popcount);
  return 0;
}

int xpgnn_shapley_expand(const uint32_t* draws, const int32_t* ind, int32_t n_out, int32_t n_elements, uint8_t* mask_rowmajor,
                         uint32_t* act, int32_t W, int32_t* popcount, void* stream) {
  XP_REQUIRE(draws, "null argument");
  if (n_out <= 0 || n_elements <= 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  if (popcount) XP_CHECK(cudaMemsetAsync(popcount, 0, sizeof(int32_t) * n_out, st));
  dim3 grid((unsigned)ceil_div(n_elements, 256), (unsigned)ceil_div(n_out, 32));
  XP_LAUNCH(shapley_expand_kernel, grid, 256, 0, st, draws, ind, n_out, n_elements, mask_rowmajor, act, W, popcount);
  return 0;
}

int xpgnn_pack_mask(const uint8_t* mask_rowmajor, int32_t S, int32_t N, uint32_t* act, int32_t W, int32_t* popcount,
                    void* stream) {
  XP_REQUIRE(mask_rowmajor && act && W * 32 >= S, "bad argument");
  if (S <= 0 || N <= 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  if (popcount) XP_CHECK(cudaMemsetAsync(popcount, 0, sizeof(int32_t) * S, st));
  dim3 grid((unsigned)ceil_div(N, 256), (unsigned)W);
  XP_LAUNCH(pack_mask_kernel, grid, 256, 0, st, mask_rowmajor, S, N, act, W, popcount);
  return 0;
}

}  // extern "C"
