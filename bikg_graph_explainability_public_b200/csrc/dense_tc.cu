// Dense row transform on the 5th-generation tensor cores (tcgen05.mma, accumulators in TMEM).
//
// out[m][n] (+)= act( sum_k in[m][k] * w[n][k] + b[n] )      (the X*W^T transforms of the GNN layers)
//
// Two arithmetic modes:
//   TF32X3 : fp32 operands split on the fly into hi + lo TF32 parts, three MMAs per K step
//            (hi*hi + lo*hi + hi*lo).  Error ~2^-20 relative: keeps the fp32 parity bar (1e-4).
//   BF16   : operands rounded to bf16, one MMA per K step (the "bf16 transforms" mode, 2e-2 bar).
// Operands are staged in shared memory in the canonical no-swizzle K-major core-matrix layout
// (8 rows x 16 bytes per core matrix) by plain vectorised loads -- except the A operand of TF32x3 transforms whose
// input is chunk-major with 32-float chunks and whose rows come from the tile table (the layer >= 1 transforms of the
// compact paths): there each 128-row x 32-float stage is gathered by TMA (gather4, 4 rows of 128 bytes per
// instruction) into the K-major SWIZZLE_128B layout, and the tensor core reads the landed fp32 rows directly as the hi
// operand -- kind::tf32 uses only the top 19 bits of an element, which is exactly the truncated hi of the split.
// Converter warps write lo = a - hi next to it.  One elected thread issues the MMAs; completion is tracked with
// tcgen05.commit -> mbarrier; the epilogue reads the accumulator tile with tcgen05.ld (32 lanes x 32 columns per warp
// instruction).
#include <cuda_bf16.h>

#include <algorithm>
#include <cstdlib>
#include <cstring>

#include "common.cuh"
#include "dense_args.cuh"

namespace xpgnn {

// ------------------------------------------------------------------ PTX wrappers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
// ablation switches of the round-1 analysis (skip stores / loads / MMAs): compiled in only with -DXPGNN_EXPERIMENTS, so
// that no environment variable can make the shipped kernel skip work
#ifdef XPGNN_EXPERIMENTS
#define XP_EXP(a, bit) ((a).exp_flags & (bit))
#else
#define XP_EXP(a, bit) false
#endif
__constant__ int g_backoff_after = 16;  // failed polls before a waiting thread starts sleeping (XPGNN_DENSE_BACKOFF)
// > 0: waiting threads SUSPEND inside mbarrier.try_wait (suspend-time hint in ns; the hardware wakes them when the phase
// completes) instead of polling -- the r02 source-level profile counted 60 % of this kernel's executed instructions in the
// polling loop of its 21 waiting warps, every poll a shared-memory operation in a kernel bound by the shared-memory pipe
// (option dense_wait_ns)
__constant__ int g_wait_hint_ns = 0;

template <bool BACKOFF = true>
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  const uint32_t addr = smem_u32(bar);
  uint32_t done = 0;
  const uint32_t hint = (uint32_t)g_wait_hint_ns;
  if (hint > 0) {
    for (uint32_t spin = 0; !done; ++spin) {
      asm volatile(
          "{\n\t.reg .pred p;\n\t"
          "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
          "selp.u32 %0, 1, 0, p;\n\t}"
          : "=r"(done)
          : "r"(addr), "r"(parity), "r"(hint)
          : "memory");
      if (spin > (1u << 22)) __trap();
    }
    return;
  }
  for (uint32_t spin = 0; !done; ++spin) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(addr), "r"(parity)
        : "memory");
    // waiting warps must not eat the issue slots / shared-memory pipe of the working ones
    if (BACKOFF && !done && spin >= (uint32_t)g_backoff_after) __nanosleep(32);
    if (spin > (1u << 24)) __trap();  // never hang the GPU: a lost arrival becomes an error
  }
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tmem_alloc(uint32_t* smem_dst, uint32_t ncols) {  // whole warp
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)), "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {  // whole warp
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
template <int KIND>  // 0: tf32, 1: f16 (bf16 operands)
__device__ __forceinline__ void umma(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  if (KIND == 0)
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
        "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
  else
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
        "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
        "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]),
        "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
        "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
        "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// shared-memory matrix descriptor, no swizzle, K-major: core matrix = 8 rows x 16 B stored contiguously
// (128 B); LBO = byte stride between core matrices adjacent in K, SBO = between 8-row groups.
__device__ __forceinline__ uint64_t smem_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3fffu);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3fffu) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3fffu) << 32;
  d |= (uint64_t)1 << 46;  // descriptor version (Blackwell)
  return d;                // base offset 0, lbo mode 0, layout type 0 (SWIZZLE_NONE)
}
// K-major SWIZZLE_128B: rows of 128 bytes, 8-row atoms of 1024 bytes (SBO), 16-byte column c of row r stored at column
// c ^ (r & 7) -- the layout TMA writes with CU_TENSOR_MAP_SWIZZLE_128B.  The atom must be 1024-byte aligned (base offset
// 0); a K step inside the atom advances the start address by its byte offset (the swizzle applies to the final address).
__device__ __forceinline__ uint64_t smem_desc_sw128(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3fffu);
  d |= (uint64_t)1 << 16;               // LBO: unused for K-major swizzled operands one atom wide
  d |= (uint64_t)(1024 >> 4) << 32;     // SBO
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;               // layout type SWIZZLE_128B
  return d;
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
// TMA gather4: rows r0 .. r3 (128 bytes each) of the 2-D tensor map -> 4 consecutive 128-byte rows at smem_dst
__device__ __forceinline__ void tma_gather4(uint32_t smem_dst, const CUtensorMap* tmap, int r0, int r1, int r2, int r3, uint64_t* bar) {
  asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile::gather4.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, %7}], [%2];" ::"r"(smem_dst),
               "l"(tmap), "r"(smem_u32(bar)), "r"(0), "r"(r0), "r"(r1), "r"(r2), "r"(r3)
               : "memory");
}
__host__ __device__ constexpr uint32_t make_idesc(int kind_fmt /*1 bf16, 2 tf32*/, int M, int N) {
  return (1u << 4) | ((uint32_t)kind_fmt << 7) | ((uint32_t)kind_fmt << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// ------------------------------------------------------------------ kernel
constexpr int TM = 128;          // rows per tile == UMMA M == TMEM lanes
constexpr int EPI_WARPS = 8;      // two per TMEM lane quarter, each takes every other 16-column block
constexpr int LOADER_GROUPS = 3;  // chunks in flight per SM
constexpr int GROUP_WARPS = 4;
constexpr int LOADER_WARPS = GROUP_WARPS * LOADER_GROUPS;
constexpr int TC_THREADS = 32 * (EPI_WARPS + LOADER_WARPS + 1);  // warps 0-7 epilogue, 8-19 loaders / converters, 20 MMA issue
// gather4 form (G4): warps 0-7 epilogue, 8-9 converters (one 16 KB lo stage per item), 10 MMA issue, 11-14 TMA producers
// (15 warps: up to 128 registers a thread)
constexpr int G4_CONV_WARPS = 2;
constexpr int G4_PROD_WARPS = 4;
constexpr int G4_THREADS = 32 * (EPI_WARPS + G4_CONV_WARPS + 1 + G4_PROD_WARPS);
constexpr int G4_LO = 2;          // lo stages (held from conversion to MMA completion)
constexpr int G4_MAX_HI = 4;      // landed hi stages (held from the TMA issue to MMA completion: more of them)
constexpr int G4_PART = 128 * 128;  // bytes of one 128-row x 32-float stage part
constexpr int MAX_DONE = 12;      // lcm(stages <= 4, LOADER_GROUPS)
constexpr int KC = 32;           // K elements per stage
constexpr int MAX_STAGES = 4;
constexpr int TR_STRIDE = 16;     // floats per row of a 32 x 16 transposition block; the four 16-byte groups of row r sit at
                                  // group ^ ((r >> 1) & 3): conflict-free row writes AND conflict-free transposed reads (the padded
                                  // stride of round 1 made half of the reads two-wavefront: r02 ncu, 84 M of 163 M LDS wavefronts)
__device__ __forceinline__ int tr_off(int row, int group) { return row * TR_STRIDE + ((group ^ ((row >> 1) & 3)) << 2); }

// MODE 0: TF32x3 (element 4 B, hi/lo copies)   MODE 1: BF16 (element 2 B)
template <int MODE>
struct TcCfg {
  static constexpr int ELT = MODE == 0 ? 4 : 2;
  static constexpr int UK = 32 / ELT;                // K elements per MMA (32 bytes)
  static constexpr int PARTS = MODE == 0 ? 2 : 1;    // hi/lo
  static constexpr int K16 = KC * ELT / 16;          // 16-byte columns of a stage row
  static constexpr int PART_BYTES = TM * KC * ELT;
  static constexpr int A_STAGE_BYTES = PART_BYTES * PARTS;
};

__device__ __forceinline__ void mbar_wait_timed(uint64_t* bar, uint32_t parity, unsigned long long* dbg, unsigned long long& acc) {
  if (dbg) {
    const long long t0 = clock64();
    mbar_wait<true>(bar, parity);
    acc += (unsigned long long)(clock64() - t0);
  } else {
    mbar_wait<true>(bar, parity);
  }
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// offset (bytes) of element group (row r, 16-byte column j) inside an operand block whose K extent is
// `k16` sixteen-byte columns: core matrices contiguous along K (LBO = 128), SBO = k16 * 128
__device__ __forceinline__ uint32_t core_off(int r, int j, int k16) { return (uint32_t)((r >> 3) * k16 * 128 + j * 128 + (r & 7) * 16); }

__device__ __forceinline__ void split_tf32(const float4& v, float4& hi, float4& lo) {
  hi.x = __uint_as_float(__float_as_uint(v.x) & 0xffffe000u); lo.x = v.x - hi.x;
  hi.y = __uint_as_float(__float_as_uint(v.y) & 0xffffe000u); lo.y = v.y - hi.y;
  hi.z = __uint_as_float(__float_as_uint(v.z) & 0xffffe000u); lo.z = v.z - hi.z;
  hi.w = __uint_as_float(__float_as_uint(v.w) & 0xffffe000u); lo.w = v.w - hi.w;
}
__device__ __forceinline__ uint2 pack_bf16(const float4& v) {
  __nv_bfloat162 p0 = __floats2bfloat162_rn(v.x, v.y), p1 = __floats2bfloat162_rn(v.z, v.w);
  uint2 r;
  r.x = *reinterpret_cast<uint32_t*>(&p0);
  r.y = *reinterpret_cast<uint32_t*>(&p1);
  return r;
}

// out of line on purpose (rare paths; the hot epilogue must stay small).  By value / through shared memory:
// a reference parameter would force the caller's registers into local memory.
__device__ __noinline__ float4 sigmoid4(float4 v) {
  v.x = apply_act(v.x, XPGNN_ACT_SIGMOID); v.y = apply_act(v.y, XPGNN_ACT_SIGMOID);
  v.z = apply_act(v.z, XPGNN_ACT_SIGMOID); v.w = apply_act(v.w, XPGNN_ACT_SIGMOID);
  return v;
}
// row-per-thread fallback for outputs that cannot be written as float4: `row16` = the thread's 16 accumulators in shared memory
__device__ __noinline__ void scalar_epilogue(const float* row16, int swz, int c0, int n_out, const float* s_bias, float* out_row, int cw_out, int cw_out_lg,
                                             int64_t out_chunk_stride, int accumulate, int act_fn, float rs) {
#pragma unroll 1
  for (int c = 0; c < 16; ++c) {
    const int n = c0 + c;
    if (n >= n_out) break;
    float x = row16[(((c >> 2) ^ swz) << 2) | (c & 3)] + s_bias[n];  // 16-byte groups are stored XOR-swizzled (tr_off)
    float* op = out_row + (cw_out ? (int64_t)(n >> cw_out_lg) * out_chunk_stride + (n & (cw_out - 1)) : (int64_t)n);
    if (accumulate) x += *op;
    *op = apply_act(x, act_fn) * rs;
  }
}

// out of line on purpose: called once per (tile, row) by the loaders, keeps their unrolled pipeline small
__device__ __noinline__ const float* resolve_in_row(const float* in, int64_t in_s_stride, int ld_in, const int32_t* rows, int rows_per_s,
                                                   int row_lo, int64_t M, int dst_lo, int dst_hi, int64_t tile, int r) {
  DenseArgs a{};  // flat row naming only (the tile table is read inline by the loaders)
  a.in_s_stride = in_s_stride; a.ld_in = ld_in; a.rows = rows; a.rows_per_s = rows_per_s; a.row_lo = row_lo; a.M = M;
  a.dst_lo = dst_lo; a.dst_hi = dst_hi;
  DenseRow row;
  return dense_resolve_row(a, tile, r, row) ? in + row.io : nullptr;
}

// Warp-specialised persistent kernel, one CTA per SM, tiles dealt round-robin:
//   loaders  (4 warps): global -> registers three K chunks ahead -> hi/lo (or bf16) operand stage in shared
//                       memory (canonical no-swizzle K-major core matrices) -> mbarrier "stage full";
//   MMA      (1 lane) : waits "stage full", issues the tcgen05.mma's of the chunk into one of TWO accumulator
//                       buffers in TMEM, commits to "stage empty" and, after the last chunk, "accumulator full";
//   epilogue (4 warps): waits "accumulator full", tcgen05.ld, bias / accumulate / activation / row scale,
//                       stores, then "accumulator empty".  It overlaps the next tile's loads and MMAs.
// G4 (MODE 0, chunk-major 32-float input, tile-table rows): the loaders are replaced by
//   TMA producers (4 warps): per item 32 gather4 (8 per warp, 4 tile rows each) into a landed "hi" stage, counted in
//                       bytes on its mbarrier; n_stages hi stages, refilled when the MMAs of the item that used them are done;
//   converters (2 warps): read the landed stage, write lo = a - (a & 0xffffe000) to one of G4_LO lo stages (same
//                       swizzled layout, so element positions match one to one), arrive "stage full".
template <int MODE, bool G4>
__global__ void __launch_bounds__(G4 ? G4_THREADS : TC_THREADS, 1)
    dense_tc_kernel(const DenseArgs a, int n_pad, uint32_t tmem_cols, int n_stages, unsigned long long* dbg, const __grid_constant__ CUtensorMap tmap) {
  static_assert(!G4 || MODE == 0, "the gather4 path feeds the TF32x3 MMAs");
  constexpr int NT = G4 ? G4_THREADS : TC_THREADS;
  constexpr int MMA_WARP = EPI_WARPS + (G4 ? G4_CONV_WARPS : LOADER_WARPS);
  using Cfg = TcCfg<MODE>;
  extern __shared__ __align__(128) uint8_t smem[];
  __shared__ uint64_t bar_full[MAX_STAGES];
  // MMAs of item i done -> bar_done[i % n_done], n_done = lcm(n_stages, LOADER_GROUPS): every barrier is then waited on by
  // exactly one loader group and in every one of its phases (a parity wait must not skip a phase)
  __shared__ uint64_t bar_done[MAX_DONE];
  __shared__ uint64_t bar_acc_full[2], bar_acc_empty[2];
  __shared__ uint32_t tmem_base_sh;
  __shared__ __align__(16) float s_bias[256];
  __shared__ __align__(16) float s_tr[EPI_WARPS * 32 * TR_STRIDE];  // epilogue transposition blocks, one per epilogue warp

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int K = a.k;                                  // multiple of KC
  const int kb16 = K * Cfg::ELT / 16;                 // 16-byte columns of a full-K row
  const uint32_t b_part_bytes = (uint32_t)n_pad * K * Cfg::ELT;
  uint8_t* sB = smem;                                      // [PARTS][n_pad x K]
  uint8_t* sA = smem + (size_t)b_part_bytes * Cfg::PARTS;  // [n_stages][PARTS][TM x KC] | G4: [n_stages] hi, [G4_LO] lo
  if (G4) sA = smem + ((smem_u32(sA) + 1023u) & ~1023u) - smem_u32(smem);  // SWIZZLE_128B atoms: 1024-byte aligned
  // G4 barriers: bar_full[G4_LO] = lo stage written (converters), hi_full = hi stage landed (TMA bytes),
  // hi_empty / lo_empty = the MMAs reading the stage are done (tcgen05.commit)
  uint64_t* hi_full = bar_done;
  uint64_t* hi_empty = bar_done + G4_MAX_HI;
  uint64_t* lo_empty = bar_done + 2 * G4_MAX_HI;

  if (warp == 0) tmem_alloc(&tmem_base_sh, tmem_cols);
  if (tid < 256) s_bias[tid] = (a.b && tid < a.n_out) ? a.b[tid] : 0.0f;
  if (tid == 0) {
    for (int s = 0; s < MAX_STAGES; ++s) mbar_init(&bar_full[s], 32 * (G4 ? G4_CONV_WARPS : GROUP_WARPS));
    for (int s = 0; s < MAX_DONE; ++s) mbar_init(&bar_done[s], (G4 && s < G4_MAX_HI) ? G4_PROD_WARPS : 1);  // G4: hi_full
    for (int s = 0; s < 2; ++s) {
      mbar_init(&bar_acc_full[s], 1);
      mbar_init(&bar_acc_empty[s], 32 * EPI_WARPS);
    }
    fence_mbar_init();
  }
  // ---- B operand (weights) resident in shared memory for the whole kernel ----
  for (int f = tid; f < n_pad * kb16; f += NT) {
    // unit f -> (row group, 16B column): lanes of a quarter warp take the 8 rows of one core matrix
    const int r = ((f >> 3) / kb16) * 8 + (f & 7);
    const int j = (f >> 3) % kb16;
    const uint32_t off = core_off(r, j, kb16);
    if (MODE == 0) {
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f), hi, lo;
      if (r < a.n_out) v = __ldg(reinterpret_cast<const float4*>(a.w + (int64_t)r * K + j * 4));
      split_tf32(v, hi, lo);
      *reinterpret_cast<float4*>(sB + off) = hi;
      *reinterpret_cast<float4*>(sB + b_part_bytes + off) = lo;
    } else {
      float4 v0 = make_float4(0.f, 0.f, 0.f, 0.f), v1 = v0;
      if (r < a.n_out) {
        v0 = __ldg(reinterpret_cast<const float4*>(a.w + (int64_t)r * K + j * 8));
        v1 = __ldg(reinterpret_cast<const float4*>(a.w + (int64_t)r * K + j * 8 + 4));
      }
      const uint2 p0 = pack_bf16(v0), p1 = pack_bf16(v1);
      *reinterpret_cast<uint4*>(sB + off) = make_uint4(p0.x, p0.y, p1.x, p1.y);
    }
  }
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_sh;
  const int n_chunks = K / KC;
  const int n_done = n_stages % LOADER_GROUPS == 0 ? n_stages : n_stages * LOADER_GROUPS;
  const int64_t n_tiles = a.rows_packed ? (int64_t)*a.n_tiles_dev : (a.M + TM - 1) / TM;
  const int64_t my_tiles = (int64_t)blockIdx.x < n_tiles ? (n_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;

  if (G4 && warp > MMA_WARP) {
    // ================= TMA producer =================
    // producer warp pw, lane l < 8 gathers tile rows 32 pw + 4 l .. + 3: row (slot, node) of K chunk kc is row
    // slot * in_s_stride / 32 + node + kc * in_chunk_stride / 32 of the [rows][32] view.  Rows without an entry read
    // row 0: the MMA rows are independent and the epilogue stores no row without an entry.  The TMA instructions of one
    // warp issue one lane after the other; several warps issue side by side.
    const int pw = warp - (MMA_WARP + 1);
    if (lane < 8) {
      const int32_t s_rows = (int32_t)(a.in_s_stride >> 5), c_rows = (int32_t)(a.in_chunk_stride >> 5);
      auto tile_entries = [&](int64_t ti_) {
        return __ldg(reinterpret_cast<const int4*>(a.rows_packed + ((int64_t)blockIdx.x + ti_ * gridDim.x) * 128 + pw * 32) + lane);
      };
      int4 nxt = my_tiles > 0 ? tile_entries(0) : make_int4(-1, -1, -1, -1);
      int64_t item = 0;
      for (int64_t ti = 0; ti < my_tiles; ++ti) {
        const int e[4] = {nxt.x, nxt.y, nxt.z, nxt.w};
        int r0[4];
#pragma unroll
        for (int p = 0; p < 4; ++p) r0[p] = e[p] < 0 ? 0 : (int32_t)((uint32_t)e[p] >> kPackShift) * s_rows + (e[p] & ((1 << kPackShift) - 1));
        if (ti + 1 < my_tiles) nxt = tile_entries(ti + 1);  // a tile ahead: in flight while this tile's chunks are issued
        for (int kc = 0; kc < n_chunks; ++kc, ++item) {
          const int hs = (int)(item % n_stages);
          if (item >= n_stages) mbar_wait(&hi_empty[hs], (uint32_t)((item / n_stages) - 1) & 1u);
          if (lane == 0) mbar_arrive_expect_tx(&hi_full[hs], G4_PART / G4_PROD_WARPS);
          __syncwarp(0xffu);
          const int c = kc * c_rows;
          tma_gather4(smem_u32(sA) + hs * G4_PART + (pw * 8 + lane) * 512, &tmap, r0[0] + c, r0[1] + c, r0[2] + c, r0[3] + c, &hi_full[hs]);
        }
      }
    }
  } else if (G4 && warp >= EPI_WARPS && warp < MMA_WARP) {
    // ================= converters =================
    // thread t owns bytes 16 (t + 64 q), q = 0..15, of the stage: one warp instruction = 512 contiguous bytes (no bank
    // conflicts); hi and lo stages share the layout, so the swizzle never has to be known here
    constexpr int CT = 32 * G4_CONV_WARPS;
    const int t = tid - EPI_WARPS * 32;
    const int64_t n_items = my_tiles * n_chunks;
    for (int64_t i = 0; i < n_items; ++i) {
      const int hs = (int)(i % n_stages), ls = (int)(i % G4_LO);
      mbar_wait(&hi_full[hs], (uint32_t)(i / n_stages) & 1u);
      if (i >= G4_LO) mbar_wait(&lo_empty[ls], (uint32_t)((i / G4_LO) - 1) & 1u);
      const float4* hi = reinterpret_cast<const float4*>(sA + (size_t)hs * G4_PART);
      float4* lo = reinterpret_cast<float4*>(sA + (size_t)(n_stages + ls) * G4_PART);
#pragma unroll
      for (int h8 = 0; h8 < G4_PART / 16 / CT; h8 += 8) {
        float4 v[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) v[q] = hi[t + CT * (h8 + q)];
#pragma unroll
        for (int q = 0; q < 8; ++q) {
          float4 h, l;
          split_tf32(v[q], h, l);
          lo[t + CT * (h8 + q)] = l;
        }
      }
      fence_proxy_async();  // generic-proxy stores -> visible to the tensor core (async proxy)
      mbar_arrive(&bar_full[ls]);
    }
  } else if (!G4 && warp >= EPI_WARPS && warp < EPI_WARPS + LOADER_WARPS) {
    // ================= loaders / converters =================
    // LOADER_GROUPS groups of 4 warps take the K chunks round-robin.  A thread has only its own chunk in flight
    // when it executes fence.proxy.async (the fence waits for every outstanding load of the thread: prefetching
    // further chunks in the same thread would serialise on it); the depth comes from the groups.
    // Inside a group a warp owns 32 rows of the tile; per chunk a thread moves 8 float4 (4 rows x 2 columns).
    const int grp = (warp - EPI_WARPS) / GROUP_WARPS, lw = (warp - EPI_WARPS) % GROUP_WARPS, lr = lane & 7, lj = lane >> 3;
    const int64_t n_items = my_tiles * n_chunks;
    // MODE 0: 16-byte columns lj and lj + 4; MODE 1: the adjacent pair 2 lj, 2 lj + 1 (one bf16 column)
    const int j0 = MODE == 0 ? lj : 2 * lj, j1 = MODE == 0 ? lj + 4 : 2 * lj + 1;
    unsigned long long w_empty = 0;
    const long long t_role0 = clock64();
    // cursor of this group: item i = (local tile ti, chunk kc), stage st; dn / dn_use = barrier and phase of item i - n_stages
    int64_t ti = 0;
    int kc = grp, st = grp % n_stages;
    while (kc >= n_chunks) { kc -= n_chunks; ++ti; }
    int64_t cur_ti = -1;
    const float* ld_row[4] = {nullptr, nullptr, nullptr, nullptr};
    int32_t nxt_e[4] = {-1, -1, -1, -1};  // tile-table entries of the next tile of this CTA, loaded a tile ahead
    int64_t nxt_ti = -1;
    for (int64_t i = grp; i < n_items; i += LOADER_GROUPS) {
      if (ti != cur_ti) {  // rows of a new tile
        const int64_t tile = (int64_t)blockIdx.x + ti * gridDim.x;
#pragma unroll
        for (int p = 0; p < 4; ++p) {
          const int r = lw * 32 + p * 8 + lr;
          if (a.rows_packed) {
            const int32_t e = nxt_ti == ti ? nxt_e[p] : __ldg(a.rows_packed + tile * 128 + r);
            ld_row[p] = e < 0 ? nullptr
                              : a.in + (int64_t)((uint32_t)e >> kPackShift) * a.in_s_stride + (int64_t)(e & ((1 << kPackShift) - 1)) * a.ld_in;
          } else {
            ld_row[p] = resolve_in_row(a.in, a.in_s_stride, a.ld_in, a.rows, a.rows_per_s, a.row_lo, a.M, a.dst_lo, a.dst_hi, tile, r);
          }
        }
        cur_ti = ti;
      }
      float4 buf[8];
      if (MODE == 1 && a.in16) {
        // bf16 operand: one 16-byte column (8 elements) per row and thread, no conversion; ld_row holds element offsets
        const int64_t o16 = dense_in_off(a, kc * KC + lj * 8);
        const float4 zero = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int p = 0; p < 4; ++p)
          buf[p] = ld_row[p] ? __ldg(reinterpret_cast<const float4*>(reinterpret_cast<const __nv_bfloat16*>(a.in) + (ld_row[p] - a.in) + o16)) : zero;
      } else {
        const int64_t o0 = dense_in_off(a, kc * KC + j0 * 4), o1 = dense_in_off(a, kc * KC + j1 * 4);
        const float4 zero = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int p = 0; p < 4; ++p) {
          buf[2 * p] = (ld_row[p] && !XP_EXP(a, 2)) ? __ldg(reinterpret_cast<const float4*>(ld_row[p] + o0)) : zero;
          buf[2 * p + 1] = (ld_row[p] && !XP_EXP(a, 2)) ? __ldg(reinterpret_cast<const float4*>(ld_row[p] + o1)) : zero;
        }
      }
      if (a.rows_packed && nxt_ti != ti + 1 && ti + 1 < my_tiles) {  // table entries of the next tile, in flight with the data
        nxt_ti = ti + 1;
#pragma unroll
        for (int p = 0; p < 4; ++p)
          nxt_e[p] = __ldg(a.rows_packed + ((int64_t)blockIdx.x + nxt_ti * gridDim.x) * 128 + lw * 32 + p * 8 + lr);
      }
      if (i >= n_stages) {  // the MMAs that read this stage (item i - n_stages) are done
        const int64_t prev = i - n_stages;
        mbar_wait_timed(&bar_done[prev % n_done], (uint32_t)(prev / n_done) & 1u, dbg, w_empty);
      }
      uint8_t* stage = sA + (size_t)st * Cfg::A_STAGE_BYTES;
#pragma unroll
      for (int p = 0; p < 4; ++p) {
        const int r = lw * 32 + p * 8 + lr;
        if (MODE == 0) {
          float4 hi, lo;
          split_tf32(buf[2 * p], hi, lo);
          *reinterpret_cast<float4*>(stage + core_off(r, lj, Cfg::K16)) = hi;
          *reinterpret_cast<float4*>(stage + Cfg::PART_BYTES + core_off(r, lj, Cfg::K16)) = lo;
          split_tf32(buf[2 * p + 1], hi, lo);
          *reinterpret_cast<float4*>(stage + core_off(r, lj + 4, Cfg::K16)) = hi;
          *reinterpret_cast<float4*>(stage + Cfg::PART_BYTES + core_off(r, lj + 4, Cfg::K16)) = lo;
        } else if (a.in16) {
          *reinterpret_cast<float4*>(stage + core_off(r, lj, Cfg::K16)) = buf[p];
        } else {
          const uint2 p0 = pack_bf16(buf[2 * p]), p1 = pack_bf16(buf[2 * p + 1]);
          *reinterpret_cast<uint4*>(stage + core_off(r, lj, Cfg::K16)) = make_uint4(p0.x, p0.y, p1.x, p1.y);
        }
      }
      fence_proxy_async();  // generic-proxy stores -> visible to the tensor core (async proxy)
      mbar_arrive(&bar_full[st]);
      // advance the cursor by LOADER_GROUPS items
      kc += LOADER_GROUPS;
      while (kc >= n_chunks) { kc -= n_chunks; ++ti; }
      st = (st + LOADER_GROUPS) % n_stages;
    }
    if (dbg && blockIdx.x == 0 && tid == EPI_WARPS * 32) {
      dbg[0] = (unsigned long long)(clock64() - t_role0);
      dbg[1] = w_empty;
    }
  } else if (warp == MMA_WARP) {
    // ================= MMA issue (one lane) =================
    if (lane == 0) {
      const uint32_t idesc = make_idesc(MODE == 0 ? 2 : 1, TM, n_pad);
      const uint32_t sA_addr = smem_u32(sA), sB_addr = smem_u32(sB);
      int64_t item = 0;
      unsigned long long w_full = 0, w_acc = 0;
      const long long t_role0 = clock64();
      for (int64_t ti = 0; ti < my_tiles; ++ti) {
        const int ab = (int)(ti & 1);
        if (ti >= 2) {  // the epilogue has drained this accumulator buffer
          mbar_wait_timed(&bar_acc_empty[ab], (uint32_t)((ti >> 1) - 1) & 1u, dbg, w_acc);
          tc_fence_after();
        }
        const uint32_t d_tmem = tmem_base + (uint32_t)(ab * n_pad);
        for (int kc = 0; kc < n_chunks; ++kc, ++item) {
          const int st = (int)(item % n_stages), ls = (int)(item % G4_LO);
          if (G4)
            mbar_wait_timed(&bar_full[ls], (uint32_t)(item / G4_LO) & 1u, dbg, w_full);
          else
            mbar_wait_timed(&bar_full[st], (uint32_t)(item / n_stages) & 1u, dbg, w_full);
          tc_fence_after();
          const uint32_t a_hi = sA_addr + st * (G4 ? G4_PART : Cfg::A_STAGE_BYTES);
          const uint32_t a_lo = G4 ? sA_addr + (n_stages + ls) * G4_PART : a_hi + Cfg::PART_BYTES;
#pragma unroll
          for (int ks = 0; ks < KC / Cfg::UK; ++ks) {
            // one MMA consumes 2 sixteen-byte columns (32 bytes of K)
            const uint32_t a_off = ks * 2 * (G4 ? 16 : 128);
            const uint32_t b_off = (kc * Cfg::K16 + ks * 2) * 128;
            const uint64_t da_hi = G4 ? smem_desc_sw128(a_hi + a_off) : smem_desc(a_hi + a_off, 128, Cfg::K16 * 128);
            const uint64_t db_hi = smem_desc(sB_addr + b_off, 128, kb16 * 128);
            const uint32_t first = (kc == 0 && ks == 0) ? 0u : 1u;
            if (XP_EXP(a, 4)) continue;
            umma<MODE>(d_tmem, da_hi, db_hi, idesc, first);
            if (MODE == 0) {
              const uint64_t da_lo = G4 ? smem_desc_sw128(a_lo + a_off) : smem_desc(a_lo + a_off, 128, Cfg::K16 * 128);
              const uint64_t db_lo = smem_desc(sB_addr + b_part_bytes + b_off, 128, kb16 * 128);
              umma<MODE>(d_tmem, da_lo, db_hi, idesc, 1u);
              umma<MODE>(d_tmem, da_hi, db_lo, idesc, 1u);
            }
          }
          if (G4) {
            umma_commit(&hi_empty[st]);
            umma_commit(&lo_empty[ls]);
          } else {
            umma_commit(&bar_done[item % n_done]);
          }
          if (kc == n_chunks - 1) umma_commit(&bar_acc_full[ab]);
        }
      }
      if (dbg && blockIdx.x == 0) {
        dbg[2] = (unsigned long long)(clock64() - t_role0);
        dbg[3] = w_full;
        dbg[4] = w_acc;
      }
    }
  } else if (warp < EPI_WARPS) {
    // ================= epilogue: TMEM -> registers -> bias / accumulate / activation / row scale -> global =================
    const int quarter = warp & 3, half = warp >> 2;  // a warp may touch TMEM lanes 32 (warp % 4) .. + 31
    const int row_in_tile = quarter * 32 + lane;      // TMEM lane == tile row
    // ReLU and identity share one branch-free path (max with 0 or -inf); sigmoid is out of line
    const float lower = a.act_fn == XPGNN_ACT_RELU ? 0.0f : -INFINITY;
    const bool vec_ok = (a.n_out & 3) == 0 && (a.ld_out & 3) == 0 && (a.out_s_stride & 3) == 0 && (a.out_chunk_stride & 3) == 0;
    float* s_t = s_tr + warp * (32 * TR_STRIDE);  // this warp's transposition block
    unsigned long long w_accfull = 0;
    const long long t_role0 = clock64();
    // tile-table entry / row scale of this thread's row, fetched one tile ahead (a DRAM round trip otherwise exposed per tile)
    int32_t nxt_e = -1;
    float nxt_rs = 1.0f;
    auto fetch_entry = [&](int64_t ti_) {
      const int64_t pos = ((int64_t)blockIdx.x + ti_ * gridDim.x) * 128 + row_in_tile;
      nxt_e = __ldg(a.rows_packed + pos);
      nxt_rs = a.rs_packed ? __ldg(a.rs_packed + pos) : 1.0f;
    };
    if (a.rows_packed && my_tiles > 0) fetch_entry(0);
    for (int64_t ti = 0; ti < my_tiles; ++ti) {
      const int ab = (int)(ti & 1);
      const int64_t tile = (int64_t)blockIdx.x + ti * gridDim.x;
      bool ok;
      int64_t oo;
      float rs;
      if (a.rows_packed) {
        const int32_t e = nxt_e;
        ok = e >= 0;
        rs = nxt_rs;
        oo = ok ? (int64_t)((uint32_t)e >> kPackShift) * a.out_s_stride + (int64_t)(e & ((1 << kPackShift) - 1)) * a.ld_out : -1;
        if (ti + 1 < my_tiles) fetch_entry(ti + 1);
      } else {
        DenseRow row;
        ok = dense_resolve_row(a, tile, row_in_tile, row);
        oo = ok ? row.oo : -1;
        rs = row.rs;
      }
      // after the transposition lane l writes 16 bytes of rows 8 i + l / 4 (i = 0..3): fetch their offsets once per tile
      int64_t oo_r[4];
      float rs_r[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        oo_r[i] = __shfl_sync(0xffffffffu, oo, i * 8 + (lane >> 2));
        rs_r[i] = __shfl_sync(0xffffffffu, rs, i * 8 + (lane >> 2));
      }
      mbar_wait_timed(&bar_acc_full[ab], (uint32_t)(ti >> 1) & 1u, dbg, w_accfull);
      tc_fence_after();
      for (int c0 = half * 16; c0 < n_pad; c0 += 32) {
        uint32_t r[16];
        tmem_ld16(tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(ab * n_pad + c0), r);
        // A thread owns one accumulator row; storing it directly would touch 32 different lines per store
        // instruction.  Transpose 32 x 16 blocks through shared memory: 4 lanes then write one 64-byte run
        // of a row, 8 rows per instruction.
        __syncwarp();
#pragma unroll
        for (int c = 0; c < 16; c += 4)
          *reinterpret_cast<uint4*>(s_t + tr_off(lane, c >> 2)) = make_uint4(r[c], r[c + 1], r[c + 2], r[c + 3]);
        __syncwarp();
        if (vec_ok) {
          const int cq = (lane & 3) * 4, n = c0 + cq;
          if (n < a.n_out) {
            const float4 bb = *reinterpret_cast<const float4*>(s_bias + n);
            const int64_t ooff = dense_out_off(a, n);
            float4 v[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) v[i] = *reinterpret_cast<const float4*>(s_t + tr_off(i * 8 + (lane >> 2), lane & 3));
            if (a.accumulate && !a.out16) {
#pragma unroll
              for (int i = 0; i < 4; ++i) {
                if (oo_r[i] < 0) continue;
                const float4 pv = *reinterpret_cast<const float4*>(a.out + oo_r[i] + ooff);
                v[i].x += pv.x; v[i].y += pv.y; v[i].z += pv.z; v[i].w += pv.w;
              }
            }
#pragma unroll
            for (int i = 0; i < 4; ++i) {  // branch free up to the (predicated) store
              v[i].x += bb.x; v[i].y += bb.y; v[i].z += bb.z; v[i].w += bb.w;
              if (a.act_fn == XPGNN_ACT_SIGMOID) {
                v[i] = sigmoid4(v[i]);
              } else {
                v[i].x = fmaxf(v[i].x, lower); v[i].y = fmaxf(v[i].y, lower); v[i].z = fmaxf(v[i].z, lower); v[i].w = fmaxf(v[i].w, lower);
              }
              v[i].x *= rs_r[i]; v[i].y *= rs_r[i]; v[i].z *= rs_r[i]; v[i].w *= rs_r[i];
            }
            if (XP_EXP(a, 1)) {
            } else if (a.out16) {
              __nv_bfloat16* out16 = reinterpret_cast<__nv_bfloat16*>(a.out);
#pragma unroll
              for (int i = 0; i < 4; ++i)
                if (oo_r[i] >= 0) *reinterpret_cast<uint2*>(out16 + oo_r[i] + ooff) = pack_bf16(v[i]);
            } else {
#pragma unroll
              for (int i = 0; i < 4; ++i)
                if (oo_r[i] >= 0) *reinterpret_cast<float4*>(a.out + oo_r[i] + ooff) = v[i];
            }
          }
        } else if (ok) {
          scalar_epilogue(s_t + lane * TR_STRIDE, (lane >> 1) & 3, c0, a.n_out, s_bias, a.out + oo, a.cw_out, a.cw_out_lg, a.out_chunk_stride, a.accumulate,
                          a.act_fn, rs);
        }
      }
      tc_fence_before();
      mbar_arrive(&bar_acc_empty[ab]);
    }
    if (dbg && blockIdx.x == 0 && tid == 0) {
      dbg[5] = (unsigned long long)(clock64() - t_role0);
      dbg[6] = w_accfull;
      dbg[7] = (unsigned long long)my_tiles;
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem_base, tmem_cols);
}

// ------------------------------------------------------------------ host
static size_t tc_b_bytes(const DenseArgs& d, int mode) {
  const int n_pad = (d.n_out + 15) / 16 * 16;
  return (size_t)n_pad * d.k * (mode == 0 ? 8 : 2);
}
static int tc_stages(const DenseArgs& d, int mode) {
  const size_t stage = mode == 0 ? TcCfg<0>::A_STAGE_BYTES : TcCfg<1>::A_STAGE_BYTES;
  const size_t budget = 204 * 1024;  // + ~22 KB static (transposition blocks, bias, barriers) < 227 KB
  const size_t b = tc_b_bytes(d, mode);
  if (b + 2 * stage > budget) return 0;
  return (int)std::min<size_t>(MAX_STAGES, (budget - b) / stage);
}

static bool tc_eligible(const DenseArgs& d, int mode) {
  if (d.k <= 0 || d.k % KC != 0 || d.n_out < 8 || d.n_out > 256) return false;
  // bf16 storage: bf16 MMA mode, tile table rows, float4-able output, no accumulate into a bf16 destination
  if ((d.in16 || d.out16) && (mode != 1 || d.accumulate || (d.n_out & 3) || (d.ld_in & 7) || (d.in_chunk_stride & 7))) return false;
  if (d.M >= (1ll << 31) - 256 || d.rows_per_s <= 0) return false;
  if (d.ld_in % 4 != 0 || d.in_s_stride % 4 != 0 || d.in_chunk_stride % 4 != 0 || ((uintptr_t)d.in & 15) != 0 || ((uintptr_t)d.w & 15) != 0)
    return false;
  return tc_stages(d, mode) >= 2;
}

// G4: landed hi stages that fit next to the weights and the G4_LO lo stages (0: the gather4 form does not apply)
static int g4_stages(const DenseArgs& d) {
  static int budget = -1;  // dynamic shared memory a CTA of the G4 kernel may use
  if (budget < 0) {
    int dev = 0, optin = 0;
    cudaFuncAttributes fa;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev) != cudaSuccess ||
        cudaFuncGetAttributes(&fa, dense_tc_kernel<0, true>) != cudaSuccess) {
      (void)cudaGetLastError();
      return 0;
    }
    budget = optin - (int)fa.sharedSizeBytes - 1024;  // 1024: alignment of the swizzled stages
  }
  const int64_t room = (int64_t)budget - (int64_t)tc_b_bytes(d, 0);
  return (int)std::min<int64_t>(G4_MAX_HI, std::max<int64_t>(room / G4_PART - G4_LO, 0));
}
// rows of the [rows][32 floats] view that the tile table can name: slots below ceil(M / slot tiles), nodes below
// in_chunk_stride / 32 (a chunk holds every node)
static int64_t g4_rows(const DenseArgs& d) {
  const int64_t slot_rows = ceil_div((int64_t)d.rows_per_s, (int64_t)TM) * TM;
  const int64_t n_slots = ceil_div(d.M, slot_rows);
  return ((n_slots - 1) * d.in_s_stride + (int64_t)(d.k / KC) * d.in_chunk_stride) / 32;
}
// TF32x3 with a chunk-major input of 32-float chunks, rows from the tile table: A by TMA gather4 (option dense_tma)
static bool g4_eligible(const DenseArgs& d, int mode) {
  if (mode != 0 || !knobs().dense_tma || !d.rows_packed || d.in16 || d.cw_in != 32 || d.ld_in != 32) return false;
  if (d.in_s_stride % 32 != 0 || d.in_chunk_stride % 32 != 0 || ((uintptr_t)d.in & 15) != 0 || ((uintptr_t)d.rows_packed & 15) != 0) return false;
  if (g4_rows(d) >= (1ll << 31)) return false;  // gather4 row coordinates are int32
  return g4_stages(d) >= 2;
}

int launch_dense_tc(const DenseArgs& d_in, int mode, cudaStream_t st) {
  DenseArgs d = d_in;
#ifdef XPGNN_EXPERIMENTS  // ablation build only (make EXPERIMENTS=1): never in the shipped library
  if (const char* e = getenv("XPGNN_DENSE_EXP")) d.exp_flags = atoi(e);
  if (const char* e = getenv("XPGNN_DENSE_BACKOFF")) {
    const int v = atoi(e);
    XP_CHECK(cudaMemcpyToSymbolAsync(g_backoff_after, &v, sizeof(int), 0, cudaMemcpyHostToDevice, st));
  }
#else
  d.exp_flags = 0;
#endif
  {
    static int hint_set = 0;  // value of g_wait_hint_ns on the device (one device per process)
    const int want = knobs().dense_wait_ns;
    if (want != hint_set) {
      XP_CHECK(cudaMemcpyToSymbolAsync(g_wait_hint_ns, &want, sizeof(int), 0, cudaMemcpyHostToDevice, st));
      hint_set = want;
    }
  }
  XP_REQUIRE(tc_eligible(d, mode), "shape not eligible for the tensor-core dense path");
  const int n_pad = (d.n_out + 15) / 16 * 16;
  uint32_t cols = 32;
  while ((int)cols < 2 * n_pad) cols <<= 1;  // two accumulator buffers
  const bool g4 = g4_eligible(d, mode);
  const int stages = g4 ? g4_stages(d) : tc_stages(d, mode);
  const size_t smem = g4 ? tc_b_bytes(d, mode) + (size_t)(stages + G4_LO) * G4_PART + 1024
                         : tc_b_bytes(d, mode) + (size_t)stages * (mode == 0 ? TcCfg<0>::A_STAGE_BYTES : TcCfg<1>::A_STAGE_BYTES);
  CUtensorMap tmap;
  memset(&tmap, 0, sizeof tmap);
  if (g4 && rows128_tensor_map(d.in, (uint64_t)g4_rows(d), true, &tmap)) return 1;
  const int64_t tiles = ceil_div(d.M, TM);
  const int grid = (int)std::min<int64_t>(tiles, kNumSMs);
  // XPGNN_DENSE_DBG=1: per-role cycle counters of CTA 0 (synchronises; diagnostics only)
#ifdef XPGNN_EXPERIMENTS
  static const bool dbg_on = getenv("XPGNN_DENSE_DBG") != nullptr;
#else
  constexpr bool dbg_on = false;
#endif
  unsigned long long* dbg = nullptr;
  if (dbg_on) {
    XP_CHECK(cudaMalloc(&dbg, 8 * sizeof(unsigned long long)));
    XP_CHECK(cudaMemsetAsync(dbg, 0, 8 * sizeof(unsigned long long), st));
  }
  void (*k)(const DenseArgs, int, uint32_t, int, unsigned long long*, const CUtensorMap) =
      g4 ? dense_tc_kernel<0, true> : (mode == 0 ? dense_tc_kernel<0, false> : dense_tc_kernel<1, false>);
  XP_CHECK(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  XP_LAUNCH(k, grid, g4 ? G4_THREADS : TC_THREADS, smem, st, d, n_pad, cols, stages, dbg, tmap);
  if (dbg_on) {
    unsigned long long h[8];
    XP_CHECK(cudaStreamSynchronize(st));
    XP_CHECK(cudaMemcpy(h, dbg, sizeof h, cudaMemcpyDeviceToHost));
    XP_CHECK(cudaFree(dbg));
    fprintf(stderr, "[dense_tc] tiles/CTA %llu stages %d | loader total %llu wait_empty %llu | mma total %llu wait_full %llu wait_acc_empty %llu | epilogue total %llu wait_acc_full %llu (cycles)\n",
            h[7], stages, h[0], h[1], h[2], h[3], h[4], h[5], h[6]);
  }
  return 0;
}

bool dense_tc_eligible(const DenseArgs& d, int mode) { return tc_eligible(d, mode); }

}  // namespace xpgnn
