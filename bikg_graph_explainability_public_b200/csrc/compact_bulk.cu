// Masked SpMM of layers >= 1 (aggregate-first: unweighted sums of pre-scaled 128-byte row pieces, out = scale * sum),
// warp-specialised: the gathers are ASYNCHRONOUS COPIES into a shared-memory ring, so the data in flight is bounded by
// shared memory instead of registers and the load issue is decoupled from the arithmetic.
//
// What the copy engines of this SM deliver for 128-byte rows (measured; profiles/r02_summary.md section 1b,
// tools/tma_gather4_probe.cu): LDGSTS (cp.async) 16 bytes per cycle per SM -- one 16-byte lane request per cycle;
// per-lane cp.async.bulk (UBLKCP takes its operands from uniform registers, so a warp issues its 32 copies one by one)
// 9 - 15; the TMA gather4 form (UTMALDG.2D.GATHER4: 4 rows of a 2-D tensor map per instruction, row indices in registers)
// 29.7 = 8.4 TB/s per GPU, TMA-unit bound; plain LDG.128 > 40 (11.3 TB/s in tools/gather_probe.cu).  Alone, this kernel is
// therefore SLOWER than the register-queue kernel (cspmm_seg_kernel, compact.cu): 19 - 36 ms per C3 tile against 11.1 when it was
// measured (8.9 now).
// But the register-queue kernel is not fabric bound either -- it is short of registers for gathers in flight -- and the TMA
// unit is idle while it runs.  MODE 3 (gather4) is built to run NEXT TO it: both kernels take 32-row blocks from the same
// in-order work counter, this one with few warps and no register queue, so the TMA unit adds its bytes per cycle to those of
// the LSU path (launch_cspmm, option seg_tma).  Sums run in stream order in both kernels: results do not depend on which
// kernel took a block.
//
//   * one SCHEDULER warp takes items (32-row blocks: slot, chunk, 128-row tile, quarter -- the numbering of
//     cspmm_seg_kernel) IN ORDER from the global work counter, loads the block's row ids / list offsets two items ahead
//     of their use and publishes a descriptor in shared memory: per row the inclusive end of its part of the gather STREAM
//     (for GCN the row itself first -- the operands are pre-scaled by deg^-1/2, so the unit self loop is one more
//     unweighted term -- then its active sources in list order), the row id and its first list entry;
//   * P PRODUCER warps walk the stream 32 positions (= one ring stage) at a time, across item boundaries, with the
//     source ids of their next stages already loading: lane = position, its row by binary search over the row ends, its
//     source id from the compacted list; then MODE 0: one bulk copy per lane (UBLKCP), MODE 1 / 2: 8 x cp.async (.cg / .ca,
//     8 lanes x 16 bytes per row piece), MODE 3: lanes 0 .. 7 issue one gather4 each (4 consecutive positions = 512 bytes
//     of the stage); completion is counted on the stage's `full` mbarrier (transaction bytes, or
//     cp.async.mbarrier.arrive.noinc);
//   * C CONSUMER warps only read shared memory: a group of 8 lanes (float4 each) owns a row, adds its pieces in stream
//     order, scales and stores it.  Rounds of 4 rows are dealt round-robin to the warps; control flow is warp-uniform
//     (groups waiting or looping on their own serialised the warp); a warp releases a stage (one arrival per warp on its
//     `empty` mbarrier) after having seen it full -- that makes an early arrival for a later use of the slot impossible --
//     and consumes rounds longer than NS / 4 stages window by window, so a row may be longer than the whole ring.
//
// Ring: NS stages x 32 slots x 128 bytes.  Rows with more than long_cnt active in-edges are not part of the stream
// (cspmm_long_kernel sums them, as for the other variants).
#include <cuda.h>

#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <tuple>
#include <utility>

#include "compact_internal.cuh"

namespace xpgnn {

namespace {

constexpr int kBgDesc = 8;   // item descriptors in flight
constexpr int kBgRows = 32;  // rows per item

struct BgDesc {
  int aend[kBgRows];     // stream positions of rows 0 .. r (inclusive prefix), relative to the item
  int v[kBgRows];        // node id | -1: no row here / hub row
  uint32_t e[kBgRows];   // first list entry of the row
  int t, c, len, live;   // live < 0: no more items
  uint32_t stage0;       // global stage index (per CTA) of the item's first stage
  int pad[3];
};

// cycle counters of CTA 0 (scheduler, producer 0, consumer 0): only in the experiment build (make EXPERIMENTS=1, XPGNN_BG_DBG=1)
#ifdef XPGNN_EXPERIMENTS
__device__ unsigned long long g_bg_dbg[16];
#define BG_TIMED(acc, stmt)                                  \
  do {                                                       \
    const long long _t0 = clock64();                         \
    stmt;                                                    \
    acc += (unsigned long long)(clock64() - _t0);            \
  } while (0)
#else
#define BG_TIMED(acc, stmt) \
  do {                      \
    stmt;                   \
  } while (0)
#endif

template <int NS>
struct BgSmem {
  alignas(128) char ring[NS][32][128];
  BgDesc desc[kBgDesc];
  uint64_t full[NS], empty[NS], dfull[kBgDesc], dempty[kBgDesc];
  int start[33];
  int nact[32];
};

__device__ __forceinline__ uint32_t bg_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void bg_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bg_u32(bar)), "r"(count));
}
__device__ __forceinline__ void bg_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bg_u32(bar)) : "memory");
}
__device__ __forceinline__ void bg_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bg_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool bg_test(uint64_t* bar, uint32_t parity) {
  uint32_t done;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(done)
      : "r"(bg_u32(bar)), "r"(parity)
      : "memory");
  return done != 0;
}
template <int SLEEP_NS>
__device__ __forceinline__ void bg_wait(uint64_t* bar, uint32_t parity) {
  for (uint32_t spin = 0; !bg_test(bar, parity); ++spin) {
    if (SLEEP_NS) __nanosleep(SLEEP_NS);
    if (spin > (1u << 22)) __trap();  // never hang the GPU: a lost arrival becomes an error
  }
}
// one bulk copy (TMA unit) global -> shared; both ends 16-byte aligned; completion in bytes on `bar`
__device__ __forceinline__ void bg_bulk_copy(uint32_t smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_dst), "l"(gmem_src),
               "r"(bytes), "r"(bg_u32(bar))
               : "memory");
}
// TMA gather4: rows r0 .. r3 (columns [0, box width)) of the 2-D tensor map -> 4 consecutive box rows at smem_dst
__device__ __forceinline__ void bg_gather4(uint32_t smem_dst, const CUtensorMap* tmap, int r0, int r1, int r2, int r3, uint64_t* bar) {
  asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile::gather4.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, %7}], [%2];" ::"r"(smem_dst),
               "l"(tmap), "r"(bg_u32(bar)), "r"(0), "r"(r0), "r"(r1), "r"(r2), "r"(r3)
               : "memory");
}
__device__ __forceinline__ void bg_add(float4& acc, const float4& x) {  // two packed adds
  asm("{\n\t.reg .b64 a0, a1, x0, x1, one;\n\t"
      "mov.b64 a0, {%0, %1};\n\tmov.b64 a1, {%2, %3};\n\tmov.b64 x0, {%4, %5};\n\tmov.b64 x1, {%6, %7};\n\t"
      "mov.b64 one, {0f3F800000, 0f3F800000};\n\t"
      "fma.rn.f32x2 a0, x0, one, a0;\n\tfma.rn.f32x2 a1, x1, one, a1;\n\t"
      "mov.b64 {%0, %1}, a0;\n\tmov.b64 {%2, %3}, a1;\n\t}"
      : "+f"(acc.x), "+f"(acc.y), "+f"(acc.z), "+f"(acc.w)
      : "f"(x.x), "f"(x.y), "f"(x.z), "f"(x.w));
}

// NS: ring stages (a power of two).  MODE 0: bulk copies (UBLKCP) | 1: cp.async.cg | 2: cp.async.ca | 3: TMA gather4.
// P / C: producer / consumer warps.  MINB: CTAs per SM the register budget is sized for (the hybrid launch shares the SM).
template <int NS, int MODE, int P, int C, int MINB>
__global__ void __launch_bounds__(32 * (1 + P + C), MINB) cspmm_bulk_kernel(const CspmmArgs a, const __grid_constant__ CUtensorMap tmap) {
  extern __shared__ __align__(128) unsigned char bg_raw[];
  BgSmem<NS>& S = *reinterpret_cast<BgSmem<NS>*>(bg_raw);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (threadIdx.x <= a.nb) S.start[threadIdx.x] = a.slot_tile_start[threadIdx.x];
  if (threadIdx.x < a.nb) S.nact[threadIdx.x] = a.slot_info[threadIdx.x].x;
  if (threadIdx.x == 0) {
    for (int i = 0; i < NS; ++i) { bg_init(&S.full[i], (MODE == 0 || MODE == 3) ? 1 : 32); bg_init(&S.empty[i], C); }
    for (int i = 0; i < kBgDesc; ++i) { bg_init(&S.dfull[i], 1); bg_init(&S.dempty[i], P + C); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  const bool gcn = a.kind == XPGNN_CONV_GCN;
  const int gself = gcn ? 1 : 0;

  if (warp == 0) {
    // ================= scheduler: items in global order -> descriptors =================
    // Software pipeline: while item n is turned into a descriptor, the metadata loads of n + 1 and n + 2 and the counter
    // fetch of n + 3 are in flight (under load a DRAM round trip is several microseconds).
    const int total = S.start[a.nb] * a.n_chunks * 4;  // 32-row blocks, ordered slot / chunk / 128-row tile / quarter
    struct Meta {
      int item, t, c, v;
      uint32_t e, f;
    };
    int t_ld = 0;
    auto grab_raw = [&]() {  // lane 0 holds the value; broadcast when it is needed
      int it = 0;
      if (lane == 0) it = atomicAdd(a.counter, 1);
      return it;
    };
    auto load_meta = [&](int item, Meta& m) {
      m.item = item;
      m.t = 0; m.c = 0; m.v = -1; m.e = 0; m.f = 0;
      if (item >= total) return;
      const int idx = item >> 2;
      while (idx >= S.start[t_ld + 1] * a.n_chunks) ++t_ld;
      const int ntb = S.start[t_ld + 1] - S.start[t_ld];
      const int rem = idx - S.start[t_ld] * a.n_chunks;
      m.t = t_ld;
      m.c = rem / ntb;
      const int i = (rem - m.c * ntb) * 128 + (item & 3) * 32 + lane;
      if (i < S.nact[t_ld]) {
        m.v = __ldcs(a.act_list + (int64_t)t_ld * a.N + i);
        const uint32_t* rp = a.rowptr_c + (int64_t)t_ld * (a.N + 1) + i;
        m.e = __ldcs(rp);
        m.f = __ldcs(rp + 1);
      }
    };
    Meta A, B;
    unsigned long long t_w0 = 0;
    const long long t_begin = clock64();
    load_meta(__shfl_sync(0xffffffffu, grab_raw(), 0), A);
    load_meta(__shfl_sync(0xffffffffu, grab_raw(), 0), B);
    int raw = grab_raw();
    uint32_t stage_next = 0;
    for (uint32_t n = 0;; ++n) {
      const int d = n % kBgDesc;
      BgDesc& D = S.desc[d];
      if (n >= kBgDesc) BG_TIMED(t_w0, bg_wait<64>(&S.dempty[d], ((n / kBgDesc) - 1) & 1));
      if (A.item >= total) {
        if (lane == 0) D.live = -1;
        __syncwarp();
        if (lane == 0) bg_arrive(&S.dfull[d]);
#ifdef XPGNN_EXPERIMENTS
        if (blockIdx.x == 0 && lane == 0) { g_bg_dbg[0] = (unsigned long long)(clock64() - t_begin); g_bg_dbg[1] = t_w0; g_bg_dbg[2] = n; }
#endif
        break;
      }
      const uint32_t cnt = A.f - A.e;
      const bool mine = A.v >= 0 && !(a.long_cnt > 0 && cnt > (uint32_t)a.long_cnt);
      int x = mine ? (int)cnt + gself : 0;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int y = __shfl_up_sync(0xffffffffu, x, o);
        if (lane >= o) x += y;
      }
      D.aend[lane] = x;
      D.v[lane] = mine ? A.v : -1;
      D.e[lane] = A.e;
      const int len = __shfl_sync(0xffffffffu, x, 31);
      if (lane == 0) { D.t = A.t; D.c = A.c; D.len = len; D.live = 1; D.stage0 = stage_next; }
      stage_next += (uint32_t)((len + 31) >> 5);
      __syncwarp();
      if (lane == 0) bg_arrive(&S.dfull[d]);
      A = B;
      load_meta(__shfl_sync(0xffffffffu, raw, 0), B);
      raw = grab_raw();
    }
  } else if (warp <= P) {
    // ================= producers: stream positions -> copies into the ring =================
    // Producer pw owns the stages whose GLOBAL index is pw mod P.  It walks them as one sequence across item boundaries
    // with the source ids of the next kAhead stages already loading (a FETCH cursor runs ahead of the ISSUE cursor), so
    // neither a stage nor the first stage of an item waits for a list load.
    constexpr int kAhead = 3;
    const int pw = warp - 1;
    const int sub = lane & 7, grp = lane >> 3;
    // ---- fetch cursor ----
    uint32_t fn = 0;        // item the cursor is in
    int fk = 0, f_nst = -1; // next stage of the item for this warp; f_nst < 0: item not opened yet
    bool f_end = false;
#ifdef XPGNN_EXPERIMENTS
    const bool bg_fake = a.l2_gather == 77;  // set through the l2_gather knob in the experiment build
#endif
    unsigned long long t_w0 = 0, t_w1 = 0, t_f = 0, n_st = 0;
    const long long t_begin = clock64();
    uint32_t done_n = 0;  // this warp has arrived on dempty of every item below done_n
    auto finish_items = [&](uint32_t upto) {
      while (done_n < upto) {
        __syncwarp();
        if (lane == 0) bg_arrive(&S.dempty[done_n % kBgDesc]);
        ++done_n;
      }
    };
    // 0: produced the next stage of this warp | 1: the next item's descriptor is not there yet (only when !may_block) | 2: end
    auto f_next = [&](int& id, uint32_t& g, uint32_t& item_no, bool may_block) -> int {
      for (;;) {
        if (f_end) return 2;
        const BgDesc& D = S.desc[fn % kBgDesc];
        if (f_nst < 0) {  // open item fn
          if (may_block) BG_TIMED(t_w0, bg_wait<32>(&S.dfull[fn % kBgDesc], (fn / kBgDesc) & 1));
          else if (!bg_test(&S.dfull[fn % kBgDesc], (fn / kBgDesc) & 1)) return 1;
          if (D.live < 0) { f_end = true; return 2; }
          f_nst = (D.len + 31) >> 5;
          fk = (int)(((uint32_t)pw + (uint32_t)P - (D.stage0 % (uint32_t)P)) % (uint32_t)P);
        }
        if (fk < f_nst) {
          const int len = D.len, pos = fk * 32 + lane;
          id = -1;
#ifdef XPGNN_EXPERIMENTS
          if (bg_fake && pos < len) {  // ceiling experiment: pseudo-random source ids without the search / the list load (WRONG sums)
            id = (int)(((uint32_t)pos * 2654435761u + D.stage0 * 40503u + (uint32_t)fk * 7919u) % (uint32_t)a.N);
          } else
#endif
          if (pos < len) {
            int r = 0;  // rows whose stream ends at or before pos
#pragma unroll
            for (int step = kBgRows / 2; step >= 1; step >>= 1)
              if (D.aend[r + step - 1] <= pos) r += step;
            const int ar = r ? D.aend[r - 1] : 0;
            if (gcn && pos == ar) id = D.v[r];
            else id = __ldcs(a.ccol + a.slot_base[D.t] + D.e[r] + (uint32_t)(pos - ar - gself));
          }
          g = D.stage0 + (uint32_t)fk;
          item_no = fn;
          fk += P;
          return 0;
        }
        ++fn;
        f_nst = -1;
        // may_block means the queue is empty: every stage this warp owns in the items before the cursor has been issued.
        // Let go of them NOW -- a warp that owns no stage in kBgDesc consecutive (short) items would otherwise wait for a
        // descriptor the scheduler can only publish after this warp's arrival on an item it is still holding.
        if (may_block) finish_items(fn);
      }
    };
    auto issue = [&](int id, uint32_t g, uint32_t item_no) {
      finish_items(item_no);  // every stage of the earlier items has been issued
      const BgDesc& D = S.desc[item_no % kBgDesc];
      const uint32_t slot = g % NS, use = g / NS;
      const int k = (int)(g - D.stage0);
      const int n_valid = min(32, D.len - k * 32);
      if (use > 0) BG_TIMED(t_w1, bg_wait<64>(&S.empty[slot], (use - 1) & 1));
      ++n_st;
      if (MODE == 3) {
        // rows of the 2-D view [all slots x chunks x nodes][32 floats] of the operand buffer: row = (t, c) base + node
        const int row_base = (int)(((int64_t)D.t * a.in_s_stride + (int64_t)D.c * a.in_chunk_stride) >> 5);
        const int n_g4 = (n_valid + 3) >> 2;
        if (lane == 0) bg_arrive_expect_tx(&S.full[slot], (uint32_t)n_g4 * 512u);
        // positions past the end of the stream are padded with the first id of the stage (loaded, never summed)
        const int id0 = __shfl_sync(0xffffffffu, id, 0);
        int r4[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int idj = __shfl_sync(0xffffffffu, id, (4 * lane + j) & 31);
          r4[j] = row_base + (idj >= 0 ? idj : id0);
        }
        __syncwarp();
        if (lane < n_g4) bg_gather4(bg_u32(&S.ring[slot][(4 * lane) & 31][0]), &tmap, r4[0], r4[1], r4[2], r4[3], &S.full[slot]);
      } else {
        const char* in_c = reinterpret_cast<const char*>(a.in + (int64_t)D.t * a.in_s_stride + (int64_t)D.c * a.in_chunk_stride);
        if (MODE == 0) {
          if (lane == 0) bg_arrive_expect_tx(&S.full[slot], (uint32_t)n_valid * 128u);
          __syncwarp();
          if (id >= 0) {
            const char* src;
            asm("mad.wide.u32 %0, %1, 128, %2;" : "=l"(src) : "r"((uint32_t)id), "l"(in_c));
            bg_bulk_copy(bg_u32(&S.ring[slot][lane][0]), src, 128u, &S.full[slot]);
          }
        } else {
          const uint32_t dst0 = bg_u32(&S.ring[slot][0][0]) + (uint32_t)sub * 16u;
          const char* in_l = in_c + sub * 16;
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const int pj = j * 4 + grp;  // slot of the stage: 8 lanes x 16 bytes each
            const int idj = __shfl_sync(0xffffffffu, id, pj);
            if (idj >= 0) {
              const char* src;
              asm("mad.wide.u32 %0, %1, 128, %2;" : "=l"(src) : "r"((uint32_t)idj), "l"(in_l));
              if (MODE == 1) asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst0 + (uint32_t)pj * 128u), "l"(src) : "memory");
              else asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(dst0 + (uint32_t)pj * 128u), "l"(src) : "memory");
            }
          }
          // the stage is full once every producer lane's copies have landed (32 arrivals, none added by the instruction)
          asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(bg_u32(&S.full[slot])) : "memory");
        }
      }
    };
    // The queue is a FIFO over kAhead register slots used round-robin (the loop is unrolled, so slot indices are compile-time
    // constants and the ids stay in registers -- their loads may still be in flight).  Entries are issued strictly in order:
    // once a refill finds the next descriptor missing, nothing is appended until the queue has drained; only an EMPTY queue
    // blocks on a descriptor, after this warp has let go of every earlier item (so the scheduler can always publish it).
    int q_id[kAhead];
    uint32_t q_g[kAhead], q_n[kAhead];
    bool q_ok[kAhead];
#pragma unroll
    for (int i = 0; i < kAhead; ++i) { q_ok[i] = false; q_id[i] = -1; q_g[i] = 0; q_n[i] = 0; }
    bool stalled = true, ended = false, live = true;  // stalled: no appends until the head finds the queue empty
    while (live) {
#pragma unroll
      for (int i = 0; i < kAhead; ++i) {
        if (live && !q_ok[i]) {  // in-order FIFO: an empty head means an empty queue
          if (ended) {
            live = false;
          } else {
            finish_items(fn);  // all of this warp's stages of the items before the cursor have been issued
            const int rc = f_next(q_id[i], q_g[i], q_n[i], true);
            if (rc == 2) { ended = true; live = false; }
            else {
              q_ok[i] = true;
              stalled = false;
#pragma unroll
              for (int j = 1; j < kAhead; ++j) {  // top the queue up behind the new head
                const int sj = (i + j) % kAhead;
                if (!stalled && !ended) {
                  const int r2 = f_next(q_id[sj], q_g[sj], q_n[sj], false);
                  q_ok[sj] = r2 == 0;
                  if (r2 == 1) stalled = true;
                  if (r2 == 2) ended = true;
                }
              }
            }
          }
        }
        if (live) {
          issue(q_id[i], q_g[i], q_n[i]);
          q_ok[i] = false;
          if (!stalled && !ended) {  // slot i becomes the tail
            int r2;
            BG_TIMED(t_f, r2 = f_next(q_id[i], q_g[i], q_n[i], false));
            q_ok[i] = r2 == 0;
            if (r2 == 1) stalled = true;
            if (r2 == 2) ended = true;
          }
        }
      }
    }
    finish_items(fn);  // fn = the item that carried the end marker
#ifdef XPGNN_EXPERIMENTS
    if (blockIdx.x == 0 && pw == 0 && lane == 0) {
      g_bg_dbg[4] = (unsigned long long)(clock64() - t_begin); g_bg_dbg[5] = t_w0; g_bg_dbg[6] = t_w1; g_bg_dbg[7] = t_f; g_bg_dbg[8] = n_st;
    }
#endif
  } else {
    // ================= consumers: a group of 8 lanes sums a row from the ring =================
    // Round k of an item = rows 4k .. 4k + 3 (one per group), dealt round-robin to the consumer warps, so all warps work
    // next to the fill front.  Releases are per WARP (C arrivals per stage): before a round the warp releases every stage
    // below the round's first one -- lanes take different stages; each stage is seen full first -- and a round longer than
    // kWin stages is consumed window by window, so no row length can hold more than kWin + 1 stages unreleased.
    constexpr int kWin = NS / 4;
    constexpr int kPar = NS < 32 ? NS : 32;
    const int cw = warp - 1 - P, sub = lane & 7, grp = lane >> 3;
    uint32_t rel = 0;   // every stage below `rel` has been released by this warp (warp-uniform)
    unsigned long long t_w0 = 0, t_w1 = 0, t_w2 = 0, n_rd = 0;
    const long long t_begin = clock64();
    auto release_to = [&](uint32_t target) {
      while (rel < target) {
        const uint32_t g = rel + (uint32_t)lane;
        if (lane < kPar && g < target) {  // no lane may wait on a use of a slot that is two uses ahead of the barrier's phase
          bg_wait<20>(&S.full[g % NS], (g / NS) & 1);
          bg_arrive(&S.empty[g % NS]);
        }
        rel = min(target, rel + (uint32_t)kPar);
      }
    };
    for (uint32_t n = 0;; ++n) {
      const int d = n % kBgDesc;
      const BgDesc& D = S.desc[d];
      BG_TIMED(t_w0, bg_wait<32>(&S.dfull[d], (n / kBgDesc) & 1));
      if (D.live < 0) break;
      const uint32_t stage0 = D.stage0;
      const int nst = (D.len + 31) >> 5;
      float* out_c = a.out + (int64_t)D.t * a.out_s_stride + (int64_t)D.c * a.out_chunk_stride + sub * 4;
      for (int k = cw; k < kBgRows / 4; k += C) {
        const int P0 = k ? D.aend[4 * k - 1] : 0, P1 = D.aend[4 * k + 3];
        if (P1 == P0 && D.v[4 * k] < 0 && D.v[4 * k + 1] < 0 && D.v[4 * k + 2] < 0 && D.v[4 * k + 3] < 0) continue;  // no rows here
        const int r = 4 * k + grp;
        const int v = D.v[r];
        const int a0 = r ? D.aend[r - 1] : 0, a1 = D.aend[r];
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
        const int sa = P0 >> 5, sb = (P1 + 31) >> 5;  // the round's positions sit in stages [sa, sb) of the item
        BG_TIMED(t_w1, release_to(stage0 + (uint32_t)sa));
        ++n_rd;
        for (int ws = sa; ws < sb; ws += kWin) {
          const int we = min(ws + kWin, sb);
          for (int gg = ws; gg < we; ++gg) {
            const uint32_t g = stage0 + (uint32_t)gg;
            BG_TIMED(t_w2, bg_wait<20>(&S.full[g % NS], (g / NS) & 1));
          }
          const int lo = max(a0, ws << 5), hi = min(a1, we << 5);
          const int n_it = __reduce_max_sync(0xffffffffu, max(hi - lo, 0));
          const uint32_t pos0 = stage0 * 32u + (uint32_t)lo;  // ring slot of position q: (stage0 * 32 + q) mod (NS * 32)
          for (int i = 0; i < n_it; i += 4) {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              if (lo + i + j < hi) {
                const uint32_t slot = (pos0 + (uint32_t)(i + j)) & (uint32_t)(NS * 32 - 1);
                bg_add(acc, *reinterpret_cast<const float4*>(&S.ring[0][0][0] + (size_t)slot * 128 + sub * 16));
              }
            }
          }
          __syncwarp();
          if (we < sb) release_to(stage0 + (uint32_t)we);
        }
        if (v >= 0) {
          const uint32_t cnt = (uint32_t)(a1 - a0 - gself);
          float sc = 0.f;  // SAGE row without an active in-edge: empty mean
          if (gcn) sc = gcn_dinv(cnt);
          else if (cnt) sc = 1.0f / (float)cnt;
          __stcs(reinterpret_cast<float4*>(out_c + (int64_t)v * 32), make_float4(acc.x * sc, acc.y * sc, acc.z * sc, acc.w * sc));
        }
        __syncwarp();
      }
      BG_TIMED(t_w1, release_to(stage0 + (uint32_t)nst));
      __syncwarp();
      if (lane == 0) bg_arrive(&S.dempty[d]);
    }
#ifdef XPGNN_EXPERIMENTS
    if (blockIdx.x == 0 && cw == 0 && lane == 0) {
      g_bg_dbg[10] = (unsigned long long)(clock64() - t_begin); g_bg_dbg[11] = t_w0; g_bg_dbg[12] = t_w1; g_bg_dbg[13] = t_w2; g_bg_dbg[14] = n_rd;
    }
#endif
  }
}

template <int NS, int MODE, int P, int C, int MINB>
int bg_launch(const CspmmArgs& a, const CUtensorMap& tmap, cudaStream_t st, int variant) {
  void (*k)(const CspmmArgs, const CUtensorMap) = cspmm_bulk_kernel<NS, MODE, P, C, MINB>;
  const int smem = (int)sizeof(BgSmem<NS>);
  XP_CHECK(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  XP_LAUNCH(k, kNumSMs, 32 * (1 + P + C), smem, st, a, tmap);
#ifdef XPGNN_EXPERIMENTS
  static const bool dbg_on = getenv("XPGNN_BG_DBG") != nullptr;
  static int n_launch = 0;
  if (dbg_on && (n_launch++ % 8) == 7) {
    unsigned long long h[16];
    XP_CHECK(cudaStreamSynchronize(st));
    XP_CHECK(cudaMemcpyFromSymbol(h, g_bg_dbg, sizeof h));
    fprintf(stderr,
            "bg dbg variant %d: sched total %llu wait_dempty %llu items %llu | prod0 total %llu wait_desc %llu wait_empty %llu fetch %llu stages %llu | "
            "cons0 total %llu wait_desc %llu release %llu wait_full %llu rounds %llu\n",
            variant, h[0], h[1], h[2], h[4], h[5], h[6], h[7], h[8], h[10], h[11], h[12], h[13], h[14]);
  }
#endif
  (void)variant;
  return 0;
}

}  // namespace

// Encoding goes through the driver entry point (no link dependency on libcuda).
typedef CUresult (*BgEncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                               const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
int rows128_tensor_map(const float* base, uint64_t rows, bool swizzle128, CUtensorMap* out) {
  static std::mutex mu;
  static std::map<std::tuple<const void*, uint64_t, bool>, CUtensorMap> cache;
  static BgEncodeFn encode = nullptr;
  std::lock_guard<std::mutex> lock(mu);
  auto it = cache.find({base, rows, swizzle128});
  if (it != cache.end()) { *out = it->second; return 0; }
  if (!encode) {
    cudaDriverEntryPointQueryResult qres;
    XP_CHECK(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", (void**)&encode, cudaEnableDefault, &qres));
    XP_REQUIRE(encode != nullptr, "cuTensorMapEncodeTiled is not available");
  }
  CUtensorMap m;
  memset(&m, 0, sizeof m);
  const cuuint64_t dims[2] = {32, rows};
  const cuuint64_t strides[1] = {128};
  const cuuint32_t box[2] = {32, 1};
  const cuuint32_t estr[2] = {1, 1};
  const CUresult r = encode(&m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                            swizzle128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  XP_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled failed");
  if (cache.size() > 64) cache.clear();
  cache[{base, rows, swizzle128}] = m;
  *out = m;
  return 0;
}

int launch_cspmm_bulk(const CspmmArgs& a, int variant, cudaStream_t st) {
  // variant = 100 * mode + ring stages (16 | 32); mode 0 bulk copies | 1 cp.async.cg | 2 cp.async.ca | 3 TMA gather4 |
  // 4 TMA gather4, the small configuration that runs next to cspmm_seg_kernel (2 producer + 4 consumer warps, 16 stages)
  const int mode = variant / 100, ns = variant % 100;
  CUtensorMap tmap;
  memset(&tmap, 0, sizeof tmap);
  if (mode >= 3) {
    XP_REQUIRE(a.in_s_stride % 32 == 0 && a.in_chunk_stride % 32 == 0, "gather4: operand strides must be whole 128-byte rows");
    const uint64_t rows = (uint64_t)((int64_t)(a.nb - 1) * a.in_s_stride + (int64_t)(a.n_chunks - 1) * a.in_chunk_stride) / 32 + (uint64_t)a.N;
    XP_REQUIRE(rows < (1ull << 31), "gather4: row index does not fit 31 bits");
    if (rows128_tensor_map(a.in, rows, false, &tmap)) return 1;
  }
  if (mode == 4) return bg_launch<16, 3, 2, 4, 2>(a, tmap, st, variant);
  if (ns >= 32) {
    if (mode == 0) return bg_launch<32, 0, 8, 8, 1>(a, tmap, st, variant);
    if (mode == 1) return bg_launch<32, 1, 8, 8, 1>(a, tmap, st, variant);
    if (mode == 2) return bg_launch<32, 2, 8, 8, 1>(a, tmap, st, variant);
    return bg_launch<32, 3, 4, 8, 1>(a, tmap, st, variant);
  }
  if (mode == 0) return bg_launch<16, 0, 8, 8, 1>(a, tmap, st, variant);
  if (mode == 1) return bg_launch<16, 1, 8, 8, 1>(a, tmap, st, variant);
  if (mode == 2) return bg_launch<16, 2, 8, 8, 1>(a, tmap, st, variant);
  return bg_launch<16, 3, 4, 8, 1>(a, tmap, st, variant);
}

}  // namespace xpgnn
