// tcgen05 scan + fused top-k' kernel for sm_100a.
//
// Replaces, on B200, the reference's SIMT distance+select kernels
//   fusedL2kNN                cpp/src/neighbors/detail/fused_l2_knn.cuh:186-508   (fp32 FFMA tile + WarpSelect)
//   interleaved_scan (dense)  cpp/src/neighbors/ivf_flat/detail/jit_lto_kernels/interleaved_scan_impl.cuh:70-206
//   coarse GEMM + select_k    cpp/src/neighbors/ivf_pq/ivf_pq_search.cuh:60-168
//   unfused distance-NN       cpp/src/distance/unfused_distance_nn.cuh:54-118
// with one warp-specialised persistent kernel:
//
//   warp 0     TMA producer : query tile (A, resident per work item) + dataset k-blocks (B ring)
//   warp 1     MMA issuer   : tcgen05.mma kind::f16 (bf16 in, fp32 accumulate in TMEM), 128x128 tiles,
//                             split-bf16 products hi*hi + lo*hi + hi*lo  (passes = 3) or hi*hi (passes = 1),
//                             plus ONE extra K=16 step per tile that adds -|x|^2/2 (three bf16 pieces of the fp32
//                             half-norm times a constant column of ones), so the accumulator already holds
//                             t = q.x - |x|^2/2 = -(score) and the epilogue has no per-element arithmetic left
//   warps 2-9  epilogue     : tcgen05.ld one accumulator row per thread (two warps per TMEM lane quarter, 64 columns
//                             each), release the TMEM buffer, then a max-tree per 32 columns against the row's running
//                             threshold; the rare hits go through a per-thread smem queue into a sorted register list.
//
// The accumulator ring is 4 x 128 TMEM columns (all 512), so MMAs run up to three tiles ahead of the slowest
// epilogue warp.  Nothing but the k' (score, position) pairs per query row ever leaves the SM: the n x nq distance
// matrix of the reference's unfused path (n*nq*4 bytes through HBM) is never materialised.
#include "common.hpp"
#include "ptx_sm100.cuh"
#include "scan_tc.cuh"
#include "timing.hpp"

#include <cuda.h>

#include <cmath>
#include <mutex>

namespace b200 {
namespace {

constexpr int kTileBytes  = 128 * 128;  // 128 rows x 64 bf16, SWIZZLE_128B
constexpr int kExtBytes   = 128 * 32;   // 128 rows x 16 bf16, SWIZZLE_32B (the half-norm K extension)
constexpr int kQueue      = 16;         // per-thread pending-insert queue entries
constexpr int kAccBufs    = 4;          // TMEM accumulator ring
constexpr int kEpiWarps   = 8;
constexpr int kEpiThreads = 32 * kEpiWarps;
constexpr int kCols       = 64;         // accumulator columns per epilogue thread and tile
constexpr int kSched      = 4;          // depth of the work-item ring between the producer and its consumers

// PASSES: 1 = hi*hi; 2 = (hi + lo)*hi (exact A side: query rows at fp32 grade against bf16-exact B rows);
//         3 = hi*hi + lo*hi + hi*lo (both sides split)
template <int KB, int PASSES>
struct cfg {
  static constexpr int NA = PASSES >= 2 ? 2 : 1;  // A planes resident in shared memory
  static constexpr int NB = PASSES == 3 ? 2 : 1;  // B planes streamed
  static constexpr int threads     = 64 + kEpiThreads;
  // KB = 1, 2: the query tile (KB k-blocks of 64) stays resident in shared memory for a whole work item.
  // KB = 0: "streamed" — any padded K (multiple of 64): the A k-block travels through the ring next to the B k-block
  //         (dims > 128; costs one extra 16 KB L2 read per plane and k-block, the tile's MMA work grows with K as well).
  static constexpr bool streamed   = KB == 0;
  static constexpr int stages      = streamed ? (PASSES == 1 ? 4 : (PASSES == 2 ? 3 : 2)) : (NB == 2 ? 3 : (NA == 2 ? 5 : 6));
  static constexpr int a_bytes     = streamed ? 0 : NA * KB * kTileBytes;
  static constexpr int b_off       = streamed ? NA * kTileBytes : 0;             // B planes inside a stage
  static constexpr int x_off       = b_off + NB * kTileBytes;                    // half-norm block (kb == 0 stage of a tile)
  static constexpr int stage_bytes = x_off + kExtBytes;
  static constexpr int n_bars      = 2 * stages + 2 + 2 * kAccBufs + 2 * kSched;
  static constexpr size_t smem     = 1024 /*align slack*/ + a_bytes + kExtBytes /*ones*/ + stages * stage_bytes +
                                 kQueue * kEpiThreads * 8 /*queues*/ + n_bars * 8 + kSched * 4 + 16;
};

// KC > 0: fused top-KC epilogue, two candidate lists per (item, query row) — one per 64-column half of the tiles.
// KC == 0: "store" epilogue — every score of the tile is written to
// out_score[out_off + row * out_row_stride + (column within the item's range)] (dense distance block).
template <int KB, int PASSES, int KC>
__global__ void __launch_bounds__(64 + kEpiThreads, 1)
tc_scan_kernel(const __grid_constant__ CUtensorMap tmA_hi, const __grid_constant__ CUtensorMap tmA_lo,
               const __grid_constant__ CUtensorMap tmB_hi, const __grid_constant__ CUtensorMap tmB_lo,
               const __grid_constant__ CUtensorMap tmB_x, const tc_item* __restrict__ items, int n_items_host,
               const int* __restrict__ n_items_dev, int kblocks_rt, int* __restrict__ sched_counter, float* __restrict__ out_score, uint32_t* __restrict__ out_pos,
               int64_t out_row_stride, tc_bound bound)
{
  using C = cfg<KB, PASSES>;
  constexpr int NA = C::NA, NB = C::NB;
  const int nkb = C::streamed ? kblocks_rt : KB;  // k-blocks of 64 per tile
  const int n_items = n_items_dev ? *n_items_dev : n_items_host;
  // 1024-byte alignment is what SWIZZLE_128B operand tiles need; declared on the array (no integer
  // round-trip of the pointer) so that the compiler keeps every access in the shared address space.
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  if (threadIdx.x == 0 && (ptx::smem_u32(smem_raw) & 1023u) != 0) __trap();
  uint8_t* sA    = smem_raw;
  uint8_t* sOnes = sA + C::a_bytes;
  uint8_t* sB    = sOnes + kExtBytes;
  uint2* qe      = reinterpret_cast<uint2*>(sB + C::stages * C::stage_bytes);  // [kQueue][kEpiThreads] {t bits, row position}
  uint64_t* bars = reinterpret_cast<uint64_t*>(qe + kQueue * kEpiThreads);
  uint64_t* full    = bars;
  uint64_t* empty   = bars + C::stages;
  uint64_t* a_full  = bars + 2 * C::stages;
  uint64_t* a_empty = a_full + 1;
  uint64_t* tfull   = a_empty + 1;       // [kAccBufs]
  uint64_t* tempty  = tfull + kAccBufs;  // [kAccBufs]
  uint64_t* s_full  = tempty + kAccBufs;  // [kSched] work-item ring: producer -> MMA issuer + epilogue
  uint64_t* s_empty = s_full + kSched;    // [kSched]
  int* s_item       = reinterpret_cast<int*>(s_empty + kSched);  // [kSched] item index, -1 = no more work
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(s_item + kSched);

  // warp-uniform by construction (shuffle broadcast): lets the compiler keep role dispatch and the issue loops convergent
  const int warp = __shfl_sync(0xffffffffu, static_cast<int>(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tmap(&tmA_hi);
    ptx::prefetch_tmap(&tmB_hi);
    ptx::prefetch_tmap(&tmB_x);
    if (NA == 2) ptx::prefetch_tmap(&tmA_lo);
    if (NB == 2) ptx::prefetch_tmap(&tmB_lo);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < C::stages; ++s) {
      ptx::mbar_init(&full[s], 1);
      ptx::mbar_init(&empty[s], 1);
    }
    ptx::mbar_init(a_full, 1);
    ptx::mbar_init(a_empty, 1);
    for (int s = 0; s < kAccBufs; ++s) {
      ptx::mbar_init(&tfull[s], 1);
      ptx::mbar_init(&tempty[s], kEpiWarps);
    }
    for (int s = 0; s < kSched; ++s) {
      ptx::mbar_init(&s_full[s], 1);
      ptx::mbar_init(&s_empty[s], 1 + kEpiWarps);
    }
    ptx::fence_barrier_init();
  }
  // the constant A-side operand of the half-norm step: every row = {1, 1, 1, 0, 0, 0, 0, 0} in BOTH 16-byte chunks
  // (identical chunks make the tile invariant under the 32-byte swizzle; the B side has zeros in its second chunk)
  if (threadIdx.x < kExtBytes / 16)
    reinterpret_cast<uint4*>(sOnes)[threadIdx.x] = make_uint4(0x3f803f80u, 0x00003f80u, 0u, 0u);
  ptx::fence_proxy_async();
  if (warp == 2) { ptx::tmem_alloc<128 * kAccBufs>(tmem_slot); }
  ptx::tc_fence_before_sync();
  __syncthreads();
  ptx::tc_fence_after_sync();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0);

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer
    // The whole warp runs the (warp-uniform) control flow, one elected lane issues: keeps the loop free of the
    // per-instruction ELECT/branch sequences a single-lane branch would get.
    // Work items are handed out dynamically (one global counter): CTAs that finish early take the next item, and the
    // items of one list — adjacent in the work list — are picked up at about the same time by different SMs, so the
    // list's tiles are read from HBM once and from L2 by the others.
    uint32_t stage = 0, phase = 0, a_phase = 0, ss = 0, sp = 0;
    int static_it = static_cast<int>(blockIdx.x);  // sched_counter == null: plain round-robin over the grid
    for (;;) {
      ptx::mbar_wait(&s_empty[ss], sp ^ 1);
      int it = 0;
      if (lane == 0) {
        if (sched_counter != nullptr) {
          it = atomicAdd(sched_counter, 1);
        } else {
          it = static_it;
          static_it += static_cast<int>(gridDim.x);
        }
        if (it >= n_items) it = -1;
        s_item[ss] = it;
        ptx::mbar_arrive(&s_full[ss]);
      }
      it = __shfl_sync(0xffffffffu, it, 0);
      if (++ss == kSched) { ss = 0; sp ^= 1; }
      if (it < 0) break;
      tc_item item = items[it];
      item.a_row0  = __shfl_sync(0xffffffffu, item.a_row0, 0);
      item.b_row0  = __shfl_sync(0xffffffffu, item.b_row0, 0);
      item.n_tiles = __shfl_sync(0xffffffffu, item.n_tiles, 0);
      if constexpr (!C::streamed) {
        ptx::mbar_wait(a_empty, a_phase ^ 1);
        if (ptx::elect_one()) {
          ptx::mbar_arrive_expect_tx(a_full, C::a_bytes);
#pragma unroll
          for (int kb = 0; kb < KB; ++kb) {
            ptx::tma_load_2d(sA + (0 * KB + kb) * kTileBytes, &tmA_hi, a_full, kb * 64, static_cast<int32_t>(item.a_row0));
            if (NA == 2)
              ptx::tma_load_2d(sA + (1 * KB + kb) * kTileBytes, &tmA_lo, a_full, kb * 64, static_cast<int32_t>(item.a_row0));
          }
        }
        a_phase ^= 1;
      }
      for (uint32_t t = 0; t < item.n_tiles; ++t) {
        const int32_t brow = static_cast<int32_t>(item.b_row0 + t * 128);
#pragma unroll
        for (int kb = 0; kb < nkb; ++kb) {
          ptx::mbar_wait(&empty[stage], phase ^ 1);
          if (ptx::elect_one()) {
            ptx::mbar_arrive_expect_tx(&full[stage], C::x_off + (kb == 0 ? kExtBytes : 0));
            uint8_t* dst = sB + stage * C::stage_bytes;
            if constexpr (C::streamed) {
              ptx::tma_load_2d(dst, &tmA_hi, &full[stage], kb * 64, static_cast<int32_t>(item.a_row0));
              if (NA == 2) ptx::tma_load_2d(dst + kTileBytes, &tmA_lo, &full[stage], kb * 64, static_cast<int32_t>(item.a_row0));
            }
            ptx::tma_load_2d(dst + C::b_off, &tmB_hi, &full[stage], kb * 64, brow);
            if (NB == 2) ptx::tma_load_2d(dst + C::b_off + kTileBytes, &tmB_lo, &full[stage], kb * 64, brow);
            if (kb == 0) ptx::tma_load_2d(dst + C::x_off, &tmB_x, &full[stage], 0, brow);
          }
          if (++stage == C::stages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer (whole warp loops, lane 0 issues)
    constexpr uint32_t idesc = ptx::make_idesc_bf16(128, 128);
    const uint32_t a_lo0   = ptx::smem_desc_lo(ptx::smem_u32(sA));
    const uint32_t b_lo0   = ptx::smem_desc_lo(ptx::smem_u32(sB));
    const uint32_t ones_lo = ptx::smem_desc_lo(ptx::smem_u32(sOnes));
    uint32_t stage = 0, phase = 0, acc = 0, acc_phase = 0, a_phase = 0, ss = 0, sp = 0;
    uint32_t b_lo = b_lo0;  // descriptor low word of the current B stage
    for (;;) {
      ptx::mbar_wait(&s_full[ss], sp);
      const int it = __shfl_sync(0xffffffffu, s_item[ss], 0);  // (also: every lane has read the slot before it is handed back)
      if (lane == 0) ptx::mbar_arrive(&s_empty[ss]);
      if (++ss == kSched) { ss = 0; sp ^= 1; }
      if (it < 0) break;
      const uint32_t n_tiles = __shfl_sync(0xffffffffu, items[it].n_tiles, 0);
      if constexpr (!C::streamed) {
        ptx::mbar_wait(a_full, a_phase);
        ptx::tc_fence_after_sync();
      }
      for (uint32_t t = 0; t < n_tiles; ++t) {
        ptx::mbar_wait(&tempty[acc], acc_phase ^ 1);
        ptx::tc_fence_after_sync();
        const uint32_t d_tmem = tmem_base + acc * 128;
#pragma unroll
        for (int kb = 0; kb < nkb; ++kb) {
          ptx::mbar_wait(&full[stage], phase);
          ptx::tc_fence_after_sync();
          if (ptx::elect_one()) {
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              // +2 per K = 16 step (32 bytes >> 4).  Resident A: k-block kb / plane p sit (p * KB + kb) * 1024 further
              // (16 KB >> 4).  Streamed A: the planes lead the stage, the B planes follow at b_off.
              const uint32_t ah = (C::streamed ? b_lo : a_lo0 + (0 * KB + kb) * 1024) + k * 2;
              const uint32_t bh = b_lo + (C::b_off >> 4) + k * 2;
              ptx::mma_bf16_ss_lohi(d_tmem, ah, ptx::kDescHiSw128, bh, ptx::kDescHiSw128, idesc, (kb | k) != 0 ? 1u : 0u);
              if (NA == 2) {
                const uint32_t al = (C::streamed ? b_lo + 1024 : a_lo0 + (1 * KB + kb) * 1024) + k * 2;
                ptx::mma_bf16_ss_lohi(d_tmem, al, ptx::kDescHiSw128, bh, ptx::kDescHiSw128, idesc, 1u);
              }
              if (NB == 2) {
                const uint32_t bl = bh + 1024;
                ptx::mma_bf16_ss_lohi(d_tmem, ah, ptx::kDescHiSw128, bl, ptx::kDescHiSw128, idesc, 1u);
              }
            }
            if (kb == 0)  // -= |x|^2/2
              ptx::mma_bf16_ss_lohi(d_tmem, ones_lo, ptx::kDescHiSw32, b_lo + (C::x_off >> 4), ptx::kDescHiSw32, idesc, 1u);
            ptx::mma_commit(&empty[stage]);  // frees the B stage once these MMAs have read it
          }
          b_lo += C::stage_bytes >> 4;
          if (++stage == C::stages) { stage = 0; phase ^= 1; b_lo = b_lo0; }
        }
        if (ptx::elect_one()) ptx::mma_commit(&tfull[acc]);  // accumulator complete -> epilogue
        if (++acc == kAccBufs) { acc = 0; acc_phase ^= 1; }
      }
      if constexpr (!C::streamed) {
        if (ptx::elect_one()) ptx::mma_commit(a_empty);  // all MMAs reading this A tile are done
        a_phase ^= 1;
      }
    }
  } else {
    // ------------------------------------------------------------------ epilogue (8 warps, 1 row x 64 columns per thread)
    const int quarter = warp & 3;             // TMEM lanes [32*quarter, 32*quarter+32) belong to this warp
    const int row     = quarter * 32 + lane;  // accumulator row == query row within the tile
    const int half    = (warp - 2) >> 2;      // which 64-column half of the tile
    const int et      = half * 128 + row;     // slot in the queue arrays
    const int col0    = half * kCols;
    const uint32_t t_lane = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) + col0;
    uint32_t acc = 0, acc_phase = 0, ss = 0, sp = 0;
    auto next_item = [&]() {
      ptx::mbar_wait(&s_full[ss], sp);
      const int it = s_item[ss];
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(&s_empty[ss]);
      if (++ss == kSched) { ss = 0; sp ^= 1; }
      return it;
    };

    // One tile: wait for the accumulator, pull this thread's 64 columns into registers, hand the TMEM buffer back.
    auto fetch_tile = [&](uint32_t (&v0)[32], uint32_t (&v1)[32]) {
      ptx::mbar_wait(&tfull[acc], acc_phase);
      ptx::tc_fence_after_sync();
      ptx::tmem_ld_32x32(t_lane + acc * 128, v0);
      ptx::tmem_ld_32x32(t_lane + acc * 128 + 32, v1);
      ptx::tmem_ld_wait();
      ptx::tc_fence_before_sync();
      // one arrival per warp: 256 per-thread arrivals on one mbarrier serialise (~1000+ cycles per tile, more than a
      // one-pass tile's MMAs)
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(&tempty[acc]);
      if (++acc == kAccBufs) { acc = 0; acc_phase ^= 1; }
    };

    if constexpr (KC == 0) {
      for (int it = next_item(); it >= 0; it = next_item()) {
        const tc_item item = items[it];
        float* orow        = out_score + item.out_off + static_cast<int64_t>(row) * out_row_stride + col0;
        const bool live    = static_cast<uint32_t>(row) < item.valid_rows;
        for (uint32_t t = 0; t < item.n_tiles; ++t) {
          uint32_t v0[32], v1[32];
          fetch_tile(v0, v1);
          if (live) {
            float4* o4 = reinterpret_cast<float4*>(orow + t * 128);
#pragma unroll
            for (int c4 = 0; c4 < 8; ++c4) {
              o4[c4]     = make_float4(-__uint_as_float(v0[c4 * 4 + 0]), -__uint_as_float(v0[c4 * 4 + 1]),
                                       -__uint_as_float(v0[c4 * 4 + 2]), -__uint_as_float(v0[c4 * 4 + 3]));
              o4[8 + c4] = make_float4(-__uint_as_float(v1[c4 * 4 + 0]), -__uint_as_float(v1[c4 * 4 + 1]),
                                       -__uint_as_float(v1[c4 * 4 + 2]), -__uint_as_float(v1[c4 * 4 + 3]));
            }
          }
        }
      }
    } else {
      // Fused top-KC over t = -(score): bigger is better.  Lists keep scores (ascending, best first).
      for (int it = next_item(); it >= 0; it = next_item()) {
        const tc_item item = items[it];
        float lv[KC > 0 ? KC : 1];
        uint32_t li[KC > 0 ? KC : 1];
#pragma unroll
        for (int j = 0; j < KC; ++j) { lv[j] = INFINITY; li[j] = 0xffffffffu; }
        // cross-item pruning bound of this row's query (see tc_bound)
        float thr0 = INFINITY, b_add = 0.f;
        int* b_key = nullptr;
        if (bound.keys != nullptr && static_cast<uint32_t>(row) < item.valid_rows) {
          const uint32_t arow = item.a_row0 + row;
          b_key               = bound.keys + (bound.idx ? bound.idx[arow] : arow);
          b_add               = bound.add ? bound.add[arow] : 0.f;
          const int kb        = *reinterpret_cast<volatile int*>(b_key);
          const float bv      = __int_as_float(kb >= 0 ? kb : kb ^ 0x7fffffff);
          thr0                = (bv - b_add) / bound.scale;
        }
        const bool live_row = static_cast<uint32_t>(row) < item.valid_rows;
        if (!live_row) thr0 = -INFINITY;  // rows past the item's queries never collect candidates
        float thr_t = -thr0;  // an element is a candidate iff t > thr_t
        int cnt     = 0;
        const int kth = (bound.kth > 0 && bound.kth < KC) ? bound.kth : KC;
        // lv[kth - 1] without a dynamically indexed (= local-memory) array: the list is sorted ascending
        auto kth_best = [&]() {
          float v = lv[0];
#pragma unroll
          for (int j = 1; j < KC; ++j) v = fmaxf(v, j < kth ? lv[j] : -INFINITY);
          return v;
        };

        auto flush = [&]() {
          for (int e = 0; e < cnt; ++e) {
            const uint2 en   = qe[e * kEpiThreads + et];
            const float s    = -__uint_as_float(en.x);
            const uint32_t p = en.y;
            if (s < lv[KC - 1]) {
#pragma unroll
              for (int j = KC - 1; j > 0; --j) {
                if (s < lv[j - 1]) { lv[j] = lv[j - 1]; li[j] = li[j - 1]; }
                else if (s < lv[j]) { lv[j] = s; li[j] = p; }
              }
              if (s < lv[0]) { lv[0] = s; li[0] = p; }
            }
          }
          cnt   = 0;
          thr_t = -fminf(thr0, kth_best());
        };

        // 32 accumulator columns: max-tree per quad, one compare for the whole chunk; hits are rare
        auto scan32 = [&](const uint32_t (&v)[32], uint32_t pos) {
          if (__any_sync(0xffffffffu, cnt > kQueue / 2)) flush();
          float qm[8];
#pragma unroll
          for (int qd = 0; qd < 8; ++qd)
            qm[qd] = fmaxf(fmaxf(__uint_as_float(v[qd * 4 + 0]), __uint_as_float(v[qd * 4 + 1])),
                           fmaxf(__uint_as_float(v[qd * 4 + 2]), __uint_as_float(v[qd * 4 + 3])));
          const float m = fmaxf(fmaxf(fmaxf(qm[0], qm[1]), fmaxf(qm[2], qm[3])), fmaxf(fmaxf(qm[4], qm[5]), fmaxf(qm[6], qm[7])));
          if (m > thr_t) {
            uint32_t pending = 0xffu;  // quads still to look at; a quad waits (and the lane flushes) when its queue is full
            do {
#pragma unroll
              for (int qd = 0; qd < 8; ++qd) {
                if ((pending >> qd) & 1u) {
                  if (!(qm[qd] > thr_t)) {
                    pending &= ~(1u << qd);
                  } else if (cnt <= kQueue - 4) {
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                      if (__uint_as_float(v[qd * 4 + e]) > thr_t) {
                        qe[cnt * kEpiThreads + et] = make_uint2(v[qd * 4 + e], pos + qd * 4 + e);
                        ++cnt;
                      }
                    }
                    pending &= ~(1u << qd);
                  }
                }
              }
              if (pending) flush();
            } while (pending);
          }
        };

        for (uint32_t t = 0; t < item.n_tiles; ++t) {
          uint32_t v0[32], v1[32];
          fetch_tile(v0, v1);
          const uint32_t pos0 = item.b_row0 + t * 128 + col0;
          scan32(v0, pos0);
          scan32(v1, pos0 + 32);
        }
        flush();
        const float my_kth = kth_best();
        if (b_key != nullptr && my_kth < INFINITY) {
          const float pub = __fmaf_rn(bound.scale, my_kth, b_add);  // same expression as the consumers of the bound
          const int kp    = __float_as_int(pub);
          atomicMin(b_key, kp >= 0 ? kp : kp ^ 0x7fffffff);
        }
        if (live_row && out_score != nullptr) {
          float* os    = out_score + item.out_off + static_cast<int64_t>(row) * out_row_stride + half * KC;
          uint32_t* op = out_pos + item.out_off + static_cast<int64_t>(row) * out_row_stride + half * KC;
#pragma unroll
          for (int j = 0; j < KC; ++j) { os[j] = lv[j]; op[j] = li[j]; }
        }
      }
    }
  }

  ptx::tc_fence_before_sync();
  __syncthreads();
  if (warp == 2) { ptx::tmem_dealloc<128 * kAccBufs>(tmem_base); }
}

// ------------------------------------------------------------------------------------ host side
using encode_fn_t = CUresult (*)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                 const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                 CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

encode_fn_t get_encode_fn()
{
  static encode_fn_t fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<encode_fn_t>(p);
  });
  B2_EXPECTS(fn != nullptr, "cuTensorMapEncodeTiled is not available from this driver");
  return fn;
}

CUtensorMap make_plane_map(const __nv_bfloat16* ptr, int64_t rows, int Kp)
{
  CUtensorMap m;
  cuuint64_t gdim[2]    = {static_cast<cuuint64_t>(Kp), static_cast<cuuint64_t>(rows)};
  cuuint64_t gstride[1] = {static_cast<cuuint64_t>(Kp) * sizeof(__nv_bfloat16)};
  cuuint32_t box[2]     = {64, 128};
  cuuint32_t estr[2]    = {1, 1};
  CUresult r = get_encode_fn()(&m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<__nv_bfloat16*>(ptr), gdim, gstride, box,
                               estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                               CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  B2_EXPECTS(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled failed with code %d (rows=%lld Kp=%d)", int(r), (long long)rows, Kp);
  return m;
}

// [rows, 16] bf16 half-norm extension plane, one 32-byte row per dataset row
CUtensorMap make_ext_map(const __nv_bfloat16* ptr, int64_t rows)
{
  CUtensorMap m;
  cuuint64_t gdim[2]    = {16, static_cast<cuuint64_t>(rows)};
  cuuint64_t gstride[1] = {16 * sizeof(__nv_bfloat16)};
  cuuint32_t box[2]     = {16, 128};
  cuuint32_t estr[2]    = {1, 1};
  CUresult r = get_encode_fn()(&m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<__nv_bfloat16*>(ptr), gdim, gstride, box,
                               estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_32B,
                               CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  B2_EXPECTS(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled (half-norm plane) failed with code %d (rows=%lld)", int(r), (long long)rows);
  return m;
}

template <int KB, int PASSES, int KC>
void launch(cudaStream_t stream, int sm_count, const CUtensorMap& a_hi, const CUtensorMap& a_lo, const CUtensorMap& b_hi,
            const CUtensorMap& b_lo, const CUtensorMap& b_x, const tc_item* items, int n_items, const int* n_items_dev,
            float* out_score, uint32_t* out_pos, int64_t out_row_stride, const tc_bound& bound, bool dynamic, int kblocks)
{
  auto kern = tc_scan_kernel<KB, PASSES, KC>;
  using C   = cfg<KB, PASSES>;
  static_assert(C::smem <= 227 * 1024, "tc_scan_kernel: shared memory budget exceeded");
  // per launch, not once: the attribute belongs to the current device's context, and one process may drive several GPUs
  // (cuvsMultiGpu*); the call costs about a microsecond
  B2_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(C::smem)));
  int grid = n_items < sm_count ? n_items : sm_count;
  dbuf<int> sched;  // the kernel's work-item counter
  if (dynamic) {
    sched.alloc(1, stream);
    B2_CUDA(cudaMemsetAsync(sched.data(), 0, sizeof(int), stream));
  }
  timed_section ts("tc_scan", stream);
  count_launch();
  kern<<<grid, C::threads, C::smem, stream>>>(a_hi, a_lo, b_hi, b_lo, b_x, items, n_items, n_items_dev, kblocks, sched.data(), out_score,
                                               out_pos, out_row_stride, bound);
  B2_CUDA(cudaGetLastError());
}

__global__ void split_planes_kernel(const float* __restrict__ x, int64_t n, int64_t ld, int d, int Kp,
                                    __nv_bfloat16* __restrict__ hi, __nv_bfloat16* __restrict__ lo, int64_t rows_pad,
                                    const float* __restrict__ row_scale)
{
  const int64_t total = rows_pad * (Kp / 2);
  for (int64_t t = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; t < total;
       t += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int64_t r = t / (Kp / 2);
    const int c     = static_cast<int>(t % (Kp / 2)) * 2;
    float v0 = 0.f, v1 = 0.f;
    if (r < n) {
      const float sc = row_scale ? row_scale[r] : 1.0f;
      if (c < d) v0 = x[r * ld + c] * sc;
      if (c + 1 < d) v1 = x[r * ld + c + 1] * sc;
    }
    const __nv_bfloat16 h0 = __float2bfloat16_rn(v0), h1 = __float2bfloat16_rn(v1);
    reinterpret_cast<__nv_bfloat162*>(hi)[t] = __nv_bfloat162(h0, h1);
    if (lo) {
      const __nv_bfloat16 l0 = __float2bfloat16_rn(v0 - __bfloat162float(h0));
      const __nv_bfloat16 l1 = __float2bfloat16_rn(v1 - __bfloat162float(h1));
      reinterpret_cast<__nv_bfloat162*>(lo)[t] = __nv_bfloat162(l0, l1);
    }
  }
}

// -hn as three bf16 pieces (exact: 3 x 8 significand bits) in columns 0..2 of a 16-wide row; +inf (padding) -> -inf
__device__ __forceinline__ void store_ext_row(__nv_bfloat16* row, float hn)
{
  const float h = -hn;
  __nv_bfloat16 p0, p1, p2;
  if (isinf(h)) {
    p0 = __float2bfloat16_rn(h);
    p1 = p2 = __float2bfloat16_rn(0.f);
  } else {
    p0             = __float2bfloat16_rn(h);
    const float r1 = h - __bfloat162float(p0);
    p1             = __float2bfloat16_rn(r1);
    const float r2 = r1 - __bfloat162float(p1);
    p2             = __float2bfloat16_rn(r2);
  }
  const __nv_bfloat16 z = __float2bfloat16_rn(0.f);
  uint4 w0, w1 = make_uint4(0, 0, 0, 0);
  __nv_bfloat162 a(p0, p1), b(p2, z);
  w0.x = *reinterpret_cast<uint32_t*>(&a);
  w0.y = *reinterpret_cast<uint32_t*>(&b);
  w0.z = w0.w = 0;
  reinterpret_cast<uint4*>(row)[0] = w0;
  reinterpret_cast<uint4*>(row)[1] = w1;
}

__global__ void half_norms_kernel(const float* __restrict__ xn, int64_t n, int64_t rows_pad, __nv_bfloat16* __restrict__ hx)
{
  int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  if (i >= rows_pad) return;
  store_ext_row(hx + i * 16, i < n ? (xn ? 0.5f * xn[i] : 0.0f) : INFINITY);
}

__global__ void pack_half_norms_kernel(const float* __restrict__ hn, int64_t rows_pad, __nv_bfloat16* __restrict__ hx)
{
  int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  if (i >= rows_pad) return;
  store_ext_row(hx + i * 16, hn[i]);
}

}  // namespace

int tc_lists_per_item() { return 2; }

bool tc_supported(int device, int d)
{
  int major = 0;
  if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, device) != cudaSuccess) return false;
  return major == 10 && d >= 1 && tc_pad_k(d) <= kTcMaxK;
}

void tc_split_planes(cudaStream_t stream, const float* x, int64_t n, int64_t ld, int d, int Kp, __nv_bfloat16* hi,
                     __nv_bfloat16* lo, int64_t rows_pad, const float* row_scale)
{
  if (rows_pad == 0) return;
  int64_t total = rows_pad * (Kp / 2);
  int blocks    = static_cast<int>(std::min<int64_t>((total + 255) / 256, 148 * 16));
  count_launch();
  split_planes_kernel<<<blocks, 256, 0, stream>>>(x, n, ld, d, Kp, hi, lo, rows_pad, row_scale);
  B2_CUDA(cudaGetLastError());
}

void tc_half_norms(cudaStream_t stream, const float* xn, int64_t n, int64_t rows_pad, __nv_bfloat16* hx)
{
  if (rows_pad == 0) return;
  count_launch();
  half_norms_kernel<<<static_cast<unsigned>((rows_pad + 255) / 256), 256, 0, stream>>>(xn, n, rows_pad, hx);
  B2_CUDA(cudaGetLastError());
}

void tc_pack_half_norms(cudaStream_t stream, const float* hn, int64_t rows_pad, __nv_bfloat16* hx)
{
  if (rows_pad == 0) return;
  count_launch();
  pack_half_norms_kernel<<<static_cast<unsigned>((rows_pad + 255) / 256), 256, 0, stream>>>(hn, rows_pad, hx);
  B2_CUDA(cudaGetLastError());
}

void tc_scan_topk(cudaStream_t stream, int device, const __nv_bfloat16* a_hi, const __nv_bfloat16* a_lo,
                  int64_t a_rows_pad, const __nv_bfloat16* b_hi, const __nv_bfloat16* b_lo, int64_t b_rows_pad, int Kp,
                  const __nv_bfloat16* hx, const tc_item* items_dev, int n_items, const int* n_items_dev, int KC, int passes,
                  float* out_score, uint32_t* out_pos, int64_t out_row_stride, const tc_bound* bound, bool dynamic_schedule)
{
  if (n_items == 0) return;  // n_items is the host-side upper bound (grid sizing); *n_items_dev, when given, is the exact count
  B2_EXPECTS(Kp >= 64 && Kp % 64 == 0 && Kp <= kTcMaxK, "tc_scan_topk: padded K must be a multiple of 64 up to %d (got %d)", kTcMaxK, Kp);
  B2_EXPECTS(KC == 0 || KC == 16 || KC == 32, "tc_scan_topk: KC must be 0 (store), 16 or 32");
  B2_EXPECTS(passes >= 1 && passes <= 3, "tc_scan_topk: passes must be 1, 2 or 3");
  B2_EXPECTS(passes == 1 || a_lo, "tc_scan_topk: the A lo plane is required for 2- and 3-pass mode");
  B2_EXPECTS(passes != 3 || b_lo, "tc_scan_topk: the B lo plane is required for 3-pass mode");
  const int sms = sm_count_of(device);
  const tc_bound bnd = bound ? *bound : tc_bound{};
  CUtensorMap mA  = make_plane_map(a_hi, a_rows_pad, Kp);
  CUtensorMap mB  = make_plane_map(b_hi, b_rows_pad, Kp);
  CUtensorMap mAl = passes >= 2 ? make_plane_map(a_lo, a_rows_pad, Kp) : mA;
  CUtensorMap mBl = passes == 3 ? make_plane_map(b_lo, b_rows_pad, Kp) : mB;
  CUtensorMap mBx = make_ext_map(hx, b_rows_pad);
  const int kb_case = Kp <= 128 ? Kp / 64 : 0;  // 0 = streamed A (any K)
#define B2_TC_CASE(KB_, P_, KC_)                                                                                       \
  if (kb_case == KB_ && passes == P_ && KC == KC_)                                                                     \
    return launch<KB_, P_, KC_>(stream, sms, mA, mAl, mB, mBl, mBx, items_dev, n_items, n_items_dev, out_score, out_pos, out_row_stride, bnd, dynamic_schedule, Kp / 64);
  B2_TC_CASE(1, 1, 16) B2_TC_CASE(1, 1, 32) B2_TC_CASE(1, 3, 16) B2_TC_CASE(1, 3, 32) B2_TC_CASE(1, 1, 0) B2_TC_CASE(1, 3, 0)
  B2_TC_CASE(2, 1, 16) B2_TC_CASE(2, 1, 32) B2_TC_CASE(2, 3, 16) B2_TC_CASE(2, 3, 32) B2_TC_CASE(2, 1, 0) B2_TC_CASE(2, 3, 0)
  B2_TC_CASE(1, 2, 16) B2_TC_CASE(1, 2, 32) B2_TC_CASE(2, 2, 16) B2_TC_CASE(2, 2, 32)
  B2_TC_CASE(0, 1, 16) B2_TC_CASE(0, 1, 32) B2_TC_CASE(0, 1, 0) B2_TC_CASE(0, 2, 16) B2_TC_CASE(0, 2, 32)
  B2_TC_CASE(0, 3, 16) B2_TC_CASE(0, 3, 32) B2_TC_CASE(0, 3, 0)
#undef B2_TC_CASE
  B2_FAIL("tc_scan_topk: no kernel for Kp=%d passes=%d KC=%d", Kp, passes, KC);
}

}  // namespace b200
