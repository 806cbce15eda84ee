// IVF-PQ fine scan for sm_100a: PQ codes streamed from HBM, decoded on the SM, contracted on tcgen05, top-k' filtered
// against per-query thresholds.
//
// Replaces   cpp/src/neighbors/ivf_pq/detail/jit_lto_kernels/compute_similarity_impl.cuh:77-173
//            (+ create_lut_impl.cuh:16-79, compute_score_impl.cuh:53-79, compute_distances_impl.cuh:58-100)
// Reference formulation: one CTA per (query, probe); LUT[pq_dim][256] in shared memory; every (query, row, subspace)
// costs one shared-memory gather; the list's codes are re-read from L2/HBM by every probing query.
// Here: work item = (list, <= NQ probing queries).  Per 128-row tile of the list
//
//   warp 0      producer   one cp.async.bulk of the tile's block of the code stream (128 * pq_dim code bytes in "lane-
//                          transposed" order + 128 half-norms = 8.7 KB at pq_dim 64) into a 2..7-deep mbarrier ring;
//                          per item one TMA box with the NQ residual rows (bf16, SWIZZLE_128B)
//   warps 2-9   decode     lane l owns subspaces l and l+32: its 16 code bytes per 16 rows arrive with one 128-bit
//                          shared load; codebook words sit at [half][code][lane] (bank == lane), so a row's 64 entries are
//                          fetched with two conflict-free LDS.32 per lane and written with two STS.32 into the 128-byte-
//                          swizzled K-major operand tile (bf16 row = 256 B).  4.5 shared-memory wavefronts per row.
//   warp 1      MMA        D[128 rows x NQ queries] (+)= Y_tile . R^T : tcgen05.mma kind::f16, M = 128 (rows), N = NQ, 8 K-steps
//                          + 1 step that adds -|y|^2/2 (three bf16 pieces x ones); accumulators in a 4-deep TMEM ring
//   warps 10-17 epilogue   thread = row, columns = queries: tcgen05.ld 32 columns, compare against the queries' running
//                          thresholds (shared memory), push the rare hits into per-query candidate buffers; a buffer that
//                          overflows is compacted to its KC best by one warp (rank by counting) and the threshold
//                          tightened; one named barrier per round of acc/2 tiles.
//
// With few probing queries per list (100M rows / 16k lists / 10k-query batches: ~30) the accumulator is 128 x 32..64
// instead of the 128 x 128 of the query-major kernel (scan_tc.cu), the rows fill the MMA's M side completely, and HBM
// traffic per row is pq_dim + 4 bytes instead of a 2 * rot_dim + 32 byte decoded row.
#include "common.hpp"
#include "ptx_sm100.cuh"
#include "scan_pq.cuh"
#include "timing.hpp"

#include <cuda.h>

#include <cmath>
#include <mutex>

namespace b200 {
namespace {

constexpr int kDecWarps   = 8;
constexpr int kEpiWarps   = 8;  // two per TMEM lane quarter: they split the (tile, chunk) units of a round
constexpr int kEpiThreads = 32 * kEpiWarps;
constexpr int kThreads    = 64 + 32 * kDecWarps + kEpiThreads;  // 576
constexpr int kEpiWarp0   = 2 + kDecWarps;                      // first epilogue warp (10: warp & 3 covers all TMEM quarters)
constexpr int kDecStages  = 2;
constexpr int kMaxAcc     = 8;   // TMEM accumulator ring: min(8, 512 / NQ) buffers of NQ columns
constexpr int kSched      = 4;   // work-item ring
constexpr int kMaxCStages = 8;
constexpr int kDecTile    = 128 * 128;  // one k-block of the decoded tile: 128 rows x 64 bf16, SWIZZLE_128B
constexpr int kExtTile    = 128 * 32;   // half-norm K extension: 128 rows x 16 bf16
constexpr int kSmemLimit  = 227 * 1024;

struct pq_args {
  const uint8_t* stream;
  const uint32_t* cb_words;
  const tc_item* items;
  const int* n_items_dev;
  int* sched;
  float* out_score;
  uint32_t* out_pos;
  int64_t out_row_stride;
  int* b_keys;
  const uint32_t* b_idx;
  const float* b_add;
  float b_scale;
  int kth;
  int n_items_host;
  int KC;
  int cap;      // candidate buffer entries per query (KC < cap <= 128)
  int cstages;  // code ring depth
  int blk;      // bytes of one tile block of the stream
};

__device__ __forceinline__ bool bar_red_or(uint32_t id, uint32_t nthreads, bool pred)
{
  uint32_t r;
  asm volatile(
    "{\n\t"
    ".reg .pred pi, po;\n\t"
    "setp.ne.u32 pi, %1, 0;\n\t"
    "bar.red.or.pred po, %2, %3, pi;\n\t"
    "selp.u32 %0, 1, 0, po;\n\t"
    "}\n"
    : "=r"(r)
    : "r"(static_cast<uint32_t>(pred)), "r"(id), "r"(nthreads)
    : "memory");
  return r != 0;
}

// monotone float -> uint32 (bigger float = bigger key); never 0 for a real float
__device__ __forceinline__ uint32_t okey(uint32_t fbits) { return (fbits & 0x80000000u) ? ~fbits : (fbits | 0x80000000u); }
__device__ __forceinline__ uint32_t okey_inv(uint32_t k) { return (k & 0x80000000u) ? (k & 0x7fffffffu) : ~k; }

// One chunk of one tile in the epilogue: this thread's row against 32 query columns.  taddr = TMEM address of the chunk,
// thr / cnt / cand point at the chunk's first column.  Returns the columns whose candidate could not be stored (buffer full).
// Deliberately NOT inlined: it is called from 2 x (tiles per round) x (chunks per warp) sites and, inlined, the kernel grew to
// 230 KB of SASS — the warps of the four roles then thrash the instruction cache (stall_no_inst was the top stall reason).
__device__ __noinline__ uint32_t pq_filter_chunk(uint32_t taddr, uint32_t pos, const float* __restrict__ thr, int* cnt,
                                                 unsigned long long* cand, int cap, uint32_t only)
{
  uint32_t v[32];
  ptx::tmem_ld_32x32(taddr, v);
  ptx::tmem_ld_wait();
  const float4* th4 = reinterpret_cast<const float4*>(thr);
  float d[32];  // margin over the column's threshold: a candidate iff d > 0 (exact: the difference of two floats keeps its sign)
#pragma unroll
  for (int j4 = 0; j4 < 8; ++j4) {
    const float4 x = th4[j4];
    d[4 * j4]     = __uint_as_float(v[4 * j4]) - x.x;
    d[4 * j4 + 1] = __uint_as_float(v[4 * j4 + 1]) - x.y;
    d[4 * j4 + 2] = __uint_as_float(v[4 * j4 + 2]) - x.z;
    d[4 * j4 + 3] = __uint_as_float(v[4 * j4 + 3]) - x.w;
  }
  float q[4];  // per group of 8 columns
#pragma unroll
  for (int g = 0; g < 4; ++g)
    q[g] = fmaxf(fmaxf(fmaxf(d[8 * g], d[8 * g + 1]), fmaxf(d[8 * g + 2], d[8 * g + 3])),
                 fmaxf(fmaxf(d[8 * g + 4], d[8 * g + 5]), fmaxf(d[8 * g + 6], d[8 * g + 7])));
  const float m = fmaxf(fmaxf(q[0], q[1]), fmaxf(q[2], q[3]));
  uint32_t left = 0;
  if (m > 0.f) {
    // rare per thread, but with 1024 scores per warp and chunk some lane is here about every other chunk: keep it short —
    // only the 8-column groups that hold a hit are looked at
#pragma unroll
    for (int g = 0; g < 4; ++g) {
      if (q[g] > 0.f) {
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          const int j = 8 * g + e;
          if (d[j] > 0.f && ((only >> j) & 1u)) {
            const int at = atomicAdd(&cnt[j], 1);
            if (at < cap) cand[j * cap + at] = (static_cast<unsigned long long>(okey(v[j])) << 32) | (~pos);
            else left |= 1u << j;
          }
        }
      }
    }
  }
  return left;
}

__device__ __forceinline__ float fmax3(float a, float b, float c)
{
  float r;
  asm("max.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(a), "f"(b), "f"(c));  // FMNMX3 (sm_100): NaN operands are ignored like fmaxf
  return r;
}

// One 32-column chunk of up to four tiles of an epilogue round: the chunk's 32 thresholds are loaded ONCE (they were 16 % of the
// kernel's shared-memory wavefronts when re-read per tile) and stay in registers while the tiles' accumulators stream through.
// taddr = TMEM address of the chunk in accumulator buffer 0; tile b of the round sits in buffer (buf0 + b) % nacc (nq columns
// per buffer) and is waited for here (t_full, parity aph, flipped where the buffer index wraps); mask = tiles of the round this
// warp owns (warp-uniform: tcgen05.ld is .sync.aligned).  Returns, per tile, the columns whose candidate could not be stored.
__device__ __forceinline__ uint4 pq_filter_round(uint32_t taddr, uint32_t buf0, uint32_t nacc, uint32_t nq, uint32_t mask, uint32_t pos0,
                                              const float* __restrict__ thr, int* cnt, unsigned long long* cand, int cap,
                                              uint64_t* t_full, uint32_t aph)
{
  float th[32];
  {
    const float4* th4 = reinterpret_cast<const float4*>(thr);
#pragma unroll
    for (int j4 = 0; j4 < 8; ++j4) {
      const float4 x = th4[j4];
      th[4 * j4] = x.x; th[4 * j4 + 1] = x.y; th[4 * j4 + 2] = x.z; th[4 * j4 + 3] = x.w;
    }
  }
  uint32_t l0 = 0, l1 = 0, l2 = 0, l3 = 0;
#pragma unroll 1
  for (uint32_t b = 0; b < 4; ++b) {
    if (!((mask >> b) & 1u)) continue;
    uint32_t ab = buf0 + b, par = aph;
    if (ab >= nacc) { ab -= nacc; par ^= 1u; }
    ptx::mbar_wait(&t_full[ab], par);
    ptx::tc_fence_after_sync();
    uint32_t v[32];
    ptx::tmem_ld_32x32(taddr + ab * nq, v);
    ptx::tmem_ld_wait();
    float q[4];
#pragma unroll
    for (int g = 0; g < 4; ++g) {
      float m = fmax3(__uint_as_float(v[8 * g]) - th[8 * g], __uint_as_float(v[8 * g + 1]) - th[8 * g + 1], __uint_as_float(v[8 * g + 2]) - th[8 * g + 2]);
      m       = fmax3(m, __uint_as_float(v[8 * g + 3]) - th[8 * g + 3], __uint_as_float(v[8 * g + 4]) - th[8 * g + 4]);
      m       = fmax3(m, __uint_as_float(v[8 * g + 5]) - th[8 * g + 5], __uint_as_float(v[8 * g + 6]) - th[8 * g + 6]);
      q[g]    = fmaxf(m, __uint_as_float(v[8 * g + 7]) - th[8 * g + 7]);
    }
    uint32_t lf = 0;
    if (fmaxf(fmax3(q[0], q[1], q[2]), q[3]) > 0.f) {
      const uint32_t pos = pos0 + b * 128u;
#pragma unroll
      for (int g = 0; g < 4; ++g) {
        if (q[g] > 0.f) {
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            const int j = 8 * g + e;
            if (__uint_as_float(v[j]) - th[j] > 0.f) {
              const int at = atomicAdd(&cnt[j], 1);
              if (at < cap) cand[j * cap + at] = (static_cast<unsigned long long>(okey(v[j])) << 32) | (~pos);
              else lf |= 1u << j;
            }
          }
        }
      }
    }
    __syncwarp();
    if (b == 0) l0 = lf;
    else if (b == 1) l1 = lf;
    else if (b == 2) l2 = lf;
    else l3 = lf;
  }
  return make_uint4(l0, l1, l2, l3);
}

// Selection inside one column's buffer by one warp, rank by counting: lane l holds entries l, l + 32, l + 64, l + 96 (64-bit keys
// order(t) << 32 | ~pos, unique, 0 = none; n <= 128); every entry is broadcast from shared memory and each lane counts how
// many beat its own.  rank 0 = best.  No dependent chain: n iterations of one LDS.64 + four compare-adds.
__device__ __forceinline__ void pq_rank_select(const unsigned long long* buf, int n, int lane, unsigned long long (&k)[4], int (&r)[4])
{
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    k[e] = lane + 32 * e < n ? buf[lane + 32 * e] : 0ull;
    r[e] = 0;
  }
  if (n <= 64) {  // (warp-uniform) the common case: buffers of <= 64 entries
#pragma unroll 4
    for (int i = 0; i < n; ++i) {
      const unsigned long long ki = buf[i];
      r[0] += ki > k[0] ? 1 : 0;
      r[1] += ki > k[1] ? 1 : 0;
    }
  } else {
#pragma unroll 2
    for (int i = 0; i < n; ++i) {
      const unsigned long long ki = buf[i];
#pragma unroll
      for (int e = 0; e < 4; ++e) r[e] += ki > k[e] ? 1 : 0;
    }
  }
}

template <int NQ, int NKB, int PASSES>
struct layout {
  static constexpr int q_tile     = NQ * 128;                       // one k-block of the residual rows
  static constexpr int q_bytes    = PASSES * NKB * q_tile;
  static constexpr int dec_stage  = NKB * kDecTile + kExtTile;
  static constexpr int ones_bytes = NQ * 32;
  static constexpr int cb_bytes   = NKB * 32768;
  static constexpr int off_q      = 0;
  static constexpr int off_dec    = off_q + q_bytes;
  static constexpr int off_ones   = off_dec + kDecStages * dec_stage;
  static constexpr int off_cb     = off_ones + ones_bytes;
  static constexpr int off_thr    = off_cb + cb_bytes;
  static constexpr int off_cnt    = off_thr + NQ * 4;
  static constexpr int off_bars   = off_cnt + NQ * 4;
  static constexpr int acc        = 512 / NQ < kMaxAcc ? 512 / NQ : kMaxAcc;  // accumulator buffers
  static constexpr int tb         = acc / 2;                                   // tiles per epilogue round (one barrier per round)
  static constexpr int n_bars     = 2 * kMaxCStages + 2 * kDecStages + 2 + 2 * kMaxAcc + 2 * kSched;
  static constexpr int off_item   = off_bars + n_bars * 8;
  static constexpr int off_tmem   = off_item + kSched * 4;
  static constexpr int off_cand   = (off_tmem + 4 + 15) / 16 * 16;   // [NQ][cap] uint2, then the code ring
  static constexpr int tmem_cols  = acc * NQ;
  static_assert(q_tile % 1024 == 0 && dec_stage % 1024 == 0, "operand tiles need 1024-byte alignment");
};

template <int NQ, int NKB, int PASSES>
__global__ void __launch_bounds__(kThreads, 1)
pq_stream_scan_kernel(const __grid_constant__ CUtensorMap tmQ_hi, const __grid_constant__ CUtensorMap tmQ_lo, const pq_args P)
{
  using L = layout<NQ, NKB, PASSES>;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  if (threadIdx.x == 0 && (ptx::smem_u32(smem_raw) & 1023u) != 0) __trap();
  uint8_t* sQ     = smem_raw + L::off_q;
  uint8_t* sDec   = smem_raw + L::off_dec;
  uint8_t* sOnes  = smem_raw + L::off_ones;
  uint32_t* sCb   = reinterpret_cast<uint32_t*>(smem_raw + L::off_cb);
  float* sThr     = reinterpret_cast<float*>(smem_raw + L::off_thr);
  int* sCnt       = reinterpret_cast<int*>(smem_raw + L::off_cnt);
  uint64_t* bars  = reinterpret_cast<uint64_t*>(smem_raw + L::off_bars);
  uint64_t* c_full  = bars;
  uint64_t* c_empty = c_full + kMaxCStages;
  uint64_t* d_full  = c_empty + kMaxCStages;
  uint64_t* d_empty = d_full + kDecStages;
  uint64_t* q_full  = d_empty + kDecStages;
  uint64_t* q_empty = q_full + 1;
  uint64_t* t_full  = q_empty + 1;
  uint64_t* t_empty = t_full + kMaxAcc;
  uint64_t* s_full  = t_empty + kMaxAcc;
  uint64_t* s_empty = s_full + kSched;
  int* s_item       = reinterpret_cast<int*>(smem_raw + L::off_item);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem_raw + L::off_tmem);
  unsigned long long* sCand = reinterpret_cast<unsigned long long*>(smem_raw + L::off_cand);  // okey(t) << 32 | ~pos
  uint8_t* sCode  = smem_raw + L::off_cand + NQ * P.cap * 8;

  const int warp = __shfl_sync(0xffffffffu, static_cast<int>(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
  const int n_items = P.n_items_dev ? *P.n_items_dev : P.n_items_host;
  const uint32_t ncs = static_cast<uint32_t>(P.cstages);

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tmap(&tmQ_hi);
    if (PASSES == 2) ptx::prefetch_tmap(&tmQ_lo);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < kMaxCStages; ++s) {
      ptx::mbar_init(&c_full[s], 1);
      ptx::mbar_init(&c_empty[s], kDecWarps);
    }
    for (int s = 0; s < kDecStages; ++s) {
      ptx::mbar_init(&d_full[s], kDecWarps);
      ptx::mbar_init(&d_empty[s], 1);
    }
    ptx::mbar_init(q_full, 1);
    ptx::mbar_init(q_empty, 1);
    for (int s = 0; s < kMaxAcc; ++s) {
      ptx::mbar_init(&t_full[s], 1);
      ptx::mbar_init(&t_empty[s], kEpiWarps);
    }
    for (int s = 0; s < kSched; ++s) {
      ptx::mbar_init(&s_full[s], 1);
      ptx::mbar_init(&s_empty[s], 1 + kDecWarps + kEpiWarps);
    }
    ptx::fence_barrier_init();
  }
  // codebook words -> shared memory ([half][code][lane]); the constant "ones" operand of the half-norm step: every row
  // {1, 1, 1, 0, 0, 0, 0, 0} in BOTH 16-byte chunks (identical chunks: invariant under the 32-byte swizzle)
  for (int i = threadIdx.x; i < L::cb_bytes / 16; i += kThreads)
    reinterpret_cast<uint4*>(sCb)[i] = reinterpret_cast<const uint4*>(P.cb_words)[i];
  for (int i = threadIdx.x; i < L::ones_bytes / 16; i += kThreads)
    reinterpret_cast<uint4*>(sOnes)[i] = make_uint4(0x3f803f80u, 0x00003f80u, 0u, 0u);
  ptx::fence_proxy_async();
  if (warp == 2) { ptx::tmem_alloc<L::tmem_cols>(tmem_slot); }
  ptx::tc_fence_before_sync();
  __syncthreads();
  ptx::tc_fence_after_sync();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0);

  if (warp == 0) {
    // ------------------------------------------------------------------ producer (whole warp loops, one elected lane issues)
    uint32_t cs = 0, cph = 0, qph = 0, ss = 0, sp = 0;
    for (;;) {
      ptx::mbar_wait(&s_empty[ss], sp ^ 1);
      int it = 0;
      if (lane == 0) {
        it = atomicAdd(P.sched, 1);
        if (it >= n_items) it = -1;
        s_item[ss] = it;
        ptx::mbar_arrive(&s_full[ss]);
      }
      it = __shfl_sync(0xffffffffu, it, 0);
      if (++ss == kSched) { ss = 0; sp ^= 1; }
      if (it < 0) break;
      tc_item item = P.items[it];
      item.a_row0  = __shfl_sync(0xffffffffu, item.a_row0, 0);
      item.b_row0  = __shfl_sync(0xffffffffu, item.b_row0, 0);
      item.n_tiles = __shfl_sync(0xffffffffu, item.n_tiles, 0);
      ptx::mbar_wait(q_empty, qph ^ 1);
      if (ptx::elect_one()) {
        ptx::mbar_arrive_expect_tx(q_full, L::q_bytes);
#pragma unroll
        for (int kb = 0; kb < NKB; ++kb) {
          ptx::tma_load_2d(sQ + kb * L::q_tile, &tmQ_hi, q_full, kb * 64, static_cast<int32_t>(item.a_row0));
          if (PASSES == 2) ptx::tma_load_2d(sQ + (NKB + kb) * L::q_tile, &tmQ_lo, q_full, kb * 64, static_cast<int32_t>(item.a_row0));
        }
      }
      qph ^= 1;
      const uint8_t* src = P.stream + static_cast<int64_t>(item.b_row0 >> 7) * P.blk;
      for (uint32_t t = 0; t < item.n_tiles; ++t) {
        ptx::mbar_wait(&c_empty[cs], cph ^ 1);
        if (ptx::elect_one()) {
          ptx::mbar_arrive_expect_tx(&c_full[cs], static_cast<uint32_t>(P.blk));
          ptx::bulk_load_1d(sCode + cs * P.blk, src + static_cast<int64_t>(t) * P.blk, static_cast<uint32_t>(P.blk), &c_full[cs]);
        }
        if (++cs == ncs) { cs = 0; cph ^= 1; }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer
    const uint32_t q_lo0   = ptx::smem_desc_lo(ptx::smem_u32(sQ));
    const uint32_t d_lo0   = ptx::smem_desc_lo(ptx::smem_u32(sDec));
    const uint32_t ones_lo = ptx::smem_desc_lo(ptx::smem_u32(sOnes));
    uint32_t ds = 0, dph = 0, acc = 0, aph = 0, qph = 0, ss = 0, sp = 0;
    for (;;) {
      ptx::mbar_wait(&s_full[ss], sp);
      const int it = __shfl_sync(0xffffffffu, s_item[ss], 0);  // (the shuffle consumes the load before the slot is handed back)
      if (lane == 0) ptx::mbar_arrive(&s_empty[ss]);
      if (++ss == kSched) { ss = 0; sp ^= 1; }
      if (it < 0) break;
      const uint32_t n_tiles = __shfl_sync(0xffffffffu, P.items[it].n_tiles, 0);
      // N of the MMA = the item's live queries rounded up to 16: a narrow item neither reads nor multiplies the unused rows
      const uint32_t n_live = min(static_cast<uint32_t>(NQ), (__shfl_sync(0xffffffffu, P.items[it].valid_rows, 0) + 15u) & ~15u);
      const uint32_t idesc  = ptx::make_idesc_bf16(128, static_cast<int>(max(n_live, 16u)));
      ptx::mbar_wait(q_full, qph);
      ptx::tc_fence_after_sync();
      for (uint32_t t = 0; t < n_tiles; ++t) {
        ptx::mbar_wait(&t_empty[acc], aph ^ 1);
        ptx::mbar_wait(&d_full[ds], dph);
        ptx::tc_fence_after_sync();
        if (ptx::elect_one()) {
          const uint32_t d_tmem = tmem_base + acc * NQ;
          const uint32_t a0     = d_lo0 + ds * (L::dec_stage >> 4);
#pragma unroll
          for (int kb = 0; kb < NKB; ++kb) {
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              const uint32_t a = a0 + kb * (kDecTile >> 4) + k * 2;  // decoded rows: the M side
              const uint32_t b = q_lo0 + kb * (L::q_tile >> 4) + k * 2;
              ptx::mma_bf16_ss_lohi(d_tmem, a, ptx::kDescHiSw128, b, ptx::kDescHiSw128, idesc, (kb | k) != 0 ? 1u : 0u);
              if (PASSES == 2)
                ptx::mma_bf16_ss_lohi(d_tmem, a, ptx::kDescHiSw128, b + NKB * (L::q_tile >> 4), ptx::kDescHiSw128, idesc, 1u);
            }
          }
          // -= |y|^2/2 : ext rows hold the three bf16 pieces of -hn/2 in both chunks, ones rows three 1s in both chunks
          ptx::mma_bf16_ss_lohi(d_tmem, a0 + NKB * (kDecTile >> 4), ptx::kDescHiSw32, ones_lo, ptx::kDescHiSw32, idesc, 1u);
          ptx::mma_commit(&d_empty[ds]);
          ptx::mma_commit(&t_full[acc]);
          // the item's residual rows may be replaced once its last MMAs have read them.  Committed by the SAME thread that
          // issued them: tcgen05.commit only tracks the executing thread's operations, and a second elect.sync is not
          // guaranteed to pick the same lane
          if (t + 1 == n_tiles) ptx::mma_commit(q_empty);
        }
        if (++ds == kDecStages) { ds = 0; dph ^= 1; }
        if (++acc == L::acc) { acc = 0; aph ^= 1; }
      }
      qph ^= 1;
    }
  } else if (warp < kEpiWarp0) {
    // ------------------------------------------------------------------ decode warps: 16 rows of every tile each
    const int dw = warp - 2;
    uint32_t offx[8];  // byte offset of this lane's word inside row x of an 8-row swizzle atom
#pragma unroll
    for (int x = 0; x < 8; ++x) offx[x] = x * 128 + ((((lane >> 2) ^ x) & 7) << 4) + ((lane & 3) << 2);
    const uint32_t cb_lane32 = ptx::smem_u32(sCb) + static_cast<uint32_t>(lane) * 4u;  // this lane's word of codebook row 0
    uint32_t cs = 0, cph = 0, ds = 0, dph = 0, ss = 0, sp = 0;
    for (;;) {
      ptx::mbar_wait(&s_full[ss], sp);
      const int it = __shfl_sync(0xffffffffu, s_item[ss], 0);  // (consumes the load before the slot is handed back)
      if (lane == 0) ptx::mbar_arrive(&s_empty[ss]);
      if (++ss == kSched) { ss = 0; sp ^= 1; }
      if (it < 0) break;
      const uint32_t n_tiles = P.items[it].n_tiles;
      for (uint32_t t = 0; t < n_tiles; ++t) {
        ptx::mbar_wait(&c_full[cs], cph);
        const uint8_t* cst = sCode + cs * P.blk;
        uint4 cw[NKB];
#pragma unroll
        for (int h = 0; h < NKB; ++h) cw[h] = *reinterpret_cast<const uint4*>(cst + dw * (NKB * 512) + h * 512 + lane * 16);
        const float hn = reinterpret_cast<const float*>(cst + NKB * 4096)[16 * dw + (lane >> 1)];
        // The ring slot is handed back only AFTER the decode below has consumed these registers.  An mbarrier arrive issued
        // right behind the loads does not wait for them: the arrive is not ordered behind outstanding LDS (the hardware only
        // scoreboards register USE), and under the tensor core's operand traffic a load can sit in the queue longer than the
        // producer needs to refill the slot from L2 — seen as one warp's 16 rows decoded from the codes of the tile that
        // occupies the slot next, with the half-norms (the tail of the block, written last) still the old ones.
        // compute-sanitizer racecheck flags exactly this pair.
        const uint32_t cs_read = cs;
        if (++cs == ncs) { cs = 0; cph ^= 1; }

        ptx::mbar_wait(&d_empty[ds], dph ^ 1);
        uint8_t* dst = sDec + ds * L::dec_stage + (2 * dw) * 1024;
#pragma unroll
        for (int h = 0; h < NKB; ++h) {
          const uint32_t w4[4] = {cw[h].x, cw[h].y, cw[h].z, cw[h].w};
          uint32_t val[16];
#pragma unroll
          for (int i = 0; i < 16; ++i) {
            // byte extract (PRMT) + scaled add (LEA) on a 32-bit shared address: 2 integer instructions per entry instead of
            // the shift / mask-or / add-base triple the generic-pointer form compiles to (A/B at 100M: 7.88 -> 7.60 ms per batch)
            const uint32_t c = __byte_perm(w4[i >> 2], 0u, 0x4440u | static_cast<uint32_t>(i & 3));
            asm("ld.shared.u32 %0, [%1];" : "=r"(val[i]) : "r"(cb_lane32 + static_cast<uint32_t>(h) * 32768u + (c << 7)));
          }
#pragma unroll
          for (int i = 0; i < 16; ++i)
            *reinterpret_cast<uint32_t*>(dst + h * kDecTile + (i >> 3) * 1024 + offx[i & 7]) = val[i];
        }
        {
          // -hn/2 as three bf16 pieces (exact), identical in both 16-byte chunks of the row; +inf (padding) -> -inf.
          // Lane l writes chunk l % 2 of row l / 2: the warp's 32 x 16 bytes are one contiguous 512-byte span, so every
          // quarter-warp of the 128-bit store covers 128 consecutive bytes = all 32 banks once (row-major lanes, l % 16 = row,
          // put lanes 0..7 at a 32-byte stride: a 2-way conflict on every store, 4 excess wavefronts per warp and tile in ncu)
          const float hh = -0.5f * hn;
          __nv_bfloat16 p0 = __float2bfloat16_rn(hh), p1 = __float2bfloat16_rn(0.f), p2 = p1;
          if (!isinf(hh)) {
            const float r1 = hh - __bfloat162float(p0);
            p1             = __float2bfloat16_rn(r1);
            p2             = __float2bfloat16_rn(r1 - __bfloat162float(p1));
          }
          const uint32_t w0 = static_cast<uint32_t>(__bfloat16_as_ushort(p0)) | (static_cast<uint32_t>(__bfloat16_as_ushort(p1)) << 16);
          const uint32_t w1 = static_cast<uint32_t>(__bfloat16_as_ushort(p2));
          *reinterpret_cast<uint4*>(sDec + ds * L::dec_stage + NKB * kDecTile + (16 * dw) * 32 + lane * 16) =
            make_uint4(w0, w1, 0u, 0u);
        }
        // every loaded register (codes of both halves, half-norm) has fed an issued instruction by now: release the slot
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive(&c_empty[cs_read]);
        ptx::fence_proxy_async();  // generic-proxy writes -> visible to the tensor core's async-proxy reads
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive(&d_full[ds]);
        if (++ds == kDecStages) { ds = 0; dph ^= 1; }
      }
    }
  } else {
    // ------------------------------------------------------------------ epilogue: thread = list row, columns = queries
    const int ew      = warp - kEpiWarp0;
    const int quarter = warp & 3;
    const int half    = ew >> 2;  // which of the lane quarter's two warps: they split the round's (tile, chunk) units
    const int row     = quarter * 32 + lane;
    const int te      = static_cast<int>(threadIdx.x) - 32 * kEpiWarp0;  // 0..127
    const uint32_t t_lane = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16);
    const int cap = P.cap, KC = P.KC;
    const int kth = (P.kth > 0 && P.kth < KC) ? P.kth : KC;
    constexpr int NCH = NQ / 32;
    uint32_t acc = 0, aph = 0, ss = 0, sp = 0;

    auto rank_select = [&](int col, unsigned long long (&k)[4], int (&r)[4]) -> int {
      const int n = min(sCnt[col], cap);
      pq_rank_select(sCand + col * cap, n, lane, k, r);
      return n;
    };
    // compaction: keep the KC best at the front, tighten the column's threshold to its kth best
    auto compact = [&](int col) {
      unsigned long long k[4];
      int r[4];
      const int n = rank_select(col, k, r);
      __syncwarp();
      unsigned long long* buf = sCand + col * cap;
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        if (k[e] != 0ull && r[e] < KC) buf[r[e]] = k[e];
        if (n >= kth && k[e] != 0ull && r[e] == kth - 1) sThr[col] = fmaxf(sThr[col], __uint_as_float(okey_inv(static_cast<uint32_t>(k[e] >> 32))));
      }
      if (lane == 0) sCnt[col] = min(n, KC);
      __syncwarp();
    };
    for (;;) {
      ptx::mbar_wait(&s_full[ss], sp);
      const int it = __shfl_sync(0xffffffffu, s_item[ss], 0);  // (consumes the load before the slot is handed back)
      if (lane == 0) ptx::mbar_arrive(&s_empty[ss]);
      if (++ss == kSched) { ss = 0; sp ^= 1; }
      if (it < 0) break;
      const tc_item item = P.items[it];
      // per-column state: running threshold in t = -(score) units (a row is a candidate iff t > thr), empty buffer
      for (int col = te; col < NQ; col += kEpiThreads) {
        float thr = INFINITY;  // columns past the item's queries never collect anything
        if (static_cast<uint32_t>(col) < item.valid_rows) {
          thr = -INFINITY;
          if (P.b_keys != nullptr) {
            const uint32_t arow = item.a_row0 + col;
            const int kb        = *reinterpret_cast<volatile int*>(P.b_keys + (P.b_idx ? P.b_idx[arow] : arow));
            const float bv      = __int_as_float(kb >= 0 ? kb : kb ^ 0x7fffffff);
            thr                 = -((bv - (P.b_add ? P.b_add[arow] : 0.f)) / P.b_scale);
          }
        }
        sThr[col] = thr;
        sCnt[col] = 0;
      }
      ptx::named_bar_sync(1, kEpiThreads);

      auto do_chunk = [&](uint32_t taddr, uint32_t pos, int c, uint32_t only) -> uint32_t {
        return pq_filter_chunk(taddr + c * 32, pos, sThr + c * 32, sCnt + c * 32, sCand + c * 32 * cap, cap, only);
      };
      constexpr int TB = L::tb;
      static_assert(TB <= 4, "pq_filter_round handles up to four tiles");
      // Work units of a round = (tile, chunk) for the chunks that hold queries; the two warps of a TMEM lane quarter split them:
      // by chunk when the item has an even number of live chunks, else in a checkerboard over (tile, chunk) — an item with
      // <= 32 probing queries (most items of a sparsely probed index) keeps BOTH warps busy on alternating tiles instead of
      // sending one of them through 32 columns of +inf thresholds.
      const int nvc = min(NCH, (static_cast<int>(item.valid_rows) + 31) >> 5);
      // rounds of TB tiles: all their accumulators are filtered, then ONE barrier decides whether any buffer overflowed
      for (uint32_t t0 = 0; t0 < item.n_tiles; t0 += TB) {
        const int nb = static_cast<int>(min(static_cast<uint32_t>(TB), item.n_tiles - t0));
        uint4 pend[NCH];  // per chunk: .x/.y/.z/.w = columns still pending in tile 0..3 of the round
        bool any_left = false;
#pragma unroll
        for (int c = 0; c < NCH; ++c) pend[c] = make_uint4(0u, 0u, 0u, 0u);
        const uint32_t live = (1u << nb) - 1u;
#pragma unroll 1  // ONE inlined copy of the round filter (its call overhead was ~15 % of the epilogue's instructions)
        for (int c = 0; c < nvc; ++c) {
          // tiles of the round whose (tile, c) unit is this warp's: all or none for an even chunk count, every other one else
          const uint32_t mask = live & ((nvc & 1) ? (0x55555555u << ((t0 + c + half) & 1u)) : ((c & 1) == half ? 0xffffffffu : 0u));
          if (mask != 0u) {  // (warp-uniform)
            pend[c] = pq_filter_round(t_lane + c * 32, acc, L::acc, NQ, mask, item.b_row0 + t0 * 128 + row, sThr + c * 32, sCnt + c * 32,
                                      sCand + c * 32 * cap, cap, t_full, aph);
            any_left |= (pend[c].x | pend[c].y | pend[c].z | pend[c].w) != 0u;
          }
        }
        __syncwarp();
        while (bar_red_or(1, kEpiThreads, any_left)) {
          for (int col = ew; col < NQ; col += kEpiWarps)
            if (sCnt[col] > cap) compact(col);  // (warp-uniform: every lane reads the same counter)
          ptx::named_bar_sync(1, kEpiThreads);
          any_left = false;
#pragma unroll
          for (int b = 0; b < TB; ++b) {
            const uint32_t ab = (acc + b) % L::acc;
#pragma unroll
            for (int c = 0; c < NCH; ++c) {
              // re-read from TMEM, re-test against the tightened thresholds.  tcgen05.ld / wait::ld are .sync.aligned: the
              // whole warp executes them together (lanes with nothing pending pass only = 0)
              uint32_t& pb = b == 0 ? pend[c].x : (b == 1 ? pend[c].y : (b == 2 ? pend[c].z : pend[c].w));
              if (__any_sync(0xffffffffu, pb != 0)) pb = do_chunk(t_lane + ab * NQ, item.b_row0 + (t0 + b) * 128 + row, c, pb);
              any_left |= pb != 0;
            }
          }
          __syncwarp();
        }
        ptx::tc_fence_before_sync();
        __syncwarp();
        if (lane == 0) {
          for (int b = 0; b < nb; ++b) ptx::mbar_arrive(&t_empty[(acc + b) % L::acc]);
        }
        acc += nb;
        if (acc >= static_cast<uint32_t>(L::acc)) { acc -= L::acc; aph ^= 1; }
      }

      // item done: every column's KC best -> global; publish the query's k-th best for the other items of the same query
      for (int col = ew; col < static_cast<int>(min(item.valid_rows, static_cast<uint32_t>(NQ))); col += kEpiWarps) {
        unsigned long long k[4];
        int r[4];
        const int n  = rank_select(col, k, r);
        const int nk = min(n, KC);
        const uint32_t arow = item.a_row0 + col;
        const int64_t o     = static_cast<int64_t>(item.out_off) + static_cast<int64_t>(col) * P.out_row_stride;
        auto emit = [&](unsigned long long key, int r) {
          if (key == 0ull || r >= KC) return;
          const float t = __uint_as_float(okey_inv(static_cast<uint32_t>(key >> 32)));
          if (P.out_score != nullptr) { P.out_score[o + r] = -t; P.out_pos[o + r] = ~static_cast<uint32_t>(key); }
          if (r == kth - 1 && P.b_keys != nullptr) {  // (n >= kth holds when such a rank exists)
            const float pub = __fmaf_rn(P.b_scale, -t, P.b_add ? P.b_add[arow] : 0.f);
            const int kp    = __float_as_int(pub);
            atomicMin(P.b_keys + (P.b_idx ? P.b_idx[arow] : arow), kp >= 0 ? kp : kp ^ 0x7fffffff);
          }
        };
#pragma unroll
        for (int e = 0; e < 4; ++e) emit(k[e], r[e]);
        if (P.out_score != nullptr)
          for (int slot = nk + lane; slot < KC; slot += 32) { P.out_score[o + slot] = INFINITY; P.out_pos[o + slot] = 0xffffffffu; }
      }
      ptx::named_bar_sync(1, kEpiThreads);  // the next item's column init must not overtake another warp's read-out
    }
  }

  ptx::tc_fence_before_sync();
  __syncthreads();
  if (warp == 2) { ptx::tmem_dealloc<L::tmem_cols>(tmem_base); }
}

// ------------------------------------------------------------------------------------ build-side kernels
// one CTA per 128-row tile: codes [128, pq_dim] -> lane-transposed 16-byte chunks + half norms
__global__ void __launch_bounds__(128)
pq_stream_build_kernel(const uint8_t* __restrict__ codes, const int64_t* __restrict__ ids, int64_t pad_id, int pq_dim,
                       const float* __restrict__ pq_centers, bool ip, uint8_t* __restrict__ stream)
{
  __shared__ __align__(16) uint8_t sc[128 * 64];
  const int64_t tile = blockIdx.x;
  const int r        = threadIdx.x;
  const int64_t row  = tile * 128 + r;
  const int64_t blk  = 128 * static_cast<int64_t>(pq_dim) + 512;
  const uint8_t* src = codes + row * pq_dim;
  float nrm = 0.f;
  for (int j = 0; j < pq_dim; ++j) {
    const int c = src[j];
    sc[r * pq_dim + j] = static_cast<uint8_t>(c);
    const float e0 = __bfloat162float(__float2bfloat16_rn(pq_centers[(static_cast<int64_t>(j) * 2 + 0) * 256 + c]));
    const float e1 = __bfloat162float(__float2bfloat16_rn(pq_centers[(static_cast<int64_t>(j) * 2 + 1) * 256 + c]));
    nrm = fmaf(e0, e0, nrm);
    nrm = fmaf(e1, e1, nrm);
  }
  __syncthreads();
  uint8_t* out  = stream + tile * blk;
  const int nh  = pq_dim / 32;
  for (int o = threadIdx.x; o < 8 * nh * 32; o += blockDim.x) {
    const int g = o / (nh * 32), h = (o / 32) % nh, l = o % 32;
    uint32_t w[4] = {0, 0, 0, 0};
#pragma unroll
    for (int i = 0; i < 16; ++i) w[i >> 2] |= static_cast<uint32_t>(sc[(16 * g + i) * pq_dim + 32 * h + l]) << ((i & 3) * 8);
    reinterpret_cast<uint4*>(out)[o] = make_uint4(w[0], w[1], w[2], w[3]);
  }
  reinterpret_cast<float*>(out + 128 * pq_dim)[r] = ids[row] == pad_id ? INFINITY : (ip ? 0.f : 0.5f * nrm);
}

// inverse of pq_stream_build_kernel: one CTA per tile, stream block -> codes [128, pq_dim] one code per byte
__global__ void __launch_bounds__(128) pq_stream_to_flat_kernel(const uint8_t* __restrict__ stream, int pq_dim, uint8_t* __restrict__ codes)
{
  __shared__ __align__(16) uint8_t sc[128 * 64];
  const int64_t tile = blockIdx.x;
  const int64_t blk  = 128 * static_cast<int64_t>(pq_dim) + 512;
  const uint8_t* in  = stream + tile * blk;
  const int nh       = pq_dim / 32;
  for (int o = threadIdx.x; o < 8 * nh * 32; o += blockDim.x) {
    const int g = o / (nh * 32), h = (o / 32) % nh, l = o % 32;
    const uint4 w = reinterpret_cast<const uint4*>(in)[o];
    const uint32_t w4[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
    for (int i = 0; i < 16; ++i) sc[(16 * g + i) * pq_dim + 32 * h + l] = static_cast<uint8_t>((w4[i >> 2] >> ((i & 3) * 8)) & 0xffu);
  }
  __syncthreads();
  uint4* out = reinterpret_cast<uint4*>(codes + tile * 128 * pq_dim);
  for (int o = threadIdx.x; o < 128 * pq_dim / 16; o += blockDim.x) out[o] = reinterpret_cast<const uint4*>(sc)[o];
}

__global__ void pq_cb_words_kernel(const float* __restrict__ pq_centers, int pq_dim, uint32_t* __restrict__ words)
{
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (pq_dim / 32) * 256 * 32) return;
  const int l = t & 31, c = (t >> 5) & 255, h = t >> 13;
  const int j = 32 * h + l;
  const __nv_bfloat16 e0 = __float2bfloat16_rn(pq_centers[(static_cast<int64_t>(j) * 2 + 0) * 256 + c]);
  const __nv_bfloat16 e1 = __float2bfloat16_rn(pq_centers[(static_cast<int64_t>(j) * 2 + 1) * 256 + c]);
  words[t] = static_cast<uint32_t>(__bfloat16_as_ushort(e0)) | (static_cast<uint32_t>(__bfloat16_as_ushort(e1)) << 16);
}

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

// residual rows [rows, Kp] bf16, box = 64 columns x `group` rows, SWIZZLE_128B
CUtensorMap make_query_map(const __nv_bfloat16* ptr, int64_t rows, int Kp, int group)
{
  CUtensorMap m;
  cuuint64_t gdim[2]    = {static_cast<cuuint64_t>(Kp), static_cast<cuuint64_t>(rows)};
  cuuint64_t gstride[1] = {static_cast<cuuint64_t>(Kp) * sizeof(__nv_bfloat16)};
  cuuint32_t box[2]     = {64, static_cast<cuuint32_t>(group)};
  cuuint32_t estr[2]    = {1, 1};
  CUresult r = get_encode_fn()(&m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<__nv_bfloat16*>(ptr), gdim, gstride, box, estr,
                               CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                               CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  B2_EXPECTS(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled (pq residual rows) failed with code %d (rows=%lld Kp=%d)", int(r), (long long)rows, Kp);
  return m;
}

template <int NQ, int NKB, int PASSES>
void launch(cudaStream_t stream, int sms, const CUtensorMap& mq_hi, const CUtensorMap& mq_lo, pq_args a, int n_items)
{
  using L   = layout<NQ, NKB, PASSES>;
  auto kern = pq_stream_scan_kernel<NQ, NKB, PASSES>;
  a.cap     = a.KC <= 16 ? (NQ == 128 ? 32 : 64) : (a.KC <= 32 ? 64 : 128);  // free slots between compactions: cap - KC
  const int fixed = L::off_cand + NQ * a.cap * 8 + 1024 /*alignment slack of the dynamic segment*/;
  a.cstages = std::min(kMaxCStages, (kSmemLimit - fixed) / a.blk);
  B2_EXPECTS(a.cstages >= 2, "pq_stream_scan: shared memory budget exceeded (NQ=%d KC=%d passes=%d)", NQ, a.KC, PASSES);
  const size_t smem = static_cast<size_t>(fixed) + static_cast<size_t>(a.cstages) * a.blk;
  B2_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
  const int grid = n_items < sms ? n_items : sms;
  timed_section ts("pq_stream_scan", stream);
  count_launch();
  kern<<<grid, kThreads, smem, stream>>>(mq_hi, mq_lo, a);
  B2_CUDA(cudaGetLastError());
}

}  // namespace

bool pq_stream_supported(int device, int pq_dim, int pq_len, int pq_bits, bool per_subspace)
{
  int major = 0;
  if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, device) != cudaSuccess) return false;
  return major == 10 && pq_bits == 8 && per_subspace && pq_len == 2 && (pq_dim == 32 || pq_dim == 64);
}

void pq_stream_build(cudaStream_t s, const uint8_t* codes, const int64_t* ids, int64_t pad_id, int64_t rows_total, int pq_dim,
                     const float* pq_centers, bool ip, uint8_t* stream, uint32_t* cb_words)
{
  B2_EXPECTS(pq_dim == 32 || pq_dim == 64, "pq_stream_build: pq_dim must be 32 or 64");
  B2_EXPECTS(rows_total % 128 == 0, "pq_stream_build: lists must be padded to 128-row tiles");
  count_launch();
  pq_cb_words_kernel<<<(pq_dim / 32) * 256 * 32 / 256, 256, 0, s>>>(pq_centers, pq_dim, cb_words);
  if (rows_total > 0) {
    count_launch();
    pq_stream_build_kernel<<<static_cast<unsigned>(rows_total / 128), 128, 0, s>>>(codes, ids, pad_id, pq_dim, pq_centers, ip, stream);
  }
  B2_CUDA(cudaGetLastError());
}

void pq_stream_to_flat(cudaStream_t s, const uint8_t* stream, int64_t rows_total, int pq_dim, uint8_t* codes)
{
  B2_EXPECTS(pq_dim == 32 || pq_dim == 64, "pq_stream_to_flat: pq_dim must be 32 or 64");
  if (rows_total == 0) return;
  count_launch();
  pq_stream_to_flat_kernel<<<static_cast<unsigned>(rows_total / 128), 128, 0, s>>>(stream, pq_dim, codes);
  B2_CUDA(cudaGetLastError());
}

int pq_stream_group(double pairs_per_list, int KC, int passes)
{
  const int64_t forced = env_int("CUVS_B200_PQ_GROUP", 0);  // tests pin the group (read per call)
  int g = pairs_per_list <= 20.0 ? 32 : (pairs_per_list <= 80.0 ? 64 : 128);
  if (forced == 32 || forced == 64 || forced == 128) g = forced;
  if ((KC > 16 || passes == 2) && g > 64) g = 64;  // shared-memory budget: wide candidate buffers / two residual planes
  if (KC > 32) g = 32;                             // 128-entry buffers (k in 33..64): 32 query columns per item
  return g;
}

void pq_stream_scan(cudaStream_t stream, int device, const __nv_bfloat16* q_hi, const __nv_bfloat16* q_lo, int64_t a_rows, int Kp,
                    const uint8_t* code_stream, const uint32_t* cb_words, int pq_dim, const tc_item* items_dev, int n_items,
                    const int* n_items_dev, int group, int KC, int passes, float* out_score, uint32_t* out_pos, int64_t out_row_stride,
                    const tc_bound* bound)
{
  if (n_items == 0) return;
  B2_EXPECTS(Kp == 2 * pq_dim && (pq_dim == 32 || pq_dim == 64), "pq_stream_scan: pq_dim must be 32 or 64 with pq_len 2 (Kp=%d)", Kp);
  B2_EXPECTS(KC == 16 || KC == 32 || KC == 64, "pq_stream_scan: KC must be 16, 32 or 64");
  B2_EXPECTS(passes == 1 || (passes == 2 && q_lo != nullptr), "pq_stream_scan: passes must be 1, or 2 with a lo plane");
  B2_EXPECTS(group == 32 || (group == 64 && KC <= 32) || (group == 128 && KC == 16 && passes == 1), "pq_stream_scan: unsupported group %d", group);
  B2_EXPECTS(a_rows >= group, "pq_stream_scan: the residual plane must hold at least one group of rows");
  pq_args a{};
  a.stream = code_stream;
  a.cb_words = cb_words;
  a.items = items_dev;
  a.n_items_dev = n_items_dev;
  a.out_score = out_score;
  a.out_pos = out_pos;
  a.out_row_stride = out_row_stride;
  if (bound != nullptr && bound->keys != nullptr) {
    a.b_keys = bound->keys;
    a.b_idx = bound->idx;
    a.b_add = bound->add;
    a.b_scale = bound->scale;
    a.kth = bound->kth;
  } else {
    a.b_scale = 1.0f;
  }
  a.n_items_host = n_items;
  a.KC = KC;
  a.blk = static_cast<int>(pq_stream_tile_bytes(pq_dim));
  dbuf<int> sched(1, stream);
  B2_CUDA(cudaMemsetAsync(sched.data(), 0, sizeof(int), stream));
  a.sched = sched.data();
  const CUtensorMap mq  = make_query_map(q_hi, a_rows, Kp, group);
  const CUtensorMap mql = passes == 2 ? make_query_map(q_lo, a_rows, Kp, group) : mq;
  const int sms = sm_count_of(device);
  const int nkb = Kp / 64;
#define B2_PQ_CASE(NQ_, NKB_, P_) \
  if (group == NQ_ && nkb == NKB_ && passes == P_) return launch<NQ_, NKB_, P_>(stream, sms, mq, mql, a, n_items);
  B2_PQ_CASE(32, 1, 1) B2_PQ_CASE(64, 1, 1) B2_PQ_CASE(128, 1, 1) B2_PQ_CASE(32, 2, 1) B2_PQ_CASE(64, 2, 1) B2_PQ_CASE(128, 2, 1)
  B2_PQ_CASE(32, 1, 2) B2_PQ_CASE(64, 1, 2) B2_PQ_CASE(32, 2, 2) B2_PQ_CASE(64, 2, 2)
#undef B2_PQ_CASE
  B2_FAIL("pq_stream_scan: no kernel for group=%d Kp=%d passes=%d", group, Kp, passes);
}

}  // namespace b200
