// Batched top-k: one CTA per row, 4-pass 8-bit radix select over order-preserving float keys,
// ordered gather of threshold ties, bitonic sort of the k survivors in shared memory.
//
// Why radix (not warp-sort queues) here: every caller on the scan path hands this kernel rows that
// are already reduced by a fused in-scan top-k (n_probes*k' candidates, n_lists coarse distances,
// n_shards*k partials), so rows are short-to-medium and L2-resident; a histogram pass reads each
// element once with perfectly coalesced 128-bit loads and needs no per-thread state, and the tie
// rule "smaller position wins" falls out of the ordered gather — which is what makes results
// reproducible against the oracle (oracle/oracle.c: oracle_select_k).
#include "common.hpp"
#include "select_k.cuh"
#include "timing.hpp"

#include <cuvs/selection/select_k.h>

#include <algorithm>
#include <cfloat>

namespace b200 {
namespace {

__device__ __forceinline__ uint32_t f2key(float v, bool select_min)
{
  uint32_t u = __float_as_uint(v);
  if ((u << 1) == 0) u = 0;  // -0.0 == +0.0 (the oracle compares floats)
  u = (u & 0x80000000u) ? ~u : (u | 0x80000000u);
  return select_min ? u : ~u;
}

template <typename T>
__device__ __forceinline__ T all_ones()
{
  return static_cast<T>(~static_cast<T>(0));
}
template <>
__device__ __forceinline__ int64_t all_ones<int64_t>()
{
  return -1;
}
template <>
__device__ __forceinline__ int32_t all_ones<int32_t>()
{
  return -1;
}

constexpr int kMaxK = 2048;

// smem: hist[256] | scalars[8] | warp_tot[32] | skeys[kpow2] (u64)
template <typename IdxIn, typename IdxOut, bool HasIdx>
__global__ void __launch_bounds__(1024) select_k_kernel(const float* __restrict__ in_val,
                                                          const IdxIn* __restrict__ in_idx,
                                                          int64_t len,
                                                          int64_t in_ld,
                                                          int k,
                                                          int kpow2,
                                                          float* __restrict__ out_val,
                                                          IdxOut* __restrict__ out_idx,
                                                          bool select_min)
{
  extern __shared__ __align__(16) unsigned char smem_raw[];
  uint32_t* hist     = reinterpret_cast<uint32_t*>(smem_raw);
  uint32_t* scal     = hist + 256;  // [0]=prefix [1]=kk [2]=lt counter [3]=running_eq
  uint32_t* warp_tot = scal + 8;
  uint64_t* skeys    = reinterpret_cast<uint64_t*>(warp_tot + 32);

  const int64_t row = blockIdx.x;
  const float* v    = in_val + row * in_ld;
  const int tid     = threadIdx.x;
  const int bs      = blockDim.x;
  const int k_eff   = len < k ? static_cast<int>(len) : k;

  for (int i = tid; i < kpow2; i += bs) skeys[i] = ~0ull;
  if (tid == 0) { scal[0] = 0; scal[1] = k_eff; scal[2] = 0; scal[3] = 0; }
  __syncthreads();

  if (k_eff > 0) {
    uint32_t prefix = 0, mask = 0;
    for (int pass = 0; pass < 4; ++pass) {
      const int shift = 24 - 8 * pass;
      for (int i = tid; i < 256; i += bs) hist[i] = 0;
      __syncthreads();
      for (int64_t i = tid; i < len; i += bs) {
        uint32_t u = f2key(v[i], select_min);
        if ((u & mask) == prefix) {
          // warp-aggregated histogram update: rows of near-equal distances pile into one bucket
          const uint32_t bucket = (u >> shift) & 255u;
          const uint32_t peers  = __match_any_sync(__activemask(), bucket);
          if ((threadIdx.x & 31) == __ffs(peers) - 1) atomicAdd(&hist[bucket], __popc(peers));
        }
      }
      __syncthreads();
      if (tid < 32) {
        // warp scan over 256 buckets (8 per lane)
        uint32_t loc[8], s = 0;
#pragma unroll
        for (int j = 0; j < 8; ++j) { loc[j] = hist[tid * 8 + j]; s += loc[j]; }
        uint32_t incl = s;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
          if (tid >= o) incl += t;
        }
        uint32_t excl = incl - s;
        const uint32_t kk = scal[1];
        __syncwarp();  // every lane has read kk before the owning lane rewrites it
        // the bucket where the cumulative count first reaches kk
        if (excl < kk && kk <= incl) {
          uint32_t c = excl;
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            if (c < kk && kk <= c + loc[j]) {
              scal[0] = prefix | (static_cast<uint32_t>(tid * 8 + j) << shift);
              scal[1] = kk - c;
            }
            c += loc[j];
          }
        }
      }
      __syncthreads();
      prefix = scal[0];
      mask |= 0xffu << shift;
      __syncthreads();
    }
    const uint32_t T       = prefix;
    const uint32_t need_eq = scal[1];
    const uint32_t n_lt    = k_eff - need_eq;

    // strictly better than the threshold: any order (sorted afterwards)
    for (int64_t i = tid; i < len; i += bs) {
      uint32_t u = f2key(v[i], select_min);
      if (u < T) {
        uint32_t slot = atomicAdd(&scal[2], 1u);
        skeys[slot]   = (static_cast<uint64_t>(u) << 32) | static_cast<uint32_t>(i);
      }
    }
    // ties at the threshold: in position order, first need_eq of them
    const int lane = tid & 31, wid = tid >> 5, nw = (bs + 31) >> 5;
    for (int64_t base = 0; base < len; base += bs) {
      int64_t i  = base + tid;
      bool flag  = (i < len) && (f2key(v[i], select_min) == T);
      uint32_t b = __ballot_sync(0xffffffffu, flag);
      if (lane == 0) warp_tot[wid] = __popc(b);
      __syncthreads();
      uint32_t off = 0, tot = 0;
      for (int w = 0; w < nw; ++w) {
        uint32_t t = warp_tot[w];
        if (w < wid) off += t;
        tot += t;
      }
      const uint32_t running = scal[3];
      if (flag) {
        uint32_t rank = running + off + __popc(b & ((1u << lane) - 1u));
        if (rank < need_eq) skeys[n_lt + rank] = (static_cast<uint64_t>(T) << 32) | static_cast<uint32_t>(i);
      }
      __syncthreads();
      if (tid == 0) scal[3] = running + tot;
      __syncthreads();
      if (running + tot >= need_eq) break;
    }
    __syncthreads();

    // bitonic sort of kpow2 composite keys, ascending (key, position)
    for (int size = 2; size <= kpow2; size <<= 1) {
      for (int stride = size >> 1; stride > 0; stride >>= 1) {
        for (int i = tid; i < (kpow2 >> 1); i += bs) {
          int lo  = (i / stride) * (stride << 1) + (i % stride);
          int hi  = lo + stride;
          bool up = ((lo & size) == 0);
          uint64_t a = skeys[lo], b2 = skeys[hi];
          if ((a > b2) == up) { skeys[lo] = b2; skeys[hi] = a; }
        }
        __syncthreads();
      }
    }
  }

  for (int j = tid; j < k; j += bs) {
    float ov;
    IdxOut oi;
    if (j < k_eff) {
      uint32_t pos = static_cast<uint32_t>(skeys[j] & 0xffffffffull);
      ov           = v[pos];
      if constexpr (HasIdx) {
        oi = static_cast<IdxOut>(in_idx[row * in_ld + pos]);
      } else {
        oi = static_cast<IdxOut>(pos);
      }
    } else {
      ov = select_min ? FLT_MAX : -FLT_MAX;
      oi = all_ones<IdxOut>();
    }
    out_val[row * k + j] = ov;
    out_idx[row * k + j] = oi;
  }
}


// ---------------------------------------------------------------------------------------------------------------------
// Medium rows (2k..32k elements, k <= 256: the coarse search's n_lists distances per query).  The radix kernel above reads
// the row six times and its first two 8-bit passes are wasted on distances (one exponent => one bucket).  Here the row is
// read ONCE into registers as composite keys K = key << 32 | position (unique, so "smaller position wins" is part of the
// order); the keys in play are binned LINEARLY over their actual [min, max] span into 2048 buckets, the bucket holding the
// k-th key is found by one warp, everything below it is a winner, and the bucket itself (a handful of keys) is finished by
// rank counting — or, if it is crowded (ties, clustered values), becomes the next span.  One global read, ~3 register passes.
constexpr int kRegThreads = 512;
constexpr int kRegBins    = 2048;
constexpr int kRegEqCap   = 1024;
constexpr int kRegMaxK    = 256;

template <int E, typename IdxIn, typename IdxOut, bool HasIdx>
__global__ void __launch_bounds__(kRegThreads, E <= 32 ? 2 : 1) select_k_reg_kernel(const float* __restrict__ in_val, const IdxIn* __restrict__ in_idx,
                                                                   int64_t len, int64_t in_ld, int k, float* __restrict__ out_val,
                                                                   IdxOut* __restrict__ out_idx, bool select_min, int sample_elems)
{
  __shared__ __align__(16) uint32_t hist[kRegBins];
  __shared__ unsigned long long okeys[kRegMaxK];
  __shared__ unsigned long long ebuf[kRegEqCap];
  __shared__ uint32_t red[2 * (kRegThreads / 32)];
  __shared__ uint32_t wtot[kRegThreads / 32];
  __shared__ uint32_t scal[8];  // [0] threshold bucket [1] keys below it [2] keys in it [3] winners stored [4] bucket keys stored

  const int64_t row = blockIdx.x;
  const float* v    = in_val + row * in_ld;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int k_eff = len < k ? static_cast<int>(len) : k;

  uint32_t u[E];
  uint32_t mn = 0xffffffffu, mx = 0u;  // bounds on the 32-bit keys are enough: the span only has to COVER the composites
#pragma unroll
  for (int j = 0; j < E; ++j) {
    const int64_t i = static_cast<int64_t>(j) * kRegThreads + tid;
    u[j] = 0u;
    if (i < len) {
      u[j] = f2key(v[i], select_min);
      mn   = min(mn, u[j]);
      mx   = max(mx, u[j]);
    }
  }
  mn = __reduce_min_sync(0xffffffffu, mn);
  mx = __reduce_max_sync(0xffffffffu, mx);
  if (lane == 0) { red[wid] = mn; red[kRegThreads / 32 + wid] = mx; }
  if (tid == 0) { scal[3] = 0; scal[4] = 0; }
  __syncthreads();
  uint32_t lo32 = red[lane & (kRegThreads / 32 - 1)], hi32 = red[kRegThreads / 32 + (lane & (kRegThreads / 32 - 1))];
  lo32 = __reduce_min_sync(0xffffffffu, lo32);
  hi32 = __reduce_max_sync(0xffffffffu, hi32);
  unsigned long long lo = static_cast<unsigned long long>(lo32) << 32, hi = (static_cast<unsigned long long>(hi32) << 32) | 0xffffffffull;
  const unsigned long long full_span = hi - lo;
  unsigned long long span = full_span;  // keys in play: lo <= K <= lo + span
  uint32_t need = static_cast<uint32_t>(k_eff);

  // Sampled upper bound.  k << len (48 probes out of 16k centres): binning the whole row spends one shared-memory atomic per
  // element on keys that cannot win.  Take the first `es` elements of every thread as a sample (es * 32 per warp, strided over
  // the row), T = max over the warps of the warp's sample MINIMUM: every warp has a key <= T, and for es * 32 ~ 0.7 len / k
  // about 1 % .. 3 % of the row lies below T, of which the k-th smallest is one with overwhelming probability (k = 48,
  // len = 16384: miss rate ~ 4e-5 on exchangeable data).  The first binning round then only counts keys <= T; if fewer than
  // `need` keys are there (adversarial order, e.g. a sorted row) the round is repeated over the full span — exactness never
  // depends on the sample.
  if (sample_elems > 0) {
    uint32_t smin = 0xffffffffu;
#pragma unroll
    for (int j = 0; j < E; ++j) {
      const int64_t i = static_cast<int64_t>(j) * kRegThreads + tid;
      if (j < sample_elems && i < len) smin = min(smin, u[j]);
    }
    smin = __reduce_min_sync(0xffffffffu, smin);
    __syncthreads();  // (red[] is still being read above)
    if (lane == 0) red[wid] = smin;
    __syncthreads();
    uint32_t t32 = red[lane & (kRegThreads / 32 - 1)];
    t32 = __reduce_max_sync(0xffffffffu, t32);
    if (t32 < hi32) span = ((static_cast<unsigned long long>(t32) << 32) | 0xffffffffull) - lo;
  }

  while (need > 0) {
    const int s = span >= static_cast<unsigned long long>(kRegBins) ? (64 - __clzll(static_cast<long long>(span))) - 11 : 0;  // (span >> s) < 2048
    for (int i = tid; i < kRegBins; i += kRegThreads) hist[i] = 0;
    if (tid == 0) scal[0] = 0xffffffffu;  // "no bucket reaches `need`" until the scan says otherwise
    __syncthreads();
#pragma unroll
    for (int j = 0; j < E; ++j) {
      const int64_t i = static_cast<int64_t>(j) * kRegThreads + tid;
      const unsigned long long K = (static_cast<unsigned long long>(u[j]) << 32) | static_cast<uint32_t>(i);
      if (i < len && K >= lo && K - lo <= span) atomicAdd(&hist[static_cast<uint32_t>((K - lo) >> s)], 1u);
    }
    __syncthreads();
    {
      // two-level scan, all 16 warps: warp w owns buckets [128 w, 128 w + 128), lane l four of them (one conflict-free 128-bit load)
      static_assert(kRegBins == 4 * kRegThreads, "one uint4 of buckets per thread");
      const uint4 h4 = reinterpret_cast<const uint4*>(hist)[tid];
      const uint32_t sum = h4.x + h4.y + h4.z + h4.w;
      uint32_t incl = sum;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
      }
      if (lane == 31) wtot[wid] = incl;
      __syncthreads();
      uint32_t c = incl - sum;
#pragma unroll
      for (int w = 0; w < kRegThreads / 32; ++w) c += w < wid ? wtot[w] : 0u;
      if (c < need && need <= c + sum) {  // exactly one thread: the bucket where the running count reaches `need`
        const uint32_t h[4] = {h4.x, h4.y, h4.z, h4.w};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          if (c < need && need <= c + h[e]) { scal[0] = tid * 4 + e; scal[1] = c; scal[2] = h[e]; }
          c += h[e];
        }
      }
    }
    __syncthreads();
    const uint32_t bstar = scal[0], below = scal[1], inb = scal[2];
    if (bstar == 0xffffffffu) {  // (block-uniform; first round only) the sampled bound cut below the k-th key: full span
      span = full_span;
      __syncthreads();
      continue;
    }
    const bool finish = inb <= static_cast<uint32_t>(kRegEqCap);
#pragma unroll
    for (int j = 0; j < E; ++j) {
      const int64_t i = static_cast<int64_t>(j) * kRegThreads + tid;
      const unsigned long long K = (static_cast<unsigned long long>(u[j]) << 32) | static_cast<uint32_t>(i);
      if (i < len && K >= lo && K - lo <= span) {
        const uint32_t b = static_cast<uint32_t>((K - lo) >> s);
        if (b < bstar) okeys[atomicAdd(&scal[3], 1u)] = K;
        else if (b == bstar && finish) ebuf[atomicAdd(&scal[4], 1u)] = K;
      }
    }
    need -= below;
    __syncthreads();
    if (finish) {
      // the bucket's `need` smallest keys, by rank counting (keys are unique)
      const uint32_t base = scal[3];
      for (uint32_t e = tid; e < inb; e += kRegThreads) {
        const unsigned long long K = ebuf[e];
        uint32_t r = 0;
        for (uint32_t o = 0; o < inb; ++o) r += ebuf[o] < K ? 1u : 0u;
        if (r < need) okeys[base + r] = K;
      }
      need = 0;
    } else {
      lo += static_cast<unsigned long long>(bstar) << s;  // (s > 0 here: with s == 0 a bucket holds one key)
      span = (1ull << s) - 1ull;
    }
    __syncthreads();
  }

  // ascending (key, position): rank counting among the k winners
  for (int t = tid; t < k; t += kRegThreads) {
    if (t < k_eff) {
      const unsigned long long K = okeys[t];
      int r = 0;
      for (int o = 0; o < k_eff; ++o) r += okeys[o] < K ? 1 : 0;
      const uint32_t pos = static_cast<uint32_t>(K);
      out_val[row * k + r] = v[pos];
      if constexpr (HasIdx) out_idx[row * k + r] = static_cast<IdxOut>(in_idx[row * in_ld + pos]);
      else out_idx[row * k + r] = static_cast<IdxOut>(pos);
    } else {
      out_val[row * k + t] = select_min ? FLT_MAX : -FLT_MAX;
      out_idx[row * k + t] = all_ones<IdxOut>();
    }
  }
}

template <typename IdxIn, typename IdxOut, bool HasIdx>
void launch(cudaStream_t stream, const float* in_val, const void* in_idx, int64_t batch, int64_t len, int64_t in_ld,
            int k, float* out_val, void* out_idx, bool select_min)
{
  if (len >= 2048 && len <= 64 * kRegThreads && k <= kRegMaxK) {
    count_launch();
    const unsigned grid = static_cast<unsigned>(batch);
    static bool carve = [] {  // two resident CTAs need ~40 KB of shared memory: ask for the carve-out once per instantiation
      cudaFuncSetAttribute(select_k_reg_kernel<8, IdxIn, IdxOut, HasIdx>, cudaFuncAttributePreferredSharedMemoryCarveout, 50);
      cudaFuncSetAttribute(select_k_reg_kernel<16, IdxIn, IdxOut, HasIdx>, cudaFuncAttributePreferredSharedMemoryCarveout, 50);
      cudaFuncSetAttribute(select_k_reg_kernel<32, IdxIn, IdxOut, HasIdx>, cudaFuncAttributePreferredSharedMemoryCarveout, 50);
      cudaFuncSetAttribute(select_k_reg_kernel<64, IdxIn, IdxOut, HasIdx>, cudaFuncAttributePreferredSharedMemoryCarveout, 50);
      return true;
    }();
    (void)carve;
    auto ii = static_cast<const IdxIn*>(in_idx);
    auto oo = static_cast<IdxOut*>(out_idx);
    // sample elements per thread for the kernel's sampled bound: 32 * es ~ 0.7 * len / k samples per warp (0 = no sampling)
    const int es = static_cast<int>(std::min<int64_t>(64, (7 * len) / (320 * static_cast<int64_t>(std::max(k, 1)))));
    if (len <= 8 * kRegThreads) select_k_reg_kernel<8, IdxIn, IdxOut, HasIdx><<<grid, kRegThreads, 0, stream>>>(in_val, ii, len, in_ld, k, out_val, oo, select_min, es);
    else if (len <= 16 * kRegThreads) select_k_reg_kernel<16, IdxIn, IdxOut, HasIdx><<<grid, kRegThreads, 0, stream>>>(in_val, ii, len, in_ld, k, out_val, oo, select_min, es);
    else if (len <= 32 * kRegThreads) select_k_reg_kernel<32, IdxIn, IdxOut, HasIdx><<<grid, kRegThreads, 0, stream>>>(in_val, ii, len, in_ld, k, out_val, oo, select_min, es);
    else select_k_reg_kernel<64, IdxIn, IdxOut, HasIdx><<<grid, kRegThreads, 0, stream>>>(in_val, ii, len, in_ld, k, out_val, oo, select_min, es);
    B2_CUDA(cudaGetLastError());
    return;
  }
  int kpow2 = 1;
  while (kpow2 < k) kpow2 <<= 1;
  if (kpow2 < 2) kpow2 = 2;
  int threads = len <= 2048 ? 128 : (len <= 32768 ? 256 : 1024);
  if (kpow2 / 2 > threads && threads < 1024) threads = kpow2 / 2 > 1024 ? 1024 : kpow2 / 2;
  size_t smem = (256 + 8 + 32) * sizeof(uint32_t) + static_cast<size_t>(kpow2) * sizeof(uint64_t);
  count_launch();
  select_k_kernel<IdxIn, IdxOut, HasIdx><<<static_cast<unsigned>(batch), threads, smem, stream>>>(
    in_val, static_cast<const IdxIn*>(in_idx), len, in_ld, k, kpow2, out_val, static_cast<IdxOut*>(out_idx), select_min);
  B2_CUDA(cudaGetLastError());
}

__global__ void merge_gather_kernel(const float* __restrict__ in_keys, const int64_t* __restrict__ in_vals,
                                    float* __restrict__ tmp_keys, int64_t* __restrict__ tmp_vals, int64_t n_parts,
                                    int64_t n_rows, int k, const int64_t* __restrict__ translations)
{
  int64_t total = n_parts * n_rows * k;
  for (int64_t t = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; t < total;
       t += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    int64_t j = t % k, r = (t / k) % n_rows, p = t / (k * n_rows);
    int64_t id = in_vals[t];
    if (translations && id >= 0 && id != INT64_MAX) id += translations[p];
    tmp_keys[(r * n_parts + p) * k + j] = in_keys[t];
    tmp_vals[(r * n_parts + p) * k + j] = id;
  }
}

}  // namespace

void select_k(cudaStream_t stream, const float* in_val, const void* in_idx, idx_kind in_kind, int64_t batch,
              int64_t len, int64_t in_ld, int k, float* out_val, void* out_idx, idx_kind out_kind, bool select_min)
{
  B2_EXPECTS(k >= 1 && k <= kMaxK, "select_k: k must be in [1, %d] (got %d)", kMaxK, k);
  B2_EXPECTS(len >= 0 && len < (int64_t(1) << 32), "select_k: row length out of range");
  B2_EXPECTS(batch < (int64_t(1) << 31), "select_k: batch too large");
  if (batch == 0) return;
  if (in_idx == nullptr) in_kind = IDX_NONE;
  if (in_kind == IDX_NONE && out_kind == IDX_I64) return launch<int64_t, int64_t, false>(stream, in_val, nullptr, batch, len, in_ld, k, out_val, out_idx, select_min);
  if (in_kind == IDX_NONE && out_kind == IDX_U32) return launch<uint32_t, uint32_t, false>(stream, in_val, nullptr, batch, len, in_ld, k, out_val, out_idx, select_min);
  if (in_kind == IDX_NONE && out_kind == IDX_I32) return launch<int32_t, int32_t, false>(stream, in_val, nullptr, batch, len, in_ld, k, out_val, out_idx, select_min);
  if (in_kind == IDX_I64 && out_kind == IDX_I64) return launch<int64_t, int64_t, true>(stream, in_val, in_idx, batch, len, in_ld, k, out_val, out_idx, select_min);
  if (in_kind == IDX_U32 && out_kind == IDX_U32) return launch<uint32_t, uint32_t, true>(stream, in_val, in_idx, batch, len, in_ld, k, out_val, out_idx, select_min);
  if (in_kind == IDX_U32 && out_kind == IDX_I64) return launch<uint32_t, int64_t, true>(stream, in_val, in_idx, batch, len, in_ld, k, out_val, out_idx, select_min);
  if (in_kind == IDX_I32 && out_kind == IDX_I32) return launch<int32_t, int32_t, true>(stream, in_val, in_idx, batch, len, in_ld, k, out_val, out_idx, select_min);
  B2_FAIL("select_k: unsupported index dtype combination (%d -> %d)", int(in_kind), int(out_kind));
}

void knn_merge_parts(cudaStream_t stream, const float* in_keys, const int64_t* in_vals, float* out_keys,
                     int64_t* out_vals, int64_t n_parts, int64_t n_rows, int k, const int64_t* translations_dev,
                     bool select_min)
{
  if (n_rows == 0) return;
  dbuf<float> tk(static_cast<size_t>(n_parts * n_rows * k), stream);
  dbuf<int64_t> tv(static_cast<size_t>(n_parts * n_rows * k), stream);
  int64_t total = n_parts * n_rows * k;
  int blocks    = static_cast<int>(std::min<int64_t>((total + 255) / 256, 65535));
  count_launch();
  merge_gather_kernel<<<blocks, 256, 0, stream>>>(in_keys, in_vals, tk.data(), tv.data(), n_parts, n_rows, k,
                                                  translations_dev);
  B2_CUDA(cudaGetLastError());
  select_k(stream, tk.data(), tv.data(), IDX_I64, n_rows, n_parts * k, n_parts * k, k, out_keys, out_vals, IDX_I64,
           select_min);
}

}  // namespace b200

using namespace b200;

static idx_kind kind_of(const DLTensor& t)
{
  if (dl_is(t, kDLInt, 64)) return IDX_I64;
  if (dl_is(t, kDLUInt, 32)) return IDX_U32;
  if (dl_is(t, kDLInt, 32)) return IDX_I32;
  B2_FAIL("index tensors must be int64, uint32 or int32");
}

extern "C" cuvsError_t cuvsSelectK(cuvsResources_t res, DLManagedTensor* in_val, DLManagedTensor* in_idx,
                                   DLManagedTensor* out_val, DLManagedTensor* out_idx, bool select_min, bool /*sorted*/)
{
  return guarded([=] {
    auto r = as_res(res);
    B2_EXPECTS(in_val && out_val && out_idx, "null tensor");
    const DLTensor& iv = in_val->dl_tensor;
    const DLTensor& ov = out_val->dl_tensor;
    const DLTensor& oi = out_idx->dl_tensor;
    B2_EXPECTS(dl_is_device(iv) && dl_is_device(ov) && dl_is_device(oi), "select_k tensors should have device compatible memory");
    B2_EXPECTS(iv.ndim == 2 && ov.ndim == 2 && oi.ndim == 2, "select_k tensors must be 2-D");
    B2_EXPECTS(dl_is(iv, kDLFloat, 32) && dl_is(ov, kDLFloat, 32), "values must be float32");
    B2_EXPECTS(dl_is_c_contiguous(iv) && dl_is_c_contiguous(ov) && dl_is_c_contiguous(oi), "select_k tensors must be row-major contiguous");
    B2_EXPECTS(ov.shape[0] == iv.shape[0] && oi.shape[0] == iv.shape[0] && ov.shape[1] == oi.shape[1], "output shape mismatch");
    const void* ii  = nullptr;
    idx_kind ikind  = IDX_NONE;
    if (in_idx) {
      const DLTensor& it = in_idx->dl_tensor;
      B2_EXPECTS(dl_is_device(it) && it.ndim == 2 && it.shape[0] == iv.shape[0] && it.shape[1] == iv.shape[1] && dl_is_c_contiguous(it), "in_idx shape mismatch");
      ikind = kind_of(it);
      ii    = dl_ptr<void>(it);
    }
    select_k(r->stream, dl_ptr<float>(iv), ii, ikind, iv.shape[0], iv.shape[1], iv.shape[1], static_cast<int>(ov.shape[1]),
             dl_ptr<float>(ov), dl_ptr<void>(oi), kind_of(oi), select_min);
  });
}

extern "C" cuvsError_t cuvsKnnMergeParts(cuvsResources_t res, DLManagedTensor* in_keys, DLManagedTensor* in_values,
                                         DLManagedTensor* out_keys, DLManagedTensor* out_values, int64_t n_parts,
                                         const int64_t* translations, bool select_min)
{
  return guarded([=] {
    auto r = as_res(res);
    B2_EXPECTS(in_keys && in_values && out_keys && out_values, "null tensor");
    const DLTensor& ik = in_keys->dl_tensor;
    const DLTensor& iv = in_values->dl_tensor;
    const DLTensor& ok = out_keys->dl_tensor;
    const DLTensor& ov = out_values->dl_tensor;
    B2_EXPECTS(dl_is_device(ik) && dl_is_device(iv) && dl_is_device(ok) && dl_is_device(ov), "merge tensors should have device compatible memory");
    B2_EXPECTS(dl_is(ik, kDLFloat, 32) && dl_is(ok, kDLFloat, 32), "keys must be float32");
    B2_EXPECTS(dl_is(iv, kDLInt, 64) && dl_is(ov, kDLInt, 64), "values must be int64");
    B2_EXPECTS(ik.ndim == 2 && ok.ndim == 2 && n_parts >= 1 && ik.shape[0] % n_parts == 0, "bad merge shapes");
    int64_t n_rows = ik.shape[0] / n_parts;
    int k          = static_cast<int>(ik.shape[1]);
    B2_EXPECTS(ok.shape[0] == n_rows && ok.shape[1] == k && ov.shape[0] == n_rows && ov.shape[1] == k, "bad output shape");
    dbuf<int64_t> tr;
    if (translations) {
      tr.alloc(static_cast<size_t>(n_parts), r->stream);
      B2_CUDA(cudaMemcpyAsync(tr.data(), translations, sizeof(int64_t) * n_parts, cudaMemcpyHostToDevice, r->stream));
    }
    knn_merge_parts(r->stream, dl_ptr<float>(ik), dl_ptr<int64_t>(iv), dl_ptr<float>(ok), dl_ptr<int64_t>(ov), n_parts,
                    n_rows, k, translations ? tr.data() : nullptr, select_min);
    if (translations) B2_CUDA(cudaStreamSynchronize(r->stream));  // `translations` is a host array owned by the caller
  });
}
