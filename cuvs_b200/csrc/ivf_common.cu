// Shared IVF / k-means machinery: see ivf_common.cuh.
#include "ivf_common.cuh"

#include "exact.cuh"
#include "ivf_lists.cuh"
#include "select_k.cuh"
#include "timing.hpp"

#include <algorithm>
#include <cfloat>
#include <cmath>
#include <vector>

namespace b200 {
namespace {

__global__ void iota_items_kernel(tc_item* items, int m_tiles, int64_t n_rows, uint32_t b_tiles, int64_t row_stride)
{
  int m = blockIdx.x * blockDim.x + threadIdx.x;
  if (m >= m_tiles) return;
  tc_item it;
  it.a_row0     = m * 128;
  it.b_row0     = 0;
  it.n_tiles    = b_tiles;
  int64_t valid = n_rows - static_cast<int64_t>(m) * 128;
  it.valid_rows = valid > 128 ? 128 : static_cast<uint32_t>(valid);
  it.out_off    = static_cast<uint64_t>(m) * 128 * row_stride;
  items[m]      = it;
}

// (query tile, centre range) items of the fused coarse search: item i = (split i / m_tiles, query tile i % m_tiles)
__global__ void split_items_kernel(tc_item* items, int m_tiles, int splits, int64_t nq, uint32_t tiles_total, int KCW)
{
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= m_tiles * splits) return;
  const int sp = i / m_tiles, m = i % m_tiles;
  const uint32_t per = (tiles_total + splits - 1) / splits;
  const uint32_t t0 = min(tiles_total, sp * per), t1 = min(tiles_total, t0 + per);
  tc_item it;
  it.a_row0     = m * 128;
  it.b_row0     = t0 * 128;
  it.n_tiles    = t1 - t0;
  const int64_t valid = nq - static_cast<int64_t>(m) * 128;
  it.valid_rows = valid > 128 ? 128 : static_cast<uint32_t>(valid);
  it.out_off    = (static_cast<uint64_t>(m) * 128 * splits + sp) * KCW;
  items[i]      = it;
}

// Fused coarse search, merge step: one CTA per query ranks the W = splits * lists * KC candidates its items kept
// (sorted lists of KC per centre range and column half) by (score, centre id) — the order select_k imposes on the dense
// score row, where position == centre id — and writes the n_probes best.  The scan rejects a centre only when its score is
// not below a full list's worst entry (its own list's, or through the bound shared between a query's items, another list's at
// an earlier time; such entries only decrease), so every centre outside the candidates scores >= floor = the minimum over
// the full lists of their worst entry.  If the n_probes-th candidate lies STRICTLY below the floor the selection — ties
// included — is the dense one; otherwise, or when fewer than n_probes candidates exist, the query is counted in *n_flagged
// and the caller redoes the batch through the dense path.
constexpr int kCoarseMergeThreads = 128;
constexpr int kCoarseMaxW         = 1024;
template <int E>  // candidates per thread: W <= E * kCoarseMergeThreads
__global__ void __launch_bounds__(kCoarseMergeThreads)
coarse_merge_kernel(const float* __restrict__ cs, const uint32_t* __restrict__ cp, int W, int KC, int n_probes, uint32_t* __restrict__ probes,
                    float* __restrict__ probe_scores, int* __restrict__ n_flagged)
{
  extern __shared__ unsigned long long ckeys[];
  __shared__ float s_floor;
  __shared__ int s_valid;
  const int64_t q = blockIdx.x;
  const int tid   = threadIdx.x;
  unsigned long long mine[E];
  int n_mine = 0;
  if (tid == 0) s_valid = 0;
  if (tid < 32) {
    float m = INFINITY;
    for (int l = tid; l * KC < W; l += 32) m = fminf(m, cs[q * W + l * KC + KC - 1]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fminf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if (tid == 0) s_floor = m;
  }
  __syncthreads();
#pragma unroll
  for (int e = 0; e < E; ++e) {
    const int c = e * kCoarseMergeThreads + tid;
    unsigned long long K = ~0ull;
    if (c < W) {
      const uint32_t pos = cp[q * W + c];
      if (pos != 0xffffffffu) {
        uint32_t u = __float_as_uint(cs[q * W + c]);
        if ((u << 1) == 0) u = 0;  // -0.0 == +0.0, as in select_k
        u = (u & 0x80000000u) ? ~u : (u | 0x80000000u);
        K = (static_cast<unsigned long long>(u) << 32) | pos;
        ++n_mine;
      }
      ckeys[c] = K;
    }
    mine[e] = K;
  }
  if (n_mine) atomicAdd(&s_valid, n_mine);
  __syncthreads();
  int rank[E];
#pragma unroll
  for (int e = 0; e < E; ++e) rank[e] = 0;
  for (int o = 0; o < W; ++o) {
    const unsigned long long Ko = ckeys[o];  // (broadcast)
#pragma unroll
    for (int e = 0; e < E; ++e) rank[e] += Ko < mine[e] ? 1 : 0;
  }
#pragma unroll
  for (int e = 0; e < E; ++e) {
    if (mine[e] != ~0ull && rank[e] < n_probes) {
      const int c       = e * kCoarseMergeThreads + tid;
      const float score = cs[q * W + c];
      probes[q * n_probes + rank[e]]       = static_cast<uint32_t>(mine[e]);
      probe_scores[q * n_probes + rank[e]] = score;
      if (rank[e] == n_probes - 1 && !(score < s_floor)) atomicAdd(n_flagged, 1);  // (strict: also rules out boundary ties)
    }
  }
  if (tid == 0 && s_valid < n_probes) atomicAdd(n_flagged, 1);
}

// best entry among the heads of the `lists` sorted candidate lists of each row
__global__ void first_of_rows_kernel(const uint32_t* __restrict__ pos, const float* __restrict__ score, int64_t n, int KC,
                                     int lists, uint32_t* __restrict__ labels, float* __restrict__ out_scores)
{
  int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  if (i >= n) return;
  const int64_t b = i * KC * lists;
  float best      = score[b];
  uint32_t bp     = pos[b];
  for (int j = 1; j < lists; ++j) {
    float s    = score[b + j * KC];
    uint32_t p = pos[b + j * KC];
    if (s < best || (s == best && p < bp)) { best = s; bp = p; }
  }
  labels[i] = bp;
  if (out_scores) out_scores[i] = best;
}

// ---- probe bucketing -----------------------------------------------------------------------
// Pairs are bucketed by (list, near/far bin): bin 0 holds a query's nearest `near_ranks` probes.  Inside a list the near
// pairs come first, so each list's FIRST 128-pair work item holds the lowest probe ranks; all first items are scheduled
// before any other item.  The per-query pruning bound (tc_bound) is therefore already tight — every query's closest
// lists have been scanned — when the bulk of the work starts, and the epilogue's insert path is rarely taken.
// Probes of empty lists (e.g. lists owned by another shard) are dropped here.
__global__ void count_probes_kernel(const uint32_t* __restrict__ probes, int64_t total, int n_probes, int probe_ld, int near_ranks,
                                    const int64_t* __restrict__ list_offsets, uint32_t* __restrict__ counts)
{
  int64_t t = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  if (t >= total) return;
  uint32_t l = probes[(t / n_probes) * probe_ld + t % n_probes];
  if (l != 0xffffffffu && list_offsets[l + 1] > list_offsets[l])
    atomicAdd(&counts[2 * l + (static_cast<int>(t % n_probes) < near_ranks ? 0 : 1)], 1u);
}

// single CTA: exclusive scans over lists of (a) pair counts, (b) "has a first item", (c) further items ceil(cnt/group) - 1
__global__ void __launch_bounds__(1024) scan_lists_kernel(const uint32_t* __restrict__ counts, int64_t n_lists, uint32_t group,
                                                           uint32_t* __restrict__ pair_off, uint32_t* __restrict__ first_off,
                                                           uint32_t* __restrict__ rest_off, int* __restrict__ n_items,
                                                           uint32_t* __restrict__ cursor)
{
  __shared__ uint32_t s_pairs[1024], s_first[1024], s_rest[1024];
  __shared__ uint32_t run_pairs, run_first, run_rest;
  if (threadIdx.x == 0) { run_pairs = 0; run_first = 0; run_rest = 0; }
  __syncthreads();
  for (int64_t base = 0; base < n_lists; base += 1024) {
    int64_t l   = base + threadIdx.x;
    uint32_t c0 = l < n_lists ? counts[2 * l] : 0;
    uint32_t c  = c0 + (l < n_lists ? counts[2 * l + 1] : 0);
    uint32_t f  = c > 0 ? 1u : 0u;
    uint32_t g  = c > 0 ? (c + group - 1) / group - 1 : 0u;
    s_pairs[threadIdx.x] = c;
    s_first[threadIdx.x] = f;
    s_rest[threadIdx.x]  = g;
    __syncthreads();
    for (int o = 1; o < 1024; o <<= 1) {
      uint32_t a = 0, b = 0, d = 0;
      if (threadIdx.x >= o) { a = s_pairs[threadIdx.x - o]; b = s_first[threadIdx.x - o]; d = s_rest[threadIdx.x - o]; }
      __syncthreads();
      s_pairs[threadIdx.x] += a;
      s_first[threadIdx.x] += b;
      s_rest[threadIdx.x]  += d;
      __syncthreads();
    }
    if (l < n_lists) {
      pair_off[2 * l]     = run_pairs + s_pairs[threadIdx.x] - c;
      pair_off[2 * l + 1] = run_pairs + s_pairs[threadIdx.x] - c + c0;
      first_off[l]        = run_first + s_first[threadIdx.x] - f;
      rest_off[l]         = run_rest + s_rest[threadIdx.x] - g;
      cursor[2 * l]       = 0;
      cursor[2 * l + 1]   = 0;
    }
    __syncthreads();
    if (threadIdx.x == 1023) { run_pairs += s_pairs[1023]; run_first += s_first[1023]; run_rest += s_rest[1023]; }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    n_items[0] = static_cast<int>(run_first + run_rest);
    n_items[1] = static_cast<int>(run_pairs);
    n_items[2] = static_cast<int>(run_first);
  }
}

__global__ void scatter_probes_kernel(const uint32_t* __restrict__ probes, int64_t total, int n_probes, int probe_ld, int near_ranks,
                                      const int64_t* __restrict__ list_offsets, const uint32_t* __restrict__ pair_off,
                                      uint32_t* __restrict__ cursor, uint32_t* __restrict__ slot_of,
                                      uint32_t* __restrict__ pair_query, uint32_t* __restrict__ pair_list)
{
  int64_t t = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  if (t >= total) return;
  uint32_t l = probes[(t / n_probes) * probe_ld + t % n_probes];
  if (l == 0xffffffffu || list_offsets[l + 1] <= list_offsets[l]) { slot_of[t] = 0xffffffffu; return; }
  const uint32_t b = 2 * l + (static_cast<int>(t % n_probes) < near_ranks ? 0 : 1);
  uint32_t slot    = pair_off[b] + atomicAdd(&cursor[b], 1u);
  slot_of[t]       = slot;
  pair_query[slot] = static_cast<uint32_t>(t / n_probes);
  pair_list[slot]  = l;
}

__global__ void make_list_items_kernel(const uint32_t* __restrict__ counts, const uint32_t* __restrict__ pair_off,
                                       const uint32_t* __restrict__ first_off, const uint32_t* __restrict__ rest_off,
                                       const int* __restrict__ n_items, const int64_t* __restrict__ list_offsets,
                                       int64_t n_lists, int KC, uint32_t max_tiles, uint32_t group, tc_item* __restrict__ items)
{
  int64_t l = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  if (l >= n_lists) return;
  uint32_t c = counts[2 * l] + counts[2 * l + 1];
  if (c == 0) return;
  const uint32_t b_row0  = static_cast<uint32_t>(list_offsets[l]);
  const uint32_t n_tiles = min(max_tiles, static_cast<uint32_t>((list_offsets[l + 1] - list_offsets[l]) / 128));
  const uint32_t n_first = static_cast<uint32_t>(n_items[2]);
  uint32_t g = (c + group - 1) / group;
  for (uint32_t j = 0; j < g; ++j) {
    tc_item it;
    it.a_row0     = pair_off[2 * l] + j * group;
    it.b_row0     = b_row0;
    it.n_tiles    = n_tiles;
    it.valid_rows = min(group, c - j * group);
    it.out_off    = static_cast<uint64_t>(it.a_row0) * KC;
    items[j == 0 ? first_off[l] : n_first + rest_off[l] + (j - 1)] = it;
  }
}

__global__ void gather_rows_kernel(const uint4* __restrict__ src, const uint32_t* __restrict__ pair_query,
                                   const int* __restrict__ n_live, int64_t rows_total, int vec_per_row, uint4* __restrict__ dst)
{
  int64_t t = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  if (t >= rows_total * vec_per_row) return;
  int64_t r = t / vec_per_row;
  int v     = static_cast<int>(t % vec_per_row);
  uint4 val = make_uint4(0, 0, 0, 0);
  if (r < *n_live) val = src[static_cast<int64_t>(pair_query[r]) * vec_per_row + v];
  dst[t] = val;
}

__global__ void gather_cands_kernel(const float* __restrict__ cs, const uint32_t* __restrict__ cp,
                                    const uint32_t* __restrict__ slot_of, int64_t total /*nq*n_probes*KC*/, int KC,
                                    float* __restrict__ out_score, uint32_t* __restrict__ out_pos)
{
  int64_t t = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  if (t >= total) return;
  int64_t pair = t / KC;
  int c        = static_cast<int>(t % KC);
  uint32_t slot = slot_of[pair];
  float s      = INFINITY;
  uint32_t p   = 0xffffffffu;
  if (slot != 0xffffffffu) {
    s = cs[static_cast<int64_t>(slot) * KC + c];
    p = cp[static_cast<int64_t>(slot) * KC + c];
  }
  out_score[t] = s;
  out_pos[t]   = p;
}

// ---- per-query merge of the probes' candidate lists ------------------------------------------
// One CTA per query.  The scan left, for every (query, probe) pair, KCW candidates (score, position) and — shared by all
// pairs of the query — an upper bound B on the query's k-th best value (tc_bound).  Every candidate that can be among the k
// best satisfies value <= B, and at least k candidates do (the list that published B), so: filter by B into shared memory
// (typically a few dozen survivors out of n_probes * KCW), sort those, emit the k best.  Replaces a gather of all
// candidates into a [nq, n_probes * KCW] matrix followed by a radix select over it.
__device__ __forceinline__ uint32_t order_key(float f)
{
  uint32_t u = __float_as_uint(f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float order_key_inv(uint32_t k)
{
  return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
}

constexpr int kMergeThreads = 256;
constexpr int kMergeCap     = 1024;

__global__ void __launch_bounds__(kMergeThreads)
merge_pairs_kernel(const float* __restrict__ cs, const uint32_t* __restrict__ cp, const uint32_t* __restrict__ slot_of,
                   const float* __restrict__ add, float scale, const int* __restrict__ bound_keys, int n_probes, int KCW,
                   int k, float* __restrict__ out_val, uint32_t* __restrict__ out_pos)
{
  __shared__ unsigned long long surv[kMergeCap];  // (order key << 32 | position)
  __shared__ unsigned long long red[kMergeThreads / 32];
  __shared__ int count;
  const int64_t q = blockIdx.x;
  if (threadIdx.x == 0) count = 0;
  __syncthreads();
  float bnd = INFINITY;
  if (bound_keys) {
    const int kb = bound_keys[q];
    bnd          = __int_as_float(kb >= 0 ? kb : kb ^ 0x7fffffff);
  }
  const int total          = n_probes * KCW;
  const uint32_t* my_slots = slot_of + q * n_probes;
  auto value_of = [&](int e, uint32_t& pos) -> float {  // candidate e of this query (FLT_MAX / 0xffffffff when empty)
    const int p         = e / KCW;
    const int c         = e - p * KCW;
    const uint32_t slot = my_slots[p];
    pos                 = 0xffffffffu;
    if (slot == 0xffffffffu) return FLT_MAX;
    pos = cp[static_cast<int64_t>(slot) * KCW + c];
    if (pos == 0xffffffffu) return FLT_MAX;
    return __fmaf_rn(scale, cs[static_cast<int64_t>(slot) * KCW + c], add ? add[slot] : 0.f);
  };
  // filter: four independent candidates per thread and trip keep the dependent slot -> position/score loads overlapped
  for (int e0 = threadIdx.x; e0 < total; e0 += 4 * kMergeThreads) {
    uint32_t slot[4], pos[4];
    float sc[4], ad[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int e = e0 + u * kMergeThreads;
      slot[u]     = e < total ? my_slots[e / KCW] : 0xffffffffu;
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int e = e0 + u * kMergeThreads;
      const int c = e % KCW;
      pos[u] = 0xffffffffu; sc[u] = 0.f; ad[u] = 0.f;
      if (slot[u] != 0xffffffffu) {
        pos[u] = cp[static_cast<int64_t>(slot[u]) * KCW + c];
        sc[u]  = cs[static_cast<int64_t>(slot[u]) * KCW + c];
        ad[u]  = add ? add[slot[u]] : 0.f;
      }
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      if (pos[u] == 0xffffffffu) continue;
      const float v = __fmaf_rn(scale, sc[u], ad[u]);
      if (v <= bnd) {
        const int at = atomicAdd(&count, 1);
        if (at < kMergeCap) surv[at] = (static_cast<unsigned long long>(order_key(v)) << 32) | pos[u];
      }
    }
  }
  __syncthreads();
  const int n = count;
  if (n <= kMergeCap) {
    int n2 = 1;
    while (n2 < n) n2 <<= 1;
    for (int i = n + threadIdx.x; i < n2; i += blockDim.x) surv[i] = ~0ull;
    __syncthreads();
    for (int size = 2; size <= n2; size <<= 1) {
      for (int stride = size >> 1; stride > 0; stride >>= 1) {
        for (int i = threadIdx.x; i < n2 / 2; i += blockDim.x) {
          const int lo = (i / stride) * stride * 2 + (i % stride);
          const int hi = lo + stride;
          const bool up = ((lo & size) == 0);
          const unsigned long long a = surv[lo], b = surv[hi];
          if ((a > b) == up) { surv[lo] = b; surv[hi] = a; }
        }
        __syncthreads();
      }
    }
    for (int j = threadIdx.x; j < k; j += blockDim.x) {
      float v      = FLT_MAX;
      uint32_t pos = 0xffffffffu;
      if (j < n) {
        v   = order_key_inv(static_cast<uint32_t>(surv[j] >> 32));
        pos = static_cast<uint32_t>(surv[j] & 0xffffffffu);
      }
      out_val[q * k + j] = v;
      out_pos[q * k + j] = pos;
    }
    return;
  }
  // More survivors than the buffer holds (no usable bound, or massive ties at it): k rounds of "smallest key above the
  // previous one" over all candidates.  Slow, but only for the rare query that gets here.
  unsigned long long last = 0;
  bool first = true;
  for (int j = 0; j < k; ++j) {
    unsigned long long best = ~0ull;
    for (int e = threadIdx.x; e < total; e += blockDim.x) {
      uint32_t pos;
      const float v = value_of(e, pos);
      if (pos == 0xffffffffu) continue;
      const unsigned long long key = (static_cast<unsigned long long>(order_key(v)) << 32) | pos;
      if ((first || key > last) && key < best) best = key;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const unsigned long long other = __shfl_xor_sync(0xffffffffu, best, o);
      best = other < best ? other : best;
    }
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = best;
    __syncthreads();
    best = red[0];
    for (int w = 1; w < kMergeThreads / 32; ++w) best = red[w] < best ? red[w] : best;
    __syncthreads();
    if (threadIdx.x == 0) {
      const bool have    = best != ~0ull;
      out_val[q * k + j] = have ? order_key_inv(static_cast<uint32_t>(best >> 32)) : FLT_MAX;
      out_pos[q * k + j] = have ? static_cast<uint32_t>(best & 0xffffffffu) : 0xffffffffu;
    }
    if (best == ~0ull) {  // exhausted: fill the rest
      for (int r = j + 1 + threadIdx.x; r < k; r += blockDim.x) { out_val[q * k + r] = FLT_MAX; out_pos[q * k + r] = 0xffffffffu; }
      return;
    }
    last  = best;
    first = false;
  }
}

// ---- k-means ---------------------------------------------------------------------------------
__global__ void strided_init_kernel(const float* __restrict__ x, int64_t n, int d, int k, float* __restrict__ centers)
{
  int64_t t = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  if (t >= static_cast<int64_t>(k) * d) return;
  int64_t c   = t / d;
  int64_t row = (c * n) / k;  // evenly spaced rows
  centers[t]  = x[row * d + (t % d)];
}

// one block per cluster: thread (column j, row lane r) sums the member rows r, r + R, ... in row order, and the R partial
// sums are added in lane order, so the result does not depend on scheduling (same input, same centres, run after run)
__global__ void segment_centers_kernel(const float* __restrict__ x, int d, int dp, const uint32_t* __restrict__ order,
                                       const int64_t* __restrict__ start, const float* __restrict__ weights,
                                       float* __restrict__ sums, float* __restrict__ counts, float* __restrict__ centers)
{
  extern __shared__ float part[];  // [R][dp] column partials, then [R] weight partials
  const int64_t l = blockIdx.x;
  const int j = threadIdx.x % dp, r = threadIdx.x / dp, R = blockDim.x / dp;
  float acc = 0.f, wacc = 0.f;
  for (int64_t p = start[l] + r; p < start[l + 1]; p += R) {
    const int64_t row = order[p];
    const float w     = weights ? weights[row] : 1.0f;
    if (j < d) acc += w * x[row * d + j];
    wacc += w;
  }
  part[r * dp + j] = acc;
  if (j == 0) part[R * dp + r] = wacc;
  __syncthreads();
  if (r != 0) return;
  float sum = 0.f, cnt = 0.f;
  for (int q = 0; q < R; ++q) { sum += part[q * dp + j]; cnt += part[R * dp + q]; }
  if (j < d) {
    sums[l * d + j] = sum;
    if (cnt > 0.f) centers[l * d + j] = sum / cnt;
  }
  if (j == 0) counts[l] = cnt;
}

__device__ __forceinline__ uint64_t mix64(uint64_t z)
{
  z += 0x9e3779b97f4a7c15ull;
  z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ull;
  z = (z ^ (z >> 27)) * 0x94d049bb133111ebull;
  return z ^ (z >> 31);
}

// one thread per cluster: small clusters jump onto a member of a large cluster
__global__ void reseed_small_kernel(const float* __restrict__ x, int64_t n, int d, const uint32_t* __restrict__ labels,
                                    const float* __restrict__ counts, int k, float avg, int iter, float* __restrict__ centers,
                                    int* __restrict__ n_reseeded)
{
  int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= k) return;
  if (counts[c] >= 0.25f * avg) return;
  for (int tries = 0; tries < 64; ++tries) {
    uint64_t h  = mix64((static_cast<uint64_t>(iter) << 40) ^ (static_cast<uint64_t>(c) << 8) ^ tries);
    int64_t row = static_cast<int64_t>(h % static_cast<uint64_t>(n));
    if (counts[labels[row]] >= avg) {
      // move most of the way to the donor point; keep a little of the donor's centre to break symmetry
      const float* donor_c = centers + static_cast<int64_t>(labels[row]) * d;
      for (int j = 0; j < d; ++j) centers[static_cast<int64_t>(c) * d + j] = 0.75f * x[row * d + j] + 0.25f * donor_c[j];
      atomicAdd(n_reseeded, 1);
      return;
    }
  }
}

__global__ void sum_scores_kernel(const float* __restrict__ s, const float* __restrict__ xn, int64_t n, double* __restrict__ out)
{
  double acc = 0;
  for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    float dist = fmaf(2.0f, s[i], xn[i]);  // |x|^2 + 2 (|c|^2/2 - x.c)
    acc += dist > 0.f ? dist : 0.0;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0) atomicAdd(out, acc);
}

}  // namespace

void tc_rows::build(cudaStream_t s, const float* x, int64_t n_, int d_, const float* xn, bool with_lo, const float* row_scale)
{
  n = n_; d = d_;
  Kp       = tc_pad_k(d);
  rows_pad = tc_pad_rows(std::max<int64_t>(n, 1));
  hi.alloc(static_cast<size_t>(rows_pad) * Kp);
  if (with_lo) lo.alloc(static_cast<size_t>(rows_pad) * Kp); else lo.release();
  hx.alloc(static_cast<size_t>(rows_pad) * 16);
  tc_split_planes(s, x, n, d, d, Kp, hi.data(), with_lo ? lo.data() : nullptr, rows_pad, row_scale);
  tc_half_norms(s, xn, n, rows_pad, hx.data());
}

void tc_rows_tmp::build(cudaStream_t s, const float* x, int64_t n_, int d_, bool with_lo, int64_t extra_pad_rows,
                        const float* row_scale)
{
  n = n_; d = d_;
  Kp       = tc_pad_k(d);
  rows_pad = tc_pad_rows(std::max<int64_t>(n, 1)) + extra_pad_rows;
  hi.alloc(static_cast<size_t>(rows_pad) * Kp, s);
  if (with_lo) lo.alloc(static_cast<size_t>(rows_pad) * Kp, s);
  tc_split_planes(s, x, n, d, d, Kp, hi.data(), with_lo ? lo.data() : nullptr, rows_pad, row_scale);
}

// Fused coarse search (large n_lists): instead of writing the dense [nq, n_lists] score block (655 MB at 10k x 16384) and
// selecting from it, the scan keeps 32 candidates per (query, centre range, column half) in its epilogue — (query tile, centre
// range) items also give the 148 SMs ~2 waves of work where one item per query tile gave 79 CTAs — and a small merge ranks
// the 2 * splits * 32 candidates per query.  Exact (same scores, same (score, id) order as the dense select) whenever the merge
// kernel's certificate holds for every query of the batch; returns false when the dense path has to run (one host read of
// the flag count per search).
static bool coarse_select_fused(resources* res, const tc_rows_tmp& q, const tc_rows& centers, int n_probes, uint32_t* probes,
                                float* probe_scores)
{
  const char* env = getenv("CUVS_B200_COARSE_FUSED");  // read per call (A/B inside one process): "0" = dense path
  if (env != nullptr && env[0] == '0') return false;
  const int KC = 32;
  if (n_probes > 2 * KC || centers.n < 4096) return false;
  auto s               = res->stream;
  const int64_t nq_pad = tc_pad_rows(q.n);
  const int m_tiles    = static_cast<int>(nq_pad / 128);
  const int64_t b_tiles = centers.rows_pad / 128;
  const int sms        = res->sm_count ? res->sm_count : 148;
  // enough items for ~2 waves of CTAs, and enough lists that the n_probes best are spread thin (>= 4 n_probes candidates:
  // with only n_probes candidates the certificate could never hold and every batch would pay for both paths)
  int splits = std::max((2 * sms + m_tiles - 1) / m_tiles, (n_probes + 15) / 16);
  splits     = static_cast<int>(std::min<int64_t>(splits, std::min<int64_t>(16, b_tiles / 4)));
  splits     = std::max(splits, 1);
  const int KCW = KC * tc_lists_per_item();
  const int W   = splits * KCW;
  if (W > kCoarseMaxW || W < 4 * n_probes) return false;
  const int n_items = m_tiles * splits;
  dbuf<tc_item> items(static_cast<size_t>(n_items), s);
  count_launch();
  split_items_kernel<<<blocks_for(n_items, 128), 128, 0, s>>>(items.data(), m_tiles, splits, q.n, static_cast<uint32_t>(b_tiles), KCW);
  B2_CUDA(cudaGetLastError());
  dbuf<float> cs(static_cast<size_t>(nq_pad) * W, s);
  dbuf<uint32_t> cp(static_cast<size_t>(nq_pad) * W, s);
  dbuf<int> bkeys(static_cast<size_t>(nq_pad) + 1, s);
  B2_CUDA(cudaMemsetAsync(bkeys.data(), tc_bound_init_byte, sizeof(int) * nq_pad, s));
  int* n_flagged = bkeys.data() + nq_pad;
  B2_CUDA(cudaMemsetAsync(n_flagged, 0, sizeof(int), s));
  tc_bound bnd;
  bnd.keys = bkeys.data();
  bnd.kth  = 0;  // lists prune at, and publish, their last (32nd) entry: that is what the merge's certificate reasons about
  const bool three = q.lo.data() != nullptr && centers.lo.data() != nullptr;
  tc_scan_topk(s, res->device, q.hi.data(), q.lo.data(), q.rows_pad, centers.hi.data(), centers.lo.data(), centers.rows_pad,
               q.Kp, centers.hx.data(), items.data(), n_items, nullptr, KC, three ? 3 : 1, cs.data(), cp.data(), W, &bnd);
  count_launch();
  {
    const unsigned grid = static_cast<unsigned>(q.n);
    const size_t smem   = static_cast<size_t>(W) * 8;
    const int per       = (W + kCoarseMergeThreads - 1) / kCoarseMergeThreads;
#define B2_CM(E_) coarse_merge_kernel<E_><<<grid, kCoarseMergeThreads, smem, s>>>(cs.data(), cp.data(), W, KC, n_probes, probes, probe_scores, n_flagged)
    if (per <= 1) B2_CM(1);
    else if (per <= 2) B2_CM(2);
    else if (per <= 4) B2_CM(4);
    else B2_CM(8);
#undef B2_CM
  }
  B2_CUDA(cudaGetLastError());
  int flagged = 0;
  B2_CUDA(cudaMemcpyAsync(&flagged, n_flagged, sizeof(int), cudaMemcpyDeviceToHost, s));
  B2_CUDA(cudaStreamSynchronize(s));
  return flagged == 0;
}

void coarse_select(resources* res, const tc_rows_tmp& q, const tc_rows& centers, int n_probes, uint32_t* probes,
                   float* probe_scores)
{
  auto s = res->stream;
  if (q.n == 0) return;
  B2_EXPECTS(q.Kp == centers.Kp, "coarse_select: dimension mismatch");
  dbuf<float> tmp_scores;
  if (!probe_scores) { tmp_scores.alloc(static_cast<size_t>(q.n) * n_probes, s); probe_scores = tmp_scores.data(); }
  if (coarse_select_fused(res, q, centers, n_probes, probes, probe_scores)) return;
  const int64_t nq_pad = tc_pad_rows(q.n);
  const int m_tiles    = static_cast<int>(nq_pad / 128);
  const int64_t ld     = centers.rows_pad;
  dbuf<tc_item> items(static_cast<size_t>(m_tiles), s);
  count_launch();
  iota_items_kernel<<<blocks_for(m_tiles, 128), 128, 0, s>>>(items.data(), m_tiles, q.n, static_cast<uint32_t>(ld / 128), ld);
  B2_CUDA(cudaGetLastError());
  dbuf<float> scores(static_cast<size_t>(nq_pad) * ld, s);
  const bool three = q.lo.data() != nullptr && centers.lo.data() != nullptr;
  tc_scan_topk(s, res->device, q.hi.data(), q.lo.data(), q.rows_pad, centers.hi.data(), centers.lo.data(), centers.rows_pad,
               q.Kp, centers.hx.data(), items.data(), m_tiles, nullptr, 0, three ? 3 : 1, scores.data(), nullptr, ld);
  select_k(s, scores.data(), nullptr, IDX_NONE, q.n, centers.n, ld, n_probes, probe_scores, probes, IDX_U32, true);
}

void assign_nearest(resources* res, const __nv_bfloat16* x_hi, const __nv_bfloat16* x_lo, int64_t n, int64_t x_rows_pad,
                    int Kp, const tc_rows& centers, uint32_t* labels, float* scores)
{
  auto s = res->stream;
  if (n == 0) return;
  B2_EXPECTS(Kp == centers.Kp, "assign_nearest: dimension mismatch");
  const int KC         = 16;
  const int lists      = tc_lists_per_item();
  const int KCW        = KC * lists;
  const int64_t chunk  = int64_t(1) << 20;  // rows per launch: bounds the (score,pos) scratch to 256 MiB
  const bool three     = x_lo != nullptr && centers.lo.data() != nullptr;
  dbuf<float> cs(static_cast<size_t>(std::min(chunk, tc_pad_rows(n))) * KCW, s);
  dbuf<uint32_t> cp(static_cast<size_t>(std::min(chunk, tc_pad_rows(n))) * KCW, s);
  dbuf<tc_item> items(static_cast<size_t>(std::min(chunk, tc_pad_rows(n)) / 128), s);
  for (int64_t r0 = 0; r0 < n; r0 += chunk) {
    const int64_t rows = std::min(chunk, n - r0);
    const int m_tiles  = static_cast<int>(tc_pad_rows(rows) / 128);
    count_launch();
    iota_items_kernel<<<blocks_for(m_tiles, 128), 128, 0, s>>>(items.data(), m_tiles, rows,
                                                                static_cast<uint32_t>(centers.rows_pad / 128), KCW);
    B2_CUDA(cudaGetLastError());
    tc_scan_topk(s, res->device, x_hi + r0 * Kp, x_lo ? x_lo + r0 * Kp : nullptr, x_rows_pad - r0, centers.hi.data(),
                 centers.lo.data(), centers.rows_pad, Kp, centers.hx.data(), items.data(), m_tiles, nullptr, KC,
                 three ? 3 : 1, cs.data(), cp.data(), KCW);
    count_launch();
    first_of_rows_kernel<<<blocks_for(rows, 256), 256, 0, s>>>(cp.data(), cs.data(), rows, KC, lists, labels + r0,
                                                               scores ? scores + r0 : nullptr);
    B2_CUDA(cudaGetLastError());
  }
}

void label_rows(resources* res, const tc_rows& centers, const float* x, int64_t n, int d, const float* row_scale, uint32_t* labels)
{
  tc_rows_tmp xp;
  xp.build(res->stream, x, n, d, true, 0, row_scale);
  assign_nearest(res, xp.hi.data(), xp.lo.data(), n, xp.rows_pad, xp.Kp, centers, labels, nullptr);
}

int64_t training_subsample(cudaStream_t s, const float* x, int64_t n, int d, uint32_t n_lists, double fraction, dbuf<float>& out)
{
  // the reference's rule: ivf_flat_build.cuh:430-455
  fraction             = std::min(1.0, std::max(fraction, 0.0));
  int64_t n_train      = std::max<int64_t>(n_lists, std::min<int64_t>(n, static_cast<int64_t>(std::llround(n * fraction))));
  n_train              = std::min<int64_t>(n_train, std::max<int64_t>(static_cast<int64_t>(n_lists) * 1024, 1 << 18));
  n_train              = std::min(n_train, n);
  const int64_t stride = std::max<int64_t>(1, n / n_train);
  n_train              = std::min(n_train, (n + stride - 1) / stride);
  out.alloc(static_cast<size_t>(n_train) * d, s);
  B2_CUDA(cudaMemcpy2DAsync(out.data(), sizeof(float) * d, x, sizeof(float) * d * stride, sizeof(float) * d, n_train,
                            cudaMemcpyDefault, s));
  return n_train;
}

const int64_t* extend_args(resources* res, DLManagedTensor* new_vectors, DLManagedTensor* new_indices, int dim, f32_matrix& v,
                           dbuf<int64_t>& ids_buf)
{
  B2_EXPECTS(new_vectors != nullptr, "new_vectors is null");
  const DLTensor& nv = new_vectors->dl_tensor;
  B2_EXPECTS(dl_is_dataset_dtype(nv), "Unsupported new_vectors DLtensor dtype: %d and bits: %d", nv.dtype.code, nv.dtype.bits);
  widen_to_f32(res, nv, v);
  B2_EXPECTS(dl_is(v.t, kDLFloat, 32) && v.t.ndim == 2 && v.t.shape[1] == dim && dl_is_c_contiguous(v.t),
             "new_vectors must be [n, dim] row-major");
  if (!new_indices) return nullptr;
  const int64_t n    = v.t.shape[0];
  const DLTensor& it = new_indices->dl_tensor;
  B2_EXPECTS(dl_is(it, kDLInt, 64) && it.shape[0] == n, "new_indices must be int64 [n]");
  if (dl_is_device(it) && it.device.device_type != kDLCUDAHost) return dl_ptr<int64_t>(it);
  ids_buf.alloc(static_cast<size_t>(n), res->stream);
  B2_CUDA(cudaMemcpyAsync(ids_buf.data(), dl_ptr<int64_t>(it), sizeof(int64_t) * n, cudaMemcpyHostToDevice, res->stream));
  return ids_buf.data();
}

void bucket_probes(resources* res, const uint32_t* probes, int64_t nq, int n_probes, int64_t n_lists,
                   const int64_t* list_offsets_dev, int KC, probe_buckets& out, int probe_ld, uint32_t max_tiles, int group)
{
  B2_EXPECTS(group >= 8 && group <= 128, "bucket_probes: group must be within [8, 128]");
  if (probe_ld <= 0) probe_ld = n_probes;
  auto s              = res->stream;
  const int64_t total = nq * n_probes;
  out.n_pairs         = total;
  out.max_items       = static_cast<int>(total / group + n_lists + 1);
  out.slot_of.alloc(static_cast<size_t>(total), s);
  out.pair_query.alloc(static_cast<size_t>(total), s);
  out.pair_list.alloc(static_cast<size_t>(total), s);
  out.items.alloc(static_cast<size_t>(out.max_items), s);
  out.n_items.alloc(4, s);
  const int near_ranks = std::max(1, n_probes / 8);
  dbuf<uint32_t> counts(static_cast<size_t>(2 * n_lists), s), pair_off(static_cast<size_t>(2 * n_lists), s),
    first_off(static_cast<size_t>(n_lists), s), rest_off(static_cast<size_t>(n_lists), s), cursor(static_cast<size_t>(2 * n_lists), s);
  B2_CUDA(cudaMemsetAsync(counts.data(), 0, sizeof(uint32_t) * 2 * n_lists, s));
  count_launch(4);
  count_probes_kernel<<<blocks_for(total, 256), 256, 0, s>>>(probes, total, n_probes, probe_ld, near_ranks, list_offsets_dev, counts.data());
  scan_lists_kernel<<<1, 1024, 0, s>>>(counts.data(), n_lists, static_cast<uint32_t>(group), pair_off.data(), first_off.data(), rest_off.data(), out.n_items.data(),
                                       cursor.data());
  scatter_probes_kernel<<<blocks_for(total, 256), 256, 0, s>>>(probes, total, n_probes, probe_ld, near_ranks, list_offsets_dev, pair_off.data(),
                                                                cursor.data(), out.slot_of.data(), out.pair_query.data(),
                                                                out.pair_list.data());
  make_list_items_kernel<<<blocks_for(n_lists, 128), 128, 0, s>>>(counts.data(), pair_off.data(), first_off.data(), rest_off.data(),
                                                                   out.n_items.data(), list_offsets_dev, n_lists, KC, max_tiles, static_cast<uint32_t>(group), out.items.data());
  B2_CUDA(cudaGetLastError());
}

void gather_rows_bf16(cudaStream_t s, const __nv_bfloat16* src, const uint32_t* pair_query, const int* n_live, int64_t rows_total,
                      int Kp, __nv_bfloat16* dst)
{
  const int vec = Kp * 2 / 16;
  count_launch();
  gather_rows_kernel<<<blocks_for(rows_total * vec, 256), 256, 0, s>>>(reinterpret_cast<const uint4*>(src), pair_query, n_live,
                                                                        rows_total, vec, reinterpret_cast<uint4*>(dst));
  B2_CUDA(cudaGetLastError());
}

void gather_probe_candidates(cudaStream_t s, const float* cs, const uint32_t* cp, const uint32_t* slot_of, int64_t nq,
                             int n_probes, int KC, float* out_score, uint32_t* out_pos)
{
  const int64_t total = nq * n_probes * KC;
  if (total == 0) return;
  count_launch();
  gather_cands_kernel<<<blocks_for(total, 256), 256, 0, s>>>(cs, cp, slot_of, total, KC, out_score, out_pos);
  B2_CUDA(cudaGetLastError());
}

bool merge_probe_candidates(cudaStream_t s, const float* cs, const uint32_t* cp, const uint32_t* slot_of, const float* add,
                            float scale, const int* bound_keys, int64_t nq, int n_probes, int KCW, int k, float* out_val,
                            uint32_t* out_pos)
{
  if (nq == 0) return true;
  // without a bound nothing is filtered: the generic gather + radix select is the better tool then
  if (bound_keys == nullptr && static_cast<int64_t>(n_probes) * KCW > kMergeCap) return false;
  count_launch();
  merge_pairs_kernel<<<static_cast<unsigned>(nq), kMergeThreads, 0, s>>>(cs, cp, slot_of, add, scale, bound_keys, n_probes, KCW, k,
                                                                          out_val, out_pos);
  B2_CUDA(cudaGetLastError());
  return true;
}

void update_centers(cudaStream_t s, const float* x, int64_t n, int d, const uint32_t* labels, const float* weights, int k,
                    float* centers, float* sums_ws, float* counts_ws)
{
  B2_EXPECTS(d >= 1 && d <= 1024, "update_centers: dim %d is out of range", d);
  dbuf<uint32_t> keys(static_cast<size_t>(n), s), order;
  B2_CUDA(cudaMemcpyAsync(keys.data(), labels, sizeof(uint32_t) * n, cudaMemcpyDeviceToDevice, s));
  iota_u32(s, order, n);
  dbuf<int64_t> start;
  group_by_key(s, keys, order, k, start);
  const int dp = (d + 31) / 32 * 32, R = std::max(1, 512 / dp);
  count_launch();
  segment_centers_kernel<<<static_cast<unsigned>(k), R * dp, sizeof(float) * (R * dp + R), s>>>(x, d, dp, order.data(), start.data(),
                                                                                                 weights, sums_ws, counts_ws, centers);
  B2_CUDA(cudaGetLastError());
}

void kmeans_train(resources* res, const float* x, int64_t n, int d, int k, int n_iters, float* centers, bool init_from_data,
                  bool balance, double* inertia, int* iters_done, double tol)
{
  auto s = res->stream;
  B2_EXPECTS(n >= 1 && k >= 1, "kmeans: empty input");
  B2_EXPECTS(tc_supported(res->device, d), "kmeans: dim %d is not supported by the tensor-core assignment kernel yet (<= 128)", d);
  if (init_from_data) {
    count_launch();
    strided_init_kernel<<<blocks_for(static_cast<int64_t>(k) * d, 256), 256, 0, s>>>(x, n, d, k, centers);
    B2_CUDA(cudaGetLastError());
  }
  // data-side planes (the dataset plays the "query" role of the scan)
  tc_rows_tmp xp;
  xp.build(s, x, n, d, true);
  dbuf<float> xn(static_cast<size_t>(n), s), cn(static_cast<size_t>(k), s), sums(static_cast<size_t>(k) * d, s),
    counts(static_cast<size_t>(k), s), scores(static_cast<size_t>(n), s);
  dbuf<uint32_t> labels(static_cast<size_t>(n), s);
  dbuf<double> acc(1, s);
  dbuf<int> n_reseeded(1, s);
  row_norms(s, x, n, d, d, xn.data());
  tc_rows cp;
  double prev = -1.0;
  int it      = 0;
  for (; it < std::max(n_iters, 1); ++it) {
    row_norms(s, centers, k, d, d, cn.data());
    cp.build(s, centers, k, d, cn.data(), true);
    assign_nearest(res, xp.hi.data(), xp.lo.data(), n, xp.rows_pad, xp.Kp, cp, labels.data(), scores.data());
    if (n_iters == 0) break;  // assignment only
    update_centers(s, x, n, d, labels.data(), nullptr, k, centers, sums.data(), counts.data());
    if (balance && k > 1) {
      B2_CUDA(cudaMemsetAsync(n_reseeded.data(), 0, sizeof(int), s));
      count_launch();
      reseed_small_kernel<<<blocks_for(k, 128), 128, 0, s>>>(x, n, d, labels.data(), counts.data(), k,
                                                              static_cast<float>(n) / k, it, centers, n_reseeded.data());
      B2_CUDA(cudaGetLastError());
    }
    if (tol > 0.0) {
      B2_CUDA(cudaMemsetAsync(acc.data(), 0, sizeof(double), s));
      count_launch();
      sum_scores_kernel<<<256, 256, 0, s>>>(scores.data(), xn.data(), n, acc.data());
      double cur = 0;
      B2_CUDA(cudaMemcpyAsync(&cur, acc.data(), sizeof(double), cudaMemcpyDeviceToHost, s));
      B2_CUDA(cudaStreamSynchronize(s));
      if (prev >= 0 && std::abs(prev - cur) <= tol * std::max(prev, 1e-30)) { prev = cur; ++it; break; }
      prev = cur;
    }
  }
  if (iters_done) *iters_done = it;
  if (inertia) {
    // inertia of the returned centres
    row_norms(s, centers, k, d, d, cn.data());
    cp.build(s, centers, k, d, cn.data(), true);
    assign_nearest(res, xp.hi.data(), xp.lo.data(), n, xp.rows_pad, xp.Kp, cp, labels.data(), scores.data());
    B2_CUDA(cudaMemsetAsync(acc.data(), 0, sizeof(double), s));
    count_launch();
    sum_scores_kernel<<<256, 256, 0, s>>>(scores.data(), xn.data(), n, acc.data());
    B2_CUDA(cudaMemcpyAsync(inertia, acc.data(), sizeof(double), cudaMemcpyDeviceToHost, s));
    B2_CUDA(cudaStreamSynchronize(s));
  }
}

}  // namespace b200
