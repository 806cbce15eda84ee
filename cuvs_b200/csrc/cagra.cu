// CAGRA: graph-walk search kernel, index from (graph, dataset), simple graph build, C boundary.
//
// Reference path being replaced (SURVEY §8a rows a14-a17):
//   index                 cpp/include/cuvs/neighbors/cagra.hpp:398-890
//   plan / parameters     cpp/src/neighbors/detail/cagra/search_plan.cuh:99-428
//   single-CTA kernel     cpp/src/neighbors/detail/cagra/jit_lto_kernels/search_single_cta_jit.cuh:55-451
//   seeds / children      .../device_common_jit.cuh:36-179     hash   .../hashmap.hpp:23-145
//   parent pickup / sort  .../search_single_cta_device_helpers.cuh:97-137, 277-623
//   C wrapper             c/src/neighbors/cagra.cpp
//
// B200 formulation (DESIGN.md §6).  The walk is a chain of ~70 dependent iterations per query, each a
// 256-byte adjacency read, ~64 random 384-byte vector gathers, a dedup against a small hash and a
// 128-way sort: it is bound by memory LATENCY, so throughput comes from the number of independent
// walks in flight, not from one walk's bandwidth.  The reference spends a whole CTA (>= 64 threads,
// ~6 __syncthreads per iteration) per query; here ONE WARP owns a query end to end:
//   * the internal top-k list and the candidate list live in registers (4 x 64-bit keys per lane),
//     sorted by a shuffle-only bitonic network — no shared-memory round trips, no block barriers;
//   * the visited set is the reference's small open-addressing hash, per warp in shared memory;
//   * distances use teams of 8 lanes with 128-bit loads (384 B row = 3 x 16 B per lane), several
//     candidates' loads issued back to back for memory-level parallelism;
//   * 16 warps per CTA and ~2.5 KB of shared memory per warp keep 48-64 walks resident per SM
//     (~8-9k concurrent walks per GPU), which is what hides the DRAM latency.
// Semantics (seeds, hash, parent selection, termination) follow the reference exactly and are
// restated on the CPU in oracle/oracle.c::oracle_cagra_search.
#include "common.hpp"
#include <cuda_fp16.h>
#include <cuvs_b200/ext.h>
#include <library_types.h>

#include "npy_io.hpp"
#include "ptx_sm100.cuh"
#include "exact.cuh"
#include "ivf_lists.cuh"
#include "select_k.cuh"
#include "timing.hpp"

#include <cuvs/neighbors/brute_force.h>
#include <cuvs/neighbors/cagra.h>
#include <cuvs/neighbors/ivf_flat.h>

#include <algorithm>
#include <cfloat>
#include <cstring>
#include <fstream>
#include <memory>
#include <vector>

namespace b200 {

struct cagra_index {
  int device              = 0;
  cuvsDistanceType metric = L2Expanded;
  int64_t n               = 0;
  int dim                 = 0;
  int ld                  = 0;  // row pitch in floats (rows padded to 16 bytes, cagra.hpp:610)
  int degree              = 0;
  const float* data       = nullptr;
  const uint32_t* graph   = nullptr;
  owned<float> data_own;
  owned<uint32_t> graph_own;
  // Optional fp16 copy of the vectors for the walk (cuvsB200CagraSetWalkPrecision): the walk is bound by random row
  // gathers from HBM, half-width rows halve its bytes; the returned neighbours are re-ranked with the fp32 rows.
  owned<__half> data16;
  int ld16 = 0;  // row pitch in halves (rows padded to 16 bytes)
};

namespace {

constexpr uint32_t kInvalid = 0xffffffffu;
constexpr uint32_t kMsb     = 0x80000000u;

__host__ __device__ __forceinline__ uint64_t xorshift64(uint64_t u)
{
  u ^= u >> 12;
  u ^= u << 25;
  u ^= u >> 27;
  return u * 0x2545F4914F6CDD1DULL;
}

// hashmap.hpp:37-73 — open addressing; returns 1 when newly inserted.  The reference file carries two probing schemes and
// compiles the linear one (#define HASHMAP_LINEAR_PROBING: index = (key ^ (key >> bitlen)) & mask, stride 1); this is its
// double-hashing branch (hashmap.hpp:52-55).  Both are exact sets while the table is not full (the plan keeps the fill rate
// <= 50 %, search_plan.cuh:256-372), so visited-set semantics — and therefore the walk — do not depend on the choice.
__device__ __forceinline__ uint32_t hash_insert(uint32_t* table, uint32_t bitlen, uint32_t key)
{
  const uint32_t size = 1u << bitlen, mask = size - 1;
  uint32_t index        = key & mask;
  const uint32_t stride = (key >> bitlen) * 2 + 1;
  for (uint32_t i = 0; i < size; ++i) {
    const uint32_t old = atomicCAS(&table[index], kInvalid, key);
    if (old == kInvalid) return 1;
    if (old == key) return 0;
    index = (index + stride) & mask;
  }
  return 0;
}

__device__ __forceinline__ uint32_t dist_key(float d)
{
  uint32_t u = __float_as_uint(d);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float key_dist(uint32_t k)
{
  uint32_t u = (k & 0x80000000u) ? (k & 0x7fffffffu) : ~k;
  return __uint_as_float(u);
}

// Bitonic sort of 32*E 64-bit keys held E per lane, striped (element index i = e*32 + lane), ascending.
template <int E>
__device__ __forceinline__ void warp_bitonic_sort(uint64_t (&k)[E], int lane)
{
  constexpr int N = 32 * E;
#pragma unroll
  for (int size = 2; size <= N; size <<= 1) {
#pragma unroll
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      if (stride >= 32) {
        const int es = stride >> 5;  // partner element offset inside the lane
#pragma unroll
        for (int e = 0; e < E; ++e) {
          if ((e & es) == 0) {
            const int i   = e * 32 + lane;
            const bool up = (i & size) == 0;
            uint64_t a = k[e], b = k[e | es];
            if ((a > b) == up) { k[e] = b; k[e | es] = a; }
          }
        }
      } else {
#pragma unroll
        for (int e = 0; e < E; ++e) {
          const int i        = e * 32 + lane;
          const bool up      = (i & size) == 0;
          const bool lower   = (lane & stride) == 0;
          const uint64_t o   = __shfl_xor_sync(0xffffffffu, k[e], stride);
          const bool take_min = (lower == up);
          k[e] = take_min ? (k[e] < o ? k[e] : o) : (k[e] > o ? k[e] : o);
        }
      }
    }
  }
}

struct cagra_launch {
  const __half* data16;  // non-null: the walk reads these rows (pitch ld16), the final list is re-ranked from `data`
  int ld16;
  const float* data;
  const uint32_t* graph;
  int64_t n;
  int dim, ld, degree;
  const float* queries;
  int64_t nq;
  int metric;  // L2Expanded or InnerProduct
  int k, itopk, search_width, min_iter, max_iter;
  uint32_t hash_bitlen, small_hash_bitlen, reset_interval;
  int num_random_samplings;
  uint64_t rand_xor_mask;
  uint32_t* hash_global;  // used when small_hash_bitlen == 0
  uint32_t* out_idx32;
  int64_t* out_idx64;
  float* out_dist;
  uint32_t* out_iters;
  const uint32_t* keep_bits;  // bitset pre-filter over node ids (bit = 1 keeps), null = none
  int64_t n_bits;
  unsigned long long* work_counter;  // next query index (persistent warps)
  // multi-walker mode (the reference's MULTI_CTA algorithm, search_multi_cta_jit.cuh:56-363): `walkers` warps per query,
  // each with its own 32-entry list and search_width 1, sharing ONE table of traversed parents per query
  int walkers;                  // 0 = single-walker kernel
  uint32_t* traversed;          // [nq << traversed_bitlen], initialised to kInvalid by the host
  uint32_t traversed_bitlen;
  unsigned long long* mc_keys;  // [nq, walkers, 32] every walker's final sorted list (dist_key << 32 | id)
  // > 0: bytes of one walk row (16-byte multiple, 16-byte aligned rows).  As soon as an iteration's fresh children are known,
  // every lane asks the copy engine for its children's rows with ONE cp.async.bulk.prefetch.L2 each (UBLKPF): all <= 64 row
  // gathers of the iteration are in flight at once, and the team loads below (2 rows per team in flight, register-bound at
  // 40 registers / 3 CTAs per SM) find them in L2 instead of paying the HBM latency 8 times in a row.
  uint32_t prefetch_row_bytes;
};

// squared L2 / negative dot between the smem query and a dataset row, computed by a team of 8 lanes
__device__ __forceinline__ float team_distance(const float* __restrict__ row, const float* __restrict__ sq, int dim, int t, bool ip)
{
  float acc = 0.f;
  // 16-byte chunks, chunk c handled by team lane c % 8
  const int n_chunks = dim >> 2;
  for (int c = t; c < n_chunks; c += 8) {
    const float4 x = __ldg(reinterpret_cast<const float4*>(row) + c);
    const float4 q = reinterpret_cast<const float4*>(sq)[c];
    if (ip) {
      acc = fmaf(-q.x, x.x, acc); acc = fmaf(-q.y, x.y, acc); acc = fmaf(-q.z, x.z, acc); acc = fmaf(-q.w, x.w, acc);
    } else {
      float d0 = q.x - x.x, d1 = q.y - x.y, d2 = q.z - x.z, d3 = q.w - x.w;
      acc = fmaf(d0, d0, acc); acc = fmaf(d1, d1, acc); acc = fmaf(d2, d2, acc); acc = fmaf(d3, d3, acc);
    }
  }
  for (int j = (n_chunks << 2) + t; j < dim; j += 8) {  // tail when dim % 4 != 0
    const float x = row[j], q = sq[j];
    if (ip) acc = fmaf(-q, x, acc);
    else { float df = q - x; acc = fmaf(df, df, acc); }
  }
  acc += __shfl_xor_sync(0xffffffffu, acc, 4);
  acc += __shfl_xor_sync(0xffffffffu, acc, 2);
  acc += __shfl_xor_sync(0xffffffffu, acc, 1);
  return acc;
}

__device__ __forceinline__ bool node_kept(const uint32_t* __restrict__ keep_bits, int64_t n_bits, uint32_t id)
{
  return static_cast<int64_t>(id) < n_bits && ((keep_bits[id >> 5] >> (id & 31)) & 1u);
}

// the same over an fp16 row (8 halves per 16-byte chunk), accumulated in fp32
__device__ __forceinline__ float team_distance_h(const __half* __restrict__ row, const float* __restrict__ sq, int dim, int t, bool ip)
{
  float acc = 0.f;
  const int n_chunks = dim >> 3;
  for (int c = t; c < n_chunks; c += 8) {
    const uint4 raw = __ldg(reinterpret_cast<const uint4*>(row) + c);
    const __half2* h = reinterpret_cast<const __half2*>(&raw);
    const float4 q0 = reinterpret_cast<const float4*>(sq)[2 * c], q1 = reinterpret_cast<const float4*>(sq)[2 * c + 1];
    const float2 x0 = __half22float2(h[0]), x1 = __half22float2(h[1]), x2 = __half22float2(h[2]), x3 = __half22float2(h[3]);
    if (ip) {
      acc = fmaf(-q0.x, x0.x, acc); acc = fmaf(-q0.y, x0.y, acc); acc = fmaf(-q0.z, x1.x, acc); acc = fmaf(-q0.w, x1.y, acc);
      acc = fmaf(-q1.x, x2.x, acc); acc = fmaf(-q1.y, x2.y, acc); acc = fmaf(-q1.z, x3.x, acc); acc = fmaf(-q1.w, x3.y, acc);
    } else {
      float d;
      d = q0.x - x0.x; acc = fmaf(d, d, acc); d = q0.y - x0.y; acc = fmaf(d, d, acc);
      d = q0.z - x1.x; acc = fmaf(d, d, acc); d = q0.w - x1.y; acc = fmaf(d, d, acc);
      d = q1.x - x2.x; acc = fmaf(d, d, acc); d = q1.y - x2.y; acc = fmaf(d, d, acc);
      d = q1.z - x3.x; acc = fmaf(d, d, acc); d = q1.w - x3.y; acc = fmaf(d, d, acc);
    }
  }
  for (int j = (n_chunks << 3) + t; j < dim; j += 8) {
    const float x = __half2float(row[j]), q = sq[j];
    if (ip) acc = fmaf(-q, x, acc);
    else { float df = q - x; acc = fmaf(df, df, acc); }
  }
  acc += __shfl_xor_sync(0xffffffffu, acc, 4);
  acc += __shfl_xor_sync(0xffffffffu, acc, 2);
  acc += __shfl_xor_sync(0xffffffffu, acc, 1);
  return acc;
}

// (fields passed by value: taking a reference to the __grid_constant__-less kernel parameter struct would force a local copy)
__device__ __forceinline__ float walk_distance(const __half* data16, int ld16, const float* data, int ld, int dim, uint32_t id,
                                               const float* __restrict__ sq, int t, bool ip)
{
  return data16 ? team_distance_h(data16 + static_cast<int64_t>(id) * ld16, sq, dim, t, ip)
                : team_distance(data + static_cast<int64_t>(id) * ld, sq, dim, t, ip);
}

// EI = itopk / 32, EC = (search_width * degree rounded up to 32) / 32 ; buffer = EI + EC keys per lane
constexpr int next_pow2(int v) { int r = 1; while (r < v) r <<= 1; return r; }

template <int EI, int EC, bool MULTI = false>
__global__ void __launch_bounds__(512, (EI <= 2 ? 3 : (EI <= 4 ? 2 : 1))) cagra_search_kernel(cagra_launch p)
{
  static_assert(!MULTI || EI == 1, "a multi-walker list is 32 entries (search_multi_cta.cuh:119-127)");
  constexpr int EB = next_pow2(EI + EC);  // the bitonic network needs a power-of-two key count; spare keys stay ~0 (sort last)
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const bool ip    = p.metric == InnerProduct;
  const int qpad   = (p.dim + 3) & ~3;
  const uint32_t small_size = p.small_hash_bitlen ? (1u << p.small_hash_bitlen) : 0u;
  const int n_cand = p.search_width * p.degree;
  // per-warp shared memory: query | hash (small) | staged ids | staged distances | parents
  const size_t per_warp = static_cast<size_t>(qpad) * 4 + static_cast<size_t>(small_size) * 4 + static_cast<size_t>(EB * 32) * 8 + 16;
  unsigned char* base   = smem_raw + per_warp * wid;
  float* sq             = reinterpret_cast<float*>(base);
  uint32_t* shash       = reinterpret_cast<uint32_t*>(sq + qpad);
  uint32_t* scand       = shash + small_size;
  float* sdist          = reinterpret_cast<float*>(scand + EB * 32);
  uint32_t* sparent     = reinterpret_cast<uint32_t*>(sdist + EB * 32);
  // Persistent warps: every warp keeps pulling queries from a global counter until the batch is drained.  Walks differ in
  // length, and a batch is only ~1.4 "waves" of resident warps: with one query per warp and CTA-granular scheduling the
  // early finishers idle and the second wave runs nearly empty.
  for (;;) {
  int64_t qi = 0;
  if (lane == 0) qi = static_cast<int64_t>(atomicAdd(p.work_counter, 1ull));
  qi = __shfl_sync(0xffffffffu, qi, 0);
  int widx = 0;  // which of the query's walkers this warp is
  if constexpr (MULTI) {
    widx = static_cast<int>(qi % p.walkers);
    qi /= p.walkers;
  }
  if (qi >= p.nq) break;

  const uint32_t bitlen = p.small_hash_bitlen ? p.small_hash_bitlen : p.hash_bitlen;
  uint32_t* table       = p.small_hash_bitlen ? shash : p.hash_global + (static_cast<size_t>(qi) << p.hash_bitlen);
  const uint32_t tsize  = 1u << bitlen;
  for (int j = lane; j < qpad; j += 32) sq[j] = j < p.dim ? p.queries[qi * p.dim + j] : 0.f;
  for (uint32_t j = lane; j < tsize; j += 32) table[j] = kInvalid;
  __syncwarp();

  const int t = lane & 7, g = lane >> 3;  // team lane / team id (4 teams of 8)
  uint64_t key[EB];

  // ---- random seeds over the whole buffer (device_common_jit.cuh:36-112)
  const int buf = p.itopk + n_cand;
#pragma unroll
  for (int e = 0; e < EB; ++e) key[e] = ~0ull;
  for (int i0 = 0; i0 < EB * 32; i0 += 4) {
    const int i        = i0 + g;  // buffer slot handled by this team
    const bool valid_i = i < buf;
    float best         = INFINITY;
    uint32_t best_id   = kInvalid;
    if (i0 < buf) {  // warp-uniform: at least one team has work
      for (int j = 0; j < p.num_random_samplings; ++j) {
        uint32_t seed = 0;
        if (valid_i) {
          // multi-walker: walker w draws the seeds a (w-th) CTA of the reference would (device_common_jit.cuh:65-74:
          // gid = block_id + num_blocks * (i + num_pickup * j))
          const uint64_t gid = MULTI ? static_cast<uint64_t>(widx) + static_cast<uint64_t>(p.walkers) * (static_cast<uint64_t>(i) + static_cast<uint64_t>(buf) * static_cast<uint64_t>(j))
                                     : static_cast<uint64_t>(i) + static_cast<uint64_t>(buf) * static_cast<uint64_t>(j);
          seed               = static_cast<uint32_t>(xorshift64(gid ^ p.rand_xor_mask) % static_cast<uint64_t>(p.n));
        }
        const float dd = walk_distance(p.data16, p.ld16, p.data, p.ld, p.dim, seed, sq, t, ip);
        if (valid_i && dd < best) { best = dd; best_id = seed; }
      }
    }
    if (t == 0) {
      if (best_id != kInvalid && hash_insert(table, bitlen, best_id) == 0) { best = INFINITY; best_id = kInvalid; }
      scand[i] = best_id;
      sdist[i] = best;
    }
  }
  __syncwarp();
#pragma unroll
  for (int e = 0; e < EB; ++e) {
    const int idx     = e * 32 + lane;
    const uint32_t id = scand[idx];
    key[e] = id == kInvalid ? ~0ull : (static_cast<uint64_t>(dist_key(sdist[idx])) << 32) | id;
  }
  __syncwarp();

  uint32_t iter = 0;
  while (true) {
    if (p.small_hash_bitlen && (iter + 1) % p.reset_interval == 0) {
      for (uint32_t j = lane; j < tsize; j += 32) table[j] = kInvalid;
      __syncwarp();
    }
    // ---- keep the itopk best of (itopk U candidates), sorted: keys 0..EI-1 after the sort
    warp_bitonic_sort<EB>(key, lane);
    if (static_cast<int>(iter + 1) == p.max_iter) break;

    // ---- pick up to search_width unvisited parents, in rank order (search_single_cta_device_helpers.cuh:97-137)
    int n_parents = 0;  // search_width <= 4 supported by this kernel; ids staged in sparent[]
#pragma unroll
    for (int e = 0; e < EI; ++e) {
      const uint32_t id   = static_cast<uint32_t>(key[e]);
      const bool unvisited = (key[e] != ~0ull) && (id & kMsb) == 0;
      uint32_t m = __ballot_sync(0xffffffffu, unvisited);
      while (m && n_parents < p.search_width) {
        const int src = __ffs(m) - 1;
        m &= m - 1;
        const uint32_t pid = __shfl_sync(0xffffffffu, id, src);
        if constexpr (MULTI) {
          // a node is expanded by exactly ONE walker of the query: the shared traversed table decides
          // (search_multi_cta_device_helpers.cuh pickup_next_parent: insert into traversed_hashmap, skip when present)
          uint32_t fresh = 0;
          if (lane == 0) fresh = hash_insert(p.traversed + (static_cast<size_t>(qi) << p.traversed_bitlen), p.traversed_bitlen, pid);
          fresh = __shfl_sync(0xffffffffu, fresh, 0);
          if (!fresh) {
            if (lane == src) key[e] |= kMsb;  // somebody else's parent: never pick it again
            continue;
          }
        }
        // mark as used; a node the filter rejects may serve as a stepping stone ONCE and then leaves the list
        // (search_single_cta_jit.cuh:297-316: filtered parents are invalidated after their children were expanded)
        if (lane == src) key[e] = (p.keep_bits != nullptr && !node_kept(p.keep_bits, p.n_bits, pid)) ? ~0ull : (key[e] | kMsb);
        if (lane == 0) sparent[n_parents] = pid;
        ++n_parents;
      }
    }
    // ---- restore the small hash with the current itopk (after a reset)
    if (p.small_hash_bitlen && (iter + 1) % p.reset_interval == 0) {
#pragma unroll
      for (int e = 0; e < EI; ++e)
        if (key[e] != ~0ull) hash_insert(table, bitlen, static_cast<uint32_t>(key[e]) & ~kMsb);
      __syncwarp();
    }
    if (n_parents == 0 && static_cast<int>(iter) >= p.min_iter) break;

    // ---- children of the parents: adjacency rows, dedup through the hash, compact the survivors
    int n_new = 0;
    __syncwarp();
    for (int pi = 0; pi < n_parents; ++pi) {
      const uint32_t parent = sparent[pi];
      for (int j0 = 0; j0 < p.degree; j0 += 32) {
        const int j    = j0 + lane;
        uint32_t child = kInvalid;
        if (j < p.degree) child = __ldg(p.graph + static_cast<int64_t>(parent) * p.degree + j);
        bool fresh = false;
        if (child != kInvalid && child < static_cast<uint32_t>(p.n)) fresh = hash_insert(table, bitlen, child) != 0;
        const uint32_t m = __ballot_sync(0xffffffffu, fresh);
        if (fresh) scand[n_new + __popc(m & ((1u << lane) - 1u))] = child;
        n_new += __popc(m);
      }
    }
    __syncwarp();
    if (p.prefetch_row_bytes != 0) {
      for (int c = lane; c < n_new; c += 32) {
        const uint32_t id = scand[c];
        const void* row   = p.data16 ? static_cast<const void*>(p.data16 + static_cast<int64_t>(id) * p.ld16)
                                     : static_cast<const void*>(p.data + static_cast<int64_t>(id) * p.ld);
        ptx::bulk_prefetch_l2(row, p.prefetch_row_bytes);  // UBLKPF: uniform-register operands -> one trip of a lane loop per row
      }
    }
    // ---- distances: 4 candidates per step (teams of 8 lanes), two steps in flight
    for (int c0 = 0; c0 < n_new; c0 += 8) {
      const int ca = c0 + g, cb = c0 + 4 + g;
      const uint32_t ida = ca < n_new ? scand[ca] : 0u, idb = cb < n_new ? scand[cb] : 0u;
      const float da = walk_distance(p.data16, p.ld16, p.data, p.ld, p.dim, ida, sq, t, ip);
      const float db = walk_distance(p.data16, p.ld16, p.data, p.ld, p.dim, idb, sq, t, ip);
      if (t == 0) {
        if (ca < n_new) sdist[ca] = da;
        if (cb < n_new) sdist[cb] = db;
      }
    }
    __syncwarp();
    // ---- candidates -> register keys EI..EB-1
#pragma unroll
    for (int e = 0; e < EB - EI; ++e) {
      const int c = e * 32 + lane;
      key[EI + e] = (e < EC && c < n_new) ? (static_cast<uint64_t>(dist_key(sdist[c])) << 32) | scand[c] : ~0ull;
    }
    __syncwarp();
    ++iter;
  }

  // ---- pre-filter post-processing (search_single_cta_jit.cuh:321-334): drop rejected nodes, valid ones move up
  if (p.keep_bits != nullptr) {
#pragma unroll
    for (int e = 0; e < EB; ++e) {
      if (e >= EI) key[e] = ~0ull;
      else if (key[e] != ~0ull && !node_kept(p.keep_bits, p.n_bits, static_cast<uint32_t>(key[e]) & ~kMsb)) key[e] = ~0ull;
    }
    warp_bitonic_sort<EB>(key, lane);
  }
  // ---- fp16 walk: exact fp32 re-rank of the best 32 entries (first register key of every lane), then the usual output
  if (p.data16 != nullptr) {
    const uint32_t my_id = key[0] != ~0ull ? (static_cast<uint32_t>(key[0]) & ~kMsb) : kInvalid;
    float my_d = 0.f;
    for (int c0 = 0; c0 < 32; c0 += 4) {  // team g scores entry c0 + g
      const uint32_t id = __shfl_sync(0xffffffffu, my_id, c0 + g);
      const float d     = team_distance(p.data + static_cast<int64_t>(id == kInvalid ? 0u : id) * p.ld, sq, p.dim, t, ip);
      const float got   = __shfl_sync(0xffffffffu, d, ((lane - c0) & 3) * 8);  // entry `lane` was scored by team lane - c0
      if (lane >= c0 && lane < c0 + 4) my_d = got;
    }
    if (my_id != kInvalid) key[0] = (static_cast<uint64_t>(dist_key(my_d)) << 32) | (static_cast<uint32_t>(key[0]));
#pragma unroll
    for (int e = 1; e < EB; ++e) key[e] = ~0ull;  // only the re-ranked 32 can be returned (k <= 32 in this mode)
    warp_bitonic_sort<EB>(key, lane);
  }
  if constexpr (MULTI) {
    // every walker hands its sorted 32-entry list to the per-query merge (cagra_merge_walkers_kernel)
    p.mc_keys[(static_cast<size_t>(qi) * p.walkers + widx) * 32 + lane] = key[0] == ~0ull ? ~0ull : (key[0] & ~static_cast<uint64_t>(kMsb));
    __syncwarp();
    continue;
  }
  // ---- results: first k entries of the sorted list
#pragma unroll
  for (int e = 0; e < EI; ++e) {
    const int r = e * 32 + lane;
    if (r < p.k) {
      const bool valid  = key[e] != ~0ull;
      const uint32_t id = valid ? (static_cast<uint32_t>(key[e]) & ~kMsb) : kInvalid;
      float d           = valid ? key_dist(static_cast<uint32_t>(key[e] >> 32)) : FLT_MAX;
      if (valid && ip) d = -d;
      if (p.out_idx32) p.out_idx32[qi * p.k + r] = id;
      if (p.out_idx64) p.out_idx64[qi * p.k + r] = valid ? static_cast<int64_t>(id) : -1;  // reference: max u32 cast
      p.out_dist[qi * p.k + r] = d;
    }
  }
  if (p.out_iters && lane == 0) p.out_iters[qi] = iter + 1;
  __syncwarp();
  }  // next query
}

// Multi-walker epilogue: one warp per query merges its walkers' lists — sort, drop the ids several walkers found (their
// keys are bit-identical: same id, same distance arithmetic), drop filtered nodes, emit the k best
// (search_multi_cta.cuh:245-262: topk over num_cta_per_query * 32 intermediate results).
template <int E>
__global__ void __launch_bounds__(128) cagra_merge_walkers_kernel(const unsigned long long* __restrict__ keys, int64_t nq, int walkers, int k,
                                                                   bool ip, const uint32_t* __restrict__ keep_bits, int64_t n_bits,
                                                                   uint32_t* __restrict__ out32, int64_t* __restrict__ out64,
                                                                   float* __restrict__ out_dist)
{
  const int lane   = threadIdx.x & 31;
  const int64_t qi = (blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x) >> 5;
  if (qi >= nq) return;
  uint64_t key[E];
#pragma unroll
  for (int e = 0; e < E; ++e) {
    key[e] = e < walkers ? keys[(static_cast<size_t>(qi) * walkers + e) * 32 + lane] : ~0ull;
    if (keep_bits != nullptr && key[e] != ~0ull && !node_kept(keep_bits, n_bits, static_cast<uint32_t>(key[e]))) key[e] = ~0ull;
  }
  warp_bitonic_sort<E>(key, lane);
  uint64_t prev[E];
#pragma unroll
  for (int e = 0; e < E; ++e) {  // striped order: element e*32 + lane; its predecessor sits in lane - 1 (or lane 31 of e - 1)
    prev[e] = __shfl_up_sync(0xffffffffu, key[e], 1);
    const uint64_t carry = __shfl_sync(0xffffffffu, key[e > 0 ? e - 1 : 0], 31);
    if (lane == 0) prev[e] = e > 0 ? carry : ~key[e];
  }
#pragma unroll
  for (int e = 0; e < E; ++e)
    if (key[e] == prev[e]) key[e] = ~0ull;
  warp_bitonic_sort<E>(key, lane);
#pragma unroll
  for (int e = 0; e < E; ++e) {
    const int r = e * 32 + lane;
    if (r < k) {
      const bool valid  = key[e] != ~0ull;
      const uint32_t id = valid ? static_cast<uint32_t>(key[e]) : kInvalid;
      float d           = valid ? key_dist(static_cast<uint32_t>(key[e] >> 32)) : FLT_MAX;
      if (valid && ip) d = -d;
      if (out32) out32[qi * k + r] = id;
      if (out64) out64[qi * k + r] = valid ? static_cast<int64_t>(id) : -1;
      out_dist[qi * k + r] = d;
    }
  }
}

struct cagra_plan {
  int itopk, max_iter, min_iter;
  uint32_t hash_bitlen, small_hash_bitlen, reset_interval;
};

// search_plan.cuh:199-372 (single-CTA branch)
cagra_plan make_plan(const cuvsCagraSearchParams& sp, int64_t n, int degree, int k)
{
  cagra_plan pl{};
  size_t itopk = sp.itopk_size ? sp.itopk_size : 64;
  if (itopk % 32) itopk += 32 - itopk % 32;
  const size_t w = std::max<size_t>(sp.search_width, 1);
  size_t mi = sp.max_iterations;
  if (mi == 0) {
    mi = itopk / w;
    int64_t reach = 1;
    while (reach < n) { reach *= std::max<int64_t>(2, degree / 2); ++mi; }
  }
  mi = std::max(mi, sp.min_iterations);
  pl.itopk = static_cast<int>(itopk);
  pl.max_iter = static_cast<int>(mi);
  pl.min_iter = static_cast<int>(sp.min_iterations);
  const float fill = sp.hashmap_max_fill_rate > 0.f ? sp.hashmap_max_fill_rate : 0.5f;
  pl.hash_bitlen = pl.small_hash_bitlen = 0;
  pl.reset_interval = 1u << 20;
  if (sp.hashmap_mode == AUTO_HASH || sp.hashmap_mode == SMALL) {
    const size_t max_visited = itopk + w * degree;
    uint32_t hb = std::max<uint32_t>(8, static_cast<uint32_t>(sp.hashmap_min_bitlen));
    while (max_visited > (size_t(1) << hb) * fill) ++hb;
    if (hb <= 13) {
      pl.small_hash_bitlen = pl.hash_bitlen = hb;
      pl.reset_interval = 1;
      while (itopk + w * degree * (pl.reset_interval + 1) <= (size_t(1) << hb) * fill) ++pl.reset_interval;
    } else {
      B2_EXPECTS(sp.hashmap_mode == AUTO_HASH, "small-hash cannot be used because the required hash size exceeds the limit (%u)", 1u << 13);
    }
  }
  if (pl.hash_bitlen == 0) {
    const size_t max_visited = itopk + w * degree * mi;
    uint32_t hb = std::max<uint32_t>(11, static_cast<uint32_t>(sp.hashmap_min_bitlen));
    while (max_visited > (size_t(1) << hb) * fill) ++hb;
    B2_EXPECTS(hb <= 20, "hash_bitlen cannot be largen than 20 (1M). You can decrease itopk_size, search_width or max_iterations to reduce the required hashmap size.");
    pl.hash_bitlen = hb;
  }
  B2_EXPECTS(k <= pl.itopk, "topk = %d must be smaller than itopk_size = %d", k, pl.itopk);
  return pl;
}

// Row bytes for the walk's bulk L2 prefetch (0 = off): rows must start on 16-byte boundaries and be a 16-byte multiple long.
// Measured on a B200 (profiles/r02_ab_cagra_prefetch.txt; 10M x 96 fp32, batch 10k): no prefetch 5.73-5.75 ms, per-lane
// prefetch.global.L2 of the row's lines 6.06-6.08 ms (slower: three CCTL per row and lane compete with the team loads for the
// LSU), bulk prefetch 5.56-5.58 ms.
static uint32_t walk_prefetch_bytes(const cagra_launch& p)
{
  const size_t pitch = p.data16 ? static_cast<size_t>(p.ld16) * 2 : static_cast<size_t>(p.ld) * 4;
  const uintptr_t base = p.data16 ? reinterpret_cast<uintptr_t>(p.data16) : reinterpret_cast<uintptr_t>(p.data);
  if (pitch % 16 != 0 || base % 16 != 0) return 0;
  const size_t row = (static_cast<size_t>(p.dim) * (p.data16 ? 2 : 4) + 15) / 16 * 16;
  return static_cast<uint32_t>(std::min(row, pitch));
}

template <int EI, int EC, bool MULTI = false>
void launch_search(cudaStream_t s, const cagra_launch& p, size_t per_warp_smem)
{
  auto kern = cagra_search_kernel<EI, EC, MULTI>;
  int warps = 16;
  while (warps > 1 && per_warp_smem * warps > 200 * 1024) warps >>= 1;
  const size_t smem = per_warp_smem * warps;
  B2_EXPECTS(per_warp_smem <= 200 * 1024, "cagra search: per-query shared memory (%zu bytes) exceeds the limit", per_warp_smem);
  B2_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
  int per_sm = 1, dev = 0, sms = 148;
  B2_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, warps * 32, smem));
  B2_CUDA(cudaGetDevice(&dev));
  B2_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  const int64_t n_walks = p.nq * (MULTI ? p.walkers : 1);
  if (MULTI) {
    // few walks: spread them over the SMs (one warp per CTA while the batch is smaller than the machine) instead of packing
    // 16 of them into one CTA — the case the reference switches to multi-CTA for (search_plan.cuh:122-131)
    while (warps > 1 && n_walks < static_cast<int64_t>(warps) * sms) warps >>= 1;
  }
  const unsigned grid = std::min<unsigned>(blocks_for(n_walks, warps), static_cast<unsigned>(std::max(per_sm, 1) * sms));
  dbuf<unsigned long long> counter(1, s);
  B2_CUDA(cudaMemsetAsync(counter.data(), 0, sizeof(unsigned long long), s));
  cagra_launch pl = p;
  pl.work_counter = counter.data();
  pl.prefetch_row_bytes = walk_prefetch_bytes(p);
  timed_section ts("cagra_search", s);
  count_launch();
  kern<<<grid, warps * 32, smem, s>>>(pl);
  B2_CUDA(cudaGetLastError());
}

__global__ void fill_u32_kernel(uint32_t* p, size_t n, uint32_t v)
{
  const size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x;
  if (i < n) p[i] = v;
}

// MULTI_CTA (search_multi_cta.cuh:100-262, plan search_plan.cuh:254-290): num_cta_per_query = max(search_width,
// ceil(itopk / 32)) walkers per query, each a 32-entry list with search_width 1 and its own small visited hash; parents are
// claimed through one traversed table per query; the walkers' lists are merged into the top-k.
void cagra_search_multi(resources* res, const cagra_index& idx, const cuvsCagraSearchParams& sp, const float* queries, int64_t nq, int k,
                        uint32_t* out32, int64_t* out64, float* out_dist, const uint32_t* keep_bits, int64_t n_bits)
{
  auto s = res->stream;
  size_t itopk = sp.itopk_size ? sp.itopk_size : 64;
  if (itopk % 32) itopk += 32 - itopk % 32;
  const int walkers = static_cast<int>(std::max<size_t>(std::max<size_t>(sp.search_width, 1), itopk / 32));
  B2_EXPECTS(walkers <= 16, "cagra multi-cta search: itopk_size / 32 = %d walkers per query exceeds the 16 this build merges", walkers);
  B2_EXPECTS(walkers * 32 >= k, "`num_cta_per_query` (%d) * 32 must be equal to or greater than `topk` (%d)", walkers, k);
  cuvsCagraSearchParams one = sp;  // the per-walker plan: itopk 32, search_width 1
  one.itopk_size   = 32;
  one.search_width = 1;
  one.hashmap_mode = AUTO_HASH;
  const cagra_plan pl = make_plan(one, idx.n, idx.degree, std::min(k, 32));
  B2_EXPECTS(pl.small_hash_bitlen != 0, "cagra multi-cta search: graph_degree %d needs a visited table beyond the small-hash limit", idx.degree);
  const int EC = (idx.degree + 31) / 32;
  cagra_launch p{};
  p.data = idx.data; p.graph = idx.graph; p.n = idx.n; p.dim = idx.dim; p.ld = idx.ld; p.degree = idx.degree;
  p.data16 = nullptr; p.ld16 = 0;
  p.queries = queries; p.nq = nq; p.metric = idx.metric == InnerProduct ? InnerProduct : L2Expanded;
  p.k = k; p.itopk = 32; p.search_width = 1; p.min_iter = pl.min_iter; p.max_iter = pl.max_iter;
  p.hash_bitlen = pl.hash_bitlen; p.small_hash_bitlen = pl.small_hash_bitlen; p.reset_interval = pl.reset_interval;
  p.num_random_samplings = static_cast<int>(std::max<uint32_t>(sp.num_random_samplings, 1));
  p.rand_xor_mask = sp.rand_xor_mask;
  p.keep_bits = keep_bits; p.n_bits = n_bits;
  p.walkers = walkers;
  // traversed table: every walker claims at most max(32, max_iter) parents (search_plan.cuh:277-290)
  const float fill = sp.hashmap_max_fill_rate > 0.f ? sp.hashmap_max_fill_rate : 0.5f;
  uint32_t tb = std::max<uint32_t>(11, static_cast<uint32_t>(sp.hashmap_min_bitlen));
  while (static_cast<size_t>(walkers) * std::max(32, pl.max_iter) > (size_t(1) << tb) * fill) ++tb;
  B2_EXPECTS(tb <= 20, "hash_bitlen cannot be largen than 20 (1M). You can decrease itopk_size, search_width or max_iterations to reduce the required hashmap size.");
  p.traversed_bitlen = tb;
  dbuf<uint32_t> trav(static_cast<size_t>(nq) << tb, s);
  dbuf<unsigned long long> keys(static_cast<size_t>(nq) * walkers * 32, s);
  p.traversed = trav.data();
  p.mc_keys   = keys.data();
  count_launch();
  fill_u32_kernel<<<blocks_for(static_cast<int64_t>(trav.size()), 256), 256, 0, s>>>(trav.data(), trav.size(), kInvalid);
  const int qpad = (idx.dim + 3) & ~3;
  int ebp = 1;
  while (ebp < 1 + EC) ebp <<= 1;
  const size_t per_warp = static_cast<size_t>(qpad) * 4 + (size_t(4) << pl.small_hash_bitlen) + static_cast<size_t>(ebp) * 32 * 8 + 16;
  if (EC == 1) launch_search<1, 1, true>(s, p, per_warp);
  else if (EC == 2) launch_search<1, 2, true>(s, p, per_warp);
  else if (EC <= 4) launch_search<1, 4, true>(s, p, per_warp);
  else B2_FAIL("cagra multi-cta search: graph_degree %d > 128 is not built", idx.degree);
  const bool ip = idx.metric == InnerProduct;
  count_launch();
  const unsigned mgrid = blocks_for(nq * 32, 128);
  if (walkers <= 1) cagra_merge_walkers_kernel<1><<<mgrid, 128, 0, s>>>(keys.data(), nq, walkers, k, ip, keep_bits, n_bits, out32, out64, out_dist);
  else if (walkers <= 2) cagra_merge_walkers_kernel<2><<<mgrid, 128, 0, s>>>(keys.data(), nq, walkers, k, ip, keep_bits, n_bits, out32, out64, out_dist);
  else if (walkers <= 4) cagra_merge_walkers_kernel<4><<<mgrid, 128, 0, s>>>(keys.data(), nq, walkers, k, ip, keep_bits, n_bits, out32, out64, out_dist);
  else if (walkers <= 8) cagra_merge_walkers_kernel<8><<<mgrid, 128, 0, s>>>(keys.data(), nq, walkers, k, ip, keep_bits, n_bits, out32, out64, out_dist);
  else cagra_merge_walkers_kernel<16><<<mgrid, 128, 0, s>>>(keys.data(), nq, walkers, k, ip, keep_bits, n_bits, out32, out64, out_dist);
  B2_CUDA(cudaGetLastError());
  if (idx.metric == L2SqrtExpanded) postprocess_distances(s, out_dist, nq * k, L2SqrtExpanded);
}

void cagra_search(resources* res, const cagra_index& idx, const cuvsCagraSearchParams& sp, const float* queries, int64_t nq, int k,
                  uint32_t* out32, int64_t* out64, float* out_dist, const uint32_t* keep_bits = nullptr, int64_t n_bits = 0)
{
  auto s = res->stream;
  if (nq == 0) return;
  B2_EXPECTS(idx.metric == L2Expanded || idx.metric == InnerProduct || idx.metric == L2SqrtExpanded,
             "cagra search: unsupported metric %d", int(idx.metric));
  B2_EXPECTS(!sp.persistent, "cagra search: the persistent (latency) mode is out of scope of this library");
  // algo selection (search_plan.cuh:122-131): AUTO -> single-CTA when itopk <= 512 and the batch has at least 2 queries per
  // SM, multi-CTA otherwise (small batches: several walkers per query keep the machine busy).  MULTI_KERNEL is served by the
  // multi-walker kernel too.
  int algo = static_cast<int>(sp.algo);
  if (algo == AUTO) {
    const size_t itopk_req = sp.itopk_size ? sp.itopk_size : 64;
    algo = (itopk_req <= 512 && static_cast<size_t>(nq) >= static_cast<size_t>(sm_count_of(res->device)) * 2) ? SINGLE_CTA : MULTI_CTA;
  }
  if (algo != SINGLE_CTA) return cagra_search_multi(res, idx, sp, queries, nq, k, out32, out64, out_dist, keep_bits, n_bits);
  const cagra_plan pl = make_plan(sp, idx.n, idx.degree, k);
  const int w         = static_cast<int>(std::max<size_t>(sp.search_width, 1));
  B2_EXPECTS(w <= 4, "cagra search: search_width > 4 is not supported by this build (got %d)", w);
  const int n_cand = w * idx.degree;
  const int EI = pl.itopk / 32, EC = (n_cand + 31) / 32;
  cagra_launch p{};
  p.data = idx.data; p.graph = idx.graph; p.n = idx.n; p.dim = idx.dim; p.ld = idx.ld; p.degree = idx.degree;
  p.data16 = (idx.data16.data() != nullptr && k <= 32) ? idx.data16.data() : nullptr; p.ld16 = idx.ld16;
  p.queries = queries; p.nq = nq; p.metric = idx.metric == InnerProduct ? InnerProduct : L2Expanded;
  p.k = k; p.itopk = pl.itopk; p.search_width = w; p.min_iter = pl.min_iter; p.max_iter = pl.max_iter;
  p.hash_bitlen = pl.hash_bitlen; p.small_hash_bitlen = pl.small_hash_bitlen; p.reset_interval = pl.reset_interval;
  p.num_random_samplings = static_cast<int>(std::max<uint32_t>(sp.num_random_samplings, 1));
  p.rand_xor_mask = sp.rand_xor_mask;
  p.out_idx32 = out32; p.out_idx64 = out64; p.out_dist = out_dist; p.out_iters = nullptr;
  p.keep_bits = keep_bits; p.n_bits = n_bits;
  dbuf<uint32_t> gh;
  if (pl.small_hash_bitlen == 0) {
    gh.alloc(static_cast<size_t>(nq) << pl.hash_bitlen, s);
    p.hash_global = gh.data();
  }
  const int qpad = (idx.dim + 3) & ~3;
  int ebp = 1;
  while (ebp < EI + EC) ebp <<= 1;
  const size_t per_warp = static_cast<size_t>(qpad) * 4 + (pl.small_hash_bitlen ? (size_t(4) << pl.small_hash_bitlen) : 0) +
                          static_cast<size_t>(ebp) * 32 * 8 + 16;
#define B2_CAGRA_CASE(EI_, EC_) if (EI == EI_ && EC == EC_) { launch_search<EI_, EC_>(s, p, per_warp); launched = true; }
  bool launched = false;
  B2_CAGRA_CASE(1, 1) B2_CAGRA_CASE(1, 2) B2_CAGRA_CASE(1, 4)
  B2_CAGRA_CASE(2, 1) B2_CAGRA_CASE(2, 2) B2_CAGRA_CASE(2, 4)
  B2_CAGRA_CASE(4, 1) B2_CAGRA_CASE(4, 2) B2_CAGRA_CASE(4, 4)
  B2_CAGRA_CASE(8, 2) B2_CAGRA_CASE(8, 4)
#undef B2_CAGRA_CASE
  B2_EXPECTS(launched, "cagra search: unsupported (itopk=%d, search_width*graph_degree=%d) combination; itopk in {32,64,128,256} and "
                       "search_width*degree in {<=32, <=64, <=128} are built", pl.itopk, n_cand);
  if (idx.metric == L2SqrtExpanded) postprocess_distances(s, out_dist, nq * k, L2SqrtExpanded);
}

// ------------------------------------------------------------------ graph build (kNN + reverse edges)
__global__ void to_half_rows_kernel(const float* __restrict__ x, int64_t n, int dim, int ld, int ld16, __half* __restrict__ out)
{
  int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  if (i >= n * ld16) return;
  const int64_t r = i / ld16;
  const int c     = static_cast<int>(i % ld16);
  out[i]          = __float2half_rn(c < dim ? x[r * ld + c] : 0.f);
}

__global__ void knn_to_graph_kernel(const int64_t* __restrict__ knn, int64_t n, int kk, int keep, uint32_t* __restrict__ graph, int degree)
{
  // forward half: the `keep` nearest neighbours (self removed)
  int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  if (i >= n) return;
  int w = 0;
  for (int j = 0; j < kk && w < degree; ++j) {
    int64_t v = knn[i * kk + j];
    if (v == i || v < 0 || v >= n) continue;
    graph[i * degree + w] = static_cast<uint32_t>(v);
    ++w;
  }
  for (; w < degree; ++w) graph[i * degree + w] = static_cast<uint32_t>((i + 1 + w) % n);  // degenerate tiny inputs
  (void)keep;
}

// each of the first `keep` forward edges (u, v) as (target v, source u), in source order
__global__ void forward_edges_kernel(const uint32_t* __restrict__ fwd, int64_t n, int degree, int keep, uint32_t* __restrict__ tgt,
                                     uint32_t* __restrict__ src)
{
  int64_t t = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  if (t >= n * keep) return;
  tgt[t] = fwd[(t / keep) * degree + t % keep];
  src[t] = static_cast<uint32_t>(t / keep);
}

// reverse edges of node v: its sources u in ascending order (edges grouped by target, stably), the first rev_cap kept
__global__ void reverse_edges_kernel(const uint32_t* __restrict__ src, const int64_t* __restrict__ start, int64_t n,
                                     uint32_t* __restrict__ rev, uint32_t* __restrict__ rev_cnt, int rev_cap)
{
  int64_t v = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  if (v >= n) return;
  const int64_t cnt = start[v + 1] - start[v];
  for (int64_t slot = 0; slot < cnt && slot < rev_cap; ++slot) rev[v * rev_cap + slot] = src[start[v] + slot];
  rev_cnt[v] = static_cast<uint32_t>(cnt);
}

// final row = first `keep` forward edges, then reverse edges not already present, then remaining forward edges
__global__ void merge_graph_kernel(const uint32_t* __restrict__ fwd, const uint32_t* __restrict__ rev, const uint32_t* __restrict__ rev_cnt,
                                   int64_t n, int degree, int keep, int rev_cap, uint32_t* __restrict__ out)
{
  int64_t u = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  if (u >= n) return;
  const uint32_t* f = fwd + u * degree;
  uint32_t* o       = out + u * degree;
  int w = 0;
  for (; w < keep; ++w) o[w] = f[w];
  const int nr = min(static_cast<int>(rev_cnt[u]), rev_cap);
  for (int j = 0; j < nr && w < degree; ++j) {
    uint32_t v = rev[u * rev_cap + j];
    bool dup = false;
    for (int q = 0; q < w; ++q) dup |= (o[q] == v);
    if (!dup && v != u) o[w++] = v;
  }
  for (int j = keep; j < degree && w < degree; ++j) {
    uint32_t v = f[j];
    bool dup = false;
    for (int q = 0; q < w; ++q) dup |= (o[q] == v);
    if (!dup) o[w++] = v;
  }
  for (int j = 0; w < degree; ++j) {  // pathological duplicates: fill with successive ids
    uint32_t v = static_cast<uint32_t>((u + 1 + j) % n);
    bool dup = false;
    for (int q = 0; q < w; ++q) dup |= (o[q] == v);
    if (!dup && v != u) o[w++] = v;
  }
}


// ---- graph optimisation (rank-based detour pruning, cpp/src/neighbors/detail/cagra/graph_core.cuh: kern_prune)
// For node A and its neighbour B at rank kAB, a 2-hop route A -> D -> B is "detourable" when D is a closer neighbour of A
// (rank kAD < kAB) and B is a neighbour of D with rank kDB < kAB.  Edges with few detours are kept first.
// One CTA per node; knn rows are sorted by distance (self excluded).
__global__ void __launch_bounds__(128) detour_count_kernel(const uint32_t* __restrict__ knn, int64_t n, int di, uint32_t* __restrict__ counts)
{
  extern __shared__ uint32_t sm[];
  uint32_t* na  = sm;        // [di] neighbours of A
  uint32_t* cnt = sm + di;   // [di]
  const int64_t a = blockIdx.x;
  for (int j = threadIdx.x; j < di; j += blockDim.x) { na[j] = knn[a * di + j]; cnt[j] = 0; }
  __syncthreads();
  for (int kad = 0; kad < di - 1; ++kad) {
    const uint32_t dn = na[kad];
    for (int kdb = threadIdx.x; kdb < di; kdb += blockDim.x) {
      const uint32_t b = knn[static_cast<int64_t>(dn) * di + kdb];
      const int lo     = max(kad, kdb) + 1;
      for (int kab = lo; kab < di; ++kab)
        if (na[kab] == b) { atomicAdd(&cnt[kab], 1u); break; }
    }
  }
  __syncthreads();
  for (int j = threadIdx.x; j < di; j += blockDim.x) counts[a * di + j] = cnt[j];
}

// keep the `degree` edges with the fewest detours (ties: closer first); one thread per node (di <= 128)
__global__ void select_pruned_kernel(const uint32_t* __restrict__ knn, const uint32_t* __restrict__ counts, int64_t n, int di, int degree,
                                     uint32_t* __restrict__ out)
{
  int64_t a = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  if (a >= n) return;
  const uint32_t* c = counts + a * di;
  const uint32_t* g = knn + a * di;
  // counting sort by detour count (counts <= di)
  int w = 0;
  for (uint32_t level = 0; level <= static_cast<uint32_t>(di) && w < degree; ++level)
    for (int j = 0; j < di && w < degree; ++j)
      if (c[j] == level) out[a * degree + w++] = g[j];
  for (int j = 0; w < degree; ++j) out[a * degree + w++] = g[j % di];
}

}  // namespace

// exact kNN graph through the library's own brute-force search (C boundary re-used internally)
static void build_knn_graph(cuvsResources_t res_h, resources* res, const float* data, int64_t n, int dim, cuvsDistanceType metric,
                            int kk, int64_t* knn_out)
{
  cuvsBruteForceIndex_t bf = nullptr;
  B2_EXPECTS(cuvsBruteForceIndexCreate(&bf) == CUVS_SUCCESS, "brute force index create failed");
  int64_t shape[2] = {n, dim};
  DLManagedTensor ds{};
  ds.dl_tensor.data = const_cast<float*>(data); ds.dl_tensor.device = DLDevice{kDLCUDA, res->device}; ds.dl_tensor.ndim = 2;
  ds.dl_tensor.dtype = DLDataType{kDLFloat, 32, 1}; ds.dl_tensor.shape = shape;
  cuvsDistanceType m = metric == InnerProduct ? InnerProduct : L2Expanded;
  if (cuvsBruteForceBuild(res_h, &ds, m, 2.0f, bf) != CUVS_SUCCESS) {
    std::string e = cuvsGetLastErrorText() ? cuvsGetLastErrorText() : "?";
    cuvsBruteForceIndexDestroy(bf);
    B2_FAIL("cagra build: kNN stage failed: %s", e.c_str());
  }
  const int64_t chunk = 16384;
  dbuf<float> dist(static_cast<size_t>(chunk) * kk, res->stream);
  for (int64_t r0 = 0; r0 < n; r0 += chunk) {
    int64_t rows = std::min(chunk, n - r0);
    int64_t qs[2] = {rows, dim}, os[2] = {rows, kk};
    DLManagedTensor q = ds, nb{}, dd{};
    q.dl_tensor.data = const_cast<float*>(data) + r0 * dim; q.dl_tensor.shape = qs;
    nb.dl_tensor.data = knn_out + r0 * kk; nb.dl_tensor.device = ds.dl_tensor.device; nb.dl_tensor.ndim = 2;
    nb.dl_tensor.dtype = DLDataType{kDLInt, 64, 1}; nb.dl_tensor.shape = os;
    dd = nb; dd.dl_tensor.data = dist.data(); dd.dl_tensor.dtype = DLDataType{kDLFloat, 32, 1};
    if (cuvsBruteForceSearch(res_h, bf, &q, &nb, &dd, cuvsFilter{0, NO_FILTER}) != CUVS_SUCCESS) {
      std::string e = cuvsGetLastErrorText() ? cuvsGetLastErrorText() : "?";
      cuvsBruteForceIndexDestroy(bf);
      B2_FAIL("cagra build: kNN stage failed: %s", e.c_str());
    }
  }
  B2_CUDA(cudaStreamSynchronize(res->stream));
  cuvsBruteForceIndexDestroy(bf);
}

// approximate kNN graph for large inputs: IVF-Flat self-search (k <= 64) in query chunks
static void build_knn_graph_ivf(cuvsResources_t res_h, resources* res, const float* data, int64_t n, int dim, cuvsDistanceType metric,
                                int kk, int64_t* knn_out)
{
  cuvsIvfFlatIndexParams_t ip = nullptr;
  cuvsIvfFlatSearchParams_t sp = nullptr;
  cuvsIvfFlatIndex_t ix = nullptr;
  auto fail = [&](const char* what) {
    std::string e = cuvsGetLastErrorText() ? cuvsGetLastErrorText() : "?";
    if (ix) cuvsIvfFlatIndexDestroy(ix);
    if (ip) cuvsIvfFlatIndexParamsDestroy(ip);
    if (sp) cuvsIvfFlatSearchParamsDestroy(sp);
    B2_FAIL("cagra build: %s failed: %s", what, e.c_str());
  };
  if (cuvsIvfFlatIndexParamsCreate(&ip) != CUVS_SUCCESS || cuvsIvfFlatSearchParamsCreate(&sp) != CUVS_SUCCESS || cuvsIvfFlatIndexCreate(&ix) != CUVS_SUCCESS)
    fail("parameter setup");
  uint32_t n_lists = 16;
  while (static_cast<int64_t>(n_lists) * n_lists < n) n_lists *= 2;  // ~sqrt(n), power of two
  ip->n_lists = n_lists; ip->metric = metric == InnerProduct ? InnerProduct : L2Expanded; ip->kmeans_n_iters = 10;
  sp->n_probes = std::max<uint32_t>(16, n_lists / 32);
  int64_t shape[2] = {n, dim};
  DLManagedTensor ds{};
  ds.dl_tensor.data = const_cast<float*>(data); ds.dl_tensor.device = DLDevice{kDLCUDA, res->device}; ds.dl_tensor.ndim = 2;
  ds.dl_tensor.dtype = DLDataType{kDLFloat, 32, 1}; ds.dl_tensor.shape = shape;
  if (cuvsIvfFlatBuild(res_h, ip, &ds, ix) != CUVS_SUCCESS) fail("kNN stage (ivf_flat build)");
  const int64_t chunk = 65536;
  dbuf<float> dist(static_cast<size_t>(chunk) * kk, res->stream);
  for (int64_t r0 = 0; r0 < n; r0 += chunk) {
    int64_t rows = std::min(chunk, n - r0);
    int64_t qs[2] = {rows, dim}, os[2] = {rows, kk};
    DLManagedTensor q = ds, nb{}, dd{};
    q.dl_tensor.data = const_cast<float*>(data) + r0 * dim; q.dl_tensor.shape = qs;
    nb.dl_tensor.data = knn_out + r0 * kk; nb.dl_tensor.device = ds.dl_tensor.device; nb.dl_tensor.ndim = 2;
    nb.dl_tensor.dtype = DLDataType{kDLInt, 64, 1}; nb.dl_tensor.shape = os;
    dd = nb; dd.dl_tensor.data = dist.data(); dd.dl_tensor.dtype = DLDataType{kDLFloat, 32, 1};
    if (cuvsIvfFlatSearch(res_h, sp, ix, &q, &nb, &dd, cuvsFilter{0, NO_FILTER}) != CUVS_SUCCESS) fail("kNN stage (ivf_flat search)");
  }
  B2_CUDA(cudaStreamSynchronize(res->stream));
  cuvsIvfFlatIndexDestroy(ix);
  cuvsIvfFlatIndexParamsDestroy(ip);
  cuvsIvfFlatSearchParamsDestroy(sp);
}

}  // namespace b200

using namespace b200;

static cagra_index& cagra_of(cuvsCagraIndex_t index)
{
  B2_EXPECTS(index != nullptr && index->addr != 0, "index is not built");
  return *reinterpret_cast<cagra_index*>(index->addr);
}

static void set_dataset(resources* r, cagra_index& idx, const DLTensor& ds_in)
{
  // float16 / int8 / uint8 datasets (c/src/neighbors/cagra.cpp:245-264) are widened to fp32 rows the index owns
  B2_EXPECTS(dl_is_dataset_dtype(ds_in), "Unsupported dataset DLtensor dtype: %d and bits: %d", ds_in.dtype.code, ds_in.dtype.bits);
  f32_matrix w;
  widen_to_f32(r, ds_in, w);
  const DLTensor& ds = w.t;
  B2_EXPECTS(ds.ndim == 2 && dl_is_c_contiguous(ds), "dataset must be a row-major 2-D tensor");
  idx.n   = ds.shape[0];
  idx.dim = static_cast<int>(ds.shape[1]);
  idx.ld  = (idx.dim + 3) & ~3;  // rows padded to 16 bytes (cagra.hpp:610)
  const bool dev = dl_is_device(ds) && ds.device.device_type != kDLCUDAHost;
  if (w.widened && idx.ld == idx.dim) {
    idx.data_own = std::move(w.own);
    idx.data     = idx.data_own.data();
  } else if (dev && idx.ld == idx.dim && (reinterpret_cast<uintptr_t>(dl_ptr<float>(ds)) & 15) == 0) {
    idx.data = dl_ptr<float>(ds);  // non-owning view, like the reference's strided_dataset view
  } else {
    idx.data_own.alloc(static_cast<size_t>(idx.n) * idx.ld);
    B2_CUDA(cudaMemsetAsync(idx.data_own.data(), 0, sizeof(float) * idx.n * idx.ld, r->stream));
    B2_CUDA(cudaMemcpy2DAsync(idx.data_own.data(), sizeof(float) * idx.ld, dl_ptr<float>(ds), sizeof(float) * idx.dim,
                              sizeof(float) * idx.dim, idx.n, cudaMemcpyDefault, r->stream));
    idx.data = idx.data_own.data();
  }
}

extern "C" {

cuvsError_t cuvsCagraIndexParamsCreate(cuvsCagraIndexParams_t* params)
{
  return guarded([=] {
    B2_EXPECTS(params != nullptr, "params is null");
    // c/src/neighbors/cagra.cpp:733-742
    auto p = new cuvsCagraIndexParams{};
    p->metric = L2Expanded; p->intermediate_graph_degree = 128; p->graph_degree = 64; p->build_algo = IVF_PQ; p->nn_descent_niter = 20;
    p->compression = nullptr;
    p->graph_build_params = new cuvsIvfPqParams{nullptr, nullptr, 1};
    *params = p;
  });
}
cuvsError_t cuvsCagraIndexParamsDestroy(cuvsCagraIndexParams_t params)
{
  return guarded([=] {
    if (!params) return;
    if (params->graph_build_params) {
      if (params->build_algo == ACE) delete static_cast<cuvsAceParams*>(params->graph_build_params);
      else delete static_cast<cuvsIvfPqParams*>(params->graph_build_params);
    }
    delete params;
  });
}
cuvsError_t cuvsCagraCompressionParamsCreate(cuvsCagraCompressionParams_t* params)
{
  return guarded([=] { *params = new cuvsCagraCompressionParams{8, 0, 0, 25, 0.0, 0.0}; });
}
cuvsError_t cuvsCagraCompressionParamsDestroy(cuvsCagraCompressionParams_t params) { return guarded([=] { delete params; }); }
cuvsError_t cuvsAceParamsCreate(cuvsAceParams_t* params)
{
  return guarded([=] { *params = new cuvsAceParams{0, 120, "/tmp/ace_build", false, 0.0, 0.0}; });
}
cuvsError_t cuvsAceParamsDestroy(cuvsAceParams_t params) { return guarded([=] { delete params; }); }
cuvsError_t cuvsCagraIndexParamsFromHnswParams(cuvsCagraIndexParams_t params, int64_t, int64_t, int M, int, enum cuvsCagraHnswHeuristicType heuristic,
                                               cuvsDistanceType metric)
{
  return guarded([=] {
    B2_EXPECTS(params != nullptr, "params is null");
    params->metric       = metric;
    params->graph_degree = heuristic == CUVS_CAGRA_HEURISTIC_SAME_GRAPH_FOOTPRINT ? static_cast<size_t>(2 * M) : static_cast<size_t>(std::max(2 * M, 32));
    params->intermediate_graph_degree = params->graph_degree * 2;
  });
}
cuvsError_t cuvsCagraExtendParamsCreate(cuvsCagraExtendParams_t* params) { return guarded([=] { *params = new cuvsCagraExtendParams{0}; }); }
cuvsError_t cuvsCagraExtendParamsDestroy(cuvsCagraExtendParams_t params) { return guarded([=] { delete params; }); }

cuvsError_t cuvsCagraSearchParamsCreate(cuvsCagraSearchParams_t* params)
{
  return guarded([=] {
    B2_EXPECTS(params != nullptr, "params is null");
    // c/src/neighbors/cagra.cpp:848-861 (unset fields are zero; algo 0 = SINGLE_CTA, hashmap_mode 0 = HASH as there)
    auto p = new cuvsCagraSearchParams{};
    p->itopk_size = 64; p->search_width = 1; p->hashmap_max_fill_rate = 0.5f; p->num_random_samplings = 1;
    p->rand_xor_mask = 0x128394; p->persistent = false; p->persistent_lifetime = 2; p->persistent_device_usage = 1.0f;
    p->hashmap_mode = AUTO_HASH; p->algo = AUTO;
    *params = p;
  });
}
cuvsError_t cuvsCagraSearchParamsDestroy(cuvsCagraSearchParams_t params) { return guarded([=] { delete params; }); }

cuvsError_t cuvsCagraIndexCreate(cuvsCagraIndex_t* index)
{
  return guarded([=] {
    B2_EXPECTS(index != nullptr, "index is null");
    *index = new cuvsCagraIndex{};
  });
}
cuvsError_t cuvsCagraIndexDestroy(cuvsCagraIndex_t index)
{
  return guarded([=] {
    if (!index) return;
    delete reinterpret_cast<cagra_index*>(index->addr);
    delete index;
  });
}
cuvsError_t cuvsCagraIndexGetDims(cuvsCagraIndex_t index, int64_t* dim) { return guarded([=] { *dim = cagra_of(index).dim; }); }
cuvsError_t cuvsCagraIndexGetSize(cuvsCagraIndex_t index, int64_t* size) { return guarded([=] { *size = cagra_of(index).n; }); }
cuvsError_t cuvsCagraIndexGetGraphDegree(cuvsCagraIndex_t index, int64_t* d) { return guarded([=] { *d = cagra_of(index).degree; }); }
cuvsError_t cuvsCagraIndexGetDataset(cuvsCagraIndex_t index, DLManagedTensor* dataset)
{
  return guarded([=] {
    auto& idx        = cagra_of(index);
    int64_t shape[2] = {idx.n, idx.dim};
    dl_fill_view(dataset, const_cast<float*>(idx.data), idx.device, DLDataType{kDLFloat, 32, 1}, 2, shape);
    if (idx.ld != idx.dim) {
      dataset->dl_tensor.strides    = new int64_t[2];
      dataset->dl_tensor.strides[0] = idx.ld;
      dataset->dl_tensor.strides[1] = 1;
      dataset->deleter = [](DLManagedTensor* self) {
        delete[] self->dl_tensor.shape; delete[] self->dl_tensor.strides;
        self->dl_tensor.shape = nullptr; self->dl_tensor.strides = nullptr;
      };
    }
  });
}
cuvsError_t cuvsCagraIndexGetGraph(cuvsCagraIndex_t index, DLManagedTensor* graph)
{
  return guarded([=] {
    auto& idx        = cagra_of(index);
    int64_t shape[2] = {idx.n, idx.degree};
    dl_fill_view(graph, const_cast<uint32_t*>(idx.graph), idx.device, DLDataType{kDLUInt, 32, 1}, 2, shape);
  });
}

cuvsError_t cuvsCagraIndexFromArgs(cuvsResources_t res, cuvsDistanceType metric, DLManagedTensor* graph_t, DLManagedTensor* dataset_t,
                                   cuvsCagraIndex_t index)
{
  return guarded([=] {
    auto r = as_res(res);
    B2_EXPECTS(graph_t && dataset_t && index, "null argument");
    const DLTensor& g = graph_t->dl_tensor;
    B2_EXPECTS(dl_is(g, kDLUInt, 32) && g.ndim == 2 && dl_is_c_contiguous(g), "graph must be a row-major uint32 matrix");
    auto idx    = std::make_unique<cagra_index>();
    idx->device = r->device;
    idx->metric = metric;
    set_dataset(r, *idx, dataset_t->dl_tensor);
    B2_EXPECTS(g.shape[0] == idx->n, "graph rows (%lld) != dataset rows (%lld)", (long long)g.shape[0], (long long)idx->n);
    B2_EXPECTS(idx->n < (int64_t(1) << 31), "cagra: at most 2^31 - 1 rows (the index MSB flags visited parents)");
    idx->degree = static_cast<int>(g.shape[1]);
    if (dl_is_device(g) && g.device.device_type != kDLCUDAHost) idx->graph = dl_ptr<uint32_t>(g);
    else {
      idx->graph_own.alloc(static_cast<size_t>(idx->n) * idx->degree);
      B2_CUDA(cudaMemcpyAsync(idx->graph_own.data(), dl_ptr<uint32_t>(g), sizeof(uint32_t) * idx->n * idx->degree, cudaMemcpyDefault, r->stream));
      idx->graph = idx->graph_own.data();
    }
    B2_CUDA(cudaStreamSynchronize(r->stream));
    if (index->addr) delete reinterpret_cast<cagra_index*>(index->addr);
    index->addr  = reinterpret_cast<uintptr_t>(idx.release());
    index->dtype = dataset_t->dl_tensor.dtype;
  });
}

cuvsError_t cuvsCagraBuild(cuvsResources_t res, cuvsCagraIndexParams_t params, DLManagedTensor* dataset_t, cuvsCagraIndex_t index)
{
  return guarded([=] {
    auto r = as_res(res);
    B2_EXPECTS(params && dataset_t && index, "null argument");
    B2_EXPECTS(params->compression == nullptr, "cagra build: VPQ compression is out of scope of this library");
    auto idx    = std::make_unique<cagra_index>();
    idx->device = r->device;
    idx->metric = params->metric;
    set_dataset(r, *idx, dataset_t->dl_tensor);
    const int64_t n = idx->n;
    B2_EXPECTS(n >= 2 && n < (int64_t(1) << 31), "cagra build: dataset size out of range");
    const int degree = static_cast<int>(std::min<int64_t>(static_cast<int64_t>(params->graph_degree), n - 1));
    B2_EXPECTS(degree >= 1, "graph_degree must be >= 1");
    // ---- kNN stage through the library's own scans: exact for small inputs, IVF-Flat self-search beyond
    const int di_want = static_cast<int>(std::max<size_t>(params->intermediate_graph_degree, static_cast<size_t>(degree)));
    const bool exact  = n <= 65536;
    const int di      = static_cast<int>(std::min<int64_t>(n - 1, exact ? std::min(di_want, 128) : std::min(di_want, 63)));
    const int kk      = di + 1;  // + self
    dbuf<float> compact;
    const float* data = idx->data;
    if (idx->ld != idx->dim) {  // the scans want unpadded rows
      compact.alloc(static_cast<size_t>(n) * idx->dim, r->stream);
      B2_CUDA(cudaMemcpy2DAsync(compact.data(), sizeof(float) * idx->dim, idx->data, sizeof(float) * idx->ld, sizeof(float) * idx->dim, n,
                                cudaMemcpyDeviceToDevice, r->stream));
      data = compact.data();
    }
    dbuf<int64_t> knn(static_cast<size_t>(n) * kk, r->stream);
    if (exact) build_knn_graph(res, r, data, n, idx->dim, idx->metric, kk, knn.data());
    else build_knn_graph_ivf(res, r, data, n, idx->dim, idx->metric, kk, knn.data());
    // ---- self-free neighbour rows, detour pruning, reverse-edge augmentation
    dbuf<uint32_t> nbr(static_cast<size_t>(n) * di, r->stream);
    count_launch(4);
    knn_to_graph_kernel<<<blocks_for(n, 128), 128, 0, r->stream>>>(knn.data(), n, kk, di, nbr.data(), di);
    dbuf<uint32_t> counts(static_cast<size_t>(n) * di, r->stream);
    detour_count_kernel<<<static_cast<unsigned>(n), 128, sizeof(uint32_t) * 2 * di, r->stream>>>(nbr.data(), n, di, counts.data());
    dbuf<uint32_t> fwd(static_cast<size_t>(n) * degree, r->stream);
    select_pruned_kernel<<<blocks_for(n, 128), 128, 0, r->stream>>>(nbr.data(), counts.data(), n, di, degree, fwd.data());
    const int keep    = std::max(1, degree / 2);
    const int rev_cap = degree;
    dbuf<uint32_t> rev(static_cast<size_t>(n) * rev_cap, r->stream), rev_cnt(static_cast<size_t>(n), r->stream);
    dbuf<uint32_t> src(static_cast<size_t>(n) * keep, r->stream);
    dbuf<int64_t> start;
    {
      dbuf<uint32_t> tgt(static_cast<size_t>(n) * keep, r->stream);
      count_launch();
      forward_edges_kernel<<<blocks_for(n * keep, 256), 256, 0, r->stream>>>(fwd.data(), n, degree, keep, tgt.data(), src.data());
      group_by_key(r->stream, tgt, src, n, start);
    }
    count_launch();
    reverse_edges_kernel<<<blocks_for(n, 256), 256, 0, r->stream>>>(src.data(), start.data(), n, rev.data(), rev_cnt.data(), rev_cap);
    idx->graph_own.alloc(static_cast<size_t>(n) * degree);
    merge_graph_kernel<<<blocks_for(n, 128), 128, 0, r->stream>>>(fwd.data(), rev.data(), rev_cnt.data(), n, degree, keep, rev_cap, idx->graph_own.data());
    B2_CUDA(cudaGetLastError());
    B2_CUDA(cudaStreamSynchronize(r->stream));
    idx->graph  = idx->graph_own.data();
    idx->degree = degree;
    if (index->addr) delete reinterpret_cast<cagra_index*>(index->addr);
    index->addr  = reinterpret_cast<uintptr_t>(idx.release());
    index->dtype = dataset_t->dl_tensor.dtype;
  });
}

cuvsError_t cuvsCagraSearch(cuvsResources_t res, cuvsCagraSearchParams_t params, cuvsCagraIndex_t index, DLManagedTensor* queries_t,
                            DLManagedTensor* neighbors_t, DLManagedTensor* distances_t, cuvsFilter filter)
{
  return guarded([=] {
    auto r = as_res(res);
    B2_EXPECTS(params && queries_t && neighbors_t && distances_t, "null argument");
    auto& idx = cagra_of(index);
    const DLTensor& queries   = queries_t->dl_tensor;
    const DLTensor& neighbors = neighbors_t->dl_tensor;
    const DLTensor& distances = distances_t->dl_tensor;
    // checks as in c/src/neighbors/cagra.cpp:646-690
    B2_EXPECTS(dl_is_device(queries), "queries should have device compatible memory");
    B2_EXPECTS(dl_is_device(neighbors), "neighbors should have device compatible memory");
    B2_EXPECTS(dl_is_device(distances), "distances should have device compatible memory");
    B2_EXPECTS(dl_is(neighbors, kDLUInt, 32) || dl_is(neighbors, kDLInt, 64), "neighbors should be of type uint32_t or int64_t");
    B2_EXPECTS(dl_is(distances, kDLFloat, 32), "distances should be of type float32");
    B2_EXPECTS(queries.dtype.code == index->dtype.code && queries.dtype.bits == index->dtype.bits, "type mismatch between index and queries");
    B2_EXPECTS(queries.ndim == 2 && neighbors.ndim == 2 && distances.ndim == 2, "queries/neighbors/distances must be 2-D");
    B2_EXPECTS(dl_is_c_contiguous(queries) && dl_is_c_contiguous(neighbors) && dl_is_c_contiguous(distances), "tensors must be row-major contiguous");
    B2_EXPECTS(queries.shape[1] == idx.dim, "queries dim (%lld) != index dim (%d)", (long long)queries.shape[1], idx.dim);
    B2_EXPECTS(neighbors.shape[0] == queries.shape[0] && distances.shape[0] == queries.shape[0] && distances.shape[1] == neighbors.shape[1], "neighbors/distances shape mismatch");
    const uint32_t* keep = nullptr;
    int64_t n_bits       = 0;
    if (filter.type != NO_FILTER) {
      B2_EXPECTS(filter.type == BITSET, "cagra search: only bitset pre-filters are supported (c/src/neighbors/cagra.cpp)");
      auto ft = reinterpret_cast<DLManagedTensor*>(filter.addr);
      B2_EXPECTS(ft != nullptr && dl_is_device(ft->dl_tensor), "prefilter should have device compatible memory");
      keep   = dl_ptr<uint32_t>(ft->dl_tensor);
      n_bits = ft->dl_tensor.shape[0] * 32;
    }
    const bool u32 = dl_is(neighbors, kDLUInt, 32);
    f32_matrix wq;
    widen_to_f32(r, queries, wq);
    cagra_search(r, idx, *params, dl_ptr<float>(wq.t), queries.shape[0], static_cast<int>(neighbors.shape[1]),
                 u32 ? dl_ptr<uint32_t>(neighbors) : nullptr, u32 ? nullptr : dl_ptr<int64_t>(neighbors), dl_ptr<float>(distances),
                 keep, n_bits);
  });
}

// cuVS index file, serialization version 5 (cpp/src/neighbors/detail/cagra/cagra_serialize.cuh:30-85, :270-320; dataset
// records cpp/src/neighbors/detail/dataset_serialize.hpp:30-200): the 4-byte dtype tag "<f4\0", then NPY records
// (npy_io.hpp) — version i4 = 5, size u4, dim u4, graph_degree u4, metric i4, graph u4 [size, graph_degree],
// content_map u4 (bit 0: dataset follows, bit 1: source indices follow); dataset = instance tag u4 (1 empty: suggested_dim
// u4 | 2 strided: cudaDataType u4, n_rows i8, dim u4, stride u4, data [n_rows, dim] without the row padding).
cuvsError_t cuvsCagraSerialize(cuvsResources_t res, const char* filename, cuvsCagraIndex_t index, bool include_dataset)
{
  return guarded([=] {
    auto r    = as_res(res);
    auto& idx = cagra_of(index);
    std::ofstream os(filename, std::ios::out | std::ios::binary);
    B2_EXPECTS(bool(os), "Cannot open file %s", filename);
    const char tag[4] = {'<', 'f', '4', 0};
    os.write(tag, 4);
    npy::write_scalar<int32_t>(os, 5);
    npy::write_scalar<uint32_t>(os, static_cast<uint32_t>(idx.n));
    npy::write_scalar<uint32_t>(os, static_cast<uint32_t>(idx.dim));
    npy::write_scalar<uint32_t>(os, static_cast<uint32_t>(idx.degree));
    npy::write_scalar<int32_t>(os, static_cast<int32_t>(idx.metric));
    std::vector<uint32_t> g(static_cast<size_t>(idx.n) * idx.degree);
    B2_CUDA(cudaMemcpyAsync(g.data(), idx.graph, g.size() * 4, cudaMemcpyDeviceToHost, r->stream));
    B2_CUDA(cudaStreamSynchronize(r->stream));
    npy::write_array<uint32_t>(os, g.data(), {idx.n, idx.degree});
    const bool with_data = include_dataset && idx.n > 0 && idx.data != nullptr;
    npy::write_scalar<uint32_t>(os, with_data ? 1u : 0u);
    if (with_data) {
      npy::write_scalar<uint32_t>(os, 2u);                       // kSerializeStridedDataset
      npy::write_scalar<uint32_t>(os, static_cast<uint32_t>(CUDA_R_32F));
      npy::write_scalar<int64_t>(os, idx.n);
      npy::write_scalar<uint32_t>(os, static_cast<uint32_t>(idx.dim));
      npy::write_scalar<uint32_t>(os, static_cast<uint32_t>(idx.ld));
      std::vector<float> d(static_cast<size_t>(idx.n) * idx.dim);
      B2_CUDA(cudaMemcpy2DAsync(d.data(), sizeof(float) * idx.dim, idx.data, sizeof(float) * idx.ld, sizeof(float) * idx.dim, idx.n, cudaMemcpyDeviceToHost, r->stream));
      B2_CUDA(cudaStreamSynchronize(r->stream));
      npy::write_array<float>(os, d.data(), {idx.n, idx.dim});
    }
    B2_EXPECTS(bool(os), "Error writing %s", filename);
  });
}

cuvsError_t cuvsCagraDeserialize(cuvsResources_t res, const char* filename, cuvsCagraIndex_t index)
{
  return guarded([=] {
    auto r = as_res(res);
    B2_EXPECTS(index && filename, "null argument");
    std::ifstream is(filename, std::ios::in | std::ios::binary);
    B2_EXPECTS(bool(is), "Cannot open file %s", filename);
    char tag[4]{};
    B2_EXPECTS(bool(is.read(tag, 4)), "cagra::deserialize: failed to read dtype prefix");
    B2_EXPECTS(tag[0] == '<' && tag[1] == 'f' && tag[2] == '4', "cagra::deserialize: serialized dtype prefix does not match requested type");
    const int ver = npy::read_scalar<int32_t>(is, filename);
    B2_EXPECTS(ver == 5, "serialization version mismatch, expected %d, got %d ", 5, ver);
    auto idx    = std::make_unique<cagra_index>();
    idx->device = r->device;
    idx->n      = npy::read_scalar<uint32_t>(is, filename);
    idx->dim    = static_cast<int>(npy::read_scalar<uint32_t>(is, filename));
    idx->degree = static_cast<int>(npy::read_scalar<uint32_t>(is, filename));
    idx->metric = static_cast<cuvsDistanceType>(npy::read_scalar<int32_t>(is, filename));
    idx->ld     = (idx->dim + 3) & ~3;
    std::vector<uint32_t> g(static_cast<size_t>(idx->n) * idx->degree);
    npy::read_array<uint32_t>(is, g.data(), static_cast<int64_t>(g.size()), filename);
    const uint32_t content_map = npy::read_scalar<uint32_t>(is, filename);
    B2_EXPECTS(content_map & 1u, "index file %s was saved without the dataset; use cuvsCagraIndexFromArgs to attach one", filename);
    const uint32_t inst = npy::read_scalar<uint32_t>(is, filename);
    B2_EXPECTS(inst == 2u, "cagra::deserialize: dataset instance tag %u is not supported by this build (strided fp32 datasets only)", inst);
    const uint32_t dt = npy::read_scalar<uint32_t>(is, filename);
    B2_EXPECTS(dt == static_cast<uint32_t>(CUDA_R_32F), "Failed to deserialize dataset: unsupported strided dataset element type %u.", dt);
    const int64_t rows = npy::read_scalar<int64_t>(is, filename);
    const uint32_t dim = npy::read_scalar<uint32_t>(is, filename);
    (void)npy::read_scalar<uint32_t>(is, filename);  // stride of the writer's device copy; rows are stored unpadded
    B2_EXPECTS(rows == idx->n && static_cast<int>(dim) == idx->dim, "cagra::deserialize: dataset [%lld, %u] does not match the graph [%lld rows], dim %d",
               (long long)rows, dim, (long long)idx->n, idx->dim);
    std::vector<float> d(static_cast<size_t>(idx->n) * idx->dim);
    npy::read_array<float>(is, d.data(), static_cast<int64_t>(d.size()), filename);
    idx->graph_own.alloc(g.size());
    idx->data_own.alloc(static_cast<size_t>(idx->n) * idx->ld);
    B2_CUDA(cudaMemcpyAsync(idx->graph_own.data(), g.data(), g.size() * 4, cudaMemcpyHostToDevice, r->stream));
    B2_CUDA(cudaMemsetAsync(idx->data_own.data(), 0, sizeof(float) * idx->n * idx->ld, r->stream));
    B2_CUDA(cudaMemcpy2DAsync(idx->data_own.data(), sizeof(float) * idx->ld, d.data(), sizeof(float) * idx->dim, sizeof(float) * idx->dim, idx->n, cudaMemcpyHostToDevice, r->stream));
    B2_CUDA(cudaStreamSynchronize(r->stream));
    idx->graph = idx->graph_own.data();
    idx->data  = idx->data_own.data();
    if (index->addr) delete reinterpret_cast<cagra_index*>(index->addr);
    index->addr  = reinterpret_cast<uintptr_t>(idx.release());
    index->dtype = DLDataType{kDLFloat, 32, 1};
  });
}

cuvsError_t cuvsCagraExtend(cuvsResources_t, cuvsCagraExtendParams_t, DLManagedTensor*, cuvsCagraIndex_t)
{
  return guarded([=] { B2_FAIL("cuvsCagraExtend: graph construction/extension is outside the scan+top-k hot path of this library (SURVEY §8a: build OUT OF SCOPE)"); });
}
cuvsError_t cuvsCagraSerializeToHnswlib(cuvsResources_t, const char*, cuvsCagraIndex_t)
{
  return guarded([=] { B2_FAIL("cuvsCagraSerializeToHnswlib: the hnswlib (CPU) path is out of scope of this library"); });
}
cuvsError_t cuvsCagraMerge(cuvsResources_t, cuvsCagraIndexParams_t, cuvsCagraIndex_t*, size_t, cuvsFilter, cuvsCagraIndex_t)
{
  return guarded([=] { B2_FAIL("cuvsCagraMerge: graph construction is outside the scan+top-k hot path of this library"); });
}

/* cuvs_b200 extension (include/cuvs_b200/ext.h): bits = 16 keeps an fp16 copy of the vectors for the graph walk (results are
 * re-ranked with the fp32 rows); bits = 32 drops it. */
cuvsError_t cuvsB200CagraSetWalkPrecision(cuvsResources_t res, cuvsCagraIndex_t index, int bits)
{
  return guarded([=] {
    auto r    = as_res(res);
    auto& idx = cagra_of(index);
    B2_EXPECTS(bits == 16 || bits == 32, "walk precision must be 16 or 32 bits");
    if (bits == 32) { idx.data16.release(); idx.ld16 = 0; return; }
    idx.ld16 = (idx.dim + 7) & ~7;
    idx.data16.alloc(static_cast<size_t>(idx.n) * idx.ld16);
    count_launch();
    to_half_rows_kernel<<<blocks_for(idx.n * idx.ld16, 256), 256, 0, r->stream>>>(idx.data, idx.n, idx.dim, idx.ld, idx.ld16, idx.data16.data());
    B2_CUDA(cudaGetLastError());
  });
}

}  // extern "C"
