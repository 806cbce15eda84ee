// IVF-PQ: index, build / extend, search, C boundary.
//
// Reference path being replaced (SURVEY §8a rows a9-a13):
//   index / list layout   cpp/include/cuvs/neighbors/ivf_pq.hpp:476-660, :235-296
//   build                 cpp/src/neighbors/ivf_pq/ivf_pq_build.cuh:1231-1390 (k-means, rotation, codebooks, encode)
//   search host logic     cpp/src/neighbors/ivf_pq/ivf_pq_search.cuh:881-1048, select_clusters :60-168
//   compute_similarity    cpp/src/neighbors/ivf_pq/detail/jit_lto_kernels/{compute_similarity,create_lut,
//                         compute_score,compute_distances}_impl.cuh
//   fp_8bit               cpp/src/neighbors/ivf_pq/ivf_pq_fp_8bit.cuh:31-100
//   C wrapper             c/src/neighbors/ivf_pq.cpp
//
// Two fine-scan kernels sit behind cuvsIvfPqSearch (DESIGN.md §5):
//   (A) pq_lut_scan_kernel — the reference's formulation restated for B200: one CTA per (query, probe),
//       LUT[pq_dim x 2^bits] in shared memory (fp32 / fp16 / fp_8bit<5>), codes streamed with 128-bit
//       loads, scores accumulated in subspace order (bit-identical to oracle/oracle.c for fp32), block-level
//       threshold filter + rank compaction for the top-k'.  Work is bound by shared-memory LUT gathers
//       (one 4-byte bank access per code) — 4.0e11 gathers per 10k-query batch at config C2.
//   (B) decoded-tile scan on tcgen05 — score(x) = sum_i lut[i, code_i] is algebraically
//       |r - y(x)|^2 with r = R q - c_rot[list] and y(x) the concatenation of the PQ centres selected by
//       the codes; the index keeps y(x) as bf16 rows (codebook entries are rounded to bf16 at training
//       time so the rows are exact), pairs are bucketed by list and each list tile is contracted against
//       up to 128 probing queries at once on the tensor cores (ivf_common.cu + scan_tc.cu).  This removes
//       the per-(query,probe) LUT build and the 4e11 shared-memory gathers altogether.
// (B) is used when lut_dtype == internal_distance_dtype == fp32 and the index holds decoded rows
// (conservative_memory_allocation == false); (A) otherwise or with CUVS_B200_PQ_PATH=lut.
#include "common.hpp"
#include "exact.cuh"
#include "ivf_common.cuh"
#include "ivf_lists.cuh"
#include "npy_io.hpp"
#include "scan_pq.cuh"
#include "select_k.cuh"
#include "timing.hpp"

#include <cuvs/neighbors/ivf_pq.h>
#include <cuvs_b200/ext.h>

#include <cuda_fp16.h>

#include <algorithm>
#include <cfloat>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <memory>
#include <random>
#include <vector>

namespace b200 {

struct ivf_pq_index {
  int device              = 0;
  cuvsDistanceType metric = L2Expanded;
  float metric_arg        = 2.0f;
  int dim = 0, dim_ext = 0, rot_dim = 0, pq_dim = 0, pq_len = 0, pq_bits = 8;
  uint32_t n_lists        = 0;
  int codebook_kind       = CUVS_IVF_PQ_CODEBOOK_GEN_PER_SUBSPACE;
  bool conservative       = false;
  uint32_t kmeans_n_iters = 20;
  owned<float> centers;      // [n_lists, dim]      (compact)
  owned<float> centers_ext;  // [n_lists, dim_ext]  (reference layout: col dim = |c|^2, rest 0)
  owned<float> centers_rot;  // [n_lists, rot_dim]
  owned<float> rotation;     // [rot_dim, dim]
  owned<float> pq_centers;   // PER_SUBSPACE [pq_dim, pq_len, book] | PER_CLUSTER [n_lists, pq_len, book]
  tc_rows centers_tc;
  list_layout lists;
  // [rows_total, pq_dim], one code per byte.  When the index is served by the code-streaming scan the stream below IS the
  // index and this flat copy is dropped after (re)building it; ensure_flat_codes() re-materialises it for the paths that
  // want rows (getters, extend, serialize, the LUT kernel).
  mutable owned<uint8_t> codes;
  owned<int64_t> ids;    // [rows_total], kPadId on padding rows
  // decoded side (path B)
  int Kp = 0;
  owned<__nv_bfloat16> yhat;  // [rows_total, Kp]
  owned<__nv_bfloat16> hx;    // [rows_total, 16] half-norm plane: |y|^2/2 (0 for inner product), +inf on padding rows
  // streamed side (path C, scan_pq.cu): lane-transposed code tiles + half norms, bank-transposed bf16x2 codebook words.
  // When the shape is served by the code-streaming kernel the decoded rows above are NOT kept (pq_dim + 4 bytes per
  // vector instead of 2 * rot_dim + 32).
  owned<uint8_t> cstream;    // [rows_total / 128, pq_stream_tile_bytes(pq_dim)]
  owned<uint32_t> cb_words;  // [pq_dim / 32, 256, 32]
  int book() const { return 1 << pq_bits; }
};

namespace {

void ensure_flat_codes(resources* res, const ivf_pq_index& idx)
{
  const size_t need = static_cast<size_t>(std::max<int64_t>(idx.lists.rows_total, 1)) * idx.pq_dim;
  if (idx.codes.data() != nullptr && idx.codes.size() >= need) return;
  B2_EXPECTS(idx.cstream.data() != nullptr, "ivf_pq: the index holds neither flat codes nor a code stream");
  idx.codes.alloc(need);
  pq_stream_to_flat(res->stream, idx.cstream.data(), idx.lists.rows_total, idx.pq_dim, idx.codes.data());
}
bool is_ip(cuvsDistanceType m) { return m == InnerProduct || m == CosineExpanded; }

// ------------------------------------------------------------------ fp_8bit<5, Signed> (ivf_pq_fp_8bit.cuh:31-100)
template <bool Signed>
struct fp8 {
  uint8_t bits;
  static constexpr uint32_t ExpMask = 15u, ValBits = 3u;
  __device__ __forceinline__ static fp8 from_float(float v)
  {
    const float kMin = 1.0f / float(1u << ExpMask);
    const float kMax = float(1u << (ExpMask + 1)) * (2.0f - 1.0f / float(1u << ValBits));
    float a = Signed ? fabsf(v) : v;
    uint8_t u;
    if (a < kMin) u = 0;
    else if (a >= kMax) u = 0xffu;
    else u = static_cast<uint8_t>((__float_as_uint(a) + (ExpMask << 23u) - 0x3f800000u) >> 20u);
    if (Signed) u = static_cast<uint8_t>((u & 0xfeu) | (v < 0 ? 1u : 0u));
    return fp8{u};
  }
  __device__ __forceinline__ float to_float() const
  {
    uint32_t u = bits;
    if (Signed) u &= ~1u;
    constexpr uint32_t kBase32 = (0x3f800000u | (0x00400000u >> ValBits)) - (ExpMask << 23);
    float r = __uint_as_float(kBase32 + (u << 20u));
    if (Signed && (bits & 1)) r = -r;
    return r;
  }
};

template <typename LutT> struct lut_conv;
template <> struct lut_conv<float> {
  __device__ static float enc(float v, bool) { return v; }
  __device__ static float dec(float v, bool) { return v; }
};
template <> struct lut_conv<__half> {
  __device__ static __half enc(float v, bool) { return __float2half_rn(v); }
  __device__ static float dec(__half v, bool) { return __half2float(v); }
};
template <> struct lut_conv<uint8_t> {
  __device__ static uint8_t enc(float v, bool sgn) { return sgn ? fp8<true>::from_float(v).bits : fp8<false>::from_float(v).bits; }
  __device__ static float dec(uint8_t v, bool sgn) { return sgn ? fp8<true>{v}.to_float() : fp8<false>{v}.to_float(); }
};

// ------------------------------------------------------------------ build-side kernels
__global__ void residual_kernel(const float* __restrict__ x_rot, const uint32_t* __restrict__ labels,
                                const float* __restrict__ centers_rot, int64_t n, int rot_dim, float* __restrict__ out)
{
  int64_t t = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  if (t >= n * rot_dim) return;
  int64_t r = t / rot_dim;
  int c     = static_cast<int>(t % rot_dim);
  out[t]    = x_rot[t] - centers_rot[static_cast<int64_t>(labels[r]) * rot_dim + c];
}

// nearest code per (point, subspace).  grid (ceil(n/128), n_books); codebook of this book in smem.
// book_of_row: PER_SUBSPACE -> blockIdx.y is the subspace; PER_CLUSTER -> handled by the caller with labels.
__global__ void __launch_bounds__(128) pq_assign_kernel(const float* __restrict__ resid /*[n, rot_dim]*/, int64_t n, int rot_dim,
                                                         int pq_dim, int pq_len, int book,
                                                         const float* __restrict__ pq_centers, int per_cluster,
                                                         const uint32_t* __restrict__ labels, uint8_t* __restrict__ codes,
                                                         const int64_t* __restrict__ dst_rows /*nullable*/)
{
  extern __shared__ float cb[];  // [pq_len][book]
  const int sub = blockIdx.y;
  if (!per_cluster) {
    for (int i = threadIdx.x; i < pq_len * book; i += blockDim.x) cb[i] = pq_centers[static_cast<int64_t>(sub) * pq_len * book + i];
    __syncthreads();
  }
  int64_t r = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  if (r >= n) return;
  const float* c = per_cluster ? pq_centers + static_cast<int64_t>(labels[r]) * pq_len * book : cb;
  float v[32];
  for (int t = 0; t < pq_len; ++t) v[t] = resid[r * rot_dim + sub * pq_len + t];
  float best = FLT_MAX;
  int bc     = 0;
  for (int code = 0; code < book; ++code) {
    float acc = 0.f;
    for (int t = 0; t < pq_len; ++t) { float df = v[t] - c[t * book + code]; acc = fmaf(df, df, acc); }
    if (acc < best) { best = acc; bc = code; }
  }
  int64_t o = dst_rows ? dst_rows[r] : r;
  codes[o * pq_dim + sub] = static_cast<uint8_t>(bc);
}

// codebook entry (book b, code) of every (row, subspace) item: key b * book + code
__global__ void pq_keys_kernel(int64_t n, int pq_dim, int book, const uint8_t* __restrict__ codes, int per_cluster,
                               const uint32_t* __restrict__ labels, uint32_t* __restrict__ keys)
{
  int64_t t = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  if (t >= n * pq_dim) return;
  const int64_t b = per_cluster ? labels[t / pq_dim] : t % pq_dim;
  keys[t]         = static_cast<uint32_t>(b * book + codes[t]);
}

// one warp per codebook entry: lanes stride over its items in item order and the lane sums are combined by a fixed shuffle
// tree, so the sums do not depend on scheduling (same input, same codebooks, run after run)
__global__ void pq_segment_sums_kernel(const float* __restrict__ resid, int rot_dim, int pq_dim, int pq_len, int book,
                                       int64_t n_entries, const uint32_t* __restrict__ order, const int64_t* __restrict__ start,
                                       float* __restrict__ sums, float* __restrict__ counts)
{
  const int64_t g = (blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x) >> 5;
  const int lane  = threadIdx.x & 31;
  if (g >= n_entries) return;
  const int64_t b = g / book, s0 = start[g], s1 = start[g + 1];
  const int code  = static_cast<int>(g % book);
  for (int j = 0; j < pq_len; ++j) {
    float acc = 0.f;
    for (int64_t p = s0 + lane; p < s1; p += 32) {
      const int64_t t = order[p];
      acc += resid[(t / pq_dim) * rot_dim + (t % pq_dim) * pq_len + j];
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (lane == 0) sums[(b * pq_len + j) * book + code] = acc;
  }
  if (lane == 0) counts[g] = static_cast<float>(s1 - s0);
}

__global__ void pq_finalize_kernel(float* __restrict__ pq_centers, const float* __restrict__ sums, const float* __restrict__ counts,
                                   int64_t n_books, int pq_len, int book, const float* __restrict__ resid, int64_t n, int rot_dim,
                                   int pq_dim, int iter, bool round_bf16)
{
  int64_t t = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  if (t >= n_books * book) return;
  int64_t b = t / book;
  int code  = static_cast<int>(t % book);
  float cnt = counts[t];
  for (int j = 0; j < pq_len; ++j) {
    float v;
    if (cnt > 0.f) v = sums[(b * pq_len + j) * book + code] / cnt;
    else {
      // empty code: re-seed from a pseudo-random training residual
      uint64_t h = (static_cast<uint64_t>(iter + 1) * 0x9e3779b97f4a7c15ull) ^ (static_cast<uint64_t>(t) * 0xbf58476d1ce4e5b9ull);
      h ^= h >> 29;
      int64_t row = static_cast<int64_t>(h % static_cast<uint64_t>(n));
      int sub     = static_cast<int>(b % pq_dim);
      v           = resid[row * rot_dim + sub * pq_len + j];
    }
    if (round_bf16) v = __bfloat162float(__float2bfloat16_rn(v));
    pq_centers[(b * pq_len + j) * book + code] = v;
  }
}

__global__ void pq_init_kernel(float* __restrict__ pq_centers, int64_t n_books, int pq_len, int book, const float* __restrict__ resid,
                               int64_t n, int rot_dim, int pq_dim)
{
  int64_t t = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  if (t >= n_books * book) return;
  int64_t b   = t / book;
  int code    = static_cast<int>(t % book);
  int64_t row = (static_cast<int64_t>(code) * n) / book;
  int sub     = static_cast<int>(b % pq_dim);
  for (int j = 0; j < pq_len; ++j) pq_centers[(b * pq_len + j) * book + code] = resid[row * rot_dim + sub * pq_len + j];
}

// decoded bf16 rows + half norms from codes (path B).  one warp per row.
__global__ void pq_decode_kernel(const uint8_t* __restrict__ codes, const int64_t* __restrict__ ids, int64_t rows, int pq_dim,
                                 int pq_len, int book, int Kp, const float* __restrict__ pq_centers, int per_cluster,
                                 const int64_t* __restrict__ list_offsets, int64_t n_lists, bool ip,
                                 const float* __restrict__ centers_rot, int rot_dim, __nv_bfloat16* __restrict__ yhat,
                                 float* __restrict__ hn)
{
  int64_t r = (blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x) >> 5;
  int lane  = threadIdx.x & 31;
  if (r >= rows) return;
  const bool pad = ids[r] == kPadId;
  int64_t list   = 0;
  if (per_cluster || ip) {  // binary search of the owning list
    int64_t lo = 0, hi = n_lists;
    while (hi - lo > 1) { int64_t mid = (lo + hi) >> 1; if (list_offsets[mid] <= r) lo = mid; else hi = mid; }
    list = lo;
  }
  float nrm = 0.f;
  for (int j = lane; j < Kp; j += 32) {
    float v = 0.f;
    if (!pad && j < pq_dim * pq_len) {
      int sub = j / pq_len, t = j % pq_len;
      int code = codes[r * pq_dim + sub];
      int64_t b = per_cluster ? list : sub;
      v = pq_centers[(b * pq_len + t) * book + code];
      if (ip) v += centers_rot[list * rot_dim + j];  // inner product scans the full reconstruction
    }
    __nv_bfloat16 hv = __float2bfloat16_rn(v);
    yhat[r * Kp + j] = hv;
    float f = __bfloat162float(hv);
    nrm = fmaf(f, f, nrm);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) nrm += __shfl_xor_sync(0xffffffffu, nrm, o);
  if (lane == 0) hn[r] = pad ? INFINITY : (ip ? 0.f : 0.5f * nrm);
}

__global__ void make_centers_ext_kernel(const float* __restrict__ centers, int64_t n_lists, int dim, int dim_ext,
                                        float* __restrict__ ext)
{
  int64_t l = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  if (l >= n_lists) return;
  float nrm = 0.f;
  for (int j = 0; j < dim; ++j) { float v = centers[l * dim + j]; ext[l * dim_ext + j] = v; nrm = fmaf(v, v, nrm); }
  for (int j = dim; j < dim_ext; ++j) ext[l * dim_ext + j] = (j == dim) ? nrm : 0.f;
}

// ------------------------------------------------------------------ search-side kernels
// per pair: r = q_rot[query] - c_rot[list] (L2) or q_rot[query] (IP) as bf16 A rows; add[slot] = |r|^2 (L2) or 0 (IP)
__global__ void pair_rows_kernel(const float* __restrict__ q_rot, const float* __restrict__ centers_rot,
                                 const uint32_t* __restrict__ pair_query, const uint32_t* __restrict__ pair_list,
                                 const int* __restrict__ n_live, int64_t rows_total, int rot_dim, int Kp, bool ip,
                                 __nv_bfloat16* __restrict__ a_hi,
                                 __nv_bfloat16* __restrict__ a_lo, float* __restrict__ add, bool ip_center_in_add)
{
  int64_t r = (blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x) >> 5;
  int lane  = threadIdx.x & 31;
  if (r >= rows_total) return;
  float nrm = 0.f;
  const bool live = r < *n_live;
  const float* qr = live ? q_rot + static_cast<int64_t>(pair_query[r]) * rot_dim : nullptr;
  const float* cr = live ? centers_rot + static_cast<int64_t>(pair_list[r]) * rot_dim : nullptr;
  for (int j = lane; j < Kp; j += 32) {
    float v = 0.f;
    if (live && j < rot_dim) v = ip ? qr[j] : qr[j] - cr[j];
    __nv_bfloat16 h = __float2bfloat16_rn(v);
    a_hi[r * Kp + j] = h;
    if (a_lo) a_lo[r * Kp + j] = __float2bfloat16_rn(v - __bfloat162float(h));
    // L2: |r|^2.  Inner product over code-only rows (the streamed scan decodes y, not c + y): -(q . c) of the pair
    nrm = (ip && ip_center_in_add) ? ((live && j < rot_dim) ? fmaf(-qr[j], cr[j], nrm) : nrm) : fmaf(v, v, nrm);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) nrm += __shfl_xor_sync(0xffffffffu, nrm, o);
  if (lane == 0 && live) add[r] = (ip && !ip_center_in_add) ? 0.f : nrm;
}

// out[q, p*KCW + c] = add[slot] + scale * s   (per-query concatenation of its probes' candidates)
__global__ void gather_pq_cands_kernel(const float* __restrict__ cs, const uint32_t* __restrict__ cp,
                                       const uint32_t* __restrict__ slot_of, const float* __restrict__ add, float scale,
                                       int64_t total, int KCW, float* __restrict__ out_score, uint32_t* __restrict__ out_pos)
{
  int64_t t = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  if (t >= total) return;
  int64_t pair  = t / KCW;
  int c         = static_cast<int>(t % KCW);
  uint32_t slot = slot_of[pair];
  float s       = FLT_MAX;
  uint32_t p    = 0xffffffffu;
  if (slot != 0xffffffffu) {
    p = cp[static_cast<int64_t>(slot) * KCW + c];
    if (p != 0xffffffffu) s = (add ? add[slot] : 0.f) + scale * cs[static_cast<int64_t>(slot) * KCW + c];
  }
  out_score[t] = s;
  out_pos[t]   = p;
}

__global__ void finish_ids_kernel(const uint32_t* __restrict__ pos, const int64_t* __restrict__ ids, float* __restrict__ dist,
                                  int64_t count, int metric, int64_t* __restrict__ out_idx)
{
  int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  if (i >= count) return;
  uint32_t p = pos[i];
  float d    = dist[i];
  if (p == 0xffffffffu) {
    out_idx[i] = INT64_MAX;  // kOutOfBoundsRecord (ivf_common.cuh:25-31)
    dist[i]    = (metric == InnerProduct) ? -FLT_MAX : FLT_MAX;
    return;
  }
  out_idx[i] = ids[p];
  // ivf_common.cuh:175-252 postprocess_distances
  if (metric == L2SqrtExpanded || metric == L2SqrtUnexpanded) d = sqrtf(fmaxf(d, 0.f));
  else if (metric == InnerProduct) d = -d;
  dist[i] = d;
}

// ---- (A) LUT scan: one CTA per (query, probe) slot ------------------------------------------------
constexpr int kLutThreads = 128;
constexpr int kLutBuf     = 256;  // candidate buffer (entries) per CTA

template <typename LutT, typename OutT>
__global__ void __launch_bounds__(kLutThreads)
pq_lut_scan_kernel(const float* __restrict__ q_rot, const float* __restrict__ centers_rot, const float* __restrict__ pq_centers,
                   int per_cluster, const uint8_t* __restrict__ codes, const int64_t* __restrict__ list_offsets,
                   const uint32_t* __restrict__ list_sizes, const uint32_t* __restrict__ pair_query,
                   const uint32_t* __restrict__ pair_list, const int* __restrict__ n_live, int rot_dim, int pq_dim, int pq_len, int pq_bits, bool ip, bool cosine,
                   int KC, float* __restrict__ out_score, uint32_t* __restrict__ out_pos, int KCW)
{
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int book     = 1 << pq_bits;
  const int lut_size = pq_dim * book;
  LutT* lut          = reinterpret_cast<LutT*>(smem_raw);
  size_t off         = (static_cast<size_t>(lut_size) * sizeof(LutT) + 15) & ~size_t(15);
  float* resid       = reinterpret_cast<float*>(smem_raw + off);              // [rot_dim] (L2: q-c ; IP: q)
  float* qc          = resid + rot_dim;                                        // [rot_dim] IP only: q*c
  float* bv          = qc + rot_dim;                                           // [kLutBuf] candidate scores
  uint32_t* bp       = reinterpret_cast<uint32_t*>(bv + kLutBuf);              // [kLutBuf] candidate rows
  float* nv          = reinterpret_cast<float*>(bp + kLutBuf);                 // compaction scratch
  uint32_t* np       = reinterpret_cast<uint32_t*>(nv + kLutBuf);
  __shared__ int s_cnt;
  __shared__ float s_thr;

  const int64_t slot = blockIdx.x;
  if (slot >= *n_live) return;  // slots of probes that hit empty lists are never populated
  const uint32_t qi = pair_query[slot], l = pair_list[slot];
  const float* qr = q_rot + static_cast<int64_t>(qi) * rot_dim;
  const float* cr = centers_rot + static_cast<int64_t>(l) * rot_dim;
  for (int j = threadIdx.x; j < rot_dim; j += blockDim.x) {
    resid[j] = ip ? qr[j] : qr[j] - cr[j];
    qc[j]    = ip ? qr[j] * cr[j] : 0.f;
  }
  if (threadIdx.x == 0) { s_cnt = 0; s_thr = FLT_MAX; }
  __syncthreads();
  // create_lut_impl.cuh:40-77
  const float* pqc = per_cluster ? pq_centers + static_cast<int64_t>(l) * pq_len * book : pq_centers;
  for (int i = threadIdx.x; i < lut_size; i += blockDim.x) {
    const int sub = i >> pq_bits, code = i & (book - 1);
    float score = 0.f;
    for (int t = 0; t < pq_len; ++t) {
      const int j  = sub * pq_len + t;
      const float c = per_cluster ? pqc[t * book + code] : pqc[(static_cast<int64_t>(sub) * pq_len + t) * book + code];
      if (!ip) {
        float df = resid[j];
        df -= c;
        score = fmaf(df, df, score);
      } else {
        score -= qc[j];
        score = fmaf(-resid[j], c, score);
      }
    }
    lut[i] = lut_conv<LutT>::enc(score, ip);
  }
  __syncthreads();

  const int64_t row0 = list_offsets[l];
  const uint32_t n   = list_sizes[l];
  const int vec16    = pq_dim / 16;  // uint4 loads per row when pq_dim % 16 == 0
  const bool aligned = (pq_dim % 16 == 0);

  auto compact = [&](int keep) {
    // rank compaction: keep the `keep` best of the buffer, sorted, at the front
    __syncthreads();
    const int m = min(s_cnt, kLutBuf);
    for (int c = threadIdx.x; c < m; c += blockDim.x) {
      const float v = bv[c];
      const uint32_t p = bp[c];
      int rank = 0;
      for (int o = 0; o < m; ++o) {
        const float v2 = bv[o];
        rank += (v2 < v || (v2 == v && bp[o] < p)) ? 1 : 0;
      }
      if (rank < keep) { nv[rank] = v; np[rank] = p; }
    }
    __syncthreads();
    const int kept = min(m, keep);
    for (int c = threadIdx.x; c < kept; c += blockDim.x) { bv[c] = nv[c]; bp[c] = np[c]; }
    if (threadIdx.x == 0) { s_cnt = kept; if (kept == keep) s_thr = nv[keep - 1]; }
    __syncthreads();
  };

  for (uint32_t base = 0; base < n; base += blockDim.x) {
    const uint32_t i = base + threadIdx.x;
    if (i < n) {
      const uint8_t* code = codes + (row0 + i) * pq_dim;
      OutT score = OutT(0.f);
      if (aligned) {
        for (int v = 0; v < vec16; ++v) {
          const uint4 w = reinterpret_cast<const uint4*>(code)[v];
          const uint32_t ws[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
          for (int b = 0; b < 16; ++b) {
            const uint32_t cdx = (ws[b >> 2] >> ((b & 3) * 8)) & 0xffu;
            score += OutT(lut_conv<LutT>::dec(lut[((v * 16 + b) << pq_bits) + cdx], ip));
          }
        }
      } else {
        for (int s = 0; s < pq_dim; ++s) score += OutT(lut_conv<LutT>::dec(lut[(s << pq_bits) + code[s]], ip));
      }
      float fs = float(score);
      if (cosine) fs += 1.0f;
      if (fs < s_thr) {
        int at = atomicAdd(&s_cnt, 1);
        if (at < kLutBuf) { bv[at] = fs; bp[at] = static_cast<uint32_t>(row0 + i); }
      }
    }
    // one snapshot of s_cnt decides for the whole CTA (compact() has barriers inside): every thread votes AFTER all pushes
    // of this round and BEFORE anyone can push again
    if (__syncthreads_or(s_cnt > kLutBuf - static_cast<int>(blockDim.x))) compact(KC);
  }
  compact(KC);
  const int kept = s_cnt;
  for (int c = threadIdx.x; c < KCW; c += blockDim.x) {
    out_score[slot * KCW + c] = c < kept ? bv[c] : FLT_MAX;
    out_pos[slot * KCW + c]   = c < kept ? bp[c] : 0xffffffffu;
  }
}

// ------------------------------------------------------------------ host helpers
uint32_t calculate_pq_dim(uint32_t dim)
{
  // cpp/src/neighbors/ivf_pq_index.cu:612-622
  if (dim >= 128) dim /= 2;
  uint32_t r = dim / 32 * 32;
  if (r > 0) return r;
  r = 1;
  while ((r << 1) <= dim) r <<= 1;
  return r;
}

// random orthonormal-column matrix [rot_dim, dim] (host Gram-Schmidt), or identity-with-padding
std::vector<float> make_rotation(int rot_dim, int dim, bool random)
{
  std::vector<float> R(static_cast<size_t>(rot_dim) * dim, 0.f);
  if (!random) {
    for (int i = 0; i < std::min(rot_dim, dim); ++i) R[static_cast<size_t>(i) * dim + i] = 1.f;
    return R;
  }
  std::mt19937_64 rng(7ull);
  std::normal_distribution<double> nd(0.0, 1.0);
  std::vector<double> M(static_cast<size_t>(rot_dim) * rot_dim);
  for (auto& v : M) v = nd(rng);
  // orthonormalise the columns of M (modified Gram-Schmidt), keep the first `dim` columns
  for (int c = 0; c < rot_dim; ++c) {
    for (int p = 0; p < c; ++p) {
      double dot = 0;
      for (int r = 0; r < rot_dim; ++r) dot += M[static_cast<size_t>(r) * rot_dim + c] * M[static_cast<size_t>(r) * rot_dim + p];
      for (int r = 0; r < rot_dim; ++r) M[static_cast<size_t>(r) * rot_dim + c] -= dot * M[static_cast<size_t>(r) * rot_dim + p];
    }
    double nrm = 0;
    for (int r = 0; r < rot_dim; ++r) nrm += M[static_cast<size_t>(r) * rot_dim + c] * M[static_cast<size_t>(r) * rot_dim + c];
    nrm = std::sqrt(std::max(nrm, 1e-30));
    for (int r = 0; r < rot_dim; ++r) M[static_cast<size_t>(r) * rot_dim + c] /= nrm;
  }
  for (int r = 0; r < rot_dim; ++r)
    for (int c = 0; c < dim; ++c) R[static_cast<size_t>(r) * dim + c] = static_cast<float>(M[static_cast<size_t>(r) * rot_dim + c]);
  return R;
}

// out[n, rot_dim] = x[n, dim] . R^T   (exact fp32, ascending-k fmaf like the oracle)
void rotate_rows(cudaStream_t s, const float* x, int64_t n, int dim, const float* R, int rot_dim, float* out)
{
  const int64_t chunk = 65535 * 64;
  for (int64_t r0 = 0; r0 < n; r0 += chunk) {
    int64_t rows = std::min(chunk, n - r0);
    exact_distance_tile(s, x + r0 * dim, rows, dim, R, rot_dim, dim, dim, nullptr, nullptr, InnerProduct, out + r0 * rot_dim, rot_dim,
                        filter_view{}, 0);
  }
}

// Residuals R x - c_rot[label] [n, rot_dim] of the device rows x [n, dim]; when `codes` is given, also the nearest PQ code of
// every (row, subspace), stored at codes[(dst_rows ? dst_rows[i] : i) * pq_dim + subspace].
dbuf<float> encode_rows(resources* res, const ivf_pq_index& idx, const float* x, int64_t n, const uint32_t* labels,
                        uint8_t* codes = nullptr, const int64_t* dst_rows = nullptr)
{
  auto s = res->stream;
  dbuf<float> xr(static_cast<size_t>(n) * idx.rot_dim, s), rs(static_cast<size_t>(n) * idx.rot_dim, s);
  rotate_rows(s, x, n, idx.dim, idx.rotation.data(), idx.rot_dim, xr.data());
  count_launch();
  residual_kernel<<<blocks_for(n * idx.rot_dim, 256), 256, 0, s>>>(xr.data(), labels, idx.centers_rot.data(), n, idx.rot_dim, rs.data());
  if (codes) {
    const size_t smem = static_cast<size_t>(idx.pq_len) * idx.book() * sizeof(float);
    count_launch();
    pq_assign_kernel<<<dim3(blocks_for(n, 128), idx.pq_dim), 128, smem, s>>>(
      rs.data(), n, idx.rot_dim, idx.pq_dim, idx.pq_len, idx.book(), idx.pq_centers.data(),
      idx.codebook_kind == CUVS_IVF_PQ_CODEBOOK_GEN_PER_CLUSTER, labels, codes, dst_rows);
  }
  B2_CUDA(cudaGetLastError());
  return rs;
}

void refresh_centers(resources* res, ivf_pq_index& idx)
{
  auto s = res->stream;
  idx.centers_ext.alloc(static_cast<size_t>(idx.n_lists) * idx.dim_ext);
  count_launch();
  make_centers_ext_kernel<<<blocks_for(idx.n_lists, 128), 128, 0, s>>>(idx.centers.data(), idx.n_lists, idx.dim, idx.dim_ext,
                                                                        idx.centers_ext.data());
  dbuf<float> cn(static_cast<size_t>(idx.n_lists), s);
  row_norms(s, idx.centers.data(), idx.n_lists, idx.dim, idx.dim, cn.data());
  idx.centers_tc.build(s, idx.centers.data(), idx.n_lists, idx.dim, is_l2(idx.metric) ? cn.data() : nullptr, true);
}

void refresh_decoded(resources* res, ivf_pq_index& idx)
{
  auto s          = res->stream;
  const int64_t R = idx.lists.rows_total;
  idx.Kp          = tc_pad_k(idx.rot_dim);
  idx.cstream.release();
  idx.cb_words.release();
  if (idx.conservative || !tc_supported(res->device, idx.rot_dim)) { idx.yhat.release(); idx.hx.release(); return; }
  if (idx.Kp == idx.rot_dim &&
      pq_stream_supported(res->device, idx.pq_dim, idx.pq_len, idx.pq_bits, idx.codebook_kind == CUVS_IVF_PQ_CODEBOOK_GEN_PER_SUBSPACE)) {
    idx.cstream.alloc(static_cast<size_t>(std::max<int64_t>(R / 128, 1)) * pq_stream_tile_bytes(idx.pq_dim));
    idx.cb_words.alloc(static_cast<size_t>(idx.pq_dim / 32) * 256 * 32);
    pq_stream_build(s, idx.codes.data(), idx.ids.data(), kPadId, R, idx.pq_dim, idx.pq_centers.data(), is_ip(idx.metric),
                    idx.cstream.data(), idx.cb_words.data());
    // A SMALL index additionally caches its decoded rows (2 * rot_dim bytes per vector, derived data): when a batch sends
    // hundreds of queries to every list (10M vectors / 1024 lists / 10k x 64 probes = 625 per list) the stream kernel would
    // decode each list once per 64 probing queries, and reading rows decoded once at build time is the better trade.  The
    // search picks per call (dense_probing below).  Budget: CUVS_B200_PQ_DECODED_BUDGET_MB (default 4096, 0 = never).
    const int64_t budget  = env_int("CUVS_B200_PQ_DECODED_BUDGET_MB", 4096) << 20;
    const bool also_rows  = R > 0 && static_cast<int64_t>(R) * idx.Kp * 2 <= budget;
    if (also_rows) {
      idx.yhat.alloc(static_cast<size_t>(std::max<int64_t>(R, 128)) * idx.Kp);
      idx.hx.alloc(static_cast<size_t>(std::max<int64_t>(R, 128)) * 16);
      dbuf<float> hn(static_cast<size_t>(R), s);
      count_launch();
      pq_decode_kernel<<<blocks_for(R * 32, 256), 256, 0, s>>>(idx.codes.data(), idx.ids.data(), R, idx.pq_dim, idx.pq_len, idx.book(),
                                                               idx.Kp, idx.pq_centers.data(), false, idx.lists.d_offsets.data(), idx.n_lists,
                                                               is_ip(idx.metric), idx.centers_rot.data(), idx.rot_dim, idx.yhat.data(),
                                                               hn.data());
      B2_CUDA(cudaGetLastError());
      tc_pack_half_norms(s, hn.data(), R, idx.hx.data());
    } else {
      idx.yhat.release();
      idx.hx.release();
    }
    if (R > 0) {  // the stream is the index: pq_dim + 4 bytes per vector (+ 8 for the id)
      B2_CUDA(cudaStreamSynchronize(s));
      idx.codes.release();
    }
    return;
  }
  idx.yhat.alloc(static_cast<size_t>(std::max<int64_t>(R, 128)) * idx.Kp);
  idx.hx.alloc(static_cast<size_t>(std::max<int64_t>(R, 128)) * 16);
  if (R == 0) return;
  dbuf<float> hn(static_cast<size_t>(R), s);
  count_launch();
  pq_decode_kernel<<<blocks_for(R * 32, 256), 256, 0, s>>>(idx.codes.data(), idx.ids.data(), R, idx.pq_dim, idx.pq_len, idx.book(),
                                                           idx.Kp, idx.pq_centers.data(),
                                                           idx.codebook_kind == CUVS_IVF_PQ_CODEBOOK_GEN_PER_CLUSTER,
                                                           idx.lists.d_offsets.data(), idx.n_lists, is_ip(idx.metric),
                                                           idx.centers_rot.data(), idx.rot_dim, idx.yhat.data(), hn.data());
  B2_CUDA(cudaGetLastError());
  tc_pack_half_norms(s, hn.data(), R, idx.hx.data());
}

void train_codebooks(resources* res, ivf_pq_index& idx, const float* resid, const uint32_t* labels, int64_t n, int n_iters)
{
  auto s             = res->stream;
  const bool per_cl  = idx.codebook_kind == CUVS_IVF_PQ_CODEBOOK_GEN_PER_CLUSTER;
  const int64_t nb   = per_cl ? idx.n_lists : idx.pq_dim;
  const int book     = idx.book();
  idx.pq_centers.alloc(static_cast<size_t>(nb) * idx.pq_len * book);
  B2_EXPECTS(idx.pq_len <= 32, "pq_len (%d) > 32 is not supported", idx.pq_len);
  B2_EXPECTS(!per_cl || true, "unreachable");
  count_launch();
  pq_init_kernel<<<blocks_for(nb * book, 128), 128, 0, s>>>(idx.pq_centers.data(), nb, idx.pq_len, book, resid, n, idx.rot_dim, idx.pq_dim);
  dbuf<uint8_t> codes(static_cast<size_t>(n) * idx.pq_dim, s);
  dbuf<uint32_t> keys(static_cast<size_t>(n) * idx.pq_dim, s), order;
  dbuf<int64_t> start;
  dbuf<float> sums(static_cast<size_t>(nb) * idx.pq_len * book, s), counts(static_cast<size_t>(nb) * book, s);
  const size_t smem = static_cast<size_t>(idx.pq_len) * book * sizeof(float);
  for (int it = 0; it < n_iters; ++it) {
    count_launch(4);
    pq_assign_kernel<<<dim3(blocks_for(n, 128), idx.pq_dim), 128, smem, s>>>(resid, n, idx.rot_dim, idx.pq_dim, idx.pq_len, book,
                                                                               idx.pq_centers.data(), per_cl, labels, codes.data(), nullptr);
    pq_keys_kernel<<<blocks_for(n * idx.pq_dim, 256), 256, 0, s>>>(n, idx.pq_dim, book, codes.data(), per_cl, labels, keys.data());
    iota_u32(s, order, n * idx.pq_dim);
    group_by_key(s, keys, order, nb * book, start);
    pq_segment_sums_kernel<<<blocks_for(nb * book * 32, 256), 256, 0, s>>>(resid, idx.rot_dim, idx.pq_dim, idx.pq_len, book, nb * book,
                                                                            order.data(), start.data(), sums.data(), counts.data());
    pq_finalize_kernel<<<blocks_for(nb * book, 128), 128, 0, s>>>(idx.pq_centers.data(), sums.data(), counts.data(), nb, idx.pq_len, book,
                                                                   resid, n, idx.rot_dim, idx.pq_dim, it, it == n_iters - 1);
    B2_CUDA(cudaGetLastError());
  }
}

// Insert the rows of `t` (ids new_ids[i] or id0 + i): codes are encoded straight into their place in the new lists, and the
// decoded rows are refreshed once at the end.
void ivf_pq_extend(resources* res, ivf_pq_index& idx, const DLTensor& t, const int64_t* new_ids, int64_t id0)
{
  if (t.shape[0] == 0) return;
  if (idx.lists.rows_total > 0) ensure_flat_codes(res, idx);
  auto label = [&](const float* x, int64_t n, uint32_t* labels) { label_rows(res, idx.centers_tc, x, n, idx.dim, nullptr, labels); };
  auto write = [&](const float* x, int64_t n, const uint32_t* labels, const int64_t* dst_rows, uint8_t* codes) {
    encode_rows(res, idx, x, n, labels, codes, dst_rows);
  };
  insert_rows(res, idx.lists, idx.codes, idx.pq_dim, idx.ids, t, idx.dim, new_ids, id0, label, write);
  refresh_decoded(res, idx);
}

void init_shape(ivf_pq_index& idx, const cuvsIvfPqIndexParams& p, int dim)
{
  idx.metric        = p.metric;
  idx.metric_arg    = p.metric_arg;
  idx.dim           = dim;
  idx.n_lists       = p.n_lists;
  idx.pq_bits       = static_cast<int>(p.pq_bits);
  idx.pq_dim        = static_cast<int>(p.pq_dim == 0 ? calculate_pq_dim(dim) : p.pq_dim);
  idx.pq_len        = (dim + idx.pq_dim - 1) / idx.pq_dim;
  idx.rot_dim       = idx.pq_dim * idx.pq_len;
  idx.dim_ext       = (dim + 1 + 7) / 8 * 8;
  idx.codebook_kind = static_cast<int>(p.codebook_kind);
  idx.conservative  = p.conservative_memory_allocation;
  idx.kmeans_n_iters = p.kmeans_n_iters;
  B2_EXPECTS(idx.pq_bits >= 4 && idx.pq_bits <= 8, "pq_bits must be within [4, 8]");
  B2_EXPECTS(idx.pq_len >= 1 && idx.pq_len <= 32, "pq_len = ceil(dim / pq_dim) = %d is outside [1, 32] (dim %d, pq_dim %d)", idx.pq_len, dim, idx.pq_dim);
  B2_EXPECTS(is_l2(p.metric) || p.metric == InnerProduct || p.metric == CosineExpanded, "ivf_pq: unsupported metric %d", int(p.metric));
  B2_EXPECTS(p.metric != CosineExpanded, "ivf_pq: cosine metric is not supported by this build yet");
}

ivf_pq_index* ivf_pq_build(resources* res, const cuvsIvfPqIndexParams& p, const DLTensor& ds)
{
  B2_EXPECTS(ds.ndim == 2 && dl_is_c_contiguous(ds), "dataset must be a row-major 2-D tensor");
  const int64_t n = ds.shape[0];
  const int d     = static_cast<int>(ds.shape[1]);
  B2_EXPECTS(n >= 1 && d >= 1, "empty dataset");
  B2_EXPECTS(p.n_lists >= 1 && static_cast<int64_t>(p.n_lists) <= n, "n_lists (%u) must be in [1, n_rows]", p.n_lists);
  B2_EXPECTS(tc_supported(res->device, d), "ivf_pq: dim %d > 128 is not supported by this build yet", d);
  auto idx    = std::make_unique<ivf_pq_index>();
  idx->device = res->device;
  init_shape(*idx, p, d);
  auto s = res->stream;

  // training subsample, k-means for the coarse centres
  dbuf<float> train;
  const int64_t n_train = training_subsample(s, dl_ptr<float>(ds), n, d, p.n_lists, p.kmeans_trainset_fraction, train);
  idx->centers.alloc(static_cast<size_t>(p.n_lists) * d);
  kmeans_train(res, train.data(), n_train, d, p.n_lists, std::max<uint32_t>(p.kmeans_n_iters, 1), idx->centers.data(), true, true, nullptr, nullptr);
  refresh_centers(res, *idx);

  // rotation and rotated centres
  std::vector<float> R = make_rotation(idx->rot_dim, d, p.force_random_rotation || idx->rot_dim != d);
  idx->rotation.alloc(R.size());
  B2_CUDA(cudaMemcpyAsync(idx->rotation.data(), R.data(), R.size() * sizeof(float), cudaMemcpyHostToDevice, s));
  B2_CUDA(cudaStreamSynchronize(s));
  idx->centers_rot.alloc(static_cast<size_t>(p.n_lists) * idx->rot_dim);
  rotate_rows(s, idx->centers.data(), p.n_lists, d, idx->rotation.data(), idx->rot_dim, idx->centers_rot.data());

  // PQ codebooks from the residuals of (a prefix of) the training set
  int64_t n_pq = std::min<int64_t>(n_train, static_cast<int64_t>(std::max<uint32_t>(p.max_train_points_per_pq_code, 1)) * idx->book());
  if (idx->codebook_kind == CUVS_IVF_PQ_CODEBOOK_GEN_PER_CLUSTER) n_pq = n_train;
  n_pq = std::max<int64_t>(n_pq, std::min<int64_t>(n_train, idx->book()));
  {
    dbuf<uint32_t> labels(static_cast<size_t>(n_pq), s);
    label_rows(res, idx->centers_tc, train.data(), n_pq, d, nullptr, labels.data());
    dbuf<float> rs = encode_rows(res, *idx, train.data(), n_pq, labels.data());
    train_codebooks(res, *idx, rs.data(), labels.data(), n_pq, std::max<uint32_t>(p.kmeans_n_iters, 1));
  }
  std::vector<int64_t> zero(p.n_lists, 0);
  idx->lists.set_sizes(s, zero);
  idx->codes.alloc(1);
  idx->ids.alloc(1);
  refresh_decoded(res, *idx);
  if (p.add_data_on_build) {
    ivf_pq_extend(res, *idx, ds, nullptr, 0);
  }
  return idx.release();
}

int env_path()  // read on every search: tests switch paths inside one process
{
  const char* e = getenv("CUVS_B200_PQ_PATH");
  if (!e) return 0;
  return strcmp(e, "lut") == 0 ? 1 : (strcmp(e, "tc") == 0 ? 2 : (strcmp(e, "stream") == 0 ? 3 : 0));  // stream: never the decoded-row cache
}

void ivf_pq_search(resources* res, const ivf_pq_index& idx, const cuvsIvfPqSearchParams& sp, const DLTensor& qt, const DLTensor& nt,
                   const DLTensor& dt)
{
  auto s           = res->stream;
  const int64_t nq = qt.shape[0];
  const int k      = static_cast<int>(nt.shape[1]);
  B2_EXPECTS(qt.shape[1] == idx.dim, "queries dim (%lld) != index dim (%d)", (long long)qt.shape[1], idx.dim);
  B2_EXPECTS(nt.shape[0] == nq && dt.shape[0] == nq && dt.shape[1] == k, "neighbors/distances shape mismatch");
  B2_EXPECTS(k >= 1 && k <= 64, "ivf_pq search: k must be in [1, 64] in this build (got %d)", k);
  B2_EXPECTS(sp.n_probes >= 1, "n_probes must be >= 1");
  B2_EXPECTS(sp.lut_dtype == CUDA_R_32F || sp.lut_dtype == CUDA_R_16F || sp.lut_dtype == CUDA_R_8U, "unsupported lut_dtype");
  B2_EXPECTS(sp.internal_distance_dtype == CUDA_R_32F || sp.internal_distance_dtype == CUDA_R_16F, "unsupported internal_distance_dtype");
  if (nq == 0) return;
  const uint32_t n_probes = std::min<uint32_t>(sp.n_probes, idx.n_lists);
  {
    // Query batching (ivf_pq_search.cuh:960-1010 loops over max_internal_batch_size): the per-(query, probe) workspaces
    // below — residual rows (Kp bf16 per pass) and 2 x KC candidate slots — are bounded to ~3 GiB; a 10k x 48-probe batch
    // needs 0.3 GiB and runs in one piece.  Slots are uint32: nq * n_probes must stay below 2^32 as well.
    const int64_t per_query = static_cast<int64_t>(n_probes) * (2 * idx.Kp * 2 + 64 * 8 + 16);
    int64_t batch = std::max<int64_t>(1, (int64_t(3) << 30) / per_query);
    batch         = std::min<int64_t>(batch, (int64_t(1) << 31) / std::max<uint32_t>(n_probes, 1));
    if (sp.max_internal_batch_size > 0 && n_probes > 256) batch = std::min<int64_t>(batch, std::max<uint32_t>(sp.max_internal_batch_size, 128));
    if (nq > batch) {
      for (int64_t q0 = 0; q0 < nq; q0 += batch) {
        const int64_t rows = std::min(batch, nq - q0);
        dl_row_slice qs(qt, q0, rows), ns(nt, q0, rows), ds(dt, q0, rows);
        ivf_pq_search(res, idx, sp, qs.t, ns.t, ds.t);
      }
      return;
    }
  }
  const float* q   = dl_ptr<float>(qt);
  int64_t* out_idx = dl_ptr<int64_t>(nt);
  float* out_dist  = dl_ptr<float>(dt);
  const bool ip    = is_ip(idx.metric);

  // ---- coarse + rotation
  tc_rows_tmp qp;
  qp.build(s, q, nq, idx.dim, true);
  dbuf<uint32_t> probes(static_cast<size_t>(nq) * n_probes, s);
  coarse_select(res, qp, idx.centers_tc, static_cast<int>(n_probes), probes.data(), nullptr);
  dbuf<float> q_rot(static_cast<size_t>(nq) * idx.rot_dim, s);
  rotate_rows(s, q, nq, idx.dim, idx.rotation.data(), idx.rot_dim, q_rot.data());

  // ---- bucket pairs by list
  // Decoded-row tensor-core scan whenever the index keeps decoded rows.  fp32 LUT + fp32 accumulation (the reference's
  // exact formulation) -> 2-pass scan: the residual is split into two bf16 planes, the decoded rows ARE bf16, so the scores
  // equal the LUT sums to fp32 rounding.  A reduced-precision LUT / accumulator request (fp16, fp8) -> 1-pass scan with the
  // residual rounded to bf16: the same class of approximation, at tensor-core speed.  CUVS_B200_PQ_PATH=lut forces the
  // faithful LUT kernel (bit-level emulation of the fp16 / fp_8bit<5> LUT entries).
  const bool reduced = !(sp.lut_dtype == CUDA_R_32F && sp.internal_distance_dtype == CUDA_R_32F);
  // (C) codes streamed + decoded on the SM — unless the index is small enough to also hold decoded rows AND this batch probes
  // densely (>= 128 queries per list on average: the per-group decode would be repeated more than twice per list)
  const bool dense_probing = idx.yhat.data() != nullptr && k <= 32 && env_path() != 3 &&
                             static_cast<double>(nq) * n_probes >= 128.0 * std::max<uint32_t>(idx.n_lists, 1);
  const bool use_stream = env_path() != 1 && idx.cstream.data() != nullptr && k <= 64 && !dense_probing;
  const bool use_tc     = use_stream || (env_path() == 1 ? false : idx.yhat.data() != nullptr);
  const int passes   = reduced ? 1 : 2;
  const int lists = use_stream ? 1 : (use_tc ? tc_lists_per_item() : 1);
  // candidates kept per (query, probe): the tensor-core epilogue keeps `lists` sorted lists of KC (one per column half of
  // the tile); for k > KC the union of the two half lists stands in for the pair's top-k (exact whenever no more than KC of
  // them fall into one half — an approximation only the k > 32 candidate-generation use case can see)
  const int KC    = k <= 16 ? 16 : (k <= 32 || (use_tc && !use_stream) ? 32 : 64);
  const int KCW   = KC * lists;
  B2_EXPECTS(KCW >= k, "ivf_pq search: k = %d exceeds the %d candidates kept per probe", k, KCW);
  // queries per work item: 128 for the query-major kernels; the streamed kernel takes the list rows as the MMA's M side
  // and 32 / 64 / 128 probing queries as N (picked from the average number of pairs per list)
  const int group = use_stream ? pq_stream_group(static_cast<double>(nq) * n_probes / std::max<uint32_t>(idx.n_lists, 1), KC, passes) : 128;
  probe_buckets pb;
  bucket_probes(res, probes.data(), nq, static_cast<int>(n_probes), idx.n_lists, idx.lists.d_offsets.data(), KCW, pb, 0, 0xffffffffu, group);
  dbuf<float> cs(static_cast<size_t>(pb.n_pairs) * KCW, s);
  dbuf<uint32_t> cp(static_cast<size_t>(pb.n_pairs) * KCW, s);
  dbuf<float> add;
  dbuf<int> bkeys;  // per-query pruning bound of the tensor-core scan (tc_bound), reused by the merge
  float scale = 1.0f;

  if (use_tc) {
    const int64_t a_rows = pb.n_pairs + 128;
    dbuf<__nv_bfloat16> a_hi(static_cast<size_t>(a_rows) * idx.Kp, s), a_lo;
    if (passes == 2) a_lo.alloc(static_cast<size_t>(a_rows) * idx.Kp, s);
    add.alloc(static_cast<size_t>(pb.n_pairs), s);
    // slots that were dropped (empty lists) are never read; slots beyond the live pairs are zero rows
    count_launch();
    pair_rows_kernel<<<blocks_for(a_rows * 32, 256), 256, 0, s>>>(q_rot.data(), idx.centers_rot.data(), pb.pair_query.data(),
                                                                   pb.pair_list.data(), pb.n_items.data() + 1, a_rows, idx.rot_dim, idx.Kp, ip,
                                                                   a_hi.data(), a_lo.data(), add.data(), use_stream);
    B2_CUDA(cudaGetLastError());
    scale = ip ? 1.0f : 2.0f;  // L2: |r|^2 + 2 (|y|^2/2 - r.y); IP: -(q.(c+y))
    {
      // probes of one query share a running bound on its k'-th best DISTANCE: d = add[slot] + scale * s
      if (k <= KC) {  // the bound tracks a k-th best out of KC kept entries
        bkeys.alloc(static_cast<size_t>(nq), s);
        B2_CUDA(cudaMemsetAsync(bkeys.data(), tc_bound_init_byte, sizeof(int) * nq, s));
      }
      tc_bound bnd;
      bnd.keys  = bkeys.data();
      bnd.idx   = pb.pair_query.data();
      bnd.add   = add.data();
      bnd.scale = scale;
      bnd.kth   = k;  // only the query's k best survive the merge below
      timed_section ts("pq_scan", s);
      if (use_stream)
        pq_stream_scan(s, res->device, a_hi.data(), a_lo.data(), a_rows, idx.Kp, idx.cstream.data(), idx.cb_words.data(), idx.pq_dim,
                       pb.items.data(), pb.max_items, pb.n_items.data(), group, KC, passes, cs.data(), cp.data(), KCW,
                       bkeys.data() ? &bnd : nullptr);
      else
        tc_scan_topk(s, res->device, a_hi.data(), a_lo.data(), a_rows, idx.yhat.data(), nullptr, std::max<int64_t>(idx.lists.rows_total, 128),
                     idx.Kp, idx.hx.data(), pb.items.data(), pb.max_items, pb.n_items.data(), KC, passes, cs.data(), cp.data(), KCW, bkeys.data() ? &bnd : nullptr);
    }
  } else {
    ensure_flat_codes(res, idx);
    const int book      = idx.book();
    const size_t lut_b  = sp.lut_dtype == CUDA_R_32F ? 4 : (sp.lut_dtype == CUDA_R_16F ? 2 : 1);
    const size_t smem   = ((static_cast<size_t>(idx.pq_dim) * book * lut_b + 15) & ~size_t(15)) + 2 * idx.rot_dim * sizeof(float) +
                        4 * kLutBuf * sizeof(float);
    B2_EXPECTS(smem <= 227 * 1024, "ivf_pq: LUT (%zu bytes) does not fit in shared memory; use a smaller lut_dtype", smem);
    const bool half_out = sp.internal_distance_dtype == CUDA_R_16F;
    const bool per_cl   = idx.codebook_kind == CUVS_IVF_PQ_CODEBOOK_GEN_PER_CLUSTER;
    const bool cosine   = idx.metric == CosineExpanded;
    // slots of dropped pairs hold garbage pair_query: only launch over the live prefix
    // (bucket_probes packs live pairs first; count is on the device -> launch over all slots, dead ones exit early)
#define B2_LUT_LAUNCH(LUT_T, OUT_T)                                                                                         \
  {                                                                                                                         \
    auto kern = pq_lut_scan_kernel<LUT_T, OUT_T>;                                                                           \
    B2_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));               \
    timed_section ts("pq_scan", s);                                                                                         \
    count_launch();                                                                                                         \
    kern<<<static_cast<unsigned>(pb.n_pairs), kLutThreads, smem, s>>>(                                                      \
      q_rot.data(), idx.centers_rot.data(), idx.pq_centers.data(), per_cl, idx.codes.data(), idx.lists.d_offsets.data(),   \
      idx.lists.d_sizes.data(), pb.pair_query.data(), pb.pair_list.data(), pb.n_items.data() + 1, idx.rot_dim, idx.pq_dim, idx.pq_len, idx.pq_bits, ip,  \
      cosine, KC, cs.data(), cp.data(), KCW);                                                                               \
  }
    if (sp.lut_dtype == CUDA_R_32F) B2_LUT_LAUNCH(float, float)
    else if (sp.lut_dtype == CUDA_R_16F && !half_out) B2_LUT_LAUNCH(__half, float)
    else if (sp.lut_dtype == CUDA_R_16F && half_out) B2_LUT_LAUNCH(__half, __half)
    else if (!half_out) B2_LUT_LAUNCH(uint8_t, float)
    else B2_LUT_LAUNCH(uint8_t, __half)
#undef B2_LUT_LAUNCH
    B2_CUDA(cudaGetLastError());
  }

  // ---- per query: concatenate its probes' candidates (already in final distance units), top-k, ids
  const int64_t cand_w = static_cast<int64_t>(n_probes) * KCW;
  dbuf<uint32_t> mp(static_cast<size_t>(nq) * k, s);
  if (!(bkeys.data() != nullptr &&
        merge_probe_candidates(s, cs.data(), cp.data(), pb.slot_of.data(), add.data(), scale, bkeys.data(), nq, static_cast<int>(n_probes),
                               KCW, k, out_dist, mp.data()))) {
    dbuf<float> gs(static_cast<size_t>(nq) * cand_w, s);
    dbuf<uint32_t> gp(static_cast<size_t>(nq) * cand_w, s);
    count_launch();
    gather_pq_cands_kernel<<<blocks_for(nq * cand_w, 256), 256, 0, s>>>(cs.data(), cp.data(), pb.slot_of.data(), use_tc ? add.data() : nullptr,
                                                                         scale, nq * cand_w, KCW, gs.data(), gp.data());
    select_k(s, gs.data(), gp.data(), IDX_U32, nq, cand_w, cand_w, k, out_dist, mp.data(), IDX_U32, true);
  }
  count_launch();
  finish_ids_kernel<<<blocks_for(nq * k, 256), 256, 0, s>>>(mp.data(), idx.ids.data(), out_dist, nq * k, int(idx.metric), out_idx);
  B2_CUDA(cudaGetLastError());
}

}  // namespace
}  // namespace b200

using namespace b200;

static ivf_pq_index& pq_of(cuvsIvfPqIndex_t index)
{
  B2_EXPECTS(index != nullptr && index->addr != 0, "index is not built");
  return *reinterpret_cast<ivf_pq_index*>(index->addr);
}

extern "C" {

cuvsError_t cuvsIvfPqIndexParamsCreate(cuvsIvfPqIndexParams_t* params)
{
  return guarded([=] {
    B2_EXPECTS(params != nullptr, "params is null");
    // defaults: c/src/neighbors/ivf_pq.cpp:348-365
    *params = new cuvsIvfPqIndexParams{L2Expanded, 2.0f, true, 1024, 20, 0.5, 8, 0, CUVS_IVF_PQ_CODEBOOK_GEN_PER_SUBSPACE,
                                       false, false, 256, CUVS_IVF_PQ_LIST_LAYOUT_INTERLEAVED};
  });
}
cuvsError_t cuvsIvfPqIndexParamsDestroy(cuvsIvfPqIndexParams_t params) { return guarded([=] { delete params; }); }

cuvsError_t cuvsIvfPqSearchParamsCreate(cuvsIvfPqSearchParams_t* params)
{
  return guarded([=] {
    B2_EXPECTS(params != nullptr, "params is null");
    *params = new cuvsIvfPqSearchParams{20, CUDA_R_32F, CUDA_R_32F, CUDA_R_32F, 4096, 1.0};
  });
}
cuvsError_t cuvsIvfPqSearchParamsDestroy(cuvsIvfPqSearchParams_t params) { return guarded([=] { delete params; }); }

cuvsError_t cuvsIvfPqIndexCreate(cuvsIvfPqIndex_t* index)
{
  return guarded([=] {
    B2_EXPECTS(index != nullptr, "index is null");
    *index = new cuvsIvfPqIndex{};
  });
}
cuvsError_t cuvsIvfPqIndexDestroy(cuvsIvfPqIndex_t index)
{
  return guarded([=] {
    if (!index) return;
    delete reinterpret_cast<ivf_pq_index*>(index->addr);
    delete index;
  });
}

cuvsError_t cuvsB200IvfPqIndexInfo(cuvsIvfPqIndex_t index, int* path, int64_t* device_bytes)
{
  return guarded([=] {
    const ivf_pq_index& idx = pq_of(index);
    if (path) *path = (idx.cstream.data() ? 2 : 0) | (idx.yhat.data() ? 1 : 0);
    if (device_bytes)
      *device_bytes = static_cast<int64_t>(idx.codes.size() + idx.ids.size() * 8 + idx.cstream.size() + idx.cb_words.size() * 4 +
                                           idx.yhat.size() * 2 + idx.hx.size() * 2 + idx.centers.size() * 4 + idx.centers_ext.size() * 4 +
                                           idx.centers_rot.size() * 4 + idx.rotation.size() * 4 + idx.pq_centers.size() * 4 +
                                           (idx.centers_tc.hi.size() + idx.centers_tc.lo.size() + idx.centers_tc.hx.size()) * 2);
  });
}

cuvsError_t cuvsIvfPqIndexGetNLists(cuvsIvfPqIndex_t index, int64_t* v) { return guarded([=] { *v = pq_of(index).n_lists; }); }
cuvsError_t cuvsIvfPqIndexGetDim(cuvsIvfPqIndex_t index, int64_t* v) { return guarded([=] { *v = pq_of(index).dim; }); }
cuvsError_t cuvsIvfPqIndexGetSize(cuvsIvfPqIndex_t index, int64_t* v) { return guarded([=] { *v = pq_of(index).lists.size; }); }
cuvsError_t cuvsIvfPqIndexGetPqDim(cuvsIvfPqIndex_t index, int64_t* v) { return guarded([=] { *v = pq_of(index).pq_dim; }); }
cuvsError_t cuvsIvfPqIndexGetPqBits(cuvsIvfPqIndex_t index, int64_t* v) { return guarded([=] { *v = pq_of(index).pq_bits; }); }
cuvsError_t cuvsIvfPqIndexGetPqLen(cuvsIvfPqIndex_t index, int64_t* v) { return guarded([=] { *v = pq_of(index).pq_len; }); }

cuvsError_t cuvsIvfPqIndexGetCenters(cuvsIvfPqIndex_t index, DLManagedTensor* centers)
{
  return guarded([=] {
    auto& idx        = pq_of(index);
    int64_t shape[2] = {idx.n_lists, idx.dim};
    dl_fill_view(centers, idx.centers.data(), idx.device, DLDataType{kDLFloat, 32, 1}, 2, shape);
  });
}
cuvsError_t cuvsIvfPqIndexGetCentersPadded(cuvsIvfPqIndex_t index, DLManagedTensor* centers)
{
  return guarded([=] {
    auto& idx        = pq_of(index);
    int64_t shape[2] = {idx.n_lists, idx.dim_ext};
    dl_fill_view(centers, idx.centers_ext.data(), idx.device, DLDataType{kDLFloat, 32, 1}, 2, shape);
  });
}
cuvsError_t cuvsIvfPqIndexGetPqCenters(cuvsIvfPqIndex_t index, DLManagedTensor* pq_centers)
{
  return guarded([=] {
    auto& idx        = pq_of(index);
    int64_t nb       = idx.codebook_kind == CUVS_IVF_PQ_CODEBOOK_GEN_PER_CLUSTER ? idx.n_lists : idx.pq_dim;
    int64_t shape[3] = {nb, idx.pq_len, idx.book()};
    dl_fill_view(pq_centers, idx.pq_centers.data(), idx.device, DLDataType{kDLFloat, 32, 1}, 3, shape);
  });
}
cuvsError_t cuvsIvfPqIndexGetCentersRot(cuvsIvfPqIndex_t index, DLManagedTensor* centers_rot)
{
  return guarded([=] {
    auto& idx        = pq_of(index);
    int64_t shape[2] = {idx.n_lists, idx.rot_dim};
    dl_fill_view(centers_rot, idx.centers_rot.data(), idx.device, DLDataType{kDLFloat, 32, 1}, 2, shape);
  });
}
cuvsError_t cuvsIvfPqIndexGetRotationMatrix(cuvsIvfPqIndex_t index, DLManagedTensor* rotation_matrix)
{
  return guarded([=] {
    auto& idx        = pq_of(index);
    int64_t shape[2] = {idx.rot_dim, idx.dim};
    dl_fill_view(rotation_matrix, idx.rotation.data(), idx.device, DLDataType{kDLFloat, 32, 1}, 2, shape);
  });
}
cuvsError_t cuvsIvfPqIndexGetListSizes(cuvsIvfPqIndex_t index, DLManagedTensor* list_sizes)
{
  return guarded([=] {
    auto& idx        = pq_of(index);
    int64_t shape[1] = {idx.n_lists};
    dl_fill_view(list_sizes, idx.lists.d_sizes.data(), idx.device, DLDataType{kDLUInt, 32, 1}, 1, shape);
  });
}

// out_codes [n_take, pq_dim * pq_bits / 8] uint8: contiguous (bit-packed for pq_bits < 8) codes of rows offset.. of a list
__global__ void pack_codes_kernel(const uint8_t* __restrict__ codes, int64_t n, int pq_dim, int pq_bits, int out_ld, uint8_t* __restrict__ out)
{
  int64_t r = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  if (r >= n) return;
  for (int b = 0; b < out_ld; ++b) out[r * out_ld + b] = 0;
  for (int j = 0; j < pq_dim; ++j) {
    uint32_t v   = codes[r * pq_dim + j];
    int bit      = j * pq_bits;
    uint32_t sh  = v << (bit & 7);
    out[r * out_ld + (bit >> 3)] |= static_cast<uint8_t>(sh & 0xff);
    if (sh >> 8) out[r * out_ld + (bit >> 3) + 1] |= static_cast<uint8_t>(sh >> 8);
  }
}

cuvsError_t cuvsIvfPqIndexUnpackContiguousListData(cuvsResources_t res, cuvsIvfPqIndex_t index, DLManagedTensor* out_codes,
                                                   uint32_t label, uint32_t offset)
{
  return guarded([=] {
    auto r    = as_res(res);
    auto& idx = pq_of(index);
    B2_EXPECTS(label < idx.n_lists, "label %u out of range", label);
    const DLTensor& oc = out_codes->dl_tensor;
    B2_EXPECTS(dl_is(oc, kDLUInt, 8) && oc.ndim == 2 && dl_is_device(oc) && dl_is_c_contiguous(oc), "out_codes must be a device uint8 matrix");
    const int out_ld = (idx.pq_dim * idx.pq_bits + 7) / 8;
    B2_EXPECTS(oc.shape[1] == out_ld, "out_codes must have %d columns", out_ld);
    const int64_t n_take = oc.shape[0];
    B2_EXPECTS(static_cast<int64_t>(offset) + n_take <= idx.lists.h_sizes[label], "offset + n_rows exceeds the list size");
    if (n_take == 0) return;
    ensure_flat_codes(r, idx);
    pack_codes_kernel<<<blocks_for(n_take, 128), 128, 0, r->stream>>>(idx.codes.data() + (idx.lists.h_offsets[label] + offset) * idx.pq_dim,
                                                                      n_take, idx.pq_dim, idx.pq_bits, out_ld, dl_ptr<uint8_t>(oc));
    B2_CUDA(cudaGetLastError());
  });
}

cuvsError_t cuvsIvfPqIndexGetListIndices(cuvsIvfPqIndex_t index, uint32_t label, DLManagedTensor* out_labels)
{
  return guarded([=] {
    auto& idx = pq_of(index);
    B2_EXPECTS(label < idx.n_lists, "label %u out of range", label);
    int64_t shape[1] = {idx.lists.h_sizes[label]};
    dl_fill_view(out_labels, idx.ids.data() + idx.lists.h_offsets[label], idx.device, DLDataType{kDLInt, 64, 1}, 1, shape);
  });
}

cuvsError_t cuvsIvfPqBuild(cuvsResources_t res, cuvsIvfPqIndexParams_t params, DLManagedTensor* dataset, cuvsIvfPqIndex_t index)
{
  return guarded([=] {
    auto r = as_res(res);
    B2_EXPECTS(params && dataset && index, "null argument");
    const DLTensor& ds = dataset->dl_tensor;
    B2_EXPECTS(dl_is_dataset_dtype(ds), "Unsupported dataset DLtensor dtype: %d and bits: %d", ds.dtype.code, ds.dtype.bits);
    if (index->addr) { delete reinterpret_cast<ivf_pq_index*>(index->addr); index->addr = 0; }
    f32_matrix w;  // float16 / int8 / uint8 datasets (c/src/neighbors/ivf_pq.cpp:80-103) are widened to fp32 rows
    widen_to_f32(r, ds, w);
    index->addr  = reinterpret_cast<uintptr_t>(ivf_pq_build(r, *params, w.t));
    index->dtype = ds.dtype;
  });
}

static void copy_in(resources* r, owned<float>& dst, const DLTensor& t, size_t count)
{
  dst.alloc(count);
  B2_CUDA(cudaMemcpyAsync(dst.data(), dl_ptr<float>(t), count * sizeof(float), cudaMemcpyDefault, r->stream));
}

cuvsError_t cuvsIvfPqBuildPrecomputed(cuvsResources_t res, cuvsIvfPqIndexParams_t params, uint32_t dim, DLManagedTensor* pq_centers,
                                      DLManagedTensor* centers, DLManagedTensor* centers_rot, DLManagedTensor* rotation_matrix,
                                      cuvsIvfPqIndex_t index)
{
  return guarded([=] {
    auto r = as_res(res);
    B2_EXPECTS(params && pq_centers && centers && index, "null argument");
    auto idx    = std::make_unique<ivf_pq_index>();
    idx->device = r->device;
    init_shape(*idx, *params, static_cast<int>(dim));
    const DLTensor& pc = pq_centers->dl_tensor;
    const DLTensor& ce = centers->dl_tensor;
    B2_EXPECTS(dl_is(pc, kDLFloat, 32) && dl_is(ce, kDLFloat, 32), "codebooks must be float32");
    B2_EXPECTS(tc_supported(r->device, idx->dim), "ivf_pq: dim %d > 128 is not supported by this build yet", idx->dim);
    const int64_t nb = idx->codebook_kind == CUVS_IVF_PQ_CODEBOOK_GEN_PER_CLUSTER ? idx->n_lists : idx->pq_dim;
    B2_EXPECTS(pc.ndim == 3 && pc.shape[0] == nb && pc.shape[1] == idx->pq_len && pc.shape[2] == idx->book(),
               "pq_centers must have extent [%lld, %d, %d]", (long long)nb, idx->pq_len, idx->book());
    B2_EXPECTS(ce.ndim == 2 && ce.shape[0] == idx->n_lists && (ce.shape[1] == idx->dim || ce.shape[1] == idx->dim_ext),
               "centers must have extent [n_lists, dim] or [n_lists, dim_ext]");
    copy_in(r, idx->pq_centers, pc, static_cast<size_t>(nb) * idx->pq_len * idx->book());
    idx->centers.alloc(static_cast<size_t>(idx->n_lists) * idx->dim);
    B2_CUDA(cudaMemcpy2DAsync(idx->centers.data(), sizeof(float) * idx->dim, dl_ptr<float>(ce), sizeof(float) * ce.shape[1],
                              sizeof(float) * idx->dim, idx->n_lists, cudaMemcpyDefault, r->stream));
    refresh_centers(r, *idx);
    if (rotation_matrix) {
      const DLTensor& rm = rotation_matrix->dl_tensor;
      B2_EXPECTS(dl_is(rm, kDLFloat, 32) && rm.ndim == 2 && rm.shape[0] == idx->rot_dim && rm.shape[1] == idx->dim,
                 "rotation_matrix must have extent [rot_dim, dim]");
      copy_in(r, idx->rotation, rm, static_cast<size_t>(idx->rot_dim) * idx->dim);
    } else {
      std::vector<float> R = make_rotation(idx->rot_dim, idx->dim, params->force_random_rotation || idx->rot_dim != idx->dim);
      idx->rotation.alloc(R.size());
      B2_CUDA(cudaMemcpyAsync(idx->rotation.data(), R.data(), R.size() * sizeof(float), cudaMemcpyHostToDevice, r->stream));
      B2_CUDA(cudaStreamSynchronize(r->stream));
    }
    if (centers_rot) {
      const DLTensor& cr = centers_rot->dl_tensor;
      B2_EXPECTS(dl_is(cr, kDLFloat, 32) && cr.ndim == 2 && cr.shape[0] == idx->n_lists && cr.shape[1] == idx->rot_dim,
                 "centers_rot must have extent [n_lists, rot_dim]");
      copy_in(r, idx->centers_rot, cr, static_cast<size_t>(idx->n_lists) * idx->rot_dim);
    } else {
      idx->centers_rot.alloc(static_cast<size_t>(idx->n_lists) * idx->rot_dim);
      rotate_rows(r->stream, idx->centers.data(), idx->n_lists, idx->dim, idx->rotation.data(), idx->rot_dim, idx->centers_rot.data());
    }
    std::vector<int64_t> zero(idx->n_lists, 0);
    idx->lists.set_sizes(r->stream, zero);
    idx->codes.alloc(1);
    idx->ids.alloc(1);
    refresh_decoded(r, *idx);
    if (index->addr) delete reinterpret_cast<ivf_pq_index*>(index->addr);
    index->addr  = reinterpret_cast<uintptr_t>(idx.release());
    index->dtype = DLDataType{kDLFloat, 32, 1};
  });
}

cuvsError_t cuvsIvfPqSearch(cuvsResources_t res, cuvsIvfPqSearchParams_t params, cuvsIvfPqIndex_t index, DLManagedTensor* queries_t,
                            DLManagedTensor* neighbors_t, DLManagedTensor* distances_t)
{
  return guarded([=] {
    auto r = as_res(res);
    B2_EXPECTS(params && queries_t && neighbors_t && distances_t, "null argument");
    auto& idx = pq_of(index);
    const DLTensor& queries   = queries_t->dl_tensor;
    const DLTensor& neighbors = neighbors_t->dl_tensor;
    const DLTensor& distances = distances_t->dl_tensor;
    B2_EXPECTS(dl_is_device(queries), "queries should have device compatible memory");
    B2_EXPECTS(dl_is_device(neighbors), "neighbors should have device compatible memory");
    B2_EXPECTS(dl_is_device(distances), "distances should have device compatible memory");
    B2_EXPECTS(dl_is(neighbors, kDLInt, 64), "neighbors should be of type int64_t");
    B2_EXPECTS(dl_is(distances, kDLFloat, 32), "distances should be of type float32");
    B2_EXPECTS(dl_is_dataset_dtype(queries), "Unsupported queries DLtensor dtype: %d and bits: %d", queries.dtype.code, queries.dtype.bits);
    B2_EXPECTS(queries.ndim == 2 && neighbors.ndim == 2 && distances.ndim == 2, "queries/neighbors/distances must be 2-D");
    B2_EXPECTS(dl_is_c_contiguous(queries) && dl_is_c_contiguous(neighbors) && dl_is_c_contiguous(distances), "tensors must be row-major contiguous");
    f32_matrix w;
    widen_to_f32(r, queries, w);
    ivf_pq_search(r, idx, *params, w.t, neighbors, distances);
  });
}

cuvsError_t cuvsIvfPqExtend(cuvsResources_t res, DLManagedTensor* new_vectors, DLManagedTensor* new_indices, cuvsIvfPqIndex_t index)
{
  return guarded([=] {
    auto r    = as_res(res);
    auto& idx = pq_of(index);
    f32_matrix v;
    dbuf<int64_t> ids_buf;
    const int64_t* ids = extend_args(r, new_vectors, new_indices, idx.dim, v, ids_buf);
    ivf_pq_extend(r, idx, v.t, ids, idx.lists.size);
  });
}

// cuVS index file, serialization version 4 (cpp/src/neighbors/ivf_pq/ivf_pq_serialize.cuh:25-86; per-list records
// cpp/src/neighbors/ivf_list.cuh:108-133): a sequence of NPY records (npy_io.hpp) —
//   version i4 = 4, size i8, dim u4, pq_bits u4, pq_dim u4, conservative_memory_allocation u1, metric i4, codebook_kind i4,
//   codes_layout i4, n_lists u4, pq_centers f4 [pq_dim | n_lists, pq_len, 2^pq_bits], centers f4 [n_lists, dim_ext],
//   centers_rot f4 [n_lists, rot_dim], rotation_matrix f4 [rot_dim, dim], list_sizes u4 [n_lists], then per list:
//   size u4 and (size > 0) codes u1 in the reference's list layout — INTERLEAVED [ceil(size/32), ceil(pq_dim/C), 32, 16]
//   with C = 128/pq_bits codes per 16-byte chunk (ivf_pq.hpp:235-296, bit order ivf_pq_codepacking.cuh:28-78), or FLAT
//   [size, ceil(pq_dim*pq_bits/8)] — and indices i8 [size].
// A cuVS build loads these files with ivf_pq::deserialize and this library loads files written by cuVS.
namespace {

// [n, pq_dim] one code per byte -> interleaved groups of 32 (host)
std::vector<uint8_t> pack_interleaved(const uint8_t* flat, int64_t n, int pq_dim, int pq_bits)
{
  const int C = 128 / pq_bits, n_chunks = (pq_dim + C - 1) / C;
  std::vector<uint8_t> out(static_cast<size_t>((n + 31) / 32) * n_chunks * 32 * 16, 0);
  for (int64_t v = 0; v < n; ++v) {
    const int64_t g = v / 32, l = v % 32;
    for (int j = 0; j < pq_dim; ++j) {
      const int bit = (j % C) * pq_bits;
      uint8_t* chunk = out.data() + ((g * n_chunks + j / C) * 32 + l) * 16;
      const uint32_t val = static_cast<uint32_t>(flat[v * pq_dim + j]) << (bit % 8);
      chunk[bit / 8] |= static_cast<uint8_t>(val & 0xffu);
      if (val >> 8) chunk[bit / 8 + 1] |= static_cast<uint8_t>(val >> 8);
    }
  }
  return out;
}
void unpack_interleaved(const uint8_t* packed, int64_t n, int pq_dim, int pq_bits, uint8_t* flat)
{
  const int C = 128 / pq_bits, n_chunks = (pq_dim + C - 1) / C;
  const uint32_t mask = (1u << pq_bits) - 1u;
  for (int64_t v = 0; v < n; ++v) {
    const int64_t g = v / 32, l = v % 32;
    for (int j = 0; j < pq_dim; ++j) {
      const int bit = (j % C) * pq_bits, byte = bit / 8;
      const uint8_t* chunk = packed + ((g * n_chunks + j / C) * 32 + l) * 16;
      uint32_t word = chunk[byte];
      if (byte + 1 < 16) word |= static_cast<uint32_t>(chunk[byte + 1]) << 8;
      flat[v * pq_dim + j] = static_cast<uint8_t>((word >> (bit % 8)) & mask);
    }
  }
}
// FLAT layout: every vector's codes bit-packed contiguously, ceil(pq_dim * pq_bits / 8) bytes per row
void unpack_flat_rows(const uint8_t* packed, int64_t n, int pq_dim, int pq_bits, uint8_t* flat)
{
  const int ld = (pq_dim * pq_bits + 7) / 8;
  const uint32_t mask = (1u << pq_bits) - 1u;
  for (int64_t v = 0; v < n; ++v)
    for (int j = 0; j < pq_dim; ++j) {
      const int bit = j * pq_bits, byte = bit / 8;
      uint32_t word = packed[v * ld + byte];
      if (byte + 1 < ld) word |= static_cast<uint32_t>(packed[v * ld + byte + 1]) << 8;
      flat[v * pq_dim + j] = static_cast<uint8_t>((word >> (bit % 8)) & mask);
    }
}

}  // namespace

cuvsError_t cuvsIvfPqSerialize(cuvsResources_t res, const char* filename, cuvsIvfPqIndex_t index)
{
  return guarded([=] {
    auto r    = as_res(res);
    auto& idx = pq_of(index);
    std::ofstream os(filename, std::ios::out | std::ios::binary);
    B2_EXPECTS(bool(os), "Cannot open file %s", filename);
    npy::write_scalar<int32_t>(os, 4);
    npy::write_scalar<int64_t>(os, idx.lists.size);
    npy::write_scalar<uint32_t>(os, static_cast<uint32_t>(idx.dim));
    npy::write_scalar<uint32_t>(os, static_cast<uint32_t>(idx.pq_bits));
    npy::write_scalar<uint32_t>(os, static_cast<uint32_t>(idx.pq_dim));
    npy::write_scalar<bool>(os, idx.conservative);
    npy::write_scalar<int32_t>(os, static_cast<int32_t>(idx.metric));
    npy::write_scalar<int32_t>(os, static_cast<int32_t>(idx.codebook_kind));
    npy::write_scalar<int32_t>(os, static_cast<int32_t>(CUVS_IVF_PQ_LIST_LAYOUT_INTERLEAVED));
    npy::write_scalar<uint32_t>(os, idx.n_lists);
    auto dump = [&](const float* p, std::vector<int64_t> shape) {
      size_t n = 1;
      for (auto e : shape) n *= static_cast<size_t>(e);
      std::vector<float> h(n);
      B2_CUDA(cudaMemcpyAsync(h.data(), p, n * sizeof(float), cudaMemcpyDeviceToHost, r->stream));
      B2_CUDA(cudaStreamSynchronize(r->stream));
      npy::write_array<float>(os, h.data(), shape);
    };
    const int64_t nb = idx.codebook_kind == CUVS_IVF_PQ_CODEBOOK_GEN_PER_CLUSTER ? idx.n_lists : idx.pq_dim;
    dump(idx.pq_centers.data(), {nb, idx.pq_len, idx.book()});
    dump(idx.centers_ext.data(), {static_cast<int64_t>(idx.n_lists), idx.dim_ext});
    dump(idx.centers_rot.data(), {static_cast<int64_t>(idx.n_lists), idx.rot_dim});
    dump(idx.rotation.data(), {idx.rot_dim, idx.dim});
    std::vector<uint32_t> sizes(idx.n_lists);
    for (uint32_t l = 0; l < idx.n_lists; ++l) sizes[l] = static_cast<uint32_t>(idx.lists.h_sizes[l]);
    npy::write_array<uint32_t>(os, sizes.data(), {static_cast<int64_t>(idx.n_lists)});
    std::vector<uint8_t> codes;
    std::vector<int64_t> ids;
    const int C = 128 / idx.pq_bits;
    ensure_flat_codes(r, idx);
    for (uint32_t l = 0; l < idx.n_lists; ++l) {
      const int64_t sz = idx.lists.h_sizes[l];
      npy::write_scalar<uint32_t>(os, static_cast<uint32_t>(sz));
      if (!sz) continue;
      codes.resize(static_cast<size_t>(sz) * idx.pq_dim);
      ids.resize(static_cast<size_t>(sz));
      B2_CUDA(cudaMemcpyAsync(codes.data(), idx.codes.data() + idx.lists.h_offsets[l] * idx.pq_dim, codes.size(), cudaMemcpyDeviceToHost, r->stream));
      B2_CUDA(cudaMemcpyAsync(ids.data(), idx.ids.data() + idx.lists.h_offsets[l], ids.size() * sizeof(int64_t), cudaMemcpyDeviceToHost, r->stream));
      B2_CUDA(cudaStreamSynchronize(r->stream));
      const std::vector<uint8_t> packed = pack_interleaved(codes.data(), sz, idx.pq_dim, idx.pq_bits);
      npy::write_array<uint8_t>(os, packed.data(), {(sz + 31) / 32, (idx.pq_dim + C - 1) / C, 32, 16});
      npy::write_array<int64_t>(os, ids.data(), {sz});
    }
    B2_EXPECTS(bool(os), "Error writing %s", filename);
  });
}

cuvsError_t cuvsIvfPqDeserialize(cuvsResources_t res, const char* filename, cuvsIvfPqIndex_t index)
{
  return guarded([=] {
    auto r = as_res(res);
    B2_EXPECTS(index && filename, "null argument");
    std::ifstream is(filename, std::ios::in | std::ios::binary);
    B2_EXPECTS(bool(is), "Cannot open file %s", filename);
    const int ver = npy::read_scalar<int32_t>(is, filename);
    B2_EXPECTS(ver == 4, "serialization version mismatch %d vs. %d", ver, 4);
    const int64_t n_rows  = npy::read_scalar<int64_t>(is, filename);
    const uint32_t dim    = npy::read_scalar<uint32_t>(is, filename);
    const uint32_t pqbits = npy::read_scalar<uint32_t>(is, filename);
    const uint32_t pqdim  = npy::read_scalar<uint32_t>(is, filename);
    const bool cma        = npy::read_scalar<uint8_t>(is, filename) != 0;
    const int32_t metric  = npy::read_scalar<int32_t>(is, filename);
    const int32_t cb_kind = npy::read_scalar<int32_t>(is, filename);
    const int32_t layout  = npy::read_scalar<int32_t>(is, filename);
    const uint32_t nlists = npy::read_scalar<uint32_t>(is, filename);
    B2_EXPECTS(cb_kind == 0 || cb_kind == 1, "ivf_pq::deserialize: invalid codebook_gen value %d", cb_kind);
    B2_EXPECTS(layout == 0 || layout == 1, "ivf_pq::deserialize: invalid list_layout value %d", layout);
    auto idx    = std::make_unique<ivf_pq_index>();
    idx->device = r->device;
    cuvsIvfPqIndexParams p{static_cast<cuvsDistanceType>(metric), 2.0f, true, nlists, 20, 0.5, pqbits, pqdim,
                           static_cast<cuvsIvfPqCodebookGen>(cb_kind), false, cma, 256, CUVS_IVF_PQ_LIST_LAYOUT_INTERLEAVED};
    init_shape(*idx, p, static_cast<int>(dim));
    auto load = [&](owned<float>& dst, size_t n) {
      std::vector<float> h(n);
      npy::read_array<float>(is, h.data(), static_cast<int64_t>(n), filename);
      dst.alloc(n);
      B2_CUDA(cudaMemcpyAsync(dst.data(), h.data(), n * sizeof(float), cudaMemcpyHostToDevice, r->stream));
      B2_CUDA(cudaStreamSynchronize(r->stream));
      return h;
    };
    const int64_t nb = idx->codebook_kind == CUVS_IVF_PQ_CODEBOOK_GEN_PER_CLUSTER ? idx->n_lists : idx->pq_dim;
    load(idx->pq_centers, static_cast<size_t>(nb) * idx->pq_len * idx->book());
    {
      // centers are stored padded: [n_lists, dim_ext] with |c|^2 in column dim (ivf_pq_index.cu:78-80)
      std::vector<float> ext = load(idx->centers_ext, static_cast<size_t>(idx->n_lists) * idx->dim_ext);
      std::vector<float> c(static_cast<size_t>(idx->n_lists) * idx->dim);
      for (uint32_t l = 0; l < idx->n_lists; ++l)
        std::copy(ext.begin() + static_cast<size_t>(l) * idx->dim_ext, ext.begin() + static_cast<size_t>(l) * idx->dim_ext + idx->dim,
                  c.begin() + static_cast<size_t>(l) * idx->dim);
      idx->centers.alloc(c.size());
      B2_CUDA(cudaMemcpyAsync(idx->centers.data(), c.data(), c.size() * sizeof(float), cudaMemcpyHostToDevice, r->stream));
      B2_CUDA(cudaStreamSynchronize(r->stream));
    }
    load(idx->centers_rot, static_cast<size_t>(idx->n_lists) * idx->rot_dim);
    load(idx->rotation, static_cast<size_t>(idx->rot_dim) * idx->dim);
    refresh_centers(r, *idx);
    std::vector<uint32_t> sizes32(idx->n_lists);
    npy::read_array<uint32_t>(is, sizes32.data(), idx->n_lists, filename);
    std::vector<int64_t> sizes(sizes32.begin(), sizes32.end());
    idx->lists.set_sizes(r->stream, sizes);
    B2_EXPECTS(idx->lists.size == n_rows, "ivf_pq::deserialize: list sizes sum to %lld, header says %lld rows", (long long)idx->lists.size,
               (long long)n_rows);
    alloc_padded(r->stream, idx->lists.rows_total, idx->pq_dim, idx->codes, idx->ids);
    std::vector<uint8_t> packed, codes;
    std::vector<int64_t> ids;
    const int C = 128 / idx->pq_bits;
    for (uint32_t l = 0; l < idx->n_lists; ++l) {
      const int64_t sz = npy::read_scalar<uint32_t>(is, filename);
      B2_EXPECTS(sz == sizes[l], "ivf_pq::deserialize: list %u holds %lld rows, list_sizes says %lld", l, (long long)sz, (long long)sizes[l]);
      if (!sz) continue;
      const int64_t pbytes = layout == 1 ? (sz + 31) / 32 * ((idx->pq_dim + C - 1) / C) * 32 * 16
                                         : sz * ((idx->pq_dim * idx->pq_bits + 7) / 8);
      packed.resize(static_cast<size_t>(pbytes));
      codes.resize(static_cast<size_t>(sz) * idx->pq_dim);
      ids.resize(static_cast<size_t>(sz));
      npy::read_array<uint8_t>(is, packed.data(), pbytes, filename);
      npy::read_array<int64_t>(is, ids.data(), sz, filename);
      if (layout == 1) unpack_interleaved(packed.data(), sz, idx->pq_dim, idx->pq_bits, codes.data());
      else unpack_flat_rows(packed.data(), sz, idx->pq_dim, idx->pq_bits, codes.data());
      B2_CUDA(cudaMemcpyAsync(idx->codes.data() + idx->lists.h_offsets[l] * idx->pq_dim, codes.data(), codes.size(), cudaMemcpyHostToDevice, r->stream));
      B2_CUDA(cudaMemcpyAsync(idx->ids.data() + idx->lists.h_offsets[l], ids.data(), ids.size() * sizeof(int64_t), cudaMemcpyHostToDevice, r->stream));
      B2_CUDA(cudaStreamSynchronize(r->stream));
    }
    refresh_decoded(r, *idx);
    if (index->addr) delete reinterpret_cast<ivf_pq_index*>(index->addr);
    index->addr  = reinterpret_cast<uintptr_t>(idx.release());
    index->dtype = DLDataType{kDLFloat, 32, 1};
  });
}

// Encode vectors with the index's quantizers: output_labels [n] uint32, output_dataset [n, ceil(pq_dim*pq_bits/8)] uint8.
cuvsError_t cuvsIvfPqTransform(cuvsResources_t res, cuvsIvfPqIndex_t index, DLManagedTensor* input_dataset, DLManagedTensor* output_labels,
                               DLManagedTensor* output_dataset)
{
  return guarded([=] {
    auto r    = as_res(res);
    auto& idx = pq_of(index);
    B2_EXPECTS(input_dataset && output_labels && output_dataset, "null argument");
    const DLTensor& x  = input_dataset->dl_tensor;
    const DLTensor& ol = output_labels->dl_tensor;
    const DLTensor& oc = output_dataset->dl_tensor;
    B2_EXPECTS(dl_is(x, kDLFloat, 32) && x.ndim == 2 && x.shape[1] == idx.dim && dl_is_device(x) && dl_is_c_contiguous(x), "input_dataset must be a device [n, dim] float32 matrix");
    const int64_t n  = x.shape[0];
    const int out_ld = (idx.pq_dim * idx.pq_bits + 7) / 8;
    B2_EXPECTS(dl_is(ol, kDLUInt, 32) && ol.shape[0] == n && dl_is_device(ol), "output_labels must be device uint32 [n]");
    B2_EXPECTS(dl_is(oc, kDLUInt, 8) && oc.ndim == 2 && oc.shape[0] == n && oc.shape[1] == out_ld && dl_is_device(oc), "output_dataset must be device uint8 [n, %d]", out_ld);
    if (n == 0) return;
    auto s = r->stream;
    uint32_t* labels = dl_ptr<uint32_t>(ol);
    label_rows(r, idx.centers_tc, dl_ptr<float>(x), n, idx.dim, nullptr, labels);
    dbuf<uint8_t> codes(static_cast<size_t>(n) * idx.pq_dim, s);
    encode_rows(r, idx, dl_ptr<float>(x), n, labels, codes.data());
    pack_codes_kernel<<<blocks_for(n, 128), 128, 0, s>>>(codes.data(), n, idx.pq_dim, idx.pq_bits, out_ld, dl_ptr<uint8_t>(oc));
    B2_CUDA(cudaGetLastError());
  });
}

}  // extern "C"
