// Exact kNN ("brute force"): index + search + C boundary.
//
// Reference path being replaced (SURVEY §8a rows a1-a4):
//   index / build      cpp/src/neighbors/brute_force.cu:32-108, detail/knn_brute_force.cuh:778-818
//   search dispatch    detail/knn_brute_force.cuh:353-539 (fused SIMT kernel for k<=64 L2, tiled cuBLAS otherwise)
//   C wrapper          c/src/neighbors/brute_force.cpp:120-330
//
// B200 design (DESIGN.md §3): the index keeps, next to the fp32 rows and their norms, the rows
// split into two bf16 planes (x = hi + lo) padded to 128-row tiles.  Search is
//   1. candidate scan on tcgen05 (scan_tc.cu): s = |x|^2/2 - q.x with split-bf16 products, a
//      register top-k' per query row per dataset split, no distance matrix in HBM;
//   2. merge of the per-split lists (select_k.cu);
//   3. exact fp32 re-scoring of the k' candidates in the oracle's arithmetic (exact.cu), which
//      also evaluates a certificate: if the k-th exact distance is not strictly below the worst
//      candidate's approximate distance minus the error budget, the query is flagged;
//   4. flagged queries (ties / duplicates at the k' boundary) are recomputed by the exact SIMT
//      path.  Result: identical to oracle/oracle.c::oracle_knn, bit for bit.
// Filtered search and shapes the tensor-core kernel does not cover (dim > 2048, k > 64)
// run on the exact SIMT path.
#include "common.hpp"
#include "exact.cuh"
#include "scan_tc.cuh"
#include "select_k.cuh"
#include "timing.hpp"

#include <cuvs/neighbors/brute_force.h>
#include <cuvs_b200/ext.h>

#include <algorithm>
#include <cfloat>
#include <cmath>
#include <cstring>
#include <fstream>
#include <memory>
#include <vector>

namespace b200 {

struct bf_index {
  int64_t n   = 0;
  int d       = 0;
  int device  = 0;
  cuvsDistanceType metric = L2Expanded;
  float metric_arg        = 2.0f;
  const float* data       = nullptr;  // [n, d] row-major on the device (view or data_own)
  owned<float> data_own;
  owned<float> norms;  // |x|^2 (always kept: the certificate needs max norm)
  float xn_max = 0.f;
  // tensor-core side
  bool tc      = false;
  int Kp       = 0;
  int64_t rows_pad = 0;
  owned<__nv_bfloat16> hi, lo;
  owned<__nv_bfloat16> hx;  // [rows_pad, 16] half-norm plane (scan_tc.cuh)
  owned<float> inv_norm;  // cosine only
};

namespace {

bool metric_supported(cuvsDistanceType m)
{
  return m == L2Expanded || m == L2SqrtExpanded || m == L2Unexpanded || m == L2SqrtUnexpanded || m == InnerProduct ||
         m == CosineExpanded;
}

__global__ void transpose_kernel(const float* __restrict__ in, float* __restrict__ out, int64_t n, int d)
{
  // in: column-major [n, d] (element (r,c) at c*n + r) -> out row-major
  int64_t t = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  if (t >= n * d) return;
  int64_t r = t / d;
  int c     = static_cast<int>(t % d);
  out[t]    = in[static_cast<int64_t>(c) * n + r];
}

__global__ void rsqrt_kernel(const float* __restrict__ xn, float* __restrict__ out, int64_t n)
{
  int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  if (i < n) out[i] = xn[i] > 0.f ? 1.0f / sqrtf(xn[i]) : 0.f;
}

__global__ void max_kernel(const float* __restrict__ v, int64_t n, float* __restrict__ out)
{
  float m = 0.f;
  for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x)
    m = fmaxf(m, v[i]);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0) atomicMax(reinterpret_cast<int*>(out), __float_as_int(m));  // m >= 0
}

__global__ void make_items_kernel(tc_item* items, int m_tiles, int splits, int64_t nq, uint32_t tiles_total, int KCW)
{
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= m_tiles * splits) return;
  // item order: split-major, so that concurrently running CTAs stream the same dataset range (L2 reuse)
  int s = i / m_tiles, m = i % m_tiles;
  uint32_t per = (tiles_total + splits - 1) / splits;
  uint32_t t0  = min(tiles_total, s * per), t1 = min(tiles_total, t0 + per);
  tc_item it;
  it.a_row0     = m * 128;
  it.b_row0     = t0 * 128;
  it.n_tiles    = t1 - t0;
  int64_t valid = nq - static_cast<int64_t>(m) * 128;
  it.valid_rows = valid > 128 ? 128 : static_cast<uint32_t>(valid);
  it.out_off    = (static_cast<uint64_t>(m) * 128 * splits + s) * KCW;
  items[i]      = it;
}

int pick_splits(int m_tiles, int64_t b_tiles, int sms)
{
  int64_t s_max = std::max<int64_t>(1, std::min<int64_t>(32, b_tiles / 8));
  int best = 1;
  double best_eff = -1;
  for (int s = 1; s <= s_max; ++s) {
    int64_t items = static_cast<int64_t>(m_tiles) * s;
    int64_t waves = (items + sms - 1) / sms;
    double eff    = static_cast<double>(items) / static_cast<double>(waves * sms);
    if (eff > best_eff + 1e-9) { best_eff = eff; best = s; }
  }
  return best;
}

}  // namespace

// ------------------------------------------------------------------------------------ build
static bf_index* bf_build(resources* res, const DLTensor& ds, cuvsDistanceType metric, float metric_arg)
{
  B2_EXPECTS(ds.ndim == 2, "dataset must be a 2-D tensor");
  B2_EXPECTS(metric_supported(metric), "brute_force: unsupported metric %d", int(metric));
  auto idx        = std::make_unique<bf_index>();
  idx->n          = ds.shape[0];
  idx->d          = static_cast<int>(ds.shape[1]);
  idx->metric     = metric;
  idx->metric_arg = metric_arg;
  idx->device     = res->device;
  auto stream     = res->stream;
  const bool c_contig = dl_is_c_contiguous(ds), f_contig = dl_is_f_contiguous(ds);
  B2_EXPECTS(c_contig || f_contig, "dataset input to cuvsBruteForceBuild must be contiguous (non-strided)");
  const float* src = dl_ptr<float>(ds);
  const size_t count = static_cast<size_t>(idx->n) * idx->d;
  if (dl_is_device(ds) && ds.device.device_type != kDLCUDAHost && c_contig) {
    idx->data = src;  // non-owning view, like the reference (brute_force.cu:60-75)
  } else {
    idx->data_own.alloc(count);
    if (c_contig) {
      B2_CUDA(cudaMemcpyAsync(idx->data_own.data(), src, count * sizeof(float), cudaMemcpyDefault, stream));
    } else {
      dbuf<float> tmp(count, stream);
      B2_CUDA(cudaMemcpyAsync(tmp.data(), src, count * sizeof(float), cudaMemcpyDefault, stream));
      if (count) transpose_kernel<<<static_cast<unsigned>((count + 255) / 256), 256, 0, stream>>>(tmp.data(), idx->data_own.data(), idx->n, idx->d);
      B2_CUDA(cudaGetLastError());
    }
    idx->data = idx->data_own.data();
  }
  idx->norms.alloc(static_cast<size_t>(std::max<int64_t>(idx->n, 1)));
  row_norms(stream, idx->data, idx->n, idx->d, idx->d, idx->norms.data());
  {
    dbuf<float> mx(1, stream);
    B2_CUDA(cudaMemsetAsync(mx.data(), 0, sizeof(float), stream));
    if (idx->n) max_kernel<<<std::min<int64_t>(1024, (idx->n + 255) / 256), 256, 0, stream>>>(idx->norms.data(), idx->n, mx.data());
    B2_CUDA(cudaGetLastError());
    B2_CUDA(cudaMemcpyAsync(&idx->xn_max, mx.data(), sizeof(float), cudaMemcpyDeviceToHost, stream));
    B2_CUDA(cudaStreamSynchronize(stream));
  }
  idx->tc = tc_supported(res->device, idx->d) && idx->n >= 1 && idx->n < (int64_t(1) << 31);
  if (idx->tc) {
    idx->Kp       = tc_pad_k(idx->d);
    idx->rows_pad = tc_pad_rows(idx->n);
    idx->hi.alloc(static_cast<size_t>(idx->rows_pad) * idx->Kp);
    idx->lo.alloc(static_cast<size_t>(idx->rows_pad) * idx->Kp);
    idx->hx.alloc(static_cast<size_t>(idx->rows_pad) * 16);
    const float* scale = nullptr;
    if (metric == CosineExpanded) {
      idx->inv_norm.alloc(static_cast<size_t>(idx->n));
      rsqrt_kernel<<<static_cast<unsigned>((idx->n + 255) / 256), 256, 0, stream>>>(idx->norms.data(), idx->inv_norm.data(), idx->n);
      B2_CUDA(cudaGetLastError());
      scale = idx->inv_norm.data();
    }
    tc_split_planes(stream, idx->data, idx->n, idx->d, idx->d, idx->Kp, idx->hi.data(), idx->lo.data(), idx->rows_pad, scale);
    const bool l2 = (metric != InnerProduct && metric != CosineExpanded);
    tc_half_norms(stream, l2 ? idx->norms.data() : nullptr, idx->n, idx->rows_pad, idx->hx.data());
  }
  return idx.release();
}

// ------------------------------------------------------------------------------------ search
static void search_exact(resources* res, const bf_index& idx, const float* q, int64_t nq, int64_t q_row0, int k,
                         int64_t* out_idx, float* out_dist, filter_view filt)
{
  auto stream = res->stream;
  if (nq == 0) return;
  const bool select_min = metric_is_min_close(idx.metric);
  const bool need_norms = (idx.metric == L2Expanded || idx.metric == L2SqrtExpanded || idx.metric == CosineExpanded);
  dbuf<float> qn;
  if (need_norms) {
    qn.alloc(static_cast<size_t>(nq), stream);
    row_norms(stream, q, nq, idx.d, idx.d, qn.data());
  }
  const int64_t n_cols = std::max<int64_t>(idx.n, 1);
  int64_t chunk = std::max<int64_t>(1, std::min<int64_t>(nq, (int64_t(1) << 28) / n_cols));
  chunk         = std::min<int64_t>(chunk, 65535 * 64);
  dbuf<float> dist(static_cast<size_t>(chunk * n_cols), stream);
  for (int64_t q0 = 0; q0 < nq; q0 += chunk) {
    int64_t qc = std::min(chunk, nq - q0);
    exact_distance_tile(stream, q + q0 * idx.d, qc, idx.d, idx.data, idx.n, idx.d, idx.d, need_norms ? qn.data() + q0 : nullptr,
                        need_norms ? idx.norms.data() : nullptr, idx.metric, dist.data(), idx.n, filt, q_row0 + q0);
    select_k(stream, dist.data(), nullptr, IDX_NONE, qc, idx.n, idx.n, k, out_dist + q0 * k, out_idx + q0 * k, IDX_I64,
             select_min);
  }
}

__global__ void mask_filtered_kernel(int64_t* idx, float* dist, int64_t count, bool select_min)
{
  int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  if (i >= count) return;
  float worst = select_min ? FLT_MAX : -FLT_MAX;
  if (dist[i] == worst) idx[i] = -1;  // nothing (or only filtered-out rows) left for this slot
}

struct bf_cands {
  dbuf<float> score;    // [nq, KCm] raw engine scores s = hn - q.x (best first)
  dbuf<uint32_t> pos;   // [nq, KCm] row positions
  dbuf<float> qn;       // [nq] |q|^2
  dbuf<float> floor;    // [nq] (KCm > KC only) min over the scan's FULL candidate lists of the list's worst kept score
  int width = 0;        // entries per query row in score / pos (KCm, or everything the scan kept when that is less)
};

// floor[q] = min over the query's lists of the list's last (= worst, lists are sorted best-first) entry; a list that is not
// full ends in +inf and constrains nothing.  Every row the scan rejected — by a list's own k'-th entry or by the bound shared
// between the splits, which is some full list's k'-th entry at an earlier time and only ever decreases — scores above it.
__global__ void list_floor_kernel(const float* __restrict__ cs, int64_t nq, int64_t row_stride, int KC, float* __restrict__ out)
{
  const int64_t q = (blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x) >> 5;
  const int lane  = threadIdx.x & 31;
  if (q >= nq) return;
  float m = INFINITY;
  for (int64_t l = lane; l * KC < row_stride; l += 32) m = fminf(m, cs[q * row_stride + l * KC + KC - 1]);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fminf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if (lane == 0) out[q] = m;
}

// Stage 1+2 of the search: split-bf16 tcgen05 scan over `splits` dataset ranges (lists of KC per column half and split) +
// merge to KCm per query (KCm == KC: the merged set's worst entry bounds everything outside it; KCm > KC, used for k above
// the fused list length: `out.floor` carries the bound for the rows that never entered a list).
static void bf_tc_candidates(resources* res, const bf_index& idx, const float* q, int64_t nq, int KC, bf_cands& out, int KCm = 0)
{
  if (KCm <= 0) KCm = KC;
  auto stream           = res->stream;
  const int64_t nq_pad  = tc_pad_rows(nq);
  const int m_tiles     = static_cast<int>(nq_pad / 128);
  const int64_t b_tiles = idx.rows_pad / 128;
  const int splits      = pick_splits(m_tiles, b_tiles, res->sm_count ? res->sm_count : 148);
  const int n_items     = m_tiles * splits;

  out.qn.alloc(static_cast<size_t>(nq), stream);
  row_norms(stream, q, nq, idx.d, idx.d, out.qn.data());
  dbuf<float> qscale;
  if (idx.metric == CosineExpanded) {
    qscale.alloc(static_cast<size_t>(nq), stream);
    rsqrt_kernel<<<static_cast<unsigned>((nq + 255) / 256), 256, 0, stream>>>(out.qn.data(), qscale.data(), nq);
    B2_CUDA(cudaGetLastError());
    count_launch();
  }
  dbuf<__nv_bfloat16> qhi(static_cast<size_t>(nq_pad) * idx.Kp, stream), qlo(static_cast<size_t>(nq_pad) * idx.Kp, stream);
  tc_split_planes(stream, q, nq, idx.d, idx.d, idx.Kp, qhi.data(), qlo.data(), nq_pad, qscale.data());

  dbuf<tc_item> items(static_cast<size_t>(n_items), stream);
  const int KCW = KC * tc_lists_per_item();  // candidates per (item, query row)
  make_items_kernel<<<(n_items + 127) / 128, 128, 0, stream>>>(items.data(), m_tiles, splits, nq, static_cast<uint32_t>(b_tiles), KCW);
  B2_CUDA(cudaGetLastError());
  count_launch();

  const int64_t row_stride = static_cast<int64_t>(splits) * KCW;
  dbuf<float> cs(static_cast<size_t>(nq_pad) * row_stride, stream);
  dbuf<uint32_t> cp(static_cast<size_t>(nq_pad) * row_stride, stream);
  // the splits of one query row share a running k'-th-best bound (scores are comparable: same query)
  dbuf<int> bkeys(static_cast<size_t>(nq_pad), stream);
  B2_CUDA(cudaMemsetAsync(bkeys.data(), tc_bound_init_byte, sizeof(int) * nq_pad, stream));
  tc_bound bnd;
  bnd.keys = bkeys.data();
  tc_scan_topk(stream, res->device, qhi.data(), qlo.data(), nq_pad, idx.hi.data(), idx.lo.data(), idx.rows_pad, idx.Kp,
               idx.hx.data(), items.data(), n_items, nullptr, KC, 3, cs.data(), cp.data(), row_stride, &bnd,
               false /*equal-sized items in split-major order: static round-robin keeps each column range L2 resident*/);
  if (KCm > KC) {
    out.floor.alloc(static_cast<size_t>(nq), stream);
    count_launch();
    list_floor_kernel<<<static_cast<unsigned>((nq * 32 + 255) / 256), 256, 0, stream>>>(cs.data(), nq, row_stride, KC, out.floor.data());
    B2_CUDA(cudaGetLastError());
  }
  out.width = static_cast<int>(std::min<int64_t>(row_stride, KCm));
  if (row_stride > KCm) {
    out.score.alloc(static_cast<size_t>(nq) * KCm, stream);
    out.pos.alloc(static_cast<size_t>(nq) * KCm, stream);
    select_k(stream, cs.data(), cp.data(), IDX_U32, nq, row_stride, row_stride, KCm, out.score.data(), out.pos.data(), IDX_U32, true);
  } else {
    out.score = std::move(cs);
    out.pos   = std::move(cp);
  }
}

static approx_map bf_approx_map(const bf_index& idx)
{
  approx_map am;
  am.eps_rel = 1.0f / 32768.0f;  // 2^-15: ~3x the split-bf16 bound 3*2^-18*2|q||x| <= 2^-16.4 (|q|^2+|x|^2), ~9x the observed max (DESIGN.md §3)
  if (idx.metric == InnerProduct) { am.sa = -1.f; am.eq = 1.f; am.ec = idx.xn_max; }
  else if (idx.metric == CosineExpanded) { am.sa = 1.f; am.sc = 1.f; am.eq = 0.f; am.ec = 2.f; }
  else { am.sa = 2.f; am.sb = 1.f; am.eq = 1.f; am.ec = idx.xn_max; }
  return am;
}

static void bf_search(resources* res, const bf_index& idx, const DLTensor& qt, const DLTensor& nt, const DLTensor& dt,
                      cuvsFilter prefilter)
{
  auto stream      = res->stream;
  const int64_t nq = qt.shape[0];
  const int k      = static_cast<int>(nt.shape[1]);
  B2_EXPECTS(qt.shape[1] == idx.d, "queries dim (%lld) != index dim (%d)", (long long)qt.shape[1], idx.d);
  B2_EXPECTS(nt.shape[0] == nq && dt.shape[0] == nq && dt.shape[1] == k, "neighbors/distances shape mismatch");
  B2_EXPECTS(k >= 1, "k must be >= 1");
  int64_t* out_idx = dl_ptr<int64_t>(nt);
  float* out_dist  = dl_ptr<float>(dt);
  if (nq == 0) return;

  // queries: row-major view or a transposed copy
  const float* q = dl_ptr<float>(qt);
  dbuf<float> qcopy;
  if (!dl_is_c_contiguous(qt)) {
    B2_EXPECTS(dl_is_f_contiguous(qt), "queries input to cuvsBruteForceSearch must be contiguous (non-strided)");
    qcopy.alloc(static_cast<size_t>(nq) * idx.d, stream);
    transpose_kernel<<<static_cast<unsigned>((nq * idx.d + 255) / 256), 256, 0, stream>>>(q, qcopy.data(), nq, idx.d);
    B2_CUDA(cudaGetLastError());
    q = qcopy.data();
  }

  filter_view filt;
  if (prefilter.type != NO_FILTER) {
    B2_EXPECTS(prefilter.type == BITSET || prefilter.type == BITMAP, "Unsupported prefilter type");
    auto ft = reinterpret_cast<DLManagedTensor*>(prefilter.addr);
    B2_EXPECTS(ft != nullptr && dl_is_device(ft->dl_tensor), "prefilter should have device compatible memory");
    filt.bits      = dl_ptr<uint32_t>(ft->dl_tensor);
    filt.kind      = prefilter.type == BITSET ? 1 : 2;
    filt.n_samples = idx.n;
  }

  const bool select_min = metric_is_min_close(idx.metric);
  // k <= 24: fused lists of 16 / 32, merged to the list length.  24 < k <= 64 (the reference's fused range,
  // knn_brute_force.cuh:447-451): fused lists of 32 per (column half, split), merged to 64 / 96 candidates, and the
  // certificate additionally uses the lists' own worst entries (bf_cands::floor) — a row of the true top-k can only be missing
  // when more than 32 of them fall into one list, which the certificate detects (flagged queries take the exact path).
  const bool use_tc     = idx.tc && filt.kind == 0 && k <= 64 && idx.n > 0;
  set_last_flagged(0);
  if (!use_tc) {
    search_exact(res, idx, q, nq, 0, k, out_idx, out_dist, filt);
    if (filt.kind)
      mask_filtered_kernel<<<static_cast<unsigned>((nq * k + 255) / 256), 256, 0, stream>>>(out_idx, out_dist, nq * k, select_min);
    postprocess_distances(stream, out_dist, nq * k, idx.metric);
    return;
  }

  // ---- tensor-core candidate scan
  const int KC  = k <= 10 ? 16 : 32;
  const int KCm = k <= 24 ? KC : (k <= 48 ? 64 : 96);
  bf_cands cand;
  bf_tc_candidates(res, idx, q, nq, KC, cand, KCm);
  const float* m_score  = cand.score.data();
  const uint32_t* m_pos = cand.pos.data();
  dbuf<float>& qn       = cand.qn;

  // ---- exact re-scoring + certificate
  const approx_map am = bf_approx_map(idx);
  dbuf<int> flags(static_cast<size_t>(nq) + 1, stream);
  B2_CUDA(cudaMemsetAsync(flags.data() + nq, 0, sizeof(int), stream));
  const bool need_xn = (idx.metric == L2Expanded || idx.metric == L2SqrtExpanded || idx.metric == CosineExpanded);
  rescore_topk(stream, q, nq, idx.d, idx.data, idx.d, idx.d, qn.data(), need_xn ? idx.norms.data() : nullptr, idx.metric,
               m_pos, m_score, cand.width, nullptr, k, out_idx, out_dist, -1, am, flags.data(), flags.data() + nq, cand.floor.data());

  // ---- certified fallback for flagged queries (rare: exact ties / duplicates at the k' boundary)
  int n_flagged = 0;
  B2_CUDA(cudaMemcpyAsync(&n_flagged, flags.data() + nq, sizeof(int), cudaMemcpyDeviceToHost, stream));
  B2_CUDA(cudaStreamSynchronize(stream));
  set_last_flagged(n_flagged);
  if (n_flagged > 0) {
    std::vector<int> hflags(static_cast<size_t>(nq));
    B2_CUDA(cudaMemcpyAsync(hflags.data(), flags.data(), sizeof(int) * nq, cudaMemcpyDeviceToHost, stream));
    B2_CUDA(cudaStreamSynchronize(stream));
    int64_t i = 0;
    while (i < nq) {
      if (!hflags[i]) { ++i; continue; }
      int64_t j = i;
      while (j < nq && hflags[j]) ++j;  // contiguous run of flagged queries
      search_exact(res, idx, q + i * idx.d, j - i, i, k, out_idx + i * k, out_dist + i * k, filter_view{});
      i = j;
    }
  }
  postprocess_distances(stream, out_dist, nq * k, idx.metric);
}

}  // namespace b200

using namespace b200;

// ------------------------------------------------------------------------------------ C boundary
extern "C" {

cuvsError_t cuvsBruteForceIndexCreate(cuvsBruteForceIndex_t* index)
{
  return guarded([=] {
    B2_EXPECTS(index != nullptr, "index is null");
    *index = new cuvsBruteForceIndex{};
  });
}

cuvsError_t cuvsBruteForceIndexDestroy(cuvsBruteForceIndex_t index)
{
  return guarded([=] {
    if (!index) return;
    delete reinterpret_cast<bf_index*>(index->addr);
    delete index;
  });
}

cuvsError_t cuvsBruteForceBuild(cuvsResources_t res, DLManagedTensor* dataset_tensor, cuvsDistanceType metric,
                                float metric_arg, cuvsBruteForceIndex_t index)
{
  return guarded([=] {
    auto r = as_res(res);
    B2_EXPECTS(dataset_tensor != nullptr && index != nullptr, "null argument");
    const DLTensor& ds = dataset_tensor->dl_tensor;
    if (dl_is(ds, kDLFloat, 32)) {
      if (index->addr) { delete reinterpret_cast<bf_index*>(index->addr); index->addr = 0; }
      index->addr  = reinterpret_cast<uintptr_t>(bf_build(r, ds, metric, metric_arg));
      index->dtype = ds.dtype;
    } else if (dl_is_dataset_dtype(ds)) {
      // float16 / int8 / uint8 (c/src/neighbors/brute_force.cpp:60-110): widened once, the index owns the fp32 copy
      f32_matrix w;
      widen_to_f32(r, ds, w);
      if (index->addr) { delete reinterpret_cast<bf_index*>(index->addr); index->addr = 0; }
      bf_index* b = bf_build(r, w.t, metric, metric_arg);
      if (b->data == w.own.data()) b->data_own = std::move(w.own);
      index->addr  = reinterpret_cast<uintptr_t>(b);
      index->dtype = ds.dtype;
    } else {
      B2_FAIL("Unsupported dataset DLtensor dtype: %d and bits: %d", ds.dtype.code, ds.dtype.bits);
    }
  });
}

cuvsError_t cuvsBruteForceSearch(cuvsResources_t res, cuvsBruteForceIndex_t index, DLManagedTensor* queries_tensor,
                                 DLManagedTensor* neighbors_tensor, DLManagedTensor* distances_tensor, cuvsFilter prefilter)
{
  return guarded([=] {
    auto r = as_res(res);
    B2_EXPECTS(index && index->addr && queries_tensor && neighbors_tensor && distances_tensor, "null argument");
    const DLTensor& queries   = queries_tensor->dl_tensor;
    const DLTensor& neighbors = neighbors_tensor->dl_tensor;
    const DLTensor& distances = distances_tensor->dl_tensor;
    // same checks / messages as c/src/neighbors/brute_force.cpp:193-206
    B2_EXPECTS(dl_is_device(queries), "queries should have device compatible memory");
    B2_EXPECTS(dl_is_device(neighbors), "neighbors should have device compatible memory");
    B2_EXPECTS(dl_is_device(distances), "distances should have device compatible memory");
    B2_EXPECTS(dl_is(neighbors, kDLInt, 64), "neighbors should be of type int64_t");
    B2_EXPECTS(dl_is(distances, kDLFloat, 32), "distances should be of type float32");
    B2_EXPECTS(queries.dtype.code == index->dtype.code, "type mismatch between index and queries");
    B2_EXPECTS(queries.ndim == 2 && neighbors.ndim == 2 && distances.ndim == 2, "queries/neighbors/distances must be 2-D");
    B2_EXPECTS(dl_is_c_contiguous(neighbors) && dl_is_c_contiguous(distances), "outputs must be row-major contiguous");
    if (dl_is(queries, kDLFloat, 32)) {
      bf_search(r, *reinterpret_cast<bf_index*>(index->addr), queries, neighbors, distances, prefilter);
    } else if (dl_is_dataset_dtype(queries) && queries.dtype.bits == index->dtype.bits) {
      f32_matrix w;
      widen_to_f32(r, queries, w);
      bf_search(r, *reinterpret_cast<bf_index*>(index->addr), w.t, neighbors, distances, prefilter);
    } else {
      B2_FAIL("Unsupported queries DLtensor dtype: %d and bits: %d", queries.dtype.code, queries.dtype.bits);
    }
  });
}

cuvsError_t cuvsB200BruteForceCandidates(cuvsResources_t res, cuvsBruteForceIndex_t index, DLManagedTensor* queries,
                                         DLManagedTensor* cand_pos, DLManagedTensor* cand_score)
{
  return guarded([=] {
    auto r = as_res(res);
    B2_EXPECTS(index && index->addr && queries && cand_pos && cand_score, "null argument");
    auto& idx           = *reinterpret_cast<bf_index*>(index->addr);
    const DLTensor& q   = queries->dl_tensor;
    const DLTensor& cp  = cand_pos->dl_tensor;
    const DLTensor& cs  = cand_score->dl_tensor;
    B2_EXPECTS(idx.tc, "index has no tensor-core planes on this device");
    B2_EXPECTS(dl_is(q, kDLFloat, 32) && dl_is_device(q) && dl_is_c_contiguous(q) && q.ndim == 2 && q.shape[1] == idx.d, "bad queries");
    const int KC = static_cast<int>(cp.shape[1]);
    B2_EXPECTS((KC == 16 || KC == 32) && dl_is(cp, kDLUInt, 32) && dl_is(cs, kDLFloat, 32) && cp.shape[0] == q.shape[0] &&
                 cs.shape[0] == q.shape[0] && cs.shape[1] == KC, "bad candidate tensors");
    bf_cands c;
    bf_tc_candidates(r, idx, dl_ptr<float>(q), q.shape[0], KC, c);
    B2_CUDA(cudaMemcpyAsync(dl_ptr<void>(cp), c.pos.data(), sizeof(uint32_t) * q.shape[0] * KC, cudaMemcpyDeviceToDevice, r->stream));
    B2_CUDA(cudaMemcpyAsync(dl_ptr<void>(cs), c.score.data(), sizeof(float) * q.shape[0] * KC, cudaMemcpyDeviceToDevice, r->stream));
    B2_CUDA(cudaStreamSynchronize(r->stream));
  });
}

// Serialization: 4-char numpy-style dtype tag ("<f4\0"), then n, dim, metric, metric_arg, rows.
// (Own container; the reference's brute_force_serialize.cu writes RAFT mdspans — compatibility is a
// "next" item, SURVEY §8f n1.)
cuvsError_t cuvsBruteForceSerialize(cuvsResources_t res, const char* filename, cuvsBruteForceIndex_t index)
{
  return guarded([=] {
    auto r = as_res(res);
    B2_EXPECTS(index && index->addr && filename, "null argument");
    auto& idx = *reinterpret_cast<bf_index*>(index->addr);
    std::vector<float> host(static_cast<size_t>(idx.n) * idx.d);
    B2_CUDA(cudaMemcpyAsync(host.data(), idx.data, host.size() * sizeof(float), cudaMemcpyDeviceToHost, r->stream));
    B2_CUDA(cudaStreamSynchronize(r->stream));
    std::ofstream os(filename, std::ios::out | std::ios::binary);
    B2_EXPECTS(bool(os), "Cannot open file %s", filename);
    const char tag[4] = {'<', 'f', '4', 0};
    os.write(tag, 4);
    int64_t n = idx.n, d = idx.d;
    int32_t m = int(idx.metric);
    os.write(reinterpret_cast<const char*>(&n), 8);
    os.write(reinterpret_cast<const char*>(&d), 8);
    os.write(reinterpret_cast<const char*>(&m), 4);
    os.write(reinterpret_cast<const char*>(&idx.metric_arg), 4);
    os.write(reinterpret_cast<const char*>(host.data()), static_cast<std::streamsize>(host.size() * sizeof(float)));
    B2_EXPECTS(bool(os), "Error writing %s", filename);
  });
}

cuvsError_t cuvsBruteForceDeserialize(cuvsResources_t res, const char* filename, cuvsBruteForceIndex_t index)
{
  return guarded([=] {
    auto r = as_res(res);
    B2_EXPECTS(index && filename, "null argument");
    std::ifstream is(filename, std::ios::in | std::ios::binary);
    B2_EXPECTS(bool(is), "Cannot open file %s", filename);
    char tag[4]{};
    B2_EXPECTS(bool(is.read(tag, 4)), "Invalid or truncated index header in file %s", filename);
    B2_EXPECTS(tag[0] == '<' && tag[1] == 'f' && tag[2] == '4', "Unsupported index dtype in %s", filename);
    int64_t n = 0, d = 0;
    int32_t m = 0;
    float marg = 0;
    is.read(reinterpret_cast<char*>(&n), 8);
    is.read(reinterpret_cast<char*>(&d), 8);
    is.read(reinterpret_cast<char*>(&m), 4);
    is.read(reinterpret_cast<char*>(&marg), 4);
    B2_EXPECTS(bool(is) && n >= 0 && d > 0, "Invalid index header in file %s", filename);
    std::vector<float> host(static_cast<size_t>(n) * d);
    is.read(reinterpret_cast<char*>(host.data()), static_cast<std::streamsize>(host.size() * sizeof(float)));
    B2_EXPECTS(bool(is), "Truncated index file %s", filename);
    int64_t shape[2] = {n, d};
    DLTensor t{};
    t.data   = host.data();
    t.device = DLDevice{kDLCPU, 0};
    t.ndim   = 2;
    t.dtype  = DLDataType{kDLFloat, 32, 1};
    t.shape  = shape;
    if (index->addr) { delete reinterpret_cast<bf_index*>(index->addr); index->addr = 0; }
    index->addr  = reinterpret_cast<uintptr_t>(bf_build(r, t, static_cast<cuvsDistanceType>(m), marg));
    index->dtype = t.dtype;
  });
}

}  // extern "C"
