// IVF-Flat: index, build / extend, search, C boundary.
//
// Reference path being replaced (SURVEY §8a rows a6-a8, a13):
//   index / list layout   cpp/include/cuvs/neighbors/ivf_flat.hpp:139-300
//   build / extend        cpp/src/neighbors/ivf_flat/ivf_flat_build.cuh:109-520 (balanced k-means + list fill)
//   search_impl           cpp/src/neighbors/ivf_flat/ivf_flat_search.cuh:41-309
//   interleaved_scan      cpp/src/neighbors/ivf_flat/detail/jit_lto_kernels/interleaved_scan_impl.cuh:70-206
//   C wrapper             c/src/neighbors/ivf_flat.cpp
//
// Search on B200 (DESIGN.md §4):
//   1. coarse: dense tcgen05 score block queries x centres (split-bf16, fp32-grade) + select_k(n_probes)
//   2. (query, probe) pairs are bucketed by list on the device (ivf_common.cu)
//   3. fine:   per (list, <=128 probing queries) work item, tcgen05 scan of the list's bf16 rows with the
//              fused top-k' epilogue — each list tile is read once per 128 probing queries, not once per query
//   4. per query: gather the candidates of its probes, keep the best few by approximate score, re-score
//      them exactly in fp32 (sum (q-x)^2 / q.x — the reference's fine-scan arithmetic) and emit ids.
#include "common.hpp"
#include "exact.cuh"
#include "ivf_common.cuh"
#include "ivf_lists.cuh"
#include "npy_io.hpp"
#include "select_k.cuh"
#include "timing.hpp"

#include <cuvs/neighbors/ivf_flat.h>
#include <cuvs_b200/ext.h>

#include <algorithm>
#include <cfloat>
#include <cmath>
#include <fstream>
#include <memory>
#include <vector>

namespace b200 {

struct ivf_flat_index {
  int device              = 0;
  cuvsDistanceType metric = L2Expanded;
  float metric_arg        = 2.0f;
  int dim                 = 0;
  uint32_t n_lists        = 0;
  bool adaptive_centers   = false;
  uint32_t kmeans_n_iters = 20;
  double kmeans_trainset_fraction = 0.5;
  owned<float> centers;  // [n_lists, dim]
  tc_rows centers_tc;    // split planes + |c|^2/2 (0 for inner product)
  list_layout lists;
  owned<float> data;         // [rows_total, dim], list-major, zero padding rows
  owned<int64_t> ids;        // [rows_total], kPadId on padding rows
  owned<float> xn;           // [rows_total] |x|^2 (cosine / certificate use)
  owned<__nv_bfloat16> hi;   // [rows_total, Kp] bf16 rows (normalised for cosine)
  owned<__nv_bfloat16> hx;   // [rows_total, 16] half-norm plane: |x|^2/2, +inf on padding rows (scan_tc.cuh)
  int Kp = 0;
};

namespace {

__global__ void half_norms_masked_kernel(const float* __restrict__ xn, const int64_t* __restrict__ ids, int64_t n, bool zero,
                                         float* __restrict__ hn)
{
  int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  if (i >= n) return;
  hn[i] = ids[i] == kPadId ? INFINITY : (zero ? 0.f : 0.5f * xn[i]);
}

// same, additionally hiding every row whose source id is not kept by the bitset (bit = 1 keeps): the filtered search
// scans against this temporary plane, so excluded rows score -inf inside the tensor-core kernel and can never be candidates
__global__ void half_norms_filtered_kernel(const float* __restrict__ xn, const int64_t* __restrict__ ids, int64_t n, bool zero,
                                           const uint32_t* __restrict__ bits, int64_t n_bits, float* __restrict__ hn)
{
  int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  if (i >= n) return;
  const int64_t id = ids[i];
  const bool keep  = id >= 0 && id < n_bits && ((bits[id >> 5] >> (id & 31)) & 1u);
  hn[i]            = keep ? (zero ? 0.f : 0.5f * xn[i]) : INFINITY;
}

__global__ void rsqrt_rows_kernel(const float* __restrict__ xn, float* __restrict__ out, int64_t n)
{
  int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  if (i < n) out[i] = xn[i] > 0.f ? 1.0f / sqrtf(xn[i]) : 0.f;
}

void refresh_tc_side(resources* res, ivf_flat_index& idx)
{
  auto s          = res->stream;
  const int64_t R = idx.lists.rows_total;
  idx.Kp          = tc_pad_k(idx.dim);
  idx.hi.alloc(static_cast<size_t>(std::max<int64_t>(R, 128)) * idx.Kp);
  idx.hx.alloc(static_cast<size_t>(std::max<int64_t>(R, 128)) * 16);
  idx.xn.alloc(static_cast<size_t>(std::max<int64_t>(R, 128)));
  if (R == 0) return;
  row_norms(s, idx.data.data(), R, idx.dim, idx.dim, idx.xn.data());
  dbuf<float> scale;
  if (idx.metric == CosineExpanded) {
    scale.alloc(static_cast<size_t>(R), s);
    count_launch();
    rsqrt_rows_kernel<<<blocks_for(R, 256), 256, 0, s>>>(idx.xn.data(), scale.data(), R);
  }
  tc_split_planes(s, idx.data.data(), R, idx.dim, idx.dim, idx.Kp, idx.hi.data(), nullptr, R, scale.data());
  count_launch();
  dbuf<float> hn(static_cast<size_t>(R), s);
  half_norms_masked_kernel<<<blocks_for(R, 256), 256, 0, s>>>(idx.xn.data(), idx.ids.data(), R, !is_l2(idx.metric), hn.data());
  B2_CUDA(cudaGetLastError());
  tc_pack_half_norms(s, hn.data(), R, idx.hx.data());
}

void refresh_centers_tc(resources* res, ivf_flat_index& idx)
{
  auto s = res->stream;
  dbuf<float> cn(static_cast<size_t>(idx.n_lists), s);
  row_norms(s, idx.centers.data(), idx.n_lists, idx.dim, idx.dim, cn.data());
  dbuf<float> scale;
  if (idx.metric == CosineExpanded) {
    scale.alloc(static_cast<size_t>(idx.n_lists), s);
    count_launch();
    rsqrt_rows_kernel<<<blocks_for(idx.n_lists, 256), 256, 0, s>>>(cn.data(), scale.data(), idx.n_lists);
  }
  idx.centers_tc.build(s, idx.centers.data(), idx.n_lists, idx.dim, is_l2(idx.metric) ? cn.data() : nullptr, true, scale.data());
}

// Append the rows of `t` (host or device, row-major fp32) with the given ids (device int64 or null => id0 + i).
void ivf_flat_extend(resources* res, ivf_flat_index& idx, const DLTensor& t, const int64_t* new_ids, int64_t id0)
{
  auto s = res->stream;
  if (t.shape[0] == 0) return;
  auto label = [&](const float* x, int64_t n, uint32_t* labels) {
    dbuf<float> scale;
    if (idx.metric == CosineExpanded) {
      dbuf<float> xn(static_cast<size_t>(n), s);
      row_norms(s, x, n, idx.dim, idx.dim, xn.data());
      scale.alloc(static_cast<size_t>(n), s);
      count_launch();
      rsqrt_rows_kernel<<<blocks_for(n, 256), 256, 0, s>>>(xn.data(), scale.data(), n);
    }
    label_rows(res, idx.centers_tc, x, n, idx.dim, scale.data(), labels);
  };
  auto write = [&](const float* x, int64_t n, const uint32_t*, const int64_t* dst_rows, float* data) {
    scatter_rows(s, x, n, idx.dim, dst_rows, data);
  };
  insert_rows(res, idx.lists, idx.data, idx.dim, idx.ids, t, idx.dim, new_ids, id0, label, write);
  refresh_tc_side(res, idx);
}

ivf_flat_index* ivf_flat_build(resources* res, const cuvsIvfFlatIndexParams& p, const DLTensor& ds)
{
  B2_EXPECTS(ds.ndim == 2, "dataset must be a 2-D tensor");
  B2_EXPECTS(dl_is_c_contiguous(ds), "dataset must be row-major contiguous");
  B2_EXPECTS(is_l2(p.metric) || p.metric == InnerProduct || p.metric == CosineExpanded, "ivf_flat: unsupported metric %d", int(p.metric));
  const int64_t n = ds.shape[0];
  const int d     = static_cast<int>(ds.shape[1]);
  B2_EXPECTS(n >= 1 && d >= 1, "empty dataset");
  B2_EXPECTS(p.n_lists >= 1 && static_cast<int64_t>(p.n_lists) <= n, "n_lists (%u) must be in [1, n_rows]", p.n_lists);
  B2_EXPECTS(tc_supported(res->device, d), "ivf_flat: dim %d > 128 is not supported by this build yet", d);
  auto idx               = std::make_unique<ivf_flat_index>();
  idx->device            = res->device;
  idx->metric            = p.metric;
  idx->metric_arg        = p.metric_arg;
  idx->dim               = d;
  idx->n_lists           = p.n_lists;
  idx->adaptive_centers  = p.adaptive_centers;
  idx->kmeans_n_iters    = p.kmeans_n_iters;
  idx->kmeans_trainset_fraction = p.kmeans_trainset_fraction;
  auto s = res->stream;

  dbuf<float> train;
  const int64_t n_train = training_subsample(s, dl_ptr<float>(ds), n, d, p.n_lists, p.kmeans_trainset_fraction, train);
  idx->centers.alloc(static_cast<size_t>(p.n_lists) * d);
  kmeans_train(res, train.data(), n_train, d, p.n_lists, std::max<uint32_t>(p.kmeans_n_iters, 1), idx->centers.data(), true, true,
               nullptr, nullptr);
  refresh_centers_tc(res, *idx);
  std::vector<int64_t> zero(p.n_lists, 0);
  idx->lists.set_sizes(s, zero);
  refresh_tc_side(res, *idx);
  if (p.add_data_on_build) ivf_flat_extend(res, *idx, ds, nullptr, 0);
  return idx.release();
}

void ivf_flat_search(resources* res, const ivf_flat_index& idx, uint32_t n_probes, const DLTensor& qt, const DLTensor& nt,
                     const DLTensor& dt, const uint32_t* keep_bits = nullptr, int64_t n_bits = 0)
{
  auto s           = res->stream;
  const int64_t nq = qt.shape[0];
  const int k      = static_cast<int>(nt.shape[1]);
  B2_EXPECTS(qt.shape[1] == idx.dim, "queries dim (%lld) != index dim (%d)", (long long)qt.shape[1], idx.dim);
  B2_EXPECTS(nt.shape[0] == nq && dt.shape[0] == nq && dt.shape[1] == k, "neighbors/distances shape mismatch");
  B2_EXPECTS(k >= 1 && k <= 64, "ivf_flat search: k must be in [1, 64] in this build (got %d)", k);
  B2_EXPECTS(n_probes >= 1, "n_probes must be >= 1");
  if (nq == 0) return;
  n_probes         = std::min<uint32_t>(n_probes, idx.n_lists);
  {
    // Query batching: the per-(query, probe) workspaces (gathered bf16 query rows, 2 x KC candidate slots, their per-query
    // concatenation) are bounded to ~3 GiB; slots are uint32, so nq * n_probes also stays below 2^31 per batch.
    const int64_t per_query = static_cast<int64_t>(n_probes) * (idx.Kp * 2 + 2 * 64 * 8 + 16);
    int64_t batch = std::max<int64_t>(1, (int64_t(3) << 30) / per_query);
    batch         = std::min<int64_t>(batch, (int64_t(1) << 31) / std::max<uint32_t>(n_probes, 1));
    if (nq > batch) {
      for (int64_t q0 = 0; q0 < nq; q0 += batch) {
        const int64_t rows = std::min(batch, nq - q0);
        dl_row_slice qs(qt, q0, rows), ns(nt, q0, rows), ds(dt, q0, rows);
        ivf_flat_search(res, idx, n_probes, qs.t, ns.t, ds.t, keep_bits, n_bits);
      }
      return;
    }
  }
  const float* q   = dl_ptr<float>(qt);
  int64_t* out_idx = dl_ptr<int64_t>(nt);
  float* out_dist  = dl_ptr<float>(dt);
  const bool select_min = idx.metric != InnerProduct;

  // ---- 1. coarse
  dbuf<float> qn(static_cast<size_t>(nq), s);
  row_norms(s, q, nq, idx.dim, idx.dim, qn.data());
  dbuf<float> qscale;
  if (idx.metric == CosineExpanded) {
    qscale.alloc(static_cast<size_t>(nq), s);
    count_launch();
    rsqrt_rows_kernel<<<blocks_for(nq, 256), 256, 0, s>>>(qn.data(), qscale.data(), nq);
  }
  tc_rows_tmp qp;
  qp.build(s, q, nq, idx.dim, true, 0, qscale.data());
  dbuf<uint32_t> probes(static_cast<size_t>(nq) * n_probes, s);
  coarse_select(res, qp, idx.centers_tc, static_cast<int>(n_probes), probes.data(), nullptr);

  // ---- 1b. bitset pre-filter (cuvs::neighbors::filtering::bitset_filter): one pass over the half-norm plane
  dbuf<__nv_bfloat16> hx_f;
  const __nv_bfloat16* hx = idx.hx.data();
  if (keep_bits != nullptr && idx.lists.rows_total > 0) {
    const int64_t R = idx.lists.rows_total;
    dbuf<float> hn(static_cast<size_t>(R), s);
    hx_f.alloc(static_cast<size_t>(std::max<int64_t>(R, 128)) * 16, s);
    count_launch();
    half_norms_filtered_kernel<<<blocks_for(R, 256), 256, 0, s>>>(idx.xn.data(), idx.ids.data(), R, !is_l2(idx.metric), keep_bits, n_bits,
                                                                   hn.data());
    B2_CUDA(cudaGetLastError());
    tc_pack_half_norms(s, hn.data(), R, hx_f.data());
    hx = hx_f.data();
  }

  // ---- 2. bucket (query, probe) pairs by list
  // The scan ranks rows by a ONE-pass bf16 score; the exact fp32 re-score below only sees what survives it.  Keep slack
  // between k and the per-list capacity (and the shared pruning bound, which tracks the KC-th best): a true top-k row whose
  // bf16 score ranks a few places late must still be a candidate.  k <= 10 -> 16 slots, k <= 32 -> 32 slots; the bound is
  // only used when KC >= 1.5 k.
  const int KC    = (k + k / 2 <= 16) ? 16 : 32;
  const bool use_bound = KC >= k + k / 2;
  const int lists = tc_lists_per_item();
  const int KCW   = KC * lists;
  B2_EXPECTS(KCW >= k, "ivf_flat search: k = %d exceeds the %d candidates kept per probe", k, KCW);
  probe_buckets pb;
  bucket_probes(res, probes.data(), nq, static_cast<int>(n_probes), idx.n_lists, idx.lists.d_offsets.data(), KCW, pb);

  // ---- 3. fine scan: gathered query rows (A) x list rows (B)
  const int64_t a_rows = pb.n_pairs + 128;
  dbuf<__nv_bfloat16> a_hi(static_cast<size_t>(a_rows) * idx.Kp, s);
  gather_rows_bf16(s, qp.hi.data(), pb.pair_query.data(), pb.n_items.data() + 1, a_rows, idx.Kp, a_hi.data());
  dbuf<float> cs(static_cast<size_t>(pb.n_pairs) * KCW, s);
  dbuf<uint32_t> cp(static_cast<size_t>(pb.n_pairs) * KCW, s);
  {
    // probes of one query share a running k'-th-best bound (same query => comparable scores)
    dbuf<int> bkeys(static_cast<size_t>(nq), s);
    B2_CUDA(cudaMemsetAsync(bkeys.data(), tc_bound_init_byte, sizeof(int) * nq, s));
    tc_bound bnd;
    bnd.keys = bkeys.data();
    bnd.idx  = pb.pair_query.data();
    timed_section ts("ivf_flat_scan", s);
    tc_scan_topk(s, res->device, a_hi.data(), nullptr, a_rows, idx.hi.data(), nullptr, std::max<int64_t>(idx.lists.rows_total, 128),
                 idx.Kp, hx, pb.items.data(), pb.max_items, pb.n_items.data(), KC, 1, cs.data(), cp.data(), KCW, use_bound ? &bnd : nullptr);
  }

  // ---- 4. per query: merge probes by approximate score, exact re-score, ids
  const int64_t cand_w = static_cast<int64_t>(n_probes) * KCW;
  dbuf<float> gs(static_cast<size_t>(nq) * cand_w, s);
  dbuf<uint32_t> gp(static_cast<size_t>(nq) * cand_w, s);
  gather_probe_candidates(s, cs.data(), cp.data(), pb.slot_of.data(), nq, static_cast<int>(n_probes), KCW, gs.data(), gp.data());
  const int kc2 = static_cast<int>(std::min<int64_t>(cand_w, std::max(32, 2 * k)));
  dbuf<float> ms(static_cast<size_t>(nq) * kc2, s);
  dbuf<uint32_t> mp(static_cast<size_t>(nq) * kc2, s);
  select_k(s, gs.data(), gp.data(), IDX_U32, nq, cand_w, cand_w, kc2, ms.data(), mp.data(), IDX_U32, true);
  cuvsDistanceType fine = idx.metric == InnerProduct ? InnerProduct : (idx.metric == CosineExpanded ? CosineExpanded : L2Unexpanded);
  rescore_topk(s, q, nq, idx.dim, idx.data.data(), idx.dim, idx.dim, qn.data(), idx.xn.data(), fine, mp.data(), nullptr, kc2,
               idx.ids.data(), k, out_idx, out_dist, INT64_MAX, approx_map{}, nullptr, nullptr);
  (void)select_min;
  postprocess_distances(s, out_dist, nq * k, idx.metric);
}

}  // namespace

}  // namespace b200

using namespace b200;

extern "C" {

cuvsError_t cuvsIvfFlatIndexParamsCreate(cuvsIvfFlatIndexParams_t* params)
{
  return guarded([=] {
    B2_EXPECTS(params != nullptr, "params is null");
    // defaults: c/src/neighbors/ivf_flat.cpp:265-277
    *params = new cuvsIvfFlatIndexParams{L2Expanded, 2.0f, true, 1024, 20, 0.5, false, false};
  });
}
cuvsError_t cuvsIvfFlatIndexParamsDestroy(cuvsIvfFlatIndexParams_t params) { return guarded([=] { delete params; }); }

cuvsError_t cuvsIvfFlatSearchParamsCreate(cuvsIvfFlatSearchParams_t* params)
{
  return guarded([=] {
    B2_EXPECTS(params != nullptr, "params is null");
    *params = new cuvsIvfFlatSearchParams{20};
  });
}
cuvsError_t cuvsIvfFlatSearchParamsDestroy(cuvsIvfFlatSearchParams_t params) { return guarded([=] { delete params; }); }

cuvsError_t cuvsIvfFlatIndexCreate(cuvsIvfFlatIndex_t* index)
{
  return guarded([=] {
    B2_EXPECTS(index != nullptr, "index is null");
    *index = new cuvsIvfFlatIndex{};
  });
}
cuvsError_t cuvsIvfFlatIndexDestroy(cuvsIvfFlatIndex_t index)
{
  return guarded([=] {
    if (!index) return;
    delete reinterpret_cast<ivf_flat_index*>(index->addr);
    delete index;
  });
}

static ivf_flat_index& flat_of(cuvsIvfFlatIndex_t index)
{
  B2_EXPECTS(index != nullptr && index->addr != 0, "index is not built");
  return *reinterpret_cast<ivf_flat_index*>(index->addr);
}

cuvsError_t cuvsIvfFlatIndexGetNLists(cuvsIvfFlatIndex_t index, int64_t* n_lists)
{
  return guarded([=] { *n_lists = flat_of(index).n_lists; });
}
cuvsError_t cuvsIvfFlatIndexGetDim(cuvsIvfFlatIndex_t index, int64_t* dim) { return guarded([=] { *dim = flat_of(index).dim; }); }
cuvsError_t cuvsIvfFlatIndexGetCenters(cuvsIvfFlatIndex_t index, DLManagedTensor* centers)
{
  return guarded([=] {
    auto& idx        = flat_of(index);
    int64_t shape[2] = {idx.n_lists, idx.dim};
    dl_fill_view(centers, idx.centers.data(), idx.device, DLDataType{kDLFloat, 32, 1}, 2, shape);
  });
}

cuvsError_t cuvsB200IvfFlatGetListSizes(cuvsIvfFlatIndex_t index, DLManagedTensor* list_sizes)
{
  return guarded([=] {
    auto& idx        = flat_of(index);
    int64_t shape[1] = {idx.n_lists};
    dl_fill_view(list_sizes, idx.lists.d_sizes.data(), idx.device, DLDataType{kDLUInt, 32, 1}, 1, shape);
  });
}
cuvsError_t cuvsB200IvfFlatGetListIndices(cuvsIvfFlatIndex_t index, uint32_t label, DLManagedTensor* ids)
{
  return guarded([=] {
    auto& idx = flat_of(index);
    B2_EXPECTS(label < idx.n_lists, "label %u out of range", label);
    int64_t shape[1] = {idx.lists.h_sizes[label]};
    dl_fill_view(ids, idx.ids.data() + idx.lists.h_offsets[label], idx.device, DLDataType{kDLInt, 64, 1}, 1, shape);
  });
}
cuvsError_t cuvsB200IvfFlatSetCenters(cuvsResources_t res, cuvsIvfFlatIndex_t index, DLManagedTensor* centers)
{
  return guarded([=] {
    auto r    = as_res(res);
    auto& idx = flat_of(index);
    B2_EXPECTS(centers != nullptr, "centers is null");
    const DLTensor& c = centers->dl_tensor;
    B2_EXPECTS(dl_is(c, kDLFloat, 32) && c.ndim == 2 && c.shape[0] == idx.n_lists && c.shape[1] == idx.dim && dl_is_c_contiguous(c),
               "centers must be float32 [n_lists, dim]");
    B2_EXPECTS(idx.lists.size == 0, "centres can only be replaced while the index is empty");
    B2_CUDA(cudaMemcpyAsync(idx.centers.data(), dl_ptr<float>(c), sizeof(float) * idx.n_lists * idx.dim, cudaMemcpyDefault, r->stream));
    refresh_centers_tc(r, idx);
  });
}
cuvsError_t cuvsB200IvfFlatGetSize(cuvsIvfFlatIndex_t index, int64_t* size) { return guarded([=] { *size = flat_of(index).lists.size; }); }

cuvsError_t cuvsIvfFlatBuild(cuvsResources_t res, cuvsIvfFlatIndexParams_t params, DLManagedTensor* dataset, cuvsIvfFlatIndex_t index)
{
  return guarded([=] {
    auto r = as_res(res);
    B2_EXPECTS(params && dataset && index, "null argument");
    const DLTensor& ds = dataset->dl_tensor;
    B2_EXPECTS(dl_is_dataset_dtype(ds), "Unsupported dataset DLtensor dtype: %d and bits: %d", ds.dtype.code, ds.dtype.bits);
    if (index->addr) { delete reinterpret_cast<ivf_flat_index*>(index->addr); index->addr = 0; }
    f32_matrix w;  // float16 / int8 / uint8 datasets (c/src/neighbors/ivf_flat.cpp dtype switch) are widened to fp32 rows
    widen_to_f32(r, ds, w);
    index->addr  = reinterpret_cast<uintptr_t>(ivf_flat_build(r, *params, w.t));
    index->dtype = ds.dtype;
  });
}

cuvsError_t cuvsIvfFlatSearch(cuvsResources_t res, cuvsIvfFlatSearchParams_t params, cuvsIvfFlatIndex_t index,
                              DLManagedTensor* queries_t, DLManagedTensor* neighbors_t, DLManagedTensor* distances_t, cuvsFilter filter)
{
  return guarded([=] {
    auto r = as_res(res);
    B2_EXPECTS(params && queries_t && neighbors_t && distances_t, "null argument");
    auto& idx = flat_of(index);
    const DLTensor& queries   = queries_t->dl_tensor;
    const DLTensor& neighbors = neighbors_t->dl_tensor;
    const DLTensor& distances = distances_t->dl_tensor;
    B2_EXPECTS(dl_is_device(queries), "queries should have device compatible memory");
    B2_EXPECTS(dl_is_device(neighbors), "neighbors should have device compatible memory");
    B2_EXPECTS(dl_is_device(distances), "distances should have device compatible memory");
    B2_EXPECTS(dl_is(neighbors, kDLInt, 64), "neighbors should be of type int64_t");
    B2_EXPECTS(dl_is(distances, kDLFloat, 32), "distances should be of type float32");
    B2_EXPECTS(queries.dtype.code == index->dtype.code && queries.dtype.bits == index->dtype.bits, "type mismatch between index and queries");
    B2_EXPECTS(queries.ndim == 2 && neighbors.ndim == 2 && distances.ndim == 2, "queries/neighbors/distances must be 2-D");
    B2_EXPECTS(dl_is_c_contiguous(queries) && dl_is_c_contiguous(neighbors) && dl_is_c_contiguous(distances), "tensors must be row-major contiguous");
    const uint32_t* keep = nullptr;
    int64_t n_bits       = 0;
    if (filter.type != NO_FILTER) {
      B2_EXPECTS(filter.type == BITSET, "ivf_flat search: only bitset pre-filters are supported (as in the reference)");
      auto ft = reinterpret_cast<DLManagedTensor*>(filter.addr);
      B2_EXPECTS(ft != nullptr && dl_is_device(ft->dl_tensor), "prefilter should have device compatible memory");
      keep   = dl_ptr<uint32_t>(ft->dl_tensor);
      n_bits = ft->dl_tensor.shape[0] * 32;
    }
    f32_matrix w;
    widen_to_f32(r, queries, w);
    ivf_flat_search(r, idx, params->n_probes, w.t, neighbors, distances, keep, n_bits);
  });
}

cuvsError_t cuvsIvfFlatExtend(cuvsResources_t res, DLManagedTensor* new_vectors, DLManagedTensor* new_indices, cuvsIvfFlatIndex_t index)
{
  return guarded([=] {
    auto r    = as_res(res);
    auto& idx = flat_of(index);
    f32_matrix v;
    dbuf<int64_t> ids_buf;
    const int64_t* ids = extend_args(r, new_vectors, new_indices, idx.dim, v, ids_buf);
    ivf_flat_extend(r, idx, v.t, ids, idx.lists.size);  // reference: new ids continue after the current size when none are given
  });
}

// cuVS index file, serialization version 4 (cpp/src/neighbors/ivf_flat/ivf_flat_serialize.cuh:25-84; per-list records
// cpp/src/neighbors/ivf_list.cuh:108-133): the 4-byte dtype tag "<f4\0", then NPY records (npy_io.hpp) —
//   version i4 = 4, size i8, dim u4, n_lists u4, metric i4, adaptive_centers u1, conservative_memory_allocation u1,
//   centers f4 [n_lists, dim], has_norms u1 (+ center_norms f4 [n_lists] for L2), list_sizes u4 [n_lists], then per list:
//   capacity u4 = size rounded up to 32 and (capacity > 0) data f4 [capacity, dim] in the reference's interleaved layout
//   (groups of 32 rows, element (r, k) at (r/32)*32*dim + (k/veclen)*32*veclen + (r%32)*veclen + k%veclen, veclen = 4 when
//   dim % 4 == 0 else 1: ivf_flat.hpp:184-201) and indices i8 [capacity] (-1 = kInvalidRecord on the padding rows).
namespace {

inline int flat_veclen(int dim) { return dim % 4 == 0 ? 4 : 1; }

}  // namespace

cuvsError_t cuvsIvfFlatSerialize(cuvsResources_t res, const char* filename, cuvsIvfFlatIndex_t index)
{
  return guarded([=] {
    auto r    = as_res(res);
    auto& idx = flat_of(index);
    std::ofstream os(filename, std::ios::out | std::ios::binary);
    B2_EXPECTS(bool(os), "Cannot open file %s", filename);
    const char tag[4] = {'<', 'f', '4', 0};
    os.write(tag, 4);
    npy::write_scalar<int32_t>(os, 4);
    npy::write_scalar<int64_t>(os, idx.lists.size);
    npy::write_scalar<uint32_t>(os, static_cast<uint32_t>(idx.dim));
    npy::write_scalar<uint32_t>(os, idx.n_lists);
    npy::write_scalar<int32_t>(os, static_cast<int32_t>(idx.metric));
    npy::write_scalar<bool>(os, idx.adaptive_centers);
    npy::write_scalar<bool>(os, false);
    std::vector<float> c(static_cast<size_t>(idx.n_lists) * idx.dim);
    B2_CUDA(cudaMemcpyAsync(c.data(), idx.centers.data(), c.size() * sizeof(float), cudaMemcpyDeviceToHost, r->stream));
    B2_CUDA(cudaStreamSynchronize(r->stream));
    npy::write_array<float>(os, c.data(), {static_cast<int64_t>(idx.n_lists), idx.dim});
    const bool has_norms = is_l2(idx.metric);
    npy::write_scalar<bool>(os, has_norms);
    if (has_norms) {
      std::vector<float> cn(idx.n_lists);
      for (uint32_t l = 0; l < idx.n_lists; ++l) {
        float acc = 0.f;
        for (int j = 0; j < idx.dim; ++j) acc = fmaf(c[static_cast<size_t>(l) * idx.dim + j], c[static_cast<size_t>(l) * idx.dim + j], acc);
        cn[l] = acc;
      }
      npy::write_array<float>(os, cn.data(), {static_cast<int64_t>(idx.n_lists)});
    }
    std::vector<uint32_t> sizes(idx.n_lists);
    for (uint32_t l = 0; l < idx.n_lists; ++l) sizes[l] = static_cast<uint32_t>(idx.lists.h_sizes[l]);
    npy::write_array<uint32_t>(os, sizes.data(), {static_cast<int64_t>(idx.n_lists)});
    std::vector<float> rows, inter;
    std::vector<int64_t> ids;
    const int dim = idx.dim, vl = flat_veclen(dim);
    for (uint32_t l = 0; l < idx.n_lists; ++l) {
      const int64_t sz = idx.lists.h_sizes[l], cap = (sz + 31) / 32 * 32;
      npy::write_scalar<uint32_t>(os, static_cast<uint32_t>(cap));
      if (!cap) continue;
      rows.resize(static_cast<size_t>(sz) * dim);
      ids.assign(static_cast<size_t>(cap), int64_t(-1));
      inter.assign(static_cast<size_t>(cap) * dim, 0.f);
      B2_CUDA(cudaMemcpyAsync(rows.data(), idx.data.data() + idx.lists.h_offsets[l] * dim, rows.size() * sizeof(float), cudaMemcpyDeviceToHost, r->stream));
      B2_CUDA(cudaMemcpyAsync(ids.data(), idx.ids.data() + idx.lists.h_offsets[l], static_cast<size_t>(sz) * sizeof(int64_t), cudaMemcpyDeviceToHost, r->stream));
      B2_CUDA(cudaStreamSynchronize(r->stream));
      for (int64_t rr = 0; rr < sz; ++rr)
        for (int k = 0; k < dim; ++k)
          inter[static_cast<size_t>((rr / 32) * 32 * dim + (k / vl) * 32 * vl + (rr % 32) * vl + k % vl)] = rows[static_cast<size_t>(rr) * dim + k];
      npy::write_array<float>(os, inter.data(), {cap, dim});
      npy::write_array<int64_t>(os, ids.data(), {cap});
    }
    B2_EXPECTS(bool(os), "Error writing %s", filename);
  });
}

cuvsError_t cuvsIvfFlatDeserialize(cuvsResources_t res, const char* filename, cuvsIvfFlatIndex_t index)
{
  return guarded([=] {
    auto r = as_res(res);
    B2_EXPECTS(index && filename, "null argument");
    std::ifstream is(filename, std::ios::in | std::ios::binary);
    B2_EXPECTS(bool(is), "Cannot open file %s", filename);
    char tag[4]{};
    B2_EXPECTS(bool(is.read(tag, 4)), "ivf_flat::deserialize: failed to read dtype prefix");
    B2_EXPECTS(tag[0] == '<' && tag[1] == 'f' && tag[2] == '4', "ivf_flat::deserialize: serialized dtype prefix does not match requested type");
    const int ver = npy::read_scalar<int32_t>(is, filename);
    B2_EXPECTS(ver == 4, "serialization version mismatch, expected %d, got %d ", 4, ver);
    const int64_t n_rows = npy::read_scalar<int64_t>(is, filename);
    auto idx      = std::make_unique<ivf_flat_index>();
    idx->device   = r->device;
    idx->dim      = static_cast<int>(npy::read_scalar<uint32_t>(is, filename));
    idx->n_lists  = npy::read_scalar<uint32_t>(is, filename);
    idx->metric   = static_cast<cuvsDistanceType>(npy::read_scalar<int32_t>(is, filename));
    idx->adaptive_centers = npy::read_scalar<uint8_t>(is, filename) != 0;
    (void)npy::read_scalar<uint8_t>(is, filename);  // conservative_memory_allocation: an allocation policy, nothing to restore
    std::vector<float> c(static_cast<size_t>(idx->n_lists) * idx->dim);
    npy::read_array<float>(is, c.data(), static_cast<int64_t>(c.size()), filename);
    if (npy::read_scalar<uint8_t>(is, filename) != 0) {
      std::vector<float> cn(idx->n_lists);  // recomputed on load (refresh_centers_tc)
      npy::read_array<float>(is, cn.data(), idx->n_lists, filename);
    }
    std::vector<uint32_t> sizes32(idx->n_lists);
    npy::read_array<uint32_t>(is, sizes32.data(), idx->n_lists, filename);
    std::vector<int64_t> sizes(sizes32.begin(), sizes32.end());
    idx->centers.alloc(c.size());
    B2_CUDA(cudaMemcpyAsync(idx->centers.data(), c.data(), c.size() * sizeof(float), cudaMemcpyHostToDevice, r->stream));
    B2_CUDA(cudaStreamSynchronize(r->stream));
    refresh_centers_tc(r, *idx);
    idx->lists.set_sizes(r->stream, sizes);
    B2_EXPECTS(idx->lists.size == n_rows, "ivf_flat::deserialize: list sizes sum to %lld, header says %lld rows", (long long)idx->lists.size,
               (long long)n_rows);
    alloc_padded(r->stream, idx->lists.rows_total, idx->dim, idx->data, idx->ids);
    std::vector<float> rows, inter;
    std::vector<int64_t> ids;
    const int dim = idx->dim, vl = flat_veclen(dim);
    for (uint32_t l = 0; l < idx->n_lists; ++l) {
      const int64_t cap = npy::read_scalar<uint32_t>(is, filename);
      const int64_t sz  = sizes[l];
      B2_EXPECTS(cap >= sz, "ivf_flat::deserialize: list %u stores %lld rows, list_sizes says %lld", l, (long long)cap, (long long)sz);
      if (!cap) continue;
      inter.resize(static_cast<size_t>(cap) * dim);
      ids.resize(static_cast<size_t>(cap));
      npy::read_array<float>(is, inter.data(), cap * dim, filename);
      npy::read_array<int64_t>(is, ids.data(), cap, filename);
      if (!sz) continue;
      rows.resize(static_cast<size_t>(sz) * dim);
      for (int64_t rr = 0; rr < sz; ++rr)
        for (int k = 0; k < dim; ++k)
          rows[static_cast<size_t>(rr) * dim + k] = inter[static_cast<size_t>((rr / 32) * 32 * dim + (k / vl) * 32 * vl + (rr % 32) * vl + k % vl)];
      B2_CUDA(cudaMemcpyAsync(idx->data.data() + idx->lists.h_offsets[l] * dim, rows.data(), rows.size() * sizeof(float), cudaMemcpyHostToDevice, r->stream));
      B2_CUDA(cudaMemcpyAsync(idx->ids.data() + idx->lists.h_offsets[l], ids.data(), static_cast<size_t>(sz) * sizeof(int64_t), cudaMemcpyHostToDevice, r->stream));
      B2_CUDA(cudaStreamSynchronize(r->stream));
    }
    refresh_tc_side(r, *idx);
    if (index->addr) delete reinterpret_cast<ivf_flat_index*>(index->addr);
    index->addr  = reinterpret_cast<uintptr_t>(idx.release());
    index->dtype = DLDataType{kDLFloat, 32, 1};
  });
}

}  // extern "C"
