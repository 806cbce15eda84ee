// k-means: cuvsKMeansFit / Predict / ClusterCost behind the C boundary.
//
// Reference path (SURVEY §8a row a18): the assignment step
//   cpp/src/cluster/detail/minClusterDistanceCompute.cu:18-165 — on sm_100 the reference *disables* its fused
//   kernel (kmeans_common.cuh:60-84) and runs cuBLAS GEMM into an n x k fp32 matrix + reduce_min_kernel
//   (unfused_distance_nn.cuh:54-118), i.e. n*k*4 bytes written and read back through HBM per iteration.
// Here the assignment is the tcgen05 scan kernel with its fused top-1 epilogue (ivf_common.cu: assign_nearest):
// the n x k score block lives in TMEM only.  Lloyd iterations, centroid update (per-cluster sums in row order, so the same
// input gives the same centroids) and the inertia reduction are plain CUDA; C wrapper semantics follow c/src/cluster/kmeans.cpp.
#include "common.hpp"
#include "exact.cuh"
#include "ivf_common.cuh"
#include "select_k.cuh"
#include "timing.hpp"

#include <cuvs/cluster/kmeans.h>

#include <algorithm>
#include <cfloat>
#include <cmath>
#include <vector>

namespace b200 {
namespace {

inline unsigned blocks_for(int64_t n, int bs) { return static_cast<unsigned>((n + bs - 1) / bs); }

__global__ void u32_to_i32_kernel(const uint32_t* in, int32_t* out, int64_t n)
{
  int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  if (i < n) out[i] = static_cast<int32_t>(in[i]);
}

__global__ void weighted_cost_kernel(const float* __restrict__ s, const float* __restrict__ xn, const float* __restrict__ w, int64_t n,
                                     double* __restrict__ out)
{
  double acc = 0;
  for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < n; i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    float dist = fmaf(2.0f, s[i], xn[i]);
    if (dist < 0.f) dist = 0.f;  // unfused_distance_nn.cuh:79-83 clamps at 0
    acc += static_cast<double>(w ? w[i] * dist : dist);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0) atomicAdd(out, acc);
}

// ---- k-means++ seeding (D^2 sampling, one centre per step).  Sampling proportional to w_i is done as
// argmax_i w_i / E_i with E_i ~ Exp(1) drawn from a counter-based hash, so a step is one pass + one 64-bit atomicMax.
__device__ __forceinline__ uint64_t mix64(uint64_t z)
{
  z += 0x9e3779b97f4a7c15ull;
  z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ull;
  z = (z ^ (z >> 27)) * 0x94d049bb133111ebull;
  return z ^ (z >> 31);
}
__global__ void kpp_step_kernel(const float* __restrict__ x, int64_t n, int d, int64_t new_row, float* __restrict__ mind, int step,
                                unsigned long long* __restrict__ best)
{
  extern __shared__ float c[];
  for (int j = threadIdx.x; j < d; j += blockDim.x) c[j] = x[new_row * d + j];
  __syncthreads();
  int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  unsigned long long key = 0;
  if (i < n) {
    float acc = 0.f;
    for (int j = 0; j < d; ++j) { float t = x[i * d + j] - c[j]; acc = fmaf(t, t, acc); }
    float m = step == 0 ? acc : fminf(mind[i], acc);
    mind[i] = m;
    const uint64_t h = mix64((static_cast<uint64_t>(step) << 40) ^ static_cast<uint64_t>(i));
    const float u    = (static_cast<float>(h >> 40) + 0.5f) * (1.0f / 16777216.0f);
    const float e    = -__logf(u);
    const float w    = m / fmaxf(e, 1e-20f);
    key = (static_cast<unsigned long long>(__float_as_uint(w)) << 32) | static_cast<uint32_t>(i);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    unsigned long long t = __shfl_xor_sync(0xffffffffu, key, o);
    key = t > key ? t : key;
  }
  if ((threadIdx.x & 31) == 0 && key) atomicMax(best, key);
}
__global__ void copy_row_kernel(const float* __restrict__ x, int64_t row, int d, float* __restrict__ dst)
{
  for (int j = threadIdx.x; j < d; j += blockDim.x) dst[j] = x[row * d + j];
}

void kmeanspp_init(resources* r, const float* x, int64_t n, int d, int k, float* centers)
{
  auto s = r->stream;
  dbuf<float> mind(static_cast<size_t>(n), s);
  dbuf<unsigned long long> best(1, s);
  int64_t row = static_cast<int64_t>(0x2545F4914F6CDD1DULL % static_cast<uint64_t>(n));  // fixed first pick (rng_state{0} analogue)
  for (int c = 0; c < k; ++c) {
    copy_row_kernel<<<1, 128, 0, s>>>(x, row, d, centers + static_cast<int64_t>(c) * d);
    if (c + 1 == k) break;
    B2_CUDA(cudaMemsetAsync(best.data(), 0, sizeof(unsigned long long), s));
    count_launch(2);
    kpp_step_kernel<<<blocks_for(n, 256), 256, d * sizeof(float), s>>>(x, n, d, row, mind.data(), c, best.data());
    unsigned long long h = 0;
    B2_CUDA(cudaMemcpyAsync(&h, best.data(), sizeof(h), cudaMemcpyDeviceToHost, s));
    B2_CUDA(cudaStreamSynchronize(s));
    row = static_cast<int64_t>(h & 0xffffffffull);
  }
  B2_CUDA(cudaGetLastError());
}

struct dev_matrix {
  const float* p = nullptr;
  dbuf<float> staged;
  int64_t n = 0;
  int d     = 0;
};

void stage(resources* r, const DLTensor& t, dev_matrix& m, const char* name)
{
  B2_EXPECTS(dl_is(t, kDLFloat, 32), "%s must be float32", name);
  B2_EXPECTS(t.ndim == 2 && dl_is_c_contiguous(t), "%s must be a row-major 2-D tensor", name);
  m.n = t.shape[0];
  m.d = static_cast<int>(t.shape[1]);
  if (dl_is_device(t) && t.device.device_type != kDLCUDAHost) m.p = dl_ptr<float>(t);
  else {
    m.staged.alloc(static_cast<size_t>(m.n) * m.d, r->stream);
    B2_CUDA(cudaMemcpyAsync(m.staged.data(), dl_ptr<float>(t), sizeof(float) * m.n * m.d, cudaMemcpyHostToDevice, r->stream));
    m.p = m.staged.data();
  }
}

// labels + inertia for fixed centroids
void predict(resources* r, const float* x, int64_t n, int d, const float* centroids, int k, const float* weights, uint32_t* labels,
             double* inertia)
{
  auto s = r->stream;
  B2_EXPECTS(tc_supported(r->device, d), "kmeans: dim %d > 128 is not supported by this build yet", d);
  tc_rows_tmp xp;
  xp.build(s, x, n, d, true);
  dbuf<float> cn(static_cast<size_t>(k), s), xn(static_cast<size_t>(n), s), scores(static_cast<size_t>(n), s);
  row_norms(s, centroids, k, d, d, cn.data());
  row_norms(s, x, n, d, d, xn.data());
  tc_rows cp;
  cp.build(s, centroids, k, d, cn.data(), true);
  assign_nearest(r, xp.hi.data(), xp.lo.data(), n, xp.rows_pad, xp.Kp, cp, labels, scores.data());
  if (inertia) {
    dbuf<double> acc(1, s);
    B2_CUDA(cudaMemsetAsync(acc.data(), 0, sizeof(double), s));
    count_launch();
    weighted_cost_kernel<<<256, 256, 0, s>>>(scores.data(), xn.data(), weights, n, acc.data());
    B2_CUDA(cudaMemcpyAsync(inertia, acc.data(), sizeof(double), cudaMemcpyDeviceToHost, s));
    B2_CUDA(cudaStreamSynchronize(s));
  }
}

struct fit_args {
  cuvsDistanceType metric;
  int n_clusters, max_iter, n_init;
  cuvsKMeansInitMethod init;
  double tol;
  bool balanced;
  int balanced_iters;
};

void fit(resources* r, const fit_args& a, DLManagedTensor* X, DLManagedTensor* sample_weight, DLManagedTensor* centroids, double* inertia,
         int* n_iter)
{
  B2_EXPECTS(X && centroids, "null argument");
  B2_EXPECTS(a.metric == L2Expanded || a.metric == L2SqrtExpanded || a.metric == L2Unexpanded || a.metric == L2SqrtUnexpanded,
             "kmeans: only (squared) euclidean metrics are supported, got %d", int(a.metric));
  B2_EXPECTS(a.n_clusters >= 1, "n_clusters must be >= 1");
  dev_matrix x;
  stage(r, X->dl_tensor, x, "X");
  const DLTensor& ct = centroids->dl_tensor;
  B2_EXPECTS(dl_is(ct, kDLFloat, 32) && ct.ndim == 2 && ct.shape[0] == a.n_clusters && ct.shape[1] == x.d && dl_is_device(ct) && dl_is_c_contiguous(ct),
             "centroids must be a device float32 [n_clusters, dim] matrix");
  B2_EXPECTS(x.n >= a.n_clusters, "number of samples (%lld) must be >= n_clusters (%d)", (long long)x.n, a.n_clusters);
  B2_EXPECTS(sample_weight == nullptr, "kmeans fit: sample weights are not supported by this build yet");
  float* c = dl_ptr<float>(ct);
  int iters = 0;
  double cost = 0;
  const int max_iter = a.balanced ? std::max(a.balanced_iters, 1) : std::max(a.max_iter, 1);
  // KMeansPlusPlus: D^2 seeding (one pass per centre) up to 4096 clusters, evenly strided rows beyond / for Random
  bool strided = a.init != Array;
  if (a.init == KMeansPlusPlus && a.n_clusters <= 4096 && x.n < (int64_t(1) << 32)) {
    kmeanspp_init(r, x.p, x.n, x.d, a.n_clusters, c);
    strided = false;
  }
  kmeans_train(r, x.p, x.n, x.d, a.n_clusters, max_iter, c, strided, a.balanced, &cost, &iters, a.balanced ? 0.0 : a.tol);
  if (inertia) *inertia = cost;
  if (n_iter) *n_iter = iters;
}

}  // namespace
}  // namespace b200

using namespace b200;

extern "C" {

cuvsError_t cuvsKMeansParamsCreate(cuvsKMeansParams_t* params)
{
  return guarded([=] {
    B2_EXPECTS(params != nullptr, "params is null");
    // defaults of cuvs::cluster::kmeans::params (cpp/include/cuvs/cluster/kmeans.hpp:37-120) as mirrored by c/src/cluster/kmeans.cpp:228-249
    *params = new cuvsKMeansParams{L2Expanded, 8, KMeansPlusPlus, 300, 1e-4, 1, 2.0, 1 << 15, 0, false, false, 20, 0, 0};
  });
}
cuvsError_t cuvsKMeansParamsDestroy(cuvsKMeansParams_t params) { return guarded([=] { delete params; }); }
cuvsError_t cuvsKMeansParamsCreate_v2(cuvsKMeansParams_v2_t* params)
{
  return guarded([=] {
    B2_EXPECTS(params != nullptr, "params is null");
    *params = new cuvsKMeansParams_v2{L2Expanded, 8, KMeansPlusPlus, 300, 1e-4, 1, 2.0, 1 << 15, 0, false, 20, 0, 0};
  });
}
cuvsError_t cuvsKMeansParamsDestroy_v2(cuvsKMeansParams_v2_t params) { return guarded([=] { delete params; }); }

cuvsError_t cuvsKMeansFit(cuvsResources_t res, cuvsKMeansParams_t p, DLManagedTensor* X, DLManagedTensor* sample_weight,
                          DLManagedTensor* centroids, double* inertia, int* n_iter)
{
  return guarded([=] {
    B2_EXPECTS(p != nullptr, "params is null");
    fit(as_res(res), fit_args{p->metric, p->n_clusters, p->max_iter, p->n_init, p->init, p->tol, p->hierarchical, p->hierarchical_n_iters}, X,
        sample_weight, centroids, inertia, n_iter);
  });
}
cuvsError_t cuvsKMeansFit_v2(cuvsResources_t res, cuvsKMeansParams_v2_t p, DLManagedTensor* X, DLManagedTensor* sample_weight,
                             DLManagedTensor* centroids, double* inertia, int* n_iter)
{
  return guarded([=] {
    B2_EXPECTS(p != nullptr, "params is null");
    fit(as_res(res), fit_args{p->metric, p->n_clusters, p->max_iter, p->n_init, p->init, p->tol, p->hierarchical, p->hierarchical_n_iters}, X,
        sample_weight, centroids, inertia, n_iter);
  });
}

static void predict_c(cuvsResources_t res, DLManagedTensor* X, DLManagedTensor* sample_weight, DLManagedTensor* centroids,
                      DLManagedTensor* labels, bool normalize_weight, double* inertia)
{
  auto r = as_res(res);
  B2_EXPECTS(X && centroids && labels, "null argument");
  dev_matrix x;
  stage(r, X->dl_tensor, x, "X");
  const DLTensor& ct = centroids->dl_tensor;
  const DLTensor& lt = labels->dl_tensor;
  B2_EXPECTS(dl_is(ct, kDLFloat, 32) && ct.ndim == 2 && ct.shape[1] == x.d && dl_is_device(ct) && dl_is_c_contiguous(ct), "centroids must be a device float32 [k, dim] matrix");
  B2_EXPECTS((dl_is(lt, kDLInt, 32) || dl_is(lt, kDLUInt, 32)) && lt.shape[0] == x.n && dl_is_device(lt), "labels must be a device int32 [n] vector");
  const float* w = nullptr;
  dbuf<float> wbuf;
  if (sample_weight) {
    const DLTensor& wt = sample_weight->dl_tensor;
    B2_EXPECTS(dl_is(wt, kDLFloat, 32) && wt.shape[0] == x.n && dl_is_device(wt), "sample_weight must be a device float32 [n] vector");
    w = dl_ptr<float>(wt);
    (void)normalize_weight;  // weights are used as given for the cost; normalisation only rescales inertia in the reference
  }
  dbuf<uint32_t> tmp(static_cast<size_t>(x.n), r->stream);
  predict(r, x.p, x.n, x.d, dl_ptr<float>(ct), static_cast<int>(ct.shape[0]), w, tmp.data(), inertia);
  count_launch();
  u32_to_i32_kernel<<<blocks_for(x.n, 256), 256, 0, r->stream>>>(tmp.data(), dl_ptr<int32_t>(lt), x.n);
  B2_CUDA(cudaGetLastError());
}

cuvsError_t cuvsKMeansPredict(cuvsResources_t res, cuvsKMeansParams_t, DLManagedTensor* X, DLManagedTensor* sample_weight,
                              DLManagedTensor* centroids, DLManagedTensor* labels, bool normalize_weight, double* inertia)
{
  return guarded([=] { predict_c(res, X, sample_weight, centroids, labels, normalize_weight, inertia); });
}
cuvsError_t cuvsKMeansPredict_v2(cuvsResources_t res, cuvsKMeansParams_v2_t, DLManagedTensor* X, DLManagedTensor* sample_weight,
                                 DLManagedTensor* centroids, DLManagedTensor* labels, bool normalize_weight, double* inertia)
{
  return guarded([=] { predict_c(res, X, sample_weight, centroids, labels, normalize_weight, inertia); });
}

cuvsError_t cuvsKMeansClusterCost(cuvsResources_t res, DLManagedTensor* X, DLManagedTensor* centroids, double* cost)
{
  return guarded([=] {
    auto r = as_res(res);
    B2_EXPECTS(X && centroids && cost, "null argument");
    dev_matrix x;
    stage(r, X->dl_tensor, x, "X");
    const DLTensor& ct = centroids->dl_tensor;
    B2_EXPECTS(dl_is(ct, kDLFloat, 32) && ct.ndim == 2 && ct.shape[1] == x.d && dl_is_device(ct) && dl_is_c_contiguous(ct), "centroids must be a device float32 [k, dim] matrix");
    dbuf<uint32_t> tmp(static_cast<size_t>(x.n), r->stream);
    predict(r, x.p, x.n, x.d, dl_ptr<float>(ct), static_cast<int>(ct.shape[0]), nullptr, tmp.data(), cost);
  });
}

}  // extern "C"
