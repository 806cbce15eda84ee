// cuvs_b200 — shared host-side infrastructure of the C-ABI library.
//
// Plays the role RAFT/rmm play behind the reference's C layer (c/src/core/c_api.cpp:30-330,
// c/src/core/exceptions.hpp:17-33, c/src/core/interop.hpp): a per-caller resources object
// (device, stream, stream-ordered workspace), exception -> cuvsError_t translation with
// thread-local error text, and DLPack validation.  Plain C++ over the CUDA runtime.
#pragma once

#include <cuda_runtime.h>
#include <dlpack/dlpack.h>

#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <stdexcept>
#include <string>
#include <vector>

#include <cuvs/core/c_api.h>
#include <cuvs/distance/distance.h>

namespace b200 {

struct error : std::runtime_error {
  using std::runtime_error::runtime_error;
};

[[noreturn]] inline void fail(const char* file, int line, const char* fmt, ...)
{
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  char msg[1200];
  snprintf(msg, sizeof(msg), "%s (%s:%d)", buf, file, line);
  throw error(msg);
}

#define B2_FAIL(...) ::b200::fail(__FILE__, __LINE__, __VA_ARGS__)
#define B2_EXPECTS(cond, ...)                      \
  do {                                             \
    if (!(cond)) { B2_FAIL(__VA_ARGS__); }         \
  } while (0)
#define B2_CUDA(call)                                                                   \
  do {                                                                                  \
    cudaError_t e__ = (call);                                                           \
    if (e__ != cudaSuccess) {                                                           \
      B2_FAIL("CUDA error %s: %s at `%s`", cudaGetErrorName(e__), cudaGetErrorString(e__), #call); \
    }                                                                                   \
  } while (0)

void set_last_error(const char* msg);  // c_api_core.cu

/** Run `fn`, translating any exception into CUVS_ERROR + thread-local text (never throws). */
template <typename Fn>
cuvsError_t guarded(Fn&& fn) noexcept
{
  try {
    fn();
    set_last_error(nullptr);
    return CUVS_SUCCESS;
  } catch (const std::exception& e) {
    set_last_error(e.what());
  } catch (...) {
    set_last_error("unknown exception");
  }
  return CUVS_ERROR;
}

/** What a cuvsResources_t points at. One per caller thread; not thread-safe (same as raft::resources). */
struct resources {
  int device            = 0;
  cudaStream_t stream   = cudaStreamPerThread;
  int sm_count          = 0;
  std::vector<int> mg_devices;  // non-empty for multi-GPU handles
  std::vector<cudaStream_t> mg_streams;
};

inline resources* as_res(cuvsResources_t r)
{
  B2_EXPECTS(r != 0, "null cuvsResources_t");
  return reinterpret_cast<resources*>(r);
}

/** Stream-ordered device buffer (cudaMallocAsync on the handle's stream; pool keeps freed blocks). */
template <typename T>
struct dbuf {
  T* p           = nullptr;
  size_t n       = 0;
  cudaStream_t s = nullptr;
  dbuf() = default;
  dbuf(size_t count, cudaStream_t stream) { alloc(count, stream); }
  dbuf(const dbuf&)            = delete;
  dbuf& operator=(const dbuf&) = delete;
  dbuf(dbuf&& o) noexcept : p(o.p), n(o.n), s(o.s) { o.p = nullptr; o.n = 0; }
  dbuf& operator=(dbuf&& o) noexcept
  {
    if (this != &o) { release(); p = o.p; n = o.n; s = o.s; o.p = nullptr; o.n = 0; }
    return *this;
  }
  void alloc(size_t count, cudaStream_t stream)
  {
    release();
    n = count;
    s = stream;
    if (count) { B2_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&p), count * sizeof(T), stream)); }
  }
  void release() noexcept
  {
    if (p) { cudaFreeAsync(p, s); p = nullptr; }
    n = 0;
  }
  ~dbuf() { release(); }
  T* data() const { return p; }
  size_t size() const { return n; }
};

/** Long-lived device allocation owned by an index object (plain cudaMalloc). */
template <typename T>
struct owned {
  T* p     = nullptr;
  size_t n = 0;
  owned() = default;
  explicit owned(size_t count) { alloc(count); }
  owned(const owned&)            = delete;
  owned& operator=(const owned&) = delete;
  owned(owned&& o) noexcept : p(o.p), n(o.n) { o.p = nullptr; o.n = 0; }
  owned& operator=(owned&& o) noexcept
  {
    if (this != &o) { release(); p = o.p; n = o.n; o.p = nullptr; o.n = 0; }
    return *this;
  }
  void alloc(size_t count)
  {
    release();
    n = count;
    if (count) { B2_CUDA(cudaMalloc(reinterpret_cast<void**>(&p), count * sizeof(T))); }
  }
  void release() noexcept
  {
    if (p) { cudaFree(p); p = nullptr; }
    n = 0;
  }
  ~owned() { release(); }
  T* data() const { return p; }
  size_t size() const { return n; }
};

// ------------------------------------------------------------------------------------ DLPack
inline bool dl_is_device(const DLTensor& t)
{
  return t.device.device_type == kDLCUDA || t.device.device_type == kDLCUDAHost ||
         t.device.device_type == kDLCUDAManaged;
}
inline bool dl_is_host(const DLTensor& t)
{
  return t.device.device_type == kDLCPU || t.device.device_type == kDLCUDAHost;
}
inline bool dl_is(const DLTensor& t, uint8_t code, uint8_t bits)
{
  return t.dtype.code == code && t.dtype.bits == bits && t.dtype.lanes == 1;
}
inline bool dl_is_c_contiguous(const DLTensor& t)
{
  if (t.strides == nullptr) return true;
  int64_t expect = 1;
  for (int i = t.ndim - 1; i >= 0; --i) {
    if (t.shape[i] != 1 && t.strides[i] != expect) return false;
    expect *= t.shape[i];
  }
  return true;
}
inline bool dl_is_f_contiguous(const DLTensor& t)
{
  if (t.strides == nullptr) return t.ndim <= 1;
  int64_t expect = 1;
  for (int i = 0; i < t.ndim; ++i) {
    if (t.shape[i] != 1 && t.strides[i] != expect) return false;
    expect *= t.shape[i];
  }
  return true;
}
// `byte_offset` is deliberately NOT applied: the reference's C layer never reads it (from_dlpack builds the mdspan from
// `tensor.data` alone: c/src/core/detail/interop.hpp:138) and its own C tests pass stack DLManagedTensors that leave the field
// uninitialised (c/tests/neighbors/run_brute_force_c.c:26-36) — honouring it would turn those callers' garbage into
// misaligned device addresses.  Producers that need an offset fold it into `data` (torch's DLPack exporter does).
template <typename T>
inline T* dl_ptr(const DLTensor& t)
{
  return reinterpret_cast<T*>(t.data);
}
inline const DLTensor& dl_req(DLManagedTensor* m, const char* name)
{
  B2_EXPECTS(m != nullptr && m->dl_tensor.data != nullptr || (m != nullptr && m->dl_tensor.ndim > 0 &&
             m->dl_tensor.shape != nullptr), "%s tensor is null", name);
  return m->dl_tensor;
}
inline void dl_expect_matrix(const DLTensor& t, const char* name)
{
  B2_EXPECTS(t.ndim == 2, "%s must be a 2-D tensor (got ndim=%d)", name, t.ndim);
}

/** Rows [r0, r0 + rows) of a C-contiguous 2-D tensor as a non-owning view (query batching inside the searches). */
struct dl_row_slice {
  DLTensor t;
  int64_t shape[2];
  dl_row_slice(const DLTensor& src, int64_t r0, int64_t rows)
  {
    t           = src;
    shape[0]    = rows;
    shape[1]    = src.shape[1];
    t.shape     = shape;
    t.strides   = nullptr;
    t.data      = static_cast<char*>(src.data) + r0 * src.shape[1] * ((src.dtype.bits * src.dtype.lanes + 7) / 8);
    t.byte_offset = 0;
  }
  dl_row_slice(const dl_row_slice&) = delete;
};

/**
 * fp32 view of a dataset / query matrix given as float32, float16, int8 or uint8 — the element types the reference's C ABI
 * dispatches on (c/src/neighbors/ivf_pq.cpp:80-103, ivf_flat.cpp, brute_force.cpp:60-110, cagra.cpp:245-264).  float32
 * passes through untouched; the narrower types are widened into an owned device buffer (host sources are staged), values
 * unchanged — the reference maps int8 / uint8 through utils::mapping<float> and scales the distances back
 * (ivf_pq_search.cuh:1043), which is the same arithmetic in different units.  All kernels of this library then run on fp32.
 */
struct f32_matrix {
  DLTensor t{};
  int64_t shape[2] = {0, 0};
  owned<float> own;      // non-empty when the source was widened
  bool widened = false;
  f32_matrix() = default;
  f32_matrix(const f32_matrix&) = delete;
};
inline bool dl_is_dataset_dtype(const DLTensor& t)
{
  return dl_is(t, kDLFloat, 32) || dl_is(t, kDLFloat, 16) || dl_is(t, kDLInt, 8) || dl_is(t, kDLUInt, 8);
}
void widen_to_f32(struct resources* res, const DLTensor& src, f32_matrix& out);

/** Fill a caller-provided DLManagedTensor as a non-owning row-major view (used by index getters). */
void dl_fill_view(DLManagedTensor* out, void* data, int device, DLDataType dt, int ndim, const int64_t* shape);

inline bool metric_is_min_close(cuvsDistanceType m) { return m != InnerProduct; }
inline bool is_l2(cuvsDistanceType m) { return m == L2Expanded || m == L2SqrtExpanded || m == L2Unexpanded || m == L2SqrtUnexpanded; }

inline unsigned blocks_for(int64_t n, int bs) { return static_cast<unsigned>((n + bs - 1) / bs); }

/** Integer value of environment variable `name`, `dflt` when it is unset. */
inline int64_t env_int(const char* name, int64_t dflt)
{
  const char* v = getenv(name);
  return v ? atoll(v) : dflt;
}

inline int sm_count_of(int device)
{
  int v = 0;
  B2_CUDA(cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, device));
  return v;
}

}  // namespace b200
