// List layout helpers (see ivf_lists.cuh).
#include "ivf_lists.cuh"
#include "timing.hpp"

#include <cub/device/device_radix_sort.cuh>

#include <algorithm>
#include <utility>

namespace b200 {
namespace {
__global__ void count_labels_kernel(const uint32_t* __restrict__ labels, int64_t n, unsigned long long* __restrict__ counts)
{
  int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  if (i < n) atomicAdd(&counts[labels[i]], 1ull);
}
__global__ void iota_kernel(uint32_t* __restrict__ v, int64_t n)
{
  int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  if (i < n) v[i] = static_cast<uint32_t>(i);
}
// start[g] = first sorted position with key >= g, for every g in [0, n_groups]
__global__ void group_starts_kernel(const uint32_t* __restrict__ sorted, int64_t n, int64_t n_groups, int64_t* __restrict__ start)
{
  int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  if (i >= n) return;
  const int64_t k    = sorted[i];
  const int64_t prev = i ? static_cast<int64_t>(sorted[i - 1]) : -1;
  for (int64_t g = prev + 1; g <= k; ++g) start[g] = i;
  if (i == n - 1)
    for (int64_t g = k + 1; g <= n_groups; ++g) start[g] = n;
}
// position of row order[p] inside its list = its rank among the rows of that list (sorted keys = labels)
__global__ void place_rows_kernel(const uint32_t* __restrict__ sorted, const uint32_t* __restrict__ order, int64_t n,
                                  const int64_t* __restrict__ start, const int64_t* __restrict__ offsets,
                                  const int64_t* __restrict__ base_fill, int64_t* __restrict__ dst)
{
  int64_t p = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  if (p >= n) return;
  const uint32_t l = sorted[p];
  dst[order[p]]    = offsets[l] + base_fill[l] + (p - start[l]);
}
__global__ void fill_pad_ids_kernel(int64_t* __restrict__ ids, int64_t n)
{
  int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  if (i < n) ids[i] = kPadId;
}
// one CTA per list
__global__ void remap_rows_kernel(const int64_t* __restrict__ from_off, const uint32_t* __restrict__ from_sizes,
                                  const int64_t* __restrict__ to_off, int64_t* __restrict__ dst_rows)
{
  const int64_t l = blockIdx.x, o = from_off[l], rows = from_off[l + 1] - o;
  for (int64_t i = threadIdx.x; i < rows; i += blockDim.x) dst_rows[o + i] = i < from_sizes[l] ? to_off[l] + i : -1;
}
template <typename T>
__global__ void scatter_rows_kernel(const T* __restrict__ src, int64_t rows, int row_elems, const int64_t* __restrict__ dst_rows,
                                    T* __restrict__ dst)
{
  int64_t t = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  if (t >= rows * row_elems) return;
  const int64_t o = dst_rows[t / row_elems];
  if (o >= 0) dst[o * row_elems + t % row_elems] = src[t];
}
__global__ void store_ids_kernel(const int64_t* __restrict__ dst_rows, int64_t n, const int64_t* __restrict__ new_ids, int64_t id0,
                                 int64_t* __restrict__ ids)
{
  int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  if (i < n) ids[dst_rows[i]] = new_ids ? new_ids[i] : id0 + i;
}
}  // namespace

void iota_u32(cudaStream_t s, dbuf<uint32_t>& v, int64_t n)
{
  B2_EXPECTS(n < (int64_t(1) << 32), "%lld items do not fit 32-bit indices", (long long)n);
  v.alloc(static_cast<size_t>(n), s);
  if (n == 0) return;
  count_launch();
  iota_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, s>>>(v.data(), n);
  B2_CUDA(cudaGetLastError());
}

void group_by_key(cudaStream_t s, dbuf<uint32_t>& keys, dbuf<uint32_t>& values, int64_t n_groups, dbuf<int64_t>& start)
{
  const int64_t n = static_cast<int64_t>(keys.size());
  B2_EXPECTS(n >= 1 && values.size() == keys.size(), "group_by_key: empty input or mismatched key / value counts");
  B2_EXPECTS(n_groups >= 1 && n_groups <= (int64_t(1) << 32), "group_by_key: %lld groups", (long long)n_groups);
  int end_bit = 1;
  while (end_bit < 32 && (int64_t(1) << end_bit) < n_groups) ++end_bit;
  dbuf<uint32_t> keys_alt(static_cast<size_t>(n), s), values_alt(static_cast<size_t>(n), s);
  cub::DoubleBuffer<uint32_t> dk(keys.data(), keys_alt.data()), dv(values.data(), values_alt.data());
  size_t tmp_bytes = 0;
  B2_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, dk, dv, n, 0, end_bit, s));
  dbuf<unsigned char> tmp(std::max<size_t>(tmp_bytes, 1), s);
  B2_CUDA(cub::DeviceRadixSort::SortPairs(tmp.data(), tmp_bytes, dk, dv, n, 0, end_bit, s));
  if (dk.Current() != keys.data()) std::swap(keys, keys_alt);
  if (dv.Current() != values.data()) std::swap(values, values_alt);
  start.alloc(static_cast<size_t>(n_groups + 1), s);
  count_launch();  // (the radix sort's own kernels are CUB's and not counted)
  group_starts_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, s>>>(keys.data(), n, n_groups, start.data());
  B2_CUDA(cudaGetLastError());
}

void list_layout::set_sizes(cudaStream_t s, const std::vector<int64_t>& sizes)
{
  n_lists = static_cast<int64_t>(sizes.size());
  h_sizes = sizes;
  h_offsets.assign(n_lists + 1, 0);
  size = 0;
  for (int64_t l = 0; l < n_lists; ++l) {
    h_offsets[l + 1] = h_offsets[l] + (sizes[l] + 127) / 128 * 128;
    size += sizes[l];
  }
  rows_total = h_offsets[n_lists];
  d_offsets.alloc(static_cast<size_t>(n_lists + 1));
  d_sizes.alloc(static_cast<size_t>(std::max<int64_t>(n_lists, 1)));
  std::vector<uint32_t> s32(sizes.begin(), sizes.end());
  B2_CUDA(cudaMemcpyAsync(d_offsets.data(), h_offsets.data(), sizeof(int64_t) * (n_lists + 1), cudaMemcpyHostToDevice, s));
  if (n_lists) B2_CUDA(cudaMemcpyAsync(d_sizes.data(), s32.data(), sizeof(uint32_t) * n_lists, cudaMemcpyHostToDevice, s));
  B2_CUDA(cudaStreamSynchronize(s));  // host vectors go out of scope
}

std::vector<int64_t> count_labels(cudaStream_t s, const uint32_t* labels, int64_t n, int64_t n_lists)
{
  dbuf<unsigned long long> c(static_cast<size_t>(n_lists), s);
  B2_CUDA(cudaMemsetAsync(c.data(), 0, sizeof(unsigned long long) * n_lists, s));
  if (n) {
    count_launch();
    count_labels_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, s>>>(labels, n, c.data());
    B2_CUDA(cudaGetLastError());
  }
  std::vector<unsigned long long> h(static_cast<size_t>(n_lists));
  B2_CUDA(cudaMemcpyAsync(h.data(), c.data(), sizeof(unsigned long long) * n_lists, cudaMemcpyDeviceToHost, s));
  B2_CUDA(cudaStreamSynchronize(s));
  return std::vector<int64_t>(h.begin(), h.end());
}

void place_rows(cudaStream_t s, const uint32_t* labels, int64_t n, const list_layout& layout,
                const std::vector<int64_t>& base_fill, int64_t* dst_rows)
{
  if (n == 0) return;
  dbuf<uint32_t> sorted(static_cast<size_t>(n), s), order;
  B2_CUDA(cudaMemcpyAsync(sorted.data(), labels, sizeof(uint32_t) * n, cudaMemcpyDeviceToDevice, s));
  iota_u32(s, order, n);
  dbuf<int64_t> start;
  group_by_key(s, sorted, order, layout.n_lists, start);
  dbuf<int64_t> fill(static_cast<size_t>(layout.n_lists), s);
  B2_CUDA(cudaMemcpyAsync(fill.data(), base_fill.data(), sizeof(int64_t) * layout.n_lists, cudaMemcpyHostToDevice, s));
  count_launch();
  place_rows_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, s>>>(sorted.data(), order.data(), n, start.data(),
                                                                             layout.d_offsets.data(), fill.data(), dst_rows);
  B2_CUDA(cudaGetLastError());
  B2_CUDA(cudaStreamSynchronize(s));  // base_fill is a host vector owned by the caller
}

template <typename T>
void alloc_padded(cudaStream_t s, int64_t rows, int row_elems, owned<T>& payload, owned<int64_t>& ids)
{
  payload.alloc(static_cast<size_t>(std::max<int64_t>(rows, 1)) * row_elems);
  ids.alloc(static_cast<size_t>(std::max<int64_t>(rows, 1)));
  B2_CUDA(cudaMemsetAsync(payload.data(), 0, sizeof(T) * static_cast<size_t>(rows) * row_elems, s));
  if (rows == 0) return;
  count_launch();
  fill_pad_ids_kernel<<<blocks_for(rows, 256), 256, 0, s>>>(ids.data(), rows);
  B2_CUDA(cudaGetLastError());
}
template void alloc_padded<float>(cudaStream_t, int64_t, int, owned<float>&, owned<int64_t>&);
template void alloc_padded<uint8_t>(cudaStream_t, int64_t, int, owned<uint8_t>&, owned<int64_t>&);

void remap_rows(cudaStream_t s, const list_layout& from, const list_layout& to, int64_t* dst_rows)
{
  count_launch();
  remap_rows_kernel<<<static_cast<unsigned>(from.n_lists), 128, 0, s>>>(from.d_offsets.data(), from.d_sizes.data(),
                                                                         to.d_offsets.data(), dst_rows);
  B2_CUDA(cudaGetLastError());
}

template <typename T>
void scatter_rows(cudaStream_t s, const T* src, int64_t rows, int row_elems, const int64_t* dst_rows, T* dst)
{
  count_launch();
  scatter_rows_kernel<T><<<blocks_for(rows * row_elems, 256), 256, 0, s>>>(src, rows, row_elems, dst_rows, dst);
  B2_CUDA(cudaGetLastError());
}
template void scatter_rows<float>(cudaStream_t, const float*, int64_t, int, const int64_t*, float*);
template void scatter_rows<uint8_t>(cudaStream_t, const uint8_t*, int64_t, int, const int64_t*, uint8_t*);
template void scatter_rows<int64_t>(cudaStream_t, const int64_t*, int64_t, int, const int64_t*, int64_t*);

void store_ids(cudaStream_t s, const int64_t* dst_rows, int64_t n, const int64_t* new_ids, int64_t id0, int64_t* ids)
{
  count_launch();
  store_ids_kernel<<<blocks_for(n, 256), 256, 0, s>>>(dst_rows, n, new_ids, id0, ids);
  B2_CUDA(cudaGetLastError());
}

}  // namespace b200
