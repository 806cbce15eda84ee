// List storage shared by IVF-Flat and IVF-PQ: rows grouped by list, every list padded to a whole
// number of 128-row tiles so that a (list, query-group) work item is tile aligned for the tcgen05 scan.
//
// The reference keeps one allocation per list with rows interleaved in groups of 32
// (cpp/include/cuvs/neighbors/ivf_flat.hpp:184-201, ivf_pq.hpp:235-296) because its scan kernel
// assigns one warp lane per row.  Here the scan is a dense tile contraction fed by TMA, so the natural
// layout is one flat K-major [rows, dim] array with lists back to back (B200: a list tile is a single
// 2-D TMA box; no per-list pointer table, no interleaving).
#pragma once
#include "common.hpp"

#include <algorithm>
#include <utility>
#include <vector>

namespace b200 {

/** id stored on the padding rows of a list (any other int64, negative ones included, is a user id). */
constexpr int64_t kPadId = INT64_MIN;

struct list_layout {
  int64_t n_lists = 0;
  std::vector<int64_t> h_sizes;    // rows per list
  std::vector<int64_t> h_offsets;  // padded start row of each list (n_lists + 1 entries, multiples of 128)
  owned<int64_t> d_offsets;
  owned<uint32_t> d_sizes;
  int64_t rows_total = 0;  // = h_offsets[n_lists]
  int64_t size       = 0;  // sum of sizes

  void set_sizes(cudaStream_t s, const std::vector<int64_t>& sizes);
};

/**
 * Computes, for rows with labels[i] (list id), a destination row inside `layout` such that rows of
 * a list are contiguous after `base_fill[l]` already-present rows: dst[i] = offsets[l] + base_fill[l] + rank.
 * Order inside a list follows the input order (stable).
 */
void place_rows(cudaStream_t s, const uint32_t* labels, int64_t n, const list_layout& layout,
                const std::vector<int64_t>& base_fill, int64_t* dst_rows);

/**
 * Deterministic grouping: sorts the pairs (keys[i], values[i]) stably by key, in place (on return both buffers hold the sorted
 * pairs; the stable order keeps the input order inside a key), and sets start[g] = the first position of key g
 * (n_groups + 1 entries, start[n_groups] = n).  Sums taken over a group in this order, or ranks taken inside it, do not
 * depend on thread scheduling, unlike atomics.  Transient device memory: 8 bytes per item (the radix sort's second key and
 * value buffers) + 8 bytes per group + CUB's small temporary storage.
 */
void group_by_key(cudaStream_t s, dbuf<uint32_t>& keys, dbuf<uint32_t>& values, int64_t n_groups, dbuf<int64_t>& start);
/** v = 0, 1, ..., n - 1 (n < 2^32: larger inputs are rejected). */
void iota_u32(cudaStream_t s, dbuf<uint32_t>& v, int64_t n);
/** counts[l] = number of rows with that label (host vector, synchronises the stream). */
std::vector<int64_t> count_labels(cudaStream_t s, const uint32_t* labels, int64_t n, int64_t n_lists);

/** Storage of empty padded lists of `rows` rows: payload [max(rows, 1) * row_elems] zeroed, ids [max(rows, 1)] = kPadId. */
template <typename T>
void alloc_padded(cudaStream_t s, int64_t rows, int row_elems, owned<T>& payload, owned<int64_t>& ids);
/** dst_rows[r] = row of `to` that row r of `from` moves to (same list, same rank in it), -1 on the padding rows of `from`. */
void remap_rows(cudaStream_t s, const list_layout& from, const list_layout& to, int64_t* dst_rows);
/** dst[dst_rows[r]] = src[r] for rows of row_elems elements; rows with dst_rows[r] < 0 are skipped. */
template <typename T>
void scatter_rows(cudaStream_t s, const T* src, int64_t rows, int row_elems, const int64_t* dst_rows, T* dst);
/** ids[dst_rows[i]] = new_ids ? new_ids[i] : id0 + i. */
void store_ids(cudaStream_t s, const int64_t* dst_rows, int64_t n, const int64_t* new_ids, int64_t id0, int64_t* ids);

/** fn(x, rows, r0) on the rows of the float tensor `t` [n, d] in device-resident chunks of at most 512 MiB; host rows are
 *  staged through one reused buffer. */
template <typename Fn>
void for_device_chunks(resources* res, const DLTensor& t, int d, Fn&& fn)
{
  const int64_t n     = t.shape[0];
  const float* p      = dl_ptr<float>(t);
  const int64_t chunk = std::max<int64_t>(1, (int64_t(1) << 27) / std::max(d, 1));
  const bool dev      = dl_is_device(t) && t.device.device_type != kDLCUDAHost;
  dbuf<float> buf;
  if (!dev) buf.alloc(static_cast<size_t>(std::min(n, chunk)) * d, res->stream);
  for (int64_t r0 = 0; r0 < n; r0 += chunk) {
    const int64_t rows = std::min(chunk, n - r0);
    if (dev) fn(p + r0 * d, rows, r0);
    else {
      B2_CUDA(cudaMemcpyAsync(buf.data(), p + r0 * d, sizeof(float) * rows * d, cudaMemcpyHostToDevice, res->stream));
      fn(buf.data(), rows, r0);
    }
  }
}

/**
 * Inserts the n >= 1 rows of `t` [n, d] (host or device) into the padded lists `lists` whose rows are `payload` (row_elems
 * elements each) and `ids`; row i gets the id new_ids[i] (device) or id0 + i.  Two passes over the chunks of `t`, so the
 * lists are laid out once per insertion:
 *   1. label(x, rows, labels) writes the list of every row of a chunk;
 *   2. after the old rows have moved to the new layout, write(x, rows, labels, dst_rows, new_payload) stores the rows of a
 *      chunk at dst_rows, behind the rows already in each list, in input order.
 * The padding rows of the new storage are zero, with id kPadId.
 */
template <typename T, typename Label, typename Write>
void insert_rows(resources* res, list_layout& lists, owned<T>& payload, int row_elems, owned<int64_t>& ids, const DLTensor& t,
                 int d, const int64_t* new_ids, int64_t id0, Label&& label, Write&& write)
{
  auto s          = res->stream;
  const int64_t n = t.shape[0];
  dbuf<uint32_t> labels(static_cast<size_t>(n), s);
  std::vector<int64_t> sizes = lists.h_sizes;
  std::vector<std::vector<int64_t>> chunk_add;
  for_device_chunks(res, t, d, [&](const float* x, int64_t rows, int64_t r0) {
    label(x, rows, labels.data() + r0);
    chunk_add.push_back(count_labels(s, labels.data() + r0, rows, lists.n_lists));
    for (int64_t l = 0; l < lists.n_lists; ++l) sizes[l] += chunk_add.back()[l];
  });
  list_layout nl;
  nl.set_sizes(s, sizes);
  owned<T> npayload;
  owned<int64_t> nids;
  alloc_padded(s, nl.rows_total, row_elems, npayload, nids);
  if (lists.rows_total > 0) {
    dbuf<int64_t> dst_old(static_cast<size_t>(lists.rows_total), s);
    remap_rows(s, lists, nl, dst_old.data());
    scatter_rows(s, payload.data(), lists.rows_total, row_elems, dst_old.data(), npayload.data());
    scatter_rows(s, ids.data(), lists.rows_total, 1, dst_old.data(), nids.data());
  }
  std::vector<int64_t> fill = lists.h_sizes;  // rows already placed in each list
  size_t ci = 0;
  for_device_chunks(res, t, d, [&](const float* x, int64_t rows, int64_t r0) {
    dbuf<int64_t> dst_new(static_cast<size_t>(rows), s);
    place_rows(s, labels.data() + r0, rows, nl, fill, dst_new.data());
    for (int64_t l = 0; l < lists.n_lists; ++l) fill[l] += chunk_add[ci][l];
    ++ci;
    write(x, rows, labels.data() + r0, dst_new.data(), npayload.data());
    store_ids(s, dst_new.data(), rows, new_ids ? new_ids + r0 : nullptr, id0 + r0, nids.data());
  });
  B2_CUDA(cudaStreamSynchronize(s));
  payload = std::move(npayload);
  ids     = std::move(nids);
  lists   = std::move(nl);
}

}  // namespace b200
