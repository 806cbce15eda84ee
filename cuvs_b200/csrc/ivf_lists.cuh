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

}  // namespace b200
