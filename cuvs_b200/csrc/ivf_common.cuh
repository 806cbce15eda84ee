// Building blocks shared by IVF-Flat, IVF-PQ and k-means (host API).
//
// Reference counterparts:
//   coarse search        cpp/src/neighbors/ivf_pq/ivf_pq_search.cuh:60-168, ivf_flat/ivf_flat_search.cuh:105-187
//   probe bookkeeping    cpp/src/neighbors/ivf_common.cuh:49-169 (chunk indices, sample -> id translation)
//   balanced k-means     cpp/src/cluster/detail/kmeans_balanced.cuh:76-1100 (EM + re-seeding of small clusters)
//   assignment step      cpp/src/cluster/detail/minClusterDistanceCompute.cu:18-165
//
// B200 formulation: instead of one CTA per (query, probe) that re-reads the probed list for every
// query (reference a8/a11), (query, probe) pairs are bucketed BY LIST on the device; each work item is
// "<= 128 queries that probe list l" x "the 128-row tiles of list l", which is a dense contraction the
// tcgen05 scan kernel (scan_tc.cu) executes with a fused top-k' epilogue.  List rows are read once per
// 128 probing queries instead of once per query.
#pragma once
#include "common.hpp"
#include "scan_tc.cuh"

#include <cuda_bf16.h>

namespace b200 {

/** bf16 split planes + half-norms of a set of row vectors, padded to 128-row tiles (the "B side"). */
struct tc_rows {
  int64_t n = 0, rows_pad = 0;
  int d = 0, Kp = 0;
  owned<__nv_bfloat16> hi, lo;
  owned<__nv_bfloat16> hx;  // [rows_pad, 16] half-norm plane
  void build(cudaStream_t s, const float* x, int64_t n_, int d_, const float* xn /*|x|^2 or null => hn = 0*/, bool with_lo,
             const float* row_scale = nullptr);
};

/** Temporary (stream-ordered) version of the above for query-side operands. */
struct tc_rows_tmp {
  int64_t n = 0, rows_pad = 0;
  int d = 0, Kp = 0;
  dbuf<__nv_bfloat16> hi, lo;
  void build(cudaStream_t s, const float* x, int64_t n_, int d_, bool with_lo, int64_t extra_pad_rows = 0,
             const float* row_scale = nullptr);
};

/**
 * Top-`n_probes` rows of `centers` for every query (smallest s = hn - q.c first): dense tcgen05 score
 * block + select_k.  probes: [nq, n_probes] uint32 (0xffffffff padding when n_probes > n_centers).
 */
void coarse_select(resources* res, const tc_rows_tmp& queries, const tc_rows& centers, int n_probes, uint32_t* probes,
                   float* probe_scores /*nullable*/);

/** labels[i] = argmin_j (hn[j] - x_i . c_j)  (nearest centre, approx = fp32-grade split products); optional score out. */
void assign_nearest(resources* res, const __nv_bfloat16* x_hi, const __nv_bfloat16* x_lo, int64_t n, int64_t x_rows_pad,
                    int Kp, const tc_rows& centers, uint32_t* labels, float* scores /*nullable*/);

/**
 * (query, probe) pairs bucketed by list, on the device.
 *   slot_of[q * n_probes + p]  -> row of the pair in list-major order (0xffffffff for padded probes)
 *   pair_query[slot]           -> query id
 *   items / n_items            -> work list for tc_scan_topk (A rows = slots, B rows = list ranges)
 */
struct probe_buckets {
  dbuf<uint32_t> slot_of, pair_query, pair_list;
  dbuf<tc_item> items;
  dbuf<int> n_items;   // device: [0] = number of work items, [1] = number of live pairs (slots in use)
  int max_items = 0;   // host upper bound
  int64_t n_pairs = 0;
};
void bucket_probes(resources* res, const uint32_t* probes, int64_t nq, int n_probes, int64_t n_lists,
                   const int64_t* list_offsets_dev /*[n_lists+1], padded row offsets (multiples of 128)*/, int KC,
                   probe_buckets& out, int probe_ld = 0 /*row stride of `probes` (0: n_probes)*/,
                   uint32_t max_tiles = 0xffffffffu /*scan at most this many tiles of each list (bound warm-up)*/,
                   int group = 128 /*pairs (A rows) per work item*/);

/** Gather bf16 rows: dst[slot] = src[pair_query[slot]] (Kp elements each); rows >= *n_live are zeroed up to rows_total. */
void gather_rows_bf16(cudaStream_t s, const __nv_bfloat16* src, const uint32_t* pair_query, const int* n_live, int64_t rows_total,
                      int Kp, __nv_bfloat16* dst);

/** Per query, concatenate the KC candidates of each of its probes: out [nq, n_probes*KC]. */
void gather_probe_candidates(cudaStream_t s, const float* cs, const uint32_t* cp, const uint32_t* slot_of, int64_t nq,
                             int n_probes, int KC, float* out_score, uint32_t* out_pos);

/**
 * Per query: the k best (value, position) among its probes' candidates, value = add[slot] + scale * score, sorted
 * ascending (ties: smaller position), missing entries (FLT_MAX, 0xffffffff).  `bound_keys` [nq] is the scan's tc_bound
 * state — an upper bound on each query's k-th best value in the same units (null: no bound).  Returns false (nothing
 * launched) when the shape needs the generic gather + select_k path instead.
 */
bool merge_probe_candidates(cudaStream_t s, const float* cs, const uint32_t* cp, const uint32_t* slot_of, const float* add,
                            float scale, const int* bound_keys, int64_t nq, int n_probes, int KCW, int k, float* out_val,
                            uint32_t* out_pos);

/**
 * Balanced-ish Lloyd k-means on the device (fp32 data, tcgen05 assignment).  `centers` [k, d] is
 * initialised from evenly strided rows when `init_from_data`, then refined for `n_iters` iterations;
 * clusters smaller than 1/4 of the average are re-seeded from members of large clusters each iteration.
 * Returns inertia of the final assignment when `inertia` != null (approximate scores).
 */
void kmeans_train(resources* res, const float* x, int64_t n, int d, int k, int n_iters, float* centers,
                  bool init_from_data, bool balance, double* inertia, int* iters_done, double tol = 0.0);

/** Sum of member rows and member counts per label (in row order: deterministic), then centers = sums / counts where counts > 0. */
void update_centers(cudaStream_t s, const float* x, int64_t n, int d, const uint32_t* labels, const float* weights,
                    int k, float* centers, float* sums_ws /*[k*d]*/, float* counts_ws /*[k]*/);

}  // namespace b200
