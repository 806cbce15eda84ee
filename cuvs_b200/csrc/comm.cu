// NCCL plumbing for the list-sharded searches + the one exchange step of the multi-GPU path:
// all-gather of the packed partial top-k, k-way merge on every rank, everything on the handle's stream.
//
// Reference being replaced: cpp/src/neighbors/mg/snmg.cuh:248-375 (row-sharded; the root collects the partials with
// ncclSend/ncclRecv inside an OpenMP region, merges with knn_merge_parts and returns through the host).
// Here (BASELINE.json north_star): the index is sharded by IVF LIST, every rank holds the same query batch, and the only
// collective is ONE ncclAllGather of [nq*k f32 | nq*k i64] per rank (1.2 MB at nq = 10k, k = 10) enqueued on the same
// stream as the scan — no host synchronisation between the shard's search and the merge.
//
// libnccl.so.2 is dlopen'ed on first use (inside a Python process that already imported torch the loader hands back
// torch's bundled NCCL; a plain C client gets the system one): libcuvs_c.so itself has no link-time NCCL dependency.
#include "comm.cuh"
#include "common.hpp"
#include "select_k.cuh"
#include "timing.hpp"

#include <cuvs_b200/ext.h>

#include <dlfcn.h>
#include <nccl.h>

#include <memory>
#include <mutex>
#include <vector>

namespace b200 {

struct nccl_api {
  decltype(&ncclGetUniqueId) get_unique_id = nullptr;
  decltype(&ncclCommInitRank) comm_init_rank = nullptr;
  decltype(&ncclCommInitAll) comm_init_all = nullptr;
  decltype(&ncclCommDestroy) comm_destroy = nullptr;
  decltype(&ncclAllGather) all_gather = nullptr;
  decltype(&ncclGroupStart) group_start = nullptr;
  decltype(&ncclGroupEnd) group_end = nullptr;
  decltype(&ncclGetErrorString) error_string = nullptr;
};

const nccl_api& nccl()
{
  static nccl_api api;
  static std::once_flag once;
  std::call_once(once, [] {
    void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
    if (!h) return;
    api.get_unique_id  = reinterpret_cast<decltype(api.get_unique_id)>(dlsym(h, "ncclGetUniqueId"));
    api.comm_init_rank = reinterpret_cast<decltype(api.comm_init_rank)>(dlsym(h, "ncclCommInitRank"));
    api.comm_init_all  = reinterpret_cast<decltype(api.comm_init_all)>(dlsym(h, "ncclCommInitAll"));
    api.comm_destroy   = reinterpret_cast<decltype(api.comm_destroy)>(dlsym(h, "ncclCommDestroy"));
    api.all_gather     = reinterpret_cast<decltype(api.all_gather)>(dlsym(h, "ncclAllGather"));
    api.group_start    = reinterpret_cast<decltype(api.group_start)>(dlsym(h, "ncclGroupStart"));
    api.group_end      = reinterpret_cast<decltype(api.group_end)>(dlsym(h, "ncclGroupEnd"));
    api.error_string   = reinterpret_cast<decltype(api.error_string)>(dlsym(h, "ncclGetErrorString"));
  });
  B2_EXPECTS(api.all_gather != nullptr && api.comm_init_rank != nullptr, "NCCL (libnccl.so.2) could not be loaded: %s", dlerror());
  return api;
}

#define B2_NCCL(call)                                                                                                  \
  do {                                                                                                                 \
    ncclResult_t r_ = (call);                                                                                          \
    if (r_ != ncclSuccess) B2_FAIL("NCCL error %d (%s) at %s:%d", int(r_), nccl().error_string ? nccl().error_string(r_) : "?", __FILE__, __LINE__); \
  } while (0)

namespace {

// per-rank payload: nq*k distances (f32), padded to 8 bytes, then nq*k ids (i64)
inline size_t packed_bytes(int64_t nq, int k) { return ((static_cast<size_t>(nq) * k * 4 + 7) & ~size_t(7)) + static_cast<size_t>(nq) * k * 8; }

__global__ void pack_partial_kernel(const float* __restrict__ d, const int64_t* __restrict__ i, int64_t count, uint8_t* __restrict__ out)
{
  const int64_t t = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  if (t >= count) return;
  reinterpret_cast<float*>(out)[t] = d[t];
  reinterpret_cast<int64_t*>(out + ((count * 4 + 7) & ~int64_t(7)))[t] = i[t];
}

// [world][packed] -> part-major keys / vals ([world * nq, k]): what knn_merge_parts takes
__global__ void unpack_parts_kernel(const uint8_t* __restrict__ in, int64_t count, int world, size_t stride, float* __restrict__ keys,
                                    int64_t* __restrict__ vals)
{
  const int64_t t = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  if (t >= count * world) return;
  const int w = static_cast<int>(t / count);
  const int64_t e = t - static_cast<int64_t>(w) * count;
  const uint8_t* p = in + static_cast<size_t>(w) * stride;
  keys[t] = reinterpret_cast<const float*>(p)[e];
  vals[t] = reinterpret_cast<const int64_t*>(p + ((count * 4 + 7) & ~int64_t(7)))[e];
}

}  // namespace

/** One NCCL communicator per participating device of THIS process (1 for the process-per-GPU mode). */
struct comm_group {
  std::vector<ncclComm_t> comms;
  std::vector<int> devices;
  int world = 1;
  int rank0 = 0;  // rank of comms[0]
  ~comm_group()
  {
    for (auto c : comms)
      if (c && nccl().comm_destroy) nccl().comm_destroy(c);
  }
};

/** Packed all-gather + merge for ONE local device (comm index `ci`), enqueued on `s`.  d / i: this rank's partial [nq, k]. */
void allgather_merge_topk(comm_group& g, int ci, cudaStream_t s, const float* d, const int64_t* i, int64_t nq, int k, bool select_min,
                          float* out_d, int64_t* out_i, dbuf<uint8_t>& send, dbuf<uint8_t>& recv, bool in_group)
{
  const int64_t count = nq * k;
  const size_t bytes  = packed_bytes(nq, k);
  if (!in_group) {  // (inside an ncclGroup the caller packed already and unpacks after ncclGroupEnd)
    send.alloc(bytes, s);
    recv.alloc(bytes * g.world, s);
    count_launch();
    pack_partial_kernel<<<blocks_for(count, 256), 256, 0, s>>>(d, i, count, send.data());
  }
  B2_NCCL(nccl().all_gather(send.data(), recv.data(), bytes, ncclUint8, g.comms[ci], s));
  if (!in_group) {
    dbuf<float> keys(static_cast<size_t>(count) * g.world, s);
    dbuf<int64_t> vals(static_cast<size_t>(count) * g.world, s);
    count_launch();
    unpack_parts_kernel<<<blocks_for(count * g.world, 256), 256, 0, s>>>(recv.data(), count, g.world, bytes, keys.data(), vals.data());
    B2_CUDA(cudaGetLastError());
    knn_merge_parts(s, keys.data(), vals.data(), out_d, out_i, g.world, nq, k, nullptr, select_min);
  }
}

/** Single-process, multi-device exchange: every device's partial -> merged result on EVERY device (grouped all-gather). */
void allgather_merge_topk_all(comm_group& g, const std::vector<cudaStream_t>& streams, const std::vector<const float*>& d,
                              const std::vector<const int64_t*>& i, int64_t nq, int k, bool select_min, const std::vector<float*>& out_d,
                              const std::vector<int64_t*>& out_i, int only_output_device /*-1: all*/)
{
  const int nd        = static_cast<int>(g.comms.size());
  const int64_t count = nq * k;
  const size_t bytes  = packed_bytes(nq, k);
  std::vector<dbuf<uint8_t>> send(nd), recv(nd);
  int prev = 0;
  cudaGetDevice(&prev);
  for (int c = 0; c < nd; ++c) {
    B2_CUDA(cudaSetDevice(g.devices[c]));
    send[c].alloc(bytes, streams[c]);
    recv[c].alloc(bytes * g.world, streams[c]);
    count_launch();
    pack_partial_kernel<<<blocks_for(count, 256), 256, 0, streams[c]>>>(d[c], i[c], count, send[c].data());
  }
  B2_NCCL(nccl().group_start());
  for (int c = 0; c < nd; ++c) B2_NCCL(nccl().all_gather(send[c].data(), recv[c].data(), bytes, ncclUint8, g.comms[c], streams[c]));
  B2_NCCL(nccl().group_end());
  for (int c = 0; c < nd; ++c) {
    if (only_output_device >= 0 && c != only_output_device) continue;
    B2_CUDA(cudaSetDevice(g.devices[c]));
    dbuf<float> keys(static_cast<size_t>(count) * g.world, streams[c]);
    dbuf<int64_t> vals(static_cast<size_t>(count) * g.world, streams[c]);
    count_launch();
    unpack_parts_kernel<<<blocks_for(count * g.world, 256), 256, 0, streams[c]>>>(recv[c].data(), count, g.world, bytes, keys.data(), vals.data());
    B2_CUDA(cudaGetLastError());
    knn_merge_parts(streams[c], keys.data(), vals.data(), out_d[c], out_i[c], g.world, nq, k, nullptr, select_min);
  }
  for (int c = 0; c < nd; ++c) {  // stream-ordered frees belong to their device's pool
    cudaSetDevice(g.devices[c]);
    send[c].release();
    recv[c].release();
  }
  cudaSetDevice(prev);
}

void destroy_comm_group(comm_group* g) { delete g; }

/** ncclCommInitAll over the given devices of this process. */
comm_group* make_local_comm_group(const std::vector<int>& devices)
{
  auto g     = std::make_unique<comm_group>();
  g->devices = devices;
  g->world   = static_cast<int>(devices.size());
  g->comms.resize(devices.size(), nullptr);
  B2_NCCL(nccl().comm_init_all(g->comms.data(), g->world, devices.data()));
  return g.release();
}

}  // namespace b200

using namespace b200;

struct cuvsB200Comm {
  std::unique_ptr<comm_group> g;
};

extern "C" {

cuvsError_t cuvsB200NcclUniqueId(void* id128)
{
  return guarded([=] {
    B2_EXPECTS(id128 != nullptr, "id buffer is null");
    static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId is expected to be 128 bytes");
    ncclUniqueId id;
    B2_NCCL(nccl().get_unique_id(&id));
    memcpy(id128, &id, sizeof(id));
  });
}

cuvsError_t cuvsB200CommCreate(cuvsResources_t res, const void* id128, int rank, int world, cuvsB200Comm_t* comm)
{
  return guarded([=] {
    auto r = as_res(res);
    B2_EXPECTS(id128 != nullptr && comm != nullptr && world >= 1 && rank >= 0 && rank < world, "cuvsB200CommCreate: bad arguments");
    ncclUniqueId id;
    memcpy(&id, id128, sizeof(id));
    auto g     = std::make_unique<comm_group>();
    g->world   = world;
    g->rank0   = rank;
    g->devices = {r->device};
    g->comms.resize(1, nullptr);
    int prev = 0;
    cudaGetDevice(&prev);
    B2_CUDA(cudaSetDevice(r->device));
    B2_NCCL(nccl().comm_init_rank(&g->comms[0], world, id, rank));
    cudaSetDevice(prev);
    *comm = new cuvsB200Comm{std::move(g)};
  });
}

cuvsError_t cuvsB200CommDestroy(cuvsB200Comm_t comm)
{
  return guarded([=] { delete comm; });
}

cuvsError_t cuvsB200AllGatherMergeTopK(cuvsResources_t res, cuvsB200Comm_t comm, DLManagedTensor* distances, DLManagedTensor* neighbors,
                                       DLManagedTensor* out_distances, DLManagedTensor* out_neighbors, bool select_min)
{
  return guarded([=] {
    auto r = as_res(res);
    B2_EXPECTS(comm != nullptr && comm->g && comm->g->comms.size() == 1, "cuvsB200AllGatherMergeTopK needs a communicator from cuvsB200CommCreate");
    B2_EXPECTS(distances && neighbors && out_distances && out_neighbors, "null tensor");
    const DLTensor& d = distances->dl_tensor;
    const DLTensor& i = neighbors->dl_tensor;
    const DLTensor& od = out_distances->dl_tensor;
    const DLTensor& oi = out_neighbors->dl_tensor;
    B2_EXPECTS(dl_is(d, kDLFloat, 32) && dl_is(i, kDLInt, 64) && dl_is(od, kDLFloat, 32) && dl_is(oi, kDLInt, 64),
               "distances must be float32 and neighbors int64 (global ids)");
    B2_EXPECTS(d.ndim == 2 && i.ndim == 2 && d.shape[0] == i.shape[0] && d.shape[1] == i.shape[1] && od.shape[0] == d.shape[0] &&
                 od.shape[1] == d.shape[1] && oi.shape[0] == d.shape[0] && oi.shape[1] == d.shape[1],
               "partial and merged tensors must all be [n_queries, k]");
    B2_EXPECTS(dl_is_device(d) && dl_is_device(i) && dl_is_device(od) && dl_is_device(oi), "device tensors expected");
    B2_EXPECTS(dl_is_c_contiguous(d) && dl_is_c_contiguous(i) && dl_is_c_contiguous(od) && dl_is_c_contiguous(oi), "contiguous tensors expected");
    dbuf<uint8_t> send, recv;
    timed_section ts("allgather_merge", r->stream);
    allgather_merge_topk(*comm->g, 0, r->stream, dl_ptr<float>(d), dl_ptr<int64_t>(i), d.shape[0], static_cast<int>(d.shape[1]), select_min,
                         dl_ptr<float>(od), dl_ptr<int64_t>(oi), send, recv, false);
  });
}

}  // extern "C"
