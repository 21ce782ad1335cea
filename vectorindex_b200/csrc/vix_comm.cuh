// vix_comm.cuh -- the communicator of the multi-GPU entry points (vix_comm_t) and the exchange steps that the list-sharded
// layout (vix_sharded.cu) and the replicated one (vix_replicated.cu) share.
#pragma once

#include "vix_index.cuh"
#include "vix_range.cuh"

#include <nccl.h>

#include <mutex>
#include <vector>

namespace vix {

// ------------------------------------------------------------------------------------------------ NCCL binding
struct NcclApi {
    void* lib = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Send)(const void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Recv)(void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*GroupStart)() = nullptr;
    ncclResult_t (*GroupEnd)() = nullptr;
    const char* (*GetErrorString)(ncclResult_t) = nullptr;
};

extern NcclApi g_nccl;
int nccl_load();

#define VIX_NCCL(expr)                                                                                  \
    do {                                                                                                \
        ncclResult_t _r = (expr);                                                                       \
        if (_r != ncclSuccess) {                                                                        \
            ::vix::set_error("NCCL error %d (%s): %s", (int)_r, ::vix::g_nccl.GetErrorString(_r), #expr); \
            return VIX_ERR_CUDA;                                                                        \
        }                                                                                               \
    } while (0)

}  // namespace vix

// ------------------------------------------------------------------------------------------------ communicator
struct vix_comm {
    ncclComm_t comm = nullptr;
    int rank = 0, world = 1, device = 0;
    std::mutex mu;
    // exchange memory: one region per rank, every region mapped into every rank (cudaIpc).  Same layout everywhere:
    //   [flags: one word per peer, then (from kStatusOffset) one status word per rank][queries: world x per x d f32]
    //   [probes: world x per x nprobe i32][results: world x nq x k u64]
    //   [bounds: nq f32 -- the list-major scan's per-query bounds the OTHER ranks found; all bits set (a NaN) = none]
    int peer_state = -1;                    // -1 undecided, 0 NCCL all-gathers, 1 peer memory
    void* local = nullptr;
    size_t local_bytes = 0;
    std::vector<void*> peer;                // base of every rank's region in THIS process (peer[rank] == local)
    void** peer_dev = nullptr;              // device copy
    uint32_t epoch = 0;                     // barriers passed so far
    size_t off_queries = 0, off_probes = 0, off_results = 0, off_bounds = 0;
    int64_t cap_nq = 0, cap_per = 0;
    int cap_d = 0, cap_nprobe = 0, cap_k = 0;
    // NCCL path: plain local buffers with the same roles
    void* gather_probes = nullptr; size_t gather_probes_bytes = 0;
    void* gather_keys = nullptr; size_t gather_keys_bytes = 0;
    // range search (and k-NN search beyond VIX_MAX_K): a second region, mapped like the first (peer memory only), grown
    // collectively and geometrically:
    //   [lims: world x (nq + 2) i64 -- each rank's local CSR row starts + its status]
    //   [bounds: world x nq u32 -- each rank's k-NN seed bounds; apart from the lims, which a fast peer may already store
    //    while this rank still reads the bounds]
    //   [keys: the global answer's sorted keys, rank by rank]
    void* range_local = nullptr;
    std::vector<void*> range_peer;
    void** range_peer_dev = nullptr;
    size_t range_off_bounds = 0, range_off_keys = 0;
    int64_t range_cap_nq = 0, range_cap_keys = 0;
    // optional phase events of the last search (vix_comm_trace): start | probes exchanged | scanned | merged
    bool trace = false;
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
};

namespace vix {

constexpr size_t kFlagBytes = 4096;         // flags[world] (u32) and the status words, padded
constexpr size_t kStatusOffset = 2048;      // status[world] (i32): the replicated calls' per-rank status of a k-NN step

// rows of the batch whose probe lists (sharded) / answer (replicated) a rank computes: blocks of `per` rows (a multiple of
// 4, so that every block of queries / probes is a whole number of 16-byte pieces)
inline int64_t block_rows(int64_t nq, int world) {
    int64_t per = (nq + world - 1) / world;
    return (per + 3) & ~(int64_t)3;
}

// Collective: make every rank's region large enough for (nq, d, nprobe, k) and map it everywhere; decides c->peer_state.
int ensure_region(vix_comm* c, int64_t nq, int d, int nprobe, int k);
// Collective (peer memory only): the range region holds nq rows of lims and `keys` keys (*grown: it was reallocated).
int ensure_range_region(vix_comm* c, int64_t nq, int64_t keys, bool* grown);
// Barrier across the ranks on the stream (peer memory): every store into the peers enqueued before it is visible after it.
int peer_barrier(vix_comm* c);
// lims_all [world][nq + 2] -> glims [nq + 1] (device), meta (host: key bases [world + 1], longest row, statuses [world]);
// synchronises the stream
int shard_range_lims(const int64_t* lims_all, int world, int64_t nq, int64_t* glims, std::vector<int64_t>& meta);
int knn_neg_zero(const vix_index* h);
int range_neg_zero(const vix_index* h);
const char* kind_name(const vix_index* h);
int stage_filter(const uint64_t* words, int64_t capacity, int mode, In<uint64_t>& staged, FilterArgs& f, const FilterArgs*& fp);

// The last step of sharded_range_exchange: range search decodes the merged rows into a new result object (*out); k-NN
// search beyond VIX_MAX_K (out == nullptr) cuts them at k into [nq x k] (dist, ids: device), after checking on the exchanged
// row starts that no row whose bound is finite came out shorter than k.
// neg_zero: the kind's zero sign (knn_neg_zero / range_neg_zero); flat_metric >= 0: the flat kind's k-NN keys (score word,
// user id), merged by shard_flat_merge with that metric's mapping.  concat: the replicated layout's range search -- every
// row comes from one rank, so the keys rank by rank are already the global rows (replica_range_concat).
struct ShardTail {
    vix_range_result** out = nullptr;
    int k = 0;
    const uint32_t* bound = nullptr;
    float* dist = nullptr;
    int64_t* ids = nullptr;
    int neg_zero = 0;
    int flat_metric = -1;
    bool concat = false;
};
// what the exchange reports for the VIX_SCAN_DEBUG lines: this rank's entries, the merged entries, the longest merged row
struct ShardTotals { int64_t mine = 0, total = 0, max_row = 0; bool grown = false; };

// The step after each rank's local pass: its sorted keys and lims [nq + 1] over the whole batch (rc: its status) -> every
// rank's lims and status -> global row starts and total (synchronises) -> the keys of every rank -> the tail's last step.
int sharded_range_exchange(vix_index* h, vix_comm* c, int64_t nq, int rc, RangeKeys& rk, bool grown, const ShardTail& t,
                           ShardTotals* st);

// vix_replicated.cu: the global CSR of the replicated range search from the ranks' keys, concatenated rank by rank (glims:
// the global row starts), decoded into r
int replica_range_concat(const u64* keys, const int64_t* glims, int64_t nq, int64_t total, int neg_zero, vix_range_result* r);

}  // namespace vix
