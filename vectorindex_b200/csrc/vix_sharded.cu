// vix_sharded.cu -- the multi-GPU steps of the search path behind the C ABI: one process per GPU, one vix_comm_t per
// process (NCCL communicator + peer-mapped exchange memory), inverted lists partitioned over the ranks in contiguous
// list-id blocks (lists are disjoint, IVFIndex.swift:370-375; top-k of a union = mergeTopK of the parts,
// TopKMerge.swift:11-61).
//
//   vix_sharded_search   every rank: probe selection for ITS block of the batch against ALL centroids (the single-GPU
//                        code path, so the probe lists equal the single-GPU ones by construction) -> the block is
//                        STORED into every peer's memory over NVLink by the producing rank (the all-gather is a store
//                        pattern + one barrier kernel) -> fused scan over the probed lists this rank owns -> local top-k
//                        packed as 8-byte keys and stored into every peer -> barrier -> k smallest keys per query.
//                        Host queries: only the rank's own block crosses PCIe, it travels to the peers with the probes.
//                        No host synchronisation inside a step; NCCL all-gathers carry the two exchanges when the ranks
//                        cannot map each other's memory (decided once, by all ranks together).
//   vix_sharded_add      assign + encode the rows this rank was handed, route every row to the rank owning its list
//                        (counts all-gathered, rows with grouped ncclSend / ncclRecv), append there already encoded.
//
// NCCL is bound at run time (dlopen of libnccl.so.2: inside a PyTorch process that is the copy torch already loaded),
// so the library itself has no link-time dependency on it and single-GPU hosts never touch it.
#include "vix_index.cuh"
#include "vix_scan.cuh"
#include "vix_topk.cuh"

#include <cub/cub.cuh>

#include <dlfcn.h>
#include <nccl.h>
#include <stdlib.h>
#include <string.h>

#include <new>
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

static NcclApi g_nccl;
static std::mutex g_nccl_mu;

static int nccl_load() {
    std::lock_guard<std::mutex> lk(g_nccl_mu);
    if (g_nccl.lib) return VIX_OK;
    const char* env = getenv("VIX_NCCL_PATH");
    const char* names[] = {env, "libnccl.so.2", "libnccl.so"};
    void* lib = nullptr;
    for (const char* n : names) {
        if (!n || !*n) continue;
        lib = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
        if (lib) break;
    }
    VIX_REQUIRE(lib, VIX_ERR_UNSUPPORTED, "multi-GPU entry points need NCCL: libnccl.so.2 could not be loaded (%s); set VIX_NCCL_PATH",
                dlerror());
    NcclApi a;
    a.lib = lib;
#define VIX_SYM(field, name)                                                                          \
    a.field = reinterpret_cast<decltype(a.field)>(dlsym(lib, name));                                    \
    VIX_REQUIRE(a.field, VIX_ERR_UNSUPPORTED, "libnccl does not export %s", name)
    VIX_SYM(GetUniqueId, "ncclGetUniqueId");
    VIX_SYM(CommInitRank, "ncclCommInitRank");
    VIX_SYM(CommDestroy, "ncclCommDestroy");
    VIX_SYM(AllGather, "ncclAllGather");
    VIX_SYM(AllReduce, "ncclAllReduce");
    VIX_SYM(Send, "ncclSend");
    VIX_SYM(Recv, "ncclRecv");
    VIX_SYM(GroupStart, "ncclGroupStart");
    VIX_SYM(GroupEnd, "ncclGroupEnd");
    VIX_SYM(GetErrorString, "ncclGetErrorString");
#undef VIX_SYM
    g_nccl = a;
    return VIX_OK;
}

#define VIX_NCCL(expr)                                                                                  \
    do {                                                                                                \
        ncclResult_t _r = (expr);                                                                       \
        if (_r != ncclSuccess) {                                                                        \
            ::vix::set_error("NCCL error %d (%s): %s", (int)_r, g_nccl.GetErrorString(_r), #expr);     \
            return VIX_ERR_CUDA;                                                                        \
        }                                                                                               \
    } while (0)

}  // namespace vix

using namespace vix;

// ------------------------------------------------------------------------------------------------ communicator
struct vix_comm {
    ncclComm_t comm = nullptr;
    int rank = 0, world = 1, device = 0;
    std::mutex mu;
    // exchange memory: one region per rank, every region mapped into every rank (cudaIpc).  Same layout everywhere:
    //   [flags: one word per peer][queries: world x per x d f32][probes: world x per x nprobe i32][results: world x nq x k u64]
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
    // optional phase events of the last search (vix_comm_trace): start | probes exchanged | scanned | merged
    bool trace = false;
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
};

namespace vix {

constexpr size_t kFlagBytes = 4096;         // flags[world] (u32), padded

static void close_peers(vix_comm* c) {
    for (int p = 0; p < (int)c->peer.size(); ++p)
        if (p != c->rank && c->peer[p]) cudaIpcCloseMemHandle(c->peer[p]);
    c->peer.clear();
    if (c->local) cudaFree(c->local);
    c->local = nullptr;
    c->local_bytes = 0;
    if (c->peer_dev) cudaFree(c->peer_dev);
    c->peer_dev = nullptr;
}

// rows of the batch whose probe lists a rank computes: blocks of `per` rows (a multiple of 4, so that every block of
// queries / probes is a whole number of 16-byte pieces)
static int64_t block_rows(int64_t nq, int world) {
    int64_t per = (nq + world - 1) / world;
    return (per + 3) & ~(int64_t)3;
}

// Collective: make every rank's region large enough for (nq, d, nprobe, k) and map it everywhere.  All ranks call this
// with the same arguments, so they agree on whether to reallocate.  Returns with c->peer_state decided.
static int ensure_region(vix_comm* c, int64_t nq, int d, int nprobe, int k) {
    if (c->peer_state == 0) return VIX_OK;
    if (c->peer_state == 1 && nq <= c->cap_nq && d <= c->cap_d && nprobe <= c->cap_nprobe && k <= c->cap_k) return VIX_OK;
    cudaStream_t s = ctx().stream;
    const int world = c->world;
    // capacity grows geometrically in the batch size
    int64_t cnq = c->cap_nq > 0 ? c->cap_nq : 1024;
    while (cnq < nq) cnq *= 2;
    const int cd = d > c->cap_d ? d : c->cap_d, cp = nprobe > c->cap_nprobe ? nprobe : c->cap_nprobe, ck = k > c->cap_k ? k : c->cap_k;
    const int64_t per = block_rows(cnq, world);
    const size_t off_q = kFlagBytes;
    const size_t off_p = off_q + (size_t)world * per * cd * 4;
    const size_t off_r = (off_p + (size_t)world * per * cp * 4 + 255) & ~(size_t)255;
    const size_t off_b = (off_r + (size_t)world * cnq * ck * 8 + 255) & ~(size_t)255;
    const size_t total = off_b + (size_t)cnq * 4;
    VIX_CUDA(cudaStreamSynchronize(s));                                   // nothing of mine still writes into a peer
    void* fresh = nullptr;
    int ok = 1;
    if (getenv("VIX_NO_P2P")) ok = 0;
    cudaIpcMemHandle_t mine;
    memset(&mine, 0, sizeof(mine));
    if (ok && cudaMalloc(&fresh, total) != cudaSuccess) { cudaGetLastError(); ok = 0; fresh = nullptr; }
    if (ok && cudaMemsetAsync(fresh, 0, kFlagBytes, s) != cudaSuccess) { cudaGetLastError(); ok = 0; }
    if (ok && cudaMemsetAsync(static_cast<char*>(fresh) + off_b, 0xFF, (size_t)cnq * 4, s) != cudaSuccess) { cudaGetLastError(); ok = 0; }
    if (ok && cudaIpcGetMemHandle(&mine, fresh) != cudaSuccess) { cudaGetLastError(); ok = 0; }
    // all-gather of (ok, handle): also the barrier behind which the old regions may go
    struct Msg { int ok; int pad; cudaIpcMemHandle_t h; };
    Scratch<Msg> dmsg;
    VIX_TRY(dmsg.alloc((size_t)world + 1));
    Msg m;
    memset(&m, 0, sizeof(m));
    m.ok = ok; m.h = mine;
    VIX_CUDA(cudaMemcpyAsync(dmsg.ptr + world, &m, sizeof(Msg), cudaMemcpyHostToDevice, s));
    VIX_NCCL(g_nccl.AllGather(dmsg.ptr + world, dmsg.ptr, sizeof(Msg), ncclUint8, c->comm, s));
    std::vector<Msg> all((size_t)world);
    VIX_CUDA(cudaMemcpyAsync(all.data(), dmsg.ptr, sizeof(Msg) * world, cudaMemcpyDeviceToHost, s));
    VIX_CUDA(cudaStreamSynchronize(s));
    close_peers(c);                                                       // every rank has drained its stream
    int all_ok = 1;
    for (int p = 0; p < world; ++p) all_ok &= all[p].ok;
    std::vector<void*> peer((size_t)world, nullptr);
    if (all_ok) {
        for (int p = 0; p < world && all_ok; ++p) {
            if (p == c->rank) { peer[p] = fresh; continue; }
            if (cudaIpcOpenMemHandle(&peer[p], all[p].h, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) {
                cudaGetLastError();
                peer[p] = nullptr;
                all_ok = 0;
            }
        }
    }
    // a rank that could not map a peer tells the others: one more (tiny) all-reduce, MIN
    Scratch<int> dflag;
    VIX_TRY(dflag.alloc(1));
    VIX_CUDA(cudaMemcpyAsync(dflag.ptr, &all_ok, 4, cudaMemcpyHostToDevice, s));
    VIX_NCCL(g_nccl.AllReduce(dflag.ptr, dflag.ptr, 1, ncclInt32, ncclMin, c->comm, s));
    VIX_CUDA(cudaMemcpyAsync(&all_ok, dflag.ptr, 4, cudaMemcpyDeviceToHost, s));
    VIX_CUDA(cudaStreamSynchronize(s));
    if (!all_ok) {
        for (int p = 0; p < world; ++p)
            if (p != c->rank && peer[p]) cudaIpcCloseMemHandle(peer[p]);
        if (fresh) cudaFree(fresh);
        c->peer_state = 0;
        return VIX_OK;
    }
    c->local = fresh; c->local_bytes = total; c->peer = peer;
    VIX_CUDA(cudaMalloc(reinterpret_cast<void**>(&c->peer_dev), sizeof(void*) * world));
    VIX_CUDA(cudaMemcpyAsync(c->peer_dev, peer.data(), sizeof(void*) * world, cudaMemcpyHostToDevice, s));
    VIX_CUDA(cudaStreamSynchronize(s));
    c->off_queries = off_q; c->off_probes = off_p; c->off_results = off_r; c->off_bounds = off_b;
    c->cap_nq = cnq; c->cap_per = per; c->cap_d = cd; c->cap_nprobe = cp; c->cap_k = ck;
    c->peer_state = 1;
    return VIX_OK;
}

// ------------------------------------------------------------------------------------------------ device pieces
// Barrier across the ranks on the stream: thread p tells peer p "rank has reached barrier `epoch`" (a release store into
// the peer's flag word for this rank) and waits until peer p has said the same (an acquire load of its word here).
// Everything the preceding kernels of this stream stored into the peers is visible there before the flag is.
__global__ void peer_barrier_kernel(void* const* __restrict__ peer_base, int world, int rank, uint32_t epoch, int* error_host) {
    const int p = (int)threadIdx.x;
    if (p >= world) return;
    __threadfence_system();
    uint32_t* remote = reinterpret_cast<uint32_t*>(peer_base[p]) + rank;
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(remote), "r"(epoch) : "memory");
    const uint32_t* mine = reinterpret_cast<const uint32_t*>(peer_base[rank]) + p;
    const long long t0 = clock64();
    for (;;) {
        uint32_t v;
        asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(mine) : "memory");
        if ((int32_t)(v - epoch) >= 0) break;
        if (clock64() - t0 > 20000000000LL) {              // ~10 s: a peer that never arrives is an error, not a hang
            if (error_host) { *reinterpret_cast<volatile int*>(error_host) = 1; __threadfence_system(); }
            break;
        }
    }
}

// bytes [offA, offA + bytesA) and [offB, offB + bytesB) of this rank's region -> the same offsets of every peer's region
__global__ void peer_push_kernel(void* const* __restrict__ peer_base, int world, int rank, size_t offA, size_t nA16,
                                 size_t offB, size_t nB16) {
    const uint4* srcA = reinterpret_cast<const uint4*>(static_cast<const char*>(peer_base[rank]) + offA);
    const uint4* srcB = reinterpret_cast<const uint4*>(static_cast<const char*>(peer_base[rank]) + offB);
    const size_t total = nA16 + nB16;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const bool inA = i < nA16;
        const size_t j = inA ? i : i - nA16;
        const uint4 v = inA ? srcA[j] : srcB[j];
        const size_t off = (inA ? offA : offB) + 16 * j;
        for (int p = 0; p < world; ++p)
            if (p != rank) *reinterpret_cast<uint4*>(static_cast<char*>(peer_base[p]) + off) = v;
    }
}

__global__ void fill_i32_kernel(int32_t* a, int64_t n, int32_t v) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) a[i] = v;
}

// local top-k -> packed keys (orderable API distance << 32 | id; ascending key order is mergeTopK's order for both
// metrics, the API distance of the inner product being -dot) -> slot `rank` of [world][nq][k] in every destination
__global__ void pack_result_keys_kernel(const float* __restrict__ dist, const int64_t* __restrict__ ids, int64_t total,
                                        void* const* __restrict__ peer_base, int world, size_t off, u64* __restrict__ local_only) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const int64_t id = ids[i];
    const u64 key = id < 0 ? kEmptyKey : make_key(dist[i], (uint32_t)id, 0);
    if (local_only) { local_only[i] = key; return; }
    for (int p = 0; p < world; ++p) reinterpret_cast<u64*>(static_cast<char*>(peer_base[p]) + off)[i] = key;
}

// keys_all: [world][nq][k] as gathered; one CTA per query selects the k smallest of its world x k keys (padding keys
// come out as NaN / id -1)
__global__ void merge_shard_keys_kernel(const u64* __restrict__ keys_all, int world, int64_t nq, int k, int P2,
                                        float* __restrict__ out_dist, int64_t* __restrict__ out_ids) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    u64* s = reinterpret_cast<u64*>(smem_raw);
    const int64_t row = blockIdx.x;
    const int nin = world * k;
    for (int i = threadIdx.x; i < P2; i += blockDim.x) {
        u64 key = kEmptyKey;
        if (i < nin) { const int r = i / k, j = i - r * k; key = keys_all[((size_t)r * nq + row) * k + j]; }
        s[i] = key;
    }
    __syncthreads();
    bitonic_sort_keys<false>(s, P2, threadIdx.x, blockDim.x);
    for (int i = threadIdx.x; i < k; i += blockDim.x) {
        const u64 key = s[i];
        const size_t o = (size_t)row * k + i;
        if (key == kEmptyKey) {
            out_dist[o] = __int_as_float(0x7fc00000);
            out_ids[o] = -1;
        } else {
            out_dist[o] = key_score(key, 0);
            out_ids[o] = (int64_t)key_id(key);
        }
    }
}

static int merge_shard_keys(const u64* keys_all, int world, int64_t nq, int k, float* out_dist, int64_t* out_ids) {
    const int P2 = next_pow2(world * k < 2 ? 2 : world * k);
    const size_t smem = (size_t)P2 * 8;
    VIX_REQUIRE(smem <= 200 * 1024, VIX_ERR_UNSUPPORTED, "shard merge: %d keys per query exceed shared memory", world * k);
    VIX_CUDA(cudaFuncSetAttribute(merge_shard_keys_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int threads = P2 / 2 < 32 ? 32 : (P2 / 2 > 256 ? 256 : P2 / 2);
    merge_shard_keys_kernel<<<(unsigned)nq, threads, smem, ctx().stream>>>(keys_all, world, nq, k, P2, out_dist, out_ids);
    VIX_LAUNCH_CHECK();
    return VIX_OK;
}

// The list-major scan's bounds (vix_scan.cuh: scan_thr_hook_t) over peer memory: a rank finds a finite bound only for the
// queries whose first probed list it owns, so the minimum over the ranks is a store of those into every peer's bound
// array, a barrier, and a minimum with what arrived here -- which is reset on the way (the next writers are behind the
// next call's first barrier, which this rank enters after the reset).
__global__ void push_bounds_kernel(const float* __restrict__ thr, int64_t nq, void* const* __restrict__ peer_base, int world, int rank,
                                   size_t off) {
    const int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= nq) return;
    const float t = thr[q];
    if (!(fabsf(t) < __int_as_float(0x7f800000))) return;
    for (int p = 0; p < world; ++p)
        if (p != rank) reinterpret_cast<float*>(static_cast<char*>(peer_base[p]) + off)[q] = t;
}
__global__ void take_bounds_kernel(float* __restrict__ thr, int64_t nq, uint32_t* __restrict__ arrived) {
    const int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= nq) return;
    const uint32_t v = arrived[q];
    arrived[q] = 0xFFFFFFFFu;
    thr[q] = fminf(thr[q], __uint_as_float(v));             // fminf(x, NaN) = x
}

static int peer_barrier(vix_comm* c) {
    c->epoch += 1;
    peer_barrier_kernel<<<1, 32 * ((c->world + 31) / 32), 0, ctx().stream>>>(c->peer_dev, c->world, c->rank, c->epoch,
                                                                              pipeline_error_flag());
    VIX_LAUNCH_CHECK();
    return VIX_OK;
}

// owner rank of a list under block boundaries bounds[world + 1]
__global__ void owner_kernel(const int32_t* __restrict__ assign, int64_t n, const int64_t* __restrict__ bounds, int world,
                             int32_t* __restrict__ owner, int32_t* __restrict__ row, unsigned long long* __restrict__ counts) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int64_t l = assign[i];
    int o = 0;
    while (o + 1 < world && l >= bounds[o + 1]) ++o;
    owner[i] = o;
    row[i] = (int32_t)i;
    atomicAdd(counts + o, 1ull);
}

__global__ void gather_rows_kernel(const int32_t* __restrict__ order, int64_t n, int m, const int32_t* __restrict__ assign,
                                   const uint8_t* __restrict__ codes, const int64_t* __restrict__ ids,
                                   int32_t* __restrict__ out_assign, uint8_t* __restrict__ out_codes, int64_t* __restrict__ out_ids) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int64_t r = order[i];
    out_assign[i] = assign[r];
    out_ids[i] = ids[r];
    for (int j = 0; j < m; ++j) out_codes[i * (int64_t)m + j] = codes[r * (int64_t)m + j];
}

}  // namespace vix

extern "C" {

int vix_comm_unique_id(void* id_out, size_t capacity) {
    VIX_TRY(nccl_load());
    VIX_REQUIRE(id_out && capacity >= sizeof(ncclUniqueId), VIX_ERR_INVALID_PARAM, "vix_comm_unique_id: needs %zu bytes",
                sizeof(ncclUniqueId));
    ncclUniqueId id;
    VIX_NCCL(g_nccl.GetUniqueId(&id));
    memcpy(id_out, &id, sizeof(id));
    return VIX_OK;
}

int vix_comm_create(const void* id, size_t id_bytes, int rank, int world, vix_comm_t** out) {
    VIX_TRY(ensure_device());
    VIX_TRY(nccl_load());
    VIX_REQUIRE(id && out, VIX_ERR_NULL_PTR, "vix_comm_create: null pointer");
    VIX_REQUIRE(id_bytes >= sizeof(ncclUniqueId), VIX_ERR_INVALID_PARAM, "vix_comm_create: the id has %zu bytes", sizeof(ncclUniqueId));
    VIX_REQUIRE(world > 0 && world <= 256 && rank >= 0 && rank < world, VIX_ERR_INVALID_PARAM, "vix_comm_create: rank / world");
    vix_comm* c = new (std::nothrow) vix_comm();
    VIX_REQUIRE(c, VIX_ERR_OOM, "vix_comm_create: out of host memory");
    c->rank = rank; c->world = world;
    cudaGetDevice(&c->device);
    ncclUniqueId uid;
    memcpy(&uid, id, sizeof(uid));
    ncclResult_t r = g_nccl.CommInitRank(&c->comm, world, uid, rank);
    if (r != ncclSuccess) {
        set_error("ncclCommInitRank failed: %s", g_nccl.GetErrorString(r));
        delete c;
        return VIX_ERR_CUDA;
    }
    *out = c;
    return VIX_OK;
}

int vix_comm_destroy(vix_comm_t* c) {
    if (!c) return VIX_OK;
    cudaDeviceSynchronize();
    close_peers(c);
    if (c->gather_probes) cudaFree(c->gather_probes);
    if (c->gather_keys) cudaFree(c->gather_keys);
    for (auto& e : c->ev) if (e) cudaEventDestroy(e);
    if (c->comm) g_nccl.CommDestroy(c->comm);
    delete c;
    return VIX_OK;
}

int vix_comm_rank(const vix_comm_t* c) { return c ? c->rank : -1; }
int vix_comm_world(const vix_comm_t* c) { return c ? c->world : 0; }
int vix_comm_uses_peer_memory(const vix_comm_t* c) { return c ? c->peer_state : -1; }

int vix_sharded_query_block(int64_t nq, int rank, int world, int64_t* first, int64_t* count) {
    VIX_REQUIRE(first && count && world > 0 && rank >= 0 && rank < world && nq >= 0, VIX_ERR_INVALID_PARAM, "vix_sharded_query_block");
    const int64_t per = block_rows(nq, world);
    const int64_t lo = nq < (int64_t)rank * per ? nq : (int64_t)rank * per;
    const int64_t hi = nq < lo + per ? nq : lo + per;
    *first = lo; *count = hi - lo;
    return VIX_OK;
}

// the list-major scan's per-query bounds -> their minimum over the ranks (vix_scan.cuh: scan_thr_hook_t)
static int thr_min_over_ranks(void* ctx, float* thr_dev, int64_t nq) {
    vix_comm* c = static_cast<vix_comm*>(ctx);
    cudaStream_t s = vix::ctx().stream;
    if (c->peer_state == 1 && nq <= c->cap_nq) {
        const unsigned grid = (unsigned)((nq + 255) / 256);
        push_bounds_kernel<<<grid, 256, 0, s>>>(thr_dev, nq, c->peer_dev, c->world, c->rank, c->off_bounds);
        VIX_LAUNCH_CHECK();
        VIX_TRY(peer_barrier(c));
        take_bounds_kernel<<<grid, 256, 0, s>>>(thr_dev, nq, reinterpret_cast<uint32_t*>(static_cast<char*>(c->local) + c->off_bounds));
        VIX_LAUNCH_CHECK();
        return VIX_OK;
    }
    VIX_NCCL(g_nccl.AllReduce(thr_dev, thr_dev, (size_t)nq, ncclFloat, ncclMin, c->comm, s));
    return VIX_OK;
}
struct ThrHookScope {
    ThrHookScope(vix_comm* c) { set_scan_thr_hook(thr_min_over_ranks, c); }
    ~ThrHookScope() { set_scan_thr_hook(nullptr, nullptr); }
};

int vix_sharded_search(vix_index_t* h, vix_comm_t* c, const float* queries, int64_t nq, int k, int nprobe, float* out_dist,
                       int64_t* out_ids) {
    VIX_TRY(ensure_device());
    VIX_REQUIRE(h && c, VIX_ERR_NULL_PTR, "vix_sharded_search: null handle");
    if (nq <= 0 || k <= 0) return VIX_OK;                             // IVFIndex.swift:866 (every rank sees the same nq, k)
    VIX_REQUIRE(queries && out_dist && out_ids, VIX_ERR_NULL_PTR, "vix_sharded_search: null pointer");
    VIX_REQUIRE(k <= VIX_MAX_K, VIX_ERR_INVALID_K, "vix_sharded_search: k > %d", VIX_MAX_K);
    std::lock_guard<std::mutex> lc(c->mu);
    std::lock_guard<std::mutex> lk(h->mu);
    VIX_REQUIRE(h->p.kind == VIX_INDEX_IVF_PQ && h->has_coarse && h->has_pq, VIX_ERR_NOT_TRAINED, "vix_sharded_search: needs a trained IVF-PQ index");
    VIX_REQUIRE(h->p.metric != VIX_METRIC_COSINE, VIX_ERR_UNSUPPORTED, "vix_sharded_search: L2 / IP only");
    if (nprobe <= 0) nprobe = h->p.nprobe;
    VIX_REQUIRE(nprobe > 0 && nprobe <= VIX_MAX_K, VIX_ERR_INVALID_K, "vix_sharded_search: nprobe");
    const int world = c->world, rank = c->rank, d = h->p.d;
    if (world == 1) return index_search_locked(h, queries, nq, k, nprobe, out_dist, out_ids, nullptr, nullptr);
    cudaStream_t s = ctx().stream;
    if (h->dirty) VIX_TRY(build_lists(h));
    VIX_TRY(ensure_region(c, nq, d, nprobe, k));
    ThrHookScope thr_scope(c);                                        // (cleared again on every way out)
    const bool host_q = !is_device_ptr(queries);
    const int64_t per = block_rows(nq, world);
    const int64_t lo = nq < (int64_t)rank * per ? nq : (int64_t)rank * per;
    const int64_t cnt = (nq < lo + per ? nq : lo + per) - lo;
    const int64_t total = nq * (int64_t)k;
    Out<float> dd;
    Out<int64_t> di;
    VIX_TRY(dd.stage(out_dist, (size_t)total));
    VIX_TRY(di.stage(out_ids, (size_t)total));
    Scratch<float> ldist;
    Scratch<int64_t> lids;
    VIX_TRY(ldist.alloc((size_t)total));
    VIX_TRY(lids.alloc((size_t)total));
    auto mark = [&](int i) { if (c->trace) cudaEventRecord(c->ev[i], s); };
    mark(0);

    if (c->peer_state == 1) {
        char* base = static_cast<char*>(c->local);
        float* qbuf = reinterpret_cast<float*>(base + c->off_queries);          // [world * per][d] (this call's per)
        int32_t* pbuf = reinterpret_cast<int32_t*>(base + c->off_probes);       // [world * per][nprobe]
        u64* rbuf = reinterpret_cast<u64*>(base + c->off_results);              // [world][nq][k]
        // 1. this rank's block of the batch: host queries cross PCIe once per rank, 1/world of the batch each
        const float* qblock = queries + (size_t)lo * d;
        if (host_q && cnt > 0) {
            VIX_CUDA(cudaMemcpyAsync(qbuf + (size_t)lo * d, qblock, (size_t)cnt * d * 4, cudaMemcpyHostToDevice, s));
            qblock = qbuf + (size_t)lo * d;
        }
        // 2. its probe lists against ALL centroids, straight into slot `rank` of the local probe buffer
        int32_t* pblock = pbuf + (size_t)rank * per * nprobe;
        if (cnt > 0)
            VIX_TRY(probe_select_fast_device(qblock, cnt, h->coarse.ptr, h->kc, d, h->p.metric, nprobe, h->coarse_norms.ptr,
                                             pblock, nullptr, h->coarse_norm_max.ptr));
        if (cnt < per) {
            const int64_t pad = (per - cnt) * nprobe;
            fill_i32_kernel<<<(unsigned)((pad + 255) / 256), 256, 0, s>>>(pblock + (size_t)cnt * nprobe, pad, -1);
            VIX_LAUNCH_CHECK();
        }
        // 3. the block travels to every peer (probes, and the queries when they came from the host), one barrier
        {
            const size_t offA = c->off_probes + (size_t)rank * per * nprobe * 4, nA = (size_t)per * nprobe * 4 / 16;
            const size_t offB = c->off_queries + (size_t)rank * per * d * 4, nB = host_q ? (size_t)per * d * 4 / 16 : 0;
            const size_t n16 = nA + nB;
            const size_t want = (n16 + 255) / 256;
            const unsigned grid = (unsigned)(want < (size_t)(2 * num_sms()) ? (want ? want : 1) : (size_t)(2 * num_sms()));
            peer_push_kernel<<<grid, 256, 0, s>>>(c->peer_dev, world, rank, offA, nA, offB, nB);
            VIX_LAUNCH_CHECK();
            VIX_TRY(peer_barrier(c));
        }
        mark(1);
        // 4. fused scan over the probed lists this rank owns
        const float* qall = host_q ? qbuf : queries;
        VIX_TRY(index_search_locked(h, qall, nq, k, nprobe, ldist.ptr, lids.ptr, nullptr, nullptr, pbuf));
        mark(2);
        // 5. its top-k leaves as packed keys for slot `rank` of every rank's result buffer; barrier; merge
        pack_result_keys_kernel<<<(unsigned)((total + 255) / 256), 256, 0, s>>>(ldist.ptr, lids.ptr, total, c->peer_dev, world,
                                                                              c->off_results + (size_t)rank * total * 8, nullptr);
        VIX_LAUNCH_CHECK();
        VIX_TRY(peer_barrier(c));
        VIX_TRY(merge_shard_keys(rbuf, world, nq, k, dd.dev, di.dev));
    } else {
        // NCCL carries the two exchanges
        In<float> dq;
        VIX_TRY(dq.stage(queries, (size_t)nq * d));
        const size_t pbytes = (size_t)world * per * nprobe * 4, kbytes = (size_t)world * total * 8;
        if (pbytes > c->gather_probes_bytes) {
            if (c->gather_probes) { VIX_CUDA(cudaStreamSynchronize(s)); cudaFree(c->gather_probes); c->gather_probes = nullptr; }
            VIX_CUDA(cudaMalloc(&c->gather_probes, pbytes));
            c->gather_probes_bytes = pbytes;
        }
        if (kbytes > c->gather_keys_bytes) {
            if (c->gather_keys) { VIX_CUDA(cudaStreamSynchronize(s)); cudaFree(c->gather_keys); c->gather_keys = nullptr; }
            VIX_CUDA(cudaMalloc(&c->gather_keys, kbytes));
            c->gather_keys_bytes = kbytes;
        }
        int32_t* pall = static_cast<int32_t*>(c->gather_probes);
        int32_t* pblock = pall + (size_t)rank * per * nprobe;
        if (cnt > 0)
            VIX_TRY(probe_select_fast_device(dq.dev + (size_t)lo * d, cnt, h->coarse.ptr, h->kc, d, h->p.metric, nprobe,
                                             h->coarse_norms.ptr, pblock, nullptr, h->coarse_norm_max.ptr));
        if (cnt < per) {
            const int64_t pad = (per - cnt) * nprobe;
            fill_i32_kernel<<<(unsigned)((pad + 255) / 256), 256, 0, s>>>(pblock + (size_t)cnt * nprobe, pad, -1);
            VIX_LAUNCH_CHECK();
        }
        VIX_NCCL(g_nccl.AllGather(pblock, pall, (size_t)per * nprobe, ncclInt32, c->comm, s));   // in place
        mark(1);
        VIX_TRY(index_search_locked(h, dq.dev, nq, k, nprobe, ldist.ptr, lids.ptr, nullptr, nullptr, pall));
        mark(2);
        u64* kall = static_cast<u64*>(c->gather_keys);
        pack_result_keys_kernel<<<(unsigned)((total + 255) / 256), 256, 0, s>>>(ldist.ptr, lids.ptr, total, nullptr, world, 0,
                                                                              kall + (size_t)rank * total);
        VIX_LAUNCH_CHECK();
        VIX_NCCL(g_nccl.AllGather(kall + (size_t)rank * total, kall, (size_t)total, ncclUint64, c->comm, s));
        VIX_TRY(merge_shard_keys(kall, world, nq, k, dd.dev, di.dev));
    }
    mark(3);
    VIX_TRY(dd.commit());
    VIX_TRY(di.commit());
    return finish(dd.is_host() || di.is_host());
}

int vix_comm_trace(vix_comm_t* c, int enabled) {
    VIX_REQUIRE(c, VIX_ERR_NULL_PTR, "vix_comm_trace: null handle");
    std::lock_guard<std::mutex> lc(c->mu);
    if (enabled)
        for (auto& e : c->ev)
            if (!e) VIX_CUDA(cudaEventCreate(&e));
    c->trace = enabled != 0;
    return VIX_OK;
}

int vix_comm_trace_get(vix_comm_t* c, float* phase_ms /* [3] */) {
    VIX_REQUIRE(c && phase_ms, VIX_ERR_NULL_PTR, "vix_comm_trace_get: null pointer");
    std::lock_guard<std::mutex> lc(c->mu);
    VIX_REQUIRE(c->trace && c->ev[3], VIX_ERR_CONTRACT, "vix_comm_trace_get: tracing is off");
    VIX_CUDA(cudaEventSynchronize(c->ev[3]));
    for (int i = 0; i < 3; ++i) VIX_CUDA(cudaEventElapsedTime(phase_ms + i, c->ev[i], c->ev[i + 1]));
    return VIX_OK;
}

int vix_sharded_add(vix_index_t* h, vix_comm_t* c, const int64_t* list_bounds, const float* x, const int64_t* ids, int64_t n) {
    VIX_TRY(ensure_device());
    VIX_REQUIRE(h && c, VIX_ERR_NULL_PTR, "vix_sharded_add: null handle");
    VIX_REQUIRE(n >= 0 && (n == 0 || (x && ids)), VIX_ERR_NULL_PTR, "vix_sharded_add: null pointer (explicit ids are required)");
    std::lock_guard<std::mutex> lc(c->mu);
    std::lock_guard<std::mutex> lk(h->mu);
    VIX_REQUIRE(h->p.kind == VIX_INDEX_IVF_PQ && h->has_coarse && h->has_pq, VIX_ERR_NOT_TRAINED, "vix_sharded_add: needs a trained IVF-PQ index");
    const int world = c->world, rank = c->rank, d = h->p.d, m = h->code_bytes();   // m: bytes per stored code
    cudaStream_t s = ctx().stream;
    // block boundaries of the list partition: given, or equal-count blocks
    std::vector<int64_t> bounds((size_t)world + 1);
    for (int r = 0; r <= world; ++r) bounds[r] = list_bounds ? list_bounds[r] : (int64_t)h->kc * r / world;
    VIX_REQUIRE(bounds[0] == 0 && bounds[world] == h->kc, VIX_ERR_INVALID_PARAM, "vix_sharded_add: bounds must run from 0 to %d", h->kc);
    for (int r = 0; r < world; ++r)
        VIX_REQUIRE(bounds[r + 1] >= bounds[r], VIX_ERR_INVALID_PARAM, "vix_sharded_add: bounds must ascend");
    // 1. assign + encode what this rank was handed
    In<float> dx;
    In<int64_t> dids;
    VIX_TRY(dx.stage(x, (size_t)n * d));
    VIX_TRY(dids.stage(ids, (size_t)n));
    Scratch<int32_t> asg, owner, row, order, owner_sorted;
    Scratch<uint8_t> codes;
    Scratch<unsigned long long> dcounts;
    Scratch<int64_t> dbounds;
    VIX_TRY(dcounts.alloc((size_t)world * (world + 1)));
    VIX_TRY(dbounds.alloc((size_t)world + 1));
    VIX_CUDA(cudaMemsetAsync(dcounts.ptr, 0, sizeof(unsigned long long) * world * (world + 1), s));
    VIX_CUDA(cudaMemcpyAsync(dbounds.ptr, bounds.data(), sizeof(int64_t) * (world + 1), cudaMemcpyHostToDevice, s));
    Scratch<int32_t> s_asg;
    Scratch<uint8_t> s_codes;
    Scratch<int64_t> s_ids;
    if (n > 0) {
        VIX_TRY(asg.alloc((size_t)n));
        VIX_TRY(codes.alloc((size_t)n * m));
        VIX_TRY(assign_lists_device(h, dx.dev, n, asg.ptr));
        unsigned long long invalid = 0;
        VIX_TRY(count_invalid_assign(asg.ptr, n, h->kc, &invalid));
        VIX_REQUIRE(invalid == 0, VIX_ERR_INVALID_PARAM, "vix_sharded_add: %llu rows have no nearest list (NaN components?)", invalid);
        VIX_TRY(encode_rows_device(h, dx.dev, n, asg.ptr, codes.ptr));
        // 2. rows ordered by owning rank (stable: rows keep their order inside a block)
        VIX_TRY(owner.alloc((size_t)n));
        VIX_TRY(row.alloc((size_t)n));
        VIX_TRY(order.alloc((size_t)n));
        VIX_TRY(owner_sorted.alloc((size_t)n));
        owner_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(asg.ptr, n, dbounds.ptr, world, owner.ptr, row.ptr,
                                                               dcounts.ptr + (size_t)world * world);
        VIX_LAUNCH_CHECK();
        int bits = 1;
        while ((1 << bits) < world) ++bits;
        size_t tmp_bytes = 0;
        VIX_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, owner.ptr, owner_sorted.ptr, row.ptr, order.ptr, (int)n, 0, bits, s));
        Scratch<unsigned char> tmp;
        VIX_TRY(tmp.alloc(tmp_bytes + 16));
        VIX_CUDA(cub::DeviceRadixSort::SortPairs(tmp.ptr, tmp_bytes, owner.ptr, owner_sorted.ptr, row.ptr, order.ptr, (int)n, 0, bits, s));
        ctx().launches += 1;
        VIX_TRY(s_asg.alloc((size_t)n));
        VIX_TRY(s_codes.alloc((size_t)n * m));
        VIX_TRY(s_ids.alloc((size_t)n));
        gather_rows_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(order.ptr, n, m, asg.ptr, codes.ptr, dids.dev, s_asg.ptr,
                                                                     s_codes.ptr, s_ids.ptr);
        VIX_LAUNCH_CHECK();
    }
    // 3. everybody learns everybody's send counts
    VIX_NCCL(g_nccl.AllGather(dcounts.ptr + (size_t)world * world, dcounts.ptr, (size_t)world, ncclUint64, c->comm, s));
    std::vector<unsigned long long> counts((size_t)world * world);
    VIX_CUDA(cudaMemcpyAsync(counts.data(), dcounts.ptr, sizeof(unsigned long long) * world * world, cudaMemcpyDeviceToHost, s));
    VIX_CUDA(cudaStreamSynchronize(s));
    std::vector<int64_t> send_off((size_t)world + 1, 0), recv_off((size_t)world + 1, 0);
    for (int p = 0; p < world; ++p) {
        send_off[p + 1] = send_off[p] + (int64_t)counts[(size_t)rank * world + p];
        recv_off[p + 1] = recv_off[p] + (int64_t)counts[(size_t)p * world + rank];
    }
    const int64_t nrecv = recv_off[world];
    // 4. rows travel to their owners
    Scratch<int32_t> r_asg;
    Scratch<uint8_t> r_codes;
    Scratch<int64_t> r_ids;
    VIX_TRY(r_asg.alloc((size_t)nrecv));
    VIX_TRY(r_codes.alloc((size_t)nrecv * m));
    VIX_TRY(r_ids.alloc((size_t)nrecv));
    VIX_NCCL(g_nccl.GroupStart());
    for (int p = 0; p < world; ++p) {
        const int64_t sc = send_off[p + 1] - send_off[p], rc = recv_off[p + 1] - recv_off[p];
        if (sc > 0) {
            VIX_NCCL(g_nccl.Send(s_asg.ptr + send_off[p], (size_t)sc, ncclInt32, p, c->comm, s));
            VIX_NCCL(g_nccl.Send(s_codes.ptr + (size_t)send_off[p] * m, (size_t)sc * m, ncclUint8, p, c->comm, s));
            VIX_NCCL(g_nccl.Send(s_ids.ptr + send_off[p], (size_t)sc, ncclInt64, p, c->comm, s));
        }
        if (rc > 0) {
            VIX_NCCL(g_nccl.Recv(r_asg.ptr + recv_off[p], (size_t)rc, ncclInt32, p, c->comm, s));
            VIX_NCCL(g_nccl.Recv(r_codes.ptr + (size_t)recv_off[p] * m, (size_t)rc * m, ncclUint8, p, c->comm, s));
            VIX_NCCL(g_nccl.Recv(r_ids.ptr + recv_off[p], (size_t)rc, ncclInt64, p, c->comm, s));
        }
    }
    VIX_NCCL(g_nccl.GroupEnd());
    // 5. append (already encoded)
    if (nrecv > 0) VIX_TRY(index_add_encoded_locked(h, r_asg.ptr, r_codes.ptr, r_ids.ptr, nrecv));
    return finish(true);
}

}  // extern "C"
