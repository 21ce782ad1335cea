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
#include "vix_comm.cuh"
#include "vix_scan.cuh"
#include "vix_topk.cuh"
#include "vix_group.cuh"
#include "vix_range.cuh"

#include <dlfcn.h>
#include <nccl.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <functional>
#include <memory>
#include <new>
#include <optional>
#include <vector>

namespace vix {

NcclApi g_nccl;
static std::mutex g_nccl_mu;

int nccl_load() {
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

}  // namespace vix

using namespace vix;

namespace vix {

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

// Collective: make every rank's region large enough for (nq, d, nprobe, k) and map it everywhere.  All ranks call this
// with the same arguments, so they agree on whether to reallocate.  Returns with c->peer_state decided.
int ensure_region(vix_comm* c, int64_t nq, int d, int nprobe, int k) {
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
// come out as NaN / id -1).  The keys hold zero distances as +0 (make_key folds -0); one GPU's IVF-PQ scan returns a zero
// inner-product distance as -0 (the API distance -score of a +0 score), its IVF-Flat scan and every L2 distance +0, so
// neg_zero (the kind's, as KnnDecode's) restores the sign.
__global__ void merge_shard_keys_kernel(const u64* __restrict__ keys_all, int world, int64_t nq, int k, int P2, int neg_zero,
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
            const float v = key_score(key, 0);
            out_dist[o] = (v == 0.0f && neg_zero) ? -0.0f : v;
            out_ids[o] = (int64_t)key_id(key);
        }
    }
}

static int merge_shard_keys(const u64* keys_all, int world, int64_t nq, int k, int neg_zero, float* out_dist, int64_t* out_ids) {
    const int P2 = next_pow2(world * k < 2 ? 2 : world * k);
    const size_t smem = (size_t)P2 * 8;
    VIX_REQUIRE(smem <= 200 * 1024, VIX_ERR_UNSUPPORTED, "shard merge: %d keys per query exceed shared memory", world * k);
    VIX_CUDA(cudaFuncSetAttribute(merge_shard_keys_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int threads = P2 / 2 < 32 ? 32 : (P2 / 2 > 256 ? 256 : P2 / 2);
    merge_shard_keys_kernel<<<(unsigned)nq, threads, smem, ctx().stream>>>(keys_all, world, nq, k, P2, neg_zero, out_dist, out_ids);
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

int peer_barrier(vix_comm* c) {
    c->epoch += 1;
    peer_barrier_kernel<<<1, 32 * ((c->world + 31) / 32), 0, ctx().stream>>>(c->peer_dev, c->world, c->rank, c->epoch,
                                                                              pipeline_error_flag());
    VIX_LAUNCH_CHECK();
    return VIX_OK;
}

// owner rank of a list under block boundaries bounds[world + 1]
__global__ void owner_kernel(const int32_t* __restrict__ assign, int64_t n, const int64_t* __restrict__ bounds, int world,
                             int32_t* __restrict__ owner, unsigned long long* __restrict__ counts) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int64_t l = assign[i];
    int o = 0;
    while (o + 1 < world && l >= bounds[o + 1]) ++o;
    owner[i] = o;
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

// the IVF-Flat sibling of gather_rows_kernel: float rows of d components
__global__ void gather_vec_rows_kernel(const int32_t* __restrict__ order, int64_t n, int d, const int32_t* __restrict__ assign,
                                       const float* __restrict__ x, const int64_t* __restrict__ ids, int32_t* __restrict__ out_assign,
                                       float* __restrict__ out_x, int64_t* __restrict__ out_ids) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int64_t r = order[i];
    out_assign[i] = assign[r];
    out_ids[i] = ids[r];
    for (int j = 0; j < d; ++j) out_x[i * (int64_t)d + j] = x[r * (int64_t)d + j];
}

// ------------------------------------------------------------------------------------------------ sharded range search
// n u64 words of src -> byte offset `off` of every rank's range region (this rank's included)
__global__ void peer_store_kernel(const u64* __restrict__ src, int64_t n, void* const* __restrict__ peer_base, int world,
                                  size_t off) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const u64 v = src[i];
        for (int p = 0; p < world; ++p) reinterpret_cast<u64*>(static_cast<char*>(peer_base[p]) + off)[i] = v;
    }
}

// lims_all: [world][nq + 2] every rank's local row starts (lims[nq] = its total) and its status.  glims[q] = the sum of the
// ranks' row starts (q = 0 .. nq), the global row starts; meta = [base: world + 1 starts of the ranks' keys in the
// concatenation][longest global row][status of every rank]
__global__ void shard_range_lims_kernel(const int64_t* __restrict__ lims_all, int world, int64_t nq, int64_t* __restrict__ glims,
                                        int64_t* __restrict__ meta) {
    const int64_t L = nq + 2;
    for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q <= nq; q += (int64_t)gridDim.x * blockDim.x) {
        int64_t g = 0, len = 0;
        for (int r = 0; r < world; ++r) {
            const int64_t* lr = lims_all + (size_t)r * L;
            g += lr[q];
            if (q < nq) len += lr[q + 1] - lr[q];
        }
        glims[q] = g;
        if (q < nq && len > 0) atomicMax(reinterpret_cast<unsigned long long*>(meta + world + 1), (unsigned long long)len);
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        int64_t acc = 0;
        for (int r = 0; r < world; ++r) {
            meta[r] = acc;
            acc += lims_all[(size_t)r * L + nq];
            meta[world + 2 + r] = lims_all[(size_t)r * L + nq + 1];
        }
        meta[world] = acc;
    }
}

// The merge of the ranks' sorted runs of every row.  keys: every rank's rows, concatenated rank by rank (rank r's from
// base[r]); lims_all as above.  Key i, at place j of rank r's run of row q, has place j + (keys of the lower ranks' runs of
// row q that are <= it) + (keys of the higher ranks' runs of row q that are < it) in the merged row q: one binary search in
// each other run.  Stable, and exact for equal keys on different ranks (one id stored in lists two ranks own): they keep
// rank order, as one GPU's rows would hold them.  Returns that place, *row = q.
// kWord: compare the high words only (the flat engine's keys, whose order within a run is (score word, row) and whose low
// word then carries the user id): ties at one word keep rank order, and inside a rank the run's own order -- together the
// global row order of one GPU holding the ranks' rows rank by rank.
template <bool kWord = false>
__device__ __forceinline__ int64_t shard_merge_place(const u64* __restrict__ keys, const int64_t* __restrict__ base,
                                                     const int64_t* __restrict__ lims_all, int world, int64_t nq, int64_t i,
                                                     int64_t* row) {
    const int64_t L = nq + 2;
    int ra = 0, rb = world;                                   // rank of i: the last r with base[r] <= i
    while (rb - ra > 1) { const int mid = (ra + rb) >> 1; if (base[mid] <= i) ra = mid; else rb = mid; }
    const int r = ra;
    const int64_t* lr = lims_all + (size_t)r * L;
    const int64_t j = i - base[r];
    int64_t qa = 0, qb = nq;                                  // its row: the last q with lr[q] <= j
    while (qb - qa > 1) { const int64_t mid = (qa + qb) >> 1; if (lr[mid] <= j) qa = mid; else qb = mid; }
    const int64_t q = qa;
    const u64 key = keys[i];
    int64_t pos = j - lr[q];
    for (int p = 0; p < world; ++p) {
        if (p == r) continue;
        const int64_t* lp = lims_all + (size_t)p * L;
        const u64* run = keys + base[p] + lp[q];
        int64_t x = 0, y = lp[q + 1] - lp[q];
        if (kWord) {
            const uint32_t w = (uint32_t)(key >> 32);
            if (p < r) {
                while (x < y) { const int64_t mid = (x + y) >> 1; if ((uint32_t)(run[mid] >> 32) <= w) x = mid + 1; else y = mid; }
            } else {
                while (x < y) { const int64_t mid = (x + y) >> 1; if ((uint32_t)(run[mid] >> 32) < w) x = mid + 1; else y = mid; }
            }
        } else if (p < r) {
            while (x < y) { const int64_t mid = (x + y) >> 1; if (run[mid] <= key) x = mid + 1; else y = mid; }
        } else {
            while (x < y) { const int64_t mid = (x + y) >> 1; if (run[mid] < key) x = mid + 1; else y = mid; }
        }
        pos += x;
    }
    *row = q;
    return pos;
}

// range search: every key to its place in the global rows (glims: their starts), decoded on the way (range_decode_key)
__global__ void __launch_bounds__(256)
shard_range_merge_kernel(const u64* __restrict__ keys, const int64_t* __restrict__ base, const int64_t* __restrict__ lims_all,
                         int world, int64_t nq, const int64_t* __restrict__ glims, int64_t total, int neg_zero,
                         float* __restrict__ out_dist, int64_t* __restrict__ out_ids) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        int64_t q;
        const int64_t place = shard_merge_place(keys, base, lims_all, world, nq, i, &q);
        const int64_t pos = glims[q] + place;
        range_decode_key(keys[i], neg_zero, out_dist + pos, out_ids + pos);
    }
}

// k-NN search beyond VIX_MAX_K: the merged rows cut at k, straight into out [nq x k]: a key is written only when its place
// is < k; the places of a row from its length (glims) to k are padded with id -1 / NaN.
//
// Exactness of the sharded route (sharded_knn_large).  Let C be a query's global candidate multiset, C = the union over
// the ranks of C_r (the probed lists rank r owns).  Each rank's seed S_r, a subset of C_r with |S_r| >= k, gives tau_r >=
// the k-th word of C; so does tau = min_r tau_r (tau_r = 0xFFFFFFFF when |S_r| < k).  The keys of C with word <= tau hold
// the true top k and every tie at the k-th distance.  The global top k restricted to C_r is a prefix of rank r's sorted
// collected row of length at most k, so cutting each row at k before the exchange loses nothing, and the merged rows cut at
// k are the one-GPU answer.  If tau != 0xFFFFFFFF, the rank that attained it holds at least k keys within it, so the merged
// row holds at least k; a shorter one means the two passes disagreed on a distance (shard_knn_short_kernel).  At most
// world x k keys per query travel, and that many only when no rank's seed reaches k.
__global__ void __launch_bounds__(256)
shard_knn_merge_kernel(const u64* __restrict__ keys, const int64_t* __restrict__ base, const int64_t* __restrict__ lims_all,
                       int world, int64_t nq, const int64_t* __restrict__ glims, int64_t total, int k, int neg_zero,
                       float* __restrict__ out_dist, int64_t* __restrict__ out_ids) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
        int64_t q;
        const int64_t place = shard_merge_place(keys, base, lims_all, world, nq, i, &q);
        if (place < k) range_decode_key(keys[i], neg_zero, out_dist + q * k + place, out_ids + q * k + place);
    }
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < nq * (int64_t)k; e += stride) {
        const int64_t q = e / k, j = e - q * k;
        if (j >= glims[q + 1] - glims[q]) { out_dist[e] = __int_as_float(0x7fc00000); out_ids[e] = -1; }
    }
}

// ---- the flat kind: keys (raw score word in the metric's order, user id), merged by word and rank (trap: one GPU orders
// flat results by (raw score, row) and maps to API distances only then -- sqrt and 1 - s can round two scores to one
// distance, and equal scores fall to the smaller ROW, i.e. the lower rank, not the smaller id)
__device__ __forceinline__ void flat_decode_key(u64 key, int order_max, int dist_mode, float* dist, int64_t* id) {
    float v = key_score(key, order_max);
    if (dist_mode == 1) v = __fsqrt_rn(v);
    else if (dist_mode == 2) v = -v;
    else if (dist_mode == 3) v = __fsub_rn(1.0f, v);
    *dist = v;
    *id = (int64_t)key_id(key);
}

// the per-rank CSR runs of the flat kind merged by (word, rank, place in the run), decoded with the flat API mapping: k > 0
// cuts every merged row at k into out [nq x k] (padding id -1 / NaN past the row's length), k == 0 writes the whole rows at
// glims
__global__ void __launch_bounds__(256)
shard_flat_merge_kernel(const u64* __restrict__ keys, const int64_t* __restrict__ base, const int64_t* __restrict__ lims_all,
                        int world, int64_t nq, const int64_t* __restrict__ glims, int64_t total, int k, int order_max,
                        int dist_mode, float* __restrict__ out_dist, int64_t* __restrict__ out_ids) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
        int64_t q;
        const int64_t place = shard_merge_place<true>(keys, base, lims_all, world, nq, i, &q);
        if (k == 0) flat_decode_key(keys[i], order_max, dist_mode, out_dist + glims[q] + place, out_ids + glims[q] + place);
        else if (place < k) flat_decode_key(keys[i], order_max, dist_mode, out_dist + q * k + place, out_ids + q * k + place);
    }
    if (k == 0) return;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < nq * (int64_t)k; e += stride) {
        const int64_t q = e / k, j = e - q * k;
        if (j >= glims[q + 1] - glims[q]) { out_dist[e] = __int_as_float(0x7fc00000); out_ids[e] = -1; }
    }
}

// k <= VIX_MAX_K: keys_all [world][nq][k], each rank's row its fused top-k (word, user id) in the flat search's order with
// its padding (kEmptyKey: no real key is, ids being < 2^32 - 1) at the end.  One CTA per query: the length of every run
// (its real keys, so that a NaN score -- word 0xFFFFFFFF -- is never confused with padding), then every real key to its
// place by shard_merge_place's word rule, the places from the merged length to k padded.
__global__ void __launch_bounds__(256)
merge_flat_keys_kernel(const u64* __restrict__ keys_all, int world, int64_t nq, int k, int order_max, int dist_mode,
                       float* __restrict__ out_dist, int64_t* __restrict__ out_ids) {
    extern __shared__ int s_len[];                               // [world]
    const int64_t q = blockIdx.x;
    for (int r = threadIdx.x; r < world; r += blockDim.x) {
        const u64* run = keys_all + ((size_t)r * nq + q) * k;
        int x = 0, y = k;
        while (x < y) { const int mid = (x + y) >> 1; if (run[mid] != kEmptyKey) x = mid + 1; else y = mid; }
        s_len[r] = x;
    }
    __syncthreads();
    int merged = 0;
    for (int r = 0; r < world; ++r) merged += s_len[r];
    for (int i = threadIdx.x; i < world * k; i += blockDim.x) {
        const int r = i / k, j = i - r * k;
        if (j >= s_len[r]) continue;
        const u64 key = keys_all[((size_t)r * nq + q) * k + j];
        const uint32_t w = (uint32_t)(key >> 32);
        int pos = j;
        for (int p = 0; p < world && pos < k; ++p) {
            if (p == r) continue;
            const u64* run = keys_all + ((size_t)p * nq + q) * k;
            int x = 0, y = s_len[p];
            if (p < r) {
                while (x < y) { const int mid = (x + y) >> 1; if ((uint32_t)(run[mid] >> 32) <= w) x = mid + 1; else y = mid; }
            } else {
                while (x < y) { const int mid = (x + y) >> 1; if ((uint32_t)(run[mid] >> 32) < w) x = mid + 1; else y = mid; }
            }
            pos += x;
        }
        if (pos < k) flat_decode_key(key, order_max, dist_mode, out_dist + q * k + pos, out_ids + q * k + pos);
    }
    for (int j = merged + threadIdx.x; j < k; j += blockDim.x) {
        out_dist[q * k + j] = __int_as_float(0x7fc00000);
        out_ids[q * k + j] = -1;
    }
}

// a rank's fused flat top-k (raw scores, local rows, -1 padding) -> keys (score word, user id of the row; row_ids == nullptr:
// the row itself) for slot `rank` of every destination, as pack_result_keys_kernel
__global__ void pack_flat_keys_kernel(const float* __restrict__ score, const int64_t* __restrict__ rows,
                                      const int64_t* __restrict__ row_ids, int64_t total, int order_max,
                                      void* const* __restrict__ peer_base, int world, size_t off, u64* __restrict__ local_only) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const int64_t r = rows[i];
    const u64 key = r < 0 ? kEmptyKey : make_key(score[i], (uint32_t)(row_ids ? row_ids[r] : r), order_max);
    if (local_only) { local_only[i] = key; return; }
    for (int p = 0; p < world; ++p) reinterpret_cast<u64*>(static_cast<char*>(peer_base[p]) + off)[i] = key;
}

// the low word of every key of the sorted rows (lims [nq + 1]) from local row to user id; the order stays (one CTA per row)
__global__ void __launch_bounds__(256)
relabel_rows_kernel(u64* __restrict__ keys, const int64_t* __restrict__ lims, int64_t nq, const int64_t* __restrict__ row_ids) {
    for (int64_t q = blockIdx.x; q < nq; q += gridDim.x)
        for (int64_t i = lims[q] + threadIdx.x; i < lims[q + 1]; i += blockDim.x) {
            const u64 key = keys[i];
            keys[i] = (key & 0xFFFFFFFF00000000ull) | (uint32_t)row_ids[(uint32_t)key];
        }
}

// flag += queries whose merged row (the sum of the ranks' trimmed rows, lims_all as above) is shorter than k although their
// bound is finite
__global__ void shard_knn_short_kernel(const int64_t* __restrict__ lims_all, int world, int64_t nq, int k,
                                       const uint32_t* __restrict__ bound, unsigned long long* __restrict__ flag) {
    const int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= nq) return;
    int64_t len = 0;
    for (int r = 0; r < world; ++r) len += lims_all[(size_t)r * (nq + 2) + q + 1] - lims_all[(size_t)r * (nq + 2) + q];
    if (len < k && bound[q] != 0xFFFFFFFFu) atomicAdd(flag, 1ull);
}

// The ranks' k-NN seed bounds over peer memory: tau [nq] -> slot `rank` of the bound slice [world][stride] of every rank's
// range region (this rank's included); after a barrier, tau = the minimum of the slots here.  The minimum is unsigned: the
// key words order like the distances (make_key), NaN's word being the largest.
__global__ void push_knn_bounds_kernel(const uint32_t* __restrict__ tau, int64_t nq, void* const* __restrict__ peer_base,
                                       int world, size_t off) {
    for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < nq; q += (int64_t)gridDim.x * blockDim.x) {
        const uint32_t v = tau[q];
        for (int p = 0; p < world; ++p) reinterpret_cast<uint32_t*>(static_cast<char*>(peer_base[p]) + off)[q] = v;
    }
}
__global__ void min_knn_bounds_kernel(const uint32_t* __restrict__ slots, int world, int64_t stride, int64_t nq,
                                      uint32_t* __restrict__ tau) {
    const int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= nq) return;
    uint32_t v = 0xFFFFFFFFu;
    for (int r = 0; r < world; ++r) v = min(v, slots[(size_t)r * stride + q]);
    tau[q] = v;
}

// lims_all [world][nq + 2] on the device -> glims [nq + 1] (device) and meta (host: base [world + 1], longest row, statuses
// [world]).  Synchronises the stream: the size of the global answer.
int shard_range_lims(const int64_t* lims_all, int world, int64_t nq, int64_t* glims, std::vector<int64_t>& meta) {
    cudaStream_t s = ctx().stream;
    Scratch<int64_t> dmeta;
    const size_t nm = 2 * (size_t)world + 2;
    VIX_TRY(dmeta.alloc(nm));
    VIX_CUDA(cudaMemsetAsync(dmeta.ptr, 0, nm * 8, s));
    const int64_t want = (nq + 1 + 255) / 256;
    const unsigned grid = (unsigned)(want < (int64_t)num_sms() * 4 ? want : (int64_t)num_sms() * 4);
    shard_range_lims_kernel<<<grid, 256, 0, s>>>(lims_all, world, nq, glims, dmeta.ptr);
    VIX_LAUNCH_CHECK();
    meta.assign(nm, 0);
    VIX_CUDA(cudaMemcpyAsync(meta.data(), dmeta.ptr, nm * 8, cudaMemcpyDeviceToHost, s));
    VIX_CUDA(cudaStreamSynchronize(s));
    return VIX_OK;
}

static int shard_range_merge(const u64* keys, const int64_t* base_dev, const int64_t* lims_all, int world, int64_t nq,
                             const int64_t* glims, int64_t total, int neg_zero, vix_range_result* r) {
    cudaStream_t s = ctx().stream;
    VIX_CUDA(cudaMemcpyAsync(r->lims, glims, (size_t)(nq + 1) * 8, cudaMemcpyDeviceToDevice, s));
    if (total == 0) return VIX_OK;
    const int64_t want = (total + 255) / 256;
    const unsigned grid = (unsigned)(want < (int64_t)num_sms() * 8 ? want : (int64_t)num_sms() * 8);
    shard_range_merge_kernel<<<grid, 256, 0, s>>>(keys, base_dev, lims_all, world, nq, glims, total, neg_zero, r->dist, r->ids);
    VIX_LAUNCH_CHECK();
    return VIX_OK;
}

static int shard_knn_merge(const u64* keys, const int64_t* base_dev, const int64_t* lims_all, int world, int64_t nq,
                           const int64_t* glims, int64_t total, int k, int neg_zero, float* out_dist, int64_t* out_ids) {
    const int64_t want = (std::max<int64_t>(total, nq * (int64_t)k) + 255) / 256;
    const unsigned grid = (unsigned)(want < (int64_t)num_sms() * 8 ? want : (int64_t)num_sms() * 8);
    shard_knn_merge_kernel<<<grid, 256, 0, ctx().stream>>>(keys, base_dev, lims_all, world, nq, glims, total, k, neg_zero,
                                                           out_dist, out_ids);
    VIX_LAUNCH_CHECK();
    return VIX_OK;
}

// the flat kind's merge of the ranks' CSR runs (shard_flat_merge_kernel; k == 0: whole rows at glims)
static int shard_flat_merge(const u64* keys, const int64_t* base_dev, const int64_t* lims_all, int world, int64_t nq,
                            const int64_t* glims, int64_t total, int k, int metric, float* out_dist, int64_t* out_ids) {
    const KnnDecode dec = flat_knn_decode(metric);
    const int64_t want = (std::max<int64_t>(total, nq * (int64_t)k) + 255) / 256;
    if (want == 0) return VIX_OK;
    const unsigned grid = (unsigned)(want < (int64_t)num_sms() * 8 ? want : (int64_t)num_sms() * 8);
    shard_flat_merge_kernel<<<grid, 256, 0, ctx().stream>>>(keys, base_dev, lims_all, world, nq, glims, total, k, dec.order_max,
                                                            dec.dist_mode, out_dist, out_ids);
    VIX_LAUNCH_CHECK();
    return VIX_OK;
}

// the flat kind's merge of k <= VIX_MAX_K: keys_all [world][nq][k] -> out [nq x k]
static int merge_flat_keys(const u64* keys_all, int world, int64_t nq, int k, int metric, float* out_dist, int64_t* out_ids) {
    if (nq == 0) return VIX_OK;
    const KnnDecode dec = flat_knn_decode(metric);
    merge_flat_keys_kernel<<<(unsigned)nq, 256, (size_t)world * 4, ctx().stream>>>(keys_all, world, nq, k, dec.order_max,
                                                                                  dec.dist_mode, out_dist, out_ids);
    VIX_LAUNCH_CHECK();
    return VIX_OK;
}

// The sign one GPU gives a zero distance (the keys hold +0): k-NN of the IVF-PQ scan with inner product -0, of the IVF-Flat
// scan +0 (it keys the distance itself); the flat engine's mapping (flat_knn_decode) restores its own.  Range search: the
// flat engine's and the IVF-PQ scan's inner product -0, IVF-Flat +0.
int knn_neg_zero(const vix_index* h) { return h->p.kind == VIX_INDEX_IVF_PQ && h->p.metric == VIX_METRIC_IP; }
int range_neg_zero(const vix_index* h) { return h->p.kind != VIX_INDEX_IVF_FLAT && h->p.metric == VIX_METRIC_IP; }

const char* kind_name(const vix_index* h) {
    return h->p.kind == VIX_INDEX_FLAT ? "flat" : h->p.kind == VIX_INDEX_IVF_FLAT ? "ivfflat" : "ivfpq";
}

// What a sharded call needs of the handle, checked on every rank before any exchange: an IVF-PQ index trained, with L2 / IP
// (the messages and codes of the IVF-PQ-only layout); an IVF-Flat index with coarse centroids (the sharded layout files
// every row into its list: there is no "rows wait for optimize()" state); a flat index as it is.
static int sharded_kind_check(const vix_index* h, const char* who) {
    if (h->p.kind == VIX_INDEX_IVF_PQ) {
        VIX_REQUIRE(h->has_coarse && h->has_pq, VIX_ERR_NOT_TRAINED, "%s: needs a trained IVF-PQ index", who);
        VIX_REQUIRE(h->p.metric != VIX_METRIC_COSINE, VIX_ERR_UNSUPPORTED, "%s: L2 / IP only", who);
    } else if (h->p.kind == VIX_INDEX_IVF_FLAT) {
        VIX_REQUIRE(h->has_coarse, VIX_ERR_NOT_TRAINED, "%s: an IVF-Flat index needs its coarse centroids (set or trained) "
                    "before it is sharded", who);
    }
    return VIX_OK;
}

static void close_range_peers(vix_comm* c) {
    for (int p = 0; p < (int)c->range_peer.size(); ++p)
        if (p != c->rank && c->range_peer[p]) cudaIpcCloseMemHandle(c->range_peer[p]);
    c->range_peer.clear();
    if (c->range_local) cudaFree(c->range_local);
    c->range_local = nullptr;
    if (c->range_peer_dev) cudaFree(c->range_peer_dev);
    c->range_peer_dev = nullptr;
    c->range_cap_nq = c->range_cap_keys = 0;
}

// Collective (peer memory only): make every rank's range region hold nq rows of lims and `keys` keys, growing it
// geometrically.  Every rank passes the same (nq, keys) -- the batch, and the global total all ranks computed -- so they
// agree on whether to grow.  A rank that cannot allocate or map makes every rank return VIX_ERR_OOM with no region left.
int ensure_range_region(vix_comm* c, int64_t nq, int64_t keys, bool* grown) {
    if (c->range_local && nq <= c->range_cap_nq && keys <= c->range_cap_keys) return VIX_OK;
    cudaStream_t s = ctx().stream;
    const int world = c->world;
    int64_t cnq = c->range_cap_nq > 1024 ? c->range_cap_nq : 1024;
    while (cnq < nq) cnq *= 2;
    int64_t ck = c->range_cap_keys > 65536 ? c->range_cap_keys : 65536;
    if (ck < keys) ck = keys + keys / 8 > 2 * ck ? keys + keys / 8 : 2 * ck;
    const size_t off_b = ((size_t)world * (cnq + 2) * 8 + 255) & ~(size_t)255;
    const size_t off_k = (off_b + (size_t)world * cnq * 4 + 255) & ~(size_t)255;
    const size_t total = off_k + (size_t)ck * 8;
    VIX_CUDA(cudaStreamSynchronize(s));                                   // nothing of mine still reads or writes the old one
    void* fresh = nullptr;
    int ok = 1;
    cudaIpcMemHandle_t mine;
    memset(&mine, 0, sizeof(mine));
    if (cudaMalloc(&fresh, total) != cudaSuccess) { cudaGetLastError(); ok = 0; fresh = nullptr; }
    if (ok && cudaIpcGetMemHandle(&mine, fresh) != cudaSuccess) { cudaGetLastError(); ok = 0; }
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
    close_range_peers(c);                                                 // every rank has drained its stream
    int all_ok = 1;
    for (int p = 0; p < world; ++p) all_ok &= all[p].ok;
    std::vector<void*> peer((size_t)world, nullptr);
    for (int p = 0; p < world && all_ok; ++p) {
        if (p == c->rank) { peer[p] = fresh; continue; }
        if (cudaIpcOpenMemHandle(&peer[p], all[p].h, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) {
            cudaGetLastError();
            peer[p] = nullptr;
            all_ok = 0;
        }
    }
    void** pdev = nullptr;
    if (all_ok && cudaMalloc(reinterpret_cast<void**>(&pdev), sizeof(void*) * world) != cudaSuccess) { cudaGetLastError(); all_ok = 0; }
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
        if (pdev) cudaFree(pdev);
        VIX_REQUIRE(false, VIX_ERR_OOM, "vix_sharded_range_search: a rank could not allocate or map a range region of %zu bytes "
                    "(%lld rows, %lld keys)", total, (long long)cnq, (long long)ck);
    }
    VIX_CUDA(cudaMemcpyAsync(pdev, peer.data(), sizeof(void*) * world, cudaMemcpyHostToDevice, s));
    VIX_CUDA(cudaStreamSynchronize(s));
    c->range_local = fresh; c->range_peer = peer; c->range_peer_dev = pdev;
    c->range_off_bounds = off_b; c->range_off_keys = off_k; c->range_cap_nq = cnq; c->range_cap_keys = ck;
    *grown = true;
    return VIX_OK;
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
    close_range_peers(c);
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

}  // extern "C"

namespace vix {

// Steps 1-3 of a sharded call: this rank's block of the batch gets its probe lists against ALL centroids, and the block
// (probes, plus the queries when they came from the host) reaches every rank -- stored into every peer's region with one
// barrier, or an NCCL all-gather.  On return px.queries / px.probes are the whole batch's queries and probe lists on the
// device.  The caller holds both mutexes and has called ensure_region.
// A flat index has no probes (px.probes stays null): only the queries travel, and over peer memory the barrier still
// comes first -- it is what orders this call's stores into the peers' regions (the result slab, the range region) after
// every peer's reads of them in the previous call.
struct BatchProbes {
    In<float> dq;
    const float* queries = nullptr;
    const int32_t* probes = nullptr;
};

static int exchange_probes(vix_index* h, vix_comm* c, const float* queries, int64_t nq, int nprobe, BatchProbes& px) {
    cudaStream_t s = ctx().stream;
    const int world = c->world, rank = c->rank, d = h->p.d;
    const bool host_q = !is_device_ptr(queries);
    const int64_t per = block_rows(nq, world);
    const int64_t lo = nq < (int64_t)rank * per ? nq : (int64_t)rank * per;
    const int64_t cnt = (nq < lo + per ? nq : lo + per) - lo;
    const bool flat = h->p.kind == VIX_INDEX_FLAT;
    if (flat) nprobe = 0;
    if (c->peer_state == 1) {
        char* base = static_cast<char*>(c->local);
        float* qbuf = reinterpret_cast<float*>(base + c->off_queries);          // [world * per][d] (this call's per)
        int32_t* pbuf = reinterpret_cast<int32_t*>(base + c->off_probes);       // [world * per][nprobe]
        // 1. this rank's block of the batch: host queries cross PCIe once per rank, 1/world of the batch each
        const float* qblock = queries + (size_t)lo * d;
        if (host_q && cnt > 0) {
            VIX_CUDA(cudaMemcpyAsync(qbuf + (size_t)lo * d, qblock, (size_t)cnt * d * 4, cudaMemcpyHostToDevice, s));
            qblock = qbuf + (size_t)lo * d;
        }
        // 2. its probe lists against ALL centroids (the selection of index_search_locked: cosine or fast, by the metric),
        //    straight into slot `rank` of the local probe buffer
        int32_t* pblock = pbuf + (size_t)rank * per * nprobe;
        if (!flat && cnt > 0) VIX_TRY(select_probes_device(h, qblock, cnt, nprobe, pblock));
        if (!flat && cnt < per) VIX_TRY(fill<int32_t>(pblock + (size_t)cnt * nprobe, (per - cnt) * nprobe, -1));
        // 3. the block travels to every peer (probes, and the queries when they came from the host), one barrier
        const size_t offA = c->off_probes + (size_t)rank * per * nprobe * 4, nA = (size_t)per * nprobe * 4 / 16;
        const size_t offB = c->off_queries + (size_t)rank * per * d * 4, nB = host_q ? (size_t)per * d * 4 / 16 : 0;
        const size_t n16 = nA + nB;
        const size_t want = (n16 + 255) / 256;
        const unsigned grid = (unsigned)(want < (size_t)(2 * num_sms()) ? (want ? want : 1) : (size_t)(2 * num_sms()));
        peer_push_kernel<<<grid, 256, 0, s>>>(c->peer_dev, world, rank, offA, nA, offB, nB);
        VIX_LAUNCH_CHECK();
        VIX_TRY(peer_barrier(c));
        px.queries = host_q ? qbuf : queries;
        px.probes = flat ? nullptr : pbuf;
        return VIX_OK;
    }
    // NCCL carries the exchange
    VIX_TRY(px.dq.stage(queries, (size_t)nq * d));
    px.queries = px.dq.dev;
    if (flat) return VIX_OK;
    const size_t pbytes = (size_t)world * per * nprobe * 4;
    if (pbytes > c->gather_probes_bytes) {
        if (c->gather_probes) { VIX_CUDA(cudaStreamSynchronize(s)); cudaFree(c->gather_probes); c->gather_probes = nullptr; }
        VIX_CUDA(cudaMalloc(&c->gather_probes, pbytes));
        c->gather_probes_bytes = pbytes;
    }
    int32_t* pall = static_cast<int32_t*>(c->gather_probes);
    int32_t* pblock = pall + (size_t)rank * per * nprobe;
    if (cnt > 0) VIX_TRY(select_probes_device(h, px.dq.dev + (size_t)lo * d, cnt, nprobe, pblock));
    if (cnt < per) VIX_TRY(fill<int32_t>(pblock + (size_t)cnt * nprobe, (per - cnt) * nprobe, -1));
    VIX_NCCL(g_nccl.AllGather(pblock, pall, (size_t)per * nprobe, ncclInt32, c->comm, s));   // in place
    px.queries = px.dq.dev;
    px.probes = pall;
    return VIX_OK;
}

// filter arguments of the C ABI -> FilterArgs over a staged copy of the words (f == nullptr when there is no filter)
int stage_filter(const uint64_t* words, int64_t capacity, int mode, In<uint64_t>& staged, FilterArgs& f,
                        const FilterArgs*& fp) {
    fp = nullptr;
    if (!words) return VIX_OK;
    VIX_TRY(staged.stage(words, (size_t)((capacity + 63) / 64)));
    f.words = staged.dev; f.cap = capacity; f.deny = mode == VIX_FILTER_DENY;
    fp = &f;
    return VIX_OK;
}

// A rank's pass of k <= VIX_MAX_K over what it holds, packed as keys for slot `rank` of every destination (peer_base, off)
// or into local_only [nq x k].  IVF kinds: the fused scan over the probed lists the rank owns (a filter sends it down the
// query-major path), keys (API distance, id).  Flat: the fused flat search over the rank's rows with raw scores, keys
// (score word in the metric's order, user id of the row) -- merged by merge_flat_keys_kernel, never on the full key.
// scanned (nullable): an event recorded between the scan and the pack (the trace's phase boundary).
static int local_knn_keys(vix_index* h, const float* dq, int64_t nq, int k, int nprobe, const int32_t* probes,
                          const FilterArgs* filter, void* const* peer_base, int world, size_t off, u64* local_only,
                          cudaEvent_t scanned = nullptr) {
    cudaStream_t s = ctx().stream;
    const int64_t total = nq * (int64_t)k;
    Scratch<float> ldist;
    Scratch<int64_t> lids;
    VIX_TRY(ldist.alloc((size_t)total));
    VIX_TRY(lids.alloc((size_t)total));
    const unsigned grid = (unsigned)((total + 255) / 256);
    if (h->p.kind == VIX_INDEX_FLAT) {
        const int d = h->p.d, metric = h->p.metric;
        Scratch<uint64_t> mask;
        VIX_TRY(filter_row_mask(h, filter, mask));
        if (mask.ptr) VIX_TRY(flat_search_masked_device(dq, nq, h->vecs.ptr, h->n, d, metric, k, mask.ptr, ldist.ptr, lids.ptr, true));
        else VIX_TRY(flat_search_auto_device(dq, nq, h->vecs.ptr, h->n, d, metric, k, nullptr, ldist.ptr, lids.ptr, true));
        if (scanned) VIX_CUDA(cudaEventRecord(scanned, s));
        pack_flat_keys_kernel<<<grid, 256, 0, s>>>(ldist.ptr, lids.ptr, h->ids.ptr, total, metric != VIX_METRIC_L2, peer_base, world,
                                                   off, local_only);
    } else {
        VIX_TRY(index_search_locked(h, dq, nq, k, nprobe, ldist.ptr, lids.ptr, nullptr, nullptr, probes, filter));
        if (scanned) VIX_CUDA(cudaEventRecord(scanned, s));
        pack_result_keys_kernel<<<grid, 256, 0, s>>>(ldist.ptr, lids.ptr, total, peer_base, world, off, local_only);
    }
    VIX_LAUNCH_CHECK();
    return VIX_OK;
}

// the merge of k <= VIX_MAX_K over the gathered keys [world][nq][k], by kind
static int merge_knn_keys(const vix_index* h, const u64* keys_all, int world, int64_t nq, int k, float* out_dist, int64_t* out_ids) {
    if (h->p.kind == VIX_INDEX_FLAT) return merge_flat_keys(keys_all, world, nq, k, h->p.metric, out_dist, out_ids);
    return merge_shard_keys(keys_all, world, nq, k, knn_neg_zero(h), out_dist, out_ids);
}

// The rank-local halves of k > VIX_MAX_K (sharded_knn_large, and the one-GPU emulation of the ranks): the seed -> tau_r;
// then, with the ranks' minimum, the collect within it and every sorted row cut at k.  IVF kinds: the kind's range scan
// over the probe prefix of the lists the rank owns / over every probed list, keys (API distance, id).  Flat: the flat
// engine's seed blocks and range kernel over the rank's rows, keys (score word, row), the cut rows relabelled to user ids
// in place (their order stays: the word, then the row).
struct LocalKnnLarge {
    IvfRangeScan scan;
    Scratch<int32_t> prefix;
    Scratch<uint64_t> mask;
    FlatKnnPass flat;
    std::function<int(const RangeOut&)> seed, collect;
    size_t seed_cap = 0, max_entries = 0;
};

static int local_knn_prepare(vix_index* h, const float* dq, int64_t nq, int k, int nprobe, const int32_t* probes,
                             const FilterArgs* filter, LocalKnnLarge& L) {
    if (h->p.kind == VIX_INDEX_FLAT) {
        VIX_TRY(filter_row_mask(h, filter, L.mask));
        VIX_TRY(flat_knn_pass(dq, nq, h->vecs.ptr, h->n, h->p.d, h->p.metric, k, L.mask.ptr, L.flat));
        L.seed = L.flat.seed;
        L.collect = L.flat.collect;
        L.seed_cap = L.flat.seed_cap;
        L.max_entries = L.flat.max_entries;
        return VIX_OK;
    }
    VIX_TRY(ivf_range_scan(h, dq, nq, nprobe, probes, filter, L.scan));
    VIX_TRY(L.prefix.alloc((size_t)nq * nprobe));
    VIX_TRY(knn_probe_prefix(probes, nq, nprobe, h->list_len.ptr, h->kc, k, L.prefix.ptr, &L.seed_cap, &L.max_entries));
    IvfRangeScan* sc = &L.scan;
    const int32_t* pre = L.prefix.ptr;
    L.seed = [sc, pre](const RangeOut& o) { return sc->run(pre, o); };
    L.collect = [sc, probes](const RangeOut& o) { return sc->run(probes, o); };
    return VIX_OK;
}

static int local_knn_seed(LocalKnnLarge& L, int64_t nq, int k, uint32_t* tau, int64_t* seed_n) {
    return knn_seed_bound(nq, k, L.seed_cap, L.seed ? &L.seed : nullptr, tau, seed_n);
}

static int local_knn_cut(vix_index* h, LocalKnnLarge& L, int64_t nq, int k, const uint32_t* tau, size_t& cap, RangeKeys& rk,
                         RangeKeys& cut, RangeInfo* ci) {
    VIX_TRY(knn_collect(nq, k, tau, L.collect, L.max_entries, cap, rk, ci, nullptr));
    VIX_TRY(knn_trim(nq, k, rk, cut));
    if (h->p.kind == VIX_INDEX_FLAT && cut.sorted) {
        const unsigned grid = (unsigned)std::min<int64_t>((int64_t)num_sms() * 8, nq);
        relabel_rows_kernel<<<grid, 256, 0, ctx().stream>>>(cut.sorted, cut.lims.ptr, nq, h->ids.ptr);
        VIX_LAUNCH_CHECK();
    }
    return VIX_OK;
}

// forward: k > VIX_MAX_K at world > 1 (below)
static int sharded_knn_large(vix_index* h, vix_comm* c, const float* queries, int64_t nq, int k, int nprobe,
                             const FilterArgs* filter, float* out_dist, int64_t* out_ids);

// vix_sharded_search and vix_sharded_search_filtered (filter == nullptr: the unfiltered step, launch for launch; k above
// VIX_MAX_K at world > 1: sharded_knn_large).  A flat index has no probes: phase 1 is empty and every rank searches its rows.
static int sharded_search(vix_index* h, vix_comm* c, const float* queries, int64_t nq, int k, int nprobe, const FilterArgs* filter,
                          float* out_dist, int64_t* out_ids) {
    std::lock_guard<std::mutex> lc(c->mu);
    std::lock_guard<std::mutex> lk(h->mu);
    VIX_TRY(sharded_kind_check(h, "vix_sharded_search"));
    const bool flat = h->p.kind == VIX_INDEX_FLAT;
    if (!flat) {
        if (nprobe <= 0) nprobe = h->p.nprobe;
        VIX_REQUIRE(nprobe > 0 && nprobe <= VIX_MAX_K, VIX_ERR_INVALID_K, "vix_sharded_search: nprobe");
    }
    const int world = c->world, rank = c->rank, d = h->p.d;
    if (world == 1) return index_search_locked(h, queries, nq, k, nprobe, out_dist, out_ids, nullptr, nullptr, nullptr, filter);
    if (!flat && h->dirty) VIX_TRY(build_lists(h));
    if (k > VIX_MAX_K) return sharded_knn_large(h, c, queries, nq, k, nprobe, filter, out_dist, out_ids);
    cudaStream_t s = ctx().stream;
    VIX_TRY(ensure_region(c, nq, d, flat ? 1 : nprobe, k));
    // the list-major scan's bounds over the ranks (only an IVF-PQ index can take that scan; cleared again on every way out)
    std::optional<ThrHookScope> thr_scope;
    if (h->p.kind == VIX_INDEX_IVF_PQ) thr_scope.emplace(c);
    const int64_t total = nq * (int64_t)k;
    Out<float> dd;
    Out<int64_t> di;
    VIX_TRY(dd.stage(out_dist, (size_t)total));
    VIX_TRY(di.stage(out_ids, (size_t)total));
    auto mark = [&](int i) { if (c->trace) cudaEventRecord(c->ev[i], s); };
    mark(0);
    // 1-3. probes of this rank's block, exchanged (flat: the queries only)
    BatchProbes px;
    VIX_TRY(exchange_probes(h, c, queries, nq, nprobe, px));
    const float* dq = px.queries;
    const int32_t* probes = px.probes;
    mark(1);
    // 4-5. the local pass; its top-k leaves as packed keys for slot `rank` of every rank's result buffer; barrier (or
    //      all-gather); merge
    if (c->peer_state == 1) {
        u64* rbuf = reinterpret_cast<u64*>(static_cast<char*>(c->local) + c->off_results);   // [world][nq][k]
        VIX_TRY(local_knn_keys(h, dq, nq, k, nprobe, probes, filter, c->peer_dev, world, c->off_results + (size_t)rank * total * 8,
                               nullptr, c->trace ? c->ev[2] : nullptr));
        VIX_TRY(peer_barrier(c));
        VIX_TRY(merge_knn_keys(h, rbuf, world, nq, k, dd.dev, di.dev));
    } else {
        const size_t kbytes = (size_t)world * total * 8;
        if (kbytes > c->gather_keys_bytes) {
            if (c->gather_keys) { VIX_CUDA(cudaStreamSynchronize(s)); cudaFree(c->gather_keys); c->gather_keys = nullptr; }
            VIX_CUDA(cudaMalloc(&c->gather_keys, kbytes));
            c->gather_keys_bytes = kbytes;
        }
        u64* kall = static_cast<u64*>(c->gather_keys);
        VIX_TRY(local_knn_keys(h, dq, nq, k, nprobe, probes, filter, nullptr, world, 0, kall + (size_t)rank * total,
                               c->trace ? c->ev[2] : nullptr));
        VIX_NCCL(g_nccl.AllGather(kall + (size_t)rank * total, kall, (size_t)total, ncclUint64, c->comm, s));
        VIX_TRY(merge_knn_keys(h, kall, world, nq, k, dd.dev, di.dev));
    }
    mark(3);
    VIX_TRY(dd.commit());
    VIX_TRY(di.commit());
    return finish(dd.is_host() || di.is_host());
}


// The step after each rank's local pass: its sorted keys and lims (rc: its status) -> every rank's lims and status (peer
// region + barrier, or all-gather) -> global row starts and total (synchronises) -> the keys of every rank (peer region +
// barrier, or grouped send / receive) -> merge, then the tail's last step.
int sharded_range_exchange(vix_index* h, vix_comm* c, int64_t nq, int rc, RangeKeys& rk, bool grown, const ShardTail& t,
                                  ShardTotals* st) {
    cudaStream_t s = ctx().stream;
    const int world = c->world, rank = c->rank;
    const int64_t L = nq + 2;
    const bool peer = c->peer_state == 1;
    const bool knn = t.out == nullptr;
    const char* who = t.concat ? "vix_replicated_range_search" : knn ? "vix_sharded_search" : "vix_sharded_range_search";
    Scratch<int64_t> mine, lims_all, glims, dbase;
    VIX_TRY(mine.alloc((size_t)L));
    VIX_TRY(lims_all.alloc((size_t)world * L));
    VIX_TRY(glims.alloc((size_t)nq + 1));
    VIX_TRY(dbase.alloc((size_t)world + 1));
    // this rank's lims and status (a rank whose local pass failed sends empty rows and its code)
    const int64_t status = rc;
    if (rc == VIX_OK) VIX_CUDA(cudaMemcpyAsync(mine.ptr, rk.lims.ptr, (size_t)(nq + 1) * 8, cudaMemcpyDeviceToDevice, s));
    else VIX_CUDA(cudaMemsetAsync(mine.ptr, 0, (size_t)(nq + 1) * 8, s));
    VIX_CUDA(cudaMemcpyAsync(mine.ptr + nq + 1, &status, 8, cudaMemcpyHostToDevice, s));
    if (peer) {
        const int64_t want = (L + 255) / 256;
        peer_store_kernel<<<(unsigned)(want < 64 ? want : 64), 256, 0, s>>>(reinterpret_cast<const u64*>(mine.ptr), L,
                                                                           c->range_peer_dev, world, (size_t)rank * L * 8);
        VIX_LAUNCH_CHECK();
        VIX_TRY(peer_barrier(c));
        VIX_CUDA(cudaMemcpyAsync(lims_all.ptr, c->range_local, (size_t)world * L * 8, cudaMemcpyDeviceToDevice, s));
    } else {
        VIX_NCCL(g_nccl.AllGather(mine.ptr, lims_all.ptr, (size_t)L, ncclInt64, c->comm, s));
    }
    // k-NN: rows shorter than k within a finite bound, counted from the row starts every rank now holds (read in the
    // synchronisation of shard_range_lims)
    Scratch<unsigned long long> dshort;
    unsigned long long short_rows = 0;
    if (knn) {
        VIX_TRY(dshort.alloc(1));
        VIX_CUDA(cudaMemsetAsync(dshort.ptr, 0, 8, s));
        shard_knn_short_kernel<<<(unsigned)((nq + 255) / 256), 256, 0, s>>>(lims_all.ptr, world, nq, t.k, t.bound, dshort.ptr);
        VIX_LAUNCH_CHECK();
        VIX_CUDA(cudaMemcpyAsync(&short_rows, dshort.ptr, 8, cudaMemcpyDeviceToHost, s));
    }
    std::vector<int64_t> meta;
    VIX_TRY(shard_range_lims(lims_all.ptr, world, nq, glims.ptr, meta));    // the second synchronisation: the global total
    if (rc != VIX_OK) return rc;                                          // (its own message stands)
    for (int p = 0; p < world; ++p)
        VIX_REQUIRE(meta[world + 2 + p] == VIX_OK, (int)meta[world + 2 + p], "%s: rank %d failed its local "
                    "scan (status %lld); no rank returns a result", who, p, (long long)meta[world + 2 + p]);
    // (every rank holds the same row starts and bounds, so every rank refuses here together)
    VIX_REQUIRE(short_rows == 0, VIX_ERR_CONTRACT, "%s (k = %d): %llu queries merged fewer than k entries within the bound "
                "the ranks' seed passes found", who, t.k, short_rows);
    const int64_t total = meta[world], max_row = meta[world + 1];
    // room for the answer on every rank, decided together
    if (peer) VIX_TRY(ensure_range_region(c, nq, total, &grown));
    vix_range_result* r = nullptr;
    Scratch<u64> kall;
    int ok = knn ? 1 : range_alloc(nq, total, &r) == VIX_OK;
    if (ok && !peer && kall.alloc((size_t)total) != VIX_OK) ok = 0;
    {
        Scratch<int> dflag;
        int rc2 = dflag.alloc(1);
        if (rc2 == VIX_OK) rc2 = cudaMemcpyAsync(dflag.ptr, &ok, 4, cudaMemcpyHostToDevice, s) == cudaSuccess ? VIX_OK : VIX_ERR_CUDA;
        if (rc2 == VIX_OK) rc2 = g_nccl.AllReduce(dflag.ptr, dflag.ptr, 1, ncclInt32, ncclMin, c->comm, s) == ncclSuccess ? VIX_OK : VIX_ERR_CUDA;
        if (rc2 == VIX_OK) rc2 = cudaMemcpyAsync(&ok, dflag.ptr, 4, cudaMemcpyDeviceToHost, s) == cudaSuccess ? VIX_OK : VIX_ERR_CUDA;
        if (rc2 == VIX_OK) rc2 = cudaStreamSynchronize(s) == cudaSuccess ? VIX_OK : VIX_ERR_CUDA;
        if (rc2 != VIX_OK || !ok) {
            range_free(r);
            VIX_REQUIRE(rc2 == VIX_OK, rc2, "%s: the allocation verdict failed", who);
            VIX_REQUIRE(false, VIX_ERR_OOM, "%s: %lld results (%lld bytes) do not fit in device memory on "
                        "every rank", who, (long long)total, (long long)total * (knn ? 8 : 12));
        }
    }
    auto fail = [&](int e) { range_free(r); return e; };
    const int64_t mine_n = meta[rank + 1] - meta[rank];
    const u64* keys = nullptr;
    if (cudaMemcpyAsync(dbase.ptr, meta.data(), ((size_t)world + 1) * 8, cudaMemcpyHostToDevice, s) != cudaSuccess)
        return fail(cuda_fail(cudaGetLastError(), "range base copy", __FILE__, __LINE__));
    if (peer) {
        // every store into a peer's region is behind this call's probe barrier, which the peer entered after its previous
        // merge had read the region
        if (mine_n > 0) {
            const int64_t want = (mine_n + 255) / 256;
            peer_store_kernel<<<(unsigned)(want < (int64_t)num_sms() * 4 ? want : (int64_t)num_sms() * 4), 256, 0, s>>>(
                rk.sorted, mine_n, c->range_peer_dev, world, c->range_off_keys + (size_t)meta[rank] * 8);
            ctx().launches += 1;
        }
        const int b = peer_barrier(c);
        if (b != VIX_OK) return fail(b);
        keys = reinterpret_cast<const u64*>(static_cast<char*>(c->range_local) + c->range_off_keys);
    } else {
        if (mine_n > 0 && cudaMemcpyAsync(kall.ptr + meta[rank], rk.sorted, (size_t)mine_n * 8, cudaMemcpyDeviceToDevice, s) != cudaSuccess)
            return fail(cuda_fail(cudaGetLastError(), "range keys copy", __FILE__, __LINE__));
        ncclResult_t nr = g_nccl.GroupStart();
        for (int p = 0; p < world && nr == ncclSuccess; ++p) {
            if (p == rank) continue;
            const int64_t np_ = meta[p + 1] - meta[p];
            if (mine_n > 0) nr = g_nccl.Send(rk.sorted, (size_t)mine_n, ncclUint64, p, c->comm, s);
            if (nr == ncclSuccess && np_ > 0) nr = g_nccl.Recv(kall.ptr + meta[p], (size_t)np_, ncclUint64, p, c->comm, s);
        }
        const ncclResult_t ne = g_nccl.GroupEnd();
        if (nr == ncclSuccess) nr = ne;
        if (nr != ncclSuccess) {
            set_error("NCCL error %d (%s): range keys exchange", (int)nr, g_nccl.GetErrorString(nr));
            return fail(VIX_ERR_CUDA);
        }
        keys = kall.ptr;
    }
    const int mr = t.concat ? replica_range_concat(keys, glims.ptr, nq, total, t.neg_zero, r)
                 : !knn ? shard_range_merge(keys, dbase.ptr, lims_all.ptr, world, nq, glims.ptr, total, t.neg_zero, r)
                 : t.flat_metric >= 0 ? shard_flat_merge(keys, dbase.ptr, lims_all.ptr, world, nq, glims.ptr, total, t.k, t.flat_metric,
                                                          t.dist, t.ids)
                 : shard_knn_merge(keys, dbase.ptr, lims_all.ptr, world, nq, glims.ptr, total, t.k, t.neg_zero, t.dist, t.ids);
    if (mr != VIX_OK) return fail(mr);
    if (getenv("VIX_SCAN_DEBUG") && !knn && !t.concat)
        fprintf(stderr, "[vix sharded range] world %d, peer %d, local %lld, total %lld, max_row %lld, grown %d, kind %s\n", world,
                peer ? 1 : 0, (long long)mine_n, (long long)total, (long long)max_row, grown ? 1 : 0, kind_name(h));
    st->mine = mine_n; st->total = total; st->max_row = max_row; st->grown = grown;
    if (!knn) *t.out = r;
    return VIX_OK;
}

// the ranks' k-NN seed bounds [nq] (device) -> their unsigned minimum, on every rank: peer memory (the bound slice of the
// range region, one barrier) or an NCCL all-reduce
static int bound_min_over_ranks(vix_comm* c, uint32_t* tau, int64_t nq) {
    cudaStream_t s = ctx().stream;
    if (c->peer_state != 1) {
        VIX_NCCL(g_nccl.AllReduce(tau, tau, (size_t)nq, ncclUint32, ncclMin, c->comm, s));
        return VIX_OK;
    }
    const int64_t stride = c->range_cap_nq;
    const int64_t want = (nq + 255) / 256;
    push_knn_bounds_kernel<<<(unsigned)(want < 64 ? want : 64), 256, 0, s>>>(tau, nq, c->range_peer_dev, c->world,
                                                                            c->range_off_bounds + (size_t)c->rank * stride * 4);
    VIX_LAUNCH_CHECK();
    VIX_TRY(peer_barrier(c));
    const uint32_t* slots = reinterpret_cast<const uint32_t*>(static_cast<char*>(c->range_local) + c->range_off_bounds);
    min_knn_bounds_kernel<<<(unsigned)want, 256, 0, s>>>(slots, c->world, stride, nq, tau);
    VIX_LAUNCH_CHECK();
    return VIX_OK;
}

// vix_sharded_search / vix_sharded_search_filtered with VIX_MAX_K < k <= VIX_MAX_K_LARGE and world > 1: the one-GPU two-pass
// route (vix_knn_large.cu) with one bound per query shared by all ranks (see shard_knn_merge_kernel for why it is exact):
//   1. the probes of the batch, exchanged as for every sharded call (flat: none);
//   2. each rank's seed over the probe prefix of the lists it owns (those it does not own have length 0; flat: the flat
//      engine's seed blocks over its rows) -> tau_r;
//   3. tau = the minimum of the tau_r over the ranks;
//   4. each rank's collect within tau over every probed list it owns (flat: its rows), each sorted row cut at k (knn_trim);
//   5. the cut rows exchanged as range search exchanges its rows, merged (flat: by score word and rank), and cut at k.
// A rank whose seed or collect fails still enters every exchange (all-ones bounds, empty rows and its status), so every
// rank returns its code.  Synchronises the stream; the handle's knn_cap is written once the call has succeeded.
static int sharded_knn_large(vix_index* h, vix_comm* c, const float* queries, int64_t nq, int k, int nprobe,
                             const FilterArgs* filter, float* out_dist, int64_t* out_ids) {
    cudaStream_t s = ctx().stream;
    const bool flat = h->p.kind == VIX_INDEX_FLAT;
    VIX_TRY(ensure_region(c, nq, h->p.d, flat ? 1 : nprobe, 1));     // (no [world x nq x k] result slab: k is large)
    bool grown = false;
    if (c->peer_state == 1) VIX_TRY(ensure_range_region(c, nq, 0, &grown));
    Out<float> dd;
    Out<int64_t> di;
    VIX_TRY(dd.stage(out_dist, (size_t)nq * k));
    VIX_TRY(di.stage(out_ids, (size_t)nq * k));
    Scratch<uint32_t> tau;
    VIX_TRY(tau.alloc((size_t)nq));
    auto mark = [&](int i) { if (c->trace) cudaEventRecord(c->ev[i], s); };
    mark(0);
    BatchProbes px;
    VIX_TRY(exchange_probes(h, c, queries, nq, nprobe, px));
    const float* dq = px.queries;
    const int32_t* probes = px.probes;
    mark(1);
    // 2. the local seed -> tau_r
    LocalKnnLarge L;
    int64_t seed_n = 0;
    int rc = local_knn_prepare(h, dq, nq, k, nprobe, probes, filter, L);
    if (rc == VIX_OK) rc = local_knn_seed(L, nq, k, tau.ptr, &seed_n);
    if (rc != VIX_OK) VIX_CUDA(cudaMemsetAsync(tau.ptr, 0xFF, (size_t)nq * 4, s));
    // 3. tau = min over the ranks
    VIX_TRY(bound_min_over_ranks(c, tau.ptr, nq));
    // 4. the local collect within tau, each row cut at k
    RangeKeys rk, cut;
    RangeInfo ci;
    size_t cap = h->knn_cap;
    if (rc == VIX_OK) rc = local_knn_cut(h, L, nq, k, tau.ptr, cap, rk, cut, &ci);
    mark(2);
    // 5. exchange, merge, cut
    ShardTail tail;
    tail.k = k; tail.bound = tau.ptr; tail.dist = dd.dev; tail.ids = di.dev;
    tail.neg_zero = knn_neg_zero(h);
    tail.flat_metric = flat ? h->p.metric : -1;
    ShardTotals st;
    VIX_TRY(sharded_range_exchange(h, c, nq, rc, cut, grown, tail, &st));
    mark(3);
    if (getenv("VIX_SCAN_DEBUG"))
        fprintf(stderr, "[vix sharded knn] world %d, peer %d, k %d, seed %lld, local %lld, sent %lld, total %lld, max_row %lld, "
                "grown %d, kind %s\n", c->world, c->peer_state == 1 ? 1 : 0, k, (long long)seed_n, (long long)ci.total,
                (long long)st.mine, (long long)st.total, (long long)st.max_row, st.grown ? 1 : 0, kind_name(h));
    VIX_TRY(dd.commit());
    VIX_TRY(di.commit());
    VIX_TRY(finish(true));
    h->knn_cap = cap;
    return VIX_OK;
}

// The test hooks' input: the ranks' lims [world][nq + 1] and rows (API distances, ids, concatenated rank by rank) -> the
// exchanged layout (lims [world][nq + 2], status 0), the packed keys, the global row starts and the ranks' key bases, as
// the exchange holds them.
struct DebugShardRuns {
    Scratch<int64_t> dlims, glims, dbase;
    Scratch<u64> keys;
    In<float> dd;
    In<int64_t> di;
    std::vector<int64_t> meta;
    int64_t total = 0;
};

static int debug_shard_runs(const char* who, const int64_t* lims_all, const float* dist_all, const int64_t* ids_all, int world,
                            int64_t nq, DebugShardRuns& in, int flat_order_max = -1) {
    cudaStream_t s = ctx().stream;
    const int64_t L = nq + 2;
    // the ranks' lims [world][nq + 1] -> the exchanged layout [world][nq + 2] (status 0)
    std::vector<int64_t> h_lims((size_t)world * (nq + 1));
    VIX_CUDA(cudaMemcpyAsync(h_lims.data(), lims_all, h_lims.size() * 8, cudaMemcpyDefault, s));
    VIX_CUDA(cudaStreamSynchronize(s));
    std::vector<int64_t> h_all((size_t)world * L, 0);
    int64_t total = 0;
    for (int r = 0; r < world; ++r) {
        const int64_t* lr = h_lims.data() + (size_t)r * (nq + 1);
        VIX_REQUIRE(lr[0] == 0, VIX_ERR_INVALID_PARAM, "%s: rank %d: lims[0] != 0", who, r);
        for (int64_t q = 0; q < nq; ++q)
            VIX_REQUIRE(lr[q + 1] >= lr[q], VIX_ERR_INVALID_PARAM, "%s: rank %d: lims descend", who, r);
        for (int64_t q = 0; q <= nq; ++q) h_all[(size_t)r * L + q] = lr[q];
        total += lr[nq];
    }
    VIX_REQUIRE(total == 0 || (dist_all && ids_all), VIX_ERR_NULL_PTR, "%s: null rows", who);
    VIX_TRY(in.dlims.alloc(h_all.size()));
    VIX_TRY(in.glims.alloc((size_t)nq + 1));
    VIX_TRY(in.dbase.alloc((size_t)world + 1));
    VIX_CUDA(cudaMemcpyAsync(in.dlims.ptr, h_all.data(), h_all.size() * 8, cudaMemcpyHostToDevice, s));
    VIX_TRY(in.dd.stage(dist_all, (size_t)total));
    VIX_TRY(in.di.stage(ids_all, (size_t)total));
    VIX_TRY(in.keys.alloc((size_t)total));
    if (total > 0) {
        if (flat_order_max >= 0)                                          // (raw scores: the flat kind's keys)
            pack_flat_keys_kernel<<<(unsigned)((total + 255) / 256), 256, 0, s>>>(in.dd.dev, in.di.dev, nullptr, total,
                                                                                flat_order_max, nullptr, world, 0, in.keys.ptr);
        else
            pack_result_keys_kernel<<<(unsigned)((total + 255) / 256), 256, 0, s>>>(in.dd.dev, in.di.dev, total, nullptr, world,
                                                                                  0, in.keys.ptr);
        VIX_LAUNCH_CHECK();
    }
    VIX_TRY(shard_range_lims(in.dlims.ptr, world, nq, in.glims.ptr, in.meta));
    VIX_CUDA(cudaMemcpyAsync(in.dbase.ptr, in.meta.data(), ((size_t)world + 1) * 8, cudaMemcpyHostToDevice, s));
    in.total = total;
    return VIX_OK;
}

}  // namespace vix

extern "C" {

int vix_sharded_search(vix_index_t* h, vix_comm_t* c, const float* queries, int64_t nq, int k, int nprobe, float* out_dist,
                       int64_t* out_ids) {
    VIX_TRY(ensure_device());
    VIX_REQUIRE(h && c, VIX_ERR_NULL_PTR, "vix_sharded_search: null handle");
    if (nq <= 0 || k <= 0) return VIX_OK;                             // IVFIndex.swift:866 (every rank sees the same nq, k)
    VIX_REQUIRE(queries && out_dist && out_ids, VIX_ERR_NULL_PTR, "vix_sharded_search: null pointer");
    VIX_REQUIRE(k <= VIX_MAX_K_LARGE, VIX_ERR_INVALID_K, "vix_sharded_search: k > %d", VIX_MAX_K_LARGE);
    VIX_REQUIRE(k <= VIX_MAX_K || nq < 0x7FFFFFFFLL, VIX_ERR_INVALID_PARAM, "vix_sharded_search: k > %d needs nq < 2^31 - 1",
                VIX_MAX_K);
    return sharded_search(h, c, queries, nq, k, nprobe, nullptr, out_dist, out_ids);
}

int vix_sharded_search_filtered(vix_index_t* h, vix_comm_t* c, const float* queries, int64_t nq, int k, int nprobe,
                                const uint64_t* filter_words, int64_t filter_capacity, int filter_mode, float* out_dist,
                                int64_t* out_ids) {
    VIX_TRY(ensure_device());
    VIX_REQUIRE(h && c, VIX_ERR_NULL_PTR, "vix_sharded_search_filtered: null handle");
    VIX_REQUIRE(filter_mode == VIX_FILTER_ALLOW || filter_mode == VIX_FILTER_DENY, VIX_ERR_INVALID_PARAM,
                "vix_sharded_search_filtered: filter_mode must be VIX_FILTER_ALLOW or VIX_FILTER_DENY");
    VIX_REQUIRE(filter_capacity >= 0, VIX_ERR_INVALID_PARAM, "vix_sharded_search_filtered: negative capacity");
    if (nq <= 0 || k <= 0) return VIX_OK;
    VIX_REQUIRE(queries && out_dist && out_ids, VIX_ERR_NULL_PTR, "vix_sharded_search_filtered: null pointer");
    VIX_REQUIRE(k <= VIX_MAX_K_LARGE, VIX_ERR_INVALID_K, "vix_sharded_search_filtered: k > %d", VIX_MAX_K_LARGE);
    VIX_REQUIRE(k <= VIX_MAX_K || nq < 0x7FFFFFFFLL, VIX_ERR_INVALID_PARAM,
                "vix_sharded_search_filtered: k > %d needs nq < 2^31 - 1", VIX_MAX_K);
    In<uint64_t> fw;
    FilterArgs f;
    const FilterArgs* fp = nullptr;
    VIX_TRY(stage_filter(filter_words, filter_capacity, filter_mode, fw, f, fp));
    return sharded_search(h, c, queries, nq, k, nprobe, fp, out_dist, out_ids);
}

int vix_sharded_range_search(vix_index_t* h, vix_comm_t* c, const float* queries, int64_t nq, float radius, int nprobe,
                             const uint64_t* filter_words, int64_t filter_capacity, int filter_mode, vix_range_result_t** out) {
    VIX_TRY(ensure_device());
    VIX_REQUIRE(h && c && out, VIX_ERR_NULL_PTR, "vix_sharded_range_search: null pointer");
    *out = nullptr;
    VIX_REQUIRE(queries || nq == 0, VIX_ERR_NULL_PTR, "vix_sharded_range_search: null queries");
    VIX_REQUIRE(nq >= 0 && nq < 0x7FFFFFFFLL, VIX_ERR_INVALID_PARAM, "vix_sharded_range_search: nq must lie in [0, 2^31 - 1)");
    VIX_REQUIRE(radius == radius, VIX_ERR_INVALID_PARAM, "vix_sharded_range_search: radius is NaN");
    VIX_REQUIRE(filter_mode == VIX_FILTER_ALLOW || filter_mode == VIX_FILTER_DENY, VIX_ERR_INVALID_PARAM,
                "vix_sharded_range_search: filter_mode must be VIX_FILTER_ALLOW or VIX_FILTER_DENY");
    VIX_REQUIRE(filter_capacity >= 0, VIX_ERR_INVALID_PARAM, "vix_sharded_range_search: negative capacity");
    std::lock_guard<std::mutex> lc(c->mu);
    std::lock_guard<std::mutex> lk(h->mu);
    VIX_TRY(sharded_kind_check(h, "vix_sharded_range_search"));
    const bool flat = h->p.kind == VIX_INDEX_FLAT;                    // (no probes: nprobe is not read, as on one GPU)
    if (!flat) {
        if (nprobe <= 0) nprobe = h->p.nprobe;
        VIX_REQUIRE(nprobe > 0 && nprobe <= VIX_MAX_K, VIX_ERR_INVALID_K, "vix_sharded_range_search: nprobe = %d (1 .. %d)", nprobe,
                    VIX_MAX_K);
    }
    if (nq == 0) return range_empty(0, out);                          // (every rank sees the same nq: no exchange)
    In<uint64_t> fw;
    FilterArgs f;
    const FilterArgs* fp = nullptr;
    VIX_TRY(stage_filter(filter_words, filter_capacity, filter_mode, fw, f, fp));
    const int world = c->world;
    if (world == 1) return index_range_locked(h, queries, nq, radius, nprobe, fp, out);
    cudaStream_t s = ctx().stream;
    if (!flat && h->dirty) VIX_TRY(build_lists(h));
    VIX_TRY(ensure_region(c, nq, h->p.d, flat ? 1 : nprobe, 1));
    bool grown = false;
    if (c->peer_state == 1) VIX_TRY(ensure_range_region(c, nq, 0, &grown));
    auto mark = [&](int i) { if (c->trace) cudaEventRecord(c->ev[i], s); };
    mark(0);
    BatchProbes px;
    VIX_TRY(exchange_probes(h, c, queries, nq, nprobe, px));
    const float* dq = px.queries;
    const int32_t* probes = px.probes;
    mark(1);
    // the local scan and sort (its one synchronisation: the local total); a failure here travels with the lims, so that
    // every rank returns it together.  Every kind's keys are (API distance, user id): the merge is the same for all.
    RangeKeys rk;
    const int rc = index_range_locked(h, dq, nq, radius, nprobe, fp, nullptr, probes, &rk);
    mark(2);
    vix_range_result* r = nullptr;
    ShardTail tail;
    tail.out = &r;
    tail.neg_zero = range_neg_zero(h);
    ShardTotals st;
    VIX_TRY(sharded_range_exchange(h, c, nq, rc, rk, grown, tail, &st));
    mark(3);
    *out = r;
    return VIX_OK;
}

int vix_debug_shard_merge(const float* dist_all, const int64_t* ids_all, int world, int64_t nq, int k, int metric,
                          float* out_dist, int64_t* out_ids) {
    VIX_TRY(ensure_device());
    VIX_REQUIRE(dist_all && ids_all && out_dist && out_ids, VIX_ERR_NULL_PTR, "vix_debug_shard_merge: null pointer");
    VIX_REQUIRE(world > 0 && world <= 256 && nq >= 0 && k > 0 && k <= VIX_MAX_K, VIX_ERR_INVALID_PARAM,
                "vix_debug_shard_merge: world / nq / k");
    if (nq == 0) return VIX_OK;
    const int64_t total = (int64_t)world * nq * k;
    In<float> dd;
    In<int64_t> di;
    Out<float> od;
    Out<int64_t> oi;
    VIX_TRY(dd.stage(dist_all, (size_t)total));
    VIX_TRY(di.stage(ids_all, (size_t)total));
    VIX_TRY(od.stage(out_dist, (size_t)nq * k));
    VIX_TRY(oi.stage(out_ids, (size_t)nq * k));
    Scratch<u64> keys;
    VIX_TRY(keys.alloc((size_t)total));
    pack_result_keys_kernel<<<(unsigned)((total + 255) / 256), 256, 0, ctx().stream>>>(dd.dev, di.dev, total, nullptr, world, 0,
                                                                                     keys.ptr);
    VIX_LAUNCH_CHECK();
    VIX_TRY(merge_shard_keys(keys.ptr, world, nq, k, metric == VIX_METRIC_IP, od.dev, oi.dev));
    VIX_TRY(od.commit());
    VIX_TRY(oi.commit());
    return finish(od.is_host() || oi.is_host());
}

int vix_debug_shard_range_merge(const int64_t* lims_all, const float* dist_all, const int64_t* ids_all, int world, int64_t nq,
                                int metric, vix_range_result_t** out) {
    VIX_TRY(ensure_device());
    VIX_REQUIRE(lims_all && out, VIX_ERR_NULL_PTR, "vix_debug_shard_range_merge: null pointer");
    *out = nullptr;
    VIX_REQUIRE(world > 0 && world <= 256 && nq >= 0 && nq < 0x7FFFFFFFLL, VIX_ERR_INVALID_PARAM,
                "vix_debug_shard_range_merge: world / nq");
    cudaStream_t s = ctx().stream;
    DebugShardRuns in;
    VIX_TRY(debug_shard_runs("vix_debug_shard_range_merge", lims_all, dist_all, ids_all, world, nq, in));
    vix_range_result* r = nullptr;
    VIX_TRY(range_alloc(nq, in.total, &r));
    const int rc = shard_range_merge(in.keys.ptr, in.dbase.ptr, in.dlims.ptr, world, nq, in.glims.ptr, in.total,
                                     metric == VIX_METRIC_IP, r);
    if (rc != VIX_OK) { range_free(r); return rc; }
    const cudaError_t e = cudaStreamSynchronize(s);                   // (meta, a host vector, is read by the copy above)
    if (e != cudaSuccess) { range_free(r); VIX_CUDA(e); }
    *out = r;
    return VIX_OK;
}

int vix_debug_shard_knn_merge(const int64_t* lims_all, const float* dist_all, const int64_t* ids_all, int world, int64_t nq,
                              int k, int metric, float* out_dist, int64_t* out_ids) {
    VIX_TRY(ensure_device());
    VIX_REQUIRE(lims_all && out_dist && out_ids, VIX_ERR_NULL_PTR, "vix_debug_shard_knn_merge: null pointer");
    VIX_REQUIRE(world > 0 && world <= 256 && nq >= 0 && nq < 0x7FFFFFFFLL && k > 0 && k <= VIX_MAX_K_LARGE,
                VIX_ERR_INVALID_PARAM, "vix_debug_shard_knn_merge: world / nq / k");
    DebugShardRuns in;
    VIX_TRY(debug_shard_runs("vix_debug_shard_knn_merge", lims_all, dist_all, ids_all, world, nq, in));
    Out<float> od;
    Out<int64_t> oi;
    VIX_TRY(od.stage(out_dist, (size_t)nq * k));
    VIX_TRY(oi.stage(out_ids, (size_t)nq * k));
    if (nq > 0)
        VIX_TRY(shard_knn_merge(in.keys.ptr, in.dbase.ptr, in.dlims.ptr, world, nq, in.glims.ptr, in.total, k,
                                metric == VIX_METRIC_IP, od.dev, oi.dev));
    VIX_TRY(od.commit());
    VIX_TRY(oi.commit());
    return finish(true);                                              // (meta, a host vector, is read by a copy)
}

int vix_debug_shard_flat_merge(const int64_t* lims_all, const float* score_all, const int64_t* ids_all, int world, int64_t nq,
                               int k, int metric, int64_t* out_lims, float* out_dist, int64_t* out_ids) {
    VIX_TRY(ensure_device());
    VIX_REQUIRE(lims_all && out_dist && out_ids, VIX_ERR_NULL_PTR, "vix_debug_shard_flat_merge: null pointer");
    VIX_REQUIRE(world > 0 && world <= 256 && nq >= 0 && nq < 0x7FFFFFFFLL && k >= 0 && k <= VIX_MAX_K_LARGE,
                VIX_ERR_INVALID_PARAM, "vix_debug_shard_flat_merge: world / nq / k");
    VIX_REQUIRE(metric == VIX_METRIC_L2 || metric == VIX_METRIC_IP || metric == VIX_METRIC_COSINE, VIX_ERR_INVALID_PARAM,
                "vix_debug_shard_flat_merge: metric");
    DebugShardRuns in;
    VIX_TRY(debug_shard_runs("vix_debug_shard_flat_merge", lims_all, score_all, ids_all, world, nq, in,
                             metric != VIX_METRIC_L2 ? 1 : 0));
    const size_t n_out = k > 0 ? (size_t)nq * k : (size_t)in.total;
    Out<float> od;
    Out<int64_t> oi;
    Out<int64_t> ol;
    VIX_TRY(od.stage(out_dist, n_out));
    VIX_TRY(oi.stage(out_ids, n_out));
    VIX_TRY(ol.stage(out_lims, out_lims ? (size_t)nq + 1 : 0));
    if (nq > 0)
        VIX_TRY(shard_flat_merge(in.keys.ptr, in.dbase.ptr, in.dlims.ptr, world, nq, in.glims.ptr, in.total, k, metric, od.dev,
                                 oi.dev));
    if (ol.dev) VIX_CUDA(cudaMemcpyAsync(ol.dev, in.glims.ptr, ((size_t)nq + 1) * 8, cudaMemcpyDeviceToDevice, ctx().stream));
    VIX_TRY(od.commit());
    VIX_TRY(oi.commit());
    VIX_TRY(ol.commit());
    return finish(true);
}

int vix_debug_sharded_emulate(vix_index_t* const* shards, int world, const float* queries, int64_t nq, int k, int nprobe,
                              float radius, const uint64_t* filter_words, int64_t filter_capacity, int filter_mode,
                              float* out_dist, int64_t* out_ids, vix_range_result_t** out_range) {
    const char* who = "vix_debug_sharded_emulate";
    VIX_TRY(ensure_device());
    VIX_REQUIRE(shards && world > 0 && world <= 256, VIX_ERR_INVALID_PARAM, "%s: shards / world", who);
    const bool range = out_range != nullptr;
    if (range) *out_range = nullptr;
    for (int r = 0; r < world; ++r) {
        VIX_REQUIRE(shards[r], VIX_ERR_NULL_PTR, "%s: null shard %d", who, r);
        for (int p = 0; p < r; ++p) VIX_REQUIRE(shards[p] != shards[r], VIX_ERR_INVALID_PARAM, "%s: shard %d repeats shard %d", who, r, p);
        VIX_REQUIRE(shards[r]->p.kind == shards[0]->p.kind && shards[r]->p.metric == shards[0]->p.metric &&
                    shards[r]->p.d == shards[0]->p.d, VIX_ERR_INVALID_PARAM, "%s: shard %d differs in kind, metric or dimension", who, r);
    }
    VIX_REQUIRE(filter_mode == VIX_FILTER_ALLOW || filter_mode == VIX_FILTER_DENY, VIX_ERR_INVALID_PARAM,
                "%s: filter_mode must be VIX_FILTER_ALLOW or VIX_FILTER_DENY", who);
    VIX_REQUIRE(filter_capacity >= 0, VIX_ERR_INVALID_PARAM, "%s: negative capacity", who);
    VIX_REQUIRE(nq >= 0 && nq < 0x7FFFFFFFLL, VIX_ERR_INVALID_PARAM, "%s: nq must lie in [0, 2^31 - 1)", who);
    VIX_REQUIRE(!range || radius == radius, VIX_ERR_INVALID_PARAM, "%s: radius is NaN", who);
    std::vector<std::unique_lock<std::mutex>> locks;
    for (int r = 0; r < world; ++r) locks.emplace_back(shards[r]->mu);
    for (int r = 0; r < world; ++r) VIX_TRY(sharded_kind_check(shards[r], who));
    vix_index* h0 = shards[0];
    const bool flat = h0->p.kind == VIX_INDEX_FLAT;
    const int d = h0->p.d;
    if (!flat) {
        if (nprobe <= 0) nprobe = h0->p.nprobe;
        VIX_REQUIRE(nprobe > 0 && nprobe <= VIX_MAX_K, VIX_ERR_INVALID_K, "%s: nprobe = %d (1 .. %d)", who, nprobe, VIX_MAX_K);
    }
    if (range && nq == 0) return range_empty(0, out_range);
    if (!range) {
        if (nq == 0 || k <= 0) return VIX_OK;
        VIX_REQUIRE(out_dist && out_ids, VIX_ERR_NULL_PTR, "%s: null outputs", who);
        VIX_REQUIRE(k <= VIX_MAX_K_LARGE, VIX_ERR_INVALID_K, "%s: k > %d", who, VIX_MAX_K_LARGE);
    }
    VIX_REQUIRE(queries, VIX_ERR_NULL_PTR, "%s: null queries", who);
    cudaStream_t s = ctx().stream;
    In<uint64_t> fw;
    FilterArgs f;
    const FilterArgs* fp = nullptr;
    VIX_TRY(stage_filter(filter_words, filter_capacity, filter_mode, fw, f, fp));
    In<float> dq;
    VIX_TRY(dq.stage(queries, (size_t)nq * d));
    // the probes of the whole batch (every rank selects them against the same centroids)
    Scratch<int32_t> pr;
    const int32_t* probes = nullptr;
    if (!flat) {
        for (int r = 0; r < world; ++r)
            if (shards[r]->dirty) VIX_TRY(build_lists(shards[r]));
        VIX_TRY(pr.alloc((size_t)nq * nprobe));
        VIX_TRY(select_probes_device(h0, dq.dev, nq, nprobe, pr.ptr));
        probes = pr.ptr;
    }
    if (!range && k <= VIX_MAX_K) {
        const int64_t total = nq * (int64_t)k;
        Out<float> dd;
        Out<int64_t> di;
        VIX_TRY(dd.stage(out_dist, (size_t)total));
        VIX_TRY(di.stage(out_ids, (size_t)total));
        Scratch<u64> keys_all;
        VIX_TRY(keys_all.alloc((size_t)world * total));
        for (int r = 0; r < world; ++r)
            VIX_TRY(local_knn_keys(shards[r], dq.dev, nq, k, nprobe, probes, fp, nullptr, world, 0, keys_all.ptr + (size_t)r * total));
        VIX_TRY(merge_knn_keys(h0, keys_all.ptr, world, nq, k, dd.dev, di.dev));
        VIX_TRY(dd.commit());
        VIX_TRY(di.commit());
        return finish(true);
    }
    // every rank's sorted rows: its range rows, or its k-NN rows within the shared bound cut at k
    std::vector<std::unique_ptr<RangeKeys>> runs;
    for (int r = 0; r < world; ++r) runs.emplace_back(new RangeKeys());
    if (range) {
        for (int r = 0; r < world; ++r)
            VIX_TRY(index_range_locked(shards[r], dq.dev, nq, radius, nprobe, fp, nullptr, probes, runs[r].get()));
    } else {
        std::vector<std::unique_ptr<LocalKnnLarge>> L;
        Scratch<uint32_t> slots, tau;
        VIX_TRY(slots.alloc((size_t)world * nq));
        VIX_TRY(tau.alloc((size_t)nq));
        for (int r = 0; r < world; ++r) {
            L.emplace_back(new LocalKnnLarge());
            int64_t seed_n = 0;
            VIX_TRY(local_knn_prepare(shards[r], dq.dev, nq, k, nprobe, probes, fp, *L[r]));
            VIX_TRY(local_knn_seed(*L[r], nq, k, slots.ptr + (size_t)r * nq, &seed_n));
        }
        min_knn_bounds_kernel<<<(unsigned)((nq + 255) / 256), 256, 0, s>>>(slots.ptr, world, nq, nq, tau.ptr);
        VIX_LAUNCH_CHECK();
        for (int r = 0; r < world; ++r) {
            RangeKeys rk;
            RangeInfo ci;
            size_t cap = shards[r]->knn_cap;
            VIX_TRY(local_knn_cut(shards[r], *L[r], nq, k, tau.ptr, cap, rk, *runs[r], &ci));
        }
    }
    // the exchanged layout, as sharded_range_exchange holds it: lims [world][nq + 2] (status 0), keys rank by rank
    const int64_t L2 = nq + 2;
    Scratch<int64_t> lims_all, glims, dbase;
    VIX_TRY(lims_all.alloc((size_t)world * L2));
    VIX_TRY(glims.alloc((size_t)nq + 1));
    VIX_TRY(dbase.alloc((size_t)world + 1));
    VIX_CUDA(cudaMemsetAsync(lims_all.ptr, 0, (size_t)world * L2 * 8, s));
    std::vector<int64_t> tot((size_t)world, 0);
    for (int r = 0; r < world; ++r) {
        VIX_CUDA(cudaMemcpyAsync(lims_all.ptr + (size_t)r * L2, runs[r]->lims.ptr, (size_t)(nq + 1) * 8, cudaMemcpyDeviceToDevice, s));
        VIX_CUDA(cudaMemcpyAsync(&tot[r], runs[r]->lims.ptr + nq, 8, cudaMemcpyDeviceToHost, s));
    }
    VIX_CUDA(cudaStreamSynchronize(s));
    int64_t total = 0;
    for (int r = 0; r < world; ++r) total += tot[r];
    Scratch<u64> keys;
    VIX_TRY(keys.alloc((size_t)total));
    for (int64_t r = 0, at = 0; r < world; at += tot[r], ++r)
        if (tot[r] > 0) VIX_CUDA(cudaMemcpyAsync(keys.ptr + at, runs[r]->sorted, (size_t)tot[r] * 8, cudaMemcpyDeviceToDevice, s));
    std::vector<int64_t> meta;
    VIX_TRY(shard_range_lims(lims_all.ptr, world, nq, glims.ptr, meta));
    VIX_CUDA(cudaMemcpyAsync(dbase.ptr, meta.data(), ((size_t)world + 1) * 8, cudaMemcpyHostToDevice, s));
    if (range) {
        vix_range_result* res = nullptr;
        VIX_TRY(range_alloc(nq, total, &res));
        int rc = shard_range_merge(keys.ptr, dbase.ptr, lims_all.ptr, world, nq, glims.ptr, total, range_neg_zero(h0), res);
        if (rc == VIX_OK) rc = finish(true);
        if (rc != VIX_OK) { range_free(res); return rc; }
        *out_range = res;
        return VIX_OK;
    }
    Out<float> dd;
    Out<int64_t> di;
    VIX_TRY(dd.stage(out_dist, (size_t)nq * k));
    VIX_TRY(di.stage(out_ids, (size_t)nq * k));
    if (flat) VIX_TRY(shard_flat_merge(keys.ptr, dbase.ptr, lims_all.ptr, world, nq, glims.ptr, total, k, h0->p.metric, dd.dev, di.dev));
    else VIX_TRY(shard_knn_merge(keys.ptr, dbase.ptr, lims_all.ptr, world, nq, glims.ptr, total, k, knn_neg_zero(h0), dd.dev, di.dev));
    VIX_TRY(dd.commit());
    VIX_TRY(di.commit());
    return finish(true);
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
    VIX_TRY(sharded_kind_check(h, "vix_sharded_add"));
    const int world = c->world, rank = c->rank, d = h->p.d;
    cudaStream_t s = ctx().stream;
    if (h->p.kind == VIX_INDEX_FLAT) {
        // rows stay on the rank that passes them: no list partition, no row exchange.  The call stays collective: the count
        // of ids outside [0, 2^32 - 1) is all-gathered before any rank stores a row, so all ranks refuse together.
        VIX_REQUIRE(!list_bounds, VIX_ERR_INVALID_PARAM, "vix_sharded_add: a flat index has no list partition (list_bounds must "
                    "be NULL)");
        In<int64_t> dids;
        VIX_TRY(dids.stage(ids, (size_t)n));
        Scratch<unsigned long long> dcounts;
        VIX_TRY(dcounts.alloc((size_t)world + 1));
        VIX_CUDA(cudaMemsetAsync(dcounts.ptr, 0, sizeof(unsigned long long) * (world + 1), s));
        VIX_TRY(count_invalid_ids_device(dids.dev, n, dcounts.ptr + world));
        VIX_NCCL(g_nccl.AllGather(dcounts.ptr + world, dcounts.ptr, 1, ncclUint64, c->comm, s));
        std::vector<unsigned long long> counts((size_t)world);
        VIX_CUDA(cudaMemcpyAsync(counts.data(), dcounts.ptr, sizeof(unsigned long long) * world, cudaMemcpyDeviceToHost, s));
        VIX_CUDA(cudaStreamSynchronize(s));
        for (int p = 0; p < world; ++p)
            VIX_REQUIRE(counts[p] == 0, VIX_ERR_INVALID_PARAM, "vix_sharded_add: rank %d was handed %llu ids outside [0, 2^32 - 1); "
                        "no rank stored any row of this call", p, counts[p]);
        return index_add_rows_locked(h, x, dids.dev, n);
    }
    const bool ivfflat = h->p.kind == VIX_INDEX_IVF_FLAT;
    const int m = ivfflat ? 0 : h->code_bytes();                          // m: bytes per stored code (IVF-PQ)
    // block boundaries of the list partition: given, or equal-count blocks
    std::vector<int64_t> bounds((size_t)world + 1);
    for (int r = 0; r <= world; ++r) bounds[r] = list_bounds ? list_bounds[r] : (int64_t)h->kc * r / world;
    VIX_REQUIRE(bounds[0] == 0 && bounds[world] == h->kc, VIX_ERR_INVALID_PARAM, "vix_sharded_add: bounds must run from 0 to %d", h->kc);
    for (int r = 0; r < world; ++r)
        VIX_REQUIRE(bounds[r + 1] >= bounds[r], VIX_ERR_INVALID_PARAM, "vix_sharded_add: bounds must ascend");
    // 1. assign what this rank was handed and count the rows no rank may store: no nearest list (NaN components) or an id
    //    outside [0, 2^32 - 1).  The count rides in the all-gather of the send counts, so every rank sees every rank's count
    //    before any row travels, and all of them refuse the call together (a rank that returned alone would leave its peers
    //    waiting in the all-gather, or holding their share of the rows).
    In<float> dx;
    In<int64_t> dids;
    VIX_TRY(dx.stage(x, (size_t)n * d));
    VIX_TRY(dids.stage(ids, (size_t)n));
    Scratch<int32_t> asg, owner, order;
    Scratch<uint8_t> codes;
    Scratch<unsigned long long> dcounts;
    Scratch<int64_t> dbounds;
    const size_t W = (size_t)world + 1;                                   // per rank: rows for each owner, then invalid rows
    VIX_TRY(dcounts.alloc(W * (world + 1)));                              // [world][W] gathered, then this rank's [W]
    VIX_TRY(dbounds.alloc((size_t)world + 1));
    VIX_CUDA(cudaMemsetAsync(dcounts.ptr, 0, sizeof(unsigned long long) * W * (world + 1), s));
    VIX_CUDA(cudaMemcpyAsync(dbounds.ptr, bounds.data(), sizeof(int64_t) * (world + 1), cudaMemcpyHostToDevice, s));
    unsigned long long* mine = dcounts.ptr + W * world;
    if (n > 0) {
        VIX_TRY(asg.alloc((size_t)n));
        VIX_TRY(assign_lists_device(h, dx.dev, n, asg.ptr));
        VIX_TRY(count_invalid_rows_device(asg.ptr, dids.dev, n, h->kc, mine + world));
        // rows ordered by owning rank (stable: rows keep their order inside a block)
        VIX_TRY(owner.alloc((size_t)n));
        VIX_TRY(order.alloc((size_t)n));
        owner_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(asg.ptr, n, dbounds.ptr, world, owner.ptr, mine);
        VIX_LAUNCH_CHECK();
        VIX_TRY(order_by_key(owner.ptr, n, world, order.ptr));
    }
    // 2. everybody learns everybody's send counts and invalid rows
    VIX_NCCL(g_nccl.AllGather(mine, dcounts.ptr, W, ncclUint64, c->comm, s));
    std::vector<unsigned long long> counts(W * world);
    VIX_CUDA(cudaMemcpyAsync(counts.data(), dcounts.ptr, sizeof(unsigned long long) * W * world, cudaMemcpyDeviceToHost, s));
    VIX_CUDA(cudaStreamSynchronize(s));
    for (int p = 0; p < world; ++p)
        VIX_REQUIRE(counts[(size_t)p * W + world] == 0, VIX_ERR_INVALID_PARAM,
                    "vix_sharded_add: rank %d was handed %llu rows with no nearest list (NaN components?) or an id outside "
                    "[0, 2^32 - 1); no rank stored any row of this call", p, counts[(size_t)p * W + world]);
    // 3. encode (IVF-PQ), in owner order; IVF-Flat rows travel as they are (4 d + 12 bytes each instead of m + 12)
    Scratch<int32_t> s_asg;
    Scratch<uint8_t> s_codes;
    Scratch<float> s_x;
    Scratch<int64_t> s_ids;
    if (n > 0) {
        VIX_TRY(s_asg.alloc((size_t)n));
        VIX_TRY(s_ids.alloc((size_t)n));
        if (ivfflat) {
            VIX_TRY(s_x.alloc((size_t)n * d));
            gather_vec_rows_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(order.ptr, n, d, asg.ptr, dx.dev, dids.dev, s_asg.ptr,
                                                                             s_x.ptr, s_ids.ptr);
        } else {
            VIX_TRY(codes.alloc((size_t)n * m));
            VIX_TRY(encode_rows_device(h, dx.dev, n, asg.ptr, codes.ptr));
            VIX_TRY(s_codes.alloc((size_t)n * m));
            gather_rows_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(order.ptr, n, m, asg.ptr, codes.ptr, dids.dev, s_asg.ptr,
                                                                         s_codes.ptr, s_ids.ptr);
        }
        VIX_LAUNCH_CHECK();
    }
    std::vector<int64_t> send_off((size_t)world + 1, 0), recv_off((size_t)world + 1, 0);
    for (int p = 0; p < world; ++p) {
        send_off[p + 1] = send_off[p] + (int64_t)counts[(size_t)rank * W + p];
        recv_off[p + 1] = recv_off[p] + (int64_t)counts[(size_t)p * W + rank];
    }
    const int64_t nrecv = recv_off[world];
    // 4. rows travel to their owners
    Scratch<int32_t> r_asg;
    Scratch<uint8_t> r_codes;
    Scratch<float> r_x;
    Scratch<int64_t> r_ids;
    VIX_TRY(r_asg.alloc((size_t)nrecv));
    if (ivfflat) VIX_TRY(r_x.alloc((size_t)nrecv * d));
    else VIX_TRY(r_codes.alloc((size_t)nrecv * m));
    VIX_TRY(r_ids.alloc((size_t)nrecv));
    VIX_NCCL(g_nccl.GroupStart());
    for (int p = 0; p < world; ++p) {
        const int64_t sc = send_off[p + 1] - send_off[p], rc = recv_off[p + 1] - recv_off[p];
        if (sc > 0) {
            VIX_NCCL(g_nccl.Send(s_asg.ptr + send_off[p], (size_t)sc, ncclInt32, p, c->comm, s));
            if (ivfflat) VIX_NCCL(g_nccl.Send(s_x.ptr + (size_t)send_off[p] * d, (size_t)sc * d, ncclFloat, p, c->comm, s));
            else VIX_NCCL(g_nccl.Send(s_codes.ptr + (size_t)send_off[p] * m, (size_t)sc * m, ncclUint8, p, c->comm, s));
            VIX_NCCL(g_nccl.Send(s_ids.ptr + send_off[p], (size_t)sc, ncclInt64, p, c->comm, s));
        }
        if (rc > 0) {
            VIX_NCCL(g_nccl.Recv(r_asg.ptr + recv_off[p], (size_t)rc, ncclInt32, p, c->comm, s));
            if (ivfflat) VIX_NCCL(g_nccl.Recv(r_x.ptr + (size_t)recv_off[p] * d, (size_t)rc * d, ncclFloat, p, c->comm, s));
            else VIX_NCCL(g_nccl.Recv(r_codes.ptr + (size_t)recv_off[p] * m, (size_t)rc * m, ncclUint8, p, c->comm, s));
            VIX_NCCL(g_nccl.Recv(r_ids.ptr + recv_off[p], (size_t)rc, ncclInt64, p, c->comm, s));
        }
    }
    VIX_NCCL(g_nccl.GroupEnd());
    // 5. append with the given assignments (IVF-PQ: already encoded)
    if (nrecv > 0) {
        if (ivfflat) VIX_TRY(index_add_assigned_locked(h, r_asg.ptr, r_x.ptr, r_ids.ptr, nrecv));
        else VIX_TRY(index_add_encoded_locked(h, r_asg.ptr, r_codes.ptr, r_ids.ptr, nrecv));
    }
    return finish(true);
}

}  // extern "C"
