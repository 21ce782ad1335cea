// vix_replicated.cu -- the replicated layout behind the C ABI: every rank holds the whole index, and a batch is split by
// query.  Rank r answers rows vix_sharded_query_block(nq, r, world) with the one-GPU code path (index_search_locked /
// index_range_locked), and the blocks are assembled on every rank:
//
//   vix_replicated_search          the rank's [cnt x k] block (distances and ids, raw bits) is stored into every peer's
//                                  region at the block's row offset, then one barrier; NCCL: an in-place all-gather.
//                                  k <= VIX_MAX_K uses the results slab of the exchange region (no host synchronisation);
//                                  above, the keys of the range region, grown collectively (the two-pass route synchronises
//                                  anyway).
//   vix_replicated_range_search    the rank's sorted keys and row starts travel with sharded_range_exchange's protocol; every
//                                  row belongs to one rank, so the keys rank by rank are the global rows: no merge, only a
//                                  decode (replica_range_concat).
//   vix_replicated_add             each rank prepares its own rows (IVF-PQ: assign + encode; IVF-Flat: assign), the rows are
//                                  all-gathered and every replica appends all of them rank by rank: identical lists.
//
// Every call over peer memory begins with a barrier: a rank stores into a peer's region only after that peer has read what
// the previous call left there.
#include "vix_comm.cuh"

#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <vector>

namespace vix {

// src [n words] -> byte offset `off` of every rank's region except `skip` (-1: every rank)
template <typename W>
__global__ void replica_store_kernel(const W* __restrict__ src, int64_t n, void* const* __restrict__ peer_base, int world, int skip,
                                     size_t off) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const W v = src[i];
        for (int p = 0; p < world; ++p)
            if (p != skip) reinterpret_cast<W*>(static_cast<char*>(peer_base[p]) + off)[i] = v;
    }
}

// rc -> status word `rank` of every rank's flags page (this rank's included)
__global__ void replica_status_store_kernel(int32_t rc, void* const* __restrict__ peer_base, int world, int rank) {
    for (int p = threadIdx.x; p < world; p += blockDim.x)
        reinterpret_cast<int32_t*>(static_cast<char*>(peer_base[p]) + kStatusOffset)[rank] = rc;
}

// asynchronous mode: a rank's failed k-NN step raises the pipeline error flag, which the next synchronising call reports
__global__ void replica_status_kernel(const int32_t* __restrict__ status, int world, int* error_host) {
    for (int p = threadIdx.x; p < world; p += blockDim.x)
        if (status[p] != VIX_OK && error_host) {
            *reinterpret_cast<volatile int*>(error_host) = 1;
            __threadfence_system();
        }
}

// a rank's block row starts [cnt + 1] (blk == nullptr: no rows) -> row starts over the whole batch [nq + 1]: the rows
// outside [lo, lo + cnt) are empty
__global__ void replica_expand_lims_kernel(const int64_t* __restrict__ blk, int64_t lo, int64_t cnt, int64_t nq,
                                           int64_t* __restrict__ out) {
    for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q <= nq; q += (int64_t)gridDim.x * blockDim.x)
        out[q] = !blk || q <= lo ? 0 : q >= lo + cnt ? blk[cnt] : blk[q - lo];
}

// The replicated range search's last step: the ranks' keys, concatenated rank by rank, are the global rows in order (rank
// r's rows are the queries of its block, and the blocks follow each other), so key i is entry i of the global CSR
__global__ void __launch_bounds__(256)
replica_range_concat_kernel(const u64* __restrict__ keys, int64_t total, int neg_zero, float* __restrict__ out_dist,
                            int64_t* __restrict__ out_ids) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x)
        range_decode_key(keys[i], neg_zero, out_dist + i, out_ids + i);
}

// the test hook's rows (API distances, ids) -> the keys a range scan collects
__global__ void replica_pack_keys_kernel(const float* __restrict__ dist, const int64_t* __restrict__ ids, int64_t n,
                                         u64* __restrict__ keys) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) keys[i] = make_key(dist[i], (uint32_t)ids[i], 0);
}

static unsigned grid_for(int64_t work, int per_sm) {
    const int64_t want = (work + 255) / 256;
    const int64_t cap = (int64_t)num_sms() * per_sm;
    return (unsigned)std::max<int64_t>(1, std::min(want, cap));
}

// `bytes` of src -> byte offset `off` of every rank's region except `skip`, in 16-, 4- or 1-byte words as alignment allows
// (the regions themselves are 256-aligned)
static int replica_store(const void* src, size_t bytes, void* const* peer_base, int world, int skip, size_t off) {
    if (bytes == 0) return VIX_OK;
    cudaStream_t s = ctx().stream;
    const uintptr_t a = reinterpret_cast<uintptr_t>(src) | (uintptr_t)off | (uintptr_t)bytes;
    if (a % 16 == 0) {
        const int64_t n = (int64_t)(bytes / 16);
        replica_store_kernel<uint4><<<grid_for(n, 4), 256, 0, s>>>(static_cast<const uint4*>(src), n, peer_base, world, skip, off);
    } else if (a % 4 == 0) {
        const int64_t n = (int64_t)(bytes / 4);
        replica_store_kernel<uint32_t><<<grid_for(n, 4), 256, 0, s>>>(static_cast<const uint32_t*>(src), n, peer_base, world, skip, off);
    } else {
        const int64_t n = (int64_t)bytes;
        replica_store_kernel<uint8_t><<<grid_for(n, 4), 256, 0, s>>>(static_cast<const uint8_t*>(src), n, peer_base, world, skip, off);
    }
    VIX_LAUNCH_CHECK();
    return VIX_OK;
}

int replica_range_concat(const u64* keys, const int64_t* glims, int64_t nq, int64_t total, int neg_zero, vix_range_result* r) {
    cudaStream_t s = ctx().stream;
    VIX_CUDA(cudaMemcpyAsync(r->lims, glims, (size_t)(nq + 1) * 8, cudaMemcpyDeviceToDevice, s));
    if (total == 0) return VIX_OK;
    replica_range_concat_kernel<<<grid_for(total, 8), 256, 0, s>>>(keys, total, neg_zero, r->dist, r->ids);
    VIX_LAUNCH_CHECK();
    return VIX_OK;
}

static int replica_expand_lims(const int64_t* blk, int64_t lo, int64_t cnt, int64_t nq, int64_t* out) {
    replica_expand_lims_kernel<<<grid_for(nq + 1, 4), 256, 0, ctx().stream>>>(blk, lo, cnt, nq, out);
    VIX_LAUNCH_CHECK();
    return VIX_OK;
}

// What a replicated call needs of the handle, checked on every rank before any exchange: the whole index (shard_world 0 /
// 1), an IVF-PQ index trained with L2 / IP, and for add an IVF-Flat index with its centroids (every row is filed into its
// list at once, as the sharded layout does).
static int replica_check(const vix_index* h, const char* who, bool add) {
    VIX_REQUIRE(h->p.shard_world <= 1, VIX_ERR_INVALID_PARAM, "%s: a replica holds the whole index (shard_world = %d; 0 or 1)",
                who, h->p.shard_world);
    if (h->p.kind == VIX_INDEX_IVF_PQ) {
        VIX_REQUIRE(h->has_coarse && h->has_pq, VIX_ERR_NOT_TRAINED, "%s: needs a trained IVF-PQ index", who);
        VIX_REQUIRE(h->p.metric != VIX_METRIC_COSINE, VIX_ERR_UNSUPPORTED, "%s: L2 / IP only", who);
    } else if (add && h->p.kind == VIX_INDEX_IVF_FLAT) {
        VIX_REQUIRE(h->has_coarse, VIX_ERR_NOT_TRAINED, "%s: an IVF-Flat index needs its coarse centroids (set or trained) "
                    "before a replicated add", who);
    }
    return VIX_OK;
}

// nprobe after the default, for the kinds that read it (one GPU: an IVF index with centroids)
static int replica_nprobe(const vix_index* h, int* nprobe, const char* who) {
    if (h->p.kind == VIX_INDEX_FLAT || !h->has_coarse) return VIX_OK;
    if (*nprobe <= 0) *nprobe = h->p.nprobe;
    VIX_REQUIRE(*nprobe > 0 && *nprobe <= VIX_MAX_K, VIX_ERR_INVALID_K, "%s: nprobe = %d (1 .. %d)", who, *nprobe, VIX_MAX_K);
    return VIX_OK;
}

static void replica_debug_line(vix_comm* c, const vix_index* h, const char* op, int64_t block, int64_t total, bool grown) {
    if (getenv("VIX_SCAN_DEBUG"))
        fprintf(stderr, "[vix replicated] world %d, peer %d, kind %s, op %s, block %lld, total %lld, grown %d\n", c->world,
                c->peer_state == 1 ? 1 : 0, kind_name(h), op, (long long)block, (long long)total, grown ? 1 : 0);
}

// vix_replicated_search and _filtered (filter == nullptr: unfiltered).  The caller checked the arguments.
static int replicated_search(vix_index* h, vix_comm* c, const float* queries, int64_t nq, int k, int nprobe, const FilterArgs* filter,
                             float* out_dist, int64_t* out_ids) {
    const char* who = filter ? "vix_replicated_search_filtered" : "vix_replicated_search";
    std::lock_guard<std::mutex> lc(c->mu);
    std::lock_guard<std::mutex> lk(h->mu);
    VIX_TRY(replica_check(h, who, false));
    VIX_TRY(replica_nprobe(h, &nprobe, who));
    const int world = c->world, rank = c->rank, d = h->p.d;
    if (world == 1) return index_search_locked(h, queries, nq, k, nprobe, out_dist, out_ids, nullptr, nullptr, nullptr, filter);
    cudaStream_t s = ctx().stream;
    const bool large = k > VIX_MAX_K;
    VIX_TRY(ensure_region(c, nq, 4, 1, large ? 1 : k));
    const bool peer = c->peer_state == 1;
    const int64_t per = block_rows(nq, world);
    const int64_t lo = std::min<int64_t>(nq, (int64_t)rank * per);
    const int64_t cnt = std::min<int64_t>(nq, lo + per) - lo;
    // Where the answer is assembled.  Peer memory: [nq x k] distances, then (256-aligned) [nq x k] ids, in the results slab of
    // the exchange region (k <= VIX_MAX_K; it holds world x nq x k keys, at least 16 bytes per entry) or in the keys of the
    // range region.  NCCL: the same for [world x per] rows in a local buffer, gathered in place.
    const int64_t rows = peer ? nq : (int64_t)world * per;
    const size_t ids_off = ((size_t)rows * k * 4 + 255) & ~(size_t)255;
    const size_t bytes = ids_off + (size_t)rows * k * 8;
    bool grown = false;
    char* base = nullptr;
    void* const* peer_base = nullptr;
    size_t region_off = 0;
    if (peer && !large) {
        base = static_cast<char*>(c->local) + c->off_results;
        peer_base = c->peer_dev;
        region_off = c->off_results;
    } else if (peer) {
        VIX_TRY(ensure_range_region(c, nq, (int64_t)((bytes + 7) / 8), &grown));
        base = static_cast<char*>(c->range_local) + c->range_off_keys;
        peer_base = c->range_peer_dev;
        region_off = c->range_off_keys;
    } else {
        if (bytes > c->gather_keys_bytes) {
            if (c->gather_keys) { VIX_CUDA(cudaStreamSynchronize(s)); cudaFree(c->gather_keys); c->gather_keys = nullptr; }
            c->gather_keys_bytes = 0;
            VIX_CUDA(cudaMalloc(&c->gather_keys, bytes));
            c->gather_keys_bytes = bytes;
        }
        base = static_cast<char*>(c->gather_keys);
    }
    float* adist = reinterpret_cast<float*>(base);
    int64_t* aids = reinterpret_cast<int64_t*>(base + ids_off);
    const int64_t row0 = peer ? lo : (int64_t)rank * per;          // the block's first row in the assembly buffer
    auto mark = [&](int i) { if (c->trace) cudaEventRecord(c->ev[i], s); };
    mark(0);
    // 1. queries in: only this rank's block (from a host pointer, only it crosses PCIe)
    if (peer) VIX_TRY(peer_barrier(c));
    In<float> dq;
    VIX_TRY(dq.stage(queries + (size_t)lo * d, (size_t)cnt * d));
    mark(1);
    // 2. the one-GPU search of the block, straight into its rows of the assembly buffer
    int rc = VIX_OK;
    if (cnt > 0) rc = index_search_locked(h, dq.dev, cnt, k, nprobe, adist + row0 * k, aids + row0 * k, nullptr, nullptr, nullptr, filter);
    mark(2);
    // 3. assembly: the block and this rank's status reach every rank
    Scratch<int32_t> st;
    const int32_t* status = nullptr;
    const size_t blk = (size_t)cnt * k;
    if (peer) {
        replica_status_store_kernel<<<1, 32 * ((world + 31) / 32), 0, s>>>(rc, c->peer_dev, world, rank);
        VIX_LAUNCH_CHECK();
        VIX_TRY(replica_store(adist + row0 * k, blk * 4, peer_base, world, rank, region_off + (size_t)row0 * k * 4));
        VIX_TRY(replica_store(aids + row0 * k, blk * 8, peer_base, world, rank, region_off + ids_off + (size_t)row0 * k * 8));
        VIX_TRY(peer_barrier(c));
        status = reinterpret_cast<const int32_t*>(static_cast<char*>(c->local) + kStatusOffset);
    } else {
        VIX_TRY(st.alloc((size_t)world));
        const int32_t mine = rc;
        VIX_CUDA(cudaMemcpyAsync(st.ptr + rank, &mine, 4, cudaMemcpyHostToDevice, s));
        VIX_NCCL(g_nccl.AllGather(st.ptr + rank, st.ptr, 1, ncclInt32, c->comm, s));
        VIX_NCCL(g_nccl.AllGather(adist + row0 * k, adist, (size_t)per * k, ncclFloat, c->comm, s));
        VIX_NCCL(g_nccl.AllGather(aids + row0 * k, aids, (size_t)per * k, ncclInt64, c->comm, s));
        status = st.ptr;
    }
    const size_t total = (size_t)nq * k;
    VIX_CUDA(cudaMemcpyAsync(out_dist, adist, total * 4, cudaMemcpyDefault, s));
    VIX_CUDA(cudaMemcpyAsync(out_ids, aids, total * 8, cudaMemcpyDefault, s));
    mark(3);
    replica_debug_line(c, h, "knn", cnt, (int64_t)total, grown);
    if (rc != VIX_OK) return rc;                                      // (its own message stands)
    const bool sync = large || !ctx().async || !is_device_ptr(out_dist) || !is_device_ptr(out_ids);
    if (!sync) {
        replica_status_kernel<<<1, 32 * ((world + 31) / 32), 0, s>>>(status, world, pipeline_error_flag());
        VIX_LAUNCH_CHECK();
        return VIX_OK;
    }
    std::vector<int32_t> hs((size_t)world);
    VIX_CUDA(cudaMemcpyAsync(hs.data(), status, (size_t)world * 4, cudaMemcpyDeviceToHost, s));
    VIX_CUDA(cudaStreamSynchronize(s));
    for (int p = 0; p < world; ++p)
        VIX_REQUIRE(hs[p] == VIX_OK, hs[p], "%s: rank %d failed its local search (status %d); no rank returns a result", who, p, hs[p]);
    return finish(true);
}

}  // namespace vix

using namespace vix;

extern "C" {

int vix_replicated_search(vix_index_t* h, vix_comm_t* c, const float* queries, int64_t nq, int k, int nprobe, float* out_dist,
                          int64_t* out_ids) {
    return vix_replicated_search_filtered(h, c, queries, nq, k, nprobe, nullptr, 0, VIX_FILTER_ALLOW, out_dist, out_ids);
}

int vix_replicated_search_filtered(vix_index_t* h, vix_comm_t* c, const float* queries, int64_t nq, int k, int nprobe,
                                   const uint64_t* filter_words, int64_t filter_capacity, int filter_mode, float* out_dist,
                                   int64_t* out_ids) {
    const char* who = filter_words ? "vix_replicated_search_filtered" : "vix_replicated_search";
    VIX_TRY(ensure_device());
    VIX_REQUIRE(h && c, VIX_ERR_NULL_PTR, "%s: null handle", who);
    VIX_REQUIRE(filter_mode == VIX_FILTER_ALLOW || filter_mode == VIX_FILTER_DENY, VIX_ERR_INVALID_PARAM,
                "%s: filter_mode must be VIX_FILTER_ALLOW or VIX_FILTER_DENY", who);
    VIX_REQUIRE(filter_capacity >= 0, VIX_ERR_INVALID_PARAM, "%s: negative capacity", who);
    if (nq <= 0 || k <= 0) return VIX_OK;                             // IVFIndex.swift:866 (every rank sees the same nq, k)
    VIX_REQUIRE(queries && out_dist && out_ids, VIX_ERR_NULL_PTR, "%s: null pointer", who);
    VIX_REQUIRE(k <= VIX_MAX_K_LARGE, VIX_ERR_INVALID_K, "%s: k > %d", who, VIX_MAX_K_LARGE);
    VIX_REQUIRE(k <= VIX_MAX_K || nq < 0x7FFFFFFFLL, VIX_ERR_INVALID_PARAM, "%s: k > %d needs nq < 2^31 - 1", who, VIX_MAX_K);
    In<uint64_t> fw;
    FilterArgs f;
    const FilterArgs* fp = nullptr;
    VIX_TRY(stage_filter(filter_words, filter_capacity, filter_mode, fw, f, fp));
    return replicated_search(h, c, queries, nq, k, nprobe, fp, out_dist, out_ids);
}

int vix_replicated_range_search(vix_index_t* h, vix_comm_t* c, const float* queries, int64_t nq, float radius, int nprobe,
                                const uint64_t* filter_words, int64_t filter_capacity, int filter_mode, vix_range_result_t** out) {
    const char* who = "vix_replicated_range_search";
    VIX_TRY(ensure_device());
    VIX_REQUIRE(h && c && out, VIX_ERR_NULL_PTR, "%s: null pointer", who);
    *out = nullptr;
    VIX_REQUIRE(queries || nq == 0, VIX_ERR_NULL_PTR, "%s: null queries", who);
    VIX_REQUIRE(nq >= 0 && nq < 0x7FFFFFFFLL, VIX_ERR_INVALID_PARAM, "%s: nq must lie in [0, 2^31 - 1)", who);
    VIX_REQUIRE(radius == radius, VIX_ERR_INVALID_PARAM, "%s: radius is NaN", who);
    VIX_REQUIRE(filter_mode == VIX_FILTER_ALLOW || filter_mode == VIX_FILTER_DENY, VIX_ERR_INVALID_PARAM,
                "%s: filter_mode must be VIX_FILTER_ALLOW or VIX_FILTER_DENY", who);
    VIX_REQUIRE(filter_capacity >= 0, VIX_ERR_INVALID_PARAM, "%s: negative capacity", who);
    std::lock_guard<std::mutex> lc(c->mu);
    std::lock_guard<std::mutex> lk(h->mu);
    VIX_TRY(replica_check(h, who, false));
    VIX_TRY(replica_nprobe(h, &nprobe, who));
    if (nq == 0) return range_empty(0, out);                          // (every rank sees the same nq: no exchange)
    In<uint64_t> fw;
    FilterArgs f;
    const FilterArgs* fp = nullptr;
    VIX_TRY(stage_filter(filter_words, filter_capacity, filter_mode, fw, f, fp));
    const int world = c->world, rank = c->rank, d = h->p.d;
    if (world == 1) return index_range_locked(h, queries, nq, radius, nprobe, fp, out);
    cudaStream_t s = ctx().stream;
    VIX_TRY(ensure_region(c, nq, 4, 1, 1));
    const bool peer = c->peer_state == 1;
    bool grown = false;
    if (peer) VIX_TRY(ensure_range_region(c, nq, 0, &grown));
    const int64_t per = block_rows(nq, world);
    const int64_t lo = std::min<int64_t>(nq, (int64_t)rank * per);
    const int64_t cnt = std::min<int64_t>(nq, lo + per) - lo;
    auto mark = [&](int i) { if (c->trace) cudaEventRecord(c->ev[i], s); };
    mark(0);
    if (peer) VIX_TRY(peer_barrier(c));
    In<float> dq;
    VIX_TRY(dq.stage(queries + (size_t)lo * d, (size_t)cnt * d));
    mark(1);
    // the block's range search (one synchronisation: its total); a failure travels with the row starts, so that every rank
    // returns it together
    RangeKeys rk, whole;
    int rc = cnt > 0 ? index_range_locked(h, dq.dev, cnt, radius, nprobe, fp, nullptr, nullptr, &rk) : VIX_OK;
    if (rc == VIX_OK) rc = whole.lims.alloc((size_t)nq + 1);
    if (rc == VIX_OK) rc = replica_expand_lims(cnt > 0 ? rk.lims.ptr : nullptr, lo, cnt, nq, whole.lims.ptr);
    whole.sorted = cnt > 0 ? rk.sorted : nullptr;
    whole.total = cnt > 0 ? rk.total : 0;
    mark(2);
    vix_range_result* r = nullptr;
    ShardTail tail;
    tail.out = &r;
    tail.neg_zero = range_neg_zero(h);
    tail.concat = true;
    ShardTotals st;
    VIX_TRY(sharded_range_exchange(h, c, nq, rc, whole, grown, tail, &st));
    mark(3);
    replica_debug_line(c, h, "range", cnt, st.total, st.grown);
    *out = r;
    return VIX_OK;
}

int vix_replicated_add(vix_index_t* h, vix_comm_t* c, const float* x, const int64_t* ids, int64_t n) {
    const char* who = "vix_replicated_add";
    VIX_TRY(ensure_device());
    VIX_REQUIRE(h && c, VIX_ERR_NULL_PTR, "%s: null handle", who);
    VIX_REQUIRE(n >= 0 && (n == 0 || (x && ids)), VIX_ERR_NULL_PTR, "%s: null pointer (explicit ids are required)", who);
    std::lock_guard<std::mutex> lc(c->mu);
    std::lock_guard<std::mutex> lk(h->mu);
    VIX_TRY(replica_check(h, who, true));
    const int world = c->world, rank = c->rank, d = h->p.d;
    const bool pq = h->p.kind == VIX_INDEX_IVF_PQ, flat = h->p.kind == VIX_INDEX_FLAT;
    const int m = pq ? h->code_bytes() : 0;
    cudaStream_t s = ctx().stream;
    // 1. this rank's rows: the list assignment (IVF kinds), and the rows no rank may store -- no nearest list (NaN
    //    components) or an id outside [0, 2^32 - 1).  [rows, invalid rows, status] of every rank are all-gathered before any
    //    row travels, so every rank refuses together.
    In<float> dx;
    In<int64_t> dids;
    VIX_TRY(dx.stage(x, (size_t)n * d));
    VIX_TRY(dids.stage(ids, (size_t)n));
    Scratch<int32_t> asg;
    Scratch<unsigned long long> dcounts;
    VIX_TRY(dcounts.alloc(3 * ((size_t)world + 1)));
    unsigned long long* mine = dcounts.ptr + 3 * (size_t)world;
    const unsigned long long head[3] = {(unsigned long long)n, 0ull, 0ull};
    VIX_CUDA(cudaMemcpyAsync(mine, head, sizeof(head), cudaMemcpyHostToDevice, s));
    int rc = VIX_OK;
    if (n > 0 && flat) rc = count_invalid_ids_device(dids.dev, n, mine + 1);
    if (n > 0 && !flat) {
        rc = asg.alloc((size_t)n);
        if (rc == VIX_OK) rc = assign_lists_device(h, dx.dev, n, asg.ptr);
        if (rc == VIX_OK) rc = count_invalid_rows_device(asg.ptr, dids.dev, n, h->kc, mine + 1);
    }
    const unsigned long long st_word = (unsigned long long)(long long)rc;
    VIX_CUDA(cudaMemcpyAsync(mine + 2, &st_word, 8, cudaMemcpyHostToDevice, s));
    VIX_NCCL(g_nccl.AllGather(mine, dcounts.ptr, 3, ncclUint64, c->comm, s));
    std::vector<unsigned long long> counts(3 * (size_t)world);
    VIX_CUDA(cudaMemcpyAsync(counts.data(), dcounts.ptr, counts.size() * 8, cudaMemcpyDeviceToHost, s));
    VIX_CUDA(cudaStreamSynchronize(s));
    if (rc != VIX_OK) return rc;
    for (int p = 0; p < world; ++p) {
        const int sp = (int)(long long)counts[3 * (size_t)p + 2];
        VIX_REQUIRE(sp == VIX_OK, sp, "%s: rank %d failed to prepare its rows (status %d); no rank stored any row of this call", who,
                    p, sp);
    }
    for (int p = 0; p < world; ++p)
        VIX_REQUIRE(counts[3 * (size_t)p + 1] == 0, VIX_ERR_INVALID_PARAM,
                    "%s: rank %d was handed %llu rows with no nearest list (NaN components?) or an id outside [0, 2^32 - 1); no "
                    "rank stored any row of this call", who, p, counts[3 * (size_t)p + 1]);
    std::vector<int64_t> off((size_t)world + 1, 0);
    for (int p = 0; p < world; ++p) off[p + 1] = off[p] + (int64_t)counts[3 * (size_t)p];
    const int64_t N = off[world];
    if (N == 0) return VIX_OK;
    // 2. IVF-PQ: encode the rows (after the check: every assignment is a list)
    Scratch<uint8_t> codes;
    if (pq && n > 0) {
        VIX_TRY(codes.alloc((size_t)n * m));
        VIX_TRY(encode_rows_device(h, dx.dev, n, asg.ptr, codes.ptr));
    }
    // 3. every rank's rows reach every rank, rank by rank: ids [N] i64, then (256-aligned) assignments [N] i32, then vectors
    //    [N x d] f32 or codes [N x m] u8
    const size_t o_asg = ((size_t)N * 8 + 255) & ~(size_t)255;
    const size_t o_row = flat ? o_asg : (o_asg + (size_t)N * 4 + 255) & ~(size_t)255;
    const size_t row_bytes = pq ? (size_t)m : (size_t)d * 4;
    const size_t bytes = o_row + (size_t)N * row_bytes;
    const void* my_rows = pq ? static_cast<const void*>(codes.ptr) : static_cast<const void*>(dx.dev);
    const int64_t o = off[rank];
    char* base = nullptr;
    Scratch<char> gathered;
    if (world > 1) VIX_TRY(ensure_region(c, 1, 4, 1, 1));
    if (world == 1) {
        if (flat) VIX_TRY(index_add_rows_locked(h, dx.dev, dids.dev, n));
        else if (pq) VIX_TRY(index_add_encoded_locked(h, asg.ptr, codes.ptr, dids.dev, n));
        else VIX_TRY(index_add_assigned_locked(h, asg.ptr, dx.dev, dids.dev, n));
        return finish(true);
    } else if (c->peer_state == 1) {
        bool grown = false;
        VIX_TRY(ensure_range_region(c, 0, (int64_t)((bytes + 7) / 8), &grown));
        VIX_TRY(peer_barrier(c));                                     // every peer has read what the last call left here
        const size_t ro = c->range_off_keys;
        VIX_TRY(replica_store(dids.dev, (size_t)n * 8, c->range_peer_dev, world, -1, ro + (size_t)o * 8));
        if (!flat) VIX_TRY(replica_store(asg.ptr, (size_t)n * 4, c->range_peer_dev, world, -1, ro + o_asg + (size_t)o * 4));
        VIX_TRY(replica_store(my_rows, (size_t)n * row_bytes, c->range_peer_dev, world, -1, ro + o_row + (size_t)o * row_bytes));
        VIX_TRY(peer_barrier(c));
        base = static_cast<char*>(c->range_local) + ro;
        replica_debug_line(c, h, "add", n, N, grown);
    } else {
        VIX_TRY(gathered.alloc(bytes));
        base = gathered.ptr;
        VIX_NCCL(g_nccl.GroupStart());
        for (int p = 0; p < world; ++p) {
            const int64_t np_ = off[p + 1] - off[p];
            if (p == rank) continue;
            if (n > 0) {
                VIX_NCCL(g_nccl.Send(dids.dev, (size_t)n, ncclInt64, p, c->comm, s));
                if (!flat) VIX_NCCL(g_nccl.Send(asg.ptr, (size_t)n, ncclInt32, p, c->comm, s));
                VIX_NCCL(g_nccl.Send(my_rows, (size_t)n * row_bytes, ncclUint8, p, c->comm, s));
            }
            if (np_ > 0) {
                VIX_NCCL(g_nccl.Recv(base + (size_t)off[p] * 8, (size_t)np_, ncclInt64, p, c->comm, s));
                if (!flat) VIX_NCCL(g_nccl.Recv(base + o_asg + (size_t)off[p] * 4, (size_t)np_, ncclInt32, p, c->comm, s));
                VIX_NCCL(g_nccl.Recv(base + o_row + (size_t)off[p] * row_bytes, (size_t)np_ * row_bytes, ncclUint8, p, c->comm, s));
            }
        }
        VIX_NCCL(g_nccl.GroupEnd());
        if (n > 0) {
            VIX_CUDA(cudaMemcpyAsync(base + (size_t)o * 8, dids.dev, (size_t)n * 8, cudaMemcpyDeviceToDevice, s));
            if (!flat) VIX_CUDA(cudaMemcpyAsync(base + o_asg + (size_t)o * 4, asg.ptr, (size_t)n * 4, cudaMemcpyDeviceToDevice, s));
            VIX_CUDA(cudaMemcpyAsync(base + o_row + (size_t)o * row_bytes, my_rows, (size_t)n * row_bytes, cudaMemcpyDeviceToDevice, s));
        }
        replica_debug_line(c, h, "add", n, N, false);
    }
    // 4. every replica appends all rows, rank 0's first
    const int64_t* all_ids = reinterpret_cast<const int64_t*>(base);
    const int32_t* all_asg = reinterpret_cast<const int32_t*>(base + o_asg);
    if (flat) VIX_TRY(index_add_rows_locked(h, reinterpret_cast<const float*>(base + o_row), all_ids, N));
    else if (pq) VIX_TRY(index_add_encoded_locked(h, all_asg, reinterpret_cast<const uint8_t*>(base + o_row), all_ids, N));
    else VIX_TRY(index_add_assigned_locked(h, all_asg, reinterpret_cast<const float*>(base + o_row), all_ids, N));
    return finish(true);
}

int vix_debug_replica_assemble(const int64_t* lims_all, const float* dist_all, const int64_t* ids_all, int world, int64_t nq, int k,
                               int metric, int kind, float* out_dist, int64_t* out_ids, vix_range_result_t** out_range) {
    const char* who = "vix_debug_replica_assemble";
    VIX_TRY(ensure_device());
    VIX_REQUIRE(world > 0 && world <= 256 && nq >= 0 && nq < 0x7FFFFFFFLL, VIX_ERR_INVALID_PARAM, "%s: world / nq", who);
    VIX_REQUIRE(kind == VIX_INDEX_FLAT || kind == VIX_INDEX_IVF_FLAT || kind == VIX_INDEX_IVF_PQ, VIX_ERR_INVALID_PARAM, "%s: kind", who);
    cudaStream_t s = ctx().stream;
    const int64_t per = block_rows(nq, world);
    if (!out_range) {
        // k-NN: every rank stores its block into every other rank's buffer at the block's rows (its own buffer holds it
        // already, as its search wrote it there); the answer is read from the last rank's buffer
        VIX_REQUIRE(k > 0 && k <= VIX_MAX_K_LARGE, VIX_ERR_INVALID_PARAM, "%s: k", who);
        VIX_REQUIRE(nq == 0 || (dist_all && ids_all && out_dist && out_ids), VIX_ERR_NULL_PTR, "%s: null pointer", who);
        if (nq == 0) return VIX_OK;
        const size_t total = (size_t)nq * k;
        // (each emulated region 256-aligned, as the cudaMalloc'ed regions of the exchange are: the stores use 16-byte words)
        const size_t ids_off = (total * 4 + 255) & ~(size_t)255, bytes = (ids_off + total * 8 + 255) & ~(size_t)255;
        In<float> dd;
        In<int64_t> di;
        VIX_TRY(dd.stage(dist_all, total));
        VIX_TRY(di.stage(ids_all, total));
        Scratch<char> regions;
        Scratch<void*> bases;
        VIX_TRY(regions.alloc(bytes * world));
        VIX_TRY(bases.alloc((size_t)world));
        std::vector<void*> hb((size_t)world);
        for (int r = 0; r < world; ++r) hb[r] = regions.ptr + bytes * r;
        VIX_CUDA(cudaMemcpyAsync(bases.ptr, hb.data(), sizeof(void*) * world, cudaMemcpyHostToDevice, s));
        for (int r = 0; r < world; ++r) {
            const int64_t lo = std::min<int64_t>(nq, (int64_t)r * per), cnt = std::min<int64_t>(nq, lo + per) - lo;
            if (cnt == 0) continue;
            char* own = static_cast<char*>(hb[r]);
            VIX_CUDA(cudaMemcpyAsync(own + (size_t)lo * k * 4, dd.dev + lo * k, (size_t)cnt * k * 4, cudaMemcpyDeviceToDevice, s));
            VIX_CUDA(cudaMemcpyAsync(own + ids_off + (size_t)lo * k * 8, di.dev + lo * k, (size_t)cnt * k * 8, cudaMemcpyDeviceToDevice, s));
            VIX_TRY(replica_store(own + (size_t)lo * k * 4, (size_t)cnt * k * 4, bases.ptr, world, r, (size_t)lo * k * 4));
            VIX_TRY(replica_store(own + ids_off + (size_t)lo * k * 8, (size_t)cnt * k * 8, bases.ptr, world, r, ids_off + (size_t)lo * k * 8));
        }
        const char* last = static_cast<const char*>(hb[world - 1]);
        VIX_CUDA(cudaMemcpyAsync(out_dist, last, total * 4, cudaMemcpyDefault, s));
        VIX_CUDA(cudaMemcpyAsync(out_ids, last + ids_off, total * 8, cudaMemcpyDefault, s));
        return finish(true);
    }
    // range: lims_all holds every rank's block row starts (count_r + 1 each, rank by rank: nq + world in all); the rows
    // follow rank by rank.  They become the exchanged layout (row starts over the whole batch, status 0), keys, the global
    // row starts, and the concatenation.
    *out_range = nullptr;
    VIX_REQUIRE(lims_all, VIX_ERR_NULL_PTR, "%s: null lims", who);
    std::vector<int64_t> hl((size_t)nq + world);
    VIX_CUDA(cudaMemcpyAsync(hl.data(), lims_all, hl.size() * 8, cudaMemcpyDefault, s));
    VIX_CUDA(cudaStreamSynchronize(s));
    const int64_t L = nq + 2;
    std::vector<int64_t> h_all((size_t)world * L, 0);
    int64_t total = 0;
    for (int r = 0, at = 0; r < world; ++r) {
        const int64_t lo = std::min<int64_t>(nq, (int64_t)r * per), cnt = std::min<int64_t>(nq, lo + per) - lo;
        const int64_t* b = hl.data() + at;
        VIX_REQUIRE(b[0] == 0, VIX_ERR_INVALID_PARAM, "%s: rank %d: lims[0] != 0", who, r);
        for (int64_t j = 0; j < cnt; ++j) VIX_REQUIRE(b[j + 1] >= b[j], VIX_ERR_INVALID_PARAM, "%s: rank %d: lims descend", who, r);
        for (int64_t q = 0; q <= nq; ++q) h_all[(size_t)r * L + q] = q <= lo ? 0 : q >= lo + cnt ? b[cnt] : b[q - lo];
        total += b[cnt];
        at += (int)(cnt + 1);
    }
    VIX_REQUIRE(total == 0 || (dist_all && ids_all), VIX_ERR_NULL_PTR, "%s: null rows", who);
    Scratch<int64_t> dlims, glims;
    Scratch<u64> keys;
    In<float> dd;
    In<int64_t> di;
    VIX_TRY(dlims.alloc(h_all.size()));
    VIX_TRY(glims.alloc((size_t)nq + 1));
    VIX_CUDA(cudaMemcpyAsync(dlims.ptr, h_all.data(), h_all.size() * 8, cudaMemcpyHostToDevice, s));
    VIX_TRY(dd.stage(dist_all, (size_t)total));
    VIX_TRY(di.stage(ids_all, (size_t)total));
    VIX_TRY(keys.alloc((size_t)total));
    if (total > 0) {
        replica_pack_keys_kernel<<<(unsigned)((total + 255) / 256), 256, 0, s>>>(dd.dev, di.dev, total, keys.ptr);
        VIX_LAUNCH_CHECK();
    }
    std::vector<int64_t> meta;
    VIX_TRY(shard_range_lims(dlims.ptr, world, nq, glims.ptr, meta));
    vix_range_result* r = nullptr;
    VIX_TRY(range_alloc(nq, total, &r));
    int rc = replica_range_concat(keys.ptr, glims.ptr, nq, total, kind != VIX_INDEX_IVF_FLAT && metric == VIX_METRIC_IP, r);
    if (rc == VIX_OK) rc = finish(true);
    if (rc != VIX_OK) { range_free(r); return rc; }
    *out_range = r;
    return VIX_OK;
}

}  // extern "C"
