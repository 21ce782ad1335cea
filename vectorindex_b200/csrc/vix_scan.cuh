// vix_scan.cuh -- interface between the index handles (vix_index.cu) and the fused IVF-PQ scan
// (vix_ivfpq_scan.cu).
#pragma once

#include "vix_common.cuh"
#include "vix_range.cuh"

namespace vix {

struct ScanArgs {
    const float* queries; int64_t nq; int d, m, ks, dsub;
    const int32_t* probes; int nprobe;            // [nq x nprobe], -1 padded
    const int32_t* order;                         // optional [nq]: work item -> query (locality order)
    const int* nq_dev;                            // optional (device): number of work items, when only the host does not know it
                                                  // (then `order` lists them and nq bounds the launch)
    int* work_counter;                            // device int[2], zeroed by the launcher: [0] queue head, [1] status
    int* status;                                  // set by the launcher (= work_counter + 1)
    int smem_bytes;                               // dynamic shared memory of the launch (set by the launcher)
    const float* coarse; int kc;                  // [kc x d]; probe ids outside [0, kc) are treated like the -1 padding
    const float* bias;                            // optional [nq x nprobe]: the per-probe term, precomputed batch-wide (large d)
    const float* lut_image;                       // optional [nq][tables][256 codes][32 slots]: the look-up tables of every query,
                                                  // compact (the scan makes the two replicas of a shared-memory row while
                                                  // copying); built batch-wide when the codebooks are large
    const float* codebooks;                       // [m x ks x dsub]
    const float* codebooks_t;                     // [ks x m x dsub]  (code-major copy for the LUT build)
    const uint32_t* tc_table; const float* tc_meta;  // optional: the list-major path's decode table + its scale / norm bound,
                                                  // built once per codebooks (tc_decode_table); absent -> built per launch
    const int64_t* list_off; const int32_t* list_len;
    const uint8_t* slot_codes; const float* slot_tx; const int64_t* slot_ids;
    const uint8_t* tc_codes;                      // the decode layout of slot_codes (below); the list-major path needs it
    // optional id filter (IDFilter.swift:115-135): ids outside [0, filter_cap) never pass; allowlist keeps set bits,
    // denylist keeps clear bits.  Applied BEFORE selection (pre-filter, IVFIndex.swift:813, 1034).
    const uint64_t* filter; int64_t filter_cap; int filter_deny;
    int metric, k, Pw, P2;
    float* out_dist; int64_t* out_ids;            // [nq x k]
    unsigned long long* scanned;                  // optional: total list entries visited
    cudaEvent_t ev_kernel[2];                     // optional: recorded around the dominant kernel of the launch
    int path;                                     // set by launch_ivfpq_scan: 0 query-major, 1 list-major (tensor cores)
    unsigned long long* phase_cycles;             // optional [3]: SM cycles in prologue / scan / tail wait, summed over CTAs
    RangeOut range;                               // range search (range.keys set): entries within range.radius go here instead
                                                  // of the top-k; launch_ivfpq_scan_classic only
};

// How the inverted lists are laid out for a given m.
//   fast:  the 16 codes of every group of 16 sub-quantisers "rotated" by the slot index (byte b of slot g holds
//          sub-quantiser (b & ~15) | ((b ^ g) & 15)) and stored chunk-blocked: inside a 32-slot chunk the 16-byte
//          piece c of slot s sits at chunk * 32 m + c * 512 + s * 16;
//   else:  plain AoS rows.  Lists start at multiples of `align` slots either way.
struct ScanLayout {
    bool fast;
    int align;    // list start / padded length granularity in slots
};
ScanLayout scan_layout(int m);

// Sharded search (vix_sharded.cu): the list-major path filters against an upper bound of every query's k-th best distance;
// on a shard the bound of a query whose near lists live on OTHER ranks is loose unless the ranks share their bounds.  The
// hook (thread-local, set around the call) is handed the per-query bounds [nq] on the stream and replaces them by the
// minimum over the ranks.  Every rank takes the same path (same shapes, same device), so the collective is matched.
typedef int (*scan_thr_hook_t)(void* ctx, float* thr_dev, int64_t nq);
void set_scan_thr_hook(scan_thr_hook_t fn, void* ctx);

int launch_ivfpq_scan(ScanArgs& a);            // picks the path
bool tc_scan_supported(const ScanArgs& a);     // would launch_ivfpq_scan take the list-major tensor-core path (vix_ivfpq_tc.cu)?
int launch_ivfpq_scan_classic(ScanArgs& a);    // query-major look-up-table scan (vix_ivfpq_scan.cu)
// bias[q x nprobe]: the per-probe term, batch-wide; with `only_flagged` [nq] just the rows of the queries flagged there
int launch_probe_bias(const ScanArgs& a, float* bias, const int* only_flagged = nullptr);
// the list-major path's decode table of a set of codebooks (dsub = 2, ks = 256, m in {16, 32, 48, 64}): table
// [kTcTableWords] fp16 pairs, meta [4] floats ([1] the table's scale, [2] the bound of a decoded residual's norm)
constexpr size_t kTcTableWords = 2 * 256 * 64;
bool tc_decode_table_shape(int m, int ks, int dsub);
// The decode layout: a second copy of the codes that only the list-major scan's decoders read (the rotated layout above
// stays the one every exact key is computed from).  Chunk-blocked like the rotated layout -- the 512-byte block of chunk
// and group grp at the same offset -- but inside a block thread t = 4 r + c (r = 0..7, c = 0..3) of the decoding warp owns
// bytes [16 t, 16 t + 16), and byte 4 v + s holds the code of slot r + 8 v, sub-quantiser 16 grp + 4 (s ^ (r & 3)) + c.
// Built for L2 indexes of the decode table's shape (tc_codes_shape), which are the only ones the list-major path takes.
bool tc_codes_shape(int metric, int m, int ks, int dsub);
int tc_decode_table(const float* codebooks, int m, uint32_t* table, float* meta);
// the list-major path's seed alone: thr[q] = the k-th smallest exact key of the first 256 vectors of the query's first
// probed list that holds vectors (+inf: fewer than k of them); k <= 64, the shapes of tc_codes_shape
int tc_seed_thresholds(const ScanArgs& a, float* thr);

}  // namespace vix
