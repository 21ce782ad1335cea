// vix_group.cuh -- grouping rows by a small integer key (list, centroid, code, owning rank) for the build side: the list
// build, both trainers, the sharded add and removal.  vix_group.cu is the only translation unit that calls CUB; the search
// path groups with counting sorts of its own and calls none of these.
//
// All functions take device pointers, run on the context stream without synchronising it, and count their launches.
#pragma once

#include "vix_common.cuh"

namespace vix {

// CUB's stable LSD radix sorts over bits [0, bits) of the keys (K = int32_t or uint32_t), and its exclusive prefix sum
template <typename K>
int sort_pairs(const K* keys_in, K* keys_out, const int32_t* vals_in, int32_t* vals_out, int64_t n, int bits);
int sort_keys(const uint32_t* keys_in, uint32_t* keys_out, int64_t n);          // all 32 bits
int exclusive_sum(const int32_t* in, int32_t* out, int64_t n);

// order[i] = the row at position i once rows are stably sorted by keys in [0, nkeys) (ceil(log2(nkeys)) key bits, at
// least 1); keys_sorted (optional) receives the keys in that order
int order_by_key(const int32_t* keys, int64_t n, int nkeys, int32_t* order, int32_t* keys_sorted = nullptr);
// counts[k] = rows with key k (keys outside [0, nkeys) are skipped), then offsets_from_counts
int key_offsets(const int32_t* keys, int64_t n, int nkeys, int32_t* counts, int64_t* off, int align = 1,
                int64_t* off_raw = nullptr);
// off[k + 1] = off[k] + roundup(counts[k], align) with off[0] = 0; off_raw (optional): the same with align 1
int offsets_from_counts(const int32_t* counts, int nkeys, int align, int64_t* off, int64_t* off_raw);

template <typename T> int iota(T* a, int64_t n, T start);                       // a[i] = start + i
template <typename T> int fill(T* a, int64_t n, T v);                           // a[i] = v
// out[i][0, d) = x[rows[i]][0, d) for i < n (I = int32_t or int64_t)
template <typename I> int gather_rows(const float* x, int d, const I* rows, int64_t n, float* out);
// out[r] = sum over e of c[r][e]^2, summed in order with separate rounded multiply and add (PQTrain.swift:299-307)
int seq_norms(const float* c, int64_t rows, int dsub, float* out);

}  // namespace vix
