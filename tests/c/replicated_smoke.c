/* Replicated indexes from a plain C11 host (no Python, no MPI): the parent forks one process per GPU and hands the NCCL id of
 * rank 0 to the others through pipes.  Every rank holds a whole flat index and a whole IVF-Flat index, contributes its own
 * slice of the rows through vix_replicated_add, and runs vix_replicated_search (k = 10 and k = 600, the route beyond 512),
 * vix_replicated_search_filtered and vix_replicated_range_search.  Every answer must equal, byte for byte, the one-GPU calls
 * on an index that received all rows, rank 0's slice first, through vix_index_add; then every replica removes the same ids
 * with vix_index_remove and the k-NN answer is checked again.  Built and run by tests/test_replicated.py with 1 or 2 ranks;
 * every rank prints "replicated == single-GPU: yes" on success. */
#define _POSIX_C_SOURCE 200809L
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <sys/types.h>
#include <sys/wait.h>
#include <unistd.h>

#include "vindex_cuda.h"

enum { D = 16, N = 3001, NQ = 19, KC = 12, KMAX = 600 };

static float frand(uint64_t* s) {
    *s = *s * 6364136223846793005ULL + 1442695040888963407ULL;
    return (float)((*s >> 40) & 0xFFFFFF) / 16777216.0f * 2.0f - 1.0f;
}

#define CHECK(call)                                                                   \
    do {                                                                              \
        int rc_ = (call);                                                             \
        if (rc_ != VIX_OK) {                                                          \
            fprintf(stderr, "%s -> %d (%s)\n", #call, rc_, vix_last_error());         \
            return 1;                                                                 \
        }                                                                             \
    } while (0)

static int make(int kind, const float* coarse, vix_index_t** out) {
    vix_index_params p;
    vix_index_params_default(&p);
    p.kind = kind;
    p.d = D;
    p.metric = VIX_METRIC_L2;
    p.nlist = KC;
    p.nprobe = 4;
    CHECK(vix_index_create(&p, out));
    if (kind == VIX_INDEX_IVF_FLAT) CHECK(vix_index_set_coarse(*out, coarse, KC));
    return 0;
}

static int range_equal(vix_range_result_t* a, vix_range_result_t* b) {
    const int64_t ta = vix_range_result_total(a), tb = vix_range_result_total(b);
    if (ta != tb) return 0;
    int64_t la[NQ + 1], lb[NQ + 1];
    float* da = malloc(sizeof(float) * (size_t)(ta + 1));
    float* db = malloc(sizeof(float) * (size_t)(ta + 1));
    int64_t* ia = malloc(sizeof(int64_t) * (size_t)(ta + 1));
    int64_t* ib = malloc(sizeof(int64_t) * (size_t)(ta + 1));
    int ok = da && db && ia && ib && vix_range_result_get(a, la, da, ia) == VIX_OK && vix_range_result_get(b, lb, db, ib) == VIX_OK &&
             !memcmp(la, lb, sizeof la) && !memcmp(da, db, sizeof(float) * (size_t)ta) && !memcmp(ia, ib, sizeof(int64_t) * (size_t)ta);
    free(da); free(db); free(ia); free(ib);
    return ok;
}

static float x[N * D], q[NQ * D], coarse[KC * D];
static int64_t ids[N];
static float d1[NQ * KMAX], d2[NQ * KMAX];
static int64_t i1[NQ * KMAX], i2[NQ * KMAX];

static int knn_equal(vix_index_t* one, vix_index_t* rep, vix_comm_t* c, int k, const uint64_t* words, int64_t cap) {
    if (words) {
        if (vix_index_search_filtered(one, q, NQ, k, 0, words, cap, VIX_FILTER_ALLOW, d1, i1) != VIX_OK) return 0;
        if (vix_replicated_search_filtered(rep, c, q, NQ, k, 0, words, cap, VIX_FILTER_ALLOW, d2, i2) != VIX_OK) return 0;
    } else {
        if (vix_index_search(one, q, NQ, k, 0, d1, i1) != VIX_OK) return 0;
        if (vix_replicated_search(rep, c, q, NQ, k, 0, d2, i2) != VIX_OK) return 0;
    }
    return !memcmp(d1, d2, sizeof(float) * (size_t)NQ * k) && !memcmp(i1, i2, sizeof(int64_t) * (size_t)NQ * k);
}

static int run_rank(int rank, int world, const unsigned char* id) {
    CHECK(vix_set_device(rank));
    vix_comm_t* c = NULL;
    CHECK(vix_comm_create(id, 128, rank, world, &c));
    uint64_t s = 7;
    for (int i = 0; i < N * D; ++i) x[i] = frand(&s);
    for (int i = 0; i < NQ * D; ++i) q[i] = frand(&s);
    for (int i = 0; i < KC * D; ++i) coarse[i] = frand(&s);
    for (int i = 0; i < N; ++i) ids[i] = 5 + 2 * (int64_t)i;
    uint64_t words[(5 + 2 * N + 63) / 64];
    memset(words, 0, sizeof words);
    for (int i = 0; i < N; i += 3) words[ids[i] >> 6] |= 1ull << (ids[i] & 63);
    const int64_t cap = 5 + 2 * N;
    int all = 1;
    for (int kind = VIX_INDEX_FLAT; kind <= VIX_INDEX_IVF_FLAT; ++kind) {
        vix_index_t *one = NULL, *rep = NULL;
        if (make(kind, coarse, &one) || make(kind, coarse, &rep)) return 1;
        CHECK(vix_index_add(one, x, ids, N));
        /* this rank's slice of the rows: ragged (rank 0 takes one row more), rank order = the one-GPU order */
        const int64_t per = N / world, lo = rank == 0 ? 0 : rank * per + 1, hi = rank == world - 1 ? N : (rank + 1) * per + 1;
        CHECK(vix_replicated_add(rep, c, x + lo * D, ids + lo, world == 1 ? N : hi - lo));
        int ok = vix_index_count(rep) == N;
        ok = ok && knn_equal(one, rep, c, 10, NULL, 0) && knn_equal(one, rep, c, KMAX, NULL, 0);
        ok = ok && knn_equal(one, rep, c, 10, words, cap) && knn_equal(one, rep, c, KMAX, words, cap);
        vix_range_result_t *ra = NULL, *rb = NULL;
        CHECK(vix_index_range_search(one, q, NQ, 1.4f, 0, NULL, 0, VIX_FILTER_ALLOW, &ra));
        CHECK(vix_replicated_range_search(rep, c, q, NQ, 1.4f, 0, NULL, 0, VIX_FILTER_ALLOW, &rb));
        ok = ok && vix_range_result_total(ra) > 0 && range_equal(ra, rb);
        vix_range_result_destroy(ra);
        vix_range_result_destroy(rb);
        /* remove: every replica passes the same ids to vix_index_remove */
        int64_t gone1 = 0, gone2 = 0;
        CHECK(vix_index_remove(one, ids, 500, &gone1));
        CHECK(vix_index_remove(rep, ids, 500, &gone2));
        ok = ok && gone1 == 500 && gone2 == 500 && knn_equal(one, rep, c, 10, NULL, 0);
        printf("rank %d %s: replicated == single-GPU: %s\n", rank, kind == VIX_INDEX_FLAT ? "flat" : "ivfflat", ok ? "yes" : "NO");
        all = all && ok;
        vix_index_destroy(one);
        vix_index_destroy(rep);
    }
    CHECK(vix_comm_destroy(c));
    return all ? 0 : 1;
}

int main(int argc, char** argv) {
    const int world = argc > 1 ? atoi(argv[1]) : 1;
    /* no CUDA call before the forks (a forked child cannot use a CUDA context its parent initialised) */
    int pipes[64][2];
    pid_t pids[64];
    if (world < 1 || world > 64) return 2;
    for (int r = 1; r < world; ++r) {
        if (pipe(pipes[r]) != 0) return 3;
        pids[r] = fork();
        if (pids[r] == 0) {
            unsigned char id[128];
            close(pipes[r][1]);
            size_t got = 0;
            while (got < sizeof(id)) { ssize_t n = read(pipes[r][0], id + got, sizeof(id) - got); if (n <= 0) return 4; got += (size_t)n; }
            return run_rank(r, world, id);
        }
        close(pipes[r][0]);
    }
    unsigned char id[128];
    if (vix_comm_unique_id(id, sizeof(id)) != VIX_OK) { fprintf(stderr, "vix_comm_unique_id: %s\n", vix_last_error()); return 5; }
    for (int r = 1; r < world; ++r) { if (write(pipes[r][1], id, sizeof(id)) != (ssize_t)sizeof(id)) return 6; close(pipes[r][1]); }
    int rc = run_rank(0, world, id);
    for (int r = 1; r < world; ++r) { int st = 0; waitpid(pids[r], &st, 0); if (!WIFEXITED(st) || WEXITSTATUS(st) != 0) rc = rc ? rc : 20 + r; }
    return rc;
}
