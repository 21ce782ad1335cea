/* The sharded flat and IVF-Flat indexes from a plain C11 host, one rank: vix_comm_create over a one-rank communicator ->
 * vix_sharded_add -> vix_sharded_search (k = 10 and k = 600, the route beyond 512) -> vix_sharded_range_search, for a flat
 * and an IVF-Flat handle.  Each answer must equal, byte for byte, the one-GPU calls on an index that received the same rows
 * through vix_index_add.  Built and run by tests/test_sharded_kinds.py; prints "sharded kinds ok". */
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "vindex_cuda.h"

enum { D = 16, N = 3000, NQ = 17, KC = 12 };

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

int main(void) {
    if (vix_device_count() < 1) {
        printf("no device\n");
        return 2;
    }
    static float x[N * D], q[NQ * D], coarse[KC * D];
    static int64_t ids[N];
    uint64_t s = 12345;
    for (int i = 0; i < N * D; ++i) x[i] = frand(&s);
    for (int i = 0; i < NQ * D; ++i) q[i] = frand(&s);
    for (int i = 0; i < KC * D; ++i) coarse[i] = x[i * 7];
    for (int i = 0; i < N; ++i) ids[i] = 5 * (int64_t)(N - i);
    unsigned char id[128];
    CHECK(vix_comm_unique_id(id, sizeof id));
    vix_comm_t* comm = NULL;
    CHECK(vix_comm_create(id, sizeof id, 0, 1, &comm));
    const int kinds[2] = {VIX_INDEX_FLAT, VIX_INDEX_IVF_FLAT};
    static float d1[NQ * 600], d2[NQ * 600];
    static int64_t i1[NQ * 600], i2[NQ * 600];
    for (int t = 0; t < 2; ++t) {
        vix_index_t *sh = NULL, *one = NULL;
        if (make(kinds[t], coarse, &sh) || make(kinds[t], coarse, &one)) return 1;
        CHECK(vix_sharded_add(sh, comm, NULL, x, ids, N));
        CHECK(vix_index_add(one, x, ids, N));
        const int ks[2] = {10, 600};
        for (int j = 0; j < 2; ++j) {
            const int k = ks[j];
            CHECK(vix_sharded_search(sh, comm, q, NQ, k, 0, d1, i1));
            CHECK(vix_index_search(one, q, NQ, k, 0, d2, i2));
            if (memcmp(d1, d2, sizeof(float) * NQ * k) || memcmp(i1, i2, sizeof(int64_t) * NQ * k)) {
                fprintf(stderr, "kind %d, k %d: sharded != one GPU\n", kinds[t], k);
                return 1;
            }
        }
        vix_range_result_t *ra = NULL, *rb = NULL;
        const float radius = d2[5];
        CHECK(vix_sharded_range_search(sh, comm, q, NQ, radius, 0, NULL, 0, VIX_FILTER_ALLOW, &ra));
        CHECK(vix_index_range_search(one, q, NQ, radius, 0, NULL, 0, VIX_FILTER_ALLOW, &rb));
        const int ok = range_equal(ra, rb);
        vix_range_result_destroy(ra);
        vix_range_result_destroy(rb);
        if (!ok) {
            fprintf(stderr, "kind %d: sharded range search != one GPU\n", kinds[t]);
            return 1;
        }
        printf("kind %d: add, search (k 10, 600), range search equal to one GPU\n", kinds[t]);
        vix_index_destroy(sh);
        vix_index_destroy(one);
    }
    CHECK(vix_comm_destroy(comm));
    printf("sharded kinds ok\n");
    return 0;
}
