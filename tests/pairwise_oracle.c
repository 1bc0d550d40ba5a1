/*
 * pairwise_oracle.c -- CPU ORACLE (test infrastructure, NOT product code) of calculate_pairwise_differences
 * (reference: SauersML/ferromic, src/stats.rs:4106-4231).  Built on first use by tests/pairwise_oracle.py.
 *
 * PARITY UNPINNED: the reference tree was not available when this was written and no reference test holds a
 * golden vector for it; the definition below (DESIGN.md §3) is a reading of the function body that has not been
 * compared with the source.
 *
 * The direct loop of the definition: pairs (i < j) of 0 .. sample_count-1 outer, in the order (0,1), (0,2), ...,
 * (1,2), ..., variants inner.  A pair is comparable at a variant when both Option genotypes are Some, and differs
 * when the two genotypes differ as whole ordered vectors (phase and length both count).  Genotypes follow
 * CompressedGenotypes (process.rs:430-536): gt[(v*n_samples + s)*stride + k], 0xFF in slot 0 => None, a later 0xFF
 * ends the genotype; samples beyond a variant's genotype list are None.
 */
#include <pthread.h>
#include <stddef.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#define PW_MISSING 0xFFu /* process.rs:438 CompressedGenotypes::MISSING */

/* same field order as orc_variants (oracle/ferromic_oracle.h) */
typedef struct {
    size_t n_variants, n_samples, stride;
    const int64_t *positions; /* 0-based */
    const uint8_t *gt;
} pw_variants;

/* genotype length, 0 => None (CompressedGenotypes::get, process.rs:479-496) */
static inline size_t gt_get(const pw_variants *vs, size_t v, size_t s, const uint8_t **gt) {
    if (s >= vs->n_samples || vs->stride == 0) return 0;
    const uint8_t *p = vs->gt + (v * vs->n_samples + s) * vs->stride;
    if (p[0] == PW_MISSING) return 0;
    size_t len = 0;
    while (len < vs->stride && p[len] != PW_MISSING) len++;
    *gt = p;
    return len;
}

static inline void pairwise_one(const pw_variants *vs, size_t i, size_t j, uint32_t *diff, uint32_t *comp,
                                int64_t *positions) {
    uint32_t d = 0, c = 0;
    for (size_t v = 0; v < vs->n_variants; v++) {
        const uint8_t *gi = NULL, *gj = NULL;
        const size_t li = gt_get(vs, v, i, &gi), lj = gt_get(vs, v, j, &gj);
        if (li == 0 || lj == 0) continue;
        c++;
        if (li != lj || memcmp(gi, gj, li) != 0) {
            if (positions) positions[d] = vs->positions[v];
            d++;
        }
    }
    *diff = d;
    if (comp) *comp = c;
}

/* differences / comparable [n_pairs]; comparable, pair_start [n_pairs + 1] and positions (room for every
 * difference; pair p's positions in site order at positions[pair_start[p]..]) may be NULL. */
void pw_pairwise_differences(const pw_variants *vs, size_t sample_count, uint32_t *differences, uint32_t *comparable,
                             uint64_t *pair_start, int64_t *positions) {
    size_t p = 0;
    uint64_t off = 0;
    for (size_t i = 0; i < sample_count; i++)
        for (size_t j = i + 1; j < sample_count; j++, p++) {
            if (pair_start) pair_start[p] = off;
            pairwise_one(vs, i, j, &differences[p], comparable ? &comparable[p] : NULL, positions ? positions + off : NULL);
            off += differences[p];
        }
    if (pair_start) pair_start[p] = off;
}

typedef struct {
    const pw_variants *vs;
    size_t n, t, nthreads;
    uint32_t *diff, *comp;
} pairwise_job;

static void *pairwise_worker(void *arg) {
    pairwise_job *jb = (pairwise_job *)arg;
    for (size_t i = jb->t; i < jb->n; i += jb->nthreads) { /* rows interleaved: row lengths fall with i */
        const size_t base = i * (2 * jb->n - i - 1) / 2;
        for (size_t j = i + 1; j < jb->n; j++)
            pairwise_one(jb->vs, i, j, &jb->diff[base + j - i - 1], jb->comp ? &jb->comp[base + j - i - 1] : NULL, NULL);
    }
    return NULL;
}

/* The same counts with rows i spread over nthreads threads (the CPU baseline of tools/bench_pairwise.py). */
void pw_pairwise_differences_mt(const pw_variants *vs, size_t sample_count, uint32_t *differences,
                                uint32_t *comparable, int nthreads) {
    if (nthreads < 1) nthreads = 1;
    pairwise_job *jobs = (pairwise_job *)calloc((size_t)nthreads, sizeof(pairwise_job));
    pthread_t *tids = (pthread_t *)calloc((size_t)nthreads, sizeof(pthread_t));
    for (int t = 0; t < nthreads; t++) {
        jobs[t] = (pairwise_job){vs, sample_count, (size_t)t, (size_t)nthreads, differences, comparable};
        pthread_create(&tids[t], NULL, pairwise_worker, &jobs[t]);
    }
    for (int t = 0; t < nthreads; t++) pthread_join(tids[t], NULL);
    free(jobs);
    free(tids);
}
