/*
 * bench_band_update.c -- one EM iteration of cPecanEm with and without --updateTheBand on the flat C-ABI, and the band update by two
 * routes, for tools/bench_band_update.py.  The batch is anchored on the device (standing in for the input cigars' anchors) with cPecanEm's
 * band (trim TRIM, expansion 10, split 3000^2), five-state default model.
 *   iteration without the update: EXPECTATIONS run + fetch of the total;
 *   device update (cpecanResidentBatch_updateAnchors): ALIGNED_PAIRS run, cpb_batch_reweight_pairs(gapGamma), cpb_batch_ordered_chain(0.85),
 *     cpb_batch_anchors_from_alignments (its device-to-host copy of the anchors included);
 *   host route, from the same run: the reference-order lists fetched, reweightAlignedPairs2 + filterPairwiseAlignmentToMakePairsOrdered on
 *     THREADS threads, the cigar of every chain and its anchors (convertPairwiseForwardStrandAlignmentToAnchorPairs + columns_match), then
 *     cpb_batch_create of a new batch with them.
 * Times are medians of REPS iterations after a warm-up, each ending in a synchronising call.  Every pair's anchors are compared.  One JSON
 * line on stdout.
 *
 *   bench_band_update SEQS.bin TRIM THREADS REPS      (SEQS.bin as for bench_decode)
 */
#include <ctype.h>
#include <inttypes.h>
#include <pthread.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>

#include "cpecan/multipleAligner.h"
#include "cpecan/pairwiseAligner.h"
#include "cpecan/pairwiseAlignment.h"
#include "cpecan_b200.h"

stList *cpecan_tripleList_construct(const int32_t *triples, int64_t n); /* host/containers.c */

static double now(void) {
    struct timespec ts;
    clock_gettime(CLOCK_MONOTONIC, &ts);
    return (double) ts.tv_sec + 1e-9 * (double) ts.tv_nsec;
}

static void *read_block(FILE *f, size_t bytes) {
    void *p = malloc(bytes ? bytes : 1);
    if (p == NULL || fread(p, 1, bytes, f) != bytes) {
        fprintf(stderr, "bench_band_update: short read\n");
        exit(2);
    }
    return p;
}

static void check(int rc, const char *what) {
    if (rc != CPB_OK) {
        fprintf(stderr, "bench_band_update: %s: %s\n", what, cpb_last_error());
        exit(1);
    }
}

static int cmp_double(const void *a, const void *b) {
    const double x = *(const double *) a, y = *(const double *) b;
    return x < y ? -1 : (x > y ? 1 : 0);
}

static double median(double *v, int n) {
    qsort(v, (size_t) n, sizeof(double), cmp_double);
    return v[n / 2];
}

typedef struct {
    int64_t n, *xOff, *yOff, trim, expansion;
    const char *seqX, *seqY;
    char **sX, **sY;
    stList **in, **anchors;
    double gapGamma;
    int64_t next;
    pthread_mutex_t lock;
} Work;

/* what cPecanRealign writes for a chain (pairs_to_alignment) and cPecanEm reads back (job_prepare) */
static stList *anchors_of_chain(stList *chain, const char *sX, const char *sY, int64_t lX, int64_t lY, int64_t trim, int64_t expansion) {
    struct List *ops = constructEmptyList(0, (void (*)(void *)) destructAlignmentOperation);
    int64_t pX = -1, pY = -1, run = 0;
    const int64_t n = stList_length(chain);
    for (int64_t i = 0; i <= n; i++) {
        const int64_t x = i < n ? stIntTuple_get(stList_get(chain, i), 1) : lX, y = i < n ? stIntTuple_get(stList_get(chain, i), 2) : lY;
        if (x - pX > 1 || y - pY > 1) {
            if (run > 0) listAppend(ops, constructAlignmentOperation(PAIRWISE_MATCH, run, 0));
            run = 0;
            if (x - pX > 1) listAppend(ops, constructAlignmentOperation(PAIRWISE_INDEL_X, x - pX - 1, 0));
            if (y - pY > 1) listAppend(ops, constructAlignmentOperation(PAIRWISE_INDEL_Y, y - pY - 1, 0));
        }
        run++;
        pX = x;
        pY = y;
    }
    if (run > 1) listAppend(ops, constructAlignmentOperation(PAIRWISE_MATCH, run - 1, 0));
    struct PairwiseAlignment *pA = constructPairwiseAlignment("x", 0, lX, 1, "y", 0, lY, 1, 0.0, ops);
    stList *all = convertPairwiseForwardStrandAlignmentToAnchorPairs(pA, trim, expansion), *kept = stList_construct3(0, (void (*)(void *)) stIntTuple_destruct);
    for (int64_t i = 0; i < stList_length(all); i++) {
        stIntTuple *t = stList_get(all, i);
        const int cx = toupper((unsigned char) sX[stIntTuple_get(t, 0)]), cy = toupper((unsigned char) sY[stIntTuple_get(t, 1)]);
        if (cx == cy && cx != 'N') stList_append(kept, stIntTuple_construct3(stIntTuple_get(t, 0), stIntTuple_get(t, 1), stIntTuple_get(t, 2)));
    }
    stList_destruct(all);
    destructPairwiseAlignment(pA);
    return kept;
}

static void *host_worker(void *arg) {
    Work *w = arg;
    for (;;) {
        pthread_mutex_lock(&w->lock);
        const int64_t i0 = w->next;
        w->next += 64;
        pthread_mutex_unlock(&w->lock);
        if (i0 >= w->n) break;
        const int64_t i1 = i0 + 64 < w->n ? i0 + 64 : w->n;
        for (int64_t i = i0; i < i1; i++) {
            const int64_t lX = w->xOff[i + 1] - w->xOff[i], lY = w->yOff[i + 1] - w->yOff[i];
            stList *chain = filterPairwiseAlignmentToMakePairsOrdered(reweightAlignedPairs2(w->in[i], lX, lY, w->gapGamma), w->sX[i], w->sY[i], 0.85f);
            w->in[i] = NULL; /* consumed */
            w->anchors[i] = anchors_of_chain(chain, w->sX[i], w->sY[i], lX, lY, w->trim, w->expansion);
            stList_destruct(chain);
        }
    }
    return NULL;
}

int main(int argc, char **argv) {
    if (argc < 5) {
        fprintf(stderr, "usage: %s SEQS.bin TRIM THREADS REPS\n", argv[0]);
        return 2;
    }
    FILE *f = fopen(argv[1], "rb");
    if (f == NULL) {
        perror(argv[1]);
        return 2;
    }
    int64_t n;
    if (fread(&n, sizeof(n), 1, f) != 1) return 2;
    int64_t *xOff = read_block(f, (size_t) (n + 1) * 8), *yOff = read_block(f, (size_t) (n + 1) * 8);
    char *seqX = read_block(f, (size_t) xOff[n]), *seqY = read_block(f, (size_t) yOff[n]);
    fclose(f);
    const int threads = atoi(argv[3]), reps = atoi(argv[4]);
    CpbParams p; /* cPecanEm's band */
    cpb_params_default(&p);
    p.constraintDiagonalTrim = atoll(argv[2]);
    p.diagonalExpansion = 10;
    p.splitMatrixBiggerThanThis = (int64_t) 3000 * 3000;
    cpb_context *ctx;
    cpb_batch *b;
    CpbModel m;
    check(cpb_context_create(0, NULL, &ctx), "context");
    check(cpb_model_default(CPB_FIVE_STATE, &m), "model");
    uint8_t *ragged = malloc((size_t) (n > 0 ? n : 1));
    memset(ragged, 1, (size_t) (n > 0 ? n : 1));
    check(cpb_batch_create_anchored(ctx, n, seqX, xOff, seqY, yOff, ragged, ragged, &p, &b), "create");
    fprintf(stderr, "bench_band_update: %" PRIi64 " pairs anchored\n", n);

    /* EM iterations: expectations alone, then expectations + update; the parts of the update */
    double *tExp = malloc((size_t) (reps + 1) * sizeof(double)), *tIt = malloc((size_t) (reps + 1) * sizeof(double));
    double *part[4];
    for (int k = 0; k < 4; k++) part[k] = malloc((size_t) (reps + 1) * sizeof(double));
    double total[CPB_HMM_LEN(5)];
    for (int r = 0; r <= reps; r++) {
        double t0 = now();
        check(cpb_batch_run(b, &m, &p, CPB_MODE_EXPECTATIONS), "expectations");
        check(cpb_batch_fetch_expectations(b, NULL, total), "fetch expectations");
        tExp[r] = 1e3 * (now() - t0);
    }
    int64_t *lOff = malloc((size_t) (n + 1) * 8), cloud = 0;
    int32_t *lTri = NULL;
    double fetchMs = 0.0;
    for (int r = 0; r <= reps; r++) {
        double t0 = now(), t1;
        check(cpb_batch_run(b, &m, &p, CPB_MODE_EXPECTATIONS), "expectations");
        check(cpb_batch_fetch_expectations(b, NULL, total), "fetch expectations");
        const double tE = now();
        check(cpb_batch_run(b, &m, &p, CPB_MODE_ALIGNED_PAIRS), "aligned pairs");
        t1 = now();
        part[0][r] = 1e3 * (t1 - tE);
        if (r == reps) { /* the host route's input, fetched from the same run (not part of the iteration's time) */
            cloud = cpb_batch_result_count(b, 0);
            lTri = malloc((size_t) (cloud > 0 ? cloud : 1) * 12);
            const double f0 = now();
            check(cpb_batch_fetch_pairs_reference_order(b, 0, lOff, lTri), "fetch lists");
            fetchMs = 1e3 * (now() - f0);
            t1 = now();
            t0 += t1 - f0;
        }
        check(cpb_batch_reweight_pairs(b, p.gapGamma), "reweight");
        double t2 = now();
        part[1][r] = 1e3 * (t2 - t1);
        check(cpb_batch_ordered_chain(b, 0.85f), "chain");
        t1 = now();
        part[2][r] = 1e3 * (t1 - t2);
        check(cpb_batch_anchors_from_alignments(b, &p), "anchors from alignments");
        t2 = now();
        part[3][r] = 1e3 * (t2 - t1);
        tIt[r] = 1e3 * (t2 - t0);
    }
    const int64_t nA = cpb_batch_anchor_count(b), nAln = cpb_batch_alignments_count(b);
    int64_t *dOff = malloc((size_t) (n + 1) * 8), *dTri = malloc((size_t) (nA > 0 ? nA : 1) * 24);
    check(cpb_batch_fetch_anchors(b, dOff, dTri), "fetch anchors");
    fprintf(stderr, "bench_band_update: device route done, %" PRIi64 " anchors\n", nA);

    /* host route from the lists of the last run */
    Work w;
    memset(&w, 0, sizeof(w));
    w.n = n;
    w.xOff = xOff;
    w.yOff = yOff;
    w.trim = p.constraintDiagonalTrim;
    w.expansion = p.diagonalExpansion;
    w.gapGamma = p.gapGamma;
    w.sX = malloc((size_t) (n > 0 ? n : 1) * sizeof(char *));
    w.sY = malloc((size_t) (n > 0 ? n : 1) * sizeof(char *));
    w.in = malloc((size_t) (n > 0 ? n : 1) * sizeof(stList *));
    w.anchors = calloc((size_t) (n > 0 ? n : 1), sizeof(stList *));
    for (int64_t i = 0; i < n; i++) {
        const int64_t lX = xOff[i + 1] - xOff[i], lY = yOff[i + 1] - yOff[i];
        w.sX[i] = malloc((size_t) lX + 1);
        w.sY[i] = malloc((size_t) lY + 1);
        memcpy(w.sX[i], seqX + xOff[i], (size_t) lX);
        memcpy(w.sY[i], seqY + yOff[i], (size_t) lY);
        w.sX[i][lX] = w.sY[i][lY] = 0;
    }
    double t0 = now();
    for (int64_t i = 0; i < n; i++) w.in[i] = cpecan_tripleList_construct(lTri + 3 * lOff[i], lOff[i + 1] - lOff[i]);
    const double listsMs = 1e3 * (now() - t0);
    pthread_mutex_init(&w.lock, NULL);
    pthread_t *th = malloc((size_t) threads * sizeof(pthread_t));
    t0 = now();
    for (int t = 0; t < threads; t++) pthread_create(&th[t], NULL, host_worker, &w);
    for (int t = 0; t < threads; t++) pthread_join(th[t], NULL);
    const double hostMs = 1e3 * (now() - t0);
    int64_t *hOff = malloc((size_t) (n + 1) * 8), hA = 0;
    hOff[0] = 0;
    for (int64_t i = 0; i < n; i++) hOff[i + 1] = hOff[i] + stList_length(w.anchors[i]);
    hA = hOff[n];
    int64_t *hTri = malloc((size_t) (hA > 0 ? hA : 1) * 24);
    for (int64_t i = 0; i < n; i++) {
        for (int64_t k = 0; k < stList_length(w.anchors[i]); k++) {
            stIntTuple *t = stList_get(w.anchors[i], k);
            for (int c = 0; c < 3; c++) hTri[3 * (hOff[i] + k) + c] = stIntTuple_get(t, c);
        }
    }
    cpb_batch *h;
    t0 = now();
    check(cpb_batch_create(ctx, n, seqX, xOff, seqY, yOff, hTri, hOff, ragged, ragged, &h), "create");
    const double createMs = 1e3 * (now() - t0);

    int64_t differ = 0, first = -1;
    for (int64_t i = 0; i < n; i++) {
        const int same = dOff[i + 1] - dOff[i] == hOff[i + 1] - hOff[i] && memcmp(dTri + 3 * dOff[i], hTri + 3 * hOff[i], (size_t) (hOff[i + 1] - hOff[i]) * 24) == 0;
        if (!same) {
            differ++;
            if (first < 0) first = i;
        }
    }
    const int64_t tab = (n + 1) * 8;
    /* bytes across the link: the device route copies the alignment and anchor offsets and the anchors back; the host route copies the list
     * back and the sequences, anchors and pair tables of the new batch over */
    const int64_t devBytes = 2 * tab + nA * 12, hostBytes = cloud * 12 + tab + xOff[n] + yOff[n] + hA * 12 + 3 * tab;
    printf("{\"pairs\": %" PRIi64 ", \"trim\": %" PRIi64 ", \"reps\": %d, \"em_iteration_ms\": %.2f, \"em_iteration_with_update_ms\": %.2f, "
           "\"update_ms\": {\"aligned_pairs_run\": %.2f, \"reweight\": %.2f, \"chain\": %.2f, \"anchors_from_alignments\": %.2f}, "
           "\"host_route_ms\": {\"fetch_reference_order\": %.2f, \"lists\": %.2f, \"reweight_chain_anchors\": %.2f, \"create\": %.2f}, "
           "\"host_threads\": %d, \"cloud_triples\": %" PRIi64 ", \"alignment_triples\": %" PRIi64 ", \"anchors\": %" PRIi64 ", "
           "\"device_route_bytes\": %" PRIi64 ", \"host_route_bytes\": %" PRIi64 ", \"pairs_checked\": %" PRIi64 ", \"pairs_differing\": %" PRIi64
           ", \"first_differing\": %" PRIi64 "}\n",
           n, p.constraintDiagonalTrim, reps, median(tExp + 1, reps), median(tIt + 1, reps), median(part[0] + 1, reps), median(part[1] + 1, reps),
           median(part[2] + 1, reps), median(part[3] + 1, reps), fetchMs, listsMs, hostMs, createMs, threads, cloud, nAln, nA, devBytes, hostBytes, n,
           differ, first);
    cpb_batch_destroy(h);
    cpb_batch_destroy(b);
    cpb_context_destroy(ctx);
    return differ != 0;
}
